// Host-side verifier: what `winterfell::verify::<Air>(proof, pub_inputs)` does for the reference
// (/root/reference/src/lib.rs:144-150 and the five sub-AIR examples; SURVEY.md section 8(f).2).  Verification is sequential,
// millisecond-scale host work in the reference too, so it stays on the CPU: it re-uses the product's own AIR descriptors
// (air_desc.cpp), the fused constraint evaluation compiled for the host (airs.cuh), the transcript (transcript.hpp) and
// the hashes (hash.cuh).  Like the prover's transcript it follows the published winterfell v0.3 protocol.
#include <algorithm>
#include <array>
#include <cstring>
#include <vector>

#include "../../../include/csg.h"
#include "../airs.cuh"
#include "air_desc.hpp"
#include "proof_common.hpp"
#include "transcript.hpp"

namespace csg {
using namespace f63;

namespace {
template <int AIR>
fe eval_merged(const AirDesc &air, const TransitionGroups &tg, const std::vector<fe> &cur, const std::vector<fe> &next, const std::vector<fe> &pv,
               const std::vector<fe> &alpha, const std::vector<fe> &beta, const std::vector<fe> &xp) {
    const size_t w = air.width, np = pv.size();
    std::vector<fe> m(2 * w);
    for (size_t c = 0; c < w; c++) { m[2 * c] = cur[c]; m[2 * c + 1] = next[c]; }
    std::vector<uint32_t> off(np + 1), mask(np + 1, 0);
    for (size_t c = 0; c <= np; c++) off[c] = (uint32_t)c;
    std::vector<fe> pvp(pv); pvp.push_back(0);
    airs::Frame f{m.data(), m.data() + 1, 2};
    airs::Periodic Pv{pvp.data(), off.data(), mask.data(), 0};
    airs::Comb C{alpha.data(), beta.data(), tg.group_of.data(), xp.data(), 1, acc192(), nullptr, 0};
    airs::eval_transition<AIR>(f, Pv, C);
    return C.sum.reduce();
}
}  // namespace
// declared in air_desc.hpp: also the host side of trace validation (validate/)
fe eval_merged_any(int id, const AirDesc &air, const TransitionGroups &tg, const std::vector<fe> &cur, const std::vector<fe> &next, const std::vector<fe> &pv,
                   const std::vector<fe> &alpha, const std::vector<fe> &beta, const std::vector<fe> &xp) {
    switch (id) {
    case 0: return eval_merged<0>(air, tg, cur, next, pv, alpha, beta, xp);
    case 1: return eval_merged<1>(air, tg, cur, next, pv, alpha, beta, xp);
    case 2: return eval_merged<2>(air, tg, cur, next, pv, alpha, beta, xp);
    case 3: return eval_merged<3>(air, tg, cur, next, pv, alpha, beta, xp);
    case 4: return eval_merged<4>(air, tg, cur, next, pv, alpha, beta, xp);
    default: return eval_merged<5>(air, tg, cur, next, pv, alpha, beta, xp);
    }
}

namespace {

struct Reader {
    const uint8_t *p; size_t len, off = 0; bool bad = false;
    const uint8_t *take(size_t n) { if (bad || off + n > len) { bad = true; return nullptr; } const uint8_t *q = p + off; off += n; return q; }
    uint64_t uint(int bytes) { const uint8_t *q = take(bytes); uint64_t v = 0; if (q) for (int i = 0; i < bytes; i++) v |= (uint64_t)q[i] << (8 * i); return v; }
    bool element(fe &out) { uint64_t v = uint(8); if (bad || v >= P) { bad = true; return false; } out = to_mont(v); return true; }
};

// in-place natural-order NTT on the host (periodic columns and the FRI remainder: at most a few thousand points, or the
// trace length for Schnorr's per-signature columns)
void host_ntt(std::vector<fe> &a, bool inverse) {
    const size_t n = a.size();
    if (n < 2) return;
    const unsigned l = ilog2_host(n);
    for (size_t i = 0; i < n; i++) {
        size_t j = 0;
        for (unsigned b = 0; b < l; b++) j |= ((i >> b) & 1) << (l - 1 - b);
        if (j > i) std::swap(a[i], a[j]);
    }
    fe w = root_of_unity(l);
    if (inverse) w = inv(w);
    std::vector<fe> tw(n / 2);
    tw[0] = ONE;
    for (size_t i = 1; i < n / 2; i++) tw[i] = mul(tw[i - 1], w);
    for (size_t h = 1; h < n; h <<= 1)
        for (size_t s = 0; s < n; s += 2 * h)
            for (size_t k = 0; k < h; k++) {
                fe u = a[s + k], v = mul(a[s + k + h], tw[k * (n / (2 * h))]);
                a[s + k] = add(u, v); a[s + k + h] = sub(u, v);
            }
    if (inverse) { fe ninv = inv(to_mont(n % P)); for (auto &v : a) v = mul(v, ninv); }
}

// root implied by a batch opening (inverse of batch_opening_nodes): false if the proof is malformed
bool batch_opening_root(int hash_fn, const uint8_t *paths, size_t plen, const std::vector<size_t> &positions, const std::vector<std::array<uint8_t, 32>> &leaves,
                        size_t nleaves, uint8_t root[32]) {
    for (size_t i = 0; i < positions.size(); i++) {
        if (positions[i] >= nleaves) return false;
        for (size_t k = 0; k < i; k++) if (positions[k] == positions[i]) return false;
    }
    std::vector<size_t> idx;
    for (size_t p : positions) idx.push_back(p & ~(size_t)1);
    std::sort(idx.begin(), idx.end());
    idx.erase(std::unique(idx.begin(), idx.end()), idx.end());
    Reader R{paths, plen};
    if (R.uint(1) != idx.size()) return false;
    std::vector<std::vector<std::array<uint8_t, 32>>> slots(idx.size());
    for (auto &s : slots) {
        size_t cnt = R.uint(1);
        for (size_t k = 0; k < cnt; k++) { const uint8_t *d = R.take(32); if (!d) return false; std::array<uint8_t, 32> a; memcpy(a.data(), d, 32); s.push_back(a); }
    }
    if (R.bad || R.off != plen) return false;
    std::vector<size_t> used(idx.size(), 0);
    auto next_node = [&](size_t slot, std::array<uint8_t, 32> &out) { if (used[slot] >= slots[slot].size()) return false; out = slots[slot][used[slot]++]; return true; };
    std::vector<size_t> cur;
    std::vector<std::array<uint8_t, 32>> val;
    for (size_t i = 0; i < idx.size(); i++) {
        uint8_t pair[64];
        for (size_t j = 0; j < 2; j++) {
            auto it = std::find(positions.begin(), positions.end(), idx[i] + j);
            std::array<uint8_t, 32> d;
            if (it != positions.end()) d = leaves[it - positions.begin()];
            else if (!next_node(i, d)) return false;
            memcpy(pair + 32 * j, d.data(), 32);
        }
        std::array<uint8_t, 32> h;
        hashes::hash_bytes(hash_fn, pair, 64, h.data());
        val.push_back(h);
        cur.push_back((nleaves + idx[i]) >> 1);
    }
    const unsigned depth = ilog2_host(nleaves);
    for (unsigned d = 1; d < depth; d++) {
        std::vector<size_t> nxt;
        std::vector<std::array<uint8_t, 32>> nval;
        for (size_t i = 0; i < cur.size(); i++) {
            const size_t node = cur[i], sib = node ^ 1;
            std::array<uint8_t, 32> nv = val[i], sv;
            if (i + 1 < cur.size() && cur[i + 1] == sib) { sv = val[i + 1]; i++; }
            else if (!next_node(i, sv)) return false;
            uint8_t pair[64];
            memcpy(pair, (node & 1) ? sv.data() : nv.data(), 32);
            memcpy(pair + 32, (node & 1) ? nv.data() : sv.data(), 32);
            std::array<uint8_t, 32> h;
            hashes::hash_bytes(hash_fn, pair, 64, h.data());
            nxt.push_back(node >> 1);
            nval.push_back(h);
        }
        cur.swap(nxt); val.swap(nval);
    }
    if (cur.size() != 1 || cur[0] != 1) return false;
    memcpy(root, val[0].data(), 32);
    return true;
}

xe fold_row(int d, const xe v[4], fe x_inv, const xe &alpha, fe zeta_inv, fe quarter) {
    xe s02 = x_add(v[0], v[2]), d02 = x_sub(v[0], v[2]), s13 = x_add(v[1], v[3]), d13 = x_scale(x_sub(v[1], v[3]), zeta_inv);
    xe c[4] = {x_add(s02, s13), x_add(d02, d13), x_sub(s02, s13), x_sub(d02, d13)};
    xe y = x_scale(alpha, x_inv), r = c[3];
    for (int j = 2; j >= 0; j--) r = x_add(x_mul(d, r, y), c[j]);
    return x_scale(r, quarter);
}
xe horner_bx(int d, const std::vector<fe> &c, const xe &x) { xe r = x_zero(); for (size_t i = c.size(); i-- > 0;) r = x_add_base(x_mul(d, r, x), c[i]); return r; }
bool read_x(Reader &R, int d, xe &out) { out = x_zero(); for (int j = 0; j < d; j++) if (!R.element(out.c[j])) return false; return true; }
// the components of E elements in order (hashing and serialisation order)
std::vector<fe> flat(int d, const xe *e, size_t n) {
    std::vector<fe> f;
    for (size_t i = 0; i < n; i++) for (int j = 0; j < d; j++) f.push_back(e[i].c[j]);
    return f;
}
std::vector<fe> flat(int d, const std::vector<xe> &v) { return flat(d, v.data(), v.size()); }
void hash_x(int hf, int d, const xe *e, size_t n, uint8_t out[32]) {
    const std::vector<fe> f = flat(d, e, n);
    hash_elements_host(hf, f.data(), f.size(), out);
}

// Merged transition constraints  sum_i result_i * coef_i  at an E-valued frame, coef_i = alpha_i + beta_i * z^adj in E.
// The AIR evaluation exists over the base field only (airs.cuh).  The frame and the periodic values are polynomials of
// degree < d in the extension generator phi; with phi replaced by a base-field point t every result_i(t) is a base-field
// value, and  S_j(t) = sum_i coef_i[j] * result_i(t)  is a polynomial in t of degree <= D*(d-1) (D the constraint degree).
// K evaluations of the fused base-field code per component j, Newton interpolation, evaluation at phi in E:
// T = sum_j phi^j * S_j(phi).  Returns false if the degree bound K assumes (16 per variable) does not hold.
bool merged_at_ext_frame(int air_id, const AirDesc &air, const TransitionGroups &tg, int d, const std::vector<xe> &cur, const std::vector<xe> &next,
                         const std::vector<xe> &pv, const std::vector<xe> &coef, xe &out) {
    const size_t w = air.width, nc = coef.size(), K = 16 * (size_t)(d - 1) + 1;
    std::vector<fe> zero_beta(nc, 0), xp(tg.adj.size(), ONE);
    std::vector<fe> c(w), nx(w), p1(pv.size()), inv_k(K, 0);
    for (size_t k = 1; k < K; k++) inv_k[k] = inv(to_mont(k));
    std::vector<std::vector<fe>> vals(d, std::vector<fe>(K));
    std::vector<std::vector<fe>> cj(d, std::vector<fe>(nc));
    for (int j = 0; j < d; j++) for (size_t i = 0; i < nc; i++) cj[j][i] = coef[i].c[j];
    for (size_t k = 0; k < K; k++) {
        const fe t = to_mont(k), t2 = sqr(t);
        for (size_t i = 0; i < w; i++) {
            c[i] = add(add(cur[i].c[0], mul(cur[i].c[1], t)), mul(cur[i].c[2], t2));
            nx[i] = add(add(next[i].c[0], mul(next[i].c[1], t)), mul(next[i].c[2], t2));
        }
        for (size_t i = 0; i < pv.size(); i++) p1[i] = add(add(pv[i].c[0], mul(pv[i].c[1], t)), mul(pv[i].c[2], t2));
        for (int j = 0; j < d; j++) vals[j][k] = eval_merged_any(air_id, air, tg, c, nx, p1, cj[j], zero_beta, xp);
    }
    xe phi = x_zero(); phi.c[1] = ONE;
    xe basis = x_one();
    out = x_zero();
    for (int j = 0; j < d; j++) {
        std::vector<fe> &dd = vals[j];
        for (size_t lvl = 1; lvl < K; lvl++)
            for (size_t k = K - 1; k >= lvl; k--) dd[k] = mul(sub(dd[k], dd[k - 1]), inv_k[lvl]);
        if (dd[K - 1] != 0) return false;
        xe r = x_zero();
        for (size_t k = K; k-- > 0;) r = x_add_base(x_mul(d, r, x_sub(phi, x_from(to_mont(k)))), dd[k]);
        out = x_add(out, x_mul(d, basis, r));
        basis = x_mul(d, basis, phi);
    }
    return true;
}

int verify_impl(int air_id, const uint64_t *pub, size_t npub, const uint8_t *proof, size_t proof_len, const csg_options *min_opt) {
    Reader R{proof, proof_len};
    const uint32_t w = (uint32_t)R.uint(1); const unsigned logn = (unsigned)R.uint(1);
    // trace meta: the reference's provers attach none; a non-empty blob would be bytes bound to nothing (proof malleability)
    if (R.uint(2) != 0) return CSG_VERIFY_MALFORMED;
    const size_t modlen = R.uint(1); const uint8_t *mod = R.take(modlen);
    csg_options o;
    o.num_queries = (uint32_t)R.uint(1);
    const size_t log_blowup = R.uint(1);
    o.grinding_factor = (uint32_t)R.uint(1);
    o.hash_fn = (uint32_t)R.uint(1); o.field_extension = (uint32_t)R.uint(1);
    const size_t log_folding = R.uint(1), log_remainder = R.uint(1);
    const size_t context_len = R.off;     // the exact context bytes seed the transcript below
    // the same ranges the prover enforces (prover.cu set_air): blowup 2..32, folding 4, remainder 4..1024, grinding below 32;
    // checked on the log2 bytes BEFORE shifting (a byte >= 32 would be undefined behaviour / wrap to a small value)
    if (R.bad || modlen != 8 || logn < 3 || logn > 40 || log_blowup < 1 || log_blowup > 5 || log_folding != 2 || log_remainder < 2 || log_remainder > 10 ||
        o.grinding_factor >= 32)
        return CSG_VERIFY_MALFORMED;
    o.blowup_factor = 1u << log_blowup; o.fri_folding_factor = 1u << log_folding; o.fri_max_remainder_size = 1u << log_remainder;
    { uint64_t m; memcpy(&m, mod, 8); if (m != P) return CSG_VERIFY_MALFORMED; }
    if (o.field_extension < CSG_FIELD_EXT_NONE || o.field_extension > CSG_FIELD_EXT_CUBIC ||
        (o.hash_fn != CSG_HASH_BLAKE3_256 && o.hash_fn != CSG_HASH_SHA3_256) || o.num_queries == 0)
        return CSG_VERIFY_MALFORMED;
    // acceptance policy of the caller: a proof whose own context is weaker than what the verifier expects is rejected, whatever
    // it proves (winterfell v0.3's verify() trusts the context inside the proof; an acceptance check must not)
    if (min_opt && (o.num_queries < min_opt->num_queries || o.blowup_factor < min_opt->blowup_factor || o.grinding_factor < min_opt->grinding_factor ||
                    o.hash_fn != min_opt->hash_fn || o.field_extension < min_opt->field_extension || o.fri_folding_factor != min_opt->fri_folding_factor ||
                    o.fri_max_remainder_size > min_opt->fri_max_remainder_size))
        return CSG_VERIFY_WEAK_OPTIONS;
    const int d = (int)o.field_extension;
    const ExtConsts xk = d > 1 ? ext_consts() : ExtConsts{};
    const size_t n = (size_t)1 << logn, b = o.blowup_factor, lde_n = n * b, nq = o.num_queries;
    const int hf = (int)o.hash_fn;
    AirDesc air;
    try { air = make_air(air_id, n, pub, npub); } catch (const std::exception &) { return CSG_VERIFY_MALFORMED; }
    if (air.width != w) return CSG_VERIFY_MALFORMED;
    const size_t ce = air.ce_blowup(), nc = air.num_constraints(), na = air.assertions.size();
    if (ce > b) return CSG_VERIFY_MALFORMED;
    try { check_remainder(lde_n, o); } catch (const std::invalid_argument &) { return CSG_VERIFY_MALFORMED; }
    const size_t nfolds = num_fri_folds(lde_n, o), nlayers = nfolds + 1;

    const size_t clen = R.uint(2); const uint8_t *commits = R.take(clen);
    if (R.bad || clen != (2 + nlayers) * 32) return CSG_VERIFY_MALFORMED;
    const size_t tv_len = R.uint(4); const uint8_t *tv = R.take(tv_len); const size_t tp_len = R.uint(4); const uint8_t *tp = R.take(tp_len);
    const size_t cv_len = R.uint(4); const uint8_t *cv = R.take(cv_len); const size_t cp_len = R.uint(4); const uint8_t *cp = R.take(cp_len);
    if (R.bad || tv_len != nq * w * 8 || cv_len != nq * ce * d * 8) return CSG_VERIFY_MALFORMED;
    std::vector<xe> ood_cur(w), ood_next(w), ood_comp(ce);
    if (R.uint(2) != (size_t)w * d * 8) return CSG_VERIFY_MALFORMED;
    for (auto &v : ood_cur) read_x(R, d, v);
    for (auto &v : ood_next) read_x(R, d, v);
    if (R.uint(2) != ce * d * 8) return CSG_VERIFY_MALFORMED;
    for (auto &v : ood_comp) read_x(R, d, v);
    if (R.bad || R.uint(1) != nfolds) return CSG_VERIFY_MALFORMED;
    struct LayerProof { const uint8_t *vals, *paths; size_t vlen, plen; };
    std::vector<LayerProof> lp(nfolds);
    for (auto &l : lp) { l.vlen = R.uint(4); l.vals = R.take(l.vlen); l.plen = R.uint(4); l.paths = R.take(l.plen); }
    const size_t rem_len = R.uint(2); const uint8_t *rem_bytes = R.take(rem_len);
    const size_t nparts = R.uint(1); const uint64_t nonce = R.uint(8);
    if (R.bad || R.off != R.len || nparts != 1) return CSG_VERIFY_MALFORMED;

    try {
        // the transcript, seeded with the exact context bytes of the proof
        ProofTranscript tr(hf, d, pub, npub, proof, context_len);
        const ProofTranscript::ConstraintCoefficients cc = tr.constraint_coefficients(commits, nc, na);
        const xe z = tr.ood_point(commits + 32);

        // out-of-domain consistency: merged constraints at z against the composition columns at z^ce
        const TransitionGroups tg = transition_groups(air);
        const BoundaryGroups bg = boundary_groups(air);
        const fe g = root_of_unity(logn);
        {
            std::vector<xe> pv;
            for (const PeriodicColumn &c : air.periodic) {
                std::vector<fe> poly(c.values);
                host_ntt(poly, true);
                pv.push_back(horner_bx(d, poly, x_pow(d, z, n / poly.size())));
            }
            std::vector<xe> xp;
            for (uint64_t adj : tg.adj) xp.push_back(x_pow(d, z, adj));
            xe t;
            if (d == 1) {
                std::vector<fe> c1, n1, p1, a1, b1, x1;
                for (auto &v : ood_cur) c1.push_back(v.c[0]);
                for (auto &v : ood_next) n1.push_back(v.c[0]);
                for (auto &v : pv) p1.push_back(v.c[0]);
                for (size_t i = 0; i < nc; i++) { a1.push_back(cc.transition[2 * i].c[0]); b1.push_back(cc.transition[2 * i + 1].c[0]); }
                for (auto &v : xp) x1.push_back(v.c[0]);
                t = x_from(eval_merged_any(air_id, air, tg, c1, n1, p1, a1, b1, x1));
            } else {
                std::vector<xe> coef(nc);
                for (size_t i = 0; i < nc; i++) coef[i] = x_add(cc.transition[2 * i], x_mul(d, cc.transition[2 * i + 1], xp[tg.group_of[i]]));
                if (!merged_at_ext_frame(air_id, air, tg, d, ood_cur, ood_next, pv, coef, t)) return CSG_VERIFY_MALFORMED;
            }
            xe lhs = x_mul(d, x_mul(d, t, x_sub(z, x_from(f63::pow(g, n - 1)))), x_inv(d, x_sub(x_pow(d, z, n), x_one()), xk));
            const fe g_inv = inv(g);
            size_t a = 0;
            for (size_t gi = 0; gi < bg.groups.size(); gi++) {
                const BoundaryGroup &G = bg.groups[gi];
                const xe xpb = x_pow(d, z, G.adj);
                xe acc = x_zero();
                for (; a < na && bg.group_of[a] == gi; a++) {
                    const Assertion &s = air.assertions[a];
                    xe v = x_from(s.values[0]);
                    if (s.values.size() > 1) {
                        std::vector<fe> poly(s.values);
                        host_ntt(poly, true);
                        v = horner_bx(d, poly, s.first_step ? x_scale(z, f63::pow(g_inv, s.first_step)) : z);
                    }
                    acc = x_add(acc, x_mul(d, x_sub(ood_cur[s.column], v), x_add(cc.boundary[2 * a], x_mul(d, cc.boundary[2 * a + 1], xpb))));
                }
                lhs = x_add(lhs, x_mul(d, acc, x_inv(d, x_sub(x_pow(d, z, G.num_steps), x_from(G.offset)), xk)));
            }
            xe rhs = x_zero(), zp = x_one();
            for (size_t r = 0; r < ce; r++) { rhs = x_add(rhs, x_mul(d, zp, ood_comp[r])); zp = x_mul(d, zp, z); }
            if (!x_eq(lhs, rhs)) return CSG_VERIFY_OOD_MISMATCH;
        }
        const ProofTranscript::DeepCoefficients dc = tr.deep_coefficients(flat(d, ood_cur).data(), flat(d, ood_next).data(), w, flat(d, ood_comp).data(), ce);
        std::vector<xe> alphas(nlayers);
        for (size_t l = 0; l < nlayers; l++) alphas[l] = tr.fri_alpha(commits + (2 + l) * 32);
        if (!tr.accept_nonce(nonce, o.grinding_factor)) return CSG_VERIFY_POW;
        const std::vector<size_t> pos = tr.query_positions(nq, lde_n);

        // openings against both commitments
        std::vector<fe> t_rows(nq * w);
        std::vector<xe> c_rows(nq * ce);
        {
            Reader T{tv, tv_len}, Cq{cv, cv_len};
            std::vector<std::array<uint8_t, 32>> lh(nq);
            uint8_t root[32];
            for (size_t i = 0; i < nq; i++) { for (size_t c = 0; c < w; c++) T.element(t_rows[i * w + c]); hash_elements_host(hf, &t_rows[i * w], w, lh[i].data()); }
            if (T.bad || !batch_opening_root(hf, tp, tp_len, pos, lh, lde_n, root) || memcmp(root, commits, 32)) return CSG_VERIFY_TRACE_QUERY;
            for (size_t i = 0; i < nq; i++) { for (size_t r = 0; r < ce; r++) read_x(Cq, d, c_rows[i * ce + r]); hash_x(hf, d, &c_rows[i * ce], ce, lh[i].data()); }
            if (Cq.bad || !batch_opening_root(hf, cp, cp_len, pos, lh, lde_n, root) || memcmp(root, commits + 32, 32)) return CSG_VERIFY_CONSTRAINT_QUERY;
        }
        // DEEP composition at the queried points
        std::vector<xe> evals(nq);
        {
            const fe offset = to_mont(GENERATOR), g_lde = root_of_unity(ilog2_host(lde_n));
            const xe zg = x_scale(z, g), zm = x_pow(d, z, ce);
            for (size_t i = 0; i < nq; i++) {
                const fe xb = mul(offset, f63::pow(g_lde, pos[i]));
                const xe x = x_from(xb);
                xe a = x_zero(), bsum = x_zero(), csum = x_zero();
                for (size_t c = 0; c < w; c++) {
                    const xe tv1 = x_from(t_rows[i * w + c]);
                    a = x_add(a, x_mul(d, dc.trace[2 * c], x_sub(tv1, ood_cur[c])));
                    bsum = x_add(bsum, x_mul(d, dc.trace[2 * c + 1], x_sub(tv1, ood_next[c])));
                }
                for (size_t r = 0; r < ce; r++) csum = x_add(csum, x_mul(d, dc.comp[r], x_sub(c_rows[i * ce + r], ood_comp[r])));
                const xe s = x_add(x_add(x_mul(d, a, x_inv(d, x_sub(x, z), xk)), x_mul(d, bsum, x_inv(d, x_sub(x, zg), xk))), x_mul(d, csum, x_inv(d, x_sub(x, zm), xk)));
                evals[i] = x_mul(d, s, x_add(dc.lambda, x_scale(dc.mu, xb)));
            }
        }
        // FRI
        std::vector<size_t> p1 = pos;
        size_t domain = lde_n, max_deg_plus_1 = n;
        const fe off_inv = inv(to_mont(GENERATOR)), quarter = inv(to_mont(4));
        for (size_t l = 0; l < nfolds; l++) {
            const size_t q = domain / 4;
            const std::vector<size_t> p2 = fold_positions(p1, domain);
            const fe ginv = inv(root_of_unity(ilog2_host(domain))), zeta_inv = f63::pow(ginv, q);
            if (lp[l].vlen != p2.size() * 4 * d * 8) return CSG_VERIFY_FRI;
            std::vector<xe> vals(p2.size() * 4);
            std::vector<std::array<uint8_t, 32>> lh(p2.size());
            Reader V{lp[l].vals, lp[l].vlen};
            for (size_t i = 0; i < p2.size(); i++) { for (int k = 0; k < 4; k++) read_x(V, d, vals[i * 4 + k]); hash_x(hf, d, &vals[i * 4], 4, lh[i].data()); }
            uint8_t root[32];
            if (V.bad || !batch_opening_root(hf, lp[l].paths, lp[l].plen, p2, lh, q, root) || memcmp(root, commits + (2 + l) * 32, 32)) return CSG_VERIFY_FRI;
            for (size_t i = 0; i < p1.size(); i++) {
                const size_t row = std::find(p2.begin(), p2.end(), p1[i] % q) - p2.begin();
                if (!x_eq(vals[row * 4 + p1[i] / q], evals[i])) return CSG_VERIFY_FRI;
            }
            std::vector<xe> folded(p2.size());
            for (size_t i = 0; i < p2.size(); i++) folded[i] = fold_row(d, &vals[i * 4], mul(off_inv, f63::pow(ginv, p2[i])), alphas[l], zeta_inv, quarter);
            if (max_deg_plus_1 % 4) return CSG_VERIFY_FRI;
            max_deg_plus_1 /= 4; domain = q; p1 = p2; evals = folded;
        }
        if (rem_len != domain * d * 8) return CSG_VERIFY_MALFORMED;
        std::vector<xe> rem(domain);
        { Reader Q{rem_bytes, rem_len}; for (auto &v : rem) read_x(Q, d, v); if (Q.bad) return CSG_VERIFY_MALFORMED; }
        {
            const size_t q = domain / 4;
            std::vector<uint8_t> nodes(2 * q * 32);
            for (size_t i = 0; i < q; i++) { xe row[4] = {rem[i], rem[i + q], rem[i + 2 * q], rem[i + 3 * q]}; hash_x(hf, d, row, 4, &nodes[(q + i) * 32]); }
            for (size_t i = q - 1; i >= 1; i--) hashes::hash_bytes(hf, &nodes[2 * i * 32], 64, &nodes[i * 32]);
            if (memcmp(&nodes[32], commits + (2 + nfolds) * 32, 32)) return CSG_VERIFY_FRI;
        }
        for (size_t i = 0; i < p1.size(); i++) if (!x_eq(rem[p1[i]], evals[i])) return CSG_VERIFY_FRI;
        if (max_deg_plus_1 - 1 >= domain - 1) return CSG_VERIFY_FRI;
        for (int j = 0; j < d; j++) {   // degree check component by component
            std::vector<fe> comp(domain);
            for (size_t i = 0; i < domain; i++) comp[i] = rem[i].c[j];
            host_ntt(comp, true);
            for (size_t i = max_deg_plus_1; i < domain; i++) if (comp[i] != 0) return CSG_VERIFY_FRI;
        }
    } catch (const std::exception &) { return CSG_VERIFY_MALFORMED; }
    return CSG_OK;
}
}  // namespace
}  // namespace csg

extern "C" int csg_verify(int air_id, const uint64_t *pub, size_t npub, const uint8_t *proof, size_t proof_len) {
    if (!pub || !proof) return CSG_VERIFY_MALFORMED;
    return csg::verify_impl(air_id, pub, npub, proof, proof_len, nullptr);
}
extern "C" int csg_verify_with_options(int air_id, const uint64_t *pub, size_t npub, const uint8_t *proof, size_t proof_len, const csg_options *min_options) {
    if (!pub || !proof || !min_options) return CSG_VERIFY_MALFORMED;
    return csg::verify_impl(air_id, pub, npub, proof, proof_len, min_options);
}
