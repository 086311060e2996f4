// The batch driver of csg_prove_many (many.cuh): Prover::prove for K independent traces of one AIR, one length and one set of
// options, stage by stage as csg_ctx::prove_loaded runs it, with every stage one launch sequence over all K proofs
// (many_kernels.cuh) and every step of the Fiat-Shamir transcript one device->host copy for the whole batch.  The K transcripts run
// on the host, one Coin per proof, spread over the host threads; a proof's transcript depends on nothing but its own trace and
// public inputs, so the bytes do not depend on the thread count.
//
// Unlike the single-proof driver this one has no low-degree split, no sharding, no extension fields, no chunked or prefetched
// copies: a batch is many short traces, where launches and round trips, not arithmetic, set the time.
#include <algorithm>
#include <array>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../constraints.cuh"
#include "../host/air_desc.hpp"
#include "../host/proof_common.hpp"
#include "../host/transcript.hpp"
#include "../ntt.cuh"
#include "../stages.cuh"
#include "many.cuh"
#include "many_kernels.cuh"

namespace csg {
using namespace f63;

namespace {

// page-locked host staging, grow-only (the traces and the constraint arguments go up in one copy each)
template <class T>
struct PinnedBuf {
    T *p = nullptr;
    size_t n = 0;
    ~PinnedBuf() { if (p) cudaFreeHost(p); }
    void reserve(size_t count) {
        if (count <= n) return;
        if (p) cudaFreeHost(p);
        p = nullptr; n = 0;
        CSG_CUDA(cudaHostAlloc((void **)&p, count * sizeof(T), cudaHostAllocDefault));
        n = count;
    }
};

// runs f(k) for k < count on the host threads; the first exception is rethrown on the calling thread.  Small batches stay on the
// calling thread: a parallel region wakes every host thread, and on a busy host one late thread holds up the region by milliseconds
// (one Rescue proof: 4-23 ms in the first region of a batch against 0.2 ms of work); from 32 proofs on the threads pay
template <class F>
void parallel_proofs(size_t count, F f) {
    std::string err;
    bool arg = false, failed = false;
#pragma omp parallel for schedule(dynamic, 4) if (count >= 32)
    for (long k = 0; k < (long)count; k++) {
        try { f((size_t)k); }
        catch (const std::invalid_argument &e) {
#pragma omp critical
            { if (!failed) { failed = true; arg = true; err = e.what(); } }
        } catch (const std::exception &e) {
#pragma omp critical
            { if (!failed) { failed = true; err = e.what(); } }
        }
    }
    if (failed) { if (arg) throw std::invalid_argument(err); throw std::runtime_error(err); }
}

// what one proof of the batch carries through the stages
struct ProofState {
    Coin coin;
    uint8_t trace_root[32], comp_root[32];
    std::vector<std::array<uint8_t, 32>> fri_roots;
    fe z = 0;
    std::vector<fe> ood_cur, ood_next, ood_comp;
    uint64_t nonce = 0;
    std::vector<size_t> pos;
    // openings, planned with offsets local to the proof
    std::vector<uint32_t> idx;
    std::vector<RowJob> rjobs;
    std::vector<DigestJob> djobs;
    Opening o_trace, o_comp;
    std::vector<Opening> o_fri;
    size_t rows_words = 0, dig_count = 0, rem_off = 0, rem_len = 0;
    size_t idx_base = 0, rows_base = 0, dig_base = 0;
    explicit ProofState(Coin c) : coin(std::move(c)) {}
};

size_t ntt_group_tmp(size_t ncols, size_t ncosets, size_t n) {   // the pass-A scratch of coset_ntt_columns (ntt.cu)
    size_t group = ncosets;
    while (group > 1 && group * ncols * n > ((size_t)1 << 29)) group = (group + 1) / 2;
    return group * ncols * n;
}

}  // namespace

class ManyProver {
  public:
    ~ManyProver() { for (auto e : ev) if (e) cudaEventDestroy(e); for (auto e : ev_cargs) if (e) cudaEventDestroy(e); }
    void prove(Stream &st, int air_id, size_t K, ManyTraces traces, int repr, size_t trace_len, const uint64_t *pubs, size_t npub,
               const csg_options *o, uint8_t **proofs, size_t *proof_lens, csg_timings &tm);

  private:
    // shape of the device tables below
    size_t n = 0, b = 0;
    unsigned logn = 0;
    RootTable roots;
    NttScratch ntt;
    CosetTables lde_tables;
    std::vector<fe> lde_shift;

    DBuf<uint64_t> d_io, d_out;
    DBuf<fe> d_polys, d_lde, d_pvals, d_pcoef, d_ptab, d_apoly, d_part, d_binv, d_comb, d_e, d_cpolys, d_clde, d_abc, d_abc_lde, d_deep, d_args, d_partial;
    DBuf<uint32_t> d_tnodes, d_cnodes, d_idx;
    DBuf<ConsArgs> d_cargs;
    DBuf<DeepArgs> d_dargs;
    DBuf<RowJob> d_rjobs;
    DBuf<DigestJob> d_djobs;
    std::vector<std::unique_ptr<DBuf<fe>>> fri_evals;         // layers 1.. ([proof][m]); layer 0 is d_deep
    std::vector<std::unique_ptr<DBuf<uint32_t>>> fri_nodes;   // [proof][16 * m/4]
    PinnedBuf<uint64_t> h_io;
    PinnedBuf<ConsArgs> h_cargs;
    cudaEvent_t ev[9] = {}, ev_cargs[2] = {};   // stage boundaries; the upload of the constraint arguments (CSG_HOST_TRACE)
    ManyWitnessScratch wit;                     // the batch witness builders' (witness_many.cu); prove does not use it
    friend ManyWitnessScratch &many_scratch(ManyProver *m);

    size_t held_bytes() const {
        size_t s = d_io.n * 8 + d_out.n * 8 + (d_tnodes.n + d_cnodes.n + d_idx.n) * 4 + d_cargs.n * sizeof(ConsArgs) + d_dargs.n * sizeof(DeepArgs) +
                   d_rjobs.n * sizeof(RowJob) + d_djobs.n * sizeof(DigestJob) + ntt.tmp.n * 8;
        for (const DBuf<fe> *p : {&d_polys, &d_lde, &d_pvals, &d_pcoef, &d_ptab, &d_apoly, &d_part, &d_binv, &d_comb, &d_e, &d_cpolys, &d_clde, &d_abc, &d_abc_lde, &d_deep, &d_args, &d_partial})
            s += p->n * 8;
        for (auto &f : fri_evals) s += f->n * 8;
        for (auto &f : fri_nodes) s += f->n * 4;
        return s;
    }
};

ManyProver *many_new() { return new ManyProver(); }
void many_delete(ManyProver *m) { delete m; }
ManyWitnessScratch &many_scratch(ManyProver *m) { return m->wit; }

void check_device_buffer(const void *p, const char *what) {
    int device = 0;
    CSG_CUDA(cudaGetDevice(&device));
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); a.type = cudaMemoryTypeUnregistered; }
    if (a.type != cudaMemoryTypeDevice || a.device != device)
        throw ManyArgError(std::string(what) + " must be device memory of the context's device (not host, pinned host or managed memory)");
}

void many_prove(ManyProver *m, Stream &st, int air_id, size_t count, ManyTraces traces, int repr, size_t trace_len, const uint64_t *pubs,
                size_t npub, const csg_options *opt, uint8_t **proofs, size_t *proof_lens, csg_timings &tm) {
    m->prove(st, air_id, count, traces, repr, trace_len, pubs, npub, opt, proofs, proof_lens, tm);
}

void ManyProver::prove(Stream &st, int air_id, size_t K, ManyTraces traces, int repr, size_t trace_len, const uint64_t *pubs, size_t npub,
                       const csg_options *o, uint8_t **proofs, size_t *proof_lens, csg_timings &tm) {
    const auto t0 = std::chrono::steady_clock::now();
    static const bool host_trace = getenv("CSG_HOST_TRACE") != nullptr;
    HostTrace trace{t0, {}};
    struct TraceScope { bool on; TraceScope(bool o_, HostTrace *t) : on(o_) { if (on) g_host_trace = t; } ~TraceScope() { if (on) g_host_trace = nullptr; } } trace_scope(host_trace, &trace);

    // ------------------------------------------------------------------ every check before anything is enqueued
    if ((!traces.host && !traces.dev) || !pubs || !proofs || !proof_lens) throw ManyArgError("null argument");
    if (K == 0 || K > MANY_MAX_COUNT) throw ManyArgError("count must be in 1..1024");
    for (size_t k = 0; k < K; k++) { proofs[k] = nullptr; proof_lens[k] = 0; }
    try { check_options(o); } catch (const std::invalid_argument &e) { throw ManyArgError(e.what()); }
    if (o->field_extension != CSG_FIELD_EXT_NONE) throw ManyUnsupported("csg_prove_many proves over the base field only (field_extension 1)");
    if (trace_len > ((size_t)1 << MANY_MAX_LOG_TRACE)) throw ManyUnsupported("csg_prove_many takes traces of at most 2^16 rows: prove longer ones with csg_prove");
    if (repr != CSG_REPR_CANONICAL && repr != CSG_REPR_MONTGOMERY) throw ManyArgError("repr must be CSG_REPR_CANONICAL or CSG_REPR_MONTGOMERY");
    if (traces.host) { for (size_t k = 0; k < K; k++) if (!traces.host[k]) throw ManyArgError("null trace"); }
    else check_device_buffer(traces.dev, "the traces");
    std::vector<AirDesc> airs(K);
    try { parallel_proofs(K, [&](size_t k) { airs[k] = make_air(air_id, trace_len, pubs + k * npub, npub); }); }
    catch (const std::invalid_argument &e) { throw ManyArgError(e.what()); }
    const AirDesc &air = airs[0];
    const size_t w = air.width, nb = o->blowup_factor, ce = air.ce_blowup(), lde_n = trace_len * nb, nc = air.num_constraints(), na = air.assertions.size();
    if (K * w > MANY_MAX_COLUMNS) throw ManyArgError("count * trace width must not exceed 65535");
    if (ce > nb) throw ManyArgError("blowup factor is smaller than the constraint evaluation blowup of this AIR");
    try { check_remainder(lde_n, *o); } catch (const std::invalid_argument &e) { throw ManyArgError(e.what()); }
    if (nc > (size_t)CONS_MAX_CONSTRAINTS || air.periodic.size() > (size_t)CONS_MAX_PERIODIC || na > (size_t)CONS_MAX_ASSERTIONS)
        throw ManyArgError("AIR exceeds the compiled table sizes");
    const TransitionGroups tg = transition_groups(air);
    const BoundaryGroups bg = boundary_groups(air);
    if (tg.adj.size() > (size_t)CONS_MAX_GROUPS || bg.groups.size() > (size_t)CONS_MAX_BGROUPS) throw ManyArgError("too many constraint groups");
    const unsigned lg = ilog2(trace_len);
    const size_t nfold = num_fri_folds(lde_n, *o), nlayers = nfold + 1, nq = o->num_queries;
    // periodic columns: runs of equal period go through the transforms together; proof k's copy of column c of run [c0, c1) of period
    // P sits at K * off(c0) + (k * (c1 - c0) + c - c0) * P of each ce coset's block of K * total elements
    struct Run { size_t c0, c1, P, off; };
    std::vector<Run> runs;
    size_t ptotal = 0;
    for (size_t c = 0; c < air.periodic.size();) {
        const size_t P = air.periodic[c].values.size();
        if (P == 0 || (P & (P - 1)) || P > trace_len) throw ManyArgError("periodic column length must be a power of two dividing the trace length");
        size_t c1 = c;
        while (c1 < air.periodic.size() && air.periodic[c1].values.size() == P) c1++;
        runs.push_back({c, c1, P, ptotal});
        ptotal += (c1 - c) * P;
        c = c1;
    }
    size_t npoly = 0;   // coefficients of the assertion sequences of one proof
    for (const Assertion &s : air.assertions) if (s.values.size() > 1) npoly += s.values.size();
    const size_t items = constraint_items_many(air_id);
    // the device footprint of the batch, from the shapes alone
    size_t layer_elems = 0, layer_nodes = 0, open_words = 0;
    for (size_t l = 0, mm = lde_n; l < nlayers; l++, mm /= 4) { if (l) layer_elems += K * mm; layer_nodes += K * 16 * (mm / 4); }
    {
        unsigned depth = ilog2(lde_n);
        open_words = K * ((nq * (w + ce + 4 * nfold) + 1024) + 8 * nq * depth * (2 + nfold) / 2 + 8);
    }
    const size_t tmp = std::max({lg > 11 ? ntt_group_tmp(K * w, nb, trace_len) : 0, lg > 11 ? ntt_group_tmp(K * ce, nb, trace_len) : 0,
                                 lg > 11 ? ntt_group_tmp(3 * K, nb, trace_len) : 0, K * w * trace_len, K * ce * trace_len});
    const size_t staged = traces.host ? K * w * trace_len : 0;   // d_io: host traces go up into it, device traces are read in place
    const size_t need = 8 * (staged + K * w * trace_len + nb * K * w * trace_len + K * ptotal * (2 + ce) + K * npoly + K * items * ce * trace_len +
                             CONS_MAX_BGROUPS * ce * trace_len + 3 * K * ce * trace_len + nb * K * ce * trace_len + 3 * K * trace_len * (1 + nb) +
                             K * lde_n + layer_elems + tmp + 2 * open_words + K * 8 * (2 * w + ce)) +
                        4 * (2 * K * 16 * lde_n + layer_nodes + open_words) + K * (sizeof(ConsArgs) + sizeof(DeepArgs));
    {
        size_t free_b = 0, total_b = 0;
        CSG_CUDA(cudaMemGetInfo(&free_b, &total_b));
        const size_t held = held_bytes();
        if (need > free_b + held) {
            char msg[200];
            snprintf(msg, sizeof msg, "the batch needs %.2f GB of device memory, %.2f GB are available", need / 1e9, (free_b + held) / 1e9);
            throw ManyArgError(msg);
        }
    }
    host_mark("checks");

    // ------------------------------------------------------------------ domain tables (kept while the shape stays)
    const int hf = (int)o->hash_fn;
    const fe g = root_of_unity(lg);
    if (trace_len != n || nb != b) {
        n = 0;   // until the tables below are complete
        roots.build(lg, st);
        const fe offset = to_mont(GENERATOR), w_lde = root_of_unity(ilog2(lde_n));
        lde_shift.assign(nb, 0);
        fe acc = offset;
        for (size_t k = 0; k < nb; k++) { lde_shift[k] = acc; acc = mul(acc, w_lde); }
        lde_tables.build(lde_shift.data(), nb, lg, st);
        n = trace_len; b = nb; logn = lg;
    }
    std::vector<fe> ce_shift(ce);
    for (size_t kc = 0; kc < ce; kc++) ce_shift[kc] = lde_shift[kc * (b / ce)];
    for (auto &e : ev) if (!e) CSG_CUDA(cudaEventCreate(&e));
    for (auto &e : ev_cargs) if (!e) CSG_CUDA(cudaEventCreate(&e));
    const unsigned long long launches0 = st.launches;
    unsigned long long lmark = launches0;
    auto stage_launches = [&](int s) { tm.stage_launches[s] = (uint32_t)(st.launches - lmark); lmark = st.launches; };
    tm = csg_timings{};

    std::vector<ProofState> ps;
    ps.reserve(K);
    for (size_t k = 0; k < K; k++) {
        Bytes seed;
        for (uint64_t v : airs[k].pub_inputs) seed.u64(v);
        write_proof_context(seed, (unsigned)w, lg, *o);
        ps.emplace_back(Coin(hf, seed.v.data(), seed.v.size()));
    }

    // ------------------------------------------------------------------ stage 1: traces up, periodic tables, LDE
    CSG_CUDA(cudaEventRecord(ev[0], st.s));
    const size_t tw = w * n;
    const uint64_t *src = traces.dev;
    if (traces.host) {
        h_io.reserve(K * tw);
        d_io.reserve(K * tw);
        parallel_proofs(K, [&](size_t k) { memcpy(h_io.p + k * tw, traces.host[k], tw * sizeof(uint64_t)); });
        CSG_CUDA(cudaMemcpyAsync(d_io.p, h_io.p, K * tw * sizeof(uint64_t), cudaMemcpyHostToDevice, st.s));
        src = d_io.p;
    }
    CSG_CUDA(cudaEventRecord(ev[1], st.s));
    host_mark("traces up");
    if (ptotal) {
        std::vector<fe> pv(K * ptotal);
        parallel_proofs(K, [&](size_t k) {
            for (const Run &r : runs)
                for (size_t c = r.c0; c < r.c1; c++)
                    memcpy(&pv[K * r.off + (k * (r.c1 - r.c0) + c - r.c0) * r.P], airs[k].periodic[c].values.data(), r.P * sizeof(fe));
        });
        d_pvals.reserve(K * ptotal); d_pcoef.reserve(K * ptotal); d_ptab.reserve(K * ptotal * ce);
        CSG_CUDA(cudaMemcpyAsync(d_pvals.p, pv.data(), pv.size() * sizeof(fe), cudaMemcpyHostToDevice, st.s));
        for (const Run &r : runs) {
            const size_t cols = K * (r.c1 - r.c0);
            intt_columns(roots, ntt, d_pvals.p + K * r.off, r.P, d_pcoef.p + K * r.off, r.P, cols, ilog2(r.P), st);
            std::vector<fe> shifts(ce);
            for (size_t kc = 0; kc < ce; kc++) shifts[kc] = f63::pow(ce_shift[kc], n / r.P);
            coset_ntt_columns(roots, ntt, d_pcoef.p + K * r.off, r.P, d_ptab.p + K * r.off, r.P, K * ptotal, cols, ilog2(r.P), shifts.data(), ce, st);
        }
    } else d_ptab.reserve(1);
    d_polys.reserve(K * tw); d_lde.reserve(b * K * tw);
    // the representation change rides on the 1/n scaling of the interpolation (as in csg_ctx::extend_and_commit_trace); intt_columns
    // writes only its output and its scratch, so a caller's device buffer is read in place
    intt_columns(roots, ntt, src, n, d_polys.p, n, K * w, logn, st, repr == CSG_REPR_MONTGOMERY ? 0 : R2, true);
    coset_ntt_columns(roots, ntt, d_polys.p, n, d_lde.p, n, K * tw, K * w, logn, lde_tables, st);
    CSG_CUDA(cudaEventRecord(ev[2], st.s));
    stage_launches(0);

    // ------------------------------------------------------------------ stage 2: trace commitments
    auto commit = [&](const fe *data, unsigned width, size_t coset_stride, size_t proof_stride, DBuf<uint32_t> &nodes, size_t nleaves, unsigned ncosets,
                      size_t rows, std::vector<std::array<uint8_t, 32>> &out) {
        const size_t tree = 16 * nleaves;
        nodes.reserve(K * tree);
        hash_rows_many(data, width, rows, ncosets, coset_stride, rows, proof_stride, K, hf, nodes.p + 8 * nleaves, tree, st);
        merkle_build_many(nodes.p, nleaves, K, tree, hf, st);
        out.resize(K);
        CSG_CUDA(cudaMemcpy2DAsync(out.data(), 32, nodes.p + 8, tree * 4, 32, K, cudaMemcpyDeviceToHost, st.s));
    };
    std::vector<std::array<uint8_t, 32>> roots_h;
    d_tnodes.reserve(K * 16 * lde_n);
    commit(d_lde.p, (unsigned)w, K * tw, tw, d_tnodes, lde_n, (unsigned)b, n, roots_h);
    CSG_CUDA(cudaEventRecord(ev[3], st.s));
    CSG_CUDA(cudaStreamSynchronize(st.s));
    stage_launches(1);
    host_mark("trace roots");

    // ------------------------------------------------------------------ stage 3: constraint coefficients and evaluation
    h_cargs.reserve(K);
    ConsArgs *T = h_cargs.p;
    {   // proof 0 carries everything that depends on the AIR and the domain only; the others start from a copy
        ConsArgs &A = T[0];
        memset(&A, 0, sizeof A);
        A.ext_degree = 1;
        A.logn = logn; A.ncosets = (unsigned)ce; A.col_stride = n; A.width = (unsigned)w;
        A.g_last = f63::pow(g, n - 1);
        A.nconstraints = (unsigned)nc; A.ngroups = (unsigned)tg.adj.size();
        for (size_t i = 0; i < nc; i++) A.group[i] = tg.group_of[i];
        for (size_t gi = 0; gi < tg.adj.size(); gi++) A.adj_mod[gi] = tg.adj[gi] % n;
        A.nbgroups = (unsigned)bg.groups.size(); A.nassertions = (unsigned)na;
        for (size_t gi = 0; gi < bg.groups.size(); gi++) { A.b_adj_mod[gi] = bg.groups[gi].adj % n; A.b_steps[gi] = bg.groups[gi].num_steps; A.b_offset[gi] = bg.groups[gi].offset; }
        for (size_t kc = 0; kc < ce; kc++) {
            const fe s = ce_shift[kc];
            A.lde_coset_stride[kc] = (unsigned long long)(kc * (b / ce)) * K * tw;
            A.shift[kc] = s;
            A.zinv[kc] = inv(sub(f63::pow(s, n), ONE));
            for (size_t gi = 0; gi < tg.adj.size(); gi++) A.shift_adj[kc][gi] = f63::pow(s, tg.adj[gi]);
            for (size_t gi = 0; gi < bg.groups.size(); gi++) { A.b_shift_adj[kc][gi] = f63::pow(s, bg.groups[gi].adj); A.b_shift_steps[kc][gi] = f63::pow(s, bg.groups[gi].num_steps); }
        }
        const fe g_inv = inv(g);
        for (size_t i = 0; i < na; i++) {
            const Assertion &s = air.assertions[i];
            A.a_col[i] = s.column; A.a_group[i] = bg.group_of[i];
            A.a_poly_len[i] = (unsigned)s.values.size();
            A.a_xoff[i] = s.first_step ? f63::pow(g_inv, s.first_step) : ONE;
        }
        A.nperiodic = (unsigned)air.periodic.size();
        A.ptab_coset_stride = K * ptotal;
        for (const Run &r : runs) for (size_t c = r.c0; c < r.c1; c++) A.pmask[c] = (unsigned)(r.P - 1);
    }
    std::vector<fe> apoly(std::max<size_t>(K * npoly, 1));
    parallel_proofs(K, [&](size_t k) {
        ProofState &p = ps[k];
        p.coin.reseed(roots_h[k].data());
        memcpy(p.trace_root, roots_h[k].data(), 32);
        ConsArgs &A = T[k];
        if (k) memcpy(&A, &T[0], sizeof A);
        for (size_t i = 0; i < nc; i++) { A.alpha[i] = p.coin.draw(); A.beta[i] = p.coin.draw(); }
        for (size_t i = 0; i < na; i++) { A.a_alpha[i] = p.coin.draw(); A.a_beta[i] = p.coin.draw(); }
        fill_rescue_tables(air_id, A);
        size_t po = k * npoly;
        for (size_t i = 0; i < na; i++) {
            const Assertion &s = airs[k].assertions[i];
            A.a_value[i] = s.values[0];
            A.a_poly_off[i] = po;
            if (s.values.size() > 1) {
                const std::vector<fe> c = interpolate_host(s.values);
                std::copy(c.begin(), c.end(), apoly.begin() + po);
                po += c.size();
            }
        }
        for (const Run &r : runs) for (size_t c = r.c0; c < r.c1; c++) A.poff[c] = (unsigned)(K * r.off + (k * (r.c1 - r.c0) + c - r.c0) * r.P);
    });
    host_mark("draw coefficients, constraint arguments");
    d_cargs.reserve(K); d_apoly.reserve(apoly.size());
    CSG_CUDA(cudaEventRecord(ev_cargs[0], st.s));
    CSG_CUDA(cudaMemcpyAsync(d_cargs.p, T, K * sizeof(ConsArgs), cudaMemcpyHostToDevice, st.s));
    CSG_CUDA(cudaEventRecord(ev_cargs[1], st.s));
    CSG_CUDA(cudaMemcpyAsync(d_apoly.p, apoly.data(), apoly.size() * sizeof(fe), cudaMemcpyHostToDevice, st.s));
    d_part.reserve(std::max<size_t>(K * items * ce * n, 1)); d_binv.reserve(CONS_MAX_BGROUPS * ce * n); d_comb.reserve(K * ce * n);
    eval_constraints_many(air_id, d_cargs.p, T[0], K, d_lde.p, tw, roots.W.p, d_ptab.p, d_apoly.p, d_part.p, d_binv.p, d_comb.p, st);
    CSG_CUDA(cudaEventRecord(ev[4], st.s));
    stage_launches(2);

    // ------------------------------------------------------------------ stage 4: composition columns and their commitments
    {
        std::vector<fe> sinv(K * ce);
        for (size_t kc = 0; kc < ce; kc++) { const fe s = inv(ce_shift[kc]); for (size_t k = 0; k < K; k++) sinv[k * ce + kc] = s; }
        std::vector<fe> mat(ce * ce);
        const fe off_n_inv = inv(f63::pow(to_mont(GENERATOR), n)), ce_inv = inv(to_mont(ce)), w_ce_inv = inv(root_of_unity(ilog2(ce)));
        for (size_t t = 0; t < ce; t++)
            for (size_t k = 0; k < ce; k++) mat[t * ce + k] = mul(mul(f63::pow(off_n_inv, t), ce_inv), f63::pow(w_ce_inv, (k * t) % ce));
        d_e.reserve(K * ce * n); d_cpolys.reserve(K * ce * n); d_clde.reserve(b * K * ce * n);
        coset_intt_columns(roots, ntt, d_comb.p, n, d_e.p, n, logn, sinv.data(), K * ce, st);
        composition_columns_many(d_e.p, d_cpolys.p, n, (unsigned)ce, mat.data(), K, st);
        coset_ntt_columns(roots, ntt, d_cpolys.p, n, d_clde.p, n, K * ce * n, K * ce, logn, lde_tables, st);
        d_cnodes.reserve(K * 16 * lde_n);
        commit(d_clde.p, (unsigned)ce, K * ce * n, ce * n, d_cnodes, lde_n, (unsigned)b, n, roots_h);
        CSG_CUDA(cudaEventRecord(ev[5], st.s));
        CSG_CUDA(cudaStreamSynchronize(st.s));   // (sinv and mat were staged by the copies that read them)
    }
    stage_launches(3);
    host_mark("composition roots");

    // ------------------------------------------------------------------ stage 5: out-of-domain frame
    const unsigned nblk = eval_polys_many_blocks(n);
    {
        std::vector<fe> pts(K * 6);   // per proof: (z, z^256), (zg, zg^256); then per proof (z^ce, (z^ce)^256)
        parallel_proofs(K, [&](size_t k) {
            ProofState &p = ps[k];
            p.coin.reseed(roots_h[k].data());
            memcpy(p.comp_root, roots_h[k].data(), 32);
            p.z = p.coin.draw();
            const fe zs[3] = {p.z, mul(p.z, g), f63::pow(p.z, ce)};
            for (int j = 0; j < 2; j++) { pts[k * 4 + 2 * j] = zs[j]; pts[k * 4 + 2 * j + 1] = f63::pow(zs[j], 256); }
            pts[K * 4 + 2 * k] = zs[2]; pts[K * 4 + 2 * k + 1] = f63::pow(zs[2], 256);
        });
        d_args.reserve(std::max<size_t>(K * 6, K * (2 * w + ce)));
        d_partial.reserve(K * (w * 2 + ce) * nblk);
        CSG_CUDA(cudaMemcpyAsync(d_args.p, pts.data(), pts.size() * sizeof(fe), cudaMemcpyHostToDevice, st.s));
        eval_polys_many(d_polys.p, n, w, K, d_args.p, 2, d_partial.p, st);
        eval_polys_many(d_cpolys.p, n, ce, K, d_args.p + K * 4, 1, d_partial.p + K * w * 2 * nblk, st);
        std::vector<fe> part(K * (w * 2 + ce) * nblk);
        CSG_CUDA(cudaMemcpyAsync(part.data(), d_partial.p, part.size() * sizeof(fe), cudaMemcpyDeviceToHost, st.s));
        CSG_CUDA(cudaStreamSynchronize(st.s));
        host_mark("ood values");
        std::vector<fe> coef(K * (2 * w + ce));
        std::vector<DeepArgs> dargs(K);
        parallel_proofs(K, [&](size_t k) {
            ProofState &p = ps[k];
            auto sum = [&](size_t at) { fe s = 0; for (unsigned x = 0; x < nblk; x++) s = add(s, part[at + x]); return s; };
            p.ood_cur.resize(w); p.ood_next.resize(w); p.ood_comp.resize(ce);
            for (size_t c = 0; c < w; c++) { p.ood_cur[c] = sum(((k * w + c) * 2) * nblk); p.ood_next[c] = sum(((k * w + c) * 2 + 1) * nblk); }
            for (size_t r = 0; r < ce; r++) p.ood_comp[r] = sum(K * w * 2 * nblk + (k * ce + r) * nblk);
            uint8_t dg[32];
            hash_elements_host(hf, p.ood_cur.data(), w, dg); p.coin.reseed(dg);
            hash_elements_host(hf, p.ood_next.data(), w, dg); p.coin.reseed(dg);
            hash_elements_host(hf, p.ood_comp.data(), ce, dg); p.coin.reseed(dg);
            // DEEP coefficients: (alpha, beta) per trace column (a third draw is discarded), one per composition column, lambda, mu
            DeepArgs &a = dargs[k];
            a = DeepArgs{};
            fe *ct = &coef[k * 2 * w], *cc = &coef[K * 2 * w + k * ce];
            for (size_t c = 0; c < w; c++) { ct[c] = p.coin.draw(); ct[w + c] = p.coin.draw(); (void)p.coin.draw(); }
            for (size_t r = 0; r < ce; r++) cc[r] = p.coin.draw();
            a.lambda = p.coin.draw(); a.mu = p.coin.draw();
            a.z = p.z; a.zg = mul(p.z, g); a.zm = f63::pow(p.z, ce);
            for (size_t c = 0; c < w; c++) { a.az = add(a.az, mul(ct[c], p.ood_cur[c])); a.bzg = add(a.bzg, mul(ct[w + c], p.ood_next[c])); }
            for (size_t r = 0; r < ce; r++) a.czm = add(a.czm, mul(cc[r], p.ood_comp[r]));
            a.ncosets = (unsigned)b;
            for (size_t s = 0; s < b; s++) a.shift[s] = lde_shift[s];
        });
        host_mark("deep coefficients");
        // ---------------------------------------------------------------- stage 6: DEEP composition
        d_dargs.reserve(K); d_abc.reserve(3 * K * n); d_abc_lde.reserve(3 * K * n * b); d_deep.reserve(K * lde_n);
        CSG_CUDA(cudaMemcpyAsync(d_args.p, coef.data(), coef.size() * sizeof(fe), cudaMemcpyHostToDevice, st.s));
        CSG_CUDA(cudaMemcpyAsync(d_dargs.p, dargs.data(), K * sizeof(DeepArgs), cudaMemcpyHostToDevice, st.s));
        combine_polys_many(d_polys.p, n, w, K, d_args.p, 2, d_abc.p, 3 * n, st);
        combine_polys_many(d_cpolys.p, n, ce, K, d_args.p + K * 2 * w, 1, d_abc.p + 2 * n, 3 * n, st);
        coset_ntt_columns(roots, ntt, d_abc.p, n, d_abc_lde.p, n, 3 * K * n, 3 * K, logn, lde_tables, st);
        deep_quotients_many(d_abc_lde.p, roots.W.p, n, K, d_dargs.p, (unsigned)b, d_deep.p, st);
        CSG_CUDA(cudaEventRecord(ev[6], st.s));
    }
    stage_launches(4);

    // ------------------------------------------------------------------ stage 7: FRI layers
    std::vector<const fe *> layer(nlayers);
    std::vector<size_t> layer_m(nlayers);
    while (fri_evals.size() < nlayers) { fri_evals.emplace_back(new DBuf<fe>()); fri_nodes.emplace_back(new DBuf<uint32_t>()); }
    layer[0] = d_deep.p; layer_m[0] = lde_n;
    for (size_t k = 0; k < K; k++) ps[k].fri_roots.resize(nlayers);
    for (size_t l = 0; l < nlayers; l++) {
        const size_t mm = layer_m[l], q = mm / 4;
        commit(layer[l], 4, 0, mm, *fri_nodes[l], q, 1, q, roots_h);
        CSG_CUDA(cudaStreamSynchronize(st.s));
        std::vector<fe> alphas(K);
        parallel_proofs(K, [&](size_t k) {
            ProofState &p = ps[k];
            memcpy(p.fri_roots[l].data(), roots_h[k].data(), 32);
            p.coin.reseed(roots_h[k].data());
            alphas[k] = p.coin.draw();
        });
        if (l + 1 == nlayers) break;
        const unsigned logm = ilog2(mm);
        FoldArgs a{};
        a.offset_inv = inv(to_mont(GENERATOR));
        const fe w_inv = inv(root_of_unity(logm));
        a.zeta_inv = f63::pow(w_inv, q); a.quarter = inv(to_mont(4));
        a.logm = logm; a.logW = roots.logn;
        if (logm > roots.logn) {
            if (logm - roots.logn > 5) throw std::runtime_error("FRI layer too large for the root table");
            for (unsigned i = 0; i < (1u << (logm - roots.logn)); i++) a.small[i] = f63::pow(w_inv, i);
        }
        fri_evals[l + 1]->reserve(K * q);
        CSG_CUDA(cudaMemcpyAsync(d_args.p, alphas.data(), K * sizeof(fe), cudaMemcpyHostToDevice, st.s));
        fri_fold4_many(layer[l], mm, roots.W.p, a, d_args.p, K, fri_evals[l + 1]->p, st);
        layer[l + 1] = fri_evals[l + 1]->p; layer_m[l + 1] = q;
    }
    CSG_CUDA(cudaEventRecord(ev[7], st.s));
    stage_launches(5);
    host_mark("fri layers");

    // ------------------------------------------------------------------ stage 8: grinding, query positions, openings
    const size_t m_last = layer_m[nlayers - 1];
    parallel_proofs(K, [&](size_t k) {
        ProofState &p = ps[k];
        uint64_t nonce = 1;
        while (p.coin.check_leading_zeros(nonce) < o->grinding_factor) nonce++;
        p.coin.reseed_with_int(nonce);
        p.nonce = nonce;
        p.pos = p.coin.draw_integers(nq, lde_n);
        // row jobs and digest jobs with offsets local to the proof
        auto plan = [&](Opening &op, const fe *data, unsigned width, unsigned ncosets, size_t coset_stride, size_t col_stride, const uint32_t *nodes,
                        size_t nleaves, const std::vector<size_t> &pos) {
            RowJob r{data, width, ncosets, coset_stride, col_stride, (unsigned)p.idx.size(), (unsigned)pos.size(), p.rows_words};
            for (size_t x : pos) p.idx.push_back((uint32_t)x);
            op.rows_off = p.rows_words; op.rows_len = pos.size() * width;
            p.rows_words += op.rows_len;
            p.rjobs.push_back(r);
            op.slots = batch_opening_nodes(nleaves, pos);
            DigestJob dj{nodes, (unsigned)p.idx.size(), 0, p.dig_count};
            for (auto &sl : op.slots) { for (uint32_t v : sl) p.idx.push_back(v); dj.count += (unsigned)sl.size(); }
            op.dig_off = p.dig_count;
            p.dig_count += dj.count;
            if (dj.count) p.djobs.push_back(dj);
        };
        plan(p.o_trace, d_lde.p + k * tw, (unsigned)w, (unsigned)b, K * tw, n, d_tnodes.p + k * 16 * lde_n, lde_n, p.pos);
        plan(p.o_comp, d_clde.p + k * ce * n, (unsigned)ce, (unsigned)b, K * ce * n, n, d_cnodes.p + k * 16 * lde_n, lde_n, p.pos);
        std::vector<size_t> fp = p.pos;
        p.o_fri.resize(nlayers - 1);
        for (size_t l = 0; l + 1 < nlayers; l++) {
            const size_t mm = layer_m[l], q = mm / 4;
            fp = fold_positions(fp, mm);
            plan(p.o_fri[l], layer[l] + k * mm, 4, 1, 0, q, fri_nodes[l]->p + k * 16 * q, q, fp);
        }
        // the remainder: its m_last elements as a one-column matrix read at positions 0 .. m_last - 1
        p.rem_off = p.rows_words; p.rem_len = m_last;
        p.rjobs.push_back(RowJob{layer[nlayers - 1] + k * m_last, 1, 1, 0, 0, (unsigned)p.idx.size(), (unsigned)m_last, p.rows_words});
        for (size_t i = 0; i < m_last; i++) p.idx.push_back((uint32_t)i);
        p.rows_words += m_last;
    });
    host_mark("grinding, positions, opening plans");
    size_t nidx = 0, nrows = 0, ndig = 0, nrj = 0, ndj = 0, max_rows = 0, max_digs = 0;
    for (ProofState &p : ps) {
        p.idx_base = nidx; p.rows_base = nrows; p.dig_base = ndig;
        nidx += p.idx.size(); nrows += p.rows_words; ndig += p.dig_count; nrj += p.rjobs.size(); ndj += p.djobs.size();
    }
    std::vector<uint32_t> idx(nidx);
    std::vector<RowJob> rj(nrj);
    std::vector<DigestJob> dj(ndj);
    {
        std::vector<size_t> rj_base(K), dj_base(K);
        for (size_t k = 0, a = 0, c = 0; k < K; k++) { rj_base[k] = a; dj_base[k] = c; a += ps[k].rjobs.size(); c += ps[k].djobs.size(); }
        for (const ProofState &p : ps) {
            for (const RowJob &r : p.rjobs) max_rows = std::max<size_t>(max_rows, (size_t)r.npos * r.width);
            for (const DigestJob &d : p.djobs) max_digs = std::max<size_t>(max_digs, d.count);
        }
        parallel_proofs(K, [&](size_t k) {
            const ProofState &p = ps[k];
            std::copy(p.idx.begin(), p.idx.end(), idx.begin() + p.idx_base);
            for (size_t j = 0; j < p.rjobs.size(); j++) {
                RowJob r = p.rjobs[j];
                r.idx_off += (unsigned)p.idx_base; r.rows_off += p.rows_base;
                rj[rj_base[k] + j] = r;
            }
            for (size_t j = 0; j < p.djobs.size(); j++) {
                DigestJob d = p.djobs[j];
                d.idx_off += (unsigned)p.idx_base; d.out_off = 2 * nrows + 8 * (p.dig_base + d.out_off);
                dj[dj_base[k] + j] = d;
            }
        });
    }
    if (nrj > 65535 || ndj > 65535) throw std::runtime_error("too many openings in one batch");
    d_idx.reserve(std::max<size_t>(nidx, 1)); d_rjobs.reserve(std::max<size_t>(nrj, 1)); d_djobs.reserve(std::max<size_t>(ndj, 1));
    d_out.reserve(nrows + 4 * ndig);
    CSG_CUDA(cudaMemcpyAsync(d_idx.p, idx.data(), nidx * sizeof(uint32_t), cudaMemcpyHostToDevice, st.s));
    CSG_CUDA(cudaMemcpyAsync(d_rjobs.p, rj.data(), nrj * sizeof(RowJob), cudaMemcpyHostToDevice, st.s));
    if (ndj) CSG_CUDA(cudaMemcpyAsync(d_djobs.p, dj.data(), ndj * sizeof(DigestJob), cudaMemcpyHostToDevice, st.s));
    gather_rows_jobs(d_rjobs.p, nrj, max_rows, d_idx.p, d_out.p, st);
    gather_digests_jobs(d_djobs.p, ndj, max_digs, d_idx.p, (uint32_t *)d_out.p, st);
    std::vector<uint64_t> out(nrows + 4 * ndig);
    CSG_CUDA(cudaMemcpyAsync(out.data(), d_out.p, out.size() * sizeof(uint64_t), cudaMemcpyDeviceToHost, st.s));
    CSG_CUDA(cudaEventRecord(ev[8], st.s));
    CSG_CUDA(cudaStreamSynchronize(st.s));
    stage_launches(6);
    host_mark("openings round trip");

    // ------------------------------------------------------------------ serialisation (write_proof, shared with csg_ctx::prove_loaded)
    const uint8_t *digs = reinterpret_cast<const uint8_t *>(out.data() + nrows);
    std::vector<Bytes> pfs(K);
    parallel_proofs(K, [&](size_t k) {
        const ProofState &p = ps[k];
        std::vector<const uint8_t *> fri_roots;
        for (auto &r : p.fri_roots) fri_roots.push_back(r.data());
        write_proof(pfs[k], (unsigned)w, logn, *o, p.trace_root, p.comp_root, fri_roots, p.o_trace, p.o_comp, p.o_fri, out.data() + p.rows_base,
                    digs + p.dig_base * 32, p.ood_cur, p.ood_next, p.ood_comp, p.rem_off, p.rem_len, p.nonce);
    });
    host_mark("serialise");
    // the last call that can fail comes before the proofs are handed out: on failure every proofs[k] stays NULL
    float *dst[8] = {&tm.h2d, &tm.lde, &tm.commit_trace, &tm.constraints, &tm.composition, &tm.ood_deep, &tm.fri, &tm.queries};
    for (int s = 0; s < 8; s++) CSG_CUDA(cudaEventElapsedTime(dst[s], ev[s], ev[s + 1]));
    float cargs_ms = 0;
    CSG_CUDA(cudaEventElapsedTime(&cargs_ms, ev_cargs[0], ev_cargs[1]));
    for (size_t k = 0; k < K; k++) {
        proofs[k] = (uint8_t *)malloc(pfs[k].v.size());
        if (!proofs[k]) {
            for (size_t j = 0; j <= k; j++) { free(proofs[j]); proofs[j] = nullptr; proof_lens[j] = 0; }
            throw std::bad_alloc();
        }
        memcpy(proofs[k], pfs[k].v.data(), pfs[k].v.size());
        proof_lens[k] = pfs[k].v.size();
    }
    tm.kernel_launches = st.launches - launches0;
    tm.total = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (host_trace) {
        host_mark("copy out");
        double prev = 0;
        fprintf(stderr, "[csg host trace] batch of %zu x (%zu x %zu), %llu launches; constraint arguments: %zu x %zu B up in %.3f ms\n", K, w, n,
                (unsigned long long)tm.kernel_launches, K, sizeof(ConsArgs), cargs_ms);
        for (auto &mk : trace.marks) { fprintf(stderr, "  %-36s +%8.1f us  (at %8.1f)\n", mk.first, mk.second - prev, mk.second); prev = mk.second; }
    }
}

}  // namespace csg
