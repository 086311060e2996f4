// Host helpers shared by the single-proof driver (prover_ctx.cuh), the batch driver (many/prove_many.cu) and the verifier: the checks
// on ProofOptions, the serialised proof context, the interpolant of an assertion sequence and the folding of query positions.
#pragma once
#include <algorithm>
#include <stdexcept>
#include <vector>

#include "../../../include/csg.h"
#include "../field.cuh"
#include "air_desc.hpp"
#include "transcript.hpp"

namespace csg {

// throws std::invalid_argument for options this library cannot prove with
inline void check_options(const csg_options *o) {
    if (!o) throw std::invalid_argument("options missing");
    if (o->field_extension < CSG_FIELD_EXT_NONE || o->field_extension > CSG_FIELD_EXT_CUBIC) throw std::invalid_argument("field extension must be None (1), Quadratic (2) or Cubic (3)");
    if (o->fri_folding_factor != 4) throw std::invalid_argument("only FRI folding factor 4 is implemented");
    if (o->hash_fn != CSG_HASH_BLAKE3_256 && o->hash_fn != CSG_HASH_SHA3_256) throw std::invalid_argument("hash function must be Blake3_256 or Sha3_256");
    if (o->num_queries == 0 || o->num_queries > 255 || o->grinding_factor >= 32) throw std::invalid_argument("num_queries in 1..255, grinding factor below 32");
    if (o->blowup_factor < 2 || o->blowup_factor > 32 || (o->blowup_factor & (o->blowup_factor - 1))) throw std::invalid_argument("blowup factor must be a power of two in 2..32");
    // winterfell caps the remainder at 1024 elements; its byte length is serialised as a u16 (8192 elements would wrap to 0)
    if (o->fri_max_remainder_size < 4 || o->fri_max_remainder_size > 1024 || (o->fri_max_remainder_size & (o->fri_max_remainder_size - 1)))
        throw std::invalid_argument("FRI remainder size must be a power of two in 4..1024");
}

// the FRI remainder layer is committed as rows of 4: it needs at least 2 rows
inline void check_remainder(size_t lde_n, const csg_options &o) {
    size_t m = lde_n;
    while (m > o.fri_max_remainder_size) m /= 4;
    if (m < 8) throw std::invalid_argument("FRI remainder would have fewer than 8 elements: raise fri_max_remainder_size");
}

// StarkProof's context: trace layout, field modulus and ProofOptions, as the coin seed and the proof header carry them
inline void write_proof_context(Bytes &w, unsigned width, unsigned logn, const csg_options &opt) {
    w.u8((uint8_t)width); w.u8((uint8_t)logn); w.u16(0);
    w.u8(8); w.u64(f63::P);
    w.u8((uint8_t)opt.num_queries); w.u8((uint8_t)ilog2_host(opt.blowup_factor)); w.u8((uint8_t)opt.grinding_factor);
    w.u8((uint8_t)opt.hash_fn); w.u8((uint8_t)opt.field_extension);
    w.u8((uint8_t)ilog2_host(opt.fri_folding_factor)); w.u8((uint8_t)ilog2_host(opt.fri_max_remainder_size));
}

// coefficients of the polynomial taking the given values on <w_len> (host, tiny: one value per signature)
inline std::vector<fe> interpolate_host(const std::vector<fe> &vals) {
    using namespace f63;
    const size_t len = vals.size();
    const fe w_inv = inv(root_of_unity(ilog2_host(len))), len_inv = inv(to_mont(len));
    std::vector<fe> c(len);
    for (size_t m = 0; m < len; m++) {
        fe s = 0, wm = f63::pow(w_inv, m), x = ONE;
        for (size_t i = 0; i < len; i++) { s = add(s, mul(vals[i], x)); x = mul(x, wm); }
        c[m] = mul(s, len_inv);
    }
    return c;
}

// positions of the next FRI layer's rows that the queries at `pos` of a layer over `domain` points open, in first-seen order
inline std::vector<size_t> fold_positions(const std::vector<size_t> &pos, size_t domain) {
    std::vector<size_t> out;
    for (size_t p : pos) { size_t f = p % (domain / 4); if (std::find(out.begin(), out.end(), f) == out.end()) out.push_back(f); }
    return out;
}

// one opening of a proof: where its rows sit among the opened words, where its path digests sit among the fetched digests, and the
// node indices of its BatchMerkleProof grouped the way serialize_nodes() writes them (batch_opening_nodes)
struct Opening { size_t rows_off = 0, rows_len = 0, dig_off = 0; std::vector<std::vector<uint32_t>> slots; };

// BatchMerkleProof::serialize_nodes() of an opening whose path digests sit at digs[32 * o.dig_off ..)
inline void write_paths(Bytes &out, const Opening &o, const uint8_t *digs) {
    out.u8((uint8_t)o.slots.size());
    size_t at = o.dig_off;
    for (auto &sl : o.slots) { out.u8((uint8_t)sl.size()); out.put(digs + at * 32, sl.size() * 32); at += sl.size(); }
}

// StarkProof::to_bytes: context, commitments, trace and constraint queries, out-of-domain frame, FRI layers and remainder,
// proof-of-work nonce.  rows / digs: the opened words and the 32-byte path digests the openings index into; the frame vectors hold
// the components of their elements in order (d per element with a field extension); the remainder is rows[rem_off, + rem_len).
inline void write_proof(Bytes &pf, unsigned width, unsigned logn, const csg_options &opt, const uint8_t *trace_root, const uint8_t *comp_root,
                        const std::vector<const uint8_t *> &fri_roots, const Opening &o_trace, const Opening &o_comp, const std::vector<Opening> &o_fri,
                        const uint64_t *rows, const uint8_t *digs, const std::vector<fe> &ood_cur, const std::vector<fe> &ood_next,
                        const std::vector<fe> &ood_comp, size_t rem_off, size_t rem_len, uint64_t nonce) {
    auto emit = [&](const Opening &o) {
        pf.u32((uint32_t)(o.rows_len * 8));
        pf.u64s(rows + o.rows_off, o.rows_len);
        Bytes paths;
        write_paths(paths, o, digs);
        pf.u32((uint32_t)paths.v.size()); pf.put(paths.v.data(), paths.v.size());
    };
    write_proof_context(pf, width, logn, opt);
    pf.u16((uint16_t)((2 + fri_roots.size()) * 32));
    pf.put(trace_root, 32); pf.put(comp_root, 32);
    for (const uint8_t *r : fri_roots) pf.put(r, 32);
    emit(o_trace);
    emit(o_comp);
    pf.u16((uint16_t)(ood_cur.size() * 8));
    for (fe v : ood_cur) pf.element(v);
    for (fe v : ood_next) pf.element(v);
    pf.u16((uint16_t)(ood_comp.size() * 8));
    for (fe v : ood_comp) pf.element(v);
    pf.u8((uint8_t)o_fri.size());
    for (const Opening &o : o_fri) emit(o);
    pf.u16((uint16_t)(rem_len * 8));
    pf.u64s(rows + rem_off, rem_len);
    pf.u8(1);
    pf.u64(nonce);
}

// number of FRI folds by 4 until the layer has at most fri_max_remainder_size elements
inline size_t num_fri_folds(size_t lde_n, const csg_options &o) { size_t r = 0, d = lde_n; while (d > o.fri_max_remainder_size) { d /= 4; r++; } return r; }

}  // namespace csg
