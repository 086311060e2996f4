// The proving context behind the C ABI of include/csg.h: device buffers, the stages of Prover::prove and the built-in transcript.
// Shared by the translation units that implement the ABI (prover.cu: level 1 / level 2; abi_witness.cu: device-side witnesses, batch
// builder, timers, sharding; abi_kernels.cu: kernel-level and debug entry points).
//
// Replaces winterfell's `Prover::prove(trace)` as the reference calls it (/root/reference/src/lib.rs:140 and the five
// sub-AIR examples): trace LDE -> commitment -> constraint evaluation -> composition commitment -> out-of-domain frame
// -> DEEP composition -> FRI -> queries, with every bulk stage on the GPU and only the Fiat-Shamir transcript, proof
// serialisation and a few hundred field operations per proof on the host.  Device data stays in Montgomery form and in
// coset-major order (ntt.cuh) from the moment the trace is loaded until rows are opened.
#pragma once
#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../include/csg.h"
#include "comm.cuh"
#include "commit.cuh"
#include "constraints.cuh"
#include "ext_stages.cuh"
#include "hash.cuh"
#include "host/air_desc.hpp"
#include "host/batch_plan.hpp"
#include "host/proof_common.hpp"
#include "host/stage_args.hpp"
#include "host/transcript.hpp"
#include "many/many.cuh"
#include "ntt.cuh"
#include "stages.cuh"
#include "validate/validate.cuh"
#include "witness.cuh"


namespace csg {
using namespace f63;

namespace {

struct StateError : std::runtime_error { using std::runtime_error::runtime_error; };
struct ArgError : std::runtime_error { using std::runtime_error::runtime_error; };

struct FriLayer {
    DBuf<fe> owned;           // evaluations of this layer (layer 0 aliases the DEEP evaluations)
    const fe *evals = nullptr;
    size_t m = 0;             // domain size of the layer
    DBuf<uint32_t> nodes;     // tree over m/4 transposed rows
    bool committed = false;
};

enum Stage { S_NONE, S_AIR, S_TRACE, S_COMMITTED, S_EVALUATED, S_COMPOSED, S_OOD, S_DEEP };

class Timer {   // device time of a stage, CUDA events on the proving stream; the events live as long as the context
  public:
    ~Timer() { for (auto &p : own_) { cudaEventDestroy(p.first); cudaEventDestroy(p.second); } }
    void start(Stream &st) {
        if (crowded()) flush();   // a level-2 caller that never reads the timings
        if (used_ == own_.size()) { cudaEvent_t a, b; CSG_CUDA(cudaEventCreate(&a)); CSG_CUDA(cudaEventCreate(&b)); own_.emplace_back(a, b); }
        l0_ = st.launches;
        CSG_CUDA(cudaEventRecord(own_[used_].first, st.s));
    }
    unsigned launches = 0;   // kernels launched between the last start() and stop()
    // blocking form: waits for the stage and returns its time (the callers that need the stage complete anyway)
    float stop(Stream &st) {
        launches = (unsigned)(st.launches - l0_);
        cudaEvent_t a = own_[used_].first, b = own_[used_].second;
        CSG_CUDA(cudaEventRecord(b, st.s)); CSG_CUDA(cudaEventSynchronize(b));
        float ms = 0; CSG_CUDA(cudaEventElapsedTime(&ms, a, b)); return ms;
    }
    // deferred form: the stage's time is written (add: added) to *dst by the next flush().  No host synchronisation per stage --
    // a proof of a small trace is a few dozen short kernels, and waiting out each stage only to read a clock cost 0.12-0.15 ms
    // of a 0.6-1.4 ms proof (tools/small_latency.py).
    void stop(Stream &st, float *dst, bool add = false) {
        launches = (unsigned)(st.launches - l0_);
        CSG_CUDA(cudaEventRecord(own_[used_].second, st.s));
        pending_.push_back({own_[used_].first, own_[used_].second, dst, add});
        used_++;
    }
    // the same for a pair of events recorded elsewhere (they must not be re-recorded before the flush)
    void span(cudaEvent_t a, cudaEvent_t b, float *dst) { pending_.push_back({a, b, dst, false}); }
    void zero(float *dst) { pending_.push_back({nullptr, nullptr, dst, false}); }   // *dst = 0, in order with the spans
    bool crowded() const { return pending_.size() >= 256; }
    void discard() { pending_.clear(); used_ = 0; }   // nobody asked for the times of the previous proof
    void flush() {
        for (const Pending &q : pending_) {
            float ms = 0;
            if (q.a) { CSG_CUDA(cudaEventSynchronize(q.b)); CSG_CUDA(cudaEventElapsedTime(&ms, q.a, q.b)); }
            *q.dst = q.add ? *q.dst + ms : ms;
        }
        pending_.clear();
        used_ = 0;
    }
  private:
    struct Pending { cudaEvent_t a, b; float *dst; bool add; };
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> own_;
    std::vector<Pending> pending_;
    size_t used_ = 0;
    unsigned long long l0_ = 0;
};

}  // namespace
}  // namespace csg

using namespace csg;

// The column chunks in which stage 1 walks a rank's column block [c_lo, c_hi).  Nothing to overlap when the trace is already
// resident: one chunk.  From host memory the extension can only start once the first chunk has arrived, so the chunks ramp up --
// 1, 3, 4, then 8 columns (8 MB first: 0.15 ms of PCIe instead of 1.2 ms; end to end 61.2 -> 60.7 ms per 1024-transaction proof,
// profiles/r2_e2e_chunks.txt); CSG_H2D_CHUNKS="a,b,c" overrides the schedule, the last entry repeating.  The sizes add up to
// c_hi - c_lo exactly: the last rank of a sharded proof owns fewer columns than columns_per_rank, and the buffers hold `width`
// columns, not world * columns_per_rank (csg_dist_trace_chunks exposes this to the CPU tests).
static std::vector<size_t> trace_chunks(bool from_host, size_t c_lo, size_t c_hi) {
    std::vector<size_t> chunks;
    if (c_hi <= c_lo) return chunks;
    if (!from_host) { chunks.push_back(c_hi - c_lo); return chunks; }
    static const std::vector<size_t> sched = [] {
        std::vector<size_t> v;
        if (const char *e = getenv("CSG_H2D_CHUNKS"))
            for (const char *q = e; *q;) { char *end; const unsigned long x = strtoul(q, &end, 10); if (end == q) break; if (x) v.push_back(x); q = *end ? end + 1 : end; }
        if (v.empty()) v = {1, 3, 4, 8};
        return v;
    }();
    for (size_t c = c_lo, k = 0; c < c_hi; k++) { const size_t sz = std::min(sched[std::min(k, sched.size() - 1)], c_hi - c); chunks.push_back(sz); c += sz; }
    return chunks;
}

// which part of a sharded proof a rank owns: a contiguous block of LDE cosets (and the ce cosets among them), and the block
// of trace columns it interpolates.  The one place this geometry is defined; csg_dist_plan exposes it to callers.
static bool shard_plan(size_t rank, size_t world, size_t b, size_t ce, size_t w, csg_shard_plan *out) {
    if (world < 1 || rank >= world || b < world || b % world || ce < 1 || ce > b || b % ce) return false;
    const size_t bl = b / world, k0 = rank * bl, cpr = (w + world - 1) / world;
    size_t kc0 = 0, cel = 0;
    for (size_t kc = 0; kc < ce; kc++) {
        const size_t k = kc * (b / ce);
        if (k >= k0 && k < k0 + bl) { if (!cel) kc0 = kc; cel++; }
    }
    const size_t c_lo = std::min(w, rank * cpr), c_hi = std::min(w, c_lo + cpr);
    *out = csg_shard_plan{(uint32_t)k0, (uint32_t)bl, (uint32_t)kc0, (uint32_t)cel, (uint32_t)c_lo, (uint32_t)(c_hi - c_lo), (uint32_t)cpr};
    return true;
}

struct csg_ctx {
    int device = 0;
    Stream st;
    std::string err;
    RootTable roots;
    NttScratch ntt;
    DBuf<fe> scratch, scratch2;
    Stage stage = S_NONE;

    AirDesc air;
    csg_options opt{};
    TransitionGroups tg;
    BoundaryGroups bg;
    size_t n = 0, b = 0, ce = 0, lde_n = 0;
    unsigned logn = 0;
    std::vector<fe> lde_shift, ce_shift;   // s_k = offset * w_lde^k ; ce cosets are the LDE cosets k = kc * (b / ce)
    // coset-sharded proof (comm.cuh): this context owns the LDE cosets [k0, k0 + bl) and the ce cosets among them; with
    // no communicator G = 1 and it owns everything.  lde_shift / ce_shift hold the OWNED cosets only.
    std::unique_ptr<Comm> comm;
    size_t G = 1, rank = 0, bl = 0, k0 = 0, cel = 0, kc0 = 0;
    DBuf<uint64_t> d_gather;               // slices under exchange
    DBuf<fe> d_xch;                        // coefficient sets of the low-degree splits under exchange
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> comm_ev;
    size_t comm_used = 0;
    Stream comm_stream;                    // the coefficient all-gather overlaps the extension of the own columns
    cudaEvent_t ev_intt = nullptr, ev_gathered = nullptr;
    std::vector<cudaEvent_t> block_ev;     // block q of the coefficient exchange has landed

    DBuf<uint64_t> d_io, d_wit_in;
    // device-side batch builder (batch_gen.cu): plan uploads, node versions, signatures; tables cached per context
    DBuf<uint64_t> d_b_accounts, d_b_txw, d_b_sigs;
    DBuf<int> d_b_left, d_b_right, d_b_refs;
    DBuf<fe> d_b_hashes, d_b_defaults, d_b_gtable;
    unsigned b_defaults_depth = 0;
    bool b_gtable_built = false;
    size_t wit_resident_ntx = 0;             // transfers whose packed records are resident in d_wit_in
    unsigned wit_resident_depth = 0;
    DBuf<fe> d_wit_finals;
    std::vector<uint64_t> wit_packed;
    const csg_tx_batch *wit_packed_for = nullptr;
    DBuf<uint32_t> d_idx, d_dig;
    DBuf<fe> d_parts, d_polys, d_lde, d_comb, d_e, d_eg, d_cpolys, d_clde, d_abc, d_abc_lde, d_deep, d_ptab, d_apoly;
    DBuf<uint32_t> d_tnodes, d_cnodes;
    // Sharded proof: each context holds the Merkle SUBTREE over its contiguous range of lde_n / G leaves (in d_tnodes / d_cnodes,
    // same heap layout, root at node 1) and a replicated copy of the top log2(G) levels (2G digests: node 1 = the root, nodes
    // G .. 2G-1 = the subtree roots of ranks 0 .. G-1).  Off for a single GPU and for traces shorter than the group.
    DBuf<uint32_t> d_ttop, d_ctop;
    bool subtrees() const { return G > 1 && n >= G; }
    // node `idx` of the whole tree (heap index) as this context can read it: see gather_digests
    uint32_t tree_ref(size_t idx) const {
        if (!subtrees()) return (uint32_t)idx;
        if (idx < 2 * G) return rank == 0 ? (0x80000000u | (uint32_t)idx) : 0xFFFFFFFFu;   // replicated: one contribution to the sum
        unsigned l = 0;
        while (((size_t)2 << l) <= idx) l++;
        const unsigned ls = l - ilog2(G);
        const size_t p = idx - ((size_t)1 << l);
        return (p >> ls) == rank ? (uint32_t)(((size_t)1 << ls) + (p & (((size_t)1 << ls) - 1))) : 0xFFFFFFFFu;
    }
    DBuf<ConsArgs> d_cargs;
    std::unique_ptr<ConsArgs> h_cargs;
    bool cargs_domain_ready = false;   // the per-AIR part of *h_cargs (domain constants, assertion polynomials) has been filled
    std::vector<std::unique_ptr<FriLayer>> fri;   // pool: buffers survive from proof to proof; nfri layers are live
    size_t nfri = 0;
    DBuf<uint64_t> d_rows;
    Timer stage_timer, query_timer;
    // The stage times of a proof are read from their event pairs only when csg_get_timings asks (some 25 pairs: 70-85 us of
    // driver calls, a tenth of a small proof); a proof nobody asked about is dropped when the next one starts.
    void flush_timers() { stage_timer.flush(); query_timer.flush(); }

    fe z = 0;
    std::vector<fe> ood_cur, ood_next, ood_comp;
    // FieldExtension::Quadratic / Cubic: d = 2 / 3; challenges, composition, OOD frame, DEEP and FRI are E-valued (ext_stages.cuh)
    int d = 1;
    ExtConsts xk{};
    xe xz{};
    std::vector<xe> xood_cur, xood_next, xood_comp;
    DBuf<fe> d_pw;
    csg_timings tm{};
    cudaEvent_t ev_a = nullptr, ev_b = nullptr;   // csg_timer_start / csg_timer_stop
    cudaEvent_t cons_ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    bool split_low_degree = getenv("CSG_NO_SPLIT") == nullptr;   // CSG_NO_SPLIT=1: evaluate every constraint on every coset (A/B testing)
    // Below this trace length the split's extra launches cost more than the arithmetic it saves (tools/small_latency.py: one
    // transaction 1.28 -> 1.18 ms, one signature 1.06 -> 0.95 ms without it; break-even at 2^14 rows).  The proof is the same
    // either way; CSG_SPLIT_MIN_ROWS=0 forces the split on small traces (tests).
    size_t split_min_rows = getenv("CSG_SPLIT_MIN_ROWS") ? strtoull(getenv("CSG_SPLIT_MIN_ROWS"), nullptr, 10) : (size_t)1 << 14;
    cudaStream_t copy_stream = nullptr;          // H2D copies of trace column chunks, overlapped with their extension
    std::vector<cudaEvent_t> chunk_ev;
    int trace_repr = CSG_REPR_CANONICAL;         // representation of the words in d_io (csg_load_trace / csg_prove_trace)
    // a trace in PAGEABLE host memory (a Rust Vec<u64>) is staged through a small ring of pinned buffers by the host threads:
    // cudaMemcpyAsync from pageable memory is a synchronous, single-threaded bounce copy inside the driver
    enum { STAGE_BUFS = 3 };
    uint64_t *stage_buf[STAGE_BUFS] = {nullptr, nullptr, nullptr};
    size_t stage_words = 0;
    cudaEvent_t stage_ev[STAGE_BUFS] = {nullptr, nullptr, nullptr};
    float h2d_ms_last = 0;
    cudaEvent_t h2d_a = nullptr, h2d_b = nullptr;   // first byte .. last byte of the overlapped H2D copy, on the copy stream
    CosetTables lde_tables;                      // per-coset scale tables of the LDE domain, built once per csg_set_air
    ManyProver *many = nullptr;                  // csg_prove_many: its own device buffers and tables, created by the first batch
    Validator *validator = nullptr;              // csg_validate_*: its own device buffers, created by the first call

    // ------------------------------------------------------------------------------------------ setup
    void set_air(int air_id, size_t trace_len, const csg_options *o, const uint64_t *pub, size_t npub) {
        try { check_options(o); } catch (const std::invalid_argument &e) { throw ArgError(e.what()); }
        // The same AIR, length, options and sharding as the last call -- a prover proving batch after batch, where only the public
        // inputs (assertion values) differ: the root table, the periodic-column tables and the coset scale tables on the device
        // stay as they are, and so does a prefetched trace.
        const bool same_shape = stage >= S_AIR && air.id == air_id && n == trace_len && memcmp(&opt, o, sizeof opt) == 0 &&
                                G == (comm ? (size_t)comm->world : 1) && rank == (comm ? (size_t)comm->rank : 0);
        bool same_periodic = same_shape;
        {
            AirDesc fresh;
            try { fresh = make_air(air_id, trace_len, pub, npub); } catch (const std::invalid_argument &e) { throw ArgError(e.what()); }
            // (the Schnorr AIR's periodic columns carry the public keys and messages: those tables follow the public inputs)
            same_periodic = same_periodic && fresh.periodic.size() == air.periodic.size();
            for (size_t c = 0; same_periodic && c < fresh.periodic.size(); c++) same_periodic = fresh.periodic[c].values == air.periodic[c].values;
            if (!(same_shape && same_periodic)) {
                // From here on the members describe the new shape while the device tables still hold the old one, and any
                // check below may throw: until this call completes the context has no AIR, so a repeated call with the same
                // arguments cannot take the fast path above, and no proof runs on the mixed state.  A prefetched trace of the
                // old shape is dropped.
                stage = S_NONE;
                if (next_pending) { CSG_CUDA(cudaStreamSynchronize(copy_stream)); next_pending = false; }
            }
            air = std::move(fresh);
        }
        if (same_shape && same_periodic) {
            tg = transition_groups(air);
            bg = boundary_groups(air);
            cargs_domain_ready = false;   // assertion values and their polynomials are refreshed by the next constraint evaluation
            nfri = 0;
            stage = S_AIR;
            return;
        }
        opt = *o;
        d = (int)o->field_extension;
        if (d > 1) xk = ext_consts();
        n = trace_len; logn = ilog2(n); b = o->blowup_factor; ce = air.ce_blowup(); lde_n = n * b;
        tg = transition_groups(air);
        bg = boundary_groups(air);
        try { check_air_shape(air, tg, bg, n, *o); } catch (const std::invalid_argument &e) { throw ArgError(e.what()); }
        G = comm ? (size_t)comm->world : 1; rank = comm ? (size_t)comm->rank : 0;
        csg_shard_plan plan;
        if (!shard_plan(rank, G, b, ce, air.width, &plan)) throw ArgError("the number of ranks of a sharded proof must divide the blowup factor");
        bl = plan.num_cosets; k0 = plan.first_coset;
        if (logn > 22) throw ArgError("trace length above 2^22 is not supported");
        roots.build(logn, st);
        const fe offset = to_mont(GENERATOR), w_lde = root_of_unity(ilog2(lde_n));
        std::vector<fe> all_shift(b);
        fe acc = offset;
        for (size_t k = 0; k < b; k++) { all_shift[k] = acc; acc = mul(acc, w_lde); }
        lde_shift.assign(all_shift.begin() + k0, all_shift.begin() + k0 + bl);
        ce_shift.clear();
        kc0 = plan.first_ce_coset; cel = plan.num_ce_cosets;
        for (size_t kc = kc0; kc < kc0 + cel; kc++) ce_shift.push_back(all_shift[kc * (b / ce)]);
        build_periodic_tables();
        lde_tables.build(lde_shift.data(), bl, logn, st);
        nfri = 0;
        stage = S_AIR;
    }

    // periodic column of period P on ce coset kc: values at y = (s_kc * w_n^i)^(n/P) = s_kc^(n/P) * w_P^i, i < P --
    // a coset LDE of the length-P column with shifts s_kc^(n/P); columns of equal period go through the NTT together
    void build_periodic_tables() {
        h_cargs.reset(new ConsArgs());
        cargs_domain_ready = false;
        ConsArgs &A = *h_cargs;
        memset(&A, 0, sizeof A);
        const PeriodicRuns pr = periodic_runs(air);
        fill_periodic_args(A, pr, 1, 0);
        d_ptab.reserve((pr.total ? pr.total : 1) * (cel ? cel : 1));
        DBuf<fe> vals, coef;
        for (const PeriodicRun &r : pr.runs) {
            const size_t P = r.P, nc = r.c1 - r.c0;
            std::vector<fe> host(nc * P);
            for (size_t c = r.c0; c < r.c1; c++) memcpy(&host[(c - r.c0) * P], air.periodic[c].values.data(), P * sizeof(fe));
            vals.reserve(nc * P); coef.reserve(nc * P);
            CSG_CUDA(cudaMemcpyAsync(vals.p, host.data(), nc * P * sizeof(fe), cudaMemcpyHostToDevice, st.s));
            intt_columns(roots, ntt, vals.p, P, coef.p, P, nc, ilog2(P), st);
            std::vector<fe> shifts(cel);
            for (size_t kc = 0; kc < cel; kc++) shifts[kc] = f63::pow(ce_shift[kc], n / P);
            if (cel) coset_ntt_columns(roots, ntt, coef.p, P, d_ptab.p + r.off, P, pr.total, nc, ilog2(P), shifts.data(), cel, st);
            CSG_CUDA(cudaStreamSynchronize(st.s));   // host staging vector goes out of scope
        }
    }

    static void check_repr(int repr) { if (repr != CSG_REPR_CANONICAL && repr != CSG_REPR_MONTGOMERY) throw ArgError("repr must be CSG_REPR_CANONICAL or CSG_REPR_MONTGOMERY"); }
    static bool is_pageable(const void *p) {
        cudaPointerAttributes a{};
        if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return true; }
        return a.type == cudaMemoryTypeUnregistered;
    }
    void load_trace(const uint64_t *trace, int repr) {
        need(S_AIR, "csg_set_air must be called first");
        check_repr(repr);
        trace_repr = repr;
        const size_t count = (size_t)air.width * n;
        Timer &t = stage_timer;
        t.start(st);
        d_io.reserve(count);
        CSG_CUDA(cudaMemcpyAsync(d_io.p, trace, count * sizeof(uint64_t), cudaMemcpyHostToDevice, st.s));
        tm.h2d = t.stop(st);
        nfri = 0;
        stage = S_TRACE;
    }
    // ---- a stream of traces: the copy of the NEXT trace runs on the copy stream under the proof of the current one.
    // Two trace buffers take turns (d_io: being proved / resident; d_next: being filled).  Proofs are synchronous calls, so
    // when a copy into d_next starts nothing in flight reads that buffer: it was d_io two proofs ago.
    DBuf<uint64_t> d_next;
    cudaEvent_t next_a = nullptr, next_b = nullptr;
    bool next_pending = false;
    int next_repr = CSG_REPR_CANONICAL;
    void prefetch_trace(const uint64_t *trace, int repr) {
        need(S_AIR, "csg_set_air must be called first");
        check_repr(repr);
        if (!trace) throw ArgError("null trace");
        if (next_pending) throw StateError("a prefetched trace is already waiting: csg_prove_prefetched proves it");
        csg_shard_plan plan;
        shard_plan(rank, G, b, ce, air.width, &plan);   // a sharded proof reads only the column block this rank interpolates
        d_next.reserve((size_t)air.width * n);
        if (!copy_stream) CSG_CUDA(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
        if (!next_a) { CSG_CUDA(cudaEventCreate(&next_a)); CSG_CUDA(cudaEventCreate(&next_b)); }
        CSG_CUDA(cudaEventRecord(next_a, copy_stream));
        if (plan.num_columns)
            CSG_CUDA(cudaMemcpyAsync(d_next.p + (size_t)plan.first_column * n, trace + (size_t)plan.first_column * n,
                                     (size_t)plan.num_columns * n * sizeof(uint64_t), cudaMemcpyHostToDevice, copy_stream));
        CSG_CUDA(cudaEventRecord(next_b, copy_stream));
        next_repr = repr;
        next_pending = true;
    }
    void prove_prefetched(const uint64_t *next_trace, int next_trace_repr, uint8_t **proof, size_t *proof_len) {
        if (!next_pending) throw StateError("csg_prefetch_trace must be called first");
        CSG_CUDA(cudaEventSynchronize(next_b));   // it ran under the previous proof; also: the caller's buffer is free from here on
        CSG_CUDA(cudaEventElapsedTime(&tm.h2d, next_a, next_b));
        std::swap(d_io.p, d_next.p); std::swap(d_io.n, d_next.n);
        trace_repr = next_repr;
        next_pending = false;
        nfri = 0;
        stage = S_TRACE;
        if (next_trace) prefetch_trace(next_trace, next_trace_repr);
        prove_loaded(proof, proof_len);
    }
    // for benchmarking with inputs already resident: the trace as left on the device by the last load_trace
    void reload_resident() {
        need(S_TRACE, "no trace has been loaded");
        nfri = 0;
        stage = S_TRACE;
        tm.h2d = 0;
    }

    void need(Stage s, const char *msg) const { if (stage < s) throw StateError(msg); }
    void download_root(const DBuf<uint32_t> &nodes, uint8_t root[32]) {
        CSG_CUDA(cudaMemcpyAsync(root, nodes.p + 8, 32, cudaMemcpyDeviceToHost, st.s));
        CSG_CUDA(cudaStreamSynchronize(st.s));
    }
    void all_to_all(const void *send, void *recv, size_t bytes) {
        comm_events();
        CSG_CUDA(cudaEventRecord(comm_ev[comm_used].first, st.s));
        comm->all_to_all(send, recv, bytes, st);
        CSG_CUDA(cudaEventRecord(comm_ev[comm_used++].second, st.s));
    }

    // ------------------------------------------------------------------------------------------ stage 1 + 2
    // Stage 1 runs column chunk by column chunk: representation change, interpolation and the `blowup` coset transforms of
    // a chunk need nothing from the other columns, so when the trace still lives in host memory (csg_prove) the H2D copy
    // of chunk c+1 overlaps the extension of chunk c.  host == nullptr: the canonical trace is already in d_io.
    // host: the whole trace, column-major, in one allocation; host_cols: one pointer per column (a TraceTable's Vec<Vec<_>>)
    void extend_and_commit_trace(uint8_t root[32], const uint64_t *host = nullptr, int host_repr = CSG_REPR_CANONICAL, const uint64_t *const *host_cols = nullptr) {
        std::vector<const uint64_t *> colptr;
        if (host || host_cols) {
            check_repr(host_repr); trace_repr = host_repr;
            colptr.resize(air.width);
            for (size_t c = 0; c < air.width; c++) {
                colptr[c] = host_cols ? host_cols[c] : host + c * n;
                if (!colptr[c]) throw ArgError("null trace column");
            }
            if (!host) host = colptr[0];
        }
        if (!host) need(S_TRACE, "csg_load_trace must be called first");
        else need(S_AIR, "csg_set_air must be called first");
        const size_t w = air.width;
        // sharded proof: this context interpolates the column block [c_lo, c_hi), the coefficient blocks are all-gathered,
        // and every context extends all columns onto its own cosets
        csg_shard_plan plan;
        shard_plan(rank, G, b, ce, w, &plan);
        const size_t cpr = plan.columns_per_rank, c_lo = plan.first_column, c_hi = c_lo + plan.num_columns, wpad = cpr * G;
        const std::vector<size_t> chunks = trace_chunks(host != nullptr, c_lo, c_hi);
        size_t CHUNK = 1;
        for (size_t s : chunks) CHUNK = std::max(CHUNK, s);
        Timer &t = stage_timer;
        t.start(st);
        d_io.reserve(w * n); d_polys.reserve(wpad * n); scratch.reserve(wpad * n); d_lde.reserve(w * n * bl);
        bool any_pageable = false;
        if (host) for (size_t c = c_lo; c < c_hi && !any_pageable; c++) any_pageable = is_pageable(colptr[c]);
        const bool staged = host && any_pageable;
        if (host) {
            if (!copy_stream) CSG_CUDA(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
            while (chunk_ev.size() < chunks.size() + 1) { cudaEvent_t e; CSG_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); chunk_ev.push_back(e); }
            if (!h2d_a) { CSG_CUDA(cudaEventCreate(&h2d_a)); CSG_CUDA(cudaEventCreate(&h2d_b)); }
            if (staged && stage_words < CHUNK * n) {
                for (auto &b : stage_buf) { if (b) cudaFreeHost(b); b = nullptr; }
                for (auto &b : stage_buf) CSG_CUDA(cudaHostAlloc((void **)&b, CHUNK * n * sizeof(uint64_t), cudaHostAllocDefault));
                stage_words = CHUNK * n;
                for (auto &e : stage_ev) if (!e) CSG_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            }
            // the copies must not overtake earlier work on the proving stream that still reads d_io
            CSG_CUDA(cudaEventRecord(chunk_ev[0], st.s));
            CSG_CUDA(cudaStreamWaitEvent(copy_stream, chunk_ev[0], 0));
            CSG_CUDA(cudaEventRecord(h2d_a, copy_stream));
        }
        for (size_t c0 = c_lo, k = 0; k < chunks.size() && c0 < c_hi; c0 += chunks[k], k++) {
            const size_t nc = std::min(chunks[k], c_hi - c0);   // never past the block: d_io holds exactly w columns
            if (host) {
                bool contiguous = true;
                for (size_t j = 1; j < nc; j++) contiguous = contiguous && colptr[c0 + j] == colptr[c0] + j * n;
                const uint64_t *src = colptr[c0];
                if (staged) {   // host threads fill a pinned buffer while the GPU extends the previous chunks
                    uint64_t *buf = stage_buf[k % STAGE_BUFS];
                    if (k >= STAGE_BUFS) CSG_CUDA(cudaEventSynchronize(stage_ev[k % STAGE_BUFS]));
                    const size_t SL = (size_t)1 << 17, per_col = (n + SL - 1) / SL;   // 1 MB slices of each column
                    const long long nsl = (long long)(per_col * nc);
#pragma omp parallel for schedule(static)
                    for (long long sl = 0; sl < nsl; sl++) {
                        const size_t j = (size_t)sl / per_col, o = ((size_t)sl % per_col) * SL;
                        memcpy(buf + j * n + o, colptr[c0 + j] + o, std::min(SL, n - o) * sizeof(uint64_t));
                    }
                    src = buf; contiguous = true;
                }
                if (contiguous) CSG_CUDA(cudaMemcpyAsync(d_io.p + c0 * n, src, nc * n * sizeof(uint64_t), cudaMemcpyHostToDevice, copy_stream));
                else for (size_t j = 0; j < nc; j++)
                    CSG_CUDA(cudaMemcpyAsync(d_io.p + (c0 + j) * n, colptr[c0 + j], n * sizeof(uint64_t), cudaMemcpyHostToDevice, copy_stream));
                if (staged) CSG_CUDA(cudaEventRecord(stage_ev[k % STAGE_BUFS], copy_stream));
                CSG_CUDA(cudaEventRecord(chunk_ev[k], copy_stream));
                if (c0 + nc >= c_hi) CSG_CUDA(cudaEventRecord(h2d_b, copy_stream));
                CSG_CUDA(cudaStreamWaitEvent(st.s, chunk_ev[k], 0));
            }
            // the representation change of the caller's words costs nothing: interpolation is linear, so the factor R^2 of
            // "canonical -> Montgomery" joins the 1/n scaling of the inverse transform (Montgomery words need no factor)
            intt_columns(roots, ntt, d_io.p + c0 * n, n, scratch.p + c0 * n, n, nc, logn, st, trace_repr == CSG_REPR_MONTGOMERY ? 0 : R2, true);
            if (G == 1) coset_ntt_columns(roots, ntt, scratch.p + c0 * n, n, d_lde.p + c0 * n, n, w * n, nc, logn, lde_tables, st);
        }
        if (G > 1) {
            // The coefficient all-gather (the largest exchange) runs on its own stream while this context already extends the
            // columns it interpolated itself; the other ranks' columns follow once they have arrived.  With 2 and 4 ranks the
            // gather is hidden entirely under the own block (47 / 24 columns); with 8 it is not (12 columns: 0.3 ms of transforms
            // against ~1 ms of gather).  CSG_COEF_BLOCKWISE=1 issues it block by block instead -- one broadcast per column block,
            // in rank order, each block extended as soon as it has landed -- but a broadcast drives one sender's links at a time
            // where the all-gather drives all of them: 10.2 against 9.6 ms for this stage at 2 ranks (profiles/r2_coef_exchange.txt).
            static const bool one_gather = getenv("CSG_COEF_BLOCKWISE") == nullptr;
            if (!comm_stream.s) CSG_CUDA(cudaStreamCreateWithFlags(&comm_stream.s, cudaStreamNonBlocking));
            if (!ev_intt) { CSG_CUDA(cudaEventCreateWithFlags(&ev_intt, cudaEventDisableTiming)); CSG_CUDA(cudaEventCreateWithFlags(&ev_gathered, cudaEventDisableTiming)); }
            while (block_ev.size() < G) { cudaEvent_t e; CSG_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); block_ev.push_back(e); }
            CSG_CUDA(cudaEventRecord(ev_intt, st.s));
            if (c_hi > c_lo) coset_ntt_columns(roots, ntt, scratch.p + c_lo * n, n, d_lde.p + c_lo * n, n, w * n, c_hi - c_lo, logn, lde_tables, st);
            CSG_CUDA(cudaStreamWaitEvent(comm_stream.s, ev_intt, 0));
            if (one_gather) {
                gather(scratch.p, cpr * n * sizeof(fe), &comm_stream);
                CSG_CUDA(cudaEventRecord(ev_gathered, comm_stream.s));
                CSG_CUDA(cudaStreamWaitEvent(st.s, ev_gathered, 0));
                if (c_lo > 0) coset_ntt_columns(roots, ntt, scratch.p, n, d_lde.p, n, w * n, c_lo, logn, lde_tables, st);
                if (c_hi < w) coset_ntt_columns(roots, ntt, scratch.p + c_hi * n, n, d_lde.p + c_hi * n, n, w * n, w - c_hi, logn, lde_tables, st);
            } else {
                for (unsigned q = 0; q < G; q++) {
                    const size_t q_lo = std::min((size_t)q * cpr, w), q_hi = std::min(q_lo + cpr, w);
                    bcast(scratch.p + (size_t)q * cpr * n, cpr * n * sizeof(fe), (int)q, &comm_stream);
                    if (q == rank || q_hi == q_lo) continue;
                    CSG_CUDA(cudaEventRecord(block_ev[q], comm_stream.s));
                    CSG_CUDA(cudaStreamWaitEvent(st.s, block_ev[q], 0));
                    coset_ntt_columns(roots, ntt, scratch.p + q_lo * n, n, d_lde.p + q_lo * n, n, w * n, q_hi - q_lo, logn, lde_tables, st);
                }
                // later stages read every block on the proving stream: it has waited for each one it transformed; an empty tail
                // block (fewer columns than ranks) still has to be in before the buffer is reused
                CSG_CUDA(cudaEventRecord(ev_gathered, comm_stream.s));
                CSG_CUDA(cudaStreamWaitEvent(st.s, ev_gathered, 0));
            }
        }
        std::swap(d_polys.p, scratch.p); std::swap(d_polys.n, scratch.n);   // d_polys = coefficients
        t.stop(st, &tm.lde); tm.stage_launches[0] = t.launches;
        if (host) {   // the copy ran under the extension: its own duration (first byte .. last byte), not time added to the proof
            nfri = 0;
            t.zero(&tm.h2d);
            if (c_hi > c_lo) t.span(h2d_a, h2d_b, &tm.h2d);
        }
        t.start(st);
        commit_rows(d_lde.p, (unsigned)w, w * n, d_tnodes, d_ttop);
        download_root(subtrees() ? d_ttop : d_tnodes, root);
        t.stop(st, &tm.commit_trace); tm.stage_launches[1] = t.launches;
        stage = S_COMMITTED;
    }

    // ------------------------------------------------------------------------------------------ exchanges of a sharded proof
    void comm_events() {
        if (comm_ev.size() == comm_used) {
            cudaEvent_t a, e;
            CSG_CUDA(cudaEventCreate(&a)); CSG_CUDA(cudaEventCreate(&e));
            comm_ev.emplace_back(a, e);
        }
    }
    void gather(void *buf, size_t bytes, Stream *on = nullptr) {
        Stream &cs = on ? *on : st;
        comm_events();
        CSG_CUDA(cudaEventRecord(comm_ev[comm_used].first, cs.s));
        comm->all_gather(buf, bytes, cs);
        CSG_CUDA(cudaEventRecord(comm_ev[comm_used++].second, cs.s));
    }
    void bcast(void *buf, size_t bytes, int root, Stream *on = nullptr) {
        Stream &cs = on ? *on : st;
        comm_events();
        CSG_CUDA(cudaEventRecord(comm_ev[comm_used].first, cs.s));
        comm->broadcast(buf, bytes, root, cs);
        CSG_CUDA(cudaEventRecord(comm_ev[comm_used++].second, cs.s));
    }
    void reduce_rows(uint64_t *buf, size_t count) {
        comm_events();
        CSG_CUDA(cudaEventRecord(comm_ev[comm_used].first, st.s));
        comm->all_reduce_sum_u64(buf, count, st);
        CSG_CUDA(cudaEventRecord(comm_ev[comm_used++].second, st.s));
    }
    float comm_ms() {
        float total = 0;
        for (size_t i = 0; i < comm_used; i++) {
            float ms = 0;
            CSG_CUDA(cudaEventSynchronize(comm_ev[i].second));
            CSG_CUDA(cudaEventElapsedTime(&ms, comm_ev[i].first, comm_ev[i].second));
            total += ms;
        }
        return total;
    }
    // Out-of-domain evaluation of a sharded proof: every context evaluates the column block it interpolated (the same block of
    // csg_dist_plan), the few hundred values are all-gathered.  vals: `per_col` values for each of this rank's columns; returns
    // the values of all `ncols` columns in column order.
    DBuf<fe> d_ood_xch;
    std::vector<fe> gather_column_values(const std::vector<fe> &mine, size_t per_col, size_t ncols) {
        csg_shard_plan plan;
        shard_plan(rank, G, b, ce, ncols, &plan);
        const size_t cpr = plan.columns_per_rank, slice = cpr * per_col;
        d_ood_xch.reserve(std::max<size_t>(slice * G, 64));
        std::vector<fe> padded(slice, 0);
        std::copy(mine.begin(), mine.end(), padded.begin());
        CSG_CUDA(cudaMemcpyAsync(d_ood_xch.p + rank * slice, padded.data(), slice * sizeof(fe), cudaMemcpyHostToDevice, st.s));
        gather(d_ood_xch.p, slice * sizeof(fe));
        std::vector<fe> all(slice * G);
        CSG_CUDA(cudaMemcpyAsync(all.data(), d_ood_xch.p, all.size() * sizeof(fe), cudaMemcpyDeviceToHost, st.s));
        CSG_CUDA(cudaStreamSynchronize(st.s));
        all.resize(ncols * per_col);   // blocks are consecutive columns; only the last one is padded
        return all;
    }
    // Row digests of a coset-major matrix into the leaves of `nodes`, then the tree.  Sharded: each context hashes the rows
    // of its cosets, the digests are all-gathered and put in natural order, and every context builds the whole tree --
    // 2^23 leaves take 0.35 ms, less than the second exchange that per-GPU subtrees would need to answer the queries.
    void commit_rows(const fe *data, unsigned width, size_t coset_stride, DBuf<uint32_t> &nodes, DBuf<uint32_t> &top) {
        const int hf = (int)opt.hash_fn;
        if (G == 1) {
            nodes.reserve(16 * lde_n);
            hash_rows(data, width, n, (unsigned)b, coset_stride, n, hf, nodes.p + 8 * lde_n, st);
            merkle_build(nodes.p, lde_n, hf, st);
            return;
        }
        if (!subtrees()) {   // a trace shorter than the group: digests all-gathered, the whole (tiny) tree on every context
            nodes.reserve(16 * lde_n);
            d_gather.reserve(4 * lde_n);
            hash_rows(data, width, n, (unsigned)bl, coset_stride, n, hf, (uint32_t *)d_gather.p + 8 * rank * bl * n, st);
            gather(d_gather.p, bl * n * 32);
            interleave_slices(d_gather.p, (uint64_t *)(nodes.p + 8 * lde_n), n, (unsigned)bl, (unsigned)G, 4, st);
            merkle_build(nodes.p, lde_n, hf, st);
            return;
        }
        // Merkle subtrees per GPU (SURVEY.md 8(e)): this context hashed the rows of its cosets, i.e. the leaves j = k + b i of ALL
        // i; the leaves of i in [q n/G, (q+1) n/G) form the contiguous range of rank q, and as hashed ([i][k]) they are one
        // contiguous chunk of the send buffer.  One all-to-all (1/G of the bytes of the all-gather it replaces), the subtree of
        // the own range, an all-gather of the G roots, and the top log2(G) levels on every context.
        const size_t nl = lde_n / G, chunk = (n / G) * bl * 32;
        nodes.reserve(16 * nl); top.reserve(16 * G);
        d_gather.reserve(8 * bl * n);                                      // send and receive buffer: n * bl digests of 4 words each
        uint64_t *send = d_gather.p, *recv = d_gather.p + 4 * bl * n;
        hash_rows(data, width, n, (unsigned)bl, coset_stride, n, hf, (uint32_t *)send, st);
        all_to_all(send, recv, chunk);
        interleave_slices(recv, (uint64_t *)(nodes.p + 8 * nl), n / G, (unsigned)bl, (unsigned)G, 4, st);
        merkle_build(nodes.p, nl, hf, st);
        CSG_CUDA(cudaMemcpyAsync(top.p + 8 * (G + rank), nodes.p + 8, 32, cudaMemcpyDeviceToDevice, st.s));
        gather(top.p + 8 * G, 32);
        merkle_build(top.p, G, hf, st);
    }

    // ------------------------------------------------------------------------------------------ stage 3
    // with a field extension, components 1.. of the coefficients are in h_cargs already (eval_constraints_x); the merged column of
    // component j lands in d_comb[j][ce coset][row]
    void eval_constraints(const fe *t_ab, const fe *b_ab) {
        need(S_COMMITTED, "the trace must be committed first");
        Timer &t = stage_timer;
        t.start(st);
        ConsArgs &A = *h_cargs;
        if (!cargs_domain_ready) {
            // everything that depends on the AIR, the domain and the public inputs only: computed for the first proof after
            // csg_set_air and kept (some 150 host exponentiations and the assertion polynomials -- a fifth of the host time of
            // a one-transaction proof)
            std::vector<size_t> lde_block(cel);
            for (size_t kc = 0; kc < cel; kc++) lde_block[kc] = (kc0 + kc) * (b / ce) - k0;
            fill_domain_args(A, air, tg, bg, n, ce_shift, lde_block, air.width * n);
            std::vector<fe> polys;
            fill_assertion_values(A, air, 0, polys);
            d_apoly.reserve(polys.size() ? polys.size() : 1);
            if (!polys.empty()) {   // pageable source: wait for the copy before `polys` goes away
                CSG_CUDA(cudaMemcpyAsync(d_apoly.p, polys.data(), polys.size() * sizeof(fe), cudaMemcpyHostToDevice, st.s));
                CSG_CUDA(cudaStreamSynchronize(st.s));
            }
            cargs_domain_ready = true;
        }
        A.ext_degree = (unsigned)d;
        for (size_t i = 0; i < air.num_constraints(); i++) { A.alpha[i] = t_ab[2 * i]; A.beta[i] = t_ab[2 * i + 1]; }
        fill_rescue_tables(air.id, A);
        for (size_t i = 0; i < air.assertions.size(); i++) { A.a_alpha[i] = b_ab[2 * i]; A.a_beta[i] = b_ab[2 * i + 1]; }
        host_mark("  cons: coefficient tables");
        d_cargs.reserve(1);
        CSG_CUDA(cudaMemcpyAsync(d_cargs.p, &A, sizeof A, cudaMemcpyHostToDevice, st.s));
        d_comb.reserve((cel ? cel : 1) * n * d);
        d_parts.reserve(constraint_scratch_elements(air.id, n, cel ? cel : 1) * d);
        host_mark("  cons: args upload, scratch");
        if (!cons_ev[0]) for (auto &e : cons_ev) CSG_CUDA(cudaEventCreate(&e));
        // the low-degree splits interpolate across the even cosets: alone, or with an exchange when every rank owns whole pairs
        const bool split = split_low_degree && n >= split_min_rows && (G == 1 || (ce == b && bl % 2 == 0));
        SplitExchange xch{(unsigned)G, (unsigned)rank, [](void *self, void *buf, size_t bytes) { static_cast<csg_ctx *>(self)->gather(buf, bytes); }, this, nullptr, 0};
        if (split && G > 1) {
            d_xch.reserve((size_t)16 * d * (ce / 2) * n);   // <= 16 polynomials per component on the even cosets of the whole proof
            xch.buf = d_xch.p; xch.buf_elems = d_xch.n;
        }
        const SplitExchange *px = split && G > 1 ? &xch : nullptr;
        if (cel && d > 1) csg::eval_constraints_ext(air.id, d_cargs.p, A, d_lde.p, roots.W.p, d_ptab.p, d_apoly.p, d_parts.p, d_comb.p, st, cons_ev,
                                                    split ? &roots : nullptr, split ? &ntt : nullptr, px);
        else if (cel) csg::eval_constraints(air.id, d_cargs.p, A, d_lde.p, roots.W.p, d_ptab.p, d_apoly.p, d_parts.p, d_comb.p, st, cons_ev,
                                            split ? &roots : nullptr, split ? &ntt : nullptr, px);
        else for (auto &e : cons_ev) CSG_CUDA(cudaEventRecord(e, st.s));
        t.stop(st, &tm.constraints);   // (`polys` is pageable memory: its copy was staged before cudaMemcpyAsync returned)
        tm.stage_launches[2] = t.launches;
        float *parts_ms[4] = {&tm.cons_rescue, &tm.cons_ecc_banks, &tm.cons_ecc_final, &tm.cons_rest};
        for (int k = 0; k < 4; k++) t.span(cons_ev[k], cons_ev[k + 1], parts_ms[k]);
        t.span(cons_ev[1], cons_ev[5], &tm.cons_ecc_low);
        stage = S_EVALUATED;
    }
    // E-valued coefficients: the constraint values are base-field elements, so component j of the merged column is the same
    // combination with component j of every coefficient; one pass, every thread accumulates all d components (constraints_ext.cu)
    void eval_constraints_x(const xe *t_ab, const xe *b_ab) {
        const size_t nc = air.num_constraints(), na = air.assertions.size();
        std::vector<fe> tj(2 * nc), bj(2 * na + 2);
        ConsArgs &A = *h_cargs;
        for (int j = 1; j < d; j++) {
            for (size_t i = 0; i < nc; i++) { A.alpha_x[j - 1][i] = t_ab[2 * i].c[j]; A.beta_x[j - 1][i] = t_ab[2 * i + 1].c[j]; }
            for (size_t i = 0; i < na; i++) { A.a_alpha_x[j - 1][i] = b_ab[2 * i].c[j]; A.a_beta_x[j - 1][i] = b_ab[2 * i + 1].c[j]; }
        }
        for (size_t i = 0; i < 2 * nc; i++) tj[i] = t_ab[i].c[0];
        for (size_t i = 0; i < 2 * na; i++) bj[i] = b_ab[i].c[0];
        eval_constraints(tj.data(), bj.data());
    }
    // ------------------------------------------------------------------------------------------ stage 4
    void commit_composition(uint8_t root[32]) {
        need(S_EVALUATED, "constraints must be evaluated first");
        Timer &t = stage_timer;
        t.start(st);
        // per-coset interpolants, divided by s_kc^m; then the cross-coset step yields the ce column polynomials
        std::vector<fe> sinv(cel);
        for (size_t kc = 0; kc < cel; kc++) sinv[kc] = inv(ce_shift[kc]);
        d_e.reserve(ce * n); d_cpolys.reserve(ce * d * n);
        const std::vector<fe> mat = composition_matrix(n, ce);
        // component j of composition column r is the base-field column r*d + j: rows hash as ce elements of E
        for (int j = 0; j < d; j++) {
        const fe *comb = d_comb.p + (size_t)j * (cel ? cel : 1) * n;
        const fe *e_all = d_e.p;
        if (G == 1) coset_intt_columns(roots, ntt, comb, n, d_e.p, n, logn, sinv.data(), ce, st);
        else {
            // every context interpolates on its ce cosets; the slices are all-gathered ("composition slices") and each context
            // runs the small cross-coset step itself.  With more ranks than ce cosets the idle ranks contribute a dummy slice.
            const size_t slot = cel ? cel : 1;
            d_eg.reserve(G * slot * n);
            if (cel) coset_intt_columns(roots, ntt, comb, n, d_eg.p + rank * slot * n, n, logn, sinv.data(), cel, st);
            gather(d_eg.p, slot * n * sizeof(fe));
            if (G <= ce) e_all = d_eg.p;
            else for (size_t kc = 0; kc < ce; kc++)
                CSG_CUDA(cudaMemcpyAsync(d_e.p + kc * n, d_eg.p + kc * (G / ce) * n, n * sizeof(fe), cudaMemcpyDeviceToDevice, st.s));
        }
        composition_columns(e_all, d_cpolys.p + (size_t)j * n, n, (unsigned)ce, mat.data(), st, (size_t)d * n);
        }
        const size_t cw = ce * d;
        d_clde.reserve(cw * n * bl);
        coset_ntt_columns(roots, ntt, d_cpolys.p, n, d_clde.p, n, cw * n, cw, logn, lde_shift.data(), bl, st);
        commit_rows(d_clde.p, (unsigned)cw, cw * n, d_cnodes, d_ctop);
        download_root(subtrees() ? d_ctop : d_cnodes, root);
        t.stop(st, &tm.composition); tm.stage_launches[3] = t.launches;
        stage = S_COMPOSED;
    }

    // ------------------------------------------------------------------------------------------ stage 5 + 6
    void ood(fe z_) {
        need(S_COMPOSED, "the composition polynomial must be committed first");
        Timer &t = stage_timer;
        t.start(st);
        z = z_;
        const size_t w = air.width;
        const fe pts[2] = {z, mul(z, root_of_unity(logn))};
        std::vector<fe> vals(2 * w);
        if (G == 1) eval_polys_at(d_polys.p, n, w, n, pts, 2, vals.data(), scratch2, st);
        else {   // own column block only (1/G of the 0.8 GB of coefficients), then a tiny all-gather: [column][point]
            csg_shard_plan plan;
            shard_plan(rank, G, b, ce, w, &plan);
            const size_t c_lo = plan.first_column, nc = plan.num_columns;
            std::vector<fe> blk(2 * nc), mine(2 * nc);
            if (nc) eval_polys_at(d_polys.p + c_lo * n, n, nc, n, pts, 2, blk.data(), scratch2, st);   // [point][column]
            for (size_t c = 0; c < nc; c++) { mine[2 * c] = blk[c]; mine[2 * c + 1] = blk[nc + c]; }
            const std::vector<fe> all = gather_column_values(mine, 2, w);
            for (size_t c = 0; c < w; c++) { vals[c] = all[2 * c]; vals[w + c] = all[2 * c + 1]; }
        }
        ood_cur.assign(vals.begin(), vals.begin() + w);
        ood_next.assign(vals.begin() + w, vals.end());
        const fe zm = f63::pow(z, ce);
        ood_comp.resize(ce);
        eval_polys_at(d_cpolys.p, n, ce, n, &zm, 1, ood_comp.data(), scratch2, st);
        t.stop(st, &tm.ood_deep); tm.stage_launches[4] = t.launches;
        stage = S_OOD;
    }
    void deep(const fe *trace_ab, const fe *comp_d, fe lambda, fe mu) {
        need(S_OOD, "the out-of-domain frame must be computed first");
        Timer &t = stage_timer;
        t.start(st);
        const size_t w = air.width;
        std::vector<fe> coef(2 * w);
        for (size_t c = 0; c < w; c++) { coef[c] = trace_ab[2 * c]; coef[w + c] = trace_ab[2 * c + 1]; }
        const DeepArgs a = deep_args(z, root_of_unity(logn), ood_cur, ood_next, ood_comp, coef.data(), comp_d, lambda, mu, lde_shift.data(), bl);
        d_abc.reserve(3 * n); d_abc_lde.reserve(3 * n * bl); d_deep.reserve(lde_n);
        combine_polys(d_polys.p, n, w, n, coef.data(), 2, d_abc.p, n, scratch2, st);
        combine_polys(d_cpolys.p, n, ce, n, comp_d, 1, d_abc.p + 2 * n, n, scratch, st);
        coset_ntt_columns(roots, ntt, d_abc.p, n, d_abc_lde.p, n, 3 * n, 3, logn, lde_shift.data(), bl, st);
        if (G == 1) deep_quotients(d_abc_lde.p, roots.W.p, n, a, d_deep.p, st);
        else {   // own rows as [i][kl], all-gather, natural order; FRI then runs whole on every context (layers are <= 64 MB)
            d_gather.reserve(lde_n);
            deep_quotients(d_abc_lde.p, roots.W.p, n, a, (fe *)d_gather.p + rank * bl * n, st);
            gather(d_gather.p, bl * n * sizeof(fe));
            interleave_slices(d_gather.p, (uint64_t *)d_deep.p, n, (unsigned)bl, (unsigned)G, 1, st);
        }
        if (fri.empty()) fri.emplace_back(new FriLayer());
        nfri = 1;
        fri[0]->evals = d_deep.p; fri[0]->m = lde_n; fri[0]->committed = false;
        t.stop(st, &tm.ood_deep, true); tm.stage_launches[4] += t.launches;   // also keeps coef alive until the copies have completed
        t.zero(&tm.fri); tm.stage_launches[5] = 0;
        stage = S_DEEP;
    }

    // ------------------------------------------------------------------------------------------ stage 5 + 6 over E
    void ood_x(const xe &z_) {
        need(S_COMPOSED, "the composition polynomial must be committed first");
        Timer &t = stage_timer;
        t.start(st);
        xz = z_;
        const size_t w = air.width, cw = ce * d;
        const xe pts[2] = {xz, x_scale(xz, root_of_unity(logn))};
        d_pw.reserve(2 * (size_t)d * n);
        ext_power_table(d, pts, 2, n, d_pw.p, st);
        std::vector<fe> vals(w * 2 * d);
        if (G == 1) dot_columns(d_polys.p, n, w, n, d_pw.p, 2 * d, vals.data(), scratch2, st);
        else {   // own column block, then the all-gather of [column][2 d] values
            csg_shard_plan plan;
            shard_plan(rank, G, b, ce, w, &plan);
            const size_t c_lo = plan.first_column, nc = plan.num_columns;
            std::vector<fe> mine(nc * 2 * d);
            if (nc) dot_columns(d_polys.p + c_lo * n, n, nc, n, d_pw.p, 2 * d, mine.data(), scratch2, st);
            vals = gather_column_values(mine, 2 * (size_t)d, w);
        }
        xood_cur.assign(w, x_zero()); xood_next.assign(w, x_zero());
        for (size_t c = 0; c < w; c++)
            for (int j = 0; j < d; j++) { xood_cur[c].c[j] = vals[c * 2 * d + j]; xood_next[c].c[j] = vals[c * 2 * d + d + j]; }
        // composition column r at z^ce: sum_j phi^j * (column (r, j) at z^ce)
        const xe zm = x_pow(d, xz, ce);
        ext_power_table(d, &zm, 1, n, d_pw.p, st);
        std::vector<fe> cv(cw * d);
        dot_columns(d_cpolys.p, n, cw, n, d_pw.p, d, cv.data(), scratch2, st);
        xe phi = x_zero(); phi.c[1] = ONE;
        xood_comp.assign(ce, x_zero());
        for (size_t r = 0; r < ce; r++) {
            xe basis = x_one();
            for (int j = 0; j < d; j++) {
                xe sv = x_zero();
                for (int k = 0; k < d; k++) sv.c[k] = cv[(r * d + j) * d + k];
                xood_comp[r] = x_add(xood_comp[r], x_mul(d, basis, sv));
                basis = x_mul(d, basis, phi);
            }
        }
        t.stop(st, &tm.ood_deep); tm.stage_launches[4] = t.launches;
        stage = S_OOD;
    }
    void deep_x(const xe *trace_ab, const xe *comp_d, const xe &lambda, const xe &mu) {
        need(S_OOD, "the out-of-domain frame must be computed first");
        Timer &t = stage_timer;
        t.start(st);
        const size_t w = air.width, cw = ce * d;
        DeepArgsX a{};
        a.d = d; a.k = xk;
        a.z = xz; a.zg = x_scale(xz, root_of_unity(logn)); a.zm = x_pow(d, xz, ce);
        a.az = x_zero(); a.bzg = x_zero(); a.czm = x_zero();
        std::vector<fe> coef(2 * (size_t)d * w), ccoef((size_t)d * cw);
        for (size_t c = 0; c < w; c++) {
            for (int j = 0; j < d; j++) { coef[(size_t)j * w + c] = trace_ab[2 * c].c[j]; coef[((size_t)d + j) * w + c] = trace_ab[2 * c + 1].c[j]; }
            a.az = x_add(a.az, x_mul(d, trace_ab[2 * c], xood_cur[c]));
            a.bzg = x_add(a.bzg, x_mul(d, trace_ab[2 * c + 1], xood_next[c]));
        }
        xe phi = x_zero(); phi.c[1] = ONE;
        for (size_t r = 0; r < ce; r++) {
            a.czm = x_add(a.czm, x_mul(d, comp_d[r], xood_comp[r]));
            xe cf = comp_d[r];    // delta_r * phi^j multiplies the base-field column (r, j)
            for (int j = 0; j < d; j++) {
                for (int k = 0; k < d; k++) ccoef[(size_t)k * cw + r * d + j] = cf.c[k];
                cf = x_mul(d, cf, phi);
            }
        }
        a.lambda = lambda; a.mu = mu; a.ncosets = (unsigned)bl;
        for (size_t k = 0; k < bl; k++) a.shift[k] = lde_shift[k];
        const size_t np = 3 * (size_t)d;
        d_abc.reserve(np * n); d_abc_lde.reserve(np * n * bl); d_deep.reserve((size_t)d * lde_n);
        combine_polys(d_polys.p, n, w, n, coef.data(), 2 * d, d_abc.p, n, scratch2, st);
        combine_polys(d_cpolys.p, n, cw, n, ccoef.data(), d, d_abc.p + 2 * (size_t)d * n, n, scratch, st);
        coset_ntt_columns(roots, ntt, d_abc.p, n, d_abc_lde.p, n, np * n, np, logn, lde_shift.data(), bl, st);
        if (G == 1) deep_quotients_ext(d_abc_lde.p, roots.W.p, n, a, d_deep.p, lde_n, st);
        else {
            d_gather.reserve((size_t)d * lde_n);
            deep_quotients_ext(d_abc_lde.p, roots.W.p, n, a, (fe *)d_gather.p + rank * bl * n, lde_n, st);
            for (int j = 0; j < d; j++) {
                gather(d_gather.p + (size_t)j * lde_n, bl * n * sizeof(fe));
                interleave_slices(d_gather.p + (size_t)j * lde_n, (uint64_t *)d_deep.p + (size_t)j * lde_n, n, (unsigned)bl, (unsigned)G, 1, st);
            }
        }
        if (fri.empty()) fri.emplace_back(new FriLayer());
        nfri = 1;
        fri[0]->evals = d_deep.p; fri[0]->m = lde_n; fri[0]->committed = false;
        t.stop(st, &tm.ood_deep, true); tm.stage_launches[4] += t.launches;
        t.zero(&tm.fri); tm.stage_launches[5] = 0;
        stage = S_DEEP;
    }

    // ------------------------------------------------------------------------------------------ stage 7
    void fri_commit_layer(uint8_t root[32]) {
        need(S_DEEP, "the DEEP composition must be computed first");
        FriLayer &L = *fri[nfri - 1];
        Timer &t = stage_timer;
        t.start(st);
        const size_t q = L.m / 4;
        L.nodes.reserve(16 * q);
        if (d == 1) hash_rows(L.evals, 4, q, 1, 0, q, (int)opt.hash_fn, L.nodes.p + 8 * q, st);
        else hash_rows(L.evals, 4 * d, q, 1, 0, q, (int)opt.hash_fn, L.nodes.p + 8 * q, st, (unsigned)d, L.m);   // rows of 4 elements of E; planes of stride m
        merkle_build(L.nodes.p, q, (int)opt.hash_fn, st);
        download_root(L.nodes, root);
        L.committed = true;
        t.stop(st, &tm.fri, true); tm.stage_launches[5] += t.launches;
    }
    void fri_fold(fe alpha) { fri_fold_x(x_from(alpha)); }
    void fri_fold_x(const xe &alpha) {
        need(S_DEEP, "the DEEP composition must be computed first");
        FriLayer &L = *fri[nfri - 1];
        if (!L.committed) throw StateError("the current FRI layer must be committed before it is folded");
        Timer &t = stage_timer;
        t.start(st);
        const size_t m = L.m, q = m / 4;
        FoldArgs a = fold_args(m, roots.logn);
        a.alpha = alpha.c[0];
        if (fri.size() == nfri) fri.emplace_back(new FriLayer());
        FriLayer &N = *fri[nfri];
        N.owned.reserve(q * d);
        if (d == 1) csg::fri_fold4(L.evals, m, roots.W.p, a, N.owned.p, st);
        else { FoldArgsX ax{a, alpha, d}; fri_fold4_ext(L.evals, m, m, roots.W.p, ax, N.owned.p, q, st); }
        N.evals = N.owned.p; N.m = q; N.committed = false;
        nfri++;
        t.stop(st, &tm.fri, true); tm.stage_launches[5] += t.launches;
    }
    size_t num_fri_folds() const { return csg::num_fri_folds(lde_n, opt); }

    // ------------------------------------------------------------------------------------------ the whole of Prover::prove
    void write_context(Bytes &w) const { write_proof_context(w, air.width, logn, opt); }
    // flattened components of E elements (serialisation / hashing order)
    std::vector<fe> flat(const std::vector<xe> &v) const {
        std::vector<fe> out;
        for (const xe &e : v) for (int j = 0; j < d; j++) out.push_back(e.c[j]);
        return out;
    }
    void prove_loaded(uint8_t **proof, size_t *proof_len, const uint64_t *host = nullptr, int host_repr = CSG_REPR_CANONICAL, const uint64_t *const *host_cols = nullptr) {
        if (!host && !host_cols) need(S_TRACE, "csg_load_trace must be called first");
        auto t0 = std::chrono::steady_clock::now();
        HostTraceScope trace(t0);
        const unsigned long long launches0 = st.launches;
        stage_timer.discard(); query_timer.discard();
        comm_used = 0;
        const size_t w = air.width, nc = air.num_constraints(), na = air.assertions.size();
        Bytes context;
        write_context(context);
        ProofTranscript tr((int)opt.hash_fn, d, air.pub_inputs.data(), air.pub_inputs.size(), context.v.data(), context.v.size());
        auto base = [](const std::vector<xe> &v) { std::vector<fe> o; for (const xe &e : v) o.push_back(e.c[0]); return o; };

        uint8_t trace_root[32], comp_root[32];
        host_mark("setup");
        extend_and_commit_trace(trace_root, host, host_repr, host_cols);
        host_mark("extend+commit trace");
        const ProofTranscript::ConstraintCoefficients cc = tr.constraint_coefficients(trace_root, nc, na);
        host_mark("draw coefficients");
        if (d == 1) eval_constraints(base(cc.transition).data(), base(cc.boundary).data());
        else eval_constraints_x(cc.transition.data(), cc.boundary.data());
        host_mark("constraints (enqueue)");
        commit_composition(comp_root);
        host_mark("composition + commit");

        const xe zz = tr.ood_point(comp_root);
        if (d == 1) ood(zz.c[0]);
        else ood_x(zz);
        const std::vector<fe> f_cur = d == 1 ? ood_cur : flat(xood_cur), f_next = d == 1 ? ood_next : flat(xood_next),
                              f_comp = d == 1 ? ood_comp : flat(xood_comp);
        const ProofTranscript::DeepCoefficients dc = tr.deep_coefficients(f_cur.data(), f_next.data(), w, f_comp.data(), ce);
        host_mark("out-of-domain frame");
        if (d == 1) deep(base(dc.trace).data(), base(dc.comp).data(), dc.lambda.c[0], dc.mu.c[0]);
        else deep_x(dc.trace.data(), dc.comp.data(), dc.lambda, dc.mu);
        host_mark("deep (enqueue)");

        const size_t nlayers = num_fri_folds() + 1;
        std::vector<std::vector<uint8_t>> fri_roots(nlayers, std::vector<uint8_t>(32));
        for (size_t l = 0; l < nlayers; l++) {
            fri_commit_layer(fri_roots[l].data());
            const xe alpha = tr.fri_alpha(fri_roots[l].data());
            if (l + 1 < nlayers) fri_fold_x(alpha);
        }
        host_mark("fri layers");

        Timer &tq = query_timer;
        tq.start(st);
        const uint64_t nonce = tr.grind(opt.grinding_factor);
        const std::vector<size_t> pos = tr.query_positions(opt.num_queries, lde_n);
        host_mark("grinding + positions");

        // every opening of the proof -- trace rows, composition rows, FRI layer rows, their Merkle paths, the remainder -- is
        // planned on the host first and fetched in ONE round trip (one index upload, a handful of gather launches, one download)
        OpenBatch B;
        const Opening o_trace = plan_trace_opening(B, pos);
        const Opening o_comp = plan_composition_opening(B, pos);
        std::vector<Opening> o_fri;
        {
            std::vector<size_t> fp = pos;
            size_t domain = lde_n;
            for (size_t l = 0; l + 1 < nlayers; l++) {
                fp = fold_positions(fp, domain);
                o_fri.push_back(plan_fri_opening(B, *fri[l], fp));
                domain /= 4;
            }
        }
        const FriLayer &last = *fri[nlayers - 1];
        const size_t rem_off = plan_remainder(B, last), rem_len = last.m * d;
        std::vector<uint64_t> rows;
        std::vector<uint8_t> digs;
        host_mark("plan openings");
        run_openings(B, rows, digs);
        host_mark("openings round trip");
        Bytes pf;
        pf.v.reserve(256 * 1024);
        std::vector<const uint8_t *> fri_root_ptrs;
        for (auto &r : fri_roots) fri_root_ptrs.push_back(r.data());
        write_proof(pf, (unsigned)w, logn, opt, trace_root, comp_root, fri_root_ptrs, o_trace, o_comp, o_fri, rows.data(), digs.data(), f_cur, f_next, f_comp,
                    rem_off, rem_len, nonce);
        tq.stop(st, &tm.queries); tm.stage_launches[6] = tq.launches;
        host_mark("serialise");
        tm.kernel_launches = st.launches - launches0;
        tm.comm = comm_ms();
        tm.total = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();

        *proof = (uint8_t *)malloc(pf.v.size());
        if (!*proof) throw std::bad_alloc();
        memcpy(*proof, pf.v.data(), pf.v.size());
        *proof_len = pf.v.size();
        host_mark("timers + copy out");
        trace.print("[csg host trace] %zu x %zu, %llu launches\n", (size_t)air.width, n, (unsigned long long)tm.kernel_launches);
        stage = S_TRACE;   // the resident trace (d_io) can be proved again
    }
    // ---- batched openings
    struct OpenBatch {
        struct Rows { const fe *data; unsigned width, ncosets; size_t coset_stride, col_stride; unsigned sub; size_t sub_stride, idx_off, npos, rows_off; };
        struct Digs { const uint32_t *nodes, *top; size_t idx_off, count, dig_off; };
        std::vector<uint32_t> idx;   // row positions and node indices of every job, concatenated
        std::vector<Rows> rows;
        std::vector<Digs> digs;
        size_t rows_words = 0, dig_count = 0, sharded_words = 0, sharded_digs = 0;   // sharded_*: leading parts summed across the ranks
        const FriLayer *rem = nullptr;   // the remainder, if planned (plan_remainder), at rows[rem_off ..)
        size_t rem_off = 0;
    };
    // rows of `data` at `pos` (sharded matrices first: their rows are summed across the ranks in one go) and the batch opening
    // of the same positions in the tree `nodes`
    Opening plan_opening(OpenBatch &B, const fe *data, unsigned width, unsigned ncosets, size_t coset_stride, size_t col_stride, unsigned sub, size_t sub_stride,
                         bool sharded, const uint32_t *nodes, size_t nleaves, const std::vector<size_t> &pos, const uint32_t *top = nullptr) {
        Opening o;
        sharded = sharded && G > 1;
        OpenBatch::Rows r{data, width, sharded ? (unsigned)bl : ncosets, coset_stride, col_stride, sub ? sub : 1, sub_stride, B.idx.size(), pos.size(), B.rows_words};
        for (size_t p : pos) {
            uint32_t v = (uint32_t)p;
            if (sharded) { const size_t k = p % b, i = p / b; v = (k >= k0 && k < k0 + bl) ? (uint32_t)((k - k0) + bl * i) : 0xFFFFFFFFu; }
            B.idx.push_back(v);
        }
        o.rows_off = B.rows_words; o.rows_len = pos.size() * width;
        B.rows_words += o.rows_len;
        if (sharded) { if (B.sharded_words != o.rows_off) throw StateError("sharded openings must be planned first"); B.sharded_words = B.rows_words; }
        B.rows.push_back(r);
        o.slots = batch_opening_nodes(nleaves, pos);
        OpenBatch::Digs dj{nodes, top, B.idx.size(), 0, B.dig_count};
        for (auto &sl : o.slots) { for (uint32_t v : sl) B.idx.push_back(top ? tree_ref(v) : v); dj.count += sl.size(); }
        o.dig_off = B.dig_count;
        B.dig_count += dj.count;
        if (top) { if (B.sharded_digs != o.dig_off) throw StateError("openings of sharded trees must be planned first"); B.sharded_digs = B.dig_count; }
        B.digs.push_back(dj);
        return o;
    }
    // the openings of the committed matrices: sharded ones first (plan_opening)
    Opening plan_trace_opening(OpenBatch &B, const std::vector<size_t> &pos) {
        return plan_opening(B, d_lde.p, (unsigned)air.width, (unsigned)b, air.width * n, n, 1, 0, true, d_tnodes.p, lde_n, pos, subtrees() ? d_ttop.p : nullptr);
    }
    Opening plan_composition_opening(OpenBatch &B, const std::vector<size_t> &pos) {
        const size_t cw = ce * d;
        return plan_opening(B, d_clde.p, (unsigned)cw, (unsigned)b, cw * n, n, 1, 0, true, d_cnodes.p, lde_n, pos, subtrees() ? d_ctop.p : nullptr);
    }
    // rows of 4 elements of E, each d components (planes of stride m)
    Opening plan_fri_opening(OpenBatch &B, const FriLayer &L, const std::vector<size_t> &pos) {
        const size_t q = L.m / 4;
        return plan_opening(B, L.evals, 4 * (unsigned)d, 1, 0, q, (unsigned)d, d == 1 ? 0 : L.m, false, L.nodes.p, q, pos);
    }
    // the last FRI layer in natural order, canonical, components of an element adjacent: returns where it sits among the opened words
    size_t plan_remainder(OpenBatch &B, const FriLayer &last) {
        B.rem = &last; B.rem_off = B.rows_words;
        B.rows_words += last.m * d;
        return B.rem_off;
    }
    void run_openings(const OpenBatch &B, std::vector<uint64_t> &rows, std::vector<uint8_t> &digs) {
        d_idx.reserve(std::max<size_t>(B.idx.size(), 1 << 16));
        d_rows.reserve(std::max<size_t>(B.rows_words, 1 << 17));
        d_dig.reserve(std::max<size_t>(B.dig_count * 8, 8 << 16));
        if (!B.idx.empty()) CSG_CUDA(cudaMemcpyAsync(d_idx.p, B.idx.data(), B.idx.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st.s));
        for (auto &r : B.rows)
            gather_rows(r.data, r.width, r.ncosets, r.coset_stride, r.col_stride, d_idx.p + r.idx_off, r.npos, d_rows.p + r.rows_off, st, r.sub, r.sub_stride);
        if (B.sharded_words) reduce_rows(d_rows.p, B.sharded_words);
        for (auto &g : B.digs) gather_digests(g.nodes, d_idx.p + g.idx_off, g.count, d_dig.p + 8 * g.dig_off, st, g.top);
        if (B.sharded_digs) reduce_rows((uint64_t *)d_dig.p, B.sharded_digs * 4);
        if (B.rem && d == 1) from_montgomery(B.rem->evals, d_rows.p + B.rem_off, B.rem->m, st);
        else if (B.rem) planes_to_canonical(B.rem->evals, B.rem->m, B.rem->m, d, d_rows.p + B.rem_off, st);
        rows.resize(B.rows_words); digs.resize(B.dig_count * 32);
        CSG_CUDA(cudaMemcpyAsync(rows.data(), d_rows.p, rows.size() * 8, cudaMemcpyDeviceToHost, st.s));
        if (!digs.empty()) CSG_CUDA(cudaMemcpyAsync(digs.data(), d_dig.p, digs.size(), cudaMemcpyDeviceToHost, st.s));
        CSG_CUDA(cudaStreamSynchronize(st.s));
    }
};

// ================================================================================================ C ABI
namespace csg_abi {
template <class F>
int guarded(csg_ctx *ctx, F f) {
    if (!ctx) return CSG_ERR_ARG;
    try {
        CSG_CUDA(cudaSetDevice(ctx->device));
        f();
        return CSG_OK;
    } catch (const ArgError &e) { ctx->err = e.what(); return CSG_ERR_ARG; }
    catch (const StateError &e) { ctx->err = e.what(); return CSG_ERR_STATE; }
    catch (const CudaError &e) { ctx->err = e.what(); return CSG_ERR_CUDA; }
    catch (const std::exception &e) { ctx->err = e.what(); return CSG_ERR_UNSUPPORTED; }
}
inline std::vector<fe> mont_vec(const uint64_t *v, size_t n) { std::vector<fe> r(n); for (size_t i = 0; i < n; i++) r[i] = to_mont(v[i] % P); return r; }
// n elements of E, d canonical words each
inline std::vector<xe> mont_xvec(const uint64_t *v, size_t n, int d) {
    std::vector<xe> r(n, x_zero());
    for (size_t i = 0; i < n; i++) for (int j = 0; j < d; j++) r[i].c[j] = to_mont(v[i * d + j] % P);
    return r;
}
}  // namespace csg_abi
using namespace csg_abi;
