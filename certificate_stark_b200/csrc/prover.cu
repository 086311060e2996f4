// libcsg: the C ABI of include/csg.h, levels 1 and 2 -- context life cycle, csg_prove*, the per-stage calls, openings.
// The context itself (every stage of Prover::prove) is prover_ctx.cuh.
#include "prover_ctx.cuh"

extern "C" {

csg_ctx *csg_create(int device) {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) return nullptr;
    if (cudaSetDevice(device) != cudaSuccess) return nullptr;
    csg_ctx *ctx = new csg_ctx();
    ctx->device = device;
    if (cudaStreamCreateWithFlags(&ctx->st.s, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return nullptr; }
    return ctx;
}
void csg_destroy(csg_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->st.s);
    cudaStream_t s = ctx->st.s;
    if (ctx->ev_a) { cudaEventDestroy(ctx->ev_a); cudaEventDestroy(ctx->ev_b); }
    for (auto e : ctx->cons_ev) if (e) cudaEventDestroy(e);
    for (auto e : ctx->chunk_ev) cudaEventDestroy(e);
    for (auto &e : ctx->comm_ev) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
    if (ctx->ev_intt) { cudaEventDestroy(ctx->ev_intt); cudaEventDestroy(ctx->ev_gathered); }
    if (ctx->comm_stream.s) { cudaStreamSynchronize(ctx->comm_stream.s); cudaStreamDestroy(ctx->comm_stream.s); }
    ctx->comm.reset();
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    for (auto b : ctx->stage_buf) if (b) cudaFreeHost(b);
    for (auto e : ctx->stage_ev) if (e) cudaEventDestroy(e);
    if (ctx->h2d_a) { cudaEventDestroy(ctx->h2d_a); cudaEventDestroy(ctx->h2d_b); }
    many_delete(ctx->many);
    delete ctx;
    cudaStreamDestroy(s);
}
const char *csg_last_error(const csg_ctx *ctx) { return ctx ? ctx->err.c_str() : "no context (CUDA device unavailable)"; }
void csg_free(void *p) { free(p); }

int csg_set_air(csg_ctx *ctx, int air_id, size_t trace_len, const csg_options *opt, const uint64_t *pub, size_t npub) {
    return guarded(ctx, [&] { ctx->set_air(air_id, trace_len, opt, pub, npub); });
}
int csg_load_trace(csg_ctx *ctx, const uint64_t *trace, int repr) { return guarded(ctx, [&] { if (!trace) throw ArgError("null trace"); ctx->load_trace(trace, repr); }); }
int csg_reload_resident_trace(csg_ctx *ctx) { return guarded(ctx, [&] { ctx->reload_resident(); }); }
int csg_prove_loaded(csg_ctx *ctx, uint8_t **proof, size_t *proof_len) {
    return guarded(ctx, [&] { if (!proof || !proof_len) throw ArgError("null output"); ctx->prove_loaded(proof, proof_len); });
}
int csg_prove(csg_ctx *ctx, int air_id, const uint64_t *trace, int repr, size_t trace_len, const uint64_t *pub, size_t npub, const csg_options *opt,
              uint8_t **proof, size_t *proof_len) {
    return guarded(ctx, [&] {
        if (!trace || !proof || !proof_len) throw ArgError("null argument");
        csg_ctx::check_repr(repr);
        ctx->set_air(air_id, trace_len, opt, pub, npub);
        ctx->prove_loaded(proof, proof_len, trace, repr);
    });
}
int csg_prove_trace(csg_ctx *ctx, const uint64_t *trace, int repr, uint8_t **proof, size_t *proof_len) {
    return guarded(ctx, [&] {
        if (!trace || !proof || !proof_len) throw ArgError("null argument");
        csg_ctx::check_repr(repr);
        ctx->need(S_AIR, "csg_set_air must be called first");
        ctx->prove_loaded(proof, proof_len, trace, repr);
    });
}
int csg_prefetch_trace(csg_ctx *ctx, const uint64_t *trace, int repr) { return guarded(ctx, [&] { ctx->prefetch_trace(trace, repr); }); }
int csg_prove_prefetched(csg_ctx *ctx, const uint64_t *next_trace, int next_repr, uint8_t **proof, size_t *proof_len) {
    return guarded(ctx, [&] {
        if (!proof || !proof_len) throw ArgError("null argument");
        ctx->prove_prefetched(next_trace, next_repr, proof, proof_len);
    });
}
// the same with one pointer per column: a winterfell TraceTable keeps each column in its own Vec
int csg_prove_columns(csg_ctx *ctx, int air_id, const uint64_t *const *columns, int repr, size_t trace_len, const uint64_t *pub, size_t npub,
                      const csg_options *opt, uint8_t **proof, size_t *proof_len) {
    return guarded(ctx, [&] {
        if (!columns || !proof || !proof_len) throw ArgError("null argument");
        csg_ctx::check_repr(repr);
        ctx->set_air(air_id, trace_len, opt, pub, npub);
        ctx->prove_loaded(proof, proof_len, nullptr, repr, columns);
    });
}
// K independent proofs of one AIR, length and options through one launch sequence (many/prove_many.cu).  The single-proof state
// (AIR, resident and prefetched traces) is left alone; only the timings are the batch's.
static int prove_many(csg_ctx *ctx, int air_id, size_t count, ManyTraces traces, int repr, size_t trace_len, const uint64_t *pubs, size_t npub,
                      const csg_options *opt, uint8_t **proofs, size_t *proof_lens) {
    if (proofs && proof_lens)   // the caller's arrays hold count entries
        for (size_t k = 0; k < count; k++) { proofs[k] = nullptr; proof_lens[k] = 0; }
    return guarded(ctx, [&] {
        if (ctx->comm && ctx->comm->world > 1) throw std::runtime_error("csg_prove_many does not run on a context attached to a group");
        if (!ctx->many) ctx->many = many_new();
        ctx->stage_timer.discard(); ctx->query_timer.discard();   // csg_get_timings reports the batch
        try { many_prove(ctx->many, ctx->st, air_id, count, traces, repr, trace_len, pubs, npub, opt, proofs, proof_lens, ctx->tm); }
        catch (const ManyArgError &e) { throw ArgError(e.what()); }
    });
}
int csg_prove_many(csg_ctx *ctx, int air_id, size_t count, const uint64_t *const *traces, int repr, size_t trace_len, const uint64_t *pubs, size_t npub,
                   const csg_options *opt, uint8_t **proofs, size_t *proof_lens) {
    return prove_many(ctx, air_id, count, ManyTraces{traces, nullptr}, repr, trace_len, pubs, npub, opt, proofs, proof_lens);
}
// the same with the K traces in one device buffer [count][width][trace_len] on the context's device, read in place
int csg_prove_many_device(csg_ctx *ctx, int air_id, size_t count, const uint64_t *traces_dev, int repr, size_t trace_len, const uint64_t *pubs,
                          size_t npub, const csg_options *opt, uint8_t **proofs, size_t *proof_lens) {
    return prove_many(ctx, air_id, count, ManyTraces{nullptr, traces_dev}, repr, trace_len, pubs, npub, opt, proofs, proof_lens);
}
// page-locked host memory for traces: the H2D copy of csg_prove / csg_prove_trace then runs at link speed under the extension
void *csg_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (!bytes || cudaHostAlloc(&p, bytes, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void csg_host_free(void *p) { if (p) cudaFreeHost(p); }
int csg_host_register(void *p, size_t bytes) {
    if (!p || !bytes) return CSG_ERR_ARG;
    if (cudaHostRegister(p, bytes, cudaHostRegisterDefault) != cudaSuccess) { cudaGetLastError(); return CSG_ERR_CUDA; }
    return CSG_OK;
}
int csg_host_unregister(void *p) {
    if (!p) return CSG_ERR_ARG;
    if (cudaHostUnregister(p) != cudaSuccess) { cudaGetLastError(); return CSG_ERR_CUDA; }
    return CSG_OK;
}
int csg_extend_and_commit_trace(csg_ctx *ctx, uint8_t root[32]) { return guarded(ctx, [&] { ctx->extend_and_commit_trace(root); }); }
int csg_eval_constraints(csg_ctx *ctx, const uint64_t *t_coeffs, const uint64_t *b_coeffs) {
    return guarded(ctx, [&] {
        ctx->need(S_AIR, "csg_set_air must be called first");
        if (ctx->d > 1) {
            std::vector<xe> t = mont_xvec(t_coeffs, 2 * ctx->air.num_constraints(), ctx->d), bb = mont_xvec(b_coeffs, 2 * ctx->air.assertions.size(), ctx->d);
            bb.push_back(x_zero());
            ctx->eval_constraints_x(t.data(), bb.data());
            return;
        }
        std::vector<fe> t = mont_vec(t_coeffs, 2 * ctx->air.num_constraints()), bb = mont_vec(b_coeffs, 2 * ctx->air.assertions.size());
        bb.push_back(0);
        ctx->eval_constraints(t.data(), bb.data());
    });
}
int csg_commit_composition(csg_ctx *ctx, uint8_t root[32]) { return guarded(ctx, [&] { ctx->commit_composition(root); }); }
int csg_ood_ext(csg_ctx *ctx, const uint64_t *z, uint64_t *frame_cur, uint64_t *frame_next, uint64_t *comp) {
    return guarded(ctx, [&] {
        if (!z || !frame_cur || !frame_next || !comp) throw ArgError("null argument");
        const int d = ctx->d;
        if (d == 1) { csg_ctx *c = ctx; c->ood(to_mont(z[0] % P)); for (size_t i = 0; i < c->air.width; i++) { frame_cur[i] = from_mont(c->ood_cur[i]); frame_next[i] = from_mont(c->ood_next[i]); }
                      for (size_t r = 0; r < c->ce; r++) comp[r] = from_mont(c->ood_comp[r]); return; }
        ctx->ood_x(mont_xvec(z, 1, d)[0]);
        for (size_t c = 0; c < ctx->air.width; c++)
            for (int j = 0; j < d; j++) { frame_cur[c * d + j] = from_mont(ctx->xood_cur[c].c[j]); frame_next[c * d + j] = from_mont(ctx->xood_next[c].c[j]); }
        for (size_t r = 0; r < ctx->ce; r++) for (int j = 0; j < d; j++) comp[r * d + j] = from_mont(ctx->xood_comp[r].c[j]);
    });
}
int csg_ood(csg_ctx *ctx, uint64_t z, uint64_t *frame_cur, uint64_t *frame_next, uint64_t *comp) {
    return guarded(ctx, [&] {
        if (ctx->d != 1) throw ArgError("with a field extension the out-of-domain point has several words: use csg_ood_ext");
        ctx->ood(to_mont(z % P));
        for (size_t c = 0; c < ctx->air.width; c++) { frame_cur[c] = from_mont(ctx->ood_cur[c]); frame_next[c] = from_mont(ctx->ood_next[c]); }
        for (size_t r = 0; r < ctx->ce; r++) comp[r] = from_mont(ctx->ood_comp[r]);
    });
}
int csg_deep(csg_ctx *ctx, const uint64_t *trace_ab, const uint64_t *comp_d, const uint64_t lambda_mu[2]) {
    return guarded(ctx, [&] {
        ctx->need(S_AIR, "csg_set_air must be called first");
        if (ctx->d > 1) {
            std::vector<xe> ab = mont_xvec(trace_ab, 2 * ctx->air.width, ctx->d), dd = mont_xvec(comp_d, ctx->ce, ctx->d), lm = mont_xvec(lambda_mu, 2, ctx->d);
            ctx->deep_x(ab.data(), dd.data(), lm[0], lm[1]);
            return;
        }
        std::vector<fe> ab = mont_vec(trace_ab, 2 * ctx->air.width), d = mont_vec(comp_d, ctx->ce);
        ctx->deep(ab.data(), d.data(), to_mont(lambda_mu[0] % P), to_mont(lambda_mu[1] % P));
    });
}
int csg_fri_commit_layer(csg_ctx *ctx, uint8_t root[32]) { return guarded(ctx, [&] { ctx->fri_commit_layer(root); }); }
int csg_fri_fold(csg_ctx *ctx, uint64_t alpha) {
    return guarded(ctx, [&] { if (ctx->d != 1) throw ArgError("with a field extension alpha has several words: use csg_fri_fold_ext"); ctx->fri_fold(to_mont(alpha % P)); });
}
int csg_fri_fold_ext(csg_ctx *ctx, const uint64_t *alpha) {
    return guarded(ctx, [&] { if (!alpha) throw ArgError("null argument"); ctx->fri_fold_x(mont_xvec(alpha, 1, ctx->d)[0]); });
}
int csg_fri_remainder(csg_ctx *ctx, uint64_t *out, size_t cap, size_t *len) {
    return guarded(ctx, [&] {
        ctx->need(S_DEEP, "the DEEP composition must be computed first");
        const FriLayer &L = *ctx->fri[ctx->nfri - 1];
        if (cap < L.m * ctx->d) throw ArgError("remainder buffer too small");
        std::vector<uint64_t> rem = ctx->remainder();
        memcpy(out, rem.data(), rem.size() * 8);
        *len = rem.size();
    });
}
// query positions handed in by the caller's coin: at most 255 (the slot count of a batch opening is one byte), distinct, inside the tree
static std::vector<size_t> checked_positions(const uint64_t *positions, size_t npos, size_t nleaves) {
    if (!positions || npos == 0 || npos > 255) throw ArgError("between 1 and 255 query positions");
    std::vector<size_t> pos(positions, positions + npos);
    std::vector<size_t> sorted(pos);
    std::sort(sorted.begin(), sorted.end());
    if (sorted.back() >= nleaves) throw ArgError("query position outside the evaluation domain");
    if (std::adjacent_find(sorted.begin(), sorted.end()) != sorted.end()) throw ArgError("query positions must be distinct");
    return pos;
}
static void copy_opening(const std::vector<uint64_t> &r, const std::vector<uint8_t> &p, uint64_t *rows, uint8_t *paths, size_t cap, size_t *paths_len) {
    if (!rows || !paths || !paths_len) throw ArgError("null output");
    if (p.size() > cap) throw ArgError("path buffer too small");
    memcpy(rows, r.data(), r.size() * 8);
    memcpy(paths, p.data(), p.size());
    *paths_len = p.size();
}
int csg_open_trace(csg_ctx *ctx, const uint64_t *positions, size_t npos, uint64_t *rows, uint8_t *paths, size_t cap, size_t *paths_len) {
    return guarded(ctx, [&] {
        ctx->need(S_COMMITTED, "the trace must be committed first");
        std::vector<size_t> pos = checked_positions(positions, npos, ctx->lde_n);
        const size_t w = ctx->air.width;
        copy_opening(ctx->open_rows(ctx->d_lde.p, (unsigned)w, (unsigned)ctx->b, w * ctx->n, ctx->n, pos, true), ctx->open_paths(ctx->d_tnodes, ctx->lde_n, pos, ctx->subtrees() ? &ctx->d_ttop : nullptr), rows, paths, cap, paths_len);
    });
}
int csg_open_composition(csg_ctx *ctx, const uint64_t *positions, size_t npos, uint64_t *rows, uint8_t *paths, size_t cap, size_t *paths_len) {
    return guarded(ctx, [&] {
        ctx->need(S_COMPOSED, "the composition polynomial must be committed first");
        std::vector<size_t> pos = checked_positions(positions, npos, ctx->lde_n);
        const size_t cw = ctx->ce * ctx->d;
        copy_opening(ctx->open_rows(ctx->d_clde.p, (unsigned)cw, (unsigned)ctx->b, cw * ctx->n, ctx->n, pos, true), ctx->open_paths(ctx->d_cnodes, ctx->lde_n, pos, ctx->subtrees() ? &ctx->d_ctop : nullptr), rows, paths, cap, paths_len);
    });
}
int csg_open_fri_layer(csg_ctx *ctx, size_t layer, const uint64_t *positions, size_t npos, uint64_t *rows, uint8_t *paths, size_t cap, size_t *paths_len) {
    return guarded(ctx, [&] {
        ctx->need(S_DEEP, "the DEEP composition must be computed first");
        if (layer >= ctx->nfri || !ctx->fri[layer]->committed) throw ArgError("no such committed FRI layer");
        const FriLayer &L = *ctx->fri[layer];
        std::vector<size_t> pos = checked_positions(positions, npos, L.m / 4);
        copy_opening(ctx->open_fri_rows(L, pos), ctx->open_paths(L.nodes, L.m / 4, pos), rows, paths, cap, paths_len);
    });
}
// debugging aid: number of elements >= p in an internal device buffer (0 = trace polys, 1 = LDE, 2 = periodic tables,

}  // extern "C"
