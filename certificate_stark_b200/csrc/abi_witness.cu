// libcsg: device-side witnesses and batch metadata, timers and the sharding entry points of include/csg.h.
#include "prover_ctx.cuh"

// the batch witness builders below: csg_get_timings then reports the build, its kernel launches and wall time
template <class F>
static int build_traces_many(csg_ctx *ctx, F build) {
    return guarded(ctx, [&] {
        if (!ctx->many) ctx->many = many_new();
        const auto t0 = std::chrono::steady_clock::now();
        const unsigned long long launches0 = ctx->st.launches;
        try { build(); }
        catch (const ManyArgError &e) { throw ArgError(e.what()); }
        ctx->stage_timer.discard(); ctx->query_timer.discard();
        ctx->tm = csg_timings{};
        ctx->tm.kernel_launches = ctx->st.launches - launches0;
        ctx->tm.total = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    });
}

extern "C" {

int csg_build_trace_transaction_device(csg_ctx *ctx, const csg_tx_batch *b) {
    return guarded(ctx, [&] {
        ctx->need(S_AIR, "csg_set_air must be called first");
        if (!b) throw ArgError("null batch");
        const size_t ntx = csg_tx_batch_size(b);
        if (ctx->air.id != CSG_AIR_TRANSACTION || ctx->n != ntx * 1024) throw ArgError("the AIR set on this context is not the transaction AIR of this batch size");
        if (csg_tx_batch_depth(b) != 15) throw ArgError("the transaction AIR is built for tree depth 15");
        // the packed record of a batch does not change: pack once per batch object (the message hashes cost ~0.2 ms each)
        std::vector<uint64_t> &packed = ctx->wit_packed;
        if (ctx->wit_packed_for != b || packed.size() != csg_tx_batch_pack(b, nullptr)) {
            packed.resize(csg_tx_batch_pack(b, nullptr));
            csg_tx_batch_pack(b, packed.data());
            ctx->wit_packed_for = b;
        }
        ctx->wit_resident_ntx = 0;   // d_wit_in is overwritten below
        Timer &t = ctx->stage_timer;
        t.start(ctx->st);
        DBuf<uint64_t> &in = ctx->d_wit_in;
        in.reserve(packed.size()); ctx->d_wit_finals.reserve(ntx * 48); ctx->d_io.reserve((size_t)ctx->air.width * ctx->n);
        CSG_CUDA(cudaMemcpyAsync(in.p, packed.data(), packed.size() * 8, cudaMemcpyHostToDevice, ctx->st.s));
        build_transaction_trace(in.p, ntx, 15, ctx->d_io.p, ctx->d_wit_finals.p, ctx->st);
        ctx->trace_repr = CSG_REPR_CANONICAL;
        ctx->tm.h2d = t.stop(ctx->st);   // here: witness generation time
        ctx->nfri = 0;
        ctx->stage = S_TRACE;
    });
}
// the standalone provers of the Merkle-update and Schnorr sub-AIRs on the device (same records, same kernels)
static void upload_records(csg_ctx *ctx, std::vector<uint64_t> &packed) {
    ctx->d_wit_in.reserve(packed.size());
    CSG_CUDA(cudaMemcpyAsync(ctx->d_wit_in.p, packed.data(), packed.size() * 8, cudaMemcpyHostToDevice, ctx->st.s));
    ctx->wit_resident_ntx = 0; ctx->wit_packed_for = nullptr;
}
int csg_build_trace_merkle_update_device(csg_ctx *ctx, const csg_tx_batch *b) {
    return guarded(ctx, [&] {
        ctx->need(S_AIR, "csg_set_air must be called first");
        if (!b) throw ArgError("null batch");
        const size_t ntx = csg_tx_batch_size(b);
        if (ctx->air.id != CSG_AIR_MERKLE_UPDATE || ctx->n != ntx * 512) throw ArgError("the AIR set on this context is not the Merkle-update AIR of this batch size");
        std::vector<uint64_t> packed(csg_tx_batch_pack(b, nullptr));
        csg_tx_batch_pack(b, packed.data());
        Timer &t = ctx->stage_timer;
        t.start(ctx->st);
        upload_records(ctx, packed);
        ctx->d_io.reserve((size_t)ctx->air.width * ctx->n);
        build_merkle_update_trace(ctx->d_wit_in.p, ntx, csg_tx_batch_depth(b), ctx->d_io.p, ctx->st);
        ctx->trace_repr = CSG_REPR_CANONICAL;
        ctx->tm.h2d = t.stop(ctx->st);
        ctx->nfri = 0; ctx->stage = S_TRACE;
    });
}
int csg_build_trace_schnorr_device(csg_ctx *ctx, const csg_sig_batch *b) {
    return guarded(ctx, [&] {
        ctx->need(S_AIR, "csg_set_air must be called first");
        if (!b) throw ArgError("null batch");
        const size_t nsig = csg_sig_batch_size(b);
        if (ctx->air.id != CSG_AIR_SCHNORR || ctx->n != nsig * 512) throw ArgError("the AIR set on this context is not the Schnorr AIR of this batch size");
        std::vector<uint64_t> packed(csg_sig_batch_pack(b, nullptr));
        csg_sig_batch_pack(b, packed.data());
        Timer &t = ctx->stage_timer;
        t.start(ctx->st);
        upload_records(ctx, packed);
        ctx->d_wit_finals.reserve(nsig * 48); ctx->d_io.reserve((size_t)ctx->air.width * ctx->n);
        build_schnorr_trace(ctx->d_wit_in.p, nsig, ctx->d_io.p, ctx->d_wit_finals.p, ctx->st);
        ctx->trace_repr = CSG_REPR_CANONICAL;
        ctx->tm.h2d = t.stop(ctx->st);
        ctx->nfri = 0; ctx->stage = S_TRACE;
    });
}
// K traces of a csg_prove_many_device batch built on the device into the caller's buffer (many/witness_many.cu).  The batch's
// scratch is its own: the single-proof state (d_wit_in, the packed batch, the resident trace) is left alone.
int csg_build_traces_many_rescue(csg_ctx *ctx, const uint64_t *seeds, size_t count, size_t chain_length, uint64_t *traces_dev, uint64_t *pubs) {
    return build_traces_many(ctx, [&] { many_build_rescue(ctx->many, ctx->st, seeds, count, chain_length, traces_dev, pubs); });
}
int csg_build_traces_many_schnorr(csg_ctx *ctx, const csg_sig_batch *b, uint64_t *traces_dev, uint64_t *pubs) {
    return build_traces_many(ctx, [&] { many_build_items(ctx->many, ctx->st, CSG_AIR_SCHNORR, b, traces_dev, pubs); });
}
int csg_build_traces_many_merkle_update(csg_ctx *ctx, const csg_tx_batch *b, uint64_t *traces_dev, uint64_t *pubs) {
    return build_traces_many(ctx, [&] { many_build_items(ctx->many, ctx->st, CSG_AIR_MERKLE_UPDATE, b, traces_dev, pubs); });
}
int csg_build_traces_many_transaction(csg_ctx *ctx, const csg_tx_batch *b, uint64_t *traces_dev, uint64_t *pubs) {
    return build_traces_many(ctx, [&] { many_build_items(ctx->many, ctx->st, CSG_AIR_TRANSACTION, b, traces_dev, pubs); });
}
// TransactionMetadata::build_random on the device: plan on the host (draws + tree shape, no hashing), hashes on the GPU
int csg_tx_batch_build_device(csg_ctx *ctx, uint64_t seed, size_t num_tx, unsigned tree_depth, uint64_t pub[14]) {
    return guarded(ctx, [&] {
        if (!pub) throw ArgError("null output");
        BatchPlan P;
        try { P = plan_tx_batch(seed, num_tx, tree_depth); } catch (const std::invalid_argument &e) { throw ArgError(e.what()); }
        Stream &st = ctx->st;
        Timer &t = ctx->stage_timer;
        t.start(st);
        const size_t total = P.level_off[P.depth + 1];
        ctx->d_b_accounts.reserve(P.accounts.size()); ctx->d_b_txw.reserve(P.tx_words.size()); ctx->d_b_sigs.reserve(14 * num_tx);
        ctx->d_b_left.reserve(total); ctx->d_b_right.reserve(total); ctx->d_b_refs.reserve(P.tx_refs.size());
        ctx->d_b_hashes.reserve(7 * total); ctx->d_b_defaults.reserve(7 * 16); ctx->d_b_gtable.reserve(64 * 16 * 12);
        ctx->d_wit_in.reserve((size_t)WIT_WORDS * num_tx);
        CSG_CUDA(cudaMemcpyAsync(ctx->d_b_accounts.p, P.accounts.data(), P.accounts.size() * 8, cudaMemcpyHostToDevice, st.s));
        CSG_CUDA(cudaMemcpyAsync(ctx->d_b_txw.p, P.tx_words.data(), P.tx_words.size() * 8, cudaMemcpyHostToDevice, st.s));
        CSG_CUDA(cudaMemcpyAsync(ctx->d_b_left.p, P.left.data(), total * 4, cudaMemcpyHostToDevice, st.s));
        CSG_CUDA(cudaMemcpyAsync(ctx->d_b_right.p, P.right.data(), total * 4, cudaMemcpyHostToDevice, st.s));
        CSG_CUDA(cudaMemcpyAsync(ctx->d_b_refs.p, P.tx_refs.data(), P.tx_refs.size() * 4, cudaMemcpyHostToDevice, st.s));
        if (ctx->b_defaults_depth != P.depth) { batch_defaults(P.depth, ctx->d_b_defaults.p, st); ctx->b_defaults_depth = P.depth; }
        if (!ctx->b_gtable_built) { batch_gtable(ctx->d_b_gtable.p, st); ctx->b_gtable_built = true; }
        BatchDevice B{P.depth, (unsigned)num_tx, P.level_off.data(), ctx->d_b_accounts.p, ctx->d_b_left.p, ctx->d_b_right.p, ctx->d_b_txw.p, ctx->d_b_refs.p,
                      ctx->d_b_hashes.p, ctx->d_b_defaults.p, ctx->d_b_gtable.p, ctx->d_b_sigs.p, ctx->d_wit_in.p};
        batch_build(B, st);
        // public inputs: the root before the first transfer and the root after the last one (TransactionProver::get_pub_inputs)
        fe roots[14];
        auto fetch = [&](int ref, fe *out) {
            const fe *src = ref >= 0 ? ctx->d_b_hashes.p + (size_t)ref * 7 : ctx->d_b_defaults.p + (size_t)(-ref - 1) * 7;
            CSG_CUDA(cudaMemcpyAsync(out, src, 7 * sizeof(fe), cudaMemcpyDeviceToHost, st.s));
        };
        fetch(P.tx_refs[32], roots); fetch(P.final_root, roots + 7);
        ctx->tm.batch_build = t.stop(st);   // synchronises: the plan's host vectors and `roots` are complete
        for (int i = 0; i < 14; i++) pub[i] = from_mont(roots[i]);
        ctx->wit_resident_ntx = num_tx; ctx->wit_resident_depth = P.depth;
        ctx->wit_packed_for = nullptr;       // d_wit_in no longer holds a host batch's records
    });
}
int csg_build_trace_transaction_resident(csg_ctx *ctx) {
    return guarded(ctx, [&] {
        ctx->need(S_AIR, "csg_set_air must be called first");
        const size_t ntx = ctx->wit_resident_ntx;
        if (!ntx) throw StateError("csg_tx_batch_build_device must be called first");
        if (ctx->air.id != CSG_AIR_TRANSACTION || ctx->n != ntx * 1024) throw ArgError("the AIR set on this context is not the transaction AIR of this batch size");
        if (ctx->wit_resident_depth != 15) throw ArgError("the transaction AIR is built for tree depth 15");
        Timer &t = ctx->stage_timer;
        t.start(ctx->st);
        ctx->d_wit_finals.reserve(ntx * 48); ctx->d_io.reserve((size_t)ctx->air.width * ctx->n);
        build_transaction_trace(ctx->d_wit_in.p, ntx, 15, ctx->d_io.p, ctx->d_wit_finals.p, ctx->st);
        ctx->trace_repr = CSG_REPR_CANONICAL;
        ctx->tm.h2d = t.stop(ctx->st);   // here: witness generation time
        ctx->nfri = 0;
        ctx->stage = S_TRACE;
    });
}
int csg_download_batch_records(csg_ctx *ctx, uint64_t *out, size_t cap_words) {
    return guarded(ctx, [&] {
        const size_t words = (size_t)WIT_WORDS * ctx->wit_resident_ntx;
        if (!words) throw StateError("no device-built batch is resident");
        if (!out || cap_words < words) throw ArgError("record buffer too small");
        CSG_CUDA(cudaMemcpyAsync(out, ctx->d_wit_in.p, words * 8, cudaMemcpyDeviceToHost, ctx->st.s));
        CSG_CUDA(cudaStreamSynchronize(ctx->st.s));
    });
}
int csg_download_trace(csg_ctx *ctx, uint64_t *trace) {
    return guarded(ctx, [&] {
        ctx->need(S_TRACE, "no trace is resident");
        CSG_CUDA(cudaMemcpyAsync(trace, ctx->d_io.p, (size_t)ctx->air.width * ctx->n * 8, cudaMemcpyDeviceToHost, ctx->st.s));
        CSG_CUDA(cudaStreamSynchronize(ctx->st.s));
    });
}
int csg_timer_start(csg_ctx *ctx) {
    return guarded(ctx, [&] {
        if (!ctx->ev_a) { CSG_CUDA(cudaEventCreate(&ctx->ev_a)); CSG_CUDA(cudaEventCreate(&ctx->ev_b)); }
        CSG_CUDA(cudaEventRecord(ctx->ev_a, ctx->st.s));
    });
}
int csg_timer_stop(csg_ctx *ctx, float *ms) {
    return guarded(ctx, [&] {
        if (!ctx->ev_a || !ms) throw StateError("csg_timer_start must be called first");
        CSG_CUDA(cudaEventRecord(ctx->ev_b, ctx->st.s));
        CSG_CUDA(cudaEventSynchronize(ctx->ev_b));
        CSG_CUDA(cudaEventElapsedTime(ms, ctx->ev_a, ctx->ev_b));
    });
}
// ---- coset-sharded proofs: attach the context to a group of `world` contexts (one per GPU) before csg_set_air
int csg_dist_unique_id(uint8_t id[128]) {
    if (!id) return CSG_ERR_ARG;
    try { nccl_unique_id(id); return CSG_OK; } catch (const std::exception &) { return CSG_ERR_UNSUPPORTED; }
}
static void check_world(int rank, int world) {
    if (world < 1 || world > 32 || (world & (world - 1)) || rank < 0 || rank >= world) throw ArgError("world must be a power of two up to 32, rank below it");
}
int csg_dist_init(csg_ctx *ctx, int rank, int world, const uint8_t id[128]) {
    return guarded(ctx, [&] {
        check_world(rank, world);
        if (!id) throw ArgError("null NCCL id");
        CSG_CUDA(cudaStreamSynchronize(ctx->st.s));
        ctx->comm.reset();
        if (world > 1) ctx->comm = make_nccl_comm(rank, world, id);
        ctx->stage = S_NONE;   // the coset ownership is fixed by csg_set_air
    });
}
int csg_dist_init_local(csg_ctx **ctxs, int world) {
    if (!ctxs) return CSG_ERR_ARG;
    for (int r = 0; r < world; r++) if (!ctxs[r]) return CSG_ERR_ARG;
    return guarded(ctxs[0], [&] {
        check_world(0, world);
        auto comms = make_local_comms(world);
        for (int r = 0; r < world; r++) {
            CSG_CUDA(cudaSetDevice(ctxs[r]->device));
            CSG_CUDA(cudaStreamSynchronize(ctxs[r]->st.s));
            ctxs[r]->comm.reset();
            if (world > 1) ctxs[r]->comm = std::move(comms[r]);
            ctxs[r]->stage = S_NONE;
        }
    });
}
int csg_dist_plan(int rank, int world, uint32_t blowup, uint32_t ce_blowup, uint32_t width, csg_shard_plan *out) {
    if (!out || rank < 0 || world < 1 || (world & (world - 1))) return CSG_ERR_ARG;
    return shard_plan((size_t)rank, (size_t)world, blowup, ce_blowup, width, out) ? CSG_OK : CSG_ERR_ARG;
}
int csg_dist_trace_chunks(int rank, int world, uint32_t blowup, uint32_t ce_blowup, uint32_t width, int from_host, uint32_t *sizes, size_t cap, size_t *count) {
    csg_shard_plan plan;
    if (!count || (cap && !sizes) || csg_dist_plan(rank, world, blowup, ce_blowup, width, &plan) != CSG_OK) return CSG_ERR_ARG;
    const std::vector<size_t> chunks = trace_chunks(from_host != 0, plan.first_column, (size_t)plan.first_column + plan.num_columns);
    *count = chunks.size();
    if (chunks.size() > cap) return CSG_ERR_ARG;
    for (size_t k = 0; k < chunks.size(); k++) sizes[k] = (uint32_t)chunks[k];
    return CSG_OK;
}
int csg_dist_info(const csg_ctx *ctx, int *rank, int *world) {
    if (!ctx || !rank || !world) return CSG_ERR_ARG;
    *rank = ctx->comm ? ctx->comm->rank : 0; *world = ctx->comm ? ctx->comm->world : 1;
    return CSG_OK;
}
int csg_get_timings(const csg_ctx *ctx, csg_timings *out) {
    if (!ctx || !out) return CSG_ERR_ARG;
    // stage times are event pairs read on demand (no host synchronisation per stage): collect the outstanding ones first
    return guarded(const_cast<csg_ctx *>(ctx), [&] { const_cast<csg_ctx *>(ctx)->flush_timers(); *out = ctx->tm; });
}


}  // extern "C"
