// libcsg: kernel-level entry points (parity tests, kernel sweep) and debugging aids of include/csg.h.
#include "prover_ctx.cuh"

extern "C" {

long long csg_debug_redc_violations(csg_ctx *) { return (long long)redc_violations(); }
long long csg_debug_redc_selftest(csg_ctx *ctx) {
    long long bad = -1;
    guarded(ctx, [&] { bad = redc_selftest(ctx->st); });
    return bad;
}
long long csg_debug_field_selftest(csg_ctx *ctx) {
    long long bad = -1;
    guarded(ctx, [&] { bad = field_selftest(ctx->st); });
    return bad;
}
// words >= p in stage buffer `which` (0 = trace coefficients, 1 = trace LDE, 2 = periodic tables, 3 = merged constraint column,
// 4 = composition columns, 5 = composition LDE), all `ext` planes of 3-5; -1 for another `which` or an error.  The copy runs on
// the proving stream, after the work queued there that writes the buffer.
long long csg_debug_count_unreduced(csg_ctx *ctx, int which) {
    if (which < 0 || which > 5) return -1;
    long long bad = -1;
    guarded(ctx, [&] {
        const DBuf<fe> *b = which == 0 ? &ctx->d_polys : which == 1 ? &ctx->d_lde : which == 2 ? &ctx->d_ptab : which == 3 ? &ctx->d_comb : which == 4 ? &ctx->d_cpolys : &ctx->d_clde;
        const size_t d = (size_t)ctx->d, cel = ctx->cel;
        size_t count = which == 0 ? ctx->air.width * ctx->n : which == 1 ? ctx->air.width * ctx->n * ctx->bl
                       : which == 2 ? (ctx->h_cargs ? ctx->h_cargs->ptab_coset_stride * cel : 0)
                       : which == 3 ? d * cel * ctx->n : which == 4 ? d * ctx->ce * ctx->n : d * ctx->ce * ctx->n * ctx->bl;
        count = std::min(count, b->n);   // a stage that has not run yet has not sized its buffer
        std::vector<fe> h(count);
        if (count) CSG_CUDA(cudaMemcpyAsync(h.data(), b->p, count * sizeof(fe), cudaMemcpyDeviceToHost, ctx->st.s));
        CSG_CUDA(cudaStreamSynchronize(ctx->st.s));
        bad = 0;
        for (fe v : h) bad += v >= P;
    });
    return bad;
}
// ---------------------------------------------------------------------------------------------- kernel-level entry points
int csg_k_lde(csg_ctx *ctx, const uint64_t *cols, size_t width, size_t n, size_t blowup, uint64_t *lde) {
    return guarded(ctx, [&] {
        if (!cols || !lde || n < 2 || (n & (n - 1)) || blowup < 1 || (blowup & (blowup - 1)) || blowup > 32) throw ArgError("bad LDE shape");
        Stream &st = ctx->st;
        RootTable rt; NttScratch sc;
        const unsigned logn = ilog2(n);
        rt.build(logn, st);
        DBuf<uint64_t> io; DBuf<fe> a, c, e;
        io.reserve(width * n * blowup); a.reserve(width * n); c.reserve(width * n); e.reserve(width * n * blowup);
        CSG_CUDA(cudaMemcpyAsync(io.p, cols, width * n * 8, cudaMemcpyHostToDevice, st.s));
        to_montgomery(io.p, a.p, width * n, st);
        intt_columns(rt, sc, a.p, n, c.p, n, width, logn, st);
        std::vector<fe> shifts(blowup);
        fe acc = to_mont(GENERATOR), w = root_of_unity(ilog2(n * blowup));
        for (size_t k = 0; k < blowup; k++) { shifts[k] = acc; acc = mul(acc, w); }
        coset_ntt_columns(rt, sc, c.p, n, e.p, n, width * n, width, logn, shifts.data(), blowup, st);
        coset_major_to_natural(e.p, (unsigned)width, (unsigned)blowup, n, io.p, st);
        CSG_CUDA(cudaMemcpyAsync(lde, io.p, width * n * blowup * 8, cudaMemcpyDeviceToHost, st.s));
        CSG_CUDA(cudaStreamSynchronize(st.s));
    });
}
int csg_k_hash_rows(csg_ctx *ctx, int hash_fn, const uint64_t *cols, size_t width, size_t rows, uint8_t *digests) {
    return guarded(ctx, [&] {
        if (!cols || !digests || !rows || !width || width > 128) throw ArgError("bad matrix shape");
        Stream &st = ctx->st;
        DBuf<uint64_t> io; DBuf<fe> a; DBuf<uint32_t> d;
        io.reserve(width * rows); a.reserve(width * rows); d.reserve(8 * rows);
        CSG_CUDA(cudaMemcpyAsync(io.p, cols, width * rows * 8, cudaMemcpyHostToDevice, st.s));
        to_montgomery(io.p, a.p, width * rows, st);
        hash_rows(a.p, (unsigned)width, rows, 1, 0, rows, hash_fn, d.p, st);
        CSG_CUDA(cudaMemcpyAsync(digests, d.p, 32 * rows, cudaMemcpyDeviceToHost, st.s));
        CSG_CUDA(cudaStreamSynchronize(st.s));
    });
}
int csg_k_merkle(csg_ctx *ctx, int hash_fn, const uint8_t *leaves, size_t nleaves, uint8_t *nodes) {
    return guarded(ctx, [&] {
        if (!leaves || !nodes || nleaves < 2 || (nleaves & (nleaves - 1))) throw ArgError("leaf count must be a power of two, at least 2");
        Stream &st = ctx->st;
        DBuf<uint32_t> d;
        d.reserve(16 * nleaves);
        CSG_CUDA(cudaMemcpyAsync(d.p + 8 * nleaves, leaves, 32 * nleaves, cudaMemcpyHostToDevice, st.s));
        merkle_build(d.p, nleaves, hash_fn, st);
        CSG_CUDA(cudaMemcpyAsync(nodes, d.p, 64 * nleaves, cudaMemcpyDeviceToHost, st.s));
        CSG_CUDA(cudaStreamSynchronize(st.s));
    });
}
int csg_k_fri_fold4(csg_ctx *ctx, const uint64_t *evals, size_t n, uint64_t alpha, uint64_t *out) {
    return guarded(ctx, [&] {
        if (!evals || !out || n < 8 || (n & (n - 1))) throw ArgError("bad FRI layer size");
        Stream &st = ctx->st;
        RootTable rt;
        const unsigned logn = ilog2(n);
        rt.build(logn, st);
        DBuf<uint64_t> io; DBuf<fe> a, r;
        io.reserve(n); a.reserve(n); r.reserve(n / 4);
        CSG_CUDA(cudaMemcpyAsync(io.p, evals, n * 8, cudaMemcpyHostToDevice, st.s));
        to_montgomery(io.p, a.p, n, st);
        FoldArgs fa{};
        fa.alpha = to_mont(alpha % P); fa.offset_inv = inv(to_mont(GENERATOR));
        fa.zeta_inv = f63::pow(inv(root_of_unity(logn)), n / 4); fa.quarter = inv(to_mont(4));
        fa.logm = logn; fa.logW = logn;
        csg::fri_fold4(a.p, n, rt.W.p, fa, r.p, st);
        from_montgomery(r.p, io.p, n / 4, st);
        CSG_CUDA(cudaMemcpyAsync(out, io.p, (n / 4) * 8, cudaMemcpyDeviceToHost, st.s));
        CSG_CUDA(cudaStreamSynchronize(st.s));
    });
}
// kernel sweep on synthetic device-resident columns: ms_out = {LDE, row hashing, Merkle tree, one FRI fold of an
// LDE-sized layer}, each the mean over `iters` runs after one warm-up
int csg_k_sweep(csg_ctx *ctx, size_t width, size_t n, size_t blowup, int hash_fn, int iters, float ms_out[4]) {
    return guarded(ctx, [&] {
        if (n < 8 || (n & (n - 1)) || blowup < 2 || (blowup & (blowup - 1)) || blowup > 32 || !width || width > 128 || iters < 1) throw ArgError("bad sweep shape");
        Stream &st = ctx->st;
        RootTable rt; NttScratch sc;
        const unsigned logn = ilog2(n);
        const size_t lde_n = n * blowup;
        rt.build(logn, st);
        DBuf<uint64_t> io; DBuf<fe> a, c, e, f; DBuf<uint32_t> nodes;
        io.reserve(width * n); a.reserve(width * n); c.reserve(width * n); e.reserve(width * lde_n); f.reserve(lde_n / 4); nodes.reserve(16 * lde_n);
        std::vector<uint64_t> host(width * n);
        uint64_t s = 0x9e3779b97f4a7c15ULL;
        for (auto &v : host) { s ^= s << 13; s ^= s >> 7; s ^= s << 17; v = s % P; }
        CSG_CUDA(cudaMemcpyAsync(io.p, host.data(), host.size() * 8, cudaMemcpyHostToDevice, st.s));
        to_montgomery(io.p, a.p, width * n, st);
        std::vector<fe> shifts(blowup);
        fe acc = to_mont(GENERATOR), w = root_of_unity(ilog2(lde_n));
        for (size_t k = 0; k < blowup; k++) { shifts[k] = acc; acc = mul(acc, w); }
        FoldArgs fa{};
        const unsigned logm = ilog2(lde_n);
        const fe w_inv = inv(w);
        fa.alpha = to_mont(12345); fa.offset_inv = inv(to_mont(GENERATOR)); fa.zeta_inv = f63::pow(w_inv, lde_n / 4); fa.quarter = inv(to_mont(4));
        fa.logm = logm; fa.logW = logn;
        for (unsigned i = 0; i < (1u << (logm - logn)); i++) fa.small[i] = f63::pow(w_inv, i);
        Timer t;
        float acc_ms[4] = {0, 0, 0, 0};
        for (int it = -1; it < iters; it++) {
            float ms[4];
            t.start(st);
            intt_columns(rt, sc, a.p, n, c.p, n, width, logn, st);
            coset_ntt_columns(rt, sc, c.p, n, e.p, n, width * n, width, logn, shifts.data(), blowup, st);
            ms[0] = t.stop(st);
            t.start(st);
            hash_rows(e.p, (unsigned)width, n, (unsigned)blowup, width * n, n, hash_fn, nodes.p + 8 * lde_n, st);
            ms[1] = t.stop(st);
            t.start(st);
            merkle_build(nodes.p, lde_n, hash_fn, st);
            ms[2] = t.stop(st);
            t.start(st);
            csg::fri_fold4(e.p, lde_n, rt.W.p, fa, f.p, st);
            ms[3] = t.stop(st);
            if (it >= 0) for (int k = 0; k < 4; k++) acc_ms[k] += ms[k];
        }
        for (int k = 0; k < 4; k++) ms_out[k] = acc_ms[k] / iters;
    });
}


}  // extern "C"
