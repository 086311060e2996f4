// See many_kernels.cuh.  Each kernel is the single-proof kernel of commit.cu / stages.cu with the proof index added to the grid.
#include "../hash.cuh"
#include "many_kernels.cuh"

namespace csg {
using namespace f63;

namespace {

template <int HASH>
__global__ void __launch_bounds__(128) hash_rows_many_kernel(const fe *__restrict__ data, unsigned width, unsigned long long n, unsigned ncosets,
                                                             unsigned long long coset_stride, unsigned long long col_stride,
                                                             unsigned long long proof_stride, uint32_t *__restrict__ leaves, unsigned long long tree_words) {
    const unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned kc = blockIdx.y, k = blockIdx.z;
    const fe *p = data + k * proof_stride + kc * coset_stride + i;
    uint32_t d[8];
    auto get = [&](uint32_t c) -> uint64_t { return from_mont(__ldg(p + c * col_stride)); };
    if (HASH == hashes::SHA3_256) hashes::k3::hash_words64(get, width, d); else hashes::b3::hash_words64(get, width, d);
    uint4 *o = reinterpret_cast<uint4 *>(leaves + k * tree_words + 8ULL * (kc + (unsigned long long)ncosets * i));
    o[0] = make_uint4(d[0], d[1], d[2], d[3]);
    o[1] = make_uint4(d[4], d[5], d[6], d[7]);
}

__device__ __forceinline__ void load_digest(const uint32_t *p, uint32_t (&d)[8]) {
    uint4 a = reinterpret_cast<const uint4 *>(p)[0], b = reinterpret_cast<const uint4 *>(p)[1];
    d[0] = a.x; d[1] = a.y; d[2] = a.z; d[3] = a.w; d[4] = b.x; d[5] = b.y; d[6] = b.z; d[7] = b.w;
}
__device__ __forceinline__ void store_digest(uint32_t *p, const uint32_t (&d)[8]) {
    reinterpret_cast<uint4 *>(p)[0] = make_uint4(d[0], d[1], d[2], d[3]);
    reinterpret_cast<uint4 *>(p)[1] = make_uint4(d[4], d[5], d[6], d[7]);
}

// one level of every tree: nodes[i] = H(nodes[2i] || nodes[2i+1]) for i in [m, 2m); tree blockIdx.y
template <int HASH>
__global__ void __launch_bounds__(256) merkle_level_many_kernel(uint32_t *nodes, unsigned long long m, unsigned long long tree_words) {
    const unsigned long long t = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
    if (t >= m) return;
    uint32_t *tree = nodes + blockIdx.y * tree_words;
    const unsigned long long i = m + t;
    uint32_t l[8], r[8], o[8];
    load_digest(tree + 16 * i, l);
    load_digest(tree + 16 * i + 8, r);
    hashes::merge(HASH, l, r, o);
    store_digest(tree + 8 * i, o);
}
// the top of each tree (levels of at most 512 nodes), one CTA per tree
template <int HASH>
__global__ void __launch_bounds__(512) merkle_top_many_kernel(uint32_t *nodes, unsigned m_first, unsigned long long tree_words) {
    uint32_t *tree = nodes + blockIdx.x * tree_words;
    for (unsigned m = m_first; m >= 1; m >>= 1) {
        if (threadIdx.x < m) {
            const unsigned i = m + threadIdx.x;
            uint32_t l[8], r[8], o[8];
            load_digest(tree + 16 * i, l);
            load_digest(tree + 16 * i + 8, r);
            hashes::merge(HASH, l, r, o);
            store_digest(tree + 8 * i, o);
        }
        __syncthreads();
    }
}

struct CrossMat { fe m[16 * 16]; };
__global__ void composition_columns_many_kernel(const fe *__restrict__ e, fe *__restrict__ cols, unsigned long long n, unsigned ce, CrossMat M) {
    const unsigned long long m = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
    if (m >= n) return;
    const unsigned long long off = blockIdx.y * (unsigned long long)ce * n;
    fe v[16];
    for (unsigned k = 0; k < ce; k++) v[k] = e[off + k * n + m];
    const unsigned long long r = m % ce, q0 = m / ce, qs = n / ce;
    for (unsigned t = 0; t < ce; t++) {
        acc192 s;
        for (unsigned k = 0; k < ce; k++) s.mac(M.m[t * ce + k], v[k]);
        cols[off + r * n + q0 + qs * t] = s.reduce();
    }
}

constexpr unsigned EVAL_THREADS = 256, EVAL_CHUNK = 32;
// eval_polys_kernel of stages.cu with the points of the column's proof read from device memory
template <int NPTS>
__global__ void __launch_bounds__(EVAL_THREADS) eval_polys_many_kernel(const fe *__restrict__ polys, unsigned long long n, unsigned ncols,
                                                                      const fe *__restrict__ pts, fe *__restrict__ partial) {
    __shared__ fe red[EVAL_THREADS];
    __shared__ fe zpow[NPTS][EVAL_CHUNK];
    const unsigned t = threadIdx.x, c = blockIdx.y;
    const fe *pp = pts + (unsigned long long)(c / ncols) * NPTS * 2;
    const unsigned long long base = blockIdx.x * (unsigned long long)(EVAL_THREADS * EVAL_CHUNK);
    const fe *poly = polys + c * n;
    if (t < NPTS * EVAL_CHUNK) zpow[t / EVAL_CHUNK][t % EVAL_CHUNK] = f63::pow(pp[2 * (t / EVAL_CHUNK) + 1], t % EVAL_CHUNK);
    __syncthreads();
    acc192 v[NPTS];
#pragma unroll 8
    for (int j = 0; j < (int)EVAL_CHUNK; j++) {
        const unsigned long long m = base + t + (unsigned long long)j * EVAL_THREADS;
        const fe cm = m < n ? poly[m] : 0;
#pragma unroll
        for (int p = 0; p < NPTS; p++) v[p].mac(cm, zpow[p][j]);
    }
#pragma unroll
    for (int p = 0; p < NPTS; p++) {
        red[t] = mul(v[p].reduce(), f63::pow(pp[2 * p], base + t));
        __syncthreads();
        for (unsigned s = EVAL_THREADS / 2; s > 0; s >>= 1) {
            if (t < s) red[t] = add(red[t], red[t + s]);
            __syncthreads();
        }
        if (t == 0) partial[((unsigned long long)c * NPTS + p) * gridDim.x + blockIdx.x] = red[0];
        __syncthreads();
    }
}

template <int NCOMB>
__global__ void combine_polys_many_kernel(const fe *__restrict__ polys, unsigned long long n, unsigned ncols, const fe *__restrict__ coef,
                                          fe *__restrict__ out, unsigned long long out_proof_stride) {
    const unsigned long long m = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
    if (m >= n) return;
    const unsigned k = blockIdx.y;
    const fe *src = polys + (unsigned long long)k * ncols * n + m, *cf = coef + (unsigned long long)k * NCOMB * ncols;
    acc192 s[NCOMB];
    for (unsigned c = 0; c < ncols; c++) {
        const fe v = src[c * n];
#pragma unroll
        for (int t = 0; t < NCOMB; t++) s[t].mac(cf[t * ncols + c], v);
    }
#pragma unroll
    for (int t = 0; t < NCOMB; t++) out[k * out_proof_stride + t * n + m] = s[t].reduce();
}

// deep_quotients_kernel of stages.cu for proof blockIdx.y, its DeepArgs in device memory
constexpr int DEEP_CHUNK = 8, DEEP_THREADS = 128;
__global__ void __launch_bounds__(DEEP_THREADS) deep_quotients_many_kernel(const fe *__restrict__ abc, const fe *__restrict__ W, unsigned long long n,
                                                                          unsigned count, const DeepArgs *__restrict__ args, fe *__restrict__ deep) {
    const unsigned kp = blockIdx.y;
    const DeepArgs *a = args + kp;
    const unsigned ncosets = a->ncosets;
    const fe z = a->z, zg = a->zg, zm = a->zm;
    const unsigned long long total = n * ncosets;
    const unsigned long long base = blockIdx.x * (unsigned long long)(DEEP_CHUNK * DEEP_THREADS) + threadIdx.x;
    fe den[DEEP_CHUNK], pre[DEEP_CHUNK], xs[DEEP_CHUNK];
    fe acc = ONE;
#pragma unroll
    for (int c = 0; c < DEEP_CHUNK; c++) {
        const unsigned long long j = base + (unsigned long long)c * DEEP_THREADS;
        fe d = ONE, x = 0;
        if (j < total) {
            x = mul(a->shift[j % ncosets], W[j / ncosets]);
            d = mul(mul(sub(x, z), sub(x, zg)), sub(x, zm));
        }
        xs[c] = x; den[c] = d; pre[c] = acc;
        acc = mul(acc, d);
    }
    fe ainv = inv(acc);
    const fe az = a->az, bzg = a->bzg, czm = a->czm, lambda = a->lambda, mu = a->mu;
    fe *out = deep + kp * total;
#pragma unroll
    for (int c = DEEP_CHUNK - 1; c >= 0; c--) {
        const unsigned long long j = base + (unsigned long long)c * DEEP_THREADS;
        const fe pinv = mul(ainv, pre[c]);
        ainv = mul(ainv, den[c]);
        if (j >= total) continue;
        const unsigned k = (unsigned)(j % ncosets);
        const unsigned long long i = j / ncosets;
        const fe x = xs[c];
        const fe *src = abc + ((unsigned long long)k * count + kp) * 3 * n + i;
        const fe na = sub(src[0], az), nb = sub(src[n], bzg), nc = sub(src[2 * n], czm);
        const fe d1 = sub(x, z), d2 = sub(x, zg), d3 = sub(x, zm);
        const fe d12 = mul(d1, d2);
        const fe i3 = mul(pinv, d12), i12 = mul(pinv, d3);
        const fe i1 = mul(i12, d2), i2 = mul(i12, d1);
        const fe s = add(add(mul(na, i1), mul(nb, i2)), mul(nc, i3));
        out[j] = mul(s, add(lambda, mul(mu, x)));
    }
}

__global__ void fri_fold4_many_kernel(const fe *__restrict__ evals, unsigned long long q, const fe *__restrict__ W, FoldArgs a,
                                      const fe *__restrict__ alphas, fe *__restrict__ out) {
    const unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
    if (i >= q) return;
    const unsigned k = blockIdx.y;
    const fe *e = evals + k * 4 * q;
    const unsigned long long N = 1ULL << a.logW;
    fe wi;   // w_m^-i
    if (a.logm <= a.logW) wi = W[(N - (i << (a.logW - a.logm))) & (N - 1)];
    else {
        const unsigned extra = a.logm - a.logW;
        wi = mul(a.small[i & ((1u << extra) - 1)], W[(N - (i >> extra)) & (N - 1)]);
    }
    const fe xinv = mul(a.offset_inv, wi);
    const fe v0 = e[i], v1 = e[i + q], v2 = e[i + 2 * q], v3 = e[i + 3 * q];
    const fe s02 = add(v0, v2), d02 = sub(v0, v2), s13 = add(v1, v3), d13 = mul(sub(v1, v3), a.zeta_inv);
    const fe c0 = add(s02, s13), c1 = add(d02, d13), c2 = sub(s02, s13), c3 = sub(d02, d13);
    const fe y = mul(alphas[k], xinv);
    fe r = c3;
    r = add(mul(r, y), c2);
    r = add(mul(r, y), c1);
    r = add(mul(r, y), c0);
    out[k * q + i] = mul(r, a.quarter);
}

// job blockIdx.y; the x-dimension strides over its elements
__global__ void gather_rows_jobs_kernel(const RowJob *__restrict__ jobs, const uint32_t *__restrict__ idx, uint64_t *__restrict__ rows) {
    const RowJob J = jobs[blockIdx.y];
    const unsigned total = J.npos * J.width;
    for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += gridDim.x * blockDim.x) {
        const unsigned r = t / J.width, c = t % J.width;
        const unsigned long long j = idx[J.idx_off + r], k = j % J.ncosets, i = j / J.ncosets;
        rows[J.rows_off + t] = from_mont(J.data[k * J.coset_stride + c * J.col_stride + i]);
    }
}
__global__ void gather_digests_jobs_kernel(const DigestJob *__restrict__ jobs, const uint32_t *__restrict__ idx, uint32_t *__restrict__ out) {
    const DigestJob J = jobs[blockIdx.y];
    for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < J.count * 8; t += gridDim.x * blockDim.x)
        out[J.out_off + t] = J.nodes[8ULL * idx[J.idx_off + (t >> 3)] + (t & 7)];
}

unsigned capped_blocks(size_t work, unsigned threads, unsigned cap) {
    const size_t g = (work + threads - 1) / threads;
    return (unsigned)(g < 1 ? 1 : g > cap ? cap : g);
}

}  // namespace

void hash_rows_many(const fe *data, unsigned width, size_t n, unsigned ncosets, size_t coset_stride, size_t col_stride, size_t proof_stride,
                    size_t count, int hash_fn, uint32_t *leaves, size_t tree_words, Stream &st) {
    if (width > 128) throw std::runtime_error("rows wider than one Blake3 chunk are not supported");
    const dim3 grid((unsigned)((n + 127) / 128), ncosets, (unsigned)count);
#define CSG_HASH_MANY(H) CSG_LAUNCH(st, hash_rows_many_kernel<H>, grid, 128, 0, data, width, (unsigned long long)n, ncosets, (unsigned long long)coset_stride, \
                                    (unsigned long long)col_stride, (unsigned long long)proof_stride, leaves, (unsigned long long)tree_words)
    if (hash_fn == hashes::SHA3_256) CSG_HASH_MANY(hashes::SHA3_256); else CSG_HASH_MANY(hashes::BLAKE3_256);
#undef CSG_HASH_MANY
}

void merkle_build_many(uint32_t *nodes, size_t nleaves, size_t count, size_t tree_words, int hash_fn, Stream &st) {
    if (nleaves < 2) throw std::runtime_error("a Merkle tree needs at least two leaves");
    size_t m = nleaves / 2;
    for (; m > 512; m >>= 1) {
        const dim3 grid((unsigned)((m + 255) / 256), (unsigned)count);
        if (hash_fn == hashes::SHA3_256) CSG_LAUNCH(st, merkle_level_many_kernel<hashes::SHA3_256>, grid, 256, 0, nodes, (unsigned long long)m, (unsigned long long)tree_words);
        else CSG_LAUNCH(st, merkle_level_many_kernel<hashes::BLAKE3_256>, grid, 256, 0, nodes, (unsigned long long)m, (unsigned long long)tree_words);
    }
    if (hash_fn == hashes::SHA3_256) CSG_LAUNCH(st, merkle_top_many_kernel<hashes::SHA3_256>, (unsigned)count, 512, 0, nodes, (unsigned)m, (unsigned long long)tree_words);
    else CSG_LAUNCH(st, merkle_top_many_kernel<hashes::BLAKE3_256>, (unsigned)count, 512, 0, nodes, (unsigned)m, (unsigned long long)tree_words);
}

void composition_columns_many(const fe *e, fe *cols, size_t n, unsigned ce, const fe *mat_host, size_t count, Stream &st) {
    if (ce > 16) throw std::runtime_error("constraint blowup above 16 is not supported");
    CrossMat M;
    for (unsigned i = 0; i < ce * ce; i++) M.m[i] = mat_host[i];
    CSG_LAUNCH(st, composition_columns_many_kernel, dim3((unsigned)((n + 255) / 256), (unsigned)count), 256, 0, e, cols, (unsigned long long)n, ce, M);
}

unsigned eval_polys_many_blocks(size_t n) { return (unsigned)((n + EVAL_THREADS * EVAL_CHUNK - 1) / (EVAL_THREADS * EVAL_CHUNK)); }

unsigned eval_polys_many(const fe *polys, size_t n, size_t ncols, size_t count, const fe *pts_dev, unsigned npts, fe *partial, Stream &st) {
    const unsigned nblk = eval_polys_many_blocks(n);
    const dim3 grid(nblk, (unsigned)(ncols * count));
    if (npts == 1) CSG_LAUNCH(st, eval_polys_many_kernel<1>, grid, EVAL_THREADS, 0, polys, (unsigned long long)n, (unsigned)ncols, pts_dev, partial);
    else if (npts == 2) CSG_LAUNCH(st, eval_polys_many_kernel<2>, grid, EVAL_THREADS, 0, polys, (unsigned long long)n, (unsigned)ncols, pts_dev, partial);
    else throw std::runtime_error("eval_polys_many: 1 or 2 points per proof");
    return nblk;
}

void combine_polys_many(const fe *polys, size_t n, size_t ncols, size_t count, const fe *coef_dev, size_t ncomb, fe *out, size_t out_proof_stride, Stream &st) {
    const dim3 grid((unsigned)((n + 255) / 256), (unsigned)count);
    if (ncomb == 1) CSG_LAUNCH(st, combine_polys_many_kernel<1>, grid, 256, 0, polys, (unsigned long long)n, (unsigned)ncols, coef_dev, out, (unsigned long long)out_proof_stride);
    else if (ncomb == 2) CSG_LAUNCH(st, combine_polys_many_kernel<2>, grid, 256, 0, polys, (unsigned long long)n, (unsigned)ncols, coef_dev, out, (unsigned long long)out_proof_stride);
    else throw std::runtime_error("combine_polys_many: 1 or 2 combinations per call");
}

void deep_quotients_many(const fe *abc, const fe *W, size_t n, size_t count, const DeepArgs *args_dev, unsigned ncosets, fe *deep, Stream &st) {
    const size_t total = n * ncosets, per_block = (size_t)DEEP_CHUNK * DEEP_THREADS;
    CSG_LAUNCH(st, deep_quotients_many_kernel, dim3((unsigned)((total + per_block - 1) / per_block), (unsigned)count), DEEP_THREADS, 0, abc, W,
               (unsigned long long)n, (unsigned)count, args_dev, deep);
}

void fri_fold4_many(const fe *evals, size_t m, const fe *W, const FoldArgs &a, const fe *alphas_dev, size_t count, fe *out, Stream &st) {
    const size_t q = m / 4;
    CSG_LAUNCH(st, fri_fold4_many_kernel, dim3((unsigned)((q + 255) / 256), (unsigned)count), 256, 0, evals, (unsigned long long)q, W, a, alphas_dev, out);
}

void gather_rows_jobs(const RowJob *jobs_dev, size_t njobs, size_t max_elems, const uint32_t *idx_dev, uint64_t *rows, Stream &st) {
    if (!njobs) return;
    CSG_LAUNCH(st, gather_rows_jobs_kernel, dim3(capped_blocks(max_elems, 256, 64), (unsigned)njobs), 256, 0, jobs_dev, idx_dev, rows);
}
void gather_digests_jobs(const DigestJob *jobs_dev, size_t njobs, size_t max_count, const uint32_t *idx_dev, uint32_t *out, Stream &st) {
    if (!njobs) return;
    CSG_LAUNCH(st, gather_digests_jobs_kernel, dim3(capped_blocks(max_count * 8, 256, 64), (unsigned)njobs), 256, 0, jobs_dev, idx_dev, out);
}

}  // namespace csg
