// The device pass of csg_validate_*: the direct constraint code of airs.cuh on the trace domain, one thread per step s < n-1 and
// blockIdx.y = trace.  The shells follow many/cons_many.cu: Rescue residuals, curve banks and the final point addition write
// partial sums, and the last kernel adds them to the linear rest per step before testing for zero -- a slot can receive values
// from several items, so no partial can be tested on its own.  Two independent random combinations (CombT<false, 2>, the
// accumulators of the degree-2 extension kernels) keep the direct Rescue form: no per-call Rescue tables.
#include <algorithm>

#include "../airs.cuh"
#include "validate.cuh"

namespace csg {
using namespace f63;

namespace {

constexpr unsigned ROW_THREADS = 128, CONV_THREADS = 256, CELL_THREADS = 128;
// blocks per SM the register allocation must allow: the curve items need about 200 registers for their Fp6 formulas with two
// accumulators: at 3 blocks (168 registers) the scalar-multiplication bank spills about 1 KB per thread, at 2 blocks (255) about
// 350 bytes, and the final addition fits (ptxas -v)
constexpr int RESCUE_MINBLOCKS = 4, ECC_MINBLOCKS = 2, REST_MINBLOCKS = 4;

__global__ void __launch_bounds__(CONV_THREADS) to_mont_kernel(const uint64_t *src, fe *mont, unsigned long long count, int montgomery) {
    for (unsigned long long i = blockIdx.x * (unsigned long long)CONV_THREADS + threadIdx.x; i < count; i += (unsigned long long)gridDim.x * CONV_THREADS) {
        uint64_t x = src[i];
        if (x >= 2 * P) x -= 2 * P;   // 2^64 < 4p: two steps reduce any word
        if (x >= P) x -= P;
        mont[i] = montgomery ? x : to_mont(x);
    }
}

struct Row {
    airs::Frame f;
    airs::Periodic pv;
};
__device__ __forceinline__ Row row_at(const ValArgs *A, const fe *mont, const fe *ptab, unsigned k, unsigned long long s) {
    const unsigned long long n = 1ULL << A->logn;
    const fe *T = mont + (unsigned long long)k * A->width * n;
    return Row{airs::Frame{T + s, T + s + 1, (size_t)n}, airs::Periodic{ptab + k * A->ptab_stride, A->poff, A->pmask, (uint32_t)s}};
}
__device__ __forceinline__ airs::CombT<false, 2> comb(const ValArgs *A) {
    return airs::CombT<false, 2>{A->alpha[0], A->beta, A->group, &A->zero, 0, acc192(), nullptr, 0, A->alpha[1], A->beta, 0};
}

// KIND 0: Rescue residual number blockIdx.z; KIND 1: scalar-multiplication bank blockIdx.z; KIND 2: final point addition.
// part[((k * items + item) * 2 + j) * n + s]: component j of the item's partial sum at step s
template <int AIR, int KIND>
__global__ void __launch_bounds__(ROW_THREADS, KIND == 0 ? RESCUE_MINBLOCKS : ECC_MINBLOCKS)
validate_item_kernel(const ValArgs *__restrict__ A, const fe *__restrict__ mont, const fe *__restrict__ ptab, fe *__restrict__ part, unsigned items) {
    const unsigned k = blockIdx.y, item = KIND == 2 ? items - 1 : (KIND == 1 ? airs::Items<AIR>::rescue : 0) + blockIdx.z;
    const unsigned long long n = 1ULL << A->logn, s = blockIdx.x * (unsigned long long)ROW_THREADS + threadIdx.x;
    if (s + 1 >= n) return;
    const Row r = row_at(A, mont, ptab, k, s);
    airs::CombT<false, 2> C = comb(A);
    if (KIND == 0) airs::eval_rescue_item<AIR>((int)blockIdx.z, r.f, r.pv, C);
    else if (KIND == 1) airs::eval_ecc_bank<AIR>((int)blockIdx.z, r.f, r.pv, C);
    else airs::eval_ecc_final<AIR>(r.f, r.pv, C);
    fe *q = part + (((unsigned long long)k * items + item) * 2) * n + s;
    q[0] = C.sum.reduce();
    q[n] = C.sum_x[0].reduce();
}

// the linear rest, the sum over the items, the test; one count per warp
template <int AIR>
__global__ void __launch_bounds__(ROW_THREADS, REST_MINBLOCKS)
validate_rest_kernel(const ValArgs *__restrict__ A, const fe *__restrict__ mont, const fe *__restrict__ ptab, const fe *__restrict__ part, unsigned items,
                     uint8_t *__restrict__ flags, unsigned long long *__restrict__ counts) {
    const unsigned k = blockIdx.y;
    const unsigned long long n = 1ULL << A->logn, s = blockIdx.x * (unsigned long long)ROW_THREADS + threadIdx.x;
    bool bad = false;
    if (s + 1 < n) {
        const Row r = row_at(A, mont, ptab, k, s);
        airs::CombT<false, 2> C = comb(A);
        airs::eval_rest<AIR>(r.f, r.pv, C);
        fe t0 = C.sum.reduce(), t1 = C.sum_x[0].reduce();
        const fe *q = part + ((unsigned long long)k * items * 2) * n + s;
        for (unsigned p = 0; p < items; p++) { t0 = add(t0, q[2 * p * n]); t1 = add(t1, q[(2 * p + 1) * n]); }
        bad = t0 != 0 || t1 != 0;
    }
    if (s < n) flags[(unsigned long long)k * n + s] = bad;
    const unsigned m = __ballot_sync(0xffffffffu, bad);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(&counts[k], (unsigned long long)__popc(m));
}

__global__ void __launch_bounds__(CELL_THREADS) validate_cells_kernel(const fe *__restrict__ mont, unsigned w, unsigned long long n, const uint32_t *__restrict__ col,
                                                                      const uint32_t *__restrict__ step, const fe *__restrict__ val, unsigned ncells,
                                                                      uint8_t *__restrict__ cflags, unsigned long long *__restrict__ counts) {
    const unsigned k = blockIdx.y, c = blockIdx.x * CELL_THREADS + threadIdx.x;
    bool bad = false;
    if (c < ncells) {
        bad = mont[((unsigned long long)k * w + col[c]) * n + step[c]] != val[(unsigned long long)k * ncells + c];
        cflags[(unsigned long long)k * ncells + c] = bad;
    }
    const unsigned m = __ballot_sync(0xffffffffu, bad);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(&counts[k], (unsigned long long)__popc(m));
}

template <int AIR>
void launch_rows(const ValArgs *args_dev, const ValArgs &h, size_t K, const fe *mont, const fe *ptab, fe *part, uint8_t *flags, unsigned long long *counts, Stream &st) {
    const unsigned long long n = 1ULL << h.logn;
    const unsigned gx = (unsigned)((n + ROW_THREADS - 1) / ROW_THREADS), gy = (unsigned)K;
    constexpr int NR = airs::Items<AIR>::rescue, NE = airs::Items<AIR>::ecc, items = NR + NE;
    if constexpr (NR > 0) CSG_LAUNCH(st, (validate_item_kernel<AIR, 0>), dim3(gx, gy, NR), ROW_THREADS, 0, args_dev, mont, ptab, part, (unsigned)items);
    if constexpr (NE > 0) {
        CSG_LAUNCH(st, (validate_item_kernel<AIR, 1>), dim3(gx, gy, 2), ROW_THREADS, 0, args_dev, mont, ptab, part, (unsigned)items);
        CSG_LAUNCH(st, (validate_item_kernel<AIR, 2>), dim3(gx, gy, 1), ROW_THREADS, 0, args_dev, mont, ptab, part, (unsigned)items);
    }
    CSG_LAUNCH(st, validate_rest_kernel<AIR>, dim3(gx, gy), ROW_THREADS, 0, args_dev, mont, ptab, (const fe *)part, (unsigned)items, flags, counts);
}

}  // namespace

void validate_to_mont(const uint64_t *src, fe *mont, size_t count, int repr, Stream &st) {
    const unsigned blocks = (unsigned)std::min<size_t>((count + CONV_THREADS - 1) / CONV_THREADS, 148 * 16);
    CSG_LAUNCH(st, to_mont_kernel, blocks, CONV_THREADS, 0, src, mont, (unsigned long long)count, repr == CSG_REPR_MONTGOMERY ? 1 : 0);
}

size_t validate_items(int air_id) {
    switch (air_id) {
    case airs::TRANSACTION: return airs::Items<airs::TRANSACTION>::rescue + airs::Items<airs::TRANSACTION>::ecc;
    case airs::MERKLE_UPDATE: return airs::Items<airs::MERKLE_UPDATE>::rescue;
    case airs::MERKLE_INIT: return airs::Items<airs::MERKLE_INIT>::rescue;
    case airs::SCHNORR: return airs::Items<airs::SCHNORR>::rescue + airs::Items<airs::SCHNORR>::ecc;
    case airs::RESCUE: return airs::Items<airs::RESCUE>::rescue;
    default: return 0;
    }
}

void validate_rows(int air_id, const ValArgs *args_dev, const ValArgs &h, size_t K, const fe *mont, const fe *ptab, fe *part, uint8_t *flags,
                   unsigned long long *counts, Stream &st) {
    switch (air_id) {
    case airs::TRANSACTION: launch_rows<airs::TRANSACTION>(args_dev, h, K, mont, ptab, part, flags, counts, st); break;
    case airs::MERKLE_UPDATE: launch_rows<airs::MERKLE_UPDATE>(args_dev, h, K, mont, ptab, part, flags, counts, st); break;
    case airs::MERKLE_INIT: launch_rows<airs::MERKLE_INIT>(args_dev, h, K, mont, ptab, part, flags, counts, st); break;
    case airs::SCHNORR: launch_rows<airs::SCHNORR>(args_dev, h, K, mont, ptab, part, flags, counts, st); break;
    case airs::RANGE: launch_rows<airs::RANGE>(args_dev, h, K, mont, ptab, part, flags, counts, st); break;
    case airs::RESCUE: launch_rows<airs::RESCUE>(args_dev, h, K, mont, ptab, part, flags, counts, st); break;
    default: throw std::runtime_error("unknown AIR id");
    }
}

void validate_cells(size_t K, const fe *mont, unsigned w, size_t n, const uint32_t *col, const uint32_t *step, const fe *val, size_t ncells,
                    uint8_t *cflags, unsigned long long *counts, Stream &st) {
    if (!ncells) return;
    CSG_LAUNCH(st, validate_cells_kernel, dim3((unsigned)((ncells + CELL_THREADS - 1) / CELL_THREADS), (unsigned)K), CELL_THREADS, 0, mont, w,
               (unsigned long long)n, col, step, val, (unsigned)ncells, cflags, counts);
}

}  // namespace csg
