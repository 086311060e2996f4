// The direct (all-coset) constraint evaluation of constraints_kernels.cuh for K proofs at once: thin shells that pick the proof's
// ConsArgs and base pointers from blockIdx.y = proof * ce + coset and then run the same device code (row_setup, airs::eval_*, CombT).
// The low-degree split is never used here: it pays off from 2^14 rows, and the proofs are the same either way.
#include "../airs.cuh"
#include "../constraints_kernels.cuh"
#include "many_kernels.cuh"

namespace csg {
using namespace f63;

namespace {

// KIND 0: Rescue residual number blockIdx.z; KIND 1: scalar-multiplication bank blockIdx.z; KIND 2: final point addition
template <int AIR, int KIND>
__global__ void __launch_bounds__(CONS_THREADS, KIND == 0 ? (AIR != airs::TRANSACTION ? CSG_RESCUE_MINBLOCKS : 4) : CSG_ECC_MINBLOCKS)
cons_item_many_kernel(const ConsArgs *__restrict__ args, unsigned ce, const fe *__restrict__ lde, unsigned long long lde_proof_stride,
                      const fe *__restrict__ W, const fe *__restrict__ ptab, fe *__restrict__ part, unsigned long long part_proof_stride) {
    __shared__ fe xp_s[airs::MAX_GROUPS][CONS_THREADS];
    const unsigned k = blockIdx.y / ce, kc = blockIdx.y % ce, item = KIND == 2 ? 2 : blockIdx.z;
    const ConsArgs *A = args + k;
    const unsigned long long n = 1ULL << A->logn, i = blockIdx.x * (unsigned long long)CONS_THREADS + threadIdx.x;
    if (i >= n) return;
    RowCtx r = row_setup(A, lde + k * lde_proof_stride, W, ptab, kc, i, xp_s);
    airs::CombT<false, 1> C{A->alpha, A->beta, A->group, &xp_s[0][threadIdx.x], (size_t)CONS_THREADS, acc192(), nullptr, 0,
                            &A->alpha_x[0][0], &A->beta_x[0][0], (size_t)CONS_MAX_CONSTRAINTS};
    C.rt = &A->rt;
    if (KIND == 0) airs::eval_rescue_item<AIR>((int)item, r.f, r.pv, C);
    else if (KIND == 1) airs::eval_ecc_bank<AIR>((int)item, r.f, r.pv, C);
    else airs::eval_ecc_final<AIR>(r.f, r.pv, C);
    part[k * part_proof_stride + ((unsigned long long)item * ce + kc) * n + i] = C.sum.reduce();
}

template <int AIR>
__global__ void __launch_bounds__(CONS_THREADS, CSG_REST_MINBLOCKS)
cons_rest_many_kernel(const ConsArgs *__restrict__ args, unsigned ce, const fe *__restrict__ lde, unsigned long long lde_proof_stride,
                      const fe *__restrict__ W, const fe *__restrict__ ptab, const fe *__restrict__ apoly, const fe *__restrict__ part,
                      unsigned long long part_proof_stride, unsigned nparts, const fe *__restrict__ binv, fe *__restrict__ out) {
    __shared__ fe xp_s[airs::MAX_GROUPS][CONS_THREADS];
    const unsigned k = blockIdx.y / ce, kc = blockIdx.y % ce;
    const ConsArgs *A = args + k;
    const unsigned long long n = 1ULL << A->logn, i = blockIdx.x * (unsigned long long)CONS_THREADS + threadIdx.x;
    if (i >= n) return;
    RowCtx r = row_setup(A, lde + k * lde_proof_stride, W, ptab, kc, i, xp_s);
    airs::CombT<false, 1> C{A->alpha, A->beta, A->group, &xp_s[0][threadIdx.x], (size_t)CONS_THREADS, acc192(), nullptr, 0,
                            &A->alpha_x[0][0], &A->beta_x[0][0], (size_t)CONS_MAX_CONSTRAINTS};
    airs::eval_rest<AIR>(r.f, r.pv, C);
    const fe x = r.x;
    const fe *pk = part + k * part_proof_stride;
    fe t = C.sum.reduce();
    for (unsigned p = 0; p < nparts; p++) t = add(t, pk[((unsigned long long)p * ce + kc) * n + i]);
    fe res = mul(mul(t, sub(x, A->g_last)), A->zinv[kc]);
    unsigned a = 0;
    for (unsigned g = 0; g < A->nbgroups; g++) {
        const fe xpb = mul(A->b_shift_adj[kc][g], W[(A->b_adj_mod[g] * i) & (n - 1)]);
        acc192 s;
        for (; a < A->nassertions && A->a_group[a] == g; a++) {
            fe v = A->a_value[a];
            if (A->a_poly_len[a] > 1) {   // Assertion::sequence: value polynomial evaluated at x * g^-first_step
                const fe *poly = apoly + A->a_poly_off[a];
                const fe y = mul(x, A->a_xoff[a]);
                v = 0;
                for (unsigned m = A->a_poly_len[a]; m-- > 0;) v = add(mul(v, y), poly[m]);
            }
            s.mac(add(A->a_alpha[a], mul(A->a_beta[a], xpb)), sub(r.f.cur(A->a_col[a]), v));
        }
        res = add(res, mul(s.reduce(), binv[((unsigned long long)g * ce + kc) * n + i]));
    }
    out[((unsigned long long)k * ce + kc) * n + i] = res;
}

template <int AIR>
void launch_many(const ConsArgs *args_dev, const ConsArgs &h, size_t count, const fe *lde, size_t lde_proof_stride, const fe *W, const fe *ptab,
                 const fe *apoly, fe *part, fe *binv, fe *out, Stream &st) {
    const unsigned long long n = 1ULL << h.logn;
    const unsigned gx = (unsigned)((n + CONS_THREADS - 1) / CONS_THREADS), ce = h.ncosets, gy = (unsigned)(ce * count);
    constexpr int NR = airs::Items<AIR>::rescue, NE = airs::Items<AIR>::ecc;
    const unsigned long long pstride = (unsigned long long)(NR + NE) * ce * n;
    if (NR > 0) CSG_LAUNCH(st, (cons_item_many_kernel<AIR, 0>), dim3(gx, gy, NR > 0 ? NR : 1), CONS_THREADS, 0, args_dev, ce, lde, (unsigned long long)lde_proof_stride, W, ptab, part, pstride);
    fe *ecc_part = part + (size_t)NR * ce * n;
    if (NE > 0) CSG_LAUNCH(st, (cons_item_many_kernel<AIR, 1>), dim3(gx, gy, 2), CONS_THREADS, 0, args_dev, ce, lde, (unsigned long long)lde_proof_stride, W, ptab, ecc_part, pstride);
    if (NE > 0) CSG_LAUNCH(st, (cons_item_many_kernel<AIR, 2>), dim3(gx, gy, 1), CONS_THREADS, 0, args_dev, ce, lde, (unsigned long long)lde_proof_stride, W, ptab, ecc_part, pstride);
    // the divisor inverses of proof 0 serve every proof of the batch
    if (h.nbgroups > 0)
        CSG_LAUNCH(st, boundary_inverse_kernel, dim3((unsigned)((n + INV_CHUNK * INV_THREADS - 1) / (INV_CHUNK * INV_THREADS)), ce, h.nbgroups),
                   INV_THREADS, 0, args_dev, W, binv);
    CSG_LAUNCH(st, cons_rest_many_kernel<AIR>, dim3(gx, gy), CONS_THREADS, 0, args_dev, ce, lde, (unsigned long long)lde_proof_stride, W, ptab, apoly,
               (const fe *)part, pstride, (unsigned)(NR + NE), (const fe *)binv, out);
}

}  // namespace

size_t constraint_items_many(int air_id) {
    switch (air_id) {
    case airs::TRANSACTION: return airs::Items<airs::TRANSACTION>::rescue + airs::Items<airs::TRANSACTION>::ecc;
    case airs::MERKLE_UPDATE: return airs::Items<airs::MERKLE_UPDATE>::rescue;
    case airs::MERKLE_INIT: return airs::Items<airs::MERKLE_INIT>::rescue;
    case airs::SCHNORR: return airs::Items<airs::SCHNORR>::rescue + airs::Items<airs::SCHNORR>::ecc;
    case airs::RESCUE: return airs::Items<airs::RESCUE>::rescue;
    default: return 0;
    }
}

void eval_constraints_many(int air_id, const ConsArgs *args_dev, const ConsArgs &h0, size_t count, const fe *lde, size_t lde_proof_stride, const fe *W,
                           const fe *ptab, const fe *apoly, fe *part, fe *binv, fe *out, Stream &st) {
    switch (air_id) {
    case airs::TRANSACTION: launch_many<airs::TRANSACTION>(args_dev, h0, count, lde, lde_proof_stride, W, ptab, apoly, part, binv, out, st); break;
    case airs::MERKLE_UPDATE: launch_many<airs::MERKLE_UPDATE>(args_dev, h0, count, lde, lde_proof_stride, W, ptab, apoly, part, binv, out, st); break;
    case airs::MERKLE_INIT: launch_many<airs::MERKLE_INIT>(args_dev, h0, count, lde, lde_proof_stride, W, ptab, apoly, part, binv, out, st); break;
    case airs::SCHNORR: launch_many<airs::SCHNORR>(args_dev, h0, count, lde, lde_proof_stride, W, ptab, apoly, part, binv, out, st); break;
    case airs::RANGE: launch_many<airs::RANGE>(args_dev, h0, count, lde, lde_proof_stride, W, ptab, apoly, part, binv, out, st); break;
    case airs::RESCUE: launch_many<airs::RESCUE>(args_dev, h0, count, lde, lde_proof_stride, W, ptab, apoly, part, binv, out, st); break;
    default: throw std::runtime_error("unknown AIR id");
    }
}

}  // namespace csg
