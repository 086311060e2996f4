// Batched kernels of csg_prove_many: the proof index is a grid dimension, every launch serves all K proofs of a batch.
//
// Layout of a batch of K proofs (w trace columns, n rows, blowup b, ce composition columns):
//   coefficients, composition columns, DEEP polynomials   [proof][column][row]
//   LDE matrices (trace, composition, DEEP)                [coset][proof][column][row]: proof k's view is the single-proof form
//                                                          (coset_stride = K*w*n, col_stride = n) at offset k*w*n
//   Merkle trees                                           [proof][2 * leaves digests], heap layout of commit.cuh
//   FRI layers                                             [proof][m]
#pragma once
#include "../constraints.cuh"
#include "../dev.cuh"
#include "../stages.cuh"

namespace csg {

// digests of the rows of K coset-major matrices (proof k at data + k * proof_stride) into the leaves of K trees
// (leaves + k * tree_words: leaf j = kc + ncosets*i of tree k)
void hash_rows_many(const fe *data, unsigned width, size_t n, unsigned ncosets, size_t coset_stride, size_t col_stride, size_t proof_stride,
                    size_t count, int hash_fn, uint32_t *leaves, size_t tree_words, Stream &st);
// the interior nodes of K trees of nleaves leaves each (tree k at nodes + k * tree_words), one launch per level
void merkle_build_many(uint32_t *nodes, size_t nleaves, size_t count, size_t tree_words, int hash_fn, Stream &st);
// cols of proof k = composition_columns of e of proof k; both [proof][ce][n]
void composition_columns_many(const fe *e, fe *cols, size_t n, unsigned ce, const fe *mat_host, size_t count, Stream &st);
// partial sums of the evaluations of count*ncols polynomials of n coefficients (polys[c * n ..], proof c / ncols) at the npts points
// of their proof: pts_dev[(proof * npts + p) * 2] = z, [.. + 1] = z^256.  partial[(c * npts + p) * nblk + blk]; returns nblk
unsigned eval_polys_many(const fe *polys, size_t n, size_t ncols, size_t count, const fe *pts_dev, unsigned npts, fe *partial, Stream &st);
unsigned eval_polys_many_blocks(size_t n);
// out[k * out_proof_stride + t * n + m] = sum_c coef_dev[(k * ncomb + t) * ncols + c] * polys[(k * ncols + c) * n + m]
void combine_polys_many(const fe *polys, size_t n, size_t ncols, size_t count, const fe *coef_dev, size_t ncomb, fe *out, size_t out_proof_stride, Stream &st);
// deep[k * n * b + j] from the LDE of the three combined polynomials of proof k, abc[(kc * count + k) * 3 * n + t * n + i]
void deep_quotients_many(const fe *abc, const fe *W, size_t n, size_t count, const DeepArgs *args_dev, unsigned ncosets, fe *deep, Stream &st);
// out[k * m/4 + i] = fold by 4 of layer k (evals[k * m ..]) with alphas_dev[k]; a.alpha is ignored
void fri_fold4_many(const fe *evals, size_t m, const fe *W, const FoldArgs &a, const fe *alphas_dev, size_t count, fe *out, Stream &st);

// opening gathers driven by job tables: one launch for every row job and one for every digest job of the batch
struct RowJob {
    const fe *data;
    unsigned width, ncosets;
    unsigned long long coset_stride, col_stride;
    unsigned idx_off, npos;
    unsigned long long rows_off;   // in words
};
struct DigestJob {
    const uint32_t *nodes;
    unsigned idx_off, count;
    unsigned long long out_off;   // in 32-bit words
};
// rows[job.rows_off + r * width + c] = canonical element (c, idx[job.idx_off + r]) of the job's coset-major matrix
void gather_rows_jobs(const RowJob *jobs_dev, size_t njobs, size_t max_elems, const uint32_t *idx_dev, uint64_t *rows, Stream &st);
// out[job.out_off + 8 * t ..] = node idx[job.idx_off + t] of the job's tree
void gather_digests_jobs(const DigestJob *jobs_dev, size_t njobs, size_t max_count, const uint32_t *idx_dev, uint32_t *out, Stream &st);

// the direct (all-coset) constraint evaluation of K proofs: args_dev[k] describes proof k, whose LDE is lde + k * lde_proof_stride;
// part: constraint_items_many(air_id) * ce * n elements per proof; binv: the boundary divisor inverses, shared by the proofs
// (they depend on the domain and the assertion shape only), CONS_MAX_BGROUPS * ce * n elements; out[k][kc][i]
void eval_constraints_many(int air_id, const ConsArgs *args_dev, const ConsArgs &h0, size_t count, const fe *lde, size_t lde_proof_stride, const fe *W,
                           const fe *ptab, const fe *apoly, fe *part, fe *binv, fe *out, Stream &st);
size_t constraint_items_many(int air_id);

}  // namespace csg
