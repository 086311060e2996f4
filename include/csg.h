/* csg.h -- C ABI of libcsg.so, the B200-native proving backend for certificate-stark.
 *
 * The reference has no FFI: its hot path is entered through the Rust trait call
 *     prover.prove(trace)                      /root/reference/src/lib.rs:140
 * (also src/schnorr/mod.rs:171, src/merkle/init/mod.rs:105, src/merkle/update/mod.rs:105, src/range/mod.rs:99,
 * benches/rescue.rs:84), which dispatches into winterfell's generic `Prover::prove` with the AIR the crate defines
 * through `impl Air` (src/air.rs:70-189 and the five sub-AIRs).  Generic Rust cannot cross an FFI boundary, so the
 * AIR is selected by id and everything the Rust side owns (trace, public inputs, ProofOptions, Fiat-Shamir
 * challenges) crosses as plain integers in CANONICAL form (BaseElement::to_repr), little-endian u64.
 *
 * Two levels are exported:
 *   1. csg_prove()            one call = Prover::prove(trace) -> StarkProof::to_bytes()
 *   2. csg_set_air() .. csg_open()   the per-stage calls a patched winterfell `generate_proof` would make,
 *                             keeping the transcript (RandomCoin) and proof serialisation on the Rust side.
 * plus the witness builders (build_trace of each prover) and a few kernel-level entry points used by the
 * parity tests and the kernel sweep.  All functions return 0 on success; they never unwind.  A context is
 * single-threaded and owns all device memory; every pointer argument is a HOST pointer owned by the caller, except the
 * traces_dev buffers of csg_prove_many_device and csg_build_traces_many_*, which are device memory the caller owns.
 */
#ifndef CSG_H
#define CSG_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

enum { CSG_OK = 0, CSG_ERR_ARG = 1, CSG_ERR_CUDA = 2, CSG_ERR_STATE = 3, CSG_ERR_UNSUPPORTED = 4, CSG_ERR_COIN = 5 };
/* csg_verify results other than CSG_OK (the VerifierError kinds of winterfell::verify) */
enum { CSG_VERIFY_MALFORMED = 16, CSG_VERIFY_OOD_MISMATCH = 17, CSG_VERIFY_POW = 18, CSG_VERIFY_TRACE_QUERY = 19,
       CSG_VERIFY_CONSTRAINT_QUERY = 20, CSG_VERIFY_FRI = 21, CSG_VERIFY_WEAK_OPTIONS = 22 };

/* AIR ids: the six `impl Air` of the reference */
enum {
    CSG_AIR_TRANSACTION = 0,   /* TransactionAir   src/air.rs:64-189            94 cols, 115 constraints */
    CSG_AIR_MERKLE_UPDATE = 1, /* MerkleAir        src/merkle/update/air.rs     65 cols, 106 constraints */
    CSG_AIR_MERKLE_INIT = 2,   /* PreMerkleAir     src/merkle/init/air.rs       58 cols,  56 constraints */
    CSG_AIR_SCHNORR = 3,       /* SchnorrAir       src/schnorr/air.rs           56 cols,  56 constraints */
    CSG_AIR_RANGE = 4,         /* RangeProofAir    src/range/air.rs              2 cols,   2 constraints */
    CSG_AIR_RESCUE = 5         /* RescueAir        benches/rescue.rs:163-268    14 cols,  14 constraints */
};
enum { CSG_HASH_BLAKE3_256 = 2, CSG_HASH_SHA3_256 = 3 }; /* HashFunction (src/lib.rs:82, examples/state-transition.rs:67-71) */
/* FieldExtension (src/lib.rs:83; the example binary takes 1/2/3, examples/state-transition.rs:62-66).  With Quadratic or Cubic
 * the challenges, composition columns, out-of-domain frame, DEEP composition and FRI layers are elements of the degree-2 / 3
 * extension: such an element crosses the ABI (and is serialised) as its 2 / 3 canonical words in order. */
enum { CSG_FIELD_EXT_NONE = 1, CSG_FIELD_EXT_QUADRATIC = 2, CSG_FIELD_EXT_CUBIC = 3 };

/* ProofOptions::new(num_queries, blowup_factor, grinding_factor, hash_fn, field_extension, fri_folding_factor,
 * fri_max_remainder_size)  -- src/lib.rs:78-86 */
typedef struct {
    uint32_t num_queries, blowup_factor, grinding_factor, hash_fn, field_extension, fri_folding_factor, fri_max_remainder_size;
} csg_options;

/* representation of the trace words handed to csg_prove / csg_load_trace / csg_prove_trace (SURVEY.md 8(b)).  winterfell's f63
 * BaseElement is a u64 in Montgomery form (R = 2^64; src/utils/ecc.rs:23-45 gives the generator through from_raw_unchecked), so
 * TraceTable column memory can cross the boundary untouched as CSG_REPR_MONTGOMERY; CSG_REPR_CANONICAL = BaseElement::to_repr(). */
enum { CSG_REPR_CANONICAL = 0, CSG_REPR_MONTGOMERY = 1 };

typedef struct csg_ctx csg_ctx;

/* ---- context ------------------------------------------------------------------------------------------------- */
csg_ctx *csg_create(int device);            /* NULL if the device cannot be opened */
void csg_destroy(csg_ctx *ctx);
const char *csg_last_error(const csg_ctx *ctx);
void csg_free(void *p);                     /* frees buffers returned by csg_prove */
/* page-locked host memory for traces (cudaHostAlloc / cudaHostRegister): from it the H2D copy runs at link speed under the trace
 * extension.  A trace in ordinary pageable memory is accepted as well: the library stages it through its own pinned buffers with
 * the host's threads (slower by the host memcpy, still overlapped).  csg_host_alloc returns NULL on failure. */
void *csg_host_alloc(size_t bytes);
void csg_host_free(void *p);
int csg_host_register(void *p, size_t bytes);
int csg_host_unregister(void *p);

/* ---- level 1: replaces `prover.prove(trace)` (src/lib.rs:140) -------------------------------------------------
 * trace: column-major [width][trace_len], exactly TraceTable's storage; repr says whether the words are canonical or Montgomery.
 * pub:   the AIR's PublicInputs as canonical words in write_into() order:
 *        TRANSACTION / MERKLE_UPDATE  initial_root[7] final_root[7]      (src/air.rs:57-62)
 *        MERKLE_INIT                  s_inputs[14] r_inputs[14] delta    (src/merkle/init/air.rs:36-42)
 *        SCHNORR                      per signature: message[28] Rx[6] s[4 LE words]  (src/schnorr/air.rs:38-46)
 *        RANGE                        number                              (src/range/air.rs:33-37)
 *        RESCUE                       seed[7] result[7]                   (benches/rescue.rs:136-141)
 * proof: malloc'ed StarkProof::to_bytes(); release with csg_free. */
int csg_prove(csg_ctx *ctx, int air_id, const uint64_t *trace, int repr, size_t trace_len, const uint64_t *pub, size_t npub,
              const csg_options *opt, uint8_t **proof, size_t *proof_len);

/* the same with one pointer per column (columns[c] -> trace_len words): a winterfell TraceTable keeps every column in its own
 * Vec<BaseElement> (TraceTable::get_column, used at src/prover.rs:107-127), so its memory crosses the boundary without being copied
 * together first */
int csg_prove_columns(csg_ctx *ctx, int air_id, const uint64_t *const *columns, int repr, size_t trace_len, const uint64_t *pub, size_t npub,
                      const csg_options *opt, uint8_t **proof, size_t *proof_len);

/* K independent proofs of one AIR, one trace length and one csg_options: traces[k] is a column-major [width][trace_len]
 * trace (repr as in csg_prove), pubs = K * npub public-input words.  proofs[k] receives a malloc'ed proof that is
 * byte-identical to what csg_prove would return for (traces[k], pubs + k*npub); release each with csg_free.  On failure
 * every proofs[k] is NULL.
 * Every stage runs as one launch sequence over all K proofs and every Fiat-Shamir step is one device->host copy for the batch, so
 * launches and round trips are paid once per batch: the call is for many small proofs (range proofs, signatures, Rescue chains).
 * The context's single-proof state (csg_set_air, the resident and the prefetched trace) is not touched; the batch keeps its own
 * device buffers, reused by the next batch of the same shape and freed by csg_destroy.  csg_get_timings then reports the batch.
 * CSG_ERR_UNSUPPORTED: field_extension 2 or 3, a context attached to a group (world > 1), trace_len > 2^16.
 * CSG_ERR_ARG: count == 0 or count > 1024, count * width > 65535, null pointers, a bad repr or npub, a batch whose device
 * footprint does not fit the free memory.  All checks run before anything is enqueued. */
int csg_prove_many(csg_ctx *ctx, int air_id, size_t count, const uint64_t *const *traces, int repr, size_t trace_len,
                   const uint64_t *pubs, size_t npub, const csg_options *opt, uint8_t **proofs, size_t *proof_lens);
/* csg_prove_many with the K traces already in device memory: traces_dev is ONE contiguous buffer [count][width][trace_len] on the
 * context's device (cudaMalloc'ed, a torch CUDA tensor, the output of csg_build_traces_many_*).  Same checks, limits, errors and
 * proof bytes as csg_prove_many; host, pinned host and managed memory and memory of another device are CSG_ERR_ARG.  The library
 * reads the buffer in place and never writes it.  The caller's writes to it must have finished before the call (synchronise the
 * stream that wrote it): the batch runs on the context's own stream. */
int csg_prove_many_device(csg_ctx *ctx, int air_id, size_t count, const uint64_t *traces_dev, int repr, size_t trace_len,
                          const uint64_t *pubs, size_t npub, const csg_options *opt, uint8_t **proofs, size_t *proof_lens);
/* ---- verification: replaces `winterfell::verify::<Air>(proof, pub_inputs)` (src/lib.rs:144-150).  Host-only, as in the
 * reference; needs no context and no GPU.  Returns CSG_OK or one of CSG_VERIFY_*. */
int csg_verify(int air_id, const uint64_t *pub, size_t npub, const uint8_t *proof, size_t proof_len);
/* csg_verify trusts the ProofOptions recorded inside the proof, as winterfell::verify does.  An acceptance check should not: this
 * form also rejects (CSG_VERIFY_WEAK_OPTIONS) a proof made with fewer queries, a smaller blowup or grinding factor, a smaller
 * field extension, another hash function or a larger FRI remainder than `min_options` -- the options the verifying side holds
 * (TransactionExample keeps them in `options`, src/lib.rs:92-98). */
int csg_verify_with_options(int air_id, const uint64_t *pub, size_t npub, const uint8_t *proof, size_t proof_len, const csg_options *min_options);

/* ---- level 2: the stages of Prover::prove, transcript on the caller's side --------------------------------------
 * call order: set_air, load_trace, [extend_and_commit_trace, eval_constraints, commit_composition, ood, deep,
 * (fri_commit_layer, fri_fold)*, fri_remainder, open]; prove_loaded() runs the bracketed part with the built-in
 * transcript.  Challenges are canonical field elements drawn by the caller's RandomCoin. */
int csg_set_air(csg_ctx *ctx, int air_id, size_t trace_len, const csg_options *opt, const uint64_t *pub, size_t npub);
int csg_load_trace(csg_ctx *ctx, const uint64_t *trace, int repr);           /* H2D copy of width*trace_len words */
int csg_prove_loaded(csg_ctx *ctx, uint8_t **proof, size_t *proof_len);      /* proof of the resident trace */
/* proof of a trace in HOST memory for the AIR set by csg_set_air: the H2D copy is pipelined with the trace extension */
int csg_prove_trace(csg_ctx *ctx, const uint64_t *trace, int repr, uint8_t **proof, size_t *proof_len);
/* A stream of traces for the AIR set by csg_set_air (a prover service proving batch after batch): the copy of the NEXT trace runs on
 * its own stream under the proof of the current one, so in the steady state a proof costs what it costs with the trace already in
 * HBM.  csg_prefetch_trace starts the copy of the first trace and returns at once; csg_prove_prefetched proves the trace that is
 * waiting and, when next_trace is not NULL, starts the copy of that one first.  The memory of a prefetched trace must stay valid
 * until the csg_prove_prefetched call that proves it has started (page-locked memory -- csg_host_alloc / csg_host_register --
 * for the copy to be asynchronous; pageable memory works but is copied synchronously).  One trace can wait at a time. */
int csg_prefetch_trace(csg_ctx *ctx, const uint64_t *trace, int repr);
int csg_prove_prefetched(csg_ctx *ctx, const uint64_t *next_trace, int next_repr, uint8_t **proof, size_t *proof_len);
int csg_reload_resident_trace(csg_ctx *ctx);                                 /* re-arm the trace left in HBM by the last csg_load_trace (benchmarks) */
int csg_extend_and_commit_trace(csg_ctx *ctx, uint8_t root[32]);             /* Trace::extend + build_commitment */
/* t_coeffs: (alpha,beta) per transition constraint; b_coeffs: (alpha,beta) per assertion in winterfell's sorted order */
int csg_eval_constraints(csg_ctx *ctx, const uint64_t *t_coeffs, const uint64_t *b_coeffs);
int csg_commit_composition(csg_ctx *ctx, uint8_t root[32]);                  /* into_poly + evaluate + commit */
/* OOD frame at z: trace polys at z and z*g (width each), composition columns at z^m (m = ce blowup) */
int csg_ood(csg_ctx *ctx, uint64_t z, uint64_t *frame_cur, uint64_t *frame_next, uint64_t *comp);
/* DEEP coefficients: per trace column (alpha, beta), per composition column delta, then (lambda, mu) */
int csg_deep(csg_ctx *ctx, const uint64_t *trace_ab, const uint64_t *comp_d, const uint64_t *lambda_mu /* 2 elements */);
/* with a field extension every challenge / frame entry of the level-2 calls is d words (t_coeffs, b_coeffs, trace_ab, comp_d,
 * lambda_mu, opened composition and FRI rows, the remainder); the two calls that take a challenge by value have pointer forms: */
int csg_ood_ext(csg_ctx *ctx, const uint64_t *z, uint64_t *frame_cur, uint64_t *frame_next, uint64_t *comp);
int csg_fri_fold_ext(csg_ctx *ctx, const uint64_t *alpha);
int csg_fri_commit_layer(csg_ctx *ctx, uint8_t root[32]);                    /* transpose/4, hash, Merkle */
int csg_fri_fold(csg_ctx *ctx, uint64_t alpha);                              /* degree-respecting projection */
int csg_fri_remainder(csg_ctx *ctx, uint64_t *out, size_t cap, size_t *len);
/* openings at the query positions (1..255 distinct positions inside the domain, else CSG_ERR_ARG): `rows` receives npos rows of the
 * opened matrix, row-major -- the caller provides npos * width words (trace: AIR width; composition: ce_blowup * d; FRI layer: 4 * d);
 * `paths` (capacity `cap` bytes) receives BatchMerkleProof::serialize_nodes() */
int csg_open_trace(csg_ctx *ctx, const uint64_t *positions, size_t npos, uint64_t *rows, uint8_t *paths, size_t cap, size_t *paths_len);
int csg_open_composition(csg_ctx *ctx, const uint64_t *positions, size_t npos, uint64_t *rows, uint8_t *paths, size_t cap, size_t *paths_len);
int csg_open_fri_layer(csg_ctx *ctx, size_t layer, const uint64_t *positions, size_t npos, uint64_t *rows, uint8_t *paths, size_t cap, size_t *paths_len);

/* ---- one proof sharded over several GPUs by LDE coset (SURVEY.md 8(e); the reference has no multi-device path) -----------
 * `world` contexts, one per GPU (world a power of two dividing the blowup factor), each owning blowup/world cosets of the
 * LDE domain: column blocks are interpolated per context and the coefficients all-gathered; extension, row hashing,
 * constraint evaluation, composition LDE and DEEP quotients run on the owned cosets only; leaf digests travel by all-to-all into
 * contiguous leaf ranges so that every context builds the Merkle subtree of its range (the G roots are all-gathered, the top
 * levels replicated; path nodes are collected from the owning contexts at opening time); per-coset composition interpolants, OOD
 * values and DEEP evaluations are all-gathered; FRI is built by every context, so every context follows the same transcript and
 * returns the same proof bytes (identical to the single-GPU proof).
 * After attaching, EVERY context of the group makes the same sequence of calls (csg_set_air .. csg_prove_loaded, or
 * csg_prove) with the same arguments; calls block until the peers arrive.
 *   csg_dist_init        one process per GPU (torchrun): NCCL; rank 0 creates the id with csg_dist_unique_id and the host
 *                        distributes it (torch.distributed broadcast, MPI, a file)
 *   csg_dist_init_local  one process, one host thread per context: peer copies; contexts may share a device (tests)
 * world = 1 detaches. */
int csg_dist_unique_id(uint8_t id[128]);
int csg_dist_init(csg_ctx *ctx, int rank, int world, const uint8_t id[128]);
int csg_dist_init_local(csg_ctx **ctxs, int world);
int csg_dist_info(const csg_ctx *ctx, int *rank, int *world);
/* what rank `rank` of `world` owns for an AIR of `width` columns and constraint-evaluation blowup `ce_blowup` (<= blowup): a
 * contiguous block of LDE cosets, the constraint-evaluation cosets among them (possibly none), and the block of trace columns
 * it interpolates -- the only columns csg_prove / csg_prove_trace read from the caller's trace on that rank.  Needs no GPU. */
typedef struct { uint32_t first_coset, num_cosets, first_ce_coset, num_ce_cosets, first_column, num_columns, columns_per_rank; } csg_shard_plan;
int csg_dist_plan(int rank, int world, uint32_t blowup, uint32_t ce_blowup, uint32_t width, csg_shard_plan *out);
/* the column chunks in which that rank walks its column block in stage 1 (copy from the caller's memory overlapped with the
 * extension when from_host != 0, one chunk for a resident trace): sizes[0 .. *count), adding up to num_columns.  *count is set even
 * when cap is too small (CSG_ERR_ARG).  Needs no GPU; the CPU tests check the geometry of every world size with it. */
int csg_dist_trace_chunks(int rank, int world, uint32_t blowup, uint32_t ce_blowup, uint32_t width, int from_host, uint32_t *sizes, size_t cap, size_t *count);

/* per-stage device times of the last proof, milliseconds (CUDA events on the proving stream) */
typedef struct {
    float h2d, lde, commit_trace, constraints, composition, ood_deep, fri, queries, total;
    uint64_t kernel_launches; /* kernels launched by the last proof */
    /* the four kernels of the constraint stage: Rescue residuals, scalar-multiplication banks, final point addition,
     * linear constraints + divisors + boundary terms (CUDA events between the launches) */
    float cons_rescue, cons_ecc_banks, cons_ecc_final, cons_rest;
    float comm; /* sharded proofs: time inside the exchanges (all-gathers, row sums), already included in the stage times */
    float cons_ecc_low; /* part of cons_ecc_banks: the curve-formula kernel on the even cosets alone (0 when the split is off) */
    /* kernels launched inside each stage, in the order lde, commit_trace, constraints, composition, ood_deep, fri, queries:
     * lets a profiler's launch list of one proof be cut into stages */
    uint32_t stage_launches[7];
    float batch_build; /* device time of the last csg_tx_batch_build_device */
} csg_timings;
int csg_get_timings(const csg_ctx *ctx, csg_timings *out);
/* CUDA events on the proving stream around an arbitrary sequence of calls (bench.py's timed region) */
int csg_timer_start(csg_ctx *ctx);
int csg_timer_stop(csg_ctx *ctx, float *ms);

/* ---- witness builders: build_trace() of each prover -------------------------------------------------------------
 * Traces are column-major canonical; `pub` receives get_pub_inputs(). */
typedef struct csg_tx_batch csg_tx_batch;   /* TransactionMetadata  (src/lib.rs:188-232) */
typedef struct csg_sig_batch csg_sig_batch; /* SchnorrExample's messages + signatures (src/schnorr/mod.rs:71-76) */
csg_tx_batch *csg_tx_batch_new(uint64_t seed, size_t num_tx, unsigned tree_depth); /* build_random, seeded (src/lib.rs:235-464) */
void csg_tx_batch_free(csg_tx_batch *b);
size_t csg_tx_batch_size(const csg_tx_batch *b);
void csg_tx_batch_roots(const csg_tx_batch *b, uint64_t initial_root[7], uint64_t final_root[7]);
int csg_build_trace_transaction(const csg_tx_batch *b, uint64_t *trace /* 94 x 1024*num_tx */, uint64_t pub[14]);   /* src/prover.rs:37-98 */
/* the same witness built ON THE DEVICE into the context's resident trace (SURVEY.md 8(f).1): call after csg_set_air for
 * CSG_AIR_TRANSACTION with trace_len = 1024 * num_tx, then csg_prove_loaded.  Only the packed batch (2.2 KB per transaction)
 * crosses PCIe.  csg_download_trace copies the resident canonical trace back (tests). */
int csg_build_trace_transaction_device(csg_ctx *ctx, const csg_tx_batch *b);
int csg_download_trace(csg_ctx *ctx, uint64_t *trace /* width x trace_len */);
/* TransactionMetadata::build_random ON THE DEVICE (SURVEY.md 8(f).4; src/lib.rs:235-464): the same seeded draws as
 * csg_tx_batch_new(seed, num_tx, tree_depth), but the depth-15 Rescue account tree, its update by every transfer, the authentication
 * paths, the signature points r.G and the message hashes are computed by kernels (the tree's history level by level: thousands of
 * independent permutations per launch instead of 32 dependent ones per transfer).  The packed witness records stay in HBM; only the
 * public inputs (root before the first transfer, root after the last) come back.  Follow with csg_set_air(TRANSACTION,
 * 1024 * num_tx, opt, pub, 14), csg_build_trace_transaction_resident, csg_prove_loaded.  csg_download_batch_records (tests) copies
 * the records back: csg_tx_batch_pack(csg_tx_batch_new(seed, ...)) bit for bit. */
int csg_tx_batch_build_device(csg_ctx *ctx, uint64_t seed, size_t num_tx, unsigned tree_depth, uint64_t pub[14]);
int csg_build_trace_transaction_resident(csg_ctx *ctx);
int csg_download_batch_records(csg_ctx *ctx, uint64_t *out /* 278 words per transfer */, size_t cap_words);
size_t csg_tx_batch_pack(const csg_tx_batch *b, uint64_t *out /* NULL: returns the word count */);
size_t csg_sig_batch_pack(const csg_sig_batch *b, uint64_t *out /* NULL: returns the word count */);
/* MerkleProver::build_trace (src/merkle/update/prover.rs:37-80) and SchnorrProver::build_trace (src/schnorr/prover.rs:52-80) on the
 * device, into the resident trace: call after csg_set_air for that AIR with trace_len = 512 * (transfers | signatures) */
int csg_build_trace_merkle_update_device(csg_ctx *ctx, const csg_tx_batch *b);
int csg_build_trace_schnorr_device(csg_ctx *ctx, const csg_sig_batch *b);
unsigned csg_tx_batch_depth(const csg_tx_batch *b);
int csg_build_trace_merkle_update(const csg_tx_batch *b, uint64_t *trace /* 65 x 512*num_tx */, uint64_t pub[14]); /* src/merkle/update/prover.rs:37-80 */
int csg_build_trace_merkle_init(const uint64_t s_inputs[14], const uint64_t r_inputs[14], uint64_t delta,
                                uint64_t *trace /* 58 x 16 */, uint64_t pub[29]);                                   /* src/merkle/init/prover.rs:35-53 */
csg_sig_batch *csg_sig_batch_new(uint64_t seed, size_t num_sig);
void csg_sig_batch_free(csg_sig_batch *b);
size_t csg_sig_batch_size(const csg_sig_batch *b);
int csg_build_trace_schnorr(const csg_sig_batch *b, uint64_t *trace /* 56 x 512*num_sig */, uint64_t *pub /* 38*num_sig */); /* src/schnorr/prover.rs:52-80 */
int csg_build_trace_range(uint64_t number, uint64_t *trace /* 2 x 64 */, uint64_t pub[1]);                          /* src/range/prover.rs:36-56 */
int csg_build_trace_rescue(const uint64_t seed[7], size_t chain_length, uint64_t *trace /* 14 x 8*len */, uint64_t pub[14]); /* benches/rescue.rs:279-321 */
/* Batch witness builders for csg_prove_many_device: build the traces of count proofs ON THE DEVICE into traces_dev, a device buffer
 * of the context's device that the caller owns and sizes [count][width][rows] (canonical words), and write the public inputs of
 * every proof to the host array pubs in csg_prove's word order.  The device has finished when they return.  count is 1..1024;
 * null pointers and a traces_dev that is not device memory of the context's device are CSG_ERR_ARG, checked before anything runs.
 * The builders keep their scratch with the batch (freed by csg_destroy) and leave the single-proof state alone.
 *   rescue:         count chains, seeds = count * 7 words (reduced mod p), rows = 8 * chain_length; chain_length a power of two
 *                   up to 8192; trace k and pubs + 14k equal csg_build_trace_rescue(seeds + 7k, chain_length)
 *   schnorr:        one proof per signature of the batch (56 x 512), pubs: 38 words per signature
 *   merkle_update:  one proof per transfer (65 x 512), pubs: 14 words per transfer (root before it, root after it)
 *   transaction:    one proof per transfer (94 x 1024), pubs as merkle_update; the batch's tree depth must be 15
 * Trace k of the last three is columns [k * rows, (k + 1) * rows) of the host builder's trace of the whole batch (for the
 * Merkle update with row 1 of columns 14 and 43 set to 1, as MerkleProver::build_trace sets them in every single proof). */
int csg_build_traces_many_rescue(csg_ctx *ctx, const uint64_t *seeds, size_t count, size_t chain_length, uint64_t *traces_dev, uint64_t *pubs);
int csg_build_traces_many_schnorr(csg_ctx *ctx, const csg_sig_batch *b, uint64_t *traces_dev, uint64_t *pubs);
int csg_build_traces_many_merkle_update(csg_ctx *ctx, const csg_tx_batch *b, uint64_t *traces_dev, uint64_t *pubs);
int csg_build_traces_many_transaction(csg_ctx *ctx, const csg_tx_batch *b, uint64_t *traces_dev, uint64_t *pubs);

/* ---- kernel-level entry points (parity tests, kernel sweep).  Host buffers in/out; values canonical ------------- */
/* per-column inverse NTT + coset LDE: cols [width][n] -> lde [width][n*blowup], natural order x_j = 3 * w^j */
int csg_k_lde(csg_ctx *ctx, const uint64_t *cols, size_t width, size_t n, size_t blowup, uint64_t *lde);
/* Blake3/SHA3 of every row of a column-major matrix [width][rows] -> rows*32 bytes */
int csg_k_hash_rows(csg_ctx *ctx, int hash_fn, const uint64_t *cols, size_t width, size_t rows, uint8_t *digests);
/* Merkle tree over nleaves 32-byte leaves -> nodes[2*nleaves][32], nodes[1] = root */
int csg_k_merkle(csg_ctx *ctx, int hash_fn, const uint8_t *leaves, size_t nleaves, uint8_t *nodes);
/* one FRI fold by 4 (domain offset 3, size n) */
int csg_k_fri_fold4(csg_ctx *ctx, const uint64_t *evals, size_t n, uint64_t alpha, uint64_t *out);
/* kernel sweep: LDE + row hash + Merkle over device-resident synthetic columns; returns per-stage ms */
int csg_k_sweep(csg_ctx *ctx, size_t width, size_t n, size_t blowup, int hash_fn, int iters, float ms_out[4]);

#ifdef __cplusplus
}
#endif
#endif
