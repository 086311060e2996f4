// csg_prove_many: K independent proofs of one AIR, one trace length and one csg_options through one launch sequence (see
// include/csg.h).  The batch driver and its kernels live in this directory; the single-proof driver (prover_ctx.cuh) owns one
// ManyProver per context, created on the first batch and deleted with the context.
#pragma once
#include <cstddef>
#include <cstdint>
#include <stdexcept>

#include "../../../include/csg.h"
#include "../dev.cuh"

namespace csg {

// a malformed batch (CSG_ERR_ARG); an unsupported one throws ManyUnsupported (CSG_ERR_UNSUPPORTED)
struct ManyArgError : std::runtime_error { using std::runtime_error::runtime_error; };
struct ManyUnsupported : std::runtime_error { using std::runtime_error::runtime_error; };

constexpr size_t MANY_MAX_COUNT = 1024;
constexpr size_t MANY_MAX_COLUMNS = 65535;       // count * width: the column transforms put columns on gridDim.y
constexpr unsigned MANY_MAX_LOG_TRACE = 16;      // longer traces: the single-proof path with its low-degree split

// where the traces of a batch are: K host traces (one pointer each, csg_prove_many) or one device buffer [K][width][trace_len] on
// the device of the stream (csg_prove_many_device), which the batch reads and never writes
struct ManyTraces {
    const uint64_t *const *host;
    const uint64_t *dev;
};
// ManyArgError unless p is device memory of the current device (not host, pinned host or managed memory, not another device's)
void check_device_buffer(const void *p, const char *what);

// device scratch of the batch witness builders (witness_many.cu): packed records, the K-item trace before it is regrouped, the
// final curve states of the Schnorr kernels, the last rows of the Rescue chains
struct ManyWitnessScratch {
    DBuf<uint64_t> records, trace, last;
    DBuf<fe> finals;
};

class ManyProver;
ManyProver *many_new();
void many_delete(ManyProver *m);
ManyWitnessScratch &many_scratch(ManyProver *m);
// Every check runs before anything is enqueued.  proofs[k] / proof_lens[k] receive malloc'ed proofs; on failure all are NULL.
// tm receives the stage times and launches of the batch.  The device of `st` must be current.
void many_prove(ManyProver *m, Stream &st, int air_id, size_t count, ManyTraces traces, int repr, size_t trace_len,
                const uint64_t *pubs, size_t npub, const csg_options *opt, uint8_t **proofs, size_t *proof_lens, csg_timings &tm);

// batch witness builders (witness_many.cu): count column-major traces [count][width][rows] into traces_dev, a device buffer of the
// current device that the caller owns, and the public inputs of each proof (csg_prove's word order) into pubs.  Every check runs
// before anything is enqueued; the device has finished when they return.  They use many_scratch(m) and nothing else of a context.
//   Rescue: RescueProver::build_trace of every seed (7 canonical words each), rows = 8 * chain_length
void many_build_rescue(ManyProver *m, Stream &st, const uint64_t *seeds, size_t count, size_t chain_length, uint64_t *traces_dev, uint64_t *pubs);
//   one proof per signature (CSG_AIR_SCHNORR, 512 rows) or per transfer (CSG_AIR_MERKLE_UPDATE, 512 rows; CSG_AIR_TRANSACTION,
//   1024 rows) from the packed records of the batch (witness.cuh); `batch` is a csg_sig_batch for Schnorr, else a csg_tx_batch
void many_build_items(ManyProver *m, Stream &st, int air_id, const void *batch, uint64_t *traces_dev, uint64_t *pubs);

}  // namespace csg
