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

class ManyProver;
ManyProver *many_new();
void many_delete(ManyProver *m);
// Every check runs before anything is enqueued.  proofs[k] / proof_lens[k] receive malloc'ed proofs; on failure all are NULL.
// tm receives the stage times and launches of the batch.  The device of `st` must be current.
void many_prove(ManyProver *m, Stream &st, int air_id, size_t count, const uint64_t *const *traces, int repr, size_t trace_len,
                const uint64_t *pubs, size_t npub, const csg_options *opt, uint8_t **proofs, size_t *proof_lens, csg_timings &tm);

}  // namespace csg
