// csg_validate_*: winterfell's debug-build `trace.validate(&air)` on the GPU (see include/csg.h).  One pass of the constraint code of
// airs.cuh over the trace domain itself -- rows (s, s+1) for s < n-1, periodic column c at step s is values[s mod P], no LDE -- plus
// a check of every asserted cell.  The kernels (kernels.cu) take the trace index in the grid, so a single trace is a batch of one.
// The single-proof driver (prover_ctx.cuh) owns one Validator per context, created on the first call and deleted with the context.
#pragma once
#include <cstddef>
#include <cstdint>
#include <vector>

#include "../../../include/csg.h"
#include "../constraints.cuh"
#include "../dev.cuh"
#include "../host/air_desc.hpp"

namespace csg {

// what the row kernels of one call share: the periodic-column layout, and two independent random combinations of the constraint
// slots.  CombT<false, 2> forms alpha[0] . result and alpha[1] . result with the coefficient alpha + beta * xp[group] of a slot:
// beta is zero and xp points at `zero`, so only alpha counts.
struct ValArgs {
    unsigned logn, width, nperiodic;
    unsigned long long ptab_stride;   // words between the periodic tables of consecutive traces (0: one table serves all)
    unsigned poff[CONS_MAX_PERIODIC], pmask[CONS_MAX_PERIODIC];
    fe alpha[2][CONS_MAX_CONSTRAINTS];
    fe beta[CONS_MAX_CONSTRAINTS];    // zero
    unsigned char group[CONS_MAX_CONSTRAINTS];
    fe zero;
};

// kernels.cu.  The trace words of K traces [K][w][n] in any 64-bit form -> Montgomery words reduced below p, into `mont` (may
// equal `src`, never written otherwise).
void validate_to_mont(const uint64_t *src, fe *mont, size_t count, int repr, Stream &st);
// part of the call per AIR: item partial sums into `part` ([K][items][2][n]), then per step the sum of everything and its test for
// zero: flags[k * n + s] = 1 if step s of trace k fails (0 for s = n-1), counts[k] += number of failing steps
void validate_rows(int air_id, const ValArgs *args_dev, const ValArgs &h, size_t K, const fe *mont, const fe *ptab, fe *part,
                   uint8_t *flags, unsigned long long *counts, Stream &st);
size_t validate_items(int air_id);   // the heavy items of an AIR (Rescue residuals, curve banks, final addition)
// asserted cells: cell c of trace k is (col[c], step[c]) with value val[k * ncells + c]; cflags[k * ncells + c] = 1 if it differs,
// counts[k] += number of failing cells
void validate_cells(size_t K, const fe *mont, unsigned w, size_t n, const uint32_t *col, const uint32_t *step, const fe *val, size_t ncells,
                    uint8_t *cflags, unsigned long long *counts, Stream &st);

// validate.cu
class Validator;
Validator *validator_new();
void validator_delete(Validator *v);
// K traces of one AIR (airs[k]: the AirDesc of trace k, from its public inputs) and length n: `host` (one trace in host memory) or
// `dev` (K traces [K][w][n] in device memory of the stream's device, read in place).  out receives K reports.  Every check on the
// arguments belongs to the caller.
void validate_traces(Validator *v, Stream &st, int air_id, const std::vector<AirDesc> &airs, const uint64_t *host, const uint64_t *dev, int repr,
                     size_t n, csg_trace_report *out);
// the device bytes validate_traces needs for K traces of width w and length n with `ptotal` periodic words and `ncells` asserted
// cells each (at most), and what the validator holds already
size_t validate_footprint(int air_id, size_t K, size_t w, size_t n, size_t ptotal, size_t ncells);
size_t validator_held(const Validator *v);

// every transition constraint slot of AIR `air` at step `step` of rows cur, next (Montgomery): result[] of evaluate_transition
std::vector<fe> transition_values(const AirDesc &air, const TransitionGroups &tg, size_t step, const std::vector<fe> &cur, const std::vector<fe> &next);

}  // namespace csg
