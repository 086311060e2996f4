// Host-side description of the six AIRs: what each `impl Air` of the reference hands to winterfell besides
// evaluate_transition -- trace width, transition-constraint degrees, periodic columns and boundary assertions.
//   TransactionAir   src/air.rs:76-108 (degrees), 175-184 (assertions), 194-380 (periodic columns)
//   MerkleAir        src/merkle/update/air.rs:46-56, 158-212, 371-401
//   PreMerkleAir     src/merkle/init/air.rs:50-150, 204-211
//   SchnorrAir       src/schnorr/air.rs:50-58, 115-299, 533-585
//   RangeProofAir    src/range/air.rs:43-105
//   RescueAir        benches/rescue.rs:163-254
// plus the winterfell-side bookkeeping derived from them (constraint groups, degree adjustments, divisors).
#pragma once
#include <cstddef>
#include <cstdint>
#include <vector>

#include "../field.cuh"

namespace csg {
using f63::fe;
inline unsigned ilog2_host(size_t n) { unsigned l = 0; while (((size_t)1 << l) < n) l++; return l; }

struct Degree { uint32_t base; std::vector<uint32_t> cycles; };   // TransitionConstraintDegree::{new, with_cycles}
struct PeriodicColumn { std::vector<fe> values; };                  // one cycle, Montgomery form; length = period
struct Assertion {                                                  // Assertion::{single, periodic, sequence}
    uint32_t column; size_t first_step, stride;                     // stride 0 = single
    std::vector<fe> values;                                         // 1 value unless a sequence
};

struct AirDesc {
    int id = -1;
    uint32_t width = 0;
    size_t trace_len = 0;
    std::vector<Degree> degrees;
    std::vector<PeriodicColumn> periodic;
    std::vector<Assertion> assertions;   // sorted the way winterfell orders them: (stride, first_step, column)
    std::vector<uint64_t> pub_inputs;    // canonical words, in PublicInputs::write_into order

    size_t num_constraints() const { return degrees.size(); }
    size_t ce_blowup() const;                            // AirContext: max over constraints of next_pow2(base + #cycles), at least 2
    size_t evaluation_degree(const Degree &d) const;     // base*(n-1) + sum (n/cycle)*(cycle-1)
};
// throws std::invalid_argument on malformed input (wrong number of public inputs, trace length not matching the AIR)
AirDesc make_air(int air_id, size_t trace_len, const uint64_t *pub, size_t npub);

// transition-constraint groups (one per distinct evaluation degree, in order of first appearance) and boundary groups
// (one per distinct divisor), with their degree adjustments: winterfell Air::get_transition_constraints /
// get_boundary_constraints
struct TransitionGroups {
    std::vector<uint8_t> group_of;       // per constraint
    std::vector<uint64_t> adj;           // per group: composition_degree + (n - 1) - evaluation_degree
};
struct BoundaryGroup { size_t num_steps, first_step, stride; uint64_t adj; fe offset; };   // divisor x^num_steps - offset
struct BoundaryGroups {
    std::vector<BoundaryGroup> groups;
    std::vector<uint32_t> group_of;      // per (sorted) assertion
};
TransitionGroups transition_groups(const AirDesc &air);
BoundaryGroups boundary_groups(const AirDesc &air);

// the merged transition constraints sum_s result_s * (alpha_s + beta_s * xp[group(s)]) of AIR `id` on one row pair, host build of
// airs.cuh (verifier.cpp); pv: the periodic values of the row.  With a one-hot alpha and beta = 0 it is result_s alone.
fe eval_merged_any(int id, const AirDesc &air, const TransitionGroups &tg, const std::vector<fe> &cur, const std::vector<fe> &next, const std::vector<fe> &pv,
                   const std::vector<fe> &alpha, const std::vector<fe> &beta, const std::vector<fe> &xp);

}  // namespace csg
