// Stage arguments that the single-proof driver (prover_ctx.cuh) and the batch driver (many/prove_many.cu) compute on the host: the
// checks on an AIR's shape, the layout of the periodic-column tables, the constraint, composition, DEEP and FRI arguments, and the
// CSG_HOST_TRACE scope.  Needs ConsArgs, DeepArgs and FoldArgs: included by nvcc translation units only.
#pragma once
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <stdexcept>
#include <vector>

#include "../constraints.cuh"
#include "../dev.cuh"
#include "../stages.cuh"
#include "air_desc.hpp"
#include "proof_common.hpp"

namespace csg {

// throws std::invalid_argument for an AIR of trace length n that does not fit these options or the compiled table sizes
inline void check_air_shape(const AirDesc &air, const TransitionGroups &tg, const BoundaryGroups &bg, size_t n, const csg_options &o) {
    if (air.ce_blowup() > o.blowup_factor) throw std::invalid_argument("blowup factor is smaller than the constraint evaluation blowup of this AIR");
    check_remainder(n * o.blowup_factor, o);
    if (air.num_constraints() > (size_t)CONS_MAX_CONSTRAINTS || air.periodic.size() > (size_t)CONS_MAX_PERIODIC ||
        air.assertions.size() > (size_t)CONS_MAX_ASSERTIONS)
        throw std::invalid_argument("AIR exceeds the compiled table sizes");
    if (tg.adj.size() > (size_t)CONS_MAX_GROUPS || bg.groups.size() > (size_t)CONS_MAX_BGROUPS) throw std::invalid_argument("too many constraint groups");
    for (const PeriodicColumn &c : air.periodic) {
        const size_t P = c.values.size();
        if (P == 0 || (P & (P - 1)) || P > n) throw std::invalid_argument("periodic column length must be a power of two dividing the trace length");
    }
}

// Periodic columns in runs of equal period: a run goes through the transforms together.  In a batch of K proofs, proof k's copy of
// column c of a run sits at at(c, K, k) of each ce coset's block of K * total elements; a single proof is K = 1, k = 0.
struct PeriodicRun {
    size_t c0, c1, P, off;
    size_t at(size_t c, size_t K, size_t k) const { return K * off + (k * (c1 - c0) + c - c0) * P; }
};
struct PeriodicRuns { std::vector<PeriodicRun> runs; size_t total = 0; };
inline PeriodicRuns periodic_runs(const AirDesc &air) {
    PeriodicRuns r;
    for (size_t c = 0; c < air.periodic.size();) {
        const size_t P = air.periodic[c].values.size();
        size_t c1 = c;
        while (c1 < air.periodic.size() && air.periodic[c1].values.size() == P) c1++;
        r.runs.push_back({c, c1, P, r.total});
        r.total += (c1 - c) * P;
        c = c1;
    }
    return r;
}
inline void fill_periodic_args(ConsArgs &A, const PeriodicRuns &pr, size_t K, size_t k) {
    A.nperiodic = pr.runs.empty() ? 0 : (unsigned)pr.runs.back().c1;
    A.ptab_coset_stride = K * pr.total;
    for (const PeriodicRun &r : pr.runs)
        for (size_t c = r.c0; c < r.c1; c++) { A.poff[c] = (unsigned)r.at(c, K, k); A.pmask[c] = (unsigned)(r.P - 1); }
}

// The part of ConsArgs that depends on the AIR and the evaluation domain only.  ce coset kc of the caller has the shift ce_shift[kc]
// and is read from block lde_block[kc] of the LDE buffer, in blocks of block_stride elements.
inline void fill_domain_args(ConsArgs &A, const AirDesc &air, const TransitionGroups &tg, const BoundaryGroups &bg, size_t n,
                             const std::vector<fe> &ce_shift, const std::vector<size_t> &lde_block, size_t block_stride) {
    using namespace f63;
    const unsigned logn = ilog2_host(n);
    const fe g = root_of_unity(logn), g_inv = inv(g);
    A.logn = logn; A.ncosets = (unsigned)ce_shift.size(); A.col_stride = n; A.width = air.width;
    A.g_last = f63::pow(g, n - 1);
    A.nconstraints = (unsigned)air.num_constraints(); A.ngroups = (unsigned)tg.adj.size();
    for (size_t i = 0; i < air.num_constraints(); i++) A.group[i] = tg.group_of[i];
    for (size_t gi = 0; gi < tg.adj.size(); gi++) A.adj_mod[gi] = tg.adj[gi] % n;
    A.nbgroups = (unsigned)bg.groups.size(); A.nassertions = (unsigned)air.assertions.size();
    for (size_t gi = 0; gi < bg.groups.size(); gi++) { A.b_adj_mod[gi] = bg.groups[gi].adj % n; A.b_steps[gi] = bg.groups[gi].num_steps; A.b_offset[gi] = bg.groups[gi].offset; }
    for (size_t kc = 0; kc < ce_shift.size(); kc++) {
        const fe s = ce_shift[kc];
        A.lde_coset_stride[kc] = (unsigned long long)(lde_block[kc] * block_stride);
        A.shift[kc] = s;
        A.zinv[kc] = inv(sub(f63::pow(s, n), ONE));
        for (size_t gi = 0; gi < tg.adj.size(); gi++) A.shift_adj[kc][gi] = f63::pow(s, tg.adj[gi]);
        for (size_t gi = 0; gi < bg.groups.size(); gi++) { A.b_shift_adj[kc][gi] = f63::pow(s, bg.groups[gi].adj); A.b_shift_steps[kc][gi] = f63::pow(s, bg.groups[gi].num_steps); }
    }
    // a sequence becomes its interpolating polynomial (fill_assertion_values), evaluated in-kernel at x * g^-first_step
    for (size_t i = 0; i < air.assertions.size(); i++) {
        const Assertion &s = air.assertions[i];
        A.a_col[i] = s.column; A.a_group[i] = bg.group_of[i];
        A.a_poly_len[i] = (unsigned)s.values.size();
        A.a_xoff[i] = s.first_step ? f63::pow(g_inv, s.first_step) : ONE;
    }
}

// the assertion values of one proof: the first value of each assertion, and the interpolants of the sequences appended to `polys`,
// whose first element sits at poly_base in the device table
inline void fill_assertion_values(ConsArgs &A, const AirDesc &air, size_t poly_base, std::vector<fe> &polys) {
    for (size_t i = 0; i < air.assertions.size(); i++) {
        const Assertion &s = air.assertions[i];
        A.a_value[i] = s.values[0];
        A.a_poly_off[i] = poly_base + polys.size();
        if (s.values.size() > 1) {
            const std::vector<fe> c = interpolate_host(s.values);
            polys.insert(polys.end(), c.begin(), c.end());
        }
    }
}

// the cross-coset step of the composition: column t = sum_k mat[t][k] * (interpolant on ce coset k, divided by its shift^m)
inline std::vector<fe> composition_matrix(size_t n, size_t ce) {
    using namespace f63;
    std::vector<fe> mat(ce * ce);
    const fe off_n_inv = inv(f63::pow(to_mont(GENERATOR), n)), ce_inv = inv(to_mont(ce)), w_ce_inv = inv(root_of_unity(ilog2_host(ce)));
    for (size_t t = 0; t < ce; t++)
        for (size_t k = 0; k < ce; k++) mat[t * ce + k] = mul(mul(f63::pow(off_n_inv, t), ce_inv), f63::pow(w_ce_inv, (k * t) % ce));
    return mat;
}

// the fold of a FRI layer of m points with a root table of 2^logW points; alpha is left to the caller
inline FoldArgs fold_args(size_t m, unsigned logW) {
    using namespace f63;
    const unsigned logm = ilog2_host(m);
    FoldArgs a{};
    a.offset_inv = inv(to_mont(GENERATOR));
    const fe w_inv = inv(root_of_unity(logm));
    a.zeta_inv = f63::pow(w_inv, m / 4); a.quarter = inv(to_mont(4));
    a.logm = logm; a.logW = logW;
    if (logm > logW) {
        if (logm - logW > 5) throw std::runtime_error("FRI layer too large for the root table");
        for (unsigned i = 0; i < (1u << (logm - logW)); i++) a.small[i] = f63::pow(w_inv, i);
    }
    return a;
}

// The base-field DEEP arguments: the three points (g generates the trace domain), the coefficient-weighted out-of-domain values and
// the shifts of the ncosets LDE cosets.  coef: the trace column coefficients as combine_polys takes them (w alphas, then w betas);
// comp_coef: one per composition column.
inline DeepArgs deep_args(fe z, fe g, const std::vector<fe> &ood_cur, const std::vector<fe> &ood_next, const std::vector<fe> &ood_comp,
                          const fe *coef, const fe *comp_coef, fe lambda, fe mu, const fe *shift, size_t ncosets) {
    using namespace f63;
    const size_t w = ood_cur.size();
    DeepArgs a{};
    a.z = z; a.zg = mul(z, g); a.zm = f63::pow(z, ood_comp.size());
    for (size_t c = 0; c < w; c++) { a.az = add(a.az, mul(coef[c], ood_cur[c])); a.bzg = add(a.bzg, mul(coef[w + c], ood_next[c])); }
    for (size_t r = 0; r < ood_comp.size(); r++) a.czm = add(a.czm, mul(comp_coef[r], ood_comp[r]));
    a.lambda = lambda; a.mu = mu; a.ncosets = (unsigned)ncosets;
    for (size_t k = 0; k < ncosets; k++) a.shift[k] = shift[k];
    return a;
}

// CSG_HOST_TRACE: host clock at the stage boundaries of one call (host_mark), printed to stderr -- where the time of a small proof
// goes: launches, round trips of the Fiat-Shamir transcript, host arithmetic
class HostTraceScope {
  public:
    explicit HostTraceScope(std::chrono::steady_clock::time_point t0) : trace_{t0, {}} { if (on()) g_host_trace = &trace_; }
    ~HostTraceScope() { if (on()) g_host_trace = nullptr; }
    HostTraceScope(const HostTraceScope &) = delete;
    HostTraceScope &operator=(const HostTraceScope &) = delete;
    static bool on() { static const bool enabled = getenv("CSG_HOST_TRACE") != nullptr; return enabled; }
    // a header line, then one line per mark
    __attribute__((format(printf, 2, 3))) void print(const char *header, ...) const {
        if (!on()) return;
        va_list ap;
        va_start(ap, header);
        vfprintf(stderr, header, ap);
        va_end(ap);
        double prev = 0;
        for (auto &m : trace_.marks) { fprintf(stderr, "  %-36s +%8.1f us  (at %8.1f)\n", m.first, m.second - prev, m.second); prev = m.second; }
    }

  private:
    HostTrace trace_;
};

}  // namespace csg
