// The host driver of csg_validate_* (validate.cuh): uploads, the device pass of kernels.cu, and the localisation of the first
// failing steps on the host, where every constraint slot of a flagged step is evaluated on its own with the host build of airs.cuh.
#include <algorithm>
#include <cstring>
#include <random>
#include <stdexcept>

#include "../host/stage_args.hpp"
#include "validate.cuh"

namespace csg {
using namespace f63;

namespace {

// the asserted cells of an AIR in report order (ascending by step, then column), with the index of their assertion and value
struct Cell { uint32_t col, step, a, j; };
std::vector<Cell> asserted_cells(const AirDesc &air) {
    std::vector<Cell> cells;
    for (size_t a = 0; a < air.assertions.size(); a++) {
        const Assertion &s = air.assertions[a];
        const size_t count = s.stride ? air.trace_len / s.stride : 1;
        for (size_t j = 0; j < count; j++)
            cells.push_back(Cell{s.column, (uint32_t)(s.first_step + j * s.stride), (uint32_t)a, (uint32_t)(s.values.size() > 1 ? j : 0)});
    }
    std::sort(cells.begin(), cells.end(), [](const Cell &x, const Cell &y) { return x.step != y.step ? x.step < y.step : x.col < y.col; });
    return cells;
}

fe random_nonzero(std::mt19937_64 &rng) {
    for (;;) { const uint64_t v = rng() % P; if (v) return to_mont(v); }
}

}  // namespace

class Validator {
  public:
    void run(Stream &st, int air_id, const std::vector<AirDesc> &airs, const uint64_t *host, const uint64_t *dev, int repr, size_t n, csg_trace_report *out);
    size_t held() const {
        return (d_mont.n + d_ptab.n + d_part.n + d_val.n) * 8 + d_flags.n + d_cflags.n + (d_col.n + d_step.n) * 4 + d_counts.n * 8 + d_args.n * sizeof(ValArgs);
    }

  private:
    DBuf<fe> d_mont, d_ptab, d_part, d_val;
    DBuf<uint8_t> d_flags, d_cflags;
    DBuf<uint32_t> d_col, d_step;
    DBuf<unsigned long long> d_counts;
    DBuf<ValArgs> d_args;
    std::mt19937_64 rng{std::random_device{}()};
};

Validator *validator_new() { return new Validator(); }
void validator_delete(Validator *v) { delete v; }
size_t validator_held(const Validator *v) { return v ? v->held() : 0; }
void validate_traces(Validator *v, Stream &st, int air_id, const std::vector<AirDesc> &airs, const uint64_t *host, const uint64_t *dev, int repr,
                     size_t n, csg_trace_report *out) {
    v->run(st, air_id, airs, host, dev, repr, n, out);
}

// a host trace goes up into the Montgomery buffer and is converted in place
size_t validate_footprint(int air_id, size_t K, size_t w, size_t n, size_t ptotal, size_t ncells) {
    return 8 * (K * w * n + K * ptotal + 2 * validate_items(air_id) * K * n + K * ncells) + K * n + K * ncells + 8 * ncells + 16 * K + sizeof(ValArgs);
}

std::vector<fe> transition_values(const AirDesc &air, const TransitionGroups &tg, size_t step, const std::vector<fe> &cur, const std::vector<fe> &next) {
    const size_t nc = air.num_constraints();
    std::vector<fe> pv(air.periodic.size());
    for (size_t c = 0; c < pv.size(); c++) pv[c] = air.periodic[c].values[step % air.periodic[c].values.size()];
    const std::vector<fe> beta(nc, 0), xp(std::max<size_t>(tg.adj.size(), 1), 0);
    std::vector<fe> out(nc);
#pragma omp parallel for schedule(dynamic) if (nc >= 16)
    for (long s = 0; s < (long)nc; s++) {
        std::vector<fe> alpha(nc, 0);
        alpha[s] = ONE;
        out[s] = eval_merged_any(air.id, air, tg, cur, next, pv, alpha, beta, xp);
    }
    return out;
}

void Validator::run(Stream &st, int air_id, const std::vector<AirDesc> &airs, const uint64_t *host, const uint64_t *dev, int repr, size_t n,
                    csg_trace_report *out) {
    const size_t K = airs.size();
    const AirDesc &air = airs[0];
    const size_t w = air.width, items = validate_items(air_id);
    const TransitionGroups tg = transition_groups(air);
    for (size_t k = 0; k < K; k++) memset(&out[k], 0, sizeof out[k]);

    // ---- arguments: the periodic layout, the two random combinations; one periodic table when every trace has the same columns
    ValArgs h;
    memset(&h, 0, sizeof h);
    h.logn = ilog2(n); h.width = (unsigned)w;
    const PeriodicRuns pr = periodic_runs(air);
    h.nperiodic = (unsigned)air.periodic.size();
    for (const PeriodicRun &r : pr.runs)
        for (size_t c = r.c0; c < r.c1; c++) { h.poff[c] = (unsigned)r.at(c, 1, 0); h.pmask[c] = (unsigned)(r.P - 1); }
    bool shared = true;
    for (size_t k = 1; k < K && shared; k++)
        for (size_t c = 0; c < air.periodic.size() && shared; c++) shared = airs[k].periodic[c].values == air.periodic[c].values;
    const size_t ntab = shared ? 1 : K;
    h.ptab_stride = shared ? 0 : pr.total;
    for (int j = 0; j < 2; j++)
        for (size_t s = 0; s < air.num_constraints(); s++) h.alpha[j][s] = random_nonzero(rng);
    std::vector<fe> ptab(std::max<size_t>(ntab * pr.total, 1));
#pragma omp parallel for if (ntab >= 32)
    for (long k = 0; k < (long)ntab; k++)
        for (const PeriodicRun &r : pr.runs)
            for (size_t c = r.c0; c < r.c1; c++) memcpy(&ptab[k * pr.total + r.at(c, 1, 0)], airs[k].periodic[c].values.data(), r.P * sizeof(fe));

    // ---- asserted cells: positions shared, values per trace
    const std::vector<Cell> cells = asserted_cells(air);
    const size_t nce = cells.size();
    std::vector<uint32_t> col(std::max<size_t>(nce, 1)), step(std::max<size_t>(nce, 1));
    for (size_t c = 0; c < nce; c++) { col[c] = cells[c].col; step[c] = cells[c].step; }
    std::vector<fe> val(std::max<size_t>(K * nce, 1));
#pragma omp parallel for if (K >= 32)
    for (long k = 0; k < (long)K; k++)
        for (size_t c = 0; c < nce; c++) val[k * nce + c] = airs[k].assertions[cells[c].a].values[cells[c].j];

    // ---- device pass
    d_mont.reserve(K * w * n); d_ptab.reserve(ptab.size()); d_part.reserve(std::max<size_t>(2 * items * K * n, 1));
    d_flags.reserve(K * n); d_cflags.reserve(std::max<size_t>(K * nce, 1)); d_col.reserve(col.size()); d_step.reserve(step.size());
    d_val.reserve(val.size()); d_counts.reserve(2 * K); d_args.reserve(1);
    CSG_CUDA(cudaMemcpyAsync(d_args.p, &h, sizeof h, cudaMemcpyHostToDevice, st.s));
    CSG_CUDA(cudaMemcpyAsync(d_ptab.p, ptab.data(), ptab.size() * sizeof(fe), cudaMemcpyHostToDevice, st.s));
    CSG_CUDA(cudaMemcpyAsync(d_col.p, col.data(), col.size() * 4, cudaMemcpyHostToDevice, st.s));
    CSG_CUDA(cudaMemcpyAsync(d_step.p, step.data(), step.size() * 4, cudaMemcpyHostToDevice, st.s));
    CSG_CUDA(cudaMemcpyAsync(d_val.p, val.data(), val.size() * sizeof(fe), cudaMemcpyHostToDevice, st.s));
    CSG_CUDA(cudaMemsetAsync(d_counts.p, 0, 2 * K * sizeof(unsigned long long), st.s));
    if (host) {
        CSG_CUDA(cudaMemcpyAsync(d_mont.p, host, K * w * n * sizeof(uint64_t), cudaMemcpyHostToDevice, st.s));
        validate_to_mont(d_mont.p, d_mont.p, K * w * n, repr, st);
    } else validate_to_mont(dev, d_mont.p, K * w * n, repr, st);
    validate_rows(air_id, d_args.p, h, K, d_mont.p, d_ptab.p, d_part.p, d_flags.p, d_counts.p, st);
    validate_cells(K, d_mont.p, (unsigned)w, n, d_col.p, d_step.p, d_val.p, nce, d_cflags.p, d_counts.p + K, st);
    std::vector<unsigned long long> counts(2 * K);
    CSG_CUDA(cudaMemcpyAsync(counts.data(), d_counts.p, counts.size() * 8, cudaMemcpyDeviceToHost, st.s));
    CSG_CUDA(cudaStreamSynchronize(st.s));

    // ---- the flags of the traces that fail
    std::vector<size_t> bad_rows, bad_cells;
    for (size_t k = 0; k < K; k++) {
        out[k].failed_steps = counts[k]; out[k].failed_cells = counts[K + k];
        if (counts[k]) bad_rows.push_back(k);
        if (counts[K + k]) bad_cells.push_back(k);
    }
    if (bad_rows.empty() && bad_cells.empty()) return;
    std::vector<uint8_t> flags(bad_rows.size() * n), cflags(bad_cells.size() * nce);
    for (size_t i = 0; i < bad_rows.size(); i++)
        CSG_CUDA(cudaMemcpyAsync(&flags[i * n], d_flags.p + bad_rows[i] * n, n, cudaMemcpyDeviceToHost, st.s));
    for (size_t i = 0; i < bad_cells.size(); i++)
        CSG_CUDA(cudaMemcpyAsync(&cflags[i * nce], d_cflags.p + bad_cells[i] * nce, nce, cudaMemcpyDeviceToHost, st.s));
    // rows s and s+1 of the first CSG_REPORT_CAP failing steps of each failing trace: each step holds at least one failing pair
    std::vector<std::vector<uint32_t>> steps(bad_rows.size());
    std::vector<std::vector<fe>> frames(bad_rows.size());
    CSG_CUDA(cudaStreamSynchronize(st.s));
    for (size_t i = 0; i < bad_rows.size(); i++) {
        for (size_t s = 0; s + 1 < n && steps[i].size() < CSG_REPORT_CAP; s++) if (flags[i * n + s]) steps[i].push_back((uint32_t)s);
        frames[i].resize(steps[i].size() * 2 * w);
        const fe *T = d_mont.p + bad_rows[i] * w * n;
        for (size_t j = 0; j < steps[i].size(); j++)   // [column][2] words: (row s, row s+1) of each column are adjacent
            CSG_CUDA(cudaMemcpy2DAsync(&frames[i][j * 2 * w], 2 * sizeof(fe), T + steps[i][j], n * sizeof(fe), 2 * sizeof(fe), w, cudaMemcpyDeviceToHost, st.s));
    }
    CSG_CUDA(cudaStreamSynchronize(st.s));

    for (size_t i = 0; i < bad_cells.size(); i++) {
        csg_trace_report &r = out[bad_cells[i]];
        for (size_t c = 0; c < nce && r.num_boundary < CSG_REPORT_CAP; c++)
            if (cflags[i * nce + c]) { r.boundary[r.num_boundary][0] = cells[c].col; r.boundary[r.num_boundary][1] = cells[c].step; r.num_boundary++; }
    }
    for (size_t i = 0; i < bad_rows.size(); i++) {
        csg_trace_report &r = out[bad_rows[i]];
        const AirDesc &a = airs[bad_rows[i]];
        std::vector<fe> cur(w), next(w);
        for (size_t j = 0; j < steps[i].size() && r.num_transition < CSG_REPORT_CAP; j++) {
            for (size_t c = 0; c < w; c++) { cur[c] = frames[i][(j * w + c) * 2]; next[c] = frames[i][(j * w + c) * 2 + 1]; }
            const std::vector<fe> v = transition_values(a, tg, steps[i][j], cur, next);
            bool any = false;
            for (size_t s = 0; s < v.size() && r.num_transition < CSG_REPORT_CAP; s++)
                if (v[s]) { r.transition[r.num_transition][0] = steps[i][j]; r.transition[r.num_transition][1] = (uint32_t)s; r.num_transition++; any = true; }
            if (!any) throw std::runtime_error("internal error: step " + std::to_string(steps[i][j]) + " failed on the device and no constraint fails on the host");
        }
    }
}

}  // namespace csg

extern "C" int csg_debug_transition_at(int air_id, size_t trace_len, const uint64_t *pub, size_t npub, size_t step, const uint64_t *cur,
                                       const uint64_t *next, uint64_t *out) {
    using namespace csg;
    if (!pub || !cur || !next || !out) return CSG_ERR_ARG;
    try {
        const AirDesc air = make_air(air_id, trace_len, pub, npub);
        if (step >= trace_len) return CSG_ERR_ARG;
        std::vector<fe> c(air.width), x(air.width);
        for (size_t i = 0; i < air.width; i++) { c[i] = to_mont(cur[i] % P); x[i] = to_mont(next[i] % P); }
        const std::vector<fe> v = transition_values(air, transition_groups(air), step, c, x);
        for (size_t s = 0; s < v.size(); s++) out[s] = from_mont(v[s]);
        return CSG_OK;
    } catch (const std::invalid_argument &) { return CSG_ERR_ARG; }
    catch (const std::exception &) { return CSG_ERR_UNSUPPORTED; }
}
