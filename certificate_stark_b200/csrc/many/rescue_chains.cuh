// K Rescue chains (RescueProver::build_trace, benches/rescue.rs:279-321) on the device, for csg_build_traces_many_rescue.
// A chain is one long dependent sequence: row i+1 is a round of row i.  The only parallelism inside a chain is the 14 state
// elements, so a chain runs on RESCUE_LANES = 16 lanes of a warp (two chains per warp, lanes 14 and 15 idle), one state element per
// lane: the two 14 x 14 MDS products exchange the state through shuffles and every lane runs the inverse S-box (a 62-bit
// exponentiation, the latency of a round) of its own element.  One thread per chain (rescue::apply_round, as the wit_* kernels
// run their chains) makes a thread run all 14 exponentiations one after the other; tools/microbench/rescue_chains.cu measures
// both mappings (DESIGN §3b).
#pragma once
#include "../dev.cuh"
#include "../rescue.cuh"

namespace csg {

constexpr unsigned RESCUE_LANES = 16, RESCUE_CHAIN_THREADS = 128;

// seeds[7k ..]: canonical words, reduced mod p here; trace + k*14*n: the column-major [14][n] trace of chain k (canonical);
// last[7k ..]: row n-1 of columns 0..6 of chain k (canonical)
__global__ void __launch_bounds__(RESCUE_CHAIN_THREADS) rescue_chains_kernel(const uint64_t *__restrict__ seeds, unsigned count, unsigned long long n,
                                                                              uint64_t *__restrict__ trace, uint64_t *__restrict__ last) {
    using namespace f63;
    const unsigned g = blockIdx.x * blockDim.x + threadIdx.x, chain = g / RESCUE_LANES, lane = g % RESCUE_LANES;
    const bool live = chain < count && lane < 14;   // every lane of the warp takes part in the shuffles
    const unsigned row_of = lane < 14 ? lane : 13;
    fe m[14], ark0[7], ark1[7];
#pragma unroll
    for (int j = 0; j < 14; j++) m[j] = CSG_TABLE(CSG_MDS)[row_of * 14 + j];
#pragma unroll
    for (int r = 0; r < 7; r++) { ark0[r] = CSG_TABLE(CSG_ARK)[r * 28 + row_of]; ark1[r] = CSG_TABLE(CSG_ARK)[r * 28 + 14 + row_of]; }
    fe s = live && lane < 7 ? to_mont(seeds[(size_t)chain * 7 + lane] % P) : 0;
    uint64_t *col = trace + ((size_t)chain * 14 + lane) * n;
    if (live) col[0] = from_mont(s);
    auto mds = [&](fe v) {
        acc128 acc;
#pragma unroll
        for (int j = 0; j < 14; j++) acc.mac(m[j], __shfl_sync(0xffffffffu, v, j, RESCUE_LANES));
        return acc.reduce();
    };
    for (unsigned long long c = 0; c < n / 8; c++) {
#pragma unroll
        for (int r = 0; r < 8; r++) {
            const unsigned long long row = c * 8 + r + 1;
            if (row == n) break;
            if (r < 7) {   // rescue::apply_round
                fe t = add(mds(rescue::cube(s)), ark0[r]);
                t = f63::pow(t, CSG_INV_ALPHA);   // qualified: the std::pow template is the better match for these arguments
                s = add(mds(t), ark1[r]);
            } else if (lane >= 7) s = 0;
            if (live) col[row] = from_mont(s);
        }
    }
    if (live && lane < 7) last[(size_t)chain * 7 + lane] = from_mont(s);
}

}  // namespace csg
