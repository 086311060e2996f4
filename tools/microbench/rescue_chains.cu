// Thread mapping of the batch Rescue witness builder (certificate_stark_b200/csrc/many/rescue_chains.cuh), measured: the
// library's 16 lanes per chain against one thread per chain running rescue::apply_round, for K chains of a given length.
// Both must write the same trace.  Prints one JSON object per (K, chain length); profiles/r4_rescue_chain_mapping.json holds a run.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o rescue_chains rescue_chains.cu && ./rescue_chains
#include <cstdio>
#include <cstring>
#include <vector>

#include "../../certificate_stark_b200/csrc/many/rescue_chains.cuh"

using namespace csg;

__global__ void __launch_bounds__(64) one_thread_per_chain_kernel(const uint64_t *seeds, unsigned count, unsigned long long n, uint64_t *trace, uint64_t *last) {
    using namespace f63;
    const unsigned k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    fe st[14];
    for (int i = 0; i < 14; i++) st[i] = i < 7 ? to_mont(seeds[(size_t)k * 7 + i] % P) : 0;
    uint64_t *t = trace + (size_t)k * 14 * n;
    for (int i = 0; i < 14; i++) t[i * n] = from_mont(st[i]);
    for (unsigned long long step = 0; step + 1 < n; step++) {
        if (step % 8 < 7) rescue::apply_round(st, step);
        else for (int i = 7; i < 14; i++) st[i] = 0;
        for (int i = 0; i < 14; i++) t[i * n + step + 1] = from_mont(st[i]);
    }
    for (int i = 0; i < 7; i++) last[(size_t)k * 7 + i] = from_mont(st[i]);
}

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { fprintf(stderr, "%s: %s\n", #x, cudaGetErrorString(e)); return 1; } } while (0)

int main() {
    const unsigned counts[] = {1, 16, 256, 1024};
    const unsigned long long lengths[] = {128, 1024, 8192};
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b));
    for (unsigned long long len : lengths)
        for (unsigned K : counts) {
            const unsigned long long n = 8 * len;
            if (K * 14ull * n * 8 > (8ull << 30)) continue;   // 1024 chains of 8192: 7.5 GB each way, skipped
            std::vector<uint64_t> seeds(7 * K);
            for (size_t i = 0; i < seeds.size(); i++) seeds[i] = 0x9e3779b97f4a7c15ull * (i + 1);
            uint64_t *d_seeds, *d_t1, *d_t2, *d_l1, *d_l2;
            const size_t words = (size_t)K * 14 * n;
            CK(cudaMalloc(&d_seeds, seeds.size() * 8)); CK(cudaMalloc(&d_t1, words * 8)); CK(cudaMalloc(&d_t2, words * 8));
            CK(cudaMalloc(&d_l1, K * 56)); CK(cudaMalloc(&d_l2, K * 56));
            CK(cudaMemcpy(d_seeds, seeds.data(), seeds.size() * 8, cudaMemcpyHostToDevice));
            float ms[2] = {0, 0};
            const int reps = len >= 8192 ? 1 : 3;
            for (int v = 0; v < 2; v++) {
                for (int rep = -1; rep < reps; rep++) {   // rep -1: warm-up
                    CK(cudaEventRecord(a));
                    if (v == 0) rescue_chains_kernel<<<(K * RESCUE_LANES + RESCUE_CHAIN_THREADS - 1) / RESCUE_CHAIN_THREADS, RESCUE_CHAIN_THREADS>>>(d_seeds, K, n, d_t1, d_l1);
                    else one_thread_per_chain_kernel<<<(K + 63) / 64, 64>>>(d_seeds, K, n, d_t2, d_l2);
                    CK(cudaEventRecord(b));
                    CK(cudaEventSynchronize(b));
                    float t = 0;
                    CK(cudaEventElapsedTime(&t, a, b));
                    if (rep >= 0) ms[v] += t / reps;
                }
            }
            std::vector<uint64_t> h1(words), h2(words);
            CK(cudaMemcpy(h1.data(), d_t1, words * 8, cudaMemcpyDeviceToHost));
            CK(cudaMemcpy(h2.data(), d_t2, words * 8, cudaMemcpyDeviceToHost));
            const bool same = memcmp(h1.data(), h2.data(), words * 8) == 0;
            printf("{\"count\": %u, \"chain_length\": %llu, \"rows\": %llu, \"lanes16_ms\": %.4f, \"one_thread_ms\": %.4f, \"same_trace\": %s}\n", K, len, n,
                   ms[0], ms[1], same ? "true" : "false");
            fflush(stdout);
            cudaFree(d_seeds); cudaFree(d_t1); cudaFree(d_t2); cudaFree(d_l1); cudaFree(d_l2);
            if (!same) return 2;
        }
    return 0;
}
