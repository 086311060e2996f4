// Batch witness builders (many.cuh): the K traces of a csg_prove_many_device batch built on the device, [K][width][rows], so that
// neither the host nor PCIe carries a trace.  Rescue chains run on their own kernel (rescue_chains.cuh); signatures, Merkle updates
// and transfers run the single-proof kernels of witness_gen.cu over the K items of a batch, then one kernel regroups that K-item
// trace [width][K * rows] into one trace per proof.  The public inputs come from the host's side of the inputs (seeds, packed
// records) except the last rows of the Rescue chains.
#include <cstring>
#include <vector>

#include "../witness.cuh"
#include "many.cuh"
#include "rescue_chains.cuh"

namespace csg {
using namespace f63;

namespace {

// out[(k * w + c) * R + r] = in[c * K * R + k * R + r]; with bit_col0 / bit_col1 >= 0 row 1 of those columns is set to 1 in every
// proof (MerkleProver::build_trace, src/merkle/update/prover.rs:72-77: the K-item kernel sets them in its first item only)
__global__ void __launch_bounds__(256) regroup_items_kernel(const uint64_t *__restrict__ in, unsigned w, unsigned K, unsigned R, uint64_t *__restrict__ out,
                                                            int bit_col0, int bit_col1) {
    const unsigned kc = blockIdx.x, k = kc / w, c = kc % w;
    const uint64_t *src = in + (size_t)c * K * R + (size_t)k * R;
    uint64_t *dst = out + (size_t)kc * R;
    const bool bits = (int)c == bit_col0 || (int)c == bit_col1;
    for (unsigned r = threadIdx.x; r < R; r += blockDim.x) dst[r] = bits && r == 1 ? 1 : src[r];
}

void check_count(size_t count) {
    if (count == 0 || count > MANY_MAX_COUNT) throw ManyArgError("count must be in 1..1024");
}

}  // namespace

void many_build_rescue(ManyProver *m, Stream &st, const uint64_t *seeds, size_t count, size_t chain_length, uint64_t *traces_dev, uint64_t *pubs) {
    if (!seeds || !traces_dev || !pubs) throw ManyArgError("null argument");
    check_count(count);
    if (!chain_length || (chain_length & (chain_length - 1)) || 8 * chain_length > ((size_t)1 << MANY_MAX_LOG_TRACE))
        throw ManyArgError("chain_length must be a power of two of at most 8192 (traces of at most 2^16 rows)");
    check_device_buffer(traces_dev, "the trace buffer");
    ManyWitnessScratch &S = many_scratch(m);
    S.records.reserve(7 * count); S.last.reserve(7 * count);
    CSG_CUDA(cudaMemcpyAsync(S.records.p, seeds, 7 * count * sizeof(uint64_t), cudaMemcpyHostToDevice, st.s));
    const unsigned blocks = (unsigned)((count * RESCUE_LANES + RESCUE_CHAIN_THREADS - 1) / RESCUE_CHAIN_THREADS);
    CSG_LAUNCH(st, rescue_chains_kernel, blocks, RESCUE_CHAIN_THREADS, 0, S.records.p, (unsigned)count, (unsigned long long)(8 * chain_length), traces_dev, S.last.p);
    std::vector<uint64_t> last(7 * count);
    CSG_CUDA(cudaMemcpyAsync(last.data(), S.last.p, last.size() * sizeof(uint64_t), cudaMemcpyDeviceToHost, st.s));
    CSG_CUDA(cudaStreamSynchronize(st.s));
    // pub = seed[7] result[7] (benches/rescue.rs:136-141), as csg_build_trace_rescue reads them from rows 0 and n-1
    for (size_t k = 0; k < count; k++)
        for (int i = 0; i < 7; i++) { pubs[k * 14 + i] = seeds[k * 7 + i] % P; pubs[k * 14 + 7 + i] = last[k * 7 + i]; }
}

void many_build_items(ManyProver *m, Stream &st, int air_id, const void *batch, uint64_t *traces_dev, uint64_t *pubs) {
    if (!batch) throw ManyArgError("null batch");
    if (!traces_dev || !pubs) throw ManyArgError("null argument");
    const bool sig = air_id == CSG_AIR_SCHNORR;
    const csg_sig_batch *sb = static_cast<const csg_sig_batch *>(batch);
    const csg_tx_batch *tb = static_cast<const csg_tx_batch *>(batch);
    const size_t K = sig ? csg_sig_batch_size(sb) : csg_tx_batch_size(tb);
    check_count(K);
    const unsigned depth = sig ? 0 : csg_tx_batch_depth(tb);
    if (air_id == CSG_AIR_TRANSACTION && depth != 15) throw ManyArgError("the transaction AIR is built for tree depth 15");
    check_device_buffer(traces_dev, "the trace buffer");
    const unsigned R = air_id == CSG_AIR_TRANSACTION ? 1024 : 512, w = air_id == CSG_AIR_TRANSACTION ? 94 : sig ? 56 : 65;
    std::vector<uint64_t> rec(sig ? csg_sig_batch_pack(sb, nullptr) : csg_tx_batch_pack(tb, nullptr));
    if (sig) csg_sig_batch_pack(sb, rec.data());
    else csg_tx_batch_pack(tb, rec.data());

    ManyWitnessScratch &S = many_scratch(m);
    S.records.reserve(rec.size()); S.trace.reserve((size_t)K * w * R); S.finals.reserve(K * 48);
    CSG_CUDA(cudaMemcpyAsync(S.records.p, rec.data(), rec.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, st.s));
    if (sig) build_schnorr_trace(S.records.p, K, S.trace.p, S.finals.p, st);
    else if (air_id == CSG_AIR_MERKLE_UPDATE) build_merkle_update_trace(S.records.p, K, depth, S.trace.p, st);
    else build_transaction_trace(S.records.p, K, 15, S.trace.p, S.finals.p, st);
    const int b0 = air_id == CSG_AIR_MERKLE_UPDATE ? 14 : -1, b1 = air_id == CSG_AIR_MERKLE_UPDATE ? 43 : -1;
    CSG_LAUNCH(st, regroup_items_kernel, (unsigned)(K * w), 256, 0, (const uint64_t *)S.trace.p, w, (unsigned)K, R, traces_dev, b0, b1);

    // public inputs from the records (Montgomery words) while the kernels run
    if (sig) {   // message[28] Rx[6] s[4] (src/schnorr/air.rs:38-46); the message's slots in the record are those of witness.cuh
        for (size_t k = 0; k < K; k++) {
            const uint64_t *T = &rec[k * WIT_WORDS];
            uint64_t *p = pubs + 38 * k;
            for (int j = 0; j < 28; j++)
                p[j] = from_mont(j < 12 ? T[WIT_S_OLD + j] : j < 24 ? T[WIT_R_OLD + j - 12] : j == 24 ? T[WIT_DELTA] : j == 25 ? T[WIT_S_OLD + 13] : T[WIT_M26 + j - 26]);
            for (int j = 0; j < 6; j++) p[28 + j] = from_mont(T[WIT_RX + j]);
            for (int j = 0; j < 4; j++) p[34 + j] = T[WIT_S + j];
        }
    } else {     // (root before transfer k, root after it): the next record's root, the batch's final root after the last transfer
        uint64_t initial[7], final_root[7];
        csg_tx_batch_roots(tb, initial, final_root);
        for (size_t k = 0; k < K; k++)
            for (int i = 0; i < 7; i++) {
                pubs[k * 14 + i] = from_mont(rec[k * WIT_WORDS + WIT_ROOT + i]);
                pubs[k * 14 + 7 + i] = k + 1 < K ? from_mont(rec[(k + 1) * WIT_WORDS + WIT_ROOT + i]) : final_root[i];
            }
    }
    CSG_CUDA(cudaStreamSynchronize(st.s));
}

}  // namespace csg
