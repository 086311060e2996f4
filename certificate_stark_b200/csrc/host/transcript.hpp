// Host side of the protocol that stays sequential: the Fiat-Shamir public coin (winterfell RandomCoin), the
// little-endian byte writer proofs are serialised with (winterfell ByteWriter / StarkProof::to_bytes, reached from
// /root/reference/examples/state-transition.rs:96) and the shape of batch Merkle openings (MerkleTree::prove_batch +
// BatchMerkleProof::serialize_nodes).  The winterfell fork (Cargo.toml:20) is not vendored in the reference tree; these
// follow the published v0.3 behaviour and are byte-compared against the CPU oracle in tests/.
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <stdexcept>
#include <vector>

#include "../ext.cuh"
#include "../hash.cuh"

namespace csg {
using f63::fe;

class Bytes {
  public:
    std::vector<uint8_t> v;
    void put(const void *p, size_t n) { const uint8_t *b = (const uint8_t *)p; v.insert(v.end(), b, b + n); }
    void u8(uint8_t x) { v.push_back(x); }
    void u16(uint16_t x) { for (int i = 0; i < 2; i++) v.push_back((uint8_t)(x >> (8 * i))); }
    void u32(uint32_t x) { for (int i = 0; i < 4; i++) v.push_back((uint8_t)(x >> (8 * i))); }
    void u64(uint64_t x) { put(&x, 8); }
    void u64s(const uint64_t *x, size_t n) { put(x, 8 * n); }   // n little-endian words at once (the opened rows of a proof)
    static_assert(__BYTE_ORDER__ == __ORDER_LITTLE_ENDIAN__, "the serialiser writes host words as little-endian bytes");
    void element(fe m) { u64(f63::from_mont(m)); }   // BaseElement::write_into: canonical little-endian
};

class Coin {
  public:
    Coin(int hash_fn, const uint8_t *seed_bytes, size_t n) : hash_fn_(hash_fn) { hashes::hash_bytes(hash_fn_, seed_bytes, n, seed_); }
    void reseed(const uint8_t digest[32]) {
        uint8_t t[64];
        memcpy(t, seed_, 32); memcpy(t + 32, digest, 32);
        hashes::hash_bytes(hash_fn_, t, 64, seed_);
        counter_ = 0;
    }
    void reseed_with_int(uint64_t v) { uint8_t t[32]; merge_with_int(v, t); memcpy(seed_, t, 32); counter_ = 0; }
    // an element of the degree-d extension: the first 8*d bytes of one output as d canonical words, the whole output
    // rejected unless every word is below p (coin.draw::<E>())
    // For d = 3 only 1.7 % of the outputs pass (each word is below p with probability 0.26), about 60 hashes per draw and
    // ~30k per proof: the outputs H(seed || counter) are independent, so they are computed a block at a time on all host threads.
    f63::xe draw_x(int d) {
        for (int i = 0; i < 1000; i++) {
            counter_++;
            const uint8_t *t = d > 1 ? output(counter_) : nullptr;
            uint8_t t1[32];
            if (!t) { merge_with_int(counter_, t1); t = t1; }
            f63::xe r = f63::x_zero();
            bool ok = true;
            for (int j = 0; j < d && ok; j++) { uint64_t v; memcpy(&v, t + 8 * j, 8); if (v >= f63::P) ok = false; else r.c[j] = f63::to_mont(v); }
            if (ok) return r;
        }
        throw std::runtime_error("random coin failed to draw a field element");
    }
    std::vector<size_t> draw_integers(size_t count, size_t domain_size) {
        if (count >= domain_size) throw std::runtime_error("more query positions than domain points");
        std::vector<size_t> out;
        for (int i = 0; i < 1000 && out.size() < count; i++) {
            size_t v = (size_t)(next_u64() & (uint64_t)(domain_size - 1));
            if (std::find(out.begin(), out.end(), v) == out.end()) out.push_back(v);
        }
        if (out.size() != count) throw std::runtime_error("random coin failed to draw enough distinct integers");
        return out;
    }
    // proof of work: zeros counted from the least significant end of the first 8 digest bytes read little-endian
    unsigned check_leading_zeros(uint64_t nonce) const { uint8_t t[32]; merge_with_int(nonce, t); return tz(t); }
    unsigned leading_zeros() const { return tz(seed_); }

  private:
    int hash_fn_;
    uint8_t seed_[32];
    uint64_t counter_ = 0;
    // outputs for the counters block_first_ .. block_first_ + block_.size()/32 - 1 under the seed they were computed for
    std::vector<uint8_t> block_;
    uint64_t block_first_ = 0;
    uint8_t block_seed_[32];
    const uint8_t *output(uint64_t ctr) {
        const bool same_seed = !block_.empty() && memcmp(block_seed_, seed_, 32) == 0;
        if (!same_seed || ctr < block_first_ || ctr >= block_first_ + block_.size() / 32) {
            // a seed that serves one draw (a FRI layer's alpha) needs ~60 outputs, one that serves hundreds keeps asking: grow
            const size_t K = same_seed ? std::min<size_t>(4 * (block_.size() / 32), 2048) : 128;
            block_.resize(K * 32);
            block_first_ = ctr;
            memcpy(block_seed_, seed_, 32);
#pragma omp parallel for schedule(static)
            for (long k = 0; k < (long)K; k++) merge_with_int(ctr + (uint64_t)k, &block_[(size_t)k * 32]);
        }
        return &block_[(size_t)(ctr - block_first_) * 32];
    }
    void merge_with_int(uint64_t v, uint8_t out[32]) const {
        uint8_t t[40];
        memcpy(t, seed_, 32);
        for (int i = 0; i < 8; i++) t[32 + i] = (uint8_t)(v >> (8 * i));
        hashes::hash_bytes(hash_fn_, t, 40, out);
    }
    uint64_t next_u64() { uint8_t t[32]; counter_++; merge_with_int(counter_, t); uint64_t v; memcpy(&v, t, 8); return v; }
    static unsigned tz(const uint8_t *d) { uint64_t h; memcpy(&h, d, 8); return h ? (unsigned)__builtin_ctzll(h) : 64; }
};

// hash of a short vector of elements (OOD frames) on the host: H(canonical little-endian bytes)
inline void hash_elements_host(int hash_fn, const fe *e, size_t n, uint8_t out[32]) {
    std::vector<uint8_t> b(n * 8);
    for (size_t i = 0; i < n; i++) { uint64_t v = f63::from_mont(e[i]); memcpy(b.data() + 8 * i, &v, 8); }
    hashes::hash_bytes(hash_fn, b.data(), b.size(), out);
}

// The Fiat-Shamir schedule of Prover::prove, one method per step in protocol order.  Both provers and the verifier draw every
// challenge through it: a proof is only valid if all three replay the same schedule.  Challenges are elements of the degree-d
// extension (d = 1: the base field, in component 0).
class ProofTranscript {
  public:
    // seeded with the public inputs as little-endian words, then the serialised proof context (write_proof_context)
    ProofTranscript(int hash_fn, int d, const uint64_t *pub, size_t npub, const uint8_t *context, size_t context_len)
        : hash_fn_(hash_fn), d_(d), coin_(seeded(hash_fn, pub, npub, context, context_len)) {}

    // (alpha, beta) per transition constraint, then per assertion
    struct ConstraintCoefficients { std::vector<f63::xe> transition, boundary; };
    ConstraintCoefficients constraint_coefficients(const uint8_t trace_root[32], size_t nconstraints, size_t nassertions) {
        coin_.reseed(trace_root);
        std::vector<f63::xe> t = draw(2 * nconstraints);
        return {std::move(t), draw(2 * nassertions)};
    }
    // the out-of-domain point z
    f63::xe ood_point(const uint8_t comp_root[32]) { coin_.reseed(comp_root); return draw(); }
    // (alpha, beta) per trace column, one coefficient per composition column, lambda and mu.  The frame is given as flat component
    // arrays: cur and next hold w elements, comp ce elements, d components each.
    struct DeepCoefficients { std::vector<f63::xe> trace, comp; f63::xe lambda, mu; };
    DeepCoefficients deep_coefficients(const fe *cur, const fe *next, size_t w, const fe *comp, size_t ce) {
        uint8_t dg[32];
        hash_elements_host(hash_fn_, cur, w * d_, dg); coin_.reseed(dg);
        hash_elements_host(hash_fn_, next, w * d_, dg); coin_.reseed(dg);
        hash_elements_host(hash_fn_, comp, ce * d_, dg); coin_.reseed(dg);
        DeepCoefficients c;
        c.trace.resize(2 * w);
        for (size_t i = 0; i < w; i++) { c.trace[2 * i] = draw(); c.trace[2 * i + 1] = draw(); (void)draw(); }   // a third per column, unused
        c.comp = draw(ce);
        c.lambda = draw(); c.mu = draw();
        return c;
    }
    // the folding challenge of a FRI layer (also drawn for the remainder layer, which is not folded)
    f63::xe fri_alpha(const uint8_t layer_root[32]) { coin_.reseed(layer_root); return draw(); }
    // proof of work: the first nonce from 1 that reaches `bits` zeros (Coin::check_leading_zeros); the coin is reseeded with it
    uint64_t grind(unsigned bits) {
        uint64_t nonce = 1;
        while (coin_.check_leading_zeros(nonce) < bits) nonce++;
        coin_.reseed_with_int(nonce);
        return nonce;
    }
    // the verifier's side of grind(): reseeds with the proof's nonce and checks its work
    bool accept_nonce(uint64_t nonce, unsigned bits) { coin_.reseed_with_int(nonce); return coin_.leading_zeros() >= bits; }
    std::vector<size_t> query_positions(size_t count, size_t domain_size) { return coin_.draw_integers(count, domain_size); }

  private:
    int hash_fn_, d_;
    Coin coin_;
    static Coin seeded(int hash_fn, const uint64_t *pub, size_t npub, const uint8_t *context, size_t context_len) {
        Bytes seed;
        seed.u64s(pub, npub);
        seed.put(context, context_len);
        return Coin(hash_fn, seed.v.data(), seed.v.size());
    }
    f63::xe draw() { return coin_.draw_x(d_); }
    std::vector<f63::xe> draw(size_t count) {
        std::vector<f63::xe> v(count);
        for (f63::xe &e : v) e = draw();
        return v;
    }
};

// Which tree nodes a batch opening of `positions` carries, grouped the way BatchMerkleProof stores them: one vector
// per pair of adjacent leaves touched, siblings appended level by level.  Node numbering: root 1, leaves at nleaves+j.
inline std::vector<std::vector<uint32_t>> batch_opening_nodes(size_t nleaves, const std::vector<size_t> &positions) {
    std::vector<size_t> idx;
    for (size_t p : positions) idx.push_back(p & ~(size_t)1);
    std::sort(idx.begin(), idx.end());
    idx.erase(std::unique(idx.begin(), idx.end()), idx.end());
    std::vector<std::vector<uint32_t>> slots(idx.size());
    std::vector<size_t> cur, nxt;
    for (size_t i = 0; i < idx.size(); i++) {
        for (size_t j = idx[i]; j < idx[i] + 2; j++)
            if (std::find(positions.begin(), positions.end(), j) == positions.end()) slots[i].push_back((uint32_t)(nleaves + j));
        cur.push_back((idx[i] + nleaves) >> 1);
    }
    unsigned depth = 0;
    while (((size_t)1 << depth) < nleaves) depth++;
    for (unsigned d = 1; d < depth; d++) {
        nxt.clear();
        for (size_t i = 0; i < cur.size(); i++) {
            size_t sib = cur[i] ^ 1;
            if (i + 1 < cur.size() && cur[i + 1] == sib) i++;
            else slots[i].push_back((uint32_t)sib);
            nxt.push_back(sib >> 1);
        }
        cur.swap(nxt);
    }
    return slots;
}

}  // namespace csg
