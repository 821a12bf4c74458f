// The device index stream of RolloutBuffer.get (mr_device_permutations): key schedule and the keyed bijection, shared by
// the kernels of ppo.cu and -- __host__ __device__ -- by the host build of tests/host/perm_host.cu, which checks them
// against the numpy restatement (tests/perm_ref.py) without a GPU.
#pragma once

#include "common.cuh"

namespace mr {

// Device-side index stream for RolloutBuffer.get when the bit-for-bit numpy stream is not asked for:
// out[i] = P(i), P a keyed bijection of [0, n) -- a 6-round Feistel network over the enclosing
// power-of-two domain (split into two halves of bits / 2 and bits - bits / 2 bits, swapped every
// round; round function = keyed 32-bit avalanche hash), cycle-walked back into range (at most 2 trips
// on average).  Every index is one thread's private computation: no sort, no atomics, one 10 MB store
// for an epoch of 1.2 M samples.  Round 1's four multiply-xorshift rounds were a narrow family with
// weak low bits (modulo 2^k a product's low bits depend only on the operands' low bits); a Feistel
// network with a strong round function has no such structure -- tests/test_device_perm_gpu.py holds it
// to chi-square tests on positions x values, successive pairs and minibatch composition.
struct PermKey {
    uint32_t key[6];
    int bits;
};
__host__ __device__ __forceinline__ uint32_t perm_round(uint32_t x, uint32_t k) {
    x ^= k;
    x *= 0x9E3779B1u;   // lowbias32-style avalanche: every output bit depends on every input bit
    x ^= x >> 16;
    x *= 0x85EBCA6Bu;
    x ^= x >> 13;
    x *= 0xC2B2AE35u;
    x ^= x >> 16;
    return x;
}
__host__ __device__ __forceinline__ uint32_t perm_feistel(uint32_t x, const PermKey& K) {
    const int lb = K.bits >> 1, rb = K.bits - lb;          // left half: high lb bits, right half: low rb bits
    uint32_t L = x >> rb, R = x & ((1u << rb) - 1u);
    int wl = lb, wr = rb;                                   // widths travel with the halves
#pragma unroll
    for (int r = 0; r < 6; ++r) {
        const uint32_t f = perm_round(R, K.key[r]) & ((1u << wl) - 1u);
        const uint32_t nl = R, nr = L ^ f;
        L = nl; R = nr;
        const int t = wl; wl = wr; wr = t;
    }
    return (L << wr) | R;   // six rounds: an even number of swaps, the halves are back at (lb, rb)
}

// the walk back into [0, n): at most 2 trips on average
__host__ __device__ __forceinline__ uint32_t perm_index(uint32_t i, int64_t n, const PermKey& K) {
    uint32_t x = i;
    do { x = perm_feistel(x, K); } while ((int64_t)x >= n);
    return x;
}

inline PermKey make_perm_key(uint64_t seed, uint64_t stream_id, int64_t n) {
    PermKey K;
    K.bits = 2;   // both Feistel halves need at least one bit
    while ((int64_t(1) << K.bits) < n) ++K.bits;
    uint64_t x = seed ^ (stream_id * 0xD1342543DE82EF95ull + 0x2545F4914F6CDD1Dull);
    for (int r = 0; r < 6; r += 2) {   // splitmix64 key schedule: two round keys per output
        uint64_t z = (x += 0x9E3779B97F4A7C15ull);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        z ^= z >> 31;
        K.key[r] = (uint32_t)z;
        K.key[r + 1] = (uint32_t)(z >> 32);
    }
    return K;
}

}  // namespace mr
