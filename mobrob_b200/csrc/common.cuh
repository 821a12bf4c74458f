// Shared helpers for libmobrob_b200: error reporting, launch accounting, and the
// device-side restatements of the reference's random streams.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/mobrob_b200.h"

namespace mr {

// Explicitly rounded fp64 operations and the 64 x 64 -> high 64 multiply: the device intrinsics, and plain IEEE
// operations in the HOST builds of the __host__ __device__ routines (tests/host/*.cu; x86-64 without -mfma does not
// contract a product and a sum).
namespace rn {
__host__ __device__ __forceinline__ double add(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
__host__ __device__ __forceinline__ double sub(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}
__host__ __device__ __forceinline__ double mul(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
__host__ __device__ __forceinline__ double root(double a) {
#ifdef __CUDA_ARCH__
    return __dsqrt_rn(a);
#else
    return sqrt(a);
#endif
}
__host__ __device__ __forceinline__ uint64_t mulhi(uint64_t a, uint64_t b) {
#ifdef __CUDA_ARCH__
    return __umul64hi(a, b);
#else
    return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}
}  // namespace rn

void set_error(const char* fmt, ...);
void count_launch(uint64_t n = 1);

#define MR_CUDA(expr)                                                                   \
    do {                                                                                \
        cudaError_t _e = (expr);                                                        \
        if (_e != cudaSuccess) {                                                        \
            mr::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                          __LINE__);                                                    \
            return MR_ERR_CUDA;                                                         \
        }                                                                               \
    } while (0)

#define MR_CHECK_LAUNCH()                                                               \
    do {                                                                                \
        mr::count_launch();                                                             \
        cudaError_t _e = cudaGetLastError();                                            \
        if (_e != cudaSuccess) {                                                        \
            mr::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e),   \
                          __FILE__, __LINE__);                                          \
            return MR_ERR_CUDA;                                                         \
        }                                                                               \
    } while (0)

#define MR_REQUIRE(cond, msg)                                                           \
    do {                                                                                \
        if (!(cond)) {                                                                  \
            mr::set_error("%s (%s:%d)", msg, __FILE__, __LINE__);                       \
            return MR_ERR_ARG;                                                          \
        }                                                                               \
    } while (0)

static inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// Function attributes (dynamic shared-memory opt-in) and SM counts are per DEVICE, and one process
// may drive several devices through this ABI (mr_env_create / mr_xchg_create take a device index):
// one-time setup is keyed by the current device, never by a process-wide flag.
constexpr int MR_MAX_DEVICES = 64;
struct OncePerDevice {
    bool done[MR_MAX_DEVICES] = {};
    // true the first time it is asked about the current device (dev receives its index)
    bool first(int* dev_out = nullptr) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MR_MAX_DEVICES) dev = 0;
        if (dev_out) *dev_out = dev;
        if (done[dev]) return false;
        done[dev] = true;
        return true;
    }
};
static inline int sm_count() {
    static int sms[MR_MAX_DEVICES] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MR_MAX_DEVICES) return 148;
    if (!sms[dev]) cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev);
    return sms[dev] ? sms[dev] : 148;
}
// entry points that must run on a handle's device switch to it for the call only
struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) cudaSetDevice(dev); else prev = -1;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// ---------------------------------------------------------------------------------------
// PCG64 (numpy's default BitGenerator) -- gymnasium Box.sample draws from
// Generator(PCG64(SeedSequence(seed))).uniform(low, high)  [GYM 0.28.1; call sites
// src/mobrob/envs/wrapper.py:126,191].  128-bit LCG, XSL-RR output, step-then-output.
struct Pcg64 {
    uint64_t hi, lo, inc_hi, inc_lo;

    __host__ __device__ __forceinline__ uint64_t next64() {
        const uint64_t MH = 0x2360ED051FC65DA4ull, ML = 0x4385DF649FCCF645ull;
        uint64_t nlo = lo * ML;
        uint64_t nhi = rn::mulhi(lo, ML) + hi * ML + lo * MH;
        uint64_t slo = nlo + inc_lo;
        uint64_t carry = slo < nlo ? 1ull : 0ull;
        hi = nhi + inc_hi + carry;
        lo = slo;
        uint64_t x = hi ^ lo;
        unsigned rot = (unsigned)(hi >> 58);
        return (x >> rot) | (x << ((64u - rot) & 63u));
    }
    __host__ __device__ __forceinline__ double next_double() {
        return (double)(next64() >> 11) * (1.0 / 9007199254740992.0);
    }
    // Generator.uniform(low, high): low + (high - low) * u, no contraction.
    __host__ __device__ __forceinline__ double uniform(double low, double high) {
        return rn::add(low, rn::mul(rn::sub(high, low), next_double()));
    }
};

// ---------------------------------------------------------------------------------------
// MT19937 as used by np.random.RandomState(seed) -- Engine.reset draws the start heading
// from a freshly seeded RandomState (engine.py:1002-1003, 633-667, 728-729).  Only the first
// 227 output words are reachable here (enough for 55 rejected goal placements; each
// rejection has probability ~0.19), so the twist only ever reads the seeding recurrence.
struct MtHead {
    uint32_t a, a1, b;
    int j;
    __host__ __device__ explicit MtHead(uint32_t seed) {
        a = seed;
        a1 = 1812433253u * (a ^ (a >> 30)) + 1u;
        uint32_t x = a1;
        for (uint32_t p = 2; p <= 397; ++p) x = 1812433253u * (x ^ (x >> 30)) + p;
        b = x;
        j = 0;
    }
    __host__ __device__ uint32_t next32() {
        uint32_t y = (a & 0x80000000u) | (a1 & 0x7fffffffu);
        uint32_t v = b ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
        a = a1;
        a1 = 1812433253u * (a1 ^ (a1 >> 30)) + (uint32_t)(j + 2);
        b = 1812433253u * (b ^ (b >> 30)) + (uint32_t)(j + 398);
        ++j;
        v ^= v >> 11;
        v ^= (v << 7) & 0x9d2c5680u;
        v ^= (v << 15) & 0xefc60000u;
        v ^= v >> 18;
        return v;
    }
    __host__ __device__ double next_double() {
        uint32_t x = next32() >> 5, y = next32() >> 6;
        return ((double)x * 67108864.0 + (double)y) / 9007199254740992.0;
    }
    __host__ __device__ double uniform(double low, double high) {
        return rn::add(low, rn::mul(rn::sub(high, low), next_double()));
    }
};

// The same generator with its whole 624-word state, for any number of draws (hazard_layout).  Word k of each round is
// twisted when it is drawn, from mt[k + 1] of the previous round and mt[k + 397] of whichever round wrote it last --
// what the reference's block twist computes.  2.5 KB: local memory, for the full resets of hazard envs only.
struct Mt19937 {
    uint32_t mt[624];
    int k;
    __host__ __device__ explicit Mt19937(uint32_t seed) {
        mt[0] = seed;
        for (int j = 1; j < 624; ++j) mt[j] = 1812433253u * (mt[j - 1] ^ (mt[j - 1] >> 30)) + (uint32_t)j;
        k = 0;
    }
    __host__ __device__ uint32_t next32() {
        const int k1 = k + 1 == 624 ? 0 : k + 1, km = k < 227 ? k + 397 : k - 227;
        const uint32_t y = (mt[k] & 0x80000000u) | (mt[k1] & 0x7fffffffu);
        uint32_t v = mt[km] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
        mt[k] = v;
        k = k1;
        v ^= v >> 11;
        v ^= (v << 7) & 0x9d2c5680u;
        v ^= (v << 15) & 0xefc60000u;
        v ^= v >> 18;
        return v;
    }
    __host__ __device__ double next_double() {
        uint32_t x = next32() >> 5, y = next32() >> 6;
        return ((double)x * 67108864.0 + (double)y) / 9007199254740992.0;
    }
    __host__ __device__ double uniform(double low, double high) {
        return rn::add(low, rn::mul(rn::sub(high, low), next_double()));
    }
};

// Engine.reset -> build_layout -> build_world_config: the heading is the first uniform after
// the robot xy pair and the accepted goal xy pair.
__host__ __device__ inline double engine_heading(uint32_t engine_seed) {
    MtHead rs(engine_seed);
    const double lo = -2 + 0.4, hi = 2 - 0.4;  // constrain_placement(extents, keepout)
    const double keep = 0.4 + 0.0 + 0.4;       // robot_keepout + margin + goal_keepout
    double rx = rs.uniform(lo, hi), ry = rs.uniform(lo, hi);
    for (int k = 0; k < 55; ++k) {
        double gx = rs.uniform(lo, hi), gy = rs.uniform(lo, hi);
        double dx = rn::sub(gx, rx), dy = rn::sub(gy, ry);
        double dist = rn::root(rn::add(rn::mul(dx, dx), rn::mul(dy, dy)));
        if (!(dist < keep)) break;
    }
    return rs.uniform(0.0, 2 * 3.141592653589793);
}

// ---------------------------------------------------------------------------------------
// Philox4x32-10: device-side action noise when the host does not supply it.
__device__ __forceinline__ uint4 philox4x32(uint4 ctr, uint2 key) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t h0 = __umulhi(M0, ctr.x), l0 = M0 * ctr.x;
        uint32_t h1 = __umulhi(M1, ctr.z), l1 = M1 * ctr.z;
        ctr = make_uint4(h1 ^ ctr.y ^ key.x, l1, h0 ^ ctr.w ^ key.y, l0);
        key.x += W0;
        key.y += W1;
    }
    return ctr;
}

// two independent standard normals from two 32-bit words (Box-Muller)
__device__ __forceinline__ float2 normal2(uint32_t u0, uint32_t u1) {
    float a = ((float)u0 + 0.5f) * (1.0f / 4294967296.0f);
    float b = ((float)u1 + 0.5f) * (1.0f / 4294967296.0f);
    a = fminf(fmaxf(a, 1e-10f), 1.0f);
    float r = sqrtf(-2.0f * logf(a));
    float s, c;
    sincospif(2.0f * b, &s, &c);
    return make_float2(r * c, r * s);
}

}  // namespace mr
