// HBM layout of the batched environment state: one slab per mr_env, every array 256-byte aligned.
// "Hot" fields are read+written by every step; "cold" arrays only by resets.
//
// Hot state is TILED: a tile holds the hot fields of 128 consecutive envs (= one block of the
// env-step kernel), field-major inside the tile, 9728 contiguous bytes:
//     px py psi vx vy om ep_ret  (f64, 1024 B each) | ctrl goal (float2, 1024 B each) | elapsed (i32, 512 B)
// A warp's loads stay 128/256-byte coalesced, every field of an env sits at a COMPILE-TIME offset
// from one per-thread address (a plain struct-of-arrays spent 8 % of the env-step kernel's
// instructions on 64-bit address arithmetic for its 10 arrays), and the block's whole input is one
// contiguous range for the L2 prefetch.
#pragma once

#include "env_car.cuh"
#include "env_point.cuh"

namespace mr {

constexpr int POINT_STATE_DIM = 15;

struct PointState {
    static constexpr int TILE = 128;
    static constexpr int F_PX = 0, F_PY = 1024, F_PSI = 2048, F_VX = 3072, F_VY = 4096, F_OM = 5120, F_EPRET = 6144,
                         F_CTRL = 7168, F_GOAL = 8192, F_ELAPSED = 9216, TILE_BYTES = 9728;
    int64_t n;
    char* hot;   // ceil(n / 128) tiles
    EnvCold cold;

    static size_t align_up(size_t x) { return (x + 255) & ~size_t(255); }
    static size_t tiles(int64_t n) { return (size_t)((n + TILE - 1) / TILE); }
    static size_t slab_bytes(int64_t n) {
        size_t b = 0;
        b += align_up(tiles(n) * TILE_BYTES);
        b += 2 * align_up(n * 32);  // pcg_init pcg_goal
        b += align_up(n * 8);       // engine_seed
        b += align_up(n * 8);       // body_xy
        b += align_up(n * 8);       // psi0
        b += align_up(n * 8);       // counts
        b += align_up(32);          // spaces
        return b;
    }
    void carve(void* slab, int64_t n_) {
        n = n_;
        char* p = static_cast<char*>(slab);
        auto take = [&](size_t bytes) { char* r = p; p += align_up(bytes); return r; };
        hot = take(tiles(n) * TILE_BYTES);
        cold.pcg_init = (uint64_t*)take(n * 32); cold.pcg_goal = (uint64_t*)take(n * 32);
        cold.engine_seed = (int64_t*)take(n * 8);
        cold.body_xy = (float2*)take(n * 8);
        cold.psi0 = (double*)take(n * 8);
        cold.counts = (int32_t*)take(n * 8);
        cold.spaces = (const float*)take(32);
    }

    // address of env i's 8-byte slot in field 0 of its tile; the other fields are at + F_*
    __device__ __forceinline__ char* slot(int64_t i) const {
        return hot + (i >> 7) * TILE_BYTES + ((int)i & (TILE - 1)) * 8;
    }
    __device__ __forceinline__ char* tile(int64_t t) const { return hot + t * TILE_BYTES; }
    template <class T>
    static __device__ __forceinline__ T& at(char* p, int off) { return *reinterpret_cast<T*>(p + off); }
    // elapsed is 4 bytes wide: lane * 4 instead of lane * 8
    static __device__ __forceinline__ int32_t& elapsed_at(char* p, int64_t i) {
        return *reinterpret_cast<int32_t*>(p + F_ELAPSED - ((int)i & (TILE - 1)) * 4);
    }

    __device__ __forceinline__ PointHot load(int64_t i) const {
        char* p = slot(i);
        PointHot h;
        h.d.px = at<double>(p, F_PX); h.d.py = at<double>(p, F_PY); h.d.psi = at<double>(p, F_PSI);
        h.d.vx = at<double>(p, F_VX); h.d.vy = at<double>(p, F_VY); h.d.om = at<double>(p, F_OM);
        const float2 c = at<float2>(p, F_CTRL), g = at<float2>(p, F_GOAL);
        h.cx = c.x; h.cz = c.y; h.gx = g.x; h.gy = g.y;
        h.elapsed = elapsed_at(p, i);
        h.ep_ret = at<double>(p, F_EPRET);
        return h;
    }
    __device__ __forceinline__ void store(int64_t i, const PointHot& h) const {
        char* p = slot(i);
        at<double>(p, F_PX) = h.d.px; at<double>(p, F_PY) = h.d.py; at<double>(p, F_PSI) = h.d.psi;
        at<double>(p, F_VX) = h.d.vx; at<double>(p, F_VY) = h.d.vy; at<double>(p, F_OM) = h.d.om;
        at<float2>(p, F_CTRL) = make_float2(h.cx, h.cz);
        at<float2>(p, F_GOAL) = make_float2(h.gx, h.gy);
        elapsed_at(p, i) = h.elapsed;
        at<double>(p, F_EPRET) = h.ep_ret;
    }
    // env-step variants: data.ctrl is overwritten by the action before anything reads it, and the
    // goal only changes in a reset -- 8 B less read and 8 B less written per env-step
    // (68 B read, 68 B written).
    __device__ __forceinline__ PointHot load_step(int64_t i) const {
        char* p = slot(i);
        PointHot h;
        h.d.px = at<double>(p, F_PX); h.d.py = at<double>(p, F_PY); h.d.psi = at<double>(p, F_PSI);
        h.d.vx = at<double>(p, F_VX); h.d.vy = at<double>(p, F_VY); h.d.om = at<double>(p, F_OM);
        const float2 g = at<float2>(p, F_GOAL);
        h.cx = 0.f; h.cz = 0.f; h.gx = g.x; h.gy = g.y;
        h.elapsed = elapsed_at(p, i);
        h.ep_ret = at<double>(p, F_EPRET);
        return h;
    }
    __device__ __forceinline__ void store_step(int64_t i, const PointHot& h, bool was_reset) const {
        char* p = slot(i);
        at<double>(p, F_PX) = h.d.px; at<double>(p, F_PY) = h.d.py; at<double>(p, F_PSI) = h.d.psi;
        at<double>(p, F_VX) = h.d.vx; at<double>(p, F_VY) = h.d.vy; at<double>(p, F_OM) = h.d.om;
        at<float2>(p, F_CTRL) = make_float2(h.cx, h.cz);
        if (was_reset) at<float2>(p, F_GOAL) = make_float2(h.gx, h.gy);
        elapsed_at(p, i) = h.elapsed;
        at<double>(p, F_EPRET) = h.ep_ret;
    }
    __device__ __forceinline__ double2 pos(int64_t i) const {
        char* p = slot(i);
        return make_double2(at<double>(p, F_PX), at<double>(p, F_PY));
    }
    // pull tile t (one block's hot input: 68 of the tile's 76 lines of 128 B -- the step never reads the ctrl
    // field) towards L2; called by a block one wave ahead of the tile's use, thread k takes line k
    __device__ __forceinline__ void prefetch_tile(int64_t t, int k) const {
        const bool ctrl_line = k >= F_CTRL / 128 && k < F_GOAL / 128;
        if (k < TILE_BYTES / 128 && !ctrl_line) asm volatile("prefetch.global.L2 [%0];" ::"l"(tile(t) + k * 128));
    }
};

}  // namespace mr

struct mr_env {
    int kind;
    int64_t n;
    int device;
    mr::EnvCfg cfg;
    void* slab;
    size_t slab_bytes;
    mr::PointState point;
    mr::CarSoA car;
    mr::car::Consts carK;
    void* scratch = nullptr;  // lazily allocated by mr_rollout_unfused
    void* haz_slab = nullptr; // mr_env_set_hazards: EnvCfg::haz's arrays
    int step_flip = 0;        // env-step kernels alternate the block order (L2 keeps the tail of the last step)
};

namespace mr {

// car env kernels (env.cu, waypoints.cu): one thread per env, the contact solver's scratch in shared memory
constexpr int CAR_THREADS = 64;
constexpr size_t CAR_SMEM = (size_t)car::SCRATCH_DOUBLES * sizeof(double) * CAR_THREADS;   // 112.5 KB: two CTAs per SM
#define MR_CAR_SCRATCH() extern __shared__ __align__(16) double car_smem[]; \
    const car::Scratch S{(uint32_t)__cvta_generic_to_shared(car_smem + threadIdx.x), (uint32_t)(CAR_THREADS * sizeof(double))}

// EnvWrapper.set_goal for the masked envs (mask NULL: all): env i's goal <- goals[i * goal_stride + 0..1]; obs (may be
// NULL) receives the masked envs' get_obs() rows.  mr_env_set_goals and mr_follow_waypoints' first waypoint.
int env_set_goals(mr_env* env, const uint8_t* mask, const float* goals, int64_t goal_stride, float* obs,
                  cudaStream_t s);

// mr_follow_waypoints' per-step path: the per-env loop state, advanced by env_step_waypoints (waypoints.cu)
struct WaypointStep {
    const float* wp;                 // [N][K][2]
    int K;
    int64_t max_steps;
    int64_t t;                       // step index of this launch (0-based)
    int32_t* cursor;                 // [N] next waypoint; K once the last one is reached
    int32_t* steps;                  // [N] steps the env has taken
    double* ret;                     // [N] sum of the rewards
    int32_t* arrival;                // [N][K]
    float* pos;                      // [max_steps + 1][N][2] or NULL
    unsigned long long* n_finished;  // envs whose loop has ended
};

// one step of the envs whose loop is still running (the others are not touched): env step with act, the step's
// arrival / return bookkeeping, the next waypoint's goal and get_obs() row for envs that just reached one
int env_step_waypoints(mr_env* env, const float* act, float* obs, const WaypointStep& w, cudaStream_t s);

}  // namespace mr
