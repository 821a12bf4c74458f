// Fused rollout (K4 + K1 + K6 + K11): replaces [SB3 2.0.0] OnPolicyAlgorithm.collect_rollouts over
// DummyVecEnv(Monitor(TimeLimit(PointEnv))) -- policy forward, Gaussian sampling, log-prob,
// action clip, env step, reward, goal-reached / time-limit flags, auto-reset, time-out
// bootstrap, Monitor episode statistics and RolloutBuffer.add -- for T steps in ONE launch.
// Reference call chain: examples/train.py:42-46 -> src/mobrob/rl_control/ppo.py:73-74 ->
// PPO.learn -> collect_rollouts -> EnvWrapper.step (src/mobrob/envs/wrapper.py:156-171).
//
// Environments are independent for the whole rollout and the parameters are frozen, so
// there is no grid-wide synchronisation: a warp owns 8 environments for all T steps.  The
// body state stays in fp64 registers of lanes 0..7, the parameters stay in shared memory,
// the two MLP towers run as the warp micro-GEMM of mlp.cuh, and the only HBM traffic is the
// rollout-buffer rows (80 B per env-step for the point robot).
#include "env_state.cuh"
#include "mlp.cuh"

#include <stdlib.h>
#include <string.h>

namespace mr {

// (warps per CTA, environments per warp): measured on B200 at 4096 envs x 296 steps (tools/time_rollout.py):
// 4x8 2.55 ms, 7x4 2.19 ms, 8x4 2.06 ms, 4x4 2.04 ms, 14x4 3.09 ms.  4 x 4 = 256 CTAs, ~7 warps per SM
// (the env step is a long fp64 dependency chain: more, smaller warps
// hide it better than 4 x 8, at the price of re-reading the weights per 4 instead of 8 samples).
constexpr int RO_WARPS_DEFAULT = 4;
constexpr int RO_E_DEFAULT = 4;

struct RolloutArgs {
    PointState st;
    EnvCfg cfg;
    const float* params;
    int O;
    int64_t T, N;
    float* last_obs;       // [N][O]  in: obs the rollout starts from; out: obs it ended on
    float* last_starts;    // [N]     in/out: _last_episode_starts
    float* obs;            // [T][N][O]
    float* act;            // [T][N][2]  unclipped actions
    float* rew;            // [T][N]
    float* starts;         // [T][N]
    float* val;            // [T][N]
    float* logp;           // [T][N]
    float* last_val;       // [N]  V(final obs)
    uint8_t* last_done;    // [N]
    const float* eps;      // [T][N][2] host-supplied N(0,1) draws, or NULL -> Philox
    uint64_t seed;
    uint64_t noise_offset; // rollout counter * T (Philox counter word)
    int64_t env_offset;    // global index of env 0 (multi-GPU sharding)
    float gamma;
    double* ep_ret;        // [T][N] Monitor's return and length of the episode that ended at (t, n), written only
    int32_t* ep_len;       //        there (episode_records puts them into the ring in SB3's order)
};

template <int RO_WARPS, int RO_E>
__global__ void __launch_bounds__(RO_WARPS * 32) point_rollout_kernel(RolloutArgs A) {
    extern __shared__ __align__(16) float smem[];
    const int O = A.O;
    SmemW W = stage_weights(smem, A.params, O);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* obsT = smem + smem_w_floats(O) + warp * (MAX_OBS * RO_E + 128 * RO_E);
    float* hbuf = obsT + MAX_OBS * RO_E;
    __syncthreads();

    const int64_t n0 = ((int64_t)blockIdx.x * RO_WARPS + warp) * RO_E;  // first env of this warp
    if (n0 >= A.N) return;
    const int n_live = (int)min((int64_t)RO_E, A.N - n0);
    const bool phys = lane < n_live;
    const int64_t n = n0 + lane;
    const float sig0 = expf(W.logstd[0]), sig1 = expf(W.logstd[1]);
    const float gamma = A.gamma;

    PointHot h;
    float start_flag = 0.f;
    if (phys) {
        h = A.st.load(n);
        start_flag = A.last_starts[n];
    }
    for (int idx = lane; idx < RO_E * O; idx += 32) {
        int e = idx / O, k = idx - e * O;
        obsT[k * RO_E + e] = e < n_live ? A.last_obs[n0 * O + idx] : 0.f;
    }
    __syncwarp();

    const int e_of = lane / 3, j_of = lane - 3 * e_of;
    // where element lane + 32 i of the tile's contiguous rows sits in the transposed tile (the division by the
    // run-time O inside the step loop was 4 % of the kernel's stall samples)
    constexpr int ROW_PASSES = (RO_E * MAX_OBS + 31) / 32;
    int tile_off[ROW_PASSES];
#pragma unroll
    for (int i = 0; i < ROW_PASSES; ++i) {
        const int idx = lane + 32 * i, e = idx / O, k = idx - e * O;
        tile_off[i] = idx < n_live * O ? k * RO_E + e : -1;
    }
    bool done_flag = false;
    for (int64_t t = 0; t < A.T; ++t) {
        // RolloutBuffer.add(obs): the tile's rows are contiguous in the [T][N][O] buffer
        {
            float* dst = A.obs + (t * A.N + n0) * O;
#pragma unroll
            for (int i = 0; i < ROW_PASSES; ++i)
                if (tile_off[i] >= 0) dst[lane + 32 * i] = obsT[tile_off[i]];
        }
        float out = warp_mlp_forward<RO_E>(W, O, obsT, hbuf, lane);
        // sample: a = mu + sigma * eps ; log-prob in torch's evaluation order
        float a = out, lp = 0.f;
        if (lane < 3 * RO_E && e_of < n_live && j_of < 2) {
            const int64_t ne = n0 + e_of;
            float z;
            if (A.eps) {
                z = A.eps[(t * A.N + ne) * 2 + j_of];
            } else {
                const uint64_t g = (uint64_t)(A.env_offset + ne);
                const uint64_t c = A.noise_offset + (uint64_t)t;
                uint4 r = philox4x32(make_uint4((uint32_t)g, (uint32_t)(g >> 32), (uint32_t)c, (uint32_t)(c >> 32)),
                                     make_uint2((uint32_t)A.seed, (uint32_t)(A.seed >> 32)));
                float2 zz = normal2(r.x, r.y);
                z = j_of == 0 ? zz.x : zz.y;
            }
            const float sig = j_of == 0 ? sig0 : sig1;
            a = __fadd_rn(out, __fmul_rn(sig, z));
            lp = normal_logprob(a, out, sig);
        }
        const int src = 3 * (lane % RO_E);
        const float a0 = __shfl_sync(0xffffffffu, a, src);
        const float a1 = __shfl_sync(0xffffffffu, a, src + 1);
        const float v = __shfl_sync(0xffffffffu, out, src + 2);
        const float logp = __fadd_rn(__shfl_sync(0xffffffffu, lp, src), __shfl_sync(0xffffffffu, lp, src + 1));

        StepResult r;
        r.trunc = false;
        float o_new[point::OBS], o_term[point::OBS];
        if (phys) {
            const int64_t row = t * A.N + n;
            reinterpret_cast<float2*>(A.act)[row] = make_float2(a0, a1);
            A.val[row] = v;
            A.logp[row] = logp;
            A.starts[row] = start_flag;
            r = point_env_step(h, A.st.cold, n, a0, a1, A.cfg, o_new, o_term);
            if (r.done) {
                A.ep_ret[row] = r.ep_r;
                A.ep_len[row] = r.ep_l;
            }
            start_flag = r.done ? 1.f : 0.f;
            done_flag = r.done;
        }
        // time-out bootstrap: reward += gamma * V(terminal_observation) where truncated
        const unsigned trunc_mask = __ballot_sync(0xffffffffu, phys && r.trunc);
        float rew = phys ? r.rew : 0.f;
        if (trunc_mask) {
            __syncwarp();
            if (phys) {
#pragma unroll
                for (int k = 0; k < point::OBS; ++k) obsT[k * RO_E + lane] = r.trunc ? o_term[k] : 0.f;
            }
            __syncwarp();
            const float tv_all = warp_mlp_forward<RO_E>(W, O, obsT, hbuf, lane);
            const float tv = __shfl_sync(0xffffffffu, tv_all, src + 2);
            if (phys && r.trunc) rew = __fadd_rn(rew, __fmul_rn(gamma, tv));
        }
        if (phys) {
            A.rew[t * A.N + n] = rew;
#pragma unroll
            for (int k = 0; k < point::OBS; ++k) obsT[k * RO_E + lane] = o_new[k];
        }
        __syncwarp();
    }

    // values of the final observation, carry-over state
    const float out = warp_mlp_forward<RO_E>(W, O, obsT, hbuf, lane);
    const float v_last = __shfl_sync(0xffffffffu, out, 3 * (lane % RO_E) + 2);
    if (phys) {
        A.last_val[n] = v_last;
        A.last_done[n] = done_flag ? 1 : 0;
        A.last_starts[n] = start_flag;
        A.st.store(n, h);
    }
    for (int idx = lane; idx < n_live * O; idx += 32) {
        int e = idx / O, k = idx - e * O;
        A.last_obs[n0 * O + idx] = obsT[k * RO_E + e];
    }
}

// ---------------------------------------------------------------------------------------------
// Monitor's finished episodes in SB3's order.  DummyVecEnv steps its envs in index order and collect_rollouts appends
// each step's infos to ep_info_buffer, so the episodes of a rollout are ordered by (step, env).  The rollout kernels
// leave them in [T][N] side buffers at the (t, n) where they ended; the done mask tells which entries are valid:
// episode_starts[t + 1], or last_done at the last step.  Two launches put the newest ring_cap of them into the ring
// (slot = global episode index % ring_cap) and advance the episode counter, with no host synchronisation.
constexpr int EPR_THREADS = 256;

__device__ __forceinline__ bool episode_ended(const float* starts, const uint8_t* last_done, int64_t t, int64_t T,
                                              int64_t N, int64_t n) {
    return t + 1 < T ? starts[(t + 1) * N + n] != 0.f : last_done[n] != 0;
}

// block t: the number of episodes that ended at step t; the counter gets the rollout's total
__global__ void __launch_bounds__(EPR_THREADS) episode_count_kernel(const float* starts, const uint8_t* last_done,
                                                                    int64_t T, int64_t N, int32_t* ep_steps,
                                                                    unsigned long long* ep_count) {
    __shared__ int part[EPR_THREADS / 32];
    const int64_t t = blockIdx.x;
    int c = 0;
    for (int64_t n = threadIdx.x; n < N; n += EPR_THREADS) c += episode_ended(starts, last_done, t, T, N, n);
    c = __reduce_add_sync(0xffffffffu, c);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int s = 0;
        for (int w = 0; w < EPR_THREADS / 32; ++w) s += part[w];
        ep_steps[t] = s;
        if (s) atomicAdd(ep_count, (unsigned long long)s);
    }
}

// block t: the episodes that ended at step t, in env order, into ring slots (first index of the step + rank) % cap
__global__ void __launch_bounds__(EPR_THREADS) episode_ring_kernel(const float* starts, const uint8_t* last_done,
                                                                   const double* ep_ret, const int32_t* ep_len,
                                                                   int64_t T, int64_t N, const int32_t* ep_steps,
                                                                   const unsigned long long* ep_count, double* ep_r,
                                                                   int32_t* ep_l, int ring_cap) {
    __shared__ long long part[EPR_THREADS / 32];
    __shared__ int warp_cnt[EPR_THREADS / 32];
    const int64_t t = blockIdx.x;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    long long later = 0;   // episodes that ended after step t
    for (int64_t s = t + 1 + threadIdx.x; s < T; s += EPR_THREADS) later += ep_steps[s];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) later += __shfl_down_sync(0xffffffffu, later, o);
    if (lane == 0) part[w] = later;
    __syncthreads();
    later = 0;
    for (int i = 0; i < EPR_THREADS / 32; ++i) later += part[i];
    const int mine = ep_steps[t];
    if (mine == 0 || later >= ring_cap) return;   // nothing ended here, or newer episodes fill the ring
    const unsigned long long first = *ep_count - (unsigned long long)(later + mine);   // global index of the step's first
    const long long skip = later + mine - ring_cap;   // > 0: the step's oldest episodes do not fit
    int base = 0;
    for (int64_t n0 = 0; n0 < N && base < mine; n0 += EPR_THREADS) {
        const int64_t n = n0 + threadIdx.x;
        const bool d = n < N && episode_ended(starts, last_done, t, T, N, n);
        const unsigned bal = __ballot_sync(0xffffffffu, d);
        if (lane == 0) warp_cnt[w] = __popc(bal);
        __syncthreads();
        int rank = base + __popc(bal & ((1u << lane) - 1u)), tot = 0;
        for (int i = 0; i < EPR_THREADS / 32; ++i) {
            rank += i < w ? warp_cnt[i] : 0;
            tot += warp_cnt[i];
        }
        if (d && rank >= skip) {
            const unsigned long long slot = (first + (unsigned long long)rank) % (unsigned long long)ring_cap;
            ep_r[slot] = ep_ret[t * N + n];
            ep_l[slot] = ep_len[t * N + n];
        }
        base += tot;
        __syncthreads();
    }
}

}  // namespace mr

using namespace mr;

static int episode_records(const float* starts, const uint8_t* last_done, const double* ep_ret, const int32_t* ep_len,
                           int64_t T, int64_t N, int32_t* ep_steps, double* ep_r, int32_t* ep_l,
                           unsigned long long* ep_count, int ring_cap, cudaStream_t stream) {
    episode_count_kernel<<<(unsigned)T, EPR_THREADS, 0, stream>>>(starts, last_done, T, N, ep_steps, ep_count);
    MR_CHECK_LAUNCH();
    episode_ring_kernel<<<(unsigned)T, EPR_THREADS, 0, stream>>>(starts, last_done, ep_ret, ep_len, T, N, ep_steps,
                                                                 ep_count, ep_r, ep_l, ring_cap);
    MR_CHECK_LAUNCH();
    return MR_OK;
}

template <int RO_WARPS, int RO_E>
static int launch_rollout_cfg(const RolloutArgs& A, int64_t n_envs, cudaStream_t stream) {
    const size_t smem = (smem_w_floats(A.O) + RO_WARPS * (MAX_OBS * RO_E + 128 * RO_E)) * sizeof(float);
    static OncePerDevice once;
    if (once.first())
        MR_CUDA(cudaFuncSetAttribute(point_rollout_kernel<RO_WARPS, RO_E>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     100 * 1024));
    const int64_t warps = (n_envs + RO_E - 1) / RO_E;
    const int blocks = (int)((warps + RO_WARPS - 1) / RO_WARPS);
    point_rollout_kernel<RO_WARPS, RO_E><<<blocks, RO_WARPS * 32, smem, stream>>>(A);
    MR_CHECK_LAUNCH();
    return MR_OK;
}

static int launch_rollout(const RolloutArgs& A, int64_t n_envs, cudaStream_t stream) {
    static int cfg = -1;   // MR_ROLLOUT_CFG = "<warps>x<envs per warp>" selects a tuning variant
    if (cfg < 0) {
        const char* e = getenv("MR_ROLLOUT_CFG");
        cfg = 0;
        if (e) {
            if (!strcmp(e, "4x8")) cfg = 1;
            else if (!strcmp(e, "4x4")) cfg = 2;
            else if (!strcmp(e, "8x4")) cfg = 3;
            else if (!strcmp(e, "14x4")) cfg = 4;
        }
    }
    switch (cfg) {
        case 1: return launch_rollout_cfg<4, 8>(A, n_envs, stream);
        case 2: return launch_rollout_cfg<4, 4>(A, n_envs, stream);
        case 3: return launch_rollout_cfg<8, 4>(A, n_envs, stream);
        case 4: return launch_rollout_cfg<14, 4>(A, n_envs, stream);
        default: return launch_rollout_cfg<RO_WARPS_DEFAULT, RO_E_DEFAULT>(A, n_envs, stream);
    }
}

extern "C" int mr_rollout(mr_env* env, const float* params, int64_t T, float* last_obs,
                          float* last_starts, float* obs, float* act, float* rew, float* starts,
                          float* val, float* logp, float* last_val, uint8_t* last_done,
                          const float* eps, uint64_t seed, uint64_t noise_offset,
                          int64_t env_offset, double gamma, double* ep_ret, int32_t* ep_len,
                          int32_t* ep_steps, double* ep_r, int32_t* ep_l, unsigned long long* ep_count,
                          int ring_cap, void* stream) {
    MR_REQUIRE(env && params && last_obs && last_starts && obs && act && rew && starts && val &&
                   logp && last_val && last_done && ep_ret && ep_len && ep_steps && ep_r && ep_l && ep_count,
               "NULL argument");
    MR_REQUIRE(env->kind == MR_ENV_POINT, "fused rollout is built for the point env");
    MR_REQUIRE(env->cfg.obs_flags == 0, "fused rollout is built for the default observation (use mr_rollout_unfused)");
    MR_REQUIRE(T > 0 && T <= INT32_MAX && ring_cap > 0, "T must be in 1 .. 2^31 - 1 and ring_cap positive");
    RolloutArgs A;
    A.st = env->point;
    A.cfg = env->cfg;
    A.params = params;
    A.O = point::OBS;
    A.T = T;
    A.N = env->n;
    A.last_obs = last_obs; A.last_starts = last_starts;
    A.obs = obs; A.act = act; A.rew = rew; A.starts = starts; A.val = val; A.logp = logp;
    A.last_val = last_val; A.last_done = last_done;
    A.eps = eps; A.seed = seed; A.noise_offset = noise_offset; A.env_offset = env_offset;
    A.gamma = (float)gamma;
    A.ep_ret = ep_ret; A.ep_len = ep_len;
    const int rc = launch_rollout(A, env->n, (cudaStream_t)stream);
    if (rc != MR_OK) return rc;
    return episode_records(starts, last_done, ep_ret, ep_len, T, env->n, ep_steps, ep_r, ep_l, ep_count, ring_cap,
                           (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------
// Unfused rollout: the same collect_rollouts semantics as mr_rollout from the stand-alone env-step kernel plus ONE
// bookkeeping kernel per step.  Used for the car, whose contact solver is too heavy to share a warp with the MLP,
// for envs with optional observation keys, and as a cross-check of the fused kernel.
namespace mr {

constexpr int RS_WARPS = 8;   // 88 KB of shared memory per block: two blocks = 16 warps per SM, 16 384 envs in one wave
constexpr int RS_E = 8;

struct StepArgs {
    const float* params;
    int O;
    int64_t N, t;
    int record;            // finish step t - 1: time-out bootstrap, reward row, episode records, start flags
    int forward;           // open step t: buffer rows, policy forward, sampling
    float* last_obs;       // [N][O]  observation the env returned (in), unchanged
    float* last_starts;    // [N]     _last_episode_starts (updated by the record half)
    float* obs; float* act; float* rew; float* starts; float* val; float* logp;   // rollout buffer, [T][N][...]
    float* last_val;       // [N]  (closing call: V of the final observation)
    const float* eps;      // [T][N][2] host-supplied draws or NULL -> Philox
    uint64_t seed, noise_offset;
    int64_t env_offset;
    float gamma;
    // outputs of the env step t - 1
    const float* rew_tmp; const uint8_t* done; const uint8_t* trunc; const float* term_obs;
    const double* ep_ret_n; const int32_t* ep_len_n;
    double* ep_ret; int32_t* ep_len;   // [T][N] episodes that ended at (t - 1, n), as in RolloutArgs
};

// Between two env steps: [RolloutBuffer.add bookkeeping of the step that just ran] + [policy forward, Gaussian
// sample, log-prob and buffer rows of the step about to run], a warp per tile of 8 envs.  Replaces, per step, two
// device-to-device copies, the noise kernel, the policy forward, the masked terminal-value forward and the record
// kernel (6 launches, ~68 us of a 242 us car step) by one launch.
__global__ void __launch_bounds__(RS_WARPS * 32) rollout_step_kernel(StepArgs A) {
    extern __shared__ __align__(16) float smem[];
    const int O = A.O;
    SmemW W = stage_weights(smem, A.params, O);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* obsT = smem + smem_w_floats(O) + warp * (MAX_OBS * RS_E + 128 * RS_E);
    float* hbuf = obsT + MAX_OBS * RS_E;
    __syncthreads();
    const float sig0 = expf(W.logstd[0]), sig1 = expf(W.logstd[1]);
    const int64_t n_tiles = (A.N + RS_E - 1) / RS_E;
    const int e_of = lane / 3, j_of = lane - 3 * e_of;
    for (int64_t tile = (int64_t)blockIdx.x * RS_WARPS + warp; tile < n_tiles; tile += (int64_t)gridDim.x * RS_WARPS) {
        const int64_t s0 = tile * RS_E;
        const int rows = (int)min((int64_t)RS_E, A.N - s0);
        const bool own = lane < rows;          // lane e owns env s0 + e for the per-env bookkeeping
        const int64_t n = s0 + lane;
        float start_flag = own ? A.last_starts[n] : 0.f;
        if (A.record) {
            const bool tr = own && A.trunc[n] != 0;
            float r = own ? A.rew_tmp[n] : 0.f;
            if (__any_sync(0xffffffffu, tr)) {   // reward += gamma * V(terminal_observation) where the episode timed out
                for (int idx = lane; idx < RS_E * O; idx += 32) {
                    const int e = idx / O, k = idx - e * O;
                    obsT[k * RS_E + e] = e < rows ? A.term_obs[s0 * O + idx] : 0.f;
                }
                __syncwarp();
                const float out = warp_mlp_forward<RS_E>(W, O, obsT, hbuf, lane);
                const float tv = __shfl_sync(0xffffffffu, out, 3 * (lane % RS_E) + 2);
                if (tr) r = __fadd_rn(r, __fmul_rn(A.gamma, tv));
            }
            if (own) {
                A.rew[(A.t - 1) * A.N + n] = r;
                const bool d = A.done[n] != 0;
                start_flag = d ? 1.f : 0.f;
                A.last_starts[n] = start_flag;
                if (d) {
                    A.ep_ret[(A.t - 1) * A.N + n] = A.ep_ret_n[n];
                    A.ep_len[(A.t - 1) * A.N + n] = A.ep_len_n[n];
                }
            }
        }
        // the observation the policy acts on: RolloutBuffer.add(obs) row + transposed tile for the forward
        for (int idx = lane; idx < RS_E * O; idx += 32) {
            const int e = idx / O, k = idx - e * O;
            const float v = e < rows ? A.last_obs[s0 * O + idx] : 0.f;
            obsT[k * RS_E + e] = v;
            if (A.forward && e < rows) A.obs[(A.t * A.N + s0) * O + idx] = v;
        }
        __syncwarp();
        const float out = warp_mlp_forward<RS_E>(W, O, obsT, hbuf, lane);
        if (!A.forward) {   // closing call: values of the final observation
            if (lane < 3 * RS_E && e_of < rows && j_of == 2) A.last_val[s0 + e_of] = out;
            continue;
        }
        const bool live = lane < 3 * RS_E && e_of < rows;
        float a = out, lp = 0.f;
        if (live && j_of < 2) {
            const int64_t ne = s0 + e_of;
            float z;
            if (A.eps) {
                z = A.eps[(A.t * A.N + ne) * 2 + j_of];
            } else {
                const uint64_t g = (uint64_t)(A.env_offset + ne);
                const uint64_t c = A.noise_offset + (uint64_t)A.t;
                const uint4 rr = philox4x32(make_uint4((uint32_t)g, (uint32_t)(g >> 32), (uint32_t)c, (uint32_t)(c >> 32)),
                                            make_uint2((uint32_t)A.seed, (uint32_t)(A.seed >> 32)));
                const float2 zz = normal2(rr.x, rr.y);
                z = j_of == 0 ? zz.x : zz.y;
            }
            const float sig = j_of == 0 ? sig0 : sig1;
            a = __fadd_rn(out, __fmul_rn(sig, z));
            lp = normal_logprob(a, out, sig);
            A.act[(A.t * A.N + ne) * 2 + j_of] = a;
        }
        const float lp1 = __shfl_down_sync(0xffffffffu, lp, 1);
        if (live && j_of == 0) A.logp[A.t * A.N + s0 + e_of] = __fadd_rn(lp, lp1);
        if (live && j_of == 2) A.val[A.t * A.N + s0 + e_of] = out;
        if (own) A.starts[A.t * A.N + n] = start_flag;
        __syncwarp();
    }
}

}  // namespace mr

extern "C" int mr_rollout_unfused(mr_env* env, const float* params, int64_t T, float* last_obs,
                                  float* last_starts, float* obs, float* act, float* rew, float* starts,
                                  float* val, float* logp, float* last_val, uint8_t* last_done,
                                  const float* eps, uint64_t seed, uint64_t noise_offset,
                                  int64_t env_offset, double gamma, double* ep_ret, int32_t* ep_len,
                                  int32_t* ep_steps, double* ep_r, int32_t* ep_l, unsigned long long* ep_count,
                                  int ring_cap, void* stream) {
    MR_REQUIRE(env && params && last_obs && last_starts && obs && act && rew && starts && val && logp &&
                   last_val && last_done && ep_ret && ep_len && ep_steps && ep_r && ep_l && ep_count, "NULL argument");
    MR_REQUIRE(T > 0 && T <= INT32_MAX && ring_cap > 0, "T must be in 1 .. 2^31 - 1 and ring_cap positive");
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t N = env->n;
    const int O = mr_env_obs_dim(env);
    MR_REQUIRE(O <= MAX_OBS, "the policy kernels take observations of at most 32 floats");
    // scratch (library-owned, one per env handle): what one env step hands to the next bookkeeping launch
    const size_t per_env = 8 + (size_t)O * 4 + 4 + 4 + 1 + 1;
    if (!env->scratch) {
        DeviceGuard guard(env->device);
        MR_CUDA(cudaMalloc(&env->scratch, per_env * N + 8 * 256));
        MR_CUDA(cudaMemsetAsync(env->scratch, 0, per_env * N + 8 * 256, s));
    }
    char* p = static_cast<char*>(env->scratch);
    auto take = [&](size_t bytes) { char* r = p; p += (bytes + 255) & ~size_t(255); return r; };
    double* ep_ret_n = (double*)take(N * 8);
    float* term_obs = (float*)take(N * O * 4);
    float* rew_tmp = (float*)take(N * 4);
    int32_t* ep_len_n = (int32_t*)take(N * 4);
    uint8_t* done = (uint8_t*)take(N);
    uint8_t* trunc = (uint8_t*)take(N);

    const size_t smem = (smem_w_floats(O) + RS_WARPS * (MAX_OBS * RS_E + 128 * RS_E)) * sizeof(float);
    static OncePerDevice once;
    if (once.first())
        MR_CUDA(cudaFuncSetAttribute(mr::rollout_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    const int64_t tiles = (N + RS_E - 1) / RS_E;
    const int blocks = (int)std::min<int64_t>((tiles + RS_WARPS - 1) / RS_WARPS, (int64_t)sm_count() * 2);
    StepArgs A;
    A.params = params; A.O = O; A.N = N;
    A.last_obs = last_obs; A.last_starts = last_starts;
    A.obs = obs; A.act = act; A.rew = rew; A.starts = starts; A.val = val; A.logp = logp; A.last_val = last_val;
    A.eps = eps; A.seed = seed; A.noise_offset = noise_offset; A.env_offset = env_offset; A.gamma = (float)gamma;
    A.rew_tmp = rew_tmp; A.done = done; A.trunc = trunc; A.term_obs = term_obs; A.ep_ret_n = ep_ret_n; A.ep_len_n = ep_len_n;
    A.ep_ret = ep_ret; A.ep_len = ep_len;
    for (int64_t t = 0; t <= T; ++t) {
        A.t = t; A.record = t > 0; A.forward = t < T;
        mr::rollout_step_kernel<<<blocks, RS_WARPS * 32, smem, s>>>(A);
        MR_CHECK_LAUNCH();
        if (t == T) break;
        const int rc = mr_env_step(env, act + t * N * 2, last_obs, rew_tmp, done, trunc, term_obs, ep_ret_n, ep_len_n, stream);
        if (rc != MR_OK) return rc;
    }
    MR_CUDA(cudaMemcpyAsync(last_done, done, N, cudaMemcpyDeviceToDevice, s));
    return episode_records(starts, last_done, ep_ret, ep_len, T, N, ep_steps, ep_r, ep_l, ep_count, ring_cap, s);
}
