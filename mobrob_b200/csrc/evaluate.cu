// Batched policy evaluation (K5): replaces [SB3 2.0.0] common/evaluation.py:evaluate_policy over the vectorised
// env -- env.reset(), then model.predict + VecEnv.step until every env has finished its share of n_eval_episodes,
// recording Monitor's info["episode"] (r, l) of each counted episode.
//
// Env i counts its first c_i = (n_episodes + i) // N finished episodes; its records go to slots off_i .. off_i + c_i - 1
// (off_i = sum of c_j over j < i, in closed form), each with the step index t at which it ended, so that the host
// can put them into SB3's (step, env index) order.  Like SB3's loop, every env keeps stepping until the LAST one has
// met its target (S steps in all): the env is left where SB3 leaves it, which matters because the next evaluation
// starts with a lazy reset that only re-places the robot if the goal was not reached.
//
// Two paths, picked from the env handle:
//   * point, default observation row: point_eval_kernel, a copy of point_rollout_kernel's structure (a warp owns a few
//     envs, fp64 body state in registers, parameters in shared memory) without any rollout-buffer traffic.  Phase 1
//     runs each warp until its envs are done and takes the max of the warps' step counts as S; phase 2 (a second
//     launch) advances every warp, without recording, to exactly S steps.
//   * the car, and point envs with optional observation keys: eval_step_kernel (record the episodes the last env step
//     finished, write the next actions) + the stand-alone mr_env_step per step, looped from C, which reads a device
//     "envs done" counter after each step to stop at exactly S.
// Both stop at max_steps at the latest (then *status = 1, the env stays consistent at S = max_steps).
#include "env_state.cuh"
#include "mlp.cuh"

namespace mr {

// same tiling as the rollout kernel's default.  On B200 at 16 384 envs (4 x 16 384 episodes, ~800 steps) 4 x 4,
// 4 x 8 and 8 x 8 came within 5 % of each other, inside run-to-run noise: the call is bound by the chain of S
// dependent steps (phase 1, then phase 2 for the warps that finished early), not by occupancy.
constexpr int EV_WARPS = 4;
constexpr int EV_E = 4;

// first slot of env i's records: sum over j < i of (E + j) // N.  With E = q N + r, (E + j) // N = q + [j >= N - r].
__host__ __device__ __forceinline__ int64_t eval_slot_offset(int64_t i, int64_t E, int64_t N) {
    const int64_t q = E / N, r = E % N;
    return q * i + (i > N - r ? i - (N - r) : 0);
}
__host__ __device__ __forceinline__ int64_t eval_target(int64_t i, int64_t E, int64_t N) { return (E + i) / N; }

// Philox draw of sample e's action component j: the rollout kernels' construction, keyed (seed, env_offset + n),
// counter noise_offset + t
__device__ __forceinline__ float eval_action(float mu, float sig, bool stochastic, uint64_t seed, uint64_t g, uint64_t c, int j) {
    if (!stochastic) return mu;
    const uint4 r = philox4x32(make_uint4((uint32_t)g, (uint32_t)(g >> 32), (uint32_t)c, (uint32_t)(c >> 32)),
                               make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const float2 zz = normal2(r.x, r.y);
    return __fadd_rn(mu, __fmul_rn(sig, j == 0 ? zz.x : zz.y));
}

struct EvalArgs {
    PointState st;
    EnvCfg cfg;
    const float* params;
    int O;
    int64_t N, E, max_steps;
    int phase;             // 1: run to the warp's targets and record; 2: advance to S without recording
    int stochastic;
    float* last_obs;       // [N][O] in: the observation of env.reset(); out: the observation after S steps
    double* ep_r;          // [E] Monitor's episode return
    int32_t* ep_l;         // [E] episode length
    int64_t* ep_t;         // [E] step index at which the episode ended
    int32_t* warp_steps;   // [warps] phase 1 -> phase 2: steps the warp has taken
    unsigned long long* S; // max over warps of the phase-1 step count
    int* status;           // 1 if max_steps ended the evaluation before every target was met
    uint64_t seed, noise_offset;
    int64_t env_offset;
};

template <int W_, int E_>
__global__ void __launch_bounds__(W_ * 32) point_eval_kernel(EvalArgs A) {
    extern __shared__ __align__(16) float smem[];
    const int O = A.O;
    SmemW W = stage_weights(smem, A.params, O);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* obsT = smem + smem_w_floats(O) + warp * (MAX_OBS * E_ + 128 * E_);
    float* hbuf = obsT + MAX_OBS * E_;
    __syncthreads();

    const int64_t wid = (int64_t)blockIdx.x * W_ + warp;
    const int64_t n0 = wid * E_;
    if (n0 >= A.N) return;
    const int n_live = (int)min((int64_t)E_, A.N - n0);
    const bool phys = lane < n_live;
    const int64_t n = n0 + lane;
    const float sig0 = expf(W.logstd[0]), sig1 = expf(W.logstd[1]);
    const bool record = A.phase == 1;

    int64_t t = 0, t_end = A.max_steps;
    if (!record) {
        t = A.warp_steps[wid];
        t_end = (int64_t)*A.S;
        if (t >= t_end) return;   // state and observation are already where phase 1 left them
    }
    int64_t target = 0, done_eps = 0, slot0 = 0;
    PointHot h;
    if (phys) {
        h = A.st.load(n);
        if (record) {
            target = eval_target(n, A.E, A.N);
            slot0 = eval_slot_offset(n, A.E, A.N);
        }
    }
    for (int idx = lane; idx < E_ * O; idx += 32) {
        const int e = idx / O, k = idx - e * O;
        obsT[k * E_ + e] = e < n_live ? A.last_obs[n0 * O + idx] : 0.f;
    }
    __syncwarp();

    const int e_of = lane / 3, j_of = lane - 3 * e_of;
    const int src = 3 * (lane % E_);
    for (; t < t_end; ++t) {
        // SB3's loop condition, per warp: stop once none of the warp's envs is short of its target
        if (record && !__any_sync(0xffffffffu, phys && done_eps < target)) break;
        const float out = warp_mlp_forward<E_>(W, O, obsT, hbuf, lane);
        float a = out;
        if (lane < 3 * E_ && e_of < n_live && j_of < 2)
            a = eval_action(out, j_of == 0 ? sig0 : sig1, A.stochastic, A.seed, (uint64_t)(A.env_offset + n0 + e_of),
                            A.noise_offset + (uint64_t)t, j_of);
        const float a0 = __shfl_sync(0xffffffffu, a, src);
        const float a1 = __shfl_sync(0xffffffffu, a, src + 1);
        float o_new[point::OBS], o_term[point::OBS];
        if (phys) {
            // point_env_step clips like predict's np.clip followed by Engine.step's clip
            const StepResult r = point_env_step(h, A.st.cold, n, a0, a1, A.cfg, o_new, o_term);
            if (record && r.done && done_eps < target) {
                const int64_t slot = slot0 + done_eps;
                A.ep_r[slot] = r.ep_r;
                A.ep_l[slot] = r.ep_l;
                A.ep_t[slot] = t;
                ++done_eps;
            }
        }
        __syncwarp();
        if (phys) {
#pragma unroll
            for (int k = 0; k < point::OBS; ++k) obsT[k * E_ + lane] = o_new[k];
        }
        __syncwarp();
    }

    if (record) {
        if (lane == 0) {
            A.warp_steps[wid] = (int32_t)t;
            atomicMax(A.S, (unsigned long long)t);
        }
        if (__any_sync(0xffffffffu, phys && done_eps < target) && lane == 0) atomicExch(A.status, 1);
    }
    if (phys) A.st.store(n, h);
    for (int idx = lane; idx < n_live * O; idx += 32) {
        const int e = idx / O, k = idx - e * O;
        A.last_obs[n0 * O + idx] = obsT[k * E_ + e];
    }
}

// ---------------------------------------------------------------------------------------------
// Per-step path: one launch between two env steps, in the mould of rollout_step_kernel.
constexpr int ES_WARPS = 8;
constexpr int ES_E = 8;

struct EvalStepArgs {
    const float* params;
    int O;
    int64_t N, E, t;
    int stochastic;
    const float* obs;                       // [N][O] the observation step t acts on
    float* act;                             // [N][2] out: step t's actions
    // outputs of env step t - 1 (read when t > 0)
    const uint8_t* done; const double* ep_ret_n; const int32_t* ep_len_n;
    int32_t* counts;                        // [N] episodes recorded so far
    unsigned long long* n_met;              // envs whose target is met
    double* ep_r; int32_t* ep_l; int64_t* ep_t;
    uint64_t seed, noise_offset;
    int64_t env_offset;
};

__global__ void __launch_bounds__(ES_WARPS * 32) eval_step_kernel(EvalStepArgs A) {
    extern __shared__ __align__(16) float smem[];
    const int O = A.O;
    SmemW W = stage_weights(smem, A.params, O);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* obsT = smem + smem_w_floats(O) + warp * (MAX_OBS * ES_E + 128 * ES_E);
    float* hbuf = obsT + MAX_OBS * ES_E;
    __syncthreads();
    const float sig0 = expf(W.logstd[0]), sig1 = expf(W.logstd[1]);
    const int64_t n_tiles = (A.N + ES_E - 1) / ES_E;
    const int e_of = lane / 3, j_of = lane - 3 * e_of;
    for (int64_t tile = (int64_t)blockIdx.x * ES_WARPS + warp; tile < n_tiles; tile += (int64_t)gridDim.x * ES_WARPS) {
        const int64_t s0 = tile * ES_E;
        const int rows = (int)min((int64_t)ES_E, A.N - s0);
        const int64_t n = s0 + lane;
        if (A.t > 0 && lane < rows && A.done[n]) {
            const int64_t target = eval_target(n, A.E, A.N);
            const int32_t k = A.counts[n];
            if (k < target) {
                const int64_t slot = eval_slot_offset(n, A.E, A.N) + k;
                A.ep_r[slot] = A.ep_ret_n[n];
                A.ep_l[slot] = A.ep_len_n[n];
                A.ep_t[slot] = A.t - 1;
                A.counts[n] = k + 1;
                if (k + 1 == target) atomicAdd(A.n_met, 1ull);
            }
        }
        for (int idx = lane; idx < ES_E * O; idx += 32) {
            const int e = idx / O, k = idx - e * O;
            obsT[k * ES_E + e] = e < rows ? A.obs[s0 * O + idx] : 0.f;
        }
        __syncwarp();
        const float out = warp_mlp_forward<ES_E>(W, O, obsT, hbuf, lane);
        if (lane < 3 * ES_E && e_of < rows && j_of < 2) {
            const int64_t ne = s0 + e_of;
            A.act[ne * 2 + j_of] = eval_action(out, j_of == 0 ? sig0 : sig1, A.stochastic, A.seed,
                                               (uint64_t)(A.env_offset + ne), A.noise_offset + (uint64_t)A.t, j_of);
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------
// Waypoint following (mr_follow_waypoints).  Fused path for the point's default row: point_eval_kernel's structure,
// each env with its own waypoint cursor and its own end; a warp ends when its envs have ended.
struct WaypointArgs {
    PointState st;
    EnvCfg cfg;
    const float* params;
    int O, K;
    int64_t N, max_steps;
    int stochastic;
    const float* wp;       // [N][K][2]
    float* last_obs;       // [N][O] out
    int32_t* arrival;      // [N][K] out (pre-filled with -1)
    double* ret;           // [N] out
    int32_t* steps;        // [N] out
    float2* pos;           // [max_steps + 1][N] out, or NULL
    uint64_t seed, noise_offset;
    int64_t env_offset;
};

template <int W_, int E_>
__global__ void __launch_bounds__(W_ * 32) point_waypoint_kernel(WaypointArgs A) {
    extern __shared__ __align__(16) float smem[];
    const int O = A.O;
    SmemW W = stage_weights(smem, A.params, O);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* obsT = smem + smem_w_floats(O) + warp * (MAX_OBS * E_ + 128 * E_);
    float* hbuf = obsT + MAX_OBS * E_;
    __syncthreads();

    const int64_t n0 = ((int64_t)blockIdx.x * W_ + warp) * E_;
    if (n0 >= A.N) return;
    const int n_live = (int)min((int64_t)E_, A.N - n0);
    const bool phys = lane < n_live;
    const int64_t n = n0 + lane;
    const float sig0 = expf(W.logstd[0]), sig1 = expf(W.logstd[1]);

    // set_goal(W[n, 0]); obs = get_obs()
    PointHot h;
    int k = 0, my_t = 0;
    double ret = 0.0;
    bool running = phys;
    if (phys) {
        h = A.st.load(n);
        h.gx = A.wp[n * A.K * 2];
        h.gy = A.wp[n * A.K * 2 + 1];
        float o[point::OBS];
        point::sensors(h.d, (double)h.cx, (double)h.cz, h.gx, h.gy, o);
#pragma unroll
        for (int j = 0; j < point::OBS; ++j) obsT[j * E_ + lane] = o[j];
        if (A.pos) A.pos[n] = make_float2((float)h.d.px, (float)h.d.py);
    } else if (lane < E_) {
        for (int j = 0; j < O; ++j) obsT[j * E_ + lane] = 0.f;
    }
    __syncwarp();

    const int e_of = lane / 3, j_of = lane - 3 * e_of;
    const int src = 3 * (lane % E_);
    int64_t t = 0;
    for (; t < A.max_steps; ++t) {
        if (!__any_sync(0xffffffffu, running)) break;
        const float out = warp_mlp_forward<E_>(W, O, obsT, hbuf, lane);
        float a = out;
        if (lane < 3 * E_ && e_of < n_live && j_of < 2)
            a = eval_action(out, j_of == 0 ? sig0 : sig1, A.stochastic, A.seed, (uint64_t)(A.env_offset + n0 + e_of),
                            A.noise_offset + (uint64_t)t, j_of);
        const float a0 = __shfl_sync(0xffffffffu, a, src);
        const float a1 = __shfl_sync(0xffffffffu, a, src + 1);
        float o_new[point::OBS], o_term[point::OBS];
        const bool stepped = running;
        if (stepped) {
            const StepResult r = point_env_step(h, A.st.cold, n, a0, a1, A.cfg, o_new, o_term);
            my_t = (int)t + 1;
            ret = rn::add(ret, r.reward);
            if (r.reach) {
                A.arrival[n * A.K + k] = my_t;
                if (++k < A.K) {   // set_goal(W[n, k]); obs = get_obs()
                    h.gx = A.wp[(n * A.K + k) * 2];
                    h.gy = A.wp[(n * A.K + k) * 2 + 1];
                    point::sensors(h.d, (double)h.cx, (double)h.cz, h.gx, h.gy, o_new);
                }
            }
            running = k < A.K && my_t < A.max_steps;
        }
        if (phys && A.pos) A.pos[(t + 1) * A.N + n] = make_float2((float)h.d.px, (float)h.d.py);
        __syncwarp();
        if (stepped) {
#pragma unroll
            for (int j = 0; j < point::OBS; ++j) obsT[j * E_ + lane] = o_new[j];
        }
        __syncwarp();
    }

    if (phys) {
        if (A.pos)   // rows past the warp's end repeat the final position
            for (int64_t r = t + 1; r <= A.max_steps; ++r) A.pos[r * A.N + n] = make_float2((float)h.d.px, (float)h.d.py);
        A.st.store(n, h);
        A.ret[n] = ret;
        A.steps[n] = my_t;
    }
    for (int idx = lane; idx < n_live * O; idx += 32) {
        const int e = idx / O, j = idx - e * O;
        A.last_obs[n0 * O + idx] = obsT[j * E_ + e];
    }
}

// per-step path: positions rows from_row .. max_steps repeat row from_row - 1
__global__ void fill_positions_kernel(float2* pos, int64_t N, int64_t from_row, int64_t max_steps) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const float2 p = pos[(from_row - 1) * N + i];
    for (int64_t r = from_row; r <= max_steps; ++r) pos[r * N + i] = p;
}

}  // namespace mr

using namespace mr;

static int eval_fused(mr_env* env, const EvalArgs& base, cudaStream_t s) {
    const size_t smem = (smem_w_floats(base.O) + EV_WARPS * (MAX_OBS * EV_E + 128 * EV_E)) * sizeof(float);
    static OncePerDevice once;
    if (once.first())
        MR_CUDA(cudaFuncSetAttribute(point_eval_kernel<EV_WARPS, EV_E>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     100 * 1024));
    const int64_t warps = (env->n + EV_E - 1) / EV_E;
    const int blocks = (int)((warps + EV_WARPS - 1) / EV_WARPS);
    EvalArgs A = base;
    MR_CUDA(cudaMallocAsync((void**)&A.warp_steps, (size_t)warps * sizeof(int32_t), s));
    for (int phase = 1; phase <= 2; ++phase) {
        A.phase = phase;
        point_eval_kernel<EV_WARPS, EV_E><<<blocks, EV_WARPS * 32, smem, s>>>(A);
        MR_CHECK_LAUNCH();
    }
    MR_CUDA(cudaFreeAsync(A.warp_steps, s));
    return MR_OK;
}

static int eval_per_step(mr_env* env, const EvalArgs& base, cudaStream_t s) {
    const int64_t N = env->n;
    const int O = base.O;
    // scratch for the env step's outputs and the per-env record counts, released on the stream at the end
    char* scratch = nullptr;
    size_t off = 0;
    auto carve = [&](size_t bytes) { const size_t at = off; off += (bytes + 255) & ~size_t(255); return at; };
    const size_t o_act = carve(N * 8), o_rew = carve(N * 4), o_ret = carve(N * 8), o_len = carve(N * 4),
                 o_cnt = carve(N * 4), o_done = carve(N), o_trunc = carve(N), o_met = carve(8);
    MR_CUDA(cudaMallocAsync((void**)&scratch, off, s));
    MR_CUDA(cudaMemsetAsync(scratch + o_cnt, 0, N * 4, s));
    MR_CUDA(cudaMemsetAsync(scratch + o_met, 0, 8, s));

    const size_t smem = (smem_w_floats(O) + ES_WARPS * (MAX_OBS * ES_E + 128 * ES_E)) * sizeof(float);
    static OncePerDevice once;
    if (once.first())
        MR_CUDA(cudaFuncSetAttribute(mr::eval_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    const int64_t tiles = (N + ES_E - 1) / ES_E;
    const int blocks = (int)std::min<int64_t>((tiles + ES_WARPS - 1) / ES_WARPS, (int64_t)sm_count() * 2);
    EvalStepArgs A;
    A.params = base.params; A.O = O; A.N = N; A.E = base.E; A.stochastic = base.stochastic;
    A.obs = base.last_obs; A.act = (float*)(scratch + o_act);
    A.done = (const uint8_t*)(scratch + o_done); A.ep_ret_n = (const double*)(scratch + o_ret);
    A.ep_len_n = (const int32_t*)(scratch + o_len);
    A.counts = (int32_t*)(scratch + o_cnt); A.n_met = (unsigned long long*)(scratch + o_met);
    A.ep_r = base.ep_r; A.ep_l = base.ep_l; A.ep_t = base.ep_t;
    A.seed = base.seed; A.noise_offset = base.noise_offset; A.env_offset = base.env_offset;

    // envs with a positive target: (E + i) // N > 0  <=>  i >= N - E
    const unsigned long long need = (unsigned long long)std::min<int64_t>(base.E, N);
    unsigned long long met = 0;
    int rc = MR_OK;
    int64_t t = 0;
    for (;; ++t) {
        A.t = t;
        mr::eval_step_kernel<<<blocks, ES_WARPS * 32, smem, s>>>(A);
        count_launch();
        cudaError_t e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaMemcpyAsync(&met, A.n_met, 8, cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) {
            set_error("evaluation step %lld: %s", (long long)t, cudaGetErrorString(e));
            rc = MR_ERR_CUDA;
            break;
        }
        if (met >= need || t == base.max_steps) break;
        rc = mr_env_step(env, A.act, base.last_obs, (float*)(scratch + o_rew), (uint8_t*)(scratch + o_done),
                         (uint8_t*)(scratch + o_trunc), nullptr, (double*)(scratch + o_ret),
                         (int32_t*)(scratch + o_len), s);
        if (rc != MR_OK) break;
    }
    cudaFreeAsync(scratch, s);
    if (rc != MR_OK) return rc;
    const unsigned long long S = (unsigned long long)t;
    const int short_of_target = met < need ? 1 : 0;
    MR_CUDA(cudaMemcpyAsync(base.S, &S, 8, cudaMemcpyHostToDevice, s));
    MR_CUDA(cudaMemcpyAsync(base.status, &short_of_target, sizeof(int), cudaMemcpyHostToDevice, s));
    MR_CUDA(cudaStreamSynchronize(s));   // the two host words live on this stack frame
    return MR_OK;
}

extern "C" int mr_evaluate(mr_env* env, const float* params, int deterministic, int64_t n_episodes, int64_t max_steps,
                           uint64_t seed, uint64_t noise_offset, int64_t env_offset, float* last_obs, double* ep_r,
                           int32_t* ep_l, int64_t* ep_t, int64_t* steps_taken, int* status, void* stream) {
    MR_REQUIRE(env && params && last_obs && steps_taken && status, "NULL argument");
    MR_REQUIRE(n_episodes >= 0 && max_steps >= 0, "n_episodes and max_steps must not be negative");
    MR_REQUIRE(n_episodes == 0 || (ep_r && ep_l && ep_t), "NULL episode record array");
    const int O = mr_env_obs_dim(env);
    MR_REQUIRE(O <= MAX_OBS, "the policy kernels take observations of at most 32 floats");
    cudaStream_t s = (cudaStream_t)stream;
    DeviceGuard guard(env->device);
    EvalArgs A;
    A.st = env->point;
    A.cfg = env->cfg;
    A.params = params;
    A.O = O;
    A.N = env->n;
    A.E = n_episodes;
    A.max_steps = max_steps;
    A.phase = 1;
    A.stochastic = deterministic ? 0 : 1;
    A.last_obs = last_obs;
    A.ep_r = ep_r; A.ep_l = ep_l; A.ep_t = ep_t;
    A.warp_steps = nullptr;
    A.S = reinterpret_cast<unsigned long long*>(steps_taken);
    A.status = status;
    A.seed = seed; A.noise_offset = noise_offset; A.env_offset = env_offset;
    if (env->kind == MR_ENV_POINT && env->cfg.obs_flags == 0 && env->cfg.haz.num == 0) {
        MR_CUDA(cudaMemsetAsync(steps_taken, 0, sizeof(int64_t), s));
        MR_CUDA(cudaMemsetAsync(status, 0, sizeof(int), s));
        return eval_fused(env, A, s);
    }
    return eval_per_step(env, A, s);
}

// Per-step path (the car, point envs with optional keys): per step, eval_step_kernel (forward + sample for every env,
// with no episode to record) then the masked env step, which leaves envs whose loop has ended untouched and does the
// waypoint bookkeeping itself -- it is the kernel that holds the car's contact scratch, which the post-switch get_obs()
// row needs.  The loop reads the device count of finished envs every WP_POLL steps: each read synchronises the stream,
// which costs about as much as a step of a few thousand envs, while a late stop costs at most WP_POLL - 1 pairs of
// launches whose threads all return at once.
constexpr int64_t WP_POLL = 16;

static int waypoints_per_step(mr_env* env, const float* params, int stochastic, const float* wp, int K,
                              int64_t max_steps, uint64_t seed, uint64_t noise_offset, int64_t env_offset,
                              float* last_obs, int32_t* arrival, double* ret, int32_t* steps, float* pos,
                              cudaStream_t s) {
    const int64_t N = env->n;
    const int O = mr_env_obs_dim(env);
    char* scratch = nullptr;
    size_t off = 0;
    auto carve = [&](size_t bytes) { const size_t at = off; off += (bytes + 255) & ~size_t(255); return at; };
    const size_t o_act = carve(N * 8), o_cur = carve(N * 4), o_done = carve(N), o_fin = carve(8);
    MR_CUDA(cudaMallocAsync((void**)&scratch, off, s));
    MR_CUDA(cudaMemsetAsync(scratch + o_cur, 0, off - o_cur, s));   // cursors, eval_step_kernel's done flags, count

    const size_t smem = (smem_w_floats(O) + ES_WARPS * (MAX_OBS * ES_E + 128 * ES_E)) * sizeof(float);
    static OncePerDevice once;
    if (once.first())
        MR_CUDA(cudaFuncSetAttribute(mr::eval_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    const int64_t tiles = (N + ES_E - 1) / ES_E;
    const int blocks = (int)std::min<int64_t>((tiles + ES_WARPS - 1) / ES_WARPS, (int64_t)sm_count() * 2);
    EvalStepArgs A{};
    A.params = params; A.O = O; A.N = N; A.E = 0; A.stochastic = stochastic;
    A.obs = last_obs; A.act = (float*)(scratch + o_act);
    A.done = (const uint8_t*)(scratch + o_done);   // all zero: no episode ever ends (no reset, no time limit)
    A.seed = seed; A.noise_offset = noise_offset; A.env_offset = env_offset;

    WaypointStep w;
    w.wp = wp; w.K = K; w.max_steps = max_steps;
    w.cursor = (int32_t*)(scratch + o_cur); w.steps = steps; w.ret = ret; w.arrival = arrival; w.pos = pos;
    w.n_finished = (unsigned long long*)(scratch + o_fin);

    int rc = env_set_goals(env, nullptr, wp, 2 * (int64_t)K, last_obs, s);
    unsigned long long finished = 0;
    int64_t t = 0;
    for (; rc == MR_OK && t < max_steps; ++t) {
        A.t = t;
        mr::eval_step_kernel<<<blocks, ES_WARPS * 32, smem, s>>>(A);
        count_launch();
        w.t = t;
        rc = env_step_waypoints(env, A.act, last_obs, w, s);
        if (rc == MR_OK && (t + 1) % WP_POLL == 0) {
            cudaError_t e = cudaMemcpyAsync(&finished, w.n_finished, 8, cudaMemcpyDeviceToHost, s);
            if (e == cudaSuccess) e = cudaStreamSynchronize(s);
            if (e != cudaSuccess) {
                set_error("waypoint step %lld: %s", (long long)t, cudaGetErrorString(e));
                rc = MR_ERR_CUDA;
            } else if (finished >= (unsigned long long)N) {
                ++t;
                break;
            }
        }
    }
    if (rc == MR_OK && pos && t < max_steps) {   // rows 0 .. t are written
        fill_positions_kernel<<<ceil_div(N, 128), 128, 0, s>>>(reinterpret_cast<float2*>(pos), N, t + 1, max_steps);
        count_launch();
    }
    cudaFreeAsync(scratch, s);
    if (rc != MR_OK) return rc;
    MR_CHECK_LAUNCH();
    return MR_OK;
}

extern "C" int mr_follow_waypoints(mr_env* env, const float* params, int deterministic, const float* waypoints,
                                   int K, int64_t max_steps, uint64_t seed, uint64_t noise_offset, int64_t env_offset,
                                   float* last_obs, int32_t* arrival, double* ret, int32_t* steps_taken,
                                   float* positions, void* stream) {
    MR_REQUIRE(env && params && waypoints && last_obs && arrival && ret && steps_taken, "NULL argument");
    MR_REQUIRE(K >= 1, "K must be at least 1");
    MR_REQUIRE(max_steps >= 1 && max_steps <= INT32_MAX, "max_steps must be in 1 .. 2^31 - 1");
    MR_REQUIRE(!env->cfg.terminate_on_goal && env->cfg.time_limit <= 0,
               "mr_follow_waypoints needs an env created with terminate_on_goal = 0 and no time limit (its "
               "auto-reset would draw a random goal)");
    const int O = mr_env_obs_dim(env);
    MR_REQUIRE(O <= MAX_OBS, "the policy kernels take observations of at most 32 floats");
    cudaStream_t s = (cudaStream_t)stream;
    DeviceGuard guard(env->device);
    const int64_t N = env->n;
    MR_CUDA(cudaMemsetAsync(arrival, 0xff, (size_t)N * K * sizeof(int32_t), s));   // -1: not reached
    MR_CUDA(cudaMemsetAsync(ret, 0, (size_t)N * sizeof(double), s));
    MR_CUDA(cudaMemsetAsync(steps_taken, 0, (size_t)N * sizeof(int32_t), s));
    const int stochastic = deterministic ? 0 : 1;
    if (env->kind != MR_ENV_POINT || env->cfg.obs_flags != 0 || env->cfg.haz.num != 0)
        return waypoints_per_step(env, params, stochastic, waypoints, K, max_steps, seed, noise_offset, env_offset,
                                  last_obs, arrival, ret, steps_taken, positions, s);
    WaypointArgs A;
    A.st = env->point; A.cfg = env->cfg; A.params = params; A.O = O; A.K = K; A.N = N; A.max_steps = max_steps;
    A.stochastic = stochastic; A.wp = waypoints; A.last_obs = last_obs; A.arrival = arrival; A.ret = ret;
    A.steps = steps_taken; A.pos = reinterpret_cast<float2*>(positions);
    A.seed = seed; A.noise_offset = noise_offset; A.env_offset = env_offset;
    const size_t smem = (smem_w_floats(O) + EV_WARPS * (MAX_OBS * EV_E + 128 * EV_E)) * sizeof(float);
    static OncePerDevice once;
    if (once.first())
        MR_CUDA(cudaFuncSetAttribute(point_waypoint_kernel<EV_WARPS, EV_E>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     100 * 1024));
    const int64_t warps = (N + EV_E - 1) / EV_E;
    point_waypoint_kernel<EV_WARPS, EV_E><<<(int)((warps + EV_WARPS - 1) / EV_WARPS), EV_WARPS * 32, smem, s>>>(A);
    MR_CHECK_LAUNCH();
    return MR_OK;
}
