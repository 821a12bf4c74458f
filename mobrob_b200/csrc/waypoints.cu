// Goal changes on the device: EnvWrapper.set_goal for a batch (mr_env_set_goals), and the per-step path of
// mr_follow_waypoints (evaluate.cu) -- a masked env step for either robot and any observation row: envs whose loop
// has ended are not touched, the others take env.step and then the reference loop's bookkeeping.
// These kernels live apart from env.cu so that its kernels keep their inlining: one more caller of car_env_step or
// car::sensors there makes nvcc outline the step from car_step_ext_kernel.
#include "env_state.cuh"

namespace mr {

constexpr int WP_THREADS = 128;

// EnvWrapper.set_goal (wrapper.py:115-117) then get_obs(): the goal changes, nothing else does (the ctrl stays stale).
// emit_obs_row with obs_flags = 0 writes the default row.
__device__ __forceinline__ void point_goal_obs_row(const PointState& st, const PointHot& h, int64_t i, const EnvCfg& cfg,
                                                   float* __restrict__ obs) {
    float o[point::OBS];
    point::sensors(h.d, (double)h.cx, (double)h.cz, h.gx, h.gy, o);
    PointExt x;
    double s, c;
    sincos(h.d.psi, &s, &c);
    point_obs_ext(h, st.cold, i, c, s, x);
    emit_obs_row<point::OBS, POINT_OBS_PRE, 3, 3>(obs + i * obs_dim_ext(point::OBS, 3, 3, cfg.obs_flags, cfg.lidar.num_bins),
                                                  o, x, cfg.obs_flags, cfg.lidar);
}

__global__ void __launch_bounds__(WP_THREADS)
point_set_goals_kernel(PointState st, const uint8_t* __restrict__ mask, const float* __restrict__ goals,
                       int64_t goal_stride, float* __restrict__ obs, EnvCfg cfg) {
    const int64_t i = (int64_t)blockIdx.x * WP_THREADS + threadIdx.x;
    if (i >= st.n || (mask && !mask[i])) return;
    PointHot h = st.load(i);
    h.gx = goals[i * goal_stride];
    h.gy = goals[i * goal_stride + 1];
    st.store(i, h);
    if (obs) point_goal_obs_row(st, h, i, cfg, obs);
}

__device__ __forceinline__ void car_goal_obs_row(const car::Consts& K, const CarSoA& st, const CarHot& h, int64_t i,
                                                 const EnvCfg& cfg, float* __restrict__ obs, const car::Scratch& S) {
    float o[car::OBS];
    car::sensors(K, h.s, (double)h.cx, (double)h.cz, h.gx, h.gy, st.contacts != 0, o, S);
    CarExt x;
    car_obs_ext(h, x);
    emit_obs_row<car::OBS, CAR_OBS_PRE, 13, 11>(obs + i * obs_dim_ext(car::OBS, 13, 11, cfg.obs_flags, cfg.lidar.num_bins),
                                                o, x, cfg.obs_flags, cfg.lidar);
}

__global__ void __launch_bounds__(CAR_THREADS)
car_set_goals_kernel(CarSoA st, car::Consts K, const uint8_t* __restrict__ mask, const float* __restrict__ goals,
                     int64_t goal_stride, float* __restrict__ obs, EnvCfg cfg) {
    MR_CAR_SCRATCH();
    const int64_t i = (int64_t)blockIdx.x * CAR_THREADS + threadIdx.x;
    if (i >= st.n || (mask && !mask[i])) return;
    CarHot h = st.load(i);
    h.gx = goals[i * goal_stride];
    h.gy = goals[i * goal_stride + 1];
    st.store(i, h);
    if (obs) car_goal_obs_row(K, st, h, i, cfg, obs, S);
}

// What the reference loop of mr_follow_waypoints does after env.step: count the step and its reward; on reaching
// the current waypoint record the arrival and set_goal the next one (returns true: the caller re-forms the row as
// get_obs()).  The env's loop ends at its last waypoint or at max_steps.
__device__ __forceinline__ bool waypoint_after_step(const WaypointStep& w, int64_t i, const StepResult& r, float& gx,
                                                    float& gy) {
    const int32_t t = w.steps[i] + 1;
    w.steps[i] = t;
    w.ret[i] = rn::add(w.ret[i], r.reward);
    int32_t k = w.cursor[i];
    bool switched = false;
    if (r.reach) {
        w.arrival[i * w.K + k] = t;
        if (++k < w.K) {
            gx = w.wp[(i * w.K + k) * 2];
            gy = w.wp[(i * w.K + k) * 2 + 1];
            switched = true;
        }
        w.cursor[i] = k;
    }
    if (k >= w.K || t >= w.max_steps) atomicAdd(w.n_finished, 1ull);
    return switched;
}

__device__ __forceinline__ bool waypoint_running(const WaypointStep& w, int64_t i) {
    return w.cursor[i] < w.K && w.steps[i] < w.max_steps;
}

__device__ __forceinline__ void waypoint_pos(const WaypointStep& w, int64_t n, int64_t i, int64_t row, double x,
                                             double y) {
    if (w.pos) reinterpret_cast<float2*>(w.pos)[row * n + i] = make_float2((float)x, (float)y);
}

// masked env step of mr_follow_waypoints (any observation row): envs whose loop has ended are left untouched
__global__ void __launch_bounds__(WP_THREADS)
point_waypoint_step_kernel(PointState st, EnvCfg cfg, const float2* __restrict__ act, float* __restrict__ obs,
                           WaypointStep w) {
    const int64_t i = (int64_t)blockIdx.x * WP_THREADS + threadIdx.x;
    if (i >= st.n) return;
    PointHot h = st.load(i);
    if (w.t == 0) waypoint_pos(w, st.n, i, 0, h.d.px, h.d.py);
    if (waypoint_running(w, i)) {
        const int O = obs_dim_ext(point::OBS, 3, 3, cfg.obs_flags, cfg.lidar.num_bins);
        const float2 a = act[i];
        float o[point::OBS], tobs[point::OBS];
        PointExt x, tx;
        const StepResult r = point_env_step(h, st.cold, i, a.x, a.y, cfg, o, tobs, &x, &tx);
        if (waypoint_after_step(w, i, r, h.gx, h.gy))
            point_goal_obs_row(st, h, i, cfg, obs);
        else
            emit_obs_row<point::OBS, POINT_OBS_PRE, 3, 3>(obs + i * O, o, x, cfg.obs_flags, cfg.lidar);
        st.store(i, h);
    }
    waypoint_pos(w, st.n, i, w.t + 1, h.d.px, h.d.py);
}

// see point_waypoint_step_kernel
__global__ void __launch_bounds__(CAR_THREADS)
car_waypoint_step_kernel(CarSoA st, car::Consts K, EnvCfg cfg, const float2* __restrict__ act, float* __restrict__ obs,
                         WaypointStep w) {
    MR_CAR_SCRATCH();
    const int64_t i = (int64_t)blockIdx.x * CAR_THREADS + threadIdx.x;
    if (i >= st.n) return;
    if (w.t == 0) waypoint_pos(w, st.n, i, 0, st.st[i], st.st[st.n + i]);
    if (waypoint_running(w, i)) {
        CarHot h = st.load(i);
        const float2 a = act[i];
        float o[car::OBS], tobs[car::OBS];
        CarExt x, tx;
        const StepResult r = car_env_step(K, h, st.cold, i, a.x, a.y, cfg, st.contacts != 0, o, tobs, S, &x, &tx);
        if (waypoint_after_step(w, i, r, h.gx, h.gy)) {
            car_goal_obs_row(K, st, h, i, cfg, obs, S);
        } else {
            const int O = obs_dim_ext(car::OBS, 13, 11, cfg.obs_flags, cfg.lidar.num_bins);
            emit_obs_row<car::OBS, CAR_OBS_PRE, 13, 11>(obs + i * O, o, x, cfg.obs_flags, cfg.lidar);
        }
        st.store(i, h);
    }
    waypoint_pos(w, st.n, i, w.t + 1, st.st[i], st.st[st.n + i]);
}

int env_set_goals(mr_env* env, const uint8_t* mask, const float* goals, int64_t goal_stride, float* obs,
                  cudaStream_t s) {
    if (env->kind == MR_ENV_POINT) {
        point_set_goals_kernel<<<ceil_div(env->n, WP_THREADS), WP_THREADS, 0, s>>>(env->point, mask, goals, goal_stride,
                                                                                   obs, env->cfg);
    } else {
        static OncePerDevice once;
        if (once.first())
            MR_CUDA(cudaFuncSetAttribute(car_set_goals_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CAR_SMEM));
        car_set_goals_kernel<<<ceil_div(env->n, CAR_THREADS), CAR_THREADS, CAR_SMEM, s>>>(env->car, env->carK, mask, goals,
                                                                                          goal_stride, obs, env->cfg);
    }
    MR_CHECK_LAUNCH();
    return MR_OK;
}

int env_step_waypoints(mr_env* env, const float* act, float* obs, const WaypointStep& w, cudaStream_t s) {
    const float2* a2 = reinterpret_cast<const float2*>(act);
    if (env->kind == MR_ENV_POINT) {
        point_waypoint_step_kernel<<<ceil_div(env->n, WP_THREADS), WP_THREADS, 0, s>>>(env->point, env->cfg, a2, obs,
                                                                                       w);
    } else {
        static OncePerDevice once;
        if (once.first())
            MR_CUDA(cudaFuncSetAttribute(car_waypoint_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)CAR_SMEM));
        car_waypoint_step_kernel<<<ceil_div(env->n, CAR_THREADS), CAR_THREADS, CAR_SMEM, s>>>(
            env->car, env->carK, env->cfg, a2, obs, w);
    }
    MR_CHECK_LAUNCH();
    return MR_OK;
}

}  // namespace mr
