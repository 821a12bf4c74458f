// Goal changes on the device: EnvWrapper.set_goal for a batch (mr_env_set_goals), and the per-step path of
// mr_follow_waypoints (evaluate.cu) -- a masked env step for either robot and any observation row: envs whose loop
// has ended are not touched, the others take env.step and then the reference loop's bookkeeping.
// These kernels live apart from env.cu so that its kernels keep their inlining: one more caller of car_env_step or
// car::sensors there makes nvcc outline the step from car_step_ext_kernel.
#include "waypoints.cuh"

namespace mr {

// EnvWrapper.set_goal (wrapper.py:115-117) then get_obs(): the goal changes, nothing else does (the ctrl stays stale).
// emit_obs_row with obs_flags = 0 writes the default row.  HAZ: the env has hazards (EnvCfg::haz.num > 0).
template <bool HAZ>
__device__ __forceinline__ void point_goal_obs_row(const PointState& st, const PointHot& h, int64_t i, const EnvCfg& cfg,
                                                   float* __restrict__ obs) {
    float o[point::OBS];
    point::sensors(h.d, (double)h.cx, (double)h.cz, h.gx, h.gy, o);
    PointExt x;
    double s, c;
    sincos(h.d.psi, &s, &c);
    point_obs_ext(h, st.cold, i, c, s, x);
    float* row = obs + i * row_dim<HAZ>(point::OBS, 3, 3, cfg);
    emit_obs_row<point::OBS, POINT_OBS_PRE, 3, 3, HAZ>(row, o, x, cfg.obs_flags, cfg.lidar);
    if constexpr (HAZ) {
        if (float* hb = hazards_block<HAZ, POINT_OBS_PRE>(row, cfg)) point_hazards_lidar(hb, h, cfg, i);
    }
}

template <bool HAZ>
__global__ void __launch_bounds__(WP_THREADS)
point_set_goals_kernel(PointState st, const uint8_t* __restrict__ mask, const float* __restrict__ goals,
                       int64_t goal_stride, float* __restrict__ obs, EnvCfg cfg) {
    const int64_t i = (int64_t)blockIdx.x * WP_THREADS + threadIdx.x;
    if (i >= st.n || (mask && !mask[i])) return;
    PointHot h = st.load(i);
    h.gx = goals[i * goal_stride];
    h.gy = goals[i * goal_stride + 1];
    st.store(i, h);
    if (obs) point_goal_obs_row<HAZ>(st, h, i, cfg, obs);
}

template <bool HAZ>
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
    if (obs) car_goal_obs_row<HAZ>(K, st, h, i, cfg, obs, S);
}

// masked env step of mr_follow_waypoints (any observation row): envs whose loop has ended are left untouched
template <bool HAZ>
__global__ void __launch_bounds__(WP_THREADS)
point_waypoint_step_kernel(PointState st, EnvCfg cfg, const float2* __restrict__ act, float* __restrict__ obs,
                           WaypointStep w) {
    const int64_t i = (int64_t)blockIdx.x * WP_THREADS + threadIdx.x;
    if (i >= st.n) return;
    PointHot h = st.load(i);
    if (w.t == 0) waypoint_pos(w, st.n, i, 0, h.d.px, h.d.py);
    if (waypoint_running(w, i)) {
        const int O = row_dim<HAZ>(point::OBS, 3, 3, cfg);
        const float2 a = act[i];
        float o[point::OBS], tobs[point::OBS];
        PointExt x, tx;
        const StepResult r = point_env_step<HAZ>(h, st.cold, i, a.x, a.y, cfg, o, tobs, &x, &tx,
                                                 hazards_block<HAZ, POINT_OBS_PRE>(obs + i * O, cfg));
        if (waypoint_after_step(w, i, r, h.gx, h.gy))
            point_goal_obs_row<HAZ>(st, h, i, cfg, obs);
        else
            emit_obs_row<point::OBS, POINT_OBS_PRE, 3, 3, HAZ>(obs + i * O, o, x, cfg.obs_flags, cfg.lidar);
        st.store(i, h);
    }
    waypoint_pos(w, st.n, i, w.t + 1, h.d.px, h.d.py);
}

int env_set_goals(mr_env* env, const uint8_t* mask, const float* goals, int64_t goal_stride, float* obs,
                  cudaStream_t s) {
    const bool haz = env->cfg.haz.num > 0;
    if (env->kind == MR_ENV_POINT) {
        auto kern = haz ? point_set_goals_kernel<true> : point_set_goals_kernel<false>;
        kern<<<ceil_div(env->n, WP_THREADS), WP_THREADS, 0, s>>>(env->point, mask, goals, goal_stride, obs, env->cfg);
    } else {
        static OncePerDevice once;
        if (once.first()) {
            MR_CUDA(cudaFuncSetAttribute(car_set_goals_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)CAR_SMEM));
            MR_CUDA(cudaFuncSetAttribute(car_set_goals_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)CAR_SMEM));
        }
        auto kern = haz ? car_set_goals_kernel<true> : car_set_goals_kernel<false>;
        kern<<<ceil_div(env->n, CAR_THREADS), CAR_THREADS, CAR_SMEM, s>>>(env->car, env->carK, mask, goals, goal_stride,
                                                                          obs, env->cfg);
    }
    MR_CHECK_LAUNCH();
    return MR_OK;
}

int env_step_waypoints(mr_env* env, const float* act, float* obs, const WaypointStep& w, cudaStream_t s) {
    const float2* a2 = reinterpret_cast<const float2*>(act);
    const bool haz = env->cfg.haz.num > 0;
    if (env->kind == MR_ENV_POINT) {
        auto kern = haz ? point_waypoint_step_kernel<true> : point_waypoint_step_kernel<false>;
        kern<<<ceil_div(env->n, WP_THREADS), WP_THREADS, 0, s>>>(env->point, env->cfg, a2, obs, w);
    } else {
        if (haz) return car_waypoint_step_hazards(env, a2, obs, w, s);
        static OncePerDevice once;
        if (once.first())
            MR_CUDA(cudaFuncSetAttribute(car_waypoint_step_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)CAR_SMEM));
        car_waypoint_step_kernel<false><<<ceil_div(env->n, CAR_THREADS), CAR_THREADS, CAR_SMEM, s>>>(
            env->car, env->carK, env->cfg, a2, obs, w);
    }
    MR_CHECK_LAUNCH();
    return MR_OK;
}

}  // namespace mr
