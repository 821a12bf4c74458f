// Device side of the waypoint kernels shared by waypoints.cu and waypoints_hazards.cu: the car's post-switch get_obs()
// row, the reference loop's per-step bookkeeping and the car's masked step.
#pragma once

#include "env_state.cuh"

namespace mr {

constexpr int WP_THREADS = 128;

template <bool HAZ>
__device__ __forceinline__ void car_goal_obs_row(const car::Consts& K, const CarSoA& st, const CarHot& h, int64_t i,
                                                 const EnvCfg& cfg, float* __restrict__ obs, const car::Scratch& S) {
    float o[car::OBS];
    car::sensors(K, h.s, (double)h.cx, (double)h.cz, h.gx, h.gy, st.contacts != 0, o, S);
    CarExt x;
    car_obs_ext(h, x);
    float* row = obs + i * row_dim<HAZ>(car::OBS, 13, 11, cfg);
    emit_obs_row<car::OBS, CAR_OBS_PRE, 13, 11, HAZ>(row, o, x, cfg.obs_flags, cfg.lidar);
    if constexpr (HAZ) {
        if (float* hb = hazards_block<HAZ, CAR_OBS_PRE>(row, cfg)) car_hazards_lidar(hb, h, cfg, i);
    }
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

// see point_waypoint_step_kernel
template <bool HAZ>
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
        float* haz_obs = nullptr;
        if constexpr (HAZ) haz_obs = hazards_block<HAZ, CAR_OBS_PRE>(obs + i * row_dim<HAZ>(car::OBS, 13, 11, cfg), cfg);
        const StepResult r = car_env_step<HAZ>(K, h, st.cold, i, a.x, a.y, cfg, st.contacts != 0, o, tobs, S, &x, &tx,
                                               haz_obs);
        if (waypoint_after_step(w, i, r, h.gx, h.gy)) {
            car_goal_obs_row<HAZ>(K, st, h, i, cfg, obs, S);
        } else {
            const int O = row_dim<HAZ>(car::OBS, 13, 11, cfg);
            emit_obs_row<car::OBS, CAR_OBS_PRE, 13, 11, HAZ>(obs + i * O, o, x, cfg.obs_flags, cfg.lidar);
        }
        st.store(i, h);
    }
    waypoint_pos(w, st.n, i, w.t + 1, st.st[i], st.st[st.n + i]);
}

// car_waypoint_step_kernel<true> (waypoints_hazards.cu)
int car_waypoint_step_hazards(mr_env* env, const float2* act, float* obs, const WaypointStep& w, cudaStream_t s);

}  // namespace mr
