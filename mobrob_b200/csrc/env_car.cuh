// Per-environment step / reset logic of the car goal env (CarEnv, src/mobrob/envs/wrapper.py:308-326)
// under the same wrapper stack as the point env (see env_point.cuh for the restated semantics).
#pragma once

#include "car_dyn.cuh"
#include "env_point.cuh"

namespace mr {

constexpr int CAR_STATE_DIM = 30;  // qpos(13) qvel(11) ctrl(2) goal(2) elapsed(1) ep_ret(1)

struct CarHot {
    car::State s;
    float cx, cz;  // data.ctrl (left, right motor)
    float gx, gy;
    int elapsed;
    double ep_ret;
};

// HBM layout: NSTATE fp64 component arrays [k][N] + the same small arrays as the point env.
struct CarSoA {
    int64_t n;
    double* st;  // [car::NSTATE][n]
    float2* ctrl;
    float2* goal;
    int32_t* elapsed;
    double* ep_ret;
    EnvCold cold;
    int contacts;

    static size_t align_up(size_t x) { return (x + 255) & ~size_t(255); }
    static size_t slab_bytes(int64_t n) {
        return align_up(n * 8 * car::NSTATE) + 2 * align_up(n * 8) + align_up(n * 4) + align_up(n * 8) +
               2 * align_up(n * 32) + 4 * align_up(n * 8) + align_up(32);
    }
    void carve(void* slab, int64_t n_) {
        n = n_;
        contacts = 1;
        char* p = static_cast<char*>(slab);
        auto take = [&](size_t bytes) { char* r = p; p += align_up(bytes); return r; };
        st = (double*)take(n * 8 * car::NSTATE);
        ctrl = (float2*)take(n * 8); goal = (float2*)take(n * 8);
        elapsed = (int32_t*)take(n * 4);
        ep_ret = (double*)take(n * 8);
        cold.pcg_init = (uint64_t*)take(n * 32); cold.pcg_goal = (uint64_t*)take(n * 32);
        cold.engine_seed = (int64_t*)take(n * 8);
        cold.body_xy = (float2*)take(n * 8);
        cold.psi0 = (double*)take(n * 8);
        cold.counts = (int32_t*)take(n * 8);
        cold.spaces = (const float*)take(32);
    }
    __device__ __forceinline__ CarHot load(int64_t i) const {
        CarHot h;
        double* d = reinterpret_cast<double*>(&h.s);
#pragma unroll
        for (int k = 0; k < car::NSTATE; ++k) d[k] = st[(int64_t)k * n + i];
        float2 c = ctrl[i], g = goal[i];
        h.cx = c.x; h.cz = c.y; h.gx = g.x; h.gy = g.y;
        h.elapsed = elapsed[i];
        h.ep_ret = ep_ret[i];
        return h;
    }
    __device__ __forceinline__ void store(int64_t i, const CarHot& h) const {
        const double* d = reinterpret_cast<const double*>(&h.s);
#pragma unroll
        for (int k = 0; k < car::NSTATE; ++k) st[(int64_t)k * n + i] = d[k];
        ctrl[i] = make_float2(h.cx, h.cz);
        goal[i] = make_float2(h.gx, h.gy);
        elapsed[i] = h.elapsed;
        ep_ret[i] = h.ep_ret;
    }
};

// see point_reset
template <bool HAZ = false>
__host__ __device__ inline void car_reset(CarHot& h, const EnvCold& cold, int64_t i, bool full,
                                          const HazardCfg* hz = nullptr) {
    if (full) {
        // Engine.reset() once (wrapper.py:190); CarEnv.set_pos only rewrites qpos[0:2] (wrapper.py:320-326)
        int64_t seed = cold.engine_seed[i] + 1;
        cold.engine_seed[i] = seed;
        Pcg64 g = load_pcg(cold.pcg_init, i);
        float x = (float)g.uniform((double)cold.spaces[0], (double)cold.spaces[2]);
        float y = (float)g.uniform((double)cold.spaces[1], (double)cold.spaces[3]);
        store_pcg(cold.pcg_init, i, g);
        double heading;
        if constexpr (HAZ) heading = hazard_reset_heading(*hz, (uint32_t)seed, i);
        else heading = engine_heading((uint32_t)seed);
        car::State& s = h.s;
        s.p[0] = (double)x; s.p[1] = (double)y; s.p[2] = 0.1;  // body pos z (car.xml:12)
        double sh, ch;
        sincos(0.5 * heading, &sh, &ch);
        s.q[0] = ch; s.q[1] = 0.0; s.q[2] = 0.0; s.q[3] = sh;  // rot2quat (world.py:52-54)
#pragma unroll
        for (int k = 0; k < 3; ++k) { s.v[k] = 0.0; s.w[k] = 0.0; s.wb[k] = 0.0; }
        s.th[0] = s.th[1] = s.s[0] = s.s[1] = 0.0;
        s.qb[0] = 1.0; s.qb[1] = s.qb[2] = s.qb[3] = 0.0;
        h.cx = h.cz = 0.f;
        cold.body_xy[i] = make_float2(x, y);
        cold.psi0[i] = heading;
        cold.counts[2 * i + 1] += 1;
    }
    Pcg64 g = load_pcg(cold.pcg_goal, i);
    h.gx = (float)g.uniform((double)cold.spaces[4], (double)cold.spaces[6]);
    h.gy = (float)g.uniform((double)cold.spaces[5], (double)cold.spaces[7]);
    store_pcg(cold.pcg_goal, i, g);
    h.elapsed = 0;
    h.ep_ret = 0.0;
    cold.counts[2 * i] += 1;
}

using CarExt = ObsExt<13, 11>;
constexpr int CAR_OBS_PRE = 15;

// data.qpos = free joint (pos, quat) + wheel angles + rear ball quat; data.qvel = free joint (linear world, angular
// body) + wheel rates + ball angular velocity: the order of mr_env_get_state's reference view.
// The lidar drops the goal's height (engine.py ego_xy): R^T (goal_x - p_x, goal_y - p_y, -p_z), not goal_compass's
// vector to the goal body at GOAL_Z -- the two differ once the chassis tilts.
__host__ __device__ inline void car_obs_ext(const CarHot& h, CarExt& x) {
    const car::State& s = h.s;
    x.ctrl[0] = h.cx; x.ctrl[1] = h.cz;
    double R[9], e[3];
    car::quat2mat(s.q, R);
    const double dv[3] = {(double)h.gx - s.p[0], (double)h.gy - s.p[1], -s.p[2]};
    car::mat3tv(R, dv, e);
    x.lidar_x = e[0];
    x.lidar_y = e[1];
    x.goal_dist = (float)exp(-point::dist2((double)h.gx, (double)h.gy, s.p[0], s.p[1]));
#pragma unroll
    for (int k = 0; k < 3; ++k) { x.qpos[k] = (float)s.p[k]; x.qvel[k] = (float)s.v[k]; x.qvel[3 + k] = (float)s.w[k]; x.qvel[8 + k] = (float)s.wb[k]; }
#pragma unroll
    for (int k = 0; k < 4; ++k) { x.qpos[3 + k] = (float)s.q[k]; x.qpos[9 + k] = (float)s.qb[k]; }
    x.qpos[7] = (float)s.th[0]; x.qpos[8] = (float)s.th[1];
    x.qvel[6] = (float)s.s[0]; x.qvel[7] = (float)s.s[1];
}

// the hazards_lidar block of the car at its current pose: R^T (h_x - p_x, h_y - p_y, -p_z), as car_obs_ext's goal
__host__ __device__ inline void car_hazards_lidar(float* dst, const CarHot& h, const EnvCfg& cfg, int64_t i) {
    double R[9];
    car::quat2mat(h.s.q, R);
    const double m[6] = {R[0], R[3], R[6], R[1], R[4], R[7]};
    hazards_lidar(dst, cfg.haz.pos + i * cfg.haz.num, cfg.haz.num, m, h.s.p[0], h.s.p[1], h.s.p[2], cfg.lidar);
}

// see point_env_step
template <bool HAZ = false>
__host__ __device__ inline StepResult car_env_step(const car::Consts& K, CarHot& h, const EnvCold& cold, int64_t i,
                                          float a0, float a1, const EnvCfg& cfg, bool contacts, float* obs,
                                          float* term_obs, const car::Scratch& S, CarExt* ext = nullptr,
                                          CarExt* term_ext = nullptr, float* haz_obs = nullptr,
                                          float* haz_term = nullptr) {
    StepResult r;
    h.cx = fminf(fmaxf(a0, -1.f), 1.f);
    h.cz = fminf(fmaxf(a1, -1.f), 1.f);
    const double prevx = h.s.p[0], prevy = h.s.p[1];
#pragma unroll 1
    for (int k = 0; k < car::FRAME_SKIP; ++k) car::substep(K, h.s, (double)h.cx, (double)h.cz, contacts, S, k > 0);
    const double gx = (double)h.gx, gy = (double)h.gy;
    const double dprev = point::dist2(gx, gy, prevx, prevy);
    const double dcur = point::dist2(gx, gy, h.s.p[0], h.s.p[1]);
    r.reach = dcur < REACH_RADIUS;
    double reward = rn::sub(dprev, dcur);
    if (r.reach) reward = rn::add(reward, REACH_BONUS);
    h.elapsed += 1;
    const bool term = r.reach && cfg.terminate_on_goal;
    const bool tl = cfg.time_limit > 0 && h.elapsed >= cfg.time_limit;
    r.done = term || tl;
    r.trunc = tl && !term;
    h.ep_ret = rn::add(h.ep_ret, reward);
    r.reward = reward;
    r.rew = (float)reward;
    r.ep_r = h.ep_ret;
    r.ep_l = h.elapsed;
    car::sensors(K, h.s, (double)h.cx, (double)h.cz, h.gx, h.gy, contacts, obs, S);
    if (ext) car_obs_ext(h, *ext);
    if constexpr (HAZ) {
        if (cfg.haz.flags & HAZ_CONSTRAIN)
            cfg.haz.cost_out[i] = hazard_cost(cfg.haz, cfg.haz.pos + i * cfg.haz.num, h.s.p[0], h.s.p[1]);
    }
    if (r.done) {
        for (int k = 0; k < car::OBS; ++k) term_obs[k] = obs[k];
        if (ext) *term_ext = *ext;
        if constexpr (HAZ) {
            if (haz_term) car_hazards_lidar(haz_term, h, cfg, i);
        }
        car_reset<HAZ>(h, cold, i, !r.reach, &cfg.haz);
        car::sensors(K, h.s, (double)h.cx, (double)h.cz, h.gx, h.gy, contacts, obs, S);
        if (ext) car_obs_ext(h, *ext);
    }
    if constexpr (HAZ) {
        if (haz_obs) car_hazards_lidar(haz_obs, h, cfg, i);
    }
    return r;
}

}  // namespace mr
