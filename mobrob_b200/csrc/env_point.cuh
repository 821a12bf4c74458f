// Per-environment step / reset logic of the point goal env, shared by the stand-alone
// VecEnv kernels (env.cu) and the fused rollout kernel (rollout.cu).
//
// Restates, per env: EnvWrapper.step/reward_fn/reached/reset (src/mobrob/envs/wrapper.py:
// 137-207), PointEnv.set_pos (wrapper.py:301-305), [GYM] TimeLimit (wrapper.py:568-569),
// [SB3] Monitor + DummyVecEnv auto-reset (src/mobrob/rl_control/ppo.py:37-48).
#pragma once

#include "point_dyn.cuh"

namespace mr {

// Engine's pseudo-lidar settings (config keys lidar_num_bins, lidar_max_dist, lidar_exp_gain, lidar_alias;
// lidar_type 'pseudo'), read by the goal_lidar block only.  32 bytes: the kernel parameters behind EnvCfg keep their
// 16-byte alignment, so the default kernels load them with the same instructions as without the lidar.
struct LidarCfg {
    int num_bins;
    int alias;          // 0 / 1
    double bin_size;    // 2 pi / num_bins, formed once on the host (make_lidar_cfg)
    double max_dist;    // <= 0: None (sensor = exp(-exp_gain * dist))
    double exp_gain;
};
constexpr double TWO_PI = 2.0 * 3.141592653589793;   // np.pi * 2

__host__ __device__ inline LidarCfg make_lidar_cfg(int num_bins, double max_dist, double exp_gain, int alias) {
    return LidarCfg{num_bins, alias ? 1 : 0, TWO_PI / num_bins, max_dist > 0.0 ? max_dist : 0.0, exp_gain};
}

struct EnvCfg {
    int time_limit;         // <= 0: no TimeLimit wrapper
    int terminate_on_goal;  // EnvWrapper(terminate_on_goal=...)
    point::K pk;            // integrator constants of the point robot (constant-bank operands)
    unsigned obs_flags;     // optional Engine.obs() keys (OBS_*); 0 = the configuration wrapper.py:293-317 builds
    LidarCfg lidar;         // OBS_GOAL_LIDAR
};

// Optional observation keys of Engine.obs() (flags src/mobrob/envs/mujoco_robots/robots/engine.py:125,140-142,
// values engine.py:1179-1180 and 1243-1248): goal_dist = exp(-|goal - pos|_xy), qpos / qvel = data.qpos / data.qvel,
// ctrl = data.ctrl (the clipped action of the last step), goal_lidar = the pseudo-lidar of the goal (engine.py:1092-1172,
// goal_lidar() below, LidarCfg::num_bins floats).  The flat row is the concatenation in SORTED key order
// (engine.py:1253-1259), so the extra keys are interleaved with the sensors:
//   accelerometer [ballangvel_rear ballquat_rear] | ctrl | goal_compass | goal_dist | goal_lidar | gyro magnetometer |
//   qpos | qvel | velocimeter
constexpr unsigned OBS_GOAL_DIST = 1u, OBS_QPOS = 2u, OBS_QVEL = 4u, OBS_CTRL = 8u, OBS_GOAL_LIDAR = 16u,
                   OBS_ALL_FLAGS = 31u;

template <int NQ, int NV>
struct ObsExt {
    float ctrl[2];
    float goal_dist;
    float qpos[NQ];
    float qvel[NV];
    double lidar_x, lidar_y;   // the goal's egocentric xy for goal_lidar: ((goal_x, goal_y, 0) - robot_pos) @ robot_mat
};

__host__ __device__ inline int obs_dim_ext(int base, int nq, int nv, unsigned f, int lidar_bins) {
    return base + ((f & OBS_CTRL) ? 2 : 0) + ((f & OBS_GOAL_DIST) ? 1 : 0) + ((f & OBS_GOAL_LIDAR) ? lidar_bins : 0) +
           ((f & OBS_QPOS) ? nq : 0) + ((f & OBS_QVEL) ? nv : 0);
}

// Engine.obs_lidar_pseudo (engine.py:1092-1172) over the goal envs' one object, the goal, at egocentric (ex, ey):
// c.num_bins floats at dst.  float64 like the reference, float32 on the store:
//   dist = |ex + i ey|, angle = atan2(ey, ex) % 2 pi, bin = int(angle / bin_size), bin_size = 2 pi / n,
//   sensor = exp(-exp_gain dist) (max_dist None) or max(0, max_dist - dist) / max_dist,
//   obs[bin] = max(obs[bin], sensor); with alias a = (angle - bin * bin_size) / bin_size:
//   obs[(bin + 1) % n] = max(., a sensor), then obs[(bin - 1) % n] = max(., (1 - a) sensor).
// The block is zero but for those (at most three) bins, which coincide for n <= 2: each update takes the value the
// earlier ones left at its index.  One deliberate deviation: angle / bin_size can round up to n (atan2 returns a tiny
// negative angle and % 2 pi rounds to 2 pi), where the reference raises IndexError; the bin is clamped to n - 1.
__host__ __device__ inline void goal_lidar(float* __restrict__ dst, double ex, double ey, const LidarCfg& c) {
    const int n = c.num_bins;
    const double dist = hypot(ex, ey);
    double angle = atan2(ey, ex);
    angle = angle < 0.0 ? angle + TWO_PI : angle + 0.0;   // Python's float %: in [0, 2 pi], -0 -> +0
    const double bin_size = c.bin_size;
    const double q = angle / bin_size;
    const int bin = q < (double)n ? (int)q : n - 1;
    const double left = c.max_dist - dist;
    const double sensor = c.max_dist > 0.0 ? (left > 0.0 ? left : 0.0) / c.max_dist : exp(-c.exp_gain * dist);
    int idx[3] = {bin, 0, 0};
    double val[3] = {sensor > 0.0 ? sensor : 0.0, 0.0, 0.0};
    int m = 1;
    if (c.alias) {
        const double alias = (angle - bin_size * bin) / bin_size;
        const double upd[3] = {0.0, alias * sensor, (1.0 - alias) * sensor};
        idx[1] = bin + 1 == n ? 0 : bin + 1;
        idx[2] = bin == 0 ? n - 1 : bin - 1;
#pragma unroll
        for (int k = 1; k < 3; ++k) {
            double cur = 0.0;
#pragma unroll
            for (int j = 0; j < k; ++j)
                if (idx[j] == idx[k]) cur = val[j];
            val[k] = upd[k] > cur ? upd[k] : cur;
        }
        m = 3;
    }
    for (int k = 0; k < n; ++k) dst[k] = 0.f;
#pragma unroll
    for (int k = 0; k < 3; ++k)
        if (k < m) dst[idx[k]] = (float)val[k];
}

// BASE floats of the default row, PRE of them in front of goal_compass (= in front of "ctrl")
template <int BASE, int PRE, int NQ, int NV>
__host__ __device__ __forceinline__ void emit_obs_row(float* __restrict__ dst, const float* base, const ObsExt<NQ, NV>& x, unsigned f,
                                                      const LidarCfg& lidar) {
    int k = 0;
#pragma unroll
    for (int j = 0; j < PRE; ++j) dst[k++] = base[j];
    if (f & OBS_CTRL) { dst[k++] = x.ctrl[0]; dst[k++] = x.ctrl[1]; }
    dst[k++] = base[PRE]; dst[k++] = base[PRE + 1];
    if (f & OBS_GOAL_DIST) dst[k++] = x.goal_dist;
    if (f & OBS_GOAL_LIDAR) { goal_lidar(dst + k, x.lidar_x, x.lidar_y, lidar); k += lidar.num_bins; }
#pragma unroll
    for (int j = PRE + 2; j < BASE - 3; ++j) dst[k++] = base[j];
    if (f & OBS_QPOS) {
#pragma unroll
        for (int j = 0; j < NQ; ++j) dst[k++] = x.qpos[j];
    }
    if (f & OBS_QVEL) {
#pragma unroll
        for (int j = 0; j < NV; ++j) dst[k++] = x.qvel[j];
    }
#pragma unroll
    for (int j = BASE - 3; j < BASE; ++j) dst[k++] = base[j];
}

// Arrays touched only by resets (and by the reference-view export).
struct EnvCold {
    uint64_t* pcg_init;    // [N][4] init_space stream
    uint64_t* pcg_goal;    // [N][4] goal_space stream
    int64_t* engine_seed;  // [N] Engine._seed
    float2* body_xy;       // [N] model.body_pos[robot][:2]
    double* psi0;          // [N] start heading (body quat)
    int32_t* counts;       // [N][2] (#resets, #full resets)
    const float* spaces;   // [8] init low (x, y), init high, goal low, goal high: EnvWrapper.init_space / goal_space
                           // (defaults wrapper.py:250-264; reset_init_space / reset_goal_space, wrapper.py:209-219)
};

struct PointHot {
    point::Dyn d;
    float cx, cz;  // data.ctrl (clipped action); survives goal-only resets
    float gx, gy;  // goal (float32, as drawn by Box.sample)
    int elapsed;   // TimeLimit._elapsed_steps == Monitor episode length
    double ep_ret; // Monitor episode return
};

struct StepResult {
    float rew;
    bool done, trunc, reach;
    double ep_r;
    int ep_l;
};

constexpr double REACH_RADIUS = 0.3;  // wrapper.py:203
constexpr double REACH_BONUS = 5.0;   // wrapper.py:151-152

__host__ __device__ __forceinline__ Pcg64 load_pcg(const uint64_t* p, int64_t i) {
    const ulonglong2* q = reinterpret_cast<const ulonglong2*>(p + 4 * i);
    ulonglong2 a = q[0], b = q[1];
    return Pcg64{a.x, a.y, b.x, b.y};
}
__host__ __device__ __forceinline__ void store_pcg(uint64_t* p, int64_t i, const Pcg64& g) {
    // the increment never changes
    *reinterpret_cast<ulonglong2*>(p + 4 * i) = make_ulonglong2(g.hi, g.lo);
}

// EnvWrapper.reset for one env.  full: re-place the robot (first reset, or goal not reached).
__host__ __device__ inline void point_reset(PointHot& h, const EnvCold& cold, int64_t i, bool full) {
    if (full) {
        // Engine.reset() (wrapper.py:190) then PointEnv.set_pos -> Engine.reset() again
        // (wrapper.py:302): the heading that survives is the one drawn with _seed + 2.
        int64_t seed = cold.engine_seed[i] + 2;
        cold.engine_seed[i] = seed;
        Pcg64 g = load_pcg(cold.pcg_init, i);
        // init_space.sample(): default extents / 2 (wrapper.py:250-256); float32 bounds, float64 arithmetic
        float x = (float)g.uniform((double)cold.spaces[0], (double)cold.spaces[2]);
        float y = (float)g.uniform((double)cold.spaces[1], (double)cold.spaces[3]);
        store_pcg(cold.pcg_init, i, g);
        double heading = engine_heading((uint32_t)seed);
        h.d.px = (double)x;
        h.d.py = (double)y;
        h.d.psi = heading;
        h.d.vx = h.d.vy = h.d.om = 0.0;  // new MjSim: qpos = qvel = ctrl = 0
        h.cx = h.cz = 0.f;
        cold.body_xy[i] = make_float2(x, y);
        cold.psi0[i] = heading;
        cold.counts[2 * i + 1] += 1;
    }
    Pcg64 g = load_pcg(cold.pcg_goal, i);
    h.gx = (float)g.uniform((double)cold.spaces[4], (double)cold.spaces[6]);  // goal_space: default extents (wrapper.py:258-264)
    h.gy = (float)g.uniform((double)cold.spaces[5], (double)cold.spaces[7]);
    store_pcg(cold.pcg_goal, i, g);
    h.elapsed = 0;
    h.ep_ret = 0.0;
    cold.counts[2 * i] += 1;
}

using PointExt = ObsExt<3, 3>;
constexpr int POINT_OBS_PRE = 3;

// qpos / qvel are the joint coordinates (two slides in the robot body's frame, one hinge), relative to the body
// pose PointEnv.set_pos wrote into the model (wrapper.py:301-305): the same view mr_env_get_state exports.
// c, s: cos / sin of the heading.  The robot frame is a pure yaw, so the lidar's egocentric goal is the compass's.
__host__ __device__ inline void point_obs_ext(const PointHot& h, const EnvCold& cold, int64_t i, double c, double s,
                                              PointExt& x) {
    x.ctrl[0] = h.cx; x.ctrl[1] = h.cz;
    const double gx = (double)h.gx - h.d.px, gy = (double)h.gy - h.d.py;
    x.lidar_x = fma(s, gy, c * gx);
    x.lidar_y = fma(-s, gx, c * gy);
    x.goal_dist = (float)exp(-point::dist2((double)h.gx, (double)h.gy, h.d.px, h.d.py));
    const float2 b = cold.body_xy[i];
    const double p0 = cold.psi0[i];
    double s0, c0;
    sincos(p0, &s0, &c0);
    const double dx = h.d.px - (double)b.x, dy = h.d.py - (double)b.y;
    x.qpos[0] = (float)(c0 * dx + s0 * dy);
    x.qpos[1] = (float)(-s0 * dx + c0 * dy);
    x.qpos[2] = (float)(h.d.psi - p0);
    x.qvel[0] = (float)(c0 * h.d.vx + s0 * h.d.vy);
    x.qvel[1] = (float)(-s0 * h.d.vx + c0 * h.d.vy);
    x.qvel[2] = (float)h.d.om;
}

// One VecEnv step of one env.  obs receives the row the VecEnv returns (post-reset when
// done); term_obs receives info["terminal_observation"] when done.  ext / term_ext (may be NULL): the optional keys
// of the same two observations.
__host__ __device__ inline StepResult point_env_step(PointHot& h, const EnvCold& cold, int64_t i,
                                            float a0, float a1, const EnvCfg& cfg, float* obs,
                                            float* term_obs, PointExt* ext = nullptr, PointExt* term_ext = nullptr) {
    StepResult r;
    h.cx = fminf(fmaxf(a0, -1.f), 1.f);  // engine.py:1401-1405
    h.cz = fminf(fmaxf(a1, -1.f), 1.f);
    const double prevx = h.d.px, prevy = h.d.py;  // _prev_pos == position before the step
    double hc, hs;  // cos / sin of the heading after the step
    point::substeps(cfg.pk, h.d, (double)h.cx, (double)h.cz, hc, hs);
    const double gx = (double)h.gx, gy = (double)h.gy;
    const double dprev = point::dist2(gx, gy, prevx, prevy);
    const double dcur = point::dist2(gx, gy, h.d.px, h.d.py);
    r.reach = dcur < REACH_RADIUS;
    double reward = rn::sub(dprev, dcur);
    if (r.reach) reward = rn::add(reward, REACH_BONUS);
    h.elapsed += 1;
    const bool term = r.reach && cfg.terminate_on_goal;
    const bool tl = cfg.time_limit > 0 && h.elapsed >= cfg.time_limit;
    r.done = term || tl;
    r.trunc = tl && !term;
    h.ep_ret = rn::add(h.ep_ret, reward);
    r.rew = (float)reward;
    r.ep_r = h.ep_ret;
    r.ep_l = h.elapsed;
    point::sensors_cs(cfg.pk, h.d, hc, hs, (double)h.cx, (double)h.cz, h.gx, h.gy, obs, dcur);
    if (ext) point_obs_ext(h, cold, i, hc, hs, *ext);
    if (r.done) {
#pragma unroll
        for (int k = 0; k < point::OBS; ++k) term_obs[k] = obs[k];
        if (ext) *term_ext = *ext;
        point_reset(h, cold, i, !r.reach);
        point::sensors(h.d, (double)h.cx, (double)h.cz, h.gx, h.gy, obs);
        if (ext) {
            double s, c;
            sincos(h.d.psi, &s, &c);
            point_obs_ext(h, cold, i, c, s, *ext);
        }
    }
    return r;
}

}  // namespace mr
