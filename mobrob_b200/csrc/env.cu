// Batched goal environment resident in HBM: state slab, stand-alone VecEnv kernels
// (step / reset / obs / state import-export).  One thread per environment, SoA state,
// observation rows staged through shared memory so the [N][O] store is fully coalesced.
#include "env_state.cuh"

#include <stdarg.h>

#include <atomic>

namespace mr {

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
void count_launch(uint64_t n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// ---------------------------------------------------------------------------------------
constexpr int STEP_THREADS = 128;
// Observation rows leave the block as one contiguous span of rows * OBS floats.  Each thread puts
// its row into shared memory as 7 float2 (dense 56-byte rows: a half-warp's 8-byte stores cover
// all 32 banks once), then the block streams the span out as float4 -- 4 load/store pairs per
// thread instead of 14 scalar ones with an index division each (that loop was 18 % of the
// env-step kernel's instructions, profiles/r01_env_step).
__device__ __forceinline__ void stage_row(float* smem, const float (&o)[point::OBS]) {
    float2* row = reinterpret_cast<float2*>(smem + threadIdx.x * point::OBS);
#pragma unroll
    for (int j = 0; j < point::OBS / 2; ++j) row[j] = make_float2(o[2 * j], o[2 * j + 1]);
}
__device__ __forceinline__ void store_rows_coalesced(float* __restrict__ dst, const float* smem,
                                                     int64_t block_start, int rows) {
    const int total = rows * point::OBS;
    float* base = dst + block_start * point::OBS;   // block_start * 56 B is a multiple of 16
    if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
        const int nvec = total >> 2;
        const float4* src4 = reinterpret_cast<const float4*>(smem);
        float4* dst4 = reinterpret_cast<float4*>(base);
#pragma unroll
        for (int v = 0; v < (STEP_THREADS * point::OBS / 4 + STEP_THREADS - 1) / STEP_THREADS; ++v) {
            const int idx = threadIdx.x + v * STEP_THREADS;
            if (idx < nvec) dst4[idx] = src4[idx];
        }
        const int idx = (nvec << 2) + threadIdx.x;
        if (idx < total) base[idx] = smem[idx];
    } else {
        for (int idx = threadIdx.x; idx < total; idx += STEP_THREADS) base[idx] = smem[idx];
    }
}

template <int MINB>
__global__ void __launch_bounds__(STEP_THREADS, MINB)
point_step_kernel(PointState st, EnvCfg cfg, const float2* __restrict__ act,
                  float* __restrict__ obs, float* __restrict__ rew, uint8_t* __restrict__ done,
                  uint8_t* __restrict__ trunc, float* __restrict__ term_obs,
                  double* __restrict__ ep_ret, int32_t* __restrict__ ep_len, int64_t pf_dist) {
    __shared__ __align__(16) float s_obs[STEP_THREADS * point::OBS];
    // pf_dist < 0: this launch walks the envs downwards.  Consecutive steps alternate, so the state a
    // step wrote last -- still dirty in the 126 MB L2 -- is what the next step reads (and overwrites)
    // first: those lines never travel to HBM in between.
    const int64_t block = pf_dist < 0 ? (int64_t)gridDim.x - 1 - blockIdx.x : (int64_t)blockIdx.x;
    const int64_t block_start = block * STEP_THREADS;
    const int64_t i = block_start + threadIdx.x;
    if (pf_dist > 1 || pf_dist < -1) {
        const int64_t bp = block + pf_dist / STEP_THREADS;   // the block that starts one wave later
        if (bp >= 0 && bp < (int64_t)gridDim.x) {
            st.prefetch_tile(bp, threadIdx.x);
            const int64_t a0 = bp * STEP_THREADS + (int64_t)(threadIdx.x - 120) * 16;   // 16 float2 = one 128-byte line
            if (threadIdx.x >= 120 && a0 + 16 <= st.n) asm volatile("prefetch.global.L2 [%0];" ::"l"(act + a0));
        }
    }
    if (i < st.n) {
        PointHot h = st.load_step(i);
        float2 a = act[i];
        float o[point::OBS], tobs[point::OBS];
        StepResult r = point_env_step(h, st.cold, i, a.x, a.y, cfg, o, tobs);
        stage_row(s_obs, o);
        st.store_step(i, h, r.done);
        rew[i] = r.rew;
        done[i] = r.done ? 1 : 0;
        trunc[i] = r.trunc ? 1 : 0;
        if (r.done) {
            if (term_obs) {
#pragma unroll
                for (int k = 0; k < point::OBS; ++k) term_obs[i * point::OBS + k] = tobs[k];
            }
            if (ep_ret) ep_ret[i] = r.ep_r;
            if (ep_len) ep_len[i] = r.ep_l;
        }
    }
    __syncthreads();
    int rows = (int)min((int64_t)STEP_THREADS, st.n - block_start);
    store_rows_coalesced(obs, s_obs, block_start, rows);
}

// Step with optional observation keys (EnvCfg::obs_flags != 0): same per-env logic, rows of obs_dim_ext floats
// written row by row (this variant is not the measured hot path; the default configuration keeps the kernel above).
__global__ void __launch_bounds__(STEP_THREADS)
point_step_ext_kernel(PointState st, EnvCfg cfg, const float2* __restrict__ act, float* __restrict__ obs,
                      float* __restrict__ rew, uint8_t* __restrict__ done, uint8_t* __restrict__ trunc,
                      float* __restrict__ term_obs, double* __restrict__ ep_ret, int32_t* __restrict__ ep_len) {
    const int64_t i = (int64_t)blockIdx.x * STEP_THREADS + threadIdx.x;
    if (i >= st.n) return;
    const int O = obs_dim_ext(point::OBS, 3, 3, cfg.obs_flags, cfg.lidar.num_bins);
    PointHot h = st.load_step(i);
    const float2 a = act[i];
    float o[point::OBS], tobs[point::OBS];
    PointExt x, tx;
    StepResult r = point_env_step(h, st.cold, i, a.x, a.y, cfg, o, tobs, &x, &tx);
    st.store_step(i, h, r.done);
    emit_obs_row<point::OBS, POINT_OBS_PRE, 3, 3>(obs + i * O, o, x, cfg.obs_flags, cfg.lidar);
    rew[i] = r.rew;
    done[i] = r.done ? 1 : 0;
    trunc[i] = r.trunc ? 1 : 0;
    if (r.done) {
        if (term_obs) emit_obs_row<point::OBS, POINT_OBS_PRE, 3, 3>(term_obs + i * O, tobs, tx, cfg.obs_flags, cfg.lidar);
        if (ep_ret) ep_ret[i] = r.ep_r;
        if (ep_len) ep_len[i] = r.ep_l;
    }
}

__device__ __forceinline__ void point_obs_row_ext(const PointState& st, const PointHot& h, int64_t i, const float (&o)[point::OBS],
                                                  const EnvCfg& cfg, float* __restrict__ obs) {
    PointExt x;
    double s, c;
    sincos(h.d.psi, &s, &c);
    point_obs_ext(h, st.cold, i, c, s, x);
    emit_obs_row<point::OBS, POINT_OBS_PRE, 3, 3>(obs + i * obs_dim_ext(point::OBS, 3, 3, cfg.obs_flags, cfg.lidar.num_bins),
                                                  o, x, cfg.obs_flags, cfg.lidar);
}

__global__ void __launch_bounds__(STEP_THREADS)
point_reset_kernel(PointState st, const uint8_t* __restrict__ mask, int first,
                   float* __restrict__ obs, EnvCfg cfg) {
    const int64_t i = (int64_t)blockIdx.x * STEP_THREADS + threadIdx.x;
    if (i >= st.n) return;
    if (mask && !mask[i]) return;
    PointHot h = st.load(i);
    bool reach = point::dist2((double)h.gx, (double)h.gy, h.d.px, h.d.py) < REACH_RADIUS;
    point_reset(h, st.cold, i, first || !reach);
    st.store(i, h);
    if (obs) {
        float o[point::OBS];
        point::sensors(h.d, (double)h.cx, (double)h.cz, h.gx, h.gy, o);
        if (cfg.obs_flags) { point_obs_row_ext(st, h, i, o, cfg, obs); return; }
#pragma unroll
        for (int k = 0; k < point::OBS; ++k) obs[i * point::OBS + k] = o[k];
    }
}

__global__ void __launch_bounds__(STEP_THREADS)
point_obs_ext_kernel(PointState st, float* __restrict__ obs, EnvCfg cfg) {
    const int64_t i = (int64_t)blockIdx.x * STEP_THREADS + threadIdx.x;
    if (i >= st.n) return;
    PointHot h = st.load(i);
    float o[point::OBS];
    point::sensors(h.d, (double)h.cx, (double)h.cz, h.gx, h.gy, o);
    point_obs_row_ext(st, h, i, o, cfg, obs);
}

__global__ void __launch_bounds__(STEP_THREADS)
point_obs_kernel(PointState st, float* __restrict__ obs) {
    __shared__ __align__(16) float s_obs[STEP_THREADS * point::OBS];
    const int64_t block_start = (int64_t)blockIdx.x * STEP_THREADS;
    const int64_t i = block_start + threadIdx.x;
    if (i < st.n) {
        PointHot h = st.load(i);
        float o[point::OBS];
        point::sensors(h.d, (double)h.cx, (double)h.cz, h.gx, h.gy, o);
        stage_row(s_obs, o);
    }
    __syncthreads();
    int rows = (int)min((int64_t)STEP_THREADS, st.n - block_start);
    store_rows_coalesced(obs, s_obs, block_start, rows);
}

// reference view: qpos(3) qvel(3) body_xy(2) psi0(1) ctrl(2) goal(2) elapsed(1) ep_ret(1)
__global__ void point_get_state_kernel(PointState st, double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= st.n) return;
    PointHot h = st.load(i);
    float2 b = st.cold.body_xy[i];
    double p0 = st.cold.psi0[i], s0, c0;
    sincos(p0, &s0, &c0);
    double dx = h.d.px - (double)b.x, dy = h.d.py - (double)b.y;
    double* o = out + i * POINT_STATE_DIM;
    o[0] = c0 * dx + s0 * dy;
    o[1] = -s0 * dx + c0 * dy;
    o[2] = h.d.psi - p0;
    o[3] = c0 * h.d.vx + s0 * h.d.vy;
    o[4] = -s0 * h.d.vx + c0 * h.d.vy;
    o[5] = h.d.om;
    o[6] = b.x; o[7] = b.y; o[8] = p0;
    o[9] = h.cx; o[10] = h.cz; o[11] = h.gx; o[12] = h.gy;
    o[13] = (double)h.elapsed; o[14] = h.ep_ret;
}

__global__ void point_set_state_kernel(PointState st, const double* __restrict__ in) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= st.n) return;
    const double* s = in + i * POINT_STATE_DIM;
    double p0 = s[8], s0, c0;
    sincos(p0, &s0, &c0);
    PointHot h;
    h.d.px = s[6] + c0 * s[0] - s0 * s[1];
    h.d.py = s[7] + s0 * s[0] + c0 * s[1];
    h.d.psi = p0 + s[2];
    h.d.vx = c0 * s[3] - s0 * s[4];
    h.d.vy = s0 * s[3] + c0 * s[4];
    h.d.om = s[5];
    h.cx = (float)s[9]; h.cz = (float)s[10]; h.gx = (float)s[11]; h.gy = (float)s[12];
    h.elapsed = (int)s[13]; h.ep_ret = s[14];
    st.cold.body_xy[i] = make_float2((float)s[6], (float)s[7]);
    st.cold.psi0[i] = p0;
    st.store(i, h);
}

__global__ void point_get_pos_kernel(PointState st, double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= st.n) return;
    const double2 p = st.pos(i);
    out[2 * i] = p.x;
    out[2 * i + 1] = p.y;
}

// ---------------------------------------------------------------------------------------
// car: same VecEnv kernels, one thread per env (state in fp64 registers; the contact solver's Delassus matrix
// in shared memory, car::SCRATCH_DOUBLES per thread)
constexpr int CAR_THREADS = 64;
constexpr size_t CAR_SMEM = (size_t)car::SCRATCH_DOUBLES * sizeof(double) * CAR_THREADS;   // 112.5 KB: two CTAs per SM
#define MR_CAR_SCRATCH() extern __shared__ __align__(16) double car_smem[]; \
    const car::Scratch S{(uint32_t)__cvta_generic_to_shared(car_smem + threadIdx.x), (uint32_t)(CAR_THREADS * sizeof(double))}

__global__ void __launch_bounds__(CAR_THREADS)
car_step_kernel(CarSoA st, car::Consts K, EnvCfg cfg, const float2* __restrict__ act,
                float* __restrict__ obs, float* __restrict__ rew, uint8_t* __restrict__ done,
                uint8_t* __restrict__ trunc, float* __restrict__ term_obs, double* __restrict__ ep_ret,
                int32_t* __restrict__ ep_len) {
    MR_CAR_SCRATCH();
    const int64_t i = (int64_t)blockIdx.x * CAR_THREADS + threadIdx.x;
    if (i >= st.n) return;
    CarHot h = st.load(i);
    float2 a = act[i];
    float o[car::OBS], tobs[car::OBS];
    StepResult r = car_env_step(K, h, st.cold, i, a.x, a.y, cfg, st.contacts != 0, o, tobs, S);
    st.store(i, h);
    for (int k = 0; k < car::OBS; ++k) obs[i * car::OBS + k] = o[k];
    rew[i] = r.rew;
    done[i] = r.done ? 1 : 0;
    trunc[i] = r.trunc ? 1 : 0;
    if (r.done) {
        if (term_obs) for (int k = 0; k < car::OBS; ++k) term_obs[i * car::OBS + k] = tobs[k];
        if (ep_ret) ep_ret[i] = r.ep_r;
        if (ep_len) ep_len[i] = r.ep_l;
    }
}

// optional observation keys (EnvCfg::obs_flags != 0), see point_step_ext_kernel
__global__ void __launch_bounds__(CAR_THREADS)
car_step_ext_kernel(CarSoA st, car::Consts K, EnvCfg cfg, const float2* __restrict__ act,
                    float* __restrict__ obs, float* __restrict__ rew, uint8_t* __restrict__ done,
                    uint8_t* __restrict__ trunc, float* __restrict__ term_obs, double* __restrict__ ep_ret,
                    int32_t* __restrict__ ep_len) {
    MR_CAR_SCRATCH();
    const int64_t i = (int64_t)blockIdx.x * CAR_THREADS + threadIdx.x;
    if (i >= st.n) return;
    const int O = obs_dim_ext(car::OBS, 13, 11, cfg.obs_flags, cfg.lidar.num_bins);
    CarHot h = st.load(i);
    float2 a = act[i];
    float o[car::OBS], tobs[car::OBS];
    CarExt x, tx;
    StepResult r = car_env_step(K, h, st.cold, i, a.x, a.y, cfg, st.contacts != 0, o, tobs, S, &x, &tx);
    st.store(i, h);
    emit_obs_row<car::OBS, CAR_OBS_PRE, 13, 11>(obs + i * O, o, x, cfg.obs_flags, cfg.lidar);
    rew[i] = r.rew;
    done[i] = r.done ? 1 : 0;
    trunc[i] = r.trunc ? 1 : 0;
    if (r.done) {
        if (term_obs) emit_obs_row<car::OBS, CAR_OBS_PRE, 13, 11>(term_obs + i * O, tobs, tx, cfg.obs_flags, cfg.lidar);
        if (ep_ret) ep_ret[i] = r.ep_r;
        if (ep_len) ep_len[i] = r.ep_l;
    }
}

__device__ __forceinline__ void car_obs_row(const CarHot& h, int64_t i, const float (&o)[car::OBS], const EnvCfg& cfg,
                                            float* __restrict__ obs) {
    if (cfg.obs_flags) {
        CarExt x;
        car_obs_ext(h, x);
        emit_obs_row<car::OBS, CAR_OBS_PRE, 13, 11>(obs + i * obs_dim_ext(car::OBS, 13, 11, cfg.obs_flags, cfg.lidar.num_bins),
                                                    o, x, cfg.obs_flags, cfg.lidar);
    } else {
        for (int k = 0; k < car::OBS; ++k) obs[i * car::OBS + k] = o[k];
    }
}

__global__ void __launch_bounds__(CAR_THREADS)
car_reset_kernel(CarSoA st, car::Consts K, const uint8_t* __restrict__ mask, int first, float* __restrict__ obs,
                 EnvCfg cfg) {
    MR_CAR_SCRATCH();
    const int64_t i = (int64_t)blockIdx.x * CAR_THREADS + threadIdx.x;
    if (i >= st.n) return;
    if (mask && !mask[i]) return;
    CarHot h = st.load(i);
    bool reach = point::dist2((double)h.gx, (double)h.gy, h.s.p[0], h.s.p[1]) < REACH_RADIUS;
    car_reset(h, st.cold, i, first || !reach);
    st.store(i, h);
    if (obs) {
        float o[car::OBS];
        car::sensors(K, h.s, (double)h.cx, (double)h.cz, h.gx, h.gy, st.contacts != 0, o, S);
        car_obs_row(h, i, o, cfg, obs);
    }
}

__global__ void __launch_bounds__(CAR_THREADS)
car_obs_kernel(CarSoA st, car::Consts K, float* __restrict__ obs, EnvCfg cfg) {
    MR_CAR_SCRATCH();
    const int64_t i = (int64_t)blockIdx.x * CAR_THREADS + threadIdx.x;
    if (i >= st.n) return;
    CarHot h = st.load(i);
    float o[car::OBS];
    car::sensors(K, h.s, (double)h.cx, (double)h.cz, h.gx, h.gy, st.contacts != 0, o, S);
    car_obs_row(h, i, o, cfg, obs);
}

// reference view: qpos(13) = p quat thL thR qb ; qvel(11) = v w sL sR wb ; ctrl goal elapsed ep_ret
// the car kernels' contact scratch exceeds the default 48 KB of dynamic shared memory: opt in once per device
static int car_smem_optin() {
    static OncePerDevice once;
    if (once.first()) {
        MR_CUDA(cudaFuncSetAttribute(car_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CAR_SMEM));
        MR_CUDA(cudaFuncSetAttribute(car_step_ext_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CAR_SMEM));
        MR_CUDA(cudaFuncSetAttribute(car_reset_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CAR_SMEM));
        MR_CUDA(cudaFuncSetAttribute(car_obs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CAR_SMEM));
    }
    return MR_OK;
}

__global__ void car_get_state_kernel(CarSoA st, double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= st.n) return;
    CarHot h = st.load(i);
    double* o = out + i * CAR_STATE_DIM;
    const car::State& s = h.s;
    o[0] = s.p[0]; o[1] = s.p[1]; o[2] = s.p[2];
    o[3] = s.q[0]; o[4] = s.q[1]; o[5] = s.q[2]; o[6] = s.q[3];
    o[7] = s.th[0]; o[8] = s.th[1];
    o[9] = s.qb[0]; o[10] = s.qb[1]; o[11] = s.qb[2]; o[12] = s.qb[3];
    o[13] = s.v[0]; o[14] = s.v[1]; o[15] = s.v[2];
    o[16] = s.w[0]; o[17] = s.w[1]; o[18] = s.w[2];
    o[19] = s.s[0]; o[20] = s.s[1];
    o[21] = s.wb[0]; o[22] = s.wb[1]; o[23] = s.wb[2];
    o[24] = h.cx; o[25] = h.cz; o[26] = h.gx; o[27] = h.gy;
    o[28] = (double)h.elapsed; o[29] = h.ep_ret;
}

__global__ void car_set_state_kernel(CarSoA st, const double* __restrict__ in) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= st.n) return;
    const double* o = in + i * CAR_STATE_DIM;
    CarHot h;
    car::State& s = h.s;
    s.p[0] = o[0]; s.p[1] = o[1]; s.p[2] = o[2];
    s.q[0] = o[3]; s.q[1] = o[4]; s.q[2] = o[5]; s.q[3] = o[6];
    s.th[0] = o[7]; s.th[1] = o[8];
    s.qb[0] = o[9]; s.qb[1] = o[10]; s.qb[2] = o[11]; s.qb[3] = o[12];
    s.v[0] = o[13]; s.v[1] = o[14]; s.v[2] = o[15];
    s.w[0] = o[16]; s.w[1] = o[17]; s.w[2] = o[18];
    s.s[0] = o[19]; s.s[1] = o[20];
    s.wb[0] = o[21]; s.wb[1] = o[22]; s.wb[2] = o[23];
    h.cx = (float)o[24]; h.cz = (float)o[25]; h.gx = (float)o[26]; h.gy = (float)o[27];
    h.elapsed = (int)o[28]; h.ep_ret = o[29];
    st.store(i, h);
}

__global__ void car_get_pos_kernel(CarSoA st, double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= st.n) return;
    out[2 * i] = st.st[i];
    out[2 * i + 1] = st.st[st.n + i];
}

// ---- mass properties of car.xml (density 5), same formulas as oracle/car_oracle.py -----------------------

car::Consts make_car_consts() { return car::make_consts(); }

}  // namespace mr

using namespace mr;

// =======================================================================================
extern "C" {

int mr_version(void) { return 101; }
const char* mr_last_error(void) { return mr::g_err; }
uint64_t mr_launch_count(void) { return mr::g_launches.load(); }

int mr_env_create(int kind, int64_t n_envs, int device, int time_limit, int terminate_on_goal,
                  mr_env** out) {
    MR_REQUIRE(out != nullptr, "out is NULL");
    MR_REQUIRE(n_envs > 0, "n_envs must be positive");
    if (kind != MR_ENV_POINT && kind != MR_ENV_CAR) {
        set_error("unknown env kind %d (0 = point, 1 = car)", kind);
        return MR_ERR_UNSUPPORTED;
    }
    DeviceGuard guard(device);   // the caller's current device is left as it was
    mr_env* e = new mr_env();
    e->kind = kind;
    e->n = n_envs;
    e->device = device;
    e->cfg.time_limit = time_limit;
    e->cfg.terminate_on_goal = terminate_on_goal ? 1 : 0;
    e->cfg.pk = point::make_k();
    e->cfg.obs_flags = 0;
    e->cfg.lidar = make_lidar_cfg(10, 0.0, 1.0, 1);   // Safety Gym's defaults: 10 bins, max_dist None, exp_gain 1, alias
    size_t bytes = kind == MR_ENV_POINT ? PointState::slab_bytes(n_envs) : CarSoA::slab_bytes(n_envs);
    cudaError_t err = cudaMalloc(&e->slab, bytes);
    if (err != cudaSuccess) {
        set_error("cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(err));
        delete e;
        return MR_ERR_ALLOC;
    }
    cudaMemset(e->slab, 0, bytes);
    e->slab_bytes = bytes;
    if (kind == MR_ENV_POINT) {
        e->point.carve(e->slab, n_envs);
    } else {
        e->car.carve(e->slab, n_envs);
        e->carK = make_car_consts();
    }
    // MujocoGoalEnv.get_init_space / get_goal_space (wrapper.py:250-264): extents / 2 and extents
    const float spaces[8] = {-1.f, -1.f, 1.f, 1.f, -2.f, -2.f, 2.f, 2.f};
    cudaMemcpy(const_cast<float*>(kind == MR_ENV_POINT ? e->point.cold.spaces : e->car.cold.spaces), spaces,
               sizeof(spaces), cudaMemcpyHostToDevice);
    *out = e;
    return MR_OK;
}

static const EnvCold& cold_of(const mr_env* env) {
    return env->kind == MR_ENV_POINT ? env->point.cold : env->car.cold;
}

// EnvWrapper.reset_init_space / reset_goal_space (wrapper.py:209-219) for every env of the batch: later resets draw
// from the new boxes.  Each env keeps its own random stream (the reference swaps in the new Box object, whose
// generator EnvWrapper.seed re-seeds at the next seeded reset).  h_init / h_goal: (low x, low y, high x, high y) in
// host memory, either may be NULL (unchanged).
int mr_env_set_spaces(mr_env* env, const float* h_init, const float* h_goal, void* stream) {
    MR_REQUIRE(env, "env is NULL");
    DeviceGuard guard(env->device);
    float* d = const_cast<float*>(cold_of(env).spaces);
    cudaStream_t s = (cudaStream_t)stream;
    for (int k = 0; k < 2; ++k) {
        const float* h = k == 0 ? h_init : h_goal;
        if (!h) continue;
        MR_REQUIRE(h[0] <= h[2] && h[1] <= h[3], "space bounds: low must not exceed high");
        MR_CUDA(cudaMemcpyAsync(d + 4 * k, h, 4 * sizeof(float), cudaMemcpyHostToDevice, s));
    }
    MR_CUDA(cudaStreamSynchronize(s));  // host buffers may be freed by the caller on return
    return MR_OK;
}

void mr_env_destroy(mr_env* env) {
    if (!env) return;
    DeviceGuard guard(env->device);
    cudaFree(env->slab);
    if (env->scratch) cudaFree(env->scratch);
    delete env;
}

int mr_env_obs_dim(const mr_env* env) {
    if (!env) return 0;
    const int bins = env->cfg.lidar.num_bins;
    return env->kind == MR_ENV_POINT ? obs_dim_ext(point::OBS, 3, 3, env->cfg.obs_flags, bins)
                                     : obs_dim_ext(car::OBS, 13, 11, env->cfg.obs_flags, bins);
}

int mr_env_set_obs_flags(mr_env* env, unsigned flags) {
    MR_REQUIRE(env, "env is NULL");
    if (flags & ~OBS_ALL_FLAGS) {
        set_error("unknown observation flag bits 0x%x (1 goal_dist, 2 qpos, 4 qvel, 8 ctrl, 16 goal_lidar)",
                  flags & ~OBS_ALL_FLAGS);
        return MR_ERR_UNSUPPORTED;
    }
    if (env->scratch && flags != env->cfg.obs_flags) {   // mr_rollout_unfused sized its scratch for the old row length
        DeviceGuard guard(env->device);
        MR_CUDA(cudaDeviceSynchronize());
        MR_CUDA(cudaFree(env->scratch));
        env->scratch = nullptr;
    }
    env->cfg.obs_flags = flags;
    return MR_OK;
}

int mr_env_set_lidar(mr_env* env, int num_bins, double max_dist, double exp_gain, int alias) {
    MR_REQUIRE(env, "env is NULL");
    MR_REQUIRE(num_bins >= 1, "lidar_num_bins must be at least 1");
    if (env->scratch && num_bins != env->cfg.lidar.num_bins && (env->cfg.obs_flags & OBS_GOAL_LIDAR)) {
        DeviceGuard guard(env->device);   // as in mr_env_set_obs_flags: the rollout scratch has the old row length
        MR_CUDA(cudaDeviceSynchronize());
        MR_CUDA(cudaFree(env->scratch));
        env->scratch = nullptr;
    }
    env->cfg.lidar = make_lidar_cfg(num_bins, max_dist, exp_gain, alias);
    return MR_OK;
}
int mr_env_state_dim(const mr_env* env) {
    return env ? (env->kind == MR_ENV_POINT ? POINT_STATE_DIM : CAR_STATE_DIM) : 0;
}

int mr_env_set_contacts(mr_env* env, int enabled) {
    MR_REQUIRE(env, "env is NULL");
    env->car.contacts = enabled ? 1 : 0;
    return MR_OK;
}


int mr_env_seed(mr_env* env, const uint64_t* h_pcg_init, const uint64_t* h_pcg_goal,
                const int64_t* h_engine_seed, void* stream) {
    MR_REQUIRE(env && h_pcg_init && h_pcg_goal && h_engine_seed, "NULL argument");
    cudaStream_t s = (cudaStream_t)stream;
    DeviceGuard guard(env->device);
    const EnvCold& c = cold_of(env);
    MR_CUDA(cudaMemcpyAsync(c.pcg_init, h_pcg_init, env->n * 32, cudaMemcpyHostToDevice, s));
    MR_CUDA(cudaMemcpyAsync(c.pcg_goal, h_pcg_goal, env->n * 32, cudaMemcpyHostToDevice, s));
    MR_CUDA(cudaMemcpyAsync(c.engine_seed, h_engine_seed, env->n * 8, cudaMemcpyHostToDevice, s));
    MR_CUDA(cudaStreamSynchronize(s));  // host buffers may be freed by the caller on return
    return MR_OK;
}

int mr_env_reset(mr_env* env, const uint8_t* mask, int first, float* obs_out, void* stream) {
    MR_REQUIRE(env, "env is NULL");
    cudaStream_t s = (cudaStream_t)stream;
    if (env->kind == MR_ENV_POINT)
        point_reset_kernel<<<ceil_div(env->n, STEP_THREADS), STEP_THREADS, 0, s>>>(env->point, mask, first, obs_out,
                                                                                   env->cfg);
    else {
        if (car_smem_optin() != MR_OK) return MR_ERR_CUDA;
        car_reset_kernel<<<ceil_div(env->n, CAR_THREADS), CAR_THREADS, CAR_SMEM, s>>>(env->car, env->carK, mask, first, obs_out,
                                                                                      env->cfg);
    }
    MR_CHECK_LAUNCH();
    return MR_OK;
}

int mr_env_step(mr_env* env, const float* act, float* obs, float* rew, uint8_t* done,
                uint8_t* trunc, float* term_obs, double* ep_ret, int32_t* ep_len, void* stream) {
    MR_REQUIRE(env && act && obs && rew && done && trunc, "NULL argument");
    cudaStream_t s = (cudaStream_t)stream;
    if (env->cfg.obs_flags) {
        const float2* a2 = reinterpret_cast<const float2*>(act);
        if (env->kind == MR_ENV_POINT) {
            point_step_ext_kernel<<<ceil_div(env->n, STEP_THREADS), STEP_THREADS, 0, s>>>(
                env->point, env->cfg, a2, obs, rew, done, trunc, term_obs, ep_ret, ep_len);
        } else {
            if (car_smem_optin() != MR_OK) return MR_ERR_CUDA;
            car_step_ext_kernel<<<ceil_div(env->n, CAR_THREADS), CAR_THREADS, CAR_SMEM, s>>>(
                env->car, env->carK, env->cfg, a2, obs, rew, done, trunc, term_obs, ep_ret, ep_len);
        }
    } else if (env->kind == MR_ENV_POINT) {
        // tuning knobs (measured on B200 at 4M envs, profiles/r01_env_step_sweep.txt): 5 blocks per SM
        // (96 registers, no spills) and a prefetch distance of 4 blocks per SM are the defaults
        static const int minb = getenv("MR_STEP_MINB") ? atoi(getenv("MR_STEP_MINB")) : 5;
        auto kern = minb == 8 ? point_step_kernel<8> : minb == 7 ? point_step_kernel<7> : minb == 6 ? point_step_kernel<6>
                    : minb == 4 ? point_step_kernel<4> : point_step_kernel<5>;
        static const int pf_blocks = getenv("MR_STEP_PF") ? atoi(getenv("MR_STEP_PF")) : 592;
        static const int flip = getenv("MR_STEP_FLIP") ? atoi(getenv("MR_STEP_FLIP")) : 1;
        const int64_t dist = pf_blocks > 0 ? (int64_t)pf_blocks * STEP_THREADS : 1;
        const bool down = flip && env->step_flip;
        env->step_flip ^= 1;
        kern<<<ceil_div(env->n, STEP_THREADS), STEP_THREADS, 0, s>>>(
            env->point, env->cfg, reinterpret_cast<const float2*>(act), obs, rew, done, trunc, term_obs, ep_ret, ep_len,
            down ? -dist : dist);
    } else {
        if (car_smem_optin() != MR_OK) return MR_ERR_CUDA;
        car_step_kernel<<<ceil_div(env->n, CAR_THREADS), CAR_THREADS, CAR_SMEM, s>>>(
            env->car, env->carK, env->cfg, reinterpret_cast<const float2*>(act), obs, rew, done, trunc, term_obs,
            ep_ret, ep_len);
    }
    MR_CHECK_LAUNCH();
    return MR_OK;
}

int mr_env_get_obs(mr_env* env, float* obs_out, void* stream) {
    MR_REQUIRE(env && obs_out, "NULL argument");
    cudaStream_t s = (cudaStream_t)stream;
    if (env->kind == MR_ENV_POINT) {
        if (env->cfg.obs_flags)
            point_obs_ext_kernel<<<ceil_div(env->n, STEP_THREADS), STEP_THREADS, 0, s>>>(env->point, obs_out, env->cfg);
        else
            point_obs_kernel<<<ceil_div(env->n, STEP_THREADS), STEP_THREADS, 0, s>>>(env->point, obs_out);
    } else {
        if (car_smem_optin() != MR_OK) return MR_ERR_CUDA;
        car_obs_kernel<<<ceil_div(env->n, CAR_THREADS), CAR_THREADS, CAR_SMEM, s>>>(env->car, env->carK, obs_out,
                                                                                    env->cfg);
    }
    MR_CHECK_LAUNCH();
    return MR_OK;
}

int mr_env_get_state(mr_env* env, double* state_out, void* stream) {
    MR_REQUIRE(env && state_out, "NULL argument");
    cudaStream_t s = (cudaStream_t)stream;
    if (env->kind == MR_ENV_POINT) point_get_state_kernel<<<ceil_div(env->n, 128), 128, 0, s>>>(env->point, state_out);
    else car_get_state_kernel<<<ceil_div(env->n, 128), 128, 0, s>>>(env->car, state_out);
    MR_CHECK_LAUNCH();
    return MR_OK;
}

int mr_env_set_state(mr_env* env, const double* state_in, void* stream) {
    MR_REQUIRE(env && state_in, "NULL argument");
    cudaStream_t s = (cudaStream_t)stream;
    if (env->kind == MR_ENV_POINT) point_set_state_kernel<<<ceil_div(env->n, 128), 128, 0, s>>>(env->point, state_in);
    else car_set_state_kernel<<<ceil_div(env->n, 128), 128, 0, s>>>(env->car, state_in);
    MR_CHECK_LAUNCH();
    return MR_OK;
}

int mr_env_get_pos(mr_env* env, double* pos_out, void* stream) {
    MR_REQUIRE(env && pos_out, "NULL argument");
    cudaStream_t s = (cudaStream_t)stream;
    if (env->kind == MR_ENV_POINT) point_get_pos_kernel<<<ceil_div(env->n, 128), 128, 0, s>>>(env->point, pos_out);
    else car_get_pos_kernel<<<ceil_div(env->n, 128), 128, 0, s>>>(env->car, pos_out);
    MR_CHECK_LAUNCH();
    return MR_OK;
}

int mr_env_get_reset_counts(mr_env* env, int32_t* out, void* stream) {
    MR_REQUIRE(env && out, "NULL argument");
    MR_CUDA(cudaMemcpyAsync(out, cold_of(env).counts, env->n * 8, cudaMemcpyDeviceToDevice,
                            (cudaStream_t)stream));
    return MR_OK;
}

}  // extern "C"
