// PPO update (K8 + K9): replaces the inner loop of [SB3 2.0.0] PPO.train -- evaluate_actions,
// per-minibatch advantage normalisation, clipped surrogate, value MSE, entropy bonus,
// backward, clip_grad_norm_, Adam -- reached in the reference through
// src/mobrob/rl_control/ppo.py:73-74 (PPOCtrl.learn -> PPO.learn).  No autograd: the
// gradients of the two 64-64 tanh towers are formed analytically.
//
// Two forms, both on the tensor cores (ppo_tc.cuh):
//   * per launch (mr_ppo_grad / mr_adam_step, looped by mr_ppo_train_epoch; parity tests, the NCCL baseline path):
//     ppo_grad_tc_kernel writes one partial gradient per CTA, ppo_reduce_kernel sums them in a fixed
//     order, adam_kernel clips by global norm and applies torch's Adam;
//   * per epoch (mr_ppo_epoch_fused; the product path): ppo_epoch_tc_kernel, one persistent
//     cooperative launch for all minibatches of an epoch.
// The update's entry points take SB3's clip_range_vf / target_kl and the update's control word as trailing
// arguments (include/mobrob_b200.h); with those off (<= 0 / NULL) they launch the default instantiations.
#include "mlp.cuh"
#include "perm.cuh"
#include "ppo_tc.cuh"

#include <stdlib.h>
#include <string.h>

namespace mr {

constexpr int STAT_SLOTS = 16;             // tail of the gradient vector
// tail layout: 0 policy_loss, 1 value_loss, 2 clip_fraction, 3 approx_kl, 4 sample count

__host__ __device__ inline int grad_stride(int O) { return ((make_layout(O).total + 3) & ~3) + STAT_SLOTS; }
__host__ __device__ inline int stat_base(int O) { return (make_layout(O).total + 3) & ~3; }

struct GradArgs {
    const float* params;
    const float* obs;       // [T][N][O]
    const float* act;       // [T][N][2]
    const float* old_logp;  // [T][N]
    const float* adv;       // [T][N]
    const float* ret;       // [T][N]
    const int64_t* perm;    // [mb_size] env-major sample ids (n * T + t)
    const int32_t* rows;    // the same samples as time-major buffer rows (t * N + n)
    const float* rec;       // epoch kernel: packed sample records [T * N][KP + 8] (mr_ppo_pack_samples)
    int64_t mb_size;
    const double* mb_stats; // (sum adv, sum adv^2, count) of the GLOBAL minibatch
    int64_t N, T;
    float clip_range, ent_coef, vf_coef;
    int normalize_adv;
    float* partials;        // [gridDim.x][grad_stride]
    const float* old_val;   // [T][N] the rollout's values (clip_range_vf; per-launch gather)
    float clip_vf;          // SB3's clip_range_vf; <= 0: off
    const int* ctrl;        // the update's control word (NULL: none); != 0 -> the update has stopped
};

// Tensor-core version (ppo_tc.cuh): even CTAs own the policy tower, odd CTAs the value tower.
// VF: value clipping compiled in (A.clip_vf > 0).
__device__ __forceinline__ bool update_stopped(const int* ctrl) {
    return ctrl != nullptr && *reinterpret_cast<const volatile int*>(ctrl) != 0;
}
template <int KP, bool VF>
__global__ void __launch_bounds__(tc::THREADS, 1) ppo_grad_tc_kernel(GradArgs A, int O) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    if (update_stopped(A.ctrl)) return;   // target_kl stopped the update at an earlier minibatch
    MR_TR(0);
    tc::Ctx C = tc::make_ctx(smem_raw, blockIdx.x & 1);
    tc::setup(C);
    tc::stage<KP>(C, A.params, O);
    const tc::Sched S{A.mb_size, A.mb_size, 1, (int)(blockIdx.x >> 1), (int)(gridDim.x >> 1)};
    tc::Pipe<KP> Q;
    tc::pipe_start<KP, false, VF>(Q, A, S, O, threadIdx.x & 127, threadIdx.x >> 7, C.tower == 0);
    __syncthreads();
    const tc::MbConst MK = tc::mb_const(A.mb_stats, 0, A.normalize_adv);
    tc::minibatch<KP, VF>(C, A, S, MK, 0, Q, O, A.partials + (size_t)blockIdx.x * grad_stride(O));
    tc::teardown(C);
}

// grad[p] = sum over CTAs; finishes the scalar terms.  One thread per parameter; the n_parts
// loads are independent, so they are issued 8 deep into 4 interleaved accumulators that are
// combined in a fixed order (deterministic for a given n_parts).
__global__ void __launch_bounds__(128)
ppo_reduce_kernel(const float* __restrict__ partials, int n_parts, int O, float ent_coef,
                  const double* __restrict__ mb_stats, float* __restrict__ grad, float rank_share,
                  const int* __restrict__ ctrl) {
    if (update_stopped(ctrl)) return;   // grad keeps the stopping minibatch's gradient
    const int stride = grad_stride(O);
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= stride) return;
    // CTA b holds tower (b & 1) only: consecutive parts of one tower are 2 rows apart
    const float* src = partials + p + (size_t)tc::param_tower(p, make_layout(O)) * stride;
    n_parts >>= 1;
    const int st2 = 2 * stride;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int b = 0;
    for (; b + 8 <= n_parts; b += 8) {
        float v[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) v[q] = __ldg(src + (size_t)(b + q) * st2);
        a0 += v[0]; a1 += v[1]; a2 += v[2]; a3 += v[3];
        a0 += v[4]; a1 += v[5]; a2 += v[6]; a3 += v[7];
    }
    for (; b < n_parts; ++b) a0 += __ldg(src + (size_t)b * st2);
    float s = (a0 + a1) + (a2 + a3);
    const ParamLayout L = make_layout(O);
    const int sb = stat_base(O);
    if (p >= L.logstd && p < L.logstd + ACT) s -= ent_coef * rank_share;  // d(-ent_coef * mean entropy)/d log_std
    if (p >= sb && p < sb + 4) s *= (float)(1.0 / mb_stats[2]);
    if (p >= sb + 4 || (p >= L.total && p < sb)) s = 0.f;
    grad[p] = s;
}

struct AdamArgs {
    float* params;
    float* exp_avg;
    float* exp_avg_sq;
    const float* grad;
    int64_t* step;      // [0] Adam step count (state["step"]); [1] launch-internal ticket (starts at 0)
    float lr, beta1, beta2, eps, max_grad_norm;
    float* info;        // [8]: total_norm, clip_coef, step, entropy_loss, then the gradient's stats tail
    int n_params;       //      (policy_loss, value_loss, clip_fraction, approx_kl)
    float target_kl;    // SB3's target_kl (<= 0: off); needs ctrl
    int* ctrl;          // the update's control word (NULL: none)
    int64_t mb;         // index of this minibatch in the update (what ctrl records on a stop)
};

constexpr int ADAM_THREADS = 256;

// SB3's entropy_loss of a minibatch, -mean(sum_j (0.5 + 0.5 log(2 pi) + log_std_j)): the Gaussian's entropy does
// not depend on the sample, only on the log_std the minibatch was evaluated with
__device__ __forceinline__ float entropy_loss_of(float ls0, float ls1) {
    return -((1.4189385332046727f + ls0) + (1.4189385332046727f + ls1));
}

// clip_grad_norm_ + torch.optim.Adam (single-tensor path, torch 2.0.1 arithmetic order).
// The vector is only 42-48 KB, so the kernel is latency-bound: one parameter per thread,
// every CTA recomputes the global norm from L2 in the same fixed order (bit-identical across
// CTAs, no inter-CTA barrier), and the last CTA to finish bumps the step counter.
// target_kl: SB3's early stop.  The approx_kl of the reduced gradient's tail (a global mean, after the
// all-reduce when several ranks train) decides in every CTA alike; on a stop nothing is stepped, CTA 0 writes the
// info row (step unchanged) and records mb + 1 in the control word, and every later launch of the update returns.
__global__ void __launch_bounds__(ADAM_THREADS) adam_kernel(AdamArgs A) {
    __shared__ double s_part[ADAM_THREADS / 32];
    __shared__ double s_bc[2];
    if (update_stopped(A.ctrl)) return;
    const int tid = threadIdx.x;
    const int64_t step = A.step[0] + 1;
    float ent_loss = 0.f;
    if (tid == 0) {
        s_bc[0] = 1.0 - pow((double)A.beta1, (double)step);
        s_bc[1] = sqrt(1.0 - pow((double)A.beta2, (double)step));
        // log_std leads the flat vector; block 0 (which writes info) reads it before its own threads update it
        if (blockIdx.x == 0) ent_loss = entropy_loss_of(A.params[0], A.params[1]);
    }
    // global grad norm: thread t sums elements t, t + 256, ... (independent loads)
    double sq = 0.0;
    {
        constexpr int U = 8;
        int p = tid;
        for (; p + (U - 1) * ADAM_THREADS < A.n_params; p += U * ADAM_THREADS) {
            float v[U];
#pragma unroll
            for (int q = 0; q < U; ++q) v[q] = __ldg(A.grad + p + q * ADAM_THREADS);
#pragma unroll
            for (int q = 0; q < U; ++q) sq += (double)v[q] * (double)v[q];
        }
        for (; p < A.n_params; p += ADAM_THREADS) {
            float v = __ldg(A.grad + p);
            sq += (double)v * (double)v;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    if ((tid & 31) == 0) s_part[tid >> 5] = sq;
    __syncthreads();
    double tot = 0.0;
#pragma unroll
    for (int w = 0; w < ADAM_THREADS / 32; ++w) tot += s_part[w];
    const float total_norm = (float)sqrt(tot);
    const float coef = fminf(A.max_grad_norm / (total_norm + 1e-6f), 1.0f);
    if (A.target_kl > 0.f && A.ctrl) {
        const int sb = (A.n_params + 3) & ~3;
        if ((double)__ldg(A.grad + sb + 3) > 1.5 * (double)A.target_kl) {
            if (blockIdx.x == 0 && tid == 0) {
                if (A.info) {
                    A.info[0] = total_norm; A.info[1] = coef; A.info[2] = (float)(step - 1); A.info[3] = ent_loss;
                    for (int q = 0; q < 4; ++q) A.info[4 + q] = A.grad[sb + q];
                }
                *A.ctrl = (int)(A.mb + 1);
            }
            return;   // every CTA: no parameter moves, the ticket is not taken
        }
    }
    tc::AdamK K;   // one arithmetic for the per-launch and the fused path (tc::adam1)
    K.coef = coef;
    K.beta1 = A.beta1; K.beta2 = A.beta2; K.omb1 = 1.f - A.beta1; K.omb2 = 1.f - A.beta2;
    K.neg_step_size = (float)(-(double)A.lr / s_bc[0]);
    K.bc2_sqrt = (float)s_bc[1];
    K.eps = A.eps;
    const int p = blockIdx.x * ADAM_THREADS + tid;
    if (p < A.n_params) {
        float m = A.exp_avg[p], v = A.exp_avg_sq[p], w = A.params[p];
        tc::adam1(A.grad[p], K, m, v, w);
        A.params[p] = w;
        A.exp_avg[p] = m;
        A.exp_avg_sq[p] = v;
    }
    if (blockIdx.x == 0 && tid == 0 && A.info) {
        A.info[0] = total_norm; A.info[1] = coef; A.info[2] = (float)step; A.info[3] = ent_loss;
        const int sb = (A.n_params + 3) & ~3;
        for (int q = 0; q < 4; ++q) A.info[4 + q] = A.grad[sb + q];
    }
    // last CTA out increments the step (every CTA has read it by then) and re-arms the ticket
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        unsigned long long* ticket = reinterpret_cast<unsigned long long*>(A.step + 1);
        if (atomicAdd(ticket, 1ull) == (unsigned long long)gridDim.x - 1) {
            A.step[0] = step;
            *ticket = 0ull;
        }
    }
}

// Per-minibatch advantage sums of one epoch's permutation: stats[mb] = (sum, sum of squares,
// count) in float64 (shifted by the first element to keep the variance well conditioned is not
// needed at float64).  One CTA per minibatch.
__global__ void __launch_bounds__(1024)
adv_stats_kernel(const float* __restrict__ adv, const int64_t* __restrict__ perm,
                 int64_t n_samples, int64_t batch, int64_t N, int64_t T,
                 double* __restrict__ stats, int n_mb) {
    // several epochs in one launch: block b serves minibatch b % n_mb of permutation b / n_mb
    perm += (int64_t)(blockIdx.x / n_mb) * n_samples;
    stats += (int64_t)(blockIdx.x / n_mb) * n_mb * 3;
    const int64_t mb = blockIdx.x % n_mb;
    const int64_t s0 = mb * batch, s1 = min(n_samples, s0 + batch);
    double s = 0.0, q = 0.0;
    constexpr int U = 4;   // independent gathers in flight per thread
    for (int64_t i0 = s0 + threadIdx.x; i0 < s1; i0 += (int64_t)U * blockDim.x) {
        float a[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t i = i0 + (int64_t)u * blockDim.x;
            a[u] = 0.f;
            if (i < s1) {
                const int64_t id = perm[i];
                const int64_t n = id / T, t = id - n * T;
                a[u] = __ldg(adv + t * N + n);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            s += (double)a[u];
            q += (double)a[u] * (double)a[u];
        }
    }
    __shared__ double sh[2][32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        q += __shfl_xor_sync(0xffffffffu, q, o);
    }
    if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = s; sh[1][threadIdx.x >> 5] = q; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double ts = 0, tq = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { ts += sh[0][w]; tq += sh[1][w]; }
        stats[3 * mb] = ts;
        stats[3 * mb + 1] = tq;
        stats[3 * mb + 2] = (double)(s1 - s0);
    }
}

// What PPO.train logs after its epochs ([SB3] PPO.train, SURVEY A.5), in one launch: means over the
// info rows of all minibatches, the last minibatch's losses, explained_variance(values, returns) over the
// flat buffer, log_std after the update.  out[12]: [0:4] mean policy_loss / value_loss / clip_fraction /
// approx_kl, [4:6] last minibatch's policy and value loss, [6] explained variance (nan if var(returns) = 0),
// [7:9] log_std, [9] mean entropy_loss, [10] last minibatch's entropy_loss, [11] rows.
// scratch: 4 doubles + a ticket (8 doubles in all), zero before the first call; the kernel re-arms it.
// ctrl (target_kl; NULL = all rows): the update's control word.  When it records a stop after k minibatches, only
// rows [0, k) are averaged, "last" means row k - 1, out[11] = k, and out[12] = row k - 1's approx_kl (out then
// has 13 floats).
__global__ void __launch_bounds__(256)
train_summary_kernel(const float* __restrict__ info, int n_rows, const float* __restrict__ values,
                     const float* __restrict__ returns, int64_t n, const float* __restrict__ params,
                     float* __restrict__ out, double* __restrict__ scratch, const int* __restrict__ ctrl) {
    __shared__ double sh[8][8];
    __shared__ bool last;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    auto block_sum = [&](double (&v)[6], int cnt) {   // results valid in thread 0
#pragma unroll
        for (int k = 0; k < 6; ++k)
            if (k < cnt) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
                if (lane == 0) sh[k][warp] = v[k];
            }
        __syncthreads();
        if (tid == 0)
            for (int k = 0; k < cnt; ++k) {
                double t = 0.0;
                for (int w = 0; w < 8; ++w) t += sh[k][w];
                v[k] = t;
            }
        __syncthreads();
    };
    double a[6] = {0, 0, 0, 0, 0, 0};
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + tid; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double y = (double)returns[i], d = y - (double)values[i];
        a[0] += y; a[1] += y * y; a[2] += d; a[3] += d * d;
    }
    block_sum(a, 4);
    if (tid == 0) {
        for (int k = 0; k < 4; ++k) atomicAdd(scratch + k, a[k]);
        __threadfence();
        unsigned long long* ticket = reinterpret_cast<unsigned long long*>(scratch + 4);
        last = atomicAdd(ticket, 1ull) == (unsigned long long)gridDim.x - 1;
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    if (ctrl) {
        const int k = *reinterpret_cast<const volatile int*>(ctrl);
        if (k > 0 && k < n_rows) n_rows = k;
    }
    double r[6] = {0, 0, 0, 0, 0, 0};
    for (int row = tid; row < n_rows; row += blockDim.x) {
        const float* q = info + 8 * (size_t)row;
        r[0] += (double)q[4]; r[1] += (double)q[5]; r[2] += (double)q[6]; r[3] += (double)q[7]; r[4] += (double)q[3];
    }
    block_sum(r, 5);
    if (tid == 0) {
        const double inv = n_rows > 0 ? 1.0 / n_rows : 0.0;
        for (int k = 0; k < 4; ++k) out[k] = (float)(r[k] * inv);
        const float* lastrow = info + 8 * (size_t)(n_rows > 0 ? n_rows - 1 : 0);
        out[4] = lastrow[4]; out[5] = lastrow[5];
        volatile double* sc = scratch;
        const double sy = sc[0], syy = sc[1], sd = sc[2], sdd = sc[3];
        const double var_y = syy / (double)n - (sy / (double)n) * (sy / (double)n);
        const double var_d = sdd / (double)n - (sd / (double)n) * (sd / (double)n);
        out[6] = var_y > 0.0 ? (float)(1.0 - var_d / var_y) : __int_as_float(0x7fc00000);
        out[7] = params[0]; out[8] = params[1];
        out[9] = (float)(r[4] * inv);
        out[10] = lastrow[3];
        out[11] = (float)n_rows;
        if (ctrl) out[12] = lastrow[7];
        for (int k = 0; k < 5; ++k) scratch[k] = 0.0;   // re-arm (ticket included: it is slot 4)
    }
}

// One packed record per buffer row (tc::Rec): [obs | 0.. | 1 at KP-1 | a0 a1 old_logp adv | ret old_value 0 0].
// One thread per (row, 16-byte quad of the record): coalesced 16-byte stores, gathers hit L1 / L2.
// values NULL: old_value = 0 (no value clipping).
__global__ void __launch_bounds__(256)
pack_samples_kernel(const float* __restrict__ obs, const float* __restrict__ act, const float* __restrict__ old_logp,
                    const float* __restrict__ adv, const float* __restrict__ ret, const float* __restrict__ values,
                    int64_t n_rows, int O, int KP, float* __restrict__ rec) {
    const int qpr = (KP + 8) >> 2;   // quads per record
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows * qpr) return;
    const int64_t r = i / qpr;
    const int qd = (int)(i - r * qpr);
    float v[4];
    if (4 * qd < KP) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int k = 4 * qd + e;
            v[e] = k < O ? obs[r * O + k] : (k == KP - 1 ? 1.f : 0.f);
        }
    } else if (4 * qd == KP) {
        v[0] = act[2 * r]; v[1] = act[2 * r + 1]; v[2] = old_logp[r]; v[3] = adv[r];
    } else {
        v[0] = ret[r]; v[1] = values ? values[r] : 0.f; v[2] = v[3] = 0.f;
    }
    reinterpret_cast<float4*>(rec)[i] = make_float4(v[0], v[1], v[2], v[3]);
}

// env-major sample ids (RolloutBuffer.swap_and_flatten order, n * T + t) -> rows of the time-major
// buffers (t * N + n), once per epoch, so that the gather in the tensor-core kernels needs no division
__global__ void __launch_bounds__(256) perm_to_rows_kernel(const int64_t* __restrict__ perm, int64_t n_samples,
                                                           int64_t N, int64_t T, int32_t* __restrict__ rows) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_samples) return;
    const unsigned id = (unsigned)perm[i];
    const unsigned n = id / (unsigned)T, t = id - n * (unsigned)T;
    rows[i] = (int32_t)((int64_t)t * N + n);
}

constexpr int MAX_PERMS = 32;   // permutations per launch (one per epoch of an update)
struct PermKeys {
    PermKey k[MAX_PERMS];
};
__global__ void __launch_bounds__(256) device_perm_kernel(int64_t* __restrict__ out, int64_t n, PermKeys Ks) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const PermKey& K = Ks.k[blockIdx.y];   // blockIdx.y: which permutation
    uint32_t x = (uint32_t)i;
    do { x = perm_feistel(x, K); } while ((int64_t)x >= n);
    out[(int64_t)blockIdx.y * n + i] = (int64_t)x;
}

// The device index stream straight to what the epoch kernel consumes: rows[e][i] = buffer row (t * N + n) of
// the sample P_e(i) = n * T + t.  No int64 permutation is materialised (97 MB per update at the bench size).
__global__ void __launch_bounds__(256) device_rows_kernel(int32_t* __restrict__ rows, int64_t n, int64_t N, int64_t T,
                                                          PermKeys Ks) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const PermKey& K = Ks.k[blockIdx.y];
    uint32_t x = (uint32_t)i;
    do { x = perm_feistel(x, K); } while ((int64_t)x >= n);
    const unsigned env = x / (unsigned)T, t = x - env * (unsigned)T;
    rows[(int64_t)blockIdx.y * n + i] = (int32_t)((int64_t)t * N + env);
}

// adv_stats_kernel on buffer rows (several epochs per launch: block b -> minibatch b % n_mb of epoch b / n_mb)
__global__ void __launch_bounds__(1024)
adv_stats_rows_kernel(const float* __restrict__ adv, const int32_t* __restrict__ rows, int64_t n_samples, int64_t batch,
                      double* __restrict__ stats, int n_mb) {
    rows += (int64_t)(blockIdx.x / n_mb) * n_samples;
    stats += (int64_t)(blockIdx.x / n_mb) * n_mb * 3;
    const int64_t mb = blockIdx.x % n_mb;
    const int64_t s0 = mb * batch, s1 = min(n_samples, s0 + batch);
    double s = 0.0, q = 0.0;
    constexpr int U = 4;   // independent gathers in flight per thread
    for (int64_t i0 = s0 + threadIdx.x; i0 < s1; i0 += (int64_t)U * blockDim.x) {
        float a[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t i = i0 + (int64_t)u * blockDim.x;
            a[u] = i < s1 ? __ldg(adv + __ldg(rows + i)) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            s += (double)a[u];
            q += (double)a[u] * (double)a[u];
        }
    }
    __shared__ double sh[2][32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        q += __shfl_xor_sync(0xffffffffu, q, o);
    }
    if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = s; sh[1][threadIdx.x >> 5] = q; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double ts = 0, tq = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { ts += sh[0][w]; tq += sh[1][w]; }
        stats[3 * mb] = ts;
        stats[3 * mb + 1] = tq;
        stats[3 * mb + 2] = (double)(s1 - s0);
    }
}

// ---------------------------------------------------------------------------------------------
// Persistent epoch kernel: every minibatch of one epoch in ONE cooperative launch (one CTA per SM).
// Per minibatch: [stage parameters] -> forward/backward (grad_minibatch) -> grid barrier ->
// each CTA reduces its slice of the gradient over all CTAs' partials [-> one-shot all-reduce over
// NVLink peer memory: push the slice into every peer's inbox as tagged 8-byte packets, spin on the
// tags, sum in rank order] -> slice
// sum of squares -> grid barrier -> global-norm clip + Adam on the slice -> grid barrier.
// Replaces 3 launches (+ an NCCL call) per minibatch; everything is summed in a fixed order, so
// parameters stay bit-identical across ranks.
struct PeerXchg {
    int world, rank;
    int* err;                           // set to 1 when a peer's packets did not arrive in time
    unsigned long long* inbox;          // local  [2][world][stride] packets {seq << 32 | float bits}
    unsigned long long* peer_inbox[8];  // peers' inboxes (NVLink-mapped)
};

struct EpochArgs {
    GradArgs G;
    int64_t n_samples, batch;
    const double* stats;       // [n_mb][3] (global minibatch sums)
    float *params, *exp_avg, *exp_avg_sq;
    int64_t* step;
    float lr, beta1, beta2, eps, max_grad_norm;
    float* grad;               // [stride] last reduced gradient
    float* info;               // [n_mb][8] or NULL
    float* acc;                // [3][2 * TL.size] rotating gradient accumulators (zero at launch)
    float* gsum;               // [2 * TL.size] gradient summed over ranks (world > 1)
    unsigned* barrier;         // [1], zero at launch
    unsigned seq0;             // exchange sequence number before this launch
    PeerXchg X;
    float target_kl;           // SB3's target_kl (<= 0: off)           } read by the EXT instantiation only
    int* ctrl;                 // the update's control word             }
    int64_t mb0;               // index of this launch's first minibatch in the update
};

__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Split barrier: work placed between arrive and wait runs under the barrier's latency (~1 us).
__device__ __forceinline__ void grid_arrive(unsigned* counter, unsigned& target, unsigned n_cta) {
    __syncthreads();
    if (threadIdx.x == 0) {
        target += n_cta;
        // arrive = one release-reduction (no return value to wait for: the first poll leaves right behind it)
        asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(counter), "r"(1u) : "memory");
    }
}
__device__ __forceinline__ void grid_wait(unsigned* counter, unsigned target) {
    if (threadIdx.x == 0) {
        while (ld_acquire_gpu(counter) < target) {}
    }
    __syncthreads();
}
__device__ __forceinline__ void grid_barrier(unsigned* counter, unsigned& target, unsigned n_cta) {
    grid_arrive(counter, target, n_cta);
    grid_wait(counter, target);
}

// ---------------------------------------------------------------------------------------------
// Tensor-core epoch kernel.  Round 1's form of it (git history: 1.86 ms per epoch on the bench
// workload) spent 47 % of its time BETWEEN the tiles of consecutive minibatches:
//   then: 148 partial vectors -> L2 | barrier | every CTA pulls its 72-float slice from 74 partials |
//       barrier | clip + Adam on the slice | barrier | every CTA pulls its tower's new parameters.
//   now (1.40 ms): every CTA adds its partial into ONE accumulator with a single bulk reduction
//       (cp.reduce.async.bulk .add.f32, shared -> L2, 22 KB) | ONE barrier | every CTA reads the
//       whole reduced gradient (one wave of 12 float4 loads per thread), derives the clip
//       coefficient itself and applies Adam to ITS tower, whose fp32 master copy and moments live in
//       its shared memory for the whole epoch (74-fold redundant arithmetic instead of two more
//       grid-wide hand-offs); the updated W2 goes straight from the Adam registers into the fp16
//       operand panel.
// Three accumulators rotate (minibatch m uses m % 3; after barrier j the CTAs clear their slices of
// buffer (j - 1) % 3, whose readers all passed barrier j - 1 ... j).  The order in which the L2
// adds the 74 contributions is not fixed, so a single-GPU run is reproducible to rounding only
// (1e-7 of the gradient); every CTA reads the same sums, so the towers' copies -- and with more
// than one rank, the ranks -- stay bit-identical.
// World > 1: after the barrier the owner of each accumulator slice pushes it to every peer (tagged
// 8-byte packets over NVLink), sums the peers' slices in rank order into `gsum`, and a
// second barrier publishes the global sum.
__device__ __forceinline__ void bulk_reduce_add_f32(float* gdst, const float* ssrc, uint32_t bytes) {
    asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f32 [%0], [%1], %2;" ::"l"(gdst),
                 "r"(umma::smem_u32(ssrc)), "r"(bytes)
                 : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_all() {
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    asm volatile("fence.proxy.async.global;" ::: "memory");   // async-proxy writes before the generic release below
}

// EXT: SB3's clip_range_vf and target_kl compiled in.  The default instantiation (EXT = false) is the kernel
// without them, instruction for instruction.
// Early stop (target_kl): after the barrier (and the exchange) of minibatch m every CTA of every rank holds the same
// reduced statistics, so each computes approx_kl = kl_sum / count itself and takes the same decision without another
// barrier.  On a stop, Adam is skipped (parameters, moments and step stay those after minibatch m - 1), CTA 0 still
// writes info row m (step unchanged) and records mb0 + m + 1 in the control word, `grad` receives minibatch m's
// gradient, and the CTAs leave the loop for the normal write-back.  A launch that finds the control word set returns
// at entry in every CTA.
template <int KP, bool EXT>
__global__ void __launch_bounds__(tc::THREADS, 1) ppo_epoch_tc_kernel(EpochArgs E, int O) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    if (EXT && update_stopped(E.ctrl)) return;   // before any barrier: the update stopped in an earlier launch
    __shared__ double s_sq[tc::WARPS];
    __shared__ float s_kl;
    __shared__ float4 s_x[8 * 32];   // peers' packets of the slice threads (tid < q4 <= 32)
    const ParamLayout L = make_layout(O);
    const tc::TowerLayout TL = tc::make_tl(O);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int G = gridDim.x, c = blockIdx.x;
    const int n_mb = (int)((E.n_samples + E.batch - 1) / E.batch);
    const int acc_floats = 2 * TL.size;
    const int nq = acc_floats >> 2;        // quads of the accumulator
    const int q4 = (nq + G - 1) / G;       // quads per CTA slice (<= 32, checked on the host)
    const int my_quad = c * q4 + tid;
    const bool slice_t = tid < q4 && my_quad < nq;
    unsigned target = 0;
    int64_t step = E.step[0];
    double b1pow = pow((double)E.beta1, (double)step), b2pow = pow((double)E.beta2, (double)step);

    MR_TR(0);
    tc::Ctx C = tc::make_ctx(smem_raw, c & 1);
    tc::setup(C);
    float* st_w = reinterpret_cast<float*>(C.base + tc::OFF_STATE);
    float* st_m = st_w + TL.size;
    float* st_v = st_m + TL.size;
    float* stage = reinterpret_cast<float*>(C.base + tc::OFF_H1);   // H1 + dZ panels are idle between minibatches
    C.p_b2 = st_w + TL.b2;
    C.p_hw = st_w + TL.hw;
    C.p_hs = st_w + TL.hs;
    GradArgs A = E.G;
    const tc::Sched S{E.n_samples, E.batch, n_mb, c >> 1, G >> 1};
    tc::Pipe<KP> Q;
    tc::pipe_start<KP, true, EXT>(Q, A, S, O, tid & 127, tid >> 7, C.tower == 0);

    // the tower's parameters and Adam moments: flat global arrays -> shared memory, TL order
    for (int i = tid; i < TL.size; i += tc::THREADS) {
        const int p = tc::tl_to_flat(i, C.tower, TL, L, O);
        st_w[i] = p >= 0 ? E.params[p] : 0.f;
        st_m[i] = p >= 0 ? E.exp_avg[p] : 0.f;
        st_v[i] = p >= 0 ? E.exp_avg_sq[p] : 0.f;
    }
    __syncthreads();
    tc::panel_w1_from_tl<KP>(C, st_w, TL, O);
    tc::panel_w2_from_tl(C, st_w, TL);
    __syncthreads();

    tc::MbConst MK = tc::mb_const(E.stats, 0, A.normalize_adv);
    for (int m = 0; m < n_mb; ++m) {
        const float inv_cnt = MK.inv_b;
        float* accb = E.acc + (size_t)(m % 3) * acc_floats;
        // every CTA has passed barrier m - 1, i.e. nobody reads the accumulator of minibatch m - 2 any more
        if (m >= 2 && slice_t)
            __stcg(reinterpret_cast<float4*>(E.acc + (size_t)((m + 1) % 3) * acc_floats) + my_quad, make_float4(0.f, 0.f, 0.f, 0.f));
        MR_TR(2);
        const tc::TileAcc T = tc::tiles<KP, true, EXT>(C, A, S, MK, m, Q, O);
        if (T.any) {
            // the lane- and row-owned sums first (they do not need the last tile's dW1 GEMM, which finishes
            // meanwhile), then dW2 from TMEM and its bulk reduction, then dW1 and the sums
            float* dst = accb + (size_t)C.tower * TL.size;
            tc::stage_sums(C, T);
            tc::stage_w2(C, MK, TL, stage);
            umma::fence_proxy_async();   // the staged block (generic writes) -> the bulk reduction's reads
            __syncthreads();
            if (tid == 0) bulk_reduce_add_f32(dst + TL.w2, stage + TL.w2, (uint32_t)(TL.w1 - TL.w2) * 4u);
            tc::stage_rest<KP>(C, MK, O, TL, stage);
            umma::fence_proxy_async();
            __syncthreads();
            MR_TR(22);
            if (tid == 0) {
                bulk_reduce_add_f32(dst + TL.w1, stage + TL.w1, (uint32_t)(TL.size - TL.w1) * 4u);
                bulk_wait_all();
            }
        }
        MR_TR(3);
        grid_arrive(E.barrier, target, G);
        // the next minibatch's constants (two L2 loads, an fp64 division and a square root): after the arrive, so
        // that they cost nothing in front of the barrier (2 % of the stall samples sat on them there)
        if (m + 1 < n_mb) MK = tc::mb_const(E.stats, m + 1, A.normalize_adv);
        // ... and this step's fp64 scalars of Adam
        ++step;
        b1pow *= (double)E.beta1;   // beta^step, carried from one pow() per launch
        b2pow *= (double)E.beta2;
        tc::AdamK K;
        K.beta1 = E.beta1; K.beta2 = E.beta2; K.omb1 = 1.f - E.beta1; K.omb2 = 1.f - E.beta2;
        K.neg_step_size = (float)(-(double)E.lr / (1.0 - b1pow));
        K.bc2_sqrt = (float)sqrt(1.0 - b2pow);
        K.eps = E.eps;
        const float ent_loss = entropy_loss_of(C.p_hs[2], C.p_hs[3]);   // (policy tower) the log_std this minibatch used
        grid_wait(E.barrier, target);
        MR_TR(4);

        const float* src = accb;
        if (E.X.world > 1) {
            // one-shot all-reduce of this CTA's accumulator slice over NVLink peer memory: tagged 8-byte
            // packets {seq, float} into every peer's inbox, summed in rank order (bit-identical everywhere)
            if (slice_t) {
                const float4 mine = __ldcg(reinterpret_cast<const float4*>(accb) + my_quad);
                const float val[4] = {mine.x, mine.y, mine.z, mine.w};
                const unsigned seq = E.seq0 + (unsigned)m + 1u;
                const int slot = seq & 1u;
                // Inbox of (slot, source rank): two regions of nq 16-byte entries, {packet 0, packet 1} and
                // {packet 2, packet 3} of every quad, so that ONE 16-byte store per thread and region makes a warp's
                // push a contiguous range (a few full NVLink writes instead of a 32-byte sector per packet: at 8 ranks
                // the scalar form sent 79 000 sector-sized writes per minibatch and rank).  Every 8-byte packet still
                // carries its own tag, so the 16-byte stores need not arrive atomically.
                unsigned long long pk[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) pk[e] = ((unsigned long long)seq << 32) | (unsigned long long)__float_as_uint(val[e]);
                const size_t ent = ((size_t)slot * E.X.world + E.X.rank) * acc_floats + 2 * (size_t)my_quad;
                for (int r = 0; r < E.X.world; ++r)
                    if (r != E.X.rank) {
                        unsigned long long* dst = E.X.peer_inbox[r] + ent;
                        asm volatile("st.global.cg.v2.u64 [%0], {%1, %2};" ::"l"(dst), "l"(pk[0]), "l"(pk[1]) : "memory");
                        asm volatile("st.global.cg.v2.u64 [%0], {%1, %2};" ::"l"(dst + 2 * (size_t)nq), "l"(pk[2]), "l"(pk[3]) : "memory");
                    }
                // pull: the four packets of every peer, four peers per wave of 16-byte loads; payloads wait in
                // shared memory.  A peer that never delivers (dead rank) ends the wait after ~4 s: the flag is
                // raised and the epoch finishes on what arrived, so the GPU is released instead of hanging.
                const unsigned long long* src0 = E.X.inbox + (size_t)slot * E.X.world * acc_floats + 2 * (size_t)my_quad;
                unsigned pending = ((1u << E.X.world) - 1u) & ~(1u << E.X.rank);
                long long t0 = 0;
                unsigned spins = 0;
                while (pending) {
#pragma unroll
                    for (int half = 0; half < 2; ++half) {
                        ulonglong2 lo[4], hi[4];
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            const int r = 4 * half + k;
                            if (pending >> r & 1u) {
                                const unsigned long long* q = src0 + (size_t)r * acc_floats;
                                asm volatile("ld.relaxed.sys.global.v2.u64 {%0, %1}, [%2];" : "=l"(lo[k].x), "=l"(lo[k].y) : "l"(q) : "memory");
                                asm volatile("ld.relaxed.sys.global.v2.u64 {%0, %1}, [%2];" : "=l"(hi[k].x), "=l"(hi[k].y) : "l"(q + 2 * (size_t)nq) : "memory");
                            }
                        }
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            const int r = 4 * half + k;
                            if ((pending >> r & 1u) && (unsigned)(lo[k].x >> 32) == seq && (unsigned)(lo[k].y >> 32) == seq &&
                                (unsigned)(hi[k].x >> 32) == seq && (unsigned)(hi[k].y >> 32) == seq) {
                                s_x[r * 32 + tid] = make_float4(__uint_as_float((unsigned)lo[k].x), __uint_as_float((unsigned)lo[k].y),
                                                                __uint_as_float((unsigned)hi[k].x), __uint_as_float((unsigned)hi[k].y));
                                pending &= ~(1u << r);
                            }
                        }
                    }
                    if (pending && (++spins & 0xFFFu) == 0) {
                        long long now;
                        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                        if (t0 == 0) t0 = now;
                        else if (now - t0 > 4000000000ll) {
                            for (int r = 0; r < E.X.world; ++r)
                                if (pending >> r & 1u) s_x[r * 32 + tid] = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (E.X.err) *E.X.err = 1;
                            pending = 0;
                        }
                    }
                }
                float tot[4] = {0.f, 0.f, 0.f, 0.f};
                for (int r = 0; r < E.X.world; ++r) {
                    const float4 v = r == E.X.rank ? mine : s_x[r * 32 + tid];
                    tot[0] += v.x; tot[1] += v.y; tot[2] += v.z; tot[3] += v.w;
                }
                __stcg(reinterpret_cast<float4*>(E.gsum) + my_quad, make_float4(tot[0], tot[1], tot[2], tot[3]));
            }
            MR_TR(5);
            grid_barrier(E.barrier, target, G);
            MR_TR(6);
            src = E.gsum;
        }

        // ---- the whole reduced gradient: clip coefficient, then Adam on the own tower -------------------
        tc::BlockRegs<KP> gOwn, gOth;
        tc::load_block(src + (size_t)C.tower * TL.size, TL, gOwn);
        tc::load_block(src + (size_t)(C.tower ^ 1) * TL.size, TL, gOth);
        MR_TR(30);
        double sq = tc::finish_block(gOwn, TL, C.tower == 0, E.G.ent_coef) + tc::finish_block(gOth, TL, C.tower != 0, E.G.ent_coef);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
        if (lane == 0) s_sq[warp] = sq;
        if (EXT) {
            // the policy block's statistics quad: (loss, clipped count, kl sum, -)
            const int q_st = (TL.st - TL.w1) >> 2;
#pragma unroll
            for (int k = 0; k < tc::BlockRegs<KP>::NR; ++k)
                if (tid + k * tc::THREADS == q_st) s_kl = (C.tower == 0 ? gOwn.r[k].z : gOth.r[k].z) * inv_cnt;
        }
        __syncthreads();
        double tot = 0.0;
#pragma unroll
        for (int w = 0; w < tc::WARPS; ++w) tot += s_sq[w];
        const float total_norm = (float)sqrt(tot);
        K.coef = fminf(E.max_grad_norm / (total_norm + 1e-6f), 1.0f);
        MR_TR(31);
        const bool stop = EXT && E.target_kl > 0.f && (double)s_kl > 1.5 * (double)E.target_kl;
        if (!stop) tc::adam_block(C, gOwn, K, TL, st_w, st_m, st_v);
        else --step;   // SB3 breaks before optimizer.step(): the count stays that of minibatch m - 1
        MR_TR(7);
        // outputs of the API, off the other CTAs' critical path: statistics row (CTA 0), last gradient (CTAs 0, 1)
        if (c < 2) {
            const int q_st = (TL.st - TL.w1) >> 2;
            if (E.info && c == 0) {
                float* row = E.info + 8 * m;
                if (tid == 0) { row[0] = total_norm; row[1] = K.coef; row[2] = (float)step; row[3] = ent_loss; }
#pragma unroll
                for (int k = 0; k < tc::BlockRegs<KP>::NR; ++k)
                    if (tid + k * tc::THREADS == q_st) {   // policy: loss, clipped count, kl; value: squared error
                        row[4] = gOwn.r[k].x * inv_cnt; row[5] = gOth.r[k].x * inv_cnt;
                        row[6] = gOwn.r[k].y * inv_cnt; row[7] = gOwn.r[k].z * inv_cnt;
                    }
            }
            if (m == n_mb - 1 || stop) {
                const int sb = stat_base(O);
                if (EXT && c == 0) {   // the host does not clear `grad` for this instantiation: the pads here
                    for (int p = L.total + tid; p < grad_stride(O); p += tc::THREADS)
                        if (p < sb || p >= sb + 4) E.grad[p] = 0.f;
                }
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    const int idx = tid + k * tc::THREADS;
                    const int p = (C.tower ? L.vw2 : L.pw2) + (idx >> 3) * HID + 8 * (idx & 7);
                    const float4 a = gOwn.o[k][0], b = gOwn.o[k][1];
                    const float v8[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
                    for (int e = 0; e < 8; ++e) E.grad[p + e] = v8[e];
                }
#pragma unroll
                for (int k = 0; k < tc::BlockRegs<KP>::NR; ++k) {
                    const int qi = tid + k * tc::THREADS;
                    const float r4[4] = {gOwn.r[k].x, gOwn.r[k].y, gOwn.r[k].z, gOwn.r[k].w};
                    if (qi < ((TL.size - TL.w1) >> 2)) {
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const int pf = tc::tl_to_flat(TL.w1 + 4 * qi + e, C.tower, TL, L, O);
                            if (pf >= 0) E.grad[pf] = r4[e];
                        }
                        if (qi == q_st) {
                            if (C.tower == 0) { E.grad[sb] = r4[0] * inv_cnt; E.grad[sb + 2] = r4[1] * inv_cnt; E.grad[sb + 3] = r4[2] * inv_cnt; }
                            else E.grad[sb + 1] = r4[0] * inv_cnt;
                        }
                    }
                }
            }
        }
        if (stop && c == 0 && tid == 0) *E.ctrl = (int)(E.mb0 + m + 1);
        __syncthreads();   // the tower's new fp32 values (other threads' Adam) -> W1 panel, head vectors
        if (stop) break;   // uniform: every CTA read the same s_kl
        if (m + 1 < n_mb) tc::panel_w1_from_tl<KP>(C, st_w, TL, O);
        MR_TR(37);
    }
    // tower state back to the flat arrays (every CTA of a tower holds the same bits: one writes)
    if (c < 2) {
        for (int i = tid; i < TL.size; i += tc::THREADS) {
            const int p = tc::tl_to_flat(i, C.tower, TL, L, O);
            if (p >= 0) {
                E.params[p] = st_w[i];
                E.exp_avg[p] = st_m[i];
                E.exp_avg_sq[p] = st_v[i];
            }
        }
    }
    if (c == 0 && tid == 0) E.step[0] = step;
    tc::teardown(C);
}

}  // namespace mr

using namespace mr;

extern "C" {

int mr_ppo_grad_stride(int obs_dim) { return grad_stride(obs_dim); }
int mr_ppo_num_params(int obs_dim) { return make_layout(obs_dim).total; }
int mr_ppo_max_parts(void) { return sm_count(); }
int mr_ppo_epoch_scratch_floats(int obs_dim) { return 4 * 2 * tc::make_tl(obs_dim).size + 64; }

int mr_ppo_adv_stats(const float* adv, const int64_t* perm, int64_t n_samples, int64_t batch_size,
                     int64_t N, int64_t T, double* stats, void* stream) {
    MR_REQUIRE(adv && perm && stats, "NULL argument");
    MR_REQUIRE(batch_size > 0 && n_samples > 0, "empty batch");
    int n_mb = ceil_div(n_samples, batch_size);
    adv_stats_kernel<<<n_mb, 1024, 0, (cudaStream_t)stream>>>(adv, perm, n_samples, batch_size, N, T, stats, n_mb);
    MR_CHECK_LAUNCH();
    return MR_OK;
}


int mr_device_permutations(uint64_t seed, const uint64_t* h_stream_ids, int count, int64_t n, int64_t* out, void* stream) {
    MR_REQUIRE(out != nullptr && h_stream_ids != nullptr, "NULL argument");
    MR_REQUIRE(n > 0 && n < (int64_t(1) << 31), "n out of range");
    MR_REQUIRE(count > 0 && count <= MAX_PERMS, "1 to 32 permutations per call");
    PermKeys Ks{};
    for (int e = 0; e < count; ++e) Ks.k[e] = make_perm_key(seed, h_stream_ids[e], n);
    device_perm_kernel<<<dim3(ceil_div(n, 256), count), 256, 0, (cudaStream_t)stream>>>(out, n, Ks);
    MR_CHECK_LAUNCH();
    return MR_OK;
}

// Everything the epochs of one update need besides the parameters, for ALL epochs in two launches: the
// per-minibatch advantage sums (mr_ppo_adv_stats) and the samples as buffer rows.  perm [n_epochs][n_samples],
// stats [n_epochs][n_mb][3], rows [n_epochs][n_samples].  The permutations do not depend on the update, so
// nothing forces these small latency-bound kernels in between the epoch kernels (30 launches, 0.5 ms per
// iteration of the bench workload; with several ranks also ten NCCL calls instead of one).
int mr_ppo_prepare_epochs(const float* adv, const int64_t* perm, int n_epochs, int64_t n_samples, int64_t batch_size,
                          int64_t N, int64_t T, double* stats, int32_t* rows, void* stream) {
    MR_REQUIRE(adv && perm && stats && rows, "NULL argument");
    MR_REQUIRE(batch_size > 0 && n_samples > 0 && n_epochs > 0, "empty batch");
    MR_REQUIRE(n_samples * n_epochs < (int64_t(1) << 40) && N * T < (int64_t(1) << 31), "sizes out of range");
    cudaStream_t s = (cudaStream_t)stream;
    const int n_mb = ceil_div(n_samples, batch_size);
    adv_stats_kernel<<<n_mb * n_epochs, 1024, 0, s>>>(adv, perm, n_samples, batch_size, N, T, stats, n_mb);
    MR_CHECK_LAUNCH();
    perm_to_rows_kernel<<<ceil_div(n_samples * n_epochs, 256), 256, 0, s>>>(perm, n_samples * n_epochs, N, T, rows);
    MR_CHECK_LAUNCH();
    return MR_OK;
}

// mr_device_permutations + mr_ppo_prepare_epochs in two launches, without materialising the int64 permutations.
int mr_ppo_prepare_epochs_device(uint64_t seed, const uint64_t* h_stream_ids, int n_epochs, const float* adv,
                                 int64_t n_samples, int64_t batch_size, int64_t N, int64_t T, double* stats,
                                 int32_t* rows, void* stream) {
    MR_REQUIRE(adv && h_stream_ids && stats && rows, "NULL argument");
    MR_REQUIRE(n_samples > 0 && n_samples == N * T && n_samples < (int64_t(1) << 31), "n_samples must equal N * T (< 2^31)");
    MR_REQUIRE(n_epochs > 0 && n_epochs <= MAX_PERMS && batch_size > 0, "1 to 32 epochs per call");
    cudaStream_t s = (cudaStream_t)stream;
    PermKeys Ks{};
    for (int e = 0; e < n_epochs; ++e) Ks.k[e] = make_perm_key(seed, h_stream_ids[e], n_samples);
    device_rows_kernel<<<dim3(ceil_div(n_samples, 256), n_epochs), 256, 0, s>>>(rows, n_samples, N, T, Ks);
    MR_CHECK_LAUNCH();
    const int n_mb = ceil_div(n_samples, batch_size);
    adv_stats_rows_kernel<<<n_mb * n_epochs, 1024, 0, s>>>(adv, rows, n_samples, batch_size, stats, n_mb);
    MR_CHECK_LAUNCH();
    return MR_OK;
}

int mr_ppo_grad(const float* params, int obs_dim, const float* obs, const float* act,
                const float* old_logp, const float* adv, const float* ret, const int64_t* perm,
                int32_t* rows, int64_t mb_size, const double* mb_stats, int64_t N, int64_t T,
                float clip_range, float ent_coef, float vf_coef, int normalize_adv, float rank_share,
                float* partials, float* grad, const float* old_values, float clip_range_vf, const int* ctrl,
                void* stream) {
    MR_REQUIRE(params && obs && act && old_logp && adv && ret && perm && rows && mb_stats && partials && grad,
               "NULL argument");
    MR_REQUIRE(obs_dim > 0 && obs_dim <= MAX_OBS, "obs_dim out of range");
    MR_REQUIRE(mb_size > 0, "empty minibatch");
    const bool vf = clip_range_vf > 0.f;
    MR_REQUIRE(!vf || old_values, "clip_range_vf needs the rollout's values");
    GradArgs A{params, obs, act, old_logp, adv, ret, perm, nullptr, nullptr, mb_size, mb_stats, N, T,
               clip_range, ent_coef, vf_coef, normalize_adv, partials, old_values, clip_range_vf, ctrl};
    static OncePerDevice once;
    if (once.first()) {
        MR_CUDA(cudaFuncSetAttribute(ppo_grad_tc_kernel<16, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_BYTES));
        MR_CUDA(cudaFuncSetAttribute(ppo_grad_tc_kernel<32, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_BYTES));
        MR_CUDA(cudaFuncSetAttribute(ppo_grad_tc_kernel<16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_BYTES));
        MR_CUDA(cudaFuncSetAttribute(ppo_grad_tc_kernel<32, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_BYTES));
    }
    const int max_parts = mr_ppo_max_parts();
    cudaStream_t s = (cudaStream_t)stream;
    MR_REQUIRE(obs_dim < 32 && max_parts >= 2, "the tensor-core kernels need obs_dim < 32");
    MR_REQUIRE(N * T < (int64_t(1) << 31), "samples are indexed with 32 bits");
    perm_to_rows_kernel<<<ceil_div(mb_size, 256), 256, 0, s>>>(perm, mb_size, N, T, rows);
    MR_CHECK_LAUNCH();
    A.rows = rows;
    // obs_dim + 1 (bias column) padded to the 16-bit MMA K of 16
    const int kp = obs_dim + 1 <= 16 ? 16 : 32;
    const int64_t tiles = (mb_size + tc::TILE - 1) / tc::TILE;
    const int grid = (int)std::min<int64_t>(2 * tiles, max_parts & ~1);
    if (kp == 16) {
        if (vf) ppo_grad_tc_kernel<16, true><<<grid, tc::THREADS, tc::SMEM_BYTES, s>>>(A, obs_dim);
        else ppo_grad_tc_kernel<16, false><<<grid, tc::THREADS, tc::SMEM_BYTES, s>>>(A, obs_dim);
    } else {
        if (vf) ppo_grad_tc_kernel<32, true><<<grid, tc::THREADS, tc::SMEM_BYTES, s>>>(A, obs_dim);
        else ppo_grad_tc_kernel<32, false><<<grid, tc::THREADS, tc::SMEM_BYTES, s>>>(A, obs_dim);
    }
    MR_CHECK_LAUNCH();
    const int stride = grad_stride(obs_dim);
    ppo_reduce_kernel<<<ceil_div(stride, 128), 128, 0, s>>>(partials, grid, obs_dim, ent_coef, mb_stats, grad,
                                                            rank_share, ctrl);
    MR_CHECK_LAUNCH();
    return MR_OK;
}

int mr_adam_step(float* params, float* exp_avg, float* exp_avg_sq, const float* grad, int n_params,
                 int64_t* step, float lr, float beta1, float beta2, float eps, float max_grad_norm,
                 float* info, float target_kl, int* ctrl, int64_t mb_index, void* stream) {
    MR_REQUIRE(params && exp_avg && exp_avg_sq && grad && step, "NULL argument");
    MR_REQUIRE(!(target_kl > 0.f) || ctrl, "target_kl needs a control word");
    AdamArgs A{params, exp_avg, exp_avg_sq, grad, step, lr, beta1, beta2, eps, max_grad_norm, info, n_params,
               target_kl, ctrl, mb_index};
    adam_kernel<<<ceil_div(n_params, ADAM_THREADS), ADAM_THREADS, 0, (cudaStream_t)stream>>>(A);
    MR_CHECK_LAUNCH();
    return MR_OK;
}

int mr_ppo_train_summary(const float* info, int n_rows, const float* values, const float* returns, int64_t n,
                         const float* params, float* out, double* scratch, const int* ctrl, void* stream) {
    MR_REQUIRE(info && values && returns && params && out && scratch, "NULL argument");
    MR_REQUIRE(n_rows > 0 && n > 0, "empty summary");
    const int grid = (int)std::min<int64_t>(sm_count(), (n + 255) / 256);
    train_summary_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(info, n_rows, values, returns, n, params, out, scratch,
                                                                 ctrl);
    MR_CHECK_LAUNCH();
    return MR_OK;
}

int mr_ppo_train_epoch(float* params, float* exp_avg, float* exp_avg_sq, int64_t* step, int obs_dim,
                       const float* obs, const float* act, const float* old_logp, const float* adv,
                       const float* ret, const int64_t* perm, int32_t* rows, int64_t n_samples,
                       int64_t batch_size, const double* stats, int64_t N, int64_t T, float clip_range,
                       float ent_coef, float vf_coef, int normalize_adv, float lr, float beta1, float beta2,
                       float eps, float max_grad_norm, float* partials, float* grad, float* info,
                       const float* old_values, float clip_range_vf, float target_kl, int* ctrl, int64_t mb0,
                       void* stream) {
    MR_REQUIRE(batch_size > 0 && n_samples > 0, "empty batch");
    const int n_params = make_layout(obs_dim).total;
    const int64_t n_mb = (n_samples + batch_size - 1) / batch_size;
    for (int64_t mb = 0; mb < n_mb; ++mb) {
        const int64_t s0 = mb * batch_size;
        const int64_t sz = std::min(batch_size, n_samples - s0);
        int rc = mr_ppo_grad(params, obs_dim, obs, act, old_logp, adv, ret, perm + s0, rows, sz, stats + 3 * mb, N, T,
                             clip_range, ent_coef, vf_coef, normalize_adv, 1.0f, partials, grad, old_values,
                             clip_range_vf, ctrl, stream);
        if (rc != MR_OK) return rc;
        rc = mr_adam_step(params, exp_avg, exp_avg_sq, grad, n_params, step, lr, beta1, beta2, eps,
                          max_grad_norm, info ? info + 8 * mb : nullptr, target_kl, ctrl, mb0 + mb, stream);
        if (rc != MR_OK) return rc;
    }
    return MR_OK;
}

#ifdef MR_TRACE
// debug build only: copy out and clear the phase trace of CTA `cta` (0 or 1); returns the count
int mr_trace_read(int cta, unsigned long long* out, int cap) {
    unsigned n = 0;
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(&n, mr::g_trace_n, sizeof(unsigned), cta * sizeof(unsigned));
    if ((int)n > cap) n = cap;
    cudaMemcpyFromSymbol(out, mr::g_trace, n * sizeof(unsigned long long), (size_t)cta * 4096 * sizeof(unsigned long long));
    unsigned z = 0;
    cudaMemcpyToSymbol(mr::g_trace_n, &z, sizeof(unsigned), cta * sizeof(unsigned));
    return (int)n;
}
#endif

struct mr_xchg {
    int world, rank, device, n_cta;
    int64_t stride;        // packets per (slot, rank) = floats of the epoch kernel's accumulator
    void* base;            // local allocation: inbox packets, then the status word
    size_t bytes;
    void* peer_base[8];
    unsigned seq;          // exchange sequence number (host mirror)
};

static int64_t xchg_stride(int obs_dim) { return 2 * (int64_t)tc::make_tl(obs_dim).size; }
static size_t xchg_inbox_bytes(int world, int64_t stride) {
    return (size_t)2 * world * stride * sizeof(unsigned long long);
}

int mr_xchg_create(int world, int rank, int device, int obs_dim, mr_xchg** out, uint8_t* h_handle_out) {
    MR_REQUIRE(out && h_handle_out, "NULL argument");
    MR_REQUIRE(world >= 1 && world <= 8 && rank >= 0 && rank < world, "bad world/rank");
    DeviceGuard guard(device);   // the caller's current device is left as it was
    mr_xchg* x = new mr_xchg();
    x->world = world; x->rank = rank; x->device = device;
    x->n_cta = mr_ppo_max_parts();
    x->stride = xchg_stride(obs_dim);
    x->bytes = xchg_inbox_bytes(world, x->stride) + 256;
    x->seq = 0;
    for (int r = 0; r < 8; ++r) x->peer_base[r] = nullptr;
    cudaError_t e = cudaMalloc(&x->base, x->bytes);
    if (e != cudaSuccess) { set_error("cudaMalloc failed: %s", cudaGetErrorString(e)); delete x; return MR_ERR_ALLOC; }
    MR_CUDA(cudaMemset(x->base, 0, x->bytes));
    cudaIpcMemHandle_t h;
    MR_CUDA(cudaIpcGetMemHandle(&h, x->base));
    static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
    memcpy(h_handle_out, &h, 64);
    x->peer_base[rank] = x->base;
    *out = x;
    return MR_OK;
}

int mr_xchg_connect(mr_xchg* x, const uint8_t* h_all_handles) {
    MR_REQUIRE(x && h_all_handles, "NULL argument");
    DeviceGuard guard(x->device);
    for (int r = 0; r < x->world; ++r) {
        if (r == x->rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, h_all_handles + 64 * r, 64);
        MR_CUDA(cudaIpcOpenMemHandle(&x->peer_base[r], h, cudaIpcMemLazyEnablePeerAccess));
    }
    return MR_OK;
}

static int* xchg_status_word(mr_xchg* x) {
    return reinterpret_cast<int*>(static_cast<char*>(x->base) + xchg_inbox_bytes(x->world, x->stride));
}

int mr_xchg_status(mr_xchg* x, int* timed_out) {
    MR_REQUIRE(x && timed_out, "NULL argument");
    DeviceGuard guard(x->device);
    MR_CUDA(cudaMemcpy(timed_out, xchg_status_word(x), sizeof(int), cudaMemcpyDeviceToHost));
    return MR_OK;
}

void mr_xchg_destroy(mr_xchg* x) {
    if (!x) return;
    DeviceGuard guard(x->device);
    for (int r = 0; r < x->world; ++r)
        if (r != x->rank && x->peer_base[r]) cudaIpcCloseMemHandle(x->peer_base[r]);
    cudaFree(x->base);
    delete x;
}

int mr_ppo_record_floats(int obs_dim) { return (obs_dim + 1 <= 16 ? 16 : 32) + 8; }

int mr_ppo_pack_samples(int obs_dim, const float* obs, const float* act, const float* old_logp, const float* adv,
                        const float* ret, const float* values, int64_t n_rows, float* rec, void* stream) {
    MR_REQUIRE(obs && act && old_logp && adv && ret && rec, "NULL argument");
    MR_REQUIRE(obs_dim > 0 && obs_dim < MAX_OBS, "obs_dim out of range (1..31: the record's row of X is obs and the ones column)");
    MR_REQUIRE(n_rows > 0, "empty buffer");
    const int kp = obs_dim + 1 <= 16 ? 16 : 32;
    const int64_t quads = n_rows * ((kp + 8) >> 2);
    pack_samples_kernel<<<ceil_div(quads, 256), 256, 0, (cudaStream_t)stream>>>(obs, act, old_logp, adv, ret, values,
                                                                                n_rows, obs_dim, kp, rec);
    MR_CHECK_LAUNCH();
    return MR_OK;
}

int mr_ppo_epoch_fused(float* params, float* exp_avg, float* exp_avg_sq, int64_t* step, int obs_dim,
                       const float* rec, const int64_t* perm, int32_t* rows, int64_t n_samples,
                       int64_t batch_size, const double* stats, int64_t N, int64_t T,
                       float clip_range, float ent_coef, float vf_coef, int normalize_adv, float lr,
                       float beta1, float beta2, float eps, float max_grad_norm, float* partials,
                       float* grad, float* info, mr_xchg* xchg, float clip_range_vf, float target_kl, int* ctrl,
                       int64_t mb0, void* stream) {
    MR_REQUIRE(params && exp_avg && exp_avg_sq && step && rec && rows && stats && partials && grad,
               "NULL argument");   // perm may be NULL: rows then already hold the epoch's samples (mr_ppo_prepare_epochs)
    MR_REQUIRE(!(target_kl > 0.f) || ctrl, "target_kl needs a control word");
    // the extended instantiation (value clipping, early stop) only where asked for: the default one is unchanged
    const bool ext = clip_range_vf > 0.f || target_kl > 0.f || ctrl != nullptr;
    MR_REQUIRE(obs_dim > 0 && obs_dim < MAX_OBS, "obs_dim out of range (1..31: the row of X is obs and the ones column)");
    MR_REQUIRE(batch_size > 0 && n_samples > 0, "empty batch");
    MR_REQUIRE(n_samples < (int64_t(1) << 31) && N * T < (int64_t(1) << 31), "samples are indexed with 32 bits");
    cudaStream_t s = (cudaStream_t)stream;
    const int n_cta = mr_ppo_max_parts();
    MR_REQUIRE((n_cta & 1) == 0, "the epoch kernel needs an even CTA count (one tower per CTA)");
    const int stride = grad_stride(obs_dim);
    const tc::TowerLayout TL = tc::make_tl(obs_dim);
    const int acc_floats = 2 * TL.size;
    MR_REQUIRE(((int64_t)n_cta + 1) * stride >= mr_ppo_epoch_scratch_floats(obs_dim), "partials scratch too small");
    MR_REQUIRE((acc_floats / 4 + n_cta - 1) / n_cta <= 32, "accumulator slice per CTA too wide");
    // Everything the launch synchronises through lives in the CALLER's scratch (`partials`), so two
    // updaters (different streams) never share a barrier word: [3 accumulators | global sum | barrier word]
    EpochArgs E;
    E.G = GradArgs{params, nullptr, nullptr, nullptr, nullptr, nullptr, perm, rows, rec, 0, stats, N, T,
                   clip_range, ent_coef, vf_coef, normalize_adv, partials};
    E.n_samples = n_samples; E.batch = batch_size; E.stats = stats;
    E.params = params; E.exp_avg = exp_avg; E.exp_avg_sq = exp_avg_sq; E.step = step;
    E.lr = lr; E.beta1 = beta1; E.beta2 = beta2; E.eps = eps; E.max_grad_norm = max_grad_norm;
    E.grad = grad; E.info = info;
    E.acc = partials;
    E.gsum = partials + 3 * (size_t)acc_floats;
    E.barrier = reinterpret_cast<unsigned*>(partials + 4 * (size_t)acc_floats);
    MR_CUDA(cudaMemsetAsync(partials, 0, (4 * (size_t)acc_floats + 16) * sizeof(float), s));
    if (!ext) MR_CUDA(cudaMemsetAsync(grad, 0, (size_t)stride * sizeof(float), s));   // (ext: the kernel clears the pads)
    E.G.clip_vf = clip_range_vf;   // the records carry old_value (mr_ppo_pack_samples' values) when this is > 0
    E.target_kl = target_kl; E.ctrl = ctrl; E.mb0 = mb0;
    E.X.world = 1; E.X.rank = 0; E.X.inbox = nullptr; E.X.err = nullptr;
    E.seq0 = 0;
    const int64_t n_mb = (n_samples + batch_size - 1) / batch_size;
    if (xchg && xchg->world > 1) {
        MR_REQUIRE(xchg->stride == acc_floats && xchg->n_cta == n_cta, "exchange buffer mismatch");
        E.X.world = xchg->world; E.X.rank = xchg->rank;
        for (int r = 0; r < xchg->world; ++r)
            E.X.peer_inbox[r] = reinterpret_cast<unsigned long long*>(xchg->peer_base[r]);
        E.X.inbox = E.X.peer_inbox[xchg->rank];
        E.X.err = xchg_status_word(xchg);
        E.seq0 = xchg->seq;
        xchg->seq += (unsigned)n_mb;
    }
    const int kp = obs_dim + 1 <= 16 ? 16 : 32;
    const size_t smem = (size_t)tc::SMEM_BYTES + 3 * (size_t)TL.size * sizeof(float);
    static OncePerDevice once;
    if (once.first()) {
        const int smem_max = (int)((size_t)tc::SMEM_BYTES + 3 * (size_t)tc::make_tl(MAX_OBS - 1).size * sizeof(float));
        MR_CUDA(cudaFuncSetAttribute(ppo_epoch_tc_kernel<16, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
        MR_CUDA(cudaFuncSetAttribute(ppo_epoch_tc_kernel<32, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
        MR_CUDA(cudaFuncSetAttribute(ppo_epoch_tc_kernel<16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
        MR_CUDA(cudaFuncSetAttribute(ppo_epoch_tc_kernel<32, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
    }
    if (perm) {
        perm_to_rows_kernel<<<ceil_div(n_samples, 256), 256, 0, s>>>(perm, n_samples, N, T, rows);
        MR_CHECK_LAUNCH();
    }
    int O = obs_dim;
    void* args[] = {&E, &O};
    const void* fn = kp == 16 ? (ext ? (const void*)ppo_epoch_tc_kernel<16, true> : (const void*)ppo_epoch_tc_kernel<16, false>)
                              : (ext ? (const void*)ppo_epoch_tc_kernel<32, true> : (const void*)ppo_epoch_tc_kernel<32, false>);
    MR_CUDA(cudaLaunchCooperativeKernel(fn, dim3(n_cta), dim3(tc::THREADS), args, smem, s));
    mr::count_launch();
    return MR_OK;
}

}  // extern "C"
