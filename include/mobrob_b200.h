/* libmobrob_b200.so -- C ABI of the B200-native goal-conditioned PPO hot path.
 *
 * The reference (ZikangXiong/mobrob) is pure Python and has no FFI of its own: its
 * boundaries are three Python protocols (EnvWrapper, SB3 VecEnv, SB3 PPO).  The host
 * layer in mobrob_b200/ mirrors those protocols and binds this library with ctypes
 * (INTEGRATION.md shows the stub).  Each entry point below names the reference
 * interface it replaces (paths relative to the reference checkout; [SB3]/[GYM]/[MJ]
 * are its un-vendored dependencies stable-baselines3 2.0.0 / gymnasium 0.28.1 /
 * MuJoCo 2.1.0).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer on the handle's device unless its name starts
 *     with h_ (host); buffers are caller-owned (torch tensors on the Python side) and
 *     only borrowed for the duration of the stream-ordered call;
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous on it;
 *   - return 0 on success, a negative mr_status otherwise; mr_last_error() gives the
 *     message (thread local); nothing throws or aborts;
 *   - there is no CPU fallback anywhere in this library.
 */
#ifndef MOBROB_B200_H
#define MOBROB_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    MR_OK = 0,
    MR_ERR_ARG = -1,
    MR_ERR_CUDA = -2,
    MR_ERR_ALLOC = -3,
    MR_ERR_UNSUPPORTED = -4
} mr_status;

enum { MR_ENV_POINT = 0, MR_ENV_CAR = 1 };

typedef struct mr_env mr_env;

int mr_version(void);
const char* mr_last_error(void);
/* number of kernels this library has launched in this process (bench.py: gpu_launches) */
uint64_t mr_launch_count(void);

/* ------------------------------------------------------------------------------------
 * Batched goal environment.  Replaces, for N environments at once,
 *   EnvWrapper.__init__/build_env        src/mobrob/envs/wrapper.py:16-37, 238-242
 *   get_env(..., terminate_on_goal, time_limit) + [GYM] TimeLimit   wrapper.py:549-571
 *   [SB3] make_vec_env / Monitor / DummyVecEnv   src/mobrob/rl_control/ppo.py:37-48
 * kind: MR_ENV_POINT (xmls/point.xml) or MR_ENV_CAR (xmls/car.xml).
 * time_limit <= 0 means no TimeLimit wrapper (examples/control.py semantics). */
int mr_env_create(int kind, int64_t n_envs, int device, int time_limit, int terminate_on_goal,
                  mr_env** out);
void mr_env_destroy(mr_env* env);
int mr_env_obs_dim(const mr_env* env);   /* point 14, car 26 (engine.py:420-567), plus the optional keys below */

/* Optional keys of Engine.obs() (config flags engine.py:125,140-142; values engine.py:1179-1180, 1243-1248; the
 * reference sets them through MujocoGoalEnv.get_robot_config, wrapper.py:235-240): bit 0 observe_goal_dist
 * (exp(-|goal - pos|), 1 float), bit 1 observe_qpos (data.qpos: point 3, car 13), bit 2 observe_qvel (data.qvel:
 * point 3, car 11), bit 3 observe_ctrl (data.ctrl, 2), bit 4 observe_goal_lidar (the pseudo-lidar of the goal,
 * engine.py:1092-1172: lidar_num_bins floats, see mr_env_set_lidar).  The row stays the concatenation in sorted key
 * order (engine.py:1253-1259).  Call before the first reset; rows of obs / term_obs then have mr_env_obs_dim floats.
 * MR_ERR_UNSUPPORTED for other bits (the natural lidar, object lidars, vision and hazards are outside the path). */
#define MR_OBS_GOAL_DIST 1u
#define MR_OBS_QPOS 2u
#define MR_OBS_QVEL 4u
#define MR_OBS_CTRL 8u
#define MR_OBS_GOAL_LIDAR 16u
int mr_env_set_obs_flags(mr_env* env, unsigned flags);
/* Engine's pseudo-lidar settings for MR_OBS_GOAL_LIDAR (config keys lidar_num_bins, lidar_max_dist, lidar_exp_gain,
 * lidar_alias; lidar_type 'pseudo'): num_bins >= 1 (else MR_ERR_ARG); max_dist <= 0 means None (sensor =
 * exp(-exp_gain * dist)), otherwise sensor = max(0, max_dist - dist) / max_dist; alias != 0 spreads each reading over
 * the two neighbouring bins.  Defaults: 10 bins, None, 1.0, alias on.  Call before the first reset, like
 * mr_env_set_obs_flags. */
int mr_env_set_lidar(mr_env* env, int num_bins, double max_dist, double exp_gain, int alias);
int mr_env_state_dim(const mr_env* env); /* doubles per env in get/set_state */

/* Test hook (car): 0 disables the floor contacts, giving the contact-free trajectories on which
 * BASELINE.json asks for 1e-5 state parity.  Default 1. */
int mr_env_set_contacts(mr_env* env, int enabled);

/* EnvWrapper.reset_init_space / reset_goal_space (wrapper.py:209-219) for every env of the batch: resets after
 * this call draw the start position / the goal from the new boxes (defaults: MujocoGoalEnv.get_init_space /
 * get_goal_space, wrapper.py:250-264).  h_init, h_goal: (low x, low y, high x, high y) float32 in host memory;
 * either may be NULL (unchanged).  Each env keeps its own random stream. */
int mr_env_set_spaces(mr_env* env, const float* h_init, const float* h_goal, void* stream);

/* EnvWrapper.seed (wrapper.py:95-107) for every env: the two gymnasium Box streams
 * (init_space -> PCG64(SeedSequence(s)), goal_space -> PCG64(SeedSequence(s + 1))) arrive as
 * raw PCG64 words [N][4] = (state_hi, state_lo, inc_hi, inc_lo); engine_seed [N] is
 * Engine._seed (engine.py:629-631).  Host pointers, copied before returning. */
int mr_env_seed(mr_env* env, const uint64_t* h_pcg_init, const uint64_t* h_pcg_goal,
                const int64_t* h_engine_seed, void* stream);

/* EnvWrapper.reset (wrapper.py:173-201) for the envs with mask[i] != 0 (mask NULL = all).
 * first != 0 forces the full robot reset of the first call (wrapper.py:182); otherwise the
 * robot is re-placed only when the goal is not reached.  Samples come from the seeded
 * reference streams on the device.  obs_out [N][O] float32 rows are written for masked envs. */
int mr_env_reset(mr_env* env, const uint8_t* mask, int first, float* obs_out, void* stream);

/* [SB3] VecEnv.step_wait over EnvWrapper.step (wrapper.py:156-171), Engine.step
 * (engine.py:1392-1464: clip, 10 x mj_step, mj_forward), reward_fn (wrapper.py:137-154),
 * reached (wrapper.py:203-207), TimeLimit, Monitor and the auto-reset.
 *   act      [N][2] f32 in     obs      [N][O] f32 out (post-reset row where done)
 *   rew      [N] f32 out       done     [N] u8 out
 *   trunc    [N] u8 out        (= info["TimeLimit.truncated"])
 *   term_obs [N][O] f32 out    (= info["terminal_observation"], written where done; may be NULL)
 *   ep_ret   [N] f64 out, ep_len [N] i32 out (= info["episode"] r / l, valid where done; may be NULL) */
int mr_env_step(mr_env* env, const float* act, float* obs, float* rew, uint8_t* done,
                uint8_t* trunc, float* term_obs, double* ep_ret, int32_t* ep_len, void* stream);

/* EnvWrapper.get_obs (wrapper.py:272-273 -> Engine.obs, engine.py:1174-1263). */
int mr_env_get_obs(mr_env* env, float* obs_out, void* stream);
/* Reference-view state, [N][state_dim] float64.
 * point (15): qpos(3) qvel(3) body_pos_xy(2) start_heading(1) ctrl(2) goal_xy(2) elapsed(1) ep_ret(1)
 * car (30):   qpos(13) qvel(11) ctrl(2) goal_xy(2) elapsed(1) ep_ret(1), MuJoCo joint order */
int mr_env_get_state(mr_env* env, double* state_out, void* stream);
int mr_env_set_state(mr_env* env, const double* state_in, void* stream);
/* EnvWrapper.get_pos (wrapper.py:269-270): world xy, [N][2] float64. */
int mr_env_get_pos(mr_env* env, double* pos_out, void* stream);
/* counters for tests: [N][2] int32 = (#resets, #full resets) */
int mr_env_get_reset_counts(mr_env* env, int32_t* out, void* stream);

/* ------------------------------------------------------------------------------------
 * Policy.  Replaces [SB3] ActorCriticPolicy("MlpPolicy") forward / predict_values /
 * predict(deterministic=True) (call sites ppo.py:50-59, examples/control.py:39).
 * params: the 13 state-dict tensors of the shipped zips flattened in state-dict order
 * (log_std, policy_net.0.w/b, policy_net.2.w/b, value_net.0.w/b, value_net.2.w/b,
 * action_net.w/b, value_net.w/b): 10437 floats for O=14, 11973 for O=26.
 *   eps  [n][2] f32 standard normal draws, or NULL for the deterministic mean
 *   act  [n][2] f32 out (unclipped: mu + exp(log_std) * eps, or mu)
 *   logp [n] f32 out (may be NULL), val [n] f32 out (may be NULL) */
int mr_policy_forward(const float* params, int obs_dim, const float* obs, const float* eps,
                      float* act, float* logp, float* val, int64_t n, void* stream);

/* [SB3] RolloutBuffer.compute_returns_and_advantage in numpy's exact dtype flow (float32 deltas,
 * float64 running advantage, no FMA) -- bit-identical to the numpy loop.
 * All arrays [T][N] f32 time-major; last_val [N] f32, last_done [N] u8. */
int mr_gae(const float* rew, const float* val, const float* ep_start, const float* last_val,
           const uint8_t* last_done, double gamma, double lam, float* adv, float* ret, int64_t T,
           int64_t N, void* stream);

/* ------------------------------------------------------------------------------------
 * PPO update.  Replaces the inner loop of [SB3] PPO.train + torch autograd +
 * clip_grad_norm_ + torch.optim.Adam (reference call chain: examples/train.py:42-46 ->
 * src/mobrob/rl_control/ppo.py:73-74 -> PPO.learn).  Rollout arrays are time-major
 * [T][N](...) float32 as in RolloutBuffer; perm holds env-major sample ids (n * T + t), i.e.
 * indices into RolloutBuffer.swap_and_flatten order, int64 like np.random.permutation. */
int mr_ppo_num_params(int obs_dim);  /* 10437 (point) / 11973 (car) */
int mr_ppo_grad_stride(int obs_dim); /* floats in a gradient vector incl. the 16-slot stats tail:
                                        [policy_loss, value_loss, clip_fraction, approx_kl, ...] */
int mr_ppo_max_parts(void);          /* CTAs the update kernels use on the current device.  The `partials`
                                        scratch below holds (mr_ppo_max_parts() + 1) rows of
                                        mr_ppo_grad_stride() floats; it is caller-owned, and everything a
                                        launch synchronises through lives in it (two updaters on different
                                        streams never share state inside the library) */
int mr_ppo_epoch_scratch_floats(int obs_dim); /* part of `partials` mr_ppo_epoch_fused zeroes per launch */

/* (sum adv, sum adv^2, count) per minibatch of one epoch's permutation -> stats [n_mb][3] f64.
 * With several ranks the host all-reduces stats so that normalisation is over the global
 * minibatch, as PPO.train normalises over the whole minibatch. */
int mr_ppo_adv_stats(const float* adv, const int64_t* perm, int64_t n_samples, int64_t batch_size,
                     int64_t N, int64_t T, double* stats, void* stream);

/* evaluate_actions + loss + analytic backward for one minibatch (perm points at its slice).
 * mb_stats = the minibatch's (global) stats triple.  rank_share = local count / global count.
 * rows [mb_size] int32 caller-owned scratch (the samples as time-major buffer rows t * N + n);
 * partials [mr_ppo_max_parts() + 1][stride] scratch; grad [stride] out: d(loss)/d(params) of this
 * rank's share (sum over ranks = SB3's gradient) followed by the stats tail. */
int mr_ppo_grad(const float* params, int obs_dim, const float* obs, const float* act,
                const float* old_logp, const float* adv, const float* ret, const int64_t* perm,
                int32_t* rows, int64_t mb_size, const double* mb_stats, int64_t N, int64_t T,
                float clip_range, float ent_coef, float vf_coef, int normalize_adv, float rank_share,
                float* partials, float* grad, const float* old_values, float clip_range_vf, const int* ctrl,
                void* stream);

/* clip_grad_norm_(max_grad_norm) then torch.optim.Adam.step (eps as given; SB3 uses 1e-5).
 * step: device int64[2]: [0] = Adam step count (state["step"]), incremented; [1] = launch-internal
 * ticket that must start at 0.  info [8] out (may be NULL):
 * total grad norm, clip coefficient, step, the minibatch's entropy_loss (from the log_std it was
 * evaluated with), then grad's stats tail (policy_loss, value_loss, clip_fraction, approx_kl) so that
 * logging needs no extra copy. */
int mr_adam_step(float* params, float* exp_avg, float* exp_avg_sq, const float* grad, int n_params,
                 int64_t* step, float lr, float beta1, float beta2, float eps, float max_grad_norm,
                 float* info, float target_kl, int* ctrl, int64_t mb_index, void* stream);

/* ------------------------------------------------------------------------------------
 * Fused rollout.  Replaces [SB3] OnPolicyAlgorithm.collect_rollouts (n_steps = T) over the
 * vectorised env, including the time-out bootstrap  reward += gamma * V(terminal_obs),
 * Monitor's episode statistics and RolloutBuffer.add, in one launch (point env; plus two
 * launches that file the finished episodes).
 *   last_obs [N][O], last_starts [N] f32 : in/out, carried between rollouts (_last_obs,
 *                                          _last_episode_starts)
 *   obs [T][N][O], act [T][N][2] (unclipped), rew/starts/val/logp [T][N] f32 : RolloutBuffer
 *   last_val [N] f32, last_done [N] u8   : inputs of compute_returns_and_advantage
 *   eps [T][N][2] f32 standard-normal draws (parity mode: torch's CPU generator cannot be
 *        reproduced on the device) or NULL -> Philox4x32-10 keyed (seed; env_offset + n,
 *        noise_offset + t)
 *   ep_ret [T][N] f64, ep_len [T][N] i32 : scratch, Monitor's info["episode"] return and length,
 *        written only at the (t, n) where an episode ended; ep_steps [T] i32 : scratch
 *   ep_r [ring_cap] f64, ep_l [ring_cap] i32, ep_count [1] u64 : ring of finished episodes in SB3's
 *        order (by step, then env index).  Episode k (0-based, counted over all rollouts) sits in
 *        slot k % ring_cap; *ep_count = number of episodes so far.  A rollout that ends more than
 *        ring_cap episodes files its newest ring_cap. */
int mr_rollout(mr_env* env, const float* params, int64_t T, float* last_obs, float* last_starts,
               float* obs, float* act, float* rew, float* starts, float* val, float* logp,
               float* last_val, uint8_t* last_done, const float* eps, uint64_t seed,
               uint64_t noise_offset, int64_t env_offset, double gamma, double* ep_ret,
               int32_t* ep_len, int32_t* ep_steps, double* ep_r, int32_t* ep_l,
               unsigned long long* ep_count, int ring_cap, void* stream);

/* What [SB3] PPO.train logs after its epochs (SURVEY A.5), in one launch and without a host round trip.
 * info [n_rows][8]: the info rows of every minibatch of the update; values / returns [n] the flat buffer;
 * params: the flat parameter vector after the update.  out [12] f32: [0:4] mean policy_gradient_loss,
 * value_loss, clip_fraction, approx_kl; [4:6] the last minibatch's policy and value loss; [6]
 * explained_variance(values, returns) (nan if var(returns) == 0); [7:9] log_std; [9] mean entropy_loss;
 * [10] the last minibatch's entropy_loss; [11] n_rows.  scratch: 8 doubles, zero before the first call.
 * ctrl: the update's control word (target_kl, below) or NULL. */
int mr_ppo_train_summary(const float* info, int n_rows, const float* values, const float* returns, int64_t n,
                         const float* params, float* out, double* scratch, const int* ctrl, void* stream);

/* One epoch of PPO.train on one GPU: for every minibatch of perm, mr_ppo_grad then mr_adam_step,
 * launched back to back from C (no host round trip between minibatches).  stats [n_mb][3] from
 * mr_ppo_adv_stats; info [n_mb][8] receives mr_adam_step's info rows (may be NULL). */
int mr_ppo_train_epoch(float* params, float* exp_avg, float* exp_avg_sq, int64_t* step, int obs_dim,
                       const float* obs, const float* act, const float* old_logp, const float* adv,
                       const float* ret, const int64_t* perm, int32_t* rows, int64_t n_samples,
                       int64_t batch_size, const double* stats, int64_t N, int64_t T, float clip_range,
                       float ent_coef, float vf_coef, int normalize_adv, float lr, float beta1, float beta2,
                       float eps, float max_grad_norm, float* partials, float* grad, float* info,
                       const float* old_values, float clip_range_vf, float target_kl, int* ctrl, int64_t mb0,
                       void* stream);

/* ------------------------------------------------------------------------------------
 * Fused epoch: every minibatch of one epoch of PPO.train in ONE cooperative launch (forward,
 * backward, gradient reduction, [all-reduce,] clip_grad_norm_, Adam; one grid barrier per
 * minibatch, two with several ranks).  With xchg != NULL the per-minibatch gradient all-reduce
 * (the reference has none: SB3 trains in one process) runs inside the kernel over NVLink peer
 * memory: each CTA pushes its slice of the reduced gradient into every peer's inbox as tagged
 * packets and sums the ranks' slices in rank order (parameters stay bit-identical on all ranks).
 * A peer that stops delivering ends the wait after ~4 s and raises the flag mr_xchg_status reads.
 * rows [n_samples] int32 caller-owned scratch, filled from perm -- or, with perm = NULL, already holding the
 * epoch's samples as buffer rows (mr_ppo_prepare_epochs).  stats: the GLOBAL minibatches' sums (all-reduced by the
 * host when several ranks train), which is all the kernel needs to know about the other ranks' shares. */
typedef struct mr_xchg mr_xchg;
/* Allocate this rank's inbox; h_handle_out receives its 64-byte CUDA IPC handle. */
int mr_xchg_create(int world, int rank, int device, int obs_dim, mr_xchg** out, uint8_t* h_handle_out);
/* h_all_handles [world][64]: every rank's handle (gathered by the host, e.g. torch.distributed). */
int mr_xchg_connect(mr_xchg* x, const uint8_t* h_all_handles);
void mr_xchg_destroy(mr_xchg* x);
/* *timed_out <- 1 if an in-kernel exchange gave up waiting for a peer since creation (synchronous read) */
int mr_xchg_status(mr_xchg* x, int* timed_out);
/* The epoch kernel gathers its minibatches from PACKED sample records, one per buffer row (t * N + n):
 * mr_ppo_record_floats(obs_dim) floats = [obs | 0.. | 1 | a0 a1 old_logp adv | ret old_value 0 0] (96 B for
 * the point robot, 160 B for the car).  mr_ppo_pack_samples builds them once per rollout (after GAE) from
 * the RolloutBuffer arrays; old_value = values (the rollout's V(s) [T][N], needed with clip_range_vf) or 0 when
 * values = NULL.  rec is caller-owned, n_rows * mr_ppo_record_floats floats. */
int mr_ppo_record_floats(int obs_dim);
int mr_ppo_pack_samples(int obs_dim, const float* obs, const float* act, const float* old_logp, const float* adv,
                        const float* ret, const float* values, int64_t n_rows, float* rec, void* stream);
int mr_ppo_epoch_fused(float* params, float* exp_avg, float* exp_avg_sq, int64_t* step, int obs_dim,
                       const float* rec, const int64_t* perm, int32_t* rows, int64_t n_samples,
                       int64_t batch_size, const double* stats, int64_t N, int64_t T,
                       float clip_range, float ent_coef, float vf_coef, int normalize_adv, float lr,
                       float beta1, float beta2, float eps, float max_grad_norm, float* partials,
                       float* grad, float* info, mr_xchg* xchg, float clip_range_vf, float target_kl, int* ctrl,
                       int64_t mb0, void* stream);

/* [SB3] PPO's clip_range_vf and target_kl: the trailing arguments of mr_ppo_grad, mr_adam_step, mr_ppo_train_epoch,
 * mr_ppo_epoch_fused and mr_ppo_train_summary.  clip_range_vf <= 0, target_kl <= 0 and ctrl = NULL turn both off
 * (and launch the default kernels).  clip_range_vf > 0: value_loss = mse(returns, old_value + clamp(V - old_value,
 * -c, c)), old_value being the rollout's values [T][N] (RolloutBuffer.values), passed as old_values to the
 * per-launch calls and packed into the records by mr_ppo_pack_samples for the fused one.  target_kl > 0 (requires
 * ctrl): per minibatch, after its losses and statistics, approx_kl > 1.5 * target_kl (compared in double) stops the
 * update: that minibatch is not applied and no later one runs.  ctrl is the update's control word, one int32 of
 * caller-owned device memory that the caller zeroes once per update; a stop after the k-th minibatch of the update
 * (counted over all its calls from mb0 / mb_index = 0) sets it to k, and every later call of the update returns at
 * entry in its kernels and changes nothing.  After a stop the info row of the stopping minibatch holds its
 * statistics with the unchanged step count, and `grad` holds its gradient (the fused call: also when a later launch
 * of the update returns at entry; the per-launch calls: on one GPU -- a host all-reduce of later minibatches still
 * sums the unchanged vector).  mr_ppo_train_summary with a ctrl recording a stop after k minibatches averages rows
 * [0, k), takes row k - 1 as "last", sets out[11] = k and out[12] = row k - 1's approx_kl (out then has 13 floats);
 * with ctrl = NULL it covers all n_rows and writes 12 floats. */

/* Same contract as mr_rollout, from the stand-alone env-step kernel plus ONE kernel between two env steps (the
 * finished step's RolloutBuffer.add bookkeeping -- time-out bootstrap, reward row, Monitor's episode records, start
 * flags -- and the next step's policy forward, Gaussian sample and log-prob), then the two episode-filing launches:
 * 2 T + 3 launches and a copy.  Works for both env kinds and
 * for envs with optional observation keys (rows of mr_env_obs_dim floats, at most 32); the car uses this path. */
int mr_rollout_unfused(mr_env* env, const float* params, int64_t T, float* last_obs, float* last_starts,
                       float* obs, float* act, float* rew, float* starts, float* val, float* logp,
                       float* last_val, uint8_t* last_done, const float* eps, uint64_t seed,
                       uint64_t noise_offset, int64_t env_offset, double gamma, double* ep_ret,
                       int32_t* ep_len, int32_t* ep_steps, double* ep_r, int32_t* ep_l,
                       unsigned long long* ep_count, int ring_cap, void* stream);

/* Device-side minibatch index streams: out[e][0..n) <- a keyed pseudo-random permutation of 0..n-1, a pure
 * function of (seed, h_stream_ids[e]); one thread per index, no sort.  `count` (1..32) permutations in one launch:
 * out [count][n], h_stream_ids [count] in host memory.  For runs that keep RolloutBuffer.get's indices on the
 * device (PPO(permutation="device")). */
int mr_device_permutations(uint64_t seed, const uint64_t* h_stream_ids, int count, int64_t n, int64_t* out,
                           void* stream);

/* What the epochs of one PPO.train need besides the parameters, for all epochs at once: per-minibatch
 * advantage sums (as mr_ppo_adv_stats) and the samples as time-major buffer rows.  perm [n_epochs][n_samples]
 * (one permutation per epoch), stats [n_epochs][n_mb][3] f64 out, rows [n_epochs][n_samples] int32 out.
 * mr_ppo_epoch_fused then takes perm = NULL and rows = the epoch's row of `rows`. */
int mr_ppo_prepare_epochs(const float* adv, const int64_t* perm, int n_epochs, int64_t n_samples, int64_t batch_size,
                          int64_t N, int64_t T, double* stats, int32_t* rows, void* stream);
/* The same with the device index streams of mr_device_permutations(seed, h_stream_ids, n_epochs, N * T), generated
 * on the fly: rows [n_epochs][N * T] and stats come out exactly as from the two calls, but the int64 permutations
 * are never written (two launches per update). */
int mr_ppo_prepare_epochs_device(uint64_t seed, const uint64_t* h_stream_ids, int n_epochs, const float* adv,
                                 int64_t n_samples, int64_t batch_size, int64_t N, int64_t T, double* stats,
                                 int32_t* rows, void* stream);

/* Batched policy evaluation.  Replaces [SB3 2.0.0] common/evaluation.py: evaluate_policy(model, env,
 * n_eval_episodes, deterministic) over the vectorised env, AFTER the caller's env.reset(): steps every env with the
 * policy until each env i has finished its target of c_i = (n_episodes + i) / N episodes, exactly as SB3's loop does
 * (all envs keep stepping until the last target is met), and records those episodes.
 *   deterministic != 0: the action mean; else mu + exp(log_std) * z, z Philox4x32-10 keyed (seed; env_offset + n,
 *        noise_offset + t) like the rollout kernels (t = step index within this call)
 *   last_obs [N][O] f32 in/out: the observation the evaluation starts from; the one it ends on
 *   ep_r [n_episodes] f64, ep_l [n_episodes] i32, ep_t [n_episodes] i64 out: Monitor's info["episode"] return and
 *        length and the step index at which the episode ended.  Env i's records fill slots off_i .. off_i + c_i - 1,
 *        off_i = c_0 + ... + c_{i-1}; SB3's list order is the records sorted by (ep_t, env index).
 *   steps_taken [1] i64 out: steps S every env has taken.  status [1] i32 out: 1 if max_steps (mandatory: no call runs
 *        unbounded) ended the evaluation before every target was met (the env is then consistent at S = max_steps).
 * The point env with the default observation row runs in one fused kernel (two launches); the car and envs with
 * optional observation keys take one launch plus mr_env_step per step, and synchronise the stream after each step. */
int mr_evaluate(mr_env* env, const float* params, int deterministic, int64_t n_episodes, int64_t max_steps,
                uint64_t seed, uint64_t noise_offset, int64_t env_offset, float* last_obs, double* ep_r,
                int32_t* ep_l, int64_t* ep_t, int64_t* steps_taken, int* status, void* stream);

/* Host-side minibatch index stream (no device work): out[0..n) <- a uniformly random permutation
 * of 0..n-1, a pure function of (seed, stream).  Replaces, for throughput runs, the
 * np.random.permutation call of [SB3 2.0.0] RolloutBuffer.get (reached from
 * src/mobrob/rl_control/ppo.py:73-74); the bit-for-bit numpy stream stays available on the Python
 * side (PPO(permutation="sb3")).  Thread-safe; `out` is host memory (pinned or pageable). */
int mr_host_permutation(uint64_t seed, uint64_t stream, int64_t n, int64_t* out);

#ifdef __cplusplus
}
#endif
#endif /* MOBROB_B200_H */
