"""PPO: the stable-baselines3 ``PPO`` surface mobrob uses, driving the CUDA hot path.

Mirrors (same names, argument meaning, zip format):
  * ``PPO(env=, seed=, tensorboard_log=, policy="MlpPolicy", n_steps, batch_size, n_epochs,
    ent_coef, gae_lambda, verbose, device, ...)``       src/mobrob/rl_control/ppo.py:50-59
  * ``.learn(total_timesteps, callback, progress_bar)``    examples/train.py:42-46
  * ``.save(path)`` / ``PPO.load(path)``                   ppo.py:76-77, src/mobrob/utils.py:15-16
  * ``.policy.state_dict() / load_state_dict()``           train.py:30-33
  * ``.predict(obs, deterministic=True)``                  examples/control.py:39
One ``learn`` iteration = mr_rollout (T steps) -> mr_gae -> n_epochs x minibatches of
(mr_ppo_grad [-> all-reduce] -> mr_adam_step), fused into mr_ppo_epoch_fused by default ->
mr_ppo_train_summary; clip_range_vf / target_kl are the update calls' trailing arguments.
Nothing here computes on the CPU except bookkeeping; there is no fallback path.
"""
from __future__ import annotations

import base64
import ctypes
import io
import json
import os
import sys
import time
import zipfile
from collections import deque

import numpy as np
import torch

from . import _lib, sharding
from .policy import MlpPolicy
from .updater import PpoUpdater
from .vec_env import GpuVecEnv

SB3_VERSION = "2.0.0"
EP_RING = 1 << 16


def _dist():
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        return dist
    return None


class Logger:
    """Keeps the reference's log keys (SURVEY appendix A.5); prints SB3-style tables."""

    def __init__(self, verbose=0, tensorboard_log=None):
        self.name_to_value = {}
        self.verbose = verbose
        self.writer = None
        if tensorboard_log:
            try:
                from torch.utils.tensorboard import SummaryWriter

                self.writer = SummaryWriter(tensorboard_log)
            except Exception:
                self.writer = None

    def record(self, key, value, exclude=None):
        """``exclude`` (SB3: output formats to leave out) is accepted and ignored."""
        self.name_to_value[key] = value

    def dump(self, step=0):
        if self.writer is not None:
            for k, v in self.name_to_value.items():
                if isinstance(v, (int, float)):
                    self.writer.add_scalar(k, v, step)
        if self.verbose >= 1:
            groups = {}
            for k, v in sorted(self.name_to_value.items()):
                g, _, name = k.partition("/")
                groups.setdefault(g, []).append((name, v))
            lines = []
            for g, items in groups.items():
                lines.append(f"| {g + '/':<24}|{'':>14} |")
                for name, v in items:
                    sv = f"{v:.3g}" if isinstance(v, float) else str(v)
                    lines.append(f"|    {name:<21}| {sv:<13} |")
            bar = "-" * 42
            print("\n".join([bar, *lines, bar]), flush=True)
        self.name_to_value = {}


class PPO:
    def __init__(self, policy="MlpPolicy", env=None, learning_rate=3e-4, n_steps=2048, batch_size=64,
                 n_epochs=10, gamma=0.99, gae_lambda=0.95, clip_range=0.2, clip_range_vf=None,
                 normalize_advantage=True, ent_coef=0.0, vf_coef=0.5, max_grad_norm=0.5, use_sde=False,
                 sde_sample_freq=-1, target_kl=None, stats_window_size=100, tensorboard_log=None,
                 policy_kwargs=None, verbose=0, seed=None, device="auto", _init_setup_model=True,
                 host_permutation=None, update_mode="fused", permutation=None):
        if policy not in ("MlpPolicy", MlpPolicy):
            raise ValueError("only MlpPolicy is built (the only policy mobrob uses)")
        if use_sde:
            raise NotImplementedError("use_sde (gSDE) is not built: it is a different policy and rollout noise model")
        if clip_range_vf is not None and not callable(clip_range_vf) and not float(clip_range_vf) > 0:
            raise ValueError(f"clip_range_vf must be positive (got {clip_range_vf}); None turns value clipping off")
        if target_kl is not None and not float(target_kl) > 0:
            # SB3 would stop every update at its first minibatch; the kernels take target_kl <= 0 as "off"
            raise ValueError(f"target_kl must be positive (got {target_kl}); None turns early stopping off")
        if policy_kwargs not in (None, {}):
            arch = (policy_kwargs or {}).get("net_arch")
            if arch not in (None, dict(pi=[64, 64], vf=[64, 64])):
                raise NotImplementedError("kernels are specialised for net_arch pi=[64,64], vf=[64,64]")
        # SB3 schedules: callables of the remaining progress (1 -> 0), evaluated before every update
        self._lr_schedule = learning_rate if callable(learning_rate) else None
        self._clip_schedule = clip_range if callable(clip_range) else None
        self._clip_vf_schedule = clip_range_vf if callable(clip_range_vf) else None
        if callable(clip_range_vf):
            clip_range_vf = float(clip_range_vf(1.0))
        self.clip_range_vf = None if clip_range_vf is None else float(clip_range_vf)
        self.target_kl = None if target_kl is None else float(target_kl)
        if callable(learning_rate):
            learning_rate = float(learning_rate(1.0))
        if callable(clip_range):
            clip_range = float(clip_range(1.0))
        self.policy_class = MlpPolicy
        self.policy_kwargs = policy_kwargs or {}
        self.learning_rate, self.n_steps, self.batch_size, self.n_epochs = learning_rate, n_steps, batch_size, n_epochs
        self.gamma, self.gae_lambda, self.clip_range = gamma, gae_lambda, clip_range
        self.normalize_advantage, self.ent_coef, self.vf_coef = normalize_advantage, ent_coef, vf_coef
        self.max_grad_norm, self.verbose, self.seed = max_grad_norm, verbose, seed
        self.tensorboard_log = tensorboard_log
        # RolloutBuffer.get's index stream.  "device" (default): mr_device_permutations, a keyed Feistel
        # bijection computed where the samples live -- nothing crosses PCIe.  "sb3": np.random.permutation
        # on the global MT19937, bit-for-bit SB3's stream, serial on the host (parity runs).  "pool": host
        # threads drawing streams keyed by (seed, iteration, epoch) one iteration ahead (permfeed.py).
        if permutation is None:
            permutation = "sb3" if host_permutation is True else "device"
        if permutation not in ("sb3", "pool", "device"):
            raise ValueError(f"Unknown permutation mode: {permutation}")
        self.permutation = permutation
        self._feeder = None
        self._train_count = 0
        self._train_stats = None
        self._train_meta = None
        self._snap_meta = None
        self._snap = None
        # target_kl: updates whose epoch count is read back from the device lazily (_settle_updates)
        self._pending_updates = deque()
        self._n_updates_at = {}
        self._current_progress_remaining = 1.0
        self._stats_window_size = stats_window_size
        self.num_timesteps = 0
        self._total_timesteps = 0
        self._num_timesteps_at_start = 0
        self._n_updates = 0
        self._episode_num = 0
        self.start_time = None
        self.ep_info_buffer = deque(maxlen=stats_window_size)
        self.ep_success_buffer = deque(maxlen=stats_window_size)
        self.env = env
        self.policy = None
        self.logger = Logger(verbose, None)
        self._rollout_count = 0
        self._ep_seen = 0
        self._last_obs = None
        self._last_episode_starts = None
        self._xchg = None
        self.update_mode = update_mode  # "fused" | "launches" (per-minibatch kernels, NCCL when sharded)
        self.rollout_mode = "fused"     # "fused" (point only) | "unfused" (stand-alone kernels; the car)
        self.gpu_time_ms = {}
        if env is not None:
            self.n_envs = env.num_envs
            self.observation_space, self.action_space = env.observation_space, env.action_space
        if _init_setup_model and env is not None:
            self._setup_model()

    # ------------------------------------------------------------------------------------------
    def _setup_model(self):
        env = self.env
        if not isinstance(env, GpuVecEnv):
            raise TypeError("mobrob_b200.PPO trains on a GpuVecEnv (the envs live in HBM)")
        self.device = env.device
        if self.seed is not None:  # set_random_seed
            import random

            random.seed(self.seed)
            np.random.seed(self.seed)
            torch.manual_seed(self.seed)
            env.seed(self.seed)
        O = env.obs_dim
        self.updater = PpoUpdater(O, self.device, lr=self.learning_rate, max_grad_norm=self.max_grad_norm,
                                  clip_range=self.clip_range, ent_coef=self.ent_coef, vf_coef=self.vf_coef,
                                  normalize_advantage=self.normalize_advantage, clip_range_vf=self.clip_range_vf,
                                  target_kl=self.target_kl)
        self.policy = MlpPolicy(O, 2, device=self.device, flat=self.updater.params, init=True)
        d = _dist()
        if d is not None:  # every rank must start from rank 0's parameters
            d.broadcast(self.updater.params, src=0)
        T, N = self.n_steps, env.num_envs
        f32 = dict(dtype=torch.float32, device=self.device)
        self.buf = dict(obs=torch.zeros((T, N, O), **f32), actions=torch.zeros((T, N, 2), **f32),
                        rewards=torch.zeros((T, N), **f32), episode_starts=torch.zeros((T, N), **f32),
                        values=torch.zeros((T, N), **f32), log_probs=torch.zeros((T, N), **f32),
                        advantages=torch.zeros((T, N), **f32), returns=torch.zeros((T, N), **f32))
        self.last_val = torch.zeros(N, **f32)
        self.last_done = torch.zeros(N, dtype=torch.uint8, device=self.device)
        self._last_obs = None
        self._last_episode_starts = None
        # Monitor's finished episodes: the ring in SB3's (step, env) order, and the rollout kernels' [T][N] records
        # it is filled from
        self.ep_r = torch.zeros(EP_RING, dtype=torch.float64, device=self.device)
        self.ep_l = torch.zeros(EP_RING, dtype=torch.int32, device=self.device)
        self.ep_count = torch.zeros(1, dtype=torch.int64, device=self.device)
        self.ep_ret_tn = torch.zeros((T, N), dtype=torch.float64, device=self.device)
        self.ep_len_tn = torch.zeros((T, N), dtype=torch.int32, device=self.device)
        self.ep_steps = torch.zeros(T, dtype=torch.int32, device=self.device)
        self.lib = _lib.load()

    def get_env(self):
        return self.env

    def set_env(self, env, force_reset=True):
        """SB3's ``m = PPO.load(path); m.set_env(env); m.learn(...)``: attach a GpuVecEnv, (re)allocate the
        rollout buffers on ITS device and keep the loaded parameters and Adam state."""
        if not isinstance(env, GpuVecEnv):
            raise TypeError("mobrob_b200.PPO trains on a GpuVecEnv (the envs live in HBM)")
        if self.policy is not None and env.obs_dim != self.updater.obs_dim:
            raise ValueError(f"observation dimension {env.obs_dim} does not match the policy's {self.updater.obs_dim}")
        old = self.updater if self.policy is not None else None
        self.env = env
        self.n_envs = env.num_envs
        self.observation_space, self.action_space = env.observation_space, env.action_space
        seed, self.seed = self.seed, None   # set_random_seed / orthogonal init belong to construction only
        self._setup_model()
        self.seed = seed
        if old is not None:
            up = self.updater
            up.params.copy_(old.params.to(up.device))
            up.exp_avg.copy_(old.exp_avg.to(up.device))
            up.exp_avg_sq.copy_(old.exp_avg_sq.to(up.device))
            up.step.copy_(old.step.to(up.device))
            up.lr, up.betas, up.eps = old.lr, old.betas, old.eps
        self._xchg = None
        self._log = None

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    # -- rollout ------------------------------------------------------------------------------------
    def collect_rollouts(self, eps: torch.Tensor | None = None):
        """Fused rollout of n_steps; eps optionally supplies the N(0,1) draws [T, N, 2]."""
        env, b = self.env, self.buf
        if self._last_obs is None:
            self._last_obs = env.reset_tensor().clone()
            self._last_episode_starts = torch.ones(env.num_envs, dtype=torch.float32, device=self.device)
        seed = int(self.seed if self.seed is not None else 0)
        fused = env.env_name == "point" and self.rollout_mode == "fused" and not getattr(env, "obs_flags", 0)
        fn = self.lib.mr_rollout if fused else self.lib.mr_rollout_unfused
        _lib.check(fn(
            env._h, self.updater.params.data_ptr(), self.n_steps, self._last_obs.data_ptr(),
            self._last_episode_starts.data_ptr(), b["obs"].data_ptr(), b["actions"].data_ptr(),
            b["rewards"].data_ptr(), b["episode_starts"].data_ptr(), b["values"].data_ptr(),
            b["log_probs"].data_ptr(), self.last_val.data_ptr(), self.last_done.data_ptr(),
            None if eps is None else eps.data_ptr(), seed, self._rollout_count * self.n_steps,
            env.first_rank, float(self.gamma), self.ep_ret_tn.data_ptr(), self.ep_len_tn.data_ptr(),
            self.ep_steps.data_ptr(), self.ep_r.data_ptr(), self.ep_l.data_ptr(), self.ep_count.data_ptr(), EP_RING,
            self._stream()))
        self._rollout_count += 1
        _lib.check(self.lib.mr_gae(b["rewards"].data_ptr(), b["values"].data_ptr(),
                                   b["episode_starts"].data_ptr(), self.last_val.data_ptr(),
                                   self.last_done.data_ptr(), float(self.gamma), float(self.gae_lambda),
                                   b["advantages"].data_ptr(), b["returns"].data_ptr(), self.n_steps,
                                   env.num_envs, self._stream()))
        self.num_timesteps += self.n_steps * env.num_envs * (self._world_size())

    def _world_size(self):
        d = _dist()
        return d.get_world_size() if d is not None else 1

    def _snapshot_async(self):
        """Enqueue the D2H reads one logging step needs -- Monitor's newest episodes (ep_info_buffer: the last W
        slots of the ring, which the rollout fills in SB3's order), the previous train()'s statistics -- into pinned
        memory; returns the event to wait for.
        Nothing here blocks the host: train() of this iteration is enqueued behind it."""
        W = self._stats_window_size
        if getattr(self, "_snap", None) is None:
            self._snap = dict(count=torch.zeros(1, dtype=torch.int64).pin_memory(),
                              r=torch.zeros(W, dtype=torch.float64).pin_memory(),
                              l=torch.zeros(W, dtype=torch.int32).pin_memory(),
                              train=torch.zeros(12, dtype=torch.float32).pin_memory())
        sn = self._snap
        idx = (self.ep_count - W + torch.arange(W, device=self.device)).clamp_(min=0) % EP_RING
        sn["count"].copy_(self.ep_count, non_blocking=True)
        sn["r"].copy_(self.ep_r[idx], non_blocking=True)
        sn["l"].copy_(self.ep_l[idx], non_blocking=True)
        if self._train_stats is not None:
            sn["train"].copy_(self._train_stats, non_blocking=True)
            self._snap_meta = self._train_meta
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.device))
        return ev

    def _drain_episodes(self, ev=None):
        """Monitor's ep_info_buffer from the last snapshot (waits for its event)."""
        if ev is None:
            ev = self._snapshot_async()
        ev.synchronize()
        sn, W = self._snap, self._stats_window_size
        total = int(sn["count"][0])
        new = min(total - self._ep_seen, W, total)
        if new > 0:
            r, l = sn["r"].numpy(), sn["l"].numpy()
            now = round(time.time() - self.env.t_start, 6)
            for i in range(W - new, W):
                self.ep_info_buffer.append({"r": round(float(r[i]), 6), "l": int(l[i]), "t": now})
        self._ep_seen = total
        self._episode_num = total

    # -- update --------------------------------------------------------------------------------------
    @property
    def host_permutation(self):
        return self.permutation != "device"

    @host_permutation.setter
    def host_permutation(self, flag):
        self.permutation = "sb3" if flag else "device"

    def _get_feeder(self):
        if self._feeder is None:
            from .permfeed import PermutationFeeder

            d = _dist()
            self._feeder = PermutationFeeder(self.n_steps * self.env.num_envs, self.n_epochs, self.device,
                                             seed=int(self.seed or 0), rank=d.get_rank() if d is not None else 0)
        return self._feeder

    def _permutation(self, n, epoch=0):
        if self.permutation == "pool":
            return self._get_feeder().get(self._train_count, epoch)
        if self.permutation == "sb3":  # RolloutBuffer.get: np.random.permutation on the global MT19937
            if getattr(self, "_pin", None) is None or self._pin.numel() != n:
                self._pin = torch.empty(n, dtype=torch.int64).pin_memory()
                self._pin_ev = None
            if self._pin_ev is not None:
                self._pin_ev.synchronize()
            self._pin.numpy()[:] = np.random.permutation(n)
            out = self._pin.to(self.device, non_blocking=True)
            self._pin_ev = torch.cuda.Event()
            self._pin_ev.record(torch.cuda.current_stream(self.device))
            return out
        # "device": keyed bijection computed by one kernel (no sort)
        if getattr(self, "_dperm", None) is None or self._dperm.numel() != n:
            self._dperm = torch.empty(n, dtype=torch.int64, device=self.device)
        out = self._dperm
        d = _dist()
        key = ((d.get_rank() if d is not None else 0) << 48) ^ (self._train_count << 16) ^ epoch
        _lib.check(self.lib.mr_device_permutations(int(self.seed or 0), (ctypes.c_uint64 * 1)(key), 1, n,
                                                   out.data_ptr(), self._stream()))
        return out

    def _stream_ids(self):
        """Keys of this update's device index streams, one per epoch: (rank, update count, epoch)."""
        d = _dist()
        rank = d.get_rank() if d is not None else 0
        return [(rank << 48) ^ (self._train_count << 16) ^ e for e in range(self.n_epochs)]

    def train(self, perms=None):
        """PPO.train: n_epochs passes of minibatch updates.  perms: optional list of int64 index
        arrays (one per epoch) for parity runs; otherwise drawn like RolloutBuffer.get."""
        up, b = self.updater, self.buf
        T, N = self.n_steps, self.env.num_envs
        n = T * N
        B = self.batch_size
        n_mb = (n + B - 1) // B
        d = _dist()
        self._update_schedules()
        rows = self.n_epochs * n_mb
        if getattr(self, "_log", None) is None or self._log.shape[0] != rows:
            # per-minibatch info rows (every row is written by the kernels), the 12 logger inputs of the
            # update (+ the stopping minibatch's approx_kl with target_kl) and the summary kernel's scratch:
            # allocated once, no per-iteration torch launches
            self._log = torch.zeros((rows, 8), dtype=torch.float32, device=self.device)
            self._train_stats_buf = torch.zeros(13, dtype=torch.float32, device=self.device)
            self._sum_scratch = torch.zeros(8, dtype=torch.float64, device=self.device)
        log = self._log
        self._settle_updates(block=False)
        up.begin_update()   # target_kl: clear the control word (nothing otherwise)
        k = 0
        if self.update_mode == "fused":
            up.pack(b)   # packed sample records, once per rollout: what the epoch kernel gathers from
            if d is not None and self._xchg is None:
                from .updater import PeerExchange

                self._xchg = PeerExchange(up.obs_dim, self.device)
        if self.update_mode == "fused" and perms is None and self.permutation == "device" and self.n_epochs <= 32:
            # the whole update's index streams, advantage sums and row indices up front (3 launches and, with
            # several ranks, ONE all-reduce), then nothing but the epoch kernels back to back
            stats_all, rows_all = up.prepare_epochs_device(b["advantages"], int(self.seed or 0), self._stream_ids(), B, N, T)
            if d is not None:
                flat, _ = sharding.allreduce_adv_stats(stats_all.view(-1, 3))
                stats_all = flat.view(self.n_epochs, n_mb, 3)
            if n % B == 0 and not os.environ.get("MR_EPOCH_LAUNCHES"):
                # whole minibatches only: the epochs are one sequence of n_epochs * n_mb minibatches over the concatenated
                # row lists -- ONE cooperative launch for the update (the tower state is staged into shared memory and
                # written back once instead of once per epoch)
                up.train_epoch_fused(None, None, stats_all.view(-1, 3), B, N, T, log[:rows], self._xchg, rows=rows_all.view(-1))
                k = rows
            else:
                for epoch in range(self.n_epochs):
                    up.train_epoch_fused(None, None, stats_all[epoch], B, N, T, log[k:k + n_mb], self._xchg, rows=rows_all[epoch],
                                         mb0=k)
                    k += n_mb
            epochs = ()
        else:
            epochs = range(self.n_epochs)
        for epoch in epochs:
            perm = perms[epoch] if perms is not None else self._permutation(n, epoch)
            if not torch.is_tensor(perm):
                perm = torch.as_tensor(np.asarray(perm, dtype=np.int64))
            perm = perm.to(self.device).contiguous()
            stats = up.adv_stats(b["advantages"], perm, B, N, T)
            share = None
            if d is not None:
                stats, share = sharding.allreduce_adv_stats(stats)
            if self.update_mode == "fused":      # one cooperative launch per epoch (+ NVLink all-reduce)
                up.train_epoch_fused(None, perm, stats, B, N, T, log[k:k + n_mb], self._xchg, mb0=k)
                k += n_mb
            elif d is None:                      # 3 launches per minibatch, looped in C
                up.train_epoch(b, perm, stats, B, N, T, log[k:k + n_mb], mb0=k)
                k += n_mb
            else:                                # NCCL all-reduce per minibatch (baseline path)
                share_h = share.cpu().tolist()
                for mb in range(n_mb):
                    sl = perm[mb * B:(mb + 1) * B]
                    up.compute_grad(b, sl, stats[mb], N, T, share_h[mb])
                    d.all_reduce(up.grad)
                    up.adam_step(log[k], mb_index=k)
                    k += 1
        if perms is None and self.permutation == "pool":
            self._feeder.release(self._train_count)
        uid = self._train_count
        self._train_count += 1
        self._train_log = (log[:, 4:], log[:, :4])
        # logger inputs of this update (mr_ppo_train_summary), read one iteration later -- SB3 records
        # train/* inside train() and dumps them with the NEXT iteration's rollout statistics
        # (target_kl: statistics over the minibatches evaluated before the stop)
        _lib.check(self.lib.mr_ppo_train_summary(log.data_ptr(), rows, b["values"].data_ptr(), b["returns"].data_ptr(),
                                                 n, up.params.data_ptr(), self._train_stats_buf.data_ptr(),
                                                 self._sum_scratch.data_ptr(), up.ctrl_ptr(), self._stream()))
        if self.target_kl is None:
            self._n_updates += self.n_epochs
        else:
            # how many epochs were entered is read back without blocking (the control word and the stopping
            # approx_kl, into pinned memory)
            ctrl_h = torch.zeros(1, dtype=torch.int32).pin_memory()
            kl_h = torch.zeros(1, dtype=torch.float32).pin_memory()
            ctrl_h.copy_(up.ctrl, non_blocking=True)
            kl_h.copy_(self._train_stats_buf[12:13], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(self.device))
            self._pending_updates.append((uid, ev, ctrl_h, kl_h, n_mb))
        self._train_stats = self._train_stats_buf[:12]
        self._train_meta = dict(update=uid, n_updates=self._n_updates if self.target_kl is None else None,
                                clip_range=self.clip_range, clip_range_vf=self.clip_range_vf, learning_rate=up.lr)

    def _settle_updates(self, upto=None, block=True):
        """target_kl: add the epochs each finished update entered to _n_updates (SB3 counts every epoch it
        enters, the one it stops in included) and print SB3's early-stopping message.  Updates are settled in
        order: all of them, those up to update id `upto`, or (block=False) those already complete."""
        while self._pending_updates:
            uid, ev, ctrl_h, kl_h, n_mb = self._pending_updates[0]
            if upto is not None and uid > upto:
                break
            if not block and not ev.query():
                break
            ev.synchronize()
            self._pending_updates.popleft()
            k = int(ctrl_h[0])
            if k > 0:
                epochs = (k + n_mb - 1) // n_mb
                if self.verbose >= 1 and self._is_rank0():
                    print(f"Early stopping at step {epochs - 1} due to reaching max kl: {float(kl_h[0]):.2f}")
            else:
                epochs = self.n_epochs
            self._n_updates += epochs
            self._n_updates_at[uid] = self._n_updates
            self._n_updates_at.pop(uid - 8, None)

    def _update_schedules(self):
        """SB3's _update_learning_rate / clip_range(progress): constant values or callables of the
        remaining progress (1 -> 0); both are per-launch kernel arguments."""
        progress = 1.0   # _update_current_progress_remaining: 1 - num_timesteps / total_timesteps
        if self._total_timesteps:
            progress = 1.0 - float(self.num_timesteps) / float(self._total_timesteps)
        self._current_progress_remaining = progress
        if self._lr_schedule is not None:
            self.learning_rate = float(self._lr_schedule(progress))
        if self._clip_schedule is not None:
            self.clip_range = float(self._clip_schedule(progress))
        if self._clip_vf_schedule is not None:
            self.clip_range_vf = float(self._clip_vf_schedule(progress))
        self.updater.lr = self.learning_rate
        self.updater.clip_range = self.clip_range
        self.updater.clip_range_vf = self.clip_range_vf
        self.updater.target_kl = self.target_kl

    def _log_train(self):
        """train/* keys of SB3's PPO.train, from the statistics snapshot of the previous update."""
        t = self._snap["train"].numpy()
        meta = self._snap_meta
        lg = self.logger
        lg.record("train/entropy_loss", float(t[9]))
        lg.record("train/policy_gradient_loss", float(t[0]))
        lg.record("train/value_loss", float(t[1]))
        lg.record("train/approx_kl", float(t[3]))
        lg.record("train/clip_fraction", float(t[2]))
        lg.record("train/loss", float(t[4] + self.ent_coef * t[10] + self.vf_coef * t[5]))
        lg.record("train/explained_variance", float(t[6]))
        lg.record("train/std", float(np.exp(t[7:9].astype(np.float32)).mean()))
        n_updates = meta["n_updates"]
        if n_updates is None:   # target_kl: the update's epoch count is in the snapshot's past, complete by now
            self._settle_updates(upto=meta["update"])
            n_updates = self._n_updates_at.get(meta["update"], self._n_updates)
        lg.record("train/n_updates", n_updates)
        lg.record("train/clip_range", meta["clip_range"])
        if meta.get("clip_range_vf") is not None:
            lg.record("train/clip_range_vf", meta["clip_range_vf"])
        lg.record("train/learning_rate", meta["learning_rate"])

    # -- learn ----------------------------------------------------------------------------------------
    def learn(self, total_timesteps, callback=None, log_interval=1, tb_log_name="PPO",
              reset_num_timesteps=True, progress_bar=False):
        if reset_num_timesteps or self.start_time is None:
            self.num_timesteps = 0 if reset_num_timesteps else self.num_timesteps
            self._num_timesteps_at_start = self.num_timesteps
            self.start_time = time.time_ns()
            self._last_obs = None
            if self.tensorboard_log:
                self.logger = Logger(self.verbose, os.path.join(self.tensorboard_log, f"{tb_log_name}_1"))
        self._total_timesteps = total_timesteps + self._num_timesteps_at_start
        if isinstance(callback, list):   # BaseAlgorithm._init_callback
            from .callbacks import CallbackList

            callback = CallbackList(callback)
        if callback is not None and hasattr(callback, "init_callback"):
            callback.init_callback(self)
            callback.on_training_start(locals(), globals())
        iteration = 0
        bar = None
        if progress_bar and self._is_rank0():
            try:
                from tqdm import tqdm

                bar = tqdm(total=total_timesteps, file=sys.stderr)
            except Exception:
                bar = None
        while self.num_timesteps < self._total_timesteps:
            before = self.num_timesteps
            if self.permutation == "pool":  # copies of this iteration overlap the rollout; next one is drawn
                f = self._get_feeder()
                f.stage(self._train_count)
                f.prefetch(self._train_count + 1)
            self.collect_rollouts()
            if callback is not None and hasattr(callback, "on_rollout_steps"):
                if callback.on_rollout_steps(self.n_steps) is False:
                    break
            iteration += 1
            if bar is not None:
                bar.update(self.num_timesteps - before)
            log_now = log_interval is not None and iteration % log_interval == 0
            had_update = self._train_stats is not None
            # SB3 logs, then trains.  Here the update is ENQUEUED first and the host formats the log
            # while the GPU works; the logged numbers are the same (snapshot taken before train()).
            ev = self._snapshot_async() if log_now else None
            self.train()
            if log_now:
                self._drain_episodes(ev)
                elapsed = max((time.time_ns() - self.start_time) / 1e9, sys.float_info.epsilon)
                fps = int((self.num_timesteps - self._num_timesteps_at_start) / elapsed)
                lg = self.logger
                if len(self.ep_info_buffer) > 0:
                    lg.record("rollout/ep_rew_mean", float(np.mean([e["r"] for e in self.ep_info_buffer])))
                    lg.record("rollout/ep_len_mean", float(np.mean([e["l"] for e in self.ep_info_buffer])))
                lg.record("time/fps", fps)
                lg.record("time/iterations", iteration)
                lg.record("time/time_elapsed", int(elapsed))
                lg.record("time/total_timesteps", self.num_timesteps)
                if had_update:
                    self._log_train()
                if self._is_rank0():
                    lg.dump(self.num_timesteps)
                else:
                    lg.name_to_value = {}
        if bar is not None:
            bar.close()
        if callback is not None and hasattr(callback, "on_training_end"):
            callback.on_training_end()
        torch.cuda.synchronize(self.device)
        return self

    @staticmethod
    def _is_rank0():
        d = _dist()
        return d is None or d.get_rank() == 0

    def predict(self, observation, state=None, episode_start=None, deterministic=False):
        return self.policy.predict(observation, state, episode_start, deterministic)

    # -- zip format (SURVEY appendix A.6) ----------------------------------------------------------------
    def _json_data(self):
        def ser(obj):
            try:
                import cloudpickle

                return base64.b64encode(cloudpickle.dumps(obj)).decode()
            except Exception:
                return ""

        def space(sp):
            return {":type:": "<class 'gymnasium.spaces.box.Box'>", ":serialized:": ser(sp),
                    "dtype": str(sp.dtype), "bounded_below": str(sp.bounded_below),
                    "bounded_above": str(sp.bounded_above), "_shape": list(sp.shape),
                    "low": str(sp.low), "high": str(sp.high), "low_repr": str(sp.low.min()),
                    "high_repr": str(sp.high.max()), "_np_random": None}

        lr, cr, cvf = self.learning_rate, self.clip_range, self.clip_range_vf
        last_obs = None if self._last_obs is None else self._last_obs.cpu().numpy()
        starts = None if self._last_episode_starts is None else self._last_episode_starts.cpu().numpy().astype(bool)
        return {
            "policy_class": {":type:": "<class 'abc.ABCMeta'>", ":serialized:": ser(MlpPolicy),
                             "__module__": "stable_baselines3.common.policies"},
            "verbose": self.verbose, "policy_kwargs": {},
            "num_timesteps": self.num_timesteps, "_total_timesteps": self._total_timesteps,
            "_num_timesteps_at_start": self._num_timesteps_at_start, "seed": self.seed,
            "action_noise": None, "start_time": self.start_time,
            "learning_rate": (lr if self._lr_schedule is None else
                              {":type:": "<class 'function'>", ":serialized:": ser(self._lr_schedule), "value": lr}),
            "tensorboard_log": self.tensorboard_log,
            "_last_obs": {":type:": "<class 'numpy.ndarray'>", ":serialized:": ser(last_obs)},
            "_last_episode_starts": {":type:": "<class 'numpy.ndarray'>", ":serialized:": ser(starts)},
            "_last_original_obs": None, "_episode_num": self._episode_num, "use_sde": False,
            "sde_sample_freq": -1,
            "_current_progress_remaining": 1.0 - self.num_timesteps / max(self._total_timesteps, 1),
            "_stats_window_size": self._stats_window_size,
            "ep_info_buffer": {":type:": "<class 'collections.deque'>", ":serialized:": ser(self.ep_info_buffer)},
            "ep_success_buffer": {":type:": "<class 'collections.deque'>", ":serialized:": ser(self.ep_success_buffer)},
            "_n_updates": self._n_updates, "n_steps": self.n_steps, "gamma": self.gamma,
            "gae_lambda": self.gae_lambda, "ent_coef": self.ent_coef, "vf_coef": self.vf_coef,
            "max_grad_norm": self.max_grad_norm, "batch_size": self.batch_size, "n_epochs": self.n_epochs,
            "clip_range": {":type:": "<class 'function'>", ":serialized:": ser(self._clip_schedule or _Constant(cr)),
                           "value": cr},
            "clip_range_vf": None if cvf is None else {
                ":type:": "<class 'function'>", ":serialized:": ser(self._clip_vf_schedule or _Constant(cvf)), "value": cvf},
            "normalize_advantage": self.normalize_advantage, "target_kl": self.target_kl,
            "observation_space": space(self.observation_space), "action_space": space(self.action_space),
            "n_envs": self.n_envs,
            "lr_schedule": {":type:": "<class 'function'>", ":serialized:": ser(self._lr_schedule or _Constant(lr)),
                            "value": lr},
        }

    def save(self, path):
        path = str(path)
        if not path.endswith(".zip"):
            path += ".zip"
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        self._settle_updates()   # target_kl: _n_updates of an update still in flight (waits for it)
        sd = {k: v.detach().cpu().clone() for k, v in self.policy.state_dict().items()}
        up = self.updater
        opt_state, off = {}, 0
        step = float(up.step[0].item())
        for i, (k, v) in enumerate(sd.items()):
            n = v.numel()
            opt_state[i] = {"step": torch.tensor(step), "exp_avg": up.exp_avg[off:off + n].view(v.shape).cpu().clone(),
                            "exp_avg_sq": up.exp_avg_sq[off:off + n].view(v.shape).cpu().clone()}
            off += n
        opt = {"state": opt_state if step > 0 else {},
               "param_groups": [{"lr": up.lr, "betas": tuple(up.betas), "eps": up.eps, "weight_decay": 0,
                                 "amsgrad": False, "maximize": False, "foreach": None, "capturable": False,
                                 "differentiable": False, "fused": None, "params": list(range(len(sd)))}]}

        def pth(obj):
            bio = io.BytesIO()
            torch.save(obj, bio)
            return bio.getvalue()

        with zipfile.ZipFile(path, "w") as z:
            z.writestr("data", json.dumps(self._json_data(), indent=4))
            z.writestr("pytorch_variables.pth", pth({}))
            z.writestr("policy.pth", pth(dict(sd)))
            z.writestr("policy.optimizer.pth", pth(opt))
            z.writestr("_stable_baselines3_version", SB3_VERSION)
            z.writestr("system_info.txt", f"- mobrob_b200 (B200-native)\n- PyTorch: {torch.__version__}\n"
                                          f"- Numpy: {np.__version__}\n- Stable-Baselines3 format: {SB3_VERSION}\n")

    @classmethod
    def load(cls, path, env=None, device="auto", custom_objects=None, print_system_info=False,
             force_reset=True, **kwargs):
        path = str(path)
        if not os.path.exists(path) and os.path.exists(path + ".zip"):
            path += ".zip"
        with zipfile.ZipFile(path) as z:
            data = json.loads(z.read("data"))
            sd = torch.load(io.BytesIO(z.read("policy.pth")), map_location="cpu", weights_only=True)
            opt = None
            if "policy.optimizer.pth" in z.namelist():
                opt = torch.load(io.BytesIO(z.read("policy.optimizer.pth")), map_location="cpu",
                                 weights_only=True)
        obs_shape = data["observation_space"].get("_shape") or [0]
        act_shape = data.get("action_space", {}).get("_shape") or [2]
        if len(obs_shape) != 1 or not 0 < int(obs_shape[0]) < 32 or list(act_shape) != [2]:
            # a robot outside the B200 path (doggo 58 -> 12, drone 12 -> 18, turtlebot3 43 -> 2): the archive can be
            # inspected and re-saved (examples/fix_pickle_warning.py), not run
            return StoredPolicy(path, data, sd, opt)
        plain = ("n_steps", "batch_size", "n_epochs", "gamma", "gae_lambda", "ent_coef", "vf_coef",
                 "max_grad_norm", "normalize_advantage", "verbose", "seed")
        ctor = {k: data[k] for k in plain if k in data}
        ctor["learning_rate"] = _stored_schedule(data.get("learning_rate", 3e-4), "learning_rate")
        ctor["clip_range"] = _stored_schedule(data.get("clip_range", 0.2), "clip_range")
        if data.get("clip_range_vf") is not None:
            ctor["clip_range_vf"] = _stored_schedule(data["clip_range_vf"], "clip_range_vf")
        if data.get("target_kl") is not None:
            ctor["target_kl"] = float(data["target_kl"])
        ctor.update(kwargs)
        model = cls("MlpPolicy", env, _init_setup_model=False, **ctor)
        for k in ("num_timesteps", "_total_timesteps", "_num_timesteps_at_start", "_n_updates", "_episode_num"):
            if k in data:
                setattr(model, k, data[k])
        obs_dim = int(data["observation_space"]["_shape"][0])
        from .spaces import Box

        model.observation_space = Box(-np.inf, np.inf, (obs_dim,), np.float32)
        model.action_space = Box(-1.0, 1.0, (2,), np.float32)
        model.n_envs = data.get("n_envs", 1)
        if env is not None:
            model._setup_model()
            up = model.updater
        else:  # inference-only handle (examples/control.py): policy + optimizer state, no buffers
            dev = torch.device("cuda", torch.cuda.current_device()) if device == "auto" else torch.device(device)
            model.device = dev
            up = PpoUpdater(obs_dim, dev, lr=ctor["learning_rate"], max_grad_norm=ctor.get("max_grad_norm", 0.5),
                            clip_range=ctor["clip_range"], ent_coef=ctor.get("ent_coef", 0.0),
                            vf_coef=ctor.get("vf_coef", 0.5),
                            normalize_advantage=ctor.get("normalize_advantage", True),
                            clip_range_vf=model.clip_range_vf, target_kl=model.target_kl)
            model.updater = up
            model.policy = MlpPolicy(obs_dim, 2, device=dev, flat=up.params, init=False)
        model.policy.load_state_dict(sd)
        if opt is not None and opt.get("state"):
            g = opt["param_groups"][0]
            up.lr, up.betas, up.eps = g["lr"], tuple(g["betas"]), g["eps"]
            st = opt["state"]
            up.exp_avg.copy_(torch.cat([st[i]["exp_avg"].reshape(-1) for i in range(len(st))]))
            up.exp_avg_sq.copy_(torch.cat([st[i]["exp_avg_sq"].reshape(-1) for i in range(len(st))]))
            up.step[0] = int(st[0]["step"])
        return model


class StoredPolicy:
    """A policy zip whose observation / action shapes are outside the CUDA path (the reference's doggo, drone and
    turtlebot3 policies): PPO.load returns this handle so that maintenance code like examples/fix_pickle_warning.py
    (load_policy(...).save(...) over every robot) keeps working.  It holds the archive's contents and writes them
    back in the same six-entry format; anything that would need the kernels raises."""

    def __init__(self, path, data, state_dict, optimizer):
        self.path, self.data, self.state_dict, self.optimizer = path, data, state_dict, optimizer
        self.num_timesteps = data.get("num_timesteps", 0)
        self.obs_shape = tuple(data["observation_space"].get("_shape") or ())
        self.act_shape = tuple(data.get("action_space", {}).get("_shape") or ())

    def save(self, path):
        path = str(path)
        if not path.endswith(".zip"):
            path += ".zip"
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)

        def pth(obj):
            bio = io.BytesIO()
            torch.save(obj, bio)
            return bio.getvalue()

        entries = [("data", json.dumps(self.data, indent=4)), ("pytorch_variables.pth", pth({})),
                   ("policy.pth", pth(dict(self.state_dict))), ("policy.optimizer.pth", pth(self.optimizer or {})),
                   ("_stable_baselines3_version", SB3_VERSION),
                   ("system_info.txt", f"- mobrob_b200 (B200-native), archive passed through\n- PyTorch: {torch.__version__}\n")]
        tmp = path + ".tmp"
        with zipfile.ZipFile(tmp, "w") as z:   # the source may be the destination (fix_pickle_warning.py saves in place)
            for name, blob in entries:
                z.writestr(name, blob)
        os.replace(tmp, path)

    def _out_of_scope(self, *a, **k):
        raise NotImplementedError(f"{os.path.basename(self.path)}: observations {self.obs_shape} -> actions {self.act_shape} "
                                  "are outside the B200 path (point and car; SURVEY.md section 2)")

    predict = learn = train = collect_rollouts = set_env = _out_of_scope


def _stored_schedule(entry, what):
    """A hyper-parameter as SB3 stores it in the zip's ``data``: a number, or a pickled schedule
    ({":serialized:": base64 cloudpickle}) -- constant_fn for the shipped zips.  A stored callable is
    returned as a callable (PPO evaluates it before every update); nothing is silently replaced."""
    if isinstance(entry, (int, float)):
        return float(entry)
    if isinstance(entry, dict):
        blob = entry.get(":serialized:")
        if blob:
            try:
                import cloudpickle

                fn = cloudpickle.loads(base64.b64decode(blob))
                if callable(fn):
                    if isinstance(fn, _Constant):
                        return fn.val
                    return fn
            except Exception:
                pass
        if isinstance(entry.get("value"), (int, float)):
            return float(entry["value"])
    raise NotImplementedError(f"cannot restore the stored {what} schedule: {str(entry)[:120]}")


class _Constant:
    """constant_fn(val) of SB3: the schedule objects stored under clip_range / lr_schedule."""

    def __init__(self, val):
        self.val = float(val)

    def __call__(self, _progress_remaining):
        return self.val
