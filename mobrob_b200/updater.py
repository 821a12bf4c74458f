"""Host wrapper around the PPO update kernels (mr_ppo_adv_stats / mr_ppo_grad / mr_adam_step).

Owns the flat parameter vector, the Adam moments and the gradient scratch as torch CUDA
tensors (so ``state_dict`` views, NCCL all-reduce and checkpointing need no extra copies).
Mirrors what [SB3] PPO.train does per minibatch; see include/mobrob_b200.h.

clip_range_vf / target_kl (None = off, the default) go to the entry points as their trailing arguments (0 / NULL
when off, which launches the default kernels).  With target_kl the update's control word (``self.ctrl``, one int32 on
the device) records an early stop; ``begin_update()`` clears it and must be called before the first launch of every
update.  The control word is passed only when target_kl is set, so the default path never runs the extended kernels.
"""
from __future__ import annotations

import torch

from . import _lib


class PpoUpdater:
    def __init__(self, obs_dim: int, device: torch.device, lr: float = 3e-4, betas=(0.9, 0.999),
                 eps: float = 1e-5, max_grad_norm: float = 0.5, clip_range: float = 0.2,
                 ent_coef: float = 0.0, vf_coef: float = 0.5, normalize_advantage: bool = True,
                 clip_range_vf: float | None = None, target_kl: float | None = None):
        self.lib = _lib.load()
        if not 0 < obs_dim < 32:
            raise ValueError(f"the PPO kernels take observations of 1..31 floats (got {obs_dim}): with the optional "
                             "observation keys, the car's qpos / qvel do not fit")
        self.obs_dim = obs_dim
        self.device = device
        self.lr, self.betas, self.eps = lr, betas, eps
        self.max_grad_norm = max_grad_norm
        self.clip_range, self.ent_coef, self.vf_coef = clip_range, ent_coef, vf_coef
        self.normalize_advantage = normalize_advantage
        self.clip_range_vf, self.target_kl = clip_range_vf, target_kl
        self.n_params = int(self.lib.mr_ppo_num_params(obs_dim))
        self.stride = int(self.lib.mr_ppo_grad_stride(obs_dim))
        with torch.cuda.device(device):
            self.max_parts = int(self.lib.mr_ppo_max_parts())
        f32 = dict(dtype=torch.float32, device=device)
        self.params = torch.zeros(self.n_params, **f32)
        self.exp_avg = torch.zeros(self.n_params, **f32)
        self.exp_avg_sq = torch.zeros(self.n_params, **f32)
        self.step = torch.zeros(2, dtype=torch.int64, device=device)  # [count, kernel ticket]
        # caller-owned scratch of the update kernels (include/mobrob_b200.h): one partial vector per
        # CTA plus one row; the fused epoch kernel keeps its accumulators and barrier word in it
        self.partials = torch.zeros((self.max_parts + 1, self.stride), **f32)
        self.grad = torch.zeros(self.stride, **f32)
        self._rows = torch.empty(0, dtype=torch.int32, device=device)
        # target_kl: k > 0 once the update stopped after its k-th minibatch (caller-owned, like the barrier word)
        self.ctrl = torch.zeros(1, dtype=torch.int32, device=device)

    def begin_update(self):
        """Clear the control word (target_kl): once per update, before its first launch."""
        if self.target_kl is not None:
            self.ctrl.zero_()

    def ctrl_ptr(self):
        """The control word as the entry points take it: only with target_kl (NULL otherwise)."""
        return self.ctrl.data_ptr() if self.target_kl is not None else None

    def rows(self, n: int) -> torch.Tensor:
        """int32 scratch for the samples as buffer rows (owned here, not by the library)."""
        if self._rows.numel() < n:
            self._rows = torch.empty(n, dtype=torch.int32, device=self.device)
        return self._rows

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def adv_stats(self, adv: torch.Tensor, perm: torch.Tensor, batch_size: int, N: int, T: int):
        n = perm.numel()
        n_mb = (n + batch_size - 1) // batch_size
        stats = torch.empty((n_mb, 3), dtype=torch.float64, device=self.device)
        _lib.check(self.lib.mr_ppo_adv_stats(adv.data_ptr(), perm.data_ptr(), n, batch_size, N, T,
                                             stats.data_ptr(), self._stream()))
        return stats

    def compute_grad(self, buf: dict, perm_slice: torch.Tensor, mb_stats: torch.Tensor, N: int, T: int,
                     rank_share: float = 1.0):
        """buf: time-major rollout tensors obs/actions/log_probs/advantages/returns (+ values with clip_range_vf)."""
        cvf = float(self.clip_range_vf or 0.0)
        _lib.check(self.lib.mr_ppo_grad(
            self.params.data_ptr(), self.obs_dim, buf["obs"].data_ptr(), buf["actions"].data_ptr(),
            buf["log_probs"].data_ptr(), buf["advantages"].data_ptr(), buf["returns"].data_ptr(),
            perm_slice.data_ptr(), self.rows(perm_slice.numel()).data_ptr(), perm_slice.numel(),
            mb_stats.data_ptr(), N, T, self.clip_range, self.ent_coef, self.vf_coef,
            int(self.normalize_advantage), rank_share, self.partials.data_ptr(), self.grad.data_ptr(),
            buf["values"].data_ptr() if cvf > 0 else None, cvf, self.ctrl_ptr(), self._stream()))
        return self.grad

    def adam_step(self, info: torch.Tensor | None = None, mb_index: int = 0):
        """mb_index: this minibatch's index in the update (what an early stop records)."""
        _lib.check(self.lib.mr_adam_step(
            self.params.data_ptr(), self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(),
            self.grad.data_ptr(), self.n_params, self.step.data_ptr(), self.lr, self.betas[0],
            self.betas[1], self.eps, self.max_grad_norm, None if info is None else info.data_ptr(),
            float(self.target_kl or 0.0), self.ctrl_ptr(), mb_index, self._stream()))

    def train_epoch(self, buf: dict, perm: torch.Tensor, stats: torch.Tensor, batch_size: int, N: int, T: int,
                    info: torch.Tensor | None = None, mb0: int = 0):
        """All minibatches of one epoch, launched from C (single-GPU path).  mb0: index of the epoch's first
        minibatch in the update (target_kl)."""
        cvf = float(self.clip_range_vf or 0.0)
        _lib.check(self.lib.mr_ppo_train_epoch(
            self.params.data_ptr(), self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(), self.step.data_ptr(),
            self.obs_dim, buf["obs"].data_ptr(), buf["actions"].data_ptr(), buf["log_probs"].data_ptr(),
            buf["advantages"].data_ptr(), buf["returns"].data_ptr(), perm.data_ptr(),
            self.rows(min(perm.numel(), batch_size)).data_ptr(), perm.numel(), batch_size,
            stats.data_ptr(), N, T, self.clip_range, self.ent_coef, self.vf_coef, int(self.normalize_advantage),
            self.lr, self.betas[0], self.betas[1], self.eps, self.max_grad_norm, self.partials.data_ptr(),
            self.grad.data_ptr(), None if info is None else info.data_ptr(),
            buf["values"].data_ptr() if cvf > 0 else None, cvf, float(self.target_kl or 0.0), self.ctrl_ptr(), mb0,
            self._stream()))

    def pack(self, buf: dict) -> torch.Tensor:
        """Packed sample records of a rollout (mr_ppo_pack_samples): what train_epoch_fused gathers from.
        Build them once per rollout, after GAE; they stay valid for all epochs of the update.  With clip_range_vf
        the records also carry buf["values"], the rollout's V(s)."""
        n_rows = buf["log_probs"].numel()
        rf = int(self.lib.mr_ppo_record_floats(self.obs_dim))
        if getattr(self, "_rec", None) is None or self._rec.numel() != n_rows * rf:
            self._rec = torch.empty(n_rows * rf, dtype=torch.float32, device=self.device)
        values = buf["values"].data_ptr() if self.clip_range_vf is not None else None
        _lib.check(self.lib.mr_ppo_pack_samples(
            self.obs_dim, buf["obs"].data_ptr(), buf["actions"].data_ptr(), buf["log_probs"].data_ptr(),
            buf["advantages"].data_ptr(), buf["returns"].data_ptr(), values, n_rows, self._rec.data_ptr(),
            self._stream()))
        return self._rec

    def prepare_epochs(self, adv: torch.Tensor, perms: torch.Tensor, batch_size: int, N: int, T: int):
        """All epochs of an update at once: perms [E, n] int64 -> (stats [E, n_mb, 3] float64, rows [E, n] int32)."""
        E, n = perms.shape
        n_mb = (n + batch_size - 1) // batch_size
        stats = torch.empty((E, n_mb, 3), dtype=torch.float64, device=self.device)
        if getattr(self, "_rows_all", None) is None or self._rows_all.shape != (E, n):
            self._rows_all = torch.empty((E, n), dtype=torch.int32, device=self.device)
        _lib.check(self.lib.mr_ppo_prepare_epochs(adv.data_ptr(), perms.data_ptr(), E, n, batch_size, N, T,
                                                  stats.data_ptr(), self._rows_all.data_ptr(), self._stream()))
        return stats, self._rows_all

    def prepare_epochs_device(self, adv: torch.Tensor, seed: int, stream_ids, batch_size: int, N: int, T: int):
        """prepare_epochs for the device index streams (seed, stream_ids), generated on the fly."""
        import ctypes

        E, n = len(stream_ids), N * T
        n_mb = (n + batch_size - 1) // batch_size
        stats = torch.empty((E, n_mb, 3), dtype=torch.float64, device=self.device)
        if getattr(self, "_rows_all", None) is None or self._rows_all.shape != (E, n):
            self._rows_all = torch.empty((E, n), dtype=torch.int32, device=self.device)
        keys = (ctypes.c_uint64 * E)(*stream_ids)
        _lib.check(self.lib.mr_ppo_prepare_epochs_device(seed, keys, E, adv.data_ptr(), n, batch_size, N, T,
                                                         stats.data_ptr(), self._rows_all.data_ptr(), self._stream()))
        return stats, self._rows_all

    def train_epoch_fused(self, buf: dict | None, perm: torch.Tensor | None, stats: torch.Tensor, batch_size: int, N: int,
                          T: int, info: torch.Tensor | None = None, xchg=None, rows: torch.Tensor | None = None,
                          mb0: int = 0):
        """One cooperative launch for the whole epoch; xchg (PeerExchange) adds the in-kernel
        NVLink all-reduce of the gradient (stats must then be the all-reduced, global sums).
        buf = the rollout arrays (packed here) or None to reuse the records of the last pack().
        Either perm (int64 env-major sample ids) or rows (one row of prepare_epochs' output) names the samples.
        mb0: index of the launch's first minibatch in the update (target_kl)."""
        rec = self.pack(buf) if buf is not None else self._rec
        n = perm.numel() if perm is not None else rows.numel()
        _lib.check(self.lib.mr_ppo_epoch_fused(
            self.params.data_ptr(), self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(), self.step.data_ptr(),
            self.obs_dim, rec.data_ptr(), None if perm is None else perm.data_ptr(),
            self.rows(n).data_ptr() if rows is None else rows.data_ptr(), n,
            batch_size, stats.data_ptr(), N, T, self.clip_range,
            self.ent_coef, self.vf_coef, int(self.normalize_advantage), self.lr, self.betas[0], self.betas[1],
            self.eps, self.max_grad_norm, self.partials.data_ptr(), self.grad.data_ptr(),
            None if info is None else info.data_ptr(), None if xchg is None else xchg.handle,
            float(self.clip_range_vf or 0.0), float(self.target_kl or 0.0), self.ctrl_ptr(), mb0, self._stream()))


class PeerExchange:
    """Per-rank inbox in CUDA-IPC-shared device memory for the in-kernel gradient all-reduce."""

    def __init__(self, obs_dim: int, device: torch.device):
        import ctypes

        import numpy as np
        import torch.distributed as dist

        self.lib = _lib.load()
        self.world, self.rank = dist.get_world_size(), dist.get_rank()
        h = ctypes.c_void_p()
        mine = np.zeros(64, dtype=np.uint8)
        _lib.check(self.lib.mr_xchg_create(self.world, self.rank, device.index or 0, obs_dim, ctypes.byref(h),
                                           mine.ctypes.data))
        self.handle = h
        allh = [None] * self.world
        dist.all_gather_object(allh, mine.tobytes())
        flat = np.frombuffer(b"".join(allh), dtype=np.uint8).copy()
        _lib.check(self.lib.mr_xchg_connect(self.handle, flat.ctypes.data))
        dist.barrier()

    def timed_out(self) -> bool:
        """True if an in-kernel exchange gave up waiting for a peer (synchronises the device)."""
        import ctypes

        flag = ctypes.c_int(0)
        _lib.check(self.lib.mr_xchg_status(self.handle, ctypes.byref(flag)))
        return bool(flag.value)

    def close(self):
        if getattr(self, "handle", None) is not None:
            self.lib.mr_xchg_destroy(self.handle)
            self.handle = None
