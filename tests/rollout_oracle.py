"""Shared references of the rollout tests: the device action noise restated in numpy, and the oracle replay of one
collect_rollouts() call (the policy on the device's observations, the environment on the device's actions).

Device noise (mobrob_b200/csrc/common.cuh, ``philox4x32`` + ``normal2``): the draw of env n at step t of a rollout is
Philox4x32-10 with counter ``(g_lo, g_hi, c_lo, c_hi)``, ``g = env_offset + n`` (the global env id) and
``c = noise_offset + t`` (``noise_offset = rollout count * n_steps``), key ``(seed_lo, seed_hi)``; words ``x`` and ``y``
go through Box-Muller: ``u = (float32(u) + 0.5f) * 2^-32``, ``r = sqrt(-2 log a)``, ``z = (r cos 2 pi b, r sin 2 pi b)``.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from oracle import point_oracle as po, sb3_oracle
from oracle.vec_oracle import GoalVecOracle

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = 0x9E3779B9, 0xBB67AE85
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32(ctr, key):
    """Philox4x32-10.  ctr: four uint32 arrays (broadcastable), key: two Python ints / uint32 arrays.
    Returns the four output words as uint32 arrays."""
    x, y, z, w = (np.asarray(c, dtype=np.uint64) & _MASK for c in ctr)
    k0, k1 = (np.asarray(k, dtype=np.uint64) & _MASK for k in key)
    for _ in range(10):
        p0, p1 = _M0 * x, _M1 * z            # exact: both factors < 2^32
        h0, l0 = p0 >> np.uint64(32), p0 & _MASK
        h1, l1 = p1 >> np.uint64(32), p1 & _MASK
        x, y, z, w = h1 ^ y ^ k0, l1, h0 ^ w ^ k1, l0
        k0 = (k0 + np.uint64(_W0)) & _MASK
        k1 = (k1 + np.uint64(_W1)) & _MASK
    return tuple(v.astype(np.uint32) for v in (x, y, z, w))


def normal2(u0, u1):
    """Box-Muller of common.cuh: two float32 standard normals from two uint32 words.  float32 throughout except
    sin / cos, taken in float64 of the float32 argument (sincospif(2b) = sin / cos of pi * 2b)."""
    scale = np.float32(1.0 / 4294967296.0)
    a = (np.asarray(u0, np.uint32).astype(np.float32) + np.float32(0.5)) * scale
    b = (np.asarray(u1, np.uint32).astype(np.float32) + np.float32(0.5)) * scale
    a = np.minimum(np.maximum(a, np.float32(1e-10)), np.float32(1.0))
    r = np.sqrt(np.float32(-2.0) * np.log(a))
    ang = np.pi * (np.float32(2.0) * b).astype(np.float64)
    return r * np.cos(ang).astype(np.float32), r * np.sin(ang).astype(np.float32)


def device_draws(seed, n_envs, T, noise_offset=0, env_offset=0):
    """The [T][N][2] N(0, 1) draws a rollout of T steps over envs env_offset .. env_offset + N - 1 takes."""
    g = np.uint64(env_offset) + np.arange(n_envs, dtype=np.uint64)[None, :]
    c = np.uint64(noise_offset) + np.arange(T, dtype=np.uint64)[:, None]
    lo = lambda v: v & _MASK                       # noqa: E731
    hi = lambda v: v >> np.uint64(32)              # noqa: E731
    s = int(seed) & ((1 << 64) - 1)
    x, y, _, _ = philox4x32((lo(g), hi(g), lo(c), hi(c)), (s & 0xFFFFFFFF, s >> 32))
    z0, z1 = normal2(x, y)
    return np.stack([z0, z1], axis=-1)


def rollout_draws(model, rollout_index):
    """The draws collect_rollouts() number `rollout_index` (0-based) of `model` takes with eps=None."""
    T, env = model.n_steps, model.env
    return device_draws(int(model.seed or 0), env.num_envs, T, rollout_index * T, env.first_rank)


def setup(golden_dir, n, T, seed, time_limit, pretrained, **ppo_kw):
    from mobrob_b200 import GpuVecEnv
    from mobrob_b200.ppo import PPO

    env = GpuVecEnv("point", n, seed=None, time_limit=time_limit, terminate_on_goal=True)
    model = PPO("MlpPolicy", env, n_steps=T, seed=seed, gae_lambda=0.5, ent_coef=0.05, **ppo_kw)
    ref_pol = sb3_oracle.MlpPolicyOracle(14)
    if pretrained:
        w = dict(np.load(os.path.join(golden_dir, "point_policy.npz")))
        model.policy.load_state_dict({k: torch.as_tensor(v) for k, v in w.items()})
        ref_pol.load_numpy(w)
    else:
        ref_pol.load_state_dict({k: v.cpu() for k, v in model.policy.state_dict().items()})
    venv = GoalVecOracle(po.PointBody(n), seed=seed, time_limit=time_limit, terminate_on_goal=True)
    return model, ref_pol, venv


def teacher_forced_check(model, ref_pol, venv, eps, first, last_obs_ref, gamma=0.99):
    """Replay the device rollout through the oracle step by step.

    The point robot's turning servo is stiff against the 2 ms timestep (explicit-Euler factor
    about -3.9 per substep inside the un-saturated band), so trajectories are sensitive to
    1e-6 differences in un-saturated actions (DESIGN.md "Sensitivity").  Parity is therefore
    checked per component on identical inputs: the policy on the device's observations, the
    environment on the device's float32 actions.

    Returns the oracle's last observation and done flags, the number of time-outs and Monitor's
    finished episodes (return, length) in SB3's order: by step, then by env index.
    """
    b = {k: v.cpu().numpy() for k, v in model.buf.items()}
    T, n = b["rewards"].shape
    obs_ref = last_obs_ref
    n_trunc = 0
    ep_infos = []
    for t in range(T):
        np.testing.assert_allclose(b["obs"][t], obs_ref, rtol=1e-5, atol=2e-6, err_msg=f"obs t={t}")
        with torch.no_grad():
            a_ref, v_ref, lp_ref = ref_pol.forward_with_noise(torch.as_tensor(b["obs"][t]), torch.as_tensor(eps[t]))
        a_scale = max(1.0, float(a_ref.abs().max()))
        assert np.abs(b["actions"][t] - a_ref.numpy()).max() <= 1e-5 * a_scale, f"actions t={t}"
        np.testing.assert_allclose(b["values"][t], v_ref.numpy(), rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(b["log_probs"][t], lp_ref.numpy(), rtol=1e-5, atol=1e-5)
        obs_ref, rew, done, info = venv.step(np.clip(b["actions"][t], -1.0, 1.0))
        trunc = done & info["truncated"]
        if trunc.any():
            with torch.no_grad():
                _, tv = ref_pol.mean_value(torch.as_tensor(info["terminal_obs"][trunc]))
            rew[trunc] += gamma * tv.numpy()
            n_trunc += int(trunc.sum())
        for i in np.nonzero(done)[0]:
            ep_infos.append((float(info["ep_r"][i]), int(info["ep_l"][i])))
        np.testing.assert_allclose(b["rewards"][t], rew, rtol=1e-5, atol=2e-6, err_msg=f"rewards t={t}")
        nxt = b["episode_starts"][t + 1] if t + 1 < T else model._last_episode_starts.cpu().numpy()
        np.testing.assert_array_equal(nxt.astype(bool), done, err_msg=f"done flags t={t}")
    np.testing.assert_array_equal(b["episode_starts"][0].astype(bool), first)
    np.testing.assert_allclose(model._last_obs.cpu().numpy(), obs_ref, rtol=1e-5, atol=2e-6)
    with torch.no_grad():
        _, lv = ref_pol.mean_value(torch.as_tensor(obs_ref))
    np.testing.assert_allclose(model.last_val.cpu().numpy(), lv.numpy(), rtol=1e-5, atol=1e-5)
    np.testing.assert_array_equal(model.last_done.cpu().numpy().astype(bool), done)
    # GAE: bit exact on the device's own inputs
    adv, ret = sb3_oracle.gae_numpy(b["rewards"], b["values"], b["episode_starts"],
                                    model.last_val.cpu().numpy(), done, gamma, model.gae_lambda)
    np.testing.assert_array_equal(b["advantages"], adv)
    np.testing.assert_array_equal(b["returns"], ret)
    return obs_ref, done, n_trunc, ep_infos
