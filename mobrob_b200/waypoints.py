"""``follow_waypoints``: run a goal-conditioned policy through a sequence of waypoints per env, on the device.

A planner drives the reference's EnvWrapper with ``set_goal`` / ``model.predict`` / ``env.step`` / ``reached()``.
For each env ``i`` independently, from its current state, the loop is::

    env.set_goal(W[i, 0]); obs = env.get_obs()
    k, t, ret = 0, 0, 0.0
    while k < K and t < max_steps:
        a, _ = model.predict(obs, deterministic=deterministic)
        obs, r, terminated, _, _ = env.step(a)          # get_env(..., terminate_on_goal=True, time_limit=None)
        t += 1; ret += r
        if terminated:                                   # reached(): |pos_xy - goal| < 0.3
            arrival[i, k] = t; k += 1
            if k < K: env.set_goal(W[i, k]); obs = env.get_obs()

An env that has finished does not move while the others run.  The whole loop is one ``mr_follow_waypoints`` call.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib

__all__ = ["follow_waypoints"]


def check_waypoints(waypoints, n_envs: int, max_steps) -> np.ndarray | torch.Tensor:
    """[N, K, 2] or [K, 2] (the same path for every env) -> [N, K, 2] float32, numpy or tensor as given."""
    if int(max_steps) < 1:
        raise ValueError(f"max_steps must be at least 1, got {max_steps}")
    shape = tuple(waypoints.shape)
    if len(shape) == 2 and shape[1] == 2:
        if shape[0] < 1:
            raise ValueError("waypoints: K must be at least 1")
        if isinstance(waypoints, torch.Tensor):
            return waypoints.to(torch.float32).unsqueeze(0).expand(n_envs, shape[0], 2)
        return np.broadcast_to(np.asarray(waypoints, np.float32), (n_envs, shape[0], 2))
    if len(shape) != 3 or shape[0] != n_envs or shape[2] != 2:
        raise ValueError(f"waypoints must have shape ({n_envs}, K, 2) or (K, 2), got {shape}")
    if shape[1] < 1:
        raise ValueError("waypoints: K must be at least 1")
    return waypoints.to(torch.float32) if isinstance(waypoints, torch.Tensor) else np.asarray(waypoints, np.float32)


def vec_env_of(env):
    """The GpuVecEnv under ``env`` (itself, or the batch of one inside a get_env wrapper), refused when its auto-reset
    would draw a random goal mid-path."""
    from .envs.wrapper import MujocoGoalEnv, TimeLimit
    from .vec_env import GpuVecEnv

    if isinstance(env, TimeLimit):
        raise ValueError("follow_waypoints: the env has a time limit; use get_env(name, time_limit=None) "
                         "(max_steps bounds the call)")
    if isinstance(env, MujocoGoalEnv):
        return env.env
    if not isinstance(env, GpuVecEnv):
        raise TypeError(f"follow_waypoints takes a GpuVecEnv or a get_env() env, got {type(env).__name__}")
    if env.terminate_on_goal or (env.time_limit or 0) > 0:
        raise ValueError("follow_waypoints: the env must not reset itself; create it with "
                         "GpuVecEnv(..., terminate_on_goal=False, time_limit=None)")
    return env


def follow_waypoints(model, env, waypoints, max_steps: int, deterministic: bool = True,
                     record_positions: bool = False) -> dict:
    """Follow ``waypoints`` ([N, K, 2] or [K, 2], float32 world xy, numpy or tensor) with ``model``'s policy on every
    env of ``env`` (a ``GpuVecEnv`` created with ``terminate_on_goal=False, time_limit=None``, or a ``get_env`` env
    without a time limit), at most ``max_steps`` steps per env.  Returns numpy arrays:

    * ``arrivals`` int64 [N, K]: the step (1-based) at which each waypoint was reached, -1 if it was not
    * ``returns`` float64 [N]: the sum of the env's rewards (reward_fn, reach bonus included)
    * ``steps`` int64 [N]: the steps each env took
    * ``positions`` float32 [max_steps + 1, N, 2] with ``record_positions``: world xy after each step (row 0: the
      start); rows past an env's end repeat its final position

    Stochastic actions (``deterministic=False``) use evaluate_policy's Philox draws and continue its counter
    (``GpuVecEnv.eval_steps``), so no draw repeats across calls."""
    venv = vec_env_of(env)
    N = venv.num_envs
    wp = check_waypoints(waypoints, N, max_steps)
    K = int(wp.shape[1])
    policy = model.policy
    if policy.obs_dim != venv.obs_dim:
        raise ValueError(f"the policy takes {policy.obs_dim} observation floats, the env emits {venv.obs_dim}")
    dev = venv.device
    wp_dev = torch.as_tensor(wp).to(device=dev, dtype=torch.float32).contiguous()
    params = policy.flat if policy.flat.device == dev else policy.flat.to(dev)
    arrival = torch.empty((N, K), dtype=torch.int32, device=dev)
    ret = torch.empty(N, dtype=torch.float64, device=dev)
    steps = torch.empty(N, dtype=torch.int32, device=dev)
    pos = torch.empty((int(max_steps) + 1, N, 2), dtype=torch.float32, device=dev) if record_positions else None
    seed = int(model.seed if getattr(model, "seed", None) is not None else 0)
    _lib.check(venv.lib.mr_follow_waypoints(venv._h, params.data_ptr(), int(bool(deterministic)), wp_dev.data_ptr(), K,
                                            int(max_steps), seed, int(venv.eval_steps), int(venv.first_rank),
                                            venv.obs.data_ptr(), arrival.data_ptr(), ret.data_ptr(), steps.data_ptr(),
                                            _lib.ptr(pos), venv._stream()))
    out = {"arrivals": arrival.cpu().numpy().astype(np.int64), "returns": ret.cpu().numpy(),
           "steps": steps.cpu().numpy().astype(np.int64)}
    venv.eval_steps += int(out["steps"].max())
    if record_positions:
        out["positions"] = pos.cpu().numpy()
    if venv is not env:   # the wrapper's host-side view: the last goal set, reward_fn's _prev_pos
        reached = out["arrivals"][0] >= 0
        env._goal = np.array(wp[0, min(int(reached.sum()), K - 1)].tolist(), dtype=np.float32)
        env._prev_pos = env.get_pos()
    return out
