"""``evaluate_policy`` of [SB3 2.0.0] ``common/evaluation.py``, with the loop on the device for a ``GpuVecEnv``.

SB3's semantics: ``env.reset()``, then env ``i`` counts its first ``(n_eval_episodes + i) // n_envs`` finished
episodes (Monitor's ``info["episode"]`` return and length), every env keeps stepping until the last one has met its
target, and the lists come out in (step, env index) order.

For a ``GpuVecEnv`` without a per-step ``callback`` and without ``render``, the whole loop is ONE call of
``mr_evaluate`` (a fused kernel for the point robot's default observation; one launch plus the env step per step
otherwise); the host only puts the records into SB3's order.  Anything else takes SB3's loop as written
(``model.predict`` + the VecEnv protocol), which is also the reference the device path is tested against.

``max_steps`` is the one addition: the evaluation stops there (``RuntimeError``) if some env has not finished its
episodes, so that a policy that never reaches a goal on an env without a time limit cannot hold the GPU forever.
"""
from __future__ import annotations

import math
import warnings

import numpy as np
import torch

from . import _lib

__all__ = ["evaluate_policy"]


def episode_targets(n_eval_episodes: int, n_envs: int) -> np.ndarray:
    """Episodes env i counts: ``(n_eval_episodes + i) // n_envs`` (SB3's ``episode_count_targets``)."""
    return (int(n_eval_episodes) + np.arange(n_envs, dtype=np.int64)) // int(n_envs)


def record_order(ep_t: np.ndarray, n_envs: int, n_eval_episodes: int) -> np.ndarray:
    """Permutation that puts the device's records (env i's episodes in consecutive slots, in the order they ended,
    ``ep_t`` = the step at which each ended) into the order SB3's loop appends them: by step, then by env index."""
    env_of_slot = np.repeat(np.arange(n_envs, dtype=np.int64), episode_targets(n_eval_episodes, n_envs))
    return np.lexsort((env_of_slot, np.asarray(ep_t)))


def resolve_max_steps(env, n_eval_episodes: int, max_steps: int | None) -> int | None:
    """The step bound of one evaluation.  An env with a time limit (a positive ``time_limit`` attribute) finishes every
    target within ``ceil(n_eval_episodes / n_envs) * time_limit`` steps, because TimeLimit truncates each episode;
    that is the default.  An env whose ``time_limit`` is None or 0 has no such bound and needs an explicit one.  A
    VecEnv that does not say (no ``time_limit`` attribute) runs unbounded, as in SB3."""
    if max_steps is not None:
        if int(max_steps) < 0:
            raise ValueError(f"max_steps must not be negative, got {max_steps}")
        return int(max_steps)
    if not hasattr(env, "time_limit"):
        return None
    tl = env.time_limit
    if not tl or int(tl) <= 0:
        raise ValueError("evaluate_policy: the env has no time limit, so an episode may never end; pass max_steps "
                         "(the most VecEnv steps the evaluation may take)")
    return math.ceil(int(n_eval_episodes) / env.num_envs) * int(tl)


def _is_gpu_vec_env(env) -> bool:
    from .vec_env import GpuVecEnv

    return isinstance(env, GpuVecEnv)


def evaluate_policy(model, env, n_eval_episodes: int = 10, deterministic: bool = True, render: bool = False,
                    callback=None, reward_threshold: float | None = None, return_episode_rewards: bool = False,
                    warn: bool = True, max_steps: int | None = None):
    """Run the policy for ``n_eval_episodes`` episodes and return ``(mean, std)`` of their rewards, or the lists of
    episode rewards and lengths with ``return_episode_rewards`` (SB3 2.0.0's signature plus ``max_steps``)."""
    gpu = _is_gpu_vec_env(env)
    # a GpuVecEnv is N x Monitor(TimeLimit(env)): its infos carry Monitor's "episode" entry
    is_monitor_wrapped = gpu
    if not is_monitor_wrapped and warn:
        warnings.warn("Evaluation environment is not wrapped with a ``Monitor`` wrapper. This may result in reporting "
                      "modified episode lengths and rewards, if other wrappers happen to modify these. Consider "
                      "wrapping environment first with ``Monitor`` wrapper.", UserWarning)
    bound = resolve_max_steps(env, n_eval_episodes, max_steps)
    if gpu and callback is None and not render:
        rewards, lengths = _evaluate_on_device(model, env, n_eval_episodes, deterministic, bound)
    else:
        rewards, lengths = _evaluate_loop(model, env, n_eval_episodes, deterministic, render, callback,
                                          is_monitor_wrapped, bound)
    mean_reward = np.mean(rewards)
    std_reward = np.std(rewards)
    if reward_threshold is not None:
        assert mean_reward > reward_threshold, f"Mean reward below threshold: {mean_reward:.2f} < {reward_threshold:.2f}"
    if return_episode_rewards:
        return rewards, lengths
    return mean_reward, std_reward


def _max_steps_error(bound):
    return RuntimeError(f"evaluate_policy: max_steps={bound} VecEnv steps were taken before every env finished its "
                        "episodes (the env is left after exactly max_steps steps)")


def _evaluate_loop(model, env, n_eval_episodes, deterministic, render, callback, is_monitor_wrapped, bound):
    """SB3 2.0.0's loop, step for step (plus the step bound)."""
    n_envs = env.num_envs
    episode_rewards, episode_lengths = [], []
    episode_counts = np.zeros(n_envs, dtype="int")
    episode_count_targets = episode_targets(n_eval_episodes, n_envs)
    current_rewards = np.zeros(n_envs)
    current_lengths = np.zeros(n_envs, dtype="int")
    observations = env.reset()
    states = None
    episode_starts = np.ones((env.num_envs,), dtype=bool)
    steps = 0
    while (episode_counts < episode_count_targets).any():
        if bound is not None and steps >= bound:
            raise _max_steps_error(bound)
        actions, states = model.predict(observations, state=states, episode_start=episode_starts,
                                        deterministic=deterministic)
        new_observations, rewards, dones, infos = env.step(actions)
        steps += 1
        current_rewards += rewards
        current_lengths += 1
        for i in range(n_envs):
            if episode_counts[i] < episode_count_targets[i]:
                reward = rewards[i]  # noqa: F841  (part of the locals() a callback receives, as in SB3)
                done = dones[i]
                info = infos[i]
                episode_starts[i] = done
                if callback is not None:
                    callback(locals(), globals())
                if dones[i]:
                    if is_monitor_wrapped:
                        if "episode" in info.keys():
                            episode_rewards.append(info["episode"]["r"])
                            episode_lengths.append(info["episode"]["l"])
                            episode_counts[i] += 1
                    else:
                        episode_rewards.append(current_rewards[i])
                        episode_lengths.append(current_lengths[i])
                        episode_counts[i] += 1
                    current_rewards[i] = 0
                    current_lengths[i] = 0
        observations = new_observations
        if render:
            env.render()
    return episode_rewards, episode_lengths


def _evaluate_on_device(model, env, n_eval_episodes, deterministic, bound):
    policy = model.policy
    if policy.obs_dim != env.obs_dim:
        raise ValueError(f"the policy takes {policy.obs_dim} observation floats, the env emits {env.obs_dim}")
    dev = env.device
    params = policy.flat if policy.flat.device == dev else policy.flat.to(dev)
    E = int(n_eval_episodes)
    obs = env.reset_tensor()
    ep_r = torch.empty(max(E, 1), dtype=torch.float64, device=dev)
    ep_l = torch.empty(max(E, 1), dtype=torch.int32, device=dev)
    ep_t = torch.empty(max(E, 1), dtype=torch.int64, device=dev)
    steps_taken = torch.zeros(1, dtype=torch.int64, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    # the stochastic draws use the training rollouts' Philox key: PPO.collect_rollouts' seed and global env index
    seed = int(model.seed if getattr(model, "seed", None) is not None else 0)
    lib = _lib.load()
    _lib.check(lib.mr_evaluate(env._h, params.data_ptr(), int(bool(deterministic)), E, int(bound),
                               seed, int(env.eval_steps), int(env.first_rank), obs.data_ptr(), ep_r.data_ptr(),
                               ep_l.data_ptr(), ep_t.data_ptr(), steps_taken.data_ptr(), status.data_ptr(),
                               env._stream()))
    steps, status = int(steps_taken.item()), int(status.item())
    env.eval_steps += steps   # the next evaluation's Philox counters start after this one's
    if status:
        raise _max_steps_error(bound)
    order = record_order(ep_t[:E].cpu().numpy(), env.num_envs, E)
    r = ep_r[:E].cpu().numpy()[order]
    l = ep_l[:E].cpu().numpy()[order]
    # Monitor rounds the return to 6 decimals in info["episode"]
    return [round(float(x), 6) for x in r], [int(x) for x in l]
