"""SB3 2.0.0 PPO.train with ``clip_range_vf`` and ``target_kl``, restated on top of oracle/sb3_oracle.py (test
infrastructure only; torch-CPU autograd is the arithmetic).

The two settings as SB3 2.0.0's PPO.train applies them, per minibatch:
  * clip_range_vf (a float, evaluated once per train()): ``values_pred = old_values + clamp(values - old_values,
    -c, c)`` and ``value_loss = mse_loss(returns, values_pred)``; ``old_values`` are RolloutBuffer.values.
  * target_kl: after the losses and their log entries (policy loss, clip fraction, value loss, entropy loss,
    approx_kl) have been appended and BEFORE the optimizer step, ``approx_kl > 1.5 * target_kl`` skips this
    minibatch's step and leaves every remaining epoch.  ``_n_updates`` counts each epoch entered, the stopping one
    included.
With both left at None, ``ppo_loss`` and ``train_epochs`` compute exactly what oracle/sb3_oracle.py computes.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle import sb3_oracle


def ppo_loss(policy, obs, actions, old_log_prob, advantages, returns, old_values=None, clip_range=0.2,
             ent_coef=0.05, vf_coef=0.5, normalize_advantage=True, clip_range_vf=None):
    """One minibatch of PPO.train.  Returns (loss, stats); stats also counts the samples whose value was clipped
    below / above (vf_low / vf_high, python ints)."""
    values, log_prob, entropy = policy.evaluate_actions(obs, actions)
    adv = advantages
    if normalize_advantage and len(adv) > 1:
        adv = (adv - adv.mean()) / (adv.std() + 1e-8)
    ratio = torch.exp(log_prob - old_log_prob)
    pl1 = adv * ratio
    pl2 = adv * torch.clamp(ratio, 1 - clip_range, 1 + clip_range)
    policy_loss = -torch.min(pl1, pl2).mean()
    clip_fraction = torch.mean((torch.abs(ratio - 1) > clip_range).float()).item()
    vf_low = vf_high = 0
    if clip_range_vf is None:
        values_pred = values
    else:
        diff = values - old_values
        values_pred = old_values + torch.clamp(diff, -clip_range_vf, clip_range_vf)
        vf_low, vf_high = int((diff < -clip_range_vf).sum()), int((diff > clip_range_vf).sum())
    value_loss = torch.nn.functional.mse_loss(returns, values_pred)
    entropy_loss = -torch.mean(entropy)
    loss = policy_loss + ent_coef * entropy_loss + vf_coef * value_loss
    with torch.no_grad():
        log_ratio = log_prob - old_log_prob
        approx_kl = torch.mean((torch.exp(log_ratio) - 1) - log_ratio).item()
    stats = dict(policy_loss=policy_loss.item(), value_loss=value_loss.item(),
                 entropy_loss=entropy_loss.item(), loss=loss.item(),
                 clip_fraction=clip_fraction, approx_kl=approx_kl, vf_low=vf_low, vf_high=vf_high)
    return loss, stats


def train_epochs(policy, optimizer, buf, n_epochs, batch_size, perms=None, rng=None, max_grad_norm=0.5,
                 clip_range_vf=None, target_kl=None, **loss_kw):
    """PPO.train over a collected buffer (buf["values"] = the rollout's values when clip_range_vf is set).
    Returns (stats per evaluated minibatch, index of the minibatch that stopped the update or None).  The stopping
    minibatch's stats are included; its step is not taken (no grad_norm entry)."""
    keys = ["obs", "actions", "log_probs", "advantages", "returns"] + (["values"] if clip_range_vf is not None else [])
    flat = {k: torch.as_tensor(sb3_oracle.flatten_env_major(buf[k])) for k in keys}
    n = flat["obs"].shape[0]
    all_stats = []
    for ep in range(n_epochs):
        idx = perms[ep] if perms is not None else (rng or np.random).permutation(n)
        for s in range(0, n, batch_size):
            b = torch.as_tensor(np.asarray(idx[s:s + batch_size], dtype=np.int64))
            old_values = flat["values"][b].flatten() if clip_range_vf is not None else None
            loss, stats = ppo_loss(policy, flat["obs"][b], flat["actions"][b], flat["log_probs"][b].flatten(),
                                   flat["advantages"][b].flatten(), flat["returns"][b].flatten(), old_values,
                                   clip_range_vf=clip_range_vf, **loss_kw)
            all_stats.append(stats)
            if target_kl is not None and stats["approx_kl"] > 1.5 * target_kl:
                return all_stats, len(all_stats) - 1
            optimizer.zero_grad()
            loss.backward()
            stats["grad_norm"] = float(torch.nn.utils.clip_grad_norm_(policy.parameters(), max_grad_norm))
            optimizer.step()
    return all_stats, None


def epochs_entered(stop, n_mb, n_epochs):
    """SB3's _n_updates increment of one train(): every epoch entered, the stopping one included."""
    return n_epochs if stop is None else stop // n_mb + 1


def pick_target_kl(kls, lo, hi, margin=0.01):
    """A target_kl whose first crossing (approx_kl > 1.5 * target_kl) falls at an index in [lo, hi) of the KL
    sequence `kls` (from a run without target_kl), with every evaluated KL at least `margin` (relative) away from
    1.5 * target_kl; of the candidates, the one with the widest margin.  Returns (target_kl, index) or None."""
    best = None
    for j in range(max(lo, 1), hi):   # the threshold sits halfway (geometrically) between max(kls[:j]) and kls[j]
        below = max(kls[:j])
        if below > 0 and kls[j] > below * (1 + margin) ** 2 and (best is None or kls[j] / below > best[0]):
            best = (kls[j] / below, j, np.sqrt(below * kls[j]))
    return None if best is None else (best[2] / 1.5, best[1])
