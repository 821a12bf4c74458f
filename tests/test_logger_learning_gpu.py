"""Observability parity (SURVEY 8f-2, appendix A.5) and a learning check.

* every key SB3's PPO dumps per iteration is emitted by ``learn()`` with the value SB3's own
  arithmetic (oracle/sb3_oracle.py: torch-CPU PPO.train) gives on the same rollout data and the same
  minibatch permutations, in SB3's order (train/* of update k are dumped with iteration k + 1);
  tensorboard events go where src/mobrob/rl_control/ppo.py:53-57 puts them;
* the bench configuration (point, 4096 envs) actually learns: the mean episode length collapses
  from the 1000-step time limit towards the shipped policy's ~100 steps.
"""
import os

import numpy as np
import pytest
import torch

from oracle import sb3_oracle

pytestmark = pytest.mark.gpu

TRAIN_KEYS = ["train/entropy_loss", "train/policy_gradient_loss", "train/value_loss", "train/approx_kl",
              "train/clip_fraction", "train/loss", "train/explained_variance", "train/std", "train/n_updates",
              "train/clip_range", "train/learning_rate"]
TIME_KEYS = ["time/fps", "time/iterations", "time/time_elapsed", "time/total_timesteps"]


def _episodes_of(bufs, last_starts):
    """(length, return) of every episode that ends inside the rollouts, in completion order, from
    RolloutBuffer.episode_starts / rewards (no time-limit truncation in this test, so the buffer's
    rewards are Monitor's)."""
    n = bufs[0]["rewards"].shape[1]
    run_l, run_r, out = np.zeros(n, np.int64), np.zeros(n), []
    starts = [b["episode_starts"] for b in bufs]
    for it, b in enumerate(bufs):
        T = b["rewards"].shape[0]
        for t in range(T):
            run_l += 1
            run_r += b["rewards"][t].astype(np.float64)
            nxt = starts[it][t + 1] if t + 1 < T else (starts[it + 1][0] if it + 1 < len(bufs) else last_starts)
            for i in np.nonzero(nxt)[0]:
                out.append((int(run_l[i]), float(run_r[i])))
                run_l[i], run_r[i] = 0, 0.0
    return out


def test_logger_keys_and_values_match_sb3(cuda_lib, golden_dir, tmp_path, monkeypatch):
    from mobrob_b200 import GpuVecEnv, ppo as ppo_mod

    n, T, B, E, iters, seed = 16, 64, 128, 3, 3, 7
    env = GpuVecEnv("point", n, seed=seed, time_limit=1000, terminate_on_goal=True)
    model = ppo_mod.PPO("MlpPolicy", env, n_steps=T, batch_size=B, n_epochs=E, seed=seed, gae_lambda=0.5, ent_coef=0.05,
                        verbose=0, permutation="sb3", tensorboard_log=str(tmp_path / "tensorboard"))
    w = dict(np.load(os.path.join(golden_dir, "point_policy.npz")))   # reaches goals: episodes end inside the rollouts
    model.policy.load_state_dict({k: torch.as_tensor(v) for k, v in w.items()})
    ref_pol = sb3_oracle.MlpPolicyOracle(14).load_numpy(w)
    opt = sb3_oracle.make_adam(ref_pol)

    dumps, perms, bufs = [], [], []
    orig_dump, orig_perm, orig_train = ppo_mod.Logger.dump, model._permutation, model.train

    def dump(self, step=0):
        dumps.append((step, dict(self.name_to_value)))
        orig_dump(self, step)

    def permutation(n_, epoch=0):
        p = orig_perm(n_, epoch)
        perms.append(p.cpu().numpy().copy())
        return p

    def train(perms_=None):
        torch.cuda.synchronize()
        bufs.append({k: v.cpu().numpy().copy() for k, v in model.buf.items()})
        return orig_train(perms_)

    monkeypatch.setattr(ppo_mod.Logger, "dump", dump)
    model._permutation, model.train = permutation, train
    model.learn(total_timesteps=iters * n * T)
    assert len(dumps) == iters and len(bufs) == iters and len(perms) == iters * E

    expect = []
    for it in range(iters):
        st = sb3_oracle.train_epochs(ref_pol, opt, bufs[it], E, B, perms=perms[E * it:E * (it + 1)], clip_range=0.2,
                                     ent_coef=0.05, vf_coef=0.5)
        y, p = bufs[it]["returns"].flatten(), bufs[it]["values"].flatten()
        expect.append({
            "train/entropy_loss": np.mean([s["entropy_loss"] for s in st]),
            "train/policy_gradient_loss": np.mean([s["policy_loss"] for s in st]),
            "train/value_loss": np.mean([s["value_loss"] for s in st]),
            "train/approx_kl": np.mean([s["approx_kl"] for s in st]),
            "train/clip_fraction": np.mean([s["clip_fraction"] for s in st]),
            "train/loss": st[-1]["loss"],
            "train/explained_variance": 1.0 - np.var(y - p) / np.var(y),
            "train/std": float(torch.exp(ref_pol.log_std.detach()).mean()),
            "train/n_updates": E * (it + 1), "train/clip_range": 0.2, "train/learning_rate": 3e-4})
    eps = _episodes_of(bufs, model._last_episode_starts.cpu().numpy())
    assert 3 <= len(eps) <= 100
    for k, (step, rec) in enumerate(dumps):
        assert step == (k + 1) * n * T
        for key in TIME_KEYS:
            assert key in rec, key
        assert rec["time/iterations"] == k + 1 and rec["time/total_timesteps"] == (k + 1) * n * T
        assert isinstance(rec["time/fps"], int) and rec["time/fps"] > 0 and isinstance(rec["time/time_elapsed"], int)
        if k == 0:
            assert not any(key.startswith("train/") for key in rec)   # SB3: nothing trained yet at the first dump
            continue
        for key in TRAIN_KEYS:
            assert key in rec, key
            tol = dict(rtol=2e-2, atol=2e-5) if key in ("train/approx_kl", "train/clip_fraction") else dict(rtol=3e-3, atol=1e-6)
            np.testing.assert_allclose(rec[key], expect[k - 1][key], err_msg=f"{key} at dump {k}", **tol)
    # Monitor's episode statistics: the last dump holds the mean over the newest 100 episodes finished so far, in
    # SB3's order -- here every one of them (< 100), those that ended on the final step of the final rollout included
    window = eps[-100:]
    got_l, got_r = dumps[-1][1]["rollout/ep_len_mean"], dumps[-1][1]["rollout/ep_rew_mean"]
    assert got_l == float(np.mean([l for l, _ in window])), (got_l, [l for l, _ in window])
    assert abs(got_r - np.mean([r for _, r in window])) < 1e-3   # buffer rewards are Monitor's rounded to float32
    # tensorboard: events under <tensorboard_log>/PPO_1 (the reference's tensorboard_log + SB3's run naming)
    run = tmp_path / "tensorboard" / "PPO_1"
    assert run.is_dir() and any(f.startswith("events.out.tfevents") for f in os.listdir(run))


def test_bench_configuration_learns(cuda_lib):
    """Point robot from scratch at the bench configuration (4096 envs x 296 steps, 10 epochs x 64
    minibatches of 18 944, device-side permutations): the policy learns to reach goals."""
    from mobrob_b200 import ppo as ppo_mod
    from mobrob_b200.rl_control.ppo import PPOCtrl

    n_envs, n_steps = 4096, 296
    ctrl = PPOCtrl(dict(policy="MlpPolicy", n_steps=n_steps, n_epochs=10, ent_coef=0.05, gae_lambda=0.5,
                        batch_size=18944, verbose=0, permutation="device"), "point", 1000, n_envs, seed=0,
                   tensorboard_log=False)
    curve = []
    orig = ppo_mod.Logger.dump

    def dump(self, step=0):
        curve.append(dict(self.name_to_value))
        orig(self, step)

    ppo_mod.Logger.dump = dump
    try:
        ctrl.learn(total_timesteps=LEARN_ITERS * n_envs * n_steps)
    finally:
        ppo_mod.Logger.dump = orig
    lens = [c.get("rollout/ep_len_mean") for c in curve if "rollout/ep_len_mean" in c]
    rews = [c.get("rollout/ep_rew_mean") for c in curve if "rollout/ep_rew_mean" in c]
    ev = [c["train/explained_variance"] for c in curve if "train/explained_variance" in c]
    std = [c["train/std"] for c in curve if "train/std" in c]
    # Monitor's window (the 100 newest episodes) starts with the lucky few that end inside the first rollouts;
    # once the 1000-step time-outs of the untrained policy arrive the mean climbs (~650 around iteration 9),
    # then collapses as the policy learns to drive to the goal (~190 from iteration ~20 on; the reference's own
    # run ends at 119 after 1e6 steps of 100-sample minibatches)
    early, late = max(lens[3:16]), float(np.mean(lens[-5:]))
    print(f"\nLEARNING point 4096 envs: ep_len_mean peak (iterations 4-16) {early:.1f} -> mean of the last five {late:.1f}; "
          f"ep_rew_mean min early {min(rews[3:16]):.2f} -> last {rews[-1]:.2f}; explained variance {ev[-1]:.3f}; "
          f"std {std[0]:.2f} -> {std[-1]:.2f} after {LEARN_ITERS} iterations ({LEARN_ITERS * n_envs * n_steps:.3g} env-steps)")
    assert early > 400.0 and late < LEARN_LEN_BOUND and late < 0.5 * early
    assert rews[-1] > 6.0 and min(rews[3:16]) < rews[-1] - 1.0
    assert ev[-1] > 0.5   # the value function explains the returns it is trained on
    assert std[-1] > 5.0 * std[0]   # exploration noise grows towards the shipped policies' bang-bang regime (sigma 20-140)


LEARN_ITERS = 40
LEARN_LEN_BOUND = 300.0
