"""Fused rollout + GAE + PPO update vs the oracle's collect_rollouts / PPO.train restatement."""
import os

import numpy as np
import pytest
import torch

from oracle import sb3_oracle
from rollout_oracle import setup as _setup, teacher_forced_check as _teacher_forced_check

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("pretrained,time_limit", [(True, 1000), (False, 40)])
def test_fused_rollout_matches_collect_rollouts(cuda_lib, golden_dir, pretrained, time_limit):
    n, T, seed = 24, 160, 5
    model, ref_pol, venv = _setup(golden_dir, n, T, seed, time_limit, pretrained, batch_size=64)
    if not pretrained:  # saturating exploration noise, like the shipped policies (log_std 3.0 / 3.6)
        sd = model.policy.state_dict()
        sd["log_std"].fill_(3.0)
        with torch.no_grad():
            ref_pol.log_std.fill_(3.0)
    obs_ref = venv.reset()
    first = np.ones(n, bool)
    g = torch.Generator().manual_seed(11)
    all_eps, total_trunc = [], 0
    for it in range(2):  # second rollout checks the carried-over state (_last_obs, episode starts)
        eps = torch.randn((T, n, 2), generator=g)
        model.collect_rollouts(eps.cuda().contiguous())
        torch.cuda.synchronize()
        obs_ref, first, n_trunc, eps_infos = _teacher_forced_check(model, ref_pol, venv, eps.numpy(), first, obs_ref)
        total_trunc += n_trunc
        all_eps += eps_infos
    model._drain_episodes()
    assert model._episode_num == len(all_eps) > 0
    if time_limit < 1000:
        assert total_trunc > 0, "no truncation happened: bootstrap untested"
    if len(all_eps) <= 100:
        got = sorted((e["l"], e["r"]) for e in model.ep_info_buffer)
        exp = sorted((l, round(r, 6)) for r, l in all_eps)
        assert [x[0] for x in got] == [x[0] for x in exp]
        np.testing.assert_allclose([x[1] for x in got], [x[1] for x in exp], rtol=1e-5, atol=1e-5)


def test_ppo_iteration_matches_sb3_arithmetic(cuda_lib, golden_dir):
    """One full learn() iteration: fused rollout + GAE on the device, then 3 epochs of minibatch
    Adam on the device vs SB3's PPO.train arithmetic (torch CPU) on the same rollout data and the
    same permutations: parameters agree to a small fraction of the update."""
    n, T, seed, B = 16, 64, 2, 128
    model, ref_pol, venv = _setup(golden_dir, n, T, seed, 60, False, batch_size=B, n_epochs=3)
    p0 = ref_pol.flat_params().clone().numpy()
    model.collect_rollouts()
    torch.cuda.synchronize()
    ref = {k: v.cpu().numpy() for k, v in model.buf.items()}
    opt = sb3_oracle.make_adam(ref_pol)
    rng = np.random.default_rng(0)
    perms = [rng.permutation(n * T).astype(np.int64) for _ in range(3)]
    stats = sb3_oracle.train_epochs(ref_pol, opt, ref, 3, B, perms=perms, clip_range=0.2, ent_coef=0.05,
                                    vf_coef=0.5)
    model.train(perms=perms)
    torch.cuda.synchronize()
    p_ref = ref_pol.flat_params().numpy()
    p = model.updater.params.cpu().numpy()
    moved = np.abs(p_ref - p0).max()
    assert moved > 5e-4
    assert np.abs(p - p_ref).max() < 2e-3 * moved + 1e-7
    tails, log = model._train_log
    np.testing.assert_allclose(tails[:, 1].cpu().numpy(), [s["value_loss"] for s in stats], rtol=1e-3)
    np.testing.assert_allclose(log[:, 0].cpu().numpy(), [s["grad_norm"] for s in stats], rtol=1e-3)
    # state_dict views share memory with the flat vector the kernels updated
    sd = model.policy.state_dict()
    np.testing.assert_array_equal(sd["log_std"].cpu().numpy(), p[:2])


def test_philox_rollout_is_deterministic_and_gaussian(cuda_lib, golden_dir):
    outs = []
    for _ in range(2):
        model, _, _ = _setup(golden_dir, 64, 128, 9, 1000, False, batch_size=64)
        model.collect_rollouts()
        torch.cuda.synchronize()
        outs.append({k: v.clone() for k, v in model.buf.items()})
        mu = torch.empty_like(model.buf["actions"]).view(-1, 2)
        obs = model.buf["obs"].view(-1, 14).contiguous()
        mu, _, _ = model.policy.forward_tensor(obs, None)
        z = (model.buf["actions"].view(-1, 2) - mu)  # log_std = 0 -> sigma = 1
        assert abs(float(z.mean())) < 0.03 and abs(float(z.std()) - 1.0) < 0.03
        assert abs(float((z[:, 0] * z[:, 1]).mean())) < 0.03
    for k in outs[0]:
        assert torch.equal(outs[0][k], outs[1][k]), k


def test_save_load_roundtrip_and_reference_zip(cuda_lib, golden_dir, tmp_path):
    from mobrob_b200.ppo import PPO

    ref = PPO.load(os.path.join(golden_dir, "policies", "point-ppo.zip"))
    assert ref.n_steps == 4000 and ref.batch_size == 100 and ref.gae_lambda == 0.5 and ref.ent_coef == 0.05
    assert int(ref.updater.step[0].item()) == 100000 and ref.updater.eps == 1e-5
    obs = np.load(os.path.join(golden_dir, "point_last_obs.npy"))
    a, _ = ref.predict(obs[0], deterministic=True)
    assert a.shape == (2,) and a.dtype == np.float32
    np.testing.assert_allclose(a, [-1.0, -0.75789261], rtol=1e-5)
    ref.observation_space, ref.action_space
    out = tmp_path / "again.zip"
    ref.save(str(out))
    again = PPO.load(str(out))
    for k, v in ref.policy.state_dict().items():
        assert torch.equal(v, again.policy.state_dict()[k])
    assert torch.equal(ref.updater.exp_avg_sq, again.updater.exp_avg_sq)
    import zipfile

    names = set(zipfile.ZipFile(out).namelist())
    assert {"data", "policy.pth", "policy.optimizer.pth", "pytorch_variables.pth",
            "_stable_baselines3_version", "system_info.txt"} <= names


def test_pretrained_point_policy_reaches_goals(cuda_lib, golden_dir):
    """BASELINE configs[1] as written: the shipped point policy, deterministic, over 16 384 seeded
    (init, goal) draws for 1000 steps -- examples/control.py:33-49 batched; success = goal reached within
    the 1000-step limit of being set.  CUDA vs oracle on the same seeds: success rates within 1 %
    (north_star), steps-to-goal within 1 %."""
    import sys

    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import eval_policy

    z = os.path.join(golden_dir, "policies", "point-ppo.zip")
    n = 16384
    g = eval_policy.evaluate_gpu(z, n, steps=1000)
    o = eval_policy.evaluate_oracle(z, n, steps=1000)
    print(f"\nCONFIG2 point 16384 goals x 1000 steps: first-goal success gpu {g['first_goal_success_rate']:.5f} "
          f"oracle {o['first_goal_success_rate']:.5f}; all goals gpu {g['all_goals_success_rate']:.5f} "
          f"({g['goals_reached']} reached, {g['timeouts']} timeouts) oracle {o['all_goals_success_rate']:.5f} "
          f"({o['goals_reached']} reached, {o['timeouts']} timeouts); mean steps to first goal gpu "
          f"{g['first_goal_mean_steps']:.2f} oracle {o['first_goal_mean_steps']:.2f}; "
          f"gpu {g['env_steps_per_s']:.3e} env-steps/s (unfused step + policy kernels)")
    assert abs(g["first_goal_success_rate"] - o["first_goal_success_rate"]) <= 0.01
    assert abs(g["all_goals_success_rate"] - o["all_goals_success_rate"]) <= 0.01
    assert o["first_goal_success_rate"] > 0.99
    assert abs(g["first_goal_mean_steps"] / o["first_goal_mean_steps"] - 1.0) <= 0.01
    assert abs(g["goals_reached"] / o["goals_reached"] - 1.0) <= 0.01
    # un-saturated deterministic actions are sensitive (DESIGN.md "Sensitivity"): single episodes may differ by a
    # few steps, the distribution does not
    assert (np.abs(g["first_len"] - o["first_len"]) <= 4).mean() > 0.99
    assert (g["first_len"] == o["first_len"]).mean() > 0.6


def test_unfused_rollout_equals_fused(cuda_lib, golden_dir):
    """mr_rollout (one launch) and mr_rollout_unfused (stand-alone kernels) are the same computation."""
    outs = []
    for mode in ("fused", "unfused"):
        model, _, _ = _setup(golden_dir, 40, 96, 4, 30, False, batch_size=64)
        model.policy.state_dict()["log_std"].fill_(2.0)
        model.rollout_mode = mode
        model.collect_rollouts()
        model.collect_rollouts()
        torch.cuda.synchronize()
        model._drain_episodes()
        outs.append(({k: v.clone() for k, v in model.buf.items()}, model._episode_num, model._last_obs.clone()))
    for k in outs[0][0]:
        assert torch.equal(outs[0][0][k], outs[1][0][k]), k
    assert outs[0][1] == outs[1][1] > 0
    assert torch.equal(outs[0][2], outs[1][2])


@pytest.mark.parametrize("n_steps,batch", [(64, 1024), (50, 1024)])
def test_single_launch_update_equals_per_epoch_launches(cuda_lib, monkeypatch, n_steps, batch):
    """PPO.train runs every epoch of the update in one cooperative launch when the rollout divides into whole
    minibatches (64 x 128 / 1024); the same update as one launch per epoch (forced by MR_EPOCH_LAUNCHES, and what a
    ragged last minibatch -- 50 x 128 = 6400 = 6 x 1024 + 256 -- takes anyway) moves the parameters identically
    up to the order in which the L2 adds the CTAs' partial gradients."""
    from mobrob_b200 import GpuVecEnv
    from mobrob_b200.ppo import PPO

    def run(per_epoch):
        if per_epoch:
            monkeypatch.setenv("MR_EPOCH_LAUNCHES", "1")
        else:
            monkeypatch.delenv("MR_EPOCH_LAUNCHES", raising=False)
        env = GpuVecEnv("point", 128, seed=3, time_limit=100, terminate_on_goal=True)
        model = PPO("MlpPolicy", env, n_steps=n_steps, batch_size=batch, n_epochs=4, seed=3, gae_lambda=0.5, ent_coef=0.05)
        start = model.updater.params.clone()
        model.learn(total_timesteps=128 * n_steps)   # one iteration: the same rollout on both sides
        torch.cuda.synchronize()
        return start, model.updater.params.clone(), model.updater.exp_avg_sq.clone(), int(model.updater.step.flatten()[0].item()), model._log.clone()

    s0, p0, v0, k0, log0 = run(False)
    s1, p1, v1, k1, log1 = run(True)
    assert torch.equal(s0, s1)
    n_mb = -(-128 * n_steps // batch)
    assert k0 == k1 == 4 * n_mb
    moved = float((p0 - s0).abs().max())
    assert moved > 5e-4
    assert float((p0 - p1).abs().max()) <= 2e-5 * moved + 1e-7
    torch.testing.assert_close(v0, v1, rtol=1e-3, atol=1e-12)
    torch.testing.assert_close(log0, log1, rtol=1e-3, atol=1e-6)   # per-minibatch norm, clip coefficient, step, losses
