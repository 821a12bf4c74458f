"""The rollout kernels in the configuration training runs: device Philox noise (eps=None), ragged env counts, sharded
env offsets, the MR_ROLLOUT_CFG tuning variants, and Monitor's episode window in SB3's order.

References: tests/rollout_oracle.py restates the device noise (pinned by tests/test_rollout_noise_cpu.py) and replays
a rollout through the oracle's policy and environment.
"""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest
import torch

from oracle import point_oracle as po
from oracle.vec_oracle import GoalVecOracle
from rollout_oracle import device_draws, rollout_draws, setup, teacher_forced_check

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEEDS = [0, 5, 2**32 + 9]


def _zero_mean_unit_sigma(model):
    """action_net = 0, log_std = 0: mu = +0 and sigma = 1 exactly, so the kernels store a = 0 + 1 * z = z."""
    sd = model.policy.state_dict()
    with torch.no_grad():
        sd["action_net.weight"].zero_()
        sd["action_net.bias"].zero_()
        sd["log_std"].zero_()


def _assert_draws(actions, z, what):
    a = actions.reshape(z.shape)
    tol = 4 * np.spacing(np.abs(z).astype(np.float32))
    bad = np.abs(a - z) > tol
    assert not bad.any(), f"{what}: {int(bad.sum())} of {bad.size} draws differ, e.g. {a[bad][:4]} vs {z[bad][:4]}"


def _assert_logp(actions, logp):
    a = actions.astype(np.float64)
    ref = -0.5 * (a ** 2).sum(axis=-1) - np.log(2 * np.pi)
    np.testing.assert_allclose(logp, ref, rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("mode", ["fused", "unfused"])
@pytest.mark.parametrize("seed", SEEDS)
def test_device_draws_are_the_restated_philox(cuda_lib, golden_dir, mode, seed):
    n, T = 37, 19
    model, _, _ = setup(golden_dir, n, T, 1, 12, False, batch_size=64)
    model.seed = seed   # set_random_seed takes seeds below 2^32 (np.random.seed); the noise key has 64 bits
    model.rollout_mode = mode
    _zero_mean_unit_sigma(model)
    for k in range(2):   # the second rollout's counters continue at n_steps
        model.collect_rollouts()
        torch.cuda.synchronize()
        act = model.buf["actions"].cpu().numpy()
        _assert_draws(act, rollout_draws(model, k), f"{mode} seed {seed} rollout {k}")
        _assert_logp(act, model.buf["log_probs"].cpu().numpy())


@pytest.mark.parametrize("fused", [True, False])
def test_draws_across_the_32_bit_word_of_the_env_id(cuda_lib, golden_dir, fused):
    """mr_rollout / mr_rollout_unfused called through the C ABI with env_offset = 2^32 - 2 and N = 5: global env ids
    2^32 - 2 .. 2^32 + 2 and step counters 2^32 - 1 .. 2^32 + 1 cross the counter's 32-bit words."""
    from mobrob_b200 import _lib
    from mobrob_b200.ppo import EP_RING

    n, T, seed = 5, 3, 5
    env_offset, noise_offset = 2**32 - 2, 2**32 - 1
    model, _, _ = setup(golden_dir, n, T, seed, 12, False, batch_size=64)
    _zero_mean_unit_sigma(model)
    b, env = model.buf, model.env
    last_obs = env.reset_tensor().clone()
    starts = torch.ones(n, dtype=torch.float32, device=model.device)
    fn = model.lib.mr_rollout if fused else model.lib.mr_rollout_unfused
    _lib.check(fn(env._h, model.updater.params.data_ptr(), T, last_obs.data_ptr(), starts.data_ptr(),
                  b["obs"].data_ptr(), b["actions"].data_ptr(), b["rewards"].data_ptr(), b["episode_starts"].data_ptr(),
                  b["values"].data_ptr(), b["log_probs"].data_ptr(), model.last_val.data_ptr(),
                  model.last_done.data_ptr(), None, seed, noise_offset, env_offset, 0.99, model.ep_ret_tn.data_ptr(),
                  model.ep_len_tn.data_ptr(), model.ep_steps.data_ptr(), model.ep_r.data_ptr(), model.ep_l.data_ptr(),
                  model.ep_count.data_ptr(), EP_RING, model._stream()))
    torch.cuda.synchronize()
    act = b["actions"].cpu().numpy()
    _assert_draws(act, device_draws(seed, n, T, noise_offset, env_offset), "C ABI")
    _assert_logp(act, b["log_probs"].cpu().numpy())


# (N, T, time_limit): a lone env, a partial warp, a partial last state tile past one and two 128-env tiles; T = 37
# with a time limit of 7 (whole warps and both sides of a tile boundary time out together, goal-reaching envs
# drift out of step), and T = 1 with a time limit of 1 (every env times out at every step)
RAGGED = [(1, 37, 7), (3, 37, 7), (130, 37, 7), (257, 37, 7), (1, 1, 1), (3, 1, 1), (130, 1, 1), (257, 1, 1)]


@pytest.mark.parametrize("mode", ["fused", "unfused"])
@pytest.mark.parametrize("gamma", [0.99, 0.9])
@pytest.mark.parametrize("n,T,time_limit", RAGGED)
def test_philox_rollout_matches_oracle_at_ragged_shapes(cuda_lib, golden_dir, n, T, time_limit, gamma, mode):
    seed = 6
    model, ref_pol, venv = setup(golden_dir, n, T, seed, time_limit, False, batch_size=64, gamma=gamma)
    model.rollout_mode = mode
    sd = model.policy.state_dict()
    with torch.no_grad():   # wider exploration: some goals are reached and those envs leave the common clock
        sd["log_std"].fill_(1.0)
        ref_pol.log_std.fill_(1.0)
    obs_ref = venv.reset()
    first = np.ones(n, bool)
    total_trunc = 0
    for k in range(2):
        model.collect_rollouts()   # eps=None: the production path
        torch.cuda.synchronize()
        obs_ref, first, n_trunc, _ = teacher_forced_check(model, ref_pol, venv, rollout_draws(model, k), first,
                                                          obs_ref, gamma=gamma)
        total_trunc += n_trunc
    assert total_trunc > 0, "no time-out: the bootstrap went untested"


def _state(model):
    out = {k: v.clone() for k, v in model.buf.items()}
    out.update(last_val=model.last_val.clone(), last_done=model.last_done.clone(), last_obs=model._last_obs.clone(),
               last_starts=model._last_episode_starts.clone())
    return out


def _rollouts(env_name, n, first_rank, mode, seed, T, time_limit, k=2):
    from mobrob_b200 import GpuVecEnv
    from mobrob_b200.ppo import PPO

    env = GpuVecEnv(env_name, n, seed=None, time_limit=time_limit, terminate_on_goal=True, first_rank=first_rank)
    model = PPO("MlpPolicy", env, n_steps=T, batch_size=64, seed=seed, gae_lambda=0.5)
    model.rollout_mode = mode
    model.policy.state_dict()["log_std"].fill_(1.0)
    out = []
    for _ in range(k):
        model.collect_rollouts()
        torch.cuda.synchronize()
        out.append(_state(model))
    return out


@pytest.mark.parametrize("env_name,mode,n,n1,T,time_limit", [
    ("point", "fused", 300, 131, 29, 11),
    ("point", "unfused", 300, 131, 29, 11),
    ("car", "unfused", 21, 8, 12, 7),
])
def test_rollout_does_not_depend_on_the_sharding(cuda_lib, env_name, mode, n, n1, T, time_limit):
    """DESIGN section 7: noise and env streams are keyed by the global env id, so one handle of N envs and two handles
    that split them with first_rank compute the same rollout, column for column, bit for bit."""
    seed = 13
    whole = _rollouts(env_name, n, 0, mode, seed, T, time_limit)
    lo = _rollouts(env_name, n1, 0, mode, seed, T, time_limit)
    hi = _rollouts(env_name, n - n1, n1, mode, seed, T, time_limit)
    for k in range(2):
        for key, full in whole[k].items():
            dim = 1 if key in ("obs", "actions", "rewards", "episode_starts", "values", "log_probs", "advantages",
                               "returns") else 0
            a, b = full.split([n1, n - n1], dim=dim)
            assert torch.equal(a, lo[k][key]), f"rollout {k} {key}: envs 0 .. {n1 - 1}"
            assert torch.equal(b, hi[k][key]), f"rollout {k} {key}: envs {n1} .. {n - 1}"
        assert bool(whole[k]["episode_starts"].any()), "no episode ended: the reset streams went untested"


_VARIANT_SCRIPT = textwrap.dedent("""
    import sys
    import numpy as np
    import torch
    sys.path.insert(0, {root!r})
    from mobrob_b200 import GpuVecEnv
    from mobrob_b200.ppo import PPO
    env = GpuVecEnv("point", 257, seed=None, time_limit=7, terminate_on_goal=True)
    model = PPO("MlpPolicy", env, n_steps=37, batch_size=64, seed=8, gae_lambda=0.5)
    model.policy.state_dict()["log_std"].fill_(1.0)
    out = {{}}
    for k in range(2):
        model.collect_rollouts()
        torch.cuda.synchronize()
        for key, v in model.buf.items():
            out[f"{{key}}_{{k}}"] = v.cpu().numpy()
        out[f"last_val_{{k}}"] = model.last_val.cpu().numpy()
        out[f"last_done_{{k}}"] = model.last_done.cpu().numpy()
        out[f"last_obs_{{k}}"] = model._last_obs.cpu().numpy()
    model._drain_episodes()
    out["ep_r"] = np.array([e["r"] for e in model.ep_info_buffer])
    out["ep_l"] = np.array([e["l"] for e in model.ep_info_buffer])
    np.savez({path!r}, **out)
""")


def test_rollout_tuning_variants_are_bit_identical(cuda_lib, tmp_path):
    """MR_ROLLOUT_CFG = 4x8 | 8x4 | 14x4 launch other instantiations of the fused kernel (4x8 maps 8 envs to a warp:
    24 live lanes in the sample and bootstrap code).  launch_rollout caches its choice per process, hence one
    subprocess per variant."""
    runs = {}
    for cfg in ("default", "4x8", "8x4", "14x4"):
        path = str(tmp_path / f"{cfg}.npz")
        env = dict(os.environ)
        env.pop("MR_ROLLOUT_CFG", None)
        if cfg != "default":
            env["MR_ROLLOUT_CFG"] = cfg
        r = subprocess.run([sys.executable, "-c", _VARIANT_SCRIPT.format(root=ROOT, path=path)], env=env, cwd=ROOT,
                           capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        runs[cfg] = dict(np.load(path))
    base = runs.pop("default")
    assert base["rewards_1"].shape == (37, 257) and base["episode_starts_0"].any() and len(base["ep_l"]) > 0
    for cfg, got in runs.items():
        assert sorted(got) == sorted(base)
        for key in base:
            np.testing.assert_array_equal(got[key], base[key], err_msg=f"MR_ROLLOUT_CFG={cfg}: {key}")


@pytest.mark.parametrize("mode", ["fused", "unfused"])
@pytest.mark.parametrize("window", [7, 100, 250])
def test_monitor_window_is_sb3s(cuda_lib, monkeypatch, mode, window):
    """learn() with far more episodes per rollout than the window holds: at every dump, ep_info_buffer is the newest
    `window` episodes in SB3's order (by step, then env index) and rollout/ep_*_mean are their means.  192 envs with a
    time limit of 10 and 4-step rollouts: a tile and a half of envs time out at the same step (rollouts 3 and 5),
    and a window of 250 then spans two rollouts."""
    from mobrob_b200 import GpuVecEnv, ppo as ppo_mod

    n, T, time_limit, iters, seed = 192, 4, 10, 6, 11
    env = GpuVecEnv("point", n, seed=None, time_limit=time_limit, terminate_on_goal=True)
    model = ppo_mod.PPO("MlpPolicy", env, n_steps=T, batch_size=256, n_epochs=1, seed=seed, gae_lambda=0.5,
                        stats_window_size=window)
    model.rollout_mode = mode
    model.policy.state_dict()["log_std"].fill_(1.0)
    actions, dumps = [], []
    orig_train, orig_dump = model.train, ppo_mod.Logger.dump

    def train(perms=None):
        torch.cuda.synchronize()
        actions.append(model.buf["actions"].cpu().numpy().copy())
        return orig_train(perms)

    def dump(self, step=0):
        dumps.append((dict(self.name_to_value), [dict(e) for e in model.ep_info_buffer], model._episode_num))
        orig_dump(self, step)

    model.train = train
    monkeypatch.setattr(ppo_mod.Logger, "dump", dump)
    model.learn(total_timesteps=iters * n * T)
    assert len(actions) == iters and len(dumps) == iters

    # SB3's order: DummyVecEnv steps the envs in index order, collect_rollouts appends each step's episodes
    venv = GoalVecOracle(po.PointBody(n), seed=seed, time_limit=time_limit, terminate_on_goal=True)
    venv.reset()
    episodes, upto, rollout_of = [], [], []
    for it, act in enumerate(actions):
        for t in range(T):
            _, _, done, info = venv.step(np.clip(act[t], -1.0, 1.0))
            for i in np.nonzero(done)[0]:
                episodes.append((float(info["ep_r"][i]), int(info["ep_l"][i])))
                rollout_of.append(it)
        upto.append(len(episodes))
    assert max(np.diff([0] + upto)) > window or window == 250, "the window never overflowed within one rollout"
    spans = False
    for k, (rec, buf, episode_num) in enumerate(dumps):
        exp = episodes[:upto[k]][-window:]
        assert episode_num == upto[k], f"dump {k}: _episode_num"
        assert [e["l"] for e in buf] == [l for _, l in exp], f"dump {k}: episode lengths / order"
        np.testing.assert_allclose([e["r"] for e in buf], [round(r, 6) for r, _ in exp], rtol=1e-5, atol=1e-5,
                                   err_msg=f"dump {k}: episode returns / order")
        if exp:
            assert rec["rollout/ep_len_mean"] == float(np.mean([e["l"] for e in buf]))
            np.testing.assert_allclose(rec["rollout/ep_len_mean"], np.mean([l for _, l in exp]), rtol=1e-12)
            np.testing.assert_allclose(rec["rollout/ep_rew_mean"], np.mean([r for r, _ in exp]), rtol=1e-5, atol=1e-5)
            spans |= len({rollout_of[i] for i in range(upto[k] - len(exp), upto[k])}) > 1
        else:
            assert "rollout/ep_len_mean" not in rec
    if window == 250:
        assert spans, "no window spanned two rollouts"
