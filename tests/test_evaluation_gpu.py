"""evaluate_policy's device path (mr_evaluate) against SB3's loop run step by step through model.predict and the VecEnv
protocol, its stochastic draws against the training rollouts', its step bound, and EvalCallback inside PPO.learn."""
import os
from collections import Counter

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ALL_KEYS = {"observe_goal_dist": True, "observe_qpos": True, "observe_qvel": True, "observe_ctrl": True}


def _noop(locals_, globals_):
    """A per-step callback: evaluate_policy then takes SB3's loop on the host."""


def _envs(name, n, seed, time_limit, robot_config=None):
    from mobrob_b200 import GpuVecEnv

    return [GpuVecEnv(name, n, seed=seed, time_limit=time_limit, terminate_on_goal=True, robot_config=robot_config)
            for _ in range(2)]


def _assert_same_env(a, b):
    assert torch.equal(a.get_state(), b.get_state())
    assert torch.equal(a.get_obs_tensor(), b.get_obs_tensor())
    assert torch.equal(a.get_reset_counts(), b.get_reset_counts())


def _check_against_loop(model, name, n, time_limit, n_eval, robot_config=None, seed=3):
    from mobrob_b200 import evaluate_policy
    from mobrob_b200.evaluation import evaluate_policy as ep2

    assert ep2 is evaluate_policy
    dev_env, loop_env = _envs(name, n, seed, time_limit, robot_config)
    for _ in range(2):   # the second evaluation starts from the first one's lazy reset
        got = evaluate_policy(model, dev_env, n_eval, deterministic=True, return_episode_rewards=True)
        exp = evaluate_policy(model, loop_env, n_eval, deterministic=True, return_episode_rewards=True, callback=_noop)
        assert len(exp[0]) == n_eval
        assert got[1] == exp[1]
        assert got[0] == exp[0]
        _assert_same_env(dev_env, loop_env)
    assert dev_env.eval_steps > 0


def test_point_fused_equals_sb3_loop(cuda_lib, golden_dir):
    from mobrob_b200.ppo import PPO

    model = PPO.load(os.path.join(golden_dir, "policies", "point-ppo.zip"))
    _check_against_loop(model, "point", 96, 200, 250)


def test_car_per_step_equals_sb3_loop(cuda_lib, golden_dir):
    from mobrob_b200.ppo import PPO

    model = PPO.load(os.path.join(golden_dir, "policies", "car-ppo.zip"))
    _check_against_loop(model, "car", 16, 50, 37)


def test_point_optional_keys_per_step_equals_sb3_loop(cuda_lib):
    from mobrob_b200 import GpuVecEnv
    from mobrob_b200.ppo import PPO

    model = PPO("MlpPolicy", GpuVecEnv("point", 8, seed=1, time_limit=30, robot_config=ALL_KEYS), n_steps=8, seed=1)
    assert model.policy.obs_dim == 23
    _check_against_loop(model, "point", 24, 30, 61, robot_config=ALL_KEYS)


def _episodes_of_rollout(model):
    model._drain_episodes()
    count = int(model.ep_count.item())
    r, l = model.ep_r[:count].cpu().numpy(), model.ep_l[:count].cpu().numpy()
    return Counter((round(float(a), 6), int(b)) for a, b in zip(r, l))


@pytest.mark.parametrize("name,n,time_limit,n_eval", [("point", 64, 40, 128), ("car", 16, 30, 24)])
def test_stochastic_draws_match_training_rollout(cuda_lib, name, n, time_limit, n_eval):
    """The first stochastic evaluation on a fresh env draws what collect_rollouts draws on an identically seeded env:
    over the steps the evaluation took, every episode it records is one the rollout finished."""
    from mobrob_b200 import GpuVecEnv, evaluate_policy
    from mobrob_b200.ppo import PPO

    seed = 7
    model = PPO("MlpPolicy", GpuVecEnv(name, n, seed=seed, time_limit=time_limit), n_steps=8, seed=seed)
    eval_env, twin = _envs(name, n, seed, time_limit)
    rew, lens = evaluate_policy(model, eval_env, n_eval, deterministic=False, return_episode_rewards=True)
    S = eval_env.eval_steps
    assert len(rew) == n_eval and 0 < S <= 2 * time_limit
    roll = PPO("MlpPolicy", GpuVecEnv(name, n, seed=seed, time_limit=time_limit), n_steps=S, seed=seed)
    roll.policy.load_state_dict(model.policy.state_dict())
    roll.collect_rollouts()
    got = Counter((r, l) for r, l in zip(rew, lens))
    rolled = _episodes_of_rollout(roll)
    assert not (got - rolled), "evaluation episodes the rollout did not produce"
    # a second call continues the Philox counters: with the counter wound back it would act differently
    second = evaluate_policy(model, eval_env, n_eval, deterministic=False, return_episode_rewards=True)
    evaluate_policy(model, twin, n_eval, deterministic=False, return_episode_rewards=True)
    assert twin.eval_steps == S
    twin.eval_steps = 0
    replay = evaluate_policy(model, twin, n_eval, deterministic=False, return_episode_rewards=True)
    assert replay != second


@pytest.mark.parametrize("name,zip_name,n,max_steps", [("point", "point-ppo.zip", 32, 25), ("car", "car-ppo.zip", 8, 12)])
def test_max_steps_without_time_limit(cuda_lib, golden_dir, name, zip_name, n, max_steps):
    from mobrob_b200 import evaluate_policy
    from mobrob_b200.ppo import PPO

    model = PPO.load(os.path.join(golden_dir, "policies", zip_name))
    dev_env, loop_env = _envs(name, n, 5, None)
    with pytest.raises(ValueError, match="max_steps"):
        evaluate_policy(model, dev_env, 4 * n)
    with pytest.raises(RuntimeError, match="max_steps"):
        evaluate_policy(model, dev_env, 4 * n, max_steps=max_steps)
    with pytest.raises(RuntimeError, match="max_steps"):
        evaluate_policy(model, loop_env, 4 * n, max_steps=max_steps, callback=_noop)
    assert dev_env.eval_steps == max_steps
    _assert_same_env(dev_env, loop_env)


def test_eval_callback_in_learn(cuda_lib, tmp_path):
    from mobrob_b200 import GpuVecEnv, evaluate_policy
    from mobrob_b200.callbacks import CheckpointCallback, EvalCallback, StopTrainingOnRewardThreshold
    from mobrob_b200.ppo import PPO

    n, T = 256, 32

    def eval_env():
        return GpuVecEnv("point", 64, seed=11, time_limit=60)

    model = PPO("MlpPolicy", GpuVecEnv("point", n, seed=0, time_limit=100), n_steps=T, batch_size=1024, n_epochs=2,
                seed=0)
    ckpt = CheckpointCallback(save_freq=20, save_path=str(tmp_path / "ckpt"))
    ev = EvalCallback(eval_env(), n_eval_episodes=100, eval_freq=20, log_path=str(tmp_path / "logs"),
                      best_model_save_path=str(tmp_path / "best"))
    model.learn(total_timesteps=3 * n * T, callback=[ckpt, ev])   # a list is wrapped in CallbackList
    z = np.load(tmp_path / "logs" / "evaluations.npz")
    assert list(z["timesteps"]) == [20 * n, 40 * n, 60 * n, 80 * n]
    assert z["results"].shape == (4, 100) and z["ep_lengths"].shape == (4, 100)
    # the first evaluation ran on the first rollout's parameters, which the checkpoint of that step holds
    first = PPO.load(str(tmp_path / "ckpt" / f"rl_model_{20 * n}_steps.zip"))
    rew, lens = evaluate_policy(first, eval_env(), 100, return_episode_rewards=True)
    assert rew == z["results"][0].tolist() and lens == z["ep_lengths"][0].tolist()
    best = PPO.load(str(tmp_path / "best" / "best_model.zip"))
    assert best.policy.obs_dim == 14
    assert ev.best_mean_reward == max(np.mean(r) for r in z["results"])

    # a new best above the threshold stops learn() at the first evaluation, before that rollout is trained on
    model = PPO("MlpPolicy", GpuVecEnv("point", n, seed=0, time_limit=100), n_steps=T, batch_size=1024, n_epochs=2,
                seed=0)
    start = model.updater.params.clone()
    ev = EvalCallback(eval_env(), callback_on_new_best=StopTrainingOnRewardThreshold(-1e9), n_eval_episodes=16,
                      eval_freq=20, verbose=0)
    model.learn(total_timesteps=3 * n * T, callback=ev)
    assert len(ev.evaluations_timesteps) == 0 and ev.n_calls == 20
    assert model._train_count == 0 and model.num_timesteps == n * T
    assert torch.equal(model.updater.params, start)
