"""observe_goal_lidar on the device: the goal_lidar block of the CUDA envs against the pseudo-lidar restatement
(tests/goal_lidar_oracle.py) on the kernels' own state and along oracle trajectories, every other column unchanged,
the batch-of-one wrapper, PPO, evaluate_policy and the car's refusal in PPO."""
import numpy as np
import pytest
import torch

import goal_lidar_oracle as L
from oracle import car_oracle as co, point_oracle as po

pytestmark = pytest.mark.gpu

KEYS = ("observe_goal_dist", "observe_qpos", "observe_qvel", "observe_ctrl")
PRE = {"point": 3, "car": 15}
BASE = {"point": 14, "car": 26}
GOAL = {"point": slice(11, 13), "car": slice(26, 28)}   # goal xy in mr_env_get_state's reference view
SETTINGS = [{}, {"lidar_num_bins": 16, "lidar_max_dist": 1.5, "lidar_alias": False},
            {"lidar_num_bins": 2, "lidar_exp_gain": 0.4}, {"lidar_num_bins": 1}, {"lidar_num_bins": 3, "lidar_max_dist": 3.0}]


def _oracle_kw(settings):
    return {k[6:]: v for k, v in settings.items()}   # lidar_num_bins -> num_bins ...


def _bins(settings):
    return settings.get("lidar_num_bins", 10)


def _at(kind, cfg):
    """First column of the goal_lidar block: after accelerometer [ball sensors] | ctrl | goal_compass | goal_dist."""
    return PRE[kind] + 2 + (2 if cfg.get("observe_ctrl") else 0) + (1 if cfg.get("observe_goal_dist") else 0)


def _oracle_block(env, settings):
    st = env.get_state().cpu().numpy()
    return L.lidar_rows(st[:, GOAL[env.env_name]], *L.robot_frames_of_state(env.env_name, st),
                        **_oracle_kw(settings)).astype(np.float32)


def _close(got, want, msg=""):
    np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-7, err_msg=msg)


@pytest.mark.parametrize("settings", SETTINGS, ids=lambda s: "-".join(f"{k[6:]}={v}" for k, v in s.items()) or "default")
@pytest.mark.parametrize("kind", ["point", "car"])
def test_block_matches_oracle_on_the_kernels_state(cuda_lib, kind, settings):
    """Reset, get_obs, every step's row (post-reset where done) and every terminal observation: the block equals the
    restatement evaluated on the state the kernels export, so no dynamics drift enters.  Start and goal boxes are
    narrowed so that goal-only resets (goal reached) happen next to the full ones (time limit)."""
    from mobrob_b200 import GpuVecEnv
    from mobrob_b200.spaces import Box

    n, tl, T = (48, 25, 120) if kind == "point" else (12, 15, 40)
    cfg = {"observe_goal_lidar": True, **settings}
    env = GpuVecEnv(kind, n, seed=4, time_limit=tl, terminate_on_goal=True, robot_config=cfg)
    # the same kernels without resets: stepped from env's state, its rows are env's terminal observations
    twin = GpuVecEnv(kind, n, seed=4, time_limit=None, terminate_on_goal=False, robot_config=cfg)
    env.reset_init_space(Box(np.full(2, -0.3, np.float32), np.full(2, 0.3, np.float32), dtype=np.float32))
    env.reset_goal_space(Box(np.full(2, -0.5, np.float32), np.full(2, 0.5, np.float32), dtype=np.float32))
    bins, at = _bins(settings), _at(kind, cfg)
    assert env.obs_dim == BASE[kind] + bins
    obs = env.reset()
    _close(obs[:, at:at + bins], _oracle_block(env, settings), "reset")
    _close(env.get_obs_tensor().cpu().numpy()[:, at:at + bins], _oracle_block(env, settings), "get_obs")
    rng = np.random.default_rng(2)
    n_term = 0
    for t in range(T):
        if t == T // 2:   # a VecEnv.reset() in mid-run: goal-only where reached, full elsewhere
            obs = env.reset()
            _close(obs[:, at:at + bins], _oracle_block(env, settings), "mid-run reset")
        a = rng.uniform(-1.5, 1.5, (n, 2)).astype(np.float32)
        twin.set_state(env.get_state())
        obs, rew, done, infos = env.step(a)
        _close(obs[:, at:at + bins], _oracle_block(env, settings), f"step {t}")
        t_obs, *_ = twin.step(a)
        _close(t_obs[:, at:at + bins], _oracle_block(twin, settings), f"step {t}, pre-reset state")
        for i in np.nonzero(done)[0]:
            n_term += 1
            _close(infos[i]["terminal_observation"][at:at + bins], t_obs[i, at:at + bins], f"terminal obs, step {t}")
    counts = env.get_reset_counts().cpu().numpy()
    assert n_term > 0
    assert (counts[:, 0] - counts[:, 1]).sum() > 0, "no goal-only reset"
    assert (counts[:, 1] > 1).sum() > 0, "no full reset after the first"


def _parity(kind, cfg, lidar, n, seed, tl, T, tol, atol):
    from mobrob_b200 import GpuVecEnv

    body = po.PointBody(n) if kind == "point" else co.CarBody(n)
    ora = L.LidarVecOracle(body, lidar=_oracle_kw(lidar), seed=seed, time_limit=tl, terminate_on_goal=True,
                           observe=cfg)
    gpu = GpuVecEnv(kind, n, seed=seed, time_limit=tl, terminate_on_goal=True, robot_config={**cfg, **lidar})
    o_ref, o_gpu = ora.reset(), gpu.reset()
    assert o_gpu.shape == o_ref.shape
    np.testing.assert_allclose(o_gpu, o_ref, rtol=tol, atol=atol)
    rng = np.random.default_rng(9)
    n_term = 0
    for t in range(T):
        a = (np.sign(rng.standard_normal((n, 2))) * rng.choice([0.4, 1.0, 1.7], (n, 2))).astype(np.float32)
        o_ref, r_ref, d_ref, info = ora.step(a)
        o_gpu, r_gpu, d_gpu, infos = gpu.step(a)
        np.testing.assert_array_equal(d_gpu, d_ref)
        np.testing.assert_allclose(o_gpu, o_ref, rtol=tol, atol=atol, err_msg=f"obs step {t}")
        np.testing.assert_allclose(r_gpu, r_ref, rtol=tol, atol=max(1e-7, atol / 10))
        for i in np.nonzero(d_ref)[0]:
            n_term += 1
            np.testing.assert_allclose(infos[i]["terminal_observation"], info["terminal_obs"][i], rtol=tol, atol=atol)
    assert n_term >= n


@pytest.mark.parametrize("cfg,lidar", [({"observe_goal_lidar": True}, {}),
                                       ({"observe_goal_lidar": True, **{k: True for k in KEYS}}, {"lidar_num_bins": 17}),
                                       ({"observe_goal_lidar": True, "observe_goal_dist": True},
                                        {"lidar_num_bins": 6, "lidar_max_dist": 2.0, "lidar_exp_gain": 0.3})],
                         ids=["lidar", "all-keys-17-bins", "goal-dist-max-dist"])
def test_point_trajectory_matches_oracle(cuda_lib, cfg, lidar):
    _parity("point", cfg, lidar, n=48, seed=3, tl=40, T=200, tol=1e-5, atol=1e-6)


def test_car_trajectory_matches_oracle(cuda_lib):
    _parity("car", {"observe_goal_lidar": True, **{k: True for k in KEYS}}, {}, n=10, seed=2, tl=20, T=45,
            tol=1e-4, atol=1e-4)   # contacts: test_car_gpu's bound


@pytest.mark.parametrize("others", [False, True], ids=["lidar-only", "with-four-keys"])
@pytest.mark.parametrize("kind", ["point", "car"])
def test_every_other_column_is_unchanged(cuda_lib, kind, others):
    """The same seed without the lidar: every column outside the block, rewards, flags and terminal rows bit-identical."""
    from mobrob_b200 import GpuVecEnv

    n, tl, T = (64, 30, 100) if kind == "point" else (12, 15, 35)
    cfg = {k: True for k in KEYS} if others else {}
    lid = GpuVecEnv(kind, n, seed=6, time_limit=tl, robot_config={**cfg, "observe_goal_lidar": True, "lidar_num_bins": 7})
    ref = GpuVecEnv(kind, n, seed=6, time_limit=tl, robot_config=cfg or None)
    at = _at(kind, cfg)
    cut = lambda o: np.delete(o, np.s_[at:at + 7], axis=-1)  # noqa: E731
    assert lid.obs_dim == ref.obs_dim + 7
    np.testing.assert_array_equal(cut(lid.reset()), ref.reset())
    rng = np.random.default_rng(1)
    n_done = 0
    for t in range(T):
        a = rng.uniform(-1.5, 1.5, (n, 2)).astype(np.float32)
        o_l, r_l, d_l, i_l = lid.step(a)
        o_r, r_r, d_r, i_r = ref.step(a)
        np.testing.assert_array_equal(cut(o_l), o_r, err_msg=f"step {t}")
        np.testing.assert_array_equal(r_l, r_r)
        np.testing.assert_array_equal(d_l, d_r)
        for i in np.nonzero(d_r)[0]:
            n_done += 1
            np.testing.assert_array_equal(cut(i_l[i]["terminal_observation"]), i_r[i]["terminal_observation"])
            assert i_l[i]["episode"]["r"] == i_r[i]["episode"]["r"] and i_l[i]["episode"]["l"] == i_r[i]["episode"]["l"]
    assert n_done > 0
    np.testing.assert_array_equal(cut(lid.get_obs_tensor().cpu().numpy()), ref.get_obs_tensor().cpu().numpy())
    assert torch.equal(lid.get_state(), ref.get_state())


@pytest.mark.parametrize("kind", ["point", "car"])
def test_wrapper_subclass_switches_the_lidar_through_get_robot_config(cuda_lib, kind):
    """As in the reference: a MujocoGoalEnv subclass overrides get_robot_config (wrapper.py:235-240)."""
    from mobrob_b200.envs.wrapper import CarEnv, PointEnv

    class WithLidar(PointEnv if kind == "point" else CarEnv):
        def get_robot_config(self):
            return {**super().get_robot_config(), "observe_goal_lidar": True, "lidar_num_bins": 8,
                    "lidar_max_dist": 3.0}

    env = WithLidar(terminate_on_goal=False)
    assert env.observation_space.shape == (BASE[kind] + 8,)
    env.seed(3)
    obs, _ = env.reset()
    at = PRE[kind] + 2
    settings = {"lidar_num_bins": 8, "lidar_max_dist": 3.0}
    _close(obs[at:at + 8], _oracle_block(env.env, settings)[0])
    assert np.count_nonzero(obs[at:at + 8]) >= 1
    for _ in range(5):
        obs, *_ = env.step(np.array([1.0, 0.3], np.float32))
    assert obs.shape == (BASE[kind] + 8,)
    _close(obs[at:at + 8], _oracle_block(env.env, settings)[0])

    class Natural(PointEnv):
        def get_robot_config(self):
            return {**super().get_robot_config(), "observe_goal_lidar": True, "lidar_type": "natural"}

    with pytest.raises(NotImplementedError, match="natural"):
        Natural()


@pytest.mark.parametrize("bins", [10, 17], ids=["24-floats", "31-floats"])
def test_ppo_learns_on_the_lidar_row(cuda_lib, tmp_path, bins):
    from mobrob_b200 import GpuVecEnv
    from mobrob_b200.ppo import PPO

    cfg = {"observe_goal_lidar": True, "lidar_num_bins": bins}
    env = GpuVecEnv("point", 256, seed=1, time_limit=100, terminate_on_goal=True, robot_config=cfg)
    model = PPO("MlpPolicy", env, n_steps=32, batch_size=1024, n_epochs=2, seed=1, verbose=0)
    first = env.reset_tensor().clone()
    model._last_obs = None
    before = model.updater.params.clone()
    model.learn(total_timesteps=2 * 256 * 32)
    O = 14 + bins
    assert model.updater.obs_dim == O and model.buf["obs"].shape[-1] == O
    assert torch.isfinite(model.updater.params).all() and not torch.equal(before, model.updater.params)
    # the rollout recorded the lidar rows the env produced
    assert torch.count_nonzero(model.buf["obs"][..., 5:5 + bins]) > 0
    act, _ = model.predict(first.cpu().numpy(), deterministic=True)
    assert act.shape == (256, 2)
    model.save(tmp_path / "lidar")
    again = PPO.load(tmp_path / "lidar", env=GpuVecEnv("point", 256, seed=2, time_limit=100, robot_config=cfg))
    assert again.updater.obs_dim == O
    torch.testing.assert_close(again.updater.params, model.updater.params, rtol=0, atol=0)
    act2, _ = again.predict(first.cpu().numpy(), deterministic=True)
    np.testing.assert_array_equal(act2, act)
    loaded = again.updater.params.clone()
    again.learn(total_timesteps=256 * 32)
    assert torch.isfinite(again.updater.params).all() and not torch.equal(loaded, again.updater.params)


def test_evaluate_policy_device_path_equals_sb3_loop(cuda_lib):
    """mr_evaluate's per-step path on a lidar point env against SB3's loop through model.predict and step()."""
    from mobrob_b200 import GpuVecEnv, evaluate_policy
    from mobrob_b200.ppo import PPO

    cfg = {"observe_goal_lidar": True, "observe_goal_dist": True, "lidar_num_bins": 12}
    model = PPO("MlpPolicy", GpuVecEnv("point", 8, seed=1, time_limit=30, robot_config=cfg), n_steps=8, seed=1)
    assert model.policy.obs_dim == 14 + 1 + 12
    dev_env, loop_env = [GpuVecEnv("point", 24, seed=3, time_limit=30, terminate_on_goal=True, robot_config=cfg)
                         for _ in range(2)]
    for _ in range(2):
        got = evaluate_policy(model, dev_env, 61, deterministic=True, return_episode_rewards=True)
        exp = evaluate_policy(model, loop_env, 61, deterministic=True, return_episode_rewards=True,
                              callback=lambda locals_, globals_: None)   # a callback takes SB3's loop on the host
        assert len(exp[0]) == 61
        assert got[1] == exp[1] and got[0] == exp[0]
        assert torch.equal(dev_env.get_state(), loop_env.get_state())
        assert torch.equal(dev_env.get_obs_tensor(), loop_env.get_obs_tensor())
    assert dev_env.eval_steps > 0


def test_car_with_lidar_is_refused_by_ppo(cuda_lib):
    from mobrob_b200 import GpuVecEnv
    from mobrob_b200.ppo import PPO

    car = GpuVecEnv("car", 8, seed=1, robot_config={"observe_goal_lidar": True})
    assert car.obs_dim == 36
    with pytest.raises(ValueError, match="1..31"):
        PPO("MlpPolicy", car, n_steps=8, batch_size=64, n_epochs=1, verbose=0)
