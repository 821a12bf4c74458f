"""Hazards on the device: the layouts and headings of full resets, the hazards_lidar block and the cost against the
restatement (tests/hazards_oracle.py) on the kernels' own state, the columns a hazard leaves alone, fixed and failing
layouts, sharding, set_goals / follow_waypoints, PPO, evaluate_policy and the batch-of-one wrapper."""
import numpy as np
import pytest
import torch

import goal_lidar_oracle as L
import hazards_oracle as H
import test_waypoints_gpu as WP

pytestmark = pytest.mark.gpu

PRE = {"point": 3, "car": 15}
BASE = {"point": 14, "car": 26}
SEED_STEP = {"point": 2, "car": 1}   # Engine resets per full reset: PointEnv.set_pos resets the Engine again
HAZ = {"hazards_num": 8, "observe_hazards": True, "constrain_hazards": True, "constrain_indicator": False,
       "hazards_size": 0.35}


def _env(kind, n, seed, cfg, **kw):
    from mobrob_b200 import GpuVecEnv

    return GpuVecEnv(kind, n, seed=seed, robot_config=cfg, **kw)


def _expected_layouts(env, seed):
    """(hazards [n][num][2], headings [n]) of each env's last full reset, from its count of full resets."""
    fulls = env.get_reset_counts().cpu().numpy()[:, 1]
    out = [H.layout(seed + env.first_rank + i + SEED_STEP[env.env_name] * int(f), env.hazards_num,
                    env.hazards["keepout"], env.hazards["locations"]) for i, f in enumerate(fulls)]
    assert all(o[0] for o in out)
    return np.stack([o[2] for o in out]), np.array([o[1] for o in out])


def _check_layouts(env, seed, msg=""):
    hz, heading = _expected_layouts(env, seed)
    np.testing.assert_array_equal(env.get_hazards().cpu().numpy(), hz, err_msg=msg)
    st = env.get_state().cpu().numpy()
    if env.env_name == "point":
        np.testing.assert_array_equal(st[:, 8], heading, err_msg=msg)
    else:   # the free joint's quaternion rot2quat(heading) of a full reset: compare where it was not moved since
        fresh = (env.get_reset_counts().cpu().numpy()[:, 1] > 0) & (st[:, 13:24] == 0).all(axis=1)
        np.testing.assert_allclose(st[fresh][:, [3, 6]], np.stack([np.cos(0.5 * heading), np.sin(0.5 * heading)], 1)[fresh],
                                   rtol=0, atol=1e-15, err_msg=msg)


def _block(env, hazards, state=None):
    st = env.get_state().cpu().numpy() if state is None else state
    bins = env.lidar[0] if env.lidar else 10
    return H.hazards_rows(hazards, *L.robot_frames_of_state(env.env_name, st), num_bins=bins).astype(np.float32)


def _at(kind):
    return PRE[kind] + 2 + 3   # ... goal_compass | gyro | hazards_lidar


@pytest.mark.parametrize("kind", ["point", "car"])
def test_layouts_rows_and_cost_on_the_kernels_state(cuda_lib, kind):
    """First and later full resets lay out the restatement's hazards and headings, goal-only resets keep them; every
    step row, terminal row and post-reset row carries the restatement's block for the kernels' exported state, and
    the cost is Engine.cost of the pre-reset position against the step's hazards."""
    from mobrob_b200.spaces import Box

    n, tl, T = (64, 25, 90) if kind == "point" else (12, 12, 30)
    env = _env(kind, n, 4, HAZ, time_limit=tl, terminate_on_goal=True)
    twin = _env(kind, n, 4, HAZ, time_limit=None, terminate_on_goal=False)   # env's step without the reset
    env.reset_init_space(Box(np.full(2, -0.3, np.float32), np.full(2, 0.3, np.float32), dtype=np.float32))
    env.reset_goal_space(Box(np.full(2, -0.5, np.float32), np.full(2, 0.5, np.float32), dtype=np.float32))
    at, tol = _at(kind), dict(rtol=1e-6, atol=1e-7)
    assert env.obs_dim == BASE[kind] + 10
    obs = env.reset()
    _check_layouts(env, 4, "first reset")
    np.testing.assert_allclose(obs[:, at:at + 10], _block(env, env.get_hazards().cpu().numpy()), **tol)
    np.testing.assert_array_equal(env.cost.cpu().numpy(), np.zeros(n))
    rng = np.random.default_rng(2)
    n_term = n_cost = 0
    for t in range(T):
        a = rng.uniform(-1.5, 1.5, (n, 2)).astype(np.float32)
        hz = env.get_hazards().cpu().numpy()
        twin.set_state(env.get_state())
        obs, rew, done, infos = env.step(a)
        t_obs, *_ = twin.step(a)
        pre = twin.get_state().cpu().numpy()
        # where no reset followed, the env's own float64 xy is the step's; twin's state went through the state view,
        # which re-forms the point's pose in the last bits
        pos = np.where(done[:, None], twin.get_pos().cpu().numpy(), env.get_pos().cpu().numpy())
        want_cost = np.array([H.cost(hz[i], pos[i], 0.35, 1.0, False) for i in range(n)])
        got_cost = np.array([d["cost"] for d in infos])
        np.testing.assert_array_equal(got_cost[~done], want_cost[~done], err_msg=f"cost step {t}")
        np.testing.assert_allclose(got_cost[done], want_cost[done], rtol=0, atol=1e-12, err_msg=f"cost step {t}")
        assert all(d["cost_hazards"] == d["cost"] for d in infos)
        n_cost += int((want_cost > 0).sum())
        _check_layouts(env, 4, f"step {t}")
        np.testing.assert_allclose(obs[:, at:at + 10], _block(env, env.get_hazards().cpu().numpy()), **tol,
                                   err_msg=f"row step {t}")
        for i in np.nonzero(done)[0]:
            n_term += 1
            np.testing.assert_allclose(infos[i]["terminal_observation"][at:at + 10], _block(env, hz[i:i + 1], pre[i:i + 1])[0],
                                       **tol, err_msg=f"terminal row step {t}")
    counts = env.get_reset_counts().cpu().numpy()
    assert n_term > 0 and n_cost > 0
    assert (counts[:, 0] - counts[:, 1]).sum() > 0, "no goal-only reset"
    assert (counts[:, 1] > 1).sum() > 0, "no full reset after the first"


@pytest.mark.parametrize("kind", ["point", "car"])
def test_hazards_only_change_the_start_heading(cuda_lib, kind):
    """Without observe_hazards / constrain_hazards a hazard env computes what the hazard-free env computes from the same
    state: only the layout's start heading differs; infos carry no cost.  The car's step is inlined differently in the
    kernels with hazards, so its float64 state may differ in the last bits; its float32 rows and rewards do not."""
    n, T = (64, 40) if kind == "point" else (12, 15)
    haz = _env(kind, n, 6, {"hazards_num": 5}, time_limit=None, terminate_on_goal=False)
    ref = _env(kind, n, 6, None, time_limit=None, terminate_on_goal=False)
    o_h, o_r = haz.reset(), ref.reset()
    assert haz.obs_dim == ref.obs_dim
    s_h, s_r = haz.get_state().cpu().numpy(), ref.get_state().cpu().numpy()
    diff = np.nonzero((s_h != s_r).any(axis=0))[0].tolist()
    assert diff == ([8] if kind == "point" else [3, 6]), diff   # psi0 / the free joint's yaw quaternion
    ref.set_state(haz.get_state())
    np.testing.assert_array_equal(haz.get_obs_tensor().cpu().numpy(), ref.get_obs_tensor().cpu().numpy())
    rng = np.random.default_rng(1)
    for t in range(T):
        a = rng.uniform(-1.5, 1.5, (n, 2)).astype(np.float32)
        o_h, r_h, d_h, i_h = haz.step(a)
        o_r, r_r, d_r, i_r = ref.step(a)
        np.testing.assert_array_equal(o_h, o_r, err_msg=f"step {t}")
        np.testing.assert_array_equal(r_h, r_r)
        assert i_h == i_r and "cost" not in i_h[0]
    if kind == "point":
        assert torch.equal(haz.get_state(), ref.get_state())
    else:
        torch.testing.assert_close(haz.get_state(), ref.get_state(), rtol=1e-12, atol=1e-12)


def test_fixed_locations_failing_layout_and_sharding(cuda_lib):
    from mobrob_b200.vec_env import ResamplingError

    locs = [(1.0, -1.0), (-1.5, 1.5)]
    env = _env("point", 16, 3, {"hazards_num": 3, "hazards_locations": locs}, time_limit=10)
    env.reset()
    hz = env.get_hazards().cpu().numpy()
    np.testing.assert_allclose(hz[:, :2], np.broadcast_to(locs, (16, 2, 2)), atol=2e-9)
    _check_layouts(env, 3)
    bad = _env("car", 2, 3, {"hazards_num": 2, "hazards_locations": [(0.5, 0.5), (0.5, 0.5)]})
    with pytest.raises(ResamplingError, match="Failed to sample layout of objects"):
        bad.reset()
    cfg = {"hazards_num": 6, "observe_hazards": True}
    whole = _env("point", 10, 9, cfg, time_limit=20)
    parts = [_env("point", 5, 9, cfg, time_limit=20, first_rank=r) for r in (0, 5)]
    o = whole.reset()
    o_parts = np.concatenate([p.reset() for p in parts])
    np.testing.assert_array_equal(o, o_parts)
    np.testing.assert_array_equal(whole.get_hazards().cpu().numpy(),
                                  np.concatenate([p.get_hazards().cpu().numpy() for p in parts]))


def _model(env_cfg, obs_dim):
    from mobrob_b200.ppo import PPO

    model = PPO("MlpPolicy", _env("point", 4, 1, env_cfg, time_limit=30), n_steps=8, seed=0)
    assert model.policy.obs_dim == obs_dim
    return model


@pytest.mark.parametrize("kind", ["point", "car"])
def test_set_goals_rows_and_follow_waypoints_equal_the_loop(cuda_lib, kind):
    from mobrob_b200 import follow_waypoints

    cfg = {"hazards_num": 6, "observe_hazards": True} if kind == "point" else {"hazards_num": 6}
    n, K, max_steps = (40, 3, 80) if kind == "point" else (16, 2, 40)
    dev, ref = WP._pair(kind, n, 5, cfg, warm=2)
    goals = np.random.default_rng(0).uniform(-2, 2, (n, 2)).astype(np.float32)
    dev.set_goals(goals)
    assert torch.equal(dev.obs, dev.get_obs_tensor())
    if kind == "point":
        np.testing.assert_allclose(dev.obs[:, 8:18].cpu().numpy(), _block(dev, dev.get_hazards().cpu().numpy()),
                                   rtol=1e-6, atol=1e-7)
    WP._same_start(dev, ref)
    model = _model(cfg, dev.obs_dim) if kind == "point" else None
    if model is None:
        from mobrob_b200.ppo import PPO
        model = PPO("MlpPolicy", _env("car", 4, 1, cfg, time_limit=30), n_steps=8, seed=0)
    W = WP._waypoints(n, K, 7, spread=0.4)
    got = follow_waypoints(model, dev, W, max_steps, record_positions=True)
    exp = WP._reference(model, ref, W, max_steps)
    if kind == "point":
        WP._check(got, exp, dev, positions=True)
    else:   # the car's masked step and its env step inline the dynamics differently: float64 equal to the last bits
        np.testing.assert_array_equal(got["arrivals"], exp["arrivals"])
        np.testing.assert_array_equal(got["steps"], exp["steps"])
        np.testing.assert_allclose(got["returns"], exp["returns"], rtol=0, atol=1e-12)
        np.testing.assert_allclose(dev.get_state().cpu().numpy(), exp["state"], rtol=0, atol=1e-12)
        np.testing.assert_allclose(got["positions"], exp["positions"].astype(np.float32), rtol=1e-6, atol=1e-6)
    assert torch.equal(dev.get_hazards(), ref.get_hazards())


def test_ppo_and_evaluate_policy_on_the_24_float_row(cuda_lib, tmp_path):
    from mobrob_b200 import evaluate_policy
    from mobrob_b200.ppo import PPO

    cfg = {"hazards_num": 8, "observe_hazards": True, "constrain_hazards": True}
    env = _env("point", 256, 1, cfg, time_limit=100, terminate_on_goal=True)
    model = PPO("MlpPolicy", env, n_steps=32, batch_size=1024, n_epochs=2, seed=1, verbose=0)
    first = env.reset_tensor().clone()
    model._last_obs = None
    before = model.updater.params.clone()
    model.learn(total_timesteps=2 * 256 * 32)
    assert model.updater.obs_dim == 24 and model.buf["obs"].shape[-1] == 24
    assert torch.isfinite(model.updater.params).all() and not torch.equal(before, model.updater.params)
    assert torch.count_nonzero(model.buf["obs"][..., 8:18]) > 0
    act, _ = model.predict(first.cpu().numpy(), deterministic=True)
    model.save(tmp_path / "hazards")
    again = PPO.load(tmp_path / "hazards", env=_env("point", 256, 2, cfg, time_limit=100))
    torch.testing.assert_close(again.updater.params, model.updater.params, rtol=0, atol=0)
    np.testing.assert_array_equal(again.predict(first.cpu().numpy(), deterministic=True)[0], act)
    loaded = again.updater.params.clone()
    again.learn(total_timesteps=256 * 32)
    assert torch.isfinite(again.updater.params).all() and not torch.equal(loaded, again.updater.params)
    dev_env, loop_env = [_env("point", 24, 3, cfg, time_limit=30, terminate_on_goal=True) for _ in range(2)]
    got = evaluate_policy(model, dev_env, 61, deterministic=True, return_episode_rewards=True)
    exp = evaluate_policy(model, loop_env, 61, deterministic=True, return_episode_rewards=True,
                          callback=lambda locals_, globals_: None)
    assert got[1] == exp[1] and got[0] == exp[0]
    assert torch.equal(dev_env.get_state(), loop_env.get_state())
    assert torch.equal(dev_env.get_hazards(), loop_env.get_hazards())


@pytest.mark.parametrize("kind", ["point", "car"])
def test_wrapper_subclass_returns_the_cost(cuda_lib, kind):
    from mobrob_b200.envs.wrapper import CarEnv, PointEnv

    class WithHazards(PointEnv if kind == "point" else CarEnv):
        def get_robot_config(self):
            return {**super().get_robot_config(), "hazards_num": 8, "hazards_size": 0.5, "hazards_keepout": 0.3,
                    "hazards_locations": [(0.3, 0.0)], "constrain_hazards": True, "observe_hazards": True}

    env = WithHazards(terminate_on_goal=False)
    assert env.observation_space.shape == (BASE[kind] + 10,)
    env.seed(3)
    obs, _ = env.reset(init_pos=np.zeros(2))   # a robot placed at the origin starts inside hazard 0 (as can happen)
    engine_seed = 3 + (3 if kind == "point" else 1)   # the point's two set_pos calls rebuild the Engine twice
    ok, heading, hz, _ = H.layout(engine_seed, 8, 0.3, [(0.3, 0.0)])
    np.testing.assert_array_equal(env.env.get_hazards().cpu().numpy()[0], hz)
    if kind == "point":
        assert env.env.get_state().cpu().numpy()[0, 8] == heading
    seen = 0.0
    for _ in range(60):
        obs, rew, term, trunc, info = env.step(np.array([1.0, 0.2], np.float32))
        p = env.get_pos()
        assert info["cost"] == info["cost_hazards"] == H.cost(hz, p, 0.5, 1.0, True)
        seen += info["cost"]
    np.testing.assert_allclose(obs[_at(kind):_at(kind) + 10], _block(env.env, hz[None])[0], rtol=1e-6, atol=1e-7)
    assert seen > 0
