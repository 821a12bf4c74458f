"""follow_waypoints and GpuVecEnv.set_goals on the device, against the planner loop they replace run step by step
through the policy forward, GpuVecEnv.step_tensor, set_goals and get_obs on a same-seed env, and against the batch-of-
one wrapper's set_goal."""
import os
import sys

import numpy as np
import pytest
import torch
from rollout_oracle import device_draws

pytestmark = pytest.mark.gpu

LIDAR = {"observe_goal_dist": True, "observe_goal_lidar": True}
EP_RET = {"point": 14, "car": 29}   # ep_ret in the reference-view state


@pytest.fixture(scope="module")
def policies(cuda_lib, golden_dir):
    from mobrob_b200.ppo import PPO

    return {name: PPO.load(os.path.join(golden_dir, "policies", f"{name}-ppo.zip")) for name in ("point", "car")}


def _model_for(env, policies, seed=0):
    """The shipped policy for the default row; a fresh seeded one for rows with optional keys."""
    from mobrob_b200 import GpuVecEnv
    from mobrob_b200.ppo import PPO

    if env.obs_flags == 0:
        return policies[env.env_name]
    return PPO("MlpPolicy", GpuVecEnv(env.env_name, 4, seed=1, time_limit=30,
                                      robot_config={"observe_goal_dist": True, "observe_goal_lidar": True}),
               n_steps=8, seed=seed)


def _pair(name, n, seed, robot_config=None, warm=0):
    """Two identical envs without auto-reset, after the seeded reset and `warm` random steps."""
    from mobrob_b200 import GpuVecEnv

    envs = [GpuVecEnv(name, n, seed=seed, time_limit=None, terminate_on_goal=False, robot_config=robot_config)
            for _ in range(2)]
    rng = np.random.default_rng(seed)
    acts = [torch.as_tensor(rng.uniform(-1, 1, (n, 2)).astype(np.float32)).cuda() for _ in range(warm)]
    for e in envs:
        e.reset_tensor()
        for a in acts:
            e.step_tensor(a)
    return envs


def _same_start(dev, ref):
    """Put both envs in one state with ep_ret = 0: dev's state, through the same set_state on both.  The reference
    loop keeps stepping envs after their own end, so after a call ref is not where dev is."""
    s = dev.get_state()
    s[:, EP_RET[dev.env_name]] = 0.0
    dev.set_state(s)
    ref.set_state(s)


def _reference(model, env, W, max_steps, deterministic=True, noise_offset=0):
    """The planner loop, every env stepping each iteration; an env's results are taken at its own stopping step
    (envs are independent, so the steps it takes after that change nothing for the others).  Needs ep_ret = 0 at the
    start: the env's float64 return accumulator then equals the loop's sum of rewards."""
    N, K = W.shape[:2]
    env.set_goals(W[:, 0])
    obs = env.get_obs_tensor()
    k = np.zeros(N, np.int64)
    t = np.zeros(N, np.int64)
    arrival = -np.ones((N, K), np.int64)
    running = np.ones(N, bool)
    ret = np.zeros(N)
    state = env.get_state().cpu().numpy()
    pos = [env.get_pos().cpu().numpy()]
    final_pos = pos[0].copy()
    eps = None if deterministic else device_draws(int(model.seed or 0), N, max_steps, noise_offset, env.first_rank)
    slot = EP_RET[env.env_name]
    for step in range(max_steps):
        if not running.any():
            break
        e = None if deterministic else torch.as_tensor(eps[step]).cuda()
        act, _, _ = model.policy.forward_tensor(obs.contiguous(), e)
        env.step_tensor(act.clamp(-1.0, 1.0).contiguous())
        obs = env.obs.clone()
        p = env.get_pos().cpu().numpy()
        s = env.get_state().cpu().numpy()
        g = W[np.arange(N), np.minimum(k, K - 1)].astype(np.float64)
        reached = np.sqrt((p[:, 0] - g[:, 0]) ** 2 + (p[:, 1] - g[:, 1]) ** 2) < 0.3
        idx = np.nonzero(running)[0]
        t[idx] += 1
        state[idx] = s[idx]
        ret[idx] = s[idx, slot]
        final_pos[idx] = p[idx]
        switch = np.zeros(N, bool)
        for i in idx:
            if reached[i]:
                arrival[i, k[i]] = t[i]
                k[i] += 1
                switch[i] = k[i] < K
        running &= (k < K) & (t < max_steps)
        if switch.any():
            sw = np.nonzero(switch)[0]
            env.set_goals(W[sw, k[sw]], indices=sw)
            obs = env.get_obs_tensor()
            state[sw] = env.get_state().cpu().numpy()[sw]   # the switch happens even on an env's last step
        pos.append(final_pos.copy())
    while len(pos) < max_steps + 1:
        pos.append(final_pos.copy())
    return {"arrivals": arrival, "returns": ret, "steps": t, "state": state, "positions": np.stack(pos)}


def _waypoints(n, K, seed, spread=0.6):
    """A path per env: waypoints a random step of at most `spread` apart, inside the goal box."""
    rng = np.random.default_rng(seed)
    start = rng.uniform(-1.5, 1.5, (n, 1, 2))
    return np.clip(start + np.cumsum(rng.uniform(-spread, spread, (n, K, 2)), axis=1), -2, 2).astype(np.float32)


def _check(got, ref, dev_env, positions=False):
    np.testing.assert_array_equal(got["arrivals"], ref["arrivals"])
    np.testing.assert_array_equal(got["steps"], ref["steps"])
    np.testing.assert_array_equal(got["returns"], ref["returns"])
    np.testing.assert_array_equal(dev_env.get_state().cpu().numpy(), ref["state"])
    if positions:
        np.testing.assert_array_equal(got["positions"], ref["positions"].astype(np.float32))


# ---- set_goals ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["point", "car"])
@pytest.mark.parametrize("robot_config", [None, LIDAR])
def test_set_goals_equals_wrapper_set_goal(cuda_lib, name, robot_config):
    from mobrob_b200.envs.wrapper import CarEnv, PointEnv

    cls = {"point": PointEnv, "car": CarEnv}[name]

    class Env(cls):
        def get_robot_config(self):
            return {**super().get_robot_config(), **(robot_config or {})}

    n = 5
    (venv, _) = _pair(name, n, 3, robot_config, warm=4)
    goals = np.random.default_rng(0).uniform(-2, 2, (n, 2)).astype(np.float32)
    for i in range(n):
        w = Env()
        w.reset(seed=3 + i)
        w.env.set_state(venv.get_state()[i:i + 1])   # the same state, stale ctrl included
        w.set_goal(goals[i])
        venv.set_goals(goals[i:i + 1], indices=[i])
        np.testing.assert_array_equal(venv.obs[i].cpu().numpy(), w.get_obs())
        np.testing.assert_array_equal(venv.get_obs_tensor()[i].cpu().numpy(), w.get_obs())
        # the wrapper's get_state / set_state round trip re-forms the point's world pose: equal up to its rounding
        np.testing.assert_allclose(venv.get_state()[i].cpu().numpy(), w.env.get_state()[0].cpu().numpy(),
                                   rtol=1e-12, atol=1e-12)
        np.testing.assert_array_equal(w.get_goal(), goals[i])
    np.testing.assert_array_equal(venv.get_goals().cpu().numpy(), goals)
    # the zero-copy path, every env
    venv.set_goals(torch.as_tensor(goals[::-1].copy()).cuda())
    np.testing.assert_array_equal(venv.get_goals().cpu().numpy(), goals[::-1])
    assert torch.equal(venv.obs, venv.get_obs_tensor())


# ---- follow_waypoints against the loop --------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 3, 130, 257])
@pytest.mark.parametrize("K", [1, 4, 8])
def test_fused_point_path_equals_loop(policies, n, K):
    from mobrob_b200 import follow_waypoints

    dev, ref = _pair("point", n, 11 + n, warm=3)
    _same_start(dev, ref)
    W = _waypoints(n, K, n * K)
    max_steps = 120   # some envs finish their path, others run out of steps
    got = follow_waypoints(policies["point"], dev, W, max_steps, record_positions=True)
    exp = _reference(policies["point"], ref, W, max_steps)
    _check(got, exp, dev, positions=True)
    if n >= 130:   # both ends of an env's loop occur
        assert (exp["steps"] == max_steps).any() and (exp["arrivals"][:, -1] >= 0).any()


@pytest.mark.parametrize("name,robot_config,n,K,max_steps",
                         [("car", None, 40, 3, 90), ("point", LIDAR, 70, 4, 100)])
def test_per_step_path_equals_loop(policies, name, robot_config, n, K, max_steps):
    from mobrob_b200 import follow_waypoints

    dev, ref = _pair(name, n, 5, robot_config, warm=2)
    _same_start(dev, ref)
    model = _model_for(dev, policies)
    W = _waypoints(n, K, 7, spread=0.4)
    got = follow_waypoints(model, dev, W, max_steps, record_positions=True)
    exp = _reference(model, ref, W, max_steps)
    _check(got, exp, dev, positions=True)
    if name == "car" and robot_config is None:
        assert (exp["arrivals"] >= 0).any()


@pytest.mark.parametrize("name", ["point", "car"])
def test_two_calls_and_stochastic_draws(policies, name):
    """Two calls in a row continue the env (and the Philox counter); the stochastic draws are keyed
    (seed; first_rank + n, eval_steps + t): the first steps follow the restated draws, a replay with the counter wound
    back repeats a call exactly, and a call with the counter continued does not."""
    from mobrob_b200 import GpuVecEnv, follow_waypoints

    n, K, T = 24, 3, 60
    dev, ref = _pair(name, n, 2)
    model = policies[name]
    W = _waypoints(n, K, 1)
    used = 0
    for path in (W, W[:, ::-1].copy()):   # deterministic, back to back, against the loop
        _same_start(dev, ref)
        got = follow_waypoints(model, dev, path, T)
        _check(got, _reference(model, ref, path, T), dev)
        used += int(got["steps"].max())
    assert dev.eval_steps == used

    envs = [GpuVecEnv(name, n, seed=4, time_limit=None, terminate_on_goal=False, first_rank=100) for _ in range(3)]
    for e in envs:
        e.reset_tensor()
    a = follow_waypoints(model, envs[0], W, 3, deterministic=False, record_positions=True)
    # the first steps against the restated draws (equal to a few float32 ulp, so compared to a tolerance)
    exp = _reference(model, envs[1], W, 3, deterministic=False)
    np.testing.assert_allclose(a["positions"], exp["positions"], rtol=0, atol=1e-5)
    assert envs[0].eval_steps == 3
    b = follow_waypoints(model, envs[0], W, T, deterministic=False)          # continues the counter at 3
    envs[2].eval_steps = 0
    c = follow_waypoints(model, envs[2], W, 3, deterministic=False)          # a replay of the first call
    for key in ("arrivals", "returns", "steps"):
        np.testing.assert_array_equal(a[key], c[key])
    b_replay_env = GpuVecEnv(name, n, seed=4, time_limit=None, terminate_on_goal=False, first_rank=100)
    b_replay_env.reset_tensor()
    b_replay_env.eval_steps = 0
    follow_waypoints(model, b_replay_env, W, 3, deterministic=False)
    b_replay_env.eval_steps = 0   # wound back: the second call would reuse the first call's draws
    b_rep = follow_waypoints(model, b_replay_env, W, T, deterministic=False)
    assert not np.array_equal(b["returns"], b_rep["returns"])


def test_baseline_config_first_goals(policies):
    """K = 1 on the shipped point policy is BASELINE configs[1]: from the seeded reset, the first goal's arrival step
    and success are tools/eval_policy.evaluate_gpu's first_len and first_ok on the same 16 384 seeds, env for env."""
    from mobrob_b200 import GpuVecEnv, follow_waypoints

    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import eval_policy

    n = 16384
    g = eval_policy.evaluate_gpu(os.path.join(os.path.dirname(__file__), "golden", "policies", "point-ppo.zip"), n,
                                 steps=1000)
    env = GpuVecEnv("point", n, seed=0, time_limit=None, terminate_on_goal=False)
    env.reset_tensor()
    W = env.get_goals()[:, None, :]
    got = follow_waypoints(policies["point"], env, W, 1000)
    ok = got["arrivals"][:, 0] >= 0
    np.testing.assert_array_equal(ok, g["first_ok"])
    np.testing.assert_array_equal(got["arrivals"][ok, 0], g["first_len"][ok])
    assert ok.mean() > 0.99


def test_wrapper_env_and_refusals(policies):
    from mobrob_b200 import GpuVecEnv, follow_waypoints, get_env

    w = get_env("point", terminate_on_goal=True)
    w.reset(seed=9)
    path = np.array([[0.5, 0.5], [0.0, 1.0]], np.float32)
    out = follow_waypoints(policies["point"], w, path, 400)
    assert out["arrivals"].shape == (1, 2) and out["returns"].shape == (1,)
    np.testing.assert_array_equal(w.get_pos(), w.env.get_pos().cpu().numpy()[0])
    for bad in (get_env("point", time_limit=100), GpuVecEnv("point", 2, time_limit=None),
                GpuVecEnv("point", 2, time_limit=50, terminate_on_goal=False)):
        with pytest.raises(ValueError, match="time_limit|terminate_on_goal"):
            follow_waypoints(policies["point"], bad, path, 10)
