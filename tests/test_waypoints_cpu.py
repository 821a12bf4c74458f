"""follow_waypoints without a GPU: argument checks, the [K, 2] broadcast, the ctypes rows of the two entry points, and
a numpy restatement of the planner loop on the oracle's point body, checked on hand-built cases."""
import numpy as np
import pytest
import torch

from oracle import point_oracle as po
from oracle.vec_oracle import GoalVecOracle


# ---- the planner loop, restated on the oracle (one single-env oracle per env: an env that has finished is not
# stepped) --------------------------------------------------------------------------------------------------------
def follow_oracle(oracles, policy, W, max_steps):
    """oracles: one GoalVecOracle of one env per path, reset, without auto-reset.  policy(obs [1, O]) -> [1, 2]."""
    N, K = W.shape[:2]
    arrival = -np.ones((N, K), np.int64)
    ret = np.zeros(N)
    steps = np.zeros(N, np.int64)
    for i, ora in enumerate(oracles):
        ora.goal[0] = W[i, 0]          # set_goal; the oracle keeps prev_pos, as reward_fn keeps _prev_pos
        obs = ora._obs()
        k = t = 0
        while k < K and t < max_steps:
            obs, r, _, info = ora.step(policy(obs))
            t += 1
            ret[i] = info["ep_r"][0]   # ep_ret accumulates the float64 rewards from the reset on
            if ora.reached()[0]:
                arrival[i, k] = t
                k += 1
                if k < K:
                    ora.goal[0] = W[i, k]
                    obs = ora._obs()
        steps[i] = t
    return arrival, ret, steps


def _oracles(n, seed=0):
    out = []
    for i in range(n):
        ora = GoalVecOracle(po.PointBody(1), seed=seed + i, time_limit=None, terminate_on_goal=False)
        ora.reset()
        out.append(ora)
    return out


def _still(obs):
    return np.zeros((1, 2), np.float32)


def test_restatement_hand_built_cases():
    oras = _oracles(3)
    p = np.stack([o.body.pos()[0] for o in oras]).astype(np.float32)
    far = np.float32(3.0)
    W = np.stack([
        np.stack([p[0], p[0] + far]),          # reached on the first step, then never
        np.stack([p[1], p[1] + 0.1]),          # two waypoints within 0.3: the second on the next step, not the same
        np.stack([p[2] + far, p[2] + far]),    # max_steps ends the path
    ])
    arrival, ret, steps = follow_oracle(oras, _still, W, 5)
    np.testing.assert_array_equal(arrival, [[1, -1], [1, 2], [-1, -1]])
    np.testing.assert_array_equal(steps, [5, 2, 5])
    # a robot at rest does not move: each step pays only the reach bonus
    np.testing.assert_array_equal(ret, [5.0, 10.0, 0.0])


def test_restatement_reward_keeps_prev_pos_across_a_switch():
    """The first step after a switch pays |g_new - p_prev| - |g_new - p_cur| (+5 on reaching)."""
    (ora,) = _oracles(1, seed=4)
    rng = np.random.default_rng(0)
    ora.goal[0] = ora.body.pos()[0].astype(np.float32)
    ora.step(rng.uniform(-1, 1, (1, 2)).astype(np.float32))
    g_new = np.array([1.5, -1.5], np.float32)
    ora.goal[0] = g_new
    p_prev = ora.body.pos()[0]
    _, r, _, _ = ora.step(np.ones((1, 2), np.float32))
    p_cur = ora.body.pos()[0]
    g = g_new.astype(np.float64)
    assert r[0] == np.float32(np.linalg.norm(g - p_prev) - np.linalg.norm(g - p_cur))


# ---- argument checks ---------------------------------------------------------------------------------------------
def test_check_waypoints_broadcast_and_errors():
    from mobrob_b200.waypoints import check_waypoints

    path = np.arange(8, dtype=np.float64).reshape(4, 2)
    w = check_waypoints(path, 3, 10)
    assert w.shape == (3, 4, 2) and w.dtype == np.float32
    np.testing.assert_array_equal(w[2], path.astype(np.float32))
    t = check_waypoints(torch.as_tensor(path), 3, 10)
    assert t.shape == (3, 4, 2) and t.dtype == torch.float32
    assert check_waypoints(np.zeros((3, 5, 2)), 3, 1).shape == (3, 5, 2)
    for bad in (np.zeros((2, 4, 2)), np.zeros((3, 4, 3)), np.zeros(4), np.zeros((3, 0, 2)), np.zeros((0, 2))):
        with pytest.raises(ValueError, match="waypoints"):
            check_waypoints(bad, 3, 10)
    for ms in (0, -1):
        with pytest.raises(ValueError, match="max_steps"):
            check_waypoints(path, 3, ms)


def test_env_configuration_is_checked():
    from mobrob_b200.envs.wrapper import TimeLimit
    from mobrob_b200.vec_env import GpuVecEnv
    from mobrob_b200.waypoints import vec_env_of

    def fake(time_limit, terminate_on_goal):
        env = object.__new__(GpuVecEnv)   # the attributes follow_waypoints reads; no device needed
        env.time_limit, env.terminate_on_goal = time_limit, terminate_on_goal
        return env

    ok = fake(None, False)
    assert vec_env_of(ok) is ok
    assert vec_env_of(fake(0, False)) is not None
    with pytest.raises(ValueError, match="terminate_on_goal=False, time_limit=None"):
        vec_env_of(fake(None, True))
    with pytest.raises(ValueError, match="terminate_on_goal=False, time_limit=None"):
        vec_env_of(fake(1000, False))
    with pytest.raises(ValueError, match="time_limit=None"):
        vec_env_of(TimeLimit(object(), 100))
    with pytest.raises(TypeError):
        vec_env_of(object())


def test_signature_rows():
    from ctypes import c_int, c_int64, c_uint64, c_void_p

    from mobrob_b200 import _lib

    P = c_void_p
    assert _lib._SIGNATURES["mr_env_set_goals"] == (c_int, [P, P, P, P, P])
    assert _lib._SIGNATURES["mr_follow_waypoints"] == (
        c_int, [P, P, c_int, P, c_int, c_int64, c_uint64, c_uint64, c_int64, P, P, P, P, P, P])
