"""observe_goal_lidar without a GPU: the pseudo-lidar restatement on geometries with known answers, the robot_config
parsing of the lidar keys, and the device routine (env_point.cuh goal_lidar, compiled for the host) against the
restatement on random egocentric vectors and settings."""
import math
import os
import shutil
import subprocess

import numpy as np
import pytest

import goal_lidar_oracle as L
from oracle import car_oracle as co, point_oracle as po

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
E1 = math.exp(-1.0)


def _lidar(x, y, **kw):
    return L.obs_lidar_pseudo([(x, y)], **kw)


def _same(got, want):
    """The same bins set, the values to the last bits (math's exp / hypot against numpy's)."""
    np.testing.assert_array_equal(got != 0, np.asarray(want) != 0)
    np.testing.assert_allclose(got, want, rtol=1e-14, atol=0)


def test_goal_straight_ahead():
    # angle 0: bin 0, alias 0 -> the upper neighbour gets 0 * sensor, the lower one (bin n - 1) 1 * sensor
    np.testing.assert_array_equal(_lidar(1.0, 0.0), [E1, 0, 0, 0, 0, 0, 0, 0, 0, E1])
    np.testing.assert_array_equal(_lidar(1.0, 0.0, alias=False), [E1] + [0] * 9)


def test_goal_behind_and_on_bin_edges():
    # 4 bins (bin_size = pi / 2 exactly): behind is angle pi, 2 bin sizes -> bin 2, alias 0
    s = math.exp(-2.0)
    np.testing.assert_array_equal(_lidar(-2.0, 0.0, num_bins=4), [0, s, s, 0])
    # to the left: pi / 2, the edge between bins 0 and 1 -> bin 1, alias 0
    np.testing.assert_array_equal(_lidar(0.0, 1.0, num_bins=4), [E1, E1, 0, 0])
    # mid-bin: pi / 4 -> bin 0, alias 1/2 on both neighbours
    s = math.exp(-math.sqrt(2.0))
    np.testing.assert_allclose(_lidar(1.0, 1.0, num_bins=4), [s, s / 2, 0, s / 2], rtol=1e-15)
    # to the right: -pi / 2 % 2 pi = 3 pi / 2 -> bin 3, alias 0
    np.testing.assert_array_equal(_lidar(0.0, -1.0, num_bins=4), [0, 0, E1, E1])


@pytest.mark.parametrize("n", [1, 2, 3, 10, 16])
def test_wrap_around_angle_is_clamped_to_the_last_bin(n):
    """atan2 of a tiny negative y is a tiny negative angle; % 2 pi rounds it to 2 pi, angle / bin_size to n: the
    reference would index obs[n] (IndexError).  The bin is n - 1, its alias ~1 (the reading leans on bin 0)."""
    x, y = 1.0, -1e-300
    angle = math.atan2(y, x) % (2 * math.pi)
    assert angle == 2 * math.pi and int(angle / (2 * math.pi / n)) == n
    got = _lidar(x, y, num_bins=n)
    want = np.zeros(n)
    want[n - 1] = E1
    want[0] = E1   # alias * sensor, alias ~1
    np.testing.assert_allclose(got, want, rtol=1e-14, atol=1e-15)   # bin n - 2: (1 - alias) * sensor ~0


@pytest.mark.parametrize("n", [1, 2, 3, 10, 16])
def test_bin_counts_and_coinciding_neighbours(n):
    """One object: the block is zero but for bin, bin + 1 and bin - 1 (mod n); for n <= 2 those coincide, and each
    max() sees what the earlier ones left."""
    rng = np.random.default_rng(n)
    for _ in range(50):
        x, y = rng.uniform(-3, 3, 2)
        dist = math.hypot(x, y)
        angle = math.atan2(y, x) % (2 * math.pi)
        size = 2 * math.pi / n
        b = min(int(angle / size), n - 1)
        a = (angle - size * b) / size
        s = math.exp(-dist)
        got = _lidar(x, y, num_bins=n)
        if n == 1:
            _same(got, [s])
        elif n == 2:
            want = np.zeros(2)
            want[b] = s
            want[1 - b] = max(a * s, (1 - a) * s)
            _same(got, want)
        else:
            want = np.zeros(n)
            want[b] = s
            want[(b + 1) % n] = a * s
            want[(b - 1) % n] = (1 - a) * s
            _same(got, want)
        assert np.count_nonzero(_lidar(x, y, num_bins=n, alias=False)) == 1


def test_sensor_modes_and_gain():
    # lidar_max_dist: linear fall-off, zero beyond it (the whole block then is zero)
    np.testing.assert_allclose(_lidar(1.0, 0.0, max_dist=3.0, alias=False), [2 / 3] + [0] * 9, rtol=1e-15)
    np.testing.assert_array_equal(_lidar(4.0, 0.0, max_dist=3.0), np.zeros(10))
    np.testing.assert_array_equal(_lidar(0.0, 0.0, max_dist=3.0, alias=False), [1.0] + [0] * 9)
    # lidar_exp_gain
    np.testing.assert_allclose(_lidar(2.0, 0.0, exp_gain=0.5, alias=False), [math.exp(-1.0)] + [0] * 9, rtol=1e-15)
    np.testing.assert_allclose(_lidar(2.0, 0.0, exp_gain=3.0, alias=False), [math.exp(-6.0)] + [0] * 9, rtol=1e-15)


def test_oracle_block_sits_between_goal_dist_and_gyro():
    for body_cls in (po.PointBody, co.CarBody):
        n = 4
        ora = L.LidarVecOracle(body_cls(n), seed=2, time_limit=30, terminate_on_goal=True,
                               observe={"observe_goal_lidar": True, "observe_goal_dist": True, "observe_ctrl": True},
                               lidar={"num_bins": 7})
        row = ora.reset()
        rng = np.random.default_rng(1)
        for _ in range(4):
            row, *_ = ora.step(rng.uniform(-1, 1, (n, 2)).astype(np.float32))
        base = ora.body.obs(ora.goal)
        plain = L.extend_obs(ora.body, base, ora.goal, {"observe_goal_dist": True, "observe_ctrl": True})
        at = ora.body.obs_pre + 2 + 2 + 1
        assert row.shape == (n, plain.shape[1] + 7)
        np.testing.assert_array_equal(np.delete(row, np.s_[at:at + 7], axis=1), plain)
        block = L.lidar_rows(ora.goal, *L.robot_frames(ora.body), num_bins=7).astype(np.float32)
        np.testing.assert_array_equal(row[:, at:at + 7], block)
        # no key on: the default row itself
        assert L.extend_obs_lidar(ora.body, base, ora.goal, {"observe_goal_lidar": False}) is base


def test_car_lidar_drops_the_goal_height():
    """The car's lidar vector is R^T (goal_xy - p_xy, -p_z), not goal_compass's vector to the goal body at GOAL_Z: they
    differ once the chassis tilts."""
    body = co.CarBody(1)
    body.full_reset(0, (0.2, -0.1), 0.3)
    tilt = np.array([math.cos(0.1), math.sin(0.1), 0.0, 0.0])   # 0.2 rad about x
    q = body.quat[0]
    body.quat[0] = [q[0] * tilt[0] - q[1] * tilt[1], q[0] * tilt[1] + q[1] * tilt[0], q[3] * tilt[1], q[3] * tilt[0]]
    goal = np.array([[1.0, 0.5]])
    pos, mat = L.robot_frames(body)
    ego = L.ego_xy(goal[0], pos[0], mat[0])
    want = co.mtv(co.quat_to_mat(body.quat), np.array([1.0 - 0.2, 0.5 + 0.1, -0.1]))[0, :2]
    np.testing.assert_allclose(ego, want, rtol=1e-14)
    compass = co.mtv(co.quat_to_mat(body.quat), np.array([1.0 - 0.2, 0.5 + 0.1, co.GOAL_Z - 0.1]))[0, :2]
    assert np.abs(ego - compass).max() > 1e-3


# ---- robot_config --------------------------------------------------------------------------------------------------
def test_robot_config_lidar_keys():
    from mobrob_b200.vec_env import lidar_of, obs_flags_of

    assert obs_flags_of({"observe_goal_lidar": True}) == 16
    assert obs_flags_of({"observe_goal_lidar": True, "observe_goal_dist": True}) == 17
    assert obs_flags_of({"observe_goal_lidar": False}) == 0
    assert lidar_of(None) == (10, None, 1.0, True)
    assert lidar_of({"lidar_num_bins": 16, "lidar_max_dist": 3, "lidar_exp_gain": 0.5, "lidar_alias": False,
                     "lidar_type": "pseudo", "observe_qpos": True}) == (16, 3.0, 0.5, False)
    assert lidar_of({"lidar_num_bins": np.int64(4)}) == (4, None, 1.0, True)
    with pytest.raises(NotImplementedError, match="natural"):
        lidar_of({"lidar_type": "natural"})
    for bad in ({"lidar_type": "sonar"}, {"lidar_num_bins": 0}, {"lidar_num_bins": -3}, {"lidar_num_bins": 2.5},
                {"lidar_num_bins": True}, {"lidar_max_dist": 0}, {"lidar_max_dist": -1.0}):
        with pytest.raises(ValueError):
            lidar_of(bad)


# ---- the device routine, compiled for the host ----------------------------------------------------------------------
@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    exe = str(tmp_path_factory.mktemp("host") / "goal_lidar_host")
    subprocess.check_call([nvcc, "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", exe,
                           os.path.join(ROOT, "tests", "host", "goal_lidar_host.cu")])
    return exe


def _cases():
    rng = np.random.default_rng(7)
    cases = []
    for k in range(3000):
        n = int(rng.choice([1, 2, 3, 4, 10, 16, 17, 32])) if k % 2 else int(rng.integers(1, 40))
        max_dist = None if rng.random() < 0.5 else float(rng.uniform(0.2, 5.0))
        gain = 1.0 if rng.random() < 0.3 else float(rng.uniform(0.05, 4.0))
        x, y = rng.uniform(-4, 4, 2) * (10.0 ** rng.integers(-3, 1))
        cases.append((x, y, max_dist, gain, n, bool(rng.integers(0, 2))))
    for n in (1, 2, 3, 4, 10, 16):   # axes, bin edges, the wrap-around clamp, the origin, negative zero
        for x, y in ((1.0, 0.0), (-2.0, 0.0), (0.0, 1.0), (0.0, -1.0), (1.0, -1e-300), (0.0, 0.0), (0.5, -0.0),
                     (-0.5, -0.0), (math.cos(2 * math.pi / n), math.sin(2 * math.pi / n))):
            for alias in (True, False):
                cases.append((x, y, None, 1.0, n, alias))
                cases.append((x, y, 1.5, 1.0, n, alias))
    return cases


def test_device_routine_matches_oracle(harness, tmp_path):
    cases = _cases()
    fin, fout = str(tmp_path / "in.bin"), str(tmp_path / "out.bin")
    rec = np.array([(x, y, 0.0 if m is None else m, g, n, a) for x, y, m, g, n, a in cases], np.float64)
    with open(fin, "wb") as f:
        np.array([len(cases)], np.int64).tofile(f)
        rec.tofile(f)
    subprocess.check_call([harness, fin, fout])
    out = np.fromfile(fout, np.float32)
    off = 0
    for x, y, m, g, n, a in cases:
        got = out[off:off + n]
        off += n
        want = L.obs_lidar_pseudo([(x, y)], num_bins=n, max_dist=m, exp_gain=g, alias=a).astype(np.float32)
        msg = f"ego ({x!r}, {y!r}) bins {n} max_dist {m} gain {g} alias {a}"
        np.testing.assert_array_equal(got != 0, want != 0, err_msg=msg)   # the same bins
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-6, err_msg=msg)
    assert off == out.size
