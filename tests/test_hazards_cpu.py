"""Hazards without a GPU: the device routines (env_point.cuh hazard_layout / hazards_lidar / hazard_cost, compiled for
the host) against the restatement in tests/hazards_oracle.py, and the parsing of the Engine's hazard keys."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import hazards_oracle as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    d = tmp_path_factory.mktemp("host")
    exe = str(d / "hazards_host")
    subprocess.check_call([nvcc, "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", exe,
                           os.path.join(ROOT, "tests", "host", "hazards_host.cu")])

    def run(records):
        fi, fo = d / "in.bin", d / "out.bin"
        np.concatenate([np.asarray(r, np.float64).ravel() for r in records]).tofile(fi)
        subprocess.check_call([exe, str(fi), str(fo)])
        return np.fromfile(fo, np.float64)
    return run


# (seed, num, keepout, locations): default Safety Gym levels, crowded floors that reject often (past MtHead's 227 words
# and past one 624-word MT round), conflicting fixed locations (every layout fails)
LAYOUTS = ([(s, 8, 0.4, ()) for s in range(1, 40)] + [(s, 32, 0.18, ()) for s in range(100, 112)] +
           [(s, 12, 0.45, ()) for s in range(200, 206)] + [(7, 3, 0.4, ((1.0, 1.0), (-1.2, 0.5))), (8, 1, 0.3, ((0.0, 0.0),))])


def _layout_record(seed, num, keepout, locs):
    return [0, seed, num, keepout, len(locs), *np.asarray(locs, np.float64).ravel()]


def test_device_layout_equals_randomstate_restatement(host):
    out = host([_layout_record(*c) for c in LAYOUTS])
    k, words = 0, []
    for seed, num, keepout, locs in LAYOUTS:
        ok, heading, hz, w = H.layout(seed, num, keepout, locs)
        words.append(w)
        got_ok, got_heading, got_hz = out[k], out[k + 1], out[k + 2:k + 2 + 2 * num].reshape(num, 2)
        k += 2 + 2 * num
        assert bool(got_ok) == ok, (seed, num)
        if ok:
            assert got_heading == heading, (seed, num)
            np.testing.assert_array_equal(got_hz, hz, err_msg=f"seed {seed}")
    assert k == len(out)
    assert max(words) > 624 and sum(w > 227 for w in words) >= 3, words


def test_layout_fixed_locations_and_failure(host):
    ok, _, hz, _ = H.layout(7, 3, 0.4, ((1.0, 1.0), (-1.2, 0.5)))
    assert ok
    np.testing.assert_allclose(hz[:2], [[1.0, 1.0], [-1.2, 0.5]], atol=2e-9)
    # two hazards fixed at one point can never keep 2 * keepout from each other: every layout fails
    rec = _layout_record(3, 2, 0.4, ((0.5, 0.5), (0.5, 0.5)))
    assert not H.layout(3, 2, 0.4, ((0.5, 0.5), (0.5, 0.5)))[0]
    assert host([rec])[0] == 0.0


def _yaw(psi):
    c, s = np.cos(psi), np.sin(psi)
    return np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])


@pytest.mark.parametrize("lidar", [{}, {"num_bins": 16, "max_dist": 1.5, "alias": False}, {"num_bins": 2, "exp_gain": 0.4},
                                   {"num_bins": 1}, {"num_bins": 7, "max_dist": 3.0}])
def test_lidar_over_several_hazards(host, lidar):
    rng = np.random.default_rng(5)
    cfg = {**{"num_bins": 10, "max_dist": None, "exp_gain": 1.0, "alias": True}, **lidar}
    recs, want = [], []
    for case in range(40):
        num = int(rng.integers(1, 9))
        hz = rng.uniform(-2, 2, (num, 2))
        if case % 5 == 0:
            hz[1:] = hz[0]          # coinciding hazards: the max keeps one
        pos = np.array([*rng.uniform(-1.5, 1.5, 2), rng.choice([0.0, 0.1])])
        R = _yaw(rng.uniform(0, 2 * np.pi))
        if pos[2]:
            R = R @ _yaw(0.0)[[0, 2, 1]][:, [0, 2, 1]]   # a tilted frame for the car's case
        m = np.concatenate([R[:, 0], R[:, 1]])        # rows of R^T
        recs.append([1, num, *hz.ravel(), *m, *pos, cfg["num_bins"], cfg["max_dist"] or 0.0, cfg["exp_gain"],
                     int(cfg["alias"])])
        want.append(H.hazards_block(hz, pos, R, **cfg))
    got = host(recs).reshape(len(want), cfg["num_bins"])
    np.testing.assert_allclose(got, np.asarray(want, np.float32), rtol=1e-6, atol=1e-7)


def test_cost_indicator_and_boundary(host):
    hz = np.array([[0.5, 0.0], [0.0, 0.5], [1.5, 1.5]])
    cases = [((0.5, 0.0), 0.3, 1.0, 0), ((0.3, 0.1), 0.3, 2.5, 0), ((0.25, 0.25), 0.4, 1.0, 0), ((1.0, 1.0), 0.3, 1.0, 0),
             ((0.8, 0.0), 0.3, 1.0, 0), ((0.8, 0.0), 0.3, 1.0, 1), ((0.5, 0.1), 0.3, 1.0, 1), ((1.0, 1.0), 0.3, 1.0, 1)]
    recs = [[2, 3, *hz.ravel(), x, y, size, c, ind] for (x, y), size, c, ind in cases]
    got = host(recs)
    want = [H.cost(hz, xy, size, c, bool(ind)) for xy, size, c, ind in cases]
    np.testing.assert_array_equal(got, want)
    # exactly at d == size the hazard counts, with a zero shaped cost: the indicator stays 0 there
    assert H.cost(hz, (0.8, 0.0), 0.3, 1.0, False) == 0.0 and got[4] == 0.0 and got[5] == 0.0
    assert got[0] == 0.3 and got[6] == 1.0 and got[7] == 0.0


def test_hazard_keys_parsing_and_refusals():
    from mobrob_b200.vec_env import HAZARD_DEFAULTS, hazards_of, obs_flags_of

    assert HAZARD_DEFAULTS["hazards_num"] == 0 and HAZARD_DEFAULTS["hazards_size"] == 0.3
    assert hazards_of(None) is None and hazards_of({"hazards_size": 0.2}) is None
    hz = hazards_of({"hazards_num": 4, "constrain_hazards": True})
    assert hz["num"] == 4 and hz["size"] == 0.3 and hz["keepout"] == 0.4 and hz["cost"] == 1.0
    assert hz["constrain"] and hz["indicator"] and hz["locations"].shape == (0, 2)
    assert hazards_of({"hazards_num": 2, "hazards_locations": [(1, 1)]})["locations"].tolist() == [[1.0, 1.0]]
    assert obs_flags_of({"hazards_num": 3, "observe_hazards": True}) == 32
    assert obs_flags_of({"hazards_num": 3, "observe_hazards": True, "observe_goal_lidar": True}) == 48
    with pytest.raises(NotImplementedError):
        obs_flags_of({"observe_hazards": True})
    with pytest.raises(NotImplementedError):
        obs_flags_of({"observe_hazards": True, "hazards_num": 0})
    with pytest.raises(NotImplementedError, match="placements"):
        hazards_of({"hazards_num": 2, "hazards_placements": [(-1, -1, 1, 1)]})
    with pytest.raises(ValueError, match="hazards_num"):
        hazards_of({"hazards_num": 33})
    with pytest.raises(ValueError, match="hazards_locations"):
        hazards_of({"hazards_num": 1, "hazards_locations": [(0, 0), (1, 1)]})
    with pytest.raises(ValueError, match="World has starting cost"):
        hazards_of({"hazards_num": 1, "constrain_hazards": True, "hazards_size": 0.8})
    # without constrain_hazards the Engine computes no cost, so a large hazard is accepted
    assert hazards_of({"hazards_num": 1, "hazards_size": 0.8})["size"] == 0.8
