"""The numpy restatement of the rollout kernels' action noise (tests/rollout_oracle.py), pinned without a GPU.

The device draws are Philox4x32-10 + Box-Muller (mobrob_b200/csrc/common.cuh); the GPU tests compare the kernels'
draws with this restatement, so the restatement itself is held to published / independently computed values here.
"""
import numpy as np
import pytest

from rollout_oracle import device_draws, normal2, philox4x32

# (seed, g, c) -> the four output words.  The first is Random123's known-answer vector (all-zero counter and key);
# all three agree with torch's host engine, at::Philox4_32(seed, subsequence=c, offset=g) (ATen/core/PhiloxRNGEngine.h)
KAT = [
    (0, 0, 0, (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    (5, 3, 7, (0xBC00579F, 0xD4321950, 0x708A3C84, 0x82C86342)),
    (2**32 + 9, 2**32 - 1, 296, (0x06794C31, 0x88CC3A86, 0xA36FAA76, 0x2859D6B7)),
]


def _words(seed, g, c):
    m = 0xFFFFFFFF
    return philox4x32((g & m, g >> 32, c & m, c >> 32), (seed & m, seed >> 32))


@pytest.mark.parametrize("seed,g,c,expect", KAT)
def test_philox_known_answers(seed, g, c, expect):
    got = tuple(int(v) for v in _words(seed, g, c))
    assert got == expect, " ".join(f"{v:08x}" for v in got)


def test_philox_vectorised_equals_scalar():
    seeds, gs, cs = [0, 5, 2**32 + 9, 2**64 - 1], [0, 1, 2**32 - 2, 2**32, 2**40 + 3], [0, 7, 2**32 + 1]
    for s in seeds:
        g = np.array(gs, dtype=np.uint64)[:, None]
        c = np.array(cs, dtype=np.uint64)[None, :]
        m = np.uint64(0xFFFFFFFF)
        vec = philox4x32((g & m, g >> np.uint64(32), c & m, c >> np.uint64(32)), (s & 0xFFFFFFFF, s >> 32))
        for i, gi in enumerate(gs):
            for j, cj in enumerate(cs):
                assert tuple(int(v[i, j]) for v in vec) == tuple(int(v) for v in _words(s, gi, cj))


def _box_muller64(u0, u1):
    """Box-Muller in float64 on the float32-quantised uniforms (u + 0.5) * 2^-32 the kernel forms."""
    q = lambda u: (np.asarray(u, np.uint32).astype(np.float32) + np.float32(0.5)).astype(np.float64) / 2**32  # noqa: E731
    a, b = np.clip(q(u0), 1e-10, 1.0), q(u1)
    r = np.sqrt(-2.0 * np.log(a))
    return r * np.cos(2 * np.pi * b), r * np.sin(2 * np.pi * b), r


def test_normal2_is_box_muller_in_float32():
    rng = np.random.default_rng(0)
    u = rng.integers(0, 2**32, size=(2, 200000), dtype=np.uint64).astype(np.uint32)
    edges = np.array([[0, 1, 2**31, 2**32 - 128, 2**32 - 1, 2**24 + 1], [0, 2**30, 2**31, 3 * 2**30, 2**32 - 1, 1]],
                     dtype=np.uint32)
    u = np.concatenate([u, edges], axis=1)
    z0, z1 = normal2(u[0], u[1])
    assert z0.dtype == np.float32 and z1.dtype == np.float32
    r0, r1, rad = _box_muller64(u[0], u[1])
    # float32 log / sqrt / product: a few ulp of the radius
    for z, r in ((z0, r0), (z1, r1)):
        assert np.all(np.abs(z - r) <= 5e-7 * np.maximum(rad, 1.0)), float((np.abs(z - r) / np.maximum(rad, 1.0)).max())
    # the top 128 words round to a = 1 in float32 (a tie at 2^32 - 128 goes to the even 2^32): radius 0, both draws exactly 0
    assert z0[-3] == 0.0 and z1[-3] == 0.0 and z0[-2] == 0.0 and z1[-2] == 0.0
    # the smallest word: a = 2^-33 stays above the 1e-10 floor, radius sqrt(66 ln 2)
    assert abs(float(np.hypot(z0[-6], z1[-6])) - np.sqrt(66 * np.log(2))) < 1e-5
    full = np.concatenate([z0[:-6], z1[:-6]])
    assert abs(full.mean()) < 0.01 and abs(full.std() - 1.0) < 0.01
    assert abs(np.mean(z0[:-6] * z1[:-6])) < 0.01


def test_device_draws_are_keyed_by_global_env_and_step():
    """The draw of (env, step) depends only on (seed, env_offset + n, noise_offset + t): a shard or a later rollout
    reads a slice of the same array, across the 32-bit word boundaries of both counters."""
    full = device_draws(9, 12, 6, noise_offset=2**32 - 3, env_offset=2**32 - 6)
    np.testing.assert_array_equal(device_draws(9, 5, 4, noise_offset=2**32 - 1, env_offset=2**32 - 2), full[2:, 4:9])
    np.testing.assert_array_equal(device_draws(9, 1, 1, noise_offset=2**32 + 2, env_offset=2**32 + 5), full[5:, 11:])
    assert full.shape == (6, 12, 2) and full.dtype == np.float32
    # every key word matters: another seed, env or step gives unrelated draws
    assert not np.any(device_draws(9 + 2**32, 12, 6, 2**32 - 3, 2**32 - 6) == full)
    assert np.all(np.abs(full[:, 1:] - full[:, :-1]) > 0) and np.all(np.abs(full[1:] - full[:-1]) > 0)
    # z = (r cos, r sin) of ONE Philox call: components x and y of the counter (g, c)
    z = device_draws(5, 1, 1, noise_offset=7, env_offset=3)[0, 0]
    w = _words(5, 3, 7)
    np.testing.assert_array_equal(z, np.array(normal2(w[0], w[1])))
