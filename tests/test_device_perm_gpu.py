"""mr_device_permutations: the keyed on-device index stream used by PPO(permutation="device")."""
import ctypes

import numpy as np
import pytest
import torch

from mobrob_b200 import _lib
from perm_ref import device_permutation as perm_ref

pytestmark = pytest.mark.gpu


def _perm(seed, stream, n):
    out = torch.full((n,), -1, dtype=torch.int64, device="cuda")
    key = (ctypes.c_uint64 * 1)(stream)
    _lib.check(_lib.load().mr_device_permutations(seed, key, 1, n, out.data_ptr(),
                                                  torch.cuda.current_stream().cuda_stream))
    return out.cpu().numpy()


def test_is_a_permutation_for_ragged_sizes(cuda_lib):
    for n in (1, 2, 3, 100, 4096, 4097, 65536, 4096 * 296):
        assert np.array_equal(np.sort(_perm(3, 7, n)), np.arange(n))


def test_matches_the_numpy_restatement_bit_for_bit(cuda_lib):
    for seed, stream, n in ((0, 0, 1), (1, 2, 2), (3, 7, 3), (5, 1 << 40, 1000), (9, 3, 65537), (0, (2 << 48) ^ (5 << 16) ^ 3, 4096 * 296)):
        np.testing.assert_array_equal(_perm(seed, stream, n), perm_ref(seed, stream, n))


def _chi2(a, b, bins):
    """Pearson statistic of the bins x bins contingency table of two integer arrays already binned."""
    tab = np.zeros((bins, bins))
    np.add.at(tab, (a, b), 1)
    e = len(a) / bins**2
    return ((tab - e) ** 2 / e).sum()


def test_chi_square_positions_values_pairs(cuda_lib):
    """No structure between where an index lands and what it is (high bits and low bits), nor between
    successive indices: Pearson statistics on 64 x 64 tables stay within 5 sigma of their 3969 degrees of
    freedom (mean 3969, sigma 89) for every key tried.  (The four multiply-xorshift rounds this replaced
    fail the low-bits table by orders of magnitude.)"""
    n, bins = 4096 * 296, 64
    dof = (bins - 1) ** 2
    lim = dof + 5 * np.sqrt(2 * dof)
    i = np.arange(n)
    for seed, stream in ((0, 0), (0, 1), (7, (3 << 48) ^ (11 << 16) ^ 9), (123456789, 5)):
        p = _perm(seed, stream, n)
        assert _chi2(i * bins // n, p * bins // n, bins) < lim          # position x value, high bits
        assert _chi2(i % bins, p % bins, bins) < lim                    # low bits
        assert _chi2(p[:-1] * bins // n, p[1:] * bins // n, bins) < lim  # successive pairs
        assert _chi2(p[:-1] % bins, p[1:] % bins, bins) < lim
        # minibatch composition: every 18 944-sample minibatch x 64 buffer regions (64 x 64 table again)
        assert _chi2(i // 18944, p * bins // n, bins) < lim
    # different epochs of one iteration (consecutive stream ids) are unrelated permutations
    a, b = _perm(0, 5 << 16, n), _perm(0, (5 << 16) ^ 1, n)
    assert _chi2(a * bins // n, b * bins // n, bins) < lim


def test_pure_function_of_seed_and_stream(cuda_lib):
    a = _perm(1, 5, 100000)
    assert np.array_equal(a, _perm(1, 5, 100000))
    assert (a != _perm(1, 6, 100000)).mean() > 0.99
    assert (a != _perm(2, 5, 100000)).mean() > 0.99


def test_minibatches_are_well_mixed(cuda_lib):
    # env-major sample ids n*T + t: every minibatch should draw evenly from all parts of the buffer
    n, mb, bins = 4096 * 296, 18944, 16
    worst = 0.0
    for s in range(4):
        p = _perm(0, s, n)
        for k in (0, 17, 63):
            h = np.bincount(p[k * mb:(k + 1) * mb] * bins // n, minlength=bins)
            worst = max(worst, np.abs(h / mb - 1 / bins).max())
        # no short-range structure: neighbours in the stream are far apart in the buffer
        assert np.median(np.abs(np.diff(p[:10000]))) > n / 8
    assert worst < 0.01


def test_prepare_epochs_device_equals_the_two_step_form(cuda_lib):
    """mr_ppo_prepare_epochs_device (index streams generated on the fly) == mr_device_permutations followed by
    mr_ppo_prepare_epochs: same buffer rows bit for bit, same per-minibatch advantage sums; and the rows are
    what numpy makes of the restated permutation."""
    from mobrob_b200.updater import PpoUpdater

    N, T, B, E, seed = 37, 64, 300, 3, 11
    n = N * T
    up = PpoUpdater(14, torch.device("cuda", 0))
    adv = torch.randn((T, N), device="cuda")
    ids = [(2 << 48) ^ (7 << 16) ^ e for e in range(E)]
    perms = torch.empty((E, n), dtype=torch.int64, device="cuda")
    keys = (ctypes.c_uint64 * E)(*ids)
    _lib.check(up.lib.mr_device_permutations(seed, keys, E, n, perms.data_ptr(), torch.cuda.current_stream().cuda_stream))
    stats_a, rows_a = up.prepare_epochs(adv, perms, B, N, T)
    rows_a = rows_a.clone()
    stats_b, rows_b = up.prepare_epochs_device(adv, seed, ids, B, N, T)
    assert torch.equal(rows_a, rows_b)
    np.testing.assert_allclose(stats_b.cpu().numpy(), stats_a.cpu().numpy(), rtol=1e-14)
    for e in range(E):
        p = perm_ref(seed, ids[e], n)
        np.testing.assert_array_equal(perms[e].cpu().numpy(), p)
        np.testing.assert_array_equal(rows_b[e].cpu().numpy(), (p % T) * N + p // T)
