"""mr_device_permutations' keyed bijection (mobrob_b200/csrc/perm.cuh), compiled for the HOST, against its numpy
restatement (tests/perm_ref.py): integer work, bit for bit, no GPU needed.  The statistical quality of the stream is
tested on the device output (tests/test_device_perm_gpu.py); this holds the arithmetic."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from perm_ref import device_permutation

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    exe = str(tmp_path_factory.mktemp("host") / "perm_host")
    subprocess.check_call([nvcc, "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", exe,
                           os.path.join(ROOT, "tests", "host", "perm_host.cu")])
    return exe


@pytest.mark.parametrize("seed,stream,n", [(0, 0, 1), (0, 1, 2), (3, 5, 3), (1, 2, 1024), (7, (3 << 48) ^ (9 << 16) ^ 4, 18944),
                                           (2**63 + 11, 2**40 + 5, 100003), (0, 17, 1212416)])
def test_host_compiled_permutation_is_the_numpy_restatement(harness, tmp_path, seed, stream, n):
    out = str(tmp_path / "perm.bin")
    subprocess.check_call([harness, str(seed), str(stream), str(n), out])
    got = np.fromfile(out, np.int64)
    np.testing.assert_array_equal(got, device_permutation(seed, stream, n))
    assert np.array_equal(np.sort(got), np.arange(n))   # a bijection of [0, n)
