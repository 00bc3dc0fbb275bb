"""CPU tests of oracle/device_rng.py, the NumPy restatement of the device RNG streams (csrc/sacx_math.cuh) that
test_gpu_rowpar_oracle.py compares the kernels' indices and normals with."""
import math

import numpy as np
import pytest

from oracle import device_rng as R


@pytest.mark.parametrize("ctr,key,want", [
    ([0, 0, 0, 0], [0, 0], "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
    ([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2, "408f276d 41c83b0e a20bc7c6 6d5451fd"),
    ([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0], "d16cfe09 94fdcceb 5001e420 24126ea1"),
])
def test_philox4x32_10_known_answers(ctr, key, want):
    """The Random123 known-answer vectors of Philox4x32-10."""
    assert " ".join("%08x" % w for w in R.philox4x32_10(ctr, key)) == want


@pytest.mark.parametrize("n", [1, 2, 3, 31, 32, 33, 1000, 4097, 2 ** 20 + 1])
def test_feistel_index_is_a_bijection(n):
    for seed, counter, agent in ((0, 0, 0), (7, 3, 0), (0x123456789ABCDEF, 2 ** 32 + 5, 9)):
        idx = R.feistel_indices(n, n, seed, counter, agent)
        assert np.array_equal(np.sort(idx), np.arange(n)), (n, seed, counter)
        # the vectorized network is the scalar one
        for i in sorted({0, n // 2, n - 1}):
            assert idx[i] == R.feistel_index(i, n, seed, counter, agent)


def test_feistel_streams_depend_on_key():
    n = 4097
    a = R.feistel_indices(64, n, 1, 0, 0)
    for other in (R.feistel_indices(64, n, 2, 0, 0), R.feistel_indices(64, n, 1, 1, 0), R.feistel_indices(64, n, 1, 0, 1)):
        assert not np.array_equal(a, other)


def test_philox_normal_uniforms_and_moments():
    """u1 is never 0 (the log stays finite), and the draws are standard normal."""
    z = np.array([R.philox_normal(5, u, w, row, j, 0) for u in range(4) for w in (1, 2) for row in range(128) for j in range(4)])
    assert np.isfinite(z).all()
    assert abs(z.mean()) < 0.06 and abs(z.std() - 1) < 0.05
    u1, u2 = R.philox_uniforms(0, 0, 1, 0, 0, 0)
    assert u1.dtype == np.float32 and 0 < u1 <= 1 and 0 <= u2 < 1
    assert R.philox_normal(0, 0, 1, 0, 0, 0) == math.sqrt(-2 * math.log(float(u1))) * math.cos(2 * math.pi * float(u2))
