"""-m gpu tests of the row-parallel kernel's pair jobs (csrc/sacx_rowpar.cuh, RpJob::pair) at shapes where the twin critics'
hidden layers pair with a weight slice each. At the shapes of test_gpu_rowpar.py only the policy's twins (shared slice) and
the critics' first layers pair; here a three-layer critic pairs its middle layer too: by TMA (32 columns per CTA, K = 64)
and by cp.async (8 columns per CTA)."""
import numpy as np
import pytest

from gpu_helpers import assert_close
from test_gpu_rowpar import _engine

pytestmark = pytest.mark.gpu

CASES = [
    # obs, act, hidden_pi, hidden_q, B, activation
    (11, 3, (256, 256), (64, 256, 64), 48, "relu"),       # critic layer 1: 64 -> 256, two TMA-staged slices in one slot
    (10, 2, (64, 128), (64, 64, 64), 40, "tanh"),         # critic layer 1: 64 -> 64, two cp.async slices in one slot
]


@pytest.mark.parametrize("obs,act,hp,hq,B,actfn", CASES)
def test_rowpar_hidden_layer_pairs_match_tile_parallel_path(obs, act, hp, hq, B, actfn, monkeypatch):
    rng = np.random.default_rng(17)
    K = 2
    idx = np.stack([rng.choice(1500, B, replace=False) for _ in range(K)]).astype(np.int64)
    e1 = rng.standard_normal((K, B, act)).astype(np.float32)
    e2 = rng.standard_normal((K, B, act)).astype(np.float32)
    names = ("batch.s2a", "batch.spi", "out.y", "out.logpi", "out.logpi_next", "out.q1", "out.q2", "out.tq1", "out.tq2",
             "out.q1_pi", "out.q2_pi", "delta.q1.0", "delta.pi.0", "block.params", "block.targets")
    out = {}
    for rowpar in (True, False):
        eng = _engine(obs, act, hp, hq, B, actfn, monkeypatch, rowpar)
        assert eng.path()[0] == ("rowpar" if rowpar else "tiles"), eng.path()
        snaps = []
        for k in range(K):
            m = eng.update_host(idx[k], e1[k], e2[k], 1)
            assert m["nonfinite"] == 0 and m["updates"] == k + 1
            snaps.append({n: eng.view(n).cpu().numpy().copy() for n in names})
        out[rowpar] = snaps
    for k in range(K):
        a, b = out[True][k], out[False][k]
        tol = 2e-5 * (3 ** k)
        for n in ("batch.s2a", "batch.spi", "out.y", "out.logpi", "out.logpi_next", "out.q1", "out.q2", "out.tq1", "out.tq2",
                  "out.q1_pi", "out.q2_pi"):
            assert_close(f"step{k} {n}", a[n], b[n], tol)
        for n in ("delta.q1.0", "delta.pi.0"):
            assert_close(f"step{k} {n}", a[n], b[n], 5 * tol)
        for n in ("block.params", "block.targets"):
            assert_close(f"step{k} {n}", a[n], b[n], 1e-4 * (2 ** k))
