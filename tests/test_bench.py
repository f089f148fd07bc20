"""bench.py --dump-outputs: the row sample stays within its 64 MB and repeats from run to run (CPU),
and the files hold what the last timed step returned for the seeded inputs (GPU)."""
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle
from gpu_util import gsi  # noqa: F401

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def bench(monkeypatch):
    for v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        monkeypatch.delenv(v, raising=False)        # bench pins these on import; restored after the test
    return importlib.import_module("bench")


@pytest.mark.parametrize("workload", ["small", "c3", "c5", "dense"])
def test_dump_rows_fit_the_budget_and_repeat(bench, workload):
    kind, grid, ell, K, p, q, _ = bench.WORKLOADS[workload]
    n, l = int(np.prod(grid)), K + p
    rows = bench.dump_rows(n, l)
    assert 8 * l * (len(rows) + 1) + 2 * 128 <= bench.DUMP_BYTES <= 64_000_000   # Z rows, S, two .npy headers
    assert np.all(np.diff(rows) > 0) and rows[0] >= 0 and rows[-1] < n
    assert np.array_equal(rows, bench.dump_rows(n, l))
    if 8 * l * (n + 1) + 4096 <= bench.DUMP_BYTES:
        assert np.array_equal(rows, np.arange(n))
    else:
        assert len(rows) > bench.DUMP_BYTES // (8 * l) - 16


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(gsi, tmp_path):
    out = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
           "--workload", "small", "--no-cpu-baseline", "--no-e2e", "--no-extras", "--no-parity",
           "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert r.returncode == 0 and lines, f"rc={r.returncode}\n{r.stdout[-2000:]}\n{r.stderr[-3000:]}"
    res = json.loads(lines[-1])
    assert res["steps"] == 2
    Z, S = np.load(out / "Z.npy"), np.load(out / "S.npy")
    assert sorted(os.listdir(out)) == ["S.npy", "Z.npy"]
    assert sum(os.path.getsize(out / f) for f in os.listdir(out)) <= 64_000_000
    n, K, p, q = 28 * 26 * 24, 200, 10, 2                     # bench.WORKLOADS["small"]: every row fits
    assert Z.dtype == S.dtype == np.float64 and Z.shape == (n, K + p) and S.shape == (K + p,)
    assert list(S[:5]) == res["sigma_head"]
    # the same seeded inputs through the library in this process give the same Z
    op = gsi.GridKernelCovMatrix("gaussian", (28, 26, 24), (9.0, 7.0, 5.0))
    Omega = np.random.default_rng(0).standard_normal((n, K + p))
    Zr, Sr = gsi.randsvd(op, K, p, q, Omega=Omega, return_singular_values=True)
    op.free()
    c = oracle.compare_Z(Z, Zr, K)
    assert c["tail_zero"] and c["sv_rel"] < 1e-12 and c["sine"] < 1e-8, c
    assert np.allclose(S, Sr, rtol=1e-12, atol=0) and np.allclose(S[:K], oracle.singvals_from_Z(Z, K), rtol=1e-12)
