"""bench.py --dump-outputs: the fields of a batched solve as float64 .npy files, a seeded sample of
the problems when the batch is larger than the cap."""
import os
import subprocess
import sys
import types

import numpy as np
import pytest

from conftest import ROOT, assert_solution_parity
import bench


def _solution(B, N, rng):
    return types.SimpleNamespace(
        x=rng.random((B, 9 * N)), cost=rng.random(B), nit=rng.integers(0, 16, B, dtype=np.int32),
        nfev=rng.integers(1, 40, B, dtype=np.int32), status=rng.integers(0, 3, B, dtype=np.int32),
        task=rng.integers(0, 6, B, dtype=np.int32), accelerations=rng.random((B, N, 3)),
        attitudes=rng.random((B, N, 3)), body_rates=rng.random((B, N, 3)), thrusts=rng.random((B, N)))


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_writes_every_field_as_float64(tmp_path):
    sol = _solution(300, 8, np.random.default_rng(1))
    bench.dump_outputs(str(tmp_path), sol)
    got = _load(tmp_path)
    assert set(got) == set(bench.DUMP_FIELDS) | {"index"}
    assert all(a.dtype == np.float64 for a in got.values())
    np.testing.assert_array_equal(got["index"], np.arange(300))
    for f in bench.DUMP_FIELDS:
        np.testing.assert_array_equal(got[f], getattr(sol, f))


def test_dump_of_a_large_batch_is_a_seeded_sample_within_the_cap(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    sol = _solution(4096, 8, np.random.default_rng(2))
    bench.dump_outputs(str(tmp_path / "a"), sol)
    bench.dump_outputs(str(tmp_path / "b"), sol)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert sum(os.path.getsize(tmp_path / "a" / (f + ".npy")) for f in a) <= 1 << 20
    idx = a["index"].astype(np.int64)
    assert 0 < len(idx) < 4096 and np.all(np.diff(idx) > 0)
    for f in bench.DUMP_FIELDS:
        np.testing.assert_array_equal(a[f], getattr(sol, f)[idx])
        np.testing.assert_array_equal(a[f], b[f])


@pytest.mark.parametrize("impl", ["reference", pytest.param("b200", marks=pytest.mark.gpu)])
def test_bench_dumps_what_its_last_timed_step_returned(impl, tmp_path, oracle_mod):
    """bench.py end to end: the files hold the timed path's result for the seeded workload
    (BatchResult of the oracle for `--impl reference`, HostSolution of the GPU solve otherwise)."""
    # the GPU leg cycles through input/output sets totalling > 2 x L2: a small batch means thousands of sets
    B = 64 if impl == "reference" else 4096
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", impl, "--batch", str(B), "--steps", "2",
           "--warmup", "1", "--no-extras", "--dump-outputs", str(tmp_path)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    got = _load(tmp_path)
    assert set(got) == set(bench.DUMP_FIELDS) | {"index"}
    np.testing.assert_array_equal(got["index"], np.arange(B))
    p0, v0, goal = bench.workload_inputs(B, 1)
    ref = oracle_mod.solve_batch(oracle_mod.make_params(horizon=8, dt=0.1), p0, v0, goal, nthreads=4)
    if impl == "reference":
        for f in bench.DUMP_FIELDS:
            np.testing.assert_array_equal(got[f], getattr(ref, f), err_msg=f)
    else:
        want = {f: getattr(ref, f) for f in bench.DUMP_FIELDS}
        assert_solution_parity(types.SimpleNamespace(**got), dict(want, fun=ref.cost, dt=0.1), "bench dump")
