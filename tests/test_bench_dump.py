"""bench.py --dump-outputs: the outputs of the last timed step as .npy files, within the size budget, and on the GPU equal to
what the step returned (its verdicts are the C oracle's CNF check of its prediction on the same seeded batch)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.conftest import ROOT


def test_dump_outputs_samples_what_does_not_fit(tmp_path):
    import bench
    big = np.arange(bench.DUMP_BYTES // 8 + 1000, dtype=np.float64)
    small = np.linspace(0, 1, 8).astype(np.float32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"prediction": big, "solved": small})
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["prediction.npy", "solved.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 * 10 ** 6
    p = np.load(tmp_path / "a" / "prediction.npy")
    assert p.dtype == np.float64 and 0 < p.size < big.size
    assert (np.diff(p) > 0).all() and (p == np.round(p)).all()        # a subset of the elements, in their order
    assert np.array_equal(np.load(tmp_path / "a" / "solved.npy"), small)
    for f in files:                                                   # the sample is fixed
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))


@pytest.mark.gpu
def test_bench_dumps_the_last_step(tmp_path):
    from oracle import pdp_oracle as po
    from pdp_solver_b200 import cnfgen
    problems, n, seed = 2, 3000, 4000
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                          "--problems", str(problems), "--n", str(n), "--iterations", "30", "--walksat", "20", "--seed", str(seed),
                          "--no-cpu-baseline", "--no-config0", "--strong-problems", "0", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    pred = np.load(tmp_path / "prediction.npy")
    solved = np.load(tmp_path / "solved.npy")
    unsat = np.load(tmp_path / "unsat_clauses.npy")
    assert pred.dtype == solved.dtype == unsat.dtype == np.float32
    assert pred.shape == (problems * n,) and solved.shape == unsat.shape == (problems,)
    assert np.isin(pred, (0.0, 1.0)).all()
    want_solved, want_unsat = po.Oracle(*cnfgen.random_batch(problems, n, 3, 4.2, seed)).cnf_eval(pred)
    assert np.array_equal(solved, want_solved) and np.array_equal(unsat, want_unsat)
