"""bench.py --dump-outputs: what the last timed solve returned, written as .npy files so that two builds can be compared
output for output.  CPU: the seeded sample and the argument checks; -m gpu: a small run whose dump is the oracle's
solve of the same problem."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")


def test_solution_sample_is_fixed_and_bounded():
    import bench
    x = np.arange(3 * bench.DUMP_SAMPLE, dtype=np.float64)
    s = bench.solution_sample(x)
    assert s.size == bench.DUMP_SAMPLE and s.size * 8 * 2 <= 64 << 20      # two quadratures within 64 MB
    assert np.all(np.diff(s) > 0)                                          # distinct entries, in index order
    np.testing.assert_array_equal(s, bench.solution_sample(x.copy()))
    small = np.arange(1000.0)
    np.testing.assert_array_equal(bench.solution_sample(small), small)


@pytest.mark.parametrize("extra", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "d"]])
def test_bench_rejects_bad_arguments(extra):
    out = subprocess.run([sys.executable, BENCH, "--gpus", "1"] + extra, capture_output=True, text=True, timeout=120)
    assert out.returncode == 2 and "error" in out.stderr


@pytest.mark.gpu
def test_dumped_solution_is_the_timed_solve(tmp_path):
    import oracle as O
    p, cells = 3, 6
    out = subprocess.run([sys.executable, BENCH, "--gpus", "1", "--steps", "2", "--warmup", "1", "--degree", str(p),
                          "--cells", str(cells), "--no-variants", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert sorted(os.listdir(tmp_path)) == ["gll_solve.npy", "gll_x.npy"]
    x, solve = np.load(tmp_path / "gll_x.npy"), np.load(tmp_path / "gll_solve.npy")
    assert x.dtype == np.float64 and solve.dtype == np.float64
    its, _, x_l2 = solve
    assert abs(its - d["config"]["iterations_per_step"]) <= 1 and x_l2 == d["check"]["x_l2"]
    m = O.OracleMesh(p, (cells,) * 3, quad=O.GLL)
    b = m.rhs()
    xo, its_o, *_ = m.cg(b, variant=1, control=0, tol=1e-6 * np.linalg.norm(b), max_its=200)
    assert x.size == m.n_dofs and abs(its - its_o) <= 1
    assert np.linalg.norm(x - xo) <= (1e-8 if its == its_o else 1e-5) * np.linalg.norm(xo)
    assert x_l2 == pytest.approx(np.linalg.norm(xo), rel=1e-5)
