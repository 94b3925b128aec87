"""Tests of bench.py's command line and of the output dump that lets two builds be compared output for output.  bench.py runs
in a subprocess throughout: importing it would change this interpreter (sys.path, bytecode writing)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import rel_l2, splitmix_src

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")


def _bench(*args, **kw):
    return subprocess.run([sys.executable, BENCH, *args], capture_output=True, text=True, **kw)


def test_steps_must_be_positive():
    r = _bench("--steps", "0")
    assert r.returncode == 2 and "--steps" in r.stderr


def test_dump_is_refused_for_the_reference_arm(tmp_path):
    r = _bench("--impl", "reference", "--dump-outputs", str(tmp_path / "d"))
    assert r.returncode == 2 and "--dump-outputs" in r.stderr
    assert not (tmp_path / "d").exists()


def test_reference_arm_times_the_steps_it_is_given():
    r = _bench("--impl", "reference", "--cells", "2", "--steps", "3", "--warmup", "0", timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["warmup"] == 0 and line["value"] > 0


def test_dump_is_a_fixed_bounded_sample(tmp_path):
    code = ("import sys, numpy as np; sys.path.insert(0, %r); import bench\n"
            "v = np.arange(bench.DUMP_MAX + 12345, dtype=np.float64)  # entry == its index\n"
            "bench.dump_outputs(sys.argv[1], 'z', v)\n"
            "bench.dump_outputs(sys.argv[2], 'z', np.linspace(-1.0, 1.0, 11, dtype=np.float32))\n"
            "print(bench.DUMP_MAX)" % ROOT)
    runs = [subprocess.run([sys.executable, "-c", code, str(tmp_path / ("big%d" % k)), str(tmp_path / "small")],
                           capture_output=True, text=True, check=True) for k in (0, 1)]
    dump_max = int(runs[0].stdout)
    a, b = np.load(tmp_path / "big0" / "z.npy"), np.load(tmp_path / "big1" / "z.npy")
    assert a.dtype == np.float64 and a.size == dump_max and np.array_equal(a, b)  # the same sample in every run
    assert np.all(np.diff(a) > 0) and a[-1] < dump_max + 12345  # distinct entries, in index order
    assert os.path.getsize(tmp_path / "big0" / "z.npy") <= 64 << 20
    small = np.load(tmp_path / "small" / "z.npy")  # below DUMP_MAX: the whole array, as float64
    assert small.dtype == np.float64 and np.array_equal(small, np.linspace(-1.0, 1.0, 11, dtype=np.float32).astype(np.float64))


@pytest.mark.gpu
def test_dump_holds_the_vcycle_output(tmp_path, oracle):
    """The dumped array is what the timed path returns: one V-cycle of the configuration's hierarchy (c1: Q2 on every level,
    Chebyshev(3)) applied to the bench's residual splitmix_src(n), here at 8^3 cells, against the oracle's V-cycle."""
    r = _bench("--config", "c1", "--cells", "8", "--steps", "2", "--warmup", "3", "--no-cpu-baseline",
               "--dump-outputs", str(tmp_path / "d"), timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    z = np.load(tmp_path / "d" / "vcycle_z.npy")
    levels = [(2, 2 ** k) for k in range(4)]  # 1 -> 8 cells
    mfs = [oracle.MatrixFree(3, p, n) for (p, n) in levels]
    trs = [oracle.Transfer(mfs[l - 1], mfs[l], "h") for l in range(1, len(levels))]
    vc = oracle.VCycle(mfs, trs, degree=3)
    vc.estimate()
    assert z.shape == (mfs[-1].n_dofs,)
    assert rel_l2(z, vc.vmult(splitmix_src(mfs[-1].n_dofs))) <= 1e-10
