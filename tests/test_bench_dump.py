"""bench.py --dump-outputs: what the chain's last timed step computed, written as float64 .npy files (row pointers in full,
column indices as a fixed seeded sample with its positions).  CPU: the sampling and the files on a stand-in result.  GPU: a
small run of bench.py end to end, its files against the oracle's chain on the same last batch, and the same files again from
a second run with the same arguments."""
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
import oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("row_ptr", "col_idx_sample", "col_idx_sample_pos")


class _Result:
    def __init__(self, p, j):
        self.p, self.j = p, j

    def export_csr(self):
        return self.p.astype(np.int64), self.j, None


def _load(d):
    return {k: np.load(os.path.join(d, k + ".npy")) for k in NAMES}


def test_dump_samples_a_large_result_at_fixed_positions(tmp_path):
    rng = np.random.default_rng(7)
    nnz = bench.DUMP_SAMPLE + 123_457
    p = np.linspace(0, nnz, 33).astype(np.int64)
    j = rng.integers(0, 1 << 24, nnz).astype(np.uint32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), _Result(p, j))
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert all(a[k].dtype == np.float64 and np.array_equal(a[k], b[k]) for k in NAMES)
    pos = a["col_idx_sample_pos"].astype(np.int64)
    assert len(pos) == bench.DUMP_SAMPLE and np.all(np.diff(pos) > 0) and pos[0] >= 0 and pos[-1] < nnz
    assert np.array_equal(a["col_idx_sample"], j[pos].astype(np.float64))
    assert np.array_equal(a["row_ptr"], p.astype(np.float64))
    assert sum(os.path.getsize(tmp_path / "a" / (k + ".npy")) for k in NAMES) <= 64 << 20


def test_dump_keeps_a_small_result_whole(tmp_path):
    p = np.array([0, 2, 2, 5], np.int64)
    j = np.array([1, 9, 0, 3, 4], np.uint32)
    bench.dump_outputs(str(tmp_path), _Result(p, j))
    a = _load(tmp_path)
    assert np.array_equal(a["col_idx_sample"], j.astype(np.float64))
    assert np.array_equal(a["col_idx_sample_pos"], np.arange(5, dtype=np.float64))


def test_dump_is_refused_where_it_is_not_implemented():
    for extra in (["--workload", "bfs"], ["--impl", "reference"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", "x"] + extra,
                           capture_output=True, text=True, cwd=ROOT)
        assert r.returncode == 2 and "--dump-outputs" in r.stderr, r.stderr
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 2 and "--steps" in r.stderr, r.stderr


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step_and_repeats_it(tmp_path):
    scale, ef, seed, nsrc, hops, steps, warmup = 10, 16, 1, 64, 3, 2, 1
    for d in ("a", "b"):
        cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--scale", str(scale), "--edge-factor", str(ef),
               "--seed", str(seed), "--sources", str(nsrc), "--hops", str(hops), "--steps", str(steps), "--warmup", str(warmup),
               "--side", "none", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / d)]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
        assert r.returncode == 0, r.stderr[-2000:]
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert all(np.array_equal(a[k], b[k]) for k in NAMES)
    A = orc.rmat_csr(scale, ef, seed)
    last = bench.pick_sources(np.diff(A.p), steps + warmup, nsrc, seed, 0)[-1]
    W, _ = bench.cpu_chain(orc, A, last, hops)
    assert np.array_equal(a["row_ptr"], W.p.astype(np.float64))
    assert np.array_equal(a["col_idx_sample"], W.j[a["col_idx_sample_pos"].astype(np.int64)].astype(np.float64))
