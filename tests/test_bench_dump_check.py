"""tools/check_bench_dump.py on a dump written by bench.dump_outputs itself (no GPU): stand-in handles hand dump_outputs the
oracle's own result arrays for two frames of a C2 step, so the checker must find the dump equal to the oracle, and must not
when one label is changed or when it is told the wrong --inflight (the frame behind a dump index shifts)."""
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOOL = os.path.join(ROOT, "tools", "check_bench_dump.py")
# frame indices of a step as bench.py's last group dumps them with --inflight 80: slots 64 and 77 -> pool frames 0 and 13
INFLIGHT = 80
DUMPED = (784, 797)


class ResultOf:
    """Stands in for a Segmenter: fetch_result() returns the given arrays."""

    def __init__(self, arrays):
        self.arrays = arrays

    def fetch_result(self):
        return {n: self.arrays[n].copy() for n in ("out_xyz", "out_label", "out_voxel", "merges_ab", "merges_w", "merges_left")}


def run_tool(out_dir, *args):
    return subprocess.run([sys.executable, TOOL, str(out_dir)] + list(args), capture_output=True, text=True, timeout=600)


@pytest.fixture(scope="module")
def oracle_results(oracle_mod):
    """The oracle's fetch_result() arrays of the pool frames behind DUMPED."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import check_bench_dump
    frames = bench.make_frames(0, min(bench.N_POOL, INFLIGHT))
    return {k: check_bench_dump.oracle_arrays((frames[check_bench_dump.frame_slot(k, INFLIGHT)], bench.FLAGS)) for k in DUMPED}


def test_checker_accepts_oracle_dump_and_rejects_wrong_ones(tmp_path, oracle_results):
    assert [(k % INFLIGHT) % bench.N_POOL for k in DUMPED] == [0, 13]
    # the labelled clouds of a VGA frame are longer than DUMP_ROWS: the checker must rebuild dump_outputs' row sample
    assert all(len(r["out_label"]) > bench.DUMP_ROWS for r in oracle_results.values())
    assert all(len(r["merges_w"]) < bench.DUMP_ROWS for r in oracle_results.values())
    bench.dump_outputs(str(tmp_path), [(k, ResultOf(oracle_results[k])) for k in DUMPED])
    assert len(os.listdir(tmp_path)) == 2 * 6

    ok = run_tool(tmp_path)
    assert ok.returncode == 0, ok.stdout + ok.stderr
    verdicts = [l for l in ok.stdout.splitlines() if l.startswith("frame ")]
    assert len(verdicts) == 12 and all(" ok " in l for l in verdicts), ok.stdout

    wrong_flight = run_tool(tmp_path, "--inflight", "64")           # 784 % 64 = 16: pool frame 16 instead of 0
    assert wrong_flight.returncode != 0 and "MISMATCH" in wrong_flight.stdout, wrong_flight.stdout

    p = os.path.join(tmp_path, "frame%04d_out_label.npy" % DUMPED[1])
    lab = np.load(p)
    lab[lab.shape[0] // 2] += 1
    np.save(p, lab)
    one_label = run_tool(tmp_path)
    assert one_label.returncode != 0, one_label.stdout
    bad = [l for l in one_label.stdout.splitlines() if "MISMATCH" in l]
    assert bad == [l for l in bad if l.startswith("frame %04d" % DUMPED[1]) and "out_label" in l and "1 of" in l] and len(bad) == 1, one_label.stdout
