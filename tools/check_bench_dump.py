#!/usr/bin/env python
"""Compare what `bench.py --dump-outputs DIR` wrote with the CPU oracle.

  python tools/check_bench_dump.py DIR [--workload c2|c3] [--inflight 80]

bench.py's sweep leg gives slot i of a step the resident copy i % inflight of the rank's min(N_POOL, inflight) distinct frames,
so frame k of the dump (rank 0) is make_frames(0, min(N_POOL, F), base)[(k % F) % min(N_POOL, F)], base 20020 for c2 and 30000
for c3.  The oracle (stamp-based merge, same vccs defaults and flags) recomputes every such frame, and its arrays are cut to
the rows bench.dump_outputs keeps: np.sort(default_rng(k).choice(n, DUMP_ROWS, replace=False)) of an array longer than
DUMP_ROWS; uint32 arrays were stored as float64.  Merge weights are held to the bar of the parity tests (close_enough in
tests/test_gpu_parity.py: 1e-6 relative, at most 0.2 % not bit-identical); everything else must be identical.
Prints one verdict per frame and array; the exit status is 1 on any mismatch or missing array."""
import argparse
import multiprocessing
import os
import re
import sys
from concurrent.futures import ProcessPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"), os.path.join(ROOT, "fast-3d-pointcloud-segmentation_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import bench  # noqa: E402  (importing it has no side effects)

ARRAYS = ("out_xyz", "out_label", "out_voxel", "merges_ab", "merges_w", "merges_left")
BASE_SEED = {"c2": 20020, "c3": 30000}


def dumped_frames(out_dir):
    """{k: {name: path}} of the frame<k>_<name>.npy files in out_dir."""
    found = {}
    for f in os.listdir(out_dir):
        m = re.fullmatch(r"frame(\d+)_(\w+)\.npy", f)
        if m:
            found.setdefault(int(m.group(1)), {})[m.group(2)] = os.path.join(out_dir, f)
    return found


def frame_slot(k, inflight):
    """Index into make_frames(0, min(N_POOL, inflight), base) of frame k of a step."""
    F = max(1, inflight)
    return (k % F) % min(bench.N_POOL, F)


def pool_frame(slot, workload):
    """bench.make_frames(0, n, BASE_SEED[workload])[slot] for any n > slot, without generating the frames before it."""
    from f3ps import synth
    return synth.make_frame(seed=BASE_SEED[workload] + slot)


def oracle_arrays(arg):
    """The oracle's fetch_result() arrays for arg = (points, merge flags), and under "counts" the sizes f3ps_get_counts reports."""
    pts, flags = arg
    import oracle_py
    o = oracle_py.Oracle()
    o.set_vccs_params()
    o.set_merge_params(merge_impl=1, **flags)
    o.set_input(pts)
    o.run(0, bench.THRESHOLD)
    out = {n: o.array(n) for n in ARRAYS}
    S, M = len(o.array("sv_label")), len(out["merges_w"])
    out["counts"] = {"n_voxels": len(o.array("keys")), "n_supervoxels": S, "n_edges": len(o.array("edges_ab")), "n_merges": M,
                     "n_segments": S - M, "n_labeled": len(out["out_label"])}      # (what f3ps_get_counts reports after a merge)
    return out


def oracle_of_pool_frame(arg):
    """oracle_arrays of pool frame `slot` of `workload` (a worker process: it generates the frame itself)."""
    slot, workload = arg
    return oracle_arrays((pool_frame(slot, workload), bench.C3_FLAGS if workload == "c3" else bench.FLAGS))


def as_dumped(k, a):
    """What bench.dump_outputs writes for frame k's array a."""
    if a.shape[0] > bench.DUMP_ROWS:
        a = a[np.sort(np.random.default_rng(k).choice(a.shape[0], bench.DUMP_ROWS, replace=False))]
    return a if a.dtype == np.float32 else a.astype(np.float64)


def compare(name, got, want):
    """(ok, detail) of one dumped array against the oracle's, cut as dumped."""
    from test_gpu_parity import close_enough
    if got.shape != want.shape or got.dtype != want.dtype:
        return False, "shape/dtype %s %s, oracle %s %s" % (got.shape, got.dtype, want.shape, want.dtype)
    equal = (got == want) | (np.isnan(got) & np.isnan(want))
    n_diff = int((~equal).sum())
    if name == "merges_w":
        return close_enough(got, want), "%d of %d weights not bit-identical" % (n_diff, got.size)
    return n_diff == 0, "%d of %d entries differ" % (n_diff, got.size)


def check(out_dir, workload="c2", inflight=80, jobs=None):
    """Prints the verdicts; returns the number of mismatching (frame, array) pairs plus missing arrays."""
    found = dumped_frames(out_dir)
    if not found:
        print("%s: no frame<k>_<name>.npy files" % out_dir)
        return 1
    slots = sorted({frame_slot(k, inflight) for k in found})
    with ProcessPoolExecutor(max_workers=jobs or min(len(slots), os.cpu_count() or 1),
                             mp_context=multiprocessing.get_context("spawn")) as ex:
        ref = dict(zip(slots, ex.map(oracle_of_pool_frame, [(s, workload) for s in slots])))
    bad = 0
    for k in sorted(found):
        s = frame_slot(k, inflight)
        for name in ARRAYS:
            if name not in found[k]:
                print("frame %04d (pool frame %d) %-11s MISSING" % (k, s, name))
                bad += 1
                continue
            ok, detail = compare(name, np.load(found[k][name]), as_dumped(k, ref[s][name]))
            print("frame %04d (pool frame %d) %-11s %s  (%s)" % (k, s, name, "ok" if ok else "MISMATCH", detail))
            bad += not ok
    print("%d frames, %d arrays: %s" % (len(found), len(found) * len(ARRAYS), "all equal to the oracle" if not bad else "%d differ" % bad))
    return bad


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("dir", help="the directory bench.py --dump-outputs wrote")
    ap.add_argument("--workload", default="c2", choices=sorted(BASE_SEED), help="the workload bench.py ran (c5 is not covered)")
    ap.add_argument("--inflight", type=int, default=80, help="bench.py's --inflight of that run")
    ap.add_argument("--jobs", type=int, default=None, help="oracle worker processes (default: one per distinct frame, at most one per core)")
    args = ap.parse_args()
    import oracle_py
    oracle_py.build()
    return 1 if check(args.dir, args.workload, args.inflight, args.jobs) else 0


if __name__ == "__main__":
    sys.exit(main())
