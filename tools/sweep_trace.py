#!/usr/bin/env python
"""Does a pipelined sweep overlap the next group's front stages (K1..K6) with the current group's merge grid?

Runs BatchPool as bench.py configures it (C2 frames resident on the device, groups of --batch frames, --workers front-stage
threads, K5 as one cluster of --cluster CTAs per frame), warms up, then traces --groups groups with torch.profiler (CUDA
activities) and prints, for every group g that has a successor:
  - the interval of grid g (merge_fast_batch_kernel);
  - the share of group g+1's front-stage kernel time that falls inside that interval;
  - when group g+1's first and last K5 (expand_cluster_kernel) ran, relative to the start of grid g.
The raw kernel records (name, stream, start, end in microseconds) go to OUT/sweep_trace_<tag>.json.

  python tools/sweep_trace.py --out DIR [--tag T] [--batch 80] [--workers 32] [--cluster 8] [--groups 4] [--warmup 3]

Which group a front-stage kernel belongs to comes from its stream: BatchPool alternates two handle sets, group g runs on set
g % 2, and every handle has its own stream.  The set-0 streams are the first `batch` streams to run a kernel in the traced
window (group 0's fronts end before group 1's begin).  A kernel on a set-X stream belongs to the first group of parity X whose
grid starts after the kernel started."""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "fast-3d-pointcloud-segmentation_b200"))
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")     # before the CUDA context exists, as bench.py does

GRID = "merge_fast_batch_kernel"
K5 = "expand_cluster_kernel"
# what follows a merge grid (on the members' streams before the batched tail, on the lead's stream after it): not front stages
TAIL = ("dense_label", "labeled_cloud", "scalars_gather")


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:
        return "nvidia-smi failed: %r" % (e,)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tag", default="run")
    ap.add_argument("--out", required=True, help="directory for the kernel records")
    ap.add_argument("--batch", type=int, default=80)
    ap.add_argument("--workers", type=int, default=32)
    ap.add_argument("--cluster", type=int, default=8)
    ap.add_argument("--groups", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()

    import numpy as np
    import torch
    from torch.profiler import ProfilerActivity, profile
    import bench
    from f3ps import sweep

    F = args.batch
    frames = bench.make_frames(0, min(bench.N_POOL, F))
    npts = len(frames[0])
    d_frames = [torch.from_numpy(frames[i % len(frames)].view(np.uint8).reshape(-1, 32).copy()).cuda() for i in range(F)]
    torch.cuda.synchronize()
    pool = sweep.BatchPool(batch=F, workers=args.workers, merge=bench.FLAGS, threshold=bench.THRESHOLD, expand_cluster=args.cluster)
    ptrs_w = [d_frames[i % F].data_ptr() for i in range(F * args.warmup)]
    ptrs = [d_frames[i % F].data_ptr() for i in range(F * args.groups)]
    pool.run(ptrs_w, on_device=True, npts=npts)
    torch.cuda.synchronize()

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        pool.run(ptrs, on_device=True, npts=npts)
        torch.cuda.synchronize()
    pool.close()
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    recs = sorted(((e["name"], int(e["args"]["stream"]), float(e["ts"]), float(e["ts"]) + float(e["dur"]))
                   for e in events if e.get("cat") == "kernel"), key=lambda r: r[2])
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "sweep_trace_%s.json" % args.tag), "w") as f:
        json.dump({"card": card(), "batch": F, "workers": args.workers, "cluster": args.cluster, "groups": args.groups,
                   "kernels": [{"name": n, "stream": s, "start": a, "end": b} for n, s, a, b in recs]}, f)

    grids = [r for r in recs if GRID in r[0]]
    if len(grids) != args.groups:
        raise SystemExit("expected %d merge grids in the trace, found %d" % (args.groups, len(grids)))
    front = [r for r in recs if GRID not in r[0] and not any(t in r[0] for t in TAIL)]
    first_seen = {}
    for n, s, a, b in front:
        first_seen.setdefault(s, a)
    streams = sorted(first_seen, key=first_seen.get)
    if len(streams) != 2 * F:
        print("note: %d streams ran front-stage kernels (expected %d)" % (len(streams), 2 * F))
    parity = {s: (0 if k < F else 1) for k, s in enumerate(streams)}
    by_group = [[] for _ in grids]
    for r in front:
        p = parity[r[1]]
        g = next((g for g in range(p, len(grids), 2) if grids[g][2] > r[2]), None)
        if g is not None:
            by_group[g].append(r)

    print("card: %s" % card())
    print("BatchPool batch=%d workers=%d cluster=%d, %d traced groups; times in ms, relative to the start of grid g" % (
        F, args.workers, args.cluster, args.groups))
    print("%3s %22s %10s %9s %16s %16s %8s" % ("g", "grid g [start, end]", "grid ms", "share", "g+1 first K5", "g+1 last K5 end", "frames"))
    t0 = grids[0][2]
    shares = []
    for g in range(len(grids) - 1):
        gs, ge = grids[g][2], grids[g][3]
        nxt = by_group[g + 1]
        tot = sum(b - a for _, _, a, b in nxt)
        inside = sum(max(0.0, min(b, ge) - max(a, gs)) for _, _, a, b in nxt)
        k5 = [r for r in nxt if K5 in r[0]]
        share = inside / tot if tot > 0 else 0.0
        shares.append(share)
        print("%3d %10.2f, %9.2f %10.2f %8.1f%% %16s %16s %8d" % (
            g, (gs - t0) / 1e3, (ge - t0) / 1e3, (ge - gs) / 1e3, 100 * share,
            "%.2f" % ((k5[0][2] - gs) / 1e3) if k5 else "-", "%.2f" % ((max(r[3] for r in k5) - gs) / 1e3) if k5 else "-", len(k5)))
    span = (max(r[3] for r in recs) - min(r[2] for r in recs)) / 1e3
    print("traced window %.2f ms for %d frames = %.3f ms/frame; mean share %.1f%%" % (
        span, F * args.groups, span / (F * args.groups), 100 * sum(shares) / max(1, len(shares))))


if __name__ == "__main__":
    main()
