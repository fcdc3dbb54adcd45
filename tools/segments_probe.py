"""Segment extraction on one GPU: f3ps_get_segment_points (device output) and f3ps_get_segment_info on the C5 room scan.

  python tools/segments_probe.py [--out profiles/segments_b200.json] [--sizes 10000000,50000000]

For each size (-v 0.01 -s 0.1, --CVX --AL) and L = 1 and 8 levels (thresholds 0.2 / L .. 0.2), level L-1 (the coarsest):
  points  f3ps_get_segment_points into torch buffers, grouping included: every call after a merge_levels groups again.  CUDA
          events around one call, median of 5 after 2 warm-up calls; a merge_levels between calls drops the kept grouping (the
          replay itself is outside the timed window).  The inputs (N x 32 B records, N x 4 B point_voxel) are larger than L2
          from 10 M points on.
  info    f3ps_get_segment_info right after f3ps_get_segment_points of the same level (the grouping is kept), host clock around
          a call that ends in a device synchronise, median of 5 after 2 warm-up calls.
  host    numpy's stable argsort path on the point labels (what a caller did before: labels out, argsort, cumulative bincount).
Algorithmic bytes (N points, N_lab of them in a segment, stride 32, passes = ceil(ceil(log2 K) / 8)):
  keys 4N + 4N + 8 N_lab, each radix pass 16 N_lab, offsets 4 N_lab, copy-out 8 N_lab (read + write), descriptors
  4 N_lab + 32 N_lab.  Achieved GB/s against the 6,536 GB/s copy peak of DESIGN.md section 3.  No target is implied.
The card's name and power limit are read in the same run and written with the numbers."""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "fast-3d-pointcloud-segmentation_b200"))

AL = dict(color_mode=0, geom_mode=1, merge_mode=1)
COPY_PEAK_GBS = 6536.0          # DESIGN.md section 3: measured copy bandwidth of the B200


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def probe(f3ps, torch, n):
    pts = f3ps.synth.make_room_scan(seed=50000, n_points=n)
    g = f3ps.Segmenter(device=0, stream=torch.cuda.current_stream().cuda_stream)      # the caller's stream, so events time the calls
    g.set_vccs_params(voxel_res=0.01, seed_res=0.1); g.set_merge_params(**AL)
    g.set_input(pts); g.extract(); g.graph()
    rows = []
    for L in (1, 8):
        thr = np.linspace(0.2 / L, 0.2, L).astype(np.float32)
        k = L - 1
        g.merge_levels(thr)
        K = int(g.levels()["n_segments"][k])
        off, _ = g.segment_points(k)
        n_lab = int(off[-1])
        t_off = torch.empty(K + 1, dtype=torch.int64, device="cuda"); t_idx = torch.empty(max(n_lab, 1), dtype=torch.int32, device="cuda")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        pts_ms, info_ms = [], []
        for rep in range(7):
            g.merge_levels(thr); g.levels(); g.voxel_labels()         # drops the kept grouping; level tables built outside the window
            torch.cuda.synchronize()
            e0.record()
            g.segment_points_device(k, t_off.data_ptr(), t_idx.data_ptr(), K + 1, t_idx.numel())
            e1.record(); torch.cuda.synchronize()
            t0 = time.perf_counter(); g.segment_info(k); t1 = time.perf_counter()
            if rep >= 2:
                pts_ms.append(e0.elapsed_time(e1)); info_ms.append((t1 - t0) * 1e3)
        pl = g.point_labels()[k]
        host = []
        for _ in range(3):
            t0 = time.perf_counter()
            lab = g.point_labels()[k]
            valid = lab != np.uint32(0xffffffff)
            np.cumsum(np.bincount(lab[valid], minlength=K)); np.nonzero(valid)[0][np.argsort(lab[valid], kind="stable")]
            host.append((time.perf_counter() - t0) * 1e3)
        del pl
        passes = max(1, math.ceil(max(1, math.ceil(math.log2(max(K, 2)))) / 8)) if K > 1 else 0
        bytes_points = 8 * n + 8 * n_lab + 16 * n_lab * passes + 4 * n_lab + 8 * n_lab
        bytes_info = 4 * n_lab + 32 * n_lab
        p_ms, i_ms = statistics.median(pts_ms), statistics.median(info_ms)
        rows.append({"points": n, "in_segments": n_lab, "levels": L, "level": k, "segments": K, "radix_passes": passes,
                     "segment_points_device_ms": p_ms, "points_algorithmic_bytes": bytes_points, "points_GB_s": bytes_points / p_ms / 1e6,
                     "points_share_of_copy_peak": bytes_points / p_ms / 1e6 / COPY_PEAK_GBS,
                     "segment_info_ms": i_ms, "info_descriptor_bytes": bytes_info, "info_GB_s": bytes_info / i_ms / 1e6,
                     "info_share_of_copy_peak": bytes_info / i_ms / 1e6 / COPY_PEAK_GBS,
                     "numpy_host_ms": statistics.median(host)})
        print(json.dumps(rows[-1]), flush=True)
        del t_off, t_idx
    del g
    torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "segments_b200.json"))
    ap.add_argument("--sizes", default="10000000,50000000")
    args = ap.parse_args()
    import torch
    import f3ps
    if not torch.cuda.is_available():
        sys.exit("segments_probe: no CUDA device; these numbers only come from a GPU run")
    torch.cuda.set_stream(torch.cuda.Stream())     # not the legacy stream (0): f3ps_create would make a private stream for that
    f3ps.build()
    res = {"card": card(), "torch_device": torch.cuda.get_device_name(0), "rows": []}
    for n in map(int, args.sizes.split(",")):
        res["rows"] += probe(f3ps, torch, n)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("card:", res["card"])


if __name__ == "__main__":
    main()
