"""Segmentation levels on one GPU: what merge_levels saves, the point-gather kernel's bandwidth, the level-table stages.

  python tools/levels_probe.py [--out profiles/levels_b200.json] [--big 50000000]

(a) C2 frame (640x480, --CVX --AL): merge_levels over the 41 auto-threshold values + voxel and point labels, against 41
    separate merges each followed by the host join (point_voxel + labelled cloud -> per-point labels).  Host clock around
    calls that end in a device synchronise, median of 5.
(b) level_point_labels_kernel on the C5 room scan (-v 0.01 -s 0.1) at 10 M and --big points, L = 1, 8 and (10 M only) 41:
    CUDA events around 50 launches after 5 warm-up launches, into a torch buffer; next to it a device-to-device copy of the
    same number of bytes, timed the same way.  Algorithmic bytes from shapes:
    4 N (point_voxel) + 4 L N (labels) + 4 Lp per point with a voxel (its table row, Lp = L padded to whole uint4s).
    The output is written once per launch (not re-read); the table is reused across launches and stays in L2 when it fits.
(c) the level-table stages (forest, prefix, dense, roots, voxel table) on C4 (10 M dense scene, --RGB --ML 0.5,
    -v 0.004 -s 0.04) and C5 (10 M room scan), from torch.profiler kernel times, next to the K7 kernel time.
The card's name and power limit are read in the same run and written with the numbers."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "fast-3d-pointcloud-segmentation_b200"))

AL = dict(color_mode=0, geom_mode=1, merge_mode=1)
RGB_ML = dict(color_mode=1, geom_mode=0, merge_mode=0, lam=0.5)
COPY_PEAK_GBS = 6536.0          # DESIGN.md section 3: measured copy bandwidth of the B200
STAGES = ("levels_forest_kernel", "levels_prefix_kernel", "levels_dense_kernel", "levels_roots_kernel", "levels_voxel_kernel")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def host_join(g, n_voxels):
    pv = g.array("point_voxel")
    r = g.fetch_result()
    vox = np.full(n_voxels, 0xffffffff, np.uint32)
    vox[r["out_voxel"]] = r["out_label"]
    return np.where(pv >= 0, vox[np.maximum(pv, 0)], np.uint32(0xffffffff))


def probe_a(f3ps):
    pts = f3ps.synth.make_frame(seed=20020)
    g = f3ps.Segmenter(); g.set_vccs_params(); g.set_merge_params(**AL); g.set_input(pts); g.extract(); g.graph()
    thr = f3ps.Segmenter.sweep_thresholds()
    V = g.counts().n_voxels

    def levels():
        g.merge_levels(thr); g.voxel_labels(); return g.point_labels()

    def separate():
        out = []
        for t in thr:
            g.merge(float(t)); out.append(host_join(g, V))
        return np.stack(out)

    res = {}
    for name, fn in (("merge_levels_ms", levels), ("separate_merges_ms", separate)):
        fn()
        ts = []
        for _ in range(5):
            t0 = time.perf_counter(); fn(); g.sync(); ts.append((time.perf_counter() - t0) * 1e3)
        res[name] = statistics.median(ts)
    res["levels"] = len(thr); res["points"] = len(pts)
    res["speedup"] = res["separate_merges_ms"] / res["merge_levels_ms"]
    return res


def build_c5(f3ps, torch, n):
    pts = f3ps.synth.make_room_scan(seed=50000, n_points=n)
    g = f3ps.Segmenter(device=0, stream=torch.cuda.current_stream().cuda_stream)      # the caller's stream, so events time the kernel
    g.set_vccs_params(voxel_res=0.01, seed_res=0.1); g.set_merge_params(**AL)
    g.set_input(pts); g.extract(); g.graph()
    return g, pts


def probe_b(f3ps, torch, big):
    rows = []
    for n in (10_000_000, big):
        g, pts = build_c5(f3ps, torch, n)
        c = g.counts(); pv = g.array("point_voxel"); valid = int((pv >= 0).sum())
        for L in (1, 8, 41):
            if L == 41 and n > 10_000_000:
                continue                                     # 41 x 50 M x 4 B does not belong in a default run
            thr = np.linspace(0.2 / L, 0.2, L).astype(np.float32)
            g.merge_levels(thr)
            out = torch.empty(L * n, dtype=torch.int32, device="cuda")
            for _ in range(5):
                g.point_labels_device(out.data_ptr(), out.numel())
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 50
            e0.record()
            for _ in range(reps):
                g.point_labels_device(out.data_ptr(), out.numel())
            e1.record(); torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / reps
            Lp = 1 if L == 1 else (L + 3) // 4 * 4
            bytes_ = 4 * n + 4 * L * n + 4 * Lp * valid
            # the same bytes as one device-to-device copy (half read, half written), timed the same way: what a launch of this
            # size reaches without the gather
            del out
            src = torch.empty(bytes_ // 8, dtype=torch.int32, device="cuda"); dst = torch.empty_like(src)
            for _ in range(5):
                dst.copy_(src)
            e0.record()
            for _ in range(reps):
                dst.copy_(src)
            e1.record(); torch.cuda.synchronize()
            copy_ms = e0.elapsed_time(e1) / reps
            del src, dst
            rows.append({"points": n, "voxels": int(c.n_voxels), "levels": L, "kernel_ms": ms, "algorithmic_bytes": bytes_,
                         "table_bytes": 4 * Lp * int(c.n_voxels), "GB_s": bytes_ / ms / 1e6, "share_of_copy_peak": bytes_ / ms / 1e6 / COPY_PEAK_GBS,
                         "same_bytes_copy_ms": copy_ms, "same_bytes_copy_share_of_copy_peak": bytes_ / copy_ms / 1e6 / COPY_PEAK_GBS})
        del g
        torch.cuda.empty_cache()
    return rows


def probe_c(f3ps, torch):
    from torch.profiler import ProfilerActivity, profile
    res = {}
    scenes = {"C4": (lambda: f3ps.synth.make_dense_scene(seed=40000), dict(voxel_res=0.004, seed_res=0.04), RGB_ML),
              "C5": (lambda: f3ps.synth.make_room_scan(seed=50000, n_points=10_000_000), dict(voxel_res=0.01, seed_res=0.1), AL)}
    for name, (make, vccs, mp) in scenes.items():
        pts = make()
        g = f3ps.Segmenter(); g.set_vccs_params(**vccs); g.set_merge_params(**mp); g.set_input(pts); g.extract(); g.graph()
        thr = f3ps.Segmenter.sweep_thresholds()
        g.merge_levels(thr); g.voxel_labels()                  # warm-up of every launch
        g.merge_levels(thr)
        k7 = g.stage_ms().get("merge_kernel")
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            g.levels(); g.voxel_labels(); g.sync()
        us = {s: 0.0 for s in STAGES}
        for ev in prof.key_averages():
            for s in STAGES:
                if s in ev.key:
                    us[s] += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        c = g.counts()
        res[name] = {"S": int(c.n_supervoxels), "V": int(c.n_voxels), "M": int(c.n_merges), "levels": len(thr), "merge_path": int(c.merge_path),
                     "k7_kernel_ms": k7, "stage_ms": {s: us[s] / 1e3 for s in STAGES}, "stages_total_ms": sum(us.values()) / 1e3}
        del g
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "levels_b200.json"))
    ap.add_argument("--big", type=int, default=50_000_000, help="points of the large leg of (b)")
    args = ap.parse_args()
    import torch
    import f3ps
    if not torch.cuda.is_available():
        sys.exit("levels_probe: no CUDA device; these numbers only come from a GPU run")
    torch.cuda.set_stream(torch.cuda.Stream())     # not the legacy stream (0): f3ps_create would make a private stream for that
    f3ps.build()
    res = {"card": card(), "torch_device": torch.cuda.get_device_name(0)}
    res["a_c2_41_levels"] = probe_a(f3ps); print(json.dumps(res["a_c2_41_levels"]), flush=True)
    res["b_point_gather"] = probe_b(f3ps, torch, args.big)
    for r in res["b_point_gather"]:
        print(json.dumps(r), flush=True)
    res["c_level_tables"] = probe_c(f3ps, torch); print(json.dumps(res["c_level_tables"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("card:", res["card"])


if __name__ == "__main__":
    main()
