#!/usr/bin/env python
"""bench.py -- headline benchmark of the supervoxel-plus-merging hot path (BASELINE.json).

Metric: Mpoints/s end-to-end segmentation (voxelize -> VCCS -> edge weights -> merge) on the
C2 workload: synthetic 640x480 RGB-D frames (307,200 points each, seed 20020 + k), flags
--CVX --AL -t 0.2.  Frames are independent (the reference's -d loop), and the serial merge stage of one frame
occupies one SM, so a sweep keeps many frames in flight.  A "step" is --rounds groups of --inflight frames through
f3ps/sweep.py: BatchPool -- K1..K6 of a frame on its own handle + stream, ONE launch of the resident merge kernel per
group (CTA i = frame i, f3ps_merge_batch), the next group's front stages overlapping it (--pool streams: one merge
kernel per stream instead).  The latency of one frame alone is reported beside it (`single_frame_latency_ms`, the
figure BASELINE.json's 2 ms target refers to).

  python bench.py --gpus N --steps K --warmup W            (our arm; torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K --warmup W   (CPU oracle port, rank 0 only)
  python bench.py --workload c5 [--points P] [--verify]    (BASELINE config 5: one cloud in slab mode, torchrun for N > 1)
  python bench.py ... --dump-outputs DIR                   (also write what the last timed step computed, see dump_outputs)

`value`  : frames resident in HBM before the timed region; CUDA events around each step (recorded after every
           handle's stream has drained), per-stage times from each handle's own events on its own stream.
`e2e`    : the same frames through the public API with HOST buffers (H2D of the points and D2H of the
           labelled voxel cloud + merge log inside the timed region).
Frames are sharded per GPU with no collective (SURVEY.md section 8e): every rank runs K
steps on its own frames ("weak" scaling); the time is the max over ranks.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "fast-3d-pointcloud-segmentation_b200"))

WORKLOAD = "C2: synthetic 640x480 RGB-D frame (307200 points), --CVX --AL -t 0.2"
FLAGS = dict(color_mode=0, geom_mode=1, merge_mode=1, lam=0.5, bins=500)
THRESHOLD = 0.2
# BASELINE config 3: the -d sweep, frames from the same generator with seeds 30000 + i, --EQ 200 -t 0.2 (SURVEY.md section 8d)
C3_WORKLOAD = "C3: synthetic VGA directory sweep (-d), frames seeded 30000+i, --EQ 200 -t 0.2"
C3_FLAGS = dict(color_mode=0, geom_mode=0, merge_mode=2, lam=0.5, bins=200)
N_POOL = 32                    # distinct synthetic frames per rank (replicated into the in-flight slots)
L2_FLUSH_BYTES = 512 << 20     # > 126 MB L2


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


TRAFFIC_FILE = os.path.join("profiles", "r02c_traffic.json")


def load_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel, per launch, from this round's ncu capture of the
    kernel the run dispatches (tools/k7_ncu.sh writes the report, tools/ncu_summary.py the JSON); None when absent."""
    try:
        with open(os.path.join(ROOT, TRAFFIC_FILE)) as f:
            return int(json.load(f)["traffic_bytes_per_launch"])
    except Exception:
        return None


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, enabled=True):
        self.index = index
        self.proc = None
        self.enabled = enabled          # one sampler per job (rank 0): eight nvidia-smi loops only perturb the launches they watch
        self.path = "/tmp/f3ps_clocks_%d.csv" % os.getpid()

    def start(self):
        if not self.enabled:
            return
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.proc:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, smax, reasons = [], [], set()
        try:
            for line in open(self.path):
                c = [x.strip() for x in line.split(",")]
                if len(c) < 9:
                    continue
                try:
                    sm.append(float(c[1])); smax.append(float(c[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.remove(self.path)
        except Exception:
            pass
        if sm:
            out = {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "reasons": sorted(reasons), "samples": len(sm)}
        return out


def make_frames(rank, count, base_seed=20020):
    from f3ps import synth
    return [synth.make_frame(seed=base_seed + rank * 1000 + i) for i in range(count)]


DUMP_FRAMES = 16        # --dump-outputs: the last frames of the last timed step
DUMP_ROWS = 1 << 15     # rows kept of one array of one frame


def dump_outputs(out_dir, results):
    """results: [(frame index within the step, Segmenter)].  Writes what Segmenter.fetch_result() hands a caller for each frame
    -- the labelled voxel cloud and the merge log -- as out_dir/frame<k>_<name>.npy: float32 stays float32, the uint32 arrays
    become float64 (exact).  An array of more than DUMP_ROWS rows keeps DUMP_ROWS of them, drawn by np.random.default_rng(k) and
    kept in order.  At most DUMP_FRAMES x 2 MiB = 32 MiB in all."""
    os.makedirs(out_dir, exist_ok=True)
    for k, seg in results:
        for name, a in seg.fetch_result().items():
            if a.shape[0] > DUMP_ROWS:
                a = a[np.sort(np.random.default_rng(k).choice(a.shape[0], DUMP_ROWS, replace=False))]
            np.save(os.path.join(out_dir, "frame%04d_%s.npy" % (k, name)), a if a.dtype == np.float32 else a.astype(np.float64))


def shared_config(workload):
    """The `config` both arms print (the driver compares the two dicts): what is measured, nothing about how."""
    flags = {"c2": "--CVX --AL -t 0.2", "c3": "--EQ 200 -t 0.2", "c5": "-v 0.01 -s 0.1 --CVX --AL -t 0.2"}[workload]
    name = {"c2": WORKLOAD, "c3": C3_WORKLOAD, "c5": C5_WORKLOAD}[workload]
    return {"workload": name, "flags": flags, "points_per_frame": 307200 if workload != "c5" else None}


# ------------------------------------------------------------------------------------------------
def run_reference(args):
    """CPU arm: the oracle port on the host cores, one frame per core per step (frames are independent
    in the reference: fresh SupervoxelClustering + Clustering per file, src/supervoxel_clustering.cpp:348,408)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py
    oracle_py.build()
    from concurrent.futures import ProcessPoolExecutor
    cores = os.cpu_count() or 1
    c3 = args.workload == "c3"
    flags = C3_FLAGS if c3 else FLAGS
    frames = make_frames(0, 1, 30000 if c3 else 20020)
    npts = len(frames[0])
    with ProcessPoolExecutor(max_workers=cores) as ex:
        def step():
            t0 = time.perf_counter()
            list(ex.map(_oracle_frame, [(frames[0], 1, flags)] * cores))
            return time.perf_counter() - t0
        for _ in range(args.warmup):
            step()
        times = [step() for _ in range(args.steps)]
    total = sum(times)
    value = cores * npts * args.steps / total / 1e6
    # the reference AS WRITTEN (std::multimap rebuilt per merge, contains() by value, src/clustering.cpp:431-468, 497-506): one frame, one core
    t_lit, _ = _oracle_frame((frames[0], 0, flags))
    line = {"impl": "reference", "impl_detail": "CPU oracle port (the reference as a whole needs PCL/OpenCV C++ and cannot be built here), stamp-based merge = same results as the literal std::multimap replay, ~30x faster -- the generous baseline: the reference's own Clustering class, compiled from its sources against container stand-ins (oracle/_ref), reproduces the same merge sequence and needs 35.8 s per VGA frame for K6 + K7 on one core", "metric": "Mpoints/s end-to-end segmentation", "value": value, "unit": "Mpoints/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": shared_config(args.workload if args.workload in ("c2", "c3") else "c2"), "run": {"frames_per_step": cores},
            "cpu_baseline": {"value": value, "unit": "Mpoints/s", "cores": cores, "kind": "port",
                             "sample": "%d VGA frames per step, one per core, CPU oracle with the stamp-based merge "
                                       "(identical results to the literal std::multimap replay, which is ~30x slower)" % cores,
                             "literal_replay": {"value": npts / t_lit / 1e6, "unit": "Mpoints/s", "cores": 1,
                                                "all_cores_estimate": cores * npts / t_lit / 1e6,
                                                "sample": "1 VGA frame, the merge loop exactly as the reference writes it: %.2f s" % t_lit}},
            "e2e": {"value": value, "unit": "Mpoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


def _oracle_frame(arg):
    pts, merge_impl, FLAGS = arg
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py
    o = oracle_py.Oracle()
    o.set_vccs_params()
    o.set_merge_params(merge_impl=merge_impl, **FLAGS)
    o.set_input(pts)
    t0 = time.perf_counter()
    o.run(0, THRESHOLD)
    return time.perf_counter() - t0, o.array("stage_ms")


def cpu_baseline(frame, FLAGS=FLAGS):
    """Rank 0, N=1: the literal CPU oracle (std::multimap replay, as the reference is written) on one frame."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py
    oracle_py.build()
    t_lit, st_lit = _oracle_frame((frame, 0, FLAGS))
    t_fix, st_fix = _oracle_frame((frame, 1, FLAGS))
    n = len(frame)
    return {"value": n / t_lit / 1e6, "unit": "Mpoints/s", "cores": 1, "kind": "port",
            "sample": "1 VGA frame (307200 points), single thread, literal std::multimap merge replay: %.2f s" % t_lit,
            "stage_ms": {k: round(float(v), 3) for k, v in zip(["voxelize", "neighbors", "normals", "seeds", "expand", "graph", "merge", "total"], st_lit)},
            "fixed_merge_value": n / t_fix / 1e6,
            "fixed_merge_note": "same oracle with the stamp-based merge (identical results): %.3f s/frame" % t_fix,
            "host_cores_available": os.cpu_count()}


# ------------------------------------------------------------------------------------------------
def sweep_leg(args, env, workload, steps, dump_dir=None):
    """One measured leg of the frame sweep (C2 or C3): resident throughput, host-buffer throughput, single-frame latency.
    dump_dir: rank 0 writes the results of the last timed step's final frames there (dump_outputs)."""
    import torch
    import f3ps
    from f3ps import sweep
    dist, world, rank, local_rank, dev = env
    flags = C3_FLAGS if workload == "c3" else FLAGS
    F = max(1, args.inflight)                 # frames in flight per GPU
    R = max(1, args.rounds)                   # frames each handle processes back to back inside one step
    n_distinct = min(N_POOL, F)
    frames = make_frames(rank, n_distinct, 30000 if workload == "c3" else 20020)
    npts = len(frames[0])
    # one resident copy per in-flight slot: a step streams F * 9.8 MB of distinct input (> L2 for F >= 13)
    d_frames = [torch.from_numpy(frames[i % n_distinct].view(np.uint8).reshape(-1, 32).copy()).to(dev) for i in range(F)]
    pinned = [torch.from_numpy(frames[i % n_distinct].view(np.uint8).reshape(-1, 32).copy()).pin_memory() for i in range(F)]
    host_views = [pinned[i % F].numpy().view(f3ps.synth.POINT_DTYPE).reshape(-1) for i in range(F * R)]
    ptrs = [d_frames[i % F].data_ptr() for i in range(F * R)]
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    if args.pool == "batch":
        # groups of F frames: K1..K6 per frame on its own handle / stream, ONE merge launch per group (CTA i = frame i)
        pool = sweep.BatchPool(batch=F, workers=args.workers or None, device=local_rank, merge=flags, threshold=THRESHOLD, expand_ctas=-args.expand_ctas, expand_cluster=args.expand_cluster)
    else:
        pool = sweep.FramePool(F, device=local_rank, merge=flags, threshold=THRESHOLD)
    stream = torch.cuda.current_stream()

    out_bytes = [0]

    def collect(seg, k):
        r = seg.fetch_result()                       # labelled voxel cloud (xyz, label, voxel index) + merge log (a, b, w, left)
        out_bytes[0] = sum(a.nbytes for a in r.values())
        return int(r["out_label"].shape[0])

    for _ in range(max(args.warmup, 3)):
        pool.run(ptrs, on_device=True, npts=npts)
    torch.cuda.synchronize()

    sampler = ClockSampler(local_rank, enabled=rank == 0)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    launches0 = sum(s.launch_count() for s in pool.segs)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    stage_acc = {}
    wall0 = time.perf_counter()
    for k in range(steps):
        flush.fill_(k & 0xff)                  # L2 flush between timed iterations (outside the events)
        torch.cuda.synchronize()
        ev[k][0].record(stream)
        pool.run(ptrs, on_device=True, npts=npts)     # joins when every handle's stream has drained
        ev[k][1].record(stream)
        torch.cuda.synchronize()
        for seg in pool.segs:                         # per-stage CUDA-event times of each handle's frame, on its own stream
            for name, ms in seg.stage_ms().items():
                stage_acc[name] = stage_acc.get(name, 0.0) + ms
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    wall = time.perf_counter() - wall0
    launches = sum(s.launch_count() for s in pool.segs) - launches0
    clocks = sampler.stop()
    t_dev = sum(a.elapsed_time(b) for a, b in ev) / 1e3          # seconds, this rank
    counts = pool.segs[0].counts()
    if dump_dir and rank == 0:
        # the handle that ran frame k of a step: BatchPool alternates two sets of F handles between groups of F frames,
        # FramePool deals the frames round-robin over its F handles; each handle still holds the last frame it ran
        last = {(k // F % 2 * F if args.pool == "batch" else 0) + k % F: k for k in range(F * R)}
        dump_outputs(dump_dir, sorted((k, pool.segs[h]) for h, k in last.items())[-DUMP_FRAMES:])

    # end-to-end through the public API with host buffers (H2D of the points, D2H of the labelled cloud + merge log)
    for i in range(2):
        pool.run(host_views, collect=collect)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for k in range(steps):
        pool.run(host_views, collect=collect)
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0

    # one frame alone on one stream: the latency the 2 ms target of BASELINE.json speaks about
    solo = pool.segs[0]
    lat = []
    for k in range(7):
        flush.fill_(k)
        torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        solo.set_blocking_wait(False)
        solo.set_expand_kernel(0, 0); solo.set_expand_sharing(0, 0)   # one frame alone: K5 as the cooperative grid over the whole GPU (the pool runs small clusters)
        solo.set_input_device(ptrs[k % F], npts, 32); solo.run(THRESHOLD)
        e1.record(stream); torch.cuda.synchronize()
        lat.append(e0.elapsed_time(e1))
    solo_stage = solo.stage_ms()
    solo_counts = solo.counts()

    tmax = torch.tensor([t_dev, t_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    t_dev_max, t_e2e_max = float(tmax[0]), float(tmax[1])
    n_segs = len(pool.segs)
    pool.close()
    del d_frames, pinned, flush
    n_frames = F * R * steps
    return dict(F=F, R=R, npts=npts, n_distinct=n_distinct, steps=steps, n_frames=n_frames, t_dev=t_dev_max, t_e2e=t_e2e_max,
                value=npts * n_frames * world / t_dev_max / 1e6, e2e=npts * n_frames * world / t_e2e_max / 1e6,
                counts=counts, solo_counts=solo_counts, stage_ms={k: v / (n_segs * steps) for k, v in stage_acc.items()},
                solo_stage=solo_stage, lat=lat, launches=int(launches), clocks=clocks, wall=wall, out_bytes=int(out_bytes[0]), frame0=frames[0])


def run_ours(args):
    os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")     # before the CUDA context exists (see f3ps_create)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cpu = None
    if world == 1 and rank == 0 and not args.no_cpu:
        # the CPU legs run BEFORE any GPU work, so the GPU-busy window of this process is the measurement alone
        try:
            cpu = cpu_baseline(make_frames(0, 1, 30000 if args.workload == "c3" else 20020)[0], C3_FLAGS if args.workload == "c3" else FLAGS)
        except Exception as e:     # the oracle is a checker; its absence must not hide the GPU number
            cpu = {"value": None, "unit": "Mpoints/s", "cores": 1, "kind": "port", "sample": "failed: %r" % (e,)}
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the f3ps path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    env = (dist, world, rank, local_rank, dev)
    m = sweep_leg(args, env, args.workload, args.steps, args.dump_outputs)
    c3 = sweep_leg(args, env, "c3", max(2, args.steps // 2)) if (args.workload == "c2" and not args.no_c3) else None

    if rank == 0:
        peak, peak_src = load_peaks()
        counts, F, R, npts = m["counts"], m["F"], m["R"], m["npts"]
        V, M = counts.n_voxels, counts.n_merges
        stage_ms = m["stage_ms"]
        # dominant kernel = the persistent merge kernel (K7); algorithmic bytes per launch (DESIGN.md):
        # 12 E (edge list) + 40 S (region statistics) + 12 M (merge log) + 16 * fold_steps (voxels streamed by the folds)
        sc = m["solo_counts"]
        solo_merge_ms = m["solo_stage"].get("merge_kernel", m["solo_stage"].get("merge", 0.0))
        alg_bytes = 12 * sc.n_edges + 40 * sc.n_supervoxels + 12 * sc.n_merges + 16 * sc.fold_steps
        ach = alg_bytes / (solo_merge_ms * 1e-3) / 1e9 if solo_merge_ms > 0 else 0.0
        e2e_bytes = 16 * npts + 16 * V + 12 * M
        t_frame = m["t_dev"] / m["n_frames"]
        traffic = load_traffic()
        line = {
            "metric": "Mpoints/s end-to-end segmentation", "value": m["value"], "unit": "Mpoints/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": m["t_dev"] / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": shared_config(args.workload),
            "run": {"step": ("%d frames per GPU in groups of %d: K1..K6 of a frame on its own handle + stream, ONE resident-merge launch "
                             "per group (CTA i = frame i), the next group's front stages overlap it (BatchPool); the reference's -d loop "
                             "processes independent files" % (F * R, F)) if args.pool == "batch" else
                            ("%d frames per GPU, %d in flight (one handle + stream each, %d frames back to back per handle; "
                             "the reference's -d loop processes independent files)" % (F * R, F, R)),
                    "pool": args.pool, "frames_per_step_per_gpu": F * R, "frames_in_flight_per_gpu": F, "distinct_frames": m["n_distinct"],
                    "l2": "L2 flushed (512 MB write) between timed steps; a step streams %d MB of input" % (F * R * npts * 32 >> 20),
                    "sharding": "frames per GPU, no collective",
                    "V": int(V), "S": int(counts.n_supervoxels), "E": int(counts.n_edges), "M": int(M)},
            "e2e": {"value": m["e2e"], "unit": "Mpoints/s", "h2d_bytes_per_step": F * R * npts * 32, "d2h_bytes_per_step": m["out_bytes"] * F * R},
            "gpu_launches": m["launches"],
            "clocks": m["clocks"],
            "ms_per_frame": t_frame * 1e3,
            "single_frame_latency_ms": {"median": statistics.median(m["lat"]), "min": min(m["lat"]),
                                        "stage_ms": {k: round(v, 4) for k, v in m["solo_stage"].items()},
                                        "us_per_merge": 1e3 * solo_merge_ms / max(1, sc.n_merges)},
            "stage_ms": {k: round(v, 4) for k, v in stage_ms.items()},
            "roofline": {"bound": "hbm", "kernel": "merge_fast_kernel (K7, one persistent CTA per frame; a serial dependency chain, not a bandwidth "
                                                   "problem: its HBM fraction is ~1e-5 by construction, the figure to read is us_per_merge; DESIGN.md section 3.7)",
                         "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                         "traffic_source": TRAFFIC_FILE if traffic is not None else None, "peak_source": peak_src,
                         "timed": "the kernel's own CUDA events on its stream, one frame alone (%.3f ms for %d merges)" % (solo_merge_ms, sc.n_merges),
                         "algorithmic_bytes_per_launch": int(alg_bytes),
                         "merge_path": int(sc.merge_path),
                         "e2e_algorithmic_bytes": e2e_bytes,
                         "e2e_achieved_gbs": e2e_bytes / t_frame / 1e9 if t_frame > 0 else 0.0,
                         "e2e_frac": e2e_bytes / t_frame / 1e9 / peak if t_frame > 0 else 0.0},
            "wall_s": m["wall"],
        }
        if c3 is not None:
            line["c3"] = {"config": shared_config("c3"), "value": c3["value"], "unit": "Mpoints/s", "e2e": c3["e2e"], "steps": c3["steps"],
                          "ms_per_frame": c3["t_dev"] / c3["n_frames"] * 1e3, "M": int(c3["counts"].n_merges),
                          "single_frame_latency_ms": statistics.median(c3["lat"]), "stage_ms": {k: round(v, 4) for k, v in c3["stage_ms"].items()}}
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


# ------------------------------------------------------------------------------------------------
C5_WORKLOAD = "C5: synthetic merged room scan, -v 0.01 -s 0.1 --CVX --AL -t 0.2, spatial slabs (Morton-key ranges) over the GPUs"
C5_VCCS = dict(voxel_res=0.01, seed_res=0.1)


def run_slab(args):
    """BASELINE config 5: ONE cloud cut into slabs over the GPUs (strong scaling).  Every rank starts with the scans it
    'recorded' (a contiguous share of the 40 scan positions) resident in HBM; a step is the whole path on the whole
    cloud, exchanges included (f3ps/slab.py); the time is the max over ranks of the CUDA-event time of the step."""
    import torch
    import torch.distributed as dist
    import f3ps
    from f3ps import slab, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the f3ps path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    comm = slab.Comm(dist if world > 1 else None, torch)
    pts = synth.make_room_scan(seed=50000, n_points=args.points, scans=synth.room_scan_share(rank, world))
    n_local = int(pts.shape[0])
    d_pts = torch.from_numpy(pts.view(np.uint8).reshape(-1, 32)).to(dev)
    del pts
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    ss = slab.SlabSegmenter(comm, device=local_rank, vccs=C5_VCCS, merge=FLAGS)
    for _ in range(max(1, args.warmup)):
        ss.run((d_pts.data_ptr(), n_local, 32), THRESHOLD)
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank, enabled=rank == 0)
    if world > 1:
        dist.barrier()
    sampler.start()
    times, stage = [], {}
    launches0 = ss.seg.launch_count()
    bytes0 = comm.bytes_moved
    for k in range(args.steps):
        flush.fill_(k & 0xff)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        info = ss.run((d_pts.data_ptr(), n_local, 32), THRESHOLD)
        times.append(info["stage_ms"]["total"])
        for name, ms in info["stage_ms"].items():
            stage[name] = stage.get(name, 0.0) + ms / args.steps
    torch.cuda.synchronize()
    launches = ss.seg.launch_count() - launches0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, [(0, ss.seg)])              # every rank holds the whole cloud's result
    keys = sorted(stage)
    t = torch.tensor([sum(times) / 1e3] + [stage[k] for k in keys], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    c = ss.seg.counts()
    verified = None
    if args.verify:
        # every rank compares its (complete) slab result with one plain handle processing the whole cloud on its own GPU
        full = synth.make_room_scan(seed=50000, n_points=args.points)
        ref = f3ps.Segmenter(device=local_rank)
        ref.set_vccs_params(**C5_VCCS); ref.set_merge_params(**FLAGS)
        ref.set_input(full); ref.run(THRESHOLD)
        names = ["keys", "voxel_xyz", "normals", "seeds", "labels", "dist", "edges_ab", "edges_w", "merges_ab", "merges_w", "out_label"]
        bad = [n for n in names if not np.array_equal(ss.seg.array(n), ref.array(n), equal_nan=ref.array(n).dtype.kind == "f")]
        okt = torch.tensor([0 if bad else 1], dtype=torch.int32, device=dev)
        if world > 1:
            dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        verified = {"identical_to_single_handle_on_every_rank": bool(int(okt[0])), "arrays": names, "differing_on_rank0": bad}
        ref.close(); del full
    if rank == 0:
        peak, peak_src = load_peaks()
        t_total = float(t[0])
        value = args.points * args.steps / t_total / 1e6
        V, M = int(c.n_voxels), int(c.n_merges)
        e2e_bytes = 16 * args.points + 16 * V + 12 * M
        t_step = t_total / args.steps
        line = {"metric": "Mpoints/s end-to-end segmentation", "value": value, "unit": "Mpoints/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(1, args.warmup), "ms_per_step": t_step * 1e3, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": dict(shared_config("c5"), points=args.points), "run": {"points": args.points, "V": V, "S": int(c.n_supervoxels), "E": int(c.n_edges), "M": M,
                           "nan_weights": int(c.nan_weights), "rounds": int(c.rounds), "sweeps": int(info["sweeps"]),
                           "own_slice_rank0": list(info["own"]), "l2": "L2 flushed between steps; the cloud is %d MB" % (args.points * 32 >> 20),
                           "sharding": "slabs = Morton-key ranges; K1/K3/K5 sweeps sharded, K2/K4/K6 on replicated tables, K7 replicas only"},
                "stage_ms_max_over_ranks": {k: round(float(v), 3) for k, v in zip(keys, t[1:].tolist())},
                "exchanged_bytes_per_step_rank0": int((comm.bytes_moved - bytes0) / args.steps),
                "gpu_launches": int(launches), "clocks": clocks, "verified": verified,
                "roofline": {"bound": "hbm", "kernel": "whole path (no single dominant kernel at this size; per-stage figures in profiles/)",
                             "achieved": e2e_bytes / t_step / 1e9, "peak": peak, "unit": "GB/s", "frac": e2e_bytes / t_step / 1e9 / peak,
                             "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_launch": e2e_bytes}}
        print(json.dumps(line))
    ss.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--inflight", type=int, default=80, help="frames per merge grid (batch pool) / frames in flight per GPU (streams pool); measured on one B200, C2: 48 -> 338, 64 -> 401, 72 -> 422, 80 -> 435, 96 -> 394 Mpoints/s resident (a merge CTA holds its SM for ~26 ms: 80 of them leave 68 SMs to the front stages of the next group)")
    ap.add_argument("--rounds", type=int, default=10, help="groups per step (batch pool) / frames each handle runs back to back inside one step (streams pool)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg (development)")
    ap.add_argument("--pool", default="batch", choices=["batch", "streams"], help="batch: one merge launch per group of --inflight frames; streams: one merge kernel per stream")
    ap.add_argument("--expand-cluster", type=int, default=8, help="batch pool: K5 of a frame as one thread-block cluster of this many CTAs (0 = cooperative grid, see --expand-ctas)")
    ap.add_argument("--expand-ctas", type=int, default=24, help="batch pool: cap of the cooperative K5 grid per frame (0 = one voxel per thread)")
    ap.add_argument("--workers", type=int, default=32, help="host threads for the front stages of a group (batch pool)")
    ap.add_argument("--workload", default="c2", choices=["c2", "c3", "c5"], help="c2: frames in flight, --CVX --AL (the headline; a short C3 leg rides along); c3: the --EQ 200 directory sweep; c5: one large cloud in slab mode")
    ap.add_argument("--no-c3", action="store_true", help="c2: skip the C3 leg")
    ap.add_argument("--points", type=int, default=50_000_000, help="c5: points of the merged scan")
    ap.add_argument("--verify", action="store_true", help="c5: compare the slab result with one handle processing the whole cloud")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the labelled voxel clouds and merge logs of the "
                    "last step's final %d frames (c5: of the cloud) as DIR/frame<k>_<name>.npy, rows sampled beyond %d" % (DUMP_FRAMES, DUMP_ROWS))
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes what the GPU path computed; the reference arm has none")
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "c5":
        return run_slab(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
