"""The benchmark's batched sweep, frame by frame, against the CPU oracle at the configuration bench.py measures: BatchPool with
80 frames per merge grid, two alternating handle sets, 32 front-stage threads, K5 as one 8-CTA cluster per frame, input
resident on the device (f3ps_set_input with on_device=1, stride 32), merges in merge_fast_batch_kernel and the batched tail
kernels.  Besides: the host-buffer (e2e) leg, the single-frame latency leg on a handle that ran the sweep, one f3ps_merge_batch
call over three parameter blocks with odd members in the later ones, and a mixed group whose handles grow and shrink between
rounds.

Every frame's fetch_result() and counts() are compared with the oracle (stamp-based merge, the reference's Clustering
sequence): merge pairs, regions left and the labelled cloud exactly, merge weights with test_gpu_parity.close_enough (FP64
libm on the host and on the device differ in the last bit now and then).  Each configuration runs once."""
import multiprocessing
import os
import sys
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

import bench
from test_gpu_parity import close_enough, hub_graph, same

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import check_bench_dump  # noqa: E402  (oracle_arrays: the oracle's fetch_result() arrays and counts of one frame)

# bench.py's argparse defaults (main()): they cannot be imported
INFLIGHT = 80            # --inflight, bench.py:524
EXPAND_CLUSTER = 8       # --expand-cluster, bench.py:528
EXPAND_CTAS = 24         # --expand-ctas, bench.py:529 (BatchPool gets -24)
WORKERS = 32             # --workers, bench.py:530
ROUNDS = 3               # groups per pool.run here: set 0 runs again while set 1's grid is in flight
THR = bench.THRESHOLD
RGB_ML = dict(color_mode=1, geom_mode=0, merge_mode=0, lam=0.5)     # --RGB --ML 0.5 (BASELINE config 4's merge flags)

EXACT = ("merges_ab", "merges_left", "out_label", "out_voxel", "out_xyz")
COUNTS = ("n_voxels", "n_supervoxels", "n_edges", "n_merges", "n_segments", "n_labeled")
SMALL_SEEDS = [2000 + i for i in range(210)]       # 160x120 frames: three parameter blocks of merge_batch, the mixed group
PHANTOM = 52                                        # 160x120 seed whose phantom leaf survives (test_gpu_parity.test_phantom_seed_leaves)
TRIPLE_SEEDS = (22030, 22049)                       # VGA frames with three seed cells on one voxel
LARGE_SEED = 777                                    # the 1280x960 frame of test_larger_frame_against_fast_oracle


def edge_clouds(S):
    """The clouds of test_gpu_parity.test_edge_cases_empty_nan_single: empty, all-NaN, one point, five points."""
    return [np.zeros(0, S.POINT_DTYPE),
            S.pack_points(np.full((300, 3), np.nan, np.float32), np.zeros(300, np.uint32)),
            S.pack_points(np.array([[0.1, 0.2, 1.0]], np.float32), np.array([0x00ff8040], np.uint32)),
            S.pack_points(np.array([[0.1, 0.2, 1.0], [0.1, 0.2, 1.0], [np.nan, 0, 1], [0.5, 0.5, 0.0], [0.3, 0.1, 2.0]], np.float32),
                          np.arange(5, dtype=np.uint32) * 0x00101010)]


def mismatches(got, c, want, where):
    """Failure lines of one frame: fetch_result() `got` and counts() `c` against the oracle's `want`; [] when it matches.
    The second value is the number of merge weights that are not bit-identical."""
    bad = []
    for n in EXACT:
        if not same(got[n], want[n]):
            bad.append("%s %s: %s vs oracle %s%s" % (where, n, got[n].shape, want[n].shape,
                                                     "" if got[n].shape != want[n].shape else ", %d entries differ" % int((got[n] != want[n]).sum())))
    a, b = got["merges_w"], want["merges_w"]
    off_bits = int((~((a == b) | (np.isnan(a) & np.isnan(b)))).sum()) if a.shape == b.shape else -1
    if not close_enough(a, b):
        bad.append("%s merges_w: beyond close_enough, %d of %d weights not bit-identical" % (where, off_bits, b.size))
    for n in COUNTS:
        if getattr(c, n) != want["counts"][n]:
            bad.append("%s counts().%s = %d, oracle %d" % (where, n, getattr(c, n), want["counts"][n]))
    return bad, max(off_bits, 0)


def report(bad, n_frames, off_bits):
    assert not bad, "%d mismatches over %d frames (%d merge weights not bit-identical in all):\n%s" % (
        len(bad), n_frames, off_bits, "\n".join(bad[:40]))


@pytest.fixture(scope="module")
def gpu():
    import f3ps
    f3ps.build()
    return f3ps


@pytest.fixture(scope="module")
def inputs(gpu):
    S = gpu.synth
    return {"c2": bench.make_frames(0, bench.N_POOL), "c3": bench.make_frames(0, bench.N_POOL, 30000),
            "small": [S.make_frame(seed=s, width=160, height=120) for s in SMALL_SEEDS],
            "phantom": S.make_frame(seed=PHANTOM, width=160, height=120),
            "triple": [S.make_frame(seed=s) for s in TRIPLE_SEEDS],
            "large": S.make_frame(seed=LARGE_SEED, width=1280, height=960),
            "edge": edge_clouds(S)}


@pytest.fixture(scope="module")
def oracle(inputs):
    """The oracle's result of every distinct frame of this module, computed once in worker processes (spawned: this process
    has a CUDA context) while the GPU tests run; oracle(key)[i] waits for it."""
    import oracle_py
    oracle_py.build()
    jobs = {"c2": [(f, bench.FLAGS) for f in inputs["c2"]], "c3": [(f, bench.C3_FLAGS) for f in inputs["c3"]],
            "small": [(f, bench.FLAGS) for f in inputs["small"]], "phantom": [(inputs["phantom"], bench.FLAGS)],
            "triple": [(f, bench.FLAGS) for f in inputs["triple"]], "large": [(inputs["large"], bench.FLAGS)],
            "edge": [(f, bench.FLAGS) for f in inputs["edge"]], "c2_rgb_ml": [(f, RGB_ML) for f in inputs["c2"]]}
    with ProcessPoolExecutor(max_workers=os.cpu_count() or 1, mp_context=multiprocessing.get_context("spawn")) as ex:
        fut = {k: [ex.submit(check_bench_dump.oracle_arrays, j) for j in js] for k, js in jobs.items()}
        yield lambda key: [f.result() for f in fut[key]]


def device_copies(torch, frames):
    """sweep_leg's resident input: one device copy per in-flight slot, slot i holding frames[i % len(frames)]."""
    return [torch.from_numpy(frames[i % len(frames)].view(np.uint8).reshape(-1, 32).copy()).to("cuda") for i in range(INFLIGHT)]


def bench_pool(sweep, flags):
    return sweep.BatchPool(batch=INFLIGHT, workers=WORKERS, expand_ctas=-EXPAND_CTAS, expand_cluster=EXPAND_CLUSTER, merge=flags, threshold=THR)


def sweep_and_compare(pool, inputs_, want, on_device=False, npts=None):
    """One pool.run over ROUNDS groups; frame k is want[(k % INFLIGHT) % len(want)].  Compares inside collect (on the pool's
    reader threads, while the other set's front stages run) and checks that frame k ran on slot k % INFLIGHT of set
    (k // INFLIGHT) % 2 and on the batch kernel."""
    n_distinct = len(want)

    def collect(seg, k):
        g, slot = k // INFLIGHT, k % INFLIGHT
        where = "frame %d (group %d, set %d, slot %d, pool frame %d)" % (k, g, g % 2, slot, slot % n_distinct)
        c = seg.counts()
        bad, off = mismatches(seg.fetch_result(), c, want[slot % n_distinct], where)
        if seg is not pool.sets[g % 2][slot]:
            bad.append("%s ran on handle %d" % (where, pool.segs.index(seg)))
        if c.merge_path != 1:
            bad.append("%s merge_path %d, not the batch kernel" % (where, c.merge_path))
        return bad, off

    got = pool.run(inputs_, on_device=on_device, npts=npts, collect=collect)
    assert len(got) == INFLIGHT * ROUNDS and all(r is not None for r in got)
    report([l for b, _ in got for l in b], len(got), sum(o for _, o in got))


@pytest.fixture(scope="module")
def c2_pool(gpu, inputs):
    """The C2 pool and its resident input as bench.py's sweep_leg builds them: one device copy per in-flight slot, ROUNDS
    groups of pointers.  Tests (a), (c) and (d) run on it in that order, as the benchmark's three legs do."""
    import torch
    from f3ps import sweep
    d_frames = device_copies(torch, inputs["c2"])
    ptrs = [d_frames[i % INFLIGHT].data_ptr() for i in range(INFLIGHT * ROUNDS)]
    pool = bench_pool(sweep, bench.FLAGS)
    yield pool, ptrs
    pool.close()
    del d_frames
    torch.cuda.synchronize()


def test_a_c2_sweep_as_bench_runs_it(c2_pool, inputs, oracle):
    """(a) C2: 3 groups of 80 device-resident frames, K5 as 8-CTA clusters, the two handle sets alternating."""
    pool, ptrs = c2_pool
    sweep_and_compare(pool, ptrs, oracle("c2"), on_device=True, npts=len(inputs["c2"][0]))


def resident_sweep(frames, flags, want):
    """sweep_and_compare on a pool of its own with `flags`, input resident on the device as in (a)."""
    import torch
    from f3ps import sweep
    d_frames = device_copies(torch, frames)
    ptrs = [d_frames[i % INFLIGHT].data_ptr() for i in range(INFLIGHT * ROUNDS)]
    pool = bench_pool(sweep, flags)
    try:
        sweep_and_compare(pool, ptrs, want, on_device=True, npts=len(frames[0]))
    finally:
        pool.close()
        del d_frames
        torch.cuda.synchronize()


def test_b_c3_sweep_eq200_in_the_batch_kernel(gpu, inputs, oracle):
    """(b) merge_mode=2 (--EQ 200, the C3 leg) through merge_fast_batch_kernel, frames seeded 30000 + i."""
    resident_sweep(inputs["c3"], bench.C3_FLAGS, oracle("c3"))


def test_b_rgb_ml_sweep_in_the_batch_kernel(gpu, inputs, oracle):
    """--RGB --ML 0.5 (RGB distance, plain normal difference, manual lambda) through merge_fast_batch_kernel on the C2 frames."""
    resident_sweep(inputs["c2"], RGB_ML, oracle("c2_rgb_ml"))


def test_c_host_buffer_leg(gpu, c2_pool, inputs, oracle):
    """sweep_leg's e2e leg on the same pool: pinned host views, results read by the reader threads of one set while the
    other set's front stages run."""
    import torch
    pool, _ = c2_pool
    frames, want = inputs["c2"], oracle("c2")
    pinned = [torch.from_numpy(frames[i % len(frames)].view(np.uint8).reshape(-1, 32).copy()).pin_memory() for i in range(INFLIGHT)]
    host_views = [pinned[i % INFLIGHT].numpy().view(gpu.synth.POINT_DTYPE).reshape(-1) for i in range(INFLIGHT * ROUNDS)]
    sweep_and_compare(pool, host_views, want)


def test_d_single_frame_latency_leg(gpu, c2_pool, inputs, oracle):
    """sweep_leg's latency leg: pool.segs[0], after sweep use, switched to the cooperative K5 grid over the whole GPU and
    non-blocking waits, runs frames alone from the device copies."""
    pool, ptrs = c2_pool
    want, npts = oracle("c2"), len(inputs["c2"][0])
    solo = pool.segs[0]
    bad, off = [], 0
    for k in (1, 0):                                  # a different frame first: the handle's last sweep frame was slot 0's
        solo.set_blocking_wait(False)
        solo.set_expand_kernel(0, 0); solo.set_expand_sharing(0, 0)
        solo.set_input_device(ptrs[k], npts, 32); solo.run(THR)
        c = solo.counts()
        b, o = mismatches(solo.fetch_result(), c, want[k % len(want)], "single frame %d (pool frame %d)" % (k, k % len(want)))
        bad += b; off += o
        if c.merge_path != 1:
            bad.append("single frame %d: merge_path %d" % (k, c.merge_path))
    report(bad, 2, off)


def fresh_result(gpu, member):
    """What a fresh handle gives a member alone: f3ps_run on its points / f3ps_merge on its graph, same kernel choice."""
    g = gpu.Segmenter(); g.set_vccs_params(); g.set_merge_params(**bench.FLAGS)
    if member.get("kernel") is not None:
        g.set_merge_kernel(member["kernel"])
    if "graph" in member:
        g.set_graph(*member["graph"]); g.merge(THR)
    else:
        g.set_input(member["pts"]); g.run(THR)
    out = (g.fetch_result(), g.counts().merge_path)
    g.close()
    return out


def test_e_merge_batch_over_three_parameter_blocks(gpu, inputs, oracle, oracle_mod):
    """One f3ps_merge_batch call over more handles than two parameter blocks hold (kFastBatchMax <= 96): every chunk has its
    own lead stream, pinned scalar buffer and tail launches, and the results are read back after every grid is in flight.
    The later chunks hold a handle forced onto the L2 variant (3) and one onto the general kernel (2) (both run alone), the
    hub graph whose first merge is wider than the batch kernel's worker threads (the CTA stops, the L2 variant continues: 6),
    the phantom-leaf frame, and the empty / all-NaN (no supervoxels: alone, no kernel) / one-point / five-point clouds.
    Every member equals a fresh handle's result and the oracle's; called twice, since cluster() restarts."""
    want_small = oracle("small")
    members = [{"name": "small %d" % s, "pts": f, "want": w, "path": 1} for s, f, w in zip(SMALL_SEEDS, inputs["small"], want_small)]
    members[100].update(kernel=3, path=3, name=members[100]["name"] + " (L2 variant)")
    members[140].update(kernel=2, path=2, name=members[140]["name"] + " (general kernel)")
    graph = hub_graph(1500)
    o = oracle_mod.Oracle(); o.set_merge_params(merge_impl=1, **bench.FLAGS); o.set_graph(*graph); o.run(7, THR)
    hub_want = {n: o.array(n) for n in ("merges_ab", "merges_w", "merges_left", "out_label")}
    extra = [(120, {"name": "hub_graph(1500)", "graph": graph, "want": None, "path": 6}),
             (130, {"name": "empty cloud", "pts": inputs["edge"][0], "want": oracle("edge")[0], "path": 0}),
             (200, {"name": "phantom frame %d" % PHANTOM, "pts": inputs["phantom"], "want": oracle("phantom")[0], "path": 1}),
             (205, {"name": "all-NaN cloud", "pts": inputs["edge"][1], "want": oracle("edge")[1], "path": 0}),
             (210, {"name": "one-point cloud", "pts": inputs["edge"][2], "want": oracle("edge")[2], "path": None}),
             (215, {"name": "five-point cloud", "pts": inputs["edge"][3], "want": oracle("edge")[3], "path": None})]
    for pos, m in extra:
        members.insert(pos, m)
    segs = []
    for m in members:
        g = gpu.Segmenter(); g.set_vccs_params(); g.set_merge_params(**bench.FLAGS)
        if m.get("kernel") is not None:
            g.set_merge_kernel(m["kernel"])
        if "graph" in m:
            g.set_graph(*m["graph"])
        else:
            g.set_input(m["pts"]); g.extract(); g.graph()
        segs.append(g)
    for m, g in zip(members, segs):
        if m["path"] is None:                        # one or five points: the batch kernel if they have supervoxels
            m["path"] = 1 if g.counts().n_supervoxels else 0
    batch_index = dict(zip((m["name"] for m in members if m["path"] in (1, 6)), range(len(members))))
    assert len(batch_index) > 2 * 96                  # three parameter blocks for any kFastBatchMax <= 96
    assert 96 <= batch_index["hub_graph(1500)"] < 192 and batch_index["phantom frame %d" % PHANTOM] >= 192
    fresh = [fresh_result(gpu, m) for m in members]
    try:
        bad, off = [], 0
        for rep in range(2):
            gpu.merge_batch(segs, THR)
            for i, (m, g, (fr, fpath)) in enumerate(zip(members, segs, fresh)):
                where = "call %d, member %d (%s)" % (rep, i, m["name"])
                got, c = g.fetch_result(), g.counts()
                if c.merge_path != m["path"] or fpath != m["path"]:
                    bad.append("%s: merge_path %d, fresh handle %d, expected %d" % (where, c.merge_path, fpath, m["path"]))
                for n in EXACT + ("merges_w",):
                    if not same(got[n], fr[n]):
                        bad.append("%s %s differs from a fresh handle's" % (where, n))
                if m["want"] is not None:
                    b, o_ = mismatches(got, c, m["want"], where)
                    bad += b; off += o_
                else:
                    for n, w in hub_want.items():
                        if not (close_enough if n == "merges_w" else same)(got[n], w):
                            bad.append("%s %s differs from the oracle" % (where, n))
        report(bad, 2 * len(members), off)
    finally:
        for g in segs:
            g.close()


def test_f_mixed_group_grows_and_shrinks(gpu, inputs, oracle):
    """One group of INFLIGHT frames through BatchPool with host input: VGA frames (two with three seed cells on one voxel),
    160x120 frames, the 1280x960 frame and the edge clouds, twice, the second time with the frame order permuted so that the
    handles of the largest frames get the smallest and the other way round.  The 1280x960 frame's graph (2,578 supervoxels,
    9,274 edges) still fits the batch kernel's shared memory, so one handle of the set is forced onto the L2 variant
    (set_merge_kernel(3)): the frame it gets runs alone beside the grid, a VGA frame in the first round, a 160x120 one in the
    second.  A handle that shrinks must not report anything of its last, larger frame: the clouds without supervoxels run
    no merge kernel (merge_path 0) on handles that ran the largest frames before."""
    from f3ps import sweep
    vga = inputs["triple"] + inputs["c2"]
    frames = vga + inputs["small"][:INFLIGHT - len(vga) - 5] + [inputs["large"]] + inputs["edge"]
    want = oracle("triple") + oracle("c2") + oracle("small")[:INFLIGHT - len(vga) - 5] + oracle("large") + oracle("edge")
    names = (["vga %d" % s for s in TRIPLE_SEEDS] + ["vga %d" % (20020 + i) for i in range(len(inputs["c2"]))] +
             ["small %d" % s for s in SMALL_SEEDS[:INFLIGHT - len(vga) - 5]] + ["1280x960 %d" % LARGE_SEED] +
             ["empty", "all-NaN", "one point", "five points"])
    assert len(frames) == len(want) == len(names) == INFLIGHT
    rng = np.random.default_rng(7)
    first = rng.permutation(INFLIGHT)
    by_size = sorted(range(INFLIGHT), key=lambda i: (len(frames[i]), i))
    swap = {by_size[r]: by_size[INFLIGHT - 1 - r] for r in range(INFLIGHT)}      # k-th smallest <-> k-th largest
    second = np.array([swap[i] for i in first])
    pool = sweep.BatchPool(batch=INFLIGHT, workers=WORKERS, expand_ctas=-EXPAND_CTAS, expand_cluster=EXPAND_CLUSTER, merge=bench.FLAGS, threshold=THR)
    beside = int(np.nonzero(first == 0)[0][0])                                   # the slot of VGA frame 22030 in the first round
    assert names[second[beside]].startswith("small")
    pool.sets[0][beside].set_merge_kernel(3)
    try:
        bad, off, sizes = [], 0, []
        for rnd, order in enumerate((first, second)):
            def collect(seg, k, order=order, rnd=rnd):
                i = int(order[k])
                where = "round %d, slot %d: frame %d (%s)" % (rnd, k, i, names[i])
                c = seg.counts()
                b, o_ = mismatches(seg.fetch_result(), c, want[i], where)
                if seg is not pool.sets[0][k]:
                    b.append("%s ran on handle %d" % (where, pool.segs.index(seg)))
                expect = 0 if c.n_supervoxels == 0 else 3 if k == beside else 1
                if c.merge_path != expect:
                    b.append("%s merge_path %d (S = %d)" % (where, c.merge_path, c.n_supervoxels))
                return b, o_, c.n_voxels
            got = pool.run([frames[i] for i in order], collect=collect)
            bad += [l for b, _, _ in got for l in b]
            off += sum(o_ for _, o_, _ in got)
            sizes.append([v for _, _, v in got])
        changed = sum(a != b for a, b in zip(*sizes))
        assert changed >= INFLIGHT - 2, "only %d of %d handles changed size between the rounds" % (changed, INFLIGHT)
        report(bad, 2 * INFLIGHT, off)
    finally:
        pool.close()
