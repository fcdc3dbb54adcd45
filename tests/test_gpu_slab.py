"""Slab mode (SURVEY.md 8e row 2): a cloud cut into Morton-range slabs over R ranks must give, on EVERY rank, the
bit-identical result of one handle processing the whole cloud.  The ranks here share cuda:0 and exchange over gloo
(staged through host memory), so the parity of the whole exchange protocol is checked on a one-GPU box; on a
multi-GPU box the same driver runs over NCCL (bench.py --workload c5)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu

ARRAYS = ["keys", "voxel_xyz", "voxel_rgb", "voxel_rgba", "voxel_count", "nbr", "nbr_count", "normals", "curvature", "seeds",
          "labels", "dist", "sv_label", "sv_xyz", "sv_rgb", "sv_normal", "sv_count", "adj", "edges_ab", "edges_dc", "edges_dg",
          "edges_w", "merges_ab", "merges_w", "merges_left", "out_xyz", "out_label", "out_voxel"]


def _cloud(case):
    from f3ps import synth
    if case == "small":
        return synth.make_frame(seed=11, width=160, height=120), dict(), dict(color_mode=0, geom_mode=1, merge_mode=1)
    if case == "vga_eq":
        return synth.make_frame(seed=30003), dict(), dict(color_mode=0, geom_mode=0, merge_mode=2, bins=200)
    if case == "nt_rgb":
        return (synth.make_frame(seed=7, width=320, height=240), dict(use_transform=False, voxel_res=0.02, seed_res=0.2),
                dict(color_mode=1, geom_mode=1, merge_mode=0, lam=0.5))
    raise KeyError(case)


def _worker(rank, world, port, case, q):
    try:
        os.environ["MASTER_ADDR"] = "127.0.0.1"
        os.environ["MASTER_PORT"] = str(port)
        dist.init_process_group("gloo", rank=rank, world_size=world)
        import f3ps
        from f3ps import slab
        pts, vccs, merge = _cloud(case)
        thr = 0.6 if case == "vga_eq" else 0.2          # --EQ weights start at ~0.44 on this frame
        n = pts.shape[0]
        cuts = [n * r // world for r in range(world + 1)]
        if case == "small" and world == 3:
            cuts = [0, 0, n // 3, n]                      # an empty share
        mine = pts[cuts[rank]:cuts[rank + 1]]
        ref = f3ps.Segmenter(device=0)
        ref.set_vccs_params(**vccs); ref.set_merge_params(**merge)
        ref.set_input(pts); ref.run(thr)
        comm = slab.Comm(dist, torch)
        ss = slab.SlabSegmenter(comm, device=0, vccs=vccs, merge=merge)
        info = ss.run(mine, thr)
        bad = []
        for name in ARRAYS:
            a, b = ss.seg.array(name), ref.array(name)
            if a.shape != b.shape or not np.array_equal(a, b, equal_nan=a.dtype.kind == "f"):
                bad.append(name)
        c, cr = ss.seg.counts(), ref.counts()
        for f in ("n_voxels", "n_seeds", "n_supervoxels", "n_edges", "n_merges", "n_segments", "depth"):
            if getattr(c, f) != getattr(cr, f):
                bad.append("counts." + f)
        # a plain handle created AFTER the slab run must be unaffected by it
        ref2 = f3ps.Segmenter(device=0)
        ref2.set_vccs_params(**vccs); ref2.set_merge_params(**merge)
        ref2.set_input(pts); ref2.run(thr)
        if not np.array_equal(ref2.array("merges_ab"), ref.array("merges_ab")):
            bad.append("second plain run differs")
        q.put((rank, bad, info["own"], info["V"], info["sweeps"], int(cr.sweeps), int(c.n_merges)))
        dist.barrier()
        dist.destroy_process_group()
    except Exception as e:                                # surfaced to the parent
        import traceback
        q.put((rank, ["exception: %s\n%s" % (e, traceback.format_exc())], None, 0, 0, 0, 0))


@pytest.mark.parametrize("case,world", [("small", 2), ("small", 3), ("vga_eq", 2), ("vga_eq", 3), ("nt_rgb", 4)],
                         ids=["small-2ranks", "small-3ranks-empty-share", "vga_eq-2ranks", "vga_eq-3ranks", "nt_rgb-4ranks"])
def test_slab_equals_single_handle(case, world):
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, case, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=600) for _ in range(world))
    for p in procs:
        p.join(timeout=120)
    for rank, bad, own, V, sweeps, ref_sweeps, merges in res:
        assert bad == [], "rank %d: %s" % (rank, bad)
        assert sweeps == ref_sweeps and merges > 0, (rank, sweeps, ref_sweeps, merges)
    # the slices tile the voxel table
    owns = [r[2] for r in res]
    assert owns[0][0] == 0 and owns[-1][1] == res[0][3]
    assert all(owns[i][1] == owns[i + 1][0] for i in range(world - 1))
    assert sum(1 for o in owns if o[1] > o[0]) >= 2       # the cloud really was cut


def test_slab_world1_equals_plain(small_frame):
    import f3ps
    from f3ps import slab
    ss = slab.SlabSegmenter(slab.Comm(None, torch), device=0, merge=dict(color_mode=0, geom_mode=1, merge_mode=1))
    ss.run(small_frame, 0.2)
    ref = f3ps.Segmenter(device=0)
    ref.set_vccs_params(); ref.set_merge_params(color_mode=0, geom_mode=1, merge_mode=1)
    ref.set_input(small_frame); ref.run(0.2)
    for name in ARRAYS:
        a, b = ss.seg.array(name), ref.array(name)
        assert a.shape == b.shape and np.array_equal(a, b, equal_nan=a.dtype.kind == "f"), name
