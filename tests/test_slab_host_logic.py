"""Host logic of slab mode on CPU: the library's splitter rule, slice bookkeeping and the collectives wrapper over a
world_size-2 gloo group (the GPU pieces between the exchanges are covered by tests/test_gpu_slab.py)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


@pytest.fixture(scope="module")
def binding():
    from f3ps import binding
    binding.build()
    return binding


def test_choose_splitters_equal_count(binding):
    from f3ps import slab
    rng = np.random.default_rng(5)
    hist = rng.integers(0, 1000, 4096)
    hist[:700] = 0
    for world in (1, 2, 3, 4, 8):
        sp = binding.slab_choose_splitters(hist, world, shift=9)
        assert sp.shape == (world - 1,) and np.all(np.diff(sp.astype(np.int64)) >= 0)
        cuts = [0] + [int(x) >> 9 for x in sp] + [4096]
        loads = [int(hist[cuts[i]:cuts[i + 1]].sum()) for i in range(world)]
        assert sum(loads) == int(hist.sum())
        if world > 1:
            assert max(loads) - min(loads) <= 2 * int(hist.max()) + 1
    # degenerate: everything in one bin -> one rank owns it all, splitters still ascend
    h = np.zeros(64, np.int64); h[10] = 99
    sp = binding.slab_choose_splitters(h, 4, shift=0)
    assert list(sp) == sorted(sp) and all(int(x) <= 64 for x in sp)
    assert list(slab.slice_bounds([3, 0, 5])) == [0, 3, 3, 8]


def _splitters_reference(hist, world, shift):
    """The splitter rule restated in numpy: cut r is the first bin boundary at or after r/world of the points (cumulative
    count >= total * r // world), never below the cut before it, at most the bin count, shifted left by `shift`."""
    hist = np.asarray(hist, np.int64)
    total = int(hist.sum())
    cum = np.cumsum(hist)
    cuts = []
    for r in range(1, world):
        b = int(np.searchsorted(cum, (total * r) // world, side="left")) + 1
        cuts.append(min(max(b, cuts[-1] if cuts else 0), hist.shape[0]))
    return np.array([np.uint64(b) << np.uint64(shift) for b in cuts], np.uint64)


def test_library_choose_splitters_equals_reference(binding):
    """f3ps_slab_choose_splitters, the one splitter rule both slab drivers (f3ps/slab.py, host/slab_host.cpp) call, against
    its restatement above, over bin counts, rank counts, shifts and degenerate histograms."""
    rng = np.random.default_rng(17)
    cases = []
    for n_bins in (1, 2, 64, 4096):
        for _ in range(6):
            h = rng.integers(0, 5000, n_bins).astype(np.uint32)
            if rng.random() < 0.5:
                h[rng.integers(0, n_bins, max(1, n_bins // 2))] = 0
            cases.append(h)
    cases += [np.zeros(64, np.uint32), np.eye(1, 64, 10, dtype=np.uint32)[0] * 99]
    for h in cases:
        for world in (1, 2, 3, 8):
            for shift in (0, 9, 33):
                want = _splitters_reference(h, world, shift)
                got = binding.slab_choose_splitters(h, world, shift)
                assert np.array_equal(got, want), (len(h), world, shift)


def _oracle_keys(pts):
    """Morton key of every point's voxel (x-major), from the oracle's voxelisation -- test-side stand-in for K1 keygen."""
    import oracle_py
    o = oracle_py.Oracle()
    o.set_vccs_params(); o.set_merge_params(color_mode=0, geom_mode=1, merge_mode=1, merge_impl=1)
    o.set_input(pts); o.run(0, 0.2)
    keys = o.array("keys").astype(np.uint64)
    pv = o.array("point_voxel")

    def spread(v):
        out = np.zeros_like(v)
        for b in range(21):
            out |= ((v >> np.uint64(b)) & np.uint64(1)) << np.uint64(3 * b)
        return out
    m = (spread(keys[:, 0]) << np.uint64(2)) | (spread(keys[:, 1]) << np.uint64(1)) | spread(keys[:, 2])
    depth = int(np.ceil(np.log2(max(2, int(keys.max()) + 1))))
    return m, pv, depth


def _worker(rank, world, port, q):
    try:
        os.environ["MASTER_ADDR"] = "127.0.0.1"
        os.environ["MASTER_PORT"] = str(port)
        dist.init_process_group("gloo", rank=rank, world_size=world)
        from f3ps import binding, slab, synth
        comm = slab.Comm(dist, torch)
        assert comm.staged and comm.world == world
        pts = synth.make_frame(seed=11, width=160, height=120)
        vox_key, pv, depth = _oracle_keys(pts)
        n = pts.shape[0]
        lo, hi = n * rank // world, n * (rank + 1) // world
        valid = np.nonzero(pv[lo:hi] >= 0)[0] + lo                       # this rank's valid points, input order
        keys = vox_key[pv[valid]]
        # the protocol of SlabSegmenter.run with numpy stand-ins for the kernels
        shift = max(0, 3 * depth - 12)
        hist = torch.from_numpy(np.bincount((keys >> np.uint64(shift)).astype(np.int64), minlength=4096).astype(np.int32))
        comm.all_reduce(hist, "sum")
        sp = binding.slab_choose_splitters(hist.numpy(), world, shift)
        dest = np.searchsorted(sp, keys, side="right")
        order = np.argsort(dest, kind="stable")
        send_counts = np.bincount(dest, minlength=world).astype(np.int64)
        send = torch.from_numpy(np.stack([valid[order].astype(np.float64), keys[order].astype(np.float64)], 1))
        cm = comm.all_gather_vec(send_counts)
        recv = comm.all_to_all_rows(send, send_counts, cm[:, rank]).numpy()
        gidx, gkey = recv[:, 0].astype(np.int64), recv[:, 1].astype(np.uint64)
        # what one process would hand this slab: all valid points in input order whose key falls in the slab
        allv = np.nonzero(pv >= 0)[0]
        allk = vox_key[pv[allv]]
        mine = np.searchsorted(sp, allk, side="right") == rank
        ok = np.array_equal(gidx, allv[mine]) and np.array_equal(gkey, allk[mine])
        # slices of a replicated table
        v_local = int(np.unique(gkey).shape[0])
        vb = slab.slice_bounds(comm.all_gather_int(v_local))
        full = torch.full((int(vb[-1]), 2), -1, dtype=torch.int64)
        full[int(vb[rank]):int(vb[rank + 1])] = torch.from_numpy(np.stack([np.unique(gkey).astype(np.int64)] * 2, 1))
        comm.gather_slices(full, vb)
        ok = ok and np.array_equal(full[:, 0].numpy().astype(np.uint64), np.unique(allk))
        flag = torch.tensor([rank], dtype=torch.int32)
        comm.all_reduce(flag, "max")
        ok = ok and int(flag[0]) == world - 1
        q.put((rank, bool(ok), int(vb[-1])))
        dist.barrier()
        dist.destroy_process_group()
    except Exception as e:
        import traceback
        q.put((rank, False, "%s\n%s" % (e, traceback.format_exc())))


def test_two_rank_gloo_exchange_protocol(oracle_mod, binding):
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=300) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
    for rank, ok, v in res:
        assert ok is True, (rank, v)
    assert res[0][2] == res[1][2] > 1000
