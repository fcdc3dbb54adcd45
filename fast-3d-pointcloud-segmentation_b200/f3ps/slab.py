"""Slab mode: ONE very large cloud on several GPUs (SURVEY.md section 8e row 2, BASELINE config 5).

The reference runs pcl::SupervoxelClustering::extract + Clustering::cluster on the whole cloud in one thread
(src/supervoxel_clustering.cpp:348-367, 408-449).  Here every rank (one process per GPU, torch.distributed)
starts with an arbitrary share of the points -- e.g. some of the scan positions of a merged room scan -- and the cloud
is cut into spatial slabs: contiguous ranges of the x-major Morton key of PCL's adjacency octree.  Because that
key order IS PCL's leaf order, a slab's voxels are a contiguous slice of the single-GPU voxel table and every
ordered float sum keeps its order, so the result is bit-identical to one handle processing the whole cloud
(tests/test_gpu_slab.py).

Everything but the exchanges is a library call (include/f3ps.h, f3ps_slab_*), the splitter rule and the assembly of the
replicated voxel table included, so this driver and host/slab_host.cpp (the same protocol over NCCL from C++) cut a cloud
in the same place by construction.

Exchanges (all on the stream the handle runs on; NCCL over NVLink when the backend is nccl):
  K1  all-reduce MIN/MAX of the transformed bounding box (6 floats)      -> same frame / key grid on every rank
      all-reduce SUM of a 4096-bin histogram of the keys' top bits       -> equal-count splitters (f3ps_slab_route)
      all-to-all of the points, 16 bytes each, to the rank owning their key range (stable: input order survives)
      all-gather of the voxel slices (40 bytes per voxel), in place      -> replicated voxel table
  K3  normals of the owned slice, all-gather of the slices (20 bytes per voxel)
  K2 (hash + 27 probes), K4 (seed grid), K5 (the expansion kernel of one handle) and K6 run on the replicated
  tables on every rank; K7 does not shard ("replicas only": one graph, strictly serial order) and is replayed by
  every rank, so every rank ends with the complete result and no broadcast is needed.
"""
import numpy as np

from . import binding


class _DevView:
    """A raw device pointer as something torch.as_tensor understands (zero copy)."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (int(nbytes),), "typestr": "|u1", "data": (int(ptr), False), "version": 2}


def device_view(torch, ptr, n, elem_bytes, dtype, device):
    """torch tensor [n, elem_bytes / itemsize] aliasing n elements at device pointer ptr."""
    if n == 0 or not ptr:
        return torch.empty((0, max(1, elem_bytes // torch.empty((), dtype=dtype).element_size())), dtype=dtype, device=device)
    raw = torch.as_tensor(_DevView(ptr, n * elem_bytes), device=device)
    return raw.view(dtype).view(n, -1)


def slice_bounds(counts):
    b = np.zeros(len(counts) + 1, np.int64)
    b[1:] = np.cumsum(counts)
    return b


class Comm:
    """The collectives the slab driver needs, on torch.distributed.  backend nccl: straight on the device tensors.
    backend gloo (CPU tests, or several ranks sharing one GPU in the parity test): staged through host memory."""

    def __init__(self, dist=None, torch=None):
        self.dist, self.torch = dist, torch
        self.on = dist is not None and dist.is_available() and dist.is_initialized()
        self.rank = dist.get_rank() if self.on else 0
        self.world = dist.get_world_size() if self.on else 1
        self.staged = self.on and dist.get_backend() != "nccl"
        self.bytes_moved = 0

    def all_reduce(self, t, op):
        if not self.on or self.world == 1:
            return t
        d = self.dist
        rop = {"min": d.ReduceOp.MIN, "max": d.ReduceOp.MAX, "sum": d.ReduceOp.SUM}[op]
        self.bytes_moved += t.numel() * t.element_size()
        if self.staged and t.is_cuda:
            h = t.cpu()
            d.all_reduce(h, op=rop)
            t.copy_(h)
        else:
            d.all_reduce(t, op=rop)
        return t

    def all_gather_int(self, value):
        if not self.on or self.world == 1:
            return [int(value)]
        t = self.torch.tensor([int(value)], dtype=self.torch.int64)
        out = [self.torch.zeros(1, dtype=self.torch.int64) for _ in range(self.world)]
        if not self.staged:
            dev = self.torch.device("cuda", self.torch.cuda.current_device())
            t = t.to(dev); out = [o.to(dev) for o in out]
        self.dist.all_gather(out, t)
        return [int(o[0]) for o in out]

    def all_gather_vec(self, vec):
        """vec: int64 numpy [k] -> [world, k]"""
        if not self.on or self.world == 1:
            return np.asarray(vec, np.int64)[None, :]
        t = self.torch.from_numpy(np.ascontiguousarray(vec, np.int64))
        out = [self.torch.zeros_like(t) for _ in range(self.world)]
        if not self.staged:
            dev = self.torch.device("cuda", self.torch.cuda.current_device())
            t = t.to(dev); out = [o.to(dev) for o in out]
        self.dist.all_gather(out, t)
        return np.stack([o.cpu().numpy() for o in out])

    def gather_slices(self, full, bounds):
        """full: tensor whose rows [bounds[r], bounds[r+1]) are valid on rank r; afterwards all rows are valid everywhere."""
        if not self.on or self.world == 1:
            return full
        for r in range(self.world):
            lo, hi = int(bounds[r]), int(bounds[r + 1])
            if hi <= lo:
                continue
            part = full[lo:hi]
            self.bytes_moved += part.numel() * part.element_size()
            if self.staged and part.is_cuda:
                h = part.cpu() if r == self.rank else self.torch.empty(part.shape, dtype=part.dtype)
                self.dist.broadcast(h, src=r)
                if r != self.rank:
                    part.copy_(h)
            else:
                self.dist.broadcast(part, src=r)
        return full

    def all_to_all_rows(self, send, send_counts, recv_counts):
        """send: [n, k] rows grouped by destination; returns [sum(recv_counts), k] rows grouped by source rank."""
        torch = self.torch
        n_recv = int(np.sum(recv_counts))
        recv = torch.empty((n_recv, send.shape[1]), dtype=send.dtype, device=send.device)
        if not self.on or self.world == 1:
            recv.copy_(send[:n_recv])
            return recv
        self.bytes_moved += int(np.sum(send_counts)) * send.shape[1] * send.element_size()
        if not self.staged:
            self.dist.all_to_all_single(recv, send[:int(np.sum(send_counts))].contiguous(),
                                        [int(c) for c in recv_counts], [int(c) for c in send_counts])
            return recv
        # gloo has no all-to-all: one scatter per source rank, on host tensors
        sb = slice_bounds(send_counts)
        rb = slice_bounds(recv_counts)
        hs = send.cpu()
        for src in range(self.world):
            dst = torch.empty((int(recv_counts[src]), send.shape[1]), dtype=send.dtype)
            if src == self.rank:
                chunks = [hs[int(sb[r]):int(sb[r + 1])].contiguous() for r in range(self.world)]
                # scatter needs equal shapes: pad to the largest chunk
                m = max(1, max(c.shape[0] for c in chunks))
                padded = [torch.zeros((m, send.shape[1]), dtype=send.dtype) for _ in chunks]
                for p, c in zip(padded, chunks):
                    p[:c.shape[0]] = c
                sizes = torch.tensor([m], dtype=torch.int64)
            else:
                padded, sizes = None, torch.zeros(1, dtype=torch.int64)
            self.dist.broadcast(sizes, src=src)
            buf = torch.zeros((int(sizes[0]), send.shape[1]), dtype=send.dtype)
            self.dist.scatter(buf, scatter_list=padded, src=src)
            dst.copy_(buf[:dst.shape[0]])
            recv[int(rb[src]):int(rb[src + 1])].copy_(dst)
        return recv


class SlabSegmenter:
    """One rank of a slab-mode run.  `run(points, threshold)` takes THIS rank's share of the cloud (numpy records of
    16 or 32 bytes, or a (device pointer, n, stride) triple) and leaves the complete result on this rank's handle
    (`self.seg`: counts(), array(...), stage getters -- identical on every rank)."""

    TOP_BITS = 12

    def __init__(self, comm, device=0, vccs=None, merge=None):
        import torch
        self.torch = torch
        self.comm = comm
        self.device = torch.device("cuda", device)
        torch.cuda.set_device(self.device)
        self.stream = torch.cuda.Stream(device=self.device)
        self.seg = binding.Segmenter(device=device, stream=self.stream.cuda_stream)
        self.seg.set_vccs_params(**(vccs or {}))
        self.seg.set_merge_params(**(merge or {}))
        self.info = {}
        self._views = {}

    def close(self):
        self.seg.close()

    def _view(self, name, dtype):
        ptr, n, eb = self.seg.slab_array(name)
        key = (ptr, n, eb, dtype)                     # the handle's buffers alternate between a few addresses: wrap each once
        v = self._views.get(key)
        if v is None:
            if len(self._views) > 64:
                self._views.clear()
            v = self._views[key] = device_view(self.torch, ptr, n, eb, dtype, self.device)
        return v

    def run(self, points, threshold=0.2, merge=True):
        torch, comm, seg = self.torch, self.comm, self.seg
        ev = []

        def tick(name):
            e = torch.cuda.Event(enable_timing=True)
            e.record(self.stream)
            ev.append((name, e))

        self._views.clear()
        with torch.cuda.stream(self.stream):
            tick("start")
            seg.slab_reset()
            if isinstance(points, tuple):
                ptr, n_local, stride = points
                seg.set_input_device(ptr, n_local, stride)
            else:
                n_local = int(points.shape[0])
                seg.set_input(points)
            # ---- K1a: the frame of the whole cloud ----
            box = torch.zeros(8, dtype=torch.int32, device=self.device)
            seg.slab_bbox(box.data_ptr())
            if comm.world > 1:
                sgn = torch.tensor(-2 ** 31, dtype=torch.int32, device=self.device)
                ob = box ^ sgn                                   # unsigned order -> signed order
                comm.all_reduce(ob[0:3], "min"); comm.all_reduce(ob[3:7], "max")
                box = ob ^ sgn
            seg.slab_set_frame(box.data_ptr())
            # ---- K1b: keys, splitters, routing ----
            hist = torch.zeros(1 << self.TOP_BITS, dtype=torch.int32, device=self.device)
            seg.slab_keys(self.TOP_BITS, hist.data_ptr())
            comm.all_reduce(hist, "sum")
            send = torch.empty((max(1, n_local), 4), dtype=torch.float32, device=self.device)
            send_counts = seg.slab_route(comm.world, hist.data_ptr(), send.data_ptr())
            tick("route")
            count_matrix = comm.all_gather_vec(send_counts)      # [src, dst]
            recv_counts = count_matrix[:, comm.rank]
            recv = comm.all_to_all_rows(send, send_counts, recv_counts)
            del send
            tick("all_to_all")
            # ---- K1c: voxels of the owned slab, then the replicated table ----
            n_recv = int(recv.shape[0])
            if n_recv:
                seg.set_input_device(recv.data_ptr(), n_recv, 16)
            else:
                seg.set_input(np.zeros((0, 4), np.float32).view(np.dtype([("xyzc", "<f4", (4,))])).reshape(0))
            seg.voxelize()
            v_local = int(seg.counts().n_voxels)
            vb = slice_bounds(comm.all_gather_int(v_local))
            V = int(vb[-1])
            lo, hi = int(vb[comm.rank]), int(vb[comm.rank + 1])
            seg.slab_set_voxels(V, lo)
            tick("voxelize")
            if V:
                comm.gather_slices(self._view("vox_xyz", torch.float32), vb)
                comm.gather_slices(self._view("vox_rgb", torch.float32), vb)
                comm.gather_slices(self._view("vox_key", torch.int64), vb)
            del recv
            tick("gather_voxels")
            # ---- K2 (replicated), K3 (owned slice + exchange), K4 (replicated) ----
            seg.neighbors()
            tick("neighbors")
            seg.normals()
            if V:
                comm.gather_slices(self._view("vox_normal", torch.float32), vb)
                comm.gather_slices(self._view("vox_curv", torch.float32), vb)
            tick("normals")
            seg.seeds()
            tick("seeds")
            # ---- K5 on the replicated table: the kernel of one handle, no exchange ----
            seg.expand()
            sweeps = int(seg.counts().sweeps)
            tick("expand")
            # ---- K6, K7 on the replicated tables ----
            seg.graph()
            tick("graph")
            if merge:
                seg.merge(threshold)
                tick("merge")
            seg.sync()
        self.stream.synchronize()
        ms = {}
        for (n0, e0), (n1, e1) in zip(ev[:-1], ev[1:]):
            ms[n1] = e0.elapsed_time(e1)
        ms["total"] = ev[0][1].elapsed_time(ev[-1][1])
        self.info = {"n_local": n_local, "n_received": n_recv, "v_local": v_local, "V": V, "own": (lo, hi), "sweeps": sweeps,
                     "send_counts": [int(c) for c in send_counts],
                     "stage_ms": ms, "bytes_exchanged": comm.bytes_moved}
        return self.info
