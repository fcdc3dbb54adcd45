"""Directory-sweep sharding (-d of the reference CLI, src/supervoxel_clustering.cpp:209-227, 303):
files are independent (fresh SupervoxelClustering + Clustering per file, :348,408), so they are dealt
round-robin to the ranks, one GPU + one stream per rank, and no data-path collective exists.  Only the
final timing / score reduction crosses ranks."""


def shard_frames(n_frames, rank, world):
    """Indices of the frames rank `rank` of `world` processes (file order is kept inside a rank)."""
    if world <= 0 or not (0 <= rank < world):
        raise ValueError("bad rank/world")
    return list(range(rank, n_frames, world))


def aggregate_throughput(points_per_rank, seconds_per_rank):
    """Whole-job Mpoints/s: all points / slowest rank's time."""
    return sum(points_per_rank) / max(seconds_per_rank) / 1e6


def reduce_sweep(local_points, local_seconds, dist=None):
    """Cross-rank reduction of a sweep with torch.distributed (sum of points, max of time)."""
    if dist is None or not dist.is_initialized():
        return local_points, local_seconds
    import torch
    t = torch.tensor([float(local_points)], dtype=torch.float64)
    m = torch.tensor([float(local_seconds)], dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    dist.all_reduce(m, op=dist.ReduceOp.MAX)
    return float(t[0]), float(m[0])


class FramePool:
    """Frames in flight on ONE GPU: `n_handles` independent f3ps handles, each with its own CUDA stream and
    host thread (ctypes releases the GIL inside every C-ABI call).  The reference processes the files of a
    -d sweep strictly one after the other (src/supervoxel_clustering.cpp:303); they are independent, and the
    serial stage of a frame (K7, one persistent CTA on one SM) leaves 147 SMs idle, so a sweep keeps several
    frames in flight.  Frame k goes to handle k % n_handles; results come back in frame order."""

    def __init__(self, n_handles, device=0, vccs=None, merge=None, threshold=0.2):
        from . import binding
        import threading
        self.segs = [binding.Segmenter(device=device) for _ in range(n_handles)]
        import os
        blocking = n_handles > max(1, (os.cpu_count() or 1) // 2)     # spinning waiters must not outnumber the cores
        for s in self.segs:
            s.set_vccs_params(**(vccs or {}))
            s.set_merge_params(**(merge or {}))
            s.set_blocking_wait(blocking)
        self.threshold = threshold
        self._threading = threading

    def close(self):
        for s in self.segs:
            s.close()
        self.segs = []

    def run(self, frames, on_device=False, npts=None, collect=None):
        """frames: list of numpy point arrays (host) or device pointers (on_device=True, npts each).
        collect(seg, k) is called on the worker thread after frame k finished (result read-back)."""
        n = len(self.segs)
        errors = []
        results = [None] * len(frames)

        def worker(w):
            seg = self.segs[w]
            try:
                for k in range(w, len(frames), n):
                    if on_device:
                        seg.set_input_device(frames[k], npts, 32)
                    else:
                        seg.set_input(frames[k])
                    seg.run(self.threshold)
                    if collect is not None:
                        results[k] = collect(seg, k)
            except Exception as e:          # surfaced to the caller, never swallowed
                errors.append(e)

        th = [self._threading.Thread(target=worker, args=(w,)) for w in range(n)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        if errors:
            raise errors[0]
        return results


class BatchPool:
    """Frames in flight on ONE GPU with the merge stage batched: groups of `batch` frames run K1..K6 on their own handles /
    streams (`workers` host threads), then ONE launch of the resident merge kernel replays the whole group, CTA i = frame i
    (f3ps_merge_batch).  Independent streams share at most 32 hardware queues, which caps FramePool at 32 overlapping merge
    kernels; a grid has no such cap.  Two handle sets alternate, so the front stages of group g+1 overlap the merge of group g.
    Results are those of Segmenter.run on every frame, in frame order."""

    def __init__(self, batch=64, workers=None, device=0, vccs=None, merge=None, threshold=0.2, expand_ctas=0, expand_cluster=8):
        if expand_ctas > 0:
            raise ValueError("expand_ctas must be <= 0: -n caps K5's cooperative grid at n CTAs")
        from . import binding
        import os
        import threading
        self.binding = binding
        self.batch = batch
        # front-stage host threads: they sleep on blocking events most of the time, and what they are for is keeping ~16 frames in
        # flight (measured: 8, 16, 32 give the same throughput on 16 cores) -- not one per core: 8 ranks x 32 threads only contend
        self.workers = workers or max(2, min(batch, 16))
        self.sets = [[binding.Segmenter(device=device) for _ in range(batch)] for _ in range(2)]
        for st in self.sets:
            for s in st:
                s.set_vccs_params(**(vccs or {}))
                s.set_merge_params(**(merge or {}))
                s.set_blocking_wait(True)
                if expand_cluster:
                    # K5 as ONE thread-block cluster per frame (hardware cluster barrier; an ordinary launch, so the frames' K5 run side
                    # by side -- cooperative launches run one at a time).  Measured on C2, groups of 96: 8 CTAs 427 Mpoints/s,
                    # cooperative grid capped at 24 CTAs 416; 1-2 CTAs per frame lose (the 32 hardware queues cap long kernels)
                    s.set_expand_kernel(2, expand_cluster)
                elif expand_ctas:
                    s.set_expand_sharing(-expand_ctas, 0)            # cooperative launch, grid capped: more frames side by side
        self.segs = self.sets[0] + self.sets[1]
        self.threshold = threshold
        self._threading = threading

    def close(self):
        for s in self.segs:
            s.close()
        self.sets, self.segs = [], []

    def run(self, frames, on_device=False, npts=None, collect=None):
        n = len(frames)
        results = [None] * n
        errors = []
        groups = [list(range(g, min(n, g + self.batch))) for g in range(0, n, self.batch)]

        import time as _time
        self.timeline = []                      # (what, group, start, end) in seconds since the start of run(): where a step's time goes
        t_run0 = _time.perf_counter()

        def front(gi):
            t_f0 = _time.perf_counter()
            st = self.sets[gi % 2]
            idx = groups[gi]

            def worker(w):
                try:
                    for j in range(w, len(idx), self.workers):
                        seg = st[j]
                        if on_device:
                            seg.set_input_device(frames[idx[j]], npts, 32)
                        else:
                            seg.set_input(frames[idx[j]])
                        seg.extract()
                        seg.graph()
                except Exception as e:
                    errors.append(e)
            th = [self._threading.Thread(target=worker, args=(w,)) for w in range(min(self.workers, len(idx)))]
            for t in th:
                t.start()
            for t in th:
                t.join()
            self.timeline.append(("front", gi, t_f0 - t_run0, _time.perf_counter() - t_run0))

        def back(gi):
            t_b0 = _time.perf_counter()
            try:
                st = self.sets[gi % 2]
                idx = groups[gi]
                self.binding.merge_batch(st[:len(idx)], self.threshold)
                self.timeline.append(("merge", gi, t_b0 - t_run0, _time.perf_counter() - t_run0))
                if collect is not None:                  # result read-back of the group, a few host threads
                    def reader(w):
                        try:
                            for j in range(w, len(idx), nread):
                                results[idx[j]] = collect(st[j], idx[j])
                        except Exception as e:
                            errors.append(e)
                    nread = max(1, min(8, len(idx)))
                    th = [self._threading.Thread(target=reader, args=(w,)) for w in range(nread)]
                    for t in th:
                        t.start()
                    for t in th:
                        t.join()
            except Exception as e:
                errors.append(e)

        prev = None
        for gi in range(len(groups)):
            f = self._threading.Thread(target=front, args=(gi,))
            f.start()
            if prev is not None:
                prev.join()                      # the set this front stage is about to reuse was merged two groups ago
            f.join()
            if errors:
                raise errors[0]
            prev = self._threading.Thread(target=back, args=(gi,))
            prev.start()
        if prev is not None:
            prev.join()
        if errors:
            raise errors[0]
        return results

