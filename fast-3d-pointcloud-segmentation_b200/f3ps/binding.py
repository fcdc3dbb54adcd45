"""ctypes binding of libf3ps.so (the C ABI in include/f3ps.h).

This is the Python-side mirror of the reference's plugin interface for the hot path
(pcl::SupervoxelClustering as driven by main() + Clustering): same parameter names,
same error behaviour (std::logic_error -> LogicError, std::invalid_argument ->
ValueError).  There is no CPU fallback: without the CUDA library or without a GPU every
call raises.
"""
import ctypes as C
import os
import subprocess

import numpy as np

PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.path.join(PKG, "libf3ps.so")

LAB_CIEDE00, RGB_EUCL = 0, 1
NORMALS_DIFF, CONVEX_NORMALS_DIFF = 0, 1
MANUAL_LAMBDA, ADAPTIVE_LAMBDA, EQUALIZATION = 0, 1, 2
STAGES = ["voxelize", "neighbors", "normals", "seeds", "expand", "graph", "merge", "total", "merge_kernel"]


class F3psError(RuntimeError):
    pass


class LogicError(F3psError):
    """std::logic_error of the reference (src/clustering.cpp:576,591,672)."""


class Counts(C.Structure):
    _fields_ = [("n_points", C.c_int64), ("n_valid", C.c_int64), ("n_voxels", C.c_int64),
                ("depth", C.c_int32), ("seed_depth", C.c_int32), ("n_seed_cells", C.c_int32),
                ("n_seeds", C.c_int32), ("n_supervoxels", C.c_int32), ("n_edges", C.c_int32),
                ("n_merges", C.c_int32), ("n_segments", C.c_int32), ("n_edges_left", C.c_int32),
                ("rounds", C.c_int32), ("sweeps", C.c_int32), ("n_labeled", C.c_int32),
                ("lambda_", C.c_float), ("max_touched", C.c_int32),
                ("fold_steps", C.c_int64), ("nan_weights", C.c_int32), ("merge_path", C.c_int32)]


class SegmentInfo(C.Structure):
    """f3ps_segment_info, one 64-byte record per segment."""
    _fields_ = [("region_label", C.c_uint32), ("n_voxels", C.c_int32), ("n_points", C.c_int64),
                ("min_xyz", C.c_float * 3), ("max_xyz", C.c_float * 3), ("centroid", C.c_float * 3), ("mean_rgb", C.c_float * 3)]


SEGMENT_INFO_DTYPE = np.dtype({"names": [f[0] for f in SegmentInfo._fields_],
                               "formats": [np.uint32, np.int32, np.int64] + [(np.float32, 3)] * 4,
                               "offsets": [getattr(SegmentInfo, f[0]).offset for f in SegmentInfo._fields_], "itemsize": 64})

_lib = None


def build(force=False):
    """Compile libf3ps.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
    srcs = [os.path.join(PKG, "csrc", f) for f in os.listdir(os.path.join(PKG, "csrc"))
            if f.endswith((".cu", ".cuh", ".S"))]
    srcs.append(os.path.join(os.path.dirname(PKG), "include", "f3ps.h"))
    if force or not os.path.exists(LIB_PATH) or any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs):
        subprocess.check_call(["make", "-C", PKG, "-s"])
    return LIB_PATH


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise F3psError("libf3ps.so is not built (run __graft_entry__.build()); there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    vp, i64, i32, f32 = C.c_void_p, C.c_int64, C.c_int32, C.c_float
    sig = {
        "f3ps_create": (C.c_int, [C.c_int, vp, C.POINTER(vp)]),
        "f3ps_destroy": (None, [vp]),
        "f3ps_last_error": (C.c_char_p, [vp]),
        "f3ps_version": (C.c_char_p, []),
        "f3ps_set_vccs_params": (C.c_int, [vp, f32, f32, f32, f32, f32, C.c_int, C.c_int]),
        "f3ps_set_merge_params": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, f32, C.c_int]),
        "f3ps_set_input": (C.c_int, [vp, vp, i64, C.c_int, C.c_int]),
        "f3ps_voxelize": (C.c_int, [vp]), "f3ps_neighbors": (C.c_int, [vp]), "f3ps_normals": (C.c_int, [vp]),
        "f3ps_seeds": (C.c_int, [vp]), "f3ps_expand": (C.c_int, [vp]), "f3ps_graph": (C.c_int, [vp]),
        "f3ps_merge": (C.c_int, [vp, f32]), "f3ps_set_merge_kernel": (C.c_int, [vp, C.c_int]), "f3ps_set_blocking_wait": (C.c_int, [vp, C.c_int]), "f3ps_extract": (C.c_int, [vp]), "f3ps_run": (C.c_int, [vp, f32]),
        "f3ps_sync": (C.c_int, [vp]),
        "f3ps_set_graph": (C.c_int, [vp, i64, vp, vp, i32, vp, vp, vp, vp, i64, vp]),
        "f3ps_get_counts": (C.c_int, [vp, C.POINTER(Counts)]),
        "f3ps_get_voxel_keys": (C.c_int, [vp, vp, i64]),
        "f3ps_get_voxel_centroids": (C.c_int, [vp, vp, vp, vp, vp, i64]),
        "f3ps_get_point_voxel": (C.c_int, [vp, vp, i64]),
        "f3ps_get_voxel_neighbors": (C.c_int, [vp, vp, vp, i64]),
        "f3ps_get_voxel_normals": (C.c_int, [vp, vp, vp, i64]),
        "f3ps_get_seeds": (C.c_int, [vp, vp, i64]),
        "f3ps_get_voxel_labels": (C.c_int, [vp, vp, vp, i64]),
        "f3ps_get_supervoxels": (C.c_int, [vp, vp, vp, vp, vp, vp, i64]),
        "f3ps_get_supervoxel_voxels": (C.c_int, [vp, vp, vp, i64, i64]),
        "f3ps_get_adjacency": (C.c_int, [vp, vp, i64]),
        "f3ps_get_edges": (C.c_int, [vp, vp, vp, vp, vp, i64]),
        "f3ps_get_cdf": (C.c_int, [vp, vp, vp, i64]),
        "f3ps_get_merge_log": (C.c_int, [vp, vp, vp, vp, i64]),
        "f3ps_get_state_regions": (C.c_int, [vp, vp, vp, vp, vp, i64]),
        "f3ps_get_state_edges": (C.c_int, [vp, vp, vp, i64]),
        "f3ps_get_labeled_cloud": (C.c_int, [vp, vp, vp, vp, i64]),
        "f3ps_get_region_mean_color": (C.c_int, [vp, i32, vp]),
        "f3ps_get_voxel_segments_device": (C.c_int, [vp, C.POINTER(vp), C.POINTER(i64)]),
        "f3ps_merge_levels": (C.c_int, [vp, vp, C.c_int]),
        "f3ps_get_levels": (C.c_int, [vp, C.POINTER(i32), vp, vp, vp, i32]),
        "f3ps_get_level_voxel_labels": (C.c_int, [vp, vp, i64, C.c_int]),
        "f3ps_get_level_point_labels": (C.c_int, [vp, vp, i64, C.c_int]),
        "f3ps_get_segment_points": (C.c_int, [vp, C.c_int, vp, vp, i32, i64, C.c_int]),
        "f3ps_get_segment_voxels": (C.c_int, [vp, C.c_int, vp, vp, i32, i64, C.c_int]),
        "f3ps_get_segment_info": (C.c_int, [vp, C.c_int, vp, i32]),
        "f3ps_stage_ms": (C.c_int, [vp, C.c_int, C.POINTER(f32)]),
        "f3ps_launch_count": (i64, [vp]),
        "f3ps_merge_profile": (C.c_int, [vp, C.POINTER(C.c_uint64 * 32)]),
        "f3ps_merge_trace": (C.c_int, [vp, i64, vp, i64]),
        "f3ps_expand_profile": (C.c_int, [vp, C.POINTER(C.c_uint64 * 8)]),
        "f3ps_test_rgb2lab": (C.c_int, [vp, vp, vp, i64]),
        "f3ps_test_lab_ciede00": (C.c_int, [vp, vp, vp, vp, i64]),
        "f3ps_test_rgb_eucl": (C.c_int, [vp, vp, vp, vp, i64]),
        "f3ps_test_sort_pairs": (C.c_int, [vp, vp, vp, i64, C.c_int]),
        "f3ps_merge_batch": (C.c_int, [C.POINTER(vp), C.c_int, f32]),
        "f3ps_set_expand_sharing": (C.c_int, [vp, C.c_int, C.c_int]),
        "f3ps_set_expand_kernel": (C.c_int, [vp, C.c_int, C.c_int]),
        "f3ps_refine": (C.c_int, [vp, C.c_int]),

        "f3ps_eval_thresholds": (C.c_int, [vp, vp, i64, vp, i64, vp, C.c_int, vp, vp, vp]),
        "f3ps_eval_label_pairs": (C.c_int, [vp, vp, vp, i64, C.c_int, C.c_int, vp, i64, vp]),
        "f3ps_slab_reset": (C.c_int, [vp]),
        "f3ps_slab_bbox": (C.c_int, [vp, vp]),
        "f3ps_slab_set_frame": (C.c_int, [vp, vp]),
        "f3ps_slab_keys": (C.c_int, [vp, C.c_int, vp]),
        "f3ps_slab_route": (C.c_int, [vp, C.c_int, vp, vp, vp]),
        "f3ps_slab_choose_splitters": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, vp]),
        "f3ps_slab_array": (C.c_int, [vp, C.c_int, C.POINTER(vp), C.POINTER(i64), C.POINTER(C.c_int)]),
        "f3ps_slab_set_voxels": (C.c_int, [vp, i64, i64]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


EXPORTED = ["f3ps_create", "f3ps_destroy", "f3ps_last_error", "f3ps_version", "f3ps_set_vccs_params",
            "f3ps_set_merge_params", "f3ps_set_input", "f3ps_voxelize", "f3ps_neighbors", "f3ps_normals", "f3ps_seeds",
            "f3ps_expand", "f3ps_graph", "f3ps_merge", "f3ps_set_merge_kernel", "f3ps_set_blocking_wait", "f3ps_extract", "f3ps_run", "f3ps_sync", "f3ps_set_graph",
            "f3ps_get_counts", "f3ps_get_voxel_keys", "f3ps_get_voxel_centroids", "f3ps_get_point_voxel",
            "f3ps_get_voxel_neighbors", "f3ps_get_voxel_normals", "f3ps_get_seeds", "f3ps_get_voxel_labels",
            "f3ps_get_supervoxels", "f3ps_get_supervoxel_voxels", "f3ps_get_adjacency", "f3ps_get_edges", "f3ps_get_cdf",
            "f3ps_get_merge_log", "f3ps_get_state_regions", "f3ps_get_state_edges", "f3ps_get_labeled_cloud", "f3ps_get_region_mean_color",
            "f3ps_get_voxel_segments_device", "f3ps_merge_levels", "f3ps_get_levels", "f3ps_get_level_voxel_labels",
            "f3ps_get_level_point_labels", "f3ps_get_segment_points", "f3ps_get_segment_voxels", "f3ps_get_segment_info", "f3ps_stage_ms", "f3ps_launch_count", "f3ps_merge_profile", "f3ps_merge_trace", "f3ps_expand_profile", "f3ps_test_rgb2lab",
            "f3ps_test_lab_ciede00", "f3ps_test_rgb_eucl", "f3ps_test_sort_pairs",
            "f3ps_merge_batch", "f3ps_set_expand_sharing", "f3ps_set_expand_kernel", "f3ps_refine", "f3ps_eval_thresholds", "f3ps_eval_label_pairs", "f3ps_slab_reset", "f3ps_slab_bbox", "f3ps_slab_set_frame", "f3ps_slab_keys", "f3ps_slab_route", "f3ps_slab_array",
            "f3ps_slab_choose_splitters", "f3ps_slab_set_voxels"]


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def slab_choose_splitters(hist, world, shift):
    """Slab mode's equal-count cuts of the key space (f3ps_slab_choose_splitters, no device needed): world-1 ascending
    Morton keys from a histogram of the keys' top bits (bin = key >> shift); rank r owns [splitters[r-1], splitters[r])."""
    h = np.ascontiguousarray(hist, np.uint32)
    out = np.zeros(max(1, world - 1), np.uint64)
    rc = lib().f3ps_slab_choose_splitters(_p(h), h.shape[0], world, shift, _p(out))
    if rc:
        raise ValueError("f3ps_slab_choose_splitters: bad arguments (status %d)" % rc)
    return out[:world - 1]


def merge_batch(segs, threshold):
    """Clustering::cluster(threshold) for many handles with one launch of the resident merge kernel (f3ps_merge_batch)."""
    if not segs:
        return
    arr = (C.c_void_p * len(segs))(*[s.h for s in segs])
    rc = lib().f3ps_merge_batch(arr, len(segs), threshold)
    if rc:
        for s in segs:
            msg = s.L.f3ps_last_error(s.h).decode()
            if msg:
                s._chk(rc)
        raise F3psError("f3ps_merge_batch failed with status %d" % rc)


class Segmenter:
    """One handle = one GPU + one stream (f3ps_create)."""

    def __init__(self, device=0, stream=None):
        self.L = lib()
        h = C.c_void_p()
        rc = self.L.f3ps_create(device, stream, C.byref(h))
        if rc:
            raise F3psError("f3ps_create failed (status %d): no usable CUDA device; there is no CPU fallback" % rc)
        self.h = h
        self._keep = None

    def close(self):
        if getattr(self, "h", None):
            self.L.f3ps_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc == 0:
            return
        msg = self.L.f3ps_last_error(self.h).decode()
        if rc == 1:
            raise ValueError(msg)
        if rc == 2:
            raise LogicError(msg)
        raise F3psError("status %d: %s" % (rc, msg))

    # ---- parameters (same defaults as the CLI, src/supervoxel_clustering.cpp:247-267) ----
    def set_vccs_params(self, voxel_res=0.008, seed_res=0.08, color=0.2, spatial=0.4, normal=1.0,
                        use_transform=True, fold_negative_z=True):
        self._chk(self.L.f3ps_set_vccs_params(self.h, voxel_res, seed_res, color, spatial, normal,
                                              int(use_transform), int(fold_negative_z)))

    def set_merge_params(self, color_mode=LAB_CIEDE00, geom_mode=NORMALS_DIFF, merge_mode=ADAPTIVE_LAMBDA, lam=0.5, bins=500):
        self._chk(self.L.f3ps_set_merge_params(self.h, color_mode, geom_mode, merge_mode, lam, bins))
        self._bins = bins

    # ---- input ----
    def set_input(self, pts):
        """pts: numpy structured array (32-byte pcl::PointXYZRGBA records) or any 16/32-byte record array."""
        pts = np.ascontiguousarray(pts)
        self._keep = pts
        self._chk(self.L.f3ps_set_input(self.h, _p(pts), pts.shape[0], pts.dtype.itemsize, 0))

    def set_input_device(self, dev_ptr, n, stride=32):
        self._chk(self.L.f3ps_set_input(self.h, C.c_void_p(dev_ptr), n, stride, 1))

    # ---- stages ----
    def voxelize(self): self._chk(self.L.f3ps_voxelize(self.h))
    def neighbors(self): self._chk(self.L.f3ps_neighbors(self.h))
    def normals(self): self._chk(self.L.f3ps_normals(self.h))
    def seeds(self): self._chk(self.L.f3ps_seeds(self.h))
    def expand(self): self._chk(self.L.f3ps_expand(self.h))
    def refine(self, num_itr=3): self._chk(self.L.f3ps_refine(self.h, num_itr))
    def graph(self): self._chk(self.L.f3ps_graph(self.h))
    def merge(self, threshold): self._chk(self.L.f3ps_merge(self.h, threshold))
    def set_merge_kernel(self, which): self._chk(self.L.f3ps_set_merge_kernel(self.h, which))
    def set_blocking_wait(self, on): self._chk(self.L.f3ps_set_blocking_wait(self.h, int(on)))
    def set_expand_kernel(self, which, cluster_ctas=0): self._chk(self.L.f3ps_set_expand_kernel(self.h, which, cluster_ctas))
    def set_expand_sharing(self, ctas_per_frame, max_concurrent=0): self._chk(self.L.f3ps_set_expand_sharing(self.h, ctas_per_frame, max_concurrent))
    def extract(self): self._chk(self.L.f3ps_extract(self.h))
    def run(self, threshold=0.2): self._chk(self.L.f3ps_run(self.h, threshold))
    def sync(self): self._chk(self.L.f3ps_sync(self.h))

    def set_graph(self, vxyz, vrgba, labels, vox_lists, centroids, normals, adj_pairs):
        """Clustering::set_initialstate on caller-supplied supervoxels (voxel index lists per supervoxel)."""
        vxyz = np.ascontiguousarray(vxyz, np.float32)
        vrgba = np.ascontiguousarray(vrgba, np.uint32)
        labels = np.ascontiguousarray(labels, np.uint32)
        order = np.concatenate(vox_lists).astype(np.int64) if len(vox_lists) else np.zeros(0, np.int64)
        off = np.zeros(len(vox_lists) + 1, np.int64)
        off[1:] = np.cumsum([len(v) for v in vox_lists])
        gx = np.ascontiguousarray(vxyz[order])
        gc = np.ascontiguousarray(vrgba[order])
        centroids = np.ascontiguousarray(centroids, np.float32)
        normals = np.ascontiguousarray(normals, np.float32)
        adj = np.ascontiguousarray(adj_pairs, np.uint32).reshape(-1, 2)
        self._graph_order = order
        self._chk(self.L.f3ps_set_graph(self.h, gx.shape[0], _p(gx), _p(gc), len(labels), _p(labels), _p(off),
                                        _p(centroids), _p(normals), adj.shape[0], _p(adj)))

    # ---- results ----
    def counts(self):
        c = Counts()
        self._chk(self.L.f3ps_get_counts(self.h, C.byref(c)))
        return c

    def stage_ms(self):
        out = {}
        v = C.c_float()
        for i, name in enumerate(STAGES):
            if self.L.f3ps_stage_ms(self.h, i, C.byref(v)) == 0:
                out[name] = v.value
        return out

    def merge_profile(self):
        a = (C.c_uint64 * 32)()
        self._chk(self.L.f3ps_merge_profile(self.h, C.byref(a)))
        v = list(a)
        if self.counts().merge_path in (1, 3, 6):  # resident kernel; cycle counters only after set_merge_kernel(4) / (5)
            return {"worker": dict(zip(["scan_publish", "wait_s1_head", "incidence_w1", "dedupe_spec_ciede", "wait_fold", "weights_stamps", "wait_w4"], v[0:7])),
                    "mean": dict(zip(["wait_voxels", "fold", "lab_publish", "wait_s1"], v[12:16])),
                    "cov": dict(zip(["wait_voxels", "fold", "eigen_publish", "wait_s1"], v[16:20])),
                    "by_touched": {k: {"merges": v[28 + i], "cycles_per_merge": (v[8 + i] // v[28 + i]) if v[28 + i] else 0}
                                   for i, k in enumerate(["T<=32", "T<=128", "T>128"])},
                    "wide": {"merges": v[31], "cycles_per_merge": (v[11] // v[31]) if v[31] else 0, "worker_total": v[7],
                             "phases": dict(zip(["entries_marks_guess", "dedupe_colour_wait_fold", "weights_classes_list", "stamps_keys_clear"], v[20:24]))},
                    "guess_misses": v[24], "ciede_evals": v[25], "sum_T": v[27]}
        return dict(zip(["argmin", "fold", "order", "delta", "stamps", "wait_scan", "sum_T", "fold_tail"], v[:8]))

    def merge_trace(self, first=None):
        """first given: set the window for the next merge (kernel choice 4).  Else: the recorded window as a [256, 32] array of
        SM clock values: worker thread 0: 0 loop top, 1 rescan done, 2 head known, 3 entries read / marks set, 4 colour deltas
        done, 5 after F, 6 weights + stamps done, 7 after W4, 8 = adjacency entries read; covariance warp: 12 head known,
        13 voxels fetched, 14 folded, 15 eigen-solve done, 21 = voxels of b; mean warp: 16 head known, 17 guess published,
        18 voxels fetched, 19 folded, 20 Lab done."""
        if first is not None:
            self._chk(self.L.f3ps_merge_trace(self.h, int(first), None, 0))
            return None
        out = np.zeros((256, 32), np.uint32)
        self._chk(self.L.f3ps_merge_trace(self.h, 0, out.ctypes.data_as(C.c_void_p), out.size))
        return out

    def expand_profile(self):
        a = (C.c_uint64 * 8)()
        self._chk(self.L.f3ps_expand_profile(self.h, C.byref(a)))
        return dict(zip(["init", "sweeps", "count", "alloc", "fill", "fold", "tail"], list(a)[:7]))

    def launch_count(self):
        return int(self.L.f3ps_launch_count(self.h))

    def array(self, name):
        """Named result arrays (the names the parity tests use for both sides)."""
        c = self.counts()
        V, S0, S, E = c.n_voxels, c.n_seeds, c.n_supervoxels, c.n_edges
        if name == "keys":
            a = np.zeros((V, 3), np.uint32); self._chk(self.L.f3ps_get_voxel_keys(self.h, _p(a), V)); return a
        if name in ("voxel_xyz", "voxel_rgb", "voxel_rgba", "voxel_count"):
            x = np.zeros((V, 3), np.float32); r = np.zeros((V, 3), np.float32); q = np.zeros(V, np.uint32); n = np.zeros(V, np.int32)
            self._chk(self.L.f3ps_get_voxel_centroids(self.h, _p(x), _p(r), _p(q), _p(n), V))
            return {"voxel_xyz": x, "voxel_rgb": r, "voxel_rgba": q, "voxel_count": n}[name]
        if name == "point_voxel":
            a = np.zeros(c.n_points, np.int32); self._chk(self.L.f3ps_get_point_voxel(self.h, _p(a), c.n_points)); return a
        if name in ("nbr", "nbr_count"):
            a = np.zeros((V, 27), np.int32); n = np.zeros(V, np.int32)
            self._chk(self.L.f3ps_get_voxel_neighbors(self.h, _p(a), _p(n), V)); return a if name == "nbr" else n
        if name in ("normals", "curvature"):
            a = np.zeros((V, 4), np.float32); k = np.zeros(V, np.float32)
            self._chk(self.L.f3ps_get_voxel_normals(self.h, _p(a), _p(k), V)); return a if name == "normals" else k
        if name == "seeds":
            a = np.zeros(S0, np.int32); self._chk(self.L.f3ps_get_seeds(self.h, _p(a), S0)); return a
        if name in ("labels", "dist"):
            a = np.zeros(V, np.uint32); d = np.zeros(V, np.float32)
            self._chk(self.L.f3ps_get_voxel_labels(self.h, _p(a), _p(d), V)); return a if name == "labels" else d
        if name in ("sv_label", "sv_xyz", "sv_rgb", "sv_normal", "sv_count"):
            l = np.zeros(S, np.uint32); x = np.zeros((S, 3), np.float32); r = np.zeros((S, 3), np.float32)
            n4 = np.zeros((S, 4), np.float32); n = np.zeros(S, np.int32)
            self._chk(self.L.f3ps_get_supervoxels(self.h, _p(l), _p(x), _p(r), _p(n4), _p(n), S))
            return {"sv_label": l, "sv_xyz": x, "sv_rgb": r, "sv_normal": n4, "sv_count": n}[name]
        if name == "adj":
            a = np.zeros((2 * E, 2), np.uint32); self._chk(self.L.f3ps_get_adjacency(self.h, _p(a), 2 * E)); return a
        if name in ("edges_ab", "edges_dc", "edges_dg", "edges_w"):
            ab = np.zeros((E, 2), np.uint32); dc = np.zeros(E, np.float32); dg = np.zeros(E, np.float32); w = np.zeros(E, np.float32)
            self._chk(self.L.f3ps_get_edges(self.h, _p(ab), _p(dc), _p(dg), _p(w), E))
            return {"edges_ab": ab, "edges_dc": dc, "edges_dg": dg, "edges_w": w}[name]
        if name in ("cdf_c", "cdf_g"):
            n = self._bins
            a = np.zeros(n, np.float32); b = np.zeros(n, np.float32)
            self._chk(self.L.f3ps_get_cdf(self.h, _p(a), _p(b), n)); return a if name == "cdf_c" else b
        if name in ("merges_ab", "merges_w", "merges_left"):
            M = c.n_merges
            ab = np.zeros((M, 2), np.uint32); w = np.zeros(M, np.float32); left = np.zeros((M, 2), np.uint32)
            self._chk(self.L.f3ps_get_merge_log(self.h, _p(ab), _p(w), _p(left), M))
            return {"merges_ab": ab, "merges_w": w, "merges_left": left}[name]
        if name in ("final_ab", "final_w"):
            n = c.n_edges_left
            ab = np.zeros((n, 2), np.uint32); w = np.zeros(n, np.float32)
            self._chk(self.L.f3ps_get_state_edges(self.h, _p(ab), _p(w), n)); return ab if name == "final_ab" else w
        if name in ("out_xyz", "out_label", "out_voxel"):
            n = c.n_labeled
            x = np.zeros((n, 3), np.float32); l = np.zeros(n, np.uint32); v = np.zeros(n, np.uint32)
            self._chk(self.L.f3ps_get_labeled_cloud(self.h, _p(x), _p(l), _p(v), n))
            return {"out_xyz": x, "out_label": l, "out_voxel": v}[name]
        raise KeyError(name)

    def fetch_result(self):
        """The result of a frame in one go: labelled voxel cloud (Clustering::get_labeled_cloud) + merge log, one size query."""
        c = self.counts()
        n, M = c.n_labeled, c.n_merges
        x = np.empty((n, 3), np.float32); l = np.empty(n, np.uint32); v = np.empty(n, np.uint32)
        self._chk(self.L.f3ps_get_labeled_cloud(self.h, _p(x), _p(l), _p(v), n))
        ab = np.empty((M, 2), np.uint32); w = np.empty(M, np.float32); left = np.empty((M, 2), np.uint32)
        self._chk(self.L.f3ps_get_merge_log(self.h, _p(ab), _p(w), _p(left), M))
        return {"out_xyz": x, "out_label": l, "out_voxel": v, "merges_ab": ab, "merges_w": w, "merges_left": left}

    def state_regions(self):
        n = self.counts().n_segments
        l = np.zeros(n, np.uint32); x = np.zeros((n, 3), np.float32); nn = np.zeros((n, 3), np.float32); k = np.zeros(n, np.int32)
        self._chk(self.L.f3ps_get_state_regions(self.h, _p(l), _p(x), _p(nn), _p(k), n))
        return l, x, nn, k

    # ---- segmentation levels: several thresholds from one merge replay ----
    def merge_levels(self, thresholds):
        """One replay, merge(max(thresholds)), recording the segmentation at every threshold (1 to 256, finite, non-decreasing)."""
        t = np.ascontiguousarray(thresholds, np.float32).ravel()
        self._chk(self.L.f3ps_merge_levels(self.h, _p(t) if t.size else None, t.size))

    def levels(self):
        """{"thresholds", "n_merges", "n_segments"} of the recorded levels (a plain merge records one: its threshold)."""
        n = self._n_levels()
        t = np.zeros(n, np.float32); m = np.zeros(n, np.int32); s = np.zeros(n, np.int32)
        self._chk(self.L.f3ps_get_levels(self.h, None, _p(t), _p(m), _p(s), n))
        return {"thresholds": t, "n_merges": m, "n_segments": s}

    def _n_levels(self):
        n = C.c_int32()
        self._chk(self.L.f3ps_get_levels(self.h, C.byref(n), None, None, None, 0))
        return n.value

    def voxel_labels(self):
        """uint32 [L, V]: the segment of every voxel at every level (0xffffffff: no supervoxel owns it)."""
        out = np.empty((self._n_levels(), self.counts().n_voxels), np.uint32)
        self._chk(self.L.f3ps_get_level_voxel_labels(self.h, _p(out), out.size, 0))
        return out

    def point_labels(self):
        """uint32 [L, N]: the segment of every input point at every level, in input order (0xffffffff: no voxel)."""
        out = np.empty((self._n_levels(), self.counts().n_points), np.uint32)
        self._chk(self.L.f3ps_get_level_point_labels(self.h, _p(out), out.size, 0))
        return out

    def point_labels_device(self, dev_ptr, capacity):
        """point_labels() into a CUDA buffer of `capacity` uint32 elements (e.g. a torch tensor's data_ptr()), enqueued on the
        handle's stream without waiting: sync() before reading it from another stream or the host."""
        self._chk(self.L.f3ps_get_level_point_labels(self.h, C.c_void_p(dev_ptr), capacity, 1))

    # ---- segment extraction: the members of every segment of one level, and one descriptor per segment ----
    def _level(self, level):
        """level index of the recorded levels; negative counts from the end (out of range: the C call's ValueError)"""
        return level + self._n_levels() if level < 0 else level

    def _segments(self, fn, level, n_members):
        k = self._level(level)
        lv = self.levels()
        K = int(lv["n_segments"][k]) if 0 <= k < len(lv["n_segments"]) else 0
        off = np.empty(K + 1, np.int64); idx = np.empty(n_members, np.int32)
        self._chk(fn(self.h, k, _p(off), _p(idx), off.size, idx.size, 0))
        return off, idx[:off[-1]]

    def segment_points(self, level=-1):
        """(offsets int64 [K+1], index int32 [n]): the input points of segment j of the level at index[offsets[j]:offsets[j+1]],
        ascending; points without a segment are left out."""
        return self._segments(self.L.f3ps_get_segment_points, level, self.counts().n_points)

    def segment_voxels(self, level=-1):
        """segment_points() over voxels (after set_graph voxel i is the i-th voxel passed in)."""
        return self._segments(self.L.f3ps_get_segment_voxels, level, self.counts().n_voxels)

    def segment_points_device(self, level, offsets_ptr, index_ptr, cap_segments, cap_points):
        """segment_points() into CUDA buffers (e.g. torch tensors' data_ptr(): int64 offsets, int32 index), enqueued on the
        handle's stream: sync() before reading them from another stream or the host."""
        self._chk(self.L.f3ps_get_segment_points(self.h, self._level(level), C.c_void_p(offsets_ptr), C.c_void_p(index_ptr),
                                                 cap_segments, cap_points, 1))

    def segment_info(self, level=-1):
        """One descriptor per segment of the level, as numpy arrays: region_label, n_voxels, n_points, min_xyz, max_xyz, centroid,
        mean_rgb (the last four [K, 3] float32)."""
        k = self._level(level)
        n = self._n_levels()
        K = int(self.levels()["n_segments"][k]) if 0 <= k < n else 0
        recs = (SegmentInfo * max(K, 1))()
        self._chk(self.L.f3ps_get_segment_info(self.h, k, recs, K))
        a = np.frombuffer(recs, SEGMENT_INFO_DTYPE, count=K)
        return {name: np.ascontiguousarray(a[name]) for name in a.dtype.names}

    def supervoxel_voxels(self):
        c = self.counts()
        cap = c.n_voxels + c.n_supervoxels          # a surviving phantom leaf is listed by its holder as well
        idx = np.zeros(cap, np.int32); off = np.zeros(c.n_supervoxels + 1, np.int64)
        self._chk(self.L.f3ps_get_supervoxel_voxels(self.h, _p(idx), _p(off), cap, c.n_supervoxels))
        return idx[:off[-1]], off

    # ---- auto-threshold sweep: Clustering::all_thresh / best_thresh (src/clustering.cpp:691-774) ----
    PERF_FIELDS = ("voi", "precision", "recall", "fscore", "wov", "fpr", "fnr")

    @staticmethod
    def sweep_thresholds(start=0.8, end=1.0, step=0.005):
        """The thresholds all_thresh visits: start, then `t += step` in float while t <= end (:711-718)."""
        start, end, step = np.float32(start), np.float32(end), np.float32(step)
        if start > end:
            start, end = end, start
        out = [start]
        t = np.float32(start + step)
        while t <= end:
            out.append(t)
            t = np.float32(t + step)
        return np.array(out, np.float32)

    def all_thresh(self, truth_label, start=0.8, end=1.0, step=0.005, extra_truth=None):
        """{threshold: performanceSet dict} for every threshold of the sweep, from one merge replay on the device."""
        for v in (start, end, step):
            if v < 0 or v > 1:
                raise IndexError("start_thresh, end_thresh and/or step_thresh outside of range [0, 1]")   # std::out_of_range (:694-698)
        thr = self.sweep_thresholds(start, end, step)
        truth = np.ascontiguousarray(truth_label, np.uint32)
        perf = np.zeros((len(thr), 7), np.float32)
        nseg = np.zeros(len(thr), np.int32); nm = np.zeros(len(thr), np.int32)
        extra = None if extra_truth is None else np.ascontiguousarray(extra_truth, np.uint32)
        self._chk(self.L.f3ps_eval_thresholds(self.h, _p(truth), truth.shape[0], _p(extra), 0 if extra is None else extra.shape[0],
                                              _p(thr), len(thr), _p(perf), _p(nseg), _p(nm)))
        self.last_sweep = {"thresholds": thr, "perf": perf, "n_segments": nseg, "n_merges": nm}
        return {float(t): dict(zip(self.PERF_FIELDS, map(float, perf[k]))) for k, t in enumerate(thr)}

    def best_thresh(self, truth_label, start=0.8, end=1.0, step=0.005):
        """(threshold, performanceSet) with the largest F-score; the first one wins ties, 0 / zeros if none is positive (:759-774)."""
        res = self.all_thresh(truth_label, start, end, step)
        best_t, best = 0.0, dict.fromkeys(self.PERF_FIELDS, 0.0)
        for t in sorted(res):
            if res[t]["fscore"] > best["fscore"]:
                best_t, best = t, res[t]
        return best_t, best

    def eval_clouds(self, seg_xyz, seg_label, truth_xyz, truth_label):
        """Testing(segm, truth).eval_performance() (/root/reference/src/testing.cpp:62-146, 239-406) for one pair of labelled clouds:
        the host pairs the points by exact xyz (compareXYZ: -0 == +0; the first truth point of an xyz wins, as std::map::insert) and
        renumbers the labels densely in ascending order -- what host/facade.cpp's Testing does --, the contingency table and the seven
        scores come from f3ps_eval_label_pairs on the device."""
        sx = np.ascontiguousarray(seg_xyz, np.float32) + np.float32(0); tx = np.ascontiguousarray(truth_xyz, np.float32) + np.float32(0)   # -0 -> +0
        su, sd = np.unique(np.asarray(seg_label, np.uint32), return_inverse=True)
        tu, td = np.unique(np.asarray(truth_label, np.uint32), return_inverse=True)
        where = {}
        for k, j in zip(map(bytes, tx.view(np.uint8).reshape(len(tx), 12)), td):
            where.setdefault(k, int(j))
        nt = len(tu)
        tl = np.array([where.get(k, nt) for k in map(bytes, sx.view(np.uint8).reshape(len(sx), 12))], np.uint32)
        sl = np.ascontiguousarray(sd, np.uint32)
        tsizes = np.bincount(td, minlength=nt).astype(np.uint64)
        perf = np.zeros(7, np.float32)
        self._chk(self.L.f3ps_eval_label_pairs(self.h, _p(sl), _p(tl), len(sl), len(su), nt, _p(tsizes), len(tx), _p(perf)))
        return dict(zip(self.PERF_FIELDS, map(float, perf)))

    # ---- slab mode (per-rank pieces; f3ps/slab.py issues the exchanges between them) ----
    SLAB_ARRAYS = {"vox_xyz": 0, "vox_rgb": 1, "vox_key": 2, "vox_normal": 3, "vox_curv": 4}

    def slab_reset(self): self._chk(self.L.f3ps_slab_reset(self.h))
    def slab_bbox(self, d_box8): self._chk(self.L.f3ps_slab_bbox(self.h, C.c_void_p(d_box8)))
    def slab_set_frame(self, d_box8): self._chk(self.L.f3ps_slab_set_frame(self.h, C.c_void_p(d_box8)))

    def slab_keys(self, top_bits, d_hist): self._chk(self.L.f3ps_slab_keys(self.h, top_bits, C.c_void_p(d_hist)))

    def slab_route(self, world, d_hist, d_send):
        """d_hist: the all-reduced key histogram (device pointer).  Returns the records packed for each destination rank."""
        counts = np.zeros(world, np.int64)
        self._chk(self.L.f3ps_slab_route(self.h, world, C.c_void_p(d_hist), C.c_void_p(d_send), _p(counts)))
        return counts

    def slab_array(self, name):
        """(device pointer, elements, bytes per element) of an array the slab driver exchanges in place."""
        ptr, n, eb = C.c_void_p(), C.c_int64(), C.c_int()
        self._chk(self.L.f3ps_slab_array(self.h, self.SLAB_ARRAYS[name], C.byref(ptr), C.byref(n), C.byref(eb)))
        return (ptr.value or 0), n.value, eb.value

    def slab_set_voxels(self, n_voxels, own_begin): self._chk(self.L.f3ps_slab_set_voxels(self.h, n_voxels, own_begin))

    # ---- device self tests ----
    def test_rgb2lab(self, rgb255):
        a = np.ascontiguousarray(rgb255, np.float32).reshape(-1, 3); o = np.zeros_like(a)
        self._chk(self.L.f3ps_test_rgb2lab(self.h, _p(a), _p(o), a.shape[0])); return o

    def test_lab_ciede00(self, l1, l2):
        a = np.ascontiguousarray(l1, np.float32).reshape(-1, 3); b = np.ascontiguousarray(l2, np.float32).reshape(-1, 3)
        o = np.zeros(a.shape[0], np.float32)
        self._chk(self.L.f3ps_test_lab_ciede00(self.h, _p(a), _p(b), _p(o), a.shape[0])); return o

    def test_rgb_eucl(self, c1, c2):
        a = np.ascontiguousarray(c1, np.float32).reshape(-1, 3); b = np.ascontiguousarray(c2, np.float32).reshape(-1, 3)
        o = np.zeros(a.shape[0], np.float32)
        self._chk(self.L.f3ps_test_rgb_eucl(self.h, _p(a), _p(b), _p(o), a.shape[0])); return o

    def test_sort_pairs(self, keys, values, key_bits):
        k = np.ascontiguousarray(keys, np.uint64).copy(); v = np.ascontiguousarray(values, np.uint32).copy()
        self._chk(self.L.f3ps_test_sort_pairs(self.h, _p(k), _p(v), k.shape[0], key_bits)); return k, v

    _bins = 500
