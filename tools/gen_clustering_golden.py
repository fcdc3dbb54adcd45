#!/usr/bin/env python
"""Golden vectors of the REFERENCE's own Clustering class (SURVEY.md section 8a rows a10-a24, the K6 / K7 half of the hot path):
/root/reference/src/clustering.cpp + clustering_state.cpp + color_utilities.cpp compiled where they lie against the stand-ins of
oracle/ref_shim/ (oracle/Makefile, target `ref` -> oracle/_ref/libref_clustering.so), driven as main() drives them
(set_initialstate + cluster(threshold), /root/reference/src/supervoxel_clustering.cpp:408-443) on
  * hub + ring graphs (a region adjacent to everything, duplicates (a,x)/(b,x), few colours -> ties) in five flag sets, and
  * the supervoxels of the 160x120 synthetic frame (1,646 supervoxels, 4,635 edges) in the three flag sets BASELINE.json names, and
  * the supervoxels of the 640x480 frame of the headline benchmark (2,274 supervoxels, 7,592 edges, --CVX --AL -t 0.2: 2,267 merges).
Inputs and the reference's outputs -- its per-merge debug lines (a, b, weight bits, edges / regions left), the adaptive lambda, the
regions that remain and the labelled cloud -- and, for three threshold sweeps, Clustering::all_thresh / best_thresh (the automatic
threshold of main(), :428-438: every threshold's seven scores and the chosen one) are committed as tests/golden/clustering_ref.npz.
Build container only."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle")); sys.path.insert(0, os.path.join(ROOT, "fast-3d-pointcloud-segmentation_b200"))
OUT = os.path.join(ROOT, "tests", "golden", "clustering_ref.npz")


def ref_lib():
    if not os.path.isdir(os.environ.get("F3PS_REFERENCE_DIR", "")):
        raise SystemExit("set F3PS_REFERENCE_DIR to a checkout of the original project: oracle/_ref/libref_clustering.so is built from its sources")
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "-s"])
    lib = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_clustering.so"))
    lib.ref_cluster.restype = C.c_int
    return lib


def ref_cluster(lib, lut, vxyz, vrgba, labels, lists, cen, nrm, adj, color, geom, merging, lam, bins, thr):
    """Clustering(color, geom, merging) [+ set_lambda / set_bins_num] . set_initialstate . cluster(thr) of the compiled reference"""
    S = len(labels)
    order = np.concatenate(lists) if S else np.zeros(0, int)
    off = np.concatenate([[0], np.cumsum([len(l) for l in lists])]).astype(np.int64)
    vx = np.ascontiguousarray(np.asarray(vxyz, np.float32)[order]); vc = np.ascontiguousarray(np.asarray(vrgba, np.uint32)[order])
    labels = np.ascontiguousarray(labels, np.uint32); cen = np.ascontiguousarray(cen, np.float32); nrm = np.ascontiguousarray(nrm, np.float32)
    adj = np.ascontiguousarray(adj, np.uint32)
    capm, cape, capp = S + 1, len(adj) + 1, len(order) + 1
    m_ab = np.zeros((capm, 2), np.uint32); m_w = np.zeros(capm, np.float32); m_left = np.zeros((capm, 2), np.uint32); nm = C.c_int64()
    f_ab = np.zeros((cape, 2), np.uint32); ne = C.c_int64()
    r_label = np.zeros(S + 1, np.uint32); r_size = np.zeros(S + 1, np.int32); r_cen = np.zeros((S + 1, 3), np.float32)
    r_n4 = np.zeros((S + 1, 4), np.float32); nr = C.c_int32()
    o_label = np.zeros(capp, np.uint32); o_xyz = np.zeros((capp, 3), np.float32); npnt = C.c_int64(); lam_out = C.c_float()
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    rc = lib.ref_cluster(p(lut), C.c_int32(S), p(labels), p(off), p(vx), p(vc), p(cen), p(nrm), C.c_int64(len(adj)), p(adj), C.c_int(color), C.c_int(geom),
                         C.c_int(merging), C.c_float(lam), C.c_int(bins), C.c_float(thr), C.c_int64(capm), p(m_ab), p(m_w), p(m_left), C.byref(nm),
                         C.c_int64(cape), p(f_ab), C.byref(ne), p(r_label), p(r_size), p(r_cen), p(r_n4), C.byref(nr), C.c_int64(capp), p(o_label), p(o_xyz),
                         C.byref(npnt), C.byref(lam_out))
    if rc:
        raise RuntimeError("the reference threw")
    M = nm.value
    return dict(merges_ab=m_ab[:M].copy(), merges_w=m_w[:M].copy(), merges_left=m_left[:M].copy(), final_ab=f_ab[:ne.value].copy(),
                region_label=r_label[:nr.value].copy(), region_size=r_size[:nr.value].copy(), region_centroid=r_cen[:nr.value].copy(),
                region_normal4=r_n4[:nr.value].copy(), out_label=o_label[:npnt.value].copy(), out_xyz=o_xyz[:npnt.value].copy(),
                lam=np.float32(lam_out.value))


def ref_all_thresh(lib, lut, vxyz, vrgba, labels, lists, cen, nrm, adj, color, geom, merging, lam, bins, truth_per_voxel, start, end, step):
    """Clustering::all_thresh + best_thresh of the compiled reference; truth_per_voxel is indexed like vxyz"""
    S = len(labels)
    order = np.concatenate(lists)
    off = np.concatenate([[0], np.cumsum([len(l) for l in lists])]).astype(np.int64)
    vx = np.ascontiguousarray(np.asarray(vxyz, np.float32)[order]); vc = np.ascontiguousarray(np.asarray(vrgba, np.uint32)[order])
    tl = np.ascontiguousarray(np.asarray(truth_per_voxel, np.uint32)[order])
    labels = np.ascontiguousarray(labels, np.uint32); cen = np.ascontiguousarray(cen, np.float32); nrm = np.ascontiguousarray(nrm, np.float32)
    adj = np.ascontiguousarray(adj, np.uint32)
    cap = 512
    out_t = np.zeros(cap, np.float32); out_p = np.zeros((cap, 7), np.float32); n = C.c_int32(); best = np.zeros(8, np.float32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    lib.ref_all_thresh.restype = C.c_int
    rc = lib.ref_all_thresh(p(lut), C.c_int32(S), p(labels), p(off), p(vx), p(vc), p(cen), p(nrm), C.c_int64(len(adj)), p(adj), C.c_int(color), C.c_int(geom),
                            C.c_int(merging), C.c_float(lam), C.c_int(bins), p(tl), C.c_float(start), C.c_float(end), C.c_float(step), C.c_int32(cap),
                            p(out_t), p(out_p), C.byref(n), p(best))
    if rc:
        raise RuntimeError("the reference threw")
    return out_t[:n.value].copy(), out_p[:n.value].copy(), best


def hub_graph(n_leaves, seed):
    """two hubs + a ring of leaves (tests/test_gpu_parity.py::test_general_merge_kernel_hub_graph, smaller)"""
    rng = np.random.default_rng(seed)
    S = n_leaves + 2
    sizes = rng.integers(3, 7, S); sizes[0] = 40; sizes[1] = 25
    V = int(sizes.sum())
    vxyz = (rng.normal(0, 1, (V, 3)) + 3).astype(np.float32)
    base = rng.integers(0, 6, S)
    vrgba = np.repeat((base * 40 + 20).astype(np.uint32), sizes) * np.uint32(0x010101) + rng.integers(0, 3, V).astype(np.uint32)
    labels = np.arange(1, S + 1, dtype=np.uint32)
    off = np.concatenate([[0], np.cumsum(sizes)])
    lists = [np.arange(off[i], off[i + 1]) for i in range(S)]
    cen = np.stack([vxyz[l].mean(0) for l in lists]).astype(np.float32)
    nrm = rng.normal(0, 1, (S, 3)).astype(np.float32); nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    pairs = {(0, 1)}
    for i in range(2, S):
        pairs.add((0, i))
        if i % 2: pairs.add((1, i))
        if i + 1 < S: pairs.add((i, i + 1))
    adj = []
    for i, j in sorted(pairs): adj += [(labels[i], labels[j]), (labels[j], labels[i])]
    return vxyz, vrgba, labels, lists, cen, nrm, np.array(sorted(adj), np.uint32)


def frame_graph(vga=False, bundled=False):
    """the supervoxels PCL's VCCS would hand to set_initialstate, from the oracle's front half on the 160x120 synthetic frame
    (vga: on the 640x480 frame bench.py's headline and the exact-merge-sequence test use, seed 20020; bundled: on the reference's
    own cloud, pcd/milk_cartoon_all_small_clorox.pcd = tests/fixtures/, loaded as main() does with z < 0 folded -- BASELINE configs[0])"""
    import oracle_py
    from f3ps import pcd, synth
    o = oracle_py.Oracle(); o.set_vccs_params(fold_negative_z=True) if bundled else o.set_vccs_params()
    o.set_merge_params(merge_impl=1, color_mode=0, geom_mode=1, merge_mode=1)
    if bundled:
        pts = pcd.read_pcd(os.path.join(ROOT, "tests", "fixtures", "milk_cartoon_all_small_clorox.pcd"))[0]
    else:
        pts = synth.make_frame(seed=20020) if vga else synth.make_frame(seed=11, width=160, height=120)
    o.set_input(pts); o.run(0, 0.2)
    labels = o.array("sv_label").copy(); vl = o.array("labels")
    lists = [np.nonzero(vl == l)[0] for l in labels]
    return (o.array("voxel_xyz").copy(), o.array("voxel_rgba").copy(), labels, lists, o.array("sv_xyz").copy(), o.array("sv_normal")[:, :3].copy(), o.array("adj").copy())


CASES = [   # name, graph, flags (color, geom, merging, lambda, bins), threshold
    ("hub60_lab_cvx_al", ("hub", 60), (0, 1, 1, 0.5, 500), 0.3),
    ("hub60_rgb_eq7", ("hub", 60), (1, 0, 2, 0.5, 7), 0.95),
    ("hub150_rgb_cvx_ml", ("hub", 150), (1, 1, 0, 0.5, 500), 0.3),
    ("hub150_lab_eq200", ("hub", 150), (0, 0, 2, 0.5, 200), 0.6),
    ("hub400_lab_cvx_al", ("hub", 400), (0, 1, 1, 0.5, 500), 0.25),
    ("frame_cvx_al", ("frame",), (0, 1, 1, 0.5, 500), 0.2),          # BASELINE configs[1]: --CVX --AL -t 0.2
    ("frame_eq200", ("frame",), (0, 0, 2, 0.5, 200), 0.5),           # configs[2]: --EQ 200 (threshold raised: under equalisation few edges are below 0.2)
    ("frame_rgb_ml", ("frame",), (1, 0, 0, 0.5, 500), 0.2),          # configs[3]: --RGB --ML 0.5
    ("vga_cvx_al", ("vga",), (0, 1, 1, 0.5, 500), 0.2),              # configs[1] at its own size: the 640x480 frame of the headline, 2,267 merges
    ("c1_launch_file", ("bundled",), (0, 1, 1, 0.5, 500), 0.2),      # configs[0]: the reference's bundled cloud, launch file flags --CVX --AL -t 0.2
    ("c1_defaults", ("bundled",), (0, 0, 1, 0.5, 500), 0.2),         # ... and the CLI defaults
]


SWEEPS = [  # name, graph, flags, (start, end, step), truth: "colour" = the hub graph's six colour classes, "coarse" = the reference's own segments at 0.35 folded to 7 classes
    ("sweep_hub150_rgb_cvx_ml", ("hub", 150), (1, 1, 0, 0.5, 500), (0.05, 0.6, 0.05), "colour"),
    ("sweep_hub400_lab_cvx_al", ("hub", 400), (0, 1, 1, 0.5, 500), (0.8, 1.0, 0.005), "colour"),       # main()'s own range: 41 thresholds
    ("sweep_frame_cvx_al", ("frame",), (0, 1, 1, 0.5, 500), (0.1, 0.5, 0.1), "coarse"),
    ("sweep_c1_defaults", ("bundled",), (0, 0, 1, 0.5, 500), (0.8, 1.0, 0.005), "single"),       # configs[0] without -t: main()'s automatic threshold; the file has no label field
]


def truth_for(kind, graph, lib, lut, flags):
    vxyz, vrgba, labels, lists, cen, nrm, adj = graph
    t = np.zeros(len(vxyz), np.uint32)
    if kind == "single":
        return t                                                    # one ground-truth segment (all labels 0)
    if kind == "colour":
        for l in lists:
            t[l] = (int(vrgba[l[0]]) & 255) // 40 + 1
        return t
    r = ref_cluster(lib, lut, *graph, *flags, 0.35)                # labelled cloud: regions ascending, voxels in list order
    # map the labelled cloud back to voxels by exact xyz (voxel centroids are distinct)
    key = {tuple(np.asarray(vxyz[v], np.float32).view(np.uint32).tolist()): v for v in range(len(vxyz))}
    for xyz, lab in zip(r["out_xyz"], r["out_label"]):
        t[key[tuple(np.asarray(xyz, np.float32).view(np.uint32).tolist())]] = int(lab) % 7 + 1
    t[t == 0] = 777                                                 # voxels of no region (none here)
    return t


def main():
    import oracle_py
    lib = ref_lib()
    lut = np.fromfile(oracle_py.LUT_PATH, np.int16)
    out = {"case_names": np.array([c[0] for c in CASES])}
    graphs = {}
    for name, gsel, flags, thr in CASES:
        if gsel not in graphs:
            graphs[gsel] = hub_graph(gsel[1], gsel[1]) if gsel[0] == "hub" else frame_graph(vga=gsel[0] == "vga", bundled=gsel[0] == "bundled")
        vxyz, vrgba, labels, lists, cen, nrm, adj = graphs[gsel]
        gname = "_".join(map(str, gsel))
        if gname + "/vxyz" not in out:
            out.update({gname + "/vxyz": vxyz, gname + "/vrgba": vrgba, gname + "/labels": labels, gname + "/voxel_order": np.concatenate(lists).astype(np.int32),
                        gname + "/voxel_offsets": np.concatenate([[0], np.cumsum([len(l) for l in lists])]).astype(np.int64), gname + "/centroids": cen,
                        gname + "/normals": nrm, gname + "/adj": adj})
        r = ref_cluster(lib, lut, vxyz, vrgba, labels, lists, cen, nrm, adj, *flags, thr)
        out[name + "/graph"] = np.array(gname); out[name + "/flags"] = np.array(flags, np.float64); out[name + "/threshold"] = np.float32(thr)
        for k, v in r.items():
            out[name + "/" + k] = v
        print("%-20s S %5d  adjacency %6d  -> %5d merges, %4d regions left, lambda %.6f" % (name, len(labels), len(adj), len(r["merges_w"]), len(r["region_label"]), r["lam"]))
    out["sweep_names"] = np.array([c[0] for c in SWEEPS])
    for name, gsel, flags, (t0, t1, dt), kind in SWEEPS:
        if gsel not in graphs:
            graphs[gsel] = hub_graph(gsel[1], gsel[1]) if gsel[0] == "hub" else frame_graph(vga=gsel[0] == "vga", bundled=gsel[0] == "bundled")
        graph = graphs[gsel]
        truth = truth_for(kind, graph, lib, lut, flags)
        thr, perf, best = ref_all_thresh(lib, lut, *graph, *flags, truth, t0, t1, dt)
        out[name + "/graph"] = np.array("_".join(map(str, gsel))); out[name + "/flags"] = np.array(flags, np.float64)
        out[name + "/range"] = np.array([t0, t1, dt], np.float32); out[name + "/truth"] = truth
        out[name + "/thresholds"] = thr; out[name + "/perf"] = perf; out[name + "/best"] = best
        print("%-26s %3d thresholds, best %.3f (F-score %.4f)" % (name, len(thr), best[0], best[4]))
    np.savez_compressed(OUT, **out)
    print("wrote %s (%d bytes)" % (OUT, os.path.getsize(OUT)))


if __name__ == "__main__":
    main()
