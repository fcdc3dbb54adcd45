"""The oracle's K6 / K7 half against the REFERENCE's own Clustering class (SURVEY.md section 8c).

/root/reference/src/clustering.cpp, clustering_state.cpp and color_utilities.cpp compile where they lie against the stand-ins of
oracle/ref_shim/ (containers, the few Eigen operations, PCL's centroid / plane fit as the oracle restates PCL, cv::cvtColor as the
cv2-pinned LUT; oracle/ref_shim/README.md) into oracle/_ref/libref_clustering.so.  tools/gen_clustering_golden.py drove it the way
main() does (set_initialstate + cluster(threshold)) on hub graphs and on the supervoxels of the 160x120 synthetic frame in the flag
sets BASELINE.json names, and committed inputs and outputs as tests/golden/clustering_ref.npz.  Here the oracle -- the literal
std::multimap replay AND the stamp-rule variant the GPU kernels implement -- must reproduce the reference's per-merge debug lines
(a, b, weight bits, edges / regions left), its adaptive lambda, the edges that remain and the labelled cloud, bit for bit.
The GPU path is compared with the same fixture in tests/test_gpu_parity.py::test_set_graph_equals_reference_clustering_golden."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "clustering_ref.npz")


def load_case(z, name):
    g = str(z[name + "/graph"])
    off = z[g + "/voxel_offsets"]; order = z[g + "/voxel_order"]
    lists = [order[off[i]:off[i + 1]] for i in range(len(off) - 1)]
    graph = (z[g + "/vxyz"], z[g + "/vrgba"], z[g + "/labels"], lists, z[g + "/centroids"], z[g + "/normals"], z[g + "/adj"])
    color, geom, merging, lam, bins = z[name + "/flags"]
    flags = dict(color_mode=int(color), geom_mode=int(geom), merge_mode=int(merging), lam=float(lam), bins=int(bins))
    want = {k: z[name + "/" + k] for k in ("merges_ab", "merges_w", "merges_left", "final_ab", "out_label", "out_xyz", "lam", "region_label", "region_size")}
    return graph, flags, float(z[name + "/threshold"]), want


def case_names():
    return [str(n) for n in np.load(GOLD)["case_names"]]


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.mark.parametrize("name", case_names())
@pytest.mark.parametrize("impl", [0, 1], ids=["literal_multimap", "stamp_rule"])
def test_oracle_reproduces_reference_clustering(oracle_mod, name, impl):
    z = np.load(GOLD)
    graph, flags, thr, want = load_case(z, name)
    o = oracle_mod.Oracle(); o.set_merge_params(merge_impl=impl, **flags)
    o.set_graph(*graph); o.run(7, thr)
    assert np.array_equal(o.array("merges_ab"), want["merges_ab"])                 # the reference's "[a, b]" per merge
    assert np.array_equal(bits(o.array("merges_w")), bits(want["merges_w"]))       # "w: %f" -- the float the multimap was keyed with
    assert np.array_equal(o.array("merges_left"), want["merges_left"])             # "left: %de/%dp"
    if flags["merge_mode"] == 1:
        lam = np.float32(dict(zip(oracle_mod.SCALARS, o.array("scalars")))["lambda"])
        assert bits(lam)[()] == bits(want["lam"])[()]                              # adaptive lambda (clustering.cpp:258-287)
    got_edges = set(map(tuple, o.array("final_ab").tolist())); ref_edges = set(map(tuple, want["final_ab"].tolist()))
    assert got_edges == ref_edges                                                   # get_currentstate(): the edges that remain
    assert np.array_equal(o.array("out_label"), want["out_label"])                 # get_labeled_cloud(): dense labels in region order
    assert np.array_equal(bits(o.array("out_xyz")), bits(want["out_xyz"]))


@pytest.mark.reference("src/clustering.cpp")
def test_oracle_reproduces_reference_clustering_live(oracle_mod):
    """fresh hub graphs (other seeds, sizes and flag sets than the committed ones) through the compiled reference class"""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import gen_clustering_golden as gen
    lib = gen.ref_lib()
    lut = np.fromfile(oracle_mod.LUT_PATH, np.int16)
    for seed, n_leaves, flags, thr in [(901, 40, (0, 0, 1, 0.5, 500), 0.4), (902, 90, (1, 1, 2, 0.5, 50), 0.7), (903, 120, (0, 1, 0, 0.3, 500), 0.35),
                                       (904, 25, (1, 0, 0, 0.9, 500), 1.0), (905, 200, (0, 1, 1, 0.5, 500), 0.3)]:
        graph = gen.hub_graph(n_leaves, seed)
        want = gen.ref_cluster(lib, lut, *graph, *flags, thr)
        for impl in (0, 1):
            o = oracle_mod.Oracle()
            o.set_merge_params(merge_impl=impl, color_mode=flags[0], geom_mode=flags[1], merge_mode=flags[2], lam=flags[3], bins=flags[4])
            o.set_graph(*graph); o.run(7, thr)
            assert np.array_equal(o.array("merges_ab"), want["merges_ab"]), (seed, impl)
            assert np.array_equal(bits(o.array("merges_w")), bits(want["merges_w"])), (seed, impl)
            assert np.array_equal(o.array("merges_left"), want["merges_left"]) and np.array_equal(o.array("out_label"), want["out_label"]), (seed, impl)


def sweep_names():
    return [str(n) for n in np.load(GOLD)["sweep_names"]]


def load_sweep(z, name):
    g = str(z[name + "/graph"])
    off = z[g + "/voxel_offsets"]; order = z[g + "/voxel_order"]
    lists = [order[off[i]:off[i + 1]] for i in range(len(off) - 1)]
    graph = (z[g + "/vxyz"], z[g + "/vrgba"], z[g + "/labels"], lists, z[g + "/centroids"], z[g + "/normals"], z[g + "/adj"])
    color, geom, merging, lam, bins = z[name + "/flags"]
    flags = dict(color_mode=int(color), geom_mode=int(geom), merge_mode=int(merging), lam=float(lam), bins=int(bins))
    return graph, flags, tuple(float(x) for x in z[name + "/range"]), z[name + "/truth"], z[name + "/thresholds"], z[name + "/perf"], z[name + "/best"]


ORDER = ("voi", "precision", "recall", "fscore", "wov", "fpr", "fnr")


@pytest.mark.parametrize("name", sweep_names())
def test_oracle_reproduces_reference_all_thresh(oracle_mod, name):
    """Clustering::all_thresh / best_thresh of the compiled reference (the automatic threshold of main(),
    /root/reference/src/supervoxel_clustering.cpp:428-438): the thresholds its float loop visits, the seven scores at each, and the
    chosen threshold.  The reference continues clustering from the previous threshold's state; the oracle restarts per threshold --
    the same result (SURVEY.md CS4), now checked against the reference's own code."""
    import oracle_testing as ot
    z = np.load(GOLD)
    graph, flags, (t0, t1, dt), truth, thr, perf, best = load_sweep(z, name)
    F = np.float32
    mine = [F(t0)]
    t = F(F(t0) + F(dt))
    while t <= F(t1):
        mine.append(t); t = F(t + F(dt))
    assert np.array_equal(np.array(mine, np.float32), thr)                          # the float loop of :711-718
    res = {}
    for k, t in enumerate(thr):
        o = oracle_mod.Oracle(); o.set_merge_params(merge_impl=1, **flags); o.set_graph(*graph); o.run(7, float(t))
        owned = np.concatenate(graph[3])                                             # the ground-truth cloud holds the voxels of the supervoxels
        got = ot.scores(o.array("out_xyz"), o.array("out_label"), graph[0][owned], truth[owned])
        res[float(t)] = got
        for j, n in enumerate(ORDER):
            tol = 1e-6 if n == "voi" else 2e-7
            assert abs(got[n] - perf[k, j]) <= tol * max(1.0, abs(perf[k, j])), (name, float(t), n, got[n], perf[k, j])
    bt, bp = ot.best_thresh(res)
    assert np.float32(bt) == best[0] and abs(bp["fscore"] - best[4]) <= 2e-7


@pytest.mark.reference("src/color_utilities.cpp")
def test_oracle_colour_distances_equal_reference_live(oracle_mod):
    """ColorUtilities::lab_ciede00 / rgb_eucl of the compiled reference on 200,000 random pairs (hue wrap-arounds, greys, identical
    colours, the corners of the gamut) against the oracle's restatement: bit for bit (same libm, same float / double mix)."""
    import ctypes as C
    import subprocess
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "-s"])
    lib = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_clustering.so"))
    rng = np.random.default_rng(2000)
    n = 200000
    lab1 = np.stack([rng.random(n) * 100, rng.random(n) * 256 - 128, rng.random(n) * 256 - 128], 1).astype(np.float32)
    lab2 = np.stack([rng.random(n) * 100, rng.random(n) * 256 - 128, rng.random(n) * 256 - 128], 1).astype(np.float32)
    lab2[:1000] = lab1[:1000]                                   # identical
    lab1[1000:3000, 1:] = 0; lab2[2000:4000, 1:] = 0            # greys (C = 0: the hue branches)
    lab2[4000:6000, 1:] = -lab1[4000:6000, 1:]                  # opposite hues (the 180-degree branches)
    lab1[6000:6100] = [[0, -128, -128]]; lab2[6000:6100] = [[100, 127.99, 127.99]]
    rgb1 = (rng.random((n, 3)) * 255).astype(np.float32); rgb2 = (rng.random((n, 3)) * 255).astype(np.float32)
    ref_de = np.zeros(n, np.float32); ref_eu = np.zeros(n, np.float32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    lib.ref_color_distances(C.c_int64(n), p(lab1), p(lab2), p(ref_de), None)
    lib.ref_color_distances(C.c_int64(n), p(rgb1), p(rgb2), None, p(ref_eu))
    o = oracle_mod.Oracle()
    step = 40                                                    # the oracle's entry points take one pair per call
    got_de = np.array([o.lab_ciede00(a, b) for a, b in zip(lab1[::step], lab2[::step])], np.float32)
    got_eu = np.array([o.rgb_eucl(a, b) for a, b in zip(rgb1[::step], rgb2[::step])], np.float32)
    assert np.array_equal(bits(got_de), bits(ref_de[::step])) and np.array_equal(bits(got_eu), bits(ref_eu[::step]))
    head = np.array([o.lab_ciede00(a, b) for a, b in zip(lab1[:6100:7], lab2[:6100:7])], np.float32)      # the constructed cases, densely
    assert np.array_equal(bits(head), bits(ref_de[:6100:7]))


@pytest.mark.reference("src/clustering.cpp")
def test_reference_exception_behaviour_live():
    """The exception types of the compiled reference, case by case: what host/facade.cpp throws and what the C ABI's status codes map to
    (F3PS_ERR_LOGIC / F3PS_ERR_INVALID_ARGUMENT / std::out_of_range; tests/test_gpu_parity.py::test_error_behaviour_matches_reference,
    tests/test_gpu_eval.py::test_eval_errors and host/facade_selftest check the product side)."""
    import ctypes as C
    import subprocess
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "-s"])
    lib = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_clustering.so"))
    NONE, LOGIC, INVALID, RANGE = 0, 1, 2, 3
    want = {0: INVALID,     # set_lambda outside [0, 1]
            1: LOGIC,       # set_lambda when the criterion is not MANUAL_LAMBDA
            2: INVALID,     # set_bins_num < 0
            3: LOGIC,       # set_bins_num when the criterion is not EQUALIZATION
            4: LOGIC,       # cluster before set_initialstate
            5: RANGE,       # all_thresh with a threshold outside [0, 1]
            6: INVALID,     # Testing with an empty segmentation
            7: INVALID,     # Testing with an empty ground truth
            8: NONE}        # lambda = 0 and lambda = 1 are accepted
    for case, code in want.items():
        assert lib.ref_exception_case(case) == code, case
