"""GPU parity tests proper: the CUDA path, called through the C ABI, against the CPU oracle on the
same seeded inputs and against the committed golden fixture.  Integer / index / key results must be
identical; float results are compared bit for bit as well (the kernels replay the scalar IEEE
sequence), which is stricter than BASELINE.json's 1e-5 relative bound on edge weights."""
import hashlib
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden", "small_frame.npz")
AL = dict(color_mode=0, geom_mode=1, merge_mode=1)
EQ = dict(color_mode=0, geom_mode=0, merge_mode=2, bins=200)
RGB_ML = dict(color_mode=1, geom_mode=0, merge_mode=0, lam=0.5)

STAGE_ARRAYS = ["keys", "voxel_xyz", "voxel_rgb", "voxel_rgba", "voxel_count", "point_voxel", "nbr_count", "nbr", "normals",
                "curvature", "seeds", "labels", "dist", "sv_label", "sv_xyz", "sv_rgb", "sv_normal", "sv_count", "adj",
                "edges_ab", "edges_dc", "edges_dg", "edges_w"]
MERGE_ARRAYS = ["merges_ab", "merges_w", "merges_left", "final_ab", "final_w", "out_label", "out_voxel", "out_xyz"]


def digest(a):
    """sha256 of an array with every NaN replaced by one canonical NaN (payload/sign of a NaN is not part of parity)."""
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), np.float32(np.nan), a).astype(np.float32)
        a = a.view(np.uint32).copy()
        a[a == 0x80000000] = 0          # -0.0 == +0.0
    return hashlib.sha256(a.tobytes()).digest()


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def same(a, b):
    a = np.asarray(a); b = np.asarray(b)
    if a.shape != b.shape:
        return False
    if a.dtype.kind == "f":
        return bool(np.all((a == b) | (np.isnan(a) & np.isnan(b))))
    return bool(np.array_equal(a, b))


@pytest.fixture(scope="module")
def gpu():
    import f3ps
    f3ps.build()
    return f3ps


def run_both(gpu, oracle_mod, pts, mp, thr, merge_impl=1, **vccs):
    g = gpu.Segmenter()
    g.set_vccs_params(**vccs)
    gm = dict(mp)
    g.set_merge_params(**gm)
    g.set_input(pts)
    g.run(thr)
    o = oracle_mod.Oracle()
    o.set_vccs_params(**vccs)
    o.set_merge_params(merge_impl=merge_impl, **mp)
    o.set_input(pts)
    o.run(0, thr)
    return g, o


# CIEDE2000 is evaluated in FP64 through libm (glibc on the host, CUDA's on the device): the two differ in the last
# double bit now and then, and about one edge in 10^4 sees that survive the final cast to float.  For these arrays the
# bar is BASELINE.json's (1e-5 relative) tightened to 1e-6 and at most 0.2 % of the entries not bit-identical.
LIBM_ARRAYS = {"edges_dc", "edges_w", "merges_w", "final_w"}


def close_enough(a, b):
    a = np.asarray(a); b = np.asarray(b)
    if a.shape != b.shape:
        return False
    ne = ~((a == b) | (np.isnan(a) & np.isnan(b)))
    if not ne.any():
        return True
    rel = np.abs(a[ne] - b[ne]) / np.maximum(np.abs(b[ne]), 1e-30)
    return bool(ne.mean() <= 2e-3 and rel.max() <= 1e-6)


def upper(adj):
    """Clustering::clear_adjacency (src/clustering.cpp:476-486): what set_initialstate keeps of the adjacency multimap."""
    adj = np.asarray(adj).reshape(-1, 2)
    return adj[adj[:, 0] <= adj[:, 1]]


def assert_parity(g, o, names):
    """'adj' is compared after clear_adjacency (a surviving phantom leaf adds a ONE-WAY pair to PCL's multimap, the C ABI
    returns the symmetric closure of what Clustering keeps).  When the reference's weights are NaN (degenerate regions) its
    multimap order is undefined behaviour, so the order of the surviving edges is not compared."""
    names = list(names)
    if "adj" in names:
        names.remove("adj")
        assert np.array_equal(upper(g.array("adj")), upper(o.array("adj"))), "adj"
    if o.scalars()["nan_weights"] > 0:
        names = [n for n in names if n not in ("final_ab", "final_w")]
    bad = [n for n in names if not (close_enough if n in LIBM_ARRAYS else same)(g.array(n), o.array(n))]
    assert not bad, "GPU differs from the oracle in: %s" % bad


def test_golden_fixture(gpu):
    """No oracle involved: the committed vectors the oracle produced (tools/gen_golden.py)."""
    gold = np.load(GOLD)
    pts = gpu.synth.pack_points(gold["xyz"], gold["rgba"])
    g = gpu.Segmenter(); g.set_vccs_params(); g.set_merge_params(**AL); g.set_input(pts); g.run(0.2)
    for n in ("keys", "voxel_count", "nbr_count", "seeds", "labels", "sv_label", "sv_count"):
        assert np.array_equal(g.array(n), gold[n]), n
    for n in ("voxel_xyz", "voxel_rgb", "normals", "nbr", "dist"):
        d = np.frombuffer(digest(g.array(n)), np.uint8)
        assert np.array_equal(d, gold[n + "_sha256"]), n
    assert np.array_equal(g.array("edges_ab"), gold["al_edges_ab"])
    assert np.array_equal(bits(g.array("edges_w")), gold["al_edges_w_bits"])
    assert np.array_equal(g.array("merges_ab"), gold["al_merges_ab"])
    assert np.array_equal(bits(g.array("merges_w")), gold["al_merges_w_bits"])
    assert np.array_equal(g.array("out_label"), gold["al_out_label"])
    assert np.array_equal(g.array("out_voxel"), gold["al_out_voxel"])
    assert np.array_equal(bits(np.array([g.counts().lambda_], np.float32)), gold["al_lambda_bits"])
    # --EQ 200: heavy exact ties, the multimap insertion order decides
    g.set_merge_params(**EQ); g.merge(float(gold["eq_threshold"][0]))
    assert np.array_equal(bits(g.array("edges_w")), gold["eq_edges_w_bits"])
    assert np.array_equal(g.array("merges_ab"), gold["eq_merges_ab"])
    assert np.array_equal(bits(g.array("merges_w")), gold["eq_merges_w_bits"])
    assert np.array_equal(g.array("out_label"), gold["eq_out_label"])


@pytest.mark.parametrize("mp,thr", [(AL, 0.2), (EQ, 0.6), (RGB_ML, 0.2)])
def test_small_frame_all_stages_literal_oracle(gpu, oracle_mod, small_frame, mp, thr):
    g, o = run_both(gpu, oracle_mod, small_frame, mp, thr, merge_impl=0)
    assert_parity(g, o, STAGE_ARRAYS + MERGE_ARRAYS)
    if mp["merge_mode"] == 2:
        assert same(g.array("cdf_c"), o.array("cdf_c")) and same(g.array("cdf_g"), o.array("cdf_g"))
    assert len(o.array("merges_w")) > 50
    assert g.counts().nan_weights == int(o.scalars()["nan_weights"]) == 0


def test_vga_frame_config2_exact_merge_sequence(gpu, oracle_mod, vga_frame):
    """BASELINE.json configs[1]: 640x480 frame, --CVX --AL -t 0.2, exact merge-sequence parity."""
    g, o = run_both(gpu, oracle_mod, vga_frame, AL, 0.2, merge_impl=1)
    assert_parity(g, o, STAGE_ARRAYS + MERGE_ARRAYS)
    c = g.counts()
    assert c.n_points == 307200 and c.n_merges == len(o.array("merges_w")) > 500
    agree = np.mean(g.array("labels") == o.array("labels"))
    assert agree >= 0.995                       # BASELINE bar; measured 1.0
    rel = np.abs(g.array("edges_w") - o.array("edges_w")) / np.abs(o.array("edges_w"))
    assert np.nanmax(rel) <= 1e-5               # BASELINE bar; measured 0


@pytest.mark.parametrize("seed", [30000, 30001, 30002])
def test_sweep_frames_config3_eq200(gpu, oracle_mod, seed):
    """configs[2] frames (seeds 30000+i), --EQ 200; threshold raised to 0.5 so merges happen under ties."""
    pts = gpu.synth.make_frame(seed=seed, width=320, height=240)
    g, o = run_both(gpu, oracle_mod, pts, EQ, 0.5, merge_impl=1)
    assert_parity(g, o, STAGE_ARRAYS + MERGE_ARRAYS)
    assert len(o.array("merges_w")) > 20


@pytest.mark.parametrize("seed,w,h", [(52, 160, 120), (127, 160, 120), (16, 160, 120), (30005, 320, 240), (22030, 640, 480), (22049, 640, 480)])
def test_phantom_seed_leaves(gpu, oracle_mod, seed, w, h):
    """Two seed cells electing one voxel: the earlier helper keeps a 'phantom' leaf (kernels_expand.cuh).  Seeds 52, 127 and 16
    keep one to the end (it is listed twice in the labelled cloud, and adds a one-way adjacency pair, so the raw multimap is
    compared after clear_adjacency).  Seed 16 is the degenerate form: two helpers on one isolated voxel -> identical centroids
    -> NaN delta_g -> NaN lambda -> every weight NaN in the reference; nothing merges and the map order is undefined.
    Seeds 22030 and 22049 (two of the 512 frames bench.py generates over 8 ranks) have THREE seed cells on one voxel: two
    phantom holders and the owner (kPhSlots in kernels_expand.cuh)."""
    pts = gpu.synth.make_frame(seed=seed, width=w, height=h)
    g, o = run_both(gpu, oracle_mod, pts, AL, 0.2, merge_impl=1)
    if seed in (22030, 22049):
        assert np.unique(o.array("seeds"), return_counts=True)[1].max() == 3
    if seed == 16:
        assert np.all(np.isnan(g.array("edges_w"))) and len(g.array("merges_w")) == 0
    assert_parity(g, o, STAGE_ARRAYS + MERGE_ARRAYS)
    if seed in (52, 127, 16):
        assert int(g.array("sv_count").sum()) > int((g.array("labels") > 0).sum())
        assert len(g.array("out_voxel")) == int(g.array("sv_count").sum())


@pytest.mark.parametrize("seed,w,h", [(11, 160, 120), (52, 160, 120), (20020, 640, 480)], ids=["small", "phantom", "vga"])
def test_expand_cluster_kernel_equals_cooperative_grid(gpu, oracle_mod, seed, w, h):
    """K5 has two launch shapes (f3ps_set_expand_kernel): the cooperative grid over the GPU (software grid barrier) and ONE
    thread-block cluster per frame (hardware cluster barrier; what sweeps use).  Every cluster size, and the cooperative grid
    capped by f3ps_set_expand_sharing, gives the cooperative grid's arrays bit for bit, and those are the oracle's."""
    pts = gpu.synth.make_frame(seed=seed, width=w, height=h)
    g, o = run_both(gpu, oracle_mod, pts, AL, 0.2, merge_impl=1)
    assert_parity(g, o, STAGE_ARRAYS)
    names = ["labels", "dist", "sv_label", "sv_count", "sv_xyz", "sv_rgb", "sv_normal", "adj", "edges_ab", "edges_w"]
    ref = {n: g.array(n).copy() for n in names}
    for ctas in (1, 3, 8, 16, 0):
        g.set_expand_kernel(2, ctas)
        g.set_input(pts); g.run(0.2)
        for n in names:
            assert same(ref[n], g.array(n)), (ctas, n)
    g.set_expand_kernel(1, 0); g.set_input(pts); g.run(0.2)
    for n in names:
        assert same(ref[n], g.array(n)), ("cooperative", n)
    g.set_expand_sharing(24, 0); g.set_input(pts); g.run(0.2)      # the cooperative grid capped at 24 CTAs (BatchPool, expand_ctas=-24)
    for n in names:
        assert same(ref[n], g.array(n)), ("cooperative, 24 CTAs", n)
    with pytest.raises(ValueError):                      # F3PS_ERR_INVALID_ARGUMENT
        g.set_expand_kernel(2, 17)
    with pytest.raises(ValueError):                      # max_concurrent != 0: K5 only runs as a cooperative grid or one cluster
        g.set_expand_sharing(24, 4)
    g.set_expand_sharing(0, 0)


@pytest.mark.parametrize("seed,w,h,itr", [(11, 160, 120, 3), (52, 160, 120, 2), (20020, 640, 480, 3)], ids=["small", "phantom", "vga"])
def test_refine_supervoxels_matches_oracle(gpu, oracle_mod, seed, w, h, itr):
    """pcl::SupervoxelClustering::refineSupervoxels (src/supervoxel_clustering.cpp:369-371): refineNormals, reseedSupervoxels and
    the expansion rounds from the helpers' current centroids, num_itr times.  f3ps_refine against the oracle's literal sequential
    restatement: refined voxel normals, labels, distances, supervoxels, and everything rebuilt on top (graph, weights, merges)."""
    pts = gpu.synth.make_frame(seed=seed, width=w, height=h)
    o = oracle_mod.Oracle(); o.set_vccs_params(); o.set_merge_params(merge_impl=1, **AL); o.set_input(pts)
    for st in (1, 2, 3, 4, 5):
        o.run(st)
    s_before = len(o.array("sv_label")); labels_before = o.array("labels").copy()
    o.refine(itr); o.run(6); o.run(7, 0.2)
    g = gpu.Segmenter(); g.set_vccs_params(); g.set_merge_params(**AL); g.set_input(pts)
    with pytest.raises(gpu.LogicError):
        g.refine(itr)                                       # "Supervoxels must be extracted before they can be refined"
    g.extract(); g.refine(itr); g.graph(); g.merge(0.2)
    assert_parity(g, o, ["normals", "curvature", "labels", "dist", "sv_label", "sv_xyz", "sv_rgb", "sv_normal", "sv_count", "adj",
                         "edges_ab", "edges_dc", "edges_dg", "edges_w", "seeds"] + MERGE_ARRAYS)
    assert len(g.array("sv_label")) <= s_before and np.mean(g.array("labels") != labels_before) > 0.01    # it did something
    g.refine(0)                                             # zero iterations: makeSupervoxels only, nothing moves
    assert same(g.array("labels"), o.array("labels"))


def test_no_transform_and_other_resolutions(gpu, oracle_mod, small_frame):
    g, o = run_both(gpu, oracle_mod, small_frame, RGB_ML, 0.2, use_transform=False, voxel_res=0.02, seed_res=0.15)
    assert_parity(g, o, STAGE_ARRAYS + MERGE_ARRAYS)
    g, o = run_both(gpu, oracle_mod, small_frame, AL, 0.3, voxel_res=0.01, seed_res=0.1, color=0.5, spatial=0.2, normal=0.7)
    assert_parity(g, o, STAGE_ARRAYS + MERGE_ARRAYS)


def test_negative_z_fold_and_packed_stride(gpu, oracle_mod, small_frame):
    p2 = small_frame.copy(); p2["z"] = -p2["z"]
    g, o = run_both(gpu, oracle_mod, p2, AL, 0.2)
    assert_parity(g, o, ["keys", "labels", "merges_ab"])
    packed = np.zeros(len(small_frame), np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("rgba", "<u4")]))
    for k in ("x", "y", "z", "rgba"):
        packed[k] = small_frame[k]
    g2 = gpu.Segmenter(); g2.set_vccs_params(); g2.set_merge_params(**AL); g2.set_input(packed); g2.run(0.2)
    g1 = gpu.Segmenter(); g1.set_vccs_params(); g1.set_merge_params(**AL); g1.set_input(small_frame); g1.run(0.2)
    for n in ("keys", "labels", "merges_ab", "merges_w"):
        assert same(g1.array(n), g2.array(n)), n


def test_edge_cases_empty_nan_single(gpu, oracle_mod):
    S = gpu.synth
    cases = [np.zeros(0, S.POINT_DTYPE),
             S.pack_points(np.full((300, 3), np.nan, np.float32), np.zeros(300, np.uint32)),
             S.pack_points(np.array([[0.1, 0.2, 1.0]], np.float32), np.array([0x00ff8040], np.uint32)),
             S.pack_points(np.array([[0.1, 0.2, 1.0], [0.1, 0.2, 1.0], [np.nan, 0, 1], [0.5, 0.5, 0.0], [0.3, 0.1, 2.0]], np.float32),
                           np.arange(5, dtype=np.uint32) * 0x00101010)]
    for pts in cases:
        g, o = run_both(gpu, oracle_mod, pts, AL, 0.2)
        assert_parity(g, o, ["keys", "voxel_xyz", "voxel_count", "point_voxel", "nbr", "seeds", "labels", "edges_ab", "merges_ab", "out_label"])


def test_ragged_sizes(gpu, oracle_mod, small_frame):
    for n in (1, 31, 257, 1023, 1025, 4097, 8191):
        g, o = run_both(gpu, oracle_mod, small_frame[:n], AL, 0.2)
        assert_parity(g, o, ["keys", "voxel_xyz", "point_voxel", "nbr", "normals", "seeds", "labels", "edges_w", "merges_ab", "out_voxel"])


def test_threshold_prefix_property_and_restart(gpu, oracle_mod, small_frame):
    """cluster(t) restarts from the initial state; a lower threshold yields a prefix of the same sequence (CS4)."""
    g = gpu.Segmenter(); g.set_vccs_params(); g.set_merge_params(**AL); g.set_input(small_frame); g.run(1.0)
    full_ab, full_w = g.array("merges_ab"), g.array("merges_w")
    for thr in (0.05, 0.2, 0.6):
        g.merge(thr)
        ab, w = g.array("merges_ab"), g.array("merges_w")
        k = len(w)
        assert np.array_equal(ab, full_ab[:k]) and np.array_equal(bits(w), bits(full_w[:k]))
        assert k == len(full_w) or not (full_w[k] < np.float32(thr))
        assert np.all(w < np.float32(thr))
    g.merge(1.0)
    assert np.array_equal(g.array("merges_ab"), full_ab)


@pytest.mark.parametrize("mp", [AL, EQ, RGB_ML], ids=["cvx_al", "eq200", "rgb_ml"])
def test_resident_and_general_merge_kernels_agree(gpu, vga_frame, small_frame, mp):
    """K7 has three kernels (resident: one SM with the weight map in shared memory / the same loop with its tables in L2, for
    graphs too large for an SM / general: everything in global memory); all replay the same sequence.
    f3ps_set_merge_kernel selects (4 = resident with phase counters)."""
    for pts, thr in ((small_frame, 0.2), (vga_frame, 0.2), (small_frame, 1.0)):
        g = gpu.Segmenter(); g.set_vccs_params(); g.set_merge_params(**mp); g.set_input(pts); g.run(thr)
        assert g.counts().merge_path == 1
        fast = {n: g.array(n).copy() for n in MERGE_ARRAYS}
        for which, path in ((2, 2), (3, 3), (4, 1), (0, 1)):
            g.set_merge_kernel(which); g.merge(thr)
            assert g.counts().merge_path == path, (which, g.counts().merge_path)
            for n in MERGE_ARRAYS:
                assert same(fast[n], g.array(n)), (which, n)
            if which == 4:
                assert g.merge_profile()["sum_T"] > 0 or g.counts().n_merges < 2
        with pytest.raises(ValueError):                   # 1 is not a kernel choice
            g.set_merge_kernel(1)


def test_frames_in_flight_pool(gpu, oracle_mod, small_frame):
    """FramePool: several handles / streams / host threads on one GPU give the same result per frame as one handle alone."""
    from f3ps import sweep, synth
    frames = [small_frame] + [synth.make_frame(seed=100 + i, width=160, height=120) for i in range(5)]
    solo = []
    g = gpu.Segmenter(); g.set_vccs_params(); g.set_merge_params(**AL)
    for f in frames:
        g.set_input(f); g.run(0.2)
        solo.append((g.array("merges_ab").copy(), g.array("out_label").copy()))
    for n_handles, blocking in ((3, False), (6, True)):
        pool = sweep.FramePool(n_handles, merge=AL, threshold=0.2)
        for s_ in pool.segs:
            s_.set_blocking_wait(blocking)
        got = pool.run(frames * 2, collect=lambda s_, k: (s_.array("merges_ab").copy(), s_.array("out_label").copy()))
        pool.close()
        for k, (ab, lab) in enumerate(got):
            assert np.array_equal(ab, solo[k % len(frames)][0]) and np.array_equal(lab, solo[k % len(frames)][1])


def test_set_graph_facade_path(gpu, oracle_mod, small_frame):
    """Clustering::set_initialstate on caller-supplied supervoxels (what the C++ facade does)."""
    o = oracle_mod.Oracle(); o.set_vccs_params(); o.set_merge_params(merge_impl=0, **AL); o.set_input(small_frame); o.run(0, 0.25)
    labels = o.array("sv_label"); vl = o.array("labels")
    lists = [np.nonzero(vl == l)[0] for l in labels]
    g = gpu.Segmenter(); g.set_merge_params(**AL)
    g.set_graph(o.array("voxel_xyz"), o.array("voxel_rgba"), labels, lists, o.array("sv_xyz"), o.array("sv_normal")[:, :3], o.array("adj"))
    g.merge(0.25)
    for n in ("edges_ab", "edges_dc", "edges_dg", "edges_w", "merges_ab", "merges_w", "merges_left", "out_label"):
        assert same(g.array(n), o.array(n)), n
    assert np.array_equal(g._graph_order[g.array("out_voxel")], o.array("out_voxel"))


def _reference_clustering_cases():
    z = np.load(os.path.join(HERE, "golden", "clustering_ref.npz"))
    return [str(n) for n in z["case_names"]]


@pytest.mark.parametrize("name", _reference_clustering_cases())
def test_set_graph_equals_reference_clustering_golden(gpu, name):
    """K6 + K7 on the device against the REFERENCE's own Clustering class: /root/reference/src/clustering.cpp + color_utilities.cpp
    compiled where they lie against the stand-ins of oracle/ref_shim/ and driven like main() (set_initialstate + cluster(threshold))
    on hub graphs and on the supervoxels of the 160x120 frame in BASELINE's flag sets; inputs and the reference's per-merge lines
    committed by tools/gen_clustering_golden.py as tests/golden/clustering_ref.npz.  Merge pairs, edge / region counts and the labelled
    cloud exact; weights to 1e-6 relative with at most 0.2 % not bit-identical (FP64 libm on the host, CUDA's on the device)."""
    from test_oracle_reference_clustering import load_case
    z = np.load(os.path.join(HERE, "golden", "clustering_ref.npz"))
    graph, flags, thr, want = load_case(z, name)
    for kernel in (0, 2, 3):                                       # automatic (shared memory), general, tables in L2
        g = gpu.Segmenter(); g.set_merge_params(**flags)
        g.set_graph(*graph)
        g.set_merge_kernel(kernel); g.merge(thr)
        assert np.array_equal(g.array("merges_ab"), want["merges_ab"]), (name, kernel)
        assert close_enough(g.array("merges_w"), want["merges_w"]), (name, kernel)
        assert np.array_equal(g.array("merges_left"), want["merges_left"]), (name, kernel)
        assert np.array_equal(g.array("out_label"), want["out_label"]), (name, kernel)
        assert set(map(tuple, g.array("final_ab").tolist())) == set(map(tuple, want["final_ab"].tolist())), (name, kernel)
        if flags["merge_mode"] == 1:
            assert abs(g.counts().lambda_ - float(want["lam"])) <= 1e-6 * float(want["lam"]), (name, kernel)


def test_error_behaviour_matches_reference(gpu):
    g = gpu.Segmenter()
    with pytest.raises(gpu.LogicError):          # cluster before set_initialstate (src/clustering.cpp:671-673)
        g.merge(0.2)
    with pytest.raises(ValueError):              # set_lambda outside [0,1] (:578-579)
        g.set_merge_params(merge_mode=gpu.MANUAL_LAMBDA, lam=1.5)
    with pytest.raises(ValueError):              # set_bins_num < 0 (:593-594)
        g.set_merge_params(merge_mode=gpu.EQUALIZATION, bins=-3)
    with pytest.raises(gpu.LogicError):
        g.voxelize()


def test_device_colour_kernels_known_answers(gpu):
    from test_oracle_color import CIEDE_KAT, RGB_KAT
    import json
    g = gpu.Segmenter()
    l1 = np.array([k[:3] for k in CIEDE_KAT], np.float32); l2 = np.array([k[3:6] for k in CIEDE_KAT], np.float32)
    exp = np.array([k[6] for k in CIEDE_KAT], np.float32)
    assert np.max(np.abs(g.test_lab_ciede00(l1, l2) - exp)) < 1e-4
    c1 = np.array([k[0] for k in RGB_KAT], np.float32); c2 = np.array([k[1] for k in RGB_KAT], np.float32)
    assert np.array_equal(g.test_rgb_eucl(c1, c2), np.array([k[2] for k in RGB_KAT], np.float32))
    kat = json.load(open(os.path.join(HERE, "golden", "lab_kat.json")))
    rgb = np.array([[float.fromhex(h) for h in r] for r in kat["rgb255_f32_hex"]], np.float32)
    lab = np.array([[float.fromhex(h) for h in r] for r in kat["lab_f32_hex"]], np.float32)
    assert np.array_equal(g.test_rgb2lab(rgb), lab)


def test_device_colour_kernels_vs_oracle_random(gpu, oracle_mod):
    g = gpu.Segmenter(); o = oracle_mod.Oracle()
    rng = np.random.default_rng(9)
    rgb = (rng.random((20000, 3)) * 255).astype(np.float32)
    lab = g.test_rgb2lab(rgb)
    ref = np.stack([o.rgb2lab(c) for c in rgb[:3000]])
    assert np.array_equal(lab[:3000], ref)
    d = g.test_lab_ciede00(lab[:10000], lab[10000:])
    refd = np.array([o.lab_ciede00(a, b) for a, b in zip(lab[:3000], lab[10000:13000])], np.float32)
    assert np.mean(d[:3000] != refd) < 1e-3 and np.max(np.abs(d[:3000] - refd) / np.maximum(refd, 1e-6)) < 1e-6


@pytest.mark.parametrize("n,bits_", [(0, 8), (1, 8), (1000, 13), (4096, 24), (100003, 30), (1 << 20, 40), (3000001, 63)])
def test_radix_sort_stable(gpu, n, bits_):
    g = gpu.Segmenter()
    rng = np.random.default_rng(n + bits_)
    keys = rng.integers(0, 1 << min(bits_, 62), n, dtype=np.uint64) if n else np.zeros(0, np.uint64)
    if n > 10:
        keys[: n // 3] = keys[n // 3: 2 * (n // 3)]          # many duplicates: stability is visible
    vals = np.arange(n, dtype=np.uint32)
    k, v = g.test_sort_pairs(keys, vals, bits_)
    order = np.argsort(keys, kind="stable")
    assert np.array_equal(k, keys[order]) and np.array_equal(v, vals[order])


def test_larger_frame_against_fast_oracle(gpu, oracle_mod):
    """1.2 M-point frame (1280x960): everything still identical (oracle with the stamp-based merge)."""
    pts = gpu.synth.make_frame(seed=777, width=1280, height=960)
    g, o = run_both(gpu, oracle_mod, pts, AL, 0.2, merge_impl=1)
    assert_parity(g, o, STAGE_ARRAYS + MERGE_ARRAYS)


def test_full_size_properties_config4(gpu):
    """configs[3] shape (10 M points, -v 0.004 -s 0.04 --RGB --ML 0.5): size-independent properties."""
    pts = gpu.synth.make_dense_scene(seed=40000)
    g = gpu.Segmenter(); g.set_vccs_params(voxel_res=0.004, seed_res=0.04); g.set_merge_params(**RGB_ML)
    g.set_input(pts); g.extract()
    c = g.counts()
    finite = np.isfinite(pts["x"]) & np.isfinite(pts["y"]) & np.isfinite(pts["z"])
    assert c.n_points == len(pts) and c.n_valid == int(finite.sum())
    keys = g.array("keys").astype(np.uint64)
    assert keys.max() < (1 << c.depth)
    cnt = g.array("voxel_count"); pv = g.array("point_voxel")
    assert int(cnt.sum()) == c.n_valid and np.array_equal(pv >= 0, finite)
    assert np.array_equal(np.bincount(pv[pv >= 0], minlength=c.n_voxels), cnt)      # checksum of the point->voxel map
    # per-voxel centroid = mean of its points (float64 check of the float32 ordered sums)
    vx = g.array("voxel_xyz").astype(np.float64)
    order = np.argsort(pv[finite], kind="stable"); fi = np.nonzero(finite)[0][order]
    starts = np.concatenate([[0], np.cumsum(cnt)])
    for v in range(0, c.n_voxels, max(1, c.n_voxels // 300)):
        idx = fi[starts[v]:starts[v + 1]]
        m = np.stack([pts["x"][idx], pts["y"][idx], pts["z"][idx]], -1).astype(np.float64).mean(0)
        assert np.allclose(vx[v], m, rtol=1e-5, atol=1e-6)
    nbrc = g.array("nbr_count"); nbr = g.array("nbr")
    assert nbrc.min() >= 1 and nbrc.max() <= 27
    rows = np.arange(0, c.n_voxels, 1009)
    for v in rows[:500]:
        for u in nbr[v, :nbrc[v]]:
            assert v in nbr[u, :nbrc[u]]
            assert np.max(np.abs(keys[u].astype(np.int64) - keys[v].astype(np.int64))) <= 1
    labels = g.array("labels")
    assert labels.max() <= c.n_seeds and np.mean(labels > 0) > 0.95
    sv = g.array("sv_label"); svc = g.array("sv_count")
    assert np.array_equal(np.bincount(labels, minlength=c.n_seeds + 1)[sv], svc)
    ab = g.array("edges_ab")
    assert np.all(ab[:, 0] < ab[:, 1]) and len(np.unique(ab, axis=0)) == len(ab)
    # merge: idempotent restart, prefix property, monotone region count
    g.merge(0.2)
    m1 = g.array("merges_ab"); left = g.array("merges_left")
    assert np.all(np.diff(left[:, 1].astype(np.int64)) == -1)
    g.merge(0.2)
    assert np.array_equal(g.array("merges_ab"), m1)
    out = g.array("out_label")
    assert len(out) == int((labels > 0).sum()) and out.max() + 1 == g.counts().n_segments


def hub_graph(n_leaves, twins=False):
    """Hub + ring graph for set_graph: hub 0 touches every leaf, hub 1 every other leaf, leaf i touches leaf i + 1.
    twins: hub 1 touches every leaf too, and the hubs share colour and normal with a centroid offset perpendicular to it
    (weight 0: the hubs merge first, a merge with 2 (n_leaves + 1) adjacency entries)."""
    rng = np.random.default_rng(n_leaves)
    S = n_leaves + 2
    sizes = rng.integers(3, 7, S)
    sizes[0] = 40; sizes[1] = 25                      # two hubs
    V = int(sizes.sum())
    vxyz = (rng.normal(0, 1, (V, 3)) + 3).astype(np.float32)
    base = rng.integers(0, 6, S)                      # few colours -> many similar weights, and exact ties under EQ
    vrgba = np.repeat((base * 40 + 20).astype(np.uint32), sizes) * np.uint32(0x010101) + rng.integers(0, 3, V).astype(np.uint32)
    labels = np.arange(1, S + 1, dtype=np.uint32)
    off = np.concatenate([[0], np.cumsum(sizes)])
    lists = [np.arange(off[i], off[i + 1]) for i in range(S)]
    cen = np.stack([vxyz[l].mean(0) for l in lists]).astype(np.float32)
    nrm = rng.normal(0, 1, (S, 3)).astype(np.float32)
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    if twins:
        vrgba[:off[2]] = np.uint32(0xffffff)
        nrm[:2] = (0, 0, 1)
        cen[1] = cen[0] + np.float32([0.5, 0, 0])
    pairs = {(0, 1)}
    for i in range(2, S):
        pairs.add((0, i))                             # hub 0 touches everything
        if i % 2 or twins:
            pairs.add((1, i))                         # hub 1 touches half: duplicates (a,x)/(b,x) when the hubs merge
        if i + 1 < S:
            pairs.add((i, i + 1))
    adj = []
    for i, j in sorted(pairs):
        adj += [(labels[i], labels[j]), (labels[j], labels[i])]
    adj = np.array(sorted(adj), np.uint32)
    return vxyz, vrgba, labels, lists, cen, nrm, adj


@pytest.mark.parametrize("n_leaves,mode", [(1500, "lab_al"), (3000, "rgb_eq"), (9000, "rgb_ml"), (33000, "rgb_ml")])
def test_general_merge_kernel_hub_graph(gpu, oracle_mod, n_leaves, mode):
    """Merges that touch thousands of edges (a region with thousands of neighbours, as floors and walls of dense scenes
    have): the general kernel's sorted path (bitonic sort in shared / global memory, mark-based dedupe, ballot-scan tie
    stamps) must replay the oracle's sequence exactly.  Hub + ring graph injected through set_graph.  With twin hubs the first
    merge has more adjacency entries than the L2 variant handles (65,534): the general kernel replays from the start."""
    twins = n_leaves >= 32767                         # (the hubs' merge then has more than 65,534 adjacency entries)
    graph = hub_graph(n_leaves, twins)
    S = n_leaves + 2
    flags = {"lab_al": dict(color_mode=0, geom_mode=1, merge_mode=1), "rgb_eq": dict(color_mode=1, geom_mode=0, merge_mode=2, bins=7),
             "rgb_ml": dict(color_mode=1, geom_mode=1, merge_mode=0, lam=0.5)}[mode]
    thr = 0.08 if twins else 0.95 if mode == "rgb_eq" else 0.3   # (twins: below the hub's merges with leaves, which the oracle replays slowly)
    o = oracle_mod.Oracle(); o.set_merge_params(merge_impl=1, **flags)
    o.set_graph(*graph); o.run(7, thr)
    g = gpu.Segmenter(); g.set_merge_params(**flags)
    g.set_graph(*graph)
    g.merge(thr)
    c = g.counts()
    # 6: the shared-memory kernel up to the first merge with more adjacency entries than it has worker threads, then the L2 variant
    # from that state; 3: the graph does not fit an SM, the L2 variant loops over the entries of such merges itself; 2: a merge with
    # more than 65,534 entries stops the L2 variant too, and the general kernel replays the whole sequence
    path = 2 if twins else 6 if S <= 4096 else 3
    assert c.merge_path == path and c.max_touched > 1024 and c.n_merges > 100, (c.merge_path, c.max_touched, c.n_merges)
    first = (c.merge_path, g.array("merges_ab").copy(), g.array("final_ab").copy(), g.array("final_w").copy(), g.array("merges_w").copy())
    g.set_merge_kernel(2); g.merge(thr)                  # the general kernel alone replays the same sequence
    assert g.counts().merge_path == 2 and np.array_equal(g.array("merges_ab"), first[1]) and np.array_equal(g.array("final_ab"), first[2])
    g.set_merge_kernel(3); g.merge(thr)                  # tables in L2: merges with more than 928 adjacency entries run in lean_wide_merge
    c3 = g.counts()
    assert c3.merge_path == (2 if twins else 3) and c3.max_touched > 1024 and c3.n_merges == c.n_merges, (c3.merge_path, c3.max_touched, c3.n_merges)
    assert np.array_equal(g.array("merges_ab"), first[1]) and np.array_equal(g.array("final_ab"), first[2])
    assert same(g.array("final_w"), first[3]) and same(g.array("merges_w"), first[4])
    g.set_merge_kernel(0); g.merge(thr)
    if n_leaves >= 9000:
        assert c.max_touched > 8192                  # the global-memory sort as well
    assert np.array_equal(g.array("merges_ab"), o.array("merges_ab"))
    assert same(g.array("merges_w"), o.array("merges_w"))
    assert np.array_equal(g.array("out_label"), o.array("out_label"))
    if S <= 4096:
        # one grid for many frames (f3ps_merge_batch; a 160x120 frame beside it makes the pair a grid): this frame's CTA stops in
        # front of its first wide merge and the handle continues from that state on the L2 variant
        from f3ps import synth
        p = gpu.Segmenter(); p.set_vccs_params(); p.set_merge_params(**flags)
        p.set_input(synth.make_frame(seed=11, width=160, height=120)); p.extract(); p.graph()
        gpu.merge_batch([g, p], thr)
        assert p.counts().merge_path == 1
        assert g.counts().merge_path == 6, g.counts().merge_path
        assert np.array_equal(g.array("merges_ab"), o.array("merges_ab")) and same(g.array("merges_w"), o.array("merges_w"))
        assert np.array_equal(g.array("out_label"), o.array("out_label"))


def test_merge_batch_equals_individual_merges(gpu):
    """f3ps_merge_batch: ONE launch of the resident merge kernel, CTA i = frame i, gives every handle exactly what
    f3ps_merge gives it alone -- mixed sizes (different slot counts), handles forced onto the general kernel and onto the
    L2 variant, a handle whose largest merge overflows the resident kernel's touched list, and the pipelined BatchPool."""
    from f3ps import synth, sweep
    frames = [synth.make_frame(seed=500 + i, width=160, height=120) for i in range(9)] + [synth.make_frame(seed=20021)]
    solo = []
    for f in frames:
        g = gpu.Segmenter(); g.set_vccs_params(); g.set_merge_params(**AL)
        g.set_input(f); g.run(0.2)
        solo.append({n: g.array(n).copy() for n in ("merges_ab", "merges_w", "merges_left", "out_label", "out_voxel")})
    segs = []
    for k, f in enumerate(frames):
        g = gpu.Segmenter(); g.set_vccs_params(); g.set_merge_params(**AL)
        if k in (3, 4):
            g.set_merge_kernel(k - 1)                     # general kernel / L2 variant: these take the individual path
        g.set_input(f); g.extract(); g.graph()
        segs.append(g)
    for rep in range(2):                                   # twice: cluster() restarts from the initial state
        gpu.merge_batch(segs, 0.2)
        for k, g in enumerate(segs):
            for n, want in solo[k].items():
                assert np.array_equal(g.array(n), want), (rep, k, n)
            assert g.counts().merge_path == {3: 2, 4: 3}.get(k, 1)
    gpu.merge_batch(segs[:5], 0.1)                         # a lower threshold: a prefix
    for k, g in enumerate(segs[:5]):
        m = g.counts().n_merges
        assert m <= len(solo[k]["merges_ab"]) and np.array_equal(g.array("merges_ab"), solo[k]["merges_ab"][:m])
    pool = sweep.BatchPool(batch=4, workers=3, merge=AL, threshold=0.2)
    got = pool.run(frames * 2, collect=lambda s_, k: (s_.array("merges_ab").copy(), s_.array("out_label").copy()))
    pool.close()
    for k, (ab, lab) in enumerate(got):
        assert np.array_equal(ab, solo[k % len(frames)]["merges_ab"]) and np.array_equal(lab, solo[k % len(frames)]["out_label"]), k
