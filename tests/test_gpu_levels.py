"""Segmentation levels (f3ps_merge_levels and the level getters): the segmentation at several thresholds from one merge replay,
per voxel and per input point.  Every level must be exactly what a fresh f3ps_merge at its threshold gives."""
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
HOST = os.path.join(ROOT, "fast-3d-pointcloud-segmentation_b200", "host")
FIXTURE = os.path.join(HERE, "fixtures", "milk_cartoon_all_small_clorox.pcd")
AL = dict(color_mode=0, geom_mode=1, merge_mode=1)
EQ200 = dict(color_mode=0, geom_mode=0, merge_mode=2, bins=200)
RGB_ML = dict(color_mode=1, geom_mode=0, merge_mode=0, lam=0.5)
SMALL_THRESHOLDS = [0.05, 0.1, 0.2, 0.5, 1.0]
NONE = np.uint32(0xffffffff)


@pytest.fixture(scope="module")
def gpu():
    import f3ps
    f3ps.build()
    return f3ps


@pytest.fixture(scope="module")
def frame_small():
    from f3ps import synth
    return synth.make_frame(seed=11, width=160, height=120)


@pytest.fixture(scope="module")
def frame_vga():
    from f3ps import synth
    return synth.make_frame(seed=20020)


@pytest.fixture(scope="module")
def room_scan_10m():
    from f3ps import synth
    return synth.make_room_scan(seed=50000, n_points=10_000_000)


def segmenter(gpu, pts, mp, kernel=0, **vccs):
    g = gpu.Segmenter(); g.set_vccs_params(**vccs); g.set_merge_params(**mp)
    g.set_merge_kernel(kernel)
    g.set_input(pts); g.extract(); g.graph()
    return g


class _DeviceWords:
    """A device array of uint32 words, seen by torch through __cuda_array_interface__ (read as int32)."""
    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": "<i4", "data": (int(ptr), False), "version": 3}


def vox_segment(gpu, g):
    """f3ps_get_voxel_segments_device, copied with torch: the words it reports (the labelled cloud's position count, which
    can be less than V; voxel v's segment is word v)."""
    import ctypes as C
    import torch
    ptr, n = C.c_void_p(), C.c_int64()
    g._chk(g.L.f3ps_get_voxel_segments_device(g.h, C.byref(ptr), C.byref(n)))
    g.sync()
    t = torch.as_tensor(_DeviceWords(ptr.value, n.value), device="cuda").clone()
    return t.cpu().numpy().view(np.uint32)


def same_as_vox_segment(labels, gpu, g):
    seg = vox_segment(gpu, g)
    n = min(len(seg), len(labels))
    return n > 0 and np.array_equal(labels[:n], seg[:n])


def check_levels_against_merges(gpu, g, thresholds):
    g.merge_levels(thresholds)
    lv = g.levels(); vl = g.voxel_labels()
    assert vl.shape == (len(thresholds), g.counts().n_voxels)
    assert np.array_equal(lv["thresholds"], np.float32(thresholds))
    assert same_as_vox_segment(vl[-1], gpu, g)
    for k, t in enumerate(thresholds):
        g.merge(t)
        c = g.counts()
        assert lv["n_merges"][k] == c.n_merges and lv["n_segments"][k] == c.n_segments, (k, t)
        assert same_as_vox_segment(vl[k], gpu, g), (k, t)
        assert np.array_equal(vl[k], g.voxel_labels()[0]), (k, t)
    return vl


def check_nesting(vl):
    for k in range(len(vl) - 1):
        fine, coarse = vl[k], vl[k + 1]
        assert np.array_equal(fine == NONE, coarse == NONE)
        pairs = np.unique(np.stack([fine[fine != NONE], coarse[fine != NONE]], 1), axis=0)
        assert len(np.unique(pairs[:, 0])) == len(pairs), k          # finer -> coarser is a function


@pytest.mark.parametrize("kernel", [0, 2, 3])
@pytest.mark.parametrize("mp", [AL, EQ200, RGB_ML], ids=["AL", "EQ200", "RGB_ML"])
def test_small_frame_levels_equal_their_own_merges(gpu, frame_small, mp, kernel):
    g = segmenter(gpu, frame_small, mp, kernel)
    vl = check_levels_against_merges(gpu, g, SMALL_THRESHOLDS)
    check_nesting(vl)
    labelled = vl[vl != NONE]
    assert labelled.size > 0


@pytest.mark.parametrize("kernel", [0, 2, 3])
def test_vga_frame_sweep_levels_equal_their_own_merges(gpu, frame_vga, kernel):
    thr = sorted(list(map(float, gpu.Segmenter.sweep_thresholds())) + [0.05, 0.2])
    g = segmenter(gpu, frame_vga, AL, kernel)
    check_nesting(check_levels_against_merges(gpu, g, thr))


def test_small_frame_levels_equal_oracle_labelled_cloud(gpu, oracle_mod, frame_small):
    g = segmenter(gpu, frame_small, AL)
    g.merge_levels(SMALL_THRESHOLDS)
    vl = g.voxel_labels()
    for k, t in enumerate(SMALL_THRESHOLDS):
        o = oracle_mod.Oracle(); o.set_vccs_params(); o.set_merge_params(merge_impl=1, **AL); o.set_input(frame_small); o.run(0, t)
        lab, vox, owner = o.array("out_label"), o.array("out_voxel"), o.array("labels")
        want = np.full(len(owner), NONE, np.uint32)
        cnt = np.bincount(vox, minlength=len(owner))
        once = cnt[vox] == 1
        want[vox[once]] = lab[once]
        assert np.array_equal(vl[k][cnt == 1], want[cnt == 1]), t
        assert np.all(vl[k][owner == 0] == NONE) and np.all(vl[k][owner != 0] != NONE), t
        for v in np.nonzero(cnt > 1)[0]:                             # a phantom leaf is listed by its holder too: the owner's entry
            assert vl[k][v] in lab[vox == v], (t, v)


def _reference_cases():
    z = np.load(os.path.join(HERE, "golden", "clustering_ref.npz"))
    return [str(n) for n in z["case_names"]]


@pytest.mark.parametrize("name", _reference_cases())
def test_set_graph_levels_equal_reference_golden(gpu, name):
    from test_oracle_reference_clustering import load_case
    z = np.load(os.path.join(HERE, "golden", "clustering_ref.npz"))
    graph, flags, thr, want = load_case(z, name)
    g = gpu.Segmenter(); g.set_merge_params(**flags)
    g.set_graph(*graph)
    g.merge_levels([thr / 2, thr])
    vl = g.voxel_labels()
    # f3ps_set_graph groups the voxels by ascending supervoxel label: out_voxel counts positions of that grouping, the level
    # labels the voxels in the order they were passed in
    labels, lists = graph[2], graph[3]
    off = np.concatenate([[0], np.cumsum([len(l) for l in lists])])
    passed_in = np.concatenate([np.arange(off[s], off[s + 1]) for s in np.argsort(labels, kind="stable")] or [np.zeros(0, int)])
    assert np.array_equal(vl[1][passed_in[g.array("out_voxel")]], want["out_label"]), name
    assert np.array_equal(g.array("out_label"), want["out_label"]), name
    check_nesting(vl)
    with pytest.raises(gpu.LogicError):
        g.point_labels()


def test_point_labels_follow_point_voxel(gpu, frame_small):
    import torch
    g = segmenter(gpu, frame_small, AL)
    g.merge_levels(SMALL_THRESHOLDS)
    pl, vl, pv = g.point_labels(), g.voxel_labels(), g.array("point_voxel")
    assert pl.shape == (len(SMALL_THRESHOLDS), len(frame_small)) and pl.dtype == np.uint32
    want = np.where(pv[None, :] >= 0, vl[:, np.maximum(pv, 0)], NONE)
    assert np.array_equal(pl, want)
    t = torch.full(pl.shape, 7, dtype=torch.int32, device="cuda")
    odd = torch.zeros(pl.size + 1, dtype=torch.int32, device="cuda")   # rows not 16-byte aligned: the scalar store path
    torch.cuda.synchronize()                                         # the fills ran on torch's stream, the handle has its own
    g.point_labels_device(t.data_ptr(), t.numel())
    g.sync()
    assert np.array_equal(t.cpu().numpy().view(np.uint32), pl)
    g.point_labels_device(odd[1:].data_ptr(), pl.size)
    g.sync()
    assert np.array_equal(odd[1:].cpu().numpy().view(np.uint32).reshape(pl.shape), pl) and int(odd[0]) == 0
    with pytest.raises(ValueError):
        g.point_labels_device(t.data_ptr(), t.numel() - 1)
    import ctypes as C
    short = np.zeros(pl.size - 1, np.uint32)
    with pytest.raises(ValueError):
        g._chk(g.L.f3ps_get_level_point_labels(g.h, short.ctypes.data_as(C.c_void_p), short.size, 0))
    with pytest.raises(ValueError):
        g._chk(g.L.f3ps_get_level_voxel_labels(g.h, short.ctypes.data_as(C.c_void_p), vl.size - 1, 0))


def test_point_labels_edge_inputs(gpu):
    S = gpu.synth
    cases = [np.zeros(0, S.POINT_DTYPE),
             S.pack_points(np.full((300, 3), np.nan, np.float32), np.zeros(300, np.uint32)),
             S.pack_points(np.array([[0.1, 0.2, 1.0]], np.float32), np.array([0x00ff8040], np.uint32)),
             S.pack_points(np.array([[0.1, 0.2, 1.0], [0.1, 0.2, 1.0], [np.nan, 0, 1], [0.5, 0.5, 0.0], [0.3, 0.1, 2.0]], np.float32),
                           np.arange(5, dtype=np.uint32) * 0x00101010)]
    for pts in cases:
        g = gpu.Segmenter(); g.set_vccs_params(); g.set_merge_params(**AL); g.set_input(pts); g.run(0.2)
        g.merge_levels([0.1, 0.2])
        pl = g.point_labels()
        assert pl.shape == (2, len(pts))
        pv, vl = g.array("point_voxel"), g.voxel_labels()
        want = np.full(pl.shape, NONE, np.uint32)
        want[:, pv >= 0] = vl[:, pv[pv >= 0]]
        assert np.array_equal(pl, want)
        finite = np.isfinite(pts["x"]) & np.isfinite(pts["y"]) & np.isfinite(pts["z"]) if len(pts) else np.zeros(0, bool)
        if not finite.any():
            assert np.all(pl == NONE)


def test_state_rules(gpu, frame_small):
    g = gpu.Segmenter(); g.set_vccs_params(); g.set_merge_params(**AL); g.set_input(frame_small)
    with pytest.raises(gpu.LogicError):
        g.levels()
    g.extract(); g.graph()
    for call in (g.levels, g.voxel_labels, g.point_labels):
        with pytest.raises(gpu.LogicError):
            call()
    for bad in ([0.2, 0.1], [0.1, float("nan")], [], [0.1] * 257, [0.1, float("inf")]):
        with pytest.raises(ValueError):
            g.merge_levels(bad)
    g.merge(1.0)
    ref = {n: g.array(n).copy() for n in ("merges_ab", "merges_w", "out_label", "out_voxel")}
    ref_c = g.counts()
    g.merge_levels(SMALL_THRESHOLDS)
    c = g.counts()
    assert (c.n_merges, c.n_segments, c.n_labeled, c.n_edges_left) == (ref_c.n_merges, ref_c.n_segments, ref_c.n_labeled, ref_c.n_edges_left)
    for n, want in ref.items():
        assert np.array_equal(g.array(n), want), n
    assert len(g.levels()["thresholds"]) == len(SMALL_THRESHOLDS)
    g.merge(0.2)                                                     # a plain merge leaves exactly one level, its threshold
    lv = g.levels()
    assert list(lv["thresholds"]) == [np.float32(0.2)] and lv["n_merges"][0] == g.counts().n_merges
    assert g.voxel_labels().shape == (1, g.counts().n_voxels) and g.point_labels().shape == (1, len(frame_small))
    thr = gpu.Segmenter.sweep_thresholds()
    g.all_thresh(np.zeros(g.counts().n_voxels, np.uint32))          # eval_thresholds leaves its last threshold
    lv = g.levels()
    assert list(lv["thresholds"]) == [thr[-1]] and lv["n_merges"][0] == g.counts().n_merges
    assert same_as_vox_segment(g.voxel_labels()[0], gpu, g)
    g.set_input(frame_small)
    with pytest.raises(gpu.LogicError):
        g.levels()


def test_merge_batch_handles_report_one_level(gpu):
    from f3ps import synth
    frames = [synth.make_frame(seed=600 + i, width=160, height=120) for i in range(4)]
    solo = []
    for f in frames:
        g = gpu.Segmenter(); g.set_vccs_params(); g.set_merge_params(**AL); g.set_input(f); g.run(0.2)
        solo.append((g.voxel_labels(), g.point_labels()))
    segs = []
    for k, f in enumerate(frames):
        g = gpu.Segmenter(); g.set_vccs_params(); g.set_merge_params(**AL)
        if k == 3:
            g.set_merge_kernel(3)                                    # the L2 variant: this handle runs on its own
        g.set_input(f); g.extract(); g.graph()
        g.merge_levels([0.05, 0.1])
        segs.append(g)
    gpu.merge_batch(segs, 0.2)
    for k, g in enumerate(segs):
        lv = g.levels()
        assert list(lv["thresholds"]) == [np.float32(0.2)] and lv["n_merges"][0] == g.counts().n_merges
        assert np.array_equal(g.voxel_labels(), solo[k][0]) and np.array_equal(g.point_labels(), solo[k][1]), k


def test_room_scan_10m_levels(gpu, room_scan_10m):
    g = gpu.Segmenter(); g.set_vccs_params(voxel_res=0.01, seed_res=0.1); g.set_merge_params(**AL)
    g.set_input(room_scan_10m); g.extract(); g.graph()
    t = 0.2
    g.merge_levels([t / 4, t / 2, t])
    c = g.counts()
    assert c.merge_path in (3, 6), c.merge_path
    vl = g.voxel_labels()
    assert same_as_vox_segment(vl[-1], gpu, g)
    lv = g.levels()
    assert lv["n_merges"][-1] == c.n_merges and lv["n_segments"][-1] == c.n_segments
    check_nesting(vl)
    pl, pv = g.point_labels(), g.array("point_voxel")
    assert pl.shape == (3, len(room_scan_10m))
    for k in range(3):
        assert np.array_equal(pl[k], np.where(pv >= 0, vl[k][np.maximum(pv, 0)], NONE)), k


def test_cli_levels_and_point_labels(gpu, tmp_path):
    from f3ps import pcd
    subprocess.check_call(["make", "-C", HOST, "-s"])
    cli = os.path.join(HOST, "supervoxel_clustering")
    base = [cli, "-p", FIXTURE, "--CVX", "--AL", "-t", "0.2"]
    plain_dir, lv_dir = tmp_path / "plain", tmp_path / "levels"
    plain_dir.mkdir(); lv_dir.mkdir()
    plain = subprocess.run(base + ["-o", str(plain_dir / "seg.pcd")], cwd=plain_dir, capture_output=True, text=True, timeout=600)
    assert plain.returncode == 0, plain.stdout + plain.stderr
    run = subprocess.run(base + ["-o", str(lv_dir / "seg.pcd"), "--levels", "0.1,0.2", "--point-labels", str(lv_dir / "out.pcd")],
                         cwd=lv_dir, capture_output=True, text=True, timeout=600)
    assert run.returncode == 0, run.stdout + run.stderr
    lines = [l for l in run.stdout.splitlines() if l.startswith("level ")]
    assert len(lines) == 2 and lines[0].startswith("level 0: threshold 0.100000 -> ") and lines[1].startswith("level 1: threshold 0.200000 -> ")
    strip = lambda out: [l for l in out.splitlines() if not l.startswith(("level ", "Clustering complete", "  stage ms"))]
    assert strip(run.stdout) == strip(plain.stdout)
    for name in sorted(os.listdir(plain_dir)):                       # -o and the score files
        assert (plain_dir / name).read_bytes() == (lv_dir / name).read_bytes(), name
    pts, _, _ = pcd.read_pcd(FIXTURE)
    g = gpu.Segmenter(); g.set_vccs_params(); g.set_merge_params(color_mode=0, geom_mode=1, merge_mode=1)
    g.set_input(pts); g.extract(); g.graph()
    g.merge_levels([0.1, 0.2])
    want = g.point_labels()
    for k in range(2):
        got, lab, _ = pcd.read_pcd(str(lv_dir / ("out_%d.pcd" % k)))
        assert len(got) == 307200 and lab is not None
        assert np.array_equal(np.asarray(lab, np.uint64).astype(np.uint32), want[k]), k
    for extra in (["--facade"], ["--slabs", "1"]):
        bad = subprocess.run(base + ["--levels", "0.1"] + extra, cwd=lv_dir, capture_output=True, text=True, timeout=600)
        assert bad.returncode == 1 and "--levels" in bad.stderr, extra


def test_cli_levels_in_directory_sweep(tmp_path):
    """With -d and -t the CLI batches the merges of a group of files; --levels sends every file through the per-file path, so
    each file's report carries its level lines, the same as a -p run of that file."""
    import shutil
    subprocess.check_call(["make", "-C", HOST, "-s"])
    cli = os.path.join(HOST, "supervoxel_clustering")
    d = tmp_path / "clouds"
    d.mkdir()
    for name in ("a.pcd", "b.pcd"):
        shutil.copy(FIXTURE, d / name)
    levels = ["--levels", "0.1,0.2"]
    single = subprocess.run([cli, "-p", FIXTURE, "--CVX", "--AL", "-t", "0.2", "--no-eval"] + levels, cwd=tmp_path, capture_output=True,
                            text=True, timeout=600)
    assert single.returncode == 0, single.stdout + single.stderr
    want = [l for l in single.stdout.splitlines() if l.startswith("level ")]
    assert len(want) == 2
    sweep = subprocess.run([cli, "-d", str(d), "--CVX", "--AL", "-t", "0.2", "--no-eval"] + levels, cwd=tmp_path, capture_output=True,
                           text=True, timeout=600)
    assert sweep.returncode == 0, sweep.stdout + sweep.stderr
    assert [l for l in sweep.stdout.splitlines() if l.startswith("level ")] == want * 2
    plain = subprocess.run([cli, "-d", str(d), "--CVX", "--AL", "-t", "0.2", "--no-eval"], cwd=tmp_path, capture_output=True, text=True,
                           timeout=600)
    assert plain.returncode == 0, plain.stdout + plain.stderr
    strip = lambda out: [l for l in out.splitlines() if not l.startswith(("level ", "Clustering complete", "  stage ms"))]
    assert strip(sweep.stdout) == strip(plain.stdout)
