"""Segment extraction (f3ps_get_segment_points / _voxels / _info): the members of every segment of a level, grouped, and one
descriptor per segment.  The oracle is numpy on the level labels of the same handle."""
import ctypes as C
import os
import shutil
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


def segmenter(gpu, pts, mp, kernel=0, **vccs):
    g = gpu.Segmenter(); g.set_vccs_params(**vccs); g.set_merge_params(**mp)
    g.set_merge_kernel(kernel)
    g.set_input(pts); g.extract(); g.graph()
    return g


def grouping(lab, K):
    """(offsets, index) of labels lab (NONE = in no segment) over K segments"""
    valid = lab != NONE
    off = np.zeros(K + 1, np.int64)
    off[1:] = np.cumsum(np.bincount(lab[valid], minlength=K))
    return off, np.nonzero(valid)[0][np.argsort(lab[valid], kind="stable")]


def check_grouping(g, points=True):
    lv = g.levels()
    labels = g.point_labels() if points else g.voxel_labels()
    for k, K in enumerate(lv["n_segments"]):
        off, idx = g.segment_points(k) if points else g.segment_voxels(k)
        want_off, want_idx = grouping(labels[k], int(K))
        assert off.dtype == np.int64 and idx.dtype == np.int32
        assert np.array_equal(off, want_off), k
        assert np.array_equal(idx, want_idx), k


def check_info(g, pts, k, fold=True):
    info = g.segment_info(k)
    pl, vl = g.point_labels()[k], g.voxel_labels()[k]
    K = int(g.levels()["n_segments"][k])
    off, idx = grouping(pl, K)
    n = np.diff(off)
    assert np.array_equal(info["n_points"], n)
    assert np.array_equal(info["n_voxels"], np.bincount(vl[vl != NONE], minlength=K))
    assert np.all(n > 0)
    xyz = np.stack([pts["x"], pts["y"], np.abs(pts["z"]) if fold else pts["z"]], 1)[idx]
    starts = off[:-1]
    assert np.array_equal(info["min_xyz"], np.minimum.reduceat(xyz, starts, axis=0))
    assert np.array_equal(info["max_xyz"], np.maximum.reduceat(xyz, starts, axis=0))
    mean = np.add.reduceat(xyz.astype(np.float64), starts, axis=0) / n[:, None]
    ulp = np.spacing(np.abs(mean).astype(np.float32)).astype(np.float64)
    assert np.all(np.abs(info["centroid"].astype(np.float64) - mean) <= ulp)
    c = pts["rgba"][idx].astype(np.int64)
    rgb = np.stack([(c >> 16) & 255, (c >> 8) & 255, c & 255], 1)
    assert np.array_equal(info["mean_rgb"], (np.add.reduceat(rgb, starts, axis=0) / n[:, None]).astype(np.float32))
    again = g.segment_info(k)
    for name, a in info.items():
        assert a.tobytes() == again[name].tobytes(), name
    return info


@pytest.mark.parametrize("kernel", [0, 2])
@pytest.mark.parametrize("mp", [AL, EQ200, RGB_ML], ids=["AL", "EQ200", "RGB_ML"])
def test_small_frame_grouping_and_info(gpu, frame_small, mp, kernel):
    g = segmenter(gpu, frame_small, mp, kernel)
    g.merge_levels(SMALL_THRESHOLDS)
    check_grouping(g, points=True)
    check_grouping(g, points=False)
    for k in range(len(SMALL_THRESHOLDS)):
        check_info(g, frame_small, k)
    labels = g.state_regions()[0]
    assert np.array_equal(g.segment_info(-1)["region_label"], labels)


def test_vga_frame_sweep_levels(gpu, frame_vga):
    thr = [float(t) for t in gpu.Segmenter.sweep_thresholds()[::8]] + [1.5]
    g = segmenter(gpu, frame_vga, AL)
    g.merge_levels(thr)
    check_grouping(g, points=True)
    check_grouping(g, points=False)
    for k in (0, len(thr) - 1):
        check_info(g, frame_vga, k)
    assert np.array_equal(g.segment_info()["region_label"], g.state_regions()[0])


def test_negative_z_is_folded(gpu, frame_small):
    pts = frame_small.copy()
    pts["z"][::2] *= -1
    g = segmenter(gpu, pts, AL)
    g.merge_levels([0.1, 0.2])
    info = check_info(g, pts, 1, fold=True)
    ref = segmenter(gpu, frame_small, AL)
    ref.merge_levels([0.1, 0.2])
    want = ref.segment_info(1)
    for name in want:
        assert np.array_equal(info[name], want[name]), name
    assert np.all(info["min_xyz"][:, 2] > 0)


def test_bundled_cloud(gpu):
    from f3ps import pcd
    pts, _, _ = pcd.read_pcd(FIXTURE)
    assert len(pts) == 307200
    g = segmenter(gpu, pts, AL)
    g.merge_levels([0.1, 0.2, 0.5])
    check_grouping(g, points=True)
    check_grouping(g, points=False)
    finite = np.isfinite(pts["x"]) & np.isfinite(pts["y"]) & np.isfinite(pts["z"])
    off, idx = g.segment_points(-1)
    assert not np.isin(np.nonzero(~finite)[0], idx).any() and (~finite).any()
    for k in range(3):
        check_info(g, pts, k)


def _reference_cases():
    z = np.load(os.path.join(HERE, "golden", "clustering_ref.npz"))
    return [str(n) for n in z["case_names"]][:3]


@pytest.mark.parametrize("name", _reference_cases())
def test_set_graph_voxels_only(gpu, name):
    from test_oracle_reference_clustering import load_case
    z = np.load(os.path.join(HERE, "golden", "clustering_ref.npz"))
    graph, flags, thr, _ = load_case(z, name)
    g = gpu.Segmenter(); g.set_merge_params(**flags)
    g.set_graph(*graph)
    g.merge_levels([thr / 2, thr])
    check_grouping(g, points=False)
    for call in (g.segment_points, g.segment_info):
        with pytest.raises(gpu.LogicError):
            call(1)


def test_device_variants(gpu, frame_small):
    import torch
    g = segmenter(gpu, frame_small, AL)
    g.merge_levels(SMALL_THRESHOLDS)
    for k in (0, 2, -1):
        off, idx = g.segment_points(k)
        t_off = torch.full((off.size,), -7, dtype=torch.int64, device="cuda")
        t_idx = torch.full((idx.size + 3,), -7, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        g.segment_points_device(k, t_off.data_ptr(), t_idx.data_ptr(), off.size, t_idx.numel())
        g.sync()
        assert np.array_equal(t_off.cpu().numpy(), off) and np.array_equal(t_idx[:idx.size].cpu().numpy(), idx), k
        assert np.all(t_idx[idx.size:].cpu().numpy() == -7)
        voff, vidx = g.segment_voxels(k)
        d_off = torch.zeros(voff.size, dtype=torch.int64, device="cuda"); d_idx = torch.zeros(vidx.size, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        g._chk(g.L.f3ps_get_segment_voxels(g.h, k % len(SMALL_THRESHOLDS), C.c_void_p(d_off.data_ptr()), C.c_void_p(d_idx.data_ptr()),
                                           voff.size, vidx.size, 1))
        g.sync()
        assert np.array_equal(d_off.cpu().numpy(), voff) and np.array_equal(d_idx.cpu().numpy(), vidx), k
    off, idx = g.segment_points(0)
    t_off = torch.zeros(off.size, dtype=torch.int64, device="cuda"); t_idx = torch.zeros(idx.size, dtype=torch.int32, device="cuda")
    with pytest.raises(ValueError):
        g.segment_points_device(0, t_off.data_ptr(), t_idx.data_ptr(), off.size - 1, idx.size)
    with pytest.raises(ValueError):
        g.segment_points_device(0, t_off.data_ptr(), t_idx.data_ptr(), off.size, idx.size - 1)


def test_rules(gpu, frame_small):
    g = gpu.Segmenter(); g.set_vccs_params(); g.set_merge_params(**AL); g.set_input(frame_small); g.extract(); g.graph()
    buf = np.zeros(4, np.int64); info = np.zeros(4, np.uint8)
    for rc in (g.L.f3ps_get_segment_points(g.h, 0, buf.ctypes.data, None, 4, 0, 0),
               g.L.f3ps_get_segment_voxels(g.h, 0, buf.ctypes.data, None, 4, 0, 0),
               g.L.f3ps_get_segment_info(g.h, 0, info.ctypes.data, 0)):
        assert rc == 2                                              # F3PS_ERR_LOGIC before any merge
    g.merge_levels([0.05, 0.5])
    for bad in (2, -3):
        for call in (g.segment_points, g.segment_voxels, g.segment_info):
            with pytest.raises(ValueError):
                call(bad)
    assert g.L.f3ps_get_segment_points(g.h, -1, buf.ctypes.data, None, 4, 0, 0) == 1
    K = int(g.levels()["n_segments"][0])
    off, idx = g.segment_points(0)
    o = np.zeros(K + 1, np.int64); i = np.zeros(idx.size, np.int32)
    assert g.L.f3ps_get_segment_points(g.h, 0, o.ctypes.data, i.ctypes.data, K, i.size, 0) == 1
    assert g.L.f3ps_get_segment_points(g.h, 0, o.ctypes.data, i.ctypes.data, K + 1, i.size - 1, 0) == 1
    assert g.L.f3ps_get_segment_points(g.h, 0, o.ctypes.data, i.ctypes.data, K + 1, i.size, 0) == 0
    recs = np.zeros(K * 64, np.uint8)
    assert g.L.f3ps_get_segment_info(g.h, 0, recs.ctypes.data, K - 1) == 1
    assert g.L.f3ps_get_segment_info(g.h, 0, recs.ctypes.data, K) == 0
    # the kept grouping belongs to one merge: a new merge, or refine + merge, groups again
    for step in ("merge", "refine"):
        before = g.segment_points(0)
        g.segment_voxels(0)
        if step == "refine":
            g.refine(1); g.graph()
        g.merge_levels([0.5, 1.0] if step == "merge" else [0.05, 0.5])
        assert step == "refine" or len(g.segment_points(0)[0]) != len(before[0])
        check_grouping(g, points=True)
        check_grouping(g, points=False)
        check_info(g, frame_small, 0)


def test_edge_inputs(gpu):
    S = gpu.synth
    cases = [np.zeros(0, S.POINT_DTYPE),
             S.pack_points(np.full((300, 3), np.nan, np.float32), np.zeros(300, np.uint32)),
             S.pack_points(np.array([[0.1, 0.2, 1.0]], np.float32), np.array([0x00ff8040], np.uint32)),
             S.pack_points(np.array([[0.1, 0.2, 1.0], [0.1, 0.2, 1.0], [np.nan, 0, 1], [0.5, 0.5, 0.0], [0.3, 0.1, 2.0]], np.float32),
                           np.arange(5, dtype=np.uint32) * 0x00101010)]
    for pts in cases:
        g = gpu.Segmenter(); g.set_vccs_params(); g.set_merge_params(**AL); g.set_input(pts); g.run(0.2)
        g.merge_levels([0.1, 0.2])
        check_grouping(g, points=True)
        check_grouping(g, points=False)
        for k in range(2):
            info = g.segment_info(k)
            K = int(g.levels()["n_segments"][k])
            assert all(len(a) == K for a in info.values())
            if K:
                check_info(g, pts, k)


def test_room_scan_10m(gpu):
    from f3ps import synth
    pts = synth.make_room_scan(seed=50000, n_points=10_000_000)
    g = segmenter(gpu, pts, AL, voxel_res=0.01, seed_res=0.1)
    g.merge_levels([0.2])
    pl = g.point_labels()[0]
    K = int(g.levels()["n_segments"][0])
    off, idx = g.segment_points(0)
    want_off, want_idx = grouping(pl, K)
    assert np.array_equal(off, want_off) and np.array_equal(idx, want_idx)
    check_info(g, pts, 0)


def _csv(path):
    rows = [l.split(",") for l in open(path).read().splitlines()]
    assert rows[0] == ["level", "threshold", "segment", "region_label", "n_points", "n_voxels", "min_x", "min_y", "min_z", "max_x", "max_y",
                       "max_z", "cx", "cy", "cz", "r", "g", "b"]
    return rows[1:]


def _want_rows(g, thresholds):
    rows = []
    for k, t in enumerate(thresholds):
        info = g.segment_info(k)
        for j in range(len(info["n_points"])):
            rows.append([k, np.float32(t), j, int(info["region_label"][j]), int(info["n_points"][j]), int(info["n_voxels"][j])] +
                        [np.float32(v) for name in ("min_xyz", "max_xyz", "centroid", "mean_rgb") for v in info[name][j]])
    return rows


def _parse(rows):
    return [[int(r[0]), np.float32(r[1]), int(r[2]), int(r[3]), int(r[4]), int(r[5])] + [np.float32(v) for v in r[6:]] for r in rows]


def test_cli_segments(gpu, tmp_path):
    from f3ps import pcd
    subprocess.check_call(["make", "-C", HOST, "-s"])
    cli = os.path.join(HOST, "supervoxel_clustering")
    base = [cli, "-p", FIXTURE, "--CVX", "--AL", "-t", "0.2", "--no-eval"]
    plain_dir, seg_dir = tmp_path / "plain", tmp_path / "seg"
    plain_dir.mkdir(); seg_dir.mkdir()
    plain = subprocess.run(base + ["-o", str(plain_dir / "out.pcd")], cwd=plain_dir, capture_output=True, text=True, timeout=600)
    assert plain.returncode == 0, plain.stdout + plain.stderr
    one = subprocess.run(base + ["-o", str(seg_dir / "out.pcd"), "--segments", str(seg_dir / "seg.csv")], cwd=seg_dir, capture_output=True,
                         text=True, timeout=600)
    assert one.returncode == 0, one.stdout + one.stderr
    assert (plain_dir / "out.pcd").read_bytes() == (seg_dir / "out.pcd").read_bytes()
    strip = lambda out: [l for l in out.splitlines() if not l.startswith(("Clustering complete", "  stage ms"))]
    assert strip(one.stdout) == strip(plain.stdout)
    many = subprocess.run(base + ["--levels", "0.1,0.2", "--segments", str(seg_dir / "levels.csv")], cwd=seg_dir, capture_output=True,
                          text=True, timeout=600)
    assert many.returncode == 0, many.stdout + many.stderr
    pts, _, _ = pcd.read_pcd(FIXTURE)
    g = gpu.Segmenter(); g.set_vccs_params(); g.set_merge_params(**AL); g.set_input(pts); g.extract(); g.graph()
    g.merge_levels([0.2])
    assert _parse(_csv(seg_dir / "seg.csv")) == _want_rows(g, [0.2])
    g.merge_levels([0.1, 0.2])
    assert _parse(_csv(seg_dir / "levels.csv")) == _want_rows(g, [0.1, 0.2])
    for extra in (["--facade"], ["--slabs", "1"]):
        bad = subprocess.run(base + ["--segments", "x.csv"] + extra, cwd=seg_dir, capture_output=True, text=True, timeout=600)
        assert bad.returncode == 1 and "--segments" in bad.stderr, extra
    d = tmp_path / "clouds"
    d.mkdir()
    for name in ("a.pcd", "b.pcd"):
        shutil.copy(FIXTURE, d / name)
    sweep = subprocess.run([cli, "-d", str(d), "--CVX", "--AL", "-t", "0.2", "--no-eval", "--segments", str(tmp_path / "seg.csv")],
                           cwd=tmp_path, capture_output=True, text=True, timeout=600)
    assert sweep.returncode == 0, sweep.stdout + sweep.stderr
    for stem in ("a", "b"):
        assert (tmp_path / (stem + "_seg.csv")).read_bytes() == (seg_dir / "seg.csv").read_bytes(), stem
