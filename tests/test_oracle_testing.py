"""The evaluation restatement (oracle/oracle_testing.py) against (i) hand-computed cases of the reference's formulas
(src/testing.cpp:239-362) and (ii) the REFERENCE's own Testing class: /root/reference/src/testing.cpp compiles where it lies against
the container stand-ins of oracle/ref_shim/ (oracle/Makefile `ref` -> oracle/_ref/libref_clustering.so); tools/gen_testing_golden.py ran
it on 38 random / adversarial labelled cloud pairs and committed inputs and scores as tests/golden/testing_ref.json."""
import ctypes as C
import json
import math
import os
import subprocess

import numpy as np
import pytest

import oracle_testing as ot

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORDER = ("voi", "precision", "recall", "fscore", "wov", "fpr", "fnr")


def _check(got, want):
    """the scores are float32 sums in the reference's order: bit-identical except where libm's logf and numpy's log differ by an ulp"""
    g = np.array([got[n] for n in ORDER], np.float32)
    for n, a, b in zip(ORDER, g, want):
        if n in ("voi",):
            assert abs(a - b) <= 1e-6 * max(1.0, abs(b)), (n, a, b)
        else:
            assert a == b or abs(a - b) <= 2e-7 * max(1.0, abs(b)), (n, a, b)


def test_restatement_equals_reference_testing_class_golden():
    d = json.load(open(os.path.join(ROOT, "tests", "golden", "testing_ref.json")))
    assert list(d["order"]) == list(ORDER) and len(d["cases"]) >= 38
    exact = 0
    for c in d["cases"]:
        want = np.array([float.fromhex(h) for h in c["scores_f32_hex"]], np.float32)
        got = ot.scores(np.array(c["seg_xyz"], np.float32), np.array(c["seg_label"], np.uint32),
                        np.array(c["truth_xyz"], np.float32), np.array(c["truth_label"], np.uint32))
        _check(got, want)
        exact += int(np.array_equal(np.array([got[n] for n in ORDER], np.float32), want))
    assert exact >= len(d["cases"]) - 4                          # (36 of 38 bit-identical when the fixture was made)


@pytest.mark.reference("src/testing.cpp")
def test_restatement_equals_reference_testing_class_live():
    """fresh random clouds through the compiled reference class (not only the committed ones)"""
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "-s", "ref"])
    lib = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_clustering.so"))
    lib.ref_testing_eval.restype = C.c_int
    lib.ref_testing_eval.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    rng = np.random.default_rng(99)
    for trial in range(25):
        n = int(rng.integers(1, 400))
        idx = rng.choice(20 ** 3, n, replace=False)
        xyz = np.stack([idx % 20, (idx // 20) % 20, idx // 400], 1).astype(np.float32) - 7
        sl = rng.integers(0, int(rng.integers(1, 9)), n).astype(np.uint32) * 13 + 5
        tl = rng.integers(0, int(rng.integers(1, 9)), n).astype(np.uint32) * 7 + 2
        ks = rng.random(n) < 0.9; kt = rng.random(n) < 0.9
        ks[0] = True; kt[-1] = True
        sx, tx = np.ascontiguousarray(xyz[ks]), np.ascontiguousarray(xyz[kt])
        s_l, t_l = np.ascontiguousarray(sl[ks]), np.ascontiguousarray(tl[kt])
        out = np.zeros(7, np.float32)
        assert lib.ref_testing_eval(sx.ctypes.data, s_l.ctypes.data, len(s_l), tx.ctypes.data, t_l.ctypes.data, len(t_l), out.ctypes.data) == 0
        _check(ot.scores(sx, s_l, tx, t_l), out)
    # an empty cloud: the reference throws std::invalid_argument (src/testing.cpp:420-441)
    z = np.zeros((0, 3), np.float32); zl = np.zeros(0, np.uint32); one = np.zeros((1, 3), np.float32); ol = np.zeros(1, np.uint32)
    assert lib.ref_testing_eval(z.ctypes.data, zl.ctypes.data, 0, one.ctypes.data, ol.ctypes.data, 1, np.zeros(7, np.float32).ctypes.data) == 1


def _cloud(n):
    return np.stack([np.arange(n, dtype=np.float32), np.zeros(n, np.float32), np.ones(n, np.float32)], 1)


def test_perfect_segmentation_scores():
    xyz = _cloud(10)
    truth = np.array([5] * 4 + [9] * 6)
    seg = np.array([0] * 4 + [1] * 6)
    s = ot.scores(xyz, seg, xyz, truth)
    assert abs(s["precision"] - 1) < 1e-6 and abs(s["recall"] - 1) < 1e-6 and abs(s["fscore"] - 1) < 1e-6
    assert abs(s["wov"] - 1) < 1e-6 and s["fpr"] == 0 and s["fnr"] == 0 and abs(s["voi"]) < 1e-6


def test_hand_computed_case():
    # truth: A = 6 points, B = 4 points; segmentation: s0 = first 5, s1 = last 5  -> inter = [[5, 0], [1, 4]]
    xyz = _cloud(10)
    truth = np.array([0] * 6 + [1] * 4)
    seg = np.array([0] * 5 + [1] * 5)
    s = ot.scores(xyz, seg, xyz, truth)
    # matches: A (larger) -> s0 (5), B -> s1 (4)
    p = (5 * 6 / 5 + 4 * 4 / 5) / 10
    r = (5 + 4) / 10
    assert abs(s["precision"] - p) < 1e-6 and abs(s["recall"] - r) < 1e-6
    assert abs(s["fscore"] - 2 * p * r / (p + r)) < 1e-6
    assert abs(s["fpr"] - (0 + 1) / 10) < 1e-6 and abs(s["fnr"] - (1 + 0) / 10) < 1e-6
    assert abs(s["wov"] - (5 * 6 / 6 + 4 * 4 / 5) / 10) < 1e-6
    hs = -2 * 0.5 * math.log(0.5); ht = -(0.6 * math.log(0.6) + 0.4 * math.log(0.4))
    mi = 0.5 * math.log(10 * 5 / (5 * 6)) + 0.1 * math.log(10 * 1 / (5 * 6)) + 0.4 * math.log(10 * 4 / (5 * 4))
    assert abs(s["voi"] - (hs + ht - 2 * mi)) < 1e-5


def test_equal_sized_truth_segments_quirk():
    # std::map<size_t, uint32_t>::insert keeps only the FIRST truth segment of a given size (testing.cpp:97-110):
    # the second 5-point truth segment is never matched and counts as false negatives.
    xyz = _cloud(10)
    truth = np.array([0] * 5 + [1] * 5)
    seg = truth.copy()
    s = ot.scores(xyz, seg, xyz, truth)
    assert abs(s["recall"] - 0.5) < 1e-6 and abs(s["fnr"] - 0.5) < 1e-6 and abs(s["precision"] - 0.5) < 1e-6


def test_partial_segmentation_and_label_gaps():
    # the segmentation covers 8 of 10 truth points (unowned voxels are absent), labels are renumbered densely
    xyz = _cloud(10)
    truth = np.array([3] * 7 + [8] * 3)
    keep = np.array([0, 1, 2, 3, 4, 5, 7, 8])
    seg = np.array([10, 10, 10, 10, 10, 10, 40, 40])
    s = ot.scores(xyz[keep], seg, xyz, truth)
    assert abs(s["recall"] - (6 + 2) / 10) < 1e-6 and abs(s["fnr"] - (1 + 1) / 10) < 1e-6 and s["fpr"] == 0


def test_sweep_thresholds_float_steps():
    thr = [np.float32(0.8)]
    t = np.float32(np.float32(0.8) + np.float32(0.005))
    while t <= np.float32(1.0):
        thr.append(t); t = np.float32(t + np.float32(0.005))
    assert len(thr) == 41 and abs(float(thr[-1]) - 0.99999982) < 1e-6       # SURVEY.md CS4
