#!/usr/bin/env python
"""Golden vectors of the REFERENCE's own Testing class (SURVEY.md section 8f row 1): random labelled cloud pairs through
oracle/_ref/libref_clustering.so -- /root/reference/src/testing.cpp compiled where it lies against the container stand-ins of
oracle/ref_shim/ (oracle/Makefile, target `ref`) -- with inputs and the seven scores committed as tests/golden/testing_ref.json.
Runs in the build container only (the GPU box has no /root/reference); the tests read the fixture.
Coordinates are small integers (exact in float32), unique inside a cloud; labels are arbitrary uint32 values."""
import ctypes as C
import json
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "oracle", "_ref", "libref_clustering.so")
OUT = os.path.join(ROOT, "tests", "golden", "testing_ref.json")


def ref_lib():
    if not os.path.isdir(os.environ.get("F3PS_REFERENCE_DIR", "")):
        raise SystemExit("set F3PS_REFERENCE_DIR to a checkout of the original project: oracle/_ref/libref_clustering.so is built from its sources")
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "-s", "ref"])
    lib = C.CDLL(LIB)
    lib.ref_testing_eval.restype = C.c_int
    lib.ref_testing_eval.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    return lib


def ref_scores(lib, sxyz, slab, txyz, tlab):
    sx = np.ascontiguousarray(sxyz, np.float32); sl = np.ascontiguousarray(slab, np.uint32)
    tx = np.ascontiguousarray(txyz, np.float32); tl = np.ascontiguousarray(tlab, np.uint32)
    out = np.zeros(7, np.float32)
    rc = lib.ref_testing_eval(sx.ctypes.data, sl.ctypes.data, len(sl), tx.ctypes.data, tl.ctypes.data, len(tl), out.ctypes.data)
    return rc, out


def make_case(rng, n_universe, n_seg_labels, n_truth_labels, keep_seg, keep_truth, blocky):
    """points of a universe of distinct grid coordinates; both clouds keep a random part of it; labels either random per point or
    in contiguous blocks (blocky: segments that mostly agree between the two clouds, like a real segmentation and its ground truth)"""
    side = int(np.ceil(n_universe ** (1 / 3))) + 1
    idx = rng.choice(side ** 3, n_universe, replace=False)
    xyz = np.stack([idx % side, (idx // side) % side, idx // (side * side)], 1).astype(np.int32) - side // 2      # negative coordinates too
    seg_names = rng.choice(1 << 20, n_seg_labels, replace=False).astype(np.uint32)
    truth_names = rng.choice(1 << 20, n_truth_labels, replace=False).astype(np.uint32)
    if blocky:
        order = np.lexsort((xyz[:, 2], xyz[:, 1], xyz[:, 0]))
        s_of = np.empty(n_universe, np.int64); t_of = np.empty(n_universe, np.int64)
        s_of[order] = np.minimum((np.arange(n_universe) * n_seg_labels) // n_universe, n_seg_labels - 1)
        cuts = np.sort(rng.choice(np.arange(1, n_universe), n_truth_labels - 1, replace=False)) if n_truth_labels > 1 else np.array([], np.int64)
        t_of[order] = np.searchsorted(cuts, np.arange(n_universe), side="right")
    else:
        s_of = rng.integers(0, n_seg_labels, n_universe); t_of = rng.integers(0, n_truth_labels, n_universe)
    ks = rng.random(n_universe) < keep_seg; kt = rng.random(n_universe) < keep_truth
    if not ks.any(): ks[0] = True
    if not kt.any(): kt[-1] = True
    ps, pt = rng.permutation(np.nonzero(ks)[0]), rng.permutation(np.nonzero(kt)[0])               # cloud order is irrelevant to the reference: shuffle
    return xyz[ps], seg_names[s_of[ps]], xyz[pt], truth_names[t_of[pt]]


def cases():
    rng = np.random.default_rng(20151307)
    out = []
    for n, ns, nt, kseg, ktr, blocky in [
            (1, 1, 1, 1.0, 1.0, False), (5, 2, 2, 1.0, 1.0, False), (40, 3, 3, 0.9, 0.9, True), (40, 1, 5, 1.0, 1.0, True), (40, 6, 1, 1.0, 1.0, True),
            (200, 4, 9, 0.8, 0.95, True), (200, 9, 4, 0.95, 0.8, True), (300, 12, 12, 1.0, 1.0, True), (300, 12, 12, 0.7, 0.7, False),
            (600, 5, 7, 0.9, 0.9, True), (600, 20, 3, 0.85, 1.0, True), (600, 3, 20, 1.0, 0.85, True), (800, 10, 10, 0.5, 0.5, True),
            (800, 2, 2, 0.99, 0.99, False), (500, 25, 25, 0.9, 0.9, True), (64, 4, 4, 1.0, 1.0, True), (64, 8, 8, 1.0, 1.0, False)]:
        for rep in range(2):
            out.append(make_case(rng, n, ns, nt, kseg, ktr, blocky))
    # truth segments of EQUAL size (std::map<size, index>::insert keeps the first: the others never get a best match)
    xyz = np.stack([np.arange(60), np.zeros(60, int), np.zeros(60, int)], 1).astype(np.int32)
    out.append((xyz, np.repeat([7, 3, 9], 20).astype(np.uint32), xyz, np.repeat([5, 1, 8, 2], 15).astype(np.uint32)))
    # disjoint clouds: no intersection at all (precision = recall = 0 -> F-score 0 by the guard)
    out.append((xyz[:30], np.repeat([1, 2], 15).astype(np.uint32), xyz[30:], np.repeat([4, 5, 6], 10).astype(np.uint32)))
    # identical clouds and labels: perfect scores
    out.append((xyz, np.repeat([1, 2, 3], 20).astype(np.uint32), xyz, np.repeat([10, 20, 30], 20).astype(np.uint32)))
    # more truth segments than segmentation segments: rows run out (match -1)
    out.append((xyz, np.repeat([1, 2], 30).astype(np.uint32), xyz, (np.arange(60) // 6).astype(np.uint32)))
    return out


def main():
    lib = ref_lib()
    recs = []
    for sxyz, slab, txyz, tlab in cases():
        rc, sc = ref_scores(lib, sxyz, slab, txyz, tlab)
        assert rc == 0
        recs.append({"seg_xyz": np.asarray(sxyz).tolist(), "seg_label": np.asarray(slab).tolist(), "truth_xyz": np.asarray(txyz).tolist(),
                     "truth_label": np.asarray(tlab).tolist(), "scores_f32_hex": [float(v).hex() for v in sc], "scores": [float(v) for v in sc]})
    with open(OUT, "w") as f:
        json.dump({"source": "/root/reference/src/testing.cpp compiled against oracle/ref_shim (tools/gen_testing_golden.py)",
                   "order": ["voi", "precision", "recall", "fscore", "wov", "fpr", "fnr"], "cases": recs}, f, separators=(",", ":"))
    print("wrote %s: %d cases, %d bytes" % (OUT, len(recs), os.path.getsize(OUT)))


if __name__ == "__main__":
    main()
