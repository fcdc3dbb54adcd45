"""Slab mode driven from C++ over NCCL (host/slab_host.cpp: one thread, stream, handle and ncclComm_t per GPU) against ONE
handle processing the whole cloud -- SURVEY.md section 8e row 2 with the host side in C++ as BASELINE's north_star asks.
host/slab_selftest cuts a synthetic room scan (with drop-outs and negative z) into uneven shares, runs the protocol of
f3ps/slab.py through NCCL, and compares every rank's voxel labels / distances, merge log and labelled cloud with the single
handle bit for bit.  On a one-GPU box the world is 1 (every collective degenerates, the routing / slicing code still runs);
with two or more visible GPUs the exchanges are real."""
import json
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "fast-3d-pointcloud-segmentation_b200", "host")

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def selftest():
    import f3ps
    f3ps.build()
    subprocess.check_call(["make", "-C", HOST, "-s"])
    exe = os.path.join(HOST, "slab_selftest")
    assert os.path.exists(exe)
    return exe


@pytest.mark.parametrize("device_shares", [1, 0], ids=["device_shares", "host_shares"])
def test_cpp_nccl_slab_mode_equals_one_handle(selftest, device_shares):
    import torch
    gpus = min(2, torch.cuda.device_count())
    out = subprocess.run([selftest, "--gpus", str(gpus), "--points", "400000", "--device-shares", str(device_shares)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    rec = json.loads(out.stdout.strip().splitlines()[-1])
    assert rec["identical_to_one_handle"] is True and rec["gpus"] == gpus
    assert rec["V"] > 10000 and rec["merges"] > 10 and rec["device_shares"] == bool(device_shares)


def test_cli_slabs_prints_the_same_merge_sequence(selftest, small_frame, tmp_path):
    """supervoxel_clustering -p cloud.pcd -t 0.2 --CVX --AL --V [--slabs N]: the reference's per-merge debug lines
    (src/clustering.cpp:390-392) and the labelled cloud written by -o are the same with and without slab mode."""
    import torch
    from f3ps import pcd
    gpus = min(2, torch.cuda.device_count())
    cli = os.path.join(HOST, "supervoxel_clustering")
    p = str(tmp_path / "cloud.pcd")
    pcd.write_pcd_binary(p, small_frame)
    outs = []
    for extra, name in (([], "one.pcd"), (["--slabs", str(gpus)], "slabs.pcd")):
        o = str(tmp_path / name)
        run = subprocess.run([cli, "-p", p, "-t", "0.2", "--CVX", "--AL", "--V", "--no-eval", "-o", o] + extra, capture_output=True, text=True, timeout=300)
        assert run.returncode == 0, run.stdout + run.stderr
        lines = [l for l in run.stdout.splitlines() if l.startswith("left:") or l.startswith("Found ")]
        assert len(lines) > 50
        outs.append((lines, open(o).read()))
    assert outs[0][0] == outs[1][0]
    assert outs[0][1] == outs[1][1]
    bad = subprocess.run([cli, "-p", p, "--slabs", "1"], capture_output=True, text=True)      # no -t: refused
    assert bad.returncode == 1 and "--slabs needs" in bad.stderr
