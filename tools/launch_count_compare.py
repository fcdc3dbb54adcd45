"""Kernel launches of one C2 f3ps_merge and of one f3ps_run, for two builds of the package (needs a GPU).

  python tools/launch_count_compare.py <package dir of build A> <package dir of build B>

A package dir holds f3ps/ and a built libf3ps.so (fast-3d-pointcloud-segmentation_b200 of a checkout).  Each build runs in
its own process on the C2 frame (seed 20020, --CVX --AL -t 0.2) and prints one JSON line."""
import json
import os
import subprocess
import sys


def count(pkg):
    sys.path.insert(0, pkg)
    import f3ps
    pts = f3ps.synth.make_frame(seed=20020)
    mp = dict(color_mode=0, geom_mode=1, merge_mode=1)
    g = f3ps.Segmenter(); g.set_vccs_params(); g.set_merge_params(**mp); g.set_input(pts); g.extract(); g.graph()
    n0 = g.launch_count(); g.merge(0.2); n1 = g.launch_count()
    r = f3ps.Segmenter(); r.set_vccs_params(); r.set_merge_params(**mp); r.set_input(pts); r.run(0.2)
    return {"package": pkg, "merge_launches": n1 - n0, "run_launches": r.launch_count(), "merges": g.counts().n_merges}


if __name__ == "__main__":
    if len(sys.argv) == 3 and sys.argv[1] == "--one":
        print(json.dumps(count(os.path.abspath(sys.argv[2]))))
    else:
        for pkg in sys.argv[1:3]:
            subprocess.check_call([sys.executable, os.path.abspath(__file__), "--one", pkg])
