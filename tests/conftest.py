import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "fast-3d-pointcloud-segmentation_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

REF_DIR = os.environ.get("F3PS_REFERENCE_DIR", "")      # a checkout of the original project's sources (oracle/Makefile, `ref`)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "reference(path): runs the original project's own code; skips unless F3PS_REFERENCE_DIR "
                                       "names a checkout of it that holds `path`")


def pytest_collection_modifyitems(config, items):
    for item in items:
        m = item.get_closest_marker("reference")
        if m and not (REF_DIR and os.path.isfile(os.path.join(REF_DIR, m.args[0]))):
            item.add_marker(pytest.mark.skip(reason="needs F3PS_REFERENCE_DIR, a checkout of the original project's sources"))


@pytest.fixture(scope="session")
def oracle_mod():
    import oracle_py
    oracle_py.build()
    return oracle_py


@pytest.fixture(scope="session")
def vga_frame():
    from f3ps import synth
    return synth.make_frame(seed=20020)


@pytest.fixture(scope="session")
def small_frame():
    """160x120 frame: same generator, ~19 k points, oracle finishes in milliseconds."""
    from f3ps import synth
    return synth.make_frame(seed=11, width=160, height=120)
