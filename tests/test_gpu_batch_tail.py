"""f3ps_merge_batch runs everything after a chunk's merge grid (labelled clouds, the scalars' read-back, the stage marks) on the
lead handle's stream, as launches over the whole chunk.  Every member must still end up exactly where f3ps_merge alone leaves it,
be usable on its own stream as soon as the call returns, and the chunk's launches must not grow with its frame count."""
import numpy as np
import pytest

from test_gpu_levels import vox_segment
from test_gpu_parity import hub_graph

pytestmark = pytest.mark.gpu

AL = dict(color_mode=0, geom_mode=1, merge_mode=1)
THR, THR2 = 0.3, 0.1


@pytest.fixture(scope="module")
def gpu():
    import f3ps
    f3ps.build()
    return f3ps


def frame_handle(gpu, pts, kernel=0):
    g = gpu.Segmenter(); g.set_vccs_params(); g.set_merge_params(**AL)
    g.set_merge_kernel(kernel)
    g.set_input(pts); g.extract(); g.graph()
    return g


def mixed_chunk(gpu):
    """C2 frames, a 160x120 frame, a frame forced onto the L2 variant (it runs on its own), and a hub graph whose CTA stops in
    front of its first wide merge and continues on the L2 variant (path 6).  Returns (handles, which of them hold points)."""
    from f3ps import synth
    segs = [frame_handle(gpu, synth.make_frame(seed=20020 + i)) for i in range(3)]
    segs.append(frame_handle(gpu, synth.make_frame(seed=11, width=160, height=120)))
    segs.append(frame_handle(gpu, synth.make_frame(seed=20023), kernel=3))
    h = gpu.Segmenter(); h.set_merge_params(**AL); h.set_graph(*hub_graph(1500))
    segs.append(h)
    return segs, [True] * 5 + [False]


def point_labels_on_device(g):
    import torch
    n = g.counts().n_points
    buf = torch.full((n,), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    g.point_labels_device(buf.data_ptr(), n)          # enqueued on the handle's stream
    g.sync()
    return buf.cpu().numpy().view(np.uint32)


def result(gpu, g, points):
    out = dict(g.fetch_result())
    c = g.counts()
    out["counts"] = np.array([c.n_merges, c.n_segments, c.n_labeled, c.merge_path])
    out["vox_segment"] = vox_segment(gpu, g)
    out["voxel_labels"] = g.voxel_labels()
    if points:
        out["point_labels_device"] = point_labels_on_device(g)
    return out


def assert_same(got, want, tag):
    assert sorted(got) == sorted(want), tag
    for k in want:
        assert got[k].dtype == want[k].dtype and np.array_equal(got[k], want[k]), (tag, k)


def test_mixed_chunk_equals_individual_merges(gpu):
    segs, points = mixed_chunk(gpu)
    want = []
    for g, p in zip(segs, points):
        g.merge(THR)
        want.append(result(gpu, g, p))
    assert want[-1]["counts"][3] == 6 and want[4]["counts"][3] == 3
    for rep in range(2):
        gpu.merge_batch(segs, THR)
        for k, (g, p) in enumerate(zip(segs, points)):
            assert_same(result(gpu, g, p), want[k], (rep, k))


def test_members_usable_on_their_own_streams_right_after(gpu):
    import torch
    segs, points = mixed_chunk(gpu)
    want, want2 = [], []
    for g, p in zip(segs, points):
        g.merge(THR2)
        want2.append(g.fetch_result())
        g.merge(THR)
        want.append((g.fetch_result(), g.point_labels() if p else None))
    bufs = [torch.full((g.counts().n_points,), -7, dtype=torch.int32, device="cuda") if p else None for g, p in zip(segs, points)]
    torch.cuda.synchronize()
    gpu.merge_batch(segs, THR)
    for k, (g, p) in enumerate(zip(segs, points)):          # no sync in between: the handle's own stream alone orders these
        if p:
            g.point_labels_device(bufs[k].data_ptr(), bufs[k].numel())
        r = g.fetch_result()
        for n, a in want[k][0].items():
            assert np.array_equal(r[n], a), (k, n)
        if p:
            g.sync()
            assert np.array_equal(bufs[k].cpu().numpy().view(np.uint32), want[k][1][0]), k
        g.merge(THR2)
        r = g.fetch_result()
        for n, a in want2[k].items():
            assert np.array_equal(r[n], a), (k, n)


@pytest.mark.parametrize("kind,path", [("c2", 1), ("hub", 6)])
def test_batch_of_one_is_merge(gpu, kind, path):
    """A batch of one handle is f3ps_merge: a lone frame that fits the shared-memory kernel runs its own build rather than a
    one-CTA grid (path 1), and a hub graph continues on the L2 variant in front of its first wide merge (path 6)."""
    from f3ps import synth

    def handle():
        if kind == "c2":
            return frame_handle(gpu, synth.make_frame(seed=20020))
        h = gpu.Segmenter(); h.set_merge_params(**AL); h.set_graph(*hub_graph(1500))
        return h
    a, b = handle(), handle()
    la, lb = a.launch_count(), b.launch_count()
    a.merge(THR)
    gpu.merge_batch([b], THR)
    assert a.counts().merge_path == b.counts().merge_path == path
    assert a.launch_count() - la == b.launch_count() - lb
    assert sorted(a.stage_ms()) == sorted(b.stage_ms())
    assert_same(result(gpu, b, kind == "c2"), result(gpu, a, kind == "c2"), kind)


def test_chunk_launches_do_not_grow_with_frames(gpu):
    from f3ps import synth
    segs = [frame_handle(gpu, synth.make_frame(seed=700 + i, width=160, height=120)) for i in range(8)]
    deltas = []
    for n in (2, 4, 8):
        before = sum(g.launch_count() for g in segs)
        gpu.merge_batch(segs[:n], 0.2)
        assert all(g.counts().merge_path == 1 for g in segs[:n])
        deltas.append(sum(g.launch_count() for g in segs) - before)
    assert deltas[0] == deltas[1] == deltas[2], deltas
