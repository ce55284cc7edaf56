"""Lens frames across GPUs (skipped on boxes with fewer than 2 GPUs): a one-shot and a progressive + adaptive lens frame of a
group equal one GPU's bit for bit; ranks given different lenses all fail before anything is enqueued."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
LENS = (True, 0.06, 2.5)
CHUNKS = (2, 2, 4, 8)


def _need_two():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    return torch.cuda.device_count()


def _scene():
    import pysqt
    data = os.path.join(os.path.dirname(HERE), "data")
    return pysqt.HostScene.load(os.path.join(data, "scene.obj"), data), pysqt.load_camera(os.path.join(data, "camera"))


def _adaptive(r, p):
    ctx0 = r.ctxs[0] if hasattr(r, "ctxs") else r
    r.render_begin(CAM, p)
    out = []
    for n in CHUNKS:
        r.render_advance(n)
        act = r.render_retire(0.1, 1e-3, 2)
        rgb8, acc = ctx0.download(p.rows, p.cols)
        out.append((acc.view(np.uint32), rgb8, ctx0.download_moments(p.rows, p.cols).view(np.uint32),
                    ctx0.download_sample_counts(p.rows, p.cols), act))
    return out


CAM = None


def test_group_lens_frames_match_single_gpu():
    import pysqt
    global CAM
    n_dev = _need_two()
    hs, CAM = _scene()
    p = pysqt.make_params(320, 200, sum(CHUNKS), max_depth=6, seed=4)
    solo = pysqt.Context(0); solo.upload(hs); solo.set_lens(*LENS)
    one = solo.render(CAM, p)
    ref = _adaptive(solo, p)
    solo.close()
    for n in range(2, n_dev + 1):
        g = pysqt.Group(list(range(n)))
        g.upload(hs)
        g.set_lens(*LENS)
        got = g.render(CAM, p)
        assert np.array_equal(got["accum"].view(np.uint32), one["accum"].view(np.uint32)) and np.array_equal(got["rgb8"], one["rgb8"]), n
        for a, b in zip(_adaptive(g, p), ref):
            for x, y in zip(a, b):
                assert np.array_equal(x, y), n
        g.close()


def test_ranks_with_different_lenses_fail_together():
    import pysqt
    _need_two()
    hs, cam = _scene()
    p = pysqt.make_params(64, 48, 4, max_depth=3, seed=1)
    g = pysqt.Group([0, 1])
    g.upload(hs)
    g.ctxs[0].set_lens(*LENS)
    g.ctxs[1].set_lens(True, 0.06, 2.0)
    with pytest.raises(pysqt.SqtError):
        g.render(cam, p)
    with pytest.raises(pysqt.SqtError):
        g.render_begin(cam, p)
    g.ctxs[1].set_lens(None)
    with pytest.raises(pysqt.SqtError):
        g.render(cam, p)
    g.set_lens(*LENS)
    g.render(cam, p)                  # the communicator is still usable once the ranks agree
    g.close()
