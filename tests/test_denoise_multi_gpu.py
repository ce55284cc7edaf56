"""The denoiser across GPUs (skipped on boxes with fewer than 2 GPUs): a group's denoised mean, RGB8 and features equal one
GPU's bit for bit, after plain chunks and after retires, in one process and under torchrun."""
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
pytestmark = pytest.mark.gpu
CHUNKS = (2, 2, 4, 8)
REL = 0.08


def _need_two():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    return torch.cuda.device_count()


def _frames(r, p):
    """(features, then per chunk the denoised mean and RGB8 at levels 1 and 5) of a frame on r (a Context or a Group);
    retires after the third chunk."""
    out = [r.download_features(p.rows, p.cols)]
    for i, n in enumerate(CHUNKS):
        r.render_advance(n)
        if i == 2:
            r.render_retire(REL, 0.0, 2)
        for levels in (1, 5):
            d = r.denoise(levels)
            out.append((d["mean"], d["rgb8"]))
    return out


def _same(got, ref):
    f, rf = got[0], ref[0]
    if not all(np.array_equal(np.asarray(f[k]).view(np.uint32), np.asarray(rf[k]).view(np.uint32)) for k in ("surface", "depth", "normal")):
        return False
    return all(np.array_equal(m.view(np.uint32), rm.view(np.uint32)) and np.array_equal(c, rc) for (m, c), (rm, rc) in zip(got[1:], ref[1:]))


def _setup():
    import pysqt
    data = os.path.join(os.path.dirname(HERE), "data")
    hs = pysqt.HostScene.load(os.path.join(data, "scene.obj"), data)
    cam = pysqt.load_camera(os.path.join(data, "camera"))
    p = pysqt.make_params(320, 200, sum(CHUNKS), max_depth=6, seed=4)
    return hs, cam, p


def _begin_with_two(r, cam, p):
    """begin + the first two samples, so that the features can be read (k >= 2)"""
    r.render_begin(cam, p)
    r.render_advance(2)


def test_group_denoise_matches_single_gpu():
    import pysqt
    n_dev = _need_two()
    hs, cam, p = _setup()
    solo = pysqt.Context(0); solo.upload(hs)
    _begin_with_two(solo, cam, p)
    ref = _frames(solo, p)
    solo.close()
    n = 2
    while n <= n_dev:
        g = pysqt.Group(list(range(n)))
        g.upload(hs)
        _begin_with_two(g, cam, p)
        assert _same(_frames(g, p), ref), "group of %d" % n
        g.close()
        n *= 2


def test_torchrun_ranks_denoise_matches_single_gpu():
    _need_two()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29643", os.path.join(HERE, "dist_denoise_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "DENOISE_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
