"""Adaptive frames across GPUs (skipped on boxes with fewer than 2 GPUs): a group adaptive frame equals one GPU's bit for bit
in sums, moments, RGB8, sample counts and active totals, in one process and under torchrun; ranks given different
tolerances fail together at retire without a hang."""
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
    """(accum, rgb8, m2, counts, noise, active) after every chunk + retire of an adaptive frame on r (a Context or a Group)."""
    ctx0 = r.ctxs[0] if hasattr(r, "ctxs") else r
    out = []
    for n in CHUNKS:
        pr = r.render_advance(n)
        act = r.render_retire(REL, 0.0, 2)
        rgb8, acc = ctx0.download(p.rows, p.cols)
        out.append((acc, rgb8, ctx0.download_moments(p.rows, p.cols), ctx0.download_sample_counts(p.rows, p.cols), pr["noise"], act))
    return out


def _same(got, ref):
    for (a, r8, m2, c, nz, act), (ra, rr8, rm2, rc, rnz, ract) in zip(got, ref):
        if not (np.array_equal(a.view(np.uint32), ra.view(np.uint32)) and np.array_equal(r8, rr8)
                and np.array_equal(m2.view(np.uint32), rm2.view(np.uint32)) and np.array_equal(c, rc)
                and np.float64(nz).tobytes() == np.float64(rnz).tobytes() and act == ract):
            return False
    return True


def test_group_adaptive_frame_matches_single_gpu():
    import pysqt
    n_dev = _need_two()
    data = os.path.join(os.path.dirname(HERE), "data")
    hs = pysqt.HostScene.load(os.path.join(data, "scene.obj"), data)
    cam = pysqt.load_camera(os.path.join(data, "camera"))
    p = pysqt.make_params(320, 200, sum(CHUNKS), max_depth=6, seed=4)
    solo = pysqt.Context(0); solo.upload(hs)
    solo.render_begin(cam, p)
    ref = _frames(solo, p)
    solo.close()
    assert ref[-1][5] < ref[0][5]
    assert (ref[-1][3] < sum(CHUNKS)).any()
    n = 2
    while n <= n_dev:
        g = pysqt.Group(list(range(n)))
        g.upload(hs)
        g.render_begin(cam, p)
        assert _same(_frames(g, p), ref), "group of %d" % n
        g.close()
        n *= 2


def test_torchrun_ranks_adaptive_frame_matches_single_gpu():
    _need_two()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29641", os.path.join(HERE, "dist_adaptive_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "ADAPTIVE_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
