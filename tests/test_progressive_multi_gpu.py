"""Progressive frames across GPUs (skipped on boxes with fewer than 2 GPUs, like test_multi_gpu.py): previews and the final
frame of a group are bit-identical to one GPU's, in one process and under torchrun, and a rank that cannot start the frame
makes every rank fail at begin without a hang."""
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
pytestmark = pytest.mark.gpu
CHUNKS = (1, 4, 3, 8)


def _need_two():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    return torch.cuda.device_count()


def _frames(r, p, chunks):
    """(accum, rgb8, m2, noise) after every chunk of a progressive frame on r (a Context or a Group)."""
    ctx0 = r.ctxs[0] if hasattr(r, "ctxs") else r
    out = []
    for n in chunks:
        pr = r.render_advance(n)
        rgb8, acc = ctx0.download(p.rows, p.cols)
        out.append((acc, rgb8, ctx0.download_moments(p.rows, p.cols), pr["noise"]))
    return out


def test_group_previews_match_single_gpu():
    import pysqt
    n_dev = _need_two()
    data = os.path.join(os.path.dirname(HERE), "data")
    hs = pysqt.HostScene.load(os.path.join(data, "scene.obj"), data)
    cam = pysqt.load_camera(os.path.join(data, "camera"))
    p = pysqt.make_params(320, 200, sum(CHUNKS), max_depth=6, seed=4)
    solo = pysqt.Context(0); solo.upload(hs)
    solo.render_begin(cam, p)
    ref = _frames(solo, p, CHUNKS)
    one_shot = solo.render(cam, p)
    solo.close()
    n = 2
    while n <= n_dev:
        g = pysqt.Group(list(range(n)))
        g.upload(hs)
        g.render_begin(cam, p)
        got = _frames(g, p, CHUNKS)
        for (a, r8, m2, nz), (ra, rr8, rm2, rnz) in zip(got, ref):
            assert np.array_equal(a.view(np.uint32), ra.view(np.uint32)), "group of %d" % n
            assert np.array_equal(r8, rr8) and np.array_equal(m2.view(np.uint32), rm2.view(np.uint32))
            assert np.array_equal(np.float64(nz).view(np.uint64), np.float64(rnz).view(np.uint64))
        assert np.array_equal(got[-1][1], one_shot["rgb8"])
        g.close()
        n *= 2
    # one rank without a scene: begin fails on every rank, nobody hangs, and the group is usable afterwards
    g = pysqt.Group([0, 1])
    g.ctxs[0].upload(hs)
    with pytest.raises(pysqt.SqtError):
        g.render_begin(cam, p)
    g.upload(hs)
    g.render_begin(cam, p)
    got = _frames(g, p, CHUNKS)
    assert np.array_equal(got[-1][0].view(np.uint32), one_shot["accum"].view(np.uint32))
    g.close()


def test_torchrun_ranks_previews_match_single_gpu():
    _need_two()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29637", os.path.join(HERE, "dist_progressive_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "PROGRESSIVE_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
