"""Context lifecycle on the B200: the group entry points reject a NULL context before running anything, and one context
that grows and shrinks every buffer family (image, sample buffer, pool slots, ray batch, scene, spheres, progressive,
adaptive and denoiser state) gives the same bits as a fresh context for every call."""
import ctypes as C

import numpy as np
import pytest

import pysqt
from common import bits, build_pair, random_rays

pytestmark = pytest.mark.gpu
SQT_E_INVALID = 1

# a grey triangle in front of an emissive one, seen by a camera at the origin looking down +x
TINY_V9 = np.array([[3, -5, -5, 3, 5, -5, 3, 0, 5], [4, -6, -6, 4, 6, -6, 4, -6, 6]], np.float32)
TINY_MATS = np.array([[0.5, 0.5, 0.5, 0.5, 0, 0, 0, 0], [0, 0.8, 0.8, 0.8, 1, 1, 1, 1]], np.float32)
TINY_CAM = np.array([0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0, 1], np.float32)
SPHERES_A = [(0.8, 0.5, -1.2, 0.6, 5), (-0.9, 1.0, 0.3, 0.45, 1), (0.0, -0.5, 1.2, 0.3, 3)]
SPHERES_B = [(0.2, 0.3, 0.4, 0.5, 2), (-0.5, -0.5, -0.5, 0.25, 1)]


def test_group_calls_reject_a_null_context(host_scene, camera):
    ctx = pysqt.Context(0)
    ctx.upload(host_scene)
    W, H, spp = 64, 48, 8
    p = pysqt.make_params(W, H, spp, max_depth=4, seed=1)
    ref = ctx.render(camera, p)
    ctx.render_begin(camera, p)
    ctx.render_advance(2)
    L = ctx.L
    arr = (C.c_void_p * 2)(ctx.h, None)
    cam, desc = pysqt.camera_struct(camera), host_scene.desc()
    st, pr, act = pysqt.Stats(), pysqt.Progress(), C.c_int64(-1)
    retire_all = pysqt.RetireParams(1e9, 1e9, 2, 0)
    dp = pysqt.DenoiseParams(1, pysqt.DENOISE_SIGMA_L, pysqt.DENOISE_SIGMA_Z, 0)
    rgb8 = np.zeros((H, W, 3), np.uint8)
    out = np.zeros((H, W, 3), np.float32)
    calls = {
        "sqt_render_group": lambda: L.sqt_render_group(arr, 2, C.byref(cam), C.byref(p), rgb8.ctypes.data, out.ctypes.data, C.byref(st)),
        "sqt_render_begin_group": lambda: L.sqt_render_begin_group(arr, 2, C.byref(cam), C.byref(p), C.byref(st)),
        "sqt_render_advance_group": lambda: L.sqt_render_advance_group(arr, 2, 3, C.byref(pr), C.byref(st)),
        "sqt_render_retire_group": lambda: L.sqt_render_retire_group(arr, 2, C.byref(retire_all), C.byref(act)),
        "sqt_denoise_group": lambda: L.sqt_denoise_group(arr, 2, C.byref(dp), rgb8.ctypes.data, out.ctypes.data, C.byref(st)),
        "sqt_upload_scene_group": lambda: L.sqt_upload_scene_group(arr, 2, C.byref(desc)),
    }
    for name, call in calls.items():
        assert call() == SQT_E_INVALID, name
    assert not rgb8.any() and not out.any() and pr.samples_done == 0 and act.value == -1
    assert st.kernel_launches == 0 and st.device_ms == 0
    # the frame begun on ctx is where it was: k = 2, nothing retired, and it still ends as the one-shot frame
    assert (ctx.download_sample_counts(H, W) == 2).all()
    assert ctx.render_advance(spp)["samples_done"] == spp
    rgb8, acc = ctx.download(H, W)
    assert np.array_equal(bits(acc), bits(ref["accum"])) and np.array_equal(rgb8, ref["rgb8"])
    ctx.close()


def _steps(hs, tiny, cam):
    """(name, call): each call brings a context into the state it needs and returns what it computed."""
    def one_shot(scene, c, w, h):
        def run(ctx):
            ctx.upload(scene)
            o = ctx.render(c, pysqt.make_params(w, h, 8, max_depth=5, seed=3))
            return [o["rgb8"], bits(o["accum"])]
        return run

    def batch(n, seed):
        def run(ctx):
            ctx.upload(hs)
            tri, dist, point = ctx.intersect_batch(*random_rays(n, seed))
            return [tri, bits(dist), bits(point)]
        return run

    def spheres(sp):
        def run(ctx):
            ctx.upload(hs)
            ctx.upload_spheres(sp)
            o = ctx.render(cam, pysqt.make_params(64, 48, 4, max_depth=4, seed=2))
            tri, dist, point = ctx.intersect_batch(*random_rays(2000, 7))
            return [o["rgb8"], bits(o["accum"]), tri, bits(dist), bits(point)]
        return run

    def progressive(w, h):
        def run(ctx):
            ctx.upload(hs)
            ctx.render_begin(cam, pysqt.make_params(w, h, 12, max_depth=5, seed=4))
            a = ctx.render_advance(4)
            active = ctx.render_retire(0.3, 0.0, 2)
            b = ctx.render_advance(4)
            dn = ctx.denoise(3)
            f = ctx.download_features(h, w)
            rgb8, acc = ctx.download(h, w)
            return [rgb8, bits(acc), bits(ctx.download_moments(h, w)), ctx.download_sample_counts(h, w), np.int64(active),
                    np.float64([a["noise"], b["noise"]]).view(np.uint64), dn["rgb8"], bits(dn["mean"]), f["surface"],
                    bits(f["depth"]), bits(f["normal"])]
        return run

    return [("one-shot tiny scene", one_shot(tiny, TINY_CAM, 64, 48)),
            ("one-shot large", one_shot(hs, cam, 200, 150)),
            ("one-shot small", one_shot(hs, cam, 64, 48)),
            ("one-shot tiny scene again", one_shot(tiny, TINY_CAM, 64, 48)),
            ("batch small", batch(1000, 1)),
            ("batch large", batch(60000, 2)),
            ("batch small again", batch(1000, 3)),
            ("spheres", spheres(SPHERES_A)),
            ("spheres re-uploaded", spheres(SPHERES_B)),
            ("progressive small", progressive(48, 32)),
            ("progressive large", progressive(160, 120)),
            ("progressive small again", progressive(48, 32)),
            ("one-shot after the frames", one_shot(hs, cam, 96, 64))]


@pytest.mark.parametrize("sbuf_mb", [None, "1"])
def test_buffer_reuse_across_sizes(host_scene, camera, monkeypatch, sbuf_mb):
    """One context runs every step in turn; each step's results equal those of the same step on a fresh context.  With a
    1 MB sample buffer the one-shot rounds split."""
    if sbuf_mb:
        monkeypatch.setenv("SQT_SBUF_MB", sbuf_mb)
    _, tiny = build_pair(TINY_V9, np.array([0, 1], np.int32), TINY_MATS)
    shared = pysqt.Context(0)
    for name, step in _steps(host_scene, tiny, camera):
        got = step(shared)
        fresh = pysqt.Context(0)
        want = step(fresh)
        fresh.close()
        assert len(got) == len(want)
        for i, (g, w) in enumerate(zip(got, want)):
            assert np.array_equal(g, w), (name, i)
    shared.close()
