"""Camera sampling on the B200 (include/sqt.h, sqt_set_lens): lens frames equal the oracle bit for bit under every
sample-buffer budget; a pinhole lens (aperture 0, no jitter) gives the plain frame; progressive and adaptive lens frames are exact
prefixes; the error rules; and the optics -- anti-aliased edges converge to the pixel's analytic coverage and a thin lens
blurs an edge by the analytic disk."""
import os

import numpy as np
import pytest

import pysqt
from oracle import oracle as O
from common import bits
import lens_oracle as LO

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LENSES = {"jitter": (1, 0.0, 1.0), "lens": (0, 0.08, 2.5), "both": (1, 0.08, 2.5)}


def ctx_with(monkeypatch, hs, **env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    c = pysqt.Context(0)
    for k in env:
        monkeypatch.delenv(k)
    c.upload(hs)
    return c


def _sphere_oracle():
    spheres = [(0.8, 0.5, -1.2, 0.6, 5), (-0.9, 1.0, 0.3, 0.45, 1), (0.0, -0.5, 1.2, 0.3, 3)]
    osc = O.Scene.load(os.path.join(ROOT, "data", "scene.obj"), os.path.join(ROOT, "data"))
    osc.make_bih()
    osc.set_spheres(spheres)
    return osc, spheres


def test_lens_frames_match_oracle(host_scene, oracle_scene, camera, monkeypatch):
    W, H, spp, depth = 64, 48, 8, 5
    osc_s, spheres = _sphere_oracle()
    for sbuf in (None, "1"):
        env = {} if sbuf is None else dict(SQT_SBUF_MB=sbuf)
        ctx = ctx_with(monkeypatch, host_scene, **env)
        for name, lens in LENSES.items():
            ctx.set_lens(*lens)
            p = pysqt.make_params(W, H, spp, max_depth=depth, seed=13)
            op = O.make_params(W, H, spp, max_depth=depth, seed=13, trig=1)
            ref = LO.render(oracle_scene, camera, op, lens)
            for cull in (True, False):
                ctx.set_leaf_cull(cull)
                out = ctx.render(camera, p)
                assert np.array_equal(bits(out["accum"]), bits(ref["accum"])), (sbuf, name, cull)
                assert np.array_equal(out["rgb8"], ref["rgb8"]), (sbuf, name, cull)
                st = out["stats"]
                assert st["samples"] == W * H * spp and st["rays_reference"] == st["rays_traced"]
            ctx.set_leaf_cull(True)
        ctx.upload_spheres(spheres)
        lens = LENSES["both"]
        ctx.set_lens(*lens)
        out = ctx.render(camera, pysqt.make_params(W, H, spp, max_depth=depth, seed=13))
        ref = LO.render(osc_s, camera, O.make_params(W, H, spp, max_depth=depth, seed=13, trig=1), lens)
        assert np.array_equal(bits(out["accum"]), bits(ref["accum"])), (sbuf, "spheres")
        ctx.close()


def test_full_size_lens_rows(gpu_ctx, host_scene, oracle_scene, camera):
    """Config 2 size (1920x1080, 8 bounces) with a lens: a few full-width rows equal orc_render_window's."""
    W, H, spp, depth, lens = 1920, 1080, 4, 8, (1, 0.05, 3.0)
    gpu_ctx.upload(host_scene)
    gpu_ctx.set_lens(*lens)
    try:
        out = gpu_ctx.render(camera, pysqt.make_params(W, H, spp, max_depth=depth, seed=2))
    finally:
        gpu_ctx.set_lens(None)
    op = O.make_params(W, H, spp, max_depth=depth, seed=2, trig=1)
    for row in (0, 537, 1079):
        want = LO.render_window(oracle_scene, camera, op, lens, row * W, (row + 1) * W)
        assert np.array_equal(bits(out["accum"][row]), bits(want)), row


def test_pinhole_lens_is_the_plain_frame(gpu_ctx, host_scene, camera):
    gpu_ctx.upload(host_scene)
    p = pysqt.make_params(96, 64, 12, max_depth=6, seed=8)
    plain = gpu_ctx.render(camera, p)
    gpu_ctx.set_lens(False, 0.0, 1.0)
    lens0 = gpu_ctx.render(camera, p)
    gpu_ctx.set_lens(None)
    again = gpu_ctx.render(camera, p)
    for r in (lens0, again):
        assert np.array_equal(bits(r["accum"]), bits(plain["accum"])) and np.array_equal(r["rgb8"], plain["rgb8"])
    assert lens0["stats"]["rays_reference"] == lens0["stats"]["rays_traced"] and lens0["stats"]["samples"] == plain["stats"]["samples"]


def test_progressive_lens_frames(gpu_ctx, host_scene, oracle_scene, camera):
    W, H, spp, depth, lens = 64, 48, 10, 4, (1, 0.1, 2.0)
    gpu_ctx.upload(host_scene)
    gpu_ctx.set_lens(*lens)
    p = pysqt.make_params(W, H, spp, max_depth=depth, seed=6)
    op = O.make_params(W, H, spp, max_depth=depth, seed=6, trig=1)
    ref = gpu_ctx.render(camera, p)
    for chunks in ([spp], [1] * spp, [3, 6, 7]):
        gpu_ctx.render_begin(camera, p)
        acc_ref = m2_ref = None
        k = 0
        for n in chunks:
            pr = gpu_ctx.render_advance(n)
            kb = min(k + n, spp)
            acc_ref, m2_ref = LO.render_range(oracle_scene, camera, op, lens, k, kb, acc_ref, m2_ref)
            k = kb
            rgb8, acc = gpu_ctx.download(H, W)
            assert pr["samples_done"] == k
            assert np.array_equal(bits(acc), bits(acc_ref)), (chunks, k)
            assert np.array_equal(bits(gpu_ctx.download_moments(H, W)), bits(m2_ref)), (chunks, k)
        assert np.array_equal(bits(acc), bits(ref["accum"])) and np.array_equal(rgb8, ref["rgb8"]), chunks
    gpu_ctx.set_lens(None)


def test_adaptive_lens_frame_is_an_exact_prefix(gpu_ctx, host_scene, oracle_scene, camera):
    W, H, spp, depth, lens = 64, 48, 32, 4, (1, 0.05, 2.0)
    gpu_ctx.upload(host_scene)
    gpu_ctx.set_lens(*lens)
    p = pysqt.make_params(W, H, spp, max_depth=depth, seed=3)
    op = O.make_params(W, H, spp, max_depth=depth, seed=3, trig=1)
    # the pixels whose centre ray misses: they are sampled and can retire (abs_tol > 0)
    org, dirs = O.make_rays(op, camera)
    tri, _, _ = gpu_ctx.intersect_batch(org, dirs)
    centre_miss = (tri < 0).reshape(H, W)
    assert centre_miss.any()
    st = gpu_ctx.render_begin(camera, p)
    assert st["rays_traced"] == 0
    for n in (4, 4, 8, 16):
        gpu_ctx.render_advance(n)
        gpu_ctx.render_retire(0.2, 1e-3, 4)
    counts = gpu_ctx.download_sample_counts(H, W)
    assert (counts < spp).any() and (counts == spp).any()
    assert (counts[centre_miss] < spp).any()
    _, acc = gpu_ctx.download(H, W)
    flat, cflat = acc.reshape(-1, 3), counts.reshape(-1)
    for n_p in np.unique(cflat):
        idx = np.nonzero(cflat == n_p)[0]
        for pix in idx[:: max(1, len(idx) // 40)]:
            want, _ = LO.prefix_window(oracle_scene, camera, op, lens, int(pix), int(pix) + 1, int(n_p))
            assert np.array_equal(bits(flat[pix]), bits(want[0])), (pix, n_p)
    gpu_ctx.set_lens(None)


def test_lens_error_rules(gpu_ctx, host_scene, camera):
    gpu_ctx.upload(host_scene)
    L, h = gpu_ctx.L, gpu_ctx.h
    import ctypes as C
    gpu_ctx.set_lens(True, 0.05, 2.0)
    for bad in [(2, 0.05, 2.0, 0), (1, -0.1, 2.0, 0), (1, float("inf"), 2.0, 0), (1, float("nan"), 2.0, 0),
                (1, 0.05, 0.0, 0), (1, 0.05, -1.0, 0), (1, 0.05, float("inf"), 0), (1, 0.05, 2.0, 1)]:
        assert L.sqt_set_lens(h, C.byref(pysqt.Lens(*bad))) == 1, bad
    # the lens is unchanged: the frame equals a frame with the lens set again
    p = pysqt.make_params(48, 32, 4, max_depth=4, seed=1)
    a = gpu_ctx.render(camera, p)
    gpu_ctx.set_lens(True, 0.05, 2.0)
    b = gpu_ctx.render(camera, p)
    assert np.array_equal(bits(a["accum"]), bits(b["accum"]))
    cast = pysqt.make_params(48, 32, 4, mode=1)
    assert L.sqt_render(h, C.byref(pysqt.camera_struct(camera)), C.byref(cast), None, None, None) == 5
    assert L.sqt_render_begin(h, C.byref(pysqt.camera_struct(camera)), C.byref(cast), None) in (5,)
    # denoise and features on a lens frame
    gpu_ctx.render_begin(camera, p)
    gpu_ctx.render_advance(2)
    dp = pysqt.DenoiseParams(2, 4.0, 0.05, 0)
    assert L.sqt_denoise(h, C.byref(dp), None, None, None) == 5
    assert L.sqt_download_features(h, None, None, None) == 5
    # advance after set_lens keeps the frame's own lens
    gpu_ctx.set_lens(None)
    gpu_ctx.render_advance(2)
    _, acc = gpu_ctx.download(32, 48)
    assert np.array_equal(bits(acc), bits(b["accum"]))
    gpu_ctx.set_lens(None)


def _emitter_scene(z, slope, c):
    """One emissive triangle (emissive 1, surfColor 0) in the plane x = z, seen by the identity camera at the origin, whose
    edge is the line yo = slope*xo + c of image offsets; the triangle covers the side below it."""
    P = lambda xo, yo: (z, z * xo, z * yo)
    v9 = np.float32([P(-8.0, slope * -8.0 + c) + P(8.0, slope * 8.0 + c) + P(0.0, -40.0)])
    mats8 = np.float32([[0, 0, 0, 0, 1, 1, 1, 1]])
    return pysqt.HostScene.from_arrays(v9, np.int32([0]), mats8)


IDENTITY = np.float32([0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0, 1])
W, H, SPP = 64, 48, 4096
SLOPE, C0 = 0.37, 0.05


def _mean(ctx, hs, lens):
    ctx.upload(hs)
    ctx.set_lens(*lens) if lens else ctx.set_lens(None)
    out = ctx.render(IDENTITY, pysqt.make_params(W, H, SPP, max_depth=1, seed=17, literal=False))
    ctx.set_lens(None)
    return out["accum"][..., 0].astype(np.float64) / SPP


def _bound(c):
    return 5 * np.sqrt(c * (1 - c) / SPP) + 1e-6


def test_anti_aliased_edge_converges_to_pixel_coverage(gpu_ctx):
    hs = _emitter_scene(3.0, SLOPE, C0)
    pin = _mean(gpu_ctx, hs, None)
    assert set(np.unique(pin)) <= {0.0, 1.0} and 0 < pin.mean() < 1
    aa = _mean(gpu_ctx, hs, (1, 0.0, 1.0))
    # hit iff yo < SLOPE*xo + C0 with xo = (fx - W/2)/W, yo = (H/2 - fy)/H: fy > g(fx)
    g = lambda fx: H / 2 - H * (SLOPE * (fx - W / 2) / W + C0)
    t = (np.arange(4096) + 0.5) / 4096 - 0.5
    y, x = np.mgrid[0:H, 0:W]
    cov = np.zeros((H, W))
    for j in range(W):
        gy = g(j + t)                                         # the edge across the pixel column
        cov[:, j] = np.clip((y[:, j, None] + 0.5) - gy[None, :], 0.0, 1.0).mean(axis=1)
    assert np.all(np.abs(aa - cov) <= _bound(cov)), np.abs(aa - cov).max()
    assert ((aa > 0) & (aa < 1)).sum() >= W


@pytest.mark.parametrize("z,f", [(3.0, 1.5), (3.0, 6.0)])
def test_thin_lens_blurs_an_edge_by_the_disk(gpu_ctx, z, f):
    A = 0.15
    hs = _emitter_scene(z, SLOPE, C0)
    m = _mean(gpu_ctx, hs, (0, A, f))
    rho = A * abs(1 / z - 1 / f)
    y, x = np.mgrid[0:H, 0:W].astype(np.float64)
    xo, yo = (x - W / 2) / W, (H / 2 - y) / H
    d = (SLOPE * xo + C0 - yo) / np.sqrt(1 + SLOPE ** 2)         # > 0: the sample point sees the emitter
    u = np.clip(-d / rho, -1, 1)
    cov = (np.arccos(u) - u * np.sqrt(1 - u * u)) / np.pi
    assert np.all(np.abs(m - cov) <= _bound(cov)), np.abs(m - cov).max()
    assert ((m > 0) & (m < 1)).sum() >= W


def test_in_focus_plane_stays_sharp(gpu_ctx):
    z = 3.0
    hs = _emitter_scene(z, SLOPE, C0)
    m = _mean(gpu_ctx, hs, (0, 0.15, z))
    y, x = np.mgrid[0:H, 0:W].astype(np.float64)
    g = H / 2 - H * (SLOPE * (x - W / 2) / W + C0)             # edge row at column x
    dpix = (y - g) / np.sqrt(1 + (H * SLOPE / W) ** 2)
    far = np.abs(dpix) > 1e-3
    assert np.all((m[far] == 0.0) | (m[far] == 1.0))
    assert np.array_equal(m[far] == 1.0, dpix[far] > 0)
