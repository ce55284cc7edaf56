"""The denoiser on the B200 (include/sqt.h: sqt_denoise, sqt_download_features): the device gives the host build's bits on the
downloaded frame, levels = 0 is the preview, mirrors pass through, the features match the oracle's primary hits, the calls
leave the frame as it was, the session rules hold, the filter lowers the error of a 16-spp preview, and the CLI."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import pysqt
from oracle import oracle as O
from common import bits
from denoise import ref as DR

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SL, SZ = pysqt.DENOISE_SIGMA_L, pysqt.DENOISE_SIGMA_Z


def ctx_with(monkeypatch, hs, **env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    c = pysqt.Context(0)
    for k in env:
        monkeypatch.delenv(k)
    c.upload(hs)
    return c


def host_denoise(ctx, hs, p, levels, k):
    """The host build of the filter on what the device holds: sums, moments, counts and features."""
    rgb8, s1 = ctx.download(p.rows, p.cols)
    s2 = ctx.download_moments(p.rows, p.cols)
    counts = ctx.download_sample_counts(p.rows, p.cols)
    feats = ctx.download_features(p.rows, p.cols)
    _, mi = hs.parsed_tris()
    mean = DR.denoise_host(s1, s2, counts, k, feats, mi, hs.mats["reflective"], levels, SL, SZ)
    return mean, rgb8, s1, counts, feats


@pytest.mark.parametrize("adaptive", [False, True])
def test_device_matches_host_build(host_scene, camera, monkeypatch, adaptive):
    """Levels 1, 3 and 5: the denoised mean bits equal the host build's, the RGB8 is the tone map of that mean; levels = 0
    is the preview's mean and RGB8; mirror pixels (material 5 of scene.obj) pass through bit for bit."""
    ctx = ctx_with(monkeypatch, host_scene)
    p = pysqt.make_params(160, 120, 16, max_depth=8, seed=5)
    ctx.render_begin(camera, p)
    ctx.render_advance(6)
    if adaptive:
        assert ctx.render_retire(0.3, 0.0, 2) < (p.rows * p.cols)
    k = ctx.render_advance(4)["samples_done"]
    counts = ctx.download_sample_counts(p.rows, p.cols)
    assert (counts < k).any() == adaptive
    base = ctx.denoise(0, SL, SZ)
    for levels in (1, 3, 5):
        want, preview, s1, counts, feats = host_denoise(ctx, host_scene, p, levels, k)
        got = ctx.denoise(levels, SL, SZ)
        assert np.array_equal(bits(got["mean"]), bits(want)), (levels, int((bits(got["mean"]) != bits(want)).sum()))
        assert np.array_equal(got["rgb8"], O.tone_map(got["mean"], 1, trig=1))
        assert not np.array_equal(bits(got["mean"]), bits(base["mean"]))
        _, mi = host_scene.parsed_tris()
        mirror = (feats["surface"] >= 0) & (mi[np.maximum(feats["surface"], 0)] == 5)
        assert mirror.sum() > 100
        assert np.array_equal(bits(got["mean"][mirror]), bits(base["mean"][mirror]))
    n = counts.astype(np.float32)
    assert np.array_equal(bits(base["mean"]), bits(s1 * (np.float32(1) / n)[..., None]))
    assert np.array_equal(base["rgb8"], preview)
    ctx.close()


def test_features_match_the_oracle(gpu_ctx, host_scene, oracle_scene, camera):
    """surface = the oracle's hit index; origin + depth * direction in binary32 = the oracle's hit point bits; unit normals
    facing the camera ray."""
    gpu_ctx.upload(host_scene)
    W, H = 200, 150
    p = pysqt.make_params(W, H, 4, max_depth=3, seed=1)
    gpu_ctx.render_begin(camera, p)
    gpu_ctx.render_advance(2)
    f = gpu_ctx.download_features(H, W)
    org, dirs = O.make_rays(O.make_params(W, H, 1), camera)
    otri, _, opoint = oracle_scene.intersect_batch(org, dirs)
    surf = f["surface"].reshape(-1)
    assert np.array_equal(surf, otri)
    hit = surf >= 0
    assert 0 < hit.sum() < W * H
    t = f["depth"].reshape(-1, 1)
    pt = (org + (t * dirs).astype(np.float32)).astype(np.float32)
    assert np.array_equal(bits(pt[hit]), bits(opoint[hit]))
    n = f["normal"].reshape(-1, 3).astype(np.float64)
    assert np.abs(np.linalg.norm(n[hit], axis=1) - 1.0).max() <= 1e-6
    assert ((n[hit] * dirs[hit]).sum(1) <= 0).all()
    assert not n[~hit].any() and not t[~hit].any()


@pytest.mark.parametrize("retire", [False, True])
def test_denoise_leaves_the_frame_as_it_was(gpu_ctx, host_scene, camera, retire):
    """Denoise (and a feature download) after every chunk: the sums, moments, counts, previews and noise are those of the
    same frame without them; without retire the final frame is sqt_render's.  Two calls on one state give the same bits."""
    gpu_ctx.upload(host_scene)
    p = pysqt.make_params(128, 96, 12, max_depth=6, seed=8)

    def frame(denoise):
        gpu_ctx.render_begin(camera, p)
        out = []
        for n in (2, 3, 3, 4):
            pr = gpu_ctx.render_advance(n)
            if retire:
                gpu_ctx.render_retire(0.2, 0.0, 2)
            if denoise:
                a = gpu_ctx.denoise(3, SL, SZ)
                gpu_ctx.download_features(p.rows, p.cols)
                b = gpu_ctx.denoise(3, SL, SZ)
                assert np.array_equal(bits(a["mean"]), bits(b["mean"])) and np.array_equal(a["rgb8"], b["rgb8"])
            rgb8, acc = gpu_ctx.download(p.rows, p.cols)
            out.append((bits(acc), rgb8, bits(gpu_ctx.download_moments(p.rows, p.cols)),
                        gpu_ctx.download_sample_counts(p.rows, p.cols), np.float64(pr["noise"]).tobytes()))
        return out

    plain, with_dn = frame(False), frame(True)
    for a, b in zip(plain, with_dn):
        for x, y in zip(a, b):
            assert np.array_equal(x, y)
    if not retire:
        ref = gpu_ctx.render(camera, p)
        assert np.array_equal(with_dn[-1][0], bits(ref["accum"])) and np.array_equal(with_dn[-1][1], ref["rgb8"])


def test_stats_and_launches(gpu_ctx, host_scene, camera):
    gpu_ctx.upload(host_scene)
    p = pysqt.make_params(160, 120, 8, max_depth=4, seed=2)
    gpu_ctx.render_begin(camera, p)
    gpu_ctx.render_advance(4)
    first = gpu_ctx.denoise(5, SL, SZ)["stats"]
    again = gpu_ctx.denoise(2, SL, SZ)["stats"]
    assert first["kernel_launches"] == 1 + 1 + 5 + 1           # features, prep, levels, tone map
    assert again["kernel_launches"] == 1 + 2 + 1                # the features of this frame are cached
    assert first["device_ms"] > 0 and first["d2h_bytes"] == p.rows * p.cols * 15 and first["d2h_ms"] > 0
    assert first["reduce_ms"] >= 0 and first["rays_traced"] == 0


def _raw_denoise(ctx, levels, sl, sz, reserved=0):
    dp = pysqt.DenoiseParams(levels, sl, sz, reserved)
    return ctx.L.sqt_denoise(ctx.h, C.byref(dp), None, None, None)


def test_session_rules(gpu_ctx, host_scene, camera):
    L = gpu_ctx.L
    gpu_ctx.upload(host_scene)
    p = pysqt.make_params(64, 48, 8, max_depth=3, seed=1)
    gpu_ctx.render(camera, p)
    assert _raw_denoise(gpu_ctx, 3, SL, SZ) == 1                                      # outside a frame
    assert L.sqt_download_features(gpu_ctx.h, None, None, None) == 1
    gpu_ctx.render_begin(camera, p)
    assert _raw_denoise(gpu_ctx, 3, SL, SZ) == 1                                      # k = 0
    gpu_ctx.render_advance(1)
    assert _raw_denoise(gpu_ctx, 3, SL, SZ) == 1                                      # k = 1
    assert L.sqt_download_features(gpu_ctx.h, None, None, None) == 1
    gpu_ctx.render_advance(1)
    for lv, sl, sz, res in [(9, SL, SZ, 0), (-1, SL, SZ, 0), (3, 0.0, SZ, 0), (3, -1.0, SZ, 0), (3, float("inf"), SZ, 0),
                            (3, float("nan"), SZ, 0), (3, SL, 0.0, 0), (3, SL, float("inf"), 0), (3, SL, SZ, 1)]:
        assert _raw_denoise(gpu_ctx, lv, sl, sz, res) == 1, (lv, sl, sz, res)
    assert L.sqt_denoise(gpu_ctx.h, None, None, None, None) == 1
    for lv in (0, 8):
        assert _raw_denoise(gpu_ctx, lv, SL, SZ) == 0
    f = gpu_ctx.download_features(p.rows, p.cols)
    assert gpu_ctx.render_advance(6)["samples_done"] == 8                             # the frame goes on
    # whatever ends a frame drops its features: a new frame of another size has its own
    gpu_ctx.render_begin(camera, pysqt.make_params(32, 24, 4, max_depth=3, seed=1))
    gpu_ctx.render_advance(2)
    g = gpu_ctx.download_features(24, 32)
    org, dirs = O.make_rays(O.make_params(32, 24, 1), camera)
    assert np.array_equal(g["surface"].reshape(-1), gpu_ctx.intersect_batch(org, dirs)[0])
    assert f["surface"].shape == (48, 64)
    for end in (lambda: gpu_ctx.tone_map(np.zeros((4, 3), np.float32)), lambda: gpu_ctx.upload(host_scene)):
        gpu_ctx.render_begin(camera, p)
        gpu_ctx.render_advance(2)
        assert _raw_denoise(gpu_ctx, 1, SL, SZ) == 0
        end()
        assert _raw_denoise(gpu_ctx, 1, SL, SZ) == 1
        assert L.sqt_download_features(gpu_ctx.h, None, None, None) == 1
    gpu_ctx.render_begin(camera, pysqt.make_params(64, 48, 8, max_depth=3, seed=1, flags=pysqt.SQT_F_NO_PRIMARY_REUSE))
    gpu_ctx.render_advance(2)
    assert _raw_denoise(gpu_ctx, 3, SL, SZ) == 5
    assert L.sqt_download_features(gpu_ctx.h, None, None, None) == 5


# Measured on one B200 (1000 W, 1965 MHz) with the default parameters: the noisy 16-spp mean of this frame has 8.70 times the
# MSE of the denoised one (0.939 against 0.108).  The bound keeps a margin of more than 2x below that.
MIN_MSE_RATIO = 4.0


def test_denoised_16spp_has_a_quarter_of_the_error_or_less(gpu_ctx, host_scene, camera):
    gpu_ctx.upload(host_scene)
    W, H = 320, 240
    ref = gpu_ctx.render(camera, pysqt.make_params(W, H, 4096, max_depth=8, seed=99))["accum"] / np.float32(4096)
    p = pysqt.make_params(W, H, 1024, max_depth=8, seed=11)
    gpu_ctx.render_begin(camera, p)
    gpu_ctx.render_advance(16)
    noisy = gpu_ctx.denoise(0, SL, SZ)["mean"]
    dn = gpu_ctx.denoise(pysqt.DENOISE_LEVELS, SL, SZ)["mean"]
    mse_noisy = float(((noisy.astype(np.float64) - ref) ** 2).mean())
    mse_dn = float(((dn.astype(np.float64) - ref) ** 2).mean())
    print("MSE noisy %.6g denoised %.6g ratio %.3f" % (mse_noisy, mse_dn, mse_noisy / mse_dn))
    assert mse_noisy >= MIN_MSE_RATIO * mse_dn


def _png_pixels(path, W, H):
    import zlib
    data = open(path, "rb").read()
    pos, idat = 8, b""
    while pos < len(data):
        n = int.from_bytes(data[pos:pos + 4], "big")
        if data[pos + 4:pos + 8] == b"IDAT":
            idat += data[pos + 8:pos + 8 + n]
        pos += 12 + n
    raw = np.frombuffer(zlib.decompress(idat), np.uint8).reshape(H, 1 + 3 * W)
    return raw[:, 1:].reshape(H, W, 3)


def test_cli_denoise(tmp_path, host_scene, camera):
    exe = os.path.join(ROOT, "squigly-trace_b200", "squigly-trace")
    a, b = tmp_path / "plain.png", tmp_path / "dn.png"
    args = [exe, "-s", "16", "-d", "96,64", "--progress=8"]
    for extra, out in (([], a), (["--denoise"], b)):
        r = subprocess.run(args + extra + ["-p", str(out)], cwd=ROOT, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr
    assert a.read_bytes() == b.read_bytes()
    assert not (tmp_path / "plain-denoised.png").exists()
    d = tmp_path / "dn-denoised.png"
    # the same calls through pysqt, with the CLI's defaults: Lib.hs's index convention, 3 bounces, seed 0, data/camera
    ctx = pysqt.Context(0)
    ctx.upload(host_scene)
    p = pysqt.make_params(96, 64, 16, max_depth=3, seed=0, literal=True)
    ctx.render_begin(camera, p)
    ctx.render_advance(8)
    ctx.render_advance(8)
    want = ctx.denoise()["rgb8"]
    ctx.close()
    assert np.array_equal(_png_pixels(d, p.cols, p.rows), want)
