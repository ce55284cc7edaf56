"""Adaptive frames on the B200 (include/sqt.h: sqt_render_retire): zero tolerances change nothing, every pixel is the exact
n_p-sample prefix of the full frame, each call retires exactly the pixels the formula picks, results do not depend on the
sample-buffer budget, work counts follow the active set, the noise estimate uses per-pixel counts, the
session rules hold, config 2 at full size, and the CLI."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import pysqt
from oracle import oracle as O
from common import bits
import progressive_ref as PR
from adaptive import ref as AR

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def ctx_with(monkeypatch, hs, **env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    c = pysqt.Context(0)
    for k in env:
        monkeypatch.delenv(k)
    c.upload(hs)
    return c


def adaptive_run(ctx, cam, p, chunks, rel, abs_tol=0.0, min_samples=2, check=None):
    """begin, then advance + retire per chunk; check(k, active_before, active_after, s1, s2, counts, outs) may look at each
    retire.  Returns the advances' results and the retires' active counts."""
    ctx.render_begin(cam, p)
    outs, acts = [], []
    for n in chunks:
        outs.append(ctx.render_advance(n))
        k = outs[-1]["samples_done"]
        if k < 2:
            continue
        if check:
            _, s1 = ctx.download(p.rows, p.cols)
            s2 = ctx.download_moments(p.rows, p.cols)
        acts.append(ctx.render_retire(rel, abs_tol, min_samples))
        if check:
            check(k, s1, s2, acts[-1])
    return outs, acts


def final(ctx, p):
    rgb8, acc = ctx.download(p.rows, p.cols)
    return rgb8, acc, ctx.download_moments(p.rows, p.cols), ctx.download_sample_counts(p.rows, p.cols)


def test_zero_tolerances_change_nothing_and_results_do_not_depend_on_the_round_width(host_scene, camera, monkeypatch):
    """Zero tolerances retire nothing: the frame is sqt_render's bit for bit.  With a tolerance, the same call sequence gives
    the same sums, moments, counts and RGB8 under every sample-buffer budget (samples per round)."""
    W, H, spp = 160, 120, 16
    p = pysqt.make_params(W, H, spp, max_depth=5, seed=9)
    results = []
    for sbuf in (None, "1"):
        env = {} if sbuf is None else dict(SQT_SBUF_MB=sbuf)
        ctx = ctx_with(monkeypatch, host_scene, **env)
        ref = ctx.render(camera, p)
        outs, acts = adaptive_run(ctx, camera, p, [3, 5, 8], 0.0, 0.0, 2)
        hits = outs[0]["stats"]["samples"] // 3
        assert acts == [hits] * 3
        rgb8, acc, _, counts = final(ctx, p)
        assert (counts == spp).all()
        assert np.array_equal(bits(acc), bits(ref["accum"])) and np.array_equal(rgb8, ref["rgb8"]), sbuf
        adaptive_run(ctx, camera, p, [2, 2, 1, 3, 8], 0.05, 0.0, 2)
        results.append(final(ctx, p))
        ctx.close()
    # the reference: a fresh context at the default budget
    ctx = ctx_with(monkeypatch, host_scene)
    adaptive_run(ctx, camera, p, [2, 2, 1, 3, 8], 0.05, 0.0, 2)
    want = final(ctx, p)
    ctx.close()
    assert 0 < (want[3] < spp).sum() < H * W
    for got in results:
        for g, w in zip(got, want):
            assert np.array_equal(g.view(np.uint8), w.view(np.uint8))


def _sphere_scene(host_scene):
    spheres = [(0.8, 0.5, -1.2, 0.6, 5), (-0.9, 1.0, 0.3, 0.45, 1), (0.0, -0.5, 1.2, 0.3, 3)]
    osc = O.Scene.load(os.path.join(ROOT, "data", "scene.obj"), os.path.join(ROOT, "data"))
    osc.make_bih()
    osc.set_spheres(spheres)
    return osc, spheres


@pytest.mark.parametrize("case", ["depth3", "depth8", "literal", "spheres"])
def test_every_pixel_is_its_exact_prefix_and_each_retire_picks_the_formula_set(host_scene, oracle_scene, camera, case):
    W, H, spp, depth, literal = 64, 48, 16, 3, False
    if case == "depth8":
        depth = 8
    if case == "literal":
        W, H, literal = 56, 40, True
    ctx = pysqt.Context(0)
    ctx.upload(host_scene)
    osc = oracle_scene
    if case == "spheres":
        osc, spheres = _sphere_scene(host_scene)
        ctx.upload_spheres(spheres)
    p = pysqt.make_params(W, H, spp, max_depth=depth, seed=5, literal=literal)
    op = O.make_params(W, H, spp, max_depth=depth, seed=5, trig=1, literal=literal)
    rows, cols = p.rows, p.cols
    chunks = (2, 2, 4, 8)
    # the oracle's sums and moments after every chunk
    snaps, a, q, kk = {}, None, None, 0
    for n in chunks:
        a, q = PR.render_range(osc, camera, op, kk, kk + n, a, q)
        kk += n
        snaps[kk] = (a.reshape(-1, 3), q.reshape(-1, 3))
    # at these sample counts a standard error below the mean retires 13 % to 30 % of the hit pixels of the four cases
    rel = 1.0
    n_pred = np.zeros(rows * cols, np.int32)            # 0 = active (numpy's bookkeeping of the retire sets)
    state = {}

    def check(k, s1, s2, active):
        if k == spp:                                    # a no-op
            assert active == state["active"]
            return
        dec = AR.retire_numpy(s1, s2, k, rel, 0.0) & (n_pred == 0)
        n_pred[dec] = k
        hits = state["hits"]
        state["active"] = hits - int((n_pred > 0).sum())
        assert active == state["active"], (case, k)

    ctx.render_begin(camera, p)
    k = 0
    for n in chunks:
        pr = ctx.render_advance(n)
        if k == 0:
            state["hits"] = pr["stats"]["samples"] // n
            state["active"] = state["hits"]
        else:
            assert pr["stats"]["samples"] == state["active"] * n, (case, k)          # work follows the active set
        k += n
        _, s1 = ctx.download(rows, cols)
        s2 = ctx.download_moments(rows, cols)
        check(k, s1, s2, ctx.render_retire(rel, 0.0, 2))
    counts = ctx.download_sample_counts(rows, cols).ravel()
    assert np.array_equal(counts, np.where(n_pred > 0, n_pred, spp))
    frac = (counts < spp).sum() / state["hits"]
    assert 0.1 <= frac <= 0.9, (case, frac)
    rgb8, acc, m2, _ = final(ctx, p)
    # the oracle's prefix of every pixel at its own count
    want_a = np.zeros((rows * cols, 3), np.float32)
    want_q = np.zeros((rows * cols, 3), np.float32)
    for kk, (a, q) in snaps.items():
        sel = counts == kk
        want_a[sel] = a[sel]
        want_q[sel] = q[sel]
    assert np.array_equal(bits(acc.reshape(-1, 3)), bits(want_a)), case
    assert np.array_equal(bits(m2.reshape(-1, 3)), bits(want_q)), case
    assert np.array_equal(rgb8, AR.tone_map(want_a, counts).reshape(rows, cols, 3)), case
    ctx.close()


def test_work_and_an_empty_active_set(gpu_ctx, host_scene, camera):
    gpu_ctx.upload(host_scene)
    W, H, spp = 80, 60, 12
    p = pysqt.make_params(W, H, spp, max_depth=6, seed=3)
    ref = gpu_ctx.render(camera, p)
    gpu_ctx.render_begin(camera, p)
    st = gpu_ctx.render_advance(2)["stats"]
    hits = st["samples"] // 2
    assert 0 < hits < W * H
    assert gpu_ctx.render_retire(0.0, 1e30, 2) == 0            # abs_tol above every error: every hit pixel retires
    pr = gpu_ctx.render_advance(3)
    assert pr["samples_done"] == 5 and pr["stats"]["kernel_launches"] == 0 and pr["stats"]["samples"] == 0
    assert gpu_ctx.render_retire(0.0, 1e30, 2) == 0
    gpu_ctx.render_advance(spp)
    rgb8, acc, _, counts = final(gpu_ctx, p)
    a2 = ref["accum"]                                           # misses are black in every frame
    hit = counts == 2
    assert hit.sum() == hits and (counts[~hit] == spp).all()
    assert not acc[~hit].any() and np.array_equal(rgb8[~hit], ref["rgb8"][~hit])
    assert np.array_equal(rgb8, AR.tone_map(acc.reshape(-1, 3), counts.ravel()).reshape(H, W, 3))
    assert a2[~hit].sum() == 0


def test_noise_uses_per_pixel_counts(gpu_ctx, host_scene, camera):
    gpu_ctx.upload(host_scene)
    W, H, spp = 96, 64, 16
    p = pysqt.make_params(W, H, spp, max_depth=5, seed=1)
    seqs = []
    for rep in range(2):
        gpu_ctx.render_begin(camera, p)
        seq = []
        for n in (2, 2, 4, 8):
            pr = gpu_ctx.render_advance(n)
            k = pr["samples_done"]
            _, acc = gpu_ctx.download(H, W)
            m2 = gpu_ctx.download_moments(H, W)
            counts = gpu_ctx.download_sample_counts(H, W)
            assert pr["noise"] == pytest.approx(AR.noise(acc, m2, counts), rel=1e-9)
            seq.append(pr["noise"])
            gpu_ctx.render_retire(0.1, 0.0, 2)
        assert (counts < spp).any()
        seqs.append(np.array(seq, np.float64))
    assert np.array_equal(seqs[0].view(np.uint64), seqs[1].view(np.uint64))


def test_session_rules(gpu_ctx, host_scene, camera):
    gpu_ctx.upload(host_scene)
    L, h = gpu_ctx.L, gpu_ctx.h
    W, H, spp = 48, 32, 8
    p = pysqt.make_params(W, H, spp, max_depth=4, seed=2)
    counts = np.zeros((H, W), np.int32)
    act = C.c_int64()

    def retire(rel=0.1, ab=0.0, mn=2, reserved=0):
        rp = pysqt.RetireParams(rel, ab, mn, reserved)
        return L.sqt_render_retire(h, C.byref(rp), C.byref(act))

    gpu_ctx.render(camera, p)
    assert retire() == 1 and "no progressive frame" in gpu_ctx.last_error()
    assert L.sqt_download_sample_counts(h, counts.ctypes.data) == 1
    gpu_ctx.render_begin(camera, p)
    assert L.sqt_download_sample_counts(h, counts.ctypes.data) == 0 and not counts.any()
    assert retire() == 1                                       # k = 0
    gpu_ctx.render_advance(1)
    assert retire() == 1                                       # k = 1
    gpu_ctx.render_advance(1)
    for bad in (dict(mn=1), dict(mn=-5), dict(rel=-0.1), dict(ab=-1e-9), dict(rel=float("nan")), dict(ab=float("nan")),
                dict(reserved=1)):
        assert retire(**bad) == 1, bad
    assert L.sqt_render_retire(h, None, None) == 1
    assert retire() == 0 and 0 < act.value < W * H
    a1 = act.value
    assert retire(mn=3) == 0 and act.value == a1               # k = 2 < min_samples: nothing retires
    gpu_ctx.render_advance(spp)
    before = gpu_ctx.download_sample_counts(H, W)
    a0 = act.value
    assert retire() == 0 and act.value == a0                   # k = spp: a no-op
    assert np.array_equal(gpu_ctx.download_sample_counts(H, W), before)
    # primary reuse off is unsupported
    gpu_ctx.render_begin(camera, pysqt.make_params(W, H, spp, max_depth=4, seed=2, flags=pysqt.SQT_F_NO_PRIMARY_REUSE))
    gpu_ctx.render_advance(2)
    assert retire() == 5
    # whatever ends a frame ends its adaptive state
    for end in ("render", "tone_map", "upload", "spheres", "begin"):
        gpu_ctx.render_begin(camera, p)
        gpu_ctx.render_advance(2)
        assert retire(ab=1e30) == 0 and act.value == 0
        if end == "render":
            gpu_ctx.render(camera, p)
        elif end == "tone_map":
            gpu_ctx.tone_map(np.ones((4, 3), np.float32))
        elif end == "upload":
            gpu_ctx.upload(host_scene)
        elif end == "spheres":
            gpu_ctx.upload_spheres([])
        if end == "begin":
            gpu_ctx.render_begin(camera, p)
            assert (gpu_ctx.download_sample_counts(H, W) == 0).all()
            st = gpu_ctx.render_advance(spp)
            assert st["stats"]["samples"] > 0 and (gpu_ctx.download_sample_counts(H, W) == spp).all()
        else:
            assert retire() == 1, end
            assert L.sqt_download_sample_counts(h, counts.ctypes.data) == 1, end


def test_config2_full_size_adaptive(gpu_ctx, host_scene, oracle_scene, camera):
    """BASELINE config 2 (1920x1080, 1024 spp, 8 bounces) in chunks of 64 with retire (min 64): the active count never rises
    and twelve sampled pixels equal the oracle's prefix at their own count."""
    gpu_ctx.upload(host_scene)
    W, H, spp = 1920, 1080, 1024
    p = pysqt.make_params(W, H, spp, max_depth=8, seed=0)
    gpu_ctx.render_begin(camera, p)
    acts = []
    while True:
        pr = gpu_ctx.render_advance(64)
        acts.append(gpu_ctx.render_retire(0.02, 0.0, 64))
        if pr["samples_done"] == spp:
            break
    assert all(b <= a for a, b in zip(acts, acts[1:])) and acts[-1] < acts[0]
    rgb8, acc = gpu_ctx.download(H, W)
    counts = gpu_ctx.download_sample_counts(H, W).ravel()
    assert (counts % 64 == 0).all() and counts.min() >= 64
    op = O.make_params(W, H, spp, max_depth=8, seed=0, trig=1)
    rng = np.random.default_rng(5)
    hit = np.flatnonzero(acc.reshape(-1, 3).sum(1) > 0)
    early, late = hit[counts[hit] < spp], hit[counts[hit] == spp]
    assert len(early) >= 6
    n_late = min(6, len(late))
    picks = list(rng.choice(early, 12 - n_late, replace=False)) + list(rng.choice(late, n_late, replace=False))
    for pix in picks:
        want, _ = AR.prefix_window(oracle_scene, camera, op, int(pix), int(pix) + 1, int(counts[pix]))
        assert np.array_equal(bits(acc.reshape(-1, 3)[pix]), bits(want[0])), "pixel %d (n_p %d)" % (pix, counts[pix])
        assert np.array_equal(rgb8.reshape(-1, 3)[pix], AR.tone_map(want, counts[pix:pix + 1])[0])


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
    assert (raw[:, 0] == 0).all()
    return raw[:, 1:].reshape(H, W, 3)


def test_cli_adaptive(tmp_path, host_scene, camera):
    exe = os.path.join(ROOT, "squigly-trace_b200", "squigly-trace")
    a, b, c = tmp_path / "plain.png", tmp_path / "zero.png", tmp_path / "tol.png"
    args = [exe, "-s", "12", "-d", "96,64"]
    runs = [subprocess.run(args + ["-p", str(a)], cwd=ROOT, capture_output=True, text=True, timeout=300),
            subprocess.run(args + ["--progress=3", "--adaptive=0", "-p", str(b)], cwd=ROOT, capture_output=True, text=True, timeout=300),
            subprocess.run(args + ["--progress=3", "--adaptive=0.3,0.001,3", "-p", str(c)], cwd=ROOT, capture_output=True, text=True,
                           timeout=300)]
    for r in runs:
        assert r.returncode == 0, r.stderr
    assert a.read_bytes() == b.read_bytes()
    lines = [l for l in runs[2].stdout.splitlines() if " samples  noise " in l]
    assert [l.split()[0] for l in lines] == ["3/12", "6/12", "9/12", "12/12"]
    active = [int(l.split("active ")[1].split()[0]) for l in lines]
    # the same calls through pysqt, with the CLI's defaults: Lib.hs's index convention, 3 bounces, seed 0, data/camera
    ctx = pysqt.Context(0)
    ctx.upload(host_scene)
    p = pysqt.make_params(96, 64, 12, max_depth=3, seed=0, literal=True)
    _, acts = adaptive_run(ctx, camera, p, [3, 3, 3, 3], 0.3, 0.001, 3)
    rgb8, _ = ctx.download(p.rows, p.cols)
    ctx.close()
    assert acts == active and acts[-1] < acts[0]
    assert np.array_equal(_png_pixels(c, p.cols, p.rows), rgb8)
