"""Progressive frames on the B200 (include/sqt.h: sqt_render_begin / sqt_render_advance): chunked frames end bit-identical to
the one-shot frame, previews and second moments match the oracle's range render, the noise estimate matches its
definition, work counts add up, and the session rules hold."""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np
import pytest

import pysqt
from oracle import oracle as O
from common import bits, build_pair
import progressive_ref as PR

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

COUNTERS = ("rays_traced", "rays_reference", "samples", "branch_visits", "child_box_tests", "tri_tests", "leaves_culled",
            "mt_pass_a", "mt_pass_u", "mt_pass_v", "mt_accept")


def ctx_with(monkeypatch, hs, **env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    c = pysqt.Context(0)
    for k in env:
        monkeypatch.delenv(k)
    c.upload(hs)
    return c


def run_chunks(ctx, cam, p, chunks):
    ctx.render_begin(cam, p)
    outs = [ctx.render_advance(n) for n in chunks]
    assert outs[-1]["samples_done"] == p.spp
    return outs


def test_chunked_final_frame_equals_one_shot(host_scene, camera, monkeypatch):
    W, H, spp = 160, 120, 16
    p = pysqt.make_params(W, H, spp, max_depth=5, seed=9)
    for sbuf in (None, "1"):          # 1 MB: 4 samples per round, so chunks of 6 and 7 straddle round boundaries
        env = {} if sbuf is None else dict(SQT_SBUF_MB=sbuf)
        ctx = ctx_with(monkeypatch, host_scene, **env)
        ref = ctx.render(camera, p)
        chunkings = [[spp], [1] * spp, [3, 5, spp - 8]] + ([[3, 6, 7], [5, 100]] if sbuf else [])
        for chunks in chunkings:
            run_chunks(ctx, camera, p, chunks)
            rgb8, acc = ctx.download(H, W)
            assert np.array_equal(bits(acc), bits(ref["accum"])), (sbuf, chunks)
            assert np.array_equal(rgb8, ref["rgb8"]), (sbuf, chunks)
        ctx.close()


def _sphere_pair(host_scene):
    spheres = [(0.8, 0.5, -1.2, 0.6, 5), (-0.9, 1.0, 0.3, 0.45, 1), (0.0, -0.5, 1.2, 0.3, 3)]
    osc = O.Scene.load(os.path.join(ROOT, "data", "scene.obj"), os.path.join(ROOT, "data"))
    osc.make_bih()
    osc.set_spheres(spheres)
    return osc, spheres


@pytest.mark.parametrize("case", ["depth3", "depth8", "literal", "no_primary_reuse", "spheres"])
def test_previews_match_oracle_range(host_scene, oracle_scene, camera, case):
    W, H, spp, depth, literal, flags = 64, 48, 10, 3, False, 0
    if case == "depth8":
        depth = 8
    if case == "literal":
        W, H, literal = 56, 40, True
    if case == "no_primary_reuse":
        flags = pysqt.SQT_F_NO_PRIMARY_REUSE
    ctx = pysqt.Context(0)
    ctx.upload(host_scene)
    osc = oracle_scene
    if case == "spheres":
        osc, spheres = _sphere_pair(host_scene)
        ctx.upload_spheres(spheres)
    p = pysqt.make_params(W, H, spp, max_depth=depth, seed=5, literal=literal, flags=flags)
    op = O.make_params(W, H, spp, max_depth=depth, seed=5, trig=1, literal=literal)
    rows, cols = p.rows, p.cols
    ctx.render_begin(camera, p)
    with pytest.raises(pysqt.SqtError):
        ctx.download(rows, cols)                 # nothing to show before the first chunk
    assert not ctx.download_moments(rows, cols).any()
    acc_ref = m2_ref = None
    k = 0
    for n in (1, 3, 4, 2):
        pr = ctx.render_advance(n)
        acc_ref, m2_ref = PR.render_range(osc, camera, op, k, k + n, acc_ref, m2_ref)
        k += n
        assert pr["samples_done"] == k and pr["samples_total"] == spp
        rgb8, acc = ctx.download(rows, cols)
        m2 = ctx.download_moments(rows, cols)
        assert np.array_equal(bits(acc), bits(acc_ref)), (case, k)
        assert np.array_equal(bits(m2), bits(m2_ref)), (case, k)
        assert np.array_equal(rgb8, O.tone_map(acc, k, trig=1)), (case, k)
    assert np.array_equal(rgb8, osc.render(camera, op)["rgb8"])
    ctx.close()


def test_noise_estimate(gpu_ctx, host_scene, camera):
    gpu_ctx.upload(host_scene)
    W, H, spp = 96, 64, 12
    p = pysqt.make_params(W, H, spp, max_depth=5, seed=1)
    seqs = []
    for rep in range(2):
        gpu_ctx.render_begin(camera, p)
        seq = []
        for n in (1, 1, 4, 6):
            pr = gpu_ctx.render_advance(n)
            k = pr["samples_done"]
            _, acc = gpu_ctx.download(H, W)
            m2 = gpu_ctx.download_moments(H, W)
            want = PR.noise(acc, m2, k)
            if k == 1:
                assert pr["noise"] == float("inf")
            else:
                assert 0 < pr["noise"] < float("inf")
                assert pr["noise"] == pytest.approx(want, rel=1e-9)
            seq.append(pr["noise"])
        assert gpu_ctx.render_advance(4)["noise"] == seq[-1]            # k = spp: nothing traced, same estimate
        seqs.append(np.array(seq, np.float64))
    assert np.array_equal(seqs[0].view(np.uint64), seqs[1].view(np.uint64))
    # a black frame: one grey, non-emissive triangle in front of the camera
    cam = np.array([0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0, 1], np.float32)
    v9 = np.array([[3, -5, -5, 3, 5, -5, 3, 0, 5]], np.float32)
    _, hs = build_pair(v9, np.zeros(1, np.int32), np.array([[0.5, 0.5, 0.5, 0.5, 0, 0, 0, 0]], np.float32))
    ctx = pysqt.Context(0)
    ctx.upload(hs)
    ctx.render_begin(cam, pysqt.make_params(32, 32, 4, max_depth=3))
    assert ctx.render_advance(1)["noise"] == float("inf")
    assert ctx.render_advance(2)["noise"] == 0.0
    ctx.close()


def test_work_counts_add_up(gpu_ctx, host_scene, camera):
    gpu_ctx.upload(host_scene)
    for flags in (0, pysqt.SQT_F_COUNT_WORK, pysqt.SQT_F_COUNT_WORK | pysqt.SQT_F_NO_PRIMARY_REUSE):
        p = pysqt.make_params(80, 60, 9, max_depth=6, seed=3, flags=flags)
        ref = gpu_ctx.render(camera, p)["stats"]
        tot = dict(gpu_ctx.render_begin(camera, p))
        for n in (2, 3, 4):
            st = gpu_ctx.render_advance(n)["stats"]
            for c in COUNTERS:
                tot[c] += st[c]
        for c in COUNTERS:
            assert tot[c] == ref[c], (flags, c)
        assert tot["samples"] == 80 * 60 * 9


def test_session_rules(gpu_ctx, host_scene, camera):
    gpu_ctx.upload(host_scene)
    L, h = gpu_ctx.L, gpu_ctx.h
    W, H, spp = 48, 32, 6
    p = pysqt.make_params(W, H, spp, max_depth=4, seed=2)
    pr = pysqt.Progress()
    buf = np.zeros((H, W, 3), np.float32)
    gpu_ctx.render(camera, p)
    assert L.sqt_render_advance(h, 1, None, None) == 1                       # no frame
    assert "no progressive frame" in gpu_ctx.last_error()
    assert L.sqt_download_moments(h, buf.ctypes.data) == 1
    for end in ("render", "tone_map", "upload", "begin_cast", "spheres"):
        gpu_ctx.render_begin(camera, p)
        gpu_ctx.render_advance(2)
        if end == "render":
            gpu_ctx.render(camera, p)
        elif end == "tone_map":
            gpu_ctx.tone_map(np.ones((4, 3), np.float32))
        elif end == "upload":
            gpu_ctx.upload(host_scene)
        elif end == "spheres":
            gpu_ctx.upload_spheres([])
        else:
            with pytest.raises(pysqt.SqtError):
                gpu_ctx.render_begin(camera, pysqt.make_params(W, H, spp, mode=1))
        assert L.sqt_render_advance(h, 1, None, None) == 1, end
        assert L.sqt_download_moments(h, buf.ctypes.data) == 1, end
    # n_samples < 1, the no-op at k = spp, unsupported modes
    ref = gpu_ctx.render(camera, p)
    gpu_ctx.render_begin(camera, p)
    assert L.sqt_render_advance(h, 0, None, None) == 1 and L.sqt_render_advance(h, -3, None, None) == 1
    gpu_ctx.render_advance(spp)
    st = gpu_ctx.render_advance(5)
    assert st["samples_done"] == spp and st["stats"]["kernel_launches"] == 0 and st["stats"]["rays_traced"] == 0
    assert L.sqt_render_advance(h, 1, C.byref(pr), None) == 0 and pr.samples_done == spp
    rgb8, acc = gpu_ctx.download(H, W)
    assert np.array_equal(bits(acc), bits(ref["accum"])) and np.array_equal(rgb8, ref["rgb8"])
    cam_struct = pysqt.camera_struct(camera)
    for bad in (pysqt.make_params(W, H, spp, mode=1), pysqt.make_params(W, H, spp, flags=pysqt.SQT_F_SPLIT_SAMPLES)):
        assert L.sqt_render_begin(h, C.byref(cam_struct), C.byref(bad), None) == 5      # SQT_E_UNSUPPORTED
    # sqt_intersect_batch between chunks leaves the frame alone
    gpu_ctx.render_begin(camera, p)
    gpu_ctx.render_advance(2)
    rng = np.random.default_rng(0)
    gpu_ctx.intersect_batch(rng.uniform(-1, 1, (5000, 3)), rng.normal(size=(5000, 3)))
    gpu_ctx.render_advance(spp)
    rgb8, acc = gpu_ctx.download(H, W)
    assert np.array_equal(bits(acc), bits(ref["accum"])) and np.array_equal(rgb8, ref["rgb8"])


def test_config2_full_size_in_chunks_of_64(gpu_ctx, host_scene, camera):
    """BASELINE config 2 (1920x1080, 1024 spp, 8 bounces) in 16 chunks of 64 spp: the one-shot frame's SHA-256."""
    gpu_ctx.upload(host_scene)
    p = pysqt.make_params(1920, 1080, 1024, max_depth=8, seed=0)
    ref = gpu_ctx.render(camera, p, want_accum=False)["rgb8"]
    outs = run_chunks(gpu_ctx, camera, p, [64] * 16)
    rgb8, _ = gpu_ctx.download(1080, 1920, want_accum=False)
    assert hashlib.sha256(rgb8.tobytes()).hexdigest() == hashlib.sha256(ref.tobytes()).hexdigest()
    noise = [o["noise"] for o in outs]
    assert all(0 < v < float("inf") for v in noise) and noise[-1] < noise[0]


def test_cli_progress_writes_the_same_png(tmp_path):
    exe = os.path.join(ROOT, "squigly-trace_b200", "squigly-trace")
    a, b = tmp_path / "plain.png", tmp_path / "progress.png"
    r1 = subprocess.run([exe, "-s", "12", "-d", "96,64", "-p", str(a)], cwd=ROOT, capture_output=True, text=True, timeout=300)
    r2 = subprocess.run([exe, "-s", "12", "-d", "96,64", "--progress=5", "-p", str(b)], cwd=ROOT, capture_output=True, text=True,
                        timeout=300)
    assert r1.returncode == 0 and r2.returncode == 0, r1.stderr + r2.stderr
    assert a.read_bytes() == b.read_bytes()
    lines = [l for l in r2.stdout.splitlines() if " samples  noise " in l]
    assert [l.split()[0] for l in lines] == ["5/12", "10/12", "12/12"]
