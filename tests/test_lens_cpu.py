"""Camera sampling (include/sqt.h, sqt_set_lens) on the CPU: the oracle's lens ray against a second, independent restatement
(tests/lens_ref.py) bit for bit; the host build of the kernels' integrator (tests/emu) against the oracle's accumulation
buffer on lens frames; the distribution of the jitter and of the lens offsets; the ABI; the CLI's argument checks."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy import stats

import pysqt
from oracle import oracle as O
from common import _p, bits, default_camera
import lens_oracle as LO
import lens_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rotated_camera():
    R = np.zeros(9, np.float32)
    O.lib().orc_rot_matrix_rads(C.c_float(0.3), C.c_float(-0.7), C.c_float(1.1), _p(R))
    return np.concatenate([np.float32([0.4, -1.3, 2.2]), R]).astype(np.float32)


def _pairs(p, n, seed):
    rng = np.random.default_rng(seed)
    return rng.integers(0, p.rows * p.cols, n), rng.integers(0, p.spp, n).astype(np.int32)


@pytest.mark.parametrize("literal", [False, True])
@pytest.mark.parametrize("rotated", [False, True])
def test_lens_rays_two_restatements_agree_bit_for_bit(literal, rotated):
    """18 lens settings x 1500 (pixel, sample) pairs per convention and camera: > 100 k pairs over the four cases."""
    cam = rotated_camera() if rotated else default_camera()
    for jitter in (0, 1):
        for aperture in (0.0, 1e-3, 0.2):
            for focus in (0.37, 2.0, 11.5):
                p = O.make_params(97, 61, 1000, seed=0x1234567890AB, literal=literal)
                pix, k = _pairs(p, 1500, 7 * jitter + int(aperture * 1000) + int(focus))
                org, dirs = LO.make_lens_rays(p, cam, (jitter, aperture, focus), pix, k)
                rorg, rdir = lens_ref.lens_rays(p, cam, pix, k, jitter, aperture, focus)
                assert np.array_equal(bits(org), bits(rorg)), (jitter, aperture, focus)
                assert np.array_equal(bits(dirs), bits(rdir)), (jitter, aperture, focus)


@pytest.mark.parametrize("literal", [False, True])
def test_pinhole_lens_rays_are_make_rays(literal):
    cam = default_camera()
    p = O.make_params(97, 61, 7, seed=3, literal=literal)
    org0, dir0 = O.make_rays(p, cam)
    pix = np.repeat(np.arange(p.rows * p.cols), 2)
    k = np.tile(np.int32([0, 6]), p.rows * p.cols)
    org, dirs = LO.make_lens_rays(p, cam, (0, 0.0, 1.5), pix, k)
    assert np.array_equal(bits(org), bits(np.repeat(org0, 2, axis=0)))
    assert np.array_equal(bits(dirs), bits(np.repeat(dir0, 2, axis=0)))


SPHERES = [(0.8, 0.5, -1.2, 0.6, 5), (-0.9, 1.0, 0.3, 0.45, 1), (0.0, -0.5, 1.2, 0.3, 3)]


@pytest.mark.parametrize("case", ["jitter", "lens", "both", "depth8", "spheres", "literal", "rank0", "rank1", "small_sbuf"])
def test_emu_lens_render_matches_oracle(host_scene, oracle_scene, camera, case):
    W, H, spp, depth, literal, rank, world = 40, 28, 6, 3, False, 0, 1
    lens = {"jitter": (1, 0.0, 1.0), "lens": (0, 0.08, 2.5)}.get(case, (1, 0.08, 2.5))
    if case == "depth8":
        depth = 8
    if case == "literal":
        literal = True
    if case in ("rank0", "rank1"):
        rank, world = int(case[-1]), 2
    emu = LO.EmuLens(host_scene)
    emu.set_sbuf_budget(W * H * 12 * 2 if case == "small_sbuf" else 1 << 20)   # 2 samples per round: 3 rounds
    osc = oracle_scene
    if case == "spheres":
        emu.set_spheres(SPHERES)
        osc = O.Scene.load(os.path.join(ROOT, "data", "scene.obj"), os.path.join(ROOT, "data"))
        osc.make_bih()
        osc.set_spheres(SPHERES)
    got = emu.render(camera, pysqt.make_params(W, H, spp, max_depth=depth, seed=11, literal=literal), lens, rank, world)
    ref = LO.render(osc, camera, O.make_params(W, H, spp, max_depth=depth, seed=11, trig=1, literal=literal, rank=rank, world=world),
                    lens)
    assert np.array_equal(bits(got["accum"]), bits(ref["accum"])), case
    assert got["samples"] == ref["samples"] and got["primary_reused"] == 0


def _emu_rays(lens, w, h, spp, pix, k):
    identity = np.float32([0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0, 1])
    return LO.emu_lens_rays(identity, pysqt.make_params(w, h, spp, seed=21), lens, pix, k)


def test_jitter_is_uniform_on_the_pixel():
    """Identity camera: d = (1, xo, yo), so the sample point of (x, y) is recovered from the direction; chi-square on 16x16."""
    W, H, spp = 64, 48, 32
    pix = np.repeat(np.arange(W * H), spp)
    k = np.tile(np.arange(spp), W * H)
    _, d = _emu_rays((1, 0.0, 1.0), W, H, spp, pix, k)
    x, y = pix % W, pix // W
    jx = d[:, 1].astype(np.float64) * W + W / 2 - x
    jy = H / 2 - d[:, 2].astype(np.float64) * H - y
    assert jx.min() >= -0.5 - 1e-4 and jx.max() <= 0.5 + 1e-4 and jy.min() >= -0.5 - 1e-4 and jy.max() <= 0.5 + 1e-4
    bx = np.clip(((jx + 0.5) * 16).astype(int), 0, 15)
    by = np.clip(((jy + 0.5) * 16).astype(int), 0, 15)
    counts = np.bincount(bx * 16 + by, minlength=256)
    assert stats.chisquare(counts).pvalue > 1e-3
    assert abs(np.corrcoef(jx, jy)[0, 1]) < 0.02


def test_lens_offsets_are_uniform_on_the_disk():
    """Identity camera, A = 0.5: the origin is the offset (0, a, b); r^2/A^2 and the angle are uniform (Kolmogorov-Smirnov),
    and every lens sample of a pixel meets the pinhole ray at t = f."""
    W, H, spp, A, f = 40, 30, 40, 0.5, 2.0
    pix = np.repeat(np.arange(W * H), spp)
    k = np.tile(np.arange(spp), W * H)
    o, d = _emu_rays((0, A, f), W, H, spp, pix, k)
    assert np.all(o[:, 0] == 0.0)
    r2 = (o[:, 1].astype(np.float64) ** 2 + o[:, 2].astype(np.float64) ** 2) / A ** 2
    ang = (np.arctan2(o[:, 2], o[:, 1]).astype(np.float64) / (2 * np.pi)) % 1.0
    assert r2.max() <= 1.0 + 1e-6
    assert stats.kstest(r2, "uniform").pvalue > 1e-3
    assert stats.kstest(ang, "uniform").pvalue > 1e-3
    _, d0 = _emu_rays((0, 0.0, f), W, H, spp, pix, k)
    focus_pt = o.astype(np.float64) + f * d.astype(np.float64)
    assert np.abs(focus_pt - f * d0.astype(np.float64)).max() < 1e-6


def test_lens_struct_and_symbol():
    assert C.sizeof(pysqt.Lens) == 16
    assert [pysqt.Lens.jitter.offset, pysqt.Lens.aperture_radius.offset, pysqt.Lens.focus_distance.offset,
            pysqt.Lens.reserved.offset] == [0, 4, 8, 12]
    lib = pysqt.b200()
    assert hasattr(lib, "sqt_set_lens") and "sqt_set_lens" in pysqt.ABI_SYMBOLS
    assert lib.sqt_abi_version() == 1


def test_lens_layout_in_c_and_integration_doc(tmp_path):
    src = tmp_path / "lens.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "sqt.h"\nint main(void){ printf("%zu %zu %zu %zu %zu\\n",'
                   ' sizeof(sqt_lens), offsetof(sqt_lens, jitter), offsetof(sqt_lens, aperture_radius),'
                   ' offsetof(sqt_lens, focus_distance), offsetof(sqt_lens, reserved)); return 0; }\n')
    exe = tmp_path / "lens"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    assert subprocess.check_output([str(exe)], text=True).split() == ["16", "0", "4", "8", "12"]
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    assert "sqt_set_lens" in doc and "instance Storable SqtLens" in doc
    for off in ("ByteOff p 0 ", "ByteOff p 4 ", "ByteOff p 8 ", "pokeByteOff p 12 "):
        assert off in doc.split("instance Storable SqtLens")[1].split("```")[0]


@pytest.mark.parametrize("args,msg", [
    (["--lens=0.1"], "Could not parse --lens"),
    (["--lens=0.1,0"], "Could not parse --lens"),
    (["--lens=-1,2"], "Could not parse --lens"),
    (["--lens=a,2"], "Could not parse --lens"),
    (["--lens=0.1,inf"], "Could not parse --lens"),
    (["--lens=0.1,2,3"], "Could not parse --lens"),
    (["--progress=4", "--aa", "--denoise"], "--denoise cannot be combined"),
    (["--progress=4", "--lens=0.1,2", "--denoise=3"], "--denoise cannot be combined"),
    (["--aa", "--cast"], "--cast cannot be combined"),
])
def test_cli_rejects_bad_lens_arguments(args, msg):
    exe = os.path.join(ROOT, "squigly-trace_b200", "squigly-trace")
    r = subprocess.run([exe, "-c", "/nonexistent"] + args, capture_output=True, text=True, timeout=60)
    assert r.returncode == 1 and msg in r.stderr, r.stderr


def test_cli_accepts_lens_arguments():
    """Well-formed --aa / --lens get past argument parsing (the run then stops at the missing camera file)."""
    exe = os.path.join(ROOT, "squigly-trace_b200", "squigly-trace")
    for args in (["--aa"], ["--lens=0.05,2.5"], ["--lens=0,1", "--aa", "--progress=8", "--adaptive=0.1"]):
        r = subprocess.run([exe, "-c", "/nonexistent/camera"] + args, capture_output=True, text=True, timeout=60)
        assert r.returncode == 1 and "lens" not in r.stderr and "Unknown flag" not in r.stderr, r.stderr
