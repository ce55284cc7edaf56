"""Denoiser (include/sqt.h: sqt_denoise), the parts that need no GPU: the sqt_denoise_params layout, the host build of the
filter (csrc/sqt_denoise.cuh) against a numpy fp64 evaluation of the header's formula, its exact structural properties,
the retire test after its error terms moved into a shared function, and the CLI's --denoise argument."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import pysqt
from adaptive import ref as AR
from denoise import ref as DR

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_denoise_params_layout_matches_ctypes_and_integration_doc(tmp_path):
    """sqt_denoise_params: gcc offsetof, the ctypes mirror and the Storable instance of INTEGRATION.md give the same numbers."""
    src = tmp_path / "dn.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "sqt.h"\nint main(void){ printf("%zu %zu %zu %zu %zu %zu\\n", '
                   'sizeof(sqt_denoise_params), _Alignof(sqt_denoise_params), offsetof(sqt_denoise_params, levels), '
                   'offsetof(sqt_denoise_params, sigma_l), offsetof(sqt_denoise_params, sigma_z), '
                   'offsetof(sqt_denoise_params, reserved)); return 0; }\n')
    exe = tmp_path / "dn"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    D = pysqt.DenoiseParams
    assert got == [C.sizeof(D), C.alignment(D), D.levels.offset, D.sigma_l.offset, D.sigma_z.offset, D.reserved.offset]
    assert got == [16, 4, 0, 4, 8, 12]
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    inst = doc[doc.index("instance Storable SqtDenoiseParams"):]
    inst = inst[:inst.index("```")]
    m = re.search(r"sizeOf _ = (\d+) ; alignment _ = (\d+)", inst)
    assert m and [int(m.group(1)), int(m.group(2))] == got[:2]
    peek = [l for l in inst.splitlines() if l.strip().startswith("peek p")][0]
    assert [int(x) for x in re.findall(r"peekByteOff p (\d+)", peek)] == got[2:5]
    poke = [l for l in inst.splitlines() if l.strip().startswith("poke p")][0]
    assert [int(x) for x in re.findall(r"pokeByteOff p (\d+)", poke)] == got[2:]


def random_frame(seed, rows=37, cols=53):
    """A random filter input with material boundaries (blocks of 4 materials), invalid pixels, mirrors (material 3),
    image borders, isolated zero-variance pixels and one zero-variance block of one colour.  Returns cv, feat, sk."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:rows, 0:cols]
    mat = ((yy // 9) + 2 * (xx // 13)) % 4
    key = (mat + 1).astype(np.int32)
    key[mat == 3] *= -1                                                  # mirrors
    key[rng.random((rows, cols)) < 0.08] = 0                             # no primary hit
    c = (rng.exponential(0.5, (rows, cols, 3)) * (1 + 4 * (rng.random((rows, cols, 1)) < 0.05))).astype(np.float32)
    v = (rng.exponential(0.02, (rows, cols)) * (rng.random((rows, cols)) > 0.05)).astype(np.float32)
    blk = (slice(2, 8), slice(2, 10))                                    # zero variance, one colour
    c[blk] = np.float32(0.3)
    v[blk] = 0
    key[blk] = 1
    n = rng.normal(size=(rows, cols, 3)) * 0.3 + np.array([0.2, 0.3, 1.0]) * (1 + mat[..., None])
    n /= np.linalg.norm(n, axis=-1, keepdims=True)
    z = (2 + 0.05 * xx + 0.5 * mat + rng.random((rows, cols)) * 0.1).astype(np.float32)
    cv = np.concatenate([c, v[..., None]], axis=-1).astype(np.float32)
    feat = np.concatenate([n, z[..., None]], axis=-1).astype(np.float32)
    sk = np.stack([np.where(key != 0, 7, 0), key], axis=-1).astype(np.int32)
    return cv, feat, sk


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("sigma_l,sigma_z", [(4.0, 0.05), (1.0, 0.5), (16.0, 0.01)])
def test_host_build_matches_numpy_per_level(seed, sigma_l, sigma_z):
    """Each of 5 levels of the host build against the fp64 formula, both fed the host build's binary32 input of that level.

    Tolerance: every weight is a product of a few correctly rounded binary32 operations (relative error a few 2^-24 each),
    except that w_n = dot^128 amplifies the dot product's relative error (3 roundings) 128 times and r = (1 + x/8)^-8 that of
    x (about 5 roundings) at most 8 times: |dw/w| <= (128 * 3 + 8 * 5 + 10) * 2^-24 ~ 2.6e-5.  c' = sum w c / sum w is a convex
    combination, so its error is at most about 2 |dw/w| max|c_q| plus the rounding of 25 sums (25 * 2^-24 max|c_q|):
    < 6e-5 max|c_q|, bounded here by 1e-4 of the largest channel within the pixel's taps.  v' = sum w^2 v / (sum w)^2 gets
    twice the weight error: 2e-4 of the largest v within the taps."""
    cv, feat, sk = random_frame(seed)
    cur = cv
    for i in range(5):
        s = 1 << i
        got = DR.emu_level(cur, feat, sk, s, sigma_l, sigma_z)
        want = DR.level_numpy(cur, feat, sk[..., 1], s, sigma_l, sigma_z)
        cmax = _tap_max(np.abs(cur[..., :3]).max(-1), s)
        vmax = _tap_max(np.abs(cur[..., 3]), s)
        err_c = np.abs(got[..., :3].astype(np.float64) - want[..., :3]).max(-1)
        err_v = np.abs(got[..., 3].astype(np.float64) - want[..., 3])
        assert (err_c <= 1e-4 * cmax).all(), (i, float((err_c / cmax).max()))
        assert (err_v <= 2e-4 * vmax + 1e-30).all(), (i, float((err_v / np.maximum(vmax, 1e-30)).max()))
        cur = got
    assert not np.array_equal(bits(cur), bits(cv))
    assert np.array_equal(bits(cur), bits(DR.emu_levels(cv, feat, sk, 5, sigma_l, sigma_z)))


def _tap_max(a, s):
    m = np.zeros_like(a, dtype=np.float64)
    for dy in range(-2, 3):
        for dx in range(-2, 3):
            m = np.maximum(m, DR._shift(a.astype(np.float64), s * dy, s * dx, 0.0))
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            m = np.maximum(m, DR._shift(a.astype(np.float64), dy, dx, 0.0))
    return np.maximum(m, 1e-30)


def test_levels_zero_is_the_identity():
    cv, feat, sk = random_frame(4)
    assert np.array_equal(bits(DR.emu_levels(cv, feat, sk, 0, 4.0, 0.05)), bits(cv))


@pytest.mark.parametrize("levels", [1, 3, 5, 8])
def test_other_materials_and_invalid_pixels_change_no_output_bit(levels):
    cv, feat, sk = random_frame(5)
    key = sk[..., 1]
    base = DR.emu_levels(cv, feat, sk, levels, 4.0, 0.05)
    rng = np.random.default_rng(levels)
    for changed in (key == 2, key == 0, key == -4):
        cv2, feat2 = cv.copy(), feat.copy()
        cv2[changed] = rng.random((int(changed.sum()), 4)).astype(np.float32) * 3
        feat2[changed, 3] += 1.0
        out = DR.emu_levels(cv2, feat2, sk, levels, 4.0, 0.05)
        same = ~changed
        assert np.array_equal(bits(out[same]), bits(base[same])), levels
    # mirrors and invalid pixels pass through bit for bit; filtered pixels do change
    through = key <= 0
    assert np.array_equal(bits(base[through]), bits(cv[through]))
    assert (bits(base[key > 0]) != bits(cv[key > 0])).any()


def test_two_runs_agree_bit_for_bit():
    cv, feat, sk = random_frame(6)
    a = DR.emu_levels(cv, feat, sk, 5, 4.0, 0.05)
    b = DR.emu_levels(cv, feat, sk, 5, 4.0, 0.05)
    assert np.array_equal(bits(a), bits(b))


def test_denoise_input_is_the_preview_mean_and_the_retire_error_term():
    """c = s1 * (1.0f/(float)n) (float32 multiply) and v = (float)e2 with e2 of the retire test, per-pixel counts included."""
    rng = np.random.default_rng(7)
    P, k = 5000, 64
    s1 = (rng.exponential(1.0, (P, 3)) * k).astype(np.float32)
    s2 = (s1 * s1 / k * (1 + rng.random((P, 3)))).astype(np.float32)
    counts = np.where(rng.random(P) < 0.5, rng.integers(2, k, P), 0).astype(np.int32)
    cv = DR.emu_input(s1, s2, k, counts)
    n = np.where(counts > 0, counts, k)
    inv = (np.float32(1.0) / n.astype(np.float32)).astype(np.float32)
    assert np.array_equal(bits(cv[:, :3]), bits(s1 * inv[:, None]))
    a, q = s1.astype(np.float64), s2.astype(np.float64)
    mu = a / n[:, None]
    var = np.maximum((q - a * mu) / (n[:, None] - 1.0), 0.0)
    e2 = ((var[:, 0] + var[:, 1]) + var[:, 2]) / n
    assert np.array_equal(bits(cv[:, 3]), bits(e2.astype(np.float32)))


@pytest.mark.parametrize("n", [2, 17, 256])
def test_retire_test_after_the_shared_error_terms_matches_numpy(n):
    rng = np.random.default_rng(100 + n)
    P = 20000
    x = (rng.exponential(1.0, size=(n, P, 3)) * rng.random((1, P, 3))).astype(np.float32)
    s1 = x.sum(0, dtype=np.float32)
    s2 = (x * x).sum(0, dtype=np.float32)
    for rel, ab in [(0.05, 0.0), (0.2, 1e-3), (0.0, 0.02)]:
        assert np.array_equal(AR.retire_emu(s1, s2, n, rel, ab), AR.retire_numpy(s1, s2, n, rel, ab))


CLI = os.path.join(ROOT, "squigly-trace_b200", "squigly-trace")


@pytest.mark.parametrize("args", [
    ["--denoise"],                                        # without --progress
    ["--denoise=3"],
    ["--progress=4", "--denoise=abc"],
    ["--progress=4", "--denoise=9"],
    ["--progress=4", "--denoise="],
    ["--progress=4", "--denoise=-1"],
    ["--progress=4", "--denoise=10"],
    ["--progress=4", "--denoise=3x"],
])
def test_cli_rejects_malformed_denoise(args, tmp_path):
    r = subprocess.run([CLI, "-s", "8", "-d", "16,16", "-p", str(tmp_path / "x.png")] + args, cwd=ROOT, capture_output=True,
                       text=True, timeout=120)
    assert r.returncode == 1
    assert "--denoise" in r.stderr and "Rendering scene" not in r.stdout
    assert not (tmp_path / "x.png").exists()
