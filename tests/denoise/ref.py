"""References for the denoiser of include/sqt.h (test infrastructure, built by `make -C tests/denoise`):

  emu_input, emu_level(s) host build of csrc/sqt_denoise.cuh (the functions the denoise kernels run), in kernel order
  level_numpy             one level of the header's filter formula, evaluated with numpy in fp64
  keys                    the filter's per-pixel key (material + 1, negated for a mirror, 0 for no hit) from the surfaces
  denoise_host            the whole filter on downloaded sums, moments, counts and features, through the host build
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

H1 = {-2: 1 / 16, -1: 1 / 4, 0: 3 / 8, 1: 1 / 4, 2: 1 / 16}


def _lib():
    global _LIB
    if _LIB is None:
        so = os.path.join(_HERE, "libemu_denoise.so")
        if not os.path.exists(so):
            subprocess.check_call(["make", "-s", "-C", _HERE])
        L = C.CDLL(so)
        L.emu_denoise_input.argtypes = [C.c_longlong, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.emu_denoise_level.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_void_p]
        L.emu_denoise_levels.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_void_p]
        _LIB = L
    return _LIB


def emu_input(s1, s2, k, counts=None):
    """(c, v) per pixel, shape s1.shape[:-1] + (4,), float32."""
    shape = np.shape(s1)[:-1]
    s1 = np.ascontiguousarray(s1, np.float32)
    s2 = np.ascontiguousarray(s2, np.float32)
    cnt = None if counts is None else np.ascontiguousarray(counts, np.int32)
    out = np.zeros(shape + (4,), np.float32)
    _lib().emu_denoise_input(int(np.prod(shape)), s1.ctypes.data, s2.ctypes.data, k, None if cnt is None else cnt.ctypes.data,
                             out.ctypes.data)
    return out


def emu_levels(cv, feat, sk, levels, sigma_l, sigma_z):
    """levels of the filter on cv (rows, cols, 4) with feat (rows, cols, 4) and sk (rows, cols, 2) int32."""
    rows, cols = cv.shape[:2]
    cv = np.ascontiguousarray(cv, np.float32)
    feat = np.ascontiguousarray(feat, np.float32)
    sk = np.ascontiguousarray(sk, np.int32)
    out = np.zeros_like(cv)
    _lib().emu_denoise_levels(rows, cols, cv.ctypes.data, feat.ctypes.data, sk.ctypes.data, levels, sigma_l, sigma_z, out.ctypes.data)
    return out


def emu_level(cv, feat, sk, s, sigma_l, sigma_z):
    """One level of step s of the host build."""
    rows, cols = cv.shape[:2]
    cv = np.ascontiguousarray(cv, np.float32)
    feat = np.ascontiguousarray(feat, np.float32)
    sk = np.ascontiguousarray(sk, np.int32)
    out = np.zeros_like(cv)
    _lib().emu_denoise_level(rows, cols, cv.ctypes.data, feat.ctypes.data, sk.ctypes.data, s, sigma_l, sigma_z, out.ctypes.data)
    return out


def _shift(a, dy, dx, fill):
    """b[y, x] = a[y + dy, x + dx], `fill` outside the image."""
    rows, cols = a.shape[:2]
    b = np.full_like(a, fill)
    ys, yd = (slice(dy, rows), slice(0, rows - dy)) if dy >= 0 else (slice(0, rows + dy), slice(-dy, rows))
    xs, xd = (slice(dx, cols), slice(0, cols - dx)) if dx >= 0 else (slice(0, cols + dx), slice(-dx, cols))
    if ys.start < ys.stop and xs.start < xs.stop:
        b[yd, xd] = a[ys, xs]
    return b


def level_numpy(cv, feat, key, s, sigma_l, sigma_z):
    """One level (step s) of the header's formula in fp64: returns (c', v') as float64 (rows, cols, 4)."""
    cv = np.asarray(cv, np.float64)
    feat = np.asarray(feat, np.float64)
    key = np.asarray(key)
    c, v = cv[..., :3], cv[..., 3]
    lum = c.sum(-1)
    skv = np.zeros(key.shape)
    sk = np.zeros(key.shape)
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            m = _shift(key, dy, dx, 0) == key
            k = (2 if dy == 0 else 1) * (2 if dx == 0 else 1)
            skv += np.where(m, k * _shift(v, dy, dx, 0.0), 0.0)
            sk += np.where(m, k, 0)
    with np.errstate(all="ignore"):
        g = np.sqrt(skv / sk)
        dl = float(np.float32(sigma_l)) * g + float(np.float32(1e-6))
        dz = float(np.float32(sigma_z)) * s * feat[..., 3]
    sw = np.zeros(key.shape)
    sc = np.zeros(c.shape)
    sv = np.zeros(key.shape)
    for dy in range(-2, 3):
        for dx in range(-2, 3):
            kq = _shift(key, s * dy, s * dx, 0)
            m = kq == key
            cq = _shift(cv, s * dy, s * dx, 0.0)
            if dy == 0 and dx == 0:
                w = np.full(key.shape, 9 / 64)
            else:
                fq = _shift(feat, s * dy, s * dx, 0.0)
                with np.errstate(all="ignore"):
                    x = np.abs(lum - cq[..., :3].sum(-1)) / dl + np.abs(feat[..., 3] - fq[..., 3]) / dz
                    wn = np.maximum(0.0, (feat[..., :3] * fq[..., :3]).sum(-1)) ** 128
                    r = (1.0 + x / 8.0) ** -8
                w = H1[dy] * H1[dx] * wn * r
            w = np.where(m, w, 0.0)
            sw += w
            sc += w[..., None] * cq[..., :3]
            sv += w * w * cq[..., 3]
    out = cv.copy()
    f = key > 0
    with np.errstate(all="ignore"):
        out[..., :3] = np.where(f[..., None], sc / sw[..., None], c)
        out[..., 3] = np.where(f, sv / (sw * sw), v)
    return out


def keys(surface, tri_material, reflective):
    """key per pixel from the surfaces (tri_out numbering; triangles only) and the materials' `reflective`."""
    surface = np.asarray(surface)
    mat = np.where(surface >= 0, np.asarray(tri_material)[np.maximum(surface, 0)], 0)
    key = (mat + 1).astype(np.int32)
    key = np.where(np.asarray(reflective)[mat] >= 1.0, -key, key)
    return np.where(surface >= 0, key, 0).astype(np.int32)


def denoise_host(s1, s2, counts, k, feats, tri_material, reflective, levels, sigma_l, sigma_z):
    """The denoised mean (rows, cols, 3) of include/sqt.h from downloaded data, through the host build."""
    surface = feats["surface"]
    cv = emu_input(s1, s2, k, counts)
    feat = np.concatenate([feats["normal"], feats["depth"][..., None]], axis=-1).astype(np.float32)
    sk = np.stack([surface + 1, keys(surface, tri_material, reflective)], axis=-1).astype(np.int32)
    return emu_levels(cv, feat, sk, levels, sigma_l, sigma_z)[..., :3]
