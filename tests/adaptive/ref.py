"""References for the adaptive frames of include/sqt.h (test infrastructure, built by `make -C tests/adaptive`):

  retire_emu      host build of retire_test (csrc/sqt_paths.cuh), the per-pixel test of the retire kernel
  retire_numpy    the header's retire formula evaluated with numpy in fp64
  noise           the noise estimate with per-pixel sample counts, in numpy fp64
  tone_map        the oracle's tone map of every pixel at its own sample count
  prefix_window   the oracle's range render over a window of pixels of a full-size frame (tests/adaptive/oracle_prefix.c)
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIBS = {}


def _so(name):
    if name not in _LIBS:
        so = os.path.join(_HERE, name)
        if not os.path.exists(so):
            subprocess.check_call(["make", "-s", "-C", _HERE])
        _LIBS[name] = C.CDLL(so)
    return _LIBS[name]


def _lib():
    L = _so("libemu_retire.so")
    L.emu_retire_test.argtypes = [C.c_longlong, C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_void_p]
    return L


def prefix_window(scene, cam12, params, pix0, pix1, k_end):
    """Sums and second moments (pix1 - pix0, 3) of pixels [pix0, pix1) after samples [0, k_end) of the frame `params`."""
    L = _so("liboracle_prefix.so")
    L.orc_render_range_window.restype = C.c_int
    L.orc_render_range_window.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_int,
                                          C.c_void_p, C.c_void_p]
    acc = np.zeros((pix1 - pix0, 3), np.float32)
    m2 = np.zeros((pix1 - pix0, 3), np.float32)
    cam12 = np.ascontiguousarray(cam12, np.float32)
    if L.orc_render_range_window(scene.h, cam12.ctypes.data, C.byref(params), pix0, pix1, 0, k_end, acc.ctypes.data, m2.ctypes.data):
        raise RuntimeError("orc_render_range_window failed")
    return acc, m2


def _f64(tol):
    """A tolerance as the backend sees it: the float of sqt_retire_params widened to double."""
    return float(np.float32(tol))


def retire_emu(s1, s2, n, rel_tol, abs_tol):
    s1 = np.ascontiguousarray(s1, np.float32).reshape(-1, 3)
    s2 = np.ascontiguousarray(s2, np.float32).reshape(-1, 3)
    out = np.zeros(len(s1), np.uint8)
    _lib().emu_retire_test(len(s1), s1.ctypes.data, s2.ctypes.data, n, _f64(rel_tol), _f64(abs_tol), out.ctypes.data)
    return out.astype(bool)


def retire_numpy(s1, s2, n, rel_tol, abs_tol):
    """Per pixel: mu_c = s1_c/n, v_c = max(0, (s2_c - s1_c*mu_c)/(n-1)), e2 = (v_r + v_g + v_b)/n, m = mu_r + mu_g + mu_b,
    t = max(rel_tol*m, abs_tol); retire iff e2 < t*t, never when a NaN turns up."""
    a = np.asarray(s1, np.float32).reshape(-1, 3).astype(np.float64)
    q = np.asarray(s2, np.float32).reshape(-1, 3).astype(np.float64)
    rel, ab = _f64(rel_tol), _f64(abs_tol)
    with np.errstate(all="ignore"):
        mu = a / float(n)
        vc = (q - a * mu) / (float(n) - 1.0)
        v = np.where(vc > 0.0, vc, 0.0)
        e2 = ((v[:, 0] + v[:, 1]) + v[:, 2]) / float(n)
        m = (mu[:, 0] + mu[:, 1]) + mu[:, 2]
        tr = rel * m
        t = np.where(tr > ab, tr, ab)
        nan = np.isnan(vc).any(axis=1) | np.isnan(m) | np.isnan(tr)
        return ~nan & (e2 < t * t)


def noise(s1, s2, counts):
    """The noise estimate of include/sqt.h with n = n_p in each pixel's terms (counts: rows x cols)."""
    a = np.asarray(s1, np.float64).reshape(-1, 3)
    q = np.asarray(s2, np.float64).reshape(-1, 3)
    n = np.asarray(counts, np.float64).reshape(-1, 1)
    mu = a / n
    var = np.maximum(0.0, (q - a * mu) / (n - 1))
    smu = mu.sum()
    if smu == 0.0:
        return 0.0
    return float(np.sqrt((var / n).sum() / a.size) / (smu / a.size))


def tone_map(accum, counts):
    """RGB8 of every pixel at its own sample count, with the oracle's tone map."""
    from oracle import oracle as O
    acc = np.ascontiguousarray(accum, np.float32)
    out = np.zeros(acc.shape, np.uint8)
    for n in np.unique(counts):
        sel = counts == n
        out[sel] = O.tone_map(acc[sel], int(n), trig=1)
    return out
