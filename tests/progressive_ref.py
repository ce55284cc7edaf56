"""References for the progressive frames of include/sqt.h (test infrastructure, built by `make -C tests/progressive`):

  render_range   the oracle's range render: continues per-pixel sums and second moments of the spp frame over samples
                 [k_begin, k_end) (tests/progressive/oracle_range.c, compiled from oracle/oracle.c)
  accumulate_m2  host build of accumulate_m2_slot (csrc/sqt_paths.cuh), the per-slot function of k_accumulate_m2
  noise          the noise estimate's definition, evaluated with numpy in fp64
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "progressive")
_LIBS = {}


def _lib(name):
    if name not in _LIBS:
        so = os.path.join(_HERE, name)
        if not os.path.exists(so):
            subprocess.check_call(["make", "-s", "-C", _HERE])
        _LIBS[name] = C.CDLL(so)
    return _LIBS[name]


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def render_range(scene, cam12, params, k_begin, k_end, accum=None, m2=None, nthreads=None):
    """Continue (accum, m2) -- float32 (rows, cols, 3), zero when None -- over samples [k_begin, k_end); returns both."""
    L = _lib("liboracle_range.so")
    L.orc_render_range.restype = C.c_int
    L.orc_render_range.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    shape = (params.rows, params.cols, 3)
    accum = np.zeros(shape, np.float32) if accum is None else np.ascontiguousarray(accum, np.float32).copy()
    m2 = np.zeros(shape, np.float32) if m2 is None else np.ascontiguousarray(m2, np.float32).copy()
    cam12 = np.ascontiguousarray(cam12, np.float32)
    rc = L.orc_render_range(scene.h, _p(cam12), C.byref(params), k_begin, k_end, _p(accum), _p(m2), nthreads or os.cpu_count())
    if rc:
        raise RuntimeError("orc_render_range failed")
    return accum, m2


def accumulate_m2(rows, cols, spp, sbuf, k0, k1, accum, m2):
    """One round of accumulate_m2_slot over every pixel; sbuf is (k1 - k0, rows*cols, 3) float32.  Updates in place."""
    L = _lib("libemu_m2.so")
    L.emu_accumulate_m2.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    sbuf = np.ascontiguousarray(sbuf, np.float32)
    assert accum.dtype == np.float32 and m2.dtype == np.float32 and accum.flags.c_contiguous and m2.flags.c_contiguous
    L.emu_accumulate_m2(rows, cols, spp, _p(sbuf), k0, k1, _p(accum), _p(m2))


def noise(s1, s2, n):
    """sqrt(sum(e2)/N) / (sum(mu)/N) with mu = s1/n, var = max(0, (s2 - s1*mu)/(n-1)), e2 = var/n, in fp64."""
    if n < 2:
        return float("inf")
    a = np.asarray(s1, np.float64).ravel()
    q = np.asarray(s2, np.float64).ravel()
    mu = a / n
    var = np.maximum(0.0, (q - a * mu) / (n - 1))
    smu = mu.sum()
    if smu == 0.0:
        return 0.0
    return float(np.sqrt((var / n).sum() / a.size) / (smu / a.size))
