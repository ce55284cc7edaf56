"""A second restatement of the camera-sampling primary ray (include/sqt.h, sqt_set_lens), written from the header and not
from oracle/oracle.c: numpy binary32, one numpy operation per operation of the header, in the header's order.  Philox and
the sqt trig come from the oracle's exported orc_philox4x32_10 / orc_sqt_sincos, which tests/test_oracle.py pins on their
own.  Test infrastructure only."""
import ctypes as C

import numpy as np

from oracle import oracle as O

f32 = np.float32


def _words(streams, seed):
    """Philox4x32-10 on counter (s lo, s hi, 0, "SQTL"), key seed, for every stream s: (n, 4) uint32."""
    L = O.lib()
    out = np.zeros((len(streams), 4), np.uint32)
    ctr, key, w = (C.c_uint32 * 4)(), (C.c_uint32 * 2)(seed & 0xFFFFFFFF, seed >> 32), (C.c_uint32 * 4)()
    for i, s in enumerate(streams.tolist()):
        ctr[0], ctr[1], ctr[2], ctr[3] = s & 0xFFFFFFFF, s >> 32, 0, 0x4C545153
        L.orc_philox4x32_10(ctr, key, w)
        out[i] = w[:]
    return out


def _r01(w):
    return w.astype(f32) * f32(2.3283064365386963e-10)        # Lib.hs:183-188: Word32 -> Float / 2^32, exact scaling


def _sincos(th):
    L = O.lib()
    s, c = np.zeros(len(th), f32), np.zeros(len(th), f32)
    a, b = C.c_float(), C.c_float()
    for i, t in enumerate(th.tolist()):
        L.orc_sqt_sincos(C.c_float(t), C.byref(a), C.byref(b))
        s[i], c[i] = a.value, b.value
    return s, c


def lens_rays(params, cam12, pix, k, jitter, aperture, focus):
    """(org, dir) of sample k[i] of pixel pix[i] = y*cols + x; params: an oracle Params (rows, cols, xdiv, ydiv, seed_stride,
    spp, seed)."""
    pix = np.asarray(pix, np.int64)
    k = np.asarray(k, np.int64)
    y, x = pix // params.cols, pix % params.cols
    s = (np.uint64(params.spp) * (x.astype(np.uint64) + y.astype(np.uint64) * np.uint64(params.seed_stride))
         + k.astype(np.uint64))
    w = _words(s, int(params.seed))
    u = [_r01(w[:, i]) for i in range(4)]
    zero = np.zeros(len(pix), f32)
    jx = u[0] - f32(0.5) if jitter else zero
    jy = u[1] - f32(0.5) if jitter else zero
    fx = x.astype(f32) + jx
    fy = y.astype(f32) + jy
    ww, hh = f32(params.xdiv), f32(params.ydiv)
    xo = (fx - ww / f32(2)) / ww
    yo = (hh / f32(2) - fy) / hh
    cam = np.asarray(cam12, f32)
    R = cam[3:]
    org = np.tile(cam[:3], (len(pix), 1))
    d = np.stack([((f32(0) + f32(1) * R[i]) + xo * R[3 + i]) + yo * R[6 + i] for i in range(3)], axis=1)
    A = f32(aperture)
    if A != f32(0):
        r = A * np.sqrt(u[2])
        th = f32(6.2831855) * u[3]
        sn, cs = _sincos(th)
        a, b = r * cs, r * sn
        inv_f = f32(1) / f32(focus)
        off = np.stack([a * R[3 + i] + b * R[6 + i] for i in range(3)], axis=1)
        org = org + off
        d = d - off * inv_f
    return org.astype(f32), d.astype(f32)
