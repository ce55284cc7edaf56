"""ctypes bindings of the camera-sampling test helpers in tests/lens: the oracle's lens ray and lens render
(liboracle_lens.so, oracle/oracle.c plus the extension) and the host build of the kernels' lens frames (libemu_lens.so,
tests/emu plus the lens render).  A lens is (jitter, aperture, focus); params are oracle Params (oracle/oracle.py) for the
oracle and pysqt RenderParams for the host build.  Test infrastructure only."""
import ctypes as C
import os

import numpy as np

import pysqt
from oracle import oracle as O

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lens")
_LIBS = {}


def _lib(name):
    if name not in _LIBS:
        path = os.path.join(HERE, name)
        if not os.path.exists(path):
            import subprocess
            subprocess.check_call(["make", "-s", "-C", HERE])
        _LIBS[name] = C.CDLL(path)
    return _LIBS[name]


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _oracle():
    L = _lib("liboracle_lens.so")
    L.orc_make_lens_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_int64,
                                     C.c_void_p, C.c_void_p]
    L.orc_lens_range.restype = C.c_int
    L.orc_lens_range.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_int64, C.c_int64,
                                 C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    return L


def make_lens_rays(params, cam12, lens, pix, k):
    """(org, dir) of sample k[i] of pixel pix[i] = y*cols + x in a frame with `lens`."""
    cam12 = np.ascontiguousarray(cam12, np.float32)
    pix = np.ascontiguousarray(pix, np.int64)
    k = np.ascontiguousarray(k, np.int32)
    org = np.zeros((len(pix), 3), np.float32)
    dirs = np.zeros((len(pix), 3), np.float32)
    _oracle().orc_make_lens_rays(C.byref(params), _p(cam12), int(lens[0]), float(lens[1]), float(lens[2]), _p(pix), _p(k),
                                 len(pix), _p(org), _p(dirs))
    return org, dirs


def _range(scene, cam12, params, lens, pix0, pix1, k0, k1, accum, m2):
    cam12 = np.ascontiguousarray(cam12, np.float32)
    smp = np.zeros(1, np.uint64)
    if _oracle().orc_lens_range(scene.h, _p(cam12), C.byref(params), int(lens[0]), float(lens[1]), float(lens[2]), pix0, pix1,
                                k0, k1, _p(accum), _p(m2), _p(smp), os.cpu_count()):
        raise RuntimeError("orc_lens_range failed")
    return int(smp[0])


def render(scene, cam12, params, lens):
    """The one-shot lens frame: sums, RGB8 (sqt trig) and samples, like oracle.Scene.render."""
    k0, k1 = 0, params.spp
    if params.world > 1 and params.split_samples:
        k0, k1 = params.spp * params.rank // params.world, params.spp * (params.rank + 1) // params.world
    acc = np.zeros((params.rows, params.cols, 3), np.float32)
    n = _range(scene, cam12, params, lens, 0, params.rows * params.cols, k0, k1, acc, None)
    return dict(accum=acc, rgb8=O.tone_map(acc, params.spp, trig=1), samples=n)


def render_window(scene, cam12, params, lens, pix_lo, pix_hi):
    """Sums (pix_hi - pix_lo, 3) of the pixels [pix_lo, pix_hi) of the one-shot lens frame."""
    acc = np.zeros((pix_hi - pix_lo, 3), np.float32)
    _range(scene, cam12, params, lens, pix_lo, pix_hi, 0, params.spp, acc, None)
    return acc


def render_range(scene, cam12, params, lens, k_begin, k_end, accum=None, m2=None):
    """Continue the frame's sums and second moments over samples [k_begin, k_end), like progressive_ref.render_range."""
    shape = (params.rows, params.cols, 3)
    accum = np.zeros(shape, np.float32) if accum is None else accum.copy()
    m2 = np.zeros(shape, np.float32) if m2 is None else m2.copy()
    _range(scene, cam12, params, lens, 0, params.rows * params.cols, k_begin, k_end, accum, m2)
    return accum, m2


def prefix_window(scene, cam12, params, lens, pix0, pix1, k_end):
    """Sums and second moments (pix1 - pix0, 3) of pixels [pix0, pix1) after samples [0, k_end)."""
    acc = np.zeros((pix1 - pix0, 3), np.float32)
    m2 = np.zeros((pix1 - pix0, 3), np.float32)
    _range(scene, cam12, params, lens, pix0, pix1, 0, k_end, acc, m2)
    return acc, m2


class EmuLens:
    """Host build of the kernels' lens frames (the integrator source of k_paths_pool with LENS)."""

    def __init__(self, host_scene):
        L = _lib("libemu_lens.so")
        L.emu_upload.restype = C.c_void_p
        L.emu_upload.argtypes = [C.c_void_p]
        L.emu_error.restype = C.c_char_p
        L.emu_error.argtypes = [C.c_void_p]
        L.emu_free.argtypes = [C.c_void_p]
        L.emu_set_spheres.argtypes = [C.c_void_p, C.c_void_p, C.c_uint]
        L.emu_set_sbuf_budget.argtypes = [C.c_longlong]
        L.emu_render_lens.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.emu_lens_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p,
                                    C.c_void_p]
        self.L = L
        self.scene = host_scene
        d = host_scene.desc()
        self.h = L.emu_upload(C.byref(d))
        err = L.emu_error(self.h)
        if err:
            raise RuntimeError(err.decode())

    def __del__(self):
        try:
            self.L.emu_free(self.h)
        except Exception:
            pass

    def set_spheres(self, spheres):
        a = np.zeros(len(spheres), pysqt.SPHERE_DT)
        for i, (cx, cy, cz, r, m) in enumerate(spheres):
            a[i]["center"] = (cx, cy, cz); a[i]["radius"] = r; a[i]["material"] = int(m)
        self._spheres = a
        self.L.emu_set_spheres(self.h, _p(a) if len(a) else None, len(a))

    def set_sbuf_budget(self, nbytes):
        self.L.emu_set_sbuf_budget(nbytes)

    def render(self, cam12, params, lens, rank=0, world=1):
        acc = np.zeros((params.rows, params.cols, 3), np.float32)
        st = np.zeros(3, np.uint64)
        cam = pysqt.camera_struct(cam12)
        l = pysqt.Lens(int(lens[0]), lens[1], lens[2], 0)
        self.L.emu_render_lens(self.h, C.byref(cam), C.byref(params), rank, world, C.byref(l), _p(acc), _p(st))
        return dict(accum=acc, rays=int(st[0]), samples=int(st[1]), primary_reused=int(st[2]))


def emu_lens_rays(cam12, params, lens, pix, k):
    """lens_ray of the host build for the (pixel, sample) pairs."""
    L = _lib("libemu_lens.so")
    L.emu_lens_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p]
    cam = pysqt.camera_struct(cam12)
    l = pysqt.Lens(int(lens[0]), lens[1], lens[2], 0)
    pix = np.ascontiguousarray(pix, np.int64)
    k = np.ascontiguousarray(k, np.int32)
    org = np.zeros((len(pix), 3), np.float32)
    dirs = np.zeros((len(pix), 3), np.float32)
    L.emu_lens_rays(C.byref(cam), C.byref(params), C.byref(l), _p(pix), _p(k), len(pix), _p(org), _p(dirs))
    return org, dirs
