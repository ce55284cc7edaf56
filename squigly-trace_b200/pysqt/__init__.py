"""pysqt -- ctypes binding of the squigly-trace B200 backend for the test and bench harness.

Two libraries, both built in-tree by `make -C squigly-trace_b200` (or __graft_entry__.build()):
  libsqt_b200.so  the product: CUDA kernels + the C ABI of include/sqt.h
  libsqt_host.so  the host mirror of Obj.hs / BIH.hs / Lib.hs `render` (C++), reached through capi.cpp

PyTorch is not involved in the data path; there is no CPU fallback -- every compute entry point raises
if the CUDA library or a B200 is missing.
"""
import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROOT = os.path.dirname(_PKG)
LIB_B200 = os.environ.get("SQT_LIB_B200") or os.path.join(_PKG, "libsqt_b200.so")      # override: A/B builds of the kernels (development)
LIB_HOST = os.path.join(_PKG, "libsqt_host.so")

SQT_F_COUNT_WORK = 1
SQT_F_SPLIT_SAMPLES = 2
SQT_F_NO_PRIMARY_REUSE = 4
SQT_F_NO_EARLY_TERMINATION = 8
SQT_COMM_ID_BYTES = 128

# every symbol include/sqt.h declares
ABI_SYMBOLS = [
    "sqt_abi_version", "sqt_create", "sqt_destroy", "sqt_last_error", "sqt_upload_scene", "sqt_intersect_batch",
    "sqt_render", "sqt_render_resident", "sqt_download_image", "sqt_tone_map", "sqt_comm_unique_id", "sqt_comm_init",
    "sqt_comm_init_all", "sqt_render_group", "sqt_measure_fp32_peak", "sqt_measure_l2_bandwidth", "sqt_device_info", "sqt_set_option", "sqt_upload_spheres",
    "sqt_upload_scene_group", "sqt_last_upload", "sqt_render_begin", "sqt_render_advance", "sqt_render_begin_group",
    "sqt_render_advance_group", "sqt_download_moments", "sqt_render_retire", "sqt_render_retire_group",
    "sqt_download_sample_counts", "sqt_denoise", "sqt_denoise_group", "sqt_download_features", "sqt_set_lens",
]


class SqtError(RuntimeError):
    pass


class Node(C.Structure):
    _fields_ = [("lmax", C.c_float), ("rmin", C.c_float), ("a", C.c_uint32), ("b", C.c_uint32)]


class Tri(C.Structure):
    _fields_ = [("v0", C.c_float * 3), ("e1", C.c_float * 3), ("e2", C.c_float * 3), ("material", C.c_uint32),
                ("orig_index", C.c_uint32), ("pad", C.c_uint32)]


class Material(C.Structure):
    _fields_ = [("reflective", C.c_float), ("surf_color", C.c_float * 3), ("emissive", C.c_float), ("emit_color", C.c_float * 3)]


class SceneDesc(C.Structure):
    _fields_ = [("root_bounds", C.c_float * 6), ("nodes", C.c_void_p), ("n_nodes", C.c_uint32), ("tris", C.c_void_p),
                ("n_tris", C.c_uint32), ("mats", C.c_void_p), ("n_mats", C.c_uint32)]


class Camera(C.Structure):
    _fields_ = [("position", C.c_float * 3), ("rotation", C.c_float * 9)]


class RenderParams(C.Structure):
    _fields_ = [("rows", C.c_int32), ("cols", C.c_int32), ("xdiv", C.c_int32), ("ydiv", C.c_int32), ("seed_stride", C.c_int32),
                ("spp", C.c_int32), ("max_depth", C.c_int32), ("mode", C.c_int32), ("seed", C.c_uint64), ("flags", C.c_uint32),
                ("reserved", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [("device_ms", C.c_double), ("primary_ms", C.c_double), ("paths_ms", C.c_double), ("tonemap_ms", C.c_double),
                ("reduce_ms", C.c_double), ("h2d_ms", C.c_double), ("d2h_ms", C.c_double), ("rays_traced", C.c_uint64),
                ("rays_reference", C.c_uint64), ("samples", C.c_uint64), ("branch_visits", C.c_uint64),
                ("child_box_tests", C.c_uint64), ("tri_tests", C.c_uint64), ("leaves_culled", C.c_uint64), ("mt_pass_a", C.c_uint64), ("mt_pass_u", C.c_uint64),
                ("mt_pass_v", C.c_uint64), ("mt_accept", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("kernel_launches", C.c_uint32), ("reserved", C.c_uint32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}


class Progress(C.Structure):
    _fields_ = [("samples_done", C.c_int32), ("samples_total", C.c_int32), ("noise", C.c_double)]


class RetireParams(C.Structure):
    _fields_ = [("rel_tol", C.c_float), ("abs_tol", C.c_float), ("min_samples", C.c_int32), ("reserved", C.c_uint32)]


MIN_SAMPLES = 16       # default min_samples of render_retire and of the CLI's --adaptive


class DenoiseParams(C.Structure):
    _fields_ = [("levels", C.c_int32), ("sigma_l", C.c_float), ("sigma_z", C.c_float), ("reserved", C.c_uint32)]


DENOISE_LEVELS, DENOISE_SIGMA_L, DENOISE_SIGMA_Z = 5, 4.0, 0.05     # defaults of denoise and of the CLI's --denoise


class Lens(C.Structure):
    _fields_ = [("jitter", C.c_uint32), ("aperture_radius", C.c_float), ("focus_distance", C.c_float), ("reserved", C.c_uint32)]


NODE_DT = np.dtype([("lmax", "<f4"), ("rmin", "<f4"), ("a", "<u4"), ("b", "<u4")])
TRI_DT = np.dtype([("v0", "<f4", 3), ("e1", "<f4", 3), ("e2", "<f4", 3), ("material", "<u4"), ("orig_index", "<u4"), ("pad", "<u4")])
SPHERE_DT = np.dtype([("center", "<f4", 3), ("radius", "<f4"), ("material", "<u4"), ("pad", "<u4", 3)])
MAT_DT = np.dtype([("reflective", "<f4"), ("surf_color", "<f4", 3), ("emissive", "<f4"), ("emit_color", "<f4", 3)])
assert NODE_DT.itemsize == 16 and TRI_DT.itemsize == 48 and MAT_DT.itemsize == 32

_b200 = None
_host = None


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def b200():
    """The product library.  Fails loudly when it has not been built."""
    global _b200
    if _b200 is None:
        if not os.path.exists(LIB_B200):
            raise SqtError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)" % LIB_B200)
        L = C.CDLL(LIB_B200, mode=C.RTLD_GLOBAL)
        L.sqt_abi_version.restype = C.c_int
        L.sqt_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.sqt_destroy.argtypes = [C.c_void_p]
        L.sqt_last_error.restype = C.c_char_p
        L.sqt_last_error.argtypes = [C.c_void_p]
        L.sqt_upload_scene.argtypes = [C.c_void_p, C.c_void_p]
        L.sqt_intersect_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sqt_render.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sqt_render_resident.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sqt_download_image.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.sqt_tone_map.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
        L.sqt_comm_unique_id.argtypes = [C.c_void_p]
        L.sqt_comm_init.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.sqt_comm_init_all.argtypes = [C.c_void_p, C.c_int]
        L.sqt_render_group.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sqt_measure_fp32_peak.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
        L.sqt_measure_l2_bandwidth.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
        L.sqt_set_option.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.sqt_upload_spheres.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
        L.sqt_upload_scene_group.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.sqt_last_upload.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.sqt_render_begin.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sqt_render_advance.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
        L.sqt_render_begin_group.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sqt_render_advance_group.argtypes = [C.c_void_p, C.c_int, C.c_int32, C.c_void_p, C.c_void_p]
        L.sqt_download_moments.argtypes = [C.c_void_p, C.c_void_p]
        L.sqt_render_retire.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.sqt_render_retire_group.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.sqt_download_sample_counts.argtypes = [C.c_void_p, C.c_void_p]
        L.sqt_denoise.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sqt_denoise_group.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sqt_download_features.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sqt_set_lens.argtypes = [C.c_void_p, C.c_void_p]
        L.sqt_device_info.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_char_p]
        for name in ABI_SYMBOLS:
            if name not in ("sqt_last_error",):
                getattr(L, name).restype = C.c_int
        _b200 = L
    return _b200


def host():
    global _host
    if _host is None:
        b200()      # libsqt_host.so links against libsqt_b200.so
        if not os.path.exists(LIB_HOST):
            raise SqtError("%s is missing: run __graft_entry__.build()" % LIB_HOST)
        L = C.CDLL(LIB_HOST)
        L.sqth_last_error.restype = C.c_char_p
        L.sqth_load.restype = C.c_void_p
        L.sqth_load.argtypes = [C.c_char_p, C.c_char_p]
        L.sqth_from_arrays.restype = C.c_void_p
        L.sqth_from_arrays.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        L.sqth_free.argtypes = [C.c_void_p]
        for f in ("sqth_n_tris", "sqth_n_nodes", "sqth_n_mats", "sqth_height", "sqth_num_leaves", "sqth_longest_leaf"):
            getattr(L, f).restype = C.c_int
            getattr(L, f).argtypes = [C.c_void_p]
        L.sqth_get_tris.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.sqth_get_flat.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sqth_desc.restype = C.c_void_p
        L.sqth_desc.argtypes = [C.c_void_p]
        L.sqth_load_camera.restype = C.c_int
        L.sqth_load_camera.argtypes = [C.c_char_p, C.c_void_p]
        L.sqth_params.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_void_p]
        L.sqth_write_png.restype = C.c_int
        L.sqth_write_png.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_int]
        _host = L
    return _host


class HostScene:
    """trisFromObj + makeBIH + flatten, done by the C++ host library."""

    def __init__(self, handle):
        if not handle:
            raise SqtError(host().sqth_last_error().decode())
        self.h = handle
        H = host()
        self.n_tris, self.n_nodes, self.n_mats = H.sqth_n_tris(handle), H.sqth_n_nodes(handle), H.sqth_n_mats(handle)
        self.root = np.zeros(6, np.float32)
        self.nodes = np.zeros(self.n_nodes, NODE_DT)
        self.tris = np.zeros(self.n_tris, TRI_DT)
        self.mats = np.zeros(self.n_mats, MAT_DT)
        H.sqth_get_flat(handle, _p(self.root), _p(self.nodes), _p(self.tris), _p(self.mats))

    @classmethod
    def load(cls, obj_path, data_dir):
        if not data_dir.endswith("/"):
            data_dir += "/"
        return cls(host().sqth_load(obj_path.encode(), data_dir.encode()))

    @classmethod
    def from_arrays(cls, v9, mat_idx, mats8):
        v9 = np.ascontiguousarray(v9, np.float32).reshape(-1, 9)
        mat_idx = np.ascontiguousarray(mat_idx, np.int32)
        mats8 = np.ascontiguousarray(mats8, np.float32).reshape(-1, 8)
        return cls(host().sqth_from_arrays(_p(v9), _p(mat_idx), len(v9), _p(mats8), len(mats8)))

    def __del__(self):
        try:
            host().sqth_free(self.h)
        except Exception:
            pass

    def stats(self):
        H = host()
        return dict(nodes=self.n_nodes, height=H.sqth_height(self.h), longest_leaf=H.sqth_longest_leaf(self.h),
                    leaves=H.sqth_num_leaves(self.h))

    def parsed_tris(self):
        v9 = np.zeros((self.n_tris, 9), np.float32)
        mi = np.zeros(self.n_tris, np.int32)
        host().sqth_get_tris(self.h, _p(v9), _p(mi))
        return v9, mi

    def desc(self):
        d = SceneDesc()
        for i in range(6):
            d.root_bounds[i] = float(self.root[i])
        d.nodes, d.n_nodes = self.nodes.ctypes.data, self.n_nodes
        d.tris, d.n_tris = self.tris.ctypes.data, self.n_tris
        d.mats, d.n_mats = self.mats.ctypes.data, self.n_mats
        return d


def load_camera(path):
    cam = np.zeros(12, np.float32)
    if host().sqth_load_camera(path.encode(), _p(cam)):
        raise SqtError(host().sqth_last_error().decode())
    return cam


def make_params(width, height, spp, max_depth=3, seed=0, mode=0, literal=False, flags=0):
    p = RenderParams()
    host().sqth_params(width, height, spp, max_depth, mode, 0 if literal else 1, seed, C.byref(p))
    p.flags = flags
    return p


def camera_struct(cam12):
    c = Camera()
    for i in range(3):
        c.position[i] = float(cam12[i])
    for i in range(9):
        c.rotation[i] = float(cam12[3 + i])
    return c


def _advance(call):
    """render_advance of a Context or a Group: call(progress, stats) makes the C call and checks it."""
    pr, st = Progress(), Stats()
    call(C.byref(pr), C.byref(st))
    return dict(samples_done=pr.samples_done, samples_total=pr.samples_total, noise=pr.noise, stats=st.as_dict())


def _denoise(shape, levels, sigma_l, sigma_z, call):
    """denoise of a Context or a Group: call(params, rgb8, mean, stats) makes the C call and checks it."""
    rows, cols = shape
    dp, st = DenoiseParams(levels, sigma_l, sigma_z, 0), Stats()
    rgb8 = np.zeros((rows, cols, 3), np.uint8)
    mean = np.zeros((rows, cols, 3), np.float32)
    call(C.byref(dp), _p(rgb8), _p(mean), C.byref(st))
    return dict(rgb8=rgb8, mean=mean, stats=st.as_dict())


class Context:
    """One sqt_ctx (one B200)."""

    def __init__(self, device=0):
        L = b200()
        h = C.c_void_p()
        rc = L.sqt_create(device, C.byref(h))
        if rc:
            raise SqtError("sqt_create failed (%d): %s" % (rc, L.sqt_last_error(None).decode()))
        self.h = h
        self.L = L
        self._shape = (0, 0)        # rows, cols of the progressive frame begun last

    def close(self):
        if self.h:
            self.L.sqt_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc, what):
        if rc:
            raise SqtError("%s failed (%d): %s" % (what, rc, self.L.sqt_last_error(self.h).decode()))

    def info(self):
        sm, ma, mi = C.c_int(), C.c_int(), C.c_int()
        name = C.create_string_buffer(128)
        self._ck(self.L.sqt_device_info(self.h, C.byref(sm), C.byref(ma), C.byref(mi), name), "sqt_device_info")
        return dict(sm_count=sm.value, cc=(ma.value, mi.value), name=name.value.decode())

    def upload(self, scene):
        d = scene.desc() if hasattr(scene, "desc") else scene
        self._keep = scene
        self._ck(self.L.sqt_upload_scene(self.h, C.byref(d)), "sqt_upload_scene")

    def last_upload(self):
        b, w, h = C.c_uint64(), C.c_double(), C.c_double()
        self._ck(self.L.sqt_last_upload(self.h, C.byref(b), C.byref(w), C.byref(h)), "sqt_last_upload")
        return dict(h2d_bytes=b.value, wall_ms=w.value, host_layout_ms=h.value)

    def upload_desc_raw(self, desc):
        return self.L.sqt_upload_scene(self.h, C.byref(desc))

    def last_error(self):
        return self.L.sqt_last_error(self.h).decode()

    def intersect_batch(self, org, dir, want_stats=False):
        org = np.ascontiguousarray(org, np.float32).reshape(-1, 3)
        dir = np.ascontiguousarray(dir, np.float32).reshape(-1, 3)
        n = len(org)
        tri = np.full(n, -2, np.int32)
        dist = np.zeros(n, np.float32)
        point = np.zeros((n, 3), np.float32)
        st = Stats()
        self._ck(self.L.sqt_intersect_batch(self.h, _p(org), _p(dir), n, _p(tri), _p(dist), _p(point),
                                            C.byref(st) if want_stats else None), "sqt_intersect_batch")
        return (tri, dist, point, st.as_dict()) if want_stats else (tri, dist, point)

    def render(self, cam12, params, want_accum=True, want_rgb8=True):
        cam = camera_struct(cam12)
        npix = params.rows * params.cols
        rgb8 = np.zeros((params.rows, params.cols, 3), np.uint8) if want_rgb8 else None
        accum = np.zeros((params.rows, params.cols, 3), np.float32) if want_accum else None
        st = Stats()
        self._ck(self.L.sqt_render(self.h, C.byref(cam), C.byref(params), _p(rgb8), _p(accum), C.byref(st)), "sqt_render")
        return dict(rgb8=rgb8, accum=accum, stats=st.as_dict())

    def render_resident(self, cam12, params):
        cam = camera_struct(cam12)
        st = Stats()
        self._ck(self.L.sqt_render_resident(self.h, C.byref(cam), C.byref(params), C.byref(st)), "sqt_render_resident")
        return st.as_dict()

    def download(self, rows, cols, want_accum=True):
        rgb8 = np.zeros((rows, cols, 3), np.uint8)
        accum = np.zeros((rows, cols, 3), np.float32) if want_accum else None
        self._ck(self.L.sqt_download_image(self.h, _p(rgb8), _p(accum)), "sqt_download_image")
        return rgb8, accum

    def render_begin(self, cam12, params):
        """Start a progressive frame (include/sqt.h): checks, allocations and the primary pass; returns the stats."""
        cam = camera_struct(cam12)
        st = Stats()
        self._shape = (params.rows, params.cols)
        self._ck(self.L.sqt_render_begin(self.h, C.byref(cam), C.byref(params), C.byref(st)), "sqt_render_begin")
        return st.as_dict()

    def render_advance(self, n_samples):
        """Trace the next n_samples samples per pixel of the progressive frame."""
        return _advance(lambda pr, st: self._ck(self.L.sqt_render_advance(self.h, n_samples, pr, st), "sqt_render_advance"))

    def download_moments(self, rows, cols):
        m2 = np.zeros((rows, cols, 3), np.float32)
        self._ck(self.L.sqt_download_moments(self.h, _p(m2)), "sqt_download_moments")
        return m2

    def render_retire(self, rel_tol, abs_tol=0.0, min_samples=MIN_SAMPLES):
        """Retire the converged pixels of the progressive frame (include/sqt.h); returns the pixels still active."""
        rp, act = RetireParams(rel_tol, abs_tol, min_samples, 0), C.c_int64()
        self._ck(self.L.sqt_render_retire(self.h, C.byref(rp), C.byref(act)), "sqt_render_retire")
        return act.value

    def download_sample_counts(self, rows, cols):
        """Samples in each pixel's sums: the k at which it retired, else samples_done."""
        n = np.zeros((rows, cols), np.int32)
        self._ck(self.L.sqt_download_sample_counts(self.h, _p(n)), "sqt_download_sample_counts")
        return n

    def denoise(self, levels=DENOISE_LEVELS, sigma_l=DENOISE_SIGMA_L, sigma_z=DENOISE_SIGMA_Z):
        """Denoised preview of the progressive frame (include/sqt.h): returns rgb8, mean and stats.  The frame is unchanged."""
        return _denoise(self._shape, levels, sigma_l, sigma_z,
                        lambda *a: self._ck(self.L.sqt_denoise(self.h, *a), "sqt_denoise"))

    def download_features(self, rows, cols):
        """Primary-hit AOVs of the progressive frame: surface (tri_out numbering, -1 = no hit), depth t, camera-facing normal."""
        surface = np.zeros((rows, cols), np.int32)
        depth = np.zeros((rows, cols), np.float32)
        normal = np.zeros((rows, cols, 3), np.float32)
        self._ck(self.L.sqt_download_features(self.h, _p(surface), _p(depth), _p(normal)), "sqt_download_features")
        return dict(surface=surface, depth=depth, normal=normal)

    def tone_map(self, mean_rgb):
        mean_rgb = np.ascontiguousarray(mean_rgb, np.float32)
        out = np.zeros(mean_rgb.shape, np.uint8)
        self._ck(self.L.sqt_tone_map(self.h, _p(mean_rgb), mean_rgb.size // 3, _p(out)), "sqt_tone_map")
        return out

    def upload_spheres(self, spheres):
        """spheres: rows (cx, cy, cz, radius, material) -- extension, see include/sqt.h"""
        a = np.zeros(len(spheres), SPHERE_DT)
        for i, (cx, cy, cz, r, m) in enumerate(spheres):
            a[i]["center"] = (cx, cy, cz); a[i]["radius"] = r; a[i]["material"] = int(m)
        self._ck(self.L.sqt_upload_spheres(self.h, _p(a) if len(a) else None, len(a)), "sqt_upload_spheres")

    def set_leaf_cull(self, on):
        self._ck(self.L.sqt_set_option(self.h, 1, 1 if on else 0), "sqt_set_option")

    def set_lens(self, jitter=False, aperture=0.0, focus=1.0):
        """Camera sampling of the frames this context starts (include/sqt.h, sqt_set_lens): box-filtered pixels and a thin
        lens of radius `aperture` focused at ray parameter `focus`.  set_lens(None) restores the reference's pinhole."""
        lens = None if jitter is None else Lens(int(bool(jitter)), aperture, focus, 0)
        self._ck(self.L.sqt_set_lens(self.h, C.byref(lens) if lens is not None else None), "sqt_set_lens")

    def comm_init(self, rank, world, uid):
        buf = (C.c_uint8 * SQT_COMM_ID_BYTES).from_buffer_copy(bytes(uid))
        self._ck(self.L.sqt_comm_init(self.h, rank, world, buf), "sqt_comm_init")

    def fp32_peak_gops(self):
        v = C.c_double()
        self._ck(self.L.sqt_measure_fp32_peak(self.h, C.byref(v)), "sqt_measure_fp32_peak")
        return v.value

    def l2_bandwidth_gbs(self):
        v = C.c_double()
        self._ck(self.L.sqt_measure_l2_bandwidth(self.h, C.byref(v)), "sqt_measure_l2_bandwidth")
        return v.value


class Group:
    """Single-process group: one context per device, ncclCommInitAll underneath (what the Haskell host uses)."""

    def __init__(self, devices):
        self.ctxs = [Context(d) for d in devices]
        self.arr = (C.c_void_p * len(self.ctxs))(*[c.h for c in self.ctxs])
        self.L = b200()
        self._ck(self.L.sqt_comm_init_all(self.arr, len(self.ctxs)), "sqt_comm_init_all")
        self._shape = (0, 0)

    def _ck(self, rc, what):
        if rc:
            raise SqtError("%s failed (%d): %s" % (what, rc, self.ctxs[0].last_error()))

    def upload(self, scene):
        d = scene.desc() if hasattr(scene, "desc") else scene
        self._keep = scene
        self._ck(self.L.sqt_upload_scene_group(self.arr, len(self.ctxs), C.byref(d)), "sqt_upload_scene_group")

    def render(self, cam12, params, want_accum=True):
        cam = camera_struct(cam12)
        rgb8 = np.zeros((params.rows, params.cols, 3), np.uint8)
        accum = np.zeros((params.rows, params.cols, 3), np.float32) if want_accum else None
        st = Stats()
        self._ck(self.L.sqt_render_group(self.arr, len(self.ctxs), C.byref(cam), C.byref(params), _p(rgb8), _p(accum), C.byref(st)),
                 "sqt_render_group")
        return dict(rgb8=rgb8, accum=accum, stats=st.as_dict())

    def render_begin(self, cam12, params):
        cam = camera_struct(cam12)
        st = Stats()
        self._shape = (params.rows, params.cols)
        self._ck(self.L.sqt_render_begin_group(self.arr, len(self.ctxs), C.byref(cam), C.byref(params), C.byref(st)),
                 "sqt_render_begin_group")
        return st.as_dict()

    def render_advance(self, n_samples):
        return _advance(lambda pr, st: self._ck(self.L.sqt_render_advance_group(self.arr, len(self.ctxs), n_samples, pr, st),
                                                "sqt_render_advance_group"))

    def render_retire(self, rel_tol, abs_tol=0.0, min_samples=MIN_SAMPLES):
        rp, act = RetireParams(rel_tol, abs_tol, min_samples, 0), C.c_int64()
        self._ck(self.L.sqt_render_retire_group(self.arr, len(self.ctxs), C.byref(rp), C.byref(act)), "sqt_render_retire_group")
        return act.value

    def download_sample_counts(self, rows, cols):
        return self.ctxs[0].download_sample_counts(rows, cols)

    def set_lens(self, jitter=False, aperture=0.0, focus=1.0):
        """The same lens on every context of the group (set_lens(None): the pinhole)."""
        for c in self.ctxs:
            c.set_lens(jitter, aperture, focus)

    def denoise(self, levels=DENOISE_LEVELS, sigma_l=DENOISE_SIGMA_L, sigma_z=DENOISE_SIGMA_Z):
        return _denoise(self._shape, levels, sigma_l, sigma_z,
                        lambda *a: self._ck(self.L.sqt_denoise_group(self.arr, len(self.ctxs), *a), "sqt_denoise_group"))

    def download_features(self, rows, cols):
        """Every rank takes part (the first call of a frame sums the features onto rank 0); rank 0's result is returned."""
        import threading
        res, errs = [None] * len(self.ctxs), []

        def run(i):
            try:
                res[i] = self.ctxs[i].download_features(rows, cols)
            except SqtError as e:
                errs.append(e)
        th = [threading.Thread(target=run, args=(i,)) for i in range(1, len(self.ctxs))]
        for t in th:
            t.start()
        run(0)
        for t in th:
            t.join()
        if errs:
            raise errs[0]
        return res[0]

    def close(self):
        for c in self.ctxs:
            c.close()


def comm_unique_id():
    buf = (C.c_uint8 * SQT_COMM_ID_BYTES)()
    rc = b200().sqt_comm_unique_id(buf)
    if rc:
        raise SqtError("sqt_comm_unique_id failed: %s" % b200().sqt_last_error(None).decode())
    return bytes(buf)


def write_png(path, rgb8):
    rgb8 = np.ascontiguousarray(rgb8, np.uint8)
    if host().sqth_write_png(path.encode(), _p(rgb8), rgb8.shape[0], rgb8.shape[1]):
        raise SqtError(host().sqth_last_error().decode())
