"""The a-priori error bound behind the exact culling (DESIGN.md section 5): an accepted Moller-Trumbore hit lies within the
bound of its triangle, and the leaf / group culling built on it never rejects a leaf with an accepted triangle.  CPU only
(tests/cull: the host build of the same source as the kernels)."""
import ctypes as C
import math
import os
from fractions import Fraction

import numpy as np
import pytest

import fuzz_slabs
from oracle import oracle as O
from common import HERE, _p, adversarial_rays, build_pair, tame_boundary_rays

U = Fraction(1, 2 ** 24)
EPS_A = Fraction(float(np.float32(1e-4)))          # the `a` guard of mollerTrumbore


def _gamma(n):
    return n * U / (1 - n * U)


SQRT3 = Fraction(math.sqrt(3.0)) * (1 + Fraction(1, 2 ** 50))
C_S = float(_gamma(6) * (2 + 1 / (1 - Fraction(4001, 1000) * U)) / EPS_A)
C_E = float((2 + U) * SQRT3 * _gamma(5) / EPS_A)
K_RHO = float(SQRT3 * _gamma(5) / EPS_A)


_LIB = None


def cull_lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(os.path.join(HERE, "cull", "libsqt_cull.so"))
        L.emu_upload.restype = C.c_void_p
        L.emu_upload.argtypes = [C.c_void_p]
        L.emu_error.restype = C.c_char_p
        L.emu_error.argtypes = [C.c_void_p]
        L.emu_free.argtypes = [C.c_void_p]
        L.cull_pairs.argtypes = [C.c_void_p] * 3 + [C.c_longlong] + [C.c_void_p] * 4
        L.cull_leaf_stats.argtypes = [C.c_void_p] * 3 + [C.c_longlong, C.c_int, C.c_void_p]
        _LIB = L
    return _LIB


def cull_pairs(tri12, org, dirs):
    n = len(org)
    acc = np.zeros(n, np.int32); t = np.zeros(n, np.float32); m = np.zeros(n, np.float32); cul = np.zeros(n, np.int32)
    cull_lib().cull_pairs(_p(tri12), _p(org), _p(dirs), n, _p(acc), _p(t), _p(m), _p(cul))
    return acc.astype(bool), t, m, cul.astype(bool)


def _point_triangle_distance(p, a, e1, e2):
    """Euclidean distance (float64) of points p from the triangles a + s e1 + t e2, s, t >= 0, s + t <= 1."""
    w = p - a
    g11, g12, g22 = (e1 * e1).sum(1), (e1 * e2).sum(1), (e2 * e2).sum(1)
    r1, r2 = (w * e1).sum(1), (w * e2).sum(1)
    det = g11 * g22 - g12 * g12
    with np.errstate(divide="ignore", invalid="ignore"):
        s = (g22 * r1 - g12 * r2) / det
        t = (g11 * r2 - g12 * r1) / det
    inside = (det > 0) & (s >= 0) & (t >= 0) & (s + t <= 1)
    d_plane = np.where(inside, np.linalg.norm(w - s[:, None] * e1 - t[:, None] * e2, axis=1), np.inf)

    def seg(q0, q):
        ll = (q * q).sum(1)
        with np.errstate(divide="ignore", invalid="ignore"):
            h = np.where(ll > 0, ((p - q0) * q).sum(1) / ll, 0.0)
        h = np.clip(h, 0.0, 1.0)
        return np.linalg.norm(p - q0 - h[:, None] * q, axis=1)

    return np.minimum(d_plane, np.minimum(seg(a, e1), np.minimum(seg(a, e2), seg(a + e1, e2 - e1))))


def adversarial_pairs(n_per_scale, seed=17):
    """Triangles at scales 2^-10 .. 2^10, slivers included, with rays aimed at their edges and vertices, most of them grazing
    (|a| just above the 1e-4 guard), origins from 1e-4 in front of the surface out to a few times the triangle's size."""
    rng = np.random.default_rng(seed)
    tris, orgs, dirs = [], [], []
    for k in range(-10, 11, 2):
        sc, n = 2.0 ** k, n_per_scale
        v0 = (rng.uniform(-2, 2, (n, 3)) * sc).astype(np.float32)
        u1 = rng.normal(size=(n, 3)); u1 /= np.linalg.norm(u1, axis=1, keepdims=True)
        w = np.cross(u1, rng.normal(size=(n, 3))); w /= np.linalg.norm(w, axis=1, keepdims=True)
        l1 = sc * rng.uniform(0.05, 1.0, (n, 1)); l2 = sc * rng.uniform(0.05, 1.0, (n, 1))
        thin = 10.0 ** rng.uniform(-3, 0, (n, 1))                      # sliver when small
        ang = rng.uniform(-1, 1, (n, 1))
        e1 = (u1 * l1).astype(np.float32)
        e2 = ((ang * u1 + thin * w) / np.sqrt(ang ** 2 + thin ** 2) * l2).astype(np.float32)
        a64, e164, e264 = v0.astype(np.float64), e1.astype(np.float64), e2.astype(np.float64)
        # target: a point on an edge or a vertex (barycentrics exactly on the boundary), nudged by a few ulps
        b = rng.uniform(0, 1, n); kind = rng.integers(0, 4, n)
        s = np.where(kind == 0, b, np.where(kind == 1, 0.0, np.where(kind == 2, b, rng.integers(0, 2, n).astype(float))))
        t = np.where(kind == 0, 0.0, np.where(kind == 1, b, np.where(kind == 2, 1.0 - b, 0.0)))
        tgt = a64 + s[:, None] * e164 + t[:, None] * e264
        tgt += rng.normal(size=(n, 3)) * sc * 1e-7
        nrm = np.cross(e164, e264); nn = np.linalg.norm(nrm, axis=1, keepdims=True)
        dl = rng.uniform(0.5, 1.15, (n, 1))                            # |d|_1 <= 2: tame directions
        p = np.cross(nrm / nn, rng.normal(size=(n, 3))); p /= np.linalg.norm(p, axis=1, keepdims=True)
        graze = rng.uniform(1.0, 1.3, (n, 1)) * 1e-4 / (dl * nn)       # sin of the angle to the plane for |a| ~ 1e-4 .. 1.3e-4
        graze = np.where(rng.uniform(size=(n, 1)) < 0.25, rng.uniform(0, 1, (n, 1)), graze)
        sphi = np.clip(graze, 0.0, 1.0) * np.where(rng.uniform(size=(n, 1)) < 0.5, -1.0, 1.0)
        d = (p * np.sqrt(1.0 - sphi ** 2) + nrm / nn * sphi) * dl
        far = sc * 10.0 ** rng.uniform(-4, 1, (n, 1))
        near = 1e-4 * dl * rng.uniform(0.8, 1.3, (n, 1))              # origins right at the t > 1e-4 limit
        dist = np.where(rng.uniform(size=(n, 1)) < 0.2, near, far)
        o = tgt - d / dl * dist
        tris.append(np.concatenate([v0, e1[:, :1], e1[:, 1:], e2[:, :2], e2[:, 2:], np.zeros((n, 3), np.float32)], 1))
        orgs.append(o.astype(np.float32)); dirs.append(d.astype(np.float32))
    return (np.ascontiguousarray(np.concatenate(tris), np.float32), np.ascontiguousarray(np.concatenate(orgs)),
            np.ascontiguousarray(np.concatenate(dirs)))


def test_bound_holds_on_adversarial_pairs():
    tri, org, dirs = adversarial_pairs(40_000)
    acc, t, marg, culled = cull_pairs(tri, org, dirs)
    safe = np.isfinite(1.0 / dirs).all(1) & (dirs != 0).all(1)
    assert acc.sum() > 50_000, "too few accepted pairs to say anything"
    assert not (acc & culled & safe).any(), "an accepted triangle was culled"
    v0, e1, e2 = tri[:, 0:3].astype(np.float64), tri[:, 3:6].astype(np.float64), tri[:, 6:9].astype(np.float64)
    o, d = org.astype(np.float64), dirs.astype(np.float64)
    s = o - v0
    a = (e1 * np.cross(d, e2)).sum(1)
    with np.errstate(divide="ignore", invalid="ignore"):
        tstar = (e2 * np.cross(s, e1)).sum(1) / a
    x = o + np.maximum(tstar, 0.0)[:, None] * d              # the ray's point at the exact crossing (or its origin)
    dist = _point_triangle_distance(x, v0, e1, e2)
    E = np.maximum(np.linalg.norm(e1, axis=1), np.linalg.norm(e2, axis=1))
    P = np.linalg.norm(d, axis=1) * E * E
    regime = acc & (K_RHO * P <= 0.5)                         # beyond it the margin covers the origin (DESIGN.md section 5)
    bound = P * (C_S * np.abs(s).sum(1) + C_E * E) * (1.0 + 2.0 * K_RHO * P) + 9.002 * float(U) * E
    r_bound = (dist / bound)[regime]
    r_margin = (dist / marg.astype(np.float64))[acc & safe]
    print("\naccepted pairs %d (%d inside the bound's regime); largest distance / bound %.3g, distance / leaf margin %.3g; "
          "median distance / bound %.3g" % (acc.sum(), regime.sum(), r_bound.max(), r_margin.max(), np.median(r_bound)))
    assert regime.sum() > 50_000
    assert r_bound.max() < 1.0 and r_margin.max() < 1.0
    assert np.all(marg.astype(np.float64)[regime & safe] >= bound[regime & safe])


def _bounce_rays(oracle_scene, camera, n, seed):
    org, dirs = O.make_rays(O.make_params(160, 90, 1), camera)
    tri, _, pt = oracle_scene.intersect_batch(org, dirs)[:3]
    rng = np.random.default_rng(seed)
    p = pt[tri >= 0][rng.integers(0, int((tri >= 0).sum()), n)]
    d = rng.normal(size=(n, 3)); d /= np.linalg.norm(d, axis=1, keepdims=True)
    return p.astype(np.float32), d.astype(np.float32)


def _cull_stats(host_scene, org, dirs):
    """cull_leaf_stats for groups of 1, 2 and 4 triangles: (leaf counters, group counters per group size)."""
    L = cull_lib()
    d = host_scene.desc()
    h = L.emu_upload(C.byref(d))
    try:
        assert not L.emu_error(h)
        org = np.ascontiguousarray(org, np.float32); dirs = np.ascontiguousarray(dirs, np.float32)
        outs = []
        for g in (1, 2, 4):
            out = np.zeros(9, np.uint64)
            L.cull_leaf_stats(h, _p(org), _p(dirs), len(org), g, _p(out))
            outs.append(out)
    finally:
        L.emu_free(h)
    return outs[0][:6], [o[6:] for o in outs]


def test_culling_loses_nothing_on_scene_obj(host_scene, oracle_scene, camera):
    v9, _ = oracle_scene.tris()
    o1, d1 = _bounce_rays(oracle_scene, camera, 20_000, seed=3)
    o2, d2 = adversarial_rays(v9, n_each=128)
    o3, d3 = tame_boundary_rays(v9, 3000)
    leaf, groups = _cull_stats(host_scene, np.concatenate([o1, o2, o3]), np.concatenate([d1, d2, d3]))
    assert leaf[4] > 1000 and leaf[2] > 0.3 * leaf[0]
    assert leaf[5] == 0, "a leaf with an accepted triangle was culled"
    for out in groups:
        assert out[1] > 0 and out[2] == 0, "a group with an accepted triangle was culled"


@pytest.mark.parametrize("kind", range(5))
def test_culling_loses_nothing_on_fuzz_scenes(kind):
    fuzz_slabs.rng = rng = np.random.default_rng(100 + kind)
    v9, mi, mats = fuzz_slabs.rand_scene(kind, 3000)
    _, hs = build_pair(v9, mi, mats)
    pts = v9.reshape(-1, 3); lo, hi = pts.min(0), pts.max(0); c = 0.5 * (lo + hi); h = 0.5 * (hi - lo) + 1e-6
    m = 6000
    org = (c + rng.uniform(-2.2, 2.2, (m, 3)) * h).astype(np.float32)
    tgt = pts[rng.integers(0, len(pts), m)] + rng.normal(size=(m, 3)) * h * 0.01
    d = tgt - org; d /= np.linalg.norm(d, axis=1, keepdims=True) + 1e-30
    o2, d2 = tame_boundary_rays(v9, 1000, seed=kind)
    o3, d3 = adversarial_rays(v9, seed=kind, n_each=64)
    leaf, groups = _cull_stats(hs, np.concatenate([org, o2, o3]), np.concatenate([d.astype(np.float32), d2, d3]))
    assert leaf[4] > 0
    assert leaf[5] == 0, "a leaf with an accepted triangle was culled"
    for out in groups:
        assert out[1] > 0 and out[2] == 0, "a group with an accepted triangle was culled"
