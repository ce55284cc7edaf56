// sqt_core.cuh -- per-ray / per-path device logic of the squigly-trace B200 backend.
//
// Everything here is SQT_HD (__host__ __device__) so that tests/ can compile the same logic with
// g++ and check it against the oracle on the CPU box (tests/emu); the product only ever runs the
// __device__ instantiation from sqt_kernels.cu.
//
// Exactness rules (SURVEY A.1, hard part 2): every FP32 operation on the intersection and shading
// path is an explicit round-to-nearest add/sub/mul/div/sqrt (X* wrappers = __f*_rn on the device,
// never contracted into FMA); min/max follow the Haskell class defaults whenever a NaN could be
// involved; comparisons are written exactly as in the reference.
#pragma once
#include <stdint.h>
#include <math.h>

#if defined(__CUDACC__)
#define SQT_HD __host__ __device__ __forceinline__
#define SQT_HD_NOINLINE __host__ __device__
#define SQT_COLD __host__ __device__ __forceinline__      // (out of line was measured: 1123 vs 1135 Mrays/s)
#else
#define SQT_HD inline
#define SQT_HD_NOINLINE
#define SQT_COLD inline
#endif

#if defined(__CUDA_ARCH__)
#define XADD(a, b) __fadd_rn((a), (b))
#define XSUB(a, b) __fsub_rn((a), (b))
#define XMUL(a, b) __fmul_rn((a), (b))
#define XDIV(a, b) __fdiv_rn((a), (b))
#define XRCP(a) __frcp_rn((a))
#define XSQRT(a) __fsqrt_rn((a))
#define SQT_FMIN(a, b) fminf((a), (b))
#define SQT_FMAX(a, b) fmaxf((a), (b))
#define SQT_LDG4(p) __ldg((const float4 *)(p))
#define SQT_PREFETCH(p) asm volatile("prefetch.global.L1 [%0];" :: "l"(p))
#else
// host build (tests/emu): compiled with -ffp-contract=off -fno-fast-math
#define XADD(a, b) ((float)((float)(a) + (float)(b)))
#define XSUB(a, b) ((float)((float)(a) - (float)(b)))
#define XMUL(a, b) ((float)((float)(a) * (float)(b)))
#define XDIV(a, b) ((float)((float)(a) / (float)(b)))
#define XRCP(a) ((float)(1.0f / (float)(a)))
#define XSQRT(a) sqrtf((a))
#define SQT_FMIN(a, b) fminf((a), (b))
#define SQT_FMAX(a, b) fmaxf((a), (b))
#define SQT_LDG4(p) (*(const float4 *)(p))
#define SQT_PREFETCH(p) ((void)0)
#if !defined(__CUDACC__)
struct alignas(16) float4 { float x, y, z, w; };
struct alignas(8) int2 { int x, y; };
#endif
#endif

namespace sqt {

// ---------------------------------------------------------------------------- device records
// Branch node, 16 B = ONE 128-bit load: exactly the reference's BIHN (BIH.hs:37) plus the two child references:
//   (lmax, rmin, L, R)      L = kLeaf? | kSlow? | axis << 28 | kTight? | index      R = kLeaf? | kTight? | index
// index = position in the branch array (child is a Branch) or in the leaf array (child is a Leaf), < 2^27.
// Side array `slabs` (not in the reference, culling only -- "subtree slabs" below), 16 B per Branch: (lo, hi) of the left
// child's conservative tight slab and (lo, hi) of the right child's; the two low mantissa bits of each lo hold the slab's
// axis, or kSlabNone (not worth a test).  kTight in a reference to a Branch says that its record has a slab worth loading.
// The traversal carries the ray's parametric interval (tmin, tmax) through the box of the subtree it is about to
// enter -- the two numbers intersectsBB (Geometry.hs:166-177) computes for that box -- and updates it per visit from
// the ONE plane in which a child box differs from its parent (BIH.hs:130-141): the classic BIH step.  That is exact
// (same compare results as recomputing all six slabs, see desc_step) whenever the child box is nested in the parent's
// on the split axis, lo[ax] <= lmax <= hi[ax] and lo[ax] <= rmin <= hi[ax]; lmax/rmin carry +-0.001 (BIH.hs:93-95), so
// a plane can stick out of the clipped box -- such nodes are flagged kSlow at upload and, like rays with a
// zero/denormal/non-finite component, take the literal six-slab path from the node's box in the side array `boxes`.
// Box of a branch (side array, slow path only), 32 B: c0 = (lo.x, lo.y, lo.z, hi.x)  c1 = (hi.y, hi.z, -, -): the
// `bbox` argument intersectBIH' receives for this node, derived at upload by copying planes (no arithmetic).
// Leaf record, 32 B = 2 x 128-bit loads: the TIGHT bounding box of the leaf's triangles and their longest edge
// (used only by the conservative leaf culling, never by the reference algorithm) and the triangle range:
//   b0 = (lo.x, lo.y, lo.z, hi.x)   b1 = (hi.y, hi.z, longest edge E, first | min(count, 31) << 27 as u32 bits)
//        a leaf of 31 or more triangles keeps its count in the spare word of its first triangle record
// Traversal stack entries, 16 B each (one 128-bit load/store), at most one per tree level:
//   phase A (near subtree in flight) : (far child ref | axis << 28, far tmin, far tmax, plane isClose compares with)
//   phase B (near hit parked, far subtree in flight) : (tri | kPhaseB, t, dist, -)
constexpr uint32_t kLeaf = 0x80000000u;
constexpr uint32_t kPhaseB = 0x40000000u;
constexpr uint32_t kSlow = 0x40000000u;
constexpr uint32_t kAxisShift = 28;
constexpr uint32_t kTight = 0x08000000u;       // reference to a Branch: slabs[index] holds a child slab worth testing
constexpr uint32_t kSlabNone = 3u;             // slab code (low mantissa bits of its lo): axis 0..2, or no slab worth a test
constexpr uint32_t kIdxMask = 0x07ffffffu;
constexpr uint32_t kLeafFirstMask = 0x07ffffffu;
constexpr uint32_t kLeafCountShift = 27;
constexpr uint32_t kLeafLong = 31u;
constexpr int kStackEntries = 48;              // at most one entry per tree level (SQT_MAX_HEIGHT)
#ifndef SQT_MAX_DEPTH
#define SQT_MAX_DEPTH 64
#endif

struct SceneView {
    const float4 *nodes;     // 1 float4 per branch
    const float4 *boxes;     // 2 float4 per branch (slow path only)
    const float4 *slabs;     // 1 float4 per branch: tight slabs of its two children (culling only)
    const float4 *leaves;    // 2 float4 per leaf
    const float4 *tris;      // 3 float4 per triangle: (v0.xyz,e1.x) (e1.yz,e2.xy) (e2.z, mat, orig, leaf count if >= 31)
    const float4 *mats;      // 3 float4 per material: (refl, surf.rgb) (emissive, emit.rgb) (ec.rgb, flags)
    const float4 *spheres;   // extension: 2 float4 per sphere: (center.xyz, radius) (material bits, -, -, -)
    const float4 *sph_nodes; // extension: BVH over the spheres, 2 float4 per node (see sphere_step); nullptr = test every sphere
    const uint32_t *sph_order;   // sphere indices in BVH leaf order
    uint32_t n_spheres;
    float root_lo[3], root_hi[3];
    uint32_t n_branches, n_tris, n_mats;
    uint32_t root_is_leaf;   // tree = Leaf: no box test at all (BIH.hs:105)
    uint32_t leaf_cull;      // 1 = skip leaves whose enlarged tight box the ray provably misses (exact, see enter_leaf)
    uint32_t planes_finite;  // every plane and box coordinate of the tree is finite (else every ray takes the literal path)
    float tame_c[3], tame_r; // rays with |o - tame_c|_1 <= tame_r and |d|_1 <= 2 may use the subtree slabs (their margins assume it)
};

struct Ray { float ox, oy, oz, dx, dy, dz; };
struct Hit { int tri; float t; float dist; };      // tri = index in leaf order, -1 = Nothing
struct Counters {
    unsigned long long branch_visits, child_box_tests, tri_tests, rays, leaves_culled;
    unsigned long long mt_pass_a, mt_pass_u, mt_pass_v, mt_accept;      // triangle tests that got past each guard
};

SQT_HD uint32_t f2u(float f) {
#if defined(__CUDA_ARCH__)
    return __float_as_uint(f);
#else
    uint32_t u; __builtin_memcpy(&u, &f, 4); return u;
#endif
}
SQT_HD float u2f(uint32_t u) {
#if defined(__CUDA_ARCH__)
    return __uint_as_float(u);
#else
    float f; __builtin_memcpy(&f, &u, 4); return f;
#endif
}

// Haskell Ord Float class defaults: max x y = if x <= y then y else x ; min x y = if x <= y then x else y
SQT_HD float hs_max(float x, float y) { return (x <= y) ? y : x; }
SQT_HD float hs_min(float x, float y) { return (x <= y) ? x : y; }
// compare a b == GT  (anything against NaN is GT)
SQT_HD bool cmp_gt(float a, float b) { return !(a < b) && !(a == b); }
SQT_HD bool finite_f(float x) { return fabsf(x) < INFINITY; }   // false for inf and NaN

// V3.hs:25-26  dot = (a*d)+(b*e)+(c*f)
SQT_HD float dot3(float a, float b, float c, float d, float e, float f) {
    return XADD(XADD(XMUL(a, d), XMUL(b, e)), XMUL(c, f));
}

// ------------------------------------------------------------------------------- slab tests
// Geometry.hs:166-177, literal: also returns the two numbers the test compares.  `fast` (the ray cannot produce a NaN
// slab value: all of origin, direction and 1/direction finite, all planes finite) uses the hardware FMNMX -- without
// NaNs min/max are exact, order-free selections whose zero sign never reaches the two comparisons; otherwise the
// Haskell class defaults decide (operand order matters with NaN).
SQT_HD bool slab_iv(float lx, float ly, float lz, float hx, float hy, float hz, const Ray &r, float dfx, float dfy, float dfz,
                    bool fast, float &tmin, float &tmax) {
    const float t1 = XMUL(XSUB(lx, r.ox), dfx), t2 = XMUL(XSUB(hx, r.ox), dfx);
    const float t3 = XMUL(XSUB(ly, r.oy), dfy), t4 = XMUL(XSUB(hy, r.oy), dfy);
    const float t5 = XMUL(XSUB(lz, r.oz), dfz), t6 = XMUL(XSUB(hz, r.oz), dfz);
    if (fast) {
        tmin = SQT_FMAX(SQT_FMAX(SQT_FMIN(t1, t2), SQT_FMIN(t3, t4)), SQT_FMIN(t5, t6));
        tmax = SQT_FMIN(SQT_FMIN(SQT_FMAX(t1, t2), SQT_FMAX(t3, t4)), SQT_FMAX(t5, t6));
    } else {
        tmin = hs_max(hs_max(hs_min(t1, t2), hs_min(t3, t4)), hs_min(t5, t6));
        tmax = hs_min(hs_min(hs_max(t1, t2), hs_max(t3, t4)), hs_max(t5, t6));
    }
    return tmax > 0.0f && tmin < tmax;
}
SQT_HD bool slab_exact(float lx, float ly, float lz, float hx, float hy, float hz, const Ray &r,
                       float dfx, float dfy, float dfz) {
    float tmin, tmax;
    return slab_iv(lx, ly, lz, hx, hy, hz, r, dfx, dfy, dfz, false, tmin, tmax);
}

// branch-free 3-way select (the compiler turns the ?: chain into divergent branches otherwise)
SQT_HD float sel3(int ax, float x, float y, float z) {
#if defined(__CUDA_ARCH__)
    float r;
    asm("{\n\t.reg .pred p1, p2;\n\tsetp.eq.s32 p1, %4, 1;\n\tsetp.eq.s32 p2, %4, 2;\n\t"
        "selp.f32 %0, %2, %1, p1;\n\tselp.f32 %0, %3, %0, p2;\n\t}"
        : "=&f"(r) : "f"(x), "f"(y), "f"(z), "r"(ax));
    return r;
#else
    return ax == 0 ? x : (ax == 1 ? y : z);
#endif
}

// ------------------------------------------------------------------------- Moller-Trumbore
// Geometry.hs:117-142 with edge1/edge2 precomputed.  Guard order a -> u -> v -> t.
SQT_HD bool moller_trumbore(const float4 &a0, const float4 &a1, const float4 &a2, const Ray &r, float &t_out,
                            float &dist_out, int &stage) {
    const float eps = 0.0001f;
    const float v0x = a0.x, v0y = a0.y, v0z = a0.z;
    const float e1x = a0.w, e1y = a1.x, e1z = a1.y;
    const float e2x = a1.z, e2y = a1.w, e2z = a2.x;
    // h = rayDir `cross` edge2
    float hx = XSUB(XMUL(r.dy, e2z), XMUL(r.dz, e2y));
    float hy = XSUB(XMUL(r.dz, e2x), XMUL(r.dx, e2z));
    float hz = XSUB(XMUL(r.dx, e2y), XMUL(r.dy, e2x));
    float a = dot3(e1x, e1y, e1z, hx, hy, hz);
    stage = 0;
    if (a > -eps && a < eps) return false;
    stage = 1;
    float f = XRCP(a);
    float sx = XSUB(r.ox, v0x), sy = XSUB(r.oy, v0y), sz = XSUB(r.oz, v0z);
    float u = XMUL(f, dot3(sx, sy, sz, hx, hy, hz));
    if (u < 0.0f || u > 1.0f) return false;
    stage = 2;
    // q = s `cross` edge1
    float qx = XSUB(XMUL(sy, e1z), XMUL(sz, e1y));
    float qy = XSUB(XMUL(sz, e1x), XMUL(sx, e1z));
    float qz = XSUB(XMUL(sx, e1y), XMUL(sy, e1x));
    float v = XMUL(f, dot3(r.dx, r.dy, r.dz, qx, qy, qz));
    if (v < 0.0f || XADD(u, v) > 1.0f) return false;
    stage = 3;
    float t = XMUL(f, dot3(e2x, e2y, e2z, qx, qy, qz));
    if (!(t > eps)) return false;
    stage = 4;
    // outInter = rayVert + t *^ rayDir ; rayDist = norm (outInter - rayVert)
    float px = XADD(r.ox, XMUL(t, r.dx)), py = XADD(r.oy, XMUL(t, r.dy)), pz = XADD(r.oz, XMUL(t, r.dz));
    float ex = XSUB(px, r.ox), ey = XSUB(py, r.oy), ez = XSUB(pz, r.oz);
    t_out = t;
    dist_out = XSQRT(dot3(ex, ey, ez, ex, ey, ez));
    return true;
}

// FILTER in front of mollerTrumbore (pool kernel): false only if the full test is certain to fail its `a` or its `u` guard.
// `a` and D = s . h are computed with the operations of the full test, in the same order; the `a` guard is the same
// comparison.  The `u` guard of the full test looks at u = RN(f * D), f = RN(1 / a); the filter decides without the division:
//   * sD = D with the sign of a applied.  sD < -1e-20 and |a| < 1e20: |f * D| >= 1e-40 > 2^-149, so u is a negative number
//     (possibly denormal, never -0) and the full test returns at `u < 0`;
//   * sD > |a| * 1.000002: D / a > 1.0000019 and two roundings of relative size 2^-24 leave u > 1: the full test returns at `u > 1`;
//   * anything else -- including every NaN and infinity, for which all comparisons are false -- goes on to the full test.
// Straight-line code, no MUFU, no branch; ~18 % of the pairs survive and are re-run by moller_trumbore itself.
SQT_HD bool moller_trumbore_au(const float4 &a0, const float4 &a1, const float4 &a2, const Ray &r, bool &pass_a) {
    const float eps = 0.0001f;
    const float v0x = a0.x, v0y = a0.y, v0z = a0.z;
    const float e1x = a0.w, e1y = a1.x, e1z = a1.y;
    const float e2x = a1.z, e2y = a1.w, e2z = a2.x;
    const float hx = XSUB(XMUL(r.dy, e2z), XMUL(r.dz, e2y));
    const float hy = XSUB(XMUL(r.dz, e2x), XMUL(r.dx, e2z));
    const float hz = XSUB(XMUL(r.dx, e2y), XMUL(r.dy, e2x));
    const float a = dot3(e1x, e1y, e1z, hx, hy, hz);
    const float sx = XSUB(r.ox, v0x), sy = XSUB(r.oy, v0y), sz = XSUB(r.oz, v0z);
    const float D = dot3(sx, sy, sz, hx, hy, hz);
    const float aa = fabsf(a), sD = (a < 0.0f) ? -D : D;
    pass_a = !(a > -eps && a < eps);
    const bool neg = sD < -1.0e-20f && aa < 1.0e20f;
    const bool big = sD > XMUL(aa, 1.000002f);
    return pass_a && !neg && !big;
}

// ------------------------------------------------------------------------- exact culling margin
// A-priori error bound of moller_trumbore (derivation: DESIGN.md section 5).  If the test accepts a triangle with edges
// |e1|, |e2| <= E for a ray (o, d), the half-line o + t d, t >= 0, passes within
//   delta = N E^2 (cS S + cE E) (1 + 2 krho N E^2)
// of the triangle, where N >= |d|_2, S >= |o - v0|_1 and also >= |o_k - plane_k| for every plane of the box tested, and the
// constants come from gamma_n bounds of the operation sequence (cS = 3 gamma_6 / 1e-4, cE = 2 sqrt3 gamma_5 / 1e-4,
// krho = sqrt3 gamma_5 / 1e-4; the last factor covers the error of `a` itself).  cull_margin returns delta plus what the
// rounding of the slab test needs, 2^-19 (|o|_inf + S) + kCullAbs, with n2 = 2N, P2 = n2 E^2 = 2 N E^2 and
//   kCullC0 = cS / 2, kCullKappa = cE / cS, kCullC1 = kCullC0 krho,
// all rounded up and C0 enlarged by (1 + 2^-19) so that the rounding of the margin's own 21 operations (all on
// non-negative values) never leaves it below the bound.
constexpr float kCullC0 = 0x1.5f9038p-8f, kCullC1 = 0x1.d092d0p-16f, kCullKappa = 0x1.ecac14p-1f;
constexpr float kCullAbs = 1.0e-4f;
SQT_HD float cull_margin(float n2, float E, float S, float omax) {
    const float P2 = n2 * (E * E);
    return P2 * (S + kCullKappa * E) * (kCullC0 + kCullC1 * P2) + (kCullAbs + 1.9073486328125e-6f * (omax + S));
}
// The margin of the leaf record (b0, b1) for ray r: N = (1 + |d|^2) / 2 >= |d| (exact for unit directions),
// S = sum_k max(|o_k - lo_k|, |o_k - hi_k|) >= |o - v0|_1 for every v0 in the box.
SQT_HD float leaf_margin(const float4 &b0, const float4 &b1, const Ray &r) {
    const float S = fmaxf(fabsf(r.ox - b0.x), fabsf(r.ox - b0.w)) + fmaxf(fabsf(r.oy - b0.y), fabsf(r.oy - b1.x)) +
                    fmaxf(fabsf(r.oz - b0.z), fabsf(r.oz - b1.y));
    const float omax = fmaxf(fmaxf(fabsf(r.ox), fabsf(r.oy)), fabsf(r.oz));
    const float n2 = 1.0f + (r.dx * r.dx + r.dy * r.dy + r.dz * r.dz);
    return cull_margin(n2, b1.z, S, omax);
}
// Leaf culling: true if the ray provably misses the tight box (b0, b1) of a leaf record enlarged by leaf_margin, i.e. no
// triangle of the leaf can be accepted.  Only for rays with finite direction components and reciprocals and finite
// origins (`safe`); a NaN or infinite margin keeps the leaf.
SQT_HD bool leaf_box_culled(const float4 &b0, const float4 &b1, const Ray &r, float dfx, float dfy, float dfz) {
    const float m = leaf_margin(b0, b1, r);
    const float lx = (b0.x - m - r.ox) * dfx, hx = (b0.w + m - r.ox) * dfx;
    const float ly = (b0.y - m - r.oy) * dfy, hy = (b1.x + m - r.oy) * dfy;
    const float lz = (b0.z - m - r.oz) * dfz, hz = (b1.y + m - r.oz) * dfz;
    const float tmin = SQT_FMAX(SQT_FMAX(SQT_FMIN(lx, hx), SQT_FMIN(ly, hy)), SQT_FMIN(lz, hz));
    const float tmax = SQT_FMIN(SQT_FMIN(SQT_FMAX(lx, hx), SQT_FMAX(ly, hy)), SQT_FMAX(lz, hz));
    return tmax < 0.0f || tmin > tmax;          // a NaN anywhere keeps the leaf
}

// ------------------------------------------------------------------------------ leaf records
// Leaf record (see "device records") of the leaf tris[first .. first + cnt): the tight box of the triangles as
// Moller-Trumbore sees them (v0, v0 + e1, v0 + e2), rounded outwards, and their longest edge, rounded up.  Used only by
// the conservative leaf culling.  Runs on the device at upload (k_leaf_records) and on the host in tests/emu.
SQT_HD_NOINLINE inline void make_leaf_record(const float4 *tris, uint32_t first, uint32_t cnt, float4 &b0, float4 &b1) {
    double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300}, e2max = 0;
    for (uint32_t t = 0; t < cnt; ++t) {
        const float4 a0 = tris[3 * (size_t)(first + t)], a1 = tris[3 * (size_t)(first + t) + 1], a2 = tris[3 * (size_t)(first + t) + 2];
        const float v0[3] = {a0.x, a0.y, a0.z}, e1[3] = {a0.w, a1.x, a1.y}, e2[3] = {a1.z, a1.w, a2.x};
        double l1 = 0, l2 = 0, l3 = 0;
        for (int k = 0; k < 3; ++k) {
            const double v[3] = {(double)v0[k], (double)v0[k] + e1[k], (double)v0[k] + e2[k]};
            for (int q = 0; q < 3; ++q) { if (v[q] < lo[k]) lo[k] = v[q]; if (v[q] > hi[k]) hi[k] = v[q]; }
            l1 += (double)e1[k] * e1[k]; l2 += (double)e2[k] * e2[k];
            l3 += ((double)e2[k] - e1[k]) * ((double)e2[k] - e1[k]);
        }
        e2max = fmax(e2max, fmax(l1, fmax(l2, l3)));
    }
    if (cnt == 0) { for (int k = 0; k < 3; ++k) lo[k] = hi[k] = 0; }
    const uint32_t c5 = cnt < kLeafLong ? cnt : kLeafLong;
    b0.x = nextafterf((float)lo[0], -INFINITY); b0.y = nextafterf((float)lo[1], -INFINITY); b0.z = nextafterf((float)lo[2], -INFINITY);
    b0.w = nextafterf((float)hi[0], INFINITY);
    b1.x = nextafterf((float)hi[1], INFINITY); b1.y = nextafterf((float)hi[2], INFINITY);
    b1.z = nextafterf((float)sqrt(e2max), INFINITY);
    b1.w = u2f((cnt ? first : 0u) | (c5 << kLeafCountShift));
}

// ------------------------------------------------------------------------------ subtree slabs
// Tight box + longest edge of everything below a Branch, aggregated bottom-up from the leaf records (2 x float4 like a
// leaf record: (lo.xyz, hi.x) (hi.yz, E, empty? as bits)), and from it the ONE-axis slab desc_step intersects the ray's
// interval with.  Runs on the device at upload (k_branch_tight / k_child_slabs) and on the host in tests/emu.
struct TightRec { float4 t0, t1; };
SQT_HD TightRec tight_of_leaf(const float4 *leaves, uint32_t leaf) {
    TightRec r; r.t0 = leaves[2 * (size_t)leaf]; r.t1 = leaves[2 * (size_t)leaf + 1];
    r.t1.w = u2f((f2u(r.t1.w) >> kLeafCountShift) == 0u ? 1u : 0u);          // an empty leaf contributes nothing
    return r;
}
SQT_HD TightRec tight_union(const TightRec &a, const TightRec &b) {
    if (f2u(a.t1.w)) return b;
    if (f2u(b.t1.w)) return a;
    TightRec r;
    r.t0.x = fminf(a.t0.x, b.t0.x); r.t0.y = fminf(a.t0.y, b.t0.y); r.t0.z = fminf(a.t0.z, b.t0.z);
    r.t0.w = fmaxf(a.t0.w, b.t0.w); r.t1.x = fmaxf(a.t1.x, b.t1.x); r.t1.y = fmaxf(a.t1.y, b.t1.y);
    r.t1.z = fmaxf(a.t1.z, b.t1.z); r.t1.w = u2f(0u);
    return r;
}
// Margin: the leaf-culling margin (cull_margin) with its per-ray quantities replaced by their maxima over tame rays --
// |d|_2 <= |d|_1 <= 2 (N = 2, n2 = 4), |origin - plane| and |origin - v0|_1 <= s_max = 3 x the root's 1-norm half extent,
// |origin|_inf <= c_max + s_max (c_max = largest root coordinate).
// The axis is the one on which the enlarged tight extent is the smallest fraction of the Branch's clipped box (c0, c1: the
// box intersectBIH' passes down, BIH.hs:130-141); the slab is worth a test (return true) if that fraction is below ratio_max.
SQT_HD bool make_slab(const TightRec &t, const float4 &c0, const float4 &c1, float s_max, float c_max, float ratio_max, float4 &slab) {
    const float m = cull_margin(4.0f, t.t1.z, s_max, c_max + s_max);
    const float tlo[3] = {t.t0.x, t.t0.y, t.t0.z}, thi[3] = {t.t0.w, t.t1.x, t.t1.y};
    const float clo[3] = {c0.x, c0.y, c0.z}, chi[3] = {c0.w, c1.x, c1.y};
    float best = 2.0f;
    int bax = 0;
    for (int k = 0; k < 3; ++k) {
        const float len = chi[k] - clo[k];
        const float a = fmaxf(tlo[k] - m, clo[k]), b = fminf(thi[k] + m, chi[k]);
        const float ratio = (len > 0.0f && len < 1.0e30f && m == m && m < 1.0e30f) ? (b - a) / len : 2.0f;
        if (ratio < best) { best = ratio; bax = k; }
    }
    slab.x = tlo[bax] - m; slab.y = thi[bax] + m; slab.z = best; slab.w = u2f((uint32_t)bax);
    return f2u(t.t1.w) == 0u && best < ratio_max;
}

// lo bound of a slab with its code in the two low mantissa bits: moved outwards by 4..7 ulps, which keeps it conservative
SQT_HD float pack_slab_lo(float lo, uint32_t code) {
    if (!(fabsf(lo) >= 1.0e-30f)) lo = -1.0e-30f;                            // zero / denormal / NaN (NaN: the code is kSlabNone)
    const uint32_t b = f2u(lo);
    return u2f((((lo > 0.0f) ? b - 4u : b + 4u) & ~3u) | code);
}
// the box intersectBIH' passes to child `side` (0 = left, 1 = right) of a Branch with box (p0, p1), BIH.hs:130-141
SQT_HD void clip_child_box(const float4 &p0, const float4 &p1, int ax, float lmax, float rmin, int side, float4 &c0, float4 &c1) {
    c0 = p0; c1 = p1;
    if (side == 0) { if (ax == 0) c0.w = lmax; else if (ax == 1) c1.x = lmax; else c1.y = lmax; }
    else           { if (ax == 0) c0.x = rmin; else if (ax == 1) c0.y = rmin; else c0.z = rmin; }
}

// ------------------------------------------------------------------------------ traversal
// intersectBIH (BIH.hs:101-141) as an explicit-stack state machine that visits exactly the
// subtrees the recursion visits, in the same order, and combines results with the same rules:
//   * the own-box test of BIH.hs:112 is evaluated for the root only -- for every other branch it
//     repeats, with identical operands, the test its parent just passed at BIH.hs:128-129;
//   * a branch whose two children are both hit pushes a "phase A" entry (far child, its interval, the plane
//     isClose looks at) and enters the near child; when that subtree returns, isClose (BIH.hs:121-123) is evaluated
//     on the near subtree's OWN result; if the far child must still be visited and near had a hit, that hit is
//     parked in the same stack slot ("phase B") and merged with min' when the far subtree returns.
//
// The machine is cut into unit steps so that a warp can run them in lock step (sqt_kernels.cuh):
//   ST_DESC  enter Branch `child` with the ray's interval (tmin, tmax) through its box: derive both child intervals
//   ST_ENTER enter Leaf `child`: fetch its record, (conservatively) cull it or become ST_LEAF
//   ST_LEAF  test ONE triangle of the current leaf, walking from the last to the first
//   ST_RET   a subtree returned `cur`: pop stack entries until one sends the ray into a far subtree
//   ST_DONE  the ray is finished, result in `cur`
//   ST_SPH   (extension) the BIH part is finished, the analytic spheres are still to be folded in (sphere_step)
enum : int { ST_DONE = 0, ST_DESC = 1, ST_LEAF = 2, ST_RET = 3, ST_EXIT = 4, ST_ENTER = 5, ST_SPH = 6 };

constexpr uint32_t kRfUnsafe = 0x40000000u, kRfTame = 0x08000000u;
struct TravLane {
    Ray r;
    float dfx, dfy, dfz;        // 1/dir (Geometry.hs:168), IEEE
    uint32_t child;             // ST_DESC: branch to visit ; ST_ENTER: leaf to enter ; ST_LEAF: first triangle of the leaf
    float tmin, tmax;           // ST_DESC: intersectsBB's two numbers for the box of `child` (fast rays only)
    int i;                      // ST_LEAF: offset of the next triangle to test (counts down to 0)
    Hit cur;                    // result of the subtree that just returned / running best of the current leaf
    int sp;                     // stack entries in use
    int state;
    uint32_t rf;                // ray flags, placed so that one LOP3 combines them with a node / reference word:
                                //   bit k (k = 0..2) set iff dir[k] > 0 (leftToRight on axis k, BIH.hs:127)
                                //   kRfUnsafe (= kSlow): some slab value of this ray can be NaN -> literal six-slab path, no FMNMX
                                //   kRfTame (= kTight): culling is on, the ray is safe and within the range the subtree-slab margins
                                //   were derived for.  Other bits are ignored (the pool kernel keeps state and sp there).
    float4 *stack;              // entry e lives at stack[e * STRIDE] (STRIDE template parameter of the steps)
};

// How a step reads the ray: from the lane's registers (one ray per lane) ...
struct LaneRay {
    const TravLane &L;
    SQT_HD explicit LaneRay(const TravLane &l) : L(l) {}
    SQT_HD float o(int ax) const { return sel3(ax, L.r.ox, L.r.oy, L.r.oz); }
    SQT_HD float d(int ax) const { return sel3(ax, L.r.dx, L.r.dy, L.r.dz); }
    SQT_HD float df(int ax) const { return sel3(ax, L.dfx, L.dfy, L.dfz); }
    SQT_HD Ray ray() const { return L.r; }
    SQT_HD void dfv(float &x, float &y, float &z) const { x = L.dfx; y = L.dfy; z = L.dfz; }
};
// ... or from a structure-of-arrays pool (k_paths_pool: word f of slot s at base[f * stride + s]; fields ox oy oz dx dy
// dz dfx dfy dfz are the first nine): the split axis indexes the array, no selects, no ray registers held over a burst
struct PoolRay {
    const uint32_t *base; int stride;
    SQT_HD PoolRay(const uint32_t *b, int st) : base(b), stride(st) {}
    SQT_HD float f(int k) const { return u2f(base[k * stride]); }
    SQT_HD float o(int ax) const { return f(ax); }
    SQT_HD float d(int ax) const { return f(3 + ax); }
    SQT_HD float df(int ax) const { return f(6 + ax); }
    SQT_HD Ray ray() const { Ray r; r.ox = f(0); r.oy = f(1); r.oz = f(2); r.dx = f(3); r.dy = f(4); r.dz = f(5); return r; }
    SQT_HD void dfv(float &x, float &y, float &z) const { x = f(6); y = f(7); z = f(8); }
};

// ---- extension: analytic spheres (no reference counterpart; semantics restated in oracle/oracle.c) ----------------
// oc = o - c ; A = d.d ; B = oc.d ; C = oc.oc - r*r ; disc = B*B - A*C ; disc < 0 -> Nothing
// t0 = (-B - sqrt disc)/A ; t1 = (-B + sqrt disc)/A ; t = first of t0, t1 that is > eps (1e-4, as mollerTrumbore)
// point = o + t *^ d ; dist = norm (point - o)     -- same conventions as Geometry.hs:134,141
SQT_HD bool ray_sphere(const float4 &s0, const Ray &r, float &t_out, float &dist_out) {
    const float eps = 0.0001f;
    const float ocx = XSUB(r.ox, s0.x), ocy = XSUB(r.oy, s0.y), ocz = XSUB(r.oz, s0.z);
    const float A = dot3(r.dx, r.dy, r.dz, r.dx, r.dy, r.dz);
    const float B = dot3(ocx, ocy, ocz, r.dx, r.dy, r.dz);
    const float C = XSUB(dot3(ocx, ocy, ocz, ocx, ocy, ocz), XMUL(s0.w, s0.w));
    const float disc = XSUB(XMUL(B, B), XMUL(A, C));
    if (!(disc >= 0.0f)) return false;
    const float sq = XSQRT(disc);
    const float t0 = XDIV(XSUB(-B, sq), A), t1 = XDIV(XADD(-B, sq), A);
    const float t = t0 > eps ? t0 : t1;
    if (!(t > eps)) return false;
    const float px = XADD(r.ox, XMUL(t, r.dx)), py = XADD(r.oy, XMUL(t, r.dy)), pz = XADD(r.oz, XMUL(t, r.dz));
    const float ex = XSUB(px, r.ox), ey = XSUB(py, r.oy), ez = XSUB(pz, r.oz);
    t_out = t;
    dist_out = XSQRT(dot3(ex, ey, ez, ex, ey, ez));
    return true;
}

// The BIH part of a ray is finished with `cur`.  Without spheres the ray is ST_DONE; with spheres (extension) it becomes
// ST_SPH and sphere_step folds them in.  Semantics (include/sqt.h, restated by the oracle): candidates in order
// [BIH hit, sphere 0, sphere 1, ..], minimumBy (comparing dist) -- the first minimal candidate wins.  Surface n_tris + k =
// sphere k.
template <class RA>
SQT_HD void finish_ray(const SceneView &sc, TravLane &L, const RA &ra) {
    L.state = sc.n_spheres ? ST_SPH : ST_DONE;
}
// every sphere in index order: the definition
SQT_COLD Hit fold_spheres(const float4 *spheres, uint32_t n_spheres, uint32_t n_tris, const Ray &r, Hit cur) {
    for (uint32_t k = 0; k < n_spheres; ++k) {
        const float4 s0 = SQT_LDG4(spheres + 2 * (size_t)k);
        float t, dist;
        if (ray_sphere(s0, r, t, dist)) {
            if (cur.tri < 0 || cmp_gt(cur.dist, dist)) { cur.tri = (int)(n_tris + k); cur.t = t; cur.dist = dist; }
        }
    }
    return cur;
}
// The same result through a bounding-volume hierarchy over the spheres (built at upload, sqt_layout.hpp), so that a ray
// tests a few spheres instead of all of them.  BVH node, 2 x float4: (lo.xyz, hi.x) (hi.yz, a, b); interior: a = low child |
// split axis << 30, b = high child; leaf: a = first entry of sph_order, b = count | kLeaf.  Boxes bound centre +- radius *
// (1 + 2^-19).  The child on the ray's side of the split is visited first, and a node is also skipped when the line
// enters its (enlarged) box farther away than the best hit so far (3).  (A 4-wide variant with the four child boxes in
// the parent was measured: 2.4x SLOWER -- its unrolled box tests and ordering need registers the path kernel does not have;
// 8 spheres per leaf with a prefetch of the sibling node: 10 % slower than 4 per leaf without.)
// Exactness.  (1) Order: the definition keeps the candidate of least dist, the earliest on ties (a later candidate replaces
// only if strictly closer).  For finite distances that is a property of the candidate SET: fold rule below = "strictly
// closer, or as close and an earlier sphere", and the BIH hit (candidate 0) is never replaced on a tie.  (2) Culling:
// ray_sphere accepts only if its computed disc = B*B - A*C >= 0.  With eps = 2^-24 every 3-term dot is off by <= 3 eps
// sum|terms|, which bounds |disc_computed - disc_exact| by 17 eps |d|^2 (|oc|^2 + r^2) < 2^-19 |d|^2 (|oc|^2 + r^2), and
// disc_exact = |d|^2 (r^2 - rho^2) with rho the distance of the centre from the ray's LINE.  An accepted sphere therefore has
// rho <= r (1 + 2^-20) + 2^-9.5 |oc|.  A node is skipped only if the line misses its box enlarged by 0.0014 * D
// (0.0014 > 2^-9.5; D = 1-norm distance of the origin to the box centre + 1-norm half extent >= |oc| of every sphere in
// it) plus 2^-18 (|box| + |o|) for the slab arithmetic itself: no skipped sphere could have been accepted.  (3) Distance:
// the same error terms put the computed t of an accepted sphere within 0.0014 |oc| / |d| of a point of the line inside the
// enlarged box, so its dist is at least (t_entry |d|)(1 - 2^-16) - 0.003 D; a node whose bound exceeds the best dist so far
// cannot hold a closer or an equally close candidate.  The bounds assume no overflow / underflow: rays with a non-finite,
// zero, huge or tiny component take the definition.
template <class RA>
SQT_HD void sphere_step(const SceneView &sc, TravLane &L, const RA &ra) {
    const Ray r = ra.ray();
    const float big = 1.0e12f, tiny = 1.0e-12f;
    const float dmax = fmaxf(fmaxf(fabsf(r.dx), fabsf(r.dy)), fabsf(r.dz)), dmin = fminf(fminf(fabsf(r.dx), fabsf(r.dy)), fabsf(r.dz));
    const float omax = fmaxf(fmaxf(fabsf(r.ox), fabsf(r.oy)), fabsf(r.oz));
    L.state = ST_DONE;
    if (!sc.sph_nodes || !(dmax < big) || !(dmin > tiny) || !(omax < big)) {
        L.cur = fold_spheres(sc.spheres, sc.n_spheres, sc.n_tris, r, L.cur);
        return;
    }
    const float dfx = 1.0f / r.dx, dfy = 1.0f / r.dy, dfz = 1.0f / r.dz;
    const float dlen = 0.99998f * sqrtf(r.dx * r.dx + r.dy * r.dy + r.dz * r.dz);       // a lower bound of |d|
    uint32_t stack[32];
    int sp = 0;
    uint32_t node = 0u;
    for (;;) {
        const float4 n0 = SQT_LDG4(sc.sph_nodes + 2 * (size_t)node), n1 = SQT_LDG4(sc.sph_nodes + 2 * (size_t)node + 1);
        const float hx = 0.5f * (n0.w - n0.x), hy = 0.5f * (n1.x - n0.y), hz = 0.5f * (n1.y - n0.z);
        const float D = fabsf(r.ox - 0.5f * (n0.x + n0.w)) + fabsf(r.oy - 0.5f * (n0.y + n1.x)) + fabsf(r.oz - 0.5f * (n0.z + n1.y)) + (hx + hy + hz);
        const float cmax = fmaxf(fmaxf(fmaxf(fabsf(n0.x), fabsf(n0.w)), fmaxf(fabsf(n0.y), fabsf(n1.x))), fmaxf(fabsf(n0.z), fabsf(n1.y)));
        const float m = 0.0014f * D + 3.814697265625e-6f * (cmax + omax);
        const float lx = (n0.x - m - r.ox) * dfx, ux = (n0.w + m - r.ox) * dfx;
        const float ly = (n0.y - m - r.oy) * dfy, uy = (n1.x + m - r.oy) * dfy;
        const float lz = (n0.z - m - r.oz) * dfz, uz = (n1.y + m - r.oz) * dfz;
        const float tmin = SQT_FMAX(SQT_FMAX(SQT_FMIN(lx, ux), SQT_FMIN(ly, uy)), SQT_FMIN(lz, uz));
        const float tmax = SQT_FMIN(SQT_FMIN(SQT_FMAX(lx, ux), SQT_FMAX(ly, uy)), SQT_FMAX(lz, uz));
        const uint32_t a = f2u(n1.z), b = f2u(n1.w);
        bool pop = true;
        const bool beyond = L.cur.tri >= 0 && tmin > 0.0f && tmin * dlen - 0.003f * D > L.cur.dist;
        if (!(tmin > tmax) && !beyond) {                        // the LINE meets the enlarged box (a NaN keeps the node), not too far away
            if (b & kLeaf) {
                const uint32_t cnt = b & ~kLeaf;
                for (uint32_t i = 0; i < cnt; ++i) {
                    const uint32_t k = sc.sph_order[a + i];
                    const float4 s0 = SQT_LDG4(sc.spheres + 2 * (size_t)k);
                    float t, dist;
                    if (ray_sphere(s0, r, t, dist)) {
                        const bool earlier = (uint32_t)L.cur.tri >= sc.n_tris && (int)(sc.n_tris + k) < L.cur.tri;
                        if (L.cur.tri < 0 || dist < L.cur.dist || (dist == L.cur.dist && earlier)) { L.cur.tri = (int)(sc.n_tris + k); L.cur.t = t; L.cur.dist = dist; }
                    }
                }
            } else {
                const uint32_t lowc = a & 0x3fffffffu, ax = a >> 30;
                const bool low_first = (ax == 0u ? r.dx : (ax == 1u ? r.dy : r.dz)) > 0.0f;
                if (sp < 32) { stack[sp++] = low_first ? b : lowc; node = low_first ? lowc : b; pop = false; }
                else {          // cannot happen with the balanced tree the library builds (depth <= 27); stay exact anyway
                    L.cur = fold_spheres(sc.spheres, sc.n_spheres, sc.n_tris, r, L.cur);
                    return;
                }
            }
        }
        if (pop) {
            if (sp == 0) return;
            node = stack[--sp];
        }
    }
}

// material index of surface `idx` (triangle in leaf order, or n_tris + sphere)
SQT_HD uint32_t surface_material(const SceneView &sc, int idx) {
    if ((uint32_t)idx >= sc.n_tris) return f2u(SQT_LDG4(sc.spheres + 2 * (size_t)((uint32_t)idx - sc.n_tris) + 1).x);
    return f2u(SQT_LDG4(sc.tris + 3 * (size_t)idx + 2).y);
}

// intersectBIH b = intersectBIH' (bounds b) (tree b)   (BIH.hs:101-102).  Expects L.r; fills df, safe, sgn.
template <bool COUNT>
SQT_HD void start_ray(const SceneView &sc, TravLane &L, Counters *cn) {
    if (COUNT) cn->rays += 1;
    L.cur.tri = -1; L.cur.t = 0.0f; L.cur.dist = 0.0f;
    L.sp = 0;
    L.dfx = XRCP(L.r.dx); L.dfy = XRCP(L.r.dy); L.dfz = XRCP(L.r.dz);
    const bool safe = sc.planes_finite && finite_f(L.dfx) && finite_f(L.dfy) && finite_f(L.dfz) && finite_f(L.r.dx) && finite_f(L.r.dy) &&
                      finite_f(L.r.dz) && finite_f(L.r.ox) && finite_f(L.r.oy) && finite_f(L.r.oz);
    const bool tame = safe && sc.leaf_cull && (fabsf(L.r.dx) + fabsf(L.r.dy) + fabsf(L.r.dz)) <= 2.0f &&
                      (fabsf(L.r.ox - sc.tame_c[0]) + fabsf(L.r.oy - sc.tame_c[1]) + fabsf(L.r.oz - sc.tame_c[2])) <= sc.tame_r;
    L.rf = (L.r.dx > 0.0f ? 1u : 0u) | (L.r.dy > 0.0f ? 2u : 0u) | (L.r.dz > 0.0f ? 4u : 0u) | (safe ? 0u : kRfUnsafe) | (tame ? kRfTame : 0u);
    L.tmin = 0.0f; L.tmax = 0.0f;
    if (sc.root_is_leaf) {                       // tree = Leaf: no box test at all (BIH.hs:105)
        L.child = 0u; L.i = (int)sc.n_tris - 1;
        if (COUNT) cn->tri_tests += sc.n_tris;
        if (sc.n_tris) L.state = ST_LEAF; else finish_ray(sc, L, LaneRay(L));
        return;
    }
    if (!slab_iv(sc.root_lo[0], sc.root_lo[1], sc.root_lo[2], sc.root_hi[0], sc.root_hi[1], sc.root_hi[2], L.r, L.dfx,
                 L.dfy, L.dfz, safe, L.tmin, L.tmax)) { finish_ray(sc, L, LaneRay(L)); return; }          // BIH.hs:112 at the root
    L.child = kTight; L.state = ST_DESC;              // the root's record is always looked at (tame rays)
}

// Entering Leaf `L.child` (index into the leaf array) (BIH.hs:105-109).
//
// Conservative leaf culling (not in the reference; exact by a forward error bound, derivation in DESIGN.md section 5).
// A triangle test can only return Just if |a| >= 1e-4 and the computed u, v, u+v pass their guards and t > 1e-4
// (Geometry.hs:117-142); then the ray passes within the bound of cull_margin of the triangle.  The leaf is skipped only
// if the ray misses the leaf's tight box enlarged by that margin (leaf_box_culled): no skipped triangle could have been
// accepted, so the traversal result is bit-identical (tests: culling on/off agree on every ray; both agree with the
// oracle).  Rays with a zero/non-finite direction component or reciprocal (`safe` false) are never culled.
template <bool COUNT, class RA>
SQT_HD void enter_step(const SceneView &sc, TravLane &L, const RA &ra, Counters *cn) {
    const float4 *lp = sc.leaves + 2 * (size_t)L.child;
    const float4 b0 = SQT_LDG4(lp), b1 = SQT_LDG4(lp + 1);
    const uint32_t w = f2u(b1.w), first = w & kLeafFirstMask;
    uint32_t count = w >> kLeafCountShift;
    L.cur.tri = -1;
    if (count == 0u) { L.state = ST_RET; return; }                        // empty leaf -> Nothing (BIH.hs:107)
    if (sc.leaf_cull && !(L.rf & kRfUnsafe)) {
        float dfx, dfy, dfz;
        ra.dfv(dfx, dfy, dfz);
        if (leaf_box_culled(b0, b1, ra.ray(), dfx, dfy, dfz)) {
            if (COUNT) cn->leaves_culled += 1;
            L.state = ST_RET;
            return;
        }
    }
    if (count == kLeafLong) count = f2u(SQT_LDG4(sc.tris + 3 * (size_t)first + 2).w);   // long leaf: count rides in its first triangle
    if (COUNT) cn->tri_tests += count;
    L.child = first;
    L.i = (int)count - 1;
    L.state = ST_LEAF;
}

// The literal path of a branch visit (rare: kSlow nodes and rays with a zero / denormal / non-finite
// component): both child boxes from the node's own box (BIH.hs:130-141), all six slabs each (Geometry.hs:166-177).
// Everything travels by value (a reference to the kernel's SceneView would force it into local memory).
SQT_COLD float4 desc_children_literal(const float4 *boxes, uint32_t node, float lmax, float rmin, int ax, float ox, float oy, float oz,
                                             float dx, float dy, float dz, float dfx, float dfy, float dfz, bool fast) {
    const float4 c0 = SQT_LDG4(boxes + 2 * (size_t)node), c1 = SQT_LDG4(boxes + 2 * (size_t)node + 1);
    Ray r; r.ox = ox; r.oy = oy; r.oz = oz; r.dx = dx; r.dy = dy; r.dz = dz;
    float4 iv;                                  // (left tmin, left tmax, right tmin, right tmax); hit <=> tmax > 0 && tmin < tmax
    slab_iv(c0.x, c0.y, c0.z, ax == 0 ? lmax : c0.w, ax == 1 ? lmax : c1.x, ax == 2 ? lmax : c1.y, r, dfx, dfy, dfz, fast, iv.x, iv.y);
    slab_iv(ax == 0 ? rmin : c0.x, ax == 1 ? rmin : c0.y, ax == 2 ? rmin : c0.z, c0.w, c1.x, c1.y, r, dfx, dfy, dfz, fast, iv.z, iv.w);
    return iv;
}

// Visit Branch L.child (BIH.hs:111-141 below the own-box test, which the parent already evaluated).
//
// Fast path (safe ray, node not kSlow).  Let t_lo[k], t_hi[k] be the six slab values of the node's box and
// near[k] = min(t_lo[k], t_hi[k]), far[k] = max(..): L.tmin = max_k near[k], L.tmax = min_k far[k] (Geometry.hs:175-176;
// without NaNs min/max are exact selections, so association does not matter).  The left box replaces hi[ax] by lmax,
// the right box lo[ax] by rmin (BIH.hs:130-141).  x -> (x - o)*df is monotone under round-to-nearest, so with
// lo[ax] <= lmax <= hi[ax] the value tl = (lmax - o)*df lies between t_lo[ax] and t_hi[ax]: for df > 0 the left box
// keeps near[ax] and lowers far[ax] to tl, hence tmin(left) = L.tmin, tmax(left) = min(L.tmax, tl); the right box
// raises near[ax] to tr and keeps far[ax]: tmin(right) = max(L.tmin, tr), tmax(right) = L.tmax.  For df < 0 left and
// right swap roles.  In both cases the child the reference calls `near` (left iff dir[ax] > 0, BIH.hs:124-127) gets
// (L.tmin, min(L.tmax, t_near_plane)) and the far child (max(L.tmin, t_far_plane), L.tmax) -- the same values (up to
// the sign of a zero, which no comparison sees) intersectsBB computes from all six slabs, at 2 subtractions,
// 2 multiplications, 2 min/max and 3 compares instead of 12 + 12 + 20 + 4.
template <bool COUNT, int STRIDE = 1, class RA>
SQT_HD void desc_step(const SceneView &sc, TravLane &L, const RA &ra, Counters *cn) {
    const uint32_t node = L.child & kIdxMask;
    const float4 q = SQT_LDG4(sc.nodes + (size_t)node);
    const bool slabs = (L.child & L.rf & kTight) != 0u;                     // known from the reference: both loads go out together
    float4 cs;
#ifdef __CUDA_ARCH__
    asm("" : "=f"(cs.x), "=f"(cs.y), "=f"(cs.z), "=f"(cs.w));                  // only read under `slabs`: no registers to initialise
#else
    cs = q;
#endif
    if (slabs) cs = SQT_LDG4(sc.slabs + (size_t)node);
    const uint32_t lb = f2u(q.z), rb = f2u(q.w);
    const int ax = (int)((lb >> kAxisShift) & 3u);
    const bool ltr = ((L.rf >> ax) & 1u) != 0u;                             // BIH.hs:127
    if (COUNT) { cn->branch_visits += 1; cn->child_box_tests += 2; }
    float n_min, n_max, f_min, f_max;                                       // intervals of the near / far child
    if (((lb | L.rf) & kSlow) == 0u) {                                      // node not kSlow and ray not kRfUnsafe
        const float o = ra.o(ax), df = ra.df(ax);
        const float tl = XMUL(XSUB(q.x, o), df), tr = XMUL(XSUB(q.y, o), df);
        n_min = L.tmin; n_max = SQT_FMIN(L.tmax, ltr ? tl : tr);
        f_min = SQT_FMAX(L.tmin, ltr ? tr : tl); f_max = L.tmax;
    } else {
        const Ray r = ra.ray();
        float dfx, dfy, dfz;
        ra.dfv(dfx, dfy, dfz);
        const float4 iv = desc_children_literal(sc.boxes, node, q.x, q.y, ax, r.ox, r.oy, r.oz, r.dx, r.dy, r.dz, dfx, dfy, dfz, !(L.rf & kRfUnsafe));
        n_min = ltr ? iv.x : iv.z; n_max = ltr ? iv.y : iv.w;
        f_min = ltr ? iv.z : iv.x; f_max = ltr ? iv.w : iv.y;
    }
    const uint32_t nref = (ltr ? lb : rb) & (kLeaf | kTight | kIdxMask), fref = (ltr ? rb : lb) & (kLeaf | kTight | kIdxMask);
    if (slabs) {
        // Subtree / leaf slabs (not in the reference; exact like the leaf culling, DESIGN.md section 5.1): every triangle below
        // a child lies inside the child's tight box, and an accepted hit lies within the a-priori margin of its triangle.  One
        // axis of that box, enlarged by the margin, is intersected with the child's interval: the interval only shrinks, so
        // the child's test -- and every test below it -- can only change from "hit" to "miss", and only where no triangle could
        // have been accepted.  A child that fails is treated like a child whose box the ray misses: the reference would have
        // visited it and got Nothing, which changes none of BIH.hs:113-126.
        const float n_lo = ltr ? cs.x : cs.z, n_hi = ltr ? cs.y : cs.w, f_lo = ltr ? cs.z : cs.x, f_hi = ltr ? cs.w : cs.y;
        const uint32_t ncode = f2u(n_lo) & 3u, fcode = f2u(f_lo) & 3u;
        if (COUNT) cn->leaves_culled += (n_max > 0.0f && n_min < n_max ? 1u : 0u) + (f_max > 0.0f && f_min < f_max ? 1u : 0u);
        if (ncode != kSlabNone) {
            const float o = ra.o((int)ncode), df = ra.df((int)ncode);
            const float t1 = (n_lo - o) * df, t2 = (n_hi - o) * df;
            n_min = SQT_FMAX(n_min, SQT_FMIN(t1, t2)); n_max = SQT_FMIN(n_max, SQT_FMAX(t1, t2));
        }
        if (fcode != kSlabNone) {
            const float o = ra.o((int)fcode), df = ra.df((int)fcode);
            const float t1 = (f_lo - o) * df, t2 = (f_hi - o) * df;
            f_min = SQT_FMAX(f_min, SQT_FMIN(t1, t2)); f_max = SQT_FMIN(f_max, SQT_FMAX(t1, t2));
        }
        if (COUNT) cn->leaves_culled -= (n_max > 0.0f && n_min < n_max ? 1u : 0u) + (f_max > 0.0f && f_min < f_max ? 1u : 0u);
    }
    const bool hit_n = n_max > 0.0f && n_min < n_max, hit_f = f_max > 0.0f && f_min < f_max;       // Geometry.hs:177
    if (!(hit_n || hit_f)) { L.cur.tri = -1; L.state = ST_RET; return; }
    if (hit_n && hit_f) {                       // phase A entry: the far child, its interval, the plane isClose compares with
        float4 e;
        e.x = u2f(fref | ((uint32_t)ax << kAxisShift)); e.y = f_min; e.z = f_max; e.w = ltr ? q.y : q.x;      // rmin : lmax
        L.stack[(size_t)L.sp * STRIDE] = e;
        L.sp += 1;
    }
    const uint32_t ref = hit_n ? nref : fref;
    L.tmin = hit_n ? n_min : f_min;
    L.tmax = hit_n ? n_max : f_max;
    L.child = ref & (kTight | kIdxMask);
    L.state = (ref & kLeaf) ? ST_ENTER : ST_DESC;
}

// One triangle of the leaf (BIH.hs:105-109): V.mapMaybe over the leaf's triangles, minimumBy (comparing dist).
// base-4.9 minimumBy = foldr1 min' with min' x y = GT -> y ; _ -> x : walk from the last triangle
// to the first, the earlier one wins unless it is strictly farther.
// the three 128-bit words of triangle `idx` (leaf order)
struct TriData { float4 a0, a1, a2; };
SQT_HD TriData tri_load(const SceneView &sc, uint32_t idx) {
    const float4 *p = sc.tris + 3 * (size_t)idx;
    TriData d; d.a0 = SQT_LDG4(p); d.a1 = SQT_LDG4(p + 1); d.a2 = SQT_LDG4(p + 2);
    return d;
}
// the fold step of minimumBy (comparing dist) for a candidate that comes EARLIER in the leaf than everything folded so far
SQT_HD void fold_earlier(Hit &cur, int tri, float t, float dist) {
    if (cur.tri < 0 || !cmp_gt(dist, cur.dist)) { cur.tri = tri; cur.t = t; cur.dist = dist; }
}
// test the already loaded triangle L.child + L.i and advance (split from the load so that callers can prefetch)
template <bool COUNT>
SQT_HD void tri_apply(TravLane &L, const Ray &r, const TriData &d, Counters *cn) {
    const uint32_t idx = L.child + (uint32_t)L.i;
    float t, dist;
    int stage;
    if (moller_trumbore(d.a0, d.a1, d.a2, r, t, dist, stage)) fold_earlier(L.cur, (int)idx, t, dist);
    if (COUNT) { cn->mt_pass_a += stage >= 1; cn->mt_pass_u += stage >= 2; cn->mt_pass_v += stage >= 3; cn->mt_accept += stage >= 4; }
    if (--L.i < 0) L.state = ST_RET;
}
template <bool COUNT>
SQT_HD void tri_step(const SceneView &sc, TravLane &L, Counters *cn) {
    const TriData d = tri_load(sc, L.child + (uint32_t)L.i);
    tri_apply<COUNT>(L, L.r, d, cn);
}
// A subtree returned `cur`: pop entries until one of them sends the ray into a far subtree (-> ST_DESC / ST_ENTER) or
// the stack is empty (-> ST_DONE).  Two kinds of entry, told apart by kPhaseB in word 0:
//   phase A : the NEAR subtree of a both-children-hit branch just returned; the entry names the far child, its
//             interval and the plane (rmin when leftToRight, else lmax) isClose compares the hit point with;
//   phase B : (tri | kPhaseB, t, dist), the parked near hit of a branch whose FAR subtree just returned.
template <int STRIDE = 1, class RA>
SQT_HD void ret_step(const SceneView &sc, TravLane &L, const RA &ra) {
    for (;;) {
        if (L.sp == 0) { finish_ray(sc, L, ra); return; }
        float4 &slot = L.stack[(size_t)(L.sp - 1) * STRIDE];
        const float4 e = slot;
        const uint32_t w = f2u(e.x);
        if (w & kPhaseB) {                                                  // far subtree returned: min' near far, near wins ties
            L.sp -= 1;
            if (L.cur.tri < 0 || !cmp_gt(e.z, L.cur.dist)) { L.cur.tri = (int)(w & ~kPhaseB); L.cur.t = e.y; L.cur.dist = e.z; }
            continue;
        }
        if (L.cur.tri >= 0) {
            const int ax = (int)((w >> kAxisShift) & 3u);
            const bool ltr = ((L.rf >> ax) & 1u) != 0u;                     // BIH.hs:127: the near child was left iff leftToRight
            const float p = XADD(ra.o(ax), XMUL(L.cur.t, ra.d(ax)));        // intersectPoint on ax
            const bool close = ltr ? (p < e.w) : (p > e.w);                 // BIH.hs:121-123
            if (close) { L.sp -= 1; continue; }
            float4 b;                                                       // park the near hit in the same slot
            b.x = u2f((uint32_t)L.cur.tri | kPhaseB); b.y = L.cur.t; b.z = L.cur.dist; b.w = 0.0f;
            slot = b;
        } else L.sp -= 1;
        L.tmin = e.y; L.tmax = e.z;
        L.child = w & (kTight | kIdxMask);
        L.state = (w & kLeaf) ? ST_ENTER : ST_DESC;
        return;
    }
}

// one lane alone, to completion (host emulation and the odd single ray)
template <bool COUNT>
SQT_HD Hit traverse(const SceneView &sc, const Ray &r, Counters *cn) {
    float4 stack[kStackEntries];
    TravLane L;
    L.stack = stack;
    L.r = r;
    start_ray<COUNT>(sc, L, cn);
    const LaneRay ra(L);
    while (L.state != ST_DONE) {
        if (L.state == ST_RET) ret_step(sc, L, ra);
        if (L.state == ST_DESC) desc_step<COUNT>(sc, L, ra, cn);
        if (L.state == ST_ENTER) enter_step<COUNT>(sc, L, ra, cn);
        if (L.state == ST_LEAF) tri_step<COUNT>(sc, L, cn);
        if (L.state == ST_SPH) sphere_step(sc, L, ra);
    }
    return L.cur;
}

// ------------------------------------------------------------------------------------- RNG
// Philox4x32-10; stream = the integer the reference hands to mkTFGen (Lib.hs:85-86), j = index of
// the Word32 in that generator's output.  counter = (stream lo, stream hi, j/4, "SQTR"), key = seed.
SQT_HD void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
#if defined(__CUDA_ARCH__)
        uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
#else
        uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t h0 = (uint32_t)(p0 >> 32), l0 = (uint32_t)p0, h1 = (uint32_t)(p1 >> 32), l1 = (uint32_t)p1;
#endif
        uint32_t n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
        c0 = n0; c1 = l1; c2 = n2; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// Lib.hs:183-188 at (0,1): Word32 -> Float (round to nearest) / 2^32 ; inclusive of 1.0
SQT_HD float random_r01(uint32_t n) {
#if defined(__CUDA_ARCH__)
    return XMUL(__uint2float_rn(n), 2.3283064365386963e-10f);
#else
    return XMUL((float)n, 2.3283064365386963e-10f);
#endif
}

// ------------------------------------------------------------------------------------ trig
// "sqt trig" (DESIGN.md section 6): plain binary32 polynomials, fixed operation order, no FMA, so the
// device and the oracle's restatement agree bit for bit.  Arguments: x in [0, 2*pi].
SQT_HD void sqt_sincos(float x, float &s_out, float &c_out) {
    const int k = (int)XADD(XMUL(x, 0.63661975f), 0.5f);
    const float kf = (float)k;
    const float r = XSUB(XSUB(XSUB(x, XMUL(kf, 1.5703125f)), XMUL(kf, 4.837512969970703125e-4f)),
                         XMUL(kf, 7.54978995489188216e-8f));
    const float z = XMUL(r, r);
    float s = XADD(XMUL(-1.9515295891e-4f, z), 8.3321608736e-3f);
    s = XSUB(XMUL(s, z), 1.6666654611e-1f);
    s = XADD(XMUL(XMUL(s, z), r), r);
    float c = XSUB(XMUL(2.443315711809948e-5f, z), 1.388731625493765e-3f);
    c = XADD(XMUL(c, z), 4.166664568298827e-2f);
    c = XMUL(XMUL(c, z), z);
    c = XSUB(c, XMUL(0.5f, z));
    c = XADD(c, 1.0f);
    const int q = k & 3;
    s_out = q == 0 ? s : (q == 1 ? c : (q == 2 ? -s : -c));
    c_out = q == 0 ? c : (q == 1 ? -s : (q == 2 ? -c : s));
}
SQT_HD float sqt_asin_core(float x, float z) {
    float p = XADD(XMUL(4.2163199048e-2f, z), 2.4181311049e-2f);
    p = XADD(XMUL(p, z), 4.5470025998e-2f);
    p = XADD(XMUL(p, z), 7.4953002686e-2f);
    p = XADD(XMUL(p, z), 1.6666752422e-1f);
    return XADD(XMUL(XMUL(p, z), x), x);
}
SQT_HD float sqt_acos(float x) {
    if (x < -0.5f) {
        const float z = XMUL(0.5f, XADD(1.0f, x)), y = XSQRT(z);
        return XSUB(3.14159265358979323846f, XMUL(2.0f, sqt_asin_core(y, z)));
    }
    if (x > 0.5f) {
        const float z = XMUL(0.5f, XSUB(1.0f, x)), y = XSQRT(z);
        return XMUL(2.0f, sqt_asin_core(y, z));
    }
    return XSUB(1.57079632679489661923f, sqt_asin_core(x, XMUL(x, x)));
}
SQT_HD float sqt_atan(float x) {   // x >= 0
    float y;
    if (x > 2.414213562373095f) { y = 1.57079632679489661923f; x = -XDIV(1.0f, x); }
    else if (x > 0.4142135623730950f) { y = 0.78539816339744830962f; x = XDIV(XSUB(x, 1.0f), XADD(x, 1.0f)); }
    else y = 0.0f;
    const float z = XMUL(x, x);
    float p = XSUB(XMUL(8.05374449538e-2f, z), 1.38776856032e-1f);
    p = XADD(XMUL(p, z), 1.99777106478e-1f);
    p = XSUB(XMUL(p, z), 3.33329491539e-1f);
    return XADD(y, XADD(XMUL(XMUL(p, z), x), x));
}

// -------------------------------------------------------------------------------- shading
struct RenderParams {
    int rows, cols, xdiv, ydiv, seed_stride, spp, max_depth, mode;
    unsigned long long seed;
    int rank, world, split_samples, primary_reuse;
    float cam_pos[3], cam_rot[9];
    int terminate_on_black;     // host proved C*L stays finite: a surface with surfColor == 0 ends the path exactly
    int lens, jitter;           // camera sampling (sqt_set_lens): a lens is set; box-filtered pixels
    float aperture, focus;      // lens radius (0 = pinhole) and focus distance
};

// makeRay (Lib.hs:107-114) + rotVert (Geometry.hs:104-107: row vector x matrix, sum = foldl (+) 0)
SQT_HD Ray make_ray(const RenderParams &p, int y, int x) {
    const float ww = (float)p.xdiv, hh = (float)p.ydiv;
    const float xo = XDIV(XSUB((float)x, XDIV(ww, 2.0f)), ww);
    const float yo = XDIV(XSUB(XDIV(hh, 2.0f), (float)y), hh);
    const float *R = p.cam_rot;
    Ray r;
    r.ox = p.cam_pos[0]; r.oy = p.cam_pos[1]; r.oz = p.cam_pos[2];
    r.dx = XADD(XADD(XADD(0.0f, XMUL(1.0f, R[0])), XMUL(xo, R[3])), XMUL(yo, R[6]));
    r.dy = XADD(XADD(XADD(0.0f, XMUL(1.0f, R[1])), XMUL(xo, R[4])), XMUL(yo, R[7]));
    r.dz = XADD(XADD(XADD(0.0f, XMUL(1.0f, R[2])), XMUL(xo, R[5])), XMUL(yo, R[8]));
    return r;
}

// the primary ray of the sample with generator seed `s` (spp*(x + y*seed_stride) + k) in a frame with a lens set: jittered
// sample point, then a thin-lens offset, in the order include/sqt.h (sqt_set_lens) writes down
SQT_HD Ray lens_ray(const RenderParams &p, int y, int x, unsigned long long s) {
    uint32_t w[4];
    philox4x32_10((uint32_t)s, (uint32_t)(s >> 32), 0u, 0x4C545153u, (uint32_t)p.seed, (uint32_t)(p.seed >> 32), w);
    const float jx = p.jitter ? XSUB(random_r01(w[0]), 0.5f) : 0.0f;
    const float jy = p.jitter ? XSUB(random_r01(w[1]), 0.5f) : 0.0f;
    const float fx = XADD((float)x, jx), fy = XADD((float)y, jy);
    const float ww = (float)p.xdiv, hh = (float)p.ydiv;
    const float xo = XDIV(XSUB(fx, XDIV(ww, 2.0f)), ww);
    const float yo = XDIV(XSUB(XDIV(hh, 2.0f), fy), hh);
    const float *R = p.cam_rot;
    Ray r;
    r.ox = p.cam_pos[0]; r.oy = p.cam_pos[1]; r.oz = p.cam_pos[2];
    r.dx = XADD(XADD(XADD(0.0f, XMUL(1.0f, R[0])), XMUL(xo, R[3])), XMUL(yo, R[6]));
    r.dy = XADD(XADD(XADD(0.0f, XMUL(1.0f, R[1])), XMUL(xo, R[4])), XMUL(yo, R[7]));
    r.dz = XADD(XADD(XADD(0.0f, XMUL(1.0f, R[2])), XMUL(xo, R[5])), XMUL(yo, R[8]));
    if (p.aperture != 0.0f) {
        const float rad = XMUL(p.aperture, XSQRT(random_r01(w[2])));
        const float th = XMUL(6.2831855f, random_r01(w[3]));
        float sn, cs;
        sqt_sincos(th, sn, cs);
        const float a = XMUL(rad, cs), b = XMUL(rad, sn), inv_f = XDIV(1.0f, p.focus);
        const float offx = XADD(XMUL(a, R[3]), XMUL(b, R[6]));
        const float offy = XADD(XMUL(a, R[4]), XMUL(b, R[7]));
        const float offz = XADD(XMUL(a, R[5]), XMUL(b, R[8]));
        r.ox = XADD(r.ox, offx); r.oy = XADD(r.oy, offy); r.oz = XADD(r.oz, offz);
        r.dx = XSUB(r.dx, XMUL(offx, inv_f)); r.dy = XSUB(r.dy, XMUL(offy, inv_f)); r.dz = XSUB(r.dz, XMUL(offz, inv_f));
    }
    return r;
}

SQT_HD float hs_signum(float x) { return x > 0.0f ? 1.0f : (x < 0.0f ? -1.0f : x); }

// bounceRay (Lib.hs:155-160) at a hit on triangle `tri` (leaf order) with hit parameter t.  The caller
// drew x = draw j (scatter iff reflective < x) and, for a scatter, v = draw j+1: scatter reuses x as the
// azimuth draw and takes v as the polar draw (SURVEY A.4).  Returns the new ray; origin = intersectPoint.
SQT_HD Ray bounce_ray(const SceneView &sc, const Ray &in, int tri, float t, bool scatter, float x, float v) {
    Ray out;
    out.ox = XADD(in.ox, XMUL(t, in.dx)); out.oy = XADD(in.oy, XMUL(t, in.dy)); out.oz = XADD(in.oz, XMUL(t, in.dz));
    float nx, ny, nz;
    if ((uint32_t)tri >= sc.n_tris) {           // extension: sphere, normal = intersectPoint - center
        const float4 s0 = SQT_LDG4(sc.spheres + 2 * (size_t)((uint32_t)tri - sc.n_tris));
        nx = XSUB(out.ox, s0.x); ny = XSUB(out.oy, s0.y); nz = XSUB(out.oz, s0.z);
    } else {
        const float4 *p = sc.tris + 3 * (size_t)tri;
        const float4 a0 = SQT_LDG4(p), a1 = SQT_LDG4(p + 1), a2 = SQT_LDG4(p + 2);
        const float e1x = a0.w, e1y = a1.x, e1z = a1.y, e2x = a1.z, e2y = a1.w, e2z = a2.x;
        // normal = (b - a) `cross` (c - a)   Geometry.hs:79-80
        nx = XSUB(XMUL(e1y, e2z), XMUL(e1z, e2y));
        ny = XSUB(XMUL(e1z, e2x), XMUL(e1x, e2z));
        nz = XSUB(XMUL(e1x, e2y), XMUL(e1y, e2x));
    }
    if (scatter) {                              // scatterRay, Lib.hs:166-172 ; randomVector Lib.hs:192-198
        const float th = XMUL(6.28318530717958647692f, x);             // 2 * pi * u
        const float ph = sqt_acos(XSUB(XMUL(2.0f, v), 1.0f));
        float sth, cth, sph, cph;
        sqt_sincos(th, sth, cth);
        sqt_sincos(ph, sph, cph);
        const float ndx = XMUL(cth, sph), ndy = XMUL(sth, sph), ndz = cph;
        const float so = hs_signum(dot3(in.dx, in.dy, in.dz, nx, ny, nz));
        const float sn = hs_signum(dot3(ndx, ndy, ndz, nx, ny, nz));
        const bool flip = (so == sn);
        out.dx = flip ? -ndx : ndx; out.dy = flip ? -ndy : ndy; out.dz = flip ? -ndz : ndz;
    } else {                                    // reflectRay, Lib.hs:176-181
        const float nn = XSQRT(dot3(nx, ny, nz, nx, ny, nz));
        const float ux = XDIV(nx, nn), uy = XDIV(ny, nn), uz = XDIV(nz, nn);
        const float k = XMUL(2.0f, dot3(ux, uy, uz, in.dx, in.dy, in.dz));
        out.dx = XSUB(in.dx, XMUL(k, ux)); out.dy = XSUB(in.dy, XMUL(k, uy)); out.dz = XSUB(in.dz, XMUL(k, uz));
    }
    return out;
}

// rgbFloatToPixelRGB (Lib.hs:93-104); floor :: Float -> Word8 wraps through Integer, NaN -> 0
SQT_HD uint8_t to_w8(float s255) {
    if (s255 != s255) return 0;
    const float f = floorf(s255);
    long long w = (fabsf(f) < 9.0e18f) ? (long long)f : 0;
    uint32_t b = (uint32_t)((unsigned long long)w & 0xffull);
    return (uint8_t)(b < 255u ? b : 255u);
}
SQT_HD void tone_map(float r, float g, float b, uint8_t out[3]) {
    const float maxc = hs_max(hs_max(r, g), b), minc = hs_min(hs_min(r, g), b);
    const float lightness = XMUL(0.5f, XADD(maxc, minc));
    const float intensity = XDIV(sqt_atan(lightness), 1.57079632679489661923f);
    const float k = XDIV(intensity, maxc);
    out[0] = to_w8(XMUL(XMUL(k, r), 255.0f));
    out[1] = to_w8(XMUL(XMUL(k, g), 255.0f));
    out[2] = to_w8(XMUL(XMUL(k, b), 255.0f));
}

}  // namespace sqt
