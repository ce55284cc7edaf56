// sqt_paths.cuh -- what a lane does BETWEEN rays: the integrator (renderPixel / raytrace / raycast,
// Lib.hs:79-151) and the two simpler ray sources (batched intersect, primary hits), written as "policies"
// with one entry point:
//
//     regen(sc, L, cn)   called when L.state == ST_DONE: consume the hit in L.cur (if a ray was in flight),
//                        then put the lane's next ray into L.r and start it -- or set ST_EXIT when the lane
//                        has no more work.
//
// k_intersect_batch, k_primary and k_raycast (sqt_kernels.cuh) run one warp-synchronous loop around these: regen for
// lanes that are done, traversal steps for lanes that are descending/returning, triangle tests for lanes inside a leaf
// (sqt_core.cuh).  The integrator kernel, k_paths_pool, keeps its rays in shared-memory pools and regenerates them with
// path_regen_warp.  Rays are independent, so any schedule yields the same per-ray results; tests/emu runs each lane to
// completion on the host with the same functions (run_lane), the integrator as PathPolicy.
//
// Integrator layout: the work item is one SAMPLE of one pixel; a frame is rendered in rounds of S samples per pixel
// whose radiances go to a sample buffer and are then added to the per-pixel sums strictly in sample order
// (accumulate_slot), so the sum is the reference's sequential `sum = foldl (+) 0` (Lib.hs:88).  A lane (or pool slot)
// whose path ends (miss, depth cut, black surface) fetches its next sample right away (path regeneration).
#pragma once
#include "sqt_core.cuh"

namespace sqt {

// per-lane tallies; 32 bits on the device (a lane traces a few thousand rays per launch; the warp sums them in 64 bits)
#if defined(__CUDA_ARCH__)
typedef unsigned int stat_t;
#else
typedef unsigned long long stat_t;
#endif
struct PathStats { stat_t rays, samples, primary_reused; };

// pixel owned by this rank for work item w (pixel-group partition: groups of 32 consecutive pixels,
// round-robin over ranks).  Returns -1 for the padding of the last group.
SQT_HD long long work_to_pixel(const RenderParams &p, long long w) {
    long long pix;
    if (p.world <= 1 || p.split_samples) pix = w;
    else pix = (((w >> 5) * (long long)p.world + (long long)p.rank) << 5) | (w & 31);
    return pix < (long long)p.rows * (long long)p.cols ? pix : -1;
}
SQT_HD long long work_items(const RenderParams &p) {
    const long long npix = (long long)p.rows * (long long)p.cols;
    if (p.world <= 1 || p.split_samples) return npix;
    const long long groups = (npix + 31) >> 5;
    const long long mine = groups > p.rank ? (groups - p.rank + p.world - 1) / p.world : 0;
    return mine << 5;
}
SQT_HD void sample_range(const RenderParams &p, int &k0, int &k1) {
    k0 = 0; k1 = p.spp;
    if (p.world > 1 && p.split_samples) {
        k0 = (int)((long long)p.spp * p.rank / p.world);
        k1 = (int)((long long)p.spp * (p.rank + 1) / p.world);
    }
}

constexpr uint32_t kMatEmits = 1u;       // emissive *^ emitColor != 0
constexpr uint32_t kMatBlack = 2u;       // surfColor == (0,0,0)

// radiance of one finished path: L_j = surfColor_j * L_{j+1} + emissive_j *^ emitColor_j, evaluated from
// the deepest shaded bounce outwards exactly like the recursion of Lib.hs:135-137 (L beyond the end = black).
SQT_HD void fold_path(const SceneView &sc, const uint16_t *pm, int last, float &lr, float &lg, float &lb) {
    lr = 0.0f; lg = 0.0f; lb = 0.0f;
    for (int b = last; b >= 0; --b) {
        const float4 *m = sc.mats + 3 * (size_t)pm[b];
        const float4 m0 = SQT_LDG4(m), m2 = SQT_LDG4(m + 2);
        lr = XADD(XMUL(m0.y, lr), m2.x);
        lg = XADD(XMUL(m0.z, lg), m2.y);
        lb = XADD(XMUL(m0.w, lb), m2.z);
    }
}

// ------------------------------------------------------------------------------- raytrace policy
// Work item = one SAMPLE of one pixel (Lib.hs:84: `raytrace r scene ray 0` for generator r).  The samples of a
// frame are rendered in rounds of `S` (a power of two) samples per pixel; within a round, item w is sample
// k0 + (w mod S) of the pixel in slot (w div S) of the round's pixel list.  A path's radiance goes to a sample
// buffer (ks-major: [ks][slot][3]); `accumulate_slot` then adds the S values of a pixel to its running sum in
// sample order, continuing from the previous round -- so the per-pixel sum is the reference's sequential
// `sum = foldl (+) 0` (Lib.hs:88) although the samples of a pixel are traced by different lanes.
struct RoundInfo {
    const int *pixel_list;     // slot -> pixel (hit pixels from k_primary), or nullptr: slot -> work_to_pixel(slot)
    const int2 *prim;          // per pixel (tri, t bits) of the primary hit, or nullptr when primary reuse is off
    float *sbuf;               // sample buffer of this round, zero-filled
    long long n_slots;         // slots in use
    long long slot_stride;     // allocation stride of one ks plane (>= n_slots)
    int log2_s;                // S = 1 << log2_s
    int k0, k1;                // samples [k0, k1) of this round, k1 - k0 <= S
};

// per-ray integrator state (what a lane -- or a pool slot -- has to remember between two rays of one path)
struct PathRay {
    uint32_t sidx;                           // index of the current sample in sbuf (without the *3)
    int j;                                   // bounce index of the hit being shaded
    unsigned long long stream;               // generator seed of the current sample: spp*(x + y*w) + k
    float saved_r; int saved_j;              // draw j+1 of a scatter is draw j of the next bounce (SURVEY A.4)
    bool any_emit, in_flight;
};
SQT_HD void path_ray_init(PathRay &q) { q.sidx = 0u; q.j = 0; q.stream = 0ull; q.saved_r = 0.0f; q.saved_j = -1; q.any_emit = false; q.in_flight = false; }

SQT_HD float path_draw(const RenderParams &p, PathRay &q, uint32_t jj) {
    if ((int)jj == q.saved_j) return q.saved_r;
    uint32_t w[4];
    philox4x32_10((uint32_t)q.stream, (uint32_t)(q.stream >> 32), jj >> 2, 0x52545153u, (uint32_t)p.seed, (uint32_t)(p.seed >> 32), w);
    const uint32_t k = jj & 3u;
    return random_r01(k == 0 ? w[0] : (k == 1 ? w[1] : (k == 2 ? w[2] : w[3])));
}

// ---- the stages of path regeneration.  path_regen strings them together for one lane; path_regen_warp (device only)
//      runs every stage for all regenerating lanes of a warp at once, so that the expensive stages (bounce, start_ray)
//      execute once with many lanes instead of once per control-flow path with a few.
struct RegenLane {
    int htri; float ht;          // the hit to shade (htri < 0: none)
    float refl;                  // `reflective` of the shaded material (Lib.hs:157)
};

// A: the ray of Lib.hs:131 came back.  Returns true when the path is over (no hit).
SQT_HD bool path_consume(PathRay &q, PathStats &st, const TravLane &L, RegenLane &g) {
    g.htri = -1; g.ht = 0.0f; g.refl = 0.0f;
    if (!q.in_flight) return false;
    q.in_flight = false;
    st.rays += 1;
    if (L.cur.tri >= 0) { g.htri = L.cur.tri; g.ht = L.cur.t; q.j += 1; return false; }
    return true;
}
// B1: the sample is finished: store its radiance (samples that never met an emitter are exactly +0, which the
//     zero-filled buffer already holds)
SQT_HD void path_finish(const SceneView &sc, const RoundInfo &rd, const uint16_t *pm, const PathRay &q, PathStats &st, RegenLane &g) {
    if (q.any_emit) {
        float lr, lg, lb;
        fold_path(sc, pm, q.j, lr, lg, lb);
        rd.sbuf[3 * (size_t)q.sidx] = lr; rd.sbuf[3 * (size_t)q.sidx + 1] = lg; rd.sbuf[3 * (size_t)q.sidx + 2] = lb;
    }
    st.samples += 1;
    g.htri = -1;
}
// B2: next sample.  0 = the queue is empty, 1 = item skipped (padding / beyond the sample range) -- fetch again,
//     2 = the primary hit is known (shade it), 3 = the primary ray has to be traced (primary reuse off, or a lens frame:
//     LENS, whose primary ray is the sample's own, lens_ray)
enum : int { NS_EMPTY = 0, NS_SKIP = 1, NS_SHADE = 2, NS_TRACE = 3 };
template <bool LENS, class Fetch>
SQT_HD int path_next_sample(const RenderParams &p, const RoundInfo &rd, Fetch &fetch, PathStats &st, PathRay &q, TravLane &L, RegenLane &g) {
    const long long w = fetch();
    if (w < 0) return NS_EMPTY;
    const long long slot = w >> rd.log2_s;
    const int ks = (int)(w & ((1ll << rd.log2_s) - 1));
    const int k = rd.k0 + ks;
    if (k >= rd.k1) return NS_SKIP;
    const long long pixel = rd.pixel_list ? (long long)rd.pixel_list[slot] : work_to_pixel(p, slot);
    if (pixel < 0) return NS_SKIP;
    const int py = (int)(pixel / p.cols), px = (int)(pixel % p.cols);
    q.stream = (unsigned long long)p.spp * ((unsigned long long)px + (unsigned long long)py * (unsigned long long)p.seed_stride)
               + (unsigned long long)k;
    q.sidx = (uint32_t)((long long)ks * rd.slot_stride + slot);
    q.any_emit = false; q.saved_j = -1;
    if constexpr (LENS) {
        L.r = lens_ray(p, py, px, q.stream);
        q.j = -1; q.in_flight = true;
        return NS_TRACE;
    }
    L.r = make_ray(p, py, px);
    if (rd.prim) {
        // the primary ray is the same for every sample of a pixel (Lib.hs:81): its hit was traced once
        const int2 ph = rd.prim[pixel];
        g.htri = ph.x; g.ht = u2f((uint32_t)ph.y); q.j = 0;
        st.primary_reused += 1;
        return NS_SHADE;
    }
    q.j = -1; q.in_flight = true;                     // primary reuse off: trace it again like Lib.hs:84 does
    return NS_TRACE;
}
// C: shade the hit of bounce j (raytrace, Lib.hs:127-137).  Returns true when the path goes on with a bounce.
SQT_HD bool path_shade(const SceneView &sc, const RenderParams &p, uint16_t *pm, PathRay &q, RegenLane &g) {
    const uint32_t mat = surface_material(sc, g.htri);
    pm[q.j] = (uint16_t)mat;
    const float4 *mp = sc.mats + 3 * (size_t)mat;
    const float4 m0 = SQT_LDG4(mp);
    const uint32_t mflags = f2u(SQT_LDG4(mp + 2).w);
    q.any_emit = q.any_emit || (mflags & kMatEmits);
    g.refl = m0.x;
    return !((q.j + 1 > p.max_depth - 1) || (p.terminate_on_black && (mflags & kMatBlack)));
}
// D: bounceRay (Lib.hs:155-160); L.r is the ray that produced the hit and becomes the bounced ray
SQT_HD void path_bounce(const SceneView &sc, const RenderParams &p, PathRay &q, TravLane &L, const RegenLane &g) {
    const float x = path_draw(p, q, (uint32_t)q.j);
    float v = 0.0f;
    const bool scatter = g.refl < x;
    if (scatter) { v = path_draw(p, q, (uint32_t)q.j + 1u); q.saved_r = v; q.saved_j = q.j + 1; } else q.saved_j = -1;
    L.r = bounce_ray(sc, L.r, g.htri, g.ht, scatter, x, v);
    q.in_flight = true;
}

// called when L.state == ST_DONE: consume the hit (if a ray was in flight), then shade / start the next sample until
// the slot has a ray to trace (-> start_ray) or the queue is empty (-> ST_EXIT).  pm: SQT_MAX_DEPTH entries of
// ray-private memory holding the material of every shaded bounce of the current path.
template <bool COUNT, bool LENS, class Fetch>
SQT_HD void path_regen(const SceneView &sc, const RenderParams &p, const RoundInfo &rd, Fetch &fetch, PathStats &st, PathRay &q,
                       uint16_t *pm, TravLane &L, Counters *cn) {
    RegenLane g;
    bool path_over = path_consume(q, st, L, g);
    for (;;) {
        if (path_over) { path_finish(sc, rd, pm, q, st, g); path_over = false; }
        if (g.htri < 0) {
            const int ns = path_next_sample<LENS>(p, rd, fetch, st, q, L, g);
            if (ns == NS_EMPTY) { L.state = ST_EXIT; return; }
            if (ns == NS_SKIP) continue;
            if (ns == NS_TRACE) { start_ray<COUNT>(sc, L, cn); return; }
        }
        if (!path_shade(sc, p, pm, q, g)) { path_over = true; continue; }
        path_bounce(sc, p, q, L, g);
        start_ray<COUNT>(sc, L, cn);
        return;
    }
}

#if defined(__CUDACC__)
// The same for all lanes of a warp at once (`mine`: this lane is ST_DONE): every stage is one convergent block, the
// loop is closed by a warp vote.  Per lane the sequence of stage calls is exactly path_regen's.
template <bool COUNT, bool LENS, class Fetch>
__device__ __forceinline__ void path_regen_warp(const SceneView &sc, const RenderParams &p, const RoundInfo &rd, Fetch &fetch, PathStats &st,
                                                PathRay &q, uint16_t *pm, TravLane &L, Counters *cn, bool mine) {
    RegenLane g;
    g.htri = -1; g.ht = 0.0f; g.refl = 0.0f;
    bool fin = false, nxt = false, shd = false, bnc = false, trace = false;
    if (mine) {
        fin = path_consume(q, st, L, g);
        nxt = !fin && g.htri < 0;
        shd = g.htri >= 0;
    }
    for (;;) {
        if (fin) { path_finish(sc, rd, pm, q, st, g); fin = false; nxt = true; }
        if (nxt) {
            const int ns = path_next_sample<LENS>(p, rd, fetch, st, q, L, g);
            if (ns == NS_EMPTY) { L.state = ST_EXIT; nxt = false; }
            else if (ns == NS_SHADE) { nxt = false; shd = true; }
            else if (ns == NS_TRACE) { nxt = false; trace = true; }
        }
        if (shd) {
            shd = false;
            if (path_shade(sc, p, pm, q, g)) bnc = true; else fin = true;
        }
        if (!__any_sync(0xffffffffu, fin || nxt)) break;
    }
    if (bnc) path_bounce(sc, p, q, L, g);
    if (bnc || trace) start_ray<COUNT>(sc, L, cn);
}
#endif

// The integrator as one lane's policy (run_lane in the host build, the reference schedule of k_paths_pool).
// LENS: a frame with a lens set (sqt_set_lens) -- a compile-time choice, so that the pinhole kernels stay as they are
template <class Fetch, bool LENS = false>
struct PathPolicy {
    const RenderParams &p;
    const RoundInfo &rd;
    Fetch &fetch;
    PathStats &st;
    PathRay q;
    uint16_t *pm;
    SQT_HD PathPolicy(const RenderParams &p_, const RoundInfo &rd_, Fetch &f_, PathStats &st_, uint16_t *pm_)
        : p(p_), rd(rd_), fetch(f_), st(st_), pm(pm_) { path_ray_init(q); }
    template <bool COUNT>
    SQT_HD void regen(const SceneView &sc, TravLane &L, Counters *cn) { path_regen<COUNT, LENS>(sc, p, rd, fetch, st, q, pm, L, cn); }
};

// avg-in-order part of renderPixel (Lib.hs:87-88): add the round's samples of one slot to the pixel's running sum,
// strictly in sample order.
SQT_HD void accumulate_slot(const RenderParams &p, const RoundInfo &rd, long long slot, float *accum) {
    const long long pixel = rd.pixel_list ? (long long)rd.pixel_list[slot] : work_to_pixel(p, slot);
    if (pixel < 0) return;
    float sr = accum[3 * pixel], sg = accum[3 * pixel + 1], sb = accum[3 * pixel + 2];
    const int n = rd.k1 - rd.k0;
    for (int ks = 0; ks < n; ++ks) {
        const long long i = 3 * ((long long)ks * rd.slot_stride + slot);
        sr = XADD(sr, rd.sbuf[i]); sg = XADD(sg, rd.sbuf[i + 1]); sb = XADD(sb, rd.sbuf[i + 2]);
    }
    accum[3 * pixel] = sr; accum[3 * pixel + 1] = sg; accum[3 * pixel + 2] = sb;
}
// the same for a progressive frame, which also keeps the per-pixel second moment: s2 = s2 + x*x over the sample
// radiances x, every operation rounded to binary32, in sample order
SQT_HD void accumulate_m2_slot(const RenderParams &p, const RoundInfo &rd, long long slot, float *accum, float *m2) {
    const long long pixel = rd.pixel_list ? (long long)rd.pixel_list[slot] : work_to_pixel(p, slot);
    if (pixel < 0) return;
    float sr = accum[3 * pixel], sg = accum[3 * pixel + 1], sb = accum[3 * pixel + 2];
    float qr = m2[3 * pixel], qg = m2[3 * pixel + 1], qb = m2[3 * pixel + 2];
    const int n = rd.k1 - rd.k0;
    for (int ks = 0; ks < n; ++ks) {
        const long long i = 3 * ((long long)ks * rd.slot_stride + slot);
        const float xr = rd.sbuf[i], xg = rd.sbuf[i + 1], xb = rd.sbuf[i + 2];
        sr = XADD(sr, xr); sg = XADD(sg, xg); sb = XADD(sb, xb);
        qr = XADD(qr, XMUL(xr, xr)); qg = XADD(qg, XMUL(xg, xg)); qb = XADD(qb, XMUL(xb, xb));
    }
    accum[3 * pixel] = sr; accum[3 * pixel + 1] = sg; accum[3 * pixel + 2] = sb;
    m2[3 * pixel] = qr; m2[3 * pixel + 1] = qg; m2[3 * pixel + 2] = qb;
}
// the per-pixel error terms of include/sqt.h for sums s1 and second moments s2 after n >= 2 samples, in fp64 and in the
// header's order: e2 (the squared standard error) and m (the mean's channel sum); returns true when a channel's variance
// is NaN.  Shared by the convergence test and the denoiser's variance.
SQT_HD bool pixel_error(const float *s1, const float *s2, int n, double &e2, double &m) {
    const double dn = (double)n;
    double mu[3], v[3];
    bool nan = false;
    for (int c = 0; c < 3; ++c) {
        const double a = (double)s1[c], q = (double)s2[c];
        mu[c] = a / dn;
        const double vc = (q - a * mu[c]) / (dn - 1.0);
        nan = nan || vc != vc;
        v[c] = vc > 0.0 ? vc : 0.0;
    }
    e2 = (v[0] + v[1] + v[2]) / dn; m = mu[0] + mu[1] + mu[2];
    return nan;
}
// the convergence test of an adaptive frame (sqt_render_retire, include/sqt.h) for one pixel; false whenever a NaN turns
// up on the way
SQT_HD bool retire_test(const float *s1, const float *s2, int n, double rel_tol, double abs_tol) {
    double e2, m;
    bool nan = pixel_error(s1, s2, n, e2, m);
    const double tr = rel_tol * m;
    const double t = tr > abs_tol ? tr : abs_tol;
    nan = nan || m != m || tr != tr;
    return !nan && e2 < t * t;
}

// samples per pixel per round: the largest power of two <= spp whose sample buffer (slots * S * 12 B) fits the budget
SQT_HD int round_log2_s(long long slots, int n_samples, long long budget_bytes) {
    int l = 0;
    while ((1 << (l + 1)) <= n_samples && slots * (long long)(1 << (l + 1)) * 12ll <= budget_bytes) ++l;
    return l;
}

// ------------------------------------------------------------------------------- batched intersect policy
// Scene.intersect over a ray batch (Geometry.hs:64): lane takes rays idx, idx + stride, ...
struct BatchPolicy {
    const float *org, *dir;
    long long n, idx, stride;
    int *tri_out; float *dist_out, *point_out;
    PathStats &st;
    bool in_flight = false;
    SQT_HD BatchPolicy(const float *o, const float *d, long long n_, long long first, long long stride_, int *t, float *di,
                       float *po, PathStats &st_)
        : org(o), dir(d), n(n_), idx(first), stride(stride_), tri_out(t), dist_out(di), point_out(po), st(st_) {}

    template <bool COUNT>
    SQT_HD void regen(const SceneView &sc, TravLane &L, Counters *cn) {
        if (in_flight) {
            in_flight = false;
            st.rays += 1;
            const bool hit = L.cur.tri >= 0;
            // triangles report their position in the parsed list, sphere k reports n_tris + k
            tri_out[idx] = !hit ? -1 : ((uint32_t)L.cur.tri >= sc.n_tris ? L.cur.tri : (int)f2u(SQT_LDG4(sc.tris + 3 * (size_t)L.cur.tri + 2).z));
            if (dist_out) dist_out[idx] = hit ? L.cur.dist : 0.0f;
            if (point_out) {
                point_out[3 * idx] = hit ? XADD(L.r.ox, XMUL(L.cur.t, L.r.dx)) : 0.0f;
                point_out[3 * idx + 1] = hit ? XADD(L.r.oy, XMUL(L.cur.t, L.r.dy)) : 0.0f;
                point_out[3 * idx + 2] = hit ? XADD(L.r.oz, XMUL(L.cur.t, L.r.dz)) : 0.0f;
            }
            idx += stride;
        }
        if (idx >= n) { L.state = ST_EXIT; return; }
        L.r.ox = org[3 * idx]; L.r.oy = org[3 * idx + 1]; L.r.oz = org[3 * idx + 2];
        L.r.dx = dir[3 * idx]; L.r.dy = dir[3 * idx + 1]; L.r.dz = dir[3 * idx + 2];
        in_flight = true;
        start_ray<COUNT>(sc, L, cn);
    }
};

// ------------------------------------------------------------------------------- primary-hit policy
// makeRay (Lib.hs:107-114) + closest hit for every owned pixel, cached as (tri, t bits)
template <class Append>
struct PrimaryPolicy {
    const RenderParams &p;
    int2 *prim;
    Append &append;            // functor: append(pixel) adds a pixel whose primary ray hit something to the pixel list
    long long nwork, w, stride, pixel = -1;
    PathStats &st;
    bool in_flight = false;
    SQT_HD PrimaryPolicy(const RenderParams &p_, int2 *prim_, Append &app_, long long nwork_, long long first, long long stride_, PathStats &st_)
        : p(p_), prim(prim_), append(app_), nwork(nwork_), w(first), stride(stride_), st(st_) {}

    template <bool COUNT>
    SQT_HD void regen(const SceneView &sc, TravLane &L, Counters *cn) {
        if (in_flight) {
            in_flight = false;
            st.rays += 1;
            int2 h; h.x = L.cur.tri; h.y = (int)f2u(L.cur.t);
            prim[pixel] = h;
            if (L.cur.tri >= 0) append(pixel);
            else {                                        // every sample of this pixel is black (Lib.hs:130): nothing to trace
                int k0, k1;
                sample_range(p, k0, k1);
                if (k1 > k0) { st.samples += (stat_t)(k1 - k0); st.primary_reused += (stat_t)(k1 - k0); }
            }
            w += stride;
        }
        for (;;) {
            if (w >= nwork) { L.state = ST_EXIT; return; }
            pixel = work_to_pixel(p, w);
            if (pixel >= 0) break;
            w += stride;
        }
        L.r = make_ray(p, (int)(pixel / p.cols), (int)(pixel % p.cols));
        in_flight = true;
        start_ray<COUNT>(sc, L, cn);
    }
};

// ------------------------------------------------------------------------------- --cast policy
// raycast (Lib.hs:141-151): primary hit + one shadow ray to the hard-coded light; every sample identical.
struct CastPolicy {
    const RenderParams &p;
    float *accum;
    long long nwork, w, stride, pixel = -1;
    PathStats &st;
    int stage = 0;                 // 0 idle, 1 primary in flight, 2 shadow in flight
    int htri = -1; float dl = 0.0f;
    SQT_HD CastPolicy(const RenderParams &p_, float *accum_, long long nwork_, long long first, long long stride_, PathStats &st_)
        : p(p_), accum(accum_), nwork(nwork_), w(first), stride(stride_), st(st_) {}

    SQT_HD void finish(const SceneView &sc, bool lit) {
        float cr = 0.0f, cg = 0.0f, cb = 0.0f;
        if (lit) {
            const uint32_t mat = surface_material(sc, htri);
            const float4 m0 = SQT_LDG4(sc.mats + 3 * (size_t)mat);
            const float kk = XDIV(2.0f, dl);                        // (2 / distanceToLight) *^ surfColor
            cr = XMUL(kk, m0.y); cg = XMUL(kk, m0.z); cb = XMUL(kk, m0.w);
        }
        int k0, k1;
        sample_range(p, k0, k1);
        float sr = 0.0f, sg = 0.0f, sb = 0.0f;
        for (int k = k0; k < k1; ++k) { sr = XADD(sr, cr); sg = XADD(sg, cg); sb = XADD(sb, cb); }
        st.samples += (stat_t)(k1 > k0 ? k1 - k0 : 0);
        accum[3 * pixel] = sr; accum[3 * pixel + 1] = sg; accum[3 * pixel + 2] = sb;
        w += stride;
        stage = 0;
    }

    template <bool COUNT>
    SQT_HD void regen(const SceneView &sc, TravLane &L, Counters *cn) {
        if (stage == 1) {
            st.rays += 1;
            if (L.cur.tri < 0) finish(sc, false);
            else {
                htri = L.cur.tri;
                const float hx = XADD(L.r.ox, XMUL(L.cur.t, L.r.dx)), hy = XADD(L.r.oy, XMUL(L.cur.t, L.r.dy)),
                            hz = XADD(L.r.oz, XMUL(L.cur.t, L.r.dz));
                // shadowRay = intersectPoint `to` hardCodedLight, light = V3 0 3 (-1) ; a `to` b = Ray a (b - a)
                const float ex = XSUB(hx, 0.0f), ey = XSUB(hy, 3.0f), ez = XSUB(hz, -1.0f);
                dl = XSQRT(dot3(ex, ey, ez, ex, ey, ez));
                L.r.ox = hx; L.r.oy = hy; L.r.oz = hz;
                L.r.dx = XSUB(0.0f, hx); L.r.dy = XSUB(3.0f, hy); L.r.dz = XSUB(-1.0f, hz);
                stage = 2;
                start_ray<COUNT>(sc, L, cn);
                return;
            }
        } else if (stage == 2) {
            st.rays += 1;
            // guard $ maybe True (\pos -> dist pos > distanceToLight) (isect geom shadowRay)
            finish(sc, !(L.cur.tri >= 0 && !(L.cur.dist > dl)));
        }
        for (;;) {
            if (w >= nwork) { L.state = ST_EXIT; return; }
            pixel = work_to_pixel(p, w);
            if (pixel >= 0) break;
            w += stride;
        }
        L.r = make_ray(p, (int)(pixel / p.cols), (int)(pixel % p.cols));
        stage = 1;
        start_ray<COUNT>(sc, L, cn);
    }
};

// One lane, run to completion on its own (tests/emu; lanes are independent so this equals any warp schedule).
template <bool COUNT, class Policy>
SQT_HD_NOINLINE void run_lane(const SceneView &sc, Policy &pol, Counters *cn) {
    float4 stack[kStackEntries];
    TravLane L;
    L.stack = stack;
    L.state = ST_DONE; L.sp = 0; L.cur.tri = -1; L.cur.t = 0.0f; L.cur.dist = 0.0f;
    L.r.ox = L.r.oy = L.r.oz = L.r.dx = L.r.dy = L.r.dz = 0.0f;
    const LaneRay ra(L);
    for (;;) {
        if (L.state == ST_DONE) pol.template regen<COUNT>(sc, L, cn);
        if (L.state == ST_EXIT) break;
        if (L.state == ST_RET) ret_step(sc, L, ra);
        if (L.state == ST_DESC) desc_step<COUNT>(sc, L, ra, cn);
        if (L.state == ST_ENTER) enter_step<COUNT>(sc, L, ra, cn);
        if (L.state == ST_LEAF) tri_step<COUNT>(sc, L, cn);
        if (L.state == ST_SPH) sphere_step(sc, L, ra);
    }
}

}  // namespace sqt
