// sqt_denoise.cuh -- the per-pixel arithmetic of sqt_denoise (include/sqt.h): primary-hit features, the filter's inputs
// and one level of the edge-aware a-trous filter.  SQT_HD like sqt_paths.cuh, so that tests/denoise builds the same
// source with g++ and compares it bit for bit with the device.  Only + - * / sqrt and comparisons appear, every one an
// explicit round-to-nearest binary32 operation (X* wrappers), so the host build and the device agree to the bit.
#pragma once
#include "sqt_paths.cuh"

namespace sqt {

// the filter's per-pixel key: 0 = no primary hit; material + 1 for a surface that is filtered; -(material + 1) for a
// perfect mirror (reflective >= 1), which is passed through.  Two pixels are neighbours iff their keys are equal and > 0.
SQT_HD int denoise_key(const SceneView &sc, int surface) {
    if (surface < 0) return 0;
    const uint32_t mat = surface_material(sc, surface);
    const float refl = SQT_LDG4(sc.mats + 3 * (size_t)mat).x;
    return refl >= 1.0f ? -(int)(mat + 1u) : (int)(mat + 1u);
}

// feature of a primary hit of ray r on `surface` (leaf order, or n_tris + sphere) at parameter t: (N, t) with N the unit
// geometric normal -- e1 x e2 for a triangle, hit - centre for a sphere, divided by its length -- turned to face the ray
// (negated when N.d > 0)
SQT_HD float4 primary_feature(const SceneView &sc, const Ray &r, int surface, float t) {
    float nx, ny, nz;
    if ((uint32_t)surface >= sc.n_tris) {
        const float4 s0 = SQT_LDG4(sc.spheres + 2 * (size_t)((uint32_t)surface - sc.n_tris));
        nx = XSUB(XADD(r.ox, XMUL(t, r.dx)), s0.x); ny = XSUB(XADD(r.oy, XMUL(t, r.dy)), s0.y); nz = XSUB(XADD(r.oz, XMUL(t, r.dz)), s0.z);
    } else {
        const float4 *p = sc.tris + 3 * (size_t)surface;
        const float4 a0 = SQT_LDG4(p), a1 = SQT_LDG4(p + 1), a2 = SQT_LDG4(p + 2);
        const float e1x = a0.w, e1y = a1.x, e1z = a1.y, e2x = a1.z, e2y = a1.w, e2z = a2.x;
        nx = XSUB(XMUL(e1y, e2z), XMUL(e1z, e2y));
        ny = XSUB(XMUL(e1z, e2x), XMUL(e1x, e2z));
        nz = XSUB(XMUL(e1x, e2y), XMUL(e1y, e2x));
    }
    const float nn = XSQRT(dot3(nx, ny, nz, nx, ny, nz));
    nx = XDIV(nx, nn); ny = XDIV(ny, nn); nz = XDIV(nz, nn);
    if (dot3(nx, ny, nz, r.dx, r.dy, r.dz) > 0.0f) { nx = -nx; ny = -ny; nz = -nz; }
    float4 f; f.x = nx; f.y = ny; f.z = nz; f.w = t;
    return f;
}

// the filter's input of one pixel with sums s1, moments s2 after n samples: (c, v) with c = s1 * (1.0f/(float)n) -- the
// values the preview's tone map sees -- and v = (float)e2, the standard-error term of retire_test
SQT_HD float4 denoise_input(const float *s1, const float *s2, int n) {
    const float inv = 1.0f / (float)n;
    double e2, m;
    (void)pixel_error(s1, s2, n, e2, m);
    float4 o; o.x = XMUL(inv, s1[0]); o.y = XMUL(inv, s1[1]); o.z = XMUL(inv, s1[2]); o.w = (float)e2;
    return o;
}

SQT_HD float denoise_h1(int d) { return d == 0 ? 0.375f : (d == 1 || d == -1 ? 0.25f : 0.0625f); }
SQT_HD float denoise_lum(const float4 &c) { return XADD(XADD(c.x, c.y), c.z); }
SQT_HD float denoise_pos(float a) { return a > 0.0f ? a : 0.0f; }      // max(0, a), NaN -> 0

// one level (step s) of the filter at pixel (y, x) of a rows x cols image: cv = the previous level's (c, v) per pixel,
// feat = (N, z), sk = (surface + 1, denoise_key) -- the key is sk.y.  Returns the pixel's (c', v') -- its input where key <= 0.
SQT_HD float4 denoise_level_pixel(const float4 *cv, const float4 *feat, const int2 *sk, int rows, int cols, int y, int x,
                                  int s, float sigma_l, float sigma_z) {
    const long long p = (long long)y * cols + x;
    const float4 cp = cv[p];
    const int kp = sk[p].y;
    if (kp <= 0) return cp;
    // SVGF's variance prefilter: g = sqrt(sum k v / sum k) over the 3x3 neighbours of the same key, k = [1,2,1] x [1,2,1]
    float skv = 0.0f, ksum = 0.0f;
    for (int dy = -1; dy <= 1; ++dy)
        for (int dx = -1; dx <= 1; ++dx) {
            const int qy = y + dy, qx = x + dx;
            if (qy < 0 || qy >= rows || qx < 0 || qx >= cols) continue;
            const long long q = (long long)qy * cols + qx;
            if (sk[q].y != kp) continue;
            const float k = (float)((dy == 0 ? 2 : 1) * (dx == 0 ? 2 : 1));
            skv = XADD(skv, XMUL(k, cv[q].w));
            ksum = XADD(ksum, k);
        }
    const float g = XSQRT(XDIV(skv, ksum));
    const float4 fp = feat[p];
    const float lp = denoise_lum(cp);
    const float dl = XADD(XMUL(sigma_l, g), 1e-6f);
    const float dz = XMUL(XMUL(sigma_z, (float)s), fp.w);
    float sw = 0.0f, sr = 0.0f, sg = 0.0f, sb = 0.0f, sv = 0.0f;
    for (int dy = -2; dy <= 2; ++dy)
        for (int dx = -2; dx <= 2; ++dx) {
            const int qy = y + s * dy, qx = x + s * dx;
            if (qy < 0 || qy >= rows || qx < 0 || qx >= cols) continue;
            const long long q = (long long)qy * cols + qx;
            if (sk[q].y != kp) continue;
            const float4 cq = cv[q];
            float w;
            if (dy == 0 && dx == 0) {
                w = 0.140625f;                                 // h1(0) * h1(0) = 9/64
            } else {
                const float4 fq = feat[q];
                const float h = XMUL(denoise_h1(dy), denoise_h1(dx));
                const float ex = XADD(XDIV(fabsf(XSUB(lp, denoise_lum(cq))), dl), XDIV(fabsf(XSUB(fp.w, fq.w)), dz));
                float wn = denoise_pos(dot3(fp.x, fp.y, fp.z, fq.x, fq.y, fq.z));
                for (int i = 0; i < 7; ++i) wn = XMUL(wn, wn);
                float r = XDIV(1.0f, XADD(1.0f, XMUL(ex, 0.125f)));
                for (int i = 0; i < 3; ++i) r = XMUL(r, r);
                w = XMUL(XMUL(h, wn), r);
            }
            sw = XADD(sw, w);
            sr = XADD(sr, XMUL(w, cq.x)); sg = XADD(sg, XMUL(w, cq.y)); sb = XADD(sb, XMUL(w, cq.z));
            sv = XADD(sv, XMUL(XMUL(w, w), cq.w));
        }
    float4 o;
    o.x = XDIV(sr, sw); o.y = XDIV(sg, sw); o.z = XDIV(sb, sw); o.w = XDIV(sv, XMUL(sw, sw));
    return o;
}

}  // namespace sqt
