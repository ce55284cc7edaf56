/* oracle_lens.c -- TEST HELPER: the oracle (oracle/oracle.c, included verbatim) extended by the camera-sampling extension
 * of include/sqt.h (sqt_set_lens), which the reference lacks: the primary ray of a sample in a frame with a lens set, and a
 * render of such frames.
 *
 * lens_ray restates the header's definition in plain C (binary32, no contraction: see Makefile).  orc_lens_range continues
 * the per-pixel sums (and, if m2 is given, second moments m2 = m2 + x*x) of the pixels [pix0, pix1) over samples
 * [k_begin, k_end) with the arithmetic of render_chunk, except that every sample traces its own lens ray: same generator
 * seeds spp*(x + y*seed_stride) + k, sums in sample order.  From zero over [0, spp) -- or a rank's sample range -- it is
 * the one-shot frame; over [0, k) the k-sample prefix of a progressive frame.  Pixels another rank owns are left as they
 * are. */
#include "../../oracle/oracle.c"

static ray lens_ray(const orc_params *p, int jitter, float aperture, float focus, int y, int x, const float *cam,
                    uint64_t stream)
{
    uint32_t ctr[4] = { (uint32_t)stream, (uint32_t)(stream >> 32), 0u, 0x4C545153u };     /* "SQTL" */
    uint32_t key[2] = { (uint32_t)p->seed, (uint32_t)(p->seed >> 32) }, w[4];
    orc_philox4x32_10(ctr, key, w);
    float jx = jitter ? random_r01(w[0]) - 0.5f : 0.0f;
    float jy = jitter ? random_r01(w[1]) - 0.5f : 0.0f;
    float fx = (float)x + jx, fy = (float)y + jy;
    float ww = (float)p->xdiv, hh = (float)p->ydiv;
    float xoffs = (fx - (ww / 2)) / ww;
    float yoffs = ((hh / 2) - fy) / hh;
    ray r = { V(cam[0], cam[1], cam[2]), rot_vert(V(1, xoffs, yoffs), cam + 3) };
    if (aperture != 0.0f) {
        const float *R = cam + 3;
        float rad = aperture * sqrtf(random_r01(w[2]));
        float th = 6.2831855f * random_r01(w[3]);
        float sn, cs;
        sqt_sincos(th, &sn, &cs);
        float a = rad * cs, b = rad * sn, inv_f = 1.0f / focus;
        v3 off = V(a * R[3] + b * R[6], a * R[4] + b * R[7], a * R[5] + b * R[8]);
        r.o = V(r.o.x + off.x, r.o.y + off.y, r.o.z + off.z);
        r.d = V(r.d.x - off.x * inv_f, r.d.y - off.y * inv_f, r.d.z - off.z * inv_f);
    }
    return r;
}

/* lens rays of n (pixel, sample) pairs: pix[i] = y*cols + x, k[i] = sample index */
void orc_make_lens_rays(const orc_params *p, const float *cam, int jitter, float aperture, float focus, const int64_t *pix,
                        const int32_t *k, int64_t n, float *org, float *dir)
{
    for (int64_t i = 0; i < n; i++) {
        int y = (int)(pix[i] / p->cols), x = (int)(pix[i] % p->cols);
        uint64_t s = (uint64_t)p->spp * ((uint64_t)x + (uint64_t)y * (uint64_t)p->seed_stride) + (uint64_t)k[i];
        ray r = lens_ray(p, jitter, aperture, focus, y, x, cam, s);
        org[3 * i] = r.o.x; org[3 * i + 1] = r.o.y; org[3 * i + 2] = r.o.z;
        dir[3 * i] = r.d.x; dir[3 * i + 1] = r.d.y; dir[3 * i + 2] = r.d.z;
    }
}

typedef struct { render_ctx rc; int jitter; float aperture, focus; int k_begin, k_end; int64_t off; float *m2; } lens_ctx;

static void lens_chunk(void *ctx, int64_t lo, int64_t hi, int tid)
{
    lens_ctx *g = (lens_ctx *)ctx;
    const orc_params *p = &g->rc.p;
    orc_counters *cn = &g->rc.cn[tid];
    for (int64_t pix = lo + g->off; pix < hi + g->off; pix++) {
        if (!owns_pixel(p, pix)) continue;
        int y = (int)(pix / p->cols), x = (int)(pix % p->cols);
        uint64_t rix = (uint64_t)p->spp * ((uint64_t)x + (uint64_t)y * (uint64_t)p->seed_stride);
        float *a = g->rc.accum + 3 * (pix - g->off), *q = g->m2 ? g->m2 + 3 * (pix - g->off) : NULL;
        v3 sum = V(a[0], a[1], a[2]), sq = q ? V(q[0], q[1], q[2]) : V(0, 0, 0);
        for (int k = g->k_begin; k < g->k_end; k++) {
            ray r = lens_ray(p, g->jitter, g->aperture, g->focus, y, x, g->rc.cam, rix + (uint64_t)k);
            v3 c = raytrace(&g->rc, rix + (uint64_t)k, r, 0, cn);
            sum = vadd(sum, c);
            sq = vadd(sq, vmul(c, c));
            g->rc.samples[tid]++;
        }
        a[0] = sum.x; a[1] = sum.y; a[2] = sum.z;
        if (q) { q[0] = sq.x; q[1] = sq.y; q[2] = sq.z; }
    }
}

/* accum_inout / m2_inout (may be NULL): (pix1 - pix0) * 3 floats; *samples_out (may be NULL): samples traced */
int orc_lens_range(orc_scene *s, const float *cam12, const orc_params *p, int jitter, float aperture, float focus, int64_t pix0,
                   int64_t pix1, int k_begin, int k_end, float *accum_inout, float *m2_inout, uint64_t *samples_out, int nthreads)
{
    if (s->n_nodes == 0 || p->mode != 0 || k_begin < 0 || k_end > p->spp || k_begin > k_end) return 1;
    if (pix0 < 0 || pix1 > (int64_t)p->rows * p->cols || pix0 > pix1) return 1;
    if (nthreads < 1) nthreads = 1;
    if (nthreads > 512) nthreads = 512;
    lens_ctx g;
    g.rc.s = s; g.rc.cam = cam12; g.rc.p = *p; g.rc.accum = accum_inout; g.rc.rgb8 = NULL;
    g.rc.cn = (orc_counters *)calloc((size_t)nthreads, sizeof(orc_counters));
    g.rc.samples = (uint64_t *)calloc((size_t)nthreads, sizeof(uint64_t));
    g.jitter = jitter; g.aperture = aperture; g.focus = focus;
    g.k_begin = k_begin; g.k_end = k_end; g.off = pix0; g.m2 = m2_inout;
    parallel_for(pix1 - pix0, 64, nthreads, lens_chunk, &g);
    uint64_t smp = 0;
    for (int t = 0; t < nthreads; t++) smp += g.rc.samples[t];
    if (samples_out) *samples_out = smp;
    free(g.rc.cn); free(g.rc.samples);
    return 0;
}
