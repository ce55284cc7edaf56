/* oracle_range.c -- TEST HELPER: the oracle (oracle/oracle.c, included verbatim) extended by a range render for the
 * progressive frames of include/sqt.h.
 *
 * orc_render_range continues the per-pixel radiance sums (accum) and second moments (m2 = m2 + x*x, every operation
 * binary32) of the spp frame described by `p` over samples [k_begin, k_end), with the arithmetic of render_chunk:
 * same rays, same generator seeds spp*(x + y*seed_stride) + k, sums in sample order.  Chunked as [0,a) + [a,b) + [b,spp)
 * it therefore gives the bits of one range [0,spp), and its sums are orc_render's accumulation buffer.  Pixels another
 * rank owns are left as they are. */
#include "../../oracle/oracle.c"

typedef struct { render_ctx rc; int k_begin, k_end; float *m2; } range_ctx;

static void range_chunk(void *ctx, int64_t lo, int64_t hi, int tid)
{
    range_ctx *g = (range_ctx *)ctx;
    const orc_params *p = &g->rc.p;
    orc_counters *cn = &g->rc.cn[tid];
    for (int64_t pix = lo; pix < hi; pix++) {
        if (!owns_pixel(p, pix)) continue;
        int y = (int)(pix / p->cols), x = (int)(pix % p->cols);
        ray r = make_ray(p, y, x, g->rc.cam);
        uint64_t rix = (uint64_t)p->spp * ((uint64_t)x + (uint64_t)y * (uint64_t)p->seed_stride);
        float *a = g->rc.accum + 3 * pix, *q = g->m2 + 3 * pix;
        v3 sum = V(a[0], a[1], a[2]), sq = V(q[0], q[1], q[2]);
        for (int k = g->k_begin; k < g->k_end; k++) {
            v3 c = raytrace(&g->rc, rix + (uint64_t)k, r, 0, cn);
            sum = vadd(sum, c);
            sq = vadd(sq, vmul(c, c));
            g->rc.samples[tid]++;
        }
        a[0] = sum.x; a[1] = sum.y; a[2] = sum.z;
        q[0] = sq.x; q[1] = sq.y; q[2] = sq.z;
    }
}

int orc_render_range(orc_scene *s, const float *cam12, const orc_params *p, int k_begin, int k_end, float *accum_inout,
                     float *m2_inout, int nthreads)
{
    if (s->n_nodes == 0 || p->mode != 0 || k_begin < 0 || k_end > p->spp || k_begin > k_end) return 1;
    if (nthreads < 1) nthreads = 1;
    if (nthreads > 512) nthreads = 512;
    range_ctx g;
    g.rc.s = s; g.rc.cam = cam12; g.rc.p = *p; g.rc.accum = accum_inout; g.rc.rgb8 = NULL;
    g.rc.cn = (orc_counters *)calloc((size_t)nthreads, sizeof(orc_counters));
    g.rc.samples = (uint64_t *)calloc((size_t)nthreads, sizeof(uint64_t));
    g.k_begin = k_begin; g.k_end = k_end; g.m2 = m2_inout;
    parallel_for((int64_t)p->rows * p->cols, 64, nthreads, range_chunk, &g);
    free(g.rc.cn); free(g.rc.samples);
    return 0;
}
