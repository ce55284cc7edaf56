/* oracle_prefix.c -- TEST HELPER: the oracle's range render (tests/progressive/oracle_range.c, itself oracle/oracle.c
 * included verbatim) restricted to the pixels [pix0, pix1) of the frame described by `p`, on the calling thread.  It gives
 * a few pixels' sums and second moments over samples [k_begin, k_end) of a full-size frame without rendering all of it. */
#include "../progressive/oracle_range.c"

int orc_render_range_window(orc_scene *s, const float *cam12, const orc_params *p, int64_t pix0, int64_t pix1, int k_begin,
                            int k_end, float *accum_inout, float *m2_inout)
{
    if (s->n_nodes == 0 || p->mode != 0 || k_begin < 0 || k_end > p->spp || k_begin > k_end) return 1;
    if (pix0 < 0 || pix1 > (int64_t)p->rows * p->cols || pix0 > pix1) return 1;
    range_ctx g;
    orc_counters cn;
    uint64_t samples = 0;
    memset(&cn, 0, sizeof cn);
    g.rc.s = s; g.rc.cam = cam12; g.rc.p = *p; g.rc.rgb8 = NULL;
    g.rc.accum = accum_inout - 3 * pix0;          /* range_chunk indexes by pixel */
    g.m2 = m2_inout - 3 * pix0;
    g.rc.cn = &cn; g.rc.samples = &samples;
    g.k_begin = k_begin; g.k_end = k_end;
    range_chunk(&g, pix0, pix1, 0);
    return 0;
}
