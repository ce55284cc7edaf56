// emu_lens.cpp -- TEST HELPER: the host build of the kernels' lens frames (sqt_set_lens, include/sqt.h).  It is tests/emu
// (emu.cpp, included verbatim: scene upload, spheres, the sample-buffer budget) plus a render that runs the integrator as the
// lens kernels instantiate it -- PathPolicy<Fetch, true>: every sample traces its own lens_ray, no primary pass, every owned
// pixel on the pixel list (k_lens_list) -- and lens_ray itself for unit tests.  Not a fallback: the product never loads it.
#include "../emu/emu.cpp"

// the render parameters of a lens frame, as sqt_backend.cu's to_device_params makes them
static RenderParams lens_params(const emu_scene *s, const sqt_camera *cam, const sqt_render_params *p, int rank, int world,
                                const sqt_lens *l) {
    RenderParams d = {};
    d.rows = p->rows; d.cols = p->cols; d.xdiv = p->xdiv; d.ydiv = p->ydiv; d.seed_stride = p->seed_stride;
    d.spp = p->spp; d.max_depth = p->max_depth; d.mode = p->mode; d.seed = p->seed;
    d.rank = rank; d.world = world; d.split_samples = (p->flags & SQT_F_SPLIT_SAMPLES) ? 1 : 0;
    d.primary_reuse = 0;
    for (int k = 0; k < 3; ++k) d.cam_pos[k] = cam->position[k];
    for (int k = 0; k < 9; ++k) d.cam_rot[k] = cam->rotation[k];
    d.terminate_on_black = (s && s->lay.terminate_on_black_ok && !(p->flags & SQT_F_NO_EARLY_TERMINATION)) ? 1 : 0;
    d.lens = 1; d.jitter = (int)l->jitter; d.aperture = l->aperture_radius; d.focus = l->focus_distance;
    return d;
}

extern "C" {

// lens_ray for n (pixel, sample) pairs (pix = y*cols + x, k = sample index)
void emu_lens_rays(const sqt_camera *cam, const sqt_render_params *p, const sqt_lens *l, const long long *pix, const int *k,
                   long long n, float *org, float *dir) {
    const RenderParams d = lens_params(nullptr, cam, p, 0, 1, l);
    for (long long i = 0; i < n; ++i) {
        const int y = (int)(pix[i] / d.cols), x = (int)(pix[i] % d.cols);
        const unsigned long long st = (unsigned long long)d.spp * ((unsigned long long)x + (unsigned long long)y * (unsigned long long)d.seed_stride) + (unsigned long long)k[i];
        const Ray r = lens_ray(d, y, x, st);
        org[3 * i] = r.ox; org[3 * i + 1] = r.oy; org[3 * i + 2] = r.oz;
        dir[3 * i] = r.dx; dir[3 * i + 1] = r.dy; dir[3 * i + 2] = r.dz;
    }
}

// One lens frame (mode 0), lanes and rounds as emu_render runs them.  stats3 = rays, samples, primary_reused
void emu_render_lens(emu_scene *s, const sqt_camera *cam, const sqt_render_params *p, int rank, int world, const sqt_lens *l,
                     float *accum, unsigned long long *stats3) {
    const RenderParams d = lens_params(s, cam, p, rank, world, l);
    const long long npix = (long long)d.rows * d.cols, nwork = work_items(d);
    std::memset(accum, 0, (size_t)npix * 12);
    Counters cn = {};
    PathStats st = {0, 0, 0};
    const long long n_lanes = 7;
    std::vector<int> pixel_list;
    for (long long w = 0; w < nwork; ++w) if (work_to_pixel(d, w) >= 0) pixel_list.push_back((int)work_to_pixel(d, w));
    int k0, k1;
    sample_range(d, k0, k1);
    RoundInfo rd = {};
    rd.pixel_list = pixel_list.data();
    rd.prim = nullptr;
    rd.n_slots = (long long)pixel_list.size();
    rd.slot_stride = nwork;
    rd.log2_s = round_log2_s(nwork, k1 - k0 > 0 ? k1 - k0 : 1, sbuf_budget);
    const int S = 1 << rd.log2_s;
    std::vector<float> sbuf((size_t)(nwork * S * 3 + 3));
    rd.sbuf = sbuf.data();
    uint16_t pm[SQT_MAX_DEPTH];
    for (int kb = k0; kb < k1; kb += S) {
        rd.k0 = kb; rd.k1 = kb + S < k1 ? kb + S : k1;
        std::fill(sbuf.begin(), sbuf.end(), 0.0f);
        const long long items = rd.n_slots << rd.log2_s;
        SeqFetch fetch{0, items};
        for (long long ln = 0; ln < n_lanes; ++ln) {
            SeqFetch part{fetch.next, ln + 1 == n_lanes ? items : std::min(items, fetch.next + (items + n_lanes - 1) / n_lanes)};
            PathPolicy<SeqFetch, true> pol(d, rd, part, st, pm);
            run_lane<true>(s->view, pol, &cn);
            fetch.next = part.n;
        }
        for (long long slot = 0; slot < rd.n_slots; ++slot) accumulate_slot(d, rd, slot, accum);
    }
    if (stats3) { stats3[0] = st.rays; stats3[1] = st.samples; stats3[2] = st.primary_reused; }
}

}  // extern "C"
