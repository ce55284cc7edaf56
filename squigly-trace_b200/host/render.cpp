// render.cpp -- `render` (Lib.hs:68-75) and the Scene plug-in (Geometry.hs:62-65) on top of the C ABI.
#include <chrono>
#include <cstdio>
#include <cstring>
#include <iostream>

#include "squigly.hpp"

namespace squigly {

// Geometry of a `Scene BIH` living on one or more B200s.
class DeviceBIH {
  public:
    DeviceBIH(const BIH &bih, int nGpus) {
        if (nGpus < 1) throw std::invalid_argument("gpus must be >= 1");
        FlatBIH flat = flattenForDevice(bih);
        const sqt_scene_desc d = flat.desc();
        ctxs_.resize(nGpus, nullptr);
        for (int g = 0; g < nGpus; ++g) {
            if (sqt_create(g, &ctxs_[g]) != SQT_OK) {
                std::string e = sqt_last_error(nullptr);
                release();
                throw std::runtime_error("sqt_create(" + std::to_string(g) + "): " + e);
            }
            check(g, sqt_upload_scene(ctxs_[g], &d), "sqt_upload_scene");     // scene replicated on every GPU
        }
        if (nGpus > 1) check(0, sqt_comm_init_all(ctxs_.data(), nGpus), "sqt_comm_init_all");
    }
    ~DeviceBIH() { release(); }
    DeviceBIH(const DeviceBIH &) = delete;
    DeviceBIH &operator=(const DeviceBIH &) = delete;

    sqt_ctx *ctx(int g = 0) const { return ctxs_[g]; }
    sqt_ctx **ctxs() const { return const_cast<sqt_ctx **>(ctxs_.data()); }
    int gpus() const { return (int)ctxs_.size(); }
    void check(int g, int rc, const char *what) const {
        if (rc != SQT_OK) throw std::runtime_error(std::string(what) + ": " + sqt_last_error(ctxs_[g]));
    }

  private:
    void release() { for (auto *&c : ctxs_) { if (c) sqt_destroy(c); c = nullptr; } }
    std::vector<sqt_ctx *> ctxs_;
};

static std::vector<std::optional<Intersection>> intersectBIHBatch(const DeviceBIH &g, const std::vector<Ray> &rays) {
    const size_t n = rays.size();
    std::vector<float> org(3 * n), dir(3 * n), dist(n), point(3 * n);
    std::vector<int32_t> tri(n);
    for (size_t i = 0; i < n; ++i) {
        org[3 * i] = rays[i].vertex.x; org[3 * i + 1] = rays[i].vertex.y; org[3 * i + 2] = rays[i].vertex.z;
        dir[3 * i] = rays[i].direction.x; dir[3 * i + 1] = rays[i].direction.y; dir[3 * i + 2] = rays[i].direction.z;
    }
    g.check(0, sqt_intersect_batch(g.ctx(), org.data(), dir.data(), (int64_t)n, tri.data(), dist.data(), point.data(), nullptr),
            "sqt_intersect_batch");
    std::vector<std::optional<Intersection>> out(n);
    for (size_t i = 0; i < n; ++i)
        if (tri[i] >= 0) out[i] = Intersection{V3{point[3 * i], point[3 * i + 1], point[3 * i + 2]}, dist[i], tri[i]};
    return out;
}

std::optional<Intersection> SceneBIH::intersect(const Ray &r) const { return intersectBatch(*geometry, {r})[0]; }

// sceneFromBIH bih = Scene bih intersectBIH   (Main.hs:55-56)
SceneBIH sceneFromBIH(const BIH &bih, int nGpus) {
    SceneBIH s;
    s.geometry = std::make_shared<DeviceBIH>(bih, nGpus);
    s.intersectBatch = &intersectBIHBatch;
    return s;
}

sqt_render_params paramsFromSettings(const Settings &s) {
    sqt_render_params p;
    std::memset(&p, 0, sizeof p);
    const int w = s.dimensions.first, h = s.dimensions.second;
    if (s.corrected) { p.rows = h; p.cols = w; }         // image is w wide and h tall
    else { p.rows = w; p.cols = h; }                      // Lib.hs:70-71: dims = (w :. h) = (rows :. cols)
    p.xdiv = w; p.ydiv = h; p.seed_stride = w;            // Lib.hs:85,108-112
    p.spp = s.samples; p.max_depth = s.bounces; p.mode = s.cast ? 1 : 0; p.seed = s.seed;
    return p;
}

// --aa / --lens: the same camera model on every GPU of the run (sqt_set_lens); without either, the reference's pinhole
static void setLens(const DeviceBIH &g, const Settings &s) {
    const bool on = s.aa || s.focus > 0.0f;
    const sqt_lens l{s.aa ? 1u : 0u, s.aperture, s.focus > 0.0f ? s.focus : 1.0f, 0u};
    for (int k = 0; k < g.gpus(); ++k) g.check(k, sqt_set_lens(g.ctx(k), on ? &l : nullptr), "sqt_set_lens");
}

RenderReport renderToBuffer(const SceneBIH &scene, const Camera &cam, const Settings &settings, std::vector<uint8_t> &rgb8,
                            std::vector<float> *accum) {
    const sqt_render_params p = paramsFromSettings(settings);
    sqt_camera c;
    c.position[0] = cam.position.x; c.position[1] = cam.position.y; c.position[2] = cam.position.z;
    std::memcpy(c.rotation, cam.rotation, sizeof c.rotation);
    RenderReport rep; rep.rows = p.rows; rep.cols = p.cols;
    rgb8.assign((size_t)p.rows * p.cols * 3, 0);
    if (accum) accum->assign((size_t)p.rows * p.cols * 3, 0.0f);
    const DeviceBIH &g = *scene.geometry;
    setLens(g, settings);
    g.check(0, sqt_render_group(g.ctxs(), g.gpus(), &c, &p, rgb8.data(), accum ? accum->data() : nullptr, &rep.stats), "sqt_render");
    return rep;
}

// --progress=N: the same frame as a progressive one (include/sqt.h) in chunks of N samples; after every chunk the preview
// overwrites the save path and one line reports samples done, the noise estimate and the elapsed time.  The last image
// is the one-shot frame bit for bit.  --adaptive: after every chunk of at least 2 samples the converged pixels retire
// (sqt_render_retire) and the line also reports the pixels still active; with zero tolerances nothing retires and the
// image is the one-shot frame as well.  --denoise: after every chunk of at least 2 samples the denoised preview
// (sqt_denoise) also goes to <savepath stem>-denoised.png; the plain preview is not affected.
static std::string denoisedPath(const std::string &path) {
    const size_t slash = path.find_last_of('/'), dot = path.find_last_of('.');
    const size_t stem = dot != std::string::npos && (slash == std::string::npos || dot > slash) ? dot : path.size();
    return path.substr(0, stem) + "-denoised" + path.substr(stem);
}

static RenderReport renderProgressive(const SceneBIH &scene, const Camera &cam, const Settings &settings) {
    const sqt_render_params p = paramsFromSettings(settings);
    if (p.mode != 0) throw std::runtime_error("--progress needs path tracing (not --cast)");
    sqt_camera c;
    c.position[0] = cam.position.x; c.position[1] = cam.position.y; c.position[2] = cam.position.z;
    std::memcpy(c.rotation, cam.rotation, sizeof c.rotation);
    RenderReport rep; rep.rows = p.rows; rep.cols = p.cols;
    std::vector<uint8_t> img((size_t)p.rows * p.cols * 3, 0);
    const DeviceBIH &g = *scene.geometry;
    const auto t0 = std::chrono::steady_clock::now();
    setLens(g, settings);
    g.check(0, sqt_render_begin_group(g.ctxs(), g.gpus(), &c, &p, &rep.stats), "sqt_render_begin");
    sqt_progress pr{0, p.spp, 0.0};
    const sqt_retire_params rp{settings.adaptiveRel, settings.adaptiveAbs, settings.adaptiveMin, 0u};
    int64_t active = -1;
    while (pr.samples_done < pr.samples_total) {
        sqt_stats st;
        g.check(0, sqt_render_advance_group(g.ctxs(), g.gpus(), settings.progress, &pr, &st), "sqt_render_advance");
        rep.stats.device_ms += st.device_ms; rep.stats.rays_traced += st.rays_traced; rep.stats.samples += st.samples;
        if (settings.adaptive && pr.samples_done >= 2)
            g.check(0, sqt_render_retire_group(g.ctxs(), g.gpus(), &rp, &active), "sqt_render_retire");
        g.check(0, sqt_download_image(g.ctx(0), img.data(), nullptr), "sqt_download_image");
        writeImage(settings.savePath, img.data(), rep.rows, rep.cols);
        if (settings.denoise >= 0 && pr.samples_done >= 2) {
            const sqt_denoise_params dp{settings.denoise, 4.0f, 0.05f, 0u};
            g.check(0, sqt_denoise_group(g.ctxs(), g.gpus(), &dp, img.data(), nullptr, nullptr), "sqt_denoise");
            writeImage(denoisedPath(settings.savePath), img.data(), rep.rows, rep.cols);
        }
        const double sec = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        if (settings.adaptive && active >= 0)
            std::printf("%d/%d samples  noise %.6g  active %lld  %.3fs\n", pr.samples_done, pr.samples_total, pr.noise, (long long)active, sec);
        else
            std::printf("%d/%d samples  noise %.6g  %.3fs\n", pr.samples_done, pr.samples_total, pr.noise, sec);
        std::fflush(stdout);
    }
    return rep;
}

RenderReport render(const SceneBIH &scene, const Camera &cam, const Settings &settings) {
    if (settings.progress > 0) return renderProgressive(scene, cam, settings);
    std::vector<uint8_t> img;
    RenderReport rep = renderToBuffer(scene, cam, settings, img, nullptr);
    writeImage(settings.savePath, img.data(), rep.rows, rep.cols);        // img `seq` writeImage savePath img
    return rep;
}

}  // namespace squigly
