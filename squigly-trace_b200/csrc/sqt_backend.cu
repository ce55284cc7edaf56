// sqt_backend.cu -- context, scene upload and the C ABI (include/sqt.h) of the squigly-trace B200 backend.
//
// The kernels live in sqt_kernels.cuh (per-ray logic in sqt_core.cuh / sqt_paths.cuh), the NCCL shim in sqt_nccl.hpp,
// the host-side derivation of the device records in sqt_layout.hpp.  Every launch is bracketed by CUDA events on the
// context's stream.
//
// There is no CPU fallback in this file: every entry point needs a compute-capability-10.x device.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stddef.h>
#include <stdio.h>
#include <string.h>
#include <atomic>
#include <chrono>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "../../include/sqt.h"
#include "sqt_kernels.cuh"
#include "sqt_layout.hpp"
#include "sqt_nccl.hpp"

// ============================================================================== context
// A grow-only allocation of `cap` elements of T in device memory or, PINNED, in page-locked host memory; the destructor
// frees it.  ensure(n) reallocates only when n exceeds the capacity, reset(n) always, at exactly n (0: free only).  The
// contents are never kept.  On a failed allocation the buffer is empty, so the next ensure tries again.
template <class T, bool PINNED = false>
struct Buffer {
    T *p = nullptr;
    size_t cap = 0;
    Buffer() = default;
    Buffer(Buffer &&o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
    Buffer &operator=(Buffer &&o) noexcept { std::swap(p, o.p); std::swap(cap, o.cap); return *this; }
    ~Buffer() { reset(0); }
    operator T *() const { return p; }
    T *operator->() const { return p; }
    cudaError_t ensure(size_t n) { return n <= cap ? cudaSuccess : reset(n); }
    cudaError_t reset(size_t n) {
        if (p) { if (PINNED) cudaFreeHost(p); else cudaFree(p); }
        p = nullptr; cap = 0;
        if (n == 0) return cudaSuccess;
        void *q = nullptr;
        const cudaError_t e = PINNED ? cudaMallocHost(&q, n * sizeof(T)) : cudaMalloc(&q, n * sizeof(T));
        if (e == cudaSuccess) { p = (T *)q; cap = n; }
        return e;
    }
};
template <class T> using Pinned = Buffer<T, true>;

// launch shape of a frame's sample rounds (prepare_render): work items, this rank's sample range, S = 1 << log2_s
struct RenderPlan { long long nwork = 0; int k0 = 0, k1 = 0, log2_s = 0; long long sbytes = 0; };

// a progressive frame (sqt_render_begin until whatever ends it, include/sqt.h): what the frame needs between two calls
struct ProgFrame {
    bool on = false;                    // a progressive frame is in progress
    int k = 0;                          // samples [0, k) are in the sums
    bool count = false;
    RenderParams d = {};
    RenderPlan pl;
    bool adaptive = false;              // retire has run in this frame: d_pixel_list / n_hit hold the active pixels
    long long n = 0;                    // this rank's active slots (the primary pass's hit count until the first retire)
    long long total = 0;                // active pixels of the whole frame after the last retire
};

struct sqt_ctx {
    int device = 0, sm_count = 0, cc_major = 0, cc_minor = 0;
    char name[128] = {0};
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[8] = {};
    std::string err;
    // scene
    bool has_scene = false;
    SceneView sc = {};
    Buffer<float4> d_slabs, d_tight; Buffer<uint32_t> d_levels;                   // subtree slabs (+ upload scratch)
    Buffer<float4> d_nodes, d_boxes, d_tris, d_mats, d_leaves, d_spheres;
    Buffer<float4> d_sph_nodes; Buffer<uint32_t> d_sph_order; int sphere_bvh = 1;  // extension: hierarchy over the spheres
    Buffer<uint2> d_ranges;             // (first, count) per leaf, input of k_leaf_records
    Buffer<uint32_t> d_flag;            // material check result
    uint64_t upload_bytes = 0; double upload_ms = 0, upload_layout_ms = 0;   // last sqt_upload_scene
    int leaf_cull = 1;
    int terminate_on_black_ok = 0;
    uint32_t tree_height = 0;
    // image buffers
    Buffer<int2> d_prim;
    Buffer<int> d_pixel_list;
    Buffer<float> d_sbuf;               // sample buffer of one round
    long long sbuf_budget = 2ll << 30;
    Buffer<float> d_accum;
    Buffer<uint8_t> d_rgb8;
    long long img_pixels = 0;
    int img_spp = 0;
    Buffer<DeviceStats> d_stats;
    Pinned<DeviceStats> h_stats;
    // batch staging
    Buffer<float> d_org, d_dir, d_dist, d_point;
    Buffer<int> d_tri;
    // pinned host staging for image I/O
    Pinned<uint8_t> h_rgb8; Pinned<float> h_accum;
    Tune tune = {12, 0, 12};
    PoolTune pool_tune = {4, 10, 16};
    float slab_ratio = kSlabRatioMax, slab_ratio_leaf = kSlabRatioMaxLeaf;   // subtree / leaf slabs: test a slab when it is at most this
                                                                             // fraction of the clipped box (SQT_SLAB_RATIO=branch[,leaf], 0 = never)
    Buffer<float4> d_gstack; Buffer<uint16_t> d_gpm; Buffer<uint4> d_gpath;     // per pool slot: stack, materials, path state
    bool comm_broken = false;           // the communicator was aborted after a rank failed
    ProgFrame prog;
    long long prog_frame = 0;           // numbers the progressive frames of this context (sqt_render_begin); never reset
    bool lens_set = false; sqt_lens lens = {};      // camera model of the frames this context starts (sqt_set_lens)
    Buffer<float> d_m2;                 // per-pixel second moment (npix * 3 floats)
    Buffer<float> d_red1, d_red2;       // rank 0 of a group: sums and moments of all ranks
    Buffer<double> d_noise; Pinned<double> h_noise;              // partial sums of k_frame_noise_part + the result (pinned copy)
    // adaptive frame (sqt_render_retire): per-pixel sample counts (0 = active) and the scratch of the list compaction
    Buffer<int> d_counts, d_redc, d_list2; Buffer<uint8_t> d_keep; Buffer<long long> d_tile;
    Buffer<long long> d_active; Pinned<long long> h_active;      // all-reduced active total; pinned (local, total)
    // denoiser (sqt_denoise / sqt_download_features): features (N, z) and (surface + 1, key) -- on rank 0 of a group the sum
    // over ranks --, the filter's ping-pong (c, v) buffers, the denoised mean and its RGB8
    Buffer<float4> d_feat, d_dn[2]; Buffer<int2> d_sk; Buffer<float> d_dn_mean; Buffer<uint8_t> d_dn_rgb8;
    long long dn_frame = -1;            // the progressive frame whose features d_feat / d_sk hold (-1: none)
    // group
    int rank = 0, world = 1;
    ncclComm_t comm = nullptr;
};

// d_flag: word 0 the material check of an upload, words 1.. the group agreement (flag + up to seven keys as (v, -v): the
// lens and, for sqt_render_begin, samples done / target spp / chunk)
constexpr int kFlagWords = 16;

static thread_local std::string g_create_err;

static int fail(sqt_ctx *c, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    if (c) c->err = buf; else g_create_err = buf;
    return code;
}
#define CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(ctx, SQT_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); } while (0)

extern "C" int sqt_abi_version(void) { return SQT_ABI_VERSION; }

extern "C" const char *sqt_last_error(const sqt_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

static int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// Environment knobs (development only; they change scheduling, never a result).  Malformed values are ignored and every
// value is clamped to a range in which the persistent kernels are guaranteed to make progress.
static void read_env_tuning(sqt_ctx *c) {
    if (const char *t = getenv("SQT_SLAB_RATIO")) {
        char *e = nullptr; double v = strtod(t, &e);
        if (e != t && v >= 0.0 && v <= 2.0) {
            c->slab_ratio = (float)v;
            if (*e == ',') { const char *u = e + 1; double w = strtod(u, &e); if (e != u && w >= 0.0 && w <= 2.0) c->slab_ratio_leaf = (float)w; }
        }
    }
    if (const char *t = getenv("SQT_POOL_TUNE")) {       // "burst_t,t_leave,c_min"
        int a, b, cm;
        if (sscanf(t, "%d,%d,%d", &a, &b, &cm) == 3) c->pool_tune = {clampi(a, 1, 64), clampi(b, 0, 31), clampi(cm, 1, 32)};
    }
    if (const char *t = getenv("SQT_SBUF_MB")) { char *e = nullptr; long long mb = strtoll(t, &e, 10); if (e != t && mb > 0 && mb < (1ll << 20)) c->sbuf_budget = mb << 20; }
    if (const char *t = getenv("SQT_TUNE")) {            // "a_leave,b_leave,c_min"
        int a, b, cm;
        if (sscanf(t, "%d,%d,%d", &a, &b, &cm) == 3) c->tune = {clampi(a, 0, 31), clampi(b, 0, 32), clampi(cm, 1, 32)};
    }
}

extern "C" int sqt_destroy(sqt_ctx *c);

extern "C" int sqt_create(int device, sqt_ctx **out) {
    if (!out) return fail(nullptr, SQT_E_INVALID, "sqt_create: out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(nullptr, SQT_E_NO_DEVICE, "no CUDA device (%s); this backend has no CPU fallback", cudaGetErrorString(e));
    if (device < 0 || device >= n) return fail(nullptr, SQT_E_INVALID, "device %d out of range (have %d)", device, n);
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return fail(nullptr, SQT_E_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (prop.major != 10)
        return fail(nullptr, SQT_E_NO_DEVICE, "device %d (%s) is compute capability %d.%d; this library is built for sm_100a only",
                    device, prop.name, prop.major, prop.minor);
    if ((e = cudaSetDevice(device)) != cudaSuccess) return fail(nullptr, SQT_E_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
    sqt_ctx *c = new sqt_ctx();
    c->device = device; c->sm_count = prop.multiProcessorCount; c->cc_major = prop.major; c->cc_minor = prop.minor;
    snprintf(c->name, sizeof c->name, "%s", prop.name);
    auto init = [&]() -> int {
        sqt_ctx *ctx = c;
        CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        for (auto &ev : c->ev) CU(cudaEventCreate(&ev));
        CU(c->d_stats.ensure(1));
        CU(c->d_flag.ensure(kFlagWords));
        CU(c->h_stats.ensure(1));
        return SQT_OK;
    };
    const int rc = init();
    if (rc) { g_create_err = c->err; sqt_destroy(c); return rc; }        // no half-built context is leaked
    read_env_tuning(c);
    *out = c;
    return SQT_OK;
}

extern "C" int sqt_destroy(sqt_ctx *c) {
    if (!c) return SQT_OK;
    cudaSetDevice(c->device);
    if (c->comm && nccl_api()->lib && !c->comm_broken) nccl_api()->CommDestroy(c->comm);
    for (auto &ev : c->ev) if (ev) cudaEventDestroy(ev);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;                           // the buffers free themselves, on c->device
    return SQT_OK;
}

extern "C" int sqt_device_info(sqt_ctx *c, int *sm_count, int *cc_major, int *cc_minor, char name_out[128]) {
    if (!c) return SQT_E_INVALID;
    if (sm_count) *sm_count = c->sm_count;
    if (cc_major) *cc_major = c->cc_major;
    if (cc_minor) *cc_minor = c->cc_minor;
    if (name_out) snprintf(name_out, 128, "%s", c->name);
    return SQT_OK;
}

// ------------------------------------------------------------------------------ scene upload
// Host: one iterative walk over the boundary tree (sqt_layout.hpp) validates it and derives the 16-byte device nodes and
// the clipped boxes (BIH.hs:130-141; plane values are copied, never computed).  Meanwhile a helper thread streams the
// triangle array -- the bulk of a large scene -- to every context of the call through two pinned staging buffers.
// Device: k_leaf_records derives the leaf records from the triangles, k_check_materials validates the material indices.
// Device allocations are kept and reused while the new scene fits them.
static double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// branches, leaves, triangles (48 bytes each) and materials (three float4 each)
static int ensure_scene_capacity(sqt_ctx *ctx, size_t n_br, size_t n_lf, size_t n_tris, size_t n_mats) {
    CU(ctx->d_nodes.ensure(n_br)); CU(ctx->d_boxes.ensure(2 * n_br));
    CU(ctx->d_slabs.ensure(n_br)); CU(ctx->d_tight.ensure(2 * n_br));
    CU(ctx->d_levels.ensure(n_br));
    CU(ctx->d_leaves.ensure(2 * n_lf)); CU(ctx->d_ranges.ensure(n_lf));
    CU(ctx->d_tris.ensure(3 * n_tris));
    CU(ctx->d_mats.ensure(3 * n_mats));
    return SQT_OK;
}

// triangles -> every context, chunk by chunk through two pinned buffers (runs on a helper thread)
static void stream_tris(sqt_ctx **ctxs, int n, const sqt_tri *tris, size_t n_tris, std::atomic<int> *status, std::string *err) {
    const size_t CH = (size_t)32 << 20, bytes = n_tris * 48;
    Pinned<char> pin[2];
    std::vector<cudaEvent_t> done(2 * (size_t)n);
    auto bail = [&](cudaError_t e, const char *what) { *err = std::string(what) + ": " + cudaGetErrorString(e); status->store(SQT_E_CUDA); };
    cudaError_t e = cudaSuccess;
    bool have_ev = false;
    do {
        if (bytes == 0) break;
        const size_t buf = bytes < CH ? bytes : CH;
        if ((e = cudaSetDevice(ctxs[0]->device)) != cudaSuccess) { bail(e, "cudaSetDevice"); break; }
        if ((e = pin[0].ensure(buf)) != cudaSuccess || (bytes > CH && (e = pin[1].ensure(buf)) != cudaSuccess)) { bail(e, "cudaMallocHost (staging)"); break; }
        for (int g = 0; g < n && e == cudaSuccess; ++g) { cudaSetDevice(ctxs[g]->device); for (int b = 0; b < 2 && e == cudaSuccess; ++b) e = cudaEventCreateWithFlags(&done[2 * g + b], cudaEventDisableTiming); }
        if (e != cudaSuccess) { bail(e, "cudaEventCreate"); break; }
        have_ev = true;
        size_t off = 0;
        for (int it = 0; off < bytes; ++it) {
            const int b = it & 1;
            const size_t len = bytes - off < CH ? bytes - off : CH;
            if (it >= 2) for (int g = 0; g < n; ++g) { cudaSetDevice(ctxs[g]->device); if ((e = cudaEventSynchronize(done[2 * g + b])) != cudaSuccess) break; }
            if (e != cudaSuccess) { bail(e, "cudaEventSynchronize"); break; }
            memcpy(pin[b], (const char *)tris + off, len);
            for (int g = 0; g < n; ++g) {
                cudaSetDevice(ctxs[g]->device);
                if ((e = cudaMemcpyAsync((char *)ctxs[g]->d_tris.p + off, pin[b], len, cudaMemcpyHostToDevice, ctxs[g]->stream)) != cudaSuccess) break;
                if ((e = cudaEventRecord(done[2 * g + b], ctxs[g]->stream)) != cudaSuccess) break;
            }
            if (e != cudaSuccess) { bail(e, "cudaMemcpyAsync (triangles)"); break; }
            off += len;
        }
        for (int g = 0; g < n; ++g) { cudaSetDevice(ctxs[g]->device); cudaStreamSynchronize(ctxs[g]->stream); }
    } while (false);
    if (have_ev) for (int g = 0; g < n; ++g) { cudaSetDevice(ctxs[g]->device); for (int b = 0; b < 2; ++b) cudaEventDestroy(done[2 * g + b]); }
}

static int upload_scene_to(sqt_ctx **ctxs, int n, const sqt_scene_desc *s) {
    sqt_ctx *ctx = ctxs[0];
    const double t0 = now_ms();
    for (int g = 0; g < n; ++g) ctxs[g]->prog.on = false;       // a new scene ends a progressive frame
    if (!s->nodes || s->n_nodes == 0) return fail(ctx, SQT_E_INVALID, "scene has no BIH nodes");
    if (s->n_tris && !s->tris) return fail(ctx, SQT_E_INVALID, "tris is NULL");
    if (s->n_tris >= (1u << 27) || s->n_nodes >= (1u << 27)) return fail(ctx, SQT_E_UNSUPPORTED, "scene too large for the 27-bit indices");
    uint32_t n_br = 0, n_lf = 0;
    for (uint32_t i = 0; i < s->n_nodes; ++i) { if (s->nodes[i].b & SQT_NODE_LEAF) ++n_lf; else ++n_br; }
    for (int g = 0; g < n; ++g) {
        sqt_ctx *c = ctxs[g];
        cudaSetDevice(c->device);
        c->has_scene = false;
        const int rc = ensure_scene_capacity(c, n_br ? n_br : 1, n_lf ? n_lf : 1, s->n_tris ? s->n_tris : 1, s->n_mats ? s->n_mats : 1);
        if (rc) { if (g) ctx->err = c->err; return rc; }
    }
    // the triangles start to flow while the host walks the tree
    std::atomic<int> tri_status{0};
    std::string tri_err;
    std::thread streamer(stream_tris, ctxs, n, s->tris, (size_t)s->n_tris, &tri_status, &tri_err);
    DeviceLayout lay;
    std::string lerr;
    const int lrc = build_device_layout(*s, lay, lerr, /*check_materials=*/false);
    const double t1 = now_ms();
    streamer.join();
    if (lrc) return fail(ctx, lrc, "%s", lerr.c_str());
    if (tri_status.load()) return fail(ctx, tri_status.load(), "%s", tri_err.c_str());
    std::vector<uint2> ranges(lay.leaf_first.size());
    for (size_t k = 0; k < ranges.size(); ++k) ranges[k] = make_uint2(lay.leaf_first[k], lay.leaf_count[k]);
    // branches sorted by depth (counting sort): the bottom-up pass of the subtree slabs runs one launch per level
    std::vector<uint32_t> level_off(lay.height + 2, 0u), level_nodes(lay.n_branches ? lay.n_branches : 1);
    for (uint32_t b = 0; b < lay.n_branches; ++b) level_off[lay.branch_depth[b] + 1]++;
    for (size_t d = 1; d < level_off.size(); ++d) level_off[d] += level_off[d - 1];
    {
        std::vector<uint32_t> fill(level_off.begin(), level_off.end() - 1);
        for (uint32_t b = 0; b < lay.n_branches; ++b) level_nodes[fill[lay.branch_depth[b]]++] = b;
    }
    const uint32_t n_leaves = n_lf;
    for (int g = 0; g < n; ++g) {
        sqt_ctx *c = ctxs[g];
        sqt_ctx *ctx = c;       // CU() reports into this context
        CU(cudaSetDevice(c->device));
        cudaStream_t st = c->stream;
        const uint32_t init_flag[2] = {0xffffffffu, 0u};
        CU(cudaMemcpyAsync(c->d_flag, init_flag, sizeof init_flag, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(c->d_nodes, lay.nodes.data(), lay.nodes.size() * sizeof(float4), cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(c->d_boxes, lay.boxes.data(), lay.boxes.size() * sizeof(float4), cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(c->d_mats, lay.mats.data(), lay.mats.size() * sizeof(float4), cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(c->d_ranges, ranges.data(), ranges.size() * sizeof(uint2), cudaMemcpyHostToDevice, st));
        if (n_leaves) {
            k_leaf_records<<<(n_leaves + 255) / 256, 256, 0, st>>>(c->d_tris, c->d_ranges, n_leaves, c->d_leaves);
            CU(cudaGetLastError());
        }
        if (s->n_tris) {
            k_check_materials<<<(s->n_tris + 255) / 256, 256, 0, st>>>(c->d_tris, s->n_tris, s->n_mats, c->d_flag);
            CU(cudaGetLastError());
        }
        if (lay.n_branches) {
            CU(cudaMemcpyAsync(c->d_levels, level_nodes.data(), (size_t)lay.n_branches * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
            for (uint32_t d = lay.height; d >= 1; --d) {                      // deepest level first
                const uint32_t lo = level_off[d], cnt = level_off[d + 1] - lo;
                if (!cnt) continue;
                k_branch_tight<<<(cnt + 255) / 256, 256, 0, st>>>(c->d_levels + lo, cnt, c->d_nodes, c->d_leaves, c->d_tight);
                CU(cudaGetLastError());
            }
            k_child_slabs<<<(lay.n_branches + 255) / 256, 256, 0, st>>>(c->d_nodes, lay.n_branches, c->d_boxes, c->d_tight, c->d_leaves, lay.s_max, lay.c_max, c->slab_ratio, c->slab_ratio_leaf, c->d_slabs);
            k_flag_slabs<<<(lay.n_branches + 255) / 256, 256, 0, st>>>(c->d_nodes, lay.n_branches, c->d_slabs);
            CU(cudaGetLastError());
        }
    }
    for (int g = 0; g < n; ++g) {
        sqt_ctx *c = ctxs[g];
        sqt_ctx *ctx = c;
        CU(cudaSetDevice(c->device));
        uint32_t flag[2] = {0, 0};
        CU(cudaMemcpyAsync(flag, c->d_flag, sizeof flag, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        if (flag[0] != 0xffffffffu) return fail(ctxs[0], SQT_E_INVALID, "triangle %u: material %u out of range", flag[0], s->tris[flag[0]].material);
        SceneView v = {};
        v.nodes = c->d_nodes; v.boxes = c->d_boxes; v.tris = c->d_tris; v.mats = c->d_mats; v.leaves = c->d_leaves; v.slabs = c->d_slabs;
        for (int k = 0; k < 3; ++k) v.tame_c[k] = lay.tame_c[k];
        v.tame_r = lay.tame_r;
        v.leaf_cull = (uint32_t)c->leaf_cull;
        for (int k = 0; k < 3; ++k) { v.root_lo[k] = s->root_bounds[k]; v.root_hi[k] = s->root_bounds[3 + k]; }
        v.n_branches = lay.n_branches; v.n_tris = s->n_tris; v.n_mats = s->n_mats;
        v.root_is_leaf = (s->nodes[0].b & SQT_NODE_LEAF) ? 1u : 0u;
        v.planes_finite = (uint32_t)lay.planes_finite;
        c->sc = v; c->has_scene = true; c->terminate_on_black_ok = lay.terminate_on_black_ok; c->tree_height = lay.height;
        c->upload_bytes = (uint64_t)s->n_tris * 48 + lay.nodes.size() * 16 + lay.boxes.size() * 16 + lay.mats.size() * 16 + ranges.size() * 8 + (uint64_t)lay.n_branches * 4 + 8;
        c->upload_layout_ms = t1 - t0;
        c->upload_ms = now_ms() - t0;
    }
    return SQT_OK;
}

extern "C" int sqt_upload_scene(sqt_ctx *ctx, const sqt_scene_desc *s) {
    if (!ctx || !s) return SQT_E_INVALID;
    return upload_scene_to(&ctx, 1, s);
}

// a group call's context array: n >= 1 contexts, none of them NULL
static bool valid_group(sqt_ctx **ctxs, int n) {
    if (!ctxs || n < 1) return false;
    for (int i = 0; i < n; ++i) if (!ctxs[i]) return false;
    return true;
}

// the same scene onto every context of a single-process group: the tree is walked once, every staged chunk of
// triangles goes to all devices
extern "C" int sqt_upload_scene_group(sqt_ctx **ctxs, int n, const sqt_scene_desc *s) {
    if (!valid_group(ctxs, n) || !s) return SQT_E_INVALID;
    return upload_scene_to(ctxs, n, s);
}

extern "C" int sqt_last_upload(const sqt_ctx *ctx, uint64_t *h2d_bytes, double *wall_ms, double *host_layout_ms) {
    if (!ctx) return SQT_E_INVALID;
    if (h2d_bytes) *h2d_bytes = ctx->upload_bytes;
    if (wall_ms) *wall_ms = ctx->upload_ms;
    if (host_layout_ms) *host_layout_ms = ctx->upload_layout_ms;
    return SQT_OK;
}

// extension: analytic spheres (include/sqt.h)
extern "C" int sqt_upload_spheres(sqt_ctx *ctx, const sqt_sphere *sp, uint32_t n) {
    if (!ctx) return SQT_E_INVALID;
    ctx->prog.on = false;
    if (!ctx->has_scene) return fail(ctx, SQT_E_NO_SCENE, "sqt_upload_spheres before sqt_upload_scene");
    if (n && !sp) return fail(ctx, SQT_E_INVALID, "spheres is NULL");
    if ((uint64_t)ctx->sc.n_tris + n >= (1u << 27)) return fail(ctx, SQT_E_UNSUPPORTED, "too many surfaces");
    CU(cudaSetDevice(ctx->device));
    std::vector<float4> ds((size_t)2 * (n ? n : 1));
    for (uint32_t k = 0; k < n; ++k) {
        if (sp[k].material >= ctx->sc.n_mats) return fail(ctx, SQT_E_INVALID, "sphere %u: material %u out of range", k, sp[k].material);
        if (!(sp[k].radius > 0.0f)) return fail(ctx, SQT_E_INVALID, "sphere %u: radius must be positive", k);
        ds[2 * k] = make_float4(sp[k].center[0], sp[k].center[1], sp[k].center[2], sp[k].radius);
        ds[2 * k + 1] = make_float4(u2f(sp[k].material), 0.0f, 0.0f, 0.0f);
    }
    ctx->d_spheres.reset(0); ctx->d_sph_nodes.reset(0); ctx->d_sph_order.reset(0);
    ctx->sc.spheres = nullptr; ctx->sc.sph_nodes = nullptr; ctx->sc.sph_order = nullptr; ctx->sc.n_spheres = 0;
    if (n == 0) return SQT_OK;
    CU(ctx->d_spheres.reset(ds.size()));
    CU(cudaMemcpy(ctx->d_spheres, ds.data(), ds.size() * sizeof(float4), cudaMemcpyHostToDevice));
    ctx->sc.spheres = ctx->d_spheres; ctx->sc.n_spheres = n;
    // a hierarchy over the spheres (sphere_step): only for finite, moderate coordinates -- the culling bound assumes no overflow
    bool tame = ctx->sphere_bvh != 0;
    for (uint32_t k = 0; k < n && tame; ++k)
        for (int q = 0; q < 4; ++q) { const float v = q < 3 ? sp[k].center[q] : sp[k].radius; if (!(fabsf(v) < 1.0e12f)) tame = false; }
    if (tame) {
        SphereBvh bvh;
        build_sphere_bvh(sp, n, bvh);
        CU(ctx->d_sph_nodes.reset(bvh.nodes.size()));
        CU(ctx->d_sph_order.reset(bvh.order.size()));
        CU(cudaMemcpy(ctx->d_sph_nodes, bvh.nodes.data(), bvh.nodes.size() * sizeof(float4), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(ctx->d_sph_order, bvh.order.data(), bvh.order.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
        ctx->sc.sph_nodes = ctx->d_sph_nodes; ctx->sc.sph_order = ctx->d_sph_order;
    }
    return SQT_OK;
}

extern "C" int sqt_set_option(sqt_ctx *ctx, int option, int value) {
    if (!ctx) return SQT_E_INVALID;
    if (option == SQT_OPT_LEAF_CULL) { ctx->leaf_cull = value ? 1 : 0; ctx->sc.leaf_cull = (uint32_t)ctx->leaf_cull; return SQT_OK; }
    if (option == SQT_OPT_SPHERE_BVH) {          // takes effect at the next sqt_upload_spheres; 0 = test every sphere for every ray (the definition)
        ctx->sphere_bvh = value ? 1 : 0;
        if (!value) { ctx->sc.sph_nodes = nullptr; ctx->sc.sph_order = nullptr; }
        return SQT_OK;
    }
    return fail(ctx, SQT_E_INVALID, "unknown option %d", option);
}

extern "C" int sqt_set_lens(sqt_ctx *ctx, const sqt_lens *l) {
    if (!ctx) return SQT_E_INVALID;
    if (!l) { ctx->lens_set = false; ctx->lens = sqt_lens{}; return SQT_OK; }
    if (l->jitter > 1u) return fail(ctx, SQT_E_INVALID, "sqt_set_lens: jitter must be 0 or 1");
    if (!(l->aperture_radius >= 0.0f) || !(l->aperture_radius < INFINITY)) return fail(ctx, SQT_E_INVALID, "sqt_set_lens: aperture_radius must be >= 0 and finite");
    if (!(l->focus_distance > 0.0f) || !(l->focus_distance < INFINITY)) return fail(ctx, SQT_E_INVALID, "sqt_set_lens: focus_distance must be > 0 and finite");
    if (l->reserved) return fail(ctx, SQT_E_INVALID, "sqt_set_lens: reserved must be 0");
    ctx->lens = *l; ctx->lens_set = true;
    return SQT_OK;
}

// ------------------------------------------------------------------------------ helpers
// the device buffers of an image of npix pixels (the pixel list has 32 entries of slack)
static int ensure_image(sqt_ctx *ctx, long long npix) {
    CU(ctx->d_prim.ensure(npix));
    CU(ctx->d_pixel_list.ensure(npix + 32));
    CU(ctx->d_accum.ensure(npix * 3));
    CU(ctx->d_rgb8.ensure(npix * 3));
    return SQT_OK;
}
// the pinned staging of an image's RGB8 and sums (also of the moments and the sample counts)
static int ensure_host_image(sqt_ctx *ctx, long long npix) {
    CU(ctx->h_rgb8.ensure(npix * 3));
    CU(ctx->h_accum.ensure(npix * 3));
    return SQT_OK;
}
// persistent launch: as many 128-lane CTAs as stay resident on the 148 SMs (never more than the work needs)
template <class K>
static int persistent_grid(sqt_ctx *ctx, K kernel, long long nwork) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 128, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
    long long grid = (long long)ctx->sm_count * per_sm, want = (nwork + 127) / 128;
    if (want < grid) grid = want ? want : 1;
    return (int)grid;
}
// k_paths_pool launch shape + the per-slot global state it needs.  `launch` false: only size the grid and make sure the
// allocations exist (the pre-pass of a render, so that nothing can fail between the ranks' agreement and the collective).
template <bool COUNT, bool LENS>
static int pool_step(sqt_ctx *ctx, const RenderParams &d, const RoundInfo &rd, int round, long long nitems, bool launch) {
    const size_t smem = kPoolSmemBytes;
    auto kern = k_paths_pool<COUNT, LENS>;
    if (smem > 48 * 1024) CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 128, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
    long long grid = (long long)ctx->sm_count * per_sm, want = (nitems + kPoolSlots - 1) / kPoolSlots;
    if (want < grid) grid = want ? want : 1;
    const long long slots = grid * kPoolSlots;
    // a ray's stack holds at most one 16-byte entry per branch on a root-to-leaf path; the stacks of a warp's slots are
    // interleaved entry by entry, so the few entries in use of all resident slots share cache lines and stay in L2
    int depth = (int)ctx->tree_height;
    if (depth > kStackEntries) depth = kStackEntries;
    if (depth < 1) depth = 1;
    // the per-path material list of a slot: max_depth entries, packed (16-byte granules) for the same reason
    int pm_stride = (d.max_depth + 7) & ~7;
    if (pm_stride > SQT_MAX_DEPTH) pm_stride = SQT_MAX_DEPTH;
    // d_gpath holds two entries per slot, so its capacity tells the slot capacity; it is emptied first, so that after a
    // failed allocation the next call allocates all three again
    if (slots > (long long)ctx->d_gpath.cap / 2 || slots * depth > (long long)ctx->d_gstack.cap) {
        const long long cap = (long long)ctx->sm_count * 16 * kPoolSlots > slots ? (long long)ctx->sm_count * 16 * kPoolSlots : slots;
        ctx->d_gpath.reset(0);
        CU(ctx->d_gstack.reset(cap * depth));
        CU(ctx->d_gpm.reset(cap * SQT_MAX_DEPTH));
        CU(ctx->d_gpath.reset(cap * 2));
    }
    if (!launch) return SQT_OK;
    kern<<<(int)grid, 128, smem, ctx->stream>>>(ctx->sc, d, rd, round, ctx->d_stats, ctx->pool_tune, ctx->d_gstack, ctx->d_gpm, ctx->d_gpath, depth, pm_stride);
    CU(cudaGetLastError());
    return SQT_OK;
}
// the pool kernel of a frame: instrumented or not, lens frame (the sample's own primary ray) or pinhole
static int pool_step_d(sqt_ctx *ctx, bool count, const RenderParams &d, const RoundInfo &rd, int round, long long nitems, bool launch) {
    if (d.lens) return count ? pool_step<true, true>(ctx, d, rd, round, nitems, launch) : pool_step<false, true>(ctx, d, rd, round, nitems, launch);
    return count ? pool_step<true, false>(ctx, d, rd, round, nitems, launch) : pool_step<false, false>(ctx, d, rd, round, nitems, launch);
}
static float ev_ms(cudaEvent_t a, cudaEvent_t b) { float ms = 0; cudaEventElapsedTime(&ms, a, b); return ms; }

// ------------------------------------------------------------------------------ intersect_batch
extern "C" int sqt_intersect_batch(sqt_ctx *ctx, const float *org, const float *dir, int64_t n, int32_t *tri_out,
                                   float *dist_out, float *point_out, sqt_stats *stats) {
    if (!ctx) return SQT_E_INVALID;
    if (!ctx->has_scene) return fail(ctx, SQT_E_NO_SCENE, "sqt_intersect_batch before sqt_upload_scene");
    if (n < 0 || (n > 0 && (!org || !dir || !tri_out))) return fail(ctx, SQT_E_INVALID, "bad batch arguments");
    if (stats) memset(stats, 0, sizeof *stats);
    if (n == 0) return SQT_OK;
    CU(cudaSetDevice(ctx->device));
    CU(ctx->d_org.ensure(n * 3)); CU(ctx->d_dir.ensure(n * 3));
    CU(ctx->d_dist.ensure(n)); CU(ctx->d_point.ensure(n * 3));
    CU(ctx->d_tri.ensure(n));
    cudaStream_t st = ctx->stream;
    CU(cudaEventRecord(ctx->ev[0], st));
    CU(cudaMemcpyAsync(ctx->d_org, org, (size_t)n * 12, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ctx->d_dir, dir, (size_t)n * 12, cudaMemcpyHostToDevice, st));
    // the counters only: n_hit is the pixel list of a progressive frame's primary pass, which this call does not end
    CU(cudaMemsetAsync(ctx->d_stats, 0, offsetof(DeviceStats, n_hit), st));
    CU(cudaEventRecord(ctx->ev[1], st));
    if (stats)      // instrumented variant: fills the visit/test counters
        k_intersect_batch<true><<<persistent_grid(ctx, k_intersect_batch<true>, n), 128, 0, st>>>(
            ctx->sc, ctx->d_org, ctx->d_dir, n, ctx->d_tri, dist_out ? ctx->d_dist.p : nullptr, point_out ? ctx->d_point.p : nullptr,
            ctx->d_stats, ctx->tune);
    else
        k_intersect_batch<false><<<persistent_grid(ctx, k_intersect_batch<false>, n), 128, 0, st>>>(
            ctx->sc, ctx->d_org, ctx->d_dir, n, ctx->d_tri, dist_out ? ctx->d_dist.p : nullptr, point_out ? ctx->d_point.p : nullptr,
            ctx->d_stats, ctx->tune);
    CU(cudaGetLastError());
    CU(cudaEventRecord(ctx->ev[2], st));
    CU(cudaMemcpyAsync(tri_out, ctx->d_tri, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    if (dist_out) CU(cudaMemcpyAsync(dist_out, ctx->d_dist, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    if (point_out) CU(cudaMemcpyAsync(point_out, ctx->d_point, (size_t)n * 12, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(ctx->h_stats, ctx->d_stats, sizeof(DeviceStats), cudaMemcpyDeviceToHost, st));
    CU(cudaEventRecord(ctx->ev[3], st));
    CU(cudaStreamSynchronize(st));
    if (stats) {
        stats->h2d_ms = ev_ms(ctx->ev[0], ctx->ev[1]); stats->device_ms = ev_ms(ctx->ev[1], ctx->ev[2]);
        stats->d2h_ms = ev_ms(ctx->ev[2], ctx->ev[3]);
        stats->rays_traced = ctx->h_stats->rays; stats->rays_reference = ctx->h_stats->rays;
        stats->branch_visits = ctx->h_stats->branch_visits; stats->child_box_tests = ctx->h_stats->child_box_tests;
        stats->tri_tests = ctx->h_stats->tri_tests; stats->leaves_culled = ctx->h_stats->leaves_culled;
        stats->mt_pass_a = ctx->h_stats->mt_pass_a; stats->mt_pass_u = ctx->h_stats->mt_pass_u;
        stats->mt_pass_v = ctx->h_stats->mt_pass_v; stats->mt_accept = ctx->h_stats->mt_accept;
        stats->h2d_bytes = (uint64_t)n * 24; stats->d2h_bytes = (uint64_t)n * (4 + (dist_out ? 4 : 0) + (point_out ? 12 : 0));
        stats->kernel_launches = 1;
    }
    return SQT_OK;
}

// ------------------------------------------------------------------------------ render
static int check_params(sqt_ctx *ctx, const sqt_camera *cam, const sqt_render_params *p) {
    if (!cam || !p) return fail(ctx, SQT_E_INVALID, "cam/params is NULL");
    if (!ctx->has_scene) return fail(ctx, SQT_E_NO_SCENE, "sqt_render before sqt_upload_scene");
    if (p->rows <= 0 || p->cols <= 0 || p->xdiv <= 0 || p->ydiv <= 0 || p->spp <= 0)
        return fail(ctx, SQT_E_INVALID, "rows/cols/xdiv/ydiv/spp must be positive");
    if (p->max_depth < 1 || p->max_depth > SQT_MAX_DEPTH) return fail(ctx, SQT_E_UNSUPPORTED, "max_depth must be in 1..%d", SQT_MAX_DEPTH);
    if (p->mode != 0 && p->mode != 1) return fail(ctx, SQT_E_INVALID, "mode must be 0 (trace) or 1 (cast)");
    if ((long long)p->rows * p->cols > (1ll << 31)) return fail(ctx, SQT_E_UNSUPPORTED, "image too large");
    if (ctx->lens_set && p->mode == 1) return fail(ctx, SQT_E_UNSUPPORTED, "cast mode (mode 1) has no lens: sqt_set_lens(ctx, NULL) first");
    return SQT_OK;
}

static RenderParams to_device_params(const sqt_ctx *ctx, const sqt_camera *cam, const sqt_render_params *p) {
    RenderParams d = {};
    d.rows = p->rows; d.cols = p->cols; d.xdiv = p->xdiv; d.ydiv = p->ydiv; d.seed_stride = p->seed_stride;
    d.spp = p->spp; d.max_depth = p->max_depth; d.mode = p->mode; d.seed = p->seed;
    d.rank = ctx->rank; d.world = ctx->world; d.split_samples = (p->flags & SQT_F_SPLIT_SAMPLES) ? 1 : 0;
    d.primary_reuse = (p->flags & SQT_F_NO_PRIMARY_REUSE) ? 0 : 1;
    for (int k = 0; k < 3; ++k) d.cam_pos[k] = cam->position[k];
    for (int k = 0; k < 9; ++k) d.cam_rot[k] = cam->rotation[k];
    d.terminate_on_black = (ctx->terminate_on_black_ok && !(p->flags & SQT_F_NO_EARLY_TERMINATION)) ? 1 : 0;
    if (ctx->lens_set) {                // every sample traces its own primary ray: no primary pass, no reuse
        d.lens = 1; d.jitter = (int)ctx->lens.jitter; d.aperture = ctx->lens.aperture_radius; d.focus = ctx->lens.focus_distance;
        d.primary_reuse = 0;
    }
    return d;
}

// Everything of a render that can fail for lack of memory or because of its arguments, done BEFORE any kernel or
// collective is enqueued: image buffers, the sample buffer of a round, the pool slots' global state.
static int prepare_render(sqt_ctx *ctx, const RenderParams &d, bool count, bool host_image, RenderPlan &pl) {
    const long long npix = (long long)d.rows * d.cols;
    int rc = ensure_image(ctx, npix); if (rc) return rc;
    if (host_image) { rc = ensure_host_image(ctx, npix); if (rc) return rc; }
    pl.nwork = work_items(d);
    if (d.mode == 1) return SQT_OK;
    sample_range(d, pl.k0, pl.k1);
    pl.log2_s = round_log2_s(pl.nwork, pl.k1 - pl.k0 > 0 ? pl.k1 - pl.k0 : 1, ctx->sbuf_budget);
    const int S = 1 << pl.log2_s;
    if ((pl.k1 - pl.k0 + S - 1) / S > 256) return fail(ctx, SQT_E_UNSUPPORTED, "more than 256 sample rounds (raise SQT_SBUF_MB)");
    pl.sbytes = pl.nwork * (long long)S * 12ll;
    CU(ctx->d_sbuf.ensure((pl.sbytes > 0 ? pl.sbytes : 12) / sizeof(float)));
    RoundInfo none = {};
    return pool_step_d(ctx, count, d, none, 0, pl.nwork << pl.log2_s, false);
}

// Multi-rank contexts: all ranks learn whether every rank got through check_params + prepare_render, with a one-word
// ncclAllReduce(max) -- a collective every rank reaches whatever happened to it locally.  Only if all agree is the
// frame (and its ncclReduce) enqueued; otherwise every rank returns an error and nobody waits in a collective.
// `keys` (the lens; progressive frames: samples done, target spp, end of the chunk) must be equal on every rank: each
// travels as (v, -v) in the same all-reduce, so max(v) == -max(-v) holds exactly when all ranks agree.
static int group_agree(sqt_ctx *ctx, int rc_local, const int32_t *keys = nullptr, int n_keys = 0) {
    if (ctx->world <= 1 || !ctx->comm) return rc_local;
    if (ctx->comm_broken) return fail(ctx, SQT_E_NCCL, "the communicator of this group was aborted after an earlier failure");
    NcclApi *na = nccl_api();
    const std::string local_err = ctx->err;
    cudaSetDevice(ctx->device);
    uint32_t *flag = ctx->d_flag + 1;
    const int nw = 1 + 2 * n_keys;
    uint32_t v[kFlagWords - 1] = {rc_local ? 1u : 0u}, out[kFlagWords - 1] = {1u};
    for (int i = 0; i < n_keys; ++i) { v[1 + 2 * i] = (uint32_t)keys[i]; v[2 + 2 * i] = (uint32_t)(-keys[i]); }
    cudaError_t e = cudaMemcpyAsync(flag, v, nw * 4, cudaMemcpyHostToDevice, ctx->stream);
    ncclResult_t r = e == cudaSuccess ? na->AllReduce(flag, flag, nw, kNcclInt32, kNcclMax, ctx->comm, ctx->stream) : 1;
    if (r == 0) e = cudaMemcpyAsync(out, flag, nw * 4, cudaMemcpyDeviceToHost, ctx->stream);
    if (r == 0 && e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (r != 0 || e != cudaSuccess) {
        na->CommAbort(ctx->comm); ctx->comm_broken = true;
        return fail(ctx, SQT_E_NCCL, "group agreement failed (%s); communicator aborted", r ? na->GetErrorString(r) : cudaGetErrorString(e));
    }
    if (rc_local) { ctx->err = local_err; return rc_local; }
    if (out[0]) return fail(ctx, SQT_E_NCCL, "another rank of the group could not start this render; nothing was enqueued");
    for (int i = 0; i < n_keys; ++i)
        if ((int32_t)out[1 + 2 * i] != -(int32_t)out[2 + 2 * i])
            return fail(ctx, SQT_E_INVALID, "the ranks of the group disagree on the frame (samples done / target spp / chunk / criteria / lens); nothing was enqueued");
    return SQT_OK;
}
// a failure after the agreement (a launch error) would leave the other ranks waiting in ncclReduce: abort the communicator
// the lens as agreement keys: (set?, jitter, aperture bits, focus bits)
static void lens_keys(const sqt_ctx *ctx, int32_t keys[4]) {
    uint32_t a = 0, f = 0;
    memcpy(&a, &ctx->lens.aperture_radius, 4); memcpy(&f, &ctx->lens.focus_distance, 4);
    keys[0] = ctx->lens_set ? 1 : 0; keys[1] = ctx->lens_set ? (int32_t)ctx->lens.jitter : 0;
    keys[2] = ctx->lens_set ? (int32_t)a : 0; keys[3] = ctx->lens_set ? (int32_t)f : 0;
}
static int group_abort(sqt_ctx *ctx, int rc) {
    if (rc && ctx->world > 1 && ctx->comm && !ctx->comm_broken) { nccl_api()->CommAbort(ctx->comm); ctx->comm_broken = true; }
    return rc;
}

// Enqueue the kernels of a render on ctx->stream (no host sync, no allocation), in three stages: frame start, sample
// rounds, finish.  A one-shot frame is start + rounds [k0, k1) + finish; a progressive frame runs the start once and
// rounds + finish once per chunk.  Events: 0 start, 1 after primary, 2 after paths, 3 after reduce, 4 after tonemap.

// the pixels among the nwork work items of this rank: all but the padding of the last pixel group, which is their tail
static long long owned_pixels(const RenderParams &d, long long nwork) {
    const long long npix = (long long)d.rows * d.cols;
    if (d.world <= 1 || d.split_samples) return npix;
    const long long groups = (npix + 31) >> 5;
    return (groups - 1) % d.world == d.rank ? nwork - (groups * 32 - npix) : nwork;
}

// frame start: zero the stats and the sums, the primary pass -- or, in a lens frame, the pixel list of every owned pixel
static int enqueue_start(sqt_ctx *ctx, const RenderParams &d, bool count, const RenderPlan &pl, uint32_t &nl) {
    const long long npix = (long long)d.rows * d.cols;
    cudaStream_t st = ctx->stream;
    CU(cudaMemsetAsync(ctx->d_stats, 0, sizeof(DeviceStats), st));
    CU(cudaMemsetAsync(ctx->d_accum, 0, (size_t)npix * 3 * sizeof(float), st));
    CU(cudaEventRecord(ctx->ev[0], st));
    if (d.mode == 0 && d.primary_reuse) {
        if (count) k_primary<true><<<persistent_grid(ctx, k_primary<true>, pl.nwork), 128, 0, st>>>(ctx->sc, d, ctx->d_prim, ctx->d_pixel_list, ctx->d_stats, ctx->tune);
        else k_primary<false><<<persistent_grid(ctx, k_primary<false>, pl.nwork), 128, 0, st>>>(ctx->sc, d, ctx->d_prim, ctx->d_pixel_list, ctx->d_stats, ctx->tune);
        CU(cudaGetLastError()); nl++;
    } else if (d.mode == 0 && d.lens) {
        const long long n = owned_pixels(d, pl.nwork);
        const long long blocks = (n + 255) / 256 < (long long)ctx->sm_count * 8 ? (n + 255) / 256 : (long long)ctx->sm_count * 8;
        k_lens_list<<<blocks > 0 ? (int)blocks : 1, 256, 0, st>>>(d, n, ctx->d_pixel_list, ctx->d_stats);
        CU(cudaGetLastError()); nl++;
    }
    CU(cudaEventRecord(ctx->ev[1], st));
    return SQT_OK;
}

// samples [ka, kb) of `nwork` slots in rounds of S = 1 << log2_s samples per pixel: trace (persistent lanes, one work
// counter per round, numbered from 0 in every call), then add in sample order -- onto the sums alone (m2 == nullptr) or
// the sums and the second moments.  nwork, log2_s: the plan's, or an adaptive frame's active slots (sqt_render_advance).
static int enqueue_rounds(sqt_ctx *ctx, const RenderParams &d, bool count, long long nwork, int log2_s, int ka, int kb, float *m2, uint32_t &nl) {
    cudaStream_t st = ctx->stream;
    if (d.mode == 1) {
        if (count) k_raycast<true><<<persistent_grid(ctx, k_raycast<true>, nwork), 128, 0, st>>>(ctx->sc, d, ctx->d_accum, ctx->d_stats, ctx->tune);
        else k_raycast<false><<<persistent_grid(ctx, k_raycast<false>, nwork), 128, 0, st>>>(ctx->sc, d, ctx->d_accum, ctx->d_stats, ctx->tune);
        CU(cudaGetLastError()); nl++;
        return SQT_OK;
    }
    RoundInfo rd = {};
    rd.pixel_list = d.primary_reuse || d.lens ? ctx->d_pixel_list.p : nullptr;
    rd.prim = d.primary_reuse ? ctx->d_prim.p : nullptr;
    rd.n_slots = nwork; rd.slot_stride = nwork;
    rd.log2_s = log2_s;
    const int S = 1 << rd.log2_s;
    rd.sbuf = ctx->d_sbuf;
    const int agrid = (int)((nwork + 255) / 256 < (long long)ctx->sm_count * 8 ? (nwork + 255) / 256 : (long long)ctx->sm_count * 8);
    int round = 0;
    for (int k = ka; k < kb; k += S, ++round) {
        rd.k0 = k; rd.k1 = k + S < kb ? k + S : kb;
        CU(cudaMemsetAsync(ctx->d_sbuf, 0, (size_t)(nwork * (long long)(rd.k1 - rd.k0) * 12ll), st));
        const int rc = pool_step_d(ctx, count, d, rd, round, nwork << rd.log2_s, true);
        if (rc) return rc;
        nl++;
        if (m2) k_accumulate_m2<<<agrid > 0 ? agrid : 1, 256, 0, st>>>(d, rd, ctx->d_accum, m2, ctx->d_stats);
        else k_accumulate<<<agrid > 0 ? agrid : 1, 256, 0, st>>>(d, rd, ctx->d_accum, ctx->d_stats);
        CU(cudaGetLastError()); nl++;
    }
    return SQT_OK;
}

// finish: the sums of all ranks onto rank 0 -- in place for a one-shot frame (sum1 == d_accum, no moments), into
// rank 0's separate buffers for a progressive one (the ranks' running sums must survive the next reduce) -- then the
// tone map with `inv` and, for a progressive frame after k samples, the noise estimate, both on rank 0; counts: the
// per-pixel sample counts of an adaptive frame (nullptr: every pixel has k samples)
static int enqueue_finish(sqt_ctx *ctx, long long npix, float inv, float *sum1, float *sum2, int k, const int *counts, uint32_t &nl) {
    cudaStream_t st = ctx->stream;
    CU(cudaEventRecord(ctx->ev[2], st));
    if (ctx->world > 1 && ctx->comm) {
        NcclApi *na = nccl_api();
        ncclResult_t r = na->Reduce(ctx->d_accum, sum1, (size_t)npix * 3, kNcclFloat32, kNcclSum, 0, ctx->comm, st);
        if (r != 0) return fail(ctx, SQT_E_NCCL, "ncclReduce failed: %s", na->GetErrorString(r));
        nl++;
        if (sum2) {
            r = na->Reduce(ctx->d_m2, sum2, (size_t)npix * 3, kNcclFloat32, kNcclSum, 0, ctx->comm, st);
            if (r != 0) return fail(ctx, SQT_E_NCCL, "ncclReduce failed: %s", na->GetErrorString(r));
            nl++;
        }
    }
    CU(cudaEventRecord(ctx->ev[3], st));
    if (ctx->rank == 0) {
        k_tonemap<<<(int)((npix + 255) / 256), 256, 0, st>>>(sum1, npix, inv, ctx->d_rgb8, counts);
        CU(cudaGetLastError()); nl++;
        if (sum2) {
            k_frame_noise_part<<<kNoiseBlocks, 256, 0, st>>>(sum1, sum2, npix * 3, k, counts, ctx->d_noise);
            k_frame_noise<<<1, kNoiseBlocks, 0, st>>>(ctx->d_noise, npix * 3, k, ctx->d_noise + 2 * kNoiseBlocks);
            CU(cudaGetLastError()); nl += 2;
            CU(cudaMemcpyAsync(ctx->h_noise, ctx->d_noise + 2 * kNoiseBlocks, sizeof(double), cudaMemcpyDeviceToHost, st));
        }
    }
    CU(cudaEventRecord(ctx->ev[4], st));
    CU(cudaMemcpyAsync(ctx->h_stats, ctx->d_stats, sizeof(DeviceStats), cudaMemcpyDeviceToHost, st));
    return SQT_OK;
}

static int enqueue_render(sqt_ctx *ctx, const RenderParams &d, bool count, const RenderPlan &pl, uint32_t *launches) {
    const long long npix = (long long)d.rows * d.cols;
    uint32_t nl = 0;
    int rc = enqueue_start(ctx, d, count, pl, nl); if (rc) return rc;
    rc = enqueue_rounds(ctx, d, count, pl.nwork, pl.log2_s, pl.k0, pl.k1, nullptr, nl); if (rc) return rc;
    rc = enqueue_finish(ctx, npix, 1.0f / (float)d.spp, ctx->d_accum, nullptr, d.spp, nullptr, nl); if (rc) return rc;
    ctx->img_pixels = npix; ctx->img_spp = d.spp;
    *launches = nl;
    return SQT_OK;
}

static void fill_stats(sqt_ctx *ctx, sqt_stats *s, uint32_t launches) {
    if (!s) return;
    s->primary_ms = ev_ms(ctx->ev[0], ctx->ev[1]); s->paths_ms = ev_ms(ctx->ev[1], ctx->ev[2]);
    s->reduce_ms = ev_ms(ctx->ev[2], ctx->ev[3]); s->tonemap_ms = ev_ms(ctx->ev[3], ctx->ev[4]);
    s->device_ms = ev_ms(ctx->ev[0], ctx->ev[4]);
    s->rays_traced = ctx->h_stats->rays; s->samples = ctx->h_stats->samples;
    s->rays_reference = ctx->h_stats->rays + ctx->h_stats->primary_reused;
    s->branch_visits = ctx->h_stats->branch_visits; s->child_box_tests = ctx->h_stats->child_box_tests;
    s->tri_tests = ctx->h_stats->tri_tests; s->leaves_culled = ctx->h_stats->leaves_culled;
    s->mt_pass_a = ctx->h_stats->mt_pass_a; s->mt_pass_u = ctx->h_stats->mt_pass_u;
    s->mt_pass_v = ctx->h_stats->mt_pass_v; s->mt_accept = ctx->h_stats->mt_accept;
    s->kernel_launches = launches;
    if (getenv("SQT_DEBUG_STATS") && ctx->h_stats->dbg[0]) {        // scheduler diagnostics of the instrumented pool kernel (development)
        const unsigned long long *d = ctx->h_stats->dbg;
        const double rays = (double)ctx->h_stats->rays;
        fprintf(stderr, "[sqt pool] per ray: T rounds %.3f (fill %.1f)  L rounds %.3f (fill %.1f)  R rounds %.3f (fill %.1f)\n", d[0] / rays, (double)d[3] / d[0],
                d[1] / rays, (double)d[4] / (d[1] ? d[1] : 1), d[2] / rays, (double)d[5] / (d[2] ? d[2] : 1));
        fprintf(stderr, "[sqt pool] T burst, lanes per step  ret:");
        for (int k = 0; k < 8; ++k) fprintf(stderr, " %.1f", (double)d[16 + k] / d[0]);
        fprintf(stderr, "  desc:");
        for (int k = 0; k < 8; ++k) fprintf(stderr, " %.1f", (double)d[8 + k] / d[0]);
        fprintf(stderr, "\n[sqt pool] L passes %.3f per L round, rays with triangles %.1f, tests %.1f, chunks %.2f per pass\n", (double)d[24] / (d[1] ? d[1] : 1),
                (double)d[25] / (d[24] ? d[24] : 1), (double)d[26] / (d[24] ? d[24] : 1), (double)d[27] / (d[24] ? d[24] : 1));
    }
}

extern "C" int sqt_render_resident(sqt_ctx *ctx, const sqt_camera *cam, const sqt_render_params *p, sqt_stats *stats) {
    if (!ctx) return SQT_E_INVALID;
    ctx->prog.on = false;
    if (stats) memset(stats, 0, sizeof *stats);
    cudaSetDevice(ctx->device);
    RenderParams d = {};
    RenderPlan pl;
    int rc = check_params(ctx, cam, p);
    if (!rc) { d = to_device_params(ctx, cam, p); rc = prepare_render(ctx, d, (p->flags & SQT_F_COUNT_WORK) != 0, false, pl); }
    int32_t keys[4];
    lens_keys(ctx, keys);
    rc = group_agree(ctx, rc, keys, 4); if (rc) return rc;
    uint32_t nl = 0;
    rc = enqueue_render(ctx, d, (p->flags & SQT_F_COUNT_WORK) != 0, pl, &nl); if (rc) return group_abort(ctx, rc);
    CU(cudaStreamSynchronize(ctx->stream));
    fill_stats(ctx, stats, nl);
    return SQT_OK;
}

// the sums (moments = false) or second moments of the frame: on rank 0 of a progressive group frame the reduced
// copies, everywhere else the context's own buffers
static float *frame_sums(sqt_ctx *ctx, bool moments) {
    const bool reduced = ctx->prog.on && ctx->world > 1 && ctx->comm && ctx->rank == 0;
    if (moments) return reduced ? ctx->d_red2 : ctx->d_m2;
    return reduced ? ctx->d_red1 : ctx->d_accum;
}

extern "C" int sqt_download_image(sqt_ctx *ctx, uint8_t *rgb8_out, float *accum_out) {
    if (!ctx) return SQT_E_INVALID;
    if (ctx->img_pixels <= 0) return fail(ctx, SQT_E_INVALID, "no rendered image to download");
    CU(cudaSetDevice(ctx->device));
    const long long npix = ctx->img_pixels;
    int rc = ensure_host_image(ctx, npix); if (rc) return rc;
    if (rgb8_out) CU(cudaMemcpyAsync(ctx->h_rgb8, ctx->d_rgb8, (size_t)npix * 3, cudaMemcpyDeviceToHost, ctx->stream));
    if (accum_out) CU(cudaMemcpyAsync(ctx->h_accum, frame_sums(ctx, false), (size_t)npix * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    if (rgb8_out) memcpy(rgb8_out, ctx->h_rgb8, (size_t)npix * 3);
    if (accum_out) memcpy(accum_out, ctx->h_accum, (size_t)npix * 12);
    return SQT_OK;
}

extern "C" int sqt_render(sqt_ctx *ctx, const sqt_camera *cam, const sqt_render_params *p, uint8_t *rgb8_out,
                          float *accum_out, sqt_stats *stats) {
    if (!ctx) return SQT_E_INVALID;
    ctx->prog.on = false;
    if (stats) memset(stats, 0, sizeof *stats);
    cudaSetDevice(ctx->device);
    RenderParams d = {};
    RenderPlan pl;
    int rc = check_params(ctx, cam, p);
    if (!rc) { d = to_device_params(ctx, cam, p); rc = prepare_render(ctx, d, (p->flags & SQT_F_COUNT_WORK) != 0, true, pl); }
    int32_t keys[4];
    lens_keys(ctx, keys);
    rc = group_agree(ctx, rc, keys, 4); if (rc) return rc;
    const long long npix = (long long)d.rows * d.cols;
    uint32_t nl = 0;
    rc = enqueue_render(ctx, d, (p->flags & SQT_F_COUNT_WORK) != 0, pl, &nl); if (rc) return group_abort(ctx, rc);
    cudaStream_t st = ctx->stream;
    const bool root = ctx->rank == 0;
    CU(cudaEventRecord(ctx->ev[5], st));
    if (root && rgb8_out) CU(cudaMemcpyAsync(ctx->h_rgb8, ctx->d_rgb8, (size_t)npix * 3, cudaMemcpyDeviceToHost, st));
    if (root && accum_out) CU(cudaMemcpyAsync(ctx->h_accum, ctx->d_accum, (size_t)npix * 12, cudaMemcpyDeviceToHost, st));
    CU(cudaEventRecord(ctx->ev[6], st));
    CU(cudaStreamSynchronize(st));
    if (root && rgb8_out) memcpy(rgb8_out, ctx->h_rgb8, (size_t)npix * 3);
    if (root && accum_out) memcpy(accum_out, ctx->h_accum, (size_t)npix * 12);
    fill_stats(ctx, stats, nl);
    if (stats) {
        stats->d2h_ms = ev_ms(ctx->ev[5], ctx->ev[6]);
        stats->d2h_bytes = root ? (uint64_t)npix * ((rgb8_out ? 3 : 0) + (accum_out ? 12 : 0)) : 0;
        stats->h2d_bytes = sizeof(RenderParams);    // camera + parameters travel as kernel arguments
    }
    return SQT_OK;
}

extern "C" int sqt_tone_map(sqt_ctx *ctx, const float *mean_rgb, int64_t npix, uint8_t *rgb8_out) {
    if (!ctx) return SQT_E_INVALID;
    ctx->prog.on = false;               // d_accum is its scratch
    if (npix < 0 || (npix > 0 && (!mean_rgb || !rgb8_out))) return fail(ctx, SQT_E_INVALID, "bad tone_map arguments");
    if (npix == 0) return SQT_OK;
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_image(ctx, npix); if (rc) return rc;
    cudaStream_t st = ctx->stream;
    CU(cudaMemcpyAsync(ctx->d_accum, mean_rgb, (size_t)npix * 12, cudaMemcpyHostToDevice, st));
    k_tonemap<<<(int)((npix + 255) / 256), 256, 0, st>>>(ctx->d_accum, npix, 1.0f, ctx->d_rgb8, nullptr);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(rgb8_out, ctx->d_rgb8, (size_t)npix * 3, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    ctx->img_pixels = 0;
    return SQT_OK;
}

// ------------------------------------------------------------------------------ progressive frames
// Every buffer a progressive frame needs beyond those of a one-shot render (prepare_render): the second moments, the
// noise reduction's partial sums, what sqt_render_retire needs (sample counts, the compaction's scratch) and, on rank 0
// of a group, the reduced sums, moments and counts.  Neither sqt_render_advance nor sqt_render_retire allocates.
static int ensure_progressive(sqt_ctx *ctx, long long npix) {
    CU(ctx->d_noise.ensure(2 * kNoiseBlocks + 1));
    CU(ctx->h_noise.ensure(1));
    CU(ctx->d_active.ensure(1));
    CU(ctx->h_active.ensure(2));
    CU(ctx->d_m2.ensure(npix * 3));
    CU(ctx->d_counts.ensure(npix));
    CU(ctx->d_list2.ensure(npix));
    CU(ctx->d_keep.ensure(npix));
    CU(ctx->d_tile.ensure(npix / kRetireTile + 1));
    if (ctx->world > 1 && ctx->comm && ctx->rank == 0) {
        CU(ctx->d_red1.ensure(npix * 3));
        CU(ctx->d_red2.ensure(npix * 3));
        CU(ctx->d_redc.ensure(npix));
    }
    return SQT_OK;
}
// the sample counts of an adaptive frame (0 = samples_done): rank 0 of a group reads the sum over ranks
static const int *frame_counts(sqt_ctx *ctx) {
    if (!ctx->prog.adaptive) return nullptr;
    return ctx->world > 1 && ctx->comm && ctx->rank == 0 ? ctx->d_redc : ctx->d_counts;
}
// a failure after the group agreement of a progressive call ends the frame, leaving no image to download
static int frame_abort(sqt_ctx *ctx, int rc) {
    ctx->prog.on = false; ctx->img_pixels = 0;
    return group_abort(ctx, rc);
}
// what retire and the denoiser read needs a frame in progress with k >= 2 samples and a pixel list (retire: primary reuse
// or a lens frame) or the primary hits (the denoiser, `prim`: primary reuse, which a lens frame does not have)
static int check_variance_frame(sqt_ctx *ctx, const char *what, bool prim) {
    if (!ctx->prog.on) return fail(ctx, SQT_E_INVALID, "%s: no progressive frame in progress", what);
    if (prim && ctx->prog.d.lens) return fail(ctx, SQT_E_UNSUPPORTED, "%s needs primary hits, which a lens frame does not trace", what);
    if (!ctx->prog.d.primary_reuse && !ctx->prog.d.lens) return fail(ctx, SQT_E_UNSUPPORTED, "%s needs primary reuse (not SQT_F_NO_PRIMARY_REUSE)", what);
    if (ctx->prog.k < 2) return fail(ctx, SQT_E_INVALID, "%s needs at least 2 samples per pixel (samples done: %d)", what, ctx->prog.k);
    return SQT_OK;
}

extern "C" int sqt_render_begin(sqt_ctx *ctx, const sqt_camera *cam, const sqt_render_params *p, sqt_stats *stats) {
    if (!ctx) return SQT_E_INVALID;
    if (stats) memset(stats, 0, sizeof *stats);
    cudaSetDevice(ctx->device);
    ctx->prog.on = false; ctx->img_pixels = 0;
    RenderParams d = {};
    RenderPlan pl;
    int rc = check_params(ctx, cam, p);
    if (!rc && p->mode != 0) rc = fail(ctx, SQT_E_UNSUPPORTED, "progressive frames trace paths (mode 0) only");
    if (!rc && (p->flags & SQT_F_SPLIT_SAMPLES)) rc = fail(ctx, SQT_E_UNSUPPORTED, "progressive frames use the pixel-group partition, not SQT_F_SPLIT_SAMPLES");
    const bool count = !rc && (p->flags & SQT_F_COUNT_WORK) != 0;
    if (!rc) { d = to_device_params(ctx, cam, p); rc = prepare_render(ctx, d, count, false, pl); }
    const long long npix = (long long)d.rows * d.cols;
    if (!rc) rc = ensure_progressive(ctx, npix);
    int32_t keys[7] = {0, rc ? 0 : p->spp, 0};
    lens_keys(ctx, keys + 3);
    rc = group_agree(ctx, rc, keys, 7); if (rc) return rc;
    cudaStream_t st = ctx->stream;
    uint32_t nl = 0;
    auto enqueue = [&]() -> int {
        CU(cudaMemsetAsync(ctx->d_m2, 0, (size_t)npix * 12, st));
        int r = enqueue_start(ctx, d, count, pl, nl); if (r) return r;
        for (int e = 2; e <= 4; ++e) CU(cudaEventRecord(ctx->ev[e], st));
        CU(cudaMemcpyAsync(ctx->h_stats, ctx->d_stats, sizeof(DeviceStats), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        return SQT_OK;
    };
    rc = enqueue(); if (rc) return frame_abort(ctx, rc);
    fill_stats(ctx, stats, nl);
    ctx->prog = ProgFrame{/*on*/ true, /*k*/ 0, count, d, pl, /*adaptive*/ false, /*n*/ (long long)ctx->h_stats->n_hit, /*total*/ 0};
    ctx->prog_frame++;
    return SQT_OK;
}

extern "C" int sqt_render_advance(sqt_ctx *ctx, int32_t n_samples, sqt_progress *progress, sqt_stats *stats) {
    if (!ctx) return SQT_E_INVALID;
    if (stats) memset(stats, 0, sizeof *stats);
    cudaSetDevice(ctx->device);
    int rc = SQT_OK;
    if (!ctx->prog.on) rc = fail(ctx, SQT_E_INVALID, "no progressive frame in progress");
    else if (n_samples < 1) rc = fail(ctx, SQT_E_INVALID, "n_samples must be at least 1");
    ProgFrame &f = ctx->prog;
    const RenderParams &d = f.d;
    const int k = f.k, spp = d.spp;
    const int kb = rc ? 0 : (n_samples >= spp - k ? spp : k + n_samples);
    const int32_t keys[3] = {rc ? 0 : k, rc ? 0 : spp, kb};
    rc = group_agree(ctx, rc, keys, 3); if (rc) return rc;
    const bool root = ctx->rank == 0;
    if (k < spp && f.adaptive && f.total == 0) {
        f.k = kb; ctx->img_spp = kb;                    // every pixel has retired: nothing to trace, the image stays
    } else if (k < spp) {
        const long long npix = (long long)d.rows * d.cols;
        // an adaptive frame traces its active slots only, in rounds as wide as the sample buffer allows for them (at
        // most the chunk: wider rounds would only skip items); results never depend on the round width
        const long long nslots = f.adaptive ? f.n : f.pl.nwork;
        const int log2_s = f.adaptive ? round_log2_s(nslots, kb - k, f.pl.sbytes) : f.pl.log2_s;
        cudaStream_t st = ctx->stream;
        uint32_t nl = 0;
        auto enqueue = [&]() -> int {
            // the counters of this call only; n_hit (the primary pass's pixel list) stays
            CU(cudaMemsetAsync(ctx->d_stats, 0, offsetof(DeviceStats, n_hit), st));
            CU(cudaMemsetAsync((char *)ctx->d_stats.p + offsetof(DeviceStats, work_next), 0, sizeof(DeviceStats) - offsetof(DeviceStats, work_next), st));
            CU(cudaEventRecord(ctx->ev[0], st));
            CU(cudaEventRecord(ctx->ev[1], st));
            int r = enqueue_rounds(ctx, d, f.count, nslots, log2_s, k, kb, ctx->d_m2, nl); if (r) return r;
            r = enqueue_finish(ctx, npix, 1.0f / (float)kb, frame_sums(ctx, false), frame_sums(ctx, true), kb, frame_counts(ctx), nl);
            if (r) return r;
            CU(cudaStreamSynchronize(st));
            return SQT_OK;
        };
        rc = enqueue();
        if (rc) return frame_abort(ctx, rc);
        fill_stats(ctx, stats, nl);
        f.k = kb; ctx->img_pixels = npix; ctx->img_spp = kb;
    }
    if (progress) {
        progress->samples_done = f.k; progress->samples_total = spp;
        progress->noise = root ? *ctx->h_noise : __builtin_nan("");
    }
    return SQT_OK;
}

extern "C" int sqt_download_moments(sqt_ctx *ctx, float *m2_out) {
    if (!ctx) return SQT_E_INVALID;
    if (!ctx->prog.on) return fail(ctx, SQT_E_INVALID, "no progressive frame in progress");
    if (!m2_out) return fail(ctx, SQT_E_INVALID, "m2_out is NULL");
    CU(cudaSetDevice(ctx->device));
    const long long npix = (long long)ctx->prog.d.rows * ctx->prog.d.cols;
    int rc = ensure_host_image(ctx, npix); if (rc) return rc;
    CU(cudaMemcpyAsync(ctx->h_accum, frame_sums(ctx, true), (size_t)npix * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    memcpy(m2_out, ctx->h_accum, (size_t)npix * 12);
    return SQT_OK;
}

// ------------------------------------------------------------------------------ adaptive frames
static uint32_t float_bits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }

extern "C" int sqt_render_retire(sqt_ctx *ctx, const sqt_retire_params *rp, int64_t *active_out) {
    if (!ctx) return SQT_E_INVALID;
    cudaSetDevice(ctx->device);
    int rc = rp ? check_variance_frame(ctx, "sqt_render_retire", false) : fail(ctx, SQT_E_INVALID, "retire params are NULL");
    if (!rc && rp->min_samples < 2) rc = fail(ctx, SQT_E_INVALID, "min_samples must be at least 2");
    if (!rc && (!(rp->rel_tol >= 0.0f) || !(rp->abs_tol >= 0.0f))) rc = fail(ctx, SQT_E_INVALID, "tolerances must be non-negative numbers");
    if (!rc && rp->reserved) rc = fail(ctx, SQT_E_INVALID, "reserved must be 0");
    ProgFrame &f = ctx->prog;
    const int k = f.k, spp = f.d.spp;
    const int32_t keys[5] = {rc ? 0 : k, rc ? 0 : spp, rc ? 0 : (int32_t)float_bits(rp->rel_tol), rc ? 0 : (int32_t)float_bits(rp->abs_tol),
                             rc ? 0 : rp->min_samples};
    rc = group_agree(ctx, rc, keys, 5); if (rc) return rc;
    const bool group = ctx->world > 1 && ctx->comm;
    const long long npix = (long long)f.d.rows * f.d.cols;
    cudaStream_t st = ctx->stream;
    // at k = spp, and before min_samples, nothing can retire: only the active total is reported
    const bool test = k < spp && k >= rp->min_samples;
    auto enqueue = [&]() -> int {
        const long long n = f.n;
        if (test) {
            if (!f.adaptive) CU(cudaMemsetAsync(ctx->d_counts, 0, (size_t)npix * sizeof(int), st));
            if (n > 0) {
                const long long tiles = (n + kRetireTile - 1) / kRetireTile;
                k_retire_mark<<<(int)tiles, 256, 0, st>>>(ctx->d_pixel_list, n, ctx->d_accum, ctx->d_m2, k,
                                                          (double)rp->rel_tol, (double)rp->abs_tol, ctx->d_counts, ctx->d_keep, ctx->d_tile);
                k_retire_scan<<<1, 1024, 0, st>>>(ctx->d_tile, tiles, &ctx->d_stats->n_hit);
                k_retire_compact<<<(int)tiles, 256, 0, st>>>(ctx->d_pixel_list, n, ctx->d_keep, ctx->d_tile, ctx->d_list2);
                CU(cudaGetLastError());
                CU(cudaMemcpyAsync(ctx->d_pixel_list, ctx->d_list2, (size_t)n * sizeof(int), cudaMemcpyDeviceToDevice, st));
            }
            if (group) {
                NcclApi *na = nccl_api();
                // a pixel's count is non-zero on its owner only, so the sum is exact
                ncclResult_t r = na->Reduce(ctx->d_counts, ctx->d_redc, (size_t)npix, kNcclInt32, kNcclSum, 0, ctx->comm, st);
                if (r != 0) return fail(ctx, SQT_E_NCCL, "ncclReduce failed: %s", na->GetErrorString(r));
            }
        }
        CU(cudaMemcpyAsync(&ctx->h_active[0], &ctx->d_stats->n_hit, sizeof(long long), cudaMemcpyDeviceToHost, st));
        if (group) {
            NcclApi *na = nccl_api();
            ncclResult_t r = na->AllReduce(&ctx->d_stats->n_hit, ctx->d_active, 1, kNcclInt64, kNcclSum, ctx->comm, st);
            if (r != 0) return fail(ctx, SQT_E_NCCL, "ncclAllReduce failed: %s", na->GetErrorString(r));
            CU(cudaMemcpyAsync(&ctx->h_active[1], ctx->d_active, sizeof(long long), cudaMemcpyDeviceToHost, st));
        }
        CU(cudaStreamSynchronize(st));
        return SQT_OK;
    };
    rc = enqueue();
    if (rc) return frame_abort(ctx, rc);
    f.n = ctx->h_active[0];
    f.total = group ? ctx->h_active[1] : ctx->h_active[0];
    if (test) f.adaptive = true;
    if (active_out) *active_out = f.total;
    return SQT_OK;
}

extern "C" int sqt_download_sample_counts(sqt_ctx *ctx, int32_t *counts_out) {
    if (!ctx) return SQT_E_INVALID;
    if (!ctx->prog.on) return fail(ctx, SQT_E_INVALID, "no progressive frame in progress");
    if (!counts_out) return fail(ctx, SQT_E_INVALID, "counts_out is NULL");
    CU(cudaSetDevice(ctx->device));
    const long long npix = (long long)ctx->prog.d.rows * ctx->prog.d.cols;
    const int k = ctx->prog.k;
    if (const int *c = frame_counts(ctx)) {
        int rc = ensure_host_image(ctx, npix); if (rc) return rc;
        CU(cudaMemcpyAsync(ctx->h_accum, c, (size_t)npix * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        memcpy(counts_out, ctx->h_accum, (size_t)npix * sizeof(int));
    } else {
        memset(counts_out, 0, (size_t)npix * sizeof(int));
    }
    for (long long i = 0; i < npix; ++i) if (!counts_out[i]) counts_out[i] = k;
    return SQT_OK;
}

// ------------------------------------------------------------------------------ denoiser
// The denoiser reads the frame and writes only its own buffers: sums, moments, counts, the preview and the pixel list stay
// as they are.  Its buffers are made on first use, before the group agreement, as ensure_progressive does.
static int ensure_denoise(sqt_ctx *ctx, long long npix) {
    if ((size_t)npix > ctx->d_feat.cap || (size_t)npix > ctx->d_sk.cap) ctx->dn_frame = -1;     // new buffers hold no features
    CU(ctx->d_feat.ensure(npix));
    CU(ctx->d_sk.ensure(npix));
    CU(ctx->d_dn[0].ensure(npix));
    CU(ctx->d_dn[1].ensure(npix));
    CU(ctx->d_dn_mean.ensure(npix * 3));
    CU(ctx->d_dn_rgb8.ensure(npix * 3));
    return SQT_OK;
}

// the checks every denoiser call shares, then the group agreement on (k, spp, levels, sigma bits); sqt_download_features
// (download) agrees on levels = -1
static int denoise_enter(sqt_ctx *ctx, bool download, int levels, float sigma_l, float sigma_z, uint32_t reserved, const char *what) {
    if (download) { levels = -1; sigma_l = sigma_z = 0.0f; reserved = 0; }
    int rc = check_variance_frame(ctx, what, true);
    if (!rc && !download && (levels > 8 || levels < 0)) rc = fail(ctx, SQT_E_INVALID, "%s: levels must be in 0..8", what);
    if (!rc && !download && (!(sigma_l > 0.0f) || !(sigma_l < INFINITY) || !(sigma_z > 0.0f) || !(sigma_z < INFINITY)))
        rc = fail(ctx, SQT_E_INVALID, "%s: sigma_l and sigma_z must be positive and finite", what);
    if (!rc && reserved) rc = fail(ctx, SQT_E_INVALID, "%s: reserved must be 0", what);
    if (!rc) rc = ensure_denoise(ctx, (long long)ctx->prog.d.rows * ctx->prog.d.cols);
    const int32_t keys[5] = {rc ? 0 : ctx->prog.k, rc ? 0 : ctx->prog.d.spp, rc ? 0 : levels, rc ? 0 : (int32_t)float_bits(sigma_l),
                             rc ? 0 : (int32_t)float_bits(sigma_z)};
    return group_agree(ctx, rc, keys, 5);
}

// enqueue the features of this frame unless they are there already: k_features on every rank, then (groups) their sum
// onto rank 0 -- every value is non-zero on its owner only, so the sum is exact.  Events 0 .. 2 bracket it.
static int enqueue_features(sqt_ctx *ctx, uint32_t &nl) {
    cudaStream_t st = ctx->stream;
    const RenderParams &d = ctx->prog.d;
    const long long npix = (long long)d.rows * d.cols;
    CU(cudaEventRecord(ctx->ev[0], st));
    const bool need = ctx->dn_frame != ctx->prog_frame;
    if (need) {
        CU(cudaMemsetAsync(ctx->d_feat, 0, (size_t)npix * sizeof(float4), st));
        CU(cudaMemsetAsync(ctx->d_sk, 0, (size_t)npix * sizeof(int2), st));
        const long long nwork = ctx->prog.pl.nwork;
        k_features<<<(int)((nwork + 255) / 256), 256, 0, st>>>(ctx->sc, d, ctx->d_prim, nwork, ctx->d_feat, ctx->d_sk);
        CU(cudaGetLastError()); nl++;
    }
    CU(cudaEventRecord(ctx->ev[1], st));
    if (need && ctx->world > 1 && ctx->comm) {
        NcclApi *na = nccl_api();
        ncclResult_t r = na->Reduce(ctx->d_sk, ctx->d_sk, (size_t)npix * 2, kNcclInt32, kNcclSum, 0, ctx->comm, st);
        // (N, z) as int32 bit patterns: adding +0 to an owner's -0.0 in f32 would give +0.0, adding the integer 0 keeps every bit
        if (r == 0) r = na->Reduce(ctx->d_feat, ctx->d_feat, (size_t)npix * 4, kNcclInt32, kNcclSum, 0, ctx->comm, st);
        if (r != 0) return fail(ctx, SQT_E_NCCL, "ncclReduce failed: %s", na->GetErrorString(r));
        nl += 2;
    }
    CU(cudaEventRecord(ctx->ev[2], st));
    return SQT_OK;
}

static void denoise_stats(sqt_ctx *ctx, sqt_stats *s, uint32_t nl, uint64_t d2h_bytes) {
    if (!s) return;
    s->device_ms = ev_ms(ctx->ev[0], ctx->ev[3]);
    s->reduce_ms = ev_ms(ctx->ev[1], ctx->ev[2]);
    s->d2h_ms = ev_ms(ctx->ev[3], ctx->ev[4]);
    s->d2h_bytes = d2h_bytes;
    s->kernel_launches = nl;
}

extern "C" int sqt_denoise(sqt_ctx *ctx, const sqt_denoise_params *dp, uint8_t *rgb8_out, float *mean_out, sqt_stats *stats) {
    if (!ctx) return SQT_E_INVALID;
    if (stats) memset(stats, 0, sizeof *stats);
    cudaSetDevice(ctx->device);
    int rc = dp ? denoise_enter(ctx, false, dp->levels, dp->sigma_l, dp->sigma_z, dp->reserved, "sqt_denoise")
                : group_agree(ctx, fail(ctx, SQT_E_INVALID, "sqt_denoise: params are NULL"));
    if (rc) return rc;
    const RenderParams &d = ctx->prog.d;
    const long long npix = (long long)d.rows * d.cols;
    const bool root = ctx->rank == 0;
    cudaStream_t st = ctx->stream;
    uint32_t nl = 0;
    auto enqueue = [&]() -> int {
        int r = enqueue_features(ctx, nl); if (r) return r;
        if (root) {
            k_denoise_prep<<<(int)((npix + 255) / 256), 256, 0, st>>>(frame_sums(ctx, false), frame_sums(ctx, true), npix, ctx->prog.k,
                                                                     frame_counts(ctx), ctx->d_dn[0], ctx->d_dn_mean);
            CU(cudaGetLastError()); nl++;
            const dim3 grid((unsigned)((d.cols + 15) / 16), (unsigned)((d.rows + 15) / 16));
            for (int i = 0; i < dp->levels; ++i) {
                k_denoise_level<<<grid, 256, 0, st>>>(ctx->d_dn[i & 1], ctx->d_feat, ctx->d_sk, d.rows, d.cols, 1 << i, dp->sigma_l, dp->sigma_z,
                                                      ctx->d_dn[(i + 1) & 1], i + 1 == dp->levels ? ctx->d_dn_mean.p : nullptr);
                CU(cudaGetLastError()); nl++;
            }
            k_tonemap<<<(int)((npix + 255) / 256), 256, 0, st>>>(ctx->d_dn_mean, npix, 1.0f, ctx->d_dn_rgb8, nullptr);
            CU(cudaGetLastError()); nl++;
        }
        CU(cudaEventRecord(ctx->ev[3], st));
        if (root && rgb8_out) CU(cudaMemcpyAsync(rgb8_out, ctx->d_dn_rgb8, (size_t)npix * 3, cudaMemcpyDeviceToHost, st));
        if (root && mean_out) CU(cudaMemcpyAsync(mean_out, ctx->d_dn_mean, (size_t)npix * 12, cudaMemcpyDeviceToHost, st));
        CU(cudaEventRecord(ctx->ev[4], st));
        CU(cudaStreamSynchronize(st));
        return SQT_OK;
    };
    rc = enqueue();
    if (rc) return frame_abort(ctx, rc);
    ctx->dn_frame = ctx->prog_frame;
    denoise_stats(ctx, stats, nl, root ? (uint64_t)npix * ((rgb8_out ? 3 : 0) + (mean_out ? 12 : 0)) : 0);
    return SQT_OK;
}

extern "C" int sqt_download_features(sqt_ctx *ctx, int32_t *surface_out, float *depth_out, float *normal_out) {
    if (!ctx) return SQT_E_INVALID;
    cudaSetDevice(ctx->device);
    int rc = denoise_enter(ctx, true, 0, 0.0f, 0.0f, 0u, "sqt_download_features");
    if (rc) return rc;
    const long long npix = (long long)ctx->prog.d.rows * ctx->prog.d.cols;
    uint32_t nl = 0;
    auto enqueue = [&]() -> int {
        int r = enqueue_features(ctx, nl); if (r) return r;
        CU(cudaEventRecord(ctx->ev[3], ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        return SQT_OK;
    };
    rc = enqueue();
    if (rc) return frame_abort(ctx, rc);
    ctx->dn_frame = ctx->prog_frame;
    if (ctx->rank != 0 || (!surface_out && !depth_out && !normal_out)) return SQT_OK;
    std::vector<float4> f((size_t)npix);
    std::vector<int2> sk((size_t)npix);
    CU(cudaMemcpy(f.data(), ctx->d_feat, (size_t)npix * sizeof(float4), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(sk.data(), ctx->d_sk, (size_t)npix * sizeof(int2), cudaMemcpyDeviceToHost));
    for (long long i = 0; i < npix; ++i) {
        if (surface_out) surface_out[i] = sk[i].x - 1;
        if (depth_out) depth_out[i] = f[i].w;
        if (normal_out) { normal_out[3 * i] = f[i].x; normal_out[3 * i + 1] = f[i].y; normal_out[3 * i + 2] = f[i].z; }
    }
    return SQT_OK;
}

// ------------------------------------------------------------------------------ group (NCCL)
extern "C" int sqt_comm_unique_id(uint8_t id_out[SQT_COMM_ID_BYTES]) {
    NcclApi *na = nccl_api();
    if (!na->lib) return fail(nullptr, SQT_E_NCCL, "%s", na->err.c_str());
    ncclUniqueId id;
    ncclResult_t r = na->GetUniqueId(&id);
    if (r != 0) return fail(nullptr, SQT_E_NCCL, "ncclGetUniqueId: %s", na->GetErrorString(r));
    memcpy(id_out, id.internal, SQT_COMM_ID_BYTES);
    return SQT_OK;
}

extern "C" int sqt_comm_init(sqt_ctx *ctx, int rank, int world, const uint8_t id_in[SQT_COMM_ID_BYTES]) {
    if (!ctx) return SQT_E_INVALID;
    if (world < 1 || rank < 0 || rank >= world) return fail(ctx, SQT_E_INVALID, "bad rank/world %d/%d", rank, world);
    if (world == 1) { ctx->rank = 0; ctx->world = 1; return SQT_OK; }
    NcclApi *na = nccl_api();
    if (!na->lib) return fail(ctx, SQT_E_NCCL, "%s", na->err.c_str());
    CU(cudaSetDevice(ctx->device));
    ncclUniqueId id; memcpy(id.internal, id_in, SQT_COMM_ID_BYTES);
    ncclResult_t r = na->CommInitRank(&ctx->comm, world, id, rank);
    if (r != 0) return fail(ctx, SQT_E_NCCL, "ncclCommInitRank: %s", na->GetErrorString(r));
    ctx->rank = rank; ctx->world = world;
    return SQT_OK;
}

extern "C" int sqt_comm_init_all(sqt_ctx **ctxs, int n) {
    if (!ctxs || n < 1) return SQT_E_INVALID;
    if (n == 1) { ctxs[0]->rank = 0; ctxs[0]->world = 1; return SQT_OK; }
    NcclApi *na = nccl_api();
    if (!na->lib) return fail(ctxs[0], SQT_E_NCCL, "%s", na->err.c_str());
    std::vector<int> devs(n); std::vector<ncclComm_t> comms(n);
    for (int i = 0; i < n; ++i) devs[i] = ctxs[i]->device;
    ncclResult_t r = na->CommInitAll(comms.data(), n, devs.data());
    if (r != 0) return fail(ctxs[0], SQT_E_NCCL, "ncclCommInitAll: %s", na->GetErrorString(r));
    for (int i = 0; i < n; ++i) { ctxs[i]->comm = comms[i]; ctxs[i]->rank = i; ctxs[i]->world = n; }
    return SQT_OK;
}

// A call on every context of a single-process group, one host thread per device from ctxs[1] on (the collectives of such
// a group must be issued concurrently) and ctxs[0] on the calling thread: call(ctx, root), root for ctxs[0] only, which
// alone gets the outputs.  A failing rank's error is reported on ctxs[0].
template <class F>
static int fan_out(sqt_ctx **ctxs, int n, F call) {
    if (!valid_group(ctxs, n)) return SQT_E_INVALID;
    if (n == 1) return call(ctxs[0], true);
    std::vector<int> rcs(n, 0);
    std::vector<std::thread> th;
    for (int i = 1; i < n; ++i) th.emplace_back([&, i]() { rcs[i] = call(ctxs[i], false); });
    rcs[0] = call(ctxs[0], true);
    for (auto &t : th) t.join();
    for (int i = 0; i < n; ++i) if (rcs[i]) { if (i) ctxs[0]->err = ctxs[i]->err; return rcs[i]; }
    return SQT_OK;
}

extern "C" int sqt_render_group(sqt_ctx **ctxs, int n, const sqt_camera *cam, const sqt_render_params *p,
                                uint8_t *rgb8_out, float *accum_out, sqt_stats *stats) {
    return fan_out(ctxs, n, [&](sqt_ctx *c, bool root) { return sqt_render(c, cam, p, root ? rgb8_out : nullptr, root ? accum_out : nullptr, root ? stats : nullptr); });
}

extern "C" int sqt_render_begin_group(sqt_ctx **ctxs, int n, const sqt_camera *cam, const sqt_render_params *p, sqt_stats *stats) {
    return fan_out(ctxs, n, [&](sqt_ctx *c, bool root) { return sqt_render_begin(c, cam, p, root ? stats : nullptr); });
}

extern "C" int sqt_render_advance_group(sqt_ctx **ctxs, int n, int32_t n_samples, sqt_progress *progress, sqt_stats *stats) {
    return fan_out(ctxs, n, [&](sqt_ctx *c, bool root) { return sqt_render_advance(c, n_samples, root ? progress : nullptr, root ? stats : nullptr); });
}

extern "C" int sqt_render_retire_group(sqt_ctx **ctxs, int n, const sqt_retire_params *rp, int64_t *active_out) {
    return fan_out(ctxs, n, [&](sqt_ctx *c, bool root) { return sqt_render_retire(c, rp, root ? active_out : nullptr); });
}

extern "C" int sqt_denoise_group(sqt_ctx **ctxs, int n, const sqt_denoise_params *dp, uint8_t *rgb8_out, float *mean_out, sqt_stats *stats) {
    return fan_out(ctxs, n, [&](sqt_ctx *c, bool root) { return sqt_denoise(c, dp, root ? rgb8_out : nullptr, root ? mean_out : nullptr, root ? stats : nullptr); });
}

// ------------------------------------------------------------------------------ roofline microbenchmarks
extern "C" int sqt_measure_fp32_peak(sqt_ctx *ctx, double *gops) {
    if (!ctx || !gops) return SQT_E_INVALID;
    CU(cudaSetDevice(ctx->device));
    Buffer<float> d; CU(d.ensure(4));
    const int iters = 4096, grid = ctx->sm_count * 8, block = 256;
    cudaStream_t st = ctx->stream;
    double best = 0;
    for (int rep = 0; rep < 5; ++rep) {
        CU(cudaEventRecord(ctx->ev[0], st));
        k_fp32_peak<<<grid, block, 0, st>>>(d, iters, 1.0000001f, 1e-7f);
        CU(cudaGetLastError());
        CU(cudaEventRecord(ctx->ev[1], st));
        CU(cudaStreamSynchronize(st));
        const double ms = ev_ms(ctx->ev[0], ctx->ev[1]);
        const double ops = (double)grid * block * iters * 32.0;
        if (rep > 0 && ops / ms * 1e-6 > best) best = ops / ms * 1e-6;
    }
    *gops = best;
    return SQT_OK;
}

extern "C" int sqt_measure_l2_bandwidth(sqt_ctx *ctx, double *gbs) {
    if (!ctx || !gbs) return SQT_E_INVALID;
    CU(cudaSetDevice(ctx->device));
    const long long bytes = 32ll << 20, n4 = bytes / 16;
    Buffer<float4> buf; Buffer<float> out;
    CU(buf.ensure(n4)); CU(out.ensure(4));
    CU(cudaMemset(buf, 0, bytes));
    cudaStream_t st = ctx->stream;
    const int grid = ctx->sm_count * 8, block = 256, reps = 16;
    double best = 0;
    for (int rep = 0; rep < 5; ++rep) {
        CU(cudaEventRecord(ctx->ev[0], st));
        k_l2_read<<<grid, block, 0, st>>>(buf, n4, reps, out);
        CU(cudaGetLastError());
        CU(cudaEventRecord(ctx->ev[1], st));
        CU(cudaStreamSynchronize(st));
        const double ms = ev_ms(ctx->ev[0], ctx->ev[1]);
        const double gb = (double)bytes * reps / ms * 1e-6;
        if (rep > 0 && gb > best) best = gb;
    }
    *gbs = best;
    return SQT_OK;
}
