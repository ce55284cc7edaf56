/*
 * sqt.h -- C ABI of the B200 (sm_100a) path-tracing backend for squigly-trace.
 *
 * This is the drop-in boundary for the reference's render hot path.  The reference has no FFI
 * today (no `foreign import` anywhere); the two function-typed seams it does have are
 *
 *   render    :: Scene a -> Camera -> Settings -> IO ()        src/Lib.hs:68-75   (caller app/Main.hs:43)
 *   intersect :: a -> Ray -> Maybe Intersection  (Scene field)  src/Geometry.hs:62-65 (chosen app/Main.hs:52-56,
 *                                                               called src/Lib.hs:131,143,150)
 *
 * Everything below `render` except `writeImage` (Lib.hs:75) moves behind sqt_render();
 * sqt_intersect_batch() is the batched form of `intersect` and carries the bit-exact contract.
 * The Haskell host keeps Obj.hs / BIH.hs / Main.hs, flattens its BIH into the records below and
 * binds these symbols with `foreign import ccall safe` (see INTEGRATION.md).
 *
 * Conventions: plain C, no C++ types, no exceptions across the boundary.  Every function returns
 * 0 on success or a non-zero SQT_E_* code; sqt_last_error(ctx) gives the message.  All pointers
 * are caller-owned HOST memory, valid for the duration of the call only; the library owns all
 * device memory.  A context is bound to one CUDA device, is not re-entrant and blocks the
 * calling thread.  There is no CPU fallback: without a usable sm_100 device sqt_create fails.
 */
#ifndef SQT_H
#define SQT_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SQT_ABI_VERSION 1

enum {
    SQT_OK = 0,
    SQT_E_INVALID = 1,      /* bad argument / malformed scene */
    SQT_E_CUDA = 2,         /* CUDA runtime error (message has the cudaError string) */
    SQT_E_NO_DEVICE = 3,    /* no CUDA device, or not compute capability 10.x */
    SQT_E_NO_SCENE = 4,     /* render/intersect before sqt_upload_scene */
    SQT_E_UNSUPPORTED = 5,  /* e.g. BIH deeper than SQT_MAX_HEIGHT, max_depth > SQT_MAX_DEPTH */
    SQT_E_NCCL = 6          /* NCCL missing or failed */
};

#define SQT_MAX_HEIGHT 48   /* deepest supported BIH (reference scene: 13) */
#define SQT_MAX_DEPTH 64    /* largest max_depth (reference: 3, Lib.hs:129) */

/* ---- flattened BIH (BIH.hs:26,37-43), nodes in any order with node 0 = root ------------------
 * Branch (BIHN axis lmax rmin) l r : a = index(l) | axis<<30 ,  b = index(r)             (axis X=0,Y=1,Z=2)
 * Leaf tris                         : a = first triangle in tris[] , b = count | 0x80000000   (lmax,rmin ignored)
 * At most 2^27 - 1 nodes and 2^27 - 1 triangles.  Child boxes are NOT stored: the library derives them exactly as
 * BIH.hs:130-141 does, by clipping the parent's box (plain copies of lmax/rmin, no arithmetic).  The `pad` word of
 * a triangle is ignored on input (the device copy uses it). */
typedef struct sqt_node {
    float lmax, rmin;
    uint32_t a, b;
} sqt_node;                              /* 16 B */
#define SQT_NODE_LEAF 0x80000000u

/* Triangles in leaf order, i.e. `flatten` (BIH.hs:50-52): each Leaf's vector is a contiguous range.
 * e1 = v1 - v0, e2 = v2 - v0 computed in binary32 on the host: identical bits to edge1/edge2 of
 * Geometry.hs:130-131, and e1 x e2 is `normal` (Geometry.hs:79-80). */
typedef struct sqt_tri {
    float v0[3], e1[3], e2[3];
    uint32_t material;                   /* index into mats[] */
    uint32_t orig_index;                 /* position in the parsed triangle list (what tri_out reports) */
    uint32_t pad;
} sqt_tri;                               /* 48 B */

/* Color.hs:78-83 */
typedef struct sqt_material {
    float reflective, surf_color[3], emissive, emit_color[3];
} sqt_material;                          /* 32 B */

/* EXTENSION (named by the north star; the reference has no sphere primitive or syntax, so the semantics are this
 * library's own and are restated in oracle/oracle.c): analytic, double-sided spheres; a ray's result is the closest of
 * the BIH hit and all sphere hits, earlier candidates of the list [BIH hit, sphere 0, sphere 1, ...] win ties.  (The
 * library finds the candidate spheres through a hierarchy of its own, see SQT_OPT_SPHERE_BVH.)  In tri_out a
 * sphere k is reported as n_tris + k. */
typedef struct sqt_sphere {
    float center[3];
    float radius;
    uint32_t material;                   /* index into mats[] */
    uint32_t pad[3];
} sqt_sphere;                            /* 32 B */

typedef struct sqt_scene_desc {
    float root_bounds[6];                /* bounds of BIH (BIH.hs:41,62-65): lo.xyz, hi.xyz */
    const sqt_node *nodes;  uint32_t n_nodes;
    const sqt_tri *tris;    uint32_t n_tris;
    const sqt_material *mats; uint32_t n_mats;
} sqt_scene_desc;

/* Geometry.hs:41 : position + rotation matrix as produced by rotMatrixRads (row-major 3x3) */
typedef struct sqt_camera {
    float position[3];
    float rotation[9];
} sqt_camera;

/* Settings that reach the hot path (Lib.hs:54-63 `samples`, `dimensions`, `cast`) plus the
 * index convention of Lib.hs:69-85,107-114 made explicit (SURVEY A.5):
 *   pixel (row y, col x):  xoffs = (x - xdiv/2)/xdiv ; yoffs = (ydiv/2 - y)/ydiv ;
 *   generator seed of sample k = spp*(x + y*seed_stride) + k.
 * Reference-literal `-d W,H`: rows=W cols=H xdiv=W ydiv=H seed_stride=W.
 * Corrected:                  rows=H cols=W xdiv=W ydiv=H seed_stride=W. */
typedef struct sqt_render_params {
    int32_t rows, cols;
    int32_t xdiv, ydiv;
    int32_t seed_stride;
    int32_t spp;
    int32_t max_depth;                   /* intersections per path; reference = 3 (Lib.hs:129) */
    int32_t mode;                        /* 0 = raytrace (Lib.hs:127), 1 = raycast / --cast (Lib.hs:141) */
    uint64_t seed;                       /* key of the counter-based RNG */
    uint32_t flags;                      /* SQT_F_* */
    uint32_t reserved;
} sqt_render_params;

#define SQT_F_COUNT_WORK      1u   /* run the instrumented kernels and fill the *_visits/_tests counters (slower) */
#define SQT_F_SPLIT_SAMPLES   2u   /* multi-GPU: split the spp range per rank instead of pixel groups */
#define SQT_F_NO_PRIMARY_REUSE 4u  /* re-trace the (identical) primary ray for every sample, as Lib.hs:81-87 does */
#define SQT_F_NO_EARLY_TERMINATION 8u /* keep tracing below a surface whose surfColor is (0,0,0), as Lib.hs:135 does
                                         (the product of such a level is exactly 0, so the image is the same) */

typedef struct sqt_stats {
    double device_ms;            /* CUDA-event time of all kernels of this call on the context's stream */
    double primary_ms, paths_ms, tonemap_ms, reduce_ms;
    double h2d_ms, d2h_ms;       /* host<->device copies of this call (0 for the *_resident entry points) */
    uint64_t rays_traced;        /* closest-hit queries actually executed on the device */
    uint64_t rays_reference;     /* queries the reference would execute for the same job (Lib.hs:131 per segment) */
    uint64_t samples;            /* paths (Lib.hs:84) */
    uint64_t branch_visits, child_box_tests, tri_tests;    /* only with SQT_F_COUNT_WORK */
    uint64_t leaves_culled;      /* leaf visits skipped by the conservative tight-box test (with SQT_F_COUNT_WORK) */
    uint64_t mt_pass_a, mt_pass_u, mt_pass_v, mt_accept;   /* triangle tests that got past the a / u / v / t guards
                                                               of Geometry.hs:118-122 (with SQT_F_COUNT_WORK) */
    uint64_t h2d_bytes, d2h_bytes;
    uint32_t kernel_launches;
    uint32_t reserved;
} sqt_stats;

typedef struct sqt_ctx sqt_ctx;

/* lifecycle ------------------------------------------------------------------------------- */
int sqt_abi_version(void);
int sqt_create(int device, sqt_ctx **out);
int sqt_destroy(sqt_ctx *ctx);
const char *sqt_last_error(const sqt_ctx *ctx);        /* ctx may be NULL: error of the last failed sqt_create */

/* replaces the in-memory `Scene BIH` value handed to render (Main.hs:39,55-56) ------------- */
int sqt_upload_scene(sqt_ctx *ctx, const sqt_scene_desc *scene);

/* The same scene onto every context of a single-process group (ctxs[0..n) on n distinct devices): the tree is walked
 * once and every staged chunk of triangles is sent to all devices.  What the Haskell host calls once per run. */
int sqt_upload_scene_group(sqt_ctx **ctxs, int n, const sqt_scene_desc *scene);

/* what the last sqt_upload_scene[_group] on this context moved and cost: bytes copied host -> device, wall time of the
 * call, and the part of it the host spent walking the tree (the rest is copies + two device kernels).  Any pointer may
 * be NULL. */
int sqt_last_upload(const sqt_ctx *ctx, uint64_t *h2d_bytes, double *wall_ms, double *host_layout_ms);

/* optional, after sqt_upload_scene: n = 0 removes the spheres again */
int sqt_upload_spheres(sqt_ctx *ctx, const sqt_sphere *spheres, uint32_t n);

/* batched Scene.intersect (Geometry.hs:64; intersectBIH BIH.hs:101-141) ---------------------
 * org/dir: n x 3 floats, xyz interleaved.  tri_out[i] = orig_index of the closest hit or -1.
 * dist_out / point_out (n x 3) may be NULL.  Bit-exact contract: same index, dist and point bits
 * as the reference algorithm on the same tree. */
int sqt_intersect_batch(sqt_ctx *ctx, const float *org, const float *dir, int64_t n,
                        int32_t *tri_out, float *dist_out, float *point_out, sqt_stats *stats_or_null);

/* replaces the body of render above writeImage (Lib.hs:70-74) --------------------------------
 * rgb8_out: rows*cols*3 bytes, row-major = massiv `Array S Ix2 (Pixel RGB Word8)`.
 * accum_out (optional): rows*cols*3 floats, per-pixel radiance SUM over samples (before the 1/spp of Lib.hs:88).
 * In a multi-rank group only rank 0 receives the image; other ranks may pass NULL. */
int sqt_render(sqt_ctx *ctx, const sqt_camera *cam, const sqt_render_params *params,
               uint8_t *rgb8_out, float *accum_out, sqt_stats *stats_or_null);

/* same job, result left in device memory (no host copies); fetch it with sqt_download_image */
int sqt_render_resident(sqt_ctx *ctx, const sqt_camera *cam, const sqt_render_params *params, sqt_stats *stats_or_null);
int sqt_download_image(sqt_ctx *ctx, uint8_t *rgb8_out, float *accum_out);

/* rgbFloatToPixelRGB (Lib.hs:93-104) on the device, for n_pixels mean colours */
int sqt_tone_map(sqt_ctx *ctx, const float *mean_rgb, int64_t n_pixels, uint8_t *rgb8_out);

/* multi-GPU: one context per GPU (one process per GPU or all in one process); the group sums the
 * per-rank accumulation buffers with ncclReduce(sum, f32) onto rank 0 ---------------------- */
#define SQT_COMM_ID_BYTES 128
int sqt_comm_unique_id(uint8_t id_out[SQT_COMM_ID_BYTES]);
int sqt_comm_init(sqt_ctx *ctx, int rank, int world, const uint8_t id[SQT_COMM_ID_BYTES]);
/* single-process form: ctxs[0..n) on n distinct devices, ncclCommInitAll underneath */
int sqt_comm_init_all(sqt_ctx **ctxs, int n);
/* render on every context of a single-process group concurrently (rank 0 gets the image) */
int sqt_render_group(sqt_ctx **ctxs, int n, const sqt_camera *cam, const sqt_render_params *params,
                     uint8_t *rgb8_out, float *accum_out, sqt_stats *stats_or_null);

/* progressive frames: one sqt_render_params job (the target spp and everything else) advanced in chunks of samples per
 * pixel, so that a host can show previews, bound the time a frame takes and stop once the image is good enough ---------
 *
 * Seeds stay keyed to the target spp: sample k of pixel (y, x) uses generator seed spp*(x + y*seed_stride) + k as in
 * sqt_render.  After k < spp samples the image is the k-sample PREFIX of the spp frame, not an spp = k render.
 *
 * sqt_render_begin     does the checks and the pre-pass of sqt_render, makes every allocation the frame needs, zero-fills
 *                      and traces the primary hits -- no paths.  Stats: what that cost.  Cast mode (mode 1) and
 *                      SQT_F_SPLIT_SAMPLES are SQT_E_UNSUPPORTED.
 * sqt_render_advance   traces samples [k, min(k + n_samples, spp)), then reduces (groups), tone-maps the preview
 *                      (rgbFloatToPixelRGB of sum * (1.0f/(float)k)) and computes the noise estimate; it allocates
 *                      nothing.  n_samples < 1 is SQT_E_INVALID; at k = spp it returns SQT_OK and launches nothing.
 *                      Summed over begin and every advance, the stats' rays / samples / counters equal sqt_render's.
 * After all spp samples, with any chunking, the sums and RGB8 equal sqt_render's for the same job bit for bit.
 * Every progressive frame also keeps the per-pixel second moment s2 = s2 + x*x over the sample radiances x (binary32,
 * sample order, from +0); sqt_download_moments reads it, sqt_download_image reads the sums and the preview (both
 * SQT_E_INVALID before the first advance / outside a frame).
 * noise (rank 0; NaN on other ranks), fp64 over all N = rows*cols*3 values after n = k samples:
 *   mu = s1/n, var = max(0, (s2 - s1*mu)/(n-1)), e2 = var/n, noise = sqrt(sum(e2)/N) / (sum(mu)/N);
 *   0 when sum(mu) = 0, +inf when k < 2.  The reduction order is fixed: the same buffers give the same bits.
 * A frame ends with sqt_render[_resident|_group], sqt_tone_map, sqt_upload_scene[_group], sqt_upload_spheres or a new
 * begin; sqt_render_advance then returns SQT_E_INVALID.  sqt_intersect_batch does not end a frame.
 * In a group every rank must make the same calls: ranks that disagree on k, the target spp or the chunk fail on every
 * rank before anything is traced. */
typedef struct sqt_progress {
    int32_t samples_done, samples_total;
    double noise;
} sqt_progress;                          /* 16 B */
int sqt_render_begin(sqt_ctx *ctx, const sqt_camera *cam, const sqt_render_params *params, sqt_stats *stats_or_null);
int sqt_render_advance(sqt_ctx *ctx, int32_t n_samples, sqt_progress *progress_or_null, sqt_stats *stats_or_null);
int sqt_render_begin_group(sqt_ctx **ctxs, int n, const sqt_camera *cam, const sqt_render_params *params, sqt_stats *stats_or_null);
int sqt_render_advance_group(sqt_ctx **ctxs, int n, int32_t n_samples, sqt_progress *progress_or_null, sqt_stats *stats_or_null);
int sqt_download_moments(sqt_ctx *ctx, float *m2_out);   /* rows*cols*3 floats: s2 of the frame in progress (rank 0) */

/* adaptive sampling in a progressive frame: between two advances, stop tracing the pixels that have converged -------
 *
 * sqt_render_retire    looks at every active pixel after k = samples_done samples and retires it when k >= min_samples
 *                      and, in fp64 and in this order (n = k: every active pixel has exactly k samples):
 *                        for c in r,g,b:  mu_c = s1_c / n ;  v_c = (s2_c - s1_c*mu_c) / (n-1) ;  v_c = v_c > 0 ? v_c : 0
 *                        e2 = (v_r + v_g + v_b) / n ;  m = mu_r + mu_g + mu_b ;  t = max(rel_tol * m, abs_tol)
 *                        retire iff e2 < t*t
 *                      (the per-value terms of the noise estimate).  The comparison is strict, so zero tolerances retire
 *                      nothing, and an all-black pixel (m = 0, e2 = 0) only retires when abs_tol > 0.  A NaN in the sums,
 *                      the moments or any of these terms means the pixel is never retired.  A retired pixel's sums and
 *                      moments are frozen and it is never traced again in this frame.  *active_out: the pixels still
 *                      active in the whole frame (all ranks).  At k = spp or k < min_samples it changes nothing.
 *                      Stopping where the data says the estimate is good enough is a known source of bias: the expected
 *                      value of an adaptive frame is not that of the spp frame.  Each pixel's VALUE is still exactly the
 *                      n_p-sample prefix of the spp frame (seeds stay keyed to the target spp).
 * sample count n_p     the samples in a pixel's sums: the k at which it retired, else samples_done (pixels without a
 *                      primary hit included).  Previews and the final image are rgbFloatToPixelRGB(sum * (1.0f/(float)n_p))
 *                      per pixel, the reciprocal correctly rounded, so a pixel with n_p = spp has sqt_render's bytes; the
 *                      noise estimate uses n = n_p in each pixel's terms.  A frame that never retires is unchanged.
 * sqt_render_advance   traces the active pixels only: stats.samples = active pixels * samples in the chunk.  With no
 *                      active pixel left it launches nothing (samples_done still moves on).
 * Errors: SQT_E_INVALID outside a frame, before k >= 2, for min_samples < 2, negative or NaN tolerances or non-zero
 * reserved; SQT_E_UNSUPPORTED for a frame begun with SQT_F_NO_PRIMARY_REUSE and without a lens (sqt_set_lens).  Whatever ends a frame ends its adaptive
 * state.  In a group every rank retires its own pixels from its own sums; ranks that disagree on k, the target spp or
 * any of the three criteria fail on every rank before anything runs.  The counts reach rank 0 by a sum over ranks, and
 * a group frame is bit-identical to one GPU's. */
typedef struct sqt_retire_params {
    float rel_tol, abs_tol;              /* error target: sqrt(e2) < max(rel_tol * m, abs_tol) */
    int32_t min_samples;                 /* >= 2 */
    uint32_t reserved;                   /* 0 */
} sqt_retire_params;                     /* 16 B */
int sqt_render_retire(sqt_ctx *ctx, const sqt_retire_params *rp, int64_t *active_out_or_null);
int sqt_render_retire_group(sqt_ctx **ctxs, int n, const sqt_retire_params *rp, int64_t *active_out_or_null);
int sqt_download_sample_counts(sqt_ctx *ctx, int32_t *counts_out);   /* rows*cols n_p of the frame in progress (rank 0) */

/* denoised previews of a progressive frame: an edge-aware a-trous wavelet filter guided by the primary hits and the
 * per-pixel variance (the spatial part of SVGF: Dammertz et al. 2010, Schied et al. 2017) -------------------------------
 *
 * Valid inside a progressive frame after k = samples_done >= 2 samples.  These calls read the frame and change nothing
 * of it: a later advance, retire, download or denoise behaves exactly as if they had not been made, and they never end
 * the frame.  The filter is biased, as every denoiser is.  It does not demodulate albedo: the scenes have no textures,
 * albedo is constant per material and no two materials are ever blended.
 * All arithmetic is binary32, one explicit rounding per operation, no contraction, only + - * / sqrt min max (so a host
 * build gives the device's bits); e2 is fp64 as in sqt_render_retire.
 * Inputs per pixel p (rank 0, after k samples):
 *   n_p    the pixel's sample count (sqt_download_sample_counts);  c_p = s1_p * (1.0f/(float)n_p) per channel, the values
 *          the preview tone-maps;  v_p = (float)e2 with e2 of sqt_render_retire's test at n = n_p;  l_p = (c_r + c_g) + c_b
 *   valid  the pixel has a primary hit; an invalid pixel's output is its input and it is never a neighbour
 *   mat_p  material of the primary hit;  z_p = its t;  N_p its unit geometric normal: e1 x e2 (triangle) or hit - centre
 *          (sphere, hit = o + t*d), divided by its length sqrt(N.N), negated when N.d > 0 (facing the camera ray)
 *   mirror reflective >= 1: this integrator's perfect mirror; the primary features say nothing about what it shows, so
 *          the pixel is passed through unfiltered
 * Level i = 0 .. levels-1, step s = 2^i, for every valid non-mirror p, reading the previous level's (c, v):
 *   g_p = sqrt(sum k_j v_j / sum k_j) over the 3x3 neighbours j of p (step 1, in the image, valid, same material, p
 *         included), k = [1,2,1] x [1,2,1], rows outer
 *   taps q = p + s*(dy, dx), dy outer, dx inner, both -2..2, skipping those outside the image, invalid or of another
 *   material:  h = h1(dy)*h1(dx) with h1(-2..2) = 1/16, 1/4, 3/8, 1/4, 1/16 ;
 *              x = |l_p - l_q| / (sigma_l*g_p + 1e-6f) + |z_p - z_q| / ((sigma_z*s)*z_p) ;
 *              w_n = max(0, N_p.N_q) squared 7 times ;  r = 1/(1 + x*0.125f) squared 3 times  ((1 + x/8)^-8 ~ exp(-x)) ;
 *              w = (h*w_n)*r, except at q = p: w = 9/64 exactly (so sum w > 0)
 *   c'_p = sum w*c_q / sum w per channel,  v'_p = sum (w*w)*v_q / (sum w * sum w), every sum in tap order from +0
 * Output: the last level's c (levels = 0: c itself, the preview's mean bit for bit) and its RGB8 = rgbFloatToPixelRGB(c)
 * (the preview's RGB8 at levels = 0).  A fixed shape, one thread per pixel, no atomics: the bits never depend on the
 * device, the SM count or the group size.
 * sqt_denoise            rank 0 gets rows*cols*3 RGB8 bytes and floats (either may be NULL); the preview is not touched.
 *                        Stats: device_ms, reduce_ms (the feature reduce), d2h_ms / d2h_bytes, kernel_launches.
 * sqt_download_features  rank 0: surface (tri_out numbering: orig_index, n_tris + k for sphere k, -1 for no hit), depth
 *                        (t) and the camera-facing normal N (rows*cols*3) the filter uses -- AOVs for an external denoiser
 *                        too.  Any pointer may be NULL.
 * Errors: SQT_E_INVALID outside a frame, k < 2, levels outside 0..8, a sigma that is not positive and finite, non-zero
 * reserved; SQT_E_UNSUPPORTED for a frame begun with SQT_F_NO_PRIMARY_REUSE or with a lens (it keeps no primary hits).
 * In a group every rank makes the same calls (sqt_download_features included); ranks that disagree on k, the target spp,
 * levels or the sigmas fail on every rank before anything runs.  The features reach rank 0 once per frame by a sum over
 * ranks (each value is non-zero on its owner only, so the sum is exact), and rank 0 filters the sums, moments and counts
 * it holds: a group result is bit-identical to one GPU's.  Whatever ends a frame drops its features. */
typedef struct sqt_denoise_params {
    int32_t levels;                      /* 0..8; 0 = the preview itself */
    float sigma_l, sigma_z;              /* > 0, finite: luminance (in units of the prefiltered standard error) and depth */
    uint32_t reserved;                   /* 0 */
} sqt_denoise_params;                    /* 16 B */
int sqt_denoise(sqt_ctx *ctx, const sqt_denoise_params *dp, uint8_t *rgb8_out, float *mean_out, sqt_stats *stats_or_null);
int sqt_denoise_group(sqt_ctx **ctxs, int n, const sqt_denoise_params *dp, uint8_t *rgb8_out, float *mean_out, sqt_stats *stats_or_null);
int sqt_download_features(sqt_ctx *ctx, int32_t *surface_out, float *depth_out, float *normal_out);

/* camera sampling (extension: the reference's makeRay, Lib.hs:107-114, sends every sample of a pixel along one ray
 * through one point of the pixel): box-filtered pixels (anti-aliasing) and a thin lens (depth of field) ----------------
 *
 * sqt_set_lens sets the context's camera model; NULL restores the reference's pinhole (the default).  Invalid fields
 * (jitter not 0 or 1, a negative or non-finite aperture, a non-positive or non-finite focus distance, non-zero reserved)
 * are SQT_E_INVALID and leave the lens unchanged.  sqt_render, sqt_render_resident, sqt_render_group and
 * sqt_render_begin[_group] read the lens when the frame starts; a progressive frame keeps the lens it began with.
 * sqt_intersect_batch ignores it (it takes the caller's rays).
 * The primary ray of sample k of pixel (y, x) in a frame with a lens set, s = spp*(x + y*seed_stride) + k the sample's
 * stream, every operation one binary32 rounding in exactly this order, no contraction:
 *   w0..w3 = Philox4x32-10(counter (s lo, s hi, 0, "SQTL" = 0x4C545153), key seed);  u_i = random_r01(w_i) (Lib.hs:183-188)
 *     (the bounce draws use counter word "SQTR": they are untouched)
 *   jx = jitter ? u0 - 0.5f : 0 ;  jy = jitter ? u1 - 0.5f : 0 ;  fx = (float)x + jx ;  fy = (float)y + jy
 *   xo = (fx - ww/2) / ww ;  yo = (hh/2 - fy) / hh        with ww = (float)xdiv, hh = (float)ydiv (jx = 0: makeRay's bits)
 *   o = position ;  d_i = ((0 + 1*R[i]) + xo*R[3+i]) + yo*R[6+i]          (rotVert, R = rotation, row-major)
 *   aperture A == 0: the ray is (o, d).  Otherwise, with f = focus_distance:
 *     r = A * sqrt(u2) ;  th = 6.2831855f * u3 ;  (sn, cs) = sqt_sincos(th)  (DESIGN.md section 6) ;  a = r*cs ;  b = r*sn
 *     off_i = a*R[3+i] + b*R[6+i] ;  inv_f = 1/f ;  o'_i = o_i + off_i ;  d'_i = d_i - off_i*inv_f
 *   so that o' + f*d' = o + f*d: every lens sample of an image point meets at ray parameter t = f (along the unnormalised
 *   camera ray), the plane in focus.  The footprint of a jittered pixel is [x - 1/2, x + 1/2] x [y - 1/2, y + 1/2] around
 *   the reference's sample point, so an anti-aliased frame stays registered with the pinhole frame.
 * A frame with a lens set traces every owned pixel's primary ray for every sample: there is no primary pass and no primary
 * reuse (SQT_F_NO_PRIMARY_REUSE changes nothing), and a pixel whose centre ray misses is sampled too.  rays_reference
 * equals rays_traced.  Seeds stay keyed to the target spp, so a progressive lens frame's preview after k samples is the
 * exact k-sample prefix and its final frame equals the one-shot lens frame bit for bit; sqt_render_retire works (every
 * owned pixel starts active); a group frame is bit-identical to one GPU's.  SQT_E_UNSUPPORTED: cast mode (mode 1) with a
 * lens, and sqt_denoise[_group] / sqt_download_features on a lens frame (they need the primary hits, which a lens frame
 * does not trace; denoising lens frames is not supported).  In a group every rank must have the same lens (or none):
 * ranks that disagree fail on every rank before anything is enqueued. */
typedef struct sqt_lens {
    uint32_t jitter;                     /* 0 or 1: box-filtered pixels */
    float aperture_radius;               /* >= 0, finite, world units; 0 = pinhole */
    float focus_distance;                /* > 0, finite: ray parameter t of the sharp plane along the unnormalised camera ray */
    uint32_t reserved;                   /* 0 */
} sqt_lens;                              /* 16 B */
int sqt_set_lens(sqt_ctx *ctx, const sqt_lens *lens_or_null);

/* measured roofline denominators on this device (microbenchmarks; see DESIGN.md) ------------- */
int sqt_measure_fp32_peak(sqt_ctx *ctx, double *gops_per_s);     /* non-fused FADD/FMUL issue rate, Gop/s */
int sqt_measure_l2_bandwidth(sqt_ctx *ctx, double *gb_per_s);    /* L2-resident 128-bit read bandwidth */

/* options: SQT_OPT_LEAF_CULL (default 1) -- skip leaves whose conservatively enlarged tight box the ray
 * misses.  Exact (DESIGN.md section 5); 0 reproduces the reference's triangle-test count one for one. */
#define SQT_OPT_LEAF_CULL 1
/* SQT_OPT_SPHERE_BVH (default 1) -- extension: find the spheres a ray can hit through a bounding-volume hierarchy built at
 * sqt_upload_spheres instead of testing every sphere for every ray.  Exact (same closest surface, same tie-break); 0
 * keeps the literal definition. */
#define SQT_OPT_SPHERE_BVH 2
int sqt_set_option(sqt_ctx *ctx, int option, int value);

/* introspection used by tests */
int sqt_device_info(sqt_ctx *ctx, int *sm_count, int *cc_major, int *cc_minor, char name_out[128]);

#ifdef __cplusplus
}
#endif
#endif /* SQT_H */
