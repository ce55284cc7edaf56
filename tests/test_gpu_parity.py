"""Parity tests proper: the CUDA path, called through the C ABI (include/sqt.h), against the CPU oracle.

Bar: bit-exact for hit index, dist, hit point, the float accumulation buffer and the RGB8 image (integer/byte/
index work and -- because the oracle restates the device's "sqt trig" polynomials and shares the counter-based
RNG -- the floating-point image too).  Against the reference-faithful libm oracle the bar is a stated RMSE.
"""
import contextlib

import numpy as np
import pytest

import pysqt
from oracle import oracle as O
from pysqt import scenes

from common import adversarial_rays, assert_same_hits, bits, build_pair, random_rays

pytestmark = pytest.mark.gpu


@contextlib.contextmanager
def no_leaf_cull(ctx):
    """The conservative leaf culling skips triangle tests the reference performs; switch it off where the test
    compares work counters with the oracle's."""
    ctx.set_leaf_cull(False)
    try:
        yield
    finally:
        ctx.set_leaf_cull(True)


def test_device_is_b200(gpu_ctx):
    info = gpu_ctx.info()
    assert info["cc"][0] == 10, info
    assert info["sm_count"] >= 100


# ------------------------------------------------------------------ closest hit, bit exact
def test_primary_rays_bit_exact(gpu_ctx, host_scene, oracle_scene, camera):
    gpu_ctx.upload(host_scene)
    org, dirs = O.make_rays(O.make_params(540, 540, 1), camera)
    want = oracle_scene.intersect_batch(org, dirs, counters=True)
    assert_same_hits(gpu_ctx.intersect_batch(org, dirs), want, "primary 540x540 (leaf culling on)")
    with no_leaf_cull(gpu_ctx):
        got = gpu_ctx.intersect_batch(org, dirs, want_stats=True)
    assert_same_hits(got, want, "primary 540x540")
    st, cn = got[3], want[3]
    # the traversal visits exactly the reference's subtrees: same branch visits and triangle tests
    assert st["branch_visits"] == int(cn[0]) and st["child_box_tests"] == int(cn[1]) and st["tri_tests"] == int(cn[3])
    assert st["rays_traced"] == len(org)


def test_gpu_matches_committed_golden_fixtures(gpu_ctx, host_scene, camera):
    """tests/golden/scene_obj_golden.json (made by tests/golden/make_golden.py with the oracle): the device must
    reproduce the hashed hit indices / dist / points of the 540x540 reference-default frame and the hashed render."""
    import json, os
    from golden.make_golden import sha
    gold = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "scene_obj_golden.json")))
    gpu_ctx.upload(host_scene)
    org, dirs = O.make_rays(O.make_params(540, 540, 1), camera)
    tri, dist, point = gpu_ctx.intersect_batch(org, dirs)
    g = gold["primary_540"]
    assert int((tri >= 0).sum()) == g["hits"]
    assert sha(tri) == g["sha_tri"] and sha(dist) == g["sha_dist"] and sha(point) == g["sha_point"]
    out = gpu_ctx.render(camera, pysqt.make_params(64, 64, 4, max_depth=3, seed=1))
    g = gold["render_64x64_4spp_d3_seed1_sqttrig"]
    assert sha(out["accum"]) == g["sha_accum"] and sha(out["rgb8"]) == g["sha_rgb8"]


def test_literal_nonsquare_primary_rays(gpu_ctx, host_scene, oracle_scene, camera):
    gpu_ctx.upload(host_scene)
    org, dirs = O.make_rays(O.make_params(320, 200, 1, literal=True), camera)
    assert_same_hits(gpu_ctx.intersect_batch(org, dirs), oracle_scene.intersect_batch(org, dirs), "literal 320,200")


def test_random_incoherent_rays_bit_exact(gpu_ctx, host_scene, oracle_scene):
    gpu_ctx.upload(host_scene)
    org, dirs = random_rays(300_000, seed=11)
    assert_same_hits(gpu_ctx.intersect_batch(org, dirs), oracle_scene.intersect_batch(org, dirs), "random")


def test_adversarial_rays_bit_exact(gpu_ctx, host_scene, oracle_scene):
    gpu_ctx.upload(host_scene)
    v9, _ = oracle_scene.tris()
    org, dirs = adversarial_rays(v9)
    assert_same_hits(gpu_ctx.intersect_batch(org, dirs), oracle_scene.intersect_batch(org, dirs), "adversarial")


def test_matches_naive_intersect_up_to_ties(gpu_ctx, host_scene, oracle_scene, camera):
    """The reference's own differential pair (naiveIntersect vs intersectBIH): same dist always, same triangle
    except exact ties."""
    gpu_ctx.upload(host_scene)
    org, dirs = O.make_rays(O.make_params(96, 96, 1), camera)
    tri, dist, _ = gpu_ctx.intersect_batch(org, dirs)
    ntri, ndist, _ = oracle_scene.intersect_batch(org, dirs, naive=True)
    assert np.array_equal((tri >= 0), (ntri >= 0))
    assert np.array_equal(bits(dist), bits(ndist))
    assert (tri != ntri).mean() < 0.01


def test_recorded_bounce_rays(gpu_ctx, host_scene, oracle_scene, camera):
    """Secondary rays: origins on surfaces (self-hit rejection by t > eps), unit scatter directions."""
    gpu_ctx.upload(host_scene)
    org, dirs = O.make_rays(O.make_params(200, 200, 1), camera)
    tri, dist, point = oracle_scene.intersect_batch(org, dirs)
    hit = tri >= 0
    rng = np.random.default_rng(3)
    d2 = rng.normal(size=(hit.sum(), 3)).astype(np.float32)
    d2 /= np.linalg.norm(d2, axis=1, keepdims=True).astype(np.float32)
    assert_same_hits(gpu_ctx.intersect_batch(point[hit], d2), oracle_scene.intersect_batch(point[hit], d2), "bounce")


def test_leaf_culling_changes_no_result(gpu_ctx, host_scene, camera):
    """2M incoherent + 1M camera rays: identical index, dist and point bits with the culling on and off, and the
    culling really skips work."""
    gpu_ctx.upload(host_scene)
    org, dirs = random_rays(2_000_000, seed=99)
    o2, d2 = O.make_rays(O.make_params(1000, 1000, 1), camera)
    org = np.concatenate([org, o2]); dirs = np.concatenate([dirs, d2])
    on = gpu_ctx.intersect_batch(org, dirs, want_stats=True)
    with no_leaf_cull(gpu_ctx):
        off = gpu_ctx.intersect_batch(org, dirs, want_stats=True)
    assert_same_hits(on, off, "cull on vs off")
    assert on[3]["leaves_culled"] > 0 and off[3]["leaves_culled"] == 0
    assert on[3]["tri_tests"] < 0.8 * off[3]["tri_tests"]


def test_empty_batch_and_errors(gpu_ctx, host_scene):
    gpu_ctx.upload(host_scene)
    tri, dist, point = gpu_ctx.intersect_batch(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32))
    assert len(tri) == 0
    fresh = pysqt.Context(0)
    with pytest.raises(pysqt.SqtError, match="before sqt_upload_scene"):
        fresh.intersect_batch(np.zeros((1, 3), np.float32), np.ones((1, 3), np.float32))
    bad = host_scene.desc()
    bad.n_mats = 0
    assert fresh.upload_desc_raw(bad) == 1 and "materials" in fresh.last_error()
    p = pysqt.make_params(8, 8, 1, max_depth=0)
    fresh.upload(host_scene)
    with pytest.raises(pysqt.SqtError, match="max_depth"):
        fresh.render(pysqt.load_camera(pysqt.ROOT + "/data/camera"), p)
    fresh.close()


@pytest.mark.parametrize("n_tris", [1, 9, 14])
def test_root_leaf_scene(gpu_ctx, n_tris):
    """Fewer than 15 triangles: the tree is a single Leaf and no box test happens at all (BIH.hs:69,105)."""
    v9, mi, mats = scenes.triangle_soup(n_tris, seed=2)
    osc, hs = build_pair(v9 * 40.0, mi, mats)
    assert hs.n_nodes == 1
    gpu_ctx.upload(hs)
    org, dirs = random_rays(20000, seed=4, lo=-1, hi=1)
    assert_same_hits(gpu_ctx.intersect_batch(org, dirs), osc.intersect_batch(org, dirs), "root leaf")


def test_degenerate_split_and_empty_leaves(gpu_ctx):
    """All centroids equal on the split axis -> one side empty -> Branch (Leaf empty) (Leaf everything), a leaf
    longer than 14 (BIH.hs:70-75)."""
    rng = np.random.default_rng(8)
    n = 40
    base = rng.uniform(-1, 1, (n, 1, 3)).astype(np.float32) * np.array([0, 1, 1], np.float32)   # x centroid identical
    offs = np.array([[0.3, 0, 0], [-0.15, 0.2, 0.1], [-0.15, -0.2, -0.1]], np.float32)
    v9 = (base * np.array([1e-3, 1e-3, 1e-3], np.float32) + offs[None]).reshape(n, 9)
    mats = np.array([[0, .5, .5, .5, 0, 0, 0, 0]], np.float32)
    osc, hs = build_pair(v9, np.zeros(n, np.int32), mats)
    assert hs.stats()["longest_leaf"] > 14
    gpu_ctx.upload(hs)
    org, dirs = random_rays(20000, seed=5, lo=-1, hi=1)
    assert_same_hits(gpu_ctx.intersect_batch(org, dirs), osc.intersect_batch(org, dirs), "degenerate")


@pytest.mark.parametrize("tune", ["12,0,12", "8,1,8"])
def test_long_leaf_with_duplicate_triangles(monkeypatch, tune):
    """A leaf of 2600 triangles (longer than the 1024 tests the warp-cooperative triangle phase takes from one leaf per
    phase) in which every triangle exists four times: all four copies are hit at exactly the same distance, so the
    result depends on the order of the min' fold (BIH.hs:105-109: the first of the minimal ones wins).  Both triangle
    phases -- tests spread over all lanes (b_leave = 0) and one test per lane and step -- must reproduce it."""
    monkeypatch.setenv("SQT_TUNE", tune)
    rng = np.random.default_rng(21)
    n0, copies = 650, 4
    base = rng.uniform(-1, 1, (n0, 1, 3)).astype(np.float32) * np.array([0, 1, 1], np.float32)   # x centroid identical
    offs = np.array([[0.3, 0, 0], [-0.15, 0.2, 0.1], [-0.15, -0.2, -0.1]], np.float32)
    v9 = (base * np.float32(2e-3) + offs[None]).reshape(n0, 9)                 # x extent dominates: the split axis is x
    v9 = np.tile(v9, (copies, 1))[rng.permutation(n0 * copies)]
    mats = np.array([[0, .5, .5, .5, 0, 0, 0, 0]], np.float32)
    osc, hs = build_pair(v9, np.zeros(len(v9), np.int32), mats)
    assert hs.stats()["longest_leaf"] == n0 * copies
    ctx = pysqt.Context(0)
    ctx.upload(hs)
    org = rng.uniform(-1, 1, (6000, 3)).astype(np.float32)
    target = rng.uniform([-0.1, -0.12, -0.06], [0.2, 0.12, 0.06], (6000, 3)).astype(np.float32)   # inside the pile of triangles
    dirs = target - org
    got, ref = ctx.intersect_batch(org, dirs), osc.intersect_batch(org, dirs)
    assert (ref[0] >= 0).mean() > 0.3
    assert_same_hits(got, ref, "long leaf, duplicates, SQT_TUNE=" + tune)
    ctx.close()


@pytest.mark.parametrize("gen,n", [("cornell", 10000), ("soup", 60000), ("mesh", 80000)])
def test_synthetic_scenes_bit_exact(gpu_ctx, gen, n):
    v9, mi, mats = {"cornell": scenes.cornell_box, "soup": scenes.triangle_soup, "mesh": scenes.subdivided_mesh}[gen](n)
    osc, hs = build_pair(v9, mi, mats)
    gpu_ctx.upload(hs)
    org, dirs = random_rays(100_000, seed=21, lo=-1.5, hi=1.5)
    want = osc.intersect_batch(org, dirs, counters=True)
    culled = gpu_ctx.intersect_batch(org, dirs, want_stats=True)
    assert_same_hits(culled, want, gen + " (leaf culling on)")
    with no_leaf_cull(gpu_ctx):
        got = gpu_ctx.intersect_batch(org, dirs, want_stats=True)
    assert_same_hits(got, want, gen)
    assert got[3]["tri_tests"] == int(want[3][3]) and got[3]["branch_visits"] == int(want[3][0])
    assert culled[3]["branch_visits"] <= got[3]["branch_visits"] and culled[3]["tri_tests"] <= got[3]["tri_tests"]      # culling skips leaves and subtrees


# ------------------------------------------------------------------ rendered image
@pytest.mark.parametrize("w,h,spp,depth,literal", [(96, 64, 8, 3, False), (64, 64, 6, 8, False), (80, 48, 5, 3, True), (48, 48, 3, 1, False)])
def test_render_bit_exact_vs_oracle(gpu_ctx, host_scene, oracle_scene, camera, w, h, spp, depth, literal):
    gpu_ctx.upload(host_scene)
    out = gpu_ctx.render(camera, pysqt.make_params(w, h, spp, max_depth=depth, seed=5, literal=literal))
    ref = oracle_scene.render(camera, O.make_params(w, h, spp, max_depth=depth, seed=5, trig=1, literal=literal))
    assert out["accum"].shape == ref["accum"].shape
    assert np.array_equal(bits(out["accum"]), bits(ref["accum"]))
    assert np.array_equal(out["rgb8"], ref["rgb8"])
    assert out["stats"]["samples"] == ref["samples"] == w * h * spp
    assert out["stats"]["rays_traced"] <= ref["rays"]


def test_render_reference_work_flags_match_oracle_counts(gpu_ctx, host_scene, oracle_scene, camera):
    """With primary reuse and early termination off the device traces exactly the reference's rays: ray count,
    branch visits and triangle tests equal the oracle's counters."""
    gpu_ctx.upload(host_scene)
    f = pysqt.SQT_F_NO_PRIMARY_REUSE | pysqt.SQT_F_NO_EARLY_TERMINATION | pysqt.SQT_F_COUNT_WORK
    with no_leaf_cull(gpu_ctx):
        out = gpu_ctx.render(camera, pysqt.make_params(72, 56, 6, max_depth=4, seed=9, flags=f))
    ref = oracle_scene.render(camera, O.make_params(72, 56, 6, max_depth=4, seed=9, trig=1))
    assert np.array_equal(bits(out["accum"]), bits(ref["accum"]))
    st, cn = out["stats"], ref["counters"]
    assert st["rays_traced"] == ref["rays"]
    assert st["branch_visits"] == cn["branch_visits"] and st["tri_tests"] == cn["tri_tests"]
    assert st["child_box_tests"] == cn["child_box_tests"]


def test_render_rmse_vs_reference_faithful_libm_oracle(gpu_ctx, host_scene, oracle_scene, camera):
    """Against the oracle in libm mode (cosf/sinf/acosf/atanf as GHC calls them): stated tolerance
    per-pixel RMSE of the mean radiance <= 2e-3 (scene radiance scale: light = 100), RGB8 may differ by 1 level
    on < 0.1% of the bytes."""
    gpu_ctx.upload(host_scene)
    w, h, spp = 128, 128, 64
    out = gpu_ctx.render(camera, pysqt.make_params(w, h, spp, max_depth=3, seed=1))
    ref = oracle_scene.render(camera, O.make_params(w, h, spp, max_depth=3, seed=1, trig=0))
    rmse = float(np.sqrt(np.mean((out["accum"] / spp - ref["accum"] / spp) ** 2)))
    assert rmse <= 2e-3, rmse
    d = np.abs(out["rgb8"].astype(int) - ref["rgb8"].astype(int))
    assert d.max() <= 1 and (d > 0).mean() < 1e-3


def test_cast_mode_bit_exact(gpu_ctx, host_scene, oracle_scene, camera):
    gpu_ctx.upload(host_scene)
    out = gpu_ctx.render(camera, pysqt.make_params(120, 90, 4, mode=1))
    ref = oracle_scene.render(camera, O.make_params(120, 90, 4, mode=1, trig=1))
    assert np.array_equal(bits(out["accum"]), bits(ref["accum"]))
    assert np.array_equal(out["rgb8"], ref["rgb8"])


def test_tone_map_bit_exact(gpu_ctx):
    rng = np.random.default_rng(0)
    x = np.concatenate([rng.uniform(0, 3, (5000, 3)), rng.uniform(0, 200, (2000, 3)), np.zeros((4, 3)),
                        np.array([[0, 0, 1e-30], [1e20, 1, 0], [np.inf, 1, 1], [0.4142135, 0.4142136, 2.4142137]])]).astype(np.float32)
    assert np.array_equal(gpu_ctx.tone_map(x), O.tone_map(x, 1, trig=1))


def test_resident_then_download_equals_render(gpu_ctx, host_scene, camera):
    gpu_ctx.upload(host_scene)
    p = pysqt.make_params(64, 48, 4, max_depth=3, seed=2)
    a = gpu_ctx.render(camera, p)
    st = gpu_ctx.render_resident(camera, p)
    rgb8, accum = gpu_ctx.download(p.rows, p.cols)
    assert np.array_equal(a["rgb8"], rgb8) and np.array_equal(bits(a["accum"]), bits(accum))
    # k_primary + one (k_paths_pool, k_accumulate) pair per sample round + k_tonemap
    assert st["rays_traced"] == a["stats"]["rays_traced"] and st["kernel_launches"] == 4


def test_many_sample_rounds_are_bit_identical(host_scene, camera, monkeypatch):
    """A tiny sample-buffer budget forces several rounds of samples; the per-pixel sums must not change."""
    monkeypatch.setenv("SQT_SBUF_MB", "1")
    small = pysqt.Context(0)
    small.upload(host_scene)
    p = pysqt.make_params(160, 120, 24, max_depth=4, seed=8)
    a = small.render(camera, p)
    small.close()
    monkeypatch.delenv("SQT_SBUF_MB")
    big = pysqt.Context(0)
    big.upload(host_scene)
    b = big.render(camera, p)
    big.close()
    assert a["stats"]["kernel_launches"] > b["stats"]["kernel_launches"]
    assert np.array_equal(bits(a["accum"]), bits(b["accum"])) and np.array_equal(a["rgb8"], b["rgb8"])


def test_every_path_kernel_scheduler_is_bit_exact(host_scene, oracle_scene, camera):
    """The path kernel schedules rays onto lanes from pools of 64 rays per warp in shared memory; the oracle traces one
    path after the other.  Scheduling must never change a result."""
    ctx = pysqt.Context(0)
    ctx.upload(host_scene)
    for w, h, spp, depth, flags in [(96, 64, 8, 8, 0), (64, 48, 5, 3, pysqt.SQT_F_NO_PRIMARY_REUSE | pysqt.SQT_F_NO_EARLY_TERMINATION),
                                    (40, 40, 3, 1, 0)]:
        out = ctx.render(camera, pysqt.make_params(w, h, spp, max_depth=depth, seed=13, flags=flags))
        ref = oracle_scene.render(camera, O.make_params(w, h, spp, max_depth=depth, seed=13, trig=1))
        assert np.array_equal(bits(out["accum"]), bits(ref["accum"])) and np.array_equal(out["rgb8"], ref["rgb8"])
        assert out["stats"]["samples"] == ref["samples"]
        if flags:
            assert out["stats"]["rays_traced"] == ref["rays"]
    ctx.close()


def test_baseline_config2_at_full_size(gpu_ctx, host_scene, oracle_scene, camera):
    """BASELINE.json configs[1] exactly: data/scene.obj, 1920x1080, 1024 spp, 8 bounces (2.1e9 samples, 5.3e9 rays).
    Size-independent checks: exact sample accounting; misses are exactly black; twelve pixels re-rendered by the
    oracle with all their 1024 samples match bit for bit (so the 16 accumulation rounds add in sample order); the
    RGB8 frame equals the oracle's tone map of the device's sums."""
    gpu_ctx.upload(host_scene)
    W, H, spp, depth = 1920, 1080, 1024, 8
    p = pysqt.make_params(W, H, spp, max_depth=depth, seed=0)
    out = gpu_ctx.render(camera, p)
    acc, st = out["accum"], out["stats"]
    assert st["samples"] == W * H * spp
    assert 5.0e9 < st["rays_traced"] < 5.6e9
    org, dirs = O.make_rays(O.make_params(W, H, 1), camera)
    miss = (gpu_ctx.intersect_batch(org, dirs)[0] < 0).reshape(H, W)
    assert np.all(acc[miss] == 0) and np.all(acc[~miss].sum(-1) >= 0)
    op = O.make_params(W, H, spp, max_depth=depth, seed=0, trig=1)
    rng = np.random.default_rng(5)
    hit_pixels = np.flatnonzero(~miss.ravel())
    for pix in rng.choice(hit_pixels, 12, replace=False):
        want = O.render_window(oracle_scene, camera, op, int(pix), int(pix) + 1)
        assert np.array_equal(bits(acc.reshape(-1, 3)[pix]), bits(want[0])), "pixel %d" % pix
    assert np.array_equal(out["rgb8"], O.tone_map(acc, spp, trig=1))


def test_schedulers_and_culling_agree_at_full_size(host_scene, camera):
    """The bench frame (1920x1080, depth 8) at 32 spp -- 170 M rays -- rendered three ways: default, without the leaf
    culling, and without primary reuse / early termination.  All three accumulation buffers must be bit-identical, and
    the last one must trace strictly more rays."""
    p = pysqt.make_params(1920, 1080, 32, max_depth=8, seed=21)
    results = {}
    for name, cull, flags in [("pool", True, 0), ("pool-nocull", False, 0),
                              ("pool-reference-work", True, pysqt.SQT_F_NO_PRIMARY_REUSE | pysqt.SQT_F_NO_EARLY_TERMINATION)]:
        ctx = pysqt.Context(0)
        ctx.upload(host_scene)
        ctx.set_leaf_cull(cull)
        pp = pysqt.make_params(1920, 1080, 32, max_depth=8, seed=21, flags=flags)
        out = ctx.render(camera, pp, want_rgb8=False)
        results[name] = (out["accum"], out["stats"])
        ctx.close()
    base = results["pool"][0]
    for name, (acc, st) in results.items():
        assert np.array_equal(bits(acc), bits(base)), name
        assert st["samples"] == 1920 * 1080 * 32
    assert results["pool"][1]["rays_traced"] == results["pool-nocull"][1]["rays_traced"]
    assert results["pool-reference-work"][1]["rays_traced"] > results["pool"][1]["rays_traced"]


def test_render_is_deterministic_and_seed_sensitive(gpu_ctx, host_scene, camera):
    gpu_ctx.upload(host_scene)
    p = pysqt.make_params(64, 64, 16, max_depth=4, seed=11)
    a = gpu_ctx.render(camera, p)["accum"]
    b = gpu_ctx.render(camera, p)["accum"]
    c = gpu_ctx.render(camera, pysqt.make_params(64, 64, 16, max_depth=4, seed=12))["accum"]
    assert np.array_equal(bits(a), bits(b))
    assert not np.array_equal(a, c)


def test_synthetic_cornell_render_bit_exact(gpu_ctx, camera):
    v9, mi, mats = scenes.cornell_box(10000)
    osc, hs = build_pair(v9, mi, mats)
    gpu_ctx.upload(hs)
    out = gpu_ctx.render(camera, pysqt.make_params(64, 48, 4, max_depth=6, seed=4))
    ref = osc.render(camera, O.make_params(64, 48, 4, max_depth=6, seed=4, trig=1))
    assert np.array_equal(bits(out["accum"]), bits(ref["accum"]))


def test_sphere_extension_bit_exact(host_scene, camera):
    """Analytic spheres (north-star extension; semantics in include/sqt.h, restated by the oracle)."""
    spheres = [(0.8, 0.5, -1.2, 0.6, 5), (-0.9, 1.0, 0.3, 0.45, 1), (0.0, -0.5, 1.2, 0.3, 3), (0.0, 3.0, 0.5, 0.25, 2)]
    osc = O.Scene.load(pysqt.ROOT + "/data/scene.obj", pysqt.ROOT + "/data")
    osc.make_bih()
    osc.set_spheres(spheres)
    ctx = pysqt.Context(0)
    ctx.upload(host_scene)
    ctx.upload_spheres(spheres)
    org, dirs = O.make_rays(O.make_params(300, 300, 1), camera)
    o2, d2 = random_rays(200000, 9)
    org = np.concatenate([org, o2]); dirs = np.concatenate([dirs, d2])
    want = osc.intersect_batch(org, dirs)
    assert_same_hits(ctx.intersect_batch(org, dirs), want, "spheres")
    assert (want[0] >= osc.n_tris).sum() > 5000
    for depth, mode in ((3, 0), (8, 0), (3, 1)):
        out = ctx.render(camera, pysqt.make_params(96, 64, 6, max_depth=depth, seed=3, mode=mode))
        ref = osc.render(camera, O.make_params(96, 64, 6, max_depth=depth, seed=3, trig=1, mode=mode))
        assert np.array_equal(bits(out["accum"]), bits(ref["accum"])) and np.array_equal(out["rgb8"], ref["rgb8"])
    bad = pysqt.np.zeros(1, pysqt.SPHERE_DT); bad[0]["radius"] = 1.0; bad[0]["material"] = 99
    assert ctx.L.sqt_upload_spheres(ctx.h, bad.ctypes.data, 1) == 1 and "material" in ctx.last_error()
    ctx.upload_spheres([])
    plain = O.Scene.load(pysqt.ROOT + "/data/scene.obj", pysqt.ROOT + "/data"); plain.make_bih()
    assert_same_hits(ctx.intersect_batch(org[:20000], dirs[:20000]), plain.intersect_batch(org[:20000], dirs[:20000]), "spheres removed")
    ctx.close()


# ------------------------------------------------------------------ full-size, size-independent properties
def test_full_size_properties_1080p(gpu_ctx, host_scene, oracle_scene, camera):
    """BASELINE config 2 geometry (1920x1080, depth 8) at a reduced spp the oracle cannot follow in full:
    (1) a random sample of pixels is re-rendered by the oracle and must match bit for bit,
    (2) pixels whose primary ray misses are exactly black, (3) sample accounting is exact,
    (4) a second run is bit-identical (dynamic work fetch does not leak into the result)."""
    gpu_ctx.upload(host_scene)
    W, H, spp, depth = 1920, 1080, 16, 8
    p = pysqt.make_params(W, H, spp, max_depth=depth, seed=77)
    out = gpu_ctx.render(camera, p)
    acc = out["accum"]
    assert out["stats"]["samples"] == W * H * spp
    org, dirs = O.make_rays(O.make_params(W, H, 1), camera)
    tri, _, _ = gpu_ctx.intersect_batch(org, dirs)
    miss = (tri < 0).reshape(H, W)
    assert np.all(acc[miss] == 0)
    rng = np.random.default_rng(0)
    op = O.make_params(W, H, spp, max_depth=depth, seed=77, trig=1)
    for r in np.sort(rng.choice(H, 6, replace=False)):
        row = O.render_window(oracle_scene, camera, op, int(r) * W, (int(r) + 1) * W)
        assert np.array_equal(bits(acc[r]), bits(row)), "row %d differs" % r
    again = gpu_ctx.render(camera, p)["accum"]
    assert np.array_equal(bits(acc), bits(again))


# ------------------------------------------------------------------ interval stepping corner cases on the device
def test_slow_nodes_and_infinite_planes_bit_exact(gpu_ctx):
    """Nodes whose +-0.001 planes leave their clipped box (literal six-slab path inside desc_step) and a tree with infinite
    planes (every ray on the literal path): same hits as the oracle, with the culling on and off."""
    from test_emu_parity import _big_overlapping_triangles
    v9, mi, mats = _big_overlapping_triangles(3000, 17)
    osc, hs = build_pair(v9, mi, mats)
    gpu_ctx.upload(hs)
    org, dirs = random_rays(200_000, 23, lo=-3, hi=3)
    o2, d2 = adversarial_rays(v9, seed=3, n_each=128)
    org = np.concatenate([org, o2]); dirs = np.concatenate([dirs, d2])
    want = osc.intersect_batch(org, dirs, counters=True)
    assert_same_hits(gpu_ctx.intersect_batch(org, dirs), want, "slow nodes")
    with no_leaf_cull(gpu_ctx):
        got = gpu_ctx.intersect_batch(org, dirs, want_stats=True)
    assert_same_hits(got, want, "slow nodes, no culling")
    assert got[3]["branch_visits"] == int(want[3][0]) and got[3]["tri_tests"] == int(want[3][3])
    out = gpu_ctx.render(default_cam(), pysqt.make_params(96, 64, 6, max_depth=6, seed=2))
    ref = osc.render(default_cam(), O.make_params(96, 64, 6, max_depth=6, seed=2, trig=1))
    assert np.array_equal(bits(out["accum"]), bits(ref["accum"]))
    v9, mi, mats = scenes.cornell_box(600)
    v9 = v9.copy(); v9[5, 0] = np.inf; v9[17, 4] = -np.inf
    osc, hs = build_pair(v9, mi, mats)
    gpu_ctx.upload(hs)
    org, dirs = random_rays(100_000, 29, lo=-2.5, hi=2.5)
    assert_same_hits(gpu_ctx.intersect_batch(org, dirs), osc.intersect_batch(org, dirs), "infinite planes")


def test_child_slabs_around_the_tame_boundary_bit_exact(gpu_ctx):
    """The device side of tests/test_emu_parity.py::test_child_slabs_are_exact_around_the_tame_boundary: a height-field mesh with
    thousands of usable child slabs; rays that switch between using and ignoring them (|d|_1 around 2, origin around twice the
    root's half extent), grazing rays, direction lengths over six decades.  Same hits as the oracle through `k_intersect_batch`
    and -- the pool kernel -- an image equal to the oracle's; with the culling off the visit counters equal the oracle's."""
    from common import tame_boundary_rays
    v9, mi, mats = scenes.subdivided_mesh(20000)
    osc, hs = build_pair(v9, mi, mats)
    gpu_ctx.upload(hs)
    org, dirs = tame_boundary_rays(v9, 60_000)
    want = osc.intersect_batch(org, dirs, counters=True)
    got = gpu_ctx.intersect_batch(org, dirs, want_stats=True)
    assert_same_hits(got, want, "child slabs on")
    with no_leaf_cull(gpu_ctx):
        off = gpu_ctx.intersect_batch(org, dirs, want_stats=True)
    assert_same_hits(off, want, "culling off")
    assert off[3]["branch_visits"] == int(want[3][0]) and off[3]["tri_tests"] == int(want[3][3])
    assert got[3]["branch_visits"] < 0.75 * off[3]["branch_visits"]
    p = dict(max_depth=6, seed=9)
    out = gpu_ctx.render(default_cam(), pysqt.make_params(128, 96, 8, **p))
    ref = osc.render(default_cam(), O.make_params(128, 96, 8, trig=1, **p))
    assert np.array_equal(bits(out["accum"]), bits(ref["accum"])) and np.array_equal(out["rgb8"], ref["rgb8"])
    assert (ref["accum"].reshape(-1, 3) != 0).any(1).sum() > 500, "the frame is meant to show the mesh"


def test_culling_and_scheduler_fuzz_on_random_scenes(gpu_ctx):
    """Random scenes of the kinds of tests/fuzz_slabs.py with random materials, on the device: `k_intersect_batch` on aimed,
    tame-boundary and adversarial rays, and a small frame through `k_primary` + `k_paths_pool` (queues, flattened leaf phase,
    filter, child slabs) -- hits, accumulation buffer and RGB8 equal the oracle's bit for bit."""
    import fuzz_slabs
    from common import tame_boundary_rays
    rng = np.random.default_rng(31337)
    fuzz_slabs.rng = rng
    cam = default_cam()
    lit = 0
    for case in range(8):
        kind = case % 5
        n = int(rng.choice([300, 3000, 12000]))
        v9, mi, mats = fuzz_slabs.rand_scene(kind, n)
        if case < 5:                                         # keep the generator's own scale for the ray tests
            osc, hs = build_pair(v9, mi, mats)
            gpu_ctx.upload(hs)
            pts = v9.reshape(-1, 3); lo, hi = pts.min(0), pts.max(0); c = 0.5 * (lo + hi); h = 0.5 * (hi - lo) + 1e-6
            m = 40_000
            org = (c + rng.uniform(-2.2, 2.2, (m, 3)) * h).astype(np.float32)
            tgt = pts[rng.integers(0, len(pts), m)] + rng.normal(size=(m, 3)) * h * 0.01
            d = tgt - org; d /= np.linalg.norm(d, axis=1, keepdims=True) + 1e-30
            d = (d * rng.choice([1.0, 1.0, 0.5, 1.15], (m, 1))).astype(np.float32)
            o2, d2 = tame_boundary_rays(v9, 4000, seed=case)
            o3, d3 = adversarial_rays(v9, seed=case, n_each=64)
            O_ = np.concatenate([org, o2, o3]); D_ = np.concatenate([d, d2, d3])
            assert_same_hits(gpu_ctx.intersect_batch(O_, D_), osc.intersect_batch(O_, D_), "fuzz scene %d (kind %d)" % (case, kind))
        v9 = (v9.reshape(-1, 3) * np.float32(1.5 / max(1e-6, float(np.abs(v9).max())))).reshape(n, 9)     # into the camera's view
        nm = 6
        mats = np.zeros((nm, 8), np.float32)
        mats[:, 0] = rng.choice([0.0, 0.3, 1.0], nm); mats[:, 1:4] = rng.uniform(0, 1, (nm, 3))
        mats[:, 4] = rng.choice([0.0, 0.0, 2.0, 10.0], nm); mats[:, 5:8] = rng.uniform(0, 1, (nm, 3))
        mats[0, 4] = 5.0
        mi = rng.integers(0, nm, n).astype(np.int32)
        osc, hs = build_pair(v9, mi, mats)
        gpu_ctx.upload(hs)
        depth = int(rng.choice([3, 8])); spp = int(rng.choice([4, 9]))
        seed = int(rng.integers(1000))
        out = gpu_ctx.render(cam, pysqt.make_params(160, 120, spp, max_depth=depth, seed=seed))
        ref = osc.render(cam, O.make_params(160, 120, spp, max_depth=depth, seed=seed, trig=1))
        assert np.array_equal(bits(out["accum"]), bits(ref["accum"])) and np.array_equal(out["rgb8"], ref["rgb8"]), "fuzz frame %d" % case
        lit += int((ref["accum"] != 0).any())
    assert lit >= 4, "most frames are meant to show lit geometry"


def default_cam():
    return pysqt.load_camera(pysqt.ROOT + "/data/camera")


# ------------------------------------------------------------------ BASELINE.json configs 3, 4, 5 at their full size
def _full_size_checks(ctx, hs, osc, cam, cfg, n_pixels, seed=0):
    """Size-independent checks in the style of test_baseline_config2_at_full_size: exact sample accounting, pixels whose
    primary ray misses are exactly black, `n_pixels` hit pixels re-rendered by the oracle with ALL their samples match bit
    for bit (so every accumulation round adds in sample order), RGB8 = the oracle's tone map of the device's sums."""
    W, H, spp, depth = cfg["width"], cfg["height"], cfg["spp"], cfg["depth"]
    ctx.upload(hs)
    out = ctx.render(cam, pysqt.make_params(W, H, spp, max_depth=depth, seed=seed))
    acc, st = out["accum"], out["stats"]
    assert st["samples"] == W * H * spp
    org, dirs = O.make_rays(O.make_params(W, H, 1), cam)
    tri = ctx.intersect_batch(org, dirs)[0]
    miss = (tri < 0).reshape(H, W)
    assert np.all(acc[miss] == 0)
    op = O.make_params(W, H, spp, max_depth=depth, seed=seed, trig=1)
    rng = np.random.default_rng(5)
    hit_pixels = np.flatnonzero(~miss.ravel())
    assert len(hit_pixels) > 1000
    for pix in rng.choice(hit_pixels, n_pixels, replace=False):
        want = O.render_window(osc, cam, op, int(pix), int(pix) + 1)
        assert np.array_equal(bits(acc.reshape(-1, 3)[pix]), bits(want[0])), "pixel %d" % pix
    assert np.array_equal(out["rgb8"], O.tone_map(acc, spp, trig=1))
    return st


def test_baseline_config3_at_full_size(gpu_ctx, camera):
    """BASELINE.json configs[2]: synthetic Cornell box (~10 k triangles, one emissive quad, mixed reflective walls) at
    1920x1080, 4096 spp, 8 bounces: 8.5e9 samples."""
    cfg = scenes.CONFIGS[2]
    osc, hs = build_pair(*scenes.config_arrays(cfg))
    st = _full_size_checks(gpu_ctx, hs, osc, camera, cfg, n_pixels=10)
    assert st["rays_traced"] > 1.5 * st["samples"]


def test_baseline_config4_at_full_size(gpu_ctx, camera):
    """BASELINE.json configs[3]: synthetic 1 M-triangle mesh (height-19 BIH, traversal bound) at 3840x2160, 256 spp."""
    cfg = scenes.CONFIGS[3]
    osc, hs = build_pair(*scenes.config_arrays(cfg))
    assert hs.n_tris > 990_000 and hs.stats()["height"] >= 18
    _full_size_checks(gpu_ctx, hs, osc, camera, cfg, n_pixels=16)


def test_baseline_config5_at_full_size(gpu_ctx, camera):
    """BASELINE.json configs[4]: 10 M-triangle soup, every material fully reflective, 16 bounces, 3840x2160, 64 spp --
    the incoherent-ray stress (480 MB of triangles; paths really bounce: more than 10 rays per sample)."""
    cfg = scenes.CONFIGS[4]
    osc, hs = build_pair(*scenes.config_arrays(cfg))
    assert hs.n_tris == 10_000_000
    st = _full_size_checks(gpu_ctx, hs, osc, camera, cfg, n_pixels=12)
    assert st["rays_traced"] > 10 * st["samples"]
    up = gpu_ctx.last_upload()
    assert up["h2d_bytes"] > 480e6


def test_ten_thousand_spheres_through_the_hierarchy(host_scene, camera):
    """Extension: 10 k analytic spheres.  The device finds a ray's candidate spheres through a bounding-volume hierarchy
    (sphere_step) instead of testing all of them; hits and the rendered frame must equal the oracle's literal definition
    (closest of [BIH hit, sphere 0, ..], earliest on ties) bit for bit, with and without the hierarchy -- on a room packed
    with overlapping spheres of every size (radii 0.003 .. 0.25) and on a cloud of small ones (0.004 .. 0.03).  Throughput:
    the cloud must render at no less than a third of the rays per second of the scene without spheres (measured 392 vs 1030
    Mrays/s, DESIGN.md: every ray pays one dependent walk down a hierarchy that does not fit L1) and far above the literal
    loop (measured 3 Mrays/s)."""
    from test_emu_parity import many_spheres
    dense, cloud = many_spheres(10_000, 5), many_spheres(10_000, 6, log_r=(-2.4, -1.5))
    osc = O.Scene.load(pysqt.ROOT + "/data/scene.obj", pysqt.ROOT + "/data")
    osc.make_bih()
    ctx = pysqt.Context(0)
    ctx.upload(host_scene)
    p = pysqt.make_params(960, 540, 16, max_depth=8, seed=3)

    def mrays():
        ctx.render_resident(camera, p)
        st = min((ctx.render_resident(camera, p) for _ in range(3)), key=lambda s: s["device_ms"])
        return st["rays_traced"] / st["device_ms"] / 1e3
    r_plain = mrays()
    org, dirs = O.make_rays(O.make_params(200, 150, 1), camera)
    o2, d2 = random_rays(60000, 9)
    v9, _ = osc.tris()
    o3, d3 = adversarial_rays(v9, seed=4, n_each=64)
    org = np.concatenate([org, o2, o3]); dirs = np.concatenate([dirs, d2, d3])
    rates = {}
    for name, sph in (("dense", dense), ("cloud", cloud)):
        osc.set_spheres(sph)
        ctx.upload(host_scene); ctx.upload_spheres(sph)
        want = osc.intersect_batch(org, dirs)
        assert_same_hits(ctx.intersect_batch(org, dirs), want, "10k spheres, " + name)
        assert (want[0] >= osc.n_tris).sum() > (20000 if name == "dense" else 2000)
        rates[name] = mrays()
        ref = osc.render(camera, O.make_params(96, 64, 4, max_depth=6, seed=3, trig=1))
        out = ctx.render(camera, pysqt.make_params(96, 64, 4, max_depth=6, seed=3))
        assert np.array_equal(bits(out["accum"]), bits(ref["accum"])) and np.array_equal(out["rgb8"], ref["rgb8"])
    ctx._ck(ctx.L.sqt_set_option(ctx.h, 2, 0), "sqt_set_option")          # SQT_OPT_SPHERE_BVH off: the literal loop
    assert_same_hits(ctx.intersect_batch(org[:20000], dirs[:20000]), tuple(w[:20000] for w in want), "10k spheres, loop")
    ctx.render_resident(camera, pysqt.make_params(240, 135, 4, max_depth=8, seed=3))
    st = ctx.render_resident(camera, pysqt.make_params(240, 135, 4, max_depth=8, seed=3))
    r_loop = st["rays_traced"] / st["device_ms"] / 1e3
    ctx.close()
    print("Mrays/s: no spheres %.0f, 10k-sphere cloud %.0f, 10k dense spheres %.0f, cloud with the literal loop %.1f" % (
        r_plain, rates["cloud"], rates["dense"], r_loop))
    assert rates["cloud"] >= r_plain / 4.0 and rates["cloud"] > 10 * r_loop
