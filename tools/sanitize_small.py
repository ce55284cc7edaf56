"""Smallest end-to-end exercise of every kernel, for compute-sanitizer (one tool per gpurun call):
intersect batch, render, cast mode, spheres, tone map, multi-round accumulation, a progressive frame, the denoiser."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "squigly-trace_b200")]
import pysqt

data = os.path.join(ROOT, "data")
hs = pysqt.HostScene.load(os.path.join(data, "scene.obj"), data)
cam = pysqt.load_camera(os.path.join(data, "camera"))
rng = np.random.default_rng(0)
os.environ["SQT_SBUF_MB"] = "1"
ctx = pysqt.Context(0)
ctx.upload(hs)
org = rng.uniform(-2, 2, (5000, 3)).astype(np.float32); d = rng.normal(size=(5000, 3)).astype(np.float32)
tri, dist, pt, st = ctx.intersect_batch(org, d, want_stats=True)
out = ctx.render(cam, pysqt.make_params(96, 54, 6, max_depth=8, seed=1))
out2 = ctx.render(cam, pysqt.make_params(64, 48, 2, max_depth=3, seed=1, flags=pysqt.SQT_F_COUNT_WORK | pysqt.SQT_F_NO_PRIMARY_REUSE))
ctx.upload_spheres([(0.8, 0.5, -1.2, 0.6, 5), (0.0, 3.0, 0.5, 0.25, 2)])
out3 = ctx.render(cam, pysqt.make_params(64, 48, 2, max_depth=4, seed=1))
out4 = ctx.render(cam, pysqt.make_params(64, 48, 2, mode=1))
ctx.tone_map(np.abs(rng.normal(size=(100, 3))).astype(np.float32))
ctx.render_begin(cam, pysqt.make_params(64, 48, 6, max_depth=5, seed=1))      # progressive: k_accumulate_m2, k_frame_noise*
for n in (1, 2, 3):
    ctx.render_advance(n)
ctx.download_moments(48, 64)
ctx.denoise(3)                              # k_features, k_denoise_prep, k_denoise_level
ctx.download_features(48, 64)
print("ok", int((tri >= 0).sum()), out["stats"]["rays_traced"], out3["stats"]["rays_traced"])
ctx.close()
