"""Small render used under ncu: data/scene.obj at a reduced frame so that one k_paths_pool launch replays quickly.
usage: python tools/prof_render.py [W H SPP DEPTH]"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "squigly-trace_b200"))
import pysqt

W, H, SPP, DEPTH = (int(x) for x in (sys.argv[1:5] if len(sys.argv) >= 5 else (480, 270, 64, 8)))
data = os.path.join(ROOT, "data")
hs = pysqt.HostScene.load(os.path.join(data, "scene.obj"), data)
cam = pysqt.load_camera(os.path.join(data, "camera"))
ctx = pysqt.Context(0)
ctx.upload(hs)
p = pysqt.make_params(W, H, SPP, max_depth=DEPTH, seed=0, flags=int(os.environ.get("SQT_PROF_FLAGS", "0")))     # 1 = instrumented kernels
for i in range(2):
    st = ctx.render_resident(cam, p)
    print("render %dx%d %dspp depth%d: device %.2f ms paths %.2f ms primary %.3f ms rays %d -> %.1f Mrays/s" % (
        W, H, SPP, DEPTH, st["device_ms"], st["paths_ms"], st["primary_ms"], st["rays_traced"], st["rays_traced"] / st["device_ms"] / 1e3))
ctx.close()
