#!/usr/bin/env python
"""bench.py -- headline benchmark of the squigly-trace B200 backend (see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload config1..config5] [--spp S] [--no-cpu-baseline] [--no-other-configs] [--dump-outputs DIR]

Default workload (BASELINE.json configs[1]): data/scene.obj + scene.sq + camera at 1920x1080, 1024 spp, max 8 bounces.
A step = one full render of that frame through the hot path.  Metric = Mrays/s, where a ray is one closest-hit
query (Lib.hs:131) ACTUALLY executed -- primary hits are traced once per pixel and reused by its samples, paths end
at surfaces with surfColor = 0; both are exact (bit-identical image), and only executed rays are counted.

  value : rays of all ranks / max-over-ranks CUDA-event time of the K timed steps (scene resident in HBM)
  e2e   : same through the host-buffer C ABI (sqt_upload_scene + sqt_render): H2D of the scene, D2H of the RGB8 frame
  roofline : FP32 (non-fused issue rate; the bit-exact path may not contract to FMA) of the dominant kernel k_paths_pool
  cpu_baseline : the oracle (C port of the reference algorithm) on the host cores, bounded sample of the same frame
  other_configs (1 GPU only): the other four BASELINE.json configs at a bounded spp, each with Mrays/s, Msamples/s,
      rays/sample, a 40 k-ray bit-exact spot check against the oracle, and a roofline on its binding resource
  intersect_batch (1 GPU only): the batched Scene.intersect entry point on 8 M incoherent rays and a 1080p pinhole fan
  frame_sha256 / per_rank : identity of rank 0's RGB8 frame and every rank's phase times (outside the timed region)

`--dump-outputs DIR` writes the frame of the last timed step as a caller of the timed path receives it (sqt_download_image):
DIR/accum.npy (per-pixel radiance sums) and DIR/rgb8.npy (the tone-mapped frame), both float32 of shape (rows, cols, 3).
When the two together would exceed 64 MB, the same seeded sample of pixels is taken from both, (n, 3) each, and its
row-major pixel indices go to DIR/pixel_index.npy (float64).  Inputs are fixed by the arguments (seeded scenes, SEED), so
two builds of the project can be compared output for output.

`--impl reference` times that oracle alone (the Haskell reference cannot be built: no GHC in the image).
Multi-GPU: launched by torchrun, one rank per GPU; pixel groups are partitioned over ranks and the accumulation
buffers summed with ncclReduce inside the library (bit-identical to 1 GPU).
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "squigly-trace_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

SEED = 0
DATA = os.path.join(ROOT, "data")
DUMP_BYTES = 64_000_000
KERNEL_VERSION = "r02-v17"         # key into profiles/r02_traffic.json (ncu DRAM bytes per k_paths_pool launch)


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0, t1):
        if not self.proc:
            return None
        time.sleep(0.25)
        self.proc.terminate()
        rows = [r for ts, r in self.rows if t0 <= ts <= t1 + 0.3 and len(r) >= 7] or [r for _, r in self.rows if len(r) >= 7]
        if not rows:
            return None
        sm = sorted(float(r[0]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][1]), "reasons": reasons, "samples": len(rows),
                "power_w_max": max(float(r[2]) for r in rows if r[2].replace(".", "").isdigit())}


def algorithmic_fp32_ops(st):
    """SURVEY 8(d), guard-aware: 3 reciprocals per ray; 24 ops per child-box test (6 sub, 6 mul, 10 min/max, 2 cmp);
    per triangle test 14 ops up to the `a` guard, +9 and the divide up to the `u` guard, +16 up to the `v` guard,
    +6 up to the `t` guard, +14 and the sqrt for an accepted hit (Geometry.hs:117-142 with edges precomputed).
    Shading (RNG, trig, bounce) is NOT counted."""
    return (3 * st["rays_traced"] + 24 * st["child_box_tests"] + 14 * st["tri_tests"] + 10 * st["mt_pass_a"]
            + 16 * st["mt_pass_u"] + 6 * st["mt_pass_v"] + 15 * st["mt_accept"])


def algorithmic_fp32_ops_upper(st):
    """SURVEY 8(d) upper bound: every triangle test charged in full (59 add/mul + div + sqrt)."""
    return 3 * st["rays_traced"] + 24 * st["child_box_tests"] + 61 * st["tri_tests"]


def _hbm_peak():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 6650.0, "fallback of B200_PROFILING.md (MEASURED_PEAKS.json absent)"


def _traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of one k_paths_pool launch, from the tracked ncu summary of THIS
    kernel version; null when the kernels changed after the last capture (never a stale constant)."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        return t.get(KERNEL_VERSION)
    except Exception:
        return None


def dump_outputs(directory, arrays):
    """arrays: name -> (rows, cols, 3) frame.  Saved as float32, whole or as one seeded pixel sample (see the module docstring)."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    out = {k: np.asarray(v, np.float32) for k, v in arrays.items()}
    npix = out["rgb8"].shape[0] * out["rgb8"].shape[1]
    per_pixel = 3 * 4 * len(out)
    if npix * per_pixel > DUMP_BYTES:
        n = (DUMP_BYTES - 4096) // (per_pixel + 8)
        idx = np.sort(np.random.default_rng(SEED).choice(npix, n, replace=False))
        out = {k: v.reshape(npix, 3)[idx] for k, v in out.items()}
        out["pixel_index"] = idx.astype(np.float64)
    for k, v in out.items():
        np.save(os.path.join(directory, k + ".npy"), v)


def workload_cfg(name):
    from pysqt import scenes
    ci = {"config1": 0, "config2": 1, "config3": 2, "config4": 3, "config5": 4}[name]
    return ci, dict(scenes.CONFIGS[ci])


def build_host_scene(cfg):
    """(HostScene, arrays or None, seconds spent generating + building the BIH on the host)"""
    import pysqt
    from pysqt import scenes
    t0 = time.time()
    arr = scenes.config_arrays(cfg)
    hs = pysqt.HostScene.load(os.path.join(DATA, "scene.obj"), DATA) if arr is None else pysqt.HostScene.from_arrays(*arr)
    return hs, arr, time.time() - t0


def build_oracle_scene(arr):
    from oracle import oracle as O
    osc = O.Scene.load(os.path.join(DATA, "scene.obj"), DATA) if arr is None else O.Scene.from_arrays(*arr)
    osc.make_bih()
    return osc


def cpu_baseline(cfg, arr, target_s=15.0):
    """Oracle (oracle/oracle.c, all host threads) on a bounded sample: the workload's full frame and depth, few spp."""
    from oracle import oracle as O
    sc = build_oracle_scene(arr)
    cam = O.load_camera(os.path.join(DATA, "camera"))
    cores = os.cpu_count() or 1
    W, H, D, lit = cfg["width"], cfg["height"], cfg["depth"], cfg["literal"]
    t0 = time.perf_counter()
    r = sc.render(cam, O.make_params(W, H, 1, max_depth=D, seed=SEED, trig=0, literal=lit), want_rgb8=False, nthreads=cores)
    t1 = time.perf_counter() - t0
    spp = int(max(1, min(64, cfg["spp"], round(target_s / max(t1, 1e-3)))))
    if spp > 1:
        t0 = time.perf_counter()
        r = sc.render(cam, O.make_params(W, H, spp, max_depth=D, seed=SEED, trig=0, literal=lit), want_rgb8=False, nthreads=cores)
        t1 = time.perf_counter() - t0
    return {"value": r["rays"] / t1 / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "port",
            "sample": "full %dx%d frame, depth %d, %d spp (%d rays, %.1f s); C port of the reference algorithm, "
                      "libm trig, no primary-hit reuse (Lib.hs:81-87)" % (W, H, D, spp, r["rays"], t1),
            "msamples_per_s": r["samples"] / t1 / 1e6, "seconds": t1, "rays": r["rays"], "spp": spp}


def run_reference(args, rank, world):
    """Reference arm: the reference's own CPU algorithm on the host cores (oracle port; GHC is not in the image)."""
    if rank != 0:
        return
    from oracle import oracle as O
    ci, cfg = workload_cfg(args.workload)
    _, arr, _ = (None, None, 0) if cfg["scene"] == "obj" else build_host_scene_arrays_only(cfg)
    sc = build_oracle_scene(arr)
    cam = O.load_camera(os.path.join(DATA, "camera"))
    cores = os.cpu_count() or 1
    W, H, D, lit = cfg["width"], cfg["height"], cfg["depth"], cfg["literal"]
    t0 = time.perf_counter()
    sc.render(cam, O.make_params(W, H, 1, max_depth=D, seed=SEED, trig=0, literal=lit), want_rgb8=False, nthreads=cores)
    probe = time.perf_counter() - t0
    budget = 150.0 / max(1, args.steps + args.warmup)            # whole run within a few minutes
    spp = int(max(1, min(64, cfg["spp"], budget / max(probe, 1e-3))))
    p = O.make_params(W, H, spp, max_depth=D, seed=SEED, trig=0, literal=lit)
    for _ in range(args.warmup):
        sc.render(cam, p, want_rgb8=True, nthreads=cores)
    rays = 0
    samples = 0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r = sc.render(cam, p, want_rgb8=True, nthreads=cores)
        rays += r["rays"]; samples += r["samples"]
    dt = time.perf_counter() - t0
    v = rays / dt / 1e6
    sample = "each step = full %dx%d frame, depth %d, %d spp (bounded sample of the %d spp job)" % (W, H, D, spp, cfg["spp"])
    print(json.dumps({
        "impl": "reference", "metric": "Mrays/s", "value": v, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": cfg["name"],
        "config": {"workload": cfg["name"], "sample": sample},
        "cpu_baseline": {"value": v, "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "msamples_per_s": samples / dt / 1e6, "gpu_launches": 0,
        "note": "C port of the reference algorithm (oracle/oracle.c), all host threads; every ray counted (the reference "
                "re-traces the primary ray of every sample); the Haskell binary cannot be built here",
    }))


def build_host_scene_arrays_only(cfg):
    from pysqt import scenes
    t0 = time.time()
    return None, scenes.config_arrays(cfg), time.time() - t0


def counted_per_ray(ctx, cam, cfg, spp_c):
    """Per-ray work of the reference algorithm (leaf culling off: equals the oracle's counters) and of what the default
    kernels execute (culling on), from instrumented renders at spp_c samples per pixel."""
    import pysqt
    pc = pysqt.make_params(cfg["width"], cfg["height"], spp_c, max_depth=cfg["depth"], seed=SEED, literal=cfg["literal"],
                           flags=pysqt.SQT_F_COUNT_WORK)
    ctx.set_leaf_cull(False)
    ref = ctx.render_resident(cam, pc)
    ctx.set_leaf_cull(True)
    exe = ctx.render_resident(cam, pc)
    return ref, exe


def roofline_block(ref, exe, rays_timed, k_ms, fp32_peak_gops, l2_peak_gbs, bound):
    """Scale the counted per-ray work to the timed ray count; fractions of the FP32 / L2 / HBM ceilings."""
    scale = rays_timed / max(1, ref["rays_traced"])
    ops_ref, ops_exe = algorithmic_fp32_ops(ref) * scale, algorithmic_fp32_ops(exe) * (rays_timed / max(1, exe["rays_traced"]))
    bytes_ref = (16 * ref["branch_visits"] + 36 * ref["tri_tests"]) * scale
    hbm, hbm_src = _hbm_peak()
    t = k_ms * 1e-3
    fp32 = {"achieved": ops_ref / t / 1e12, "peak": fp32_peak_gops / 1e3, "unit": "TFLOP/s", "frac": ops_ref / t / 1e9 / fp32_peak_gops,
            "frac_executed": ops_exe / t / 1e9 / fp32_peak_gops}
    mem_gbs = bytes_ref / t / 1e9
    per_ray = {k: ref[k] / max(1, ref["rays_traced"]) for k in ("branch_visits", "child_box_tests", "tri_tests", "mt_pass_a", "mt_pass_u", "mt_pass_v", "mt_accept")}
    per_ray_exe = {k: exe[k] / max(1, exe["rays_traced"]) for k in ("branch_visits", "tri_tests", "leaves_culled")}
    out = {"bound": bound, "kernel": "k_paths_pool", "kernel_ms": k_ms,
           "fp32": fp32, "l2": {"achieved": mem_gbs, "peak": l2_peak_gbs, "unit": "GB/s", "frac": mem_gbs / l2_peak_gbs},
           "hbm": {"achieved": mem_gbs, "peak": hbm, "unit": "GB/s", "frac": mem_gbs / hbm, "peak_source": hbm_src},
           "per_ray_reference_algorithm": per_ray, "per_ray_executed": per_ray_exe,
           "algorithmic_bytes_per_ray": bytes_ref / max(1, rays_timed), "algorithmic_fp32_ops_per_ray": ops_ref / max(1, rays_timed)}
    sel = out[{"fp32": "fp32", "l2": "l2", "hbm": "hbm"}[bound]]
    out.update({"achieved": sel["achieved"], "peak": sel["peak"], "unit": sel["unit"], "frac": sel["frac"]})
    return out


def other_config_block(ctx, cam, ci, fp32_peak, l2_peak, budget_s=8.0):
    """One of the non-headline BASELINE configs at a bounded spp on this GPU."""
    import numpy as np
    import pysqt
    from pysqt import scenes
    from oracle import oracle as O
    cfg = dict(scenes.CONFIGS[ci])
    hs, arr, t_build = build_host_scene(cfg)
    t0 = time.time(); ctx.upload(hs); t_up = time.time() - t0
    up = ctx.last_upload()
    W, H, D, lit = cfg["width"], cfg["height"], cfg["depth"], cfg["literal"]
    probe_spp = max(1, min(cfg["spp"], 2))
    st = ctx.render_resident(cam, pysqt.make_params(W, H, probe_spp, max_depth=D, seed=SEED, literal=lit))
    st = ctx.render_resident(cam, pysqt.make_params(W, H, probe_spp, max_depth=D, seed=SEED, literal=lit))
    spp = int(max(1, min(cfg["spp"], budget_s * 1e3 / max(st["device_ms"], 1e-3) * probe_spp)))
    if spp > 4:
        spp = 1 << (spp.bit_length() - 1) if spp < cfg["spp"] else cfg["spp"]
    p = pysqt.make_params(W, H, spp, max_depth=D, seed=SEED, literal=lit)
    st = ctx.render_resident(cam, p)
    rgb8, _ = ctx.download(p.rows, p.cols, want_accum=False)
    ref, exe = counted_per_ray(ctx, cam, cfg, max(1, spp // 8))
    bound = {0: "fp32", 1: "fp32", 2: "fp32", 3: "l2", 4: "hbm"}[ci]
    roof = roofline_block(ref, exe, st["rays_traced"], st["paths_ms"], fp32_peak, l2_peak, bound)
    # parity spot check: 20 k incoherent + 20 k camera rays against the oracle, bit for bit (checker use, untimed)
    osc = build_oracle_scene(arr)
    lo, hi = hs.root[:3], hs.root[3:]
    rng = np.random.default_rng(ci)
    org = rng.uniform(lo, hi, (20000, 3)).astype(np.float32); d = rng.normal(size=(20000, 3)).astype(np.float32)
    o2, d2 = O.make_rays(O.make_params(200, 100, 1), cam)
    org = np.concatenate([org, o2]); d = np.concatenate([d, d2])
    g = ctx.intersect_batch(org, d); w = osc.intersect_batch(org, d)
    exact = bool(np.array_equal(g[0], w[0]) and np.array_equal(g[1].view(np.uint32), w[1].view(np.uint32))
                 and np.array_equal(g[2].view(np.uint32), w[2].view(np.uint32)))
    return {"config": cfg["name"], "tris": hs.n_tris, "bih": hs.stats(), "scene_bytes": int(up["h2d_bytes"]), "spp_run": spp,
            "spp_config": cfg["spp"], "depth": D, "device_ms": st["device_ms"], "paths_ms": st["paths_ms"], "primary_ms": st["primary_ms"],
            "rays": st["rays_traced"], "samples": st["samples"], "mrays_per_s": st["rays_traced"] / st["device_ms"] / 1e3,
            "msamples_per_s": st["samples"] / st["device_ms"] / 1e3, "rays_per_sample": st["rays_traced"] / max(1, st["samples"]),
            "mrays_reference_equivalent_per_s": st["rays_reference"] / st["device_ms"] / 1e3,
            "host_build_s": round(t_build, 2), "upload_s": round(t_up, 3), "upload_host_layout_ms": up["host_layout_ms"],
            "parity_40k_rays_bit_exact": exact, "hit_fraction": float((g[0] >= 0).mean()),
            "frame_sha256": hashlib.sha256(rgb8.tobytes()).hexdigest(), "roofline": roof}


def intersect_batch_block(ctx):
    """The bit-exact test boundary sqt_intersect_batch as a secondary metric (data/scene.obj)."""
    import numpy as np
    import pysqt
    hs = pysqt.HostScene.load(os.path.join(DATA, "scene.obj"), DATA)
    ctx.upload(hs)
    n = 8_000_000
    rng = np.random.default_rng(1)
    org = rng.uniform(-2.5, 2.5, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    lo, hi = hs.root[:3].astype(np.float64), hs.root[3:].astype(np.float64)
    c = 0.5 * (lo + hi); eye = c + np.array([0.3, -1.0, 0.25]) * float((hi - lo).max())
    fwd = (c - eye) / np.linalg.norm(c - eye); right = np.cross(fwd, [0, 0, 1.0]); right /= np.linalg.norm(right); up = np.cross(right, fwd)
    gx, gy = np.meshgrid(np.linspace(-0.6, 0.6, 1920), np.linspace(-0.34, 0.34, 1080))
    pd = (fwd[None, :] + gx.reshape(-1, 1) * right[None, :] + gy.reshape(-1, 1) * up[None, :]).astype(np.float32)
    po = np.tile(eye.astype(np.float32), (len(pd), 1))
    out = {}
    for name, o_, d_ in (("incoherent_8M", org, d), ("pinhole_1080p", po, pd)):
        best = None
        for _ in range(3):
            tri, dist, point, st = ctx.intersect_batch(o_, d_, want_stats=True)
            best = st if best is None or st["device_ms"] < best["device_ms"] else best
        out[name] = {"rays": len(o_), "device_ms": best["device_ms"], "mrays_per_s": len(o_) / best["device_ms"] / 1e3,
                     "e2e_ms": best["device_ms"] + best["h2d_ms"] + best["d2h_ms"], "hit_fraction": float((tri >= 0).mean())}
    return out


def run_ours(args, rank, world, local_rank):
    import numpy as np
    import torch
    import pysqt

    # NCCL prints its version banner with printf on stdout when NCCL_DEBUG is set in the environment: keep fd 1
    # pointed at stderr until the one JSON line is ready.
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 backend has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    ci, cfg = workload_cfg(args.workload)
    if args.spp:
        cfg["spp"] = args.spp
    W, H, SPP, DEPTH, LIT = cfg["width"], cfg["height"], cfg["spp"], cfg["depth"], cfg["literal"]
    hs, arr, t_host = build_host_scene(cfg)
    cam = pysqt.load_camera(os.path.join(DATA, "camera"))
    ctx = pysqt.Context(local_rank)
    ctx.upload(hs)
    if world > 1:
        box = [pysqt.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        ctx.comm_init(rank, world, box[0])
    p = pysqt.make_params(W, H, SPP, max_depth=DEPTH, seed=SEED, literal=LIT)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # > 126 MB L2

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def reduce_sum(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- device-resident steps -------------------------------------------------------------
    for _ in range(args.warmup):
        ctx.render_resident(cam, p)
        flush.zero_()
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    wall0 = time.time()
    dev_ms = paths_ms = 0.0
    rays = samples = launches = rays_ref = 0
    per_step = []
    phase = {"primary_ms": 0.0, "paths_ms": 0.0, "reduce_ms": 0.0, "tonemap_ms": 0.0, "device_ms": 0.0}
    for _ in range(args.steps):
        st = ctx.render_resident(cam, p)            # CUDA events on the library's stream bracket every kernel
        dev_ms += st["device_ms"]; paths_ms += st["paths_ms"]
        rays += st["rays_traced"]; samples += st["samples"]; launches += st["kernel_launches"]; rays_ref += st["rays_reference"]
        per_step.append(st["device_ms"])
        for k in phase:
            phase[k] += st[k] / args.steps
        flush.zero_()                                # L2 flush between timed iterations (outside the events)
    barrier()
    wall1 = time.time()
    clocks = sampler.stop(wall0, wall1) if sampler else None
    T = reduce_max(dev_ms)
    total_rays = reduce_sum(rays)
    total_rays_ref = reduce_sum(rays_ref)
    total_samples = reduce_sum(samples)
    total_launches = reduce_sum(launches)
    value = total_rays / (T * 1e-3) / 1e6
    # identity of the frame and where every rank spent its time (outside the timed region)
    frame_sha = None
    if rank == 0:
        rgb8, accum = ctx.download(p.rows, p.cols, want_accum=bool(args.dump_outputs))
        frame_sha = hashlib.sha256(rgb8.tobytes()).hexdigest()
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"accum": accum, "rgb8": rgb8})
    per_rank = [dict(rank=rank, **{k: round(v, 3) for k, v in phase.items()})]
    if dist is not None:
        gathered = [None] * world
        dist.all_gather_object(gathered, per_rank[0])
        per_rank = gathered

    # ---- end to end through the host-buffer ABI ---------------------------------------------
    e_steps = max(1, min(args.steps, 8))
    ctx.upload(hs); ctx.render(cam, p, want_accum=False)
    barrier()
    e_rays = 0
    t0 = time.perf_counter()
    d2h = h2d = 0
    up_ms = 0.0
    for _ in range(e_steps):
        ctx.upload(hs)                               # H2D: nodes + triangles + materials (bytes counted by the library)
        up = ctx.last_upload()
        out = ctx.render(cam, p, want_accum=False)   # D2H: RGB8 frame on rank 0
        e_rays += out["stats"]["rays_traced"]; d2h = out["stats"]["d2h_bytes"]
        h2d = up["h2d_bytes"] + out["stats"]["h2d_bytes"]; up_ms += up["wall_ms"] / e_steps
    barrier()
    e_T = reduce_max(time.perf_counter() - t0)
    e_value = reduce_sum(e_rays) / e_T / 1e6

    # ---- roofline of the dominant kernel (k_paths_pool) ---------------------------------------
    # Numerator = the REFERENCE ALGORITHM's work for this ray set (SURVEY 8(d)): per-ray averages counted by the
    # instrumented kernels with the leaf culling off (branch visits and triangle tests then equal the oracle's counters
    # one for one, tests/test_gpu_parity.py) at 1/8 of the spp, scaled to the timed ray count.
    roof = None
    fp32_peak = ctx.fp32_peak_gops()
    l2_peak = ctx.l2_bandwidth_gbs()
    ref_cnt, exe_cnt = counted_per_ray(ctx, cam, cfg, max(1, SPP // 8))
    barrier()
    if rank == 0:
        k_ms = paths_ms / args.steps
        roof = roofline_block(ref_cnt, exe_cnt, rays / args.steps, k_ms, fp32_peak, l2_peak, "fp32")
        tr = _traffic()
        roof.update({
            "traffic": tr["dram_bytes_per_launch"] if tr else None,
            "traffic_source": (tr["source"] if tr else "no ncu capture of kernel version %s yet" % KERNEL_VERSION),
            "peak_source": "measured live: non-fused FADD/FMUL issue rate of this GPU (sqt_measure_fp32_peak); FMA contraction is "
                           "forbidden on the bit-exact path, so this is the FP32 ceiling (MEASURED_PEAKS.json has no FP32 figure)",
            "kernel_ms_note": "all k_paths_pool + k_accumulate launches of one frame (one pair per sample round)",
            "kernel_share_of_step": paths_ms / dev_ms,
            "frac_note": "frac = reference-algorithm FP32 ops (guard-aware, SURVEY 8d) / time / measured peak; frac_executed "
                         "(fp32.frac_executed) counts only the work the default kernels execute (conservative leaf culling "
                         "skips about half of the triangle tests) and is the utilisation figure",
            "frac_executed": roof["fp32"]["frac_executed"],
            "counted_at_spp": max(1, SPP // 8)})

    extra = {}
    if rank == 0 and world == 1:
        if not args.no_cpu_baseline:
            extra["cpu_baseline"] = cpu_baseline(cfg, arr)
        if not args.no_other_configs:
            blocks = []
            for oc in (0, 1, 2, 3, 4):
                if oc == ci:
                    continue
                try:
                    blocks.append(other_config_block(ctx, cam, oc, fp32_peak, l2_peak))
                except Exception as e:      # a failing side block must not cost the headline line
                    blocks.append({"config": oc + 1, "error": repr(e)})
            extra["other_configs"] = blocks
            try:
                extra["intersect_batch"] = intersect_batch_block(ctx)
            except Exception as e:
                extra["intersect_batch"] = {"error": repr(e)}

    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    if rank == 0:
        line = {
            "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": T / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "%s (%d triangles), camera data/camera" % (cfg["name"], hs.n_tris),
            "config": {"workload": cfg["name"], "width": W, "height": H, "spp": SPP, "max_depth": DEPTH,
                       "index_convention": "literal (Lib.hs:69-85)" if LIT else "corrected (rows=%d, cols=%d)" % (H, W),
                       "partition": "pixel groups of 32, round-robin over ranks", "l2_flush": "256 MiB device write between steps",
                       "kernel_version": KERNEL_VERSION},
            "msamples_per_s": total_samples / (T * 1e-3) / 1e6,
            "mrays_reference_equivalent_per_s": total_rays_ref / (T * 1e-3) / 1e6,
            "rays_per_step": total_rays / args.steps, "per_step_ms": per_step,
            "e2e": {"value": e_value, "unit": "Mrays/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": e_T / e_steps * 1e3, "steps": e_steps, "upload_ms_per_step": up_ms,
                    "bytes_source": "sqt_last_upload + sqt_stats (counted by the library)"},
            "gpu_launches": int(total_launches), "clocks": clocks, "roofline": roof,
            "frame_sha256": frame_sha, "per_rank": per_rank,
            "cpu_baseline": extra.get("cpu_baseline"),
            "wall_ms_per_step": (wall1 - wall0) / args.steps * 1e3,
        }
        for k in ("other_configs", "intersect_batch"):
            if k in extra:
                line[k] = extra[k]
        print(json.dumps(line))
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="config2", choices=["config1", "config2", "config3", "config4", "config5"])
    ap.add_argument("--spp", type=int, default=0, help="override the workload's samples per pixel (a reduced run; stated in config.spp)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frame of the last timed step to DIR as .npy files (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours (the reference arm sizes its sample by timing)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # not under torchrun: relaunch as one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus), "--master-addr",
               "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__), "--gpus", str(args.gpus), "--steps", str(args.steps),
               "--warmup", str(args.warmup), "--workload", args.workload, "--spp", str(args.spp)] \
            + (["--no-cpu-baseline"] if args.no_cpu_baseline else []) + (["--no-other-configs"] if args.no_other_configs else []) \
            + (["--dump-outputs", os.path.abspath(args.dump_outputs)] if args.dump_outputs else [])
        raise SystemExit(subprocess.call(cmd))
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
