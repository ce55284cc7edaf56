"""Worker for test_progressive_multi_gpu.py: one rank per GPU (torchrun).  A progressive frame over the ranks' communicator
gives, after every chunk, rank 0 the sums, second moments, preview and noise estimate of one GPU bit for bit; ranks that
disagree on the chunk fail together before anything is traced."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path[:0] = [ROOT, os.path.join(ROOT, "squigly-trace_b200"), HERE]
import pysqt

CHUNKS = (1, 4, 3, 8)


def frames(ctx, p):
    out = []
    for n in CHUNKS:
        pr = ctx.render_advance(n)
        rgb8, acc = ctx.download(p.rows, p.cols)
        out.append((acc, rgb8, ctx.download_moments(p.rows, p.cols), pr["noise"]))
    return out


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    saved = os.dup(1); os.dup2(2, 1)                      # NCCL banner off stdout
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    data = os.path.join(ROOT, "data")
    hs = pysqt.HostScene.load(os.path.join(data, "scene.obj"), data)
    cam = pysqt.load_camera(os.path.join(data, "camera"))
    p = pysqt.make_params(320, 200, sum(CHUNKS), max_depth=6, seed=4)
    solo = pysqt.Context(local); solo.upload(hs)          # no communicator: renders the whole frame alone
    grp = pysqt.Context(local); grp.upload(hs)
    box = [pysqt.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    grp.comm_init(rank, world, box[0])
    ok = True
    grp.render_begin(cam, p)
    got = frames(grp, p)
    if rank == 0:
        solo.render_begin(cam, p)
        ref = frames(solo, p)
        for (a, r8, m2, nz), (ra, rr8, rm2, rnz) in zip(got, ref):
            ok &= bool(np.array_equal(a.view(np.uint32), ra.view(np.uint32)) and np.array_equal(r8, rr8)
                       and np.array_equal(m2.view(np.uint32), rm2.view(np.uint32)) and np.float64(nz).tobytes() == np.float64(rnz).tobytes())
    else:
        ok &= all(np.isnan(g[3]) for g in got)
    # ranks asking for different chunks: every rank fails, nothing is traced, the frame can go on afterwards
    grp.render_begin(cam, p)
    try:
        grp.render_advance(2 + rank)
        ok = False
    except pysqt.SqtError:
        pass
    ok &= grp.render_advance(sum(CHUNKS))["samples_done"] == sum(CHUNKS)
    flag = torch.tensor([0 if ok else 1], device="cuda")
    dist.all_reduce(flag)
    dist.barrier()
    os.dup2(saved, 1)
    if rank == 0:
        print("PROGRESSIVE_OK" if int(flag.item()) == 0 else "PROGRESSIVE_MISMATCH", flush=True)
    grp.close(); solo.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
