"""Worker for test_adaptive_multi_gpu.py: one rank per GPU (torchrun).  An adaptive frame over the ranks' communicator gives
rank 0, after every chunk and retire, the sums, moments, preview, sample counts, noise and active total of one GPU bit for
bit, and every rank the same active total; ranks that disagree on the tolerance fail together at retire."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path[:0] = [ROOT, os.path.join(ROOT, "squigly-trace_b200"), HERE]
import pysqt
from test_adaptive_multi_gpu import CHUNKS, _frames, _same


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
    got = _frames(grp, p)
    acts = torch.tensor([g[5] for g in got], device="cuda")
    acts0 = acts.clone()
    dist.broadcast(acts0, src=0)
    ok &= bool(torch.equal(acts, acts0))                  # every rank returns the whole frame's active total
    if rank == 0:
        solo.render_begin(cam, p)
        ok &= _same(got, _frames(solo, p))
    # ranks with different tolerances: every rank fails at retire, nothing runs, the frame goes on afterwards
    grp.render_begin(cam, p)
    grp.render_advance(4)
    try:
        grp.render_retire(0.05 + 0.01 * rank, 0.0, 2)
        ok = False
    except pysqt.SqtError:
        pass
    grp.render_retire(0.05, 0.0, 2)
    ok &= grp.render_advance(sum(CHUNKS))["samples_done"] == sum(CHUNKS)
    flag = torch.tensor([0 if ok else 1], device="cuda")
    dist.all_reduce(flag)
    dist.barrier()
    os.dup2(saved, 1)
    if rank == 0:
        print("ADAPTIVE_OK" if int(flag.item()) == 0 else "ADAPTIVE_MISMATCH", flush=True)
    grp.close(); solo.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
