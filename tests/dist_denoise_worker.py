"""Worker for test_denoise_multi_gpu.py: one rank per GPU (torchrun).  Rank 0 of a group frame gets, after every chunk (and
after a retire), the denoised mean and RGB8 and the features of one GPU bit for bit; ranks that disagree on the levels
fail together and the frame goes on."""
import os
import sys

import torch
import torch.distributed as dist

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path[:0] = [ROOT, os.path.join(ROOT, "squigly-trace_b200"), HERE]
import pysqt
from test_denoise_multi_gpu import CHUNKS, _begin_with_two, _frames, _same, _setup


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    saved = os.dup(1); os.dup2(2, 1)                      # NCCL banner off stdout
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    hs, cam, p = _setup()
    solo = pysqt.Context(local); solo.upload(hs)          # no communicator: renders the whole frame alone
    grp = pysqt.Context(local); grp.upload(hs)
    box = [pysqt.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    grp.comm_init(rank, world, box[0])
    ok = True
    _begin_with_two(grp, cam, p)
    got = _frames(grp, p)
    if rank == 0:
        _begin_with_two(solo, cam, p)
        ok &= _same(got, _frames(solo, p))
    # ranks with different levels: every rank fails, nothing runs, the frame goes on afterwards
    _begin_with_two(grp, cam, p)
    try:
        grp.denoise(2 + rank)
        ok = False
    except pysqt.SqtError:
        pass
    grp.denoise(2)
    ok &= grp.render_advance(sum(CHUNKS))["samples_done"] == sum(CHUNKS)
    flag = torch.tensor([0 if ok else 1], device="cuda")
    dist.all_reduce(flag)
    dist.barrier()
    os.dup2(saved, 1)
    if rank == 0:
        print("DENOISE_OK" if int(flag.item()) == 0 else "DENOISE_MISMATCH", flush=True)
    grp.close(); solo.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
