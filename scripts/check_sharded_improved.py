"""LSD_improved over GPUs (dist.ShardedLSDImproved: pass 1 on column shards, morphology / merge / back-off on whole frames after one
all-to-all of the mask, pass 2 on the frame-range description of each rank's weight map) against the single-GPU flow.LSD_improved on
rank 0's whole clip, for alg_ver 2 and 1.  Against flow.LSD_improved: the iteration counts and convergence of both passes, relF(L)
and relF(S) and the mask agreement on rank 0's columns.  flow.LSD_improved returns neither its weight map nor its rank sequences, so
those are compared against the same driver at world size 1 on rank 0 (tests/test_gpu_lsd_improved.py shows that the world-1 driver
gives flow.LSD_improved's weight map and rank sequences): the agreement of the stitched weight map and both passes' ranks.  Exits
non-zero unless iterations and ranks are equal, the weight-map agreement is >= 0.9999 and relF <= 1e-4.  The choreography is also
covered by tests/test_dist_gloo_lsd_improved.py on CPU ranks.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29523 scripts/check_sharded_improved.py
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import background_subtraction_b200 as B  # noqa: E402
from background_subtraction_b200 import dist as bdist, synth  # noqa: E402


class Solo:
    world, rank = 1, 0

    def all_reduce_sum(self, t):
        pass

    def all_reduce_max(self, t):
        pass


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def main():
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    rows, cols, frames = 100, 131, 37
    video, _ = synth.make_clip(rows, cols, frames, seed=9, n_rect=5)
    cube = np.asfortranarray(video.reshape(frames, cols, rows).transpose(2, 1, 0).astype(np.float64))
    c0, c1 = bdist.shard_columns(cols, world, rank)
    ok = True
    for alg_ver in (2, 1):
        drv = bdist.ShardedLSDImproved(bdist.TorchComm())
        S, mask, L, _im, _mean, _shp, it, conv, git, gconv = drv.run(np.asfortranarray(cube[:, c0:c1, :]), cube.shape, alg_ver)
        torch.cuda.synchronize()
        parts = [None] * world
        dist.all_gather_object(parts, drv.weight_frames.cpu().numpy())
        if rank == 0:
            S0, mask0, L0, _i0, _m0, _s0, it0, conv0, git0, gconv0 = B.LSD_improved(cube.copy(order='F'), 0, frames - 1, 1, alg_ver=alg_ver)
            one = bdist.ShardedLSDImproved(Solo())                 # world 1: the rank sequences and the weight map of the same clip
            one.run(cube.copy(order='F'), cube.shape, alg_ver)
            wf = np.concatenate(parts, axis=0)
            agree = float((wf == one.weight_frames.cpu().numpy()).mean())
            rl = rel(L, L0[:, c0:c1, :])
            rs = rel(S, S0.reshape(rows, cols, frames, order='F')[:, c0:c1, :].reshape(-1, frames, order='F'))
            same = (it, conv, git, gconv) == (it0, conv0, git0, gconv0) and drv.pass1_log == one.pass1_log and drv.pass2_log == one.pass2_log
            good = same and agree >= 0.9999 and rl <= 1e-4 and rs <= 1e-4
            print("alg_ver %d %dx%dx%d on %d ranks: pass 1 iter=%d ranks=%s | pass 2 iter=%d ranks=%s | flow.LSD_improved: pass 1 "
                  "iter=%d, pass 2 iter=%d | iterations vs flow.LSD_improved, ranks vs the world-1 driver: %s | weight map agreement "
                  "vs the world-1 driver %.6f | vs flow.LSD_improved on rank 0 columns: relF(L) %.3e relF(S) %.3e mask agreement %.6f %s"
                  % (alg_ver, rows, cols, frames, world, git, drv.pass1_log[2], it, drv.pass2_log[2], git0, it0,
                     "equal" if same else "DIFFER", agree, rl, rs, float((mask == mask0[:, c0:c1, :]).mean()), "ok" if good else "FAIL"),
                  flush=True)
            ok = ok and good
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.broadcast(flag, 0)
    dist.destroy_process_group()
    return 0 if int(flag.item()) == 1 else 1


if __name__ == "__main__":
    sys.exit(main())
