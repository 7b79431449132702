"""The graph modes that run their prox on whole frames (generic per-frame graphs with a background, LSD_improved-style centre windows
+ background) and the l1 RPCA, sharded over GPUs (dist.ShardedLSD: frame re-sharding around the prox, bsub_step_prox_block on each
rank's frames) against the single-GPU solve of the same clip on rank 0: same iterations and rank sequence, relF(S) <= 1e-4 on rank
0's columns.  The choreography is also covered by tests/test_dist_gloo_graph_modes.py on CPU ranks and the frame blocks by
tests/test_gpu_sharded_graph.py on one GPU.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29521 scripts/check_sharded_modes.py
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


def problems(rows, cols, frames):
    """mode -> CudaStepSolver keyword arguments; per-frame descriptions differ from frame to frame"""
    rng = np.random.default_rng(7)
    graphs, bg = [], []
    for f in range(frames):
        if f % 2:
            g = B.getGraphSPAMS_all_groups((rows, cols), (2, 5))
            g['eta_g'] = rng.uniform(0.5, 2.0, len(g['eta_g']))
        else:
            centres = np.where(rng.random((rows, cols)) < 0.15, rng.uniform(0.5, 2.0, (rows, cols)), -1.0)
            g = B.get_proximal_graph_group_centers((rows, cols), 2, centres)
        graphs.append(g)
        bg.append(rng.random(rows * cols) < 0.4)
    wm = np.where(rng.random((rows, cols, frames)) < 0.2, rng.uniform(0.5, 3.0, (rows, cols, frames)), 0.0)
    wm = np.where(rng.random((rows, cols, frames)) > 0.6, -1.0, wm)
    return {"generic_bg": dict(graphs=graphs, background_masks=bg, graph_cols=cols), "centre_bg": dict(weight_mask=wm),
            "l1": dict(l1=True)}


def solve(D, rows, cols, frames, c0, c1, comm, kw):
    cl = c1 - c0
    shard = np.ascontiguousarray(D.reshape(frames, cols, rows)[:, c0:c1, :].reshape(frames, rows * cl))
    if "l1" not in kw:
        kw = dict(kw, frames=bdist.shard_frames(frames, comm.world, comm.rank))
    s = bdist.CudaStepSolver(rows, cl, frames, rows * cols, **kw)
    s.load(shard)
    drv = bdist.ShardedLSD(s, comm)
    drv.solve()
    drv.finish(2.0, want_mask=False)
    torch.cuda.synchronize()
    return s.status(), s.dec.download('S', dtype=np.float32), [l['svp'] for l in s.dec.log()]


def main():
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    rows, cols, frames = 96, 129, 31
    video, _ = synth.make_clip(rows, cols, frames, seed=5, n_rect=3)
    D = synth.preprocess_u8(video)
    c0, c1 = bdist.shard_columns(cols, world, rank)
    ok = True
    for mode, kw in problems(rows, cols, frames).items():
        st, S, svp = solve(D, rows, cols, frames, c0, c1, bdist.TorchComm(), kw)
        if rank == 0:
            st1, S1, svp1 = solve(D, rows, cols, frames, 0, cols, Solo(), kw)
            S1 = S1.reshape(cols, rows, frames)[c0:c1].reshape(-1, frames)
            rel = float(np.linalg.norm(S - S1) / max(np.linalg.norm(S1), 1e-30))
            good = st.iter == st1.iter and svp == svp1 and rel <= 1e-4 and bool(st.converged)
            print("%s %dx%dx%d on %d ranks: iter=%d err=%.3e svp=%s | single: iter=%d err=%.3e | relF(S) on rank 0 columns %.3e %s"
                  % (mode, rows, cols, frames, world, st.iter, st.err, svp, st1.iter, st1.err, rel, "ok" if good else "FAIL"), flush=True)
            ok = ok and good
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.broadcast(flag, 0)
    dist.destroy_process_group()
    return 0 if int(flag.item()) == 1 else 1


if __name__ == "__main__":
    sys.exit(main())
