"""Time per decomposition of the graph modes sharded over N GPUs (dist.ShardedLSD: G_S re-sharded by frames around the prox,
bsub_step_prox_block on each rank's frames), at N = 1 and at every N in {2, 4, 8} the machine has; one JSON file with the GPU name
and power limit read in the same run.  Cases:
  * generic: (5,5) all-window graph (the generic kernel) on WaterSurface 128x160x48 (tests/golden);
  * centre_bg: radius-1 centre windows + background from an LSD_improved-style [h, w, t] weight map on a synthetic 240x320x200 clip.
At N = 1 the same clip also goes through bsub_run on the whole-clip handle (the public solver's path): the two times, iteration
counts, rank sequences and relF(S) between them.  Each time is one solve after the handle is built and D is loaded, ending in a
device synchronise on every rank (host clock, max over the ranks); a small solve of each case runs first as warm-up.
A GPU already runs the clusters of different frames concurrently, so sharding gains only where a rank's frames need more than one
wave of them; N > 1 figures not measured are written as "not measured".

    python -m torch.distributed.run --nnodes=1 --nproc-per-node <GPUs> --master-addr 127.0.0.1 --master-port 29523 \\
        scripts/bench_sharded_graph.py [--out profiles/r3_sharded_graph_line.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import background_subtraction_b200 as B  # noqa: E402
from background_subtraction_b200 import dist as bdist, synth  # noqa: E402


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


class Solo:
    world, rank = 1, 0

    def all_reduce_sum(self, t):
        pass

    def all_reduce_max(self, t):
        pass


def cases():
    cube = np.load(os.path.join(ROOT, "tests", "golden", "watersurface_u8.npz"))["ImData"]
    rows, cols, n = cube.shape
    ws = np.ascontiguousarray(cube.transpose(2, 1, 0)).reshape(n, rows * cols)
    yield ("generic", "WaterSurface", rows, cols, ws, dict(graphs=B.getGraphSPAMS_all_groups((rows, cols), (5, 5)), graph_cols=cols))
    rows, cols, n = 240, 320, 200
    video, _ = synth.make_clip(rows, cols, n, seed=0, n_rect=6, period=300)
    rng = np.random.default_rng(1)
    wm = np.where(rng.random((rows, cols, n)) < 0.1, rng.uniform(0.5, 3.0, (rows, cols, n)), 0.0)
    wm = np.where(rng.random((rows, cols, n)) > 0.5, -1.0, wm)
    yield ("centre_bg", "synthetic", rows, cols, video, dict(weight_mask=wm))


def shard_solve(D, rows, cols, kw, comm):
    """ShardedLSD over comm's ranks; (seconds of the solve, status, S of this shard, rank sequence)"""
    n = D.shape[0]
    c0, c1 = bdist.shard_columns(cols, comm.world, comm.rank)
    shard = np.ascontiguousarray(D.reshape(n, cols, rows)[:, c0:c1, :].reshape(n, rows * (c1 - c0)))
    s = bdist.CudaStepSolver(rows, c1 - c0, n, rows * cols, frames=bdist.shard_frames(n, comm.world, comm.rank), **kw)
    s.load(shard)
    drv = bdist.ShardedLSD(s, comm)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    drv.solve()
    drv.finish(2.0, want_mask=False)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return dt, s.status(), s.dec.download('S', dtype=np.float32), [l['svp'] for l in s.dec.log()]


def run_solve(D, rows, cols, kw):
    """bsub_run on the whole-clip handle the public solver builds (lsd_decomposition / center_window_decomposition)"""
    n, m = D.shape
    route = (B.api.route_weight_mask(kw["weight_mask"], m, n) if "weight_mask" in kw else
             B.api.route_graphs(kw["graphs"], m, n, (rows, cols)))
    dec = B.Decomposition(B.make_config(m, n, route.prox, route.rows, route.cols))
    dec.set_route(route)
    dec.load(D)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    dec.run()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return dt, dec.status(), dec.download('S', dtype=np.float32), [l['svp'] for l in dec.log()]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_sharded_graph_line.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sharded_graph: needs a CUDA device")
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    name, power = gpu_identity()
    groups = {N: dist.new_group(list(range(N))) for N in (2, 4, 8) if N <= world}
    out = {"gpu": name, "power_limit_and_max_sm_clock": power, "gpus_on_machine": world, "cases": []}
    for mode, clip, rows, cols, video, kw in cases():
        D = synth.preprocess_u8(video)                                            # [n][m] float32
        res = {"mode": mode, "clip": clip, "rows": rows, "cols": cols, "frames": int(D.shape[0])}
        if rank == 0:
            small = D[:8]                                                          # warm-up: modules, kernel attributes
            wkw = dict(kw, weight_mask=kw["weight_mask"][:, :, :8]) if "weight_mask" in kw else kw
            shard_solve(small, rows, cols, wkw, Solo())
            t_run, st0, S0, svp0 = run_solve(D, rows, cols, kw)
            t1, st1, S1, svp1 = shard_solve(D, rows, cols, kw, Solo())
            res["N1"] = {"bsub_run_s": t_run, "bsub_run_iters": int(st0.iter), "sharded_s": t1, "sharded_iters": int(st1.iter),
                         "same_ranks": svp0 == svp1, "ranks": svp1, "converged": bool(st1.converged),
                         "relF_S_vs_bsub_run": float(np.linalg.norm(S1 - S0) / max(np.linalg.norm(S0), 1e-30))}
            print(json.dumps(res), file=sys.stderr, flush=True)
        dist.barrier()
        for N in (2, 4, 8):
            if N > world:
                res["N%d" % N] = "not measured"
                continue
            if rank < N:
                dt, st, _S, svp = shard_solve(D, rows, cols, kw, bdist.TorchComm(groups[N]))
                t = torch.tensor([dt], dtype=torch.float64, device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MAX, group=groups[N])
                res["N%d" % N] = {"sharded_s": float(t.item()), "iters": int(st.iter), "ranks": svp, "converged": bool(st.converged)}
            dist.barrier()
        out["cases"].append(res)
    if rank == 0:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f)
        print(json.dumps(out))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
