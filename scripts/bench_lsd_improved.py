"""Time LSD_improved (lsd_improvement.py --alg_ver 1/2) end to end: the single-GPU flow.LSD_improved and dist.ShardedLSDImproved at
N = 1 (and at N = world under torchrun), with the driver's per-phase times (pre-processing, pass 1, mask + all-to-all, back-off,
pass 2, final mask), and the outputs of the two compared in the same run.  One JSON file with the GPU name and power limit read in
the same run.  Workloads (synthetic clips of synth.make_clip): 240x320x200 with alg_ver 2 and 1080x1920x60 with alg_ver 1.  Each
time is one call on a host clock ending in a device synchronise (max over the ranks), after a small warm-up call of both paths;
every phase boundary synchronises the device, so the phases add up to the driver's total.

    python scripts/bench_lsd_improved.py [--out profiles/r3_lsd_improved_line.json]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node <GPUs> --master-addr 127.0.0.1 --master-port 29524 \\
        scripts/bench_lsd_improved.py
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

WORKLOADS = [("qvga200", 240, 320, 200, 2), ("1080p60", 1080, 1920, 60, 1)]


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


def clip(rows, cols, frames, seed=0):
    video, _ = synth.make_clip(rows, cols, frames, seed=seed, n_rect=6)
    return np.asfortranarray(video.reshape(frames, cols, rows).transpose(2, 1, 0).astype(np.float64))


def run_driver(cube, alg_ver, comm):
    """(total seconds, phase seconds, outputs) of ShardedLSDImproved on this rank's columns"""
    h, w, t = cube.shape
    c0, c1 = bdist.shard_columns(w, comm.world, comm.rank)
    part = np.asfortranarray(cube[:, c0:c1, :])
    phases, start = {}, {}

    def hook(name, phase):
        torch.cuda.synchronize()
        if phase == 'begin':
            start[name] = time.perf_counter()
        else:
            phases[name] = time.perf_counter() - start[name]
    drv = bdist.ShardedLSDImproved(comm)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = drv.run(part, cube.shape, alg_ver, hooks=hook)
    torch.cuda.synchronize()
    return time.perf_counter() - t0, phases, out, drv


def run_flow(cube, alg_ver):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = B.LSD_improved(cube, 0, cube.shape[2] - 1, 1, alg_ver=alg_ver)
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_lsd_improved_line.json"))
    ap.add_argument("--workloads", default=",".join(w[0] for w in WORKLOADS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_lsd_improved: needs a CUDA device")
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    name, power = gpu_identity()
    out = {"gpu": name, "power_limit_and_max_sm_clock": power, "gpus": world, "workloads": []}
    for alg_ver in (2, 1):                                    # warm-up of both paths: modules, kernel attributes
        small = clip(48, 60, 8, seed=1)
        if rank == 0:
            run_flow(small.copy(order='F'), alg_ver)
            run_driver(small.copy(order='F'), alg_ver, Solo())
    for label, rows, cols, frames, alg_ver in WORKLOADS:
        if label not in args.workloads.split(","):
            continue
        cube = clip(rows, cols, frames)
        res = {"workload": label, "rows": rows, "cols": cols, "frames": frames, "alg_ver": alg_ver}
        if rank == 0:
            t_flow, ref = run_flow(cube.copy(order='F'), alg_ver)
            t1, ph1, o1, d1 = run_driver(cube.copy(order='F'), alg_ver, Solo())
            S0, mask0, L0, _i, _m, _s, it0, conv0, git0, gconv0 = ref
            S1, mask1, L1, _i1, _m1, _s1, it1, conv1, git1, gconv1 = o1
            res["flow_LSD_improved"] = {"seconds": t_flow, "pass1_iters": git0, "pass2_iters": it0, "converged": [gconv0, conv0]}
            res["driver_N1"] = {"seconds": t1, "phases_s": ph1, "pass1_iters": git1, "pass2_iters": it1, "converged": [gconv1, conv1],
                                "relF_L_vs_flow": rel(L1, L0), "relF_S_vs_flow": rel(S1, S0),
                                "mask_agreement_vs_flow": float((mask1 == mask0).mean())}
            print(json.dumps(res), file=sys.stderr, flush=True)
            del ref, o1, d1
        if world > 1:
            dist.barrier()
            tN, phN, oN, dN = run_driver(cube, alg_ver, bdist.TorchComm())
            t = torch.tensor([tN], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            res["driver_N%d" % world] = {"seconds": float(t.item()), "phases_s_rank0": phN, "pass1_iters": oN[8], "pass2_iters": oN[6]}
        out["workloads"].append(res)
    if rank == 0:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f)
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
