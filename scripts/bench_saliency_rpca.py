"""Cost of the stage-2 saliency RPCA (executeSaliencyRPCA, csrc/rpca_batch.cu) on device-resident synthetic clips.  One JSON line
with the GPU name and power limit and, per clip (h x w x t):
  * total_ms: one executeSaliencyRPCA call (both stacks), median over --reps after one warm-up call at that shape;
  * per stack (X-T: w slices of h x t, Y-T: h slices of w x t): ms and slices/s of the stack's compute_RPCA batch (median over --reps),
    min / median / max of the iteration counts, slices that hit the iteration cap, the kernel that serves the shape, and
    bytes_per_s_lower_bound = sum(iters) * 28 B * rows * cols / time.  28 B per element and iteration is the traffic of one power
    sweep (D, S, Q read) plus the shrink pass (D, Q read; S, Q written) of the global-memory kernel; every extra power sweep adds 12 B,
    and the first iteration and the ||D||_2 estimate are not counted, so the real traffic is higher.  For the shared-memory kernel the
    figure is the same count over time, not traffic to HBM or L2.
Times come from CUDA events around calls that end in a device synchronise.  A clip that raises is recorded with its error.
Clips: 240x320x289 (the reference's default clip, shared-memory kernel), 240x320x862 (the reference clip at full length),
480x640x300 and 1080x1920x300 (global-memory kernel).
   python scripts/bench_saliency_rpca.py [--reps 3] [--clips 240x320x289,...] [--root DIR]
--root imports the package from another checkout (to time two versions with the same script)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLIPS = "240x320x289,240x320x862,480x640x300,1080x1920x300"


def gpu_identity():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


def fits_shared_memory(rows, cols):
    """A copy of the launcher's routing rule (bsub_rpca_rank1_batch_dev in csrc/rpca_batch.cu, which names this copy): the
    shared-memory kernel when a cluster of <= 8 CTAs holds the slice.  Only labels the rows; keep it in step with the C loop."""
    if cols > 640:
        return False
    for c in (1, 2, 4, 8):
        r = -(-rows // c)
        width = cols + 4
        if 4 * (4 * r * cols + 2 * cols + r + 8 * cols + width + 2 * c * width + 24) <= 220 * 1024:
            return True
    return False


def event_ms(torch, fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    r = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), r


def clip_case(torch, B, flow, synth, h, w, t, reps):
    res = {"clip": "%dx%dx%d" % (h, w, t)}
    video, _ = synth.make_clip(h, w, t, seed=5, n_rect=6)
    v = torch.from_numpy(video.reshape(t, w, h).transpose(0, 2, 1).astype(np.float32)).cuda()     # [t, h, w], 0..255
    try:
        B.executeSaliencyRPCA(v, 1)                                                                  # warm-up at this shape
    except Exception as e:                                                                           # noqa: BLE001
        res["error"] = str(e)
        return res
    res["total_ms"] = float(np.median([event_ms(torch, lambda: B.executeSaliencyRPCA(v, 1))[0] for _ in range(reps)]))
    for tag, stack in (("xt", v.permute(2, 1, 0).contiguous()), ("yt", v.permute(1, 2, 0).contiguous())):
        n, rows, cols = (int(s) for s in stack.shape)
        tol_l1 = rows * cols * 1e-4

        def run():
            return flow.inexact_alm_rpca_batch(stack, delta=1.0, tol_l1=tol_l1, max_iter=500, return_info=True)
        times, info = [], None
        for _ in range(reps):
            dt, (_L, _S, info) = event_ms(torch, run)
            times.append(dt)
        ms = float(np.median(times))
        its = np.abs(info["iters"].astype(np.int64))
        res[tag] = {"slices": n, "rows": rows, "cols": cols, "kernel": "shared" if fits_shared_memory(rows, cols) else "global",
                    "ms": ms, "slices_per_s": n / (ms * 1e-3), "iters_min": int(its.min()), "iters_median": float(np.median(its)),
                    "iters_max": int(its.max()), "not_converged": int(np.sum(info["iters"] < 0)),
                    "bytes_per_s_lower_bound": float(its.sum()) * 28.0 * rows * cols / (ms * 1e-3)}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--clips", default=CLIPS)
    ap.add_argument("--root", default=ROOT)
    args = ap.parse_args()
    if args.reps < 1:
        ap.error("--reps must be >= 1")
    sys.path.insert(0, os.path.abspath(args.root))
    import torch
    import background_subtraction_b200 as B
    from background_subtraction_b200 import flow, synth
    if not torch.cuda.is_available():
        raise SystemExit("bench_saliency_rpca: needs a CUDA device")
    name, power = gpu_identity()
    out = {"gpu": name, "power_limit_and_max_sm_clock": power, "root": os.path.abspath(args.root), "reps": args.reps, "clips": []}
    for spec in args.clips.split(","):
        h, w, t = (int(s) for s in spec.split("x"))
        out["clips"].append(clip_case(torch, B, flow, synth, h, w, t, args.reps))
        print(json.dumps(out["clips"][-1]), file=sys.stderr, flush=True)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
