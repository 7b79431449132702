"""Cost of the generic graph prox (csrc/prox_graph.cu): one JSON line with the GPU name and power limit, and per clip
  * prox_ms: one prox(G, lambda/mu0, graph) call at the first ALM iteration's threshold (the most sweeps), (5,5) windows, median of
    `--reps` calls after one warm-up; includes the host-side colouring and upload of the graph (done once per call);
  * solve_ms: one whole inexact_alm_lsd with the same graph (device-resident input, ends in a device synchronise), with the
    iteration count, converged flag and the prox counters of bsub_debug_graph (sweeps of all calls, calls, calls at the cap);
  * for WaterSurface also the 3x3 all-windows graph through the generic kernel against its dedicated tile kernel.
Clips: WaterSurface 128x160x48 (tests/golden) and a synthetic 240x320x200 clip.
   python scripts/bench_graph_generic.py [--reps 3] [--skip-synthetic-solve]"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import background_subtraction_b200 as B  # noqa: E402
from background_subtraction_b200 import _cabi as C, synth  # noqa: E402


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, r


def first_threshold(D):
    """lambda / mu0 of inexact_alm_lsd.py:102-114 (lambda = 1/(sqrt(max(m, n)) delta), mu0 = 12.5 / ||D||_2, delta = 10)."""
    m, n = D.shape
    return (1.0 / (np.sqrt(max(m, n)) * 10.0)) * np.linalg.norm(D, 2) / 12.5


def prox_time(fn, reps):
    fn()
    times = []
    for _ in range(reps):
        dt, (_, sw) = timed(fn)
        times.append(dt)
    return float(np.median(times)), int(sw)


def clip_case(name, video_u8, rows, cols, reps, solve):
    n = video_u8.shape[0]
    Dt = torch.from_numpy(synth.preprocess_u8(video_u8)).cuda()          # [n][m] float32
    D = Dt.t()                                                            # m x n view, the reference's layout
    Dh = D.double().cpu().numpy()
    lam = first_threshold(Dh)
    g55 = B.getGraphSPAMS_all_groups((rows, cols), (5, 5))
    res = {"clip": name, "rows": rows, "cols": cols, "frames": n, "graph": "windows 5x5", "prox_lambda": lam}
    res["prox_ms"], res["prox_sweeps"] = prox_time(lambda: B.prox(D, lam, g55, tol=1e-6, return_sweeps=True), reps)
    if solve:
        dt, dec = timed(lambda: B.lsd_decomposition(D, graphs=g55, graph_tol=1e-6, graph_max_sweeps=20000))
        st = dec.status()
        cnt = (ctypes.c_int64 * 4)()
        C.check(dec.lib.bsub_debug_graph(dec.h, cnt))
        res.update(solve_ms=dt, iters=int(st.iter), converged=bool(st.converged), ranks=[l['svp'] for l in dec.log()],
                   prox_sweeps_total=int(cnt[1]), prox_calls=int(cnt[2]), prox_calls_at_cap=int(cnt[3]))
        dec.close()
    else:
        res["solve_ms"] = "not measured"
    return res, D, lam


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--skip-synthetic-solve", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_graph_generic: needs a CUDA device")
    name, power = gpu_identity()
    out = {"gpu": name, "power_limit_and_max_sm_clock": power, "cases": []}
    cube = np.load(os.path.join(ROOT, "tests", "golden", "watersurface_u8.npz"))["ImData"]
    rows, cols, n = cube.shape
    ws, D, lam = clip_case("WaterSurface", np.ascontiguousarray(cube.transpose(2, 1, 0)).reshape(n, rows * cols), rows, cols,
                           args.reps, True)
    g33 = B.getGraphSPAMS_all_groups((rows, cols), (3, 3))
    ws["windows3x3_tile_kernel_ms"], ws["windows3x3_tile_outer_iters"] = prox_time(
        lambda: B.prox(D, lam, g33, tol=1e-6, return_sweeps=True), args.reps)
    ws["windows3x3_generic_kernel_ms"], ws["windows3x3_generic_sweeps"] = prox_time(
        lambda: B.api._prox_generic(D, lam, g33, tol=1e-6, return_sweeps=True), args.reps)
    a = B.prox(D, lam, g33, tol=1e-6)
    b = B.api._prox_generic(D, lam, g33, tol=1e-6)
    ws["windows3x3_max_abs_diff"] = float((a - b).abs().max())
    out["cases"].append(ws)
    print(json.dumps(ws), file=sys.stderr, flush=True)
    video, _ = synth.make_clip(240, 320, 200, seed=0, n_rect=6, period=300)
    syn, _, _ = clip_case("synthetic", video, 240, 320, args.reps, not args.skip_synthetic_solve)
    out["cases"].append(syn)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
