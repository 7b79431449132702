#!/usr/bin/env python
"""bench.py -- headline benchmark: frames/s decomposed, synthetic 1920x1080 x 300 frames, flat-3x3 LSD (BASELINE.json).

  python bench.py --gpus 1 --steps K --warmup W                  # this repo (CUDA, sm_100a)
  python bench.py --impl reference --gpus N --steps K --warmup W  # the reference algorithm on the host cores
  torchrun ... bench.py --gpus N ...                              # N > 1: pixel-column shards, NCCL Gram all-reduce
  python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR # also write what the last timed step computed (dump_outputs)

A "step" is one complete decomposition of the resident clip: init norms, all ALM iterations, materialisation of L and
the foreground mask.  `value` is timed with CUDA events with D already in HBM; `e2e` is the same job through the
public host-buffer API (pinned float32 D in, L + S + mask out) with both PCIe directions inside the timed region.
One JSON line is printed by rank 0.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (rows, cols, frames, seed, rectangles)
    "synthetic_1080p_300": (1080, 1920, 300, 0, 6),
    "synthetic_4k_600": (2160, 3840, 600, 1, 12),
    "synthetic_qvga_200": (240, 320, 200, 100, 3),
    "synthetic_small": (240, 320, 48, 5, 3),
    # the reference's own clip (BASELINE.json config 1): data/WaterSurface.mat, kept as tests/golden/watersurface_u8.npz
    "watersurface": (128, 160, 48, None, None),
    # BASELINE.json configs 2 and 5 (scripts/bench_flows.py): the precomputed_main flow on the committed input/ fixture, and 64
    # independent 320x240x200 clips spread over the GPUs
    "highway_flow": (120, 160, 289, None, None),
    "batch64_qvga_200": (240, 320, 200, 100, 3),
    # the reference's default LSD() mode (overlapping 3x3 windows, spams.proximalGraph) on its own clip and at the headline size
    "watersurface_graph": (128, 160, 48, None, None),
    "synthetic_qvga_200_graph": (240, 320, 200, 100, 3),
    "synthetic_1080p_300_graph": (1080, 1920, 300, 0, 6),
    "synthetic_1080p_30_graph": (1080, 1920, 30, 0, 6),       # the first 10th of the period of that clip (the prox cost is per frame)
}
FLOW_WORKLOADS = ("highway_flow", "batch64_qvga_200")         # and every *_graph workload: scripts/bench_flows.py
DUMP_SAMPLE = 1 << 22          # --dump-outputs: entries kept per matrix (3 x 16 MB of float32, within a 64 MB budget)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="synthetic_1080p_300", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-sample-div", type=int, default=0,
                    help="CPU baseline: keep rows/div x cols/(2 div) of every frame (0 = 4: a 1/32 window of 1080p, ~20 s of CPU work)")
    ap.add_argument("--tile-rows", type=int, default=0)
    ap.add_argument("--cluster-frames", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write L, S and the mask of the last timed step to DIR/<name>.npy (a fixed seeded sample of "
                         "%d entries each, plus float64 per-frame sums), so that two builds can be compared output for output "
                         "(one GPU, --impl b200; not the *_graph, highway_flow and batch64_qvga_200 workloads)" % DUMP_SAMPLE)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._pump, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2])); power.append(float(p[3]))
            except ValueError:
                continue
            for nm, v in zip(names, p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        # "under load" = samples in the upper half of the power range seen
        thr = 0.5 * (min(power) + max(power))
        load = [s for s, pw in zip(sm, power) if pw >= thr] or sm
        return {"sm_mhz": float(np.median(load)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "power_w_max": float(max(power)), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------------------------
def cpu_port_solve(D64, rows, cols, threads, keep=False):
    """The oracle port of inexact_alm_lsd (flat 3x3) + foreground_mask on the host cores (float64, NumPy/LAPACK +
    the OpenMP C prox) -- test/bench infrastructure, not the product.  The thread count is set explicitly: torchrun exports
    OMP_NUM_THREADS=1, which would otherwise halve the N > 1 reference arm (VERDICT r1)."""
    from oracle import alm_oracle as O
    os.environ["OMP_NUM_THREADS"] = str(threads)
    groups = O.flat_groups_nonoverlap((rows, cols), (3, 3))
    try:
        from threadpoolctl import threadpool_limits
        ctx = threadpool_limits(limits=threads)
    except Exception:                                       # pragma: no cover
        import contextlib
        ctx = contextlib.nullcontext()
    with ctx:
        t0 = time.perf_counter()
        L, S, it, conv = O.inexact_alm_lsd(D64, groups=groups)
        mask = O.foreground_mask(D64, L, S)
        dt = time.perf_counter() - t0
    return (dt, it, conv, L, S, mask) if keep else (dt, it, conv)


def cpu_sample(video_u8, rows, cols, frames, div):
    """Bounded sample of the same workload: a (rows/div) x (cols/(2 div)) window of every frame (all reference costs are
    linear in the pixel count -- SURVEY 8d); rows a multiple of 12 and cols of 3, so that the 3x3 tiling is unchanged and the
    same window also runs through the CUDA fast path for the parity figures."""
    if div <= 1:
        r, c = rows, cols
    else:
        r = max(12, (rows // div) // 12 * 12)
        c = max(3, (cols // (2 * div)) // 3 * 3)
    cube = video_u8.reshape(frames, cols, rows)[:, :c, :r]                 # [n][col][row]
    x = cube.astype(np.float64)
    lo, hi = float(video_u8.min()), float(video_u8.max())
    x = (x - lo) / (hi - lo)
    x -= x.mean()
    D = np.asfortranarray(x.reshape(frames, c * r).T)                       # m x n, F-order
    return D, r, c


def load_video(workload):
    """uint8 clip [frames][m], frame-major with the reference's pixel order p = j*rows + i."""
    rows, cols, frames, seed, nrect = WORKLOADS[workload]
    if workload.startswith("watersurface"):
        cube = np.load(os.path.join(ROOT, "tests", "golden", "watersurface_u8.npz"))["ImData"]       # [rows, cols, frames]
        return np.ascontiguousarray(cube.transpose(2, 1, 0)).reshape(frames, rows * cols)
    from background_subtraction_b200 import synth
    return synth.make_clip(rows, cols, frames, seed=seed, n_rect=nrect)[0]


def dump_outputs(path, outputs):
    """--dump-outputs: `outputs` maps a name to a device matrix [frames][pixels].  Each is written as DIR/<name>.npy
    (float32): whole when it has at most DUMP_SAMPLE entries, else the entries at one seeded sample of (frame, pixel)
    positions that is the same for every output and every run.  DIR/<name>_frame_sums.npy (float64 [frames]) holds the
    per-frame sums of the whole matrix, so that a difference outside the sample shows too; they are device reductions
    whose summation order is not fixed, so compare them with a tolerance, not bit for bit."""
    import torch
    os.makedirs(path, exist_ok=True)
    n, m = next(iter(outputs.values())).shape
    idx = None
    if n * m > DUMP_SAMPLE:
        idx = torch.from_numpy(np.sort(np.random.default_rng(0).choice(n * m, size=DUMP_SAMPLE, replace=False))).cuda()
    for name, x in outputs.items():
        entries = x.reshape(-1) if idx is None else x[idx // m, idx % m]
        sums = torch.cat([x[f0:f0 + 16].to(torch.float64).sum(1) for f0 in range(0, n, 16)])
        np.save(os.path.join(path, name + ".npy"), entries.to(torch.float32).cpu().numpy())
        np.save(os.path.join(path, name + "_frame_sums.npy"), sums.cpu().numpy())


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU algorithm (oracle port; the reference itself is pure Python and is not
    present on the GPU box) on all host cores, bounded sample, same metric/config."""
    if rank != 0:
        return None
    rows, cols, frames, seed, nrect = WORKLOADS[args.workload]
    threads = os.cpu_count() or 1
    video = load_video(args.workload)
    D, r, c = cpu_sample(video, rows, cols, frames, (args.cpu_sample_div or 4) if rows * cols > 200000 else 1)
    scale = (rows * cols) / float(r * c)
    times = []
    for i in range(args.warmup + args.steps):
        dt, it, conv = cpu_port_solve(D, r, c, threads)
        if i >= args.warmup:
            times.append(dt)
    t = float(np.mean(times)) * scale
    val = frames / t
    sample = f"{r}x{c} pixel window of every frame ({r * c}/{rows * cols} of the pixels), full solve, time scaled x{scale:.1f}"
    return {"impl": "reference", "metric": "frames/s decomposed", "value": val, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "reference fixture (WaterSurface)" if args.workload == "watersurface" else "synthetic",
            "config": {"workload": args.workload, "rows": rows, "cols": cols, "frames": frames, "prox": "flat 3x3 l_inf (LSD)",
                       "delta": 10},
            "cpu_baseline": {"value": val, "unit": "frames/s", "cores": threads, "kind": "port", "sample": sample,
                             "iters": it, "converged": bool(conv)},
            "e2e": {"value": val, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


# ---------------------------------------------------------------------------------------------------------------
def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    flow = args.workload in FLOW_WORKLOADS or args.workload.endswith("_graph")
    if args.dump_outputs and (args.impl != "b200" or world > 1 or flow):
        raise SystemExit("bench.py: --dump-outputs is implemented for --impl b200 on one GPU, workloads %s"
                         % ", ".join(w for w in sorted(WORKLOADS) if w not in FLOW_WORKLOADS and not w.endswith("_graph")))
    if args.impl == "reference":
        out = run_reference(args, rank, world)
        if out is not None:
            print(json.dumps(out), flush=True)
        return 0

    import torch
    import torch.distributed as dist
    import background_subtraction_b200 as B
    from background_subtraction_b200 import synth
    from background_subtraction_b200 import dist as bdist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the CUDA path is the product; there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if flow:
        sys.path.insert(0, os.path.join(ROOT, "scripts"))
        import bench_flows
        if args.workload == "highway_flow":
            out = bench_flows.highway_flow(args, rank, world, ClockSampler)
        elif args.workload.endswith("_graph"):
            rows, cols, frames, seed, nrect = WORKLOADS[args.workload]
            out = bench_flows.graph_lsd(args, rank, world, ClockSampler, rows, cols, frames, load_video(args.workload), args.workload)
        else:
            out = bench_flows.batch_clips(args, rank, world, local_rank, ClockSampler)
        if out is not None:
            print(json.dumps(out), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return 0
    comm = bdist.TorchComm()
    rows, cols, frames, seed, nrect = WORKLOADS[args.workload]
    m = rows * cols

    # ---- data: every rank generates the same seeded clip and keeps its column shard ----
    t_gen = time.perf_counter()
    video = load_video(args.workload)
    c0, c1 = bdist.shard_columns(cols, world, rank)
    cols_local = c1 - c0
    m_local = rows * cols_local
    lo, hi = float(video.min()), float(video.max())
    mean = float(video.mean(dtype=np.float64))
    shard_u8 = np.ascontiguousarray(video.reshape(frames, cols, rows)[:, c0:c1, :].reshape(frames, m_local))
    scale = 1.0 / (hi - lo)
    mean_n = (mean - lo) * scale
    D_host = torch.empty((frames, m_local), dtype=torch.float32).pin_memory()
    Dh = D_host.numpy()
    stepf = max(1, (1 << 24) // m_local)
    for f0 in range(0, frames, stepf):
        Dh[f0:f0 + stepf] = ((shard_u8[f0:f0 + stepf].astype(np.float64) - lo) * scale - mean_n).astype(np.float32)
    t_gen = time.perf_counter() - t_gen

    solver = bdist.CudaStepSolver(rows, cols_local, frames, m, tile_rows=args.tile_rows, cluster_frames=args.cluster_frames)
    solver.load(Dh)
    torch.cuda.synchronize()
    driver = bdist.ShardedLSD(solver, comm, fence=bdist.cuda_fence)

    # ---- per-kernel timing hooks (CUDA events on the launching stream) ----
    stream = torch.cuda.current_stream()
    ev = {"gram": [], "solve": [], "project": [], "shrink": []}
    pending = {}

    def hooks(name, phase):
        e = torch.cuda.Event(enable_timing=True)
        e.record(stream)
        if phase == 'begin':
            pending[name] = e
        else:
            ev[name][-1].append((pending.pop(name), e))

    marks, mark_host = [], []

    def mark(tag):
        e = torch.cuda.Event(enable_timing=True)
        e.record(stream)
        marks.append((tag, e))
        mark_host.append((tag, time.perf_counter()))

    def one_step(timed):
        if timed:
            mark('start')
            for k in ev:
                ev[k].append([])                      # one event list per timed step
        driver.solve(hooks if timed else None)
        if timed:
            mark('solved')
            solver.finalize()
            mark('L')
        out = driver.finish(2.0, want_mask=True)
        if timed:
            mark('finished')
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    mask = None
    for _ in range(max(args.warmup, 0)):
        mask = one_step(False)         # keep the result like the timed loop does: same allocator state (two mask buffers alive)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    gc.collect()
    gc.disable()          # as timeit does: a generation-2 collection inside the host-bound finish phase costs ~20 ms of GPU idle time
    e0.record(stream)
    for _ in range(args.steps):
        mask = one_step(True)
    e1.record(stream)
    barrier()
    gc.enable()
    clocks = sampler.stop() if rank == 0 else None
    ms_total = e0.elapsed_time(e1)
    tmax = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_step = float(tmax.item()) / args.steps
    st = solver.status()
    iters = int(st.iter)
    if args.dump_outputs:                   # before the e2e leg below reloads this solver handle
        dump_outputs(args.dump_outputs, {"L": solver.dec.device_tensor('L'), "S": solver.dec.device_tensor('S'), "mask": mask})

    info = solver.dec.debug_info()

    def phase_ms(name, first=0):
        # only the `iters` real ALM iterations of every step (the host enqueues up to run_ahead extra ones, which exit at once)
        v = [a.elapsed_time(b) for step in ev[name] for a, b in step[first:iters]]
        return (float(np.mean(v)) if v else 0.0), len(v)

    # coarse breakdown of a step: solve (init + loop) vs finish (L + mask)
    seg = {}
    for (t0, e_0), (t1, e_1) in zip(marks[:-1], marks[1:]):
        if t0 != 'finished':
            seg.setdefault(t0 + '->' + t1, []).append(e_0.elapsed_time(e_1))
    breakdown = {k: float(np.mean(v)) for k, v in seg.items()}
    if os.environ.get("BSUB_BENCH_TRACE"):
        sys.stderr.write("segments per step (device ms): %s\n" % {k: [round(x, 2) for x in v] for k, v in seg.items()})
        sys.stderr.write("host ms at marks: %s\n" % [(t, round((h - mark_host[0][1]) * 1e3, 2)) for t, h in mark_host])
    use_i8 = bool(info["use_i8"])
    gram_first_ms = float(np.mean([s[0][0].elapsed_time(s[0][1]) for s in ev["gram"] if s])) if ev["gram"] else 0.0
    gram_ms, n_gram = phase_ms("gram", 1 if use_i8 else 0)      # int8 path: iteration 1 has no Gram (W_1 = c D, eigenpairs of the initialisation)
    solve_ms, n_solve = phase_ms("solve", 1 if use_i8 else 0)
    # from iteration 2 on the shrink pass is project_planes_kernel + shrink_flat_kernel (rank <= 8) when the int8 path is on
    two_kernel = bool(info.get("use_proj")) and bool(info.get("flat_stages"))
    proj_ms, n_proj = phase_ms("project", 1)
    shrink_ms, n_shrink = phase_ms("shrink", 1 if two_kernel else 0)
    shrink1_ms = float(np.mean([s[0][0].elapsed_time(s[0][1]) for s in ev["shrink"] if s])) if ev["shrink"] else 0.0
    counters = solver.dec.counters()
    # kernels launched per enqueued iteration: gram_dmma, gram_reduce, (gram_i8, gram_i8_finish), eig, (project), shrink_stream,
    # (shrink_flat, rebuild_S x2 when S is stored lazily), shrink_tma, control_post x2; per step: rowsum, Gram(D) (quantize_D + gram_i8 +
    # finish, or gram_dmma + reduce), eig, init_Y (not with the int8 path), (rebuild_S x2), lowrank, absmax/maxS, mask_stats, mask_write
    per_iter = 2 + (2 if use_i8 else 0) + 1 + (1 if info.get("use_proj") else 0) + (2 if info["use_stream"] else 1) + \
        (3 if two_kernel else 0) + 2
    gpu_launches = int(args.steps * (driver.iters_enqueued * per_iter + (10 if use_i8 else 9) + (2 if two_kernel else 0)))

    # ---- end to end through the public host-buffer API (single GPU only) ----
    # Every clip: H2D of D from pinned memory, bsub_run, D2H of L, S and the mask -- all inside the timed region.  PCIe moves
    # 8.1 GB per clip (~150 ms), about as long as the solve itself, so a serving loop keeps several clips in flight (default 4,
    # BSUB_E2E_CLIPS): one solver handle per clip, each driven by its own host thread and stream, so the copies of one clip
    # overlap the kernels of the others -- and the 8-SM eigensolve of one clip runs beside the streaming kernels of another,
    # which is why this throughput can exceed the one-clip-at-a-time `value`.  `serial_ms_per_step` is the latency of one
    # clip alone (nothing overlapped).
    e2e = None

    def measure_e2e(nwork):
        import ctypes
        from background_subtraction_b200 import _cabi as C
        decs = [solver.dec] + [bdist.CudaStepSolver(rows, cols_local, frames, m, tile_rows=args.tile_rows,
                                                    cluster_frames=args.cluster_frames, store_S_lazily=True).dec for _ in range(nwork - 1)]
        outs = [tuple(torch.empty((frames, m), dtype=dt).pin_memory() for dt in (torch.float32, torch.float32, torch.uint8))
                for _ in range(nwork)]

        tlog = []

        def e2e_clip(dec, bufs, tag=None):
            Lh, Sh, Mh = bufs
            t = [time.perf_counter()]
            dec.load(Dh)                                        # H2D from pinned memory
            t.append(time.perf_counter())
            dec.run()                                           # the C loop (bsub_run)
            t.append(time.perf_counter())
            C.check(dec.lib.bsub_download_f32(dec.h, 0, ctypes.c_void_p(Lh.data_ptr()), m, dec.stream()))
            t.append(time.perf_counter())
            C.check(dec.lib.bsub_download_f32(dec.h, 1, ctypes.c_void_p(Sh.data_ptr()), m, dec.stream()))
            t.append(time.perf_counter())
            C.check(dec.lib.bsub_mask_host(dec.h, 2.0, ctypes.c_void_p(Mh.data_ptr()), dec.stream()))
            t.append(time.perf_counter())
            if tag is not None:
                tlog.append((tag, t))

        def worker(i, nclips, errs, gate, stagger_s):
            try:
                torch.cuda.set_device(local_rank)
                with torch.cuda.stream(torch.cuda.Stream()):
                    torch.cuda.current_stream().synchronize()   # stream exists before the clock starts
                    gate.wait()
                    time.sleep(i * stagger_s)                   # inside the timed region: de-phase the handles
                    for _ in range(nclips):
                        e2e_clip(decs[i], outs[i], tag=i)
            except Exception as ex:                             # surfaced after join
                errs.append(ex)
                try:
                    gate.abort()
                except Exception:
                    pass

        for i in range(nwork):                                  # warm-up of every handle
            e2e_clip(decs[i], outs[i])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_clip(decs[0], outs[0])
        torch.cuda.synchronize()
        dt_serial = (time.perf_counter() - t0) / args.steps
        same = all(bool(torch.equal(outs[0][2], outs[i][2])) for i in range(1, nwork))   # all handles must produce the same mask
        torch.cuda.synchronize()
        nclips_each = max(2 * args.steps, 6)
        errs, gate = [], threading.Barrier(nwork + 1)
        th = [threading.Thread(target=worker, args=(i, nclips_each, errs, gate, dt_serial / nwork)) for i in range(nwork)]
        for t in th:
            t.start()
        gate.wait()
        t0 = time.perf_counter()
        for t in th:
            t.join()
        torch.cuda.synchronize()
        if errs:
            raise errs[0]
        dt = (time.perf_counter() - t0) / (nwork * nclips_each)
        if os.environ.get("BSUB_BENCH_TRACE"):
            for tag, t in sorted(tlog, key=lambda x: x[1][0]):
                sys.stderr.write("e2e worker %d: start %.1f  load %.1f run %.1f L %.1f S %.1f mask %.1f ms\n" % (
                    tag, (t[0] - t0) * 1e3, *[(b_ - a_) * 1e3 for a_, b_ in zip(t[:-1], t[1:])]))
        res = {"value": frames / dt, "unit": "frames/s", "h2d_bytes_per_step": int(4 * frames * m),
               "d2h_bytes_per_step": int(9 * frames * m), "ms_per_step": dt * 1e3, "clips_in_flight": nwork,
               "clips_timed": nwork * nclips_each, "serial_ms_per_step": dt_serial * 1e3, "serial_value": frames / dt_serial,
               "handles_agree": same,
               "what": "pinned float32 D in; float32 L, S and uint8 mask out (bsub_load_D_f32_host, bsub_run, bsub_download_f32 x2, "
                       "bsub_mask_host), %d clips in flight, one solver handle + host thread + stream each" % nwork}
        # ---- other shapes of the same public call, one clip at a time (latency figures) ----
        variants = {}
        dec0, (Lh, Sh, Mh) = decs[0], outs[0]
        u8_pinned = torch.from_numpy(shard_u8).pin_memory()
        u8_np = u8_pinned.numpy()

        def timed(fn, reps):
            fn()
            torch.cuda.synchronize()
            t_ = time.perf_counter()
            for _ in range(reps):
                fn()
            torch.cuda.synchronize()
            return (time.perf_counter() - t_) / reps

        def clip_u8_full():                                     # uint8 frames in (device-side LSD() pre-processing), L + S + mask out
            dec0.load_u8(u8_np, force=(lo, hi, mean))
            dec0.run()
            C.check(dec0.lib.bsub_download_f32(dec0.h, 0, ctypes.c_void_p(Lh.data_ptr()), m, dec0.stream()))
            C.check(dec0.lib.bsub_download_f32(dec0.h, 1, ctypes.c_void_p(Sh.data_ptr()), m, dec0.stream()))
            C.check(dec0.lib.bsub_mask_host(dec0.h, 2.0, ctypes.c_void_p(Mh.data_ptr()), dec0.stream()))

        def clip_u8_mask():                                     # uint8 frames in, foreground mask out (L, S stay on the device)
            dec0.load_u8(u8_np, force=(lo, hi, mean))
            dec0.run()
            C.check(dec0.lib.bsub_mask_host(dec0.h, 2.0, ctypes.c_void_p(Mh.data_ptr()), dec0.stream()))

        for name, fn, h2d, d2h in (("u8_in_L_S_mask_out", clip_u8_full, frames * m, 9 * frames * m),
                                   ("u8_in_mask_out", clip_u8_mask, frames * m, frames * m)):
            try:
                t_ = timed(fn, max(2, args.steps))
                variants[name] = {"ms_per_step": t_ * 1e3, "value": frames / t_, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)}
            except Exception as ex:
                variants[name] = {"error": str(ex)[:200]}
        # the reference-shaped call: inexact_alm_lsd(float64 ndarray) -> float64 L, S (pageable memory both ways) + foreground mask
        try:
            del decs[1:]
            gc.collect()
            D64 = np.asfortranarray(Dh.T.astype(np.float64)) if frames * m <= 700_000_000 else None
            if D64 is not None:
                groups_full = B.get_proximal_flat_groups_nonoverlap((rows, cols), (3, 3))

                def dropin():
                    dec_d = B.lsd_decomposition(D64, groups=groups_full, img_shape=(rows, cols))
                    L_, S_, it_, cv_ = B.api._finish(dec_d, D64, False)
                    mk_ = dec_d.mask(2)
                    dec_d.close()
                    return L_, S_, mk_
                t0_ = time.perf_counter()
                dropin()
                t_ = time.perf_counter() - t0_
                variants["dropin_f64_pageable"] = {"ms_per_step": t_ * 1e3, "value": frames / t_, "h2d_bytes_per_step": int(8 * frames * m),
                                                   "d2h_bytes_per_step": int(17 * frames * m),
                                                   "what": "inexact_alm_lsd(D float64 ndarray) -> float64 L, S + mask; one cold call incl. handle creation"}
        except Exception as ex:
            variants["dropin_f64_pageable"] = {"error": str(ex)[:200]}
        res["variants"] = variants
        return res

    if not args.no_e2e and world == 1:
        # pinned host buffers (5.6 GB per clip in flight) and one solver handle (~18.5 GB of HBM) per clip: fall back to fewer
        # clips in flight if the box cannot give that much
        tried = []
        for nw in dict.fromkeys([max(1, int(os.environ.get("BSUB_E2E_CLIPS", "4"))), 2, 1]):
            try:
                e2e = measure_e2e(nw)
                break
            except Exception as ex:
                tried.append("%d clips in flight: %s" % (nw, str(ex)[:160]))
                gc.collect()
                torch.cuda.empty_cache()
        if e2e is None:
            e2e = {"value": None, "unit": "frames/s", "h2d_bytes_per_step": None, "d2h_bytes_per_step": None,
                   "what": "e2e failed: " + "; ".join(tried)}
        elif tried:
            e2e["fell_back_after"] = tried
    elif world > 1:
        e2e = {"value": None, "unit": "frames/s", "h2d_bytes_per_step": None, "d2h_bytes_per_step": None,
               "what": "not measured for N > 1"}

    # foreground fraction over the whole frame (all shards)
    mcount = torch.tensor([float(mask.sum(dtype=torch.float64).item()), float(mask.numel())], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(mcount)
    mask_fraction = float((mcount[0] / mcount[1]).item())
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant kernel (per launch, algorithmic bytes; DESIGN.md section 5) ----
    peak, peak_src = measured_peaks()
    elems_local = float(frames) * m_local
    c3 = use_i8 and 256 < frames <= 384 and os.environ.get("BSUB_NO_GRAM_CLUSTER") is None
    gram_name = ("gram_i8_c3_kernel" if c3 else "gram_i8_kernel") if use_i8 else "gram_dmma_kernel"
    if two_kernel:
        # bytes per matrix element that the kernels are designed to move (DESIGN.md 4.4): projection reads the 4 digit bytes;
        # the single-pass kernel reads D, Y and writes Y and the 4 digit bytes of the next W, plus S when the iteration may be
        # the last one (the residual of the previous iteration within 4x of the tolerance: 2 of 19 iterations here)
        flat_b = 16.0 + 4.0 * 2 / max(iters - 1, 1)
        kern = {
            "shrink_flat_kernel": {"ms": shrink_ms, "launches": n_shrink, "alg_bytes": flat_b * elems_local, "bound": "hbm"},
            "project_planes_kernel": {"ms": proj_ms, "launches": n_proj, "alg_bytes": 4.0 * elems_local, "bound": "hbm"},
        }
        shrink_pass_ms = shrink_ms + proj_ms
    else:
        shrink_name = "shrink_stream_kernel" if info["use_stream"] else ("shrink_tma_kernel" if info["use_tma"] else "shrink_kernel")
        kern = {shrink_name: {"ms": shrink_ms, "launches": n_shrink, "alg_bytes": (24.0 if use_i8 else 20.0) * elems_local, "bound": "hbm"}}
        shrink_pass_ms = shrink_ms
    kern[gram_name] = {"ms": gram_ms, "launches": n_gram, "alg_bytes": (4.0 if use_i8 else 12.0) * elems_local,
                       "bound": "hbm" if use_i8 else "fp64 tensor pipe"}
    kern["eig_kernel"] = {"ms": solve_ms, "launches": n_solve, "alg_bytes": 8.0 * frames * frames, "bound": "latency",
                          "warm_started_iterations": counters.get("eig_fast_iters")}
    if two_kernel:
        kern["shrink_stream_kernel (iteration 1)"] = {"ms": shrink1_ms, "launches": args.steps, "alg_bytes": 16.0 * elems_local, "bound": "hbm"}
    for k in kern.values():
        k["gbs"] = (k["alg_bytes"] / (k["ms"] * 1e-3) / 1e9) if k["ms"] > 0 else 0.0
        k["share"] = (k["ms"] * k["launches"]) / (ms_step * args.steps) if ms_step > 0 else 0.0
    # The contract's figure for the "shrinkage/update pass" (SURVEY 8d): 20 B per element (read D, S, Y; write S, Y) over the time
    # of the whole pass -- here projection + single-pass kernel.  What the two kernels really move is in `kernels`.
    dom = "shrink_flat_kernel" if two_kernel else next(iter(kern))
    achieved = 20.0 * elems_local / (shrink_pass_ms * 1e-3) / 1e9 if shrink_pass_ms > 0 else 0.0
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            with open(tp) as f:
                traffic = json.load(f).get("%s@%d" % (args.workload, world), {}).get(dom)
        except Exception:
            traffic = None
    moved = sum(k["alg_bytes"] for n_, k in kern.items() if n_ in ("shrink_flat_kernel", "project_planes_kernel")) if two_kernel else kern[dom]["alg_bytes"]
    roofline = {"kernel": dom + (" (+ project_planes_kernel: the shrinkage/update pass)" if two_kernel else ""), "bound": "hbm",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "frac_of_8TBs_spec": achieved / 8000.0,
                "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": 20.0 * elems_local,
                "pass_ms": shrink_pass_ms,
                "designed_bytes_per_launch": moved, "achieved_designed_bytes": moved / (shrink_pass_ms * 1e-3) / 1e9 if shrink_pass_ms > 0 else 0.0,
                "frac_designed_bytes": (moved / (shrink_pass_ms * 1e-3) / 1e9 / peak) if shrink_pass_ms > 0 else 0.0,
                "whole_iteration_frac": (32.0 * elems_local / ((shrink_pass_ms + gram_ms + solve_ms) * 1e-3) / 1e9 / peak)
                if (shrink_pass_ms + gram_ms + solve_ms) > 0 else 0.0,
                "note": "achieved = SURVEY 8(d)'s 20 B/element / time of the pass (CUDA events on the launching stream, iterations 2..last); "
                        "designed_bytes = what the kernels are built to move (DESIGN.md 4.4); whole_iteration_frac = 32 B/element / "
                        "(pass + Gram + eigensolve)"}

    cpu = None
    parity = None
    if not args.no_cpu_baseline and world == 1:
        D64, r, c = cpu_sample(video, rows, cols, frames, (args.cpu_sample_div or 4) if rows * cols > 200000 else 1)
        threads = os.cpu_count() or 1
        dt, it_c, conv_c, L_c, S_c, mask_c = cpu_port_solve(D64, r, c, threads, keep=True)
        sc = (rows * cols) / float(r * c)
        cpu = {"value": frames / (dt * sc), "unit": "frames/s", "cores": threads, "kind": "port",
               "sample": f"{r}x{c} pixel window of every frame ({r * c}/{rows * cols} of the pixels), full solve {dt:.1f} s, scaled x{sc:.1f}",
               "iters": it_c, "converged": bool(conv_c)}
        # the same window through the CUDA path (same kernels as the timed run when frames > 256): parity next to the numbers
        try:
            dec_s = B.lsd_decomposition(D64, groups=B.get_proximal_flat_groups_nonoverlap((r, c), (3, 3)), img_shape=(r, c))
            st_s = dec_s.status()
            L_g, S_g, mask_g = dec_s.download('L'), dec_s.download('S'), dec_s.mask(2)
            rel = lambda a_, b_: float(np.linalg.norm(a_ - b_) / max(np.linalg.norm(b_), 1e-300))    # noqa: E731
            parity = {"window": f"{r}x{c}x{frames}", "iters_gpu": int(st_s.iter), "iters_oracle": int(it_c), "relF_L": rel(L_g, L_c),
                      "relF_S": rel(S_g, S_c), "mask_agreement": float((mask_g == mask_c).mean()), "paths": dec_s.debug_info(),
                      "eig_warm_started_iterations": dec_s.eig_fast_count()}
            dec_s.close()
        except Exception as ex:                             # reported, never hidden
            parity = {"error": str(ex)[:300]}

    out = {"metric": "frames/s decomposed", "value": frames / (ms_step * 1e-3), "unit": "frames/s", "n_gpus": world,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
           "scaling": "strong", "vs_baseline": None,
           "dtype": "f32 (state) / exact int8-slice Gram on tcgen05 + f64 eigensolve" if use_i8 else "f32 (state) / f64 Gram + eigensolve",
           "data": "reference fixture (WaterSurface)" if args.workload == "watersurface" else "synthetic",
           "config": {"workload": args.workload, "rows": rows, "cols": cols, "frames": frames, "prox": "flat 3x3 l_inf (LSD)",
                      "delta": 10, "sharding": f"pixel columns over {world} GPU(s)", "l2": "inputs (2.5 GB/matrix) larger than L2",
                      "tile_rows": info["stream_R"] if info["use_stream"] else solver.dec.cfg.tile_rows, "paths": info,
                      "timing": "CUDA events on the launching stream; inputs 2.5 GB per matrix >> 126 MB L2 (no flush needed)"},
           "alm_iters": iters, "converged": bool(st.converged), "rank_L": int(st.svp), "err": float(st.err),
           "mask_fraction": mask_fraction,
           "kernels": kern, "roofline": roofline, "cpu_baseline": cpu, "parity_vs_oracle": parity, "e2e": e2e, "gpu_launches": gpu_launches,
           "counters": counters,
           "clocks": clocks, "datagen_s": t_gen, "breakdown_ms": breakdown,
           "iters_enqueued": driver.iters_enqueued}
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
