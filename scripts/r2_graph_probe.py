"""Round-2 probe: graph-mode (overlapping windows) LSD; used under ncu to capture prox_graph3_tile_kernel (the first launch is ALM
iteration 1, the expensive one) and to look at the outer-iteration statistics of the prox (bsub_debug_graph).
   python scripts/r2_graph_probe.py [max_iter [rows cols frames [graph_max_sweeps]]]     (no shape: the WaterSurface clip)"""
import ctypes, os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import background_subtraction_b200 as B
from background_subtraction_b200 import _cabi as C, synth

max_iter = int(sys.argv[1]) if len(sys.argv) > 1 else 500
if len(sys.argv) > 4:
    rows, cols, n = (int(v) for v in sys.argv[2:5])
    video, _ = synth.make_clip(rows, cols, n, seed=0, n_rect=6, period=300)
else:
    cube = np.load(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "watersurface_u8.npz"))["ImData"]
    rows, cols, n = cube.shape
    video = np.ascontiguousarray(cube.transpose(2, 1, 0)).reshape(n, rows * cols)
cap = int(sys.argv[5]) if len(sys.argv) > 5 else 0
D = torch.from_numpy(synth.preprocess_u8(video)).cuda()
dec = B.Decomposition(B.make_config(rows * cols, n, C.PROX_GRAPH_LINF, rows, cols, max_iter=max_iter, graph_max_sweeps=cap))
dec.set_graph_windows(None)
for rep in range(2 if len(sys.argv) <= 4 else 1):
    dec.load(D)
    torch.cuda.synchronize(); t0 = time.perf_counter()
    dec.run(); st = dec.status()
    torch.cuda.synchronize(); dt = time.perf_counter() - t0
    out = (ctypes.c_int64 * 4)()
    C.check(dec.lib.bsub_debug_graph(dec.h, out))
    print("%dx%dx%d rep %d ms %.1f iters %d conv %d | prox outer iterations: last call %d, total %d over %d calls, %d calls hit the cap"
          % (rows, cols, n, rep, dt * 1e3, st.iter, st.converged, out[0], out[1], out[2], out[3]), flush=True)
print("svp", [l['svp'] for l in dec.log()], "err", ["%.2e" % l['err'] for l in dec.log()])
