"""-m "not gpu": host side of the sharded graph modes -- the frame-range entry points resolve, their host code adds no device code
(they launch the existing prox kernels, so no kernel's registers or spills can change), the kernel choice the public solvers and
dist.CudaStepSolver share (api.route_graphs / route_weight_mask), and the argument checks CudaStepSolver and the window operators
make before any device work."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

import background_subtraction_b200 as B
from background_subtraction_b200 import _cabi as C
from background_subtraction_b200 import api, build, dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ("bsub_set_frame_windows", "bsub_set_frame_center_windows", "bsub_set_frame_graphs", "bsub_step_prox_block")


def test_new_symbols_resolve():
    lib = C.load()
    hdr = open(os.path.join(ROOT, "include", "bsub_b200.h")).read()
    for name in NEW:
        assert hasattr(lib, name) and name in C.SIGNATURES
        assert re.search(r"\bint %s\(" % name, hdr)


def test_solver_host_code_has_no_kernels(tmp_path):
    src = os.path.join(build.CSRC, "solver.cu")
    cmd = [build.NVCC] + build.ARCH_FLAGS + [f for f in build.COMMON if not f.startswith("--use_fast_math")] + \
        ["-Xptxas", "-v", "-c", src, "-o", str(tmp_path / "solver.o")]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, check=True).stdout
    assert "Function properties" not in out and "Compiling entry function" not in out, out


def test_route_picks_the_kernels_of_the_public_solvers():
    h, w, n = 9, 12, 4
    m = h * w
    r = api.route_graphs(B.getGraphSPAMS_all_groups((h, w), (3, 3)), m, n, (h, w))
    assert (r.prox, r.rows, r.cols, r.eta) == (C.PROX_GRAPH_LINF, h, w, None)
    g = B.getGraphSPAMS_all_groups((h, w), (3, 3))
    g['eta_g'] = np.linspace(0.5, 2.0, len(g['eta_g']))
    r = api.route_graphs(g, m, n, (h, w))
    assert r.prox == C.PROX_GRAPH_LINF and np.array_equal(r.eta, g['eta_g'])
    r = api.route_graphs(B.getGraphSPAMS_all_groups((h, w), (2, 5)), m, n, (h, w))
    assert (r.prox, r.rows, r.cols, r.frame_graph.tolist(), r.background) == (C.PROX_GRAPH_GENERIC, h, w, [0] * n, None)
    rng = np.random.default_rng(0)
    wms = [np.where(rng.random((h, w)) < 0.3, 1.5, -1.0) for _ in range(n)]
    bgs = [(wm < 0).flatten(order='F') for wm in wms]
    r = api.route_graphs([B.get_proximal_graph_group_centers((h, w), 1, wm) for wm in wms], m, n, (h, w), background_masks=bgs)
    assert (r.prox, r.rows, r.cols) == (C.PROX_GRAPH_CENTER_BG, h, w)
    assert np.array_equal(r.background, np.stack(bgs).astype(np.uint8)) and r.eta.shape == (n, m)
    r2 = api.route_weight_mask(np.stack(wms, axis=2), m, n)
    assert r2.prox == C.PROX_GRAPH_CENTER_BG and np.array_equal(r2.eta, r.eta) and np.array_equal(r2.background, r.background)
    r = api.route_graphs([B.get_proximal_graph_group_centers((h, w), 2, wm) for wm in wms], m, n, (h, w), background_masks=bgs)
    assert r.prox == C.PROX_GRAPH_GENERIC and len(r.csc) == n and r.background.shape == (n, m)


@pytest.mark.parametrize("kw,msg", [
    (dict(graphs={}, l1=True, graph_cols=6), "mutually exclusive"),
    (dict(weight_mask=np.zeros((3, 6, 4)), blocks=(None, None, None)), "mutually exclusive"),
    (dict(background_masks=[None] * 4), "background_masks needs graphs"),
    (dict(graphs=B.getGraphSPAMS_all_groups((3, 6), (2, 2))), "graphs needs graph_cols"),
    (dict(weight_mask=np.zeros((3, 6, 4)), graph_cols=5), "weight_mask has 6 columns"),
    (dict(frames=(0, 2)), "frames applies to the graph modes"),
])
def test_step_solver_checks_its_arguments(kw, msg):
    with pytest.raises(Exception, match=msg):
        dist.CudaStepSolver(3, 3, 4, 18, **kw)


def test_step_prox_frames_is_gone():
    """bsub_step_prox_block serves every graph mode on frame shards, unit-weight windows included: the older entry point is gone."""
    lib = C.load()
    hdr = open(os.path.join(ROOT, "include", "bsub_b200.h")).read()
    assert not hasattr(lib, "bsub_step_prox_frames")
    assert "bsub_step_prox_frames" not in C.SIGNATURES and "bsub_step_prox_frames" not in hdr


@pytest.mark.parametrize("fn,eta,msg", [
    ("bsub_prox_graph3_dev", [1.0, float("nan")], r"bsub_prox_graph3_dev: eta\[1\] = nan is not finite and >= 0"),
    ("bsub_prox_graph3_dev", [-0.5, 1.0], r"eta\[0\] = -0.5 is not finite and >= 0"),
    ("bsub_prox_graph3_dev", [1.0, 2.0], "bsub_prox_graph3_dev: bad argument"),
    ("bsub_prox_center3_dev", [0.5, float("nan")], r"bsub_prox_center3_dev: eta\[1\] = nan is not finite"),
    ("bsub_prox_center3_dev", [-1.0, 2.0], "bsub_prox_center3_dev: bad argument"),
])
def test_window_operators_check_eta_first(fn, eta, msg):
    """NULL matrices: the weights are checked first, so bad ones are reported and good ones fail only on the NULL pointers --
    nothing reaches the device either way.  A 3 x 4 image has two 3 x 3 windows; the centre map of one 1 x 2 frame, two entries."""
    lib = C.load()
    sw = ctypes.c_int32(0)
    if fn == "bsub_prox_graph3_dev":
        e = np.asarray(eta, dtype=np.float64)
        rc = lib.bsub_prox_graph3_dev(None, None, 12, 3, 4, 1, 0.1, e.ctypes.data_as(C.c_double_p), 10, 1e-6, ctypes.byref(sw), None)
    else:
        e = np.asarray(eta, dtype=np.float32)
        rc = lib.bsub_prox_center3_dev(None, None, 2, 1, 2, 1, 0.1, e.ctypes.data_as(C.c_float_p), 10, 1e-6, ctypes.byref(sw), None)
    assert rc != 0
    assert re.search(msg, lib.bsub_last_error().decode())
