"""-m "not gpu": host side of the generic graph prox (any non-nested SPAMS graph, one per frame): the packing helper, the input
validation of the C entry point (which rejects bad graphs before anything reaches the device) and the build of its kernel."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest
import scipy.sparse as ssp

import background_subtraction_b200 as B
from background_subtraction_b200 import _cabi as C
from background_subtraction_b200 import api, build
from oracle import alm_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _graph(indptr, indices, eta, m, nested=False):
    ng = len(indptr) - 1
    gv = ssp.csc_matrix((np.ones(len(indices), dtype=bool), np.asarray(indices, dtype=np.int32), np.asarray(indptr, dtype=np.int32)),
                        shape=(m, ng))
    groups = ssp.csc_matrix((ng, ng), dtype=bool)
    if nested:
        groups = ssp.csc_matrix((np.ones(1, dtype=bool), ([0], [1])), shape=(ng, ng))
    return {'eta_g': np.asarray(eta, dtype=np.float64), 'groups': groups, 'groups_var': gv}


def test_pack_round_trips_the_csc_arrays():
    for shape, win in (((9, 11), (5, 5)), ((7, 6), (2, 4)), ((5, 8), (1, 6))):
        g = B.getGraphSPAMS_all_groups(shape, win)
        csc, fg = B.pack_graphs(g, shape[0] * shape[1], 4)
        assert len(csc) == 1 and fg.tolist() == [0, 0, 0, 0]
        ip, ix, eta = O.graph_all_groups(shape, win)
        assert np.array_equal(csc[0][0], ip) and np.array_equal(csc[0][1], ix) and np.array_equal(csc[0][2], eta)
        assert csc[0][0].dtype == np.int32 and csc[0][1].dtype == np.int32 and csc[0][2].dtype == np.float64


def test_pack_dedupes_shared_graphs():
    shape = (8, 10)
    m = 80
    rng = np.random.default_rng(1)
    wms = [np.where(rng.random(shape) < 0.3, 1.0, -1.0) for _ in range(3)]
    ga = B.get_proximal_graph_group_centers(shape, 2, wms[0])
    ga_copy = B.get_proximal_graph_group_centers(shape, 2, wms[0])           # equal arrays, another object
    gb = B.get_proximal_graph_group_centers(shape, 2, wms[1])
    csc, fg = B.pack_graphs([ga, gb, ga, ga_copy, gb], m, 5)
    assert len(csc) == 2 and fg.tolist() == [0, 1, 0, 0, 1]
    p, i, e = O.graph_group_centers(shape, 2, wms[1])
    assert np.array_equal(csc[1][0], p) and np.array_equal(csc[1][1], i) and np.array_equal(csc[1][2], e)
    gc = B.get_proximal_graph_group_centers(shape, 2, wms[2])
    assert len(B.pack_graphs([ga, gc, gb], m, 3)[0]) == 3


def test_pack_rejects_bad_graphs():
    m = 12
    good = _graph([0, 3, 5], [0, 1, 2, 4, 11], [1.0, 0.5], m)
    B.pack_graphs(good, m, 2)
    with pytest.raises(Exception, match="nested groups"):
        B.pack_graphs(_graph([0, 3, 5], [0, 1, 2, 4, 11], [1.0, 0.5], m, nested=True), m, 2)
    with pytest.raises(Exception, match="graph has 12 variables, matrix has 13 rows"):
        B.pack_graphs(good, 13, 2)
    bad = _graph([0, 3, 5], [0, 1, 2, 4, 11], [1.0, 0.5], m)
    bad['groups_var'].indices[4] = 12                                      # scipy does not check bounds on construction
    with pytest.raises(Exception, match="out of range"):
        B.pack_graphs(bad, m, 2)
    with pytest.raises(Exception, match="same pixel twice"):
        B.pack_graphs(_graph([0, 3, 5], [0, 1, 0, 4, 11], [1.0, 0.5], m), m, 2)
    with pytest.raises(Exception, match="finite and >= 0"):
        B.pack_graphs(_graph([0, 3, 5], [0, 1, 2, 4, 11], [1.0, -0.5], m), m, 2)
    with pytest.raises(Exception, match="eta_g has 3 entries"):
        B.pack_graphs(_graph([0, 3, 5], [0, 1, 2, 4, 11], [1.0, 0.5, 2.0], m), m, 2)
    with pytest.raises(Exception, match="one graph per frame"):
        B.pack_graphs([good, good], m, 3)


def _call_prox_graph_dev(n_graphs, frame_graph, graphs, m, n):
    """bsub_prox_graph_dev with NULL matrices: the graph checks come first, so a bad graph is reported and a good one
    fails only on the NULL pointers -- nothing is launched either way."""
    lib = C.load()
    keep = [(np.ascontiguousarray(p, dtype=np.int32), np.ascontiguousarray(i, dtype=np.int32), np.ascontiguousarray(e, dtype=np.float64))
            for p, i, e in graphs]
    ng, ip, ix, et = api._graph_pointers(keep)
    fg = None if frame_graph is None else np.ascontiguousarray(frame_graph, dtype=np.int32)
    rc = lib.bsub_prox_graph_dev(None, None, m, m, n, 0.1, n_graphs, None if fg is None else fg.ctypes.data_as(C.c_int32_p),
                                 ng.ctypes.data_as(C.c_int64_p), ip, ix, et, 100, 1e-7, None, None)
    return rc, lib.bsub_last_error().decode()


@pytest.mark.parametrize("graph,frame_graph,msg", [
    (([0, 2, 4], [0, 1, 2, 9], [1.0, 1.0]), [0, 0], "bad argument"),              # valid graph: only the NULL matrices fail
    (([0, 2, 4], [0, 1, 2, 10], [1.0, 1.0]), [0, 0], "holds pixel 10, not in"),
    (([0, 2, 4], [0, 1, 2, -1], [1.0, 1.0]), [0, 0], "holds pixel -1, not in"),
    (([0, 2, 4], [0, 1, 3, 3], [1.0, 1.0]), [0, 0], "holds pixel 3 twice"),
    (([0, 2, 4], [0, 1, 2, 3], [1.0, -1.0]), [0, 0], "is not finite and >= 0"),
    (([0, 2, 4], [0, 1, 2, 3], [1.0, float("nan")]), [0, 0], "is not finite and >= 0"),
    (([0, 2, 4], [0, 1, 2, 3], [1.0, float("inf")]), [0, 0], "is not finite and >= 0"),
    (([0, 3, 2], [0, 1, 2, 3], [1.0, 1.0]), [0, 0], "indptr decreases"),
    (([1, 2, 4], [0, 1, 2, 3], [1.0, 1.0]), [0, 0], "indptr\\[0\\] = 1"),
    (([0, 2, 4], [0, 1, 2, 3], [1.0, 1.0]), [0, 1], "frame_graph\\[1\\] = 1 is not a graph index"),
    (([0, 2, 4], [0, 1, 2, 3], [1.0, 1.0]), [0, -1], "frame_graph\\[1\\] = -1 is not a graph index"),
])
def test_c_entry_point_validates_before_any_launch(graph, frame_graph, msg):
    rc, err = _call_prox_graph_dev(1, frame_graph, [graph], 10, 2)
    assert rc != 0 and re.search(msg, err), err


def test_c_entry_point_needs_frame_graph_for_several_graphs():
    g = ([0, 2], [0, 1], [1.0])
    rc, err = _call_prox_graph_dev(2, None, [g, g], 10, 2)
    assert rc != 0 and "frame_graph is required" in err


def test_new_symbols_resolve():
    lib = C.load()
    for name in ("bsub_set_graphs", "bsub_prox_graph_dev"):
        assert hasattr(lib, name) and name in C.SIGNATURES
    assert C.PROX_GRAPH_GENERIC == 5
    hdr = open(os.path.join(ROOT, "include", "bsub_b200.h")).read()
    assert re.search(r"BSUB_PROX_GRAPH_GENERIC\s*=\s*5", hdr)


def test_generic_graph_kernels_do_not_spill(tmp_path):
    """The generic prox kernels keep everything in registers and shared memory (ptxas reports no local-memory spills)."""
    src = os.path.join(build.CSRC, "prox_graph.cu")
    cmd = [build.NVCC] + build.ARCH_FLAGS + [f for f in build.COMMON if not f.startswith("--use_fast_math")] + \
        ["-Xptxas", "-v", "-c", src, "-o", str(tmp_path / "prox_graph.o")]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, check=True).stdout
    props = re.findall(r"Function properties for (\S+)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", out)
    names = [p[0] for p in props]
    assert any("prox_graph_generic_kernel" in n for n in names) and any("prox_graph_generic_stats_kernel" in n for n in names), out
    for name, stack, st, ld in props:
        assert (int(stack), int(st), int(ld)) == (0, 0, 0), (name, stack, st, ld)
