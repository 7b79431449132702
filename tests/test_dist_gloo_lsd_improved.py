"""-m "not gpu": LSD_improved over ranks (dist.ShardedLSDImproved) on CPU ranks over gloo.  Each rank runs the real driver -- the
pre-processing all-reduces, pass 1 through ShardedLSD, the all-to-all of the pass-1 mask to whole frames, the morphology, merge and
back-off on its own frames, pass 2 on the frame-range description of its weight map -- around NumPy stand-ins for the step solvers
and the per-frame work (the oracle's apply_morph_ops / merge_masks).  The stitched result must equal the oracle's whole-clip
improved_LSD_weight_mask + LSD_improved_from_weight_mask: identical weight map, same iterations and ranks in both passes."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROWS, COLS = 22, 24                   # rows >= 21: disk radius 1 at the first ratio; rows % 3 != 0


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def make_cube(rows, cols, t, dense, seed=0):
    """[h, w, t] clip, 0..255 float64: smooth background, noise, and a blob across the middle column (the column-shard boundary of
    two ranks) whose left half is taller than its right half, so a morphology per column shard differs from the whole-frame one.
    dense: four 9 x 9 blobs at random places in every frame, enough foreground for the mask-percentage back-off to run."""
    rng = np.random.default_rng(seed)
    ii, jj = np.meshgrid(np.arange(rows), np.arange(cols), indexing='ij')
    bg = 0.4 + 0.2 * np.sin(ii / 5.0) * np.cos(jj / 7.0)
    cube = np.empty((rows, cols, t))
    mid = cols // 2
    for f in range(t):
        img = bg * (1 + 0.05 * np.sin(2 * np.pi * f / t)) + 0.01 * rng.standard_normal((rows, cols))
        r0 = (2 + 2 * f) % (rows - 8)
        img[r0:r0 + 7, mid - 4:mid] = 0.95
        img[r0 + 2:r0 + 5, mid:mid + 3] = 0.95
        if dense:
            for k in range(4):
                a, b = rng.integers(0, rows - 9), rng.integers(0, cols - 9)
                img[a:a + 9, b:b + 9] = 0.05 if k % 2 else 0.9
        cube[:, :, f] = img
    return np.asfortranarray(np.round(cube * 255))


def numpy_ops():
    """NumPy stand-ins for dist.CudaImprovedOps (float64 step solvers of tests/np_step_solver.py and the oracle's morphology)."""
    from np_step_solver import NumpyStepSolver
    from oracle import alm_oracle as O
    from oracle import flow_oracle as F
    from test_dist_gloo_graph_modes import modes_solver_class

    def frame_mask(cls):
        class Masked(cls):
            def mask_device(self, sigmas=2.0):            # uint8 [n][m_local], like CudaStepSolver.mask_device
                return torch.from_numpy(np.ascontiguousarray(super().mask_device(sigmas).T).astype(np.uint8))
        return Masked

    class NumpyImprovedOps:
        device = "cpu"

        def __init__(self):
            self.weight_calls = 0

        def matrix(self, D):
            return np.asfortranarray(np.asarray(D).T)

        def pass1(self, D, rows, cols_local, n, m_global, alg_ver):
            if alg_ver == 2:
                return frame_mask(NumpyStepSolver)(D, rows, cols_local, n, m_global, delta=1.0)
            s = frame_mask(modes_solver_class())(D, rows, cols_local, n, m_global, l1=True)
            s.lam = 1.0 / (np.sqrt(max(m_global, n)) * 10.0)           # inexact_alm_rpca(delta=10.0)
            return s

        def pass2(self, D, rows, cols_local, n, m_global, cols, frames, weight):
            f0, f1 = frames
            graphs, bg = [None] * n, np.zeros((n, rows * cols), dtype=bool)
            for f in range(f0, f1):
                wm = weight[f - f0].numpy().reshape(cols, rows).T
                graphs[f] = O.graph_group_centers((rows, cols), 1, wm)
                bg[f] = weight[f - f0].numpy() < 0
            return frame_mask(modes_solver_class())(D, rows, cols_local, n, m_global, cols_full=cols, graphs=graphs, background=bg,
                                                    frames=frames)

        def summary(self, s):
            return s.iter, s.converged, [l[1] for l in s.log]

        def close(self, s):
            pass

        def weight_map(self, mask, rows, cols, disk_ratio, weights):
            self.weight_calls += 1
            nf = int(mask.shape[0])
            if nf == 0:
                return torch.zeros((0, rows * cols), dtype=torch.float64), 0
            cube = mask.numpy().reshape(nf, cols, rows).transpose(2, 1, 0) != 0
            wm = F.merge_masks((cube, F.apply_morph_ops(cube, disk_ratio)), weights)
            flat = np.ascontiguousarray(wm.transpose(2, 1, 0)).reshape(nf, rows * cols)
            return torch.from_numpy(flat), int(np.sum(flat > 0))

        def outputs(self, s, mask, rows, cols_local, n, like):
            return s.S, mask.numpy().T.reshape((rows, cols_local, n), order='F') != 0, s.L.reshape((rows, cols_local, n), order='F')

    return NumpyImprovedOps()


def _worker(rank, world, port, t, alg_ver, dense, out_dir):
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from background_subtraction_b200 import dist as bdist
    cube = make_cube(ROWS, COLS, t, dense)
    c0, c1 = bdist.shard_columns(COLS, world, rank)
    ops = numpy_ops()
    drv = bdist.ShardedLSDImproved(bdist.TorchComm(), ops=ops, run_ahead=2)
    S, S_mask, L, im1, mean, shape, it, conv, git, gconv = drv.run(np.asfortranarray(cube[:, c0:c1, :]), (ROWS, COLS, t), alg_ver)
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), S=S, S_mask=S_mask, L=L, im1=im1, mean=mean, it=it, conv=conv, git=git,
             gconv=gconv, svp1=drv.pass1_log[2], svp2=drv.pass2_log[2], wf=drv.weight_frames.numpy(), frames=drv.frames,
             calls=ops.weight_calls, shape=shape)
    dist.destroy_process_group()


@pytest.mark.parametrize("world,t,alg_ver,dense", [(2, 8, 2, False), (2, 8, 1, True), (3, 2, 2, True)])
def test_sharded_lsd_improved_matches_oracle(tmp_path, world, t, alg_ver, dense):
    port = _free_port()
    mp.spawn(_worker, args=(world, port, t, alg_ver, dense, str(tmp_path)), nprocs=world, join=True)
    sys.path.insert(0, ROOT)
    from background_subtraction_b200 import dist as bdist
    from oracle import alm_oracle as O
    from oracle import flow_oracle as F
    cube = make_cube(ROWS, COLS, t, dense)
    shape = (ROWS, COLS, t)
    D, x, mean = O.normalize_and_center(cube)
    wm, it1, conv1 = F.improved_LSD_weight_mask(D, shape, alg_ver=alg_ver)
    L, S, it2, conv2, mask = F.LSD_improved_from_weight_mask(D, shape, wm)
    log1, log2 = [], []                                     # the rank sequences of the same two solves
    if alg_ver == 2:
        O.inexact_alm_lsd(D, groups=O.flat_groups_nonoverlap(shape[:2], (3, 3)), delta=1.0, log=log1)
    else:
        O.inexact_alm_rpca(D, delta=10.0, log=log1)
    O.inexact_alm_lsd_with_background(D, [O.graph_group_centers(shape[:2], 1, wm[:, :, i]) for i in range(t)],
                                      [(wm[:, :, i] < 0).flatten(order='F') for i in range(t)], log=log2)
    parts = [np.load(os.path.join(str(tmp_path), "rank%d.npz" % r)) for r in range(world)]
    assert [tuple(p["frames"]) for p in parts] == [bdist.shard_frames(t, world, r) for r in range(world)]
    if world == 3:
        assert tuple(parts[2]["frames"]) == (2, 2)                # a rank without a frame
    steps = int(parts[0]["calls"]) - 1
    assert steps >= 2 if alg_ver == 1 else steps == 0 if not dense else steps >= 1
    for p in parts:
        assert int(p["calls"]) - 1 == steps and tuple(p["shape"]) == shape
        assert int(p["git"]) == it1 and bool(p["gconv"]) == conv1 and p["svp1"].tolist() == [l["svp"] for l in log1]
        assert int(p["it"]) == it2 and bool(p["conv"]) == conv2 and p["svp2"].tolist() == [l["svp"] for l in log2]
        assert abs(float(p["mean"]) - mean) <= 1e-15
    wf = np.concatenate([p["wf"] for p in parts], axis=0)                  # [t][h * w], frame-major
    assert np.array_equal(wf, np.ascontiguousarray(wm.transpose(2, 1, 0)).reshape(t, -1))
    assert np.array_equal(np.concatenate([p["im1"] for p in parts], axis=1), x)
    Ls = np.concatenate([p["L"] for p in parts], axis=1).reshape(D.shape, order='F')
    Ss = np.concatenate([p["S"].reshape((ROWS, -1, t), order='F') for p in parts], axis=1).reshape(D.shape, order='F')
    assert np.abs(Ls - L).max() <= 1e-9 and np.abs(Ss - S).max() <= 1e-9
    assert np.array_equal(np.concatenate([p["S_mask"] for p in parts], axis=1), mask)


def test_driver_rejects_bad_arguments():
    """Before any collective: a downsampled run (resizing couples columns), an unknown alg_ver, a cube that is not the rank's
    shard_columns."""
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
    from background_subtraction_b200 import dist as bdist

    class Comm:
        world, rank = 2, 1

    cube = make_cube(ROWS, COLS, 4, False)
    drv = bdist.ShardedLSDImproved(Comm(), ops=numpy_ops())
    c0, c1 = bdist.shard_columns(COLS, 2, 1)
    with pytest.raises(Exception, match="downsample_ratio must be 1"):
        drv.run(cube[:, c0:c1], (ROWS, COLS, 4), 2, downsample_ratio=2)
    with pytest.raises(Exception, match="LSD_improved wrong alg ver"):
        drv.run(cube[:, c0:c1], (ROWS, COLS, 4), 3)
    with pytest.raises(Exception, match=r"rank 1 of 2 owns columns \[12, 24\) of the 24, so its cube must be \[22, 12, 4\]"):
        drv.run(cube[:, :c0 + 3], (ROWS, COLS, 4), 2)
