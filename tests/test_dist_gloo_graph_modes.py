"""-m "not gpu": the sharded driver (background-subtraction_b200/dist.py) in the graph modes that run their prox on whole frames
(per-frame generic graphs, the same plus the l2 shrink of each frame's background) and in the l1 mode, on 2 CPU ranks over gloo.
Each rank runs the real ShardedLSD choreography around a NumPy step solver that proxes only the frames of its own range
(shard_frames: 7 frames -> 4 + 3); the stitched result must equal the oracle's whole-clip solve."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROWS, COLS, N, WORLD = 12, 15, 7, 2


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _clip():
    from background_subtraction_b200 import synth
    from oracle import alm_oracle as O
    video, _ = synth.make_clip(ROWS, COLS, N, seed=11, n_rect=2)
    cube = np.asfortranarray(video.reshape(N, COLS, ROWS).transpose(2, 1, 0))
    D, _x, _mean = O.normalize_and_center(cube)
    return D


def frame_graphs(rows, cols, n, seed=3):
    """One graph per frame, different in every frame so that a graph taken for the wrong frame changes the result: centre windows
    of radius 1 or 2 at random centres with random weights, 2 x 4 all-windows with random weights, and one frame (3) with no
    window.  Background masks (bool [n][rows * cols]): random, frame 5 empty."""
    from oracle import alm_oracle as O
    rng = np.random.default_rng(seed)
    graphs, bg = [], np.zeros((n, rows * cols), dtype=bool)
    for f in range(n):
        if f == 3:
            graphs.append((np.zeros(1, dtype=np.int32), np.zeros(0, dtype=np.int32), np.zeros(0, dtype=np.float64)))
        elif f % 3 == 1:
            ip, ix, _ = O.graph_all_groups((rows, cols), (2, 4))
            graphs.append((ip, ix, rng.uniform(0.5, 2.0, len(ip) - 1)))
        else:
            centres = np.where(rng.random((rows, cols)) < 0.25, rng.uniform(0.5, 2.0, (rows, cols)), 0.0)
            graphs.append(O.graph_group_centers((rows, cols), 1 + f % 2, centres))
        if f != 5:
            bg[f] = rng.random(rows * cols) < 0.4
    return graphs, bg


def modes_solver_class():
    from np_step_solver import NumpyStepSolver
    from oracle import alm_oracle as O

    class ModesStepSolver(NumpyStepSolver):
        """The NumPy step solver plus the whole-frame graph modes (prox of the frames [f0, f1) of the clip only) and the l1 mode."""

        def __init__(self, D_local, rows, cols_local, n, m_global, cols_full=None, graphs=None, background=None, frames=None,
                     l1=False):
            if l1:
                super().__init__(D_local, rows, cols_local, n, m_global, delta=1.0, mu_scale=1.25, rho=1.2)
            else:
                super().__init__(D_local, rows, cols_local, n, m_global, graph_cols=cols_full)
            self.l1, self.graphs, self.background = l1, graphs, background
            self.frame_range = None if l1 else tuple(frames)

        def prox_frames(self, Uf, Vf, rows, cols, nf):
            if self.done_flag or nf == 0: return
            f0, m = self.frame_range[0], rows * cols
            U = np.asfortranarray(Uf[:nf, :m].numpy().T)
            V = O.prox_by_frame(U, self.lam / self.mu, self.graphs[f0:f0 + nf], tol=1e-13)
            if self.background is not None:
                V = O.apply_background_shrinkage_operator(U, V, 100.0 * self.lam / self.mu, self.background[f0:f0 + nf])
            Vf[:nf, :m] = torch.from_numpy(np.ascontiguousarray(V.T))

        def init_local(self):
            super().init_local()
            if self.l1:
                self.sv = self.d                     # inexact_alm_rpca: no sv prediction

        def solve(self):
            if not self.l1:
                return super().solve()
            if self.done_flag: return
            G = self.sum_buf[:self.ngram].numpy().reshape(self.n, self.n)
            w, v = np.linalg.eigh(G)
            s = np.sqrt(np.maximum(w[::-1][:self.sv], 0)); v = v[:, ::-1][:, :self.sv]
            self.iter += 1
            self.svp, self.sv = O.rank_logic(s, self.sv, self.mu, self.d, use_sv_prediction=False)
            self.P = (v[:, :self.svp] * (1 - 1 / (self.mu * s[:self.svp]))) @ v[:, :self.svp].T

        def shrink(self):
            if not self.l1:
                return super().shrink()
            if self.done_flag: return
            self.L = self.W @ self.P
            G_S = self.D - self.L + self.Y / self.mu
            self.S = np.sign(G_S) * np.maximum(np.abs(G_S) - self.lam / self.mu, 0)
            Z = self.D - self.L - self.S
            self.Y = self.Y + self.mu * Z
            self.sum_buf[self.ngram:self.ngram + 4] = torch.tensor([float((Z * Z).sum()), float(np.count_nonzero(self.S)), 0.0, 0.0],
                                                                  dtype=torch.float64)
            self.mu *= self.rho

    return ModesStepSolver


def _worker(rank, world, port, mode, out_dir):
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from background_subtraction_b200 import dist as bdist
    D = _clip()
    graphs, bg = frame_graphs(ROWS, COLS, N)
    c0, c1 = bdist.shard_columns(COLS, world, rank)
    f0, f1 = bdist.shard_frames(N, world, rank)
    cls = modes_solver_class()
    solver = cls(D[c0 * ROWS:c1 * ROWS, :], ROWS, c1 - c0, N, ROWS * COLS, cols_full=COLS, graphs=graphs,
                 background=bg if mode == "background" else None, frames=(f0, f1), l1=mode == "l1")
    driver = bdist.ShardedLSD(solver, bdist.TorchComm(), run_ahead=2)
    driver.solve()
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), L=solver.L, S=solver.S, iters=solver.iter, conv=solver.converged,
             svp=[l[1] for l in solver.log], f0=f0, f1=f1)
    dist.destroy_process_group()


@pytest.mark.parametrize("mode", ["generic", "background", "l1"])
def test_sharded_modes_match_oracle(tmp_path, mode):
    port = _free_port()
    mp.spawn(_worker, args=(WORLD, port, mode, str(tmp_path)), nprocs=WORLD, join=True)
    sys.path.insert(0, ROOT)
    from oracle import alm_oracle as O
    D = _clip()
    graphs, bg = frame_graphs(ROWS, COLS, N)
    log = []
    if mode == "generic":
        L, S, it, conv = O.inexact_alm_lsd(D, graphs=graphs, log=log)
    elif mode == "background":
        L, S, it, conv = O.inexact_alm_lsd_with_background(D, graphs, list(bg), log=log)
    else:
        L, S, it, conv = O.inexact_alm_rpca(D, log=log)
    parts = [np.load(os.path.join(str(tmp_path), "rank%d.npz" % r)) for r in range(WORLD)]
    assert [(int(p["f0"]), int(p["f1"])) for p in parts] == [(0, 4), (4, 7)]
    Ls = np.vstack([p["L"] for p in parts]); Ss = np.vstack([p["S"] for p in parts])
    for p in parts:
        assert int(p["iters"]) == it and bool(p["conv"]) == conv and p["svp"].tolist() == [l["svp"] for l in log]
    assert np.abs(Ls - L).max() <= 1e-9 and np.abs(Ss - S).max() <= 1e-9


def test_sharded_driver_rejects_a_foreign_frame_range():
    """The frames a rank proxes are the ones the exchange brings it: a solver that describes others is refused up front."""
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
    from background_subtraction_b200 import dist as bdist

    class Comm:
        world, rank = 2, 1

    cls = modes_solver_class()
    graphs, _ = frame_graphs(ROWS, COLS, N)
    D = _clip()
    s = cls(D[:ROWS * 9, :], ROWS, 9, N, ROWS * COLS, cols_full=COLS, graphs=graphs, frames=(0, 4))
    with pytest.raises(Exception, match=r"describes frames \[0, 4\), but rank 1 of 2 owns \[4, 7\)"):
        bdist.ShardedLSD(s, Comm())
    bdist.ShardedLSD(cls(D[:ROWS * 9, :], ROWS, 9, N, ROWS * COLS, cols_full=COLS, graphs=graphs, frames=(4, 7)), Comm())
