"""Pixel-row sharded multi-GPU driver (one process per GPU, torch.distributed for the plumbing).

The path shards by image columns (pixel index p = j*rows + i, so a block of whole columns is a contiguous pixel
range of every frame): rank r owns the column triples [t0, t1) so that no 3x3 tile straddles two ranks
(SURVEY.md section 8e).  Per ALM iteration there is ONE exchange (two in the l2-block and graph modes, see ShardedLSD): an all-reduce(SUM) of a single buffer that holds the
frames x frames fp64 Gram partial of iteration k+1 followed by the 4 scalars of iteration k (sum Z^2, ||S||_0, ...).  The
shrink pass of iteration k advances mu itself (local data only), the Gram of k+1 is enqueued right behind it, and the
residual / stop test of iteration k is evaluated after the joint message has arrived; an iteration that turns out to be
the last one has then cost one surplus Gram pass.  At init: all-reduce(SUM) Gram(D) and all-reduce(MAX) of the row-sum
maximum; at the end all-reduce(MAX), then (SUM) of the foreground-mask statistics.
The stop decision is identical on every rank by construction: a rank leaves the loop at the first loop index `it` for
which the device-written status says "done at iteration k" with k <= it - run_ahead, where the fence of iteration
it - run_ahead has completed -- never on a flag it merely happened to see early (ranks that left at different indices
would issue different numbers of collectives).  The eigensolve is replicated (bit-identical inputs after the all-reduce), so no
broadcast is needed.  The same driver runs world_size == 1 without any collective.

The numerical work is done by a *step solver* object; the product one is `CudaStepSolver` (libbsub_b200.so through
the C ABI).  The collective choreography is backend-agnostic (`comm` only needs all_reduce_sum / all_reduce_max on
array-like buffers), which is what the world_size-2 gloo tests on CPU exercise with a NumPy stand-in step solver.
"""
import ctypes

import numpy as np

from . import _cabi as C
from . import api


def shard_columns(cols, world, rank):
    """Column range [c0, c1) of `rank`: whole column triples, as even as possible."""
    ntrip = (cols + 2) // 3
    base, extra = divmod(ntrip, world)
    t0 = rank * base + min(rank, extra)
    t1 = t0 + base + (1 if rank < extra else 0)
    return min(3 * t0, cols), min(3 * t1, cols)


def shard_frames(n, world, rank):
    """Frame range [f0, f1) of `rank` for the frame-wise re-sharding of the overlapping-window prox: as even as possible."""
    base, extra = divmod(n, world)
    f0 = rank * base + min(rank, extra)
    return f0, f0 + base + (1 if rank < extra else 0)


class TorchComm:
    """all-reduce (and the all-to-all of the overlapping-window mode) on torch tensors over torch.distributed (NCCL on GPUs, gloo
    on CPU)."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist = dist
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0

    def all_reduce_sum(self, t):
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM, group=self.group)

    def all_reduce_max(self, t):
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX, group=self.group)

    def exchange(self, recv, send):
        """all-to-all: send[q] goes to rank q, recv[q] arrives from rank q (contiguous tensors, sizes agreed by construction)."""
        if self.world == 1:
            recv[0].copy_(send[0])
            return
        if self.dist.get_backend(self.group) == "nccl":
            self.dist.all_to_all(recv, send, group=self.group)
            return
        recv[self.rank].copy_(send[self.rank])          # gloo has no all-to-all: pairwise non-blocking sends / receives
        reqs = []
        for q in range(self.world):
            if q != self.rank:
                if send[q].numel():
                    reqs.append(self.dist.isend(send[q], q, group=self.group))
                if recv[q].numel():
                    reqs.append(self.dist.irecv(recv[q], q, group=self.group))
        for r_ in reqs:
            r_.wait()


class CudaStepSolver:
    """Thin object view of the bsub_step_* C entry points for one shard."""

    def __init__(self, rows, cols_local, n, m_global, delta=None, max_iter=500, tile_rows=0, cluster_frames=0, store_S_lazily=True,
                 blocks=None, use_sv_prediction=True, graph_cols=None, graphs=None, background_masks=None, weight_mask=None, l1=False,
                 frames=None):
        """blocks = (labels uint8 [n][rows * cols_local] of THIS shard's pixels, lam_ptr int32 [n + 1], lam float64) selects the
        group-sparse solver (inexact_alm_group_sparse_RPCA, /root/reference/group_sparse_RPCA.py:45-126: l2 blocks per frame,
        mu0 = 1.25 / ||D||_2, stop on rank 0); lam_ptr / lam are the same on every rank.  graph_cols = number of image columns of the
        WHOLE frame alone selects the reference's default LSD() mode (overlapping 3x3 windows with unit weights,
        /root/reference/inexact_alm_lsd.py:13-57): the prox then runs on whole frames after a frame-wise re-sharding (ShardedLSD).
        The other graph modes also run their prox on whole frames, those of `frames` = (f0, f1), which must be
        shard_frames(n, world, rank) (default: all n frames, one rank); they take the public solvers' descriptions of the WHOLE
        frame (rows x graph_cols pixels), and api.route_graphs / api.route_weight_mask pick the kernel as those solvers do:
          graphs = SPAMS graph dict or per-frame list, with graph_cols: inexact_alm_lsd(graphs=...);
          graphs + background_masks (list of n boolean masks of the whole frame): inexact_alm_lsd_with_background;
          weight_mask = [h, w, t] map of build_improved_LSD_graphs: center_window_decomposition (LSD_improved's second pass).
        l1=True: inexact_alm_rpca (elementwise soft threshold, /root/reference/lsd_improvement.py:123-196: delta 1.0, mu0 =
        1.25 / ||D||_2, rho 1.2, no sv prediction), which shards without any exchange.  Default: flat 3x3 l_inf groups (LSD)."""
        if sum(x is not None for x in (blocks, graphs, weight_mask)) + bool(l1) > 1:
            raise Exception("CudaStepSolver: blocks, graphs, weight_mask and l1 are mutually exclusive")
        if background_masks is not None and graphs is None:
            raise Exception("CudaStepSolver: background_masks needs graphs")
        route = None
        if weight_mask is not None:
            gc = int(np.shape(weight_mask)[1])
            if graph_cols is not None and graph_cols != gc:
                raise Exception("CudaStepSolver: weight_mask has %d columns, graph_cols = %d" % (gc, graph_cols))
            route = api.route_weight_mask(weight_mask, rows * gc, n, (rows, gc))
        elif graphs is not None:
            if graph_cols is None:
                raise Exception("CudaStepSolver: graphs needs graph_cols, the number of columns of the whole frame")
            route = api.route_graphs(graphs, rows * graph_cols, n, (rows, graph_cols), background_masks=background_masks)
        self.frame_range = None
        if route is not None:
            graph_cols = route.cols
            self.frame_range = (0, n) if frames is None else (int(frames[0]), int(frames[1]))
        elif frames is not None:
            raise Exception("CudaStepSolver: frames applies to the graph modes given by graphs or weight_mask")
        elif graph_cols is not None and not l1:
            if blocks is not None:
                raise Exception("CudaStepSolver: blocks and graph_cols are mutually exclusive")
            route = api.GraphRoute(C.PROX_GRAPH_LINF, rows, graph_cols)      # unit weights: frame_range stays None
        if delta is None:
            delta = 1.0 if l1 else 10
        self.rows, self.cols_local, self.graph_cols = rows, cols_local, graph_cols
        # store_S_lazily: let the single-pass shrink kernel skip the store of S in iterations that cannot be the last (it is
        # rebuilt from D, Y and the digit planes at the end).  A clipped digit pass in such an iteration stops EVERY rank with
        # done == 5 in the same iteration (the flag is part of the all-reduced scalars); ShardedLSD then repeats the solve
        # with S stored every time.
        self.m = rows * cols_local
        if route is not None:
            cfg = api.make_config(self.m, n, route.prox, rows, cols_local, delta=delta, m_global=m_global, d_global=min(m_global, n),
                                  max_iter=max_iter)
            self.lazy_S = False
            self.dec = api.Decomposition(cfg)
            self.dec.set_frame_route(route, *(self.frame_range or (0, n)))
        elif l1:
            cfg = api.make_config(self.m, n, C.PROX_L1, 0, 0, delta=delta, mu_scale=1.25, rho=1.2, use_sv_prediction=False,
                                  m_global=m_global, d_global=min(m_global, n), max_iter=max_iter, tile_rows=tile_rows,
                                  cluster_frames=cluster_frames, flags=0 if store_S_lazily else C.FLAG_ALWAYS_STORE_S)
            self.lazy_S = bool(store_S_lazily)
            self.dec = api.Decomposition(cfg)
        elif blocks is None:
            cfg = api.make_config(self.m, n, C.PROX_FLAT_LINF, rows, cols_local, delta=delta, m_global=m_global,
                                  d_global=min(m_global, n), max_iter=max_iter, tile_rows=tile_rows,
                                  cluster_frames=cluster_frames, flags=0 if store_S_lazily else C.FLAG_ALWAYS_STORE_S)
            self.lazy_S = bool(store_S_lazily)
            self.dec = api.Decomposition(cfg)
            self.dec.set_flat_groups(api.get_proximal_flat_groups_nonoverlap((rows, cols_local), api.BLOCK_SIZE))
        else:
            cfg = api.make_config(self.m, n, C.PROX_BLOCK_L2, rows, cols_local, delta=delta, mu_scale=1.25, break_on_rank0=True,
                                  use_sv_prediction=use_sv_prediction, m_global=m_global, d_global=min(m_global, n), max_iter=max_iter)
            self.lazy_S = False
            self.dec = api.Decomposition(cfg)
            self.dec.set_blocks(*blocks)
        self.lib, self.h = self.dec.lib, self.dec.h
        self.n = n
        self.block_sums = None
        if blocks is not None:
            bp, bc = ctypes.c_void_p(), ctypes.c_int64(0)
            C.check(self.lib.bsub_block_sums_buffer(self.h, ctypes.byref(bp), ctypes.byref(bc)))
            import torch as _torch
            self.block_sums = api._wrap_device(bp.value, (bc.value,), _torch.float64)
        sp, mp = ctypes.c_void_p(), ctypes.c_void_p()
        sc, mc = ctypes.c_int64(0), ctypes.c_int64(0)
        C.check(self.lib.bsub_comm_buffers(self.h, ctypes.byref(sp), ctypes.byref(sc), ctypes.byref(mp), ctypes.byref(mc)))
        import torch
        self.sum_buf = api._wrap_device(sp.value, (sc.value,), torch.float64)
        self.max_buf = api._wrap_device(mp.value, (mc.value,), torch.float64)
        self.ngram = sc.value - 16

    def _s(self):
        return self.dec.stream()

    def load(self, D):
        self.dec.load(D)

    def init_local(self):
        C.check(self.lib.bsub_step_init_local(self.h, self._s()))

    def init_finish(self):
        C.check(self.lib.bsub_step_init_finish(self.h, self._s()))

    def gram(self):
        C.check(self.lib.bsub_step_gram(self.h, self._s()))

    def solve(self):
        C.check(self.lib.bsub_step_solve(self.h, self._s()))

    def project(self):
        C.check(self.lib.bsub_step_project(self.h, self._s()))

    def shrink(self):
        C.check(self.lib.bsub_step_shrink(self.h, self._s()))

    def shrink_a(self):
        C.check(self.lib.bsub_step_shrink_a(self.h, self._s()))

    def shrink_b(self):
        C.check(self.lib.bsub_step_shrink_b(self.h, self._s()))

    def graph_split(self):
        """(rows, columns of the whole frame) when the prox has to run on whole frames (overlapping-window mode), else None."""
        return (self.rows, self.graph_cols) if self.graph_cols is not None else None

    def prox_buffers(self):
        """G_S of this pixel shard (valid after shrink_a) and the S it expects before shrink_b: torch views [n][m_local]."""
        import torch
        gp, sp, ld = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_int64(0)
        C.check(self.lib.bsub_step_prox_buffers(self.h, ctypes.byref(gp), ctypes.byref(sp), ctypes.byref(ld)))
        return (api._wrap_device(gp.value, (self.n, ld.value), torch.float32)[:, :self.m],
                api._wrap_device(sp.value, (self.n, ld.value), torch.float32)[:, :self.m])

    def frames_like(self, nf, ldf):
        import torch
        return torch.empty((max(nf, 1), ldf), dtype=torch.float32, device="cuda")

    def prox_frames(self, Uf, Vf, rows, cols, nf):
        """Prox of this rank's nf whole frames (rows of Uf / Vf, row stride Uf.stride(0)) at this handle's lambda / mu."""
        # the unit-weight window description (frame_range None) holds no per-frame data: frames [0, nf) of it prox any nf frames
        self.prox_block(Uf, Vf, self.frame_range[0] if self.frame_range is not None else 0, nf)

    def prox_block(self, Uf, Vf, f0, nf):
        """Prox of the whole frames [f0, f0 + nf) of the clip, held in the rows of Uf / Vf: any block of this solver's frame range."""
        C.check(self.lib.bsub_step_prox_block(self.h, ctypes.c_void_p(Uf.data_ptr()), ctypes.c_void_p(Vf.data_ptr()), int(Uf.stride(0)),
                                              int(f0), int(nf), self._s()))

    def debug_graph(self):
        """bsub_debug_graph: outer iterations of the last prox call, their total, calls, calls that hit graph_max_sweeps."""
        out = (ctypes.c_int64 * 4)()
        C.check(self.lib.bsub_debug_graph(self.h, out))
        return list(out)

    def block_sums_view(self):
        """l2-block mode: per-(frame, group) sums of squares of this shard, to be all-reduced between shrink_a and shrink_b."""
        return self.block_sums

    def finish_iter(self):
        C.check(self.lib.bsub_step_finish_iter(self.h, self._s()))

    def gram_view(self):
        return self.sum_buf[:self.ngram]

    def tail_view(self):
        return self.sum_buf[self.ngram:self.ngram + 4]

    def sum_view(self):
        """Gram partial + the 4 scalars of the previous iteration (+ the error bound of the int8 Gram in slot 8): one
        all-reduce message per ALM iteration."""
        return self.sum_buf[:self.ngram + 9]

    def mask_tail_view(self):
        return self.sum_buf[self.ngram + 4:self.ngram + 8]

    def max_view(self):
        return self.max_buf

    needs_fence = True          # the status word is written by the device: only look at it behind a fence

    def done(self):
        """Non-blocking look at the device-written status word."""
        return self.dec.poll().done != 0

    def done_by(self, k):
        """True iff the solve stopped at an iteration <= k (the caller has fenced iteration k)."""
        st = self.dec.poll()
        return st.done != 0 and st.iter <= k

    def wait_iter(self, k):
        pass

    def needs_restart(self):
        """done == 5: a digit pass clipped while S was not being stored (see bsub_set_always_store_S); blocking read."""
        return self.lazy_S and self.dec.status().done == 5

    def store_S_always(self):
        self.lazy_S = False
        C.check(self.lib.bsub_set_always_store_S(self.h, 1))

    def status(self):
        return self.dec.status()

    def finalize(self):
        self.dec.finalize()

    def mask_stats(self, phase):
        C.check(self.lib.bsub_mask_stats_local(self.h, phase, self._s()))

    def mask_device(self, sigmas=2.0):
        import torch
        out = torch.empty((self.n, self.m), dtype=torch.uint8, device="cuda")
        C.check(self.lib.bsub_mask_dev(self.h, float(sigmas), ctypes.c_void_p(out.data_ptr()), self._s()))
        return out


class ShardedLSD:
    """inexact_alm_lsd (flat 3x3 groups), inexact_alm_rpca (l1), inexact_alm_group_sparse_RPCA (l2 blocks, one more all-reduce per
    iteration: the per-(frame, group) sums of squares) or a graph mode -- any graph, with or without the background shrink (the
    prox runs on whole frames after an all-to-all to a frame sharding, _prox_on_frames) -- over `comm.world` shards; the step
    solver decides which.  A step solver with a `frame_range` must describe the frames shard_frames gives this rank.  hooks: optional callbacks
    hooks[name](phase) with phase in {'begin', 'end'} around 'gram', 'solve', 'shrink' for timing."""

    def __init__(self, solver, comm, run_ahead=3, max_iter=500, fence=None):
        self.s, self.comm, self.run_ahead, self.max_iter = solver, comm, max(1, int(run_ahead)), max_iter
        # callable(iteration) -> object with .synchronize(); bounds host run-ahead.  Mandatory for a device-side solver.
        if fence is None and getattr(solver, "needs_fence", False):
            fence = cuda_fence
        self.fence = fence
        self.iters_enqueued = 0
        fr = getattr(solver, "frame_range", None)           # the frames this rank's prox gets from the exchange
        if fr is not None and tuple(fr) != shard_frames(solver.n, comm.world, comm.rank):
            raise Exception("ShardedLSD: the step solver describes frames [%d, %d), but rank %d of %d owns [%d, %d) (shard_frames)"
                            % ((fr[0], fr[1], comm.rank, comm.world) + shard_frames(solver.n, comm.world, comm.rank)))

    def solve(self, hooks=None):
        s, comm = self.s, self.comm
        hk = hooks or (lambda name, phase: None)
        s.init_local()
        comm.all_reduce_sum(s.gram_view())
        comm.all_reduce_max(s.max_view())
        s.init_finish()
        fences = []
        self.iters_enqueued = 0
        # body `it` (0-based): Gram of iteration it+1 | all-reduce(Gram + scalars of iteration it) | stop test of iteration it |
        # eigensolve and shrink of iteration it+1.  One more body than iterations: the last one only closes iteration max_iter.
        for it in range(self.max_iter + 1 + self.run_ahead):
            if it >= self.run_ahead:
                closed = it - self.run_ahead            # iterations whose stop test is known to have run
                if self.fence is not None:
                    fences[closed].synchronize()
                if closed >= 1 and s.done_by(closed):
                    break
            hk('gram', 'begin'); s.gram(); comm.all_reduce_sum(s.sum_view())
            if it >= 1:
                s.finish_iter()
            hk('gram', 'end')
            hk('solve', 'begin'); s.solve(); hk('solve', 'end')
            if hooks is not None and hasattr(s, 'project'):      # timed runs: the projection as a phase of its own
                hk('project', 'begin'); s.project(); hk('project', 'end')
            hk('shrink', 'begin')
            bs = s.block_sums_view() if hasattr(s, 'block_sums_view') else None
            gs = s.graph_split() if hasattr(s, 'graph_split') else None
            if gs is not None:                  # overlapping windows: the prox of a frame needs the whole image
                s.shrink_a(); self._prox_on_frames(gs); s.shrink_b()
            elif bs is None:
                s.shrink()
            else:                               # l2 blocks: the groups span the shards (group_sparse_RPCA.py:29-40)
                s.shrink_a(); comm.all_reduce_sum(bs); s.shrink_b()
            hk('shrink', 'end')
            if self.fence is not None:
                fences.append(self.fence(it))
            self.iters_enqueued += 1
        if getattr(s, "lazy_S", False) and s.needs_restart():
            s.store_S_always()
            return self.solve(hooks)
        return self

    def _prox_on_frames(self, geometry):
        """G_S is sharded by pixel columns, the overlapping-window prox couples the pixels of a frame but not the frames: all-to-all
        to a FRAME sharding (rank r gets whole frames [f0_r, f1_r)), prox, all-to-all back into S.  Exact (no halo approximation);
        3 x the shard per rank over NVLink per iteration, small against the prox itself."""
        s, comm = self.s, self.comm
        rows, cols = geometry
        W, r = comm.world, comm.rank
        U, S = s.prox_buffers()                                  # [n][m_local]
        n = U.shape[0]
        f0, f1 = shard_frames(n, W, r)
        nf = f1 - f0
        if W == 1:
            s.prox_frames(U, S, rows, cols, nf)
            return
        cr = [shard_columns(cols, W, q) for q in range(W)]
        fr = [shard_frames(n, W, q) for q in range(W)]
        m_full = rows * cols
        ldf = (m_full + 31) // 32 * 32
        Uf, Vf = s.frames_like(nf, ldf), s.frames_like(nf, ldf)
        # S travels too: once the solve has stopped (the host runs a few iterations ahead of the device-side flag) the prox kernel
        # returns at its first line, and what comes back must then be the S that is already there
        for src, dst in ((U, Uf), (S, Vf)):
            send = [src[a:b, :].contiguous() for a, b in fr]
            recv = [U.new_empty((nf, (c1 - c0) * rows)) for c0, c1 in cr]
            comm.exchange(recv, send)
            for (c0, c1), t in zip(cr, recv):
                dst[:nf, c0 * rows:c1 * rows] = t
        s.prox_frames(Uf, Vf, rows, cols, nf)
        send = [Vf[:nf, c0 * rows:c1 * rows].contiguous() for c0, c1 in cr]
        recv = [U.new_empty((b - a, U.shape[1])) for a, b in fr]
        comm.exchange(recv, send)
        for (a, b), t in zip(fr, recv):
            S[a:b, :] = t

    def finish(self, sigmas=2.0, want_mask=True):
        s, comm = self.s, self.comm
        s.finalize()
        if not want_mask:
            return None
        s.mask_stats(0)
        comm.all_reduce_max(s.max_view())
        s.mask_stats(1)
        comm.all_reduce_sum(s.mask_tail_view())
        return s.mask_device(sigmas)


def cuda_fence(_it):
    import torch
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream())
    return ev
