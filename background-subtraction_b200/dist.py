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


def columns_to_frames(comm, src, dst, rows, cols):
    """all-to-all from the column sharding to the frame sharding: src [n][rows * cols_local] holds this rank's pixel columns
    (shard_columns) of every frame; rows [0, nf) of dst [>= nf][>= rows * cols] receive the whole frames shard_frames gives this rank."""
    W = comm.world
    n = src.shape[0]
    cr = [shard_columns(cols, W, q) for q in range(W)]
    fr = [shard_frames(n, W, q) for q in range(W)]
    nf = fr[comm.rank][1] - fr[comm.rank][0]
    send = [src[a:b, :].contiguous() for a, b in fr]
    recv = [src.new_empty((nf, (c1 - c0) * rows)) for c0, c1 in cr]
    comm.exchange(recv, send)
    for (c0, c1), t in zip(cr, recv):
        dst[:nf, c0 * rows:c1 * rows] = t


def frames_to_columns(comm, src, dst, rows, cols):
    """The way back: rows [0, nf) of src hold this rank's whole frames (shard_frames); dst [n][rows * cols_local] receives this rank's
    pixel columns of every frame."""
    W = comm.world
    n = dst.shape[0]
    cr = [shard_columns(cols, W, q) for q in range(W)]
    fr = [shard_frames(n, W, q) for q in range(W)]
    nf = fr[comm.rank][1] - fr[comm.rank][0]
    send = [src[:nf, c0 * rows:c1 * rows].contiguous() for c0, c1 in cr]
    recv = [dst.new_empty((b - a, dst.shape[1])) for a, b in fr]
    comm.exchange(recv, send)
    for (a, b), t in zip(fr, recv):
        dst[a:b, :] = t


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
          weight_mask = [h, w, t] map of build_improved_LSD_graphs: center_window_decomposition (LSD_improved's second pass);
          or, with graph_cols, a CUDA float32 tensor [f1 - f0][rows * graph_cols] holding only the map of `frames`, already on the
          device (bsub_set_frame_weight_map_dev; what ShardedLSDImproved builds).
        l1=True: inexact_alm_rpca (elementwise soft threshold, /root/reference/lsd_improvement.py:123-196: delta 1.0, mu0 =
        1.25 / ||D||_2, rho 1.2, no sv prediction), which shards without any exchange.  Default: flat 3x3 l_inf groups (LSD)."""
        if sum(x is not None for x in (blocks, graphs, weight_mask)) + bool(l1) > 1:
            raise Exception("CudaStepSolver: blocks, graphs, weight_mask and l1 are mutually exclusive")
        if background_masks is not None and graphs is None:
            raise Exception("CudaStepSolver: background_masks needs graphs")
        route = None
        frame_map = api._is_torch(weight_mask)
        if frame_map:
            if graph_cols is None:
                raise Exception("CudaStepSolver: a device weight_mask of the rank's frames needs graph_cols")
            route = api.GraphRoute(C.PROX_GRAPH_CENTER_BG, rows, graph_cols)
        elif weight_mask is not None:
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
            if frame_map:
                f0, f1 = self.frame_range
                if int(weight_mask.shape[0]) != f1 - f0:
                    raise Exception("CudaStepSolver: the device weight_mask has %d frames, frames = [%d, %d)"
                                    % (int(weight_mask.shape[0]), f0, f1))
                self.dec.set_frame_weight_map(weight_mask, rows, graph_cols, f0)
            else:
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
        m_full = rows * cols
        ldf = (m_full + 31) // 32 * 32
        Uf, Vf = s.frames_like(nf, ldf), s.frames_like(nf, ldf)
        # S travels too: once the solve has stopped (the host runs a few iterations ahead of the device-side flag) the prox kernel
        # returns at its first line, and what comes back must then be the S that is already there
        columns_to_frames(comm, U, Uf, rows, cols)
        columns_to_frames(comm, S, Vf, rows, cols)
        s.prox_frames(Uf, Vf, rows, cols, nf)
        frames_to_columns(comm, Vf, S, rows, cols)

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


class CudaImprovedOps:
    """What ShardedLSDImproved computes with on this GPU: the step solvers of the two passes, the per-frame morphology and merge,
    and the results.  The gloo tests substitute NumPy stand-ins (same methods) so that the driver's own code runs on CPU ranks."""

    device = "cuda"

    def matrix(self, D):
        """D shard, [n][m_local] frame-major (NumPy float64 or torch) -> the float32 device copy both passes load."""
        import torch
        if api._is_torch(D):
            return D.to(device="cuda", dtype=torch.float32).contiguous()
        # rounded to float32 on the host (round to nearest, as the device conversion of bsub_load_D_f64_host): half the bytes to copy
        return torch.from_numpy(np.ascontiguousarray(D, dtype=np.float32)).to("cuda")

    def pass1(self, D, rows, cols_local, n, m_global, alg_ver):
        """improved_LSD_weight_mask's first solve: inexact_alm_lsd on the flat 3x3 groups at delta 1.0 (alg_ver 2) or
        inexact_alm_rpca at delta 10.0 (alg_ver 1)."""
        s = CudaStepSolver(rows, cols_local, n, m_global, delta=10.0 if alg_ver == 1 else 1.0, l1=alg_ver == 1)
        s.load(D)
        return s

    def pass2(self, D, rows, cols_local, n, m_global, cols, frames, weight):
        """center_window_decomposition (delta 10) of the frame range `frames` described by weight [nf][rows * cols]."""
        s = CudaStepSolver(rows, cols_local, n, m_global, graph_cols=cols, weight_mask=weight, frames=frames)
        s.load(D)
        return s

    def summary(self, s):
        """(iterations, converged, rank of L per iteration) of a finished solve."""
        st = s.status()
        return int(st.iter), bool(st.converged), [l['svp'] for l in s.dec.log()]

    def close(self, s):
        s.dec.close()

    def weight_map(self, mask, rows, cols, disk_ratio, weights):
        """merge_masks((S_mask, apply_morph_ops(S_mask, disk_ratio)), weights) on the frames of mask (uint8 [nf][rows * cols], on the
        device) -> (float32 [nf][rows * cols] map, -1 = background; number of its positive entries)."""
        import torch
        from . import flow
        nf = int(mask.shape[0])
        if nf == 0:
            return torch.empty((0, rows * cols), dtype=torch.float32, device="cuda"), 0
        morph = flow.morph_frames_dev(mask, rows, cols, flow.disk_radius('disk', disk_ratio * rows))
        out = torch.where(mask != 0, float(weights[0]), torch.where(morph != 0, float(weights[1]), -1.0)).to(torch.float32)
        return out, int((out > 0).sum())

    def outputs(self, s, mask, rows, cols_local, n, like):
        """(S [rows * cols_local, n], S_mask [rows, cols_local, n] bool, L [rows, cols_local, n]) as LSD_improved returns them:
        torch CUDA tensors for a torch input, else NumPy (float64 L / S)."""
        shape = (rows, cols_local, n)
        S_mask = mask.view(n, cols_local, rows).permute(2, 1, 0) != 0
        if api._is_torch(like):
            L = s.dec.device_tensor('L').clone().t()
            S = s.dec.device_tensor('S').clone().t()
            return S, S_mask, L.reshape(cols_local, rows, n).permute(1, 0, 2)
        return s.dec.download('S'), np.ascontiguousarray(S_mask.cpu().numpy()), s.dec.download('L').reshape(shape, order='F')


class ShardedLSDImproved:
    """flow.LSD_improved (/root/reference/lsd_improvement.py:441-487) over `comm.world` GPUs, one call of run() per rank on the rank's
    image columns shard_columns(w, world, rank) of the [h, w, t] clip:
      pre-processing   normalizeImage and the mean from three all-reduces (MAX of -min, MAX of the shifted max, SUM);
      pass 1           ShardedLSD on the column shard (flat 3x3 at delta 1.0, or l1 at delta 10.0) and its foreground mask;
      columns->frames  one all-to-all of the uint8 mask: this rank gets whole frames shard_frames(t, world, rank);
      back-off         morphology, merge and the mask-percentage back-off (flow.mask_backoff) on those frames, with one all-reduce
                       of the positive count per step: every rank takes the same steps;
      pass 2           the centre-window solve of ShardedLSD, its prox described by exactly the weight map of those frames (device
                       tensor, no host round trip), and its mask.
    The disk morphology couples neighbouring columns but not frames, so the frame sharding is exact: no halo, no approximation.  A
    rank with no frame (t < world) takes part in every collective.  `ops` supplies the solvers and the per-frame work
    (CudaImprovedOps); the choreography does not know whether it drives CUDA or NumPy.  After run(): weight_frames = this rank's
    frames of the weight map (float32 [nf][h * w]), frames = (f0, f1), pass1_log / pass2_log = (iterations, converged, ranks)."""

    def __init__(self, comm, ops=None, run_ahead=3):
        self.comm, self.ops, self.run_ahead = comm, ops if ops is not None else CudaImprovedOps(), run_ahead
        self.weight_frames = self.frames = self.pass1_log = self.pass2_log = None

    def _all_reduce(self, value, op, dtype):
        import torch
        buf = torch.tensor([value], dtype=dtype, device=self.ops.device)
        op(buf)
        return buf.item()

    def run(self, cube, shape, alg_ver=2, downsample_ratio=1, hooks=None):
        """cube: this rank's columns [h, cols_local, t] (NumPy, normalised in place like the reference does, or a torch tensor);
        shape: (h, w, t) of the whole clip.  hooks(name, 'begin' | 'end') around 'pre', 'pass1', 'mask', 'backoff', 'pass2',
        'final_mask'.  Returns (S, S_mask, L_recon, ImData1, ImMean, shape, iterations, converged, graph_iter, graph_converged) of
        LSD_improved, restricted to this rank's columns (ImMean and shape are the whole clip's)."""
        import torch
        from . import flow
        comm, ops = self.comm, self.ops
        hk = hooks or (lambda name, phase: None)
        if downsample_ratio != 1:
            raise Exception("ShardedLSDImproved: downsample_ratio must be 1 (resizing couples columns: resize the clip first)")
        if alg_ver not in (1, 2):
            raise Exception("LSD_improved wrong alg ver")
        h, w, t = (int(v) for v in shape)
        c0, c1 = shard_columns(w, comm.world, comm.rank)
        cl = c1 - c0
        if tuple(int(v) for v in cube.shape) != (h, cl, t):
            raise Exception("ShardedLSDImproved: rank %d of %d owns columns [%d, %d) of the %d, so its cube must be [%d, %d, %d], not %s"
                            % (comm.rank, comm.world, c0, c1, w, h, cl, t, tuple(cube.shape)))
        on_torch = api._is_torch(cube)
        hk('pre', 'begin')
        x = cube.to(torch.float64) if on_torch else np.asarray(cube, dtype=np.float64)
        lo = -self._all_reduce(-float(x.min()), comm.all_reduce_max, torch.float64)
        x -= lo
        hi = self._all_reduce(float(x.max()), comm.all_reduce_max, torch.float64)
        x *= 1.0 / hi
        mean = self._all_reduce(float(x.sum()), comm.all_reduce_sum, torch.float64) / (h * w * t)
        x2 = x - mean
        D = ops.matrix(x2.permute(2, 1, 0).reshape(t, cl * h) if on_torch else np.ascontiguousarray(x2.transpose(2, 1, 0)).reshape(t, cl * h))
        del x2
        hk('pre', 'end')

        hk('pass1', 'begin')
        s1 = ops.pass1(D, h, cl, t, h * w, alg_ver)
        drv = ShardedLSD(s1, comm, run_ahead=self.run_ahead)
        drv.solve()
        hk('pass1', 'end')
        hk('mask', 'begin')
        mask = drv.finish(2.0)                                  # [t][h * cl] uint8
        self.pass1_log = ops.summary(s1)
        ops.close(s1)
        del s1, drv
        f0, f1 = self.frames = shard_frames(t, comm.world, comm.rank)
        if comm.world == 1:
            mask_f = mask
        else:
            mask_f = mask.new_zeros((max(f1 - f0, 1), h * w))
            columns_to_frames(comm, mask, mask_f, h, w)
            mask_f = mask_f[:f1 - f0]
        hk('mask', 'end')

        hk('backoff', 'begin')

        def weight_for(disk_ratio):
            wf, count = ops.weight_map(mask_f, h, w, disk_ratio, (1, 1.5))
            return wf, int(self._all_reduce(int(count), comm.all_reduce_sum, torch.int64))
        self.weight_frames = flow.mask_backoff(weight_for, h, h * w * t)
        hk('backoff', 'end')

        hk('pass2', 'begin')
        s2 = ops.pass2(D, h, cl, t, h * w, w, (f0, f1), self.weight_frames)
        drv = ShardedLSD(s2, comm, run_ahead=self.run_ahead)
        drv.solve()
        hk('pass2', 'end')
        hk('final_mask', 'begin')
        mask2 = drv.finish(2.0)
        self.pass2_log = ops.summary(s2)
        S, S_mask, L_recon = ops.outputs(s2, mask2, h, cl, t, cube)
        hk('final_mask', 'end')
        it, conv, _ = self.pass2_log
        git, gconv, _ = self.pass1_log
        return S, S_mask, L_recon, x, mean, (h, w, t), it, conv, git, gconv


def cuda_fence(_it):
    import torch
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream())
    return ev
