"""-m gpu: the frame-range centre-window description built on the device from a weight map (bsub_set_frame_weight_map_dev) against
the one built on the host (bsub_set_frame_center_windows), its errors, and LSD_improved through dist.ShardedLSDImproved at world
size 1 against flow.LSD_improved."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import rel_fro

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
H, W, T = 47, 61, 12                                            # H % 3 != 0


@pytest.fixture(scope="module")
def B():
    import background_subtraction_b200 as B
    return B


def _weight_map(seed=3):
    """[h, w, t]: positive window weights, negative background, zeros; frame 4 has no window, frame 7 no background."""
    rng = np.random.default_rng(seed)
    wm = np.zeros((H, W, T))
    for f in range(T):
        r = rng.random((H, W))
        if f != 4:
            wm[:, :, f] = np.where(r < 0.25, rng.uniform(0.5, 3.0, (H, W)), 0.0)
        if f != 7:
            wm[:, :, f] = np.where(r > 0.55, rng.uniform(-2.0, -0.1, (H, W)), wm[:, :, f])
    return wm


def _device_frames(wm, f0, f1, pad=5):
    """frames [f0, f1) of the map as a float32 CUDA tensor [nf][H * W] with a row pitch of H * W + pad"""
    import torch
    flat = np.ascontiguousarray(wm.transpose(2, 1, 0)).reshape(T, H * W)[f0:f1].astype(np.float32)
    big = torch.zeros((f1 - f0, H * W + pad), dtype=torch.float32, device="cuda")
    big[:, :H * W] = torch.from_numpy(flat).cuda()
    return big[:, :H * W]


def _solvers(D, wm, f0, f1):
    """Two initialised step solvers whose prox describes frames [f0, f1): from the host map and from the device map."""
    from background_subtraction_b200 import dist as bdist
    out = []
    for kw in (dict(weight_mask=wm), dict(weight_mask=_device_frames(wm, f0, f1), graph_cols=W)):
        s = bdist.CudaStepSolver(H, W, T, H * W, frames=(f0, f1), **kw)
        s.load(np.ascontiguousarray(D.T, dtype=np.float32))
        s.init_local()
        s.init_finish()
        out.append(s)
    return out


def _prox(s, U, f0, nf):
    import torch
    V = torch.zeros_like(U)
    s.prox_block(U, V, f0, nf)
    torch.cuda.synchronize()
    return V


@pytest.fixture(scope="module")
def D():
    rng = np.random.default_rng(1)
    return np.asfortranarray(rng.standard_normal((H * W, T)) * 0.1)


@pytest.mark.parametrize("f0,f1", [(0, T), (3, 8), (11, T)])
def test_device_map_proxes_like_host_map(B, D, f0, f1):
    import torch
    wm = _weight_map()
    host, dev = _solvers(D, wm, f0, f1)
    nf = f1 - f0
    g = torch.Generator(device="cuda").manual_seed(f0)
    U = torch.randn((nf, H * W + 32), device="cuda", generator=g) * 0.05
    for a, b in ((f0, f1), (f0 + nf // 2, f1)):                # the whole range and a block at its end
        assert torch.equal(_prox(host, U[a - f0:], a, b - a), _prox(dev, U[a - f0:], a, b - a))


def test_non_finite_entry_is_reported_and_old_description_kept(B, D):
    import torch
    wm = _weight_map()
    f0, f1 = 2, 9
    host, dev = _solvers(D, wm, f0, f1)
    U = torch.randn((f1 - f0, H * W), device="cuda") * 0.05
    for bad in (float("nan"), float("inf"), -float("inf")):
        w = _device_frames(wm, f0, f1)
        w[3, 17] = bad
        w[5, 2] = bad                                            # a later bad entry: the first one is reported
        with pytest.raises(Exception, match=r"weight\[3\]\[17\] \(frame 5, pixel 17\) = -?(nan|inf) is not finite"):
            dev.dec.set_frame_weight_map(w, H, W, f0)
        assert torch.equal(_prox(host, U, f0, f1 - f0), _prox(dev, U, f0, f1 - f0))


def test_empty_range_and_bad_arguments(B, D):
    import torch
    from background_subtraction_b200 import _cabi as C
    from background_subtraction_b200 import dist as bdist
    s = bdist.CudaStepSolver(H, W, T, H * W, weight_mask=torch.zeros((0, H * W), device="cuda"), graph_cols=W, frames=(T, T))
    s.load(np.ascontiguousarray(D.T, dtype=np.float32))
    s.init_local()
    s.init_finish()
    U = torch.zeros((1, H * W), device="cuda")
    s.prox_block(U, U, T, 0)
    C.check(s.lib.bsub_set_frame_weight_map_dev(s.h, H, W, 5, 0, None, 0, s._s()))      # nf = 0: no map, any ld
    w = _device_frames(_weight_map(), 0, 2)
    with pytest.raises(Exception, match="ld = %d is less than rows\\*cols" % (H * W - 1)):
        C.check(s.lib.bsub_set_frame_weight_map_dev(s.h, H, W, 0, 2, ctypes.c_void_p(w.data_ptr()), H * W - 1, s._s()))
    with pytest.raises(Exception, match="null argument"):
        C.check(s.lib.bsub_set_frame_weight_map_dev(s.h, H, W, 0, 2, None, H * W, s._s()))
    with pytest.raises(Exception, match=r"frames \[11, 13\) are not a range of the 12 frames"):
        s.dec.set_frame_weight_map(w, H, W, 11)
    with pytest.raises(Exception, match="bad frame geometry"):
        C.check(s.lib.bsub_set_frame_weight_map_dev(s.h, 0, W, 0, 2, ctypes.c_void_p(w.data_ptr()), H * W, s._s()))
    dec = B.Decomposition(B.make_config(H * W, T, C.PROX_GRAPH_LINF, H, W))
    with pytest.raises(Exception, match="not created with BSUB_PROX_GRAPH_CENTER_BG"):
        dec.set_frame_weight_map(w, H, W, 0)
    with pytest.raises(Exception, match="the device weight_mask has 2 frames, frames = \\[0, 12\\)"):
        bdist.CudaStepSolver(H, W, T, H * W, weight_mask=w, graph_cols=W)


class Solo:
    world, rank = 1, 0

    def all_reduce_sum(self, t_):
        pass

    def all_reduce_max(self, t_):
        pass


def _counting_ops():
    """CudaImprovedOps that counts the weight maps the back-off asks for."""
    from background_subtraction_b200 import dist as bdist

    class Ops(bdist.CudaImprovedOps):
        calls = 0

        def weight_map(self, *a):
            self.calls += 1
            return super().weight_map(*a)
    return Ops()


def _single_gpu_logs(B, D, shape, alg_ver, wm):
    """Rank sequences of the two solves flow.LSD_improved runs (the same calls, kept open to read their logs)."""
    from background_subtraction_b200 import _cabi as C
    h, w, t = shape
    if alg_ver == 2:
        dec1 = B.lsd_decomposition(D, groups=B.get_proximal_flat_groups_nonoverlap((h, w), (3, 3)), delta=1.0, img_shape=(h, w))
    else:
        dec1 = B.Decomposition(B.make_config(h * w, t, C.PROX_L1, 0, 0, delta=10.0, mu_scale=1.25, rho=1.2, use_sv_prediction=False))
        dec1.load(D)
        dec1.run()
    dec2 = B.center_window_decomposition(D, wm, img_shape=(h, w))
    return [l['svp'] for l in dec1.log()], [l['svp'] for l in dec2.log()]


def _cases(watersurface_u8):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_dist_gloo_lsd_improved import make_cube
    return {"watersurface": (np.asfortranarray(watersurface_u8[40:88, 50:110, 0:16].astype(np.float64)), 2),
            "dense_backoff": (make_cube(22, 24, 8, dense=True), 1)}


@pytest.mark.parametrize("case", ["watersurface", "dense_backoff"])
def test_driver_at_world_one_matches_LSD_improved(B, watersurface_u8, case):
    import torch
    from background_subtraction_b200 import dist as bdist
    cube, alg_ver = _cases(watersurface_u8)[case]
    shape = cube.shape
    h, w, t = shape
    ref = B.LSD_improved(cube.copy(order='F'), 0, t - 1, 1, alg_ver=alg_ver)
    S0, mask0, L0, im0, mean0, _shp, it0, conv0, git0, gconv0 = ref
    D = (im0 - mean0).reshape((h * w, t), order='F')
    prox, mode = (B.get_proximal_flat_groups_nonoverlap((h, w), (3, 3)), "NONOVERLAPPING_GROUPS") if alg_ver == 2 else (None, None)
    wm0, _i, _c = B.improved_LSD_weight_mask(D, shape, (1, 1.5), delta=1.0, proximal_object=prox, mode=mode)
    svp1, svp2 = _single_gpu_logs(B, D, shape, alg_ver, wm0)

    ops = _counting_ops()
    drv = bdist.ShardedLSDImproved(Solo(), ops=ops)
    S, mask, L, im1, mean, shp, it, conv, git, gconv = drv.run(cube.copy(order='F'), shape, alg_ver)
    torch.cuda.synchronize()
    if case == "dense_backoff":
        assert ops.calls >= 3                              # the back-off took at least two steps
    assert shp == shape and np.array_equal(im1, im0) and mean == mean0
    assert (git, gconv, drv.pass1_log[2]) == (git0, gconv0, svp1)
    assert (it, conv, drv.pass2_log[2]) == (it0, conv0, svp2)
    wf = drv.weight_frames.cpu().numpy()
    assert np.array_equal(wf, np.ascontiguousarray(wm0.transpose(2, 1, 0)).reshape(t, -1))
    assert rel_fro(L, L0) <= 1e-6 and rel_fro(S, S0) <= 1e-6
    assert mask.shape == shape and (mask == mask0).mean() >= 0.9999


def test_driver_on_a_torch_cube_matches_the_numpy_cube(B, watersurface_u8):
    """A CUDA tensor cube: the pre-processing on the device and the outputs as CUDA tensors in LSD_improved's layout.  Only the
    summation order of the mean differs from the NumPy run (ImData1 is bit-identical)."""
    import torch
    from background_subtraction_b200 import dist as bdist
    cube = np.asfortranarray(watersurface_u8[40:88, 50:110, 0:16].astype(np.float64))
    shape = cube.shape
    h, w, t = shape
    ref = bdist.ShardedLSDImproved(Solo())
    S0, mask0, L0, im0, mean0, _s, it0, conv0, git0, gconv0 = ref.run(cube.copy(order='F'), shape, 2)
    drv = bdist.ShardedLSDImproved(Solo())
    S, mask, L, im1, mean, shp, it, conv, git, gconv = drv.run(torch.from_numpy(cube.copy()).cuda(), shape, 2)
    torch.cuda.synchronize()
    assert all(torch.is_tensor(x) and x.is_cuda for x in (S, mask, L, im1))
    assert tuple(S.shape) == (h * w, t) and tuple(mask.shape) == shape and tuple(L.shape) == shape and mask.dtype == torch.bool
    assert shp == shape and np.array_equal(im1.cpu().numpy(), im0) and abs(mean - mean0) <= 1e-15
    assert (it, conv, git, gconv) == (it0, conv0, git0, gconv0)
    assert drv.pass1_log == ref.pass1_log and drv.pass2_log == ref.pass2_log
    assert (drv.weight_frames.cpu().numpy() == ref.weight_frames.cpu().numpy()).mean() >= 0.9999
    assert rel_fro(L.cpu().numpy(), L0) <= 1e-5 and rel_fro(S.cpu().numpy(), S0) <= 1e-5
    assert (mask.cpu().numpy() == mask0).mean() >= 0.9999


def test_two_rank_nccl_lsd_improved_matches_single_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29523", os.path.join(ROOT, "scripts", "check_sharded_improved.py")]
    out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
