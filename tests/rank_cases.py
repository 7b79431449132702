"""Seeded clips whose ALM solves climb or fall through the rank bands that choose the shrink kernel (common.cuh).

The solver picks its shrink route on the device from the rank svp of each iteration: <= 8 takes the single-pass kernel
(shrink_flat.cu) once the digit planes of W exist, 9..16 the streamed kernel (shrink_stream.cu), reading T = Vr^T W from
project.cu when the planes exist, and > 16 the TMA cluster kernel (shrink_tma.cu), which writes no planes.  Each case below
records which bands and band changes its float64 oracle run visits; tests/test_host_rank_routes.py checks those claims and the
distance of every rank decision from its threshold, so that a device solve of a case can be held to the oracle's exact rank
sequence.

Clip: D = sum_k r^k img_k t_k^T (img_k a smooth random image of unit norm, t_k a random unit vector over the frames), scaled to
||D||_2 = 40, plus rectangles of 0.4 moving down one row per frame, rounded to float32.
"""
import numpy as np
from scipy.ndimage import gaussian_filter

BANDS = ("<=8", "9-16", ">16")


def band(svp):
    return BANDS[0] if svp <= 8 else (BANDS[1] if svp <= 16 else BANDS[2])


def make_clip(rows, cols, n, seed, K=24, r=0.85, n_rect=3, norm_two=40.0):
    """m x n float64 (values exactly representable in float32), pixels in F order."""
    rng = np.random.default_rng(seed)
    m = rows * cols
    D = np.zeros((m, n))
    for k in range(K):
        img = gaussian_filter(rng.standard_normal((rows, cols)), 2, mode='wrap').flatten(order='F')
        t = rng.standard_normal(n)
        D += r ** k * np.outer(img / np.linalg.norm(img), t / np.linalg.norm(t))
    D *= norm_two / np.linalg.norm(D, 2)
    cube = D.reshape(rows, cols, n, order='F')
    for _ in range(n_rect):
        h, w = rng.integers(rows // 8, rows // 4 + 1), rng.integers(cols // 8, cols // 4 + 1)
        i0, j0 = rng.integers(0, rows - h), rng.integers(0, cols - w)
        for f in range(n):
            i = (i0 + f) % (rows - h)
            cube[i:i + h, j0:j0 + w, f] += 0.4
    return np.asfortranarray(cube.reshape(m, n, order='F').astype(np.float32).astype(np.float64))


# mode: 'l1' = inexact_alm_rpca (rho 1.2, no rank prediction: sv = d), 'flat' = inexact_alm_lsd with 3x3 flat groups and the
# first rank guess sv0; max_iter: where the solve is stopped (default: it converges).  bands: the set of bands the solve
# visits; transitions: the band changes it makes (from, to); final: the band of the rank L is built from.
#
# No case jumps from rank <= 8 in an iteration >= 2 straight to > 16 (the rebuild of a stale S before the TMA kernel in
# solver.cu): neither the geometric spectra below nor a few two-level ones (2 or 4 strong components over 16 at 0.3 of their
# weight) produced it under l1; the largest jump seen was 4 -> 11.  Flat LSD cannot make it below 170 frames: with rank
# prediction an iteration looks at sv <= svp_prev + round(0.05 d) singular values, so svp_prev <= 8 caps the next rank at 16
# whatever sv0 and delta are.
CASES = {
    "l1_climb": dict(mode="l1", shape=(48, 60, 40), seed=1, clip=dict(),
                     bands={"<=8", "9-16", ">16"}, transitions={("<=8", "9-16"), ("9-16", ">16")}, final=">16"),
    "l1_climb_odd_m": dict(mode="l1", shape=(47, 61, 40), seed=2, clip=dict(),
                           bands={"<=8", "9-16", ">16"}, transitions={("<=8", "9-16"), ("9-16", ">16")}, final=">16"),
    # 300 frames: three 128-frame blocks in the int8 Gram and the 8-CTA eigensolver over all 300 eigenpairs; stopped after
    # 12 iterations (the rank keeps climbing to ~50 and later decisions come within 1e-3 of their threshold)
    "l1_climb_n300": dict(mode="l1", shape=(48, 60, 300), seed=3, clip=dict(n_rect=1), max_iter=12,
                          bands={"<=8", "9-16", ">16"}, transitions={("<=8", "9-16"), ("9-16", ">16")}, final=">16"),
    "flat_descent": dict(mode="flat", sv0=20, shape=(48, 60, 40), seed=0, clip=dict(r=0.75, n_rect=1),
                         bands={">16", "9-16", "<=8"}, transitions={(">16", "9-16"), ("9-16", "<=8")}, final="<=8"),
    "flat_mid": dict(mode="flat", sv0=20, shape=(48, 60, 40), seed=0, clip=dict(r=0.75),
                     bands={">16", "9-16"}, transitions={(">16", "9-16")}, final="9-16"),
    "flat_high": dict(mode="flat", sv0=20, shape=(48, 60, 40), seed=0, clip=dict(r=0.93, K=28),
                      bands={">16"}, transitions=set(), final=">16"),
}


def clip_of(case):
    rows, cols, n = case["shape"]
    return make_clip(rows, cols, n, case["seed"], **case["clip"])


def oracle_solve(case, D, max_iter=None, log=None):
    """The float64 oracle loop of the case's mode -> (L, S, iterations, converged, Y)."""
    from oracle import alm_oracle as O
    if max_iter is None:
        max_iter = case.get("max_iter", 500)
    rows, cols, _n = case["shape"]
    if case["mode"] == "l1":
        def prox(G, lam, mu):
            return np.sign(G) * np.maximum(np.abs(G) - lam / mu, 0)
        return O._alm(D, prox, 1.25, 1.0, rho=1.2, use_sv_prediction=False, max_iter=max_iter, log=log, return_Y=True)
    groups = O.flat_groups_nonoverlap((rows, cols), (3, 3))

    def prox(G, lam, mu):
        return O.prox_flat(G, lam / mu, groups)
    return O._alm(D, prox, 12.5, 10, sv0=case["sv0"], max_iter=max_iter, log=log, return_Y=True)


def boundary_margin(log):
    """Per iteration, min |sigma_i mu - 1| over i in {svp - 1, svp}: how far the rank decision is from flipping."""
    out = []
    for entry in log:
        s, mu, svp = entry["sigma"], entry["mu"], entry["svp"]
        out.append(min(abs(s[i] * mu - 1) for i in (svp - 1, svp) if 0 <= i < s.size))
    return out


def band_changes(svp):
    """1-based iterations whose rank lies in another band than the rank of the iteration before."""
    return [k + 1 for k in range(1, len(svp)) if band(svp[k]) != band(svp[k - 1])]
