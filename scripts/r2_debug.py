"""Round-2 debugging probe (GPU): isolates three parity questions with environment toggles."""
import os, sys, json
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import background_subtraction_b200 as B
from background_subtraction_b200 import synth
from oracle import alm_oracle as O

def rel(a, b): return float(np.linalg.norm(a - b) / np.linalg.norm(b))

def with_env(env, fn):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return fn()
    finally:
        for k, v in old.items():
            if v is None: os.environ.pop(k, None)
            else: os.environ[k] = v

# ---- 1. generic groups, one iteration
ws = np.asfortranarray(np.load("tests/golden/watersurface_u8.npz")["ImData"])
D, _x, _m = O.normalize_and_center(ws[:40, :50, :12])
groups = O.flat_groups_nonoverlap((40, 50), (4, 2))
m, n = D.shape
lam = 1.0 / (np.sqrt(max(m, n)) * 10)
norm_two = np.linalg.norm(D, 2); dual = max(norm_two, np.linalg.norm(D, np.inf) / lam); mu = 12.5 / norm_two
Y0 = D / dual
u, s, vh = np.linalg.svd(D + Y0 / mu, full_matrices=False)
svp, _ = O.rank_logic(s[:10], 10, mu, min(m, n))
Lr = (u[:, :svp] * (s[:svp] - 1 / mu)) @ vh[:svp, :]
Sr = O.prox_flat(D - Lr + Y0 / mu, lam / mu, groups)
olog = []
O.inexact_alm_lsd(D, groups=groups, log=olog, max_iter=1)
print("oracle it1: svp", olog[0]['svp'], "mine", svp, "sigma*mu", np.round(olog[0]['sigma'] * mu, 4))
for env in ({}, {"BSUB_NO_I8": "1"}, {"BSUB_NO_STREAM": "1", "BSUB_NO_I8": "1"}):
    def run():
        dec = B.lsd_decomposition(D, groups=groups, max_iter=1)
        st = dec.status()
        return st.iter, st.svp, rel(dec.download('S'), Sr), rel(dec.download('L'), Lr), rel(dec.download('Y'), Y0 + mu * (D - Lr - Sr))
    print("generic groups", env, "iter, svp, relS, relL, relY:", with_env(env, run))

# ---- 2. n = 600 last-iteration rank
video, _ = synth.make_clip(48, 60, 600, seed=33, n_rect=2)
D6 = np.asfortranarray(synth.preprocess_u8(video).T.astype(np.float64))
g6 = B.get_proximal_flat_groups_nonoverlap((48, 60), (3, 3))
olog = []
O.inexact_alm_lsd(D6, groups=g6, log=olog)
print("oracle n600 svp", [l['svp'] for l in olog])
for l in olog[-3:]:
    print("  oracle iter", l['iter'], "sigma*mu", np.round(l['sigma'] * l['mu'], 5))
for env in ({}, {"BSUB_NO_EIG_FAST": "1"}, {"BSUB_NO_I8": "1"}, {"BSUB_NO_FLAT": "1"}, {"BSUB_NO_PROJ": "1"}):
    def run():
        dec = B.lsd_decomposition(D6, groups=g6, img_shape=(48, 60))
        return [l['svp'] for l in dec.log()], dec.counters()
    print("n600", env, with_env(env, run))

# ---- 3. WaterSurface delta = 1
Dw, _x, _m = O.normalize_and_center(ws)
gw = B.get_proximal_flat_groups_nonoverlap((128, 160), (3, 3))
for env in ({}, {"BSUB_NO_EIG_FAST": "1"}, {"BSUB_NO_I8": "1"}):
    def run():
        dec = B.lsd_decomposition(Dw, groups=gw, delta=1)
        lg = dec.log()
        return dec.status().iter, [l['svp'] for l in lg], ["%.4e" % l['err'] for l in lg[-3:]], dec.counters()
    print("ws delta1", env, with_env(env, run))
