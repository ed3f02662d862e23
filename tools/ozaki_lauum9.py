"""[profiles/ozaki_lauum9_r2s.log is the record of this script when the nine-digit product ran as three diagonal windows, with a
128 x 256-tile variant for the tenth diagonal; both are retired, the product now runs as two windows, see csrc/ozaki_i8.cuh.]
The W^T W product of the inverse (lauum) on the INT8 tensor cores with NINE 7-bit digits:
accuracy of NLML + gradient vs the committed N = 32768 oracle golden and stage times.   python tools/ozaki_lauum9.py"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "gaussianprocessregression.jl_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
from gpr_sm100a import _ffi
import make_golden_config3 as m3

ctx = _ffi.get_context()
rng = np.random.default_rng(5)
# raw product check first: W^T W of a well-conditioned upper-triangular-ish matrix, 9 digits vs FP64
for n in (2048,):
    A = rng.standard_normal((n, n))
    A2 = A * np.exp(rng.uniform(-8, 0, (n, 1)))          # rows spanning e^-8 .. 1 under one scale per column (what W looks like)
    for name, M in (("gauss", A), ("row-decay", A2)):
        ref = M.T @ M
        for S in (8, 9):
            Cm, ms = _ffi.dbg_ozaki_dgemm(ctx, 1.0, M, M, 0.0, np.zeros((n, n)), S=S, flags=0)
            print(f"raw A^T A ({name}) n={n} S={S}: max err / max|C| {np.abs(Cm - ref).max() / np.abs(ref).max():.2e}  ({ms:.3f} ms)", flush=True)
n = 8192
A = rng.standard_normal((n, n))
for S, fl in ((8, 0), (9, 0), (9, 3)):
    Cm, ms = _ffi.dbg_ozaki_dgemm(ctx, 1.0, A, A, 0.0, np.zeros((n, n)), S=S, flags=fl, reps=5)
    print(f"timing 8192^3 S={S} flags={fl}: {ms:.3f} ms -> {2 * n ** 3 / ms / 1e9:.1f} TFLOP/s FP64-equivalent (full product count)", flush=True)
g = np.load(os.path.join(ROOT, "tests", "golden", "config3_n32768.npz"))
x, y, hp = m3.inputs()
mh = _ffi.ModelHandle(ctx, [1, 1, 2], 8, x, y)
for lau, pan in ((0, 32768), (9, 32768), (9, 8192)):
    ctx.set_option("ozaki", -1)
    ctx.set_option("ozaki_lauum", lau)
    ctx.set_option("ozaki_panel", pan)
    mh.nlml_grad(hp * 1.001)
    F, G = mh.nlml_grad(hp)
    t = mh.timings()
    relF = abs(F - float(g["F"])) / abs(float(g["F"]))
    relG = float((np.abs(G - g["G"]) / np.maximum(np.abs(g["G"]), 1e-8 * np.linalg.norm(g["G"]))).max())
    print(f"ozaki_lauum={lau} panel={pan}: eval {t['eval']:.1f} ms (potrf {t['potrf']:.1f}, trtri {t['trtri']:.1f}, lauum {t['lauum']:.1f}); "
          f"vs oracle: relF {relF:.2e} relG {relG:.2e}", flush=True)
ctx.set_option("ozaki_lauum", 9)
ctx.set_option("ozaki_panel", 32768)
mh.close()
