"""Batched epilogue of the INT8 kernels (ctx option ozaki_epi = 1; launch flag 16384 = the first, column-serial form) against the serial one:
  1. isolated products in every form the dbg entry reaches: BIT-identical results, and the time of a large product with beta != 0;
  2. the tile-mapped forms (GEMM_MAP_UPPER / KUPTO) through the block-cyclic driver with 2 ranks on one device: identical F, G;
  3. one model (config 2 golden, N = 8192): F, G, predictive mean / variance and the split-predict mean (Hadamard epilogue) identical
     between the two forms, F and G against the committed oracle golden;
  4. the benchmark model (N = 32768): evaluation time with the option off / on, F and G identical, against the oracle golden.
python tools/oz_epi_check.py

NEEDS profiles/ozaki_batched_epilogue_r2ar.patch applied (git apply) and a rebuild: the shipped library has the serial epilogue only and no
"ozaki_epi" option.  Record of the one run: profiles/ozaki_batched_epilogue_check_r2ar.log; reading in DESIGN.md section 9."""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "gaussianprocessregression.jl_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
from gpr_sm100a import _ffi

t00 = time.time()
SER = 16384
ctx = _ffi.get_context()
rng = np.random.default_rng(31)
bad = 0
# ---- 1. isolated products ----
cases = []
for beta in (0.0, 0.5):
    for (M, N, K, S, fl) in ((256, 384, 640, 8, 0), (512, 512, 1024, 8, 1), (384, 384, 384, 8, 1 | 2), (512, 512, 512, 8, 64), (512, 512, 512, 8, 1 | 64),
                             (512, 640, 1024, 7, 0), (256, 256, 512, 6, 0),
                             (512, 512, 1024, 8, 512), (768, 512, 1024, 8, 512 | 1), (1024, 1024, 1024, 8, 512 | 1 | 2), (512, 512, 640, 8, 512 | 64),
                             (640, 640, 1024, 9, 0), (640, 640, 640, 9, 1 | 2)):
        cases.append((M, N, K, S, fl, beta))
for (M, N, K, S, fl, beta) in cases:
    if fl & 2:
        A = np.tril(rng.standard_normal((K, M)))
        for J in range(M // 128):
            A[:128 * J, 128 * J:128 * (J + 1)] = 1e30
        B = A
    elif S == 9:
        A = rng.standard_normal((K, M)) * np.exp(rng.uniform(-8, 0, (K, M)))
        B = A
    else:
        A, B = rng.standard_normal((K, M)), rng.standard_normal((K, N))
    A, B = np.asfortranarray(A), np.asfortranarray(B)
    C0 = np.asfortranarray(rng.standard_normal((M, N)))
    C1, _ = _ffi.dbg_ozaki_dgemm(ctx, -1.0, A, B, beta, C0, S=S, flags=fl | SER)
    C2, _ = _ffi.dbg_ozaki_dgemm(ctx, -1.0, A, B, beta, C0, S=S, flags=fl)
    ok = bool(np.array_equal(C1, C2))
    bad += not ok
    if not ok:
        print(f"MISMATCH M={M} N={N} K={K} S={S} flags={fl} beta={beta}: max diff {np.abs(C1 - C2).max():.3e}", flush=True)
print(f"1. {len(cases)} isolated products, serial vs batched epilogue: {'all bit-identical' if bad == 0 else str(bad) + ' MISMATCHES'}  [{time.time() - t00:.0f} s]", flush=True)
n = 4096
A = np.asfortranarray(rng.standard_normal((n, n)))
C0 = np.asfortranarray(rng.standard_normal((n, n)))
for (S, fl, what) in ((8, 0, "8 digits single pass"), (8, 512, "8 digits two windows"), (9, 0, "9 digits two windows")):
    C1, ms1 = _ffi.dbg_ozaki_dgemm(ctx, -1.0, A, A, 1.0, C0, S=S, flags=fl | SER, reps=3)
    C2, ms2 = _ffi.dbg_ozaki_dgemm(ctx, -1.0, A, A, 1.0, C0, S=S, flags=fl, reps=3)
    same = bool(np.array_equal(C1, C2))
    bad += not same
    print(f"   {n}^3, beta = 1, {what}: serial {ms1:.3f} ms, batched {ms2:.3f} ms ({ms1 / ms2:.3f} x), bit-identical {same}", flush=True)
del A, C0, C1, C2

# ---- 2. tile-mapped forms through the block-cyclic driver (2 ranks on device 0) ----
import make_golden_config2 as mg2

x2, y2, sets = mg2.inputs()
g2 = np.load(os.path.join(ROOT, "tests", "golden", "config2_n8192.npz"))
hpA = sets["A"]
res = {}
for epi in (0, 1):
    mc = _ffi.MultiContext([0, 0], nb=1024)
    mc.set_option("ozaki", 8)
    mc.set_option("ozaki_kchunk", 2048)
    mc.set_option("ozaki_epi", epi)
    mm = _ffi.MultiModelHandle(mc, [1, 2], 8, x2, y2)
    res[epi] = mm.nlml_grad(hpA)
    mm.close(); mc.close()
same = res[0][0] == res[1][0] and bool(np.array_equal(res[0][1], res[1][1]))
bad += not same
relF = abs(res[1][0] - float(g2["F_A"])) / abs(float(g2["F_A"]))
relG = float((np.abs(res[1][1] - g2["G_A"]) / np.maximum(np.abs(g2["G_A"]), 1e-8 * np.linalg.norm(g2["G_A"]))).max())
print(f"2. block-cyclic driver, 2 ranks, INT8 tile-mapped forms (N = 8192): F, G identical between the epilogues {same}; vs oracle relF {relF:.2e} relG {relG:.2e}  [{time.time() - t00:.0f} s]",
      flush=True)

# ---- 3. one model, every product path of the single-GPU handle ----
out = {}
xp = np.asfortranarray(rng.random((8, 4096)))
xe, xq = np.asfortranarray(0.5 * rng.random((8, 1024))), np.asfortranarray(0.5 * rng.random((8, 1024)))
for epi in (0, 1):
    ctx.set_option("ozaki_epi", epi)
    ctx.set_option("ozaki", 8)
    mh = _ffi.ModelHandle(ctx, [1, 2], 8, x2, y2)
    F, G = mh.nlml_grad(hpA)
    mu, var, _ = mh.predict(xp, want_var=True)
    ms_, _ = mh.split_predict(xe, xq, var_range=None, want_var=False)
    out[epi] = (F, G.copy(), mu.copy(), var.copy(), ms_.copy(), mh.route())
    mh.close()
ctx.set_option("ozaki", -1)
same = out[0][0] == out[1][0] and all(bool(np.array_equal(out[0][i], out[1][i])) for i in (1, 2, 3, 4))
bad += not same
relF = abs(out[1][0] - float(g2["F_A"])) / abs(float(g2["F_A"]))
relG = float((np.abs(out[1][1] - g2["G_A"]) / np.maximum(np.abs(g2["G_A"]), 1e-8 * np.linalg.norm(g2["G_A"]))).max())
print(f"3. model N = 8192 (route {out[1][5]}): F, G, predictive mean, variance, split mean identical between the epilogues {same}; vs oracle relF {relF:.2e} relG {relG:.2e}"
      f"  [{time.time() - t00:.0f} s]", flush=True)

# ---- 4. the benchmark model ----
import make_golden_config3 as m3

g = np.load(os.path.join(ROOT, "tests", "golden", "config3_n32768.npz"))
x, y, hp = m3.inputs()
mh = _ffi.ModelHandle(ctx, [1, 1, 2], 8, x, y)
r4 = {}
for epi in (0, 1, 0):
    ctx.set_option("ozaki_epi", epi)
    mh.nlml_grad(hp * 1.001)
    ts = []
    for rep in range(3):
        F, G = mh.nlml_grad(hp * (1 + 1e-9 * rep) if rep < 2 else hp)
        ts.append(mh.timings())
    t = {k: float(np.mean([q[k] for q in ts])) for k in ts[0]}
    relF = abs(F - float(g["F"])) / abs(float(g["F"]))
    relG = float((np.abs(G - g["G"]) / np.maximum(np.abs(g["G"]), 1e-8 * np.linalg.norm(g["G"]))).max())
    r4.setdefault(epi, (F, G.copy()))
    print(f"4. ozaki_epi={epi}: eval {t['eval']:.1f} ms (potrf {t['potrf']:.1f}, trtri {t['trtri']:.1f}, lauum {t['lauum']:.1f}); relF {relF:.2e} relG {relG:.2e}", flush=True)
same = r4[0][0] == r4[1][0] and bool(np.array_equal(r4[0][1], r4[1][1]))
bad += not same
print(f"   F, G identical between the epilogues: {same}")
mh.close()
print(f"RESULT: {'OK' if bad == 0 else 'FAILED (' + str(bad) + ')'}  [{time.time() - t00:.0f} s]")
sys.exit(1 if bad else 0)
