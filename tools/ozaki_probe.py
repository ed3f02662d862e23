"""Rate of the INT8 product kernels at 8192^3 (csrc/ozaki_i8.cuh), single CTAs against CTA pairs (tcgen05 cta_group::2, flag 2048),
with the timing probe's no-reload form (flag 256: the k-tiles after the first two reuse the staged digit planes, results are garbage)
beside the real one.  Cycles are per 128 x 64 x 32 of integer work per SM at an assumed 1.965 GHz, i.e. the time of one M128 N64 K32
UTCIMMA of the single-CTA kernel; a pair's M256 instruction does two such units, one on each SM.  The pair forms must return the same
bits as the single-CTA forms."""
import os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "gaussianprocessregression.jl_b200"))
from gpr_sm100a import _ffi
ctx = _ffi.get_context()
rng = np.random.default_rng(0)
n = 8192
A = np.asfortranarray(rng.standard_normal((n, n)))
C0 = np.zeros((n, n), order="F")
PAIR, NORELOAD, WIN = 2048, 256, 512
forms = {8: ((0, "single pass"), (NORELOAD, "single pass, no reload"), (PAIR, "single pass, pairs"), (PAIR | NORELOAD, "single pass, pairs, no reload"),
             (WIN, "two windows"), (WIN | PAIR, "two windows, pairs")),
         9: ((0, "two windows"), (PAIR, "two windows, pairs")),
         7: ((0, "single pass"), (PAIR, "single pass, pairs")),
         6: ((0, "single pass"), (PAIR, "single pass, pairs"))}
for S, fl in forms.items():
    ref = {}
    for flags, name in fl:
        C, ms = _ffi.dbg_ozaki_dgemm(ctx, 1.0, A, A, 0.0, C0, S=S, flags=flags, reps=4)
        pairs = S * (S + 1) // 2
        units_per_sm = (n // 128) * (n // 64) * (n // 32) * pairs / 148
        clk = ms * 1e-3 * 1.965e9 / units_per_sm
        same = ""
        if not flags & NORELOAD:
            key = flags & ~PAIR
            if key in ref:
                same = ", bit-identical to single CTAs" if np.array_equal(C, ref[key]) else ", DIFFERS from single CTAs"
            else:
                ref[key] = C
        print(f"S={S} {name}: {ms:.3f} ms, {2 * n ** 3 / ms / 1e9:.1f} TFLOP/s-equiv, ~{clk:.1f} clk per 128x64x32 per SM, "
              f"int8 {2 * n ** 3 * pairs / ms / 1e12:.2f} POPS{same}", flush=True)
