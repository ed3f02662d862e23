"""Outputs and launch counts of a fixed set of narrow-model calls (shapes that the shared-memory kernels take) ->
parent/narrow_calls.npz (a directory of its own: the oracle does not reproduce these).  tests/test_wide_inputs.py
compares the current library with them bit for bit: the wide-input kernels must leave every shape that ran before
them on the same kernels, with the same results.

    python tests/golden/make_golden_narrow.py [--lib path/to/libgpr_sm100a.so] [--out parent/narrow_calls.npz]

Needs a GPU.  The committed file was written by the library of the commit before the wide-input kernels."""
import argparse
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "gaussianprocessregression.jl_b200"))


def problem(D, N, ncomp_se, matern, seed):
    rng = np.random.default_rng(seed)
    x = np.asfortranarray(rng.random((D, N)))
    y = np.sin(3 * x).sum(0) + 0.1 * rng.standard_normal(N)
    types = [1] * ncomp_se + ([3] if matern else []) + [2]
    nk = ncomp_se + (1 if matern else 0)
    hp = np.concatenate([np.concatenate([[0.5 + rng.random()], rng.uniform(0.5, 1.5, D) / np.sqrt(D)]) for _ in range(nk)] + [[0.3]])
    return types, x, y, hp, rng


def calls(_ffi):
    """name -> array of results; name + '_launches' -> launches the call enqueued"""
    out = {}
    ctx = _ffi.Context(0)

    def launches(name, fn):
        l0 = ctx.launch_count()
        res = fn()
        out[name + "_launches"] = np.array(ctx.launch_count() - l0)
        return res

    for D, ncomp_se, matern, tag in ((8, 1, False, "se_d8"), (64, 1, False, "se_d64"), (8, 1, True, "se_matern_d8")):
        types, x, y, hp, rng = problem(D, 1000, ncomp_se, matern, 17 + D)
        m = _ffi.ModelHandle(ctx, types, D, x, y)
        F, G = launches("nlml_grad_" + tag, lambda: m.nlml_grad(hp))
        out["nlml_grad_" + tag] = np.concatenate([[F], G])
        if tag == "se_d8":
            xp = np.asfortranarray(rng.random((D, 300)))
            mu, var, cov = launches("predict_" + tag, lambda: m.predict(xp, want_var=True, want_cov=True))
            out["predict_" + tag] = np.concatenate([mu.ravel(), var, cov.ravel()])
            xe, xq = np.asfortranarray(0.5 * rng.random((D, 12))), np.asfortranarray(0.5 * rng.random((D, 9)))
            smu, svar = launches("split_predict_" + tag, lambda: m.split_predict(xe, xq, var_range=(1, 12)))
            out["split_predict_" + tag] = np.concatenate([smu.ravel(), svar.ravel()])
        m.close()
    ctx.close()

    types, x, y, hp, _ = problem(8, 1000, 1, False, 99)
    mc = _ffi.MultiContext([0, 0], nb=256)
    mm = _ffi.MultiModelHandle(mc, types, 8, x, y)
    l0 = mc.launch_count()
    F, G = mm.nlml_grad(hp)
    out["mgpu_nlml_grad_g2_launches"] = np.array(mc.launch_count() - l0)
    out["mgpu_nlml_grad_g2"] = np.concatenate([[F], G])
    mm.close()
    mc.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=None)
    ap.add_argument("--out", default=os.path.join(HERE, "parent", "narrow_calls.npz"))
    args = ap.parse_args()
    from gpr_sm100a import _ffi
    if args.lib:
        _ffi.LIB_PATH = os.path.abspath(args.lib)
    np.savez(args.out, **calls(_ffi))
    print("wrote", args.out)


if __name__ == "__main__":
    main()
