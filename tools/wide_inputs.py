"""Stage times of high-dimensional models (the chunked covariance build and the wide gradient reduction) -> profiles/wide_inputs.json

    python tools/wide_inputs.py [--n 32768] [--evals 3] [--out profiles/wide_inputs.json]

For each shape: GPR_T_KBUILD, GPR_T_GRAD and GPR_T_EVAL of one gpr_nlml_grad (median over --evals after one warm-up,
each at a slightly different hp so that every call builds, factors and inverts),
and F, G against the oracle's formulas (tests/test_wide_inputs.py ref_loss_grad) at a sampled size (N = 1024, same D).
D = 64 runs the shared-memory kernels and is the baseline of the others.  Prediction: points/s of mean + variance at
D = 512; a torch.profiler table of device time per kernel of one evaluation at D = 512.  The card's name and power limit are read in the same run and stored beside the numbers."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "gaussianprocessregression.jl_b200"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

SHAPES = [("SE+noise", 64), ("SE+noise", 65), ("SE+noise", 128), ("SE+noise", 512), ("SE+noise", 1024), ("SE+SE+noise", 256)]


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:   # noqa: BLE001  (recorded, not fatal)
        return f"unavailable: {e}"


def kernel_profile(m, hp):
    """Device time per kernel name of one gpr_nlml_grad (torch.profiler, CUDA activities: every kernel of the process), in a
    run of its own after a warm-up evaluation"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    m.nlml_grad(hp * (1.0 + 2e-6))
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        m.nlml_grad(hp * (1.0 + 3e-6))
        torch.cuda.synchronize()
    rows = []
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None)
        if us is None:
            us = getattr(e, "cuda_time_total", 0.0)
        if us > 0:
            rows.append({"kernel": e.key[:160], "ms": us / 1e3, "calls": e.count})
    rows.sort(key=lambda r: -r["ms"])
    for r in rows[:12]:
        print(f"  {r['ms']:9.3f} ms  {r['calls']:6d}  {r['kernel']}", flush=True)
    return {"D": 512, "what": "one NLML + gradient, SE + noise, device time per kernel name", "kernels": rows[:25]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=32768)
    ap.add_argument("--evals", type=int, default=3)
    ap.add_argument("--n-check", type=int, default=1024)
    ap.add_argument("--m-pred", type=int, default=32768)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "wide_inputs.json"))
    args = ap.parse_args()
    import gpr_oracle as o
    from gpr_sm100a import _ffi
    from test_wide_inputs import grad_err, ref_loss_grad, wide_problem
    covs = {"SE+noise": (o.SE, o.NOISE), "SE+SE+noise": (o.SE, o.SE, o.NOISE)}
    types = {o.SE: 1, o.NOISE: 2}
    res = {"gpu": gpu_info(), "n": args.n, "evals": args.evals, "shapes": []}
    ctx = _ffi.Context(0)
    for name, D in SHAPES:
        cov = covs[name]
        x, y, hp, _ = wide_problem(cov, args.n, D, D)
        m = _ffi.ModelHandle(ctx, [types[c] for c in cov], D, x, y)
        rows = []
        for k in range(args.evals + 1):
            m.nlml_grad(hp * (1.0 + 1e-6 * k))     # a new hp every time: the same hp reuses the cached factor
            t = m.timings()
            rows.append([t["kbuild"], t["grad"], t["eval"]])
        m.close()
        med = np.median(np.array(rows[1:]), axis=0)
        xs, ys, hs, _ = wide_problem(cov, args.n_check, D, D + 1)
        ms = _ffi.ModelHandle(ctx, [types[c] for c in cov], D, xs, ys)
        F, G = ms.nlml_grad(hs)
        ms.close()
        Fo, Go, cond = ref_loss_grad(cov, hs, xs, ys)
        row = {"cov": name, "D": D, "P": len(hp), "kbuild_ms": med[0], "grad_ms": med[1], "eval_ms": med[2],
               "check_n": args.n_check, "relF": abs(F - Fo) / abs(Fo), "relG": grad_err(G, Go), "cond": cond}
        print(json.dumps(row), flush=True)
        res["shapes"].append(row)
    cov, D = covs["SE+noise"], 512
    x, y, hp, rng = wide_problem(cov, args.n, D, 7)
    m = _ffi.ModelHandle(ctx, [1, 2], D, x, y)
    res["profile"] = kernel_profile(m, hp)
    m.update_cache(hp)
    xp = np.asfortranarray(rng.random((D, args.m_pred)))
    m.predict(xp[:, :1024], want_var=True)
    best = None
    for _ in range(3):
        t0 = time.perf_counter()
        m.predict(xp, want_var=True)     # returns after the device-to-host copy of mean and variance
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    t = m.timings()
    m.close()
    ctx.close()
    res["predict"] = {"D": D, "n": args.n, "m": args.m_pred, "seconds": best, "points_per_s": args.m_pred / best,
                      "pred_kstar_ms": t["pred_kstar"], "pred_trsm_ms": t["pred_trsm"]}
    print(json.dumps(res["predict"]), flush=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
