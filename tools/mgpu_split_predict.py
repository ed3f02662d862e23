"""Split prediction on Cmap(+, xe, xq) grids on the block-cyclic multi-GPU model (gpr_mgpu_split_predict): the q columns
sharded over the ranks for the mean, the var_range rows through the explicit-inverse quadratic form (include/gpr_sm100a.h,
DESIGN.md 7).

    python tools/mgpu_split_predict.py [--ne 4096] [--nq 4096] [--n 131072] [--base-n 32768] [--skip big,base] [--out FILE]

One JSON record (default profiles/mgpu_split_predict.json) with the card name and power limit read in the same call.  Every
timed figure is the second of two identical calls (the first warms workspaces and modules up); wall = host clock around the
call, which returns after every rank's queue has finished; phases = the library's CUDA-event timings (gpr_mgpu_timings).
  base  config 4's grid (ne = nq = 4096) on the benchmark model (bench.py: N = base-n, D = 8, SE + SE + noise), var_range 1:3
        and mean only, with G = 1 and G = every visible GPU, and single-GPU gpr_split_predict in the same process: max mean
        (relative) and variance (over sum sigma^2) differences.
  big   the same grid on config 5's model (N = n, D = 16, SE + noise) on every visible GPU.  The oracle and the single-GPU
        path cannot run at this N: invariants instead (0 <= var <= prior on the var rows, the prior elsewhere).
A leg that the box cannot run is recorded as not measured; nothing falls back."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "gaussianprocessregression.jl_b200"))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from mgpu_predict_kinv import card, config5_model  # noqa: E402

VAR_RANGE = (1, 3)


def grid(D, ne, nq, seed):
    rng = np.random.default_rng(seed)
    return np.asfortranarray(0.5 * rng.random((D, ne))), np.asfortranarray(0.5 * rng.random((D, nq)))


def timed(h, xe, xq, var_range):
    """two calls into the same caller-owned arrays; the second one is timed"""
    ne, nq = xe.shape[1], xq.shape[1]
    mean = np.empty((ne, nq), order="F")
    var = np.empty(ne * nq) if var_range else None
    for _ in range(2):
        t0 = time.perf_counter()
        h.split_predict(xe, xq, var_range=var_range, want_var=var_range is not None, mean_out=mean, var_out=var)
        dt = time.perf_counter() - t0
    tm = h.timings()
    keys = ("split_build", "split_gemm", "split_d2h") + (("pred_kstar", "pred_trsm", "pred_rownorm", "pred_mean") if var_range else ())
    return mean, var, {"wall_s": round(dt, 4), "phase_ms": {k: round(tm[k], 2) for k in keys}}


def mean_flop(ne, nq, N, nk):
    return 2.0 * ne * nq * N * nk


def run_mgpu(x, y, hp, types, G, nb, xe, xq):
    from gpr_sm100a import _ffi
    mc = _ffi.MultiContext(list(range(G)), nb=nb)
    mm = _ffi.MultiModelHandle(mc, types, x.shape[0], x, y)
    t0 = time.perf_counter()
    mm.update_cache(hp)
    t_fac = time.perf_counter() - t0
    mu, var, rv = timed(mm, xe, xq, VAR_RANGE)
    mu0, _, rm = timed(mm, xe, xq, None)
    mm.close(); mc.close()
    nk = sum(1 for t in types if t != 2)
    row = {"gpus": G, "nb": nb, "update_cache_s": round(t_fac, 2), "var_rows": rv, "mean_only": rm,
           "mean_gemm_tflops_all_ranks": mean_flop(xe.shape[1], xq.shape[1], x.shape[1], nk) / (rm["phase_ms"]["split_gemm"] * 1e-3) / 1e12,
           "var_points_per_s": (VAR_RANGE[1] - VAR_RANGE[0] + 1) * xq.shape[1] / (sum(rv["phase_ms"][k] for k in rv["phase_ms"]
                                                                                    if k.startswith("pred")) * 1e-3),
           "mean_only_equals_mean_with_var": bool(np.array_equal(mu, mu0))}
    return mu, var, row


def prior_of(hp, types, D):
    off, s = 0, 0.0
    for t in types:
        s += hp[off] ** 2
        off += 1 if t == 2 else D + 1
    return s


def base_leg(args, ndev, rec):
    import bench
    from gpr_sm100a import _ffi
    N, D = args.base_n, 8
    x, y, hp = bench.make_problem(N, D)
    types = [1, 1, 2]
    prior = prior_of(hp, types, D)
    xe, xq = grid(D, args.ne, args.nq, 4)
    ctx = _ffi.Context(0)
    m1 = _ffi.ModelHandle(ctx, types, D, x, y)
    m1.update_cache(hp)
    mu1, var1, r1 = timed(m1, xe, xq, VAR_RANGE)
    _, _, r1m = timed(m1, xe, xq, None)
    m1.close(); ctx.close()
    out = {"N": N, "D": D, "ne": args.ne, "nq": args.nq, "var_range": VAR_RANGE,
           "single_gpu_gpr_split_predict": {"var_rows": r1, "mean_only": r1m}, "mgpu": []}
    for G in sorted({1, ndev}):
        mu, var, row = run_mgpu(x, y, hp, types, G, 1024, xe, xq)
        row["mean_rel_vs_single"] = float(np.abs(mu - mu1).max() / np.abs(mu1).max())
        row["var_abs_over_prior_vs_single"] = float(np.abs(var - var1).max() / prior)
        out["mgpu"].append(row)
        print(json.dumps(row), flush=True)
    if ndev == 1:
        out["gpus_2_4_8"] = "not measured: the box has 1 GPU"
    rec["base"] = out


def big_leg(args, ndev, rec):
    x, y, hp = config5_model(args.n)
    D = x.shape[0]
    types = [1, 2]
    prior = prior_of(hp, types, D)
    xe, xq = grid(D, args.ne, args.nq, 5)
    mu, var, row = run_mgpu(x, y, hp, types, ndev, 2048, xe, xq)
    v2 = var.reshape(args.ne, args.nq)
    rows = v2[VAR_RANGE[0] - 1:VAR_RANGE[1]]
    row.update({"N": args.n, "D": D, "var_rows_in_0_prior": bool(rows.min() >= 0.0 and rows.max() <= prior),
                "other_rows_equal_prior": bool(np.all(np.delete(v2, np.arange(VAR_RANGE[0] - 1, VAR_RANGE[1]), axis=0) == prior)),
                "mean_finite": bool(np.isfinite(mu).all())})
    if ndev == 1:
        row["gpus_2_4_8"] = "not measured: the box has 1 GPU"
    rec["big"] = row
    print(json.dumps(row), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ne", type=int, default=4096)
    ap.add_argument("--nq", type=int, default=4096)
    ap.add_argument("--n", type=int, default=131072)
    ap.add_argument("--base-n", type=int, default=32768)
    ap.add_argument("--skip", default="", help="comma list of legs to leave out: base, big")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "mgpu_split_predict.json"))
    args = ap.parse_args()
    from gpr_sm100a import _ffi
    ndev = _ffi.device_count()
    if ndev < 1:
        sys.exit("no sm_100-class GPU: nothing to measure")
    skip = set(filter(None, args.skip.split(",")))
    rec = {"tool": "tools/mgpu_split_predict.py", "card": card(), "devices": ndev, "torchrun_leg": "not measured"}
    if "base" not in skip:
        base_leg(args, ndev, rec)
    if "big" not in skip:
        big_leg(args, ndev, rec)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({"written": args.out}), flush=True)


if __name__ == "__main__":
    main()
