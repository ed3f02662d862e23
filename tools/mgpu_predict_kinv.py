"""Posterior prediction on the block-cyclic multi-GPU model (gpr_mgpu_update_cache + gpr_mgpu_predict): the
explicit-inverse quadratic form split over the ranks that own the columns of K^-1 (include/gpr_sm100a.h, DESIGN.md 7).

    python tools/mgpu_predict_kinv.py [--n 131072] [--m 16384] [--gpus 1,2,4,8] [--nb 2048] [--base-n 32768] [--out FILE]
    python tools/mgpu_predict_kinv.py --dist-worker DIR      (one process per GPU under torchrun; started by the above)

One JSON record (default profiles/mgpu_predict_kinv.json) with the card name and power limit read in the same call:
  scaling   config 5's model (N = 131072, D = 16, SquaredExp()+WhiteNoise(), sigma = 1, l = 0.4, sigma_n = 0.1), M general test
            points with mean and diagonal variance on every GPU count the box has: points/s, per-rank TFLOP/s of the product
            (M N^2 / G over its CUDA-event time), the fix-up kernel's GB/s (16 M N / G bytes), the K(x, xp) build and the sum over
            the ranks.  The oracle cannot run at this N: invariants instead -- the largest two GPU counts agree to 1e-9 sum sigma^2,
            the mean equals K(xp, x) alpha for 32 sampled points (alpha fetched, product on the host), 0 <= var <= prior.
  baseline  N = base-n on the benchmark model (bench.py): single-GPU gpr_predict against the multi-GPU path with G = 1.
  nccl      the same prediction with one process per GPU (torchrun, transport 2) on >= 2 GPUs: outputs identical across the
            processes and equal to the single-process run to 1e-9 sum sigma^2.
A count that does not fit the box is recorded as such; nothing falls back."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "gaussianprocessregression.jl_b200"))
sys.path.insert(0, ROOT)


def config5_model(N, D=16):
    rng = np.random.default_rng(5005)
    x = np.asfortranarray(rng.random((D, N)))
    y = np.sin(3 * x).sum(0) + 0.1 * rng.standard_normal(N)
    hp = np.concatenate([[1.0], 0.4 * np.ones(D), [0.1]])
    return x, y, hp


def se_rows(xs, x, hp):
    """K(xs, x) of SquaredExp()+WhiteNoise() for general test points (no noise, no jitter): host check only"""
    sig, ell = hp[0], hp[1:-1]
    a, b = xs * ell[:, None], x * ell[:, None]
    d = (a * a).sum(0)[:, None] + (b * b).sum(0)[None, :] - 2.0 * a.T @ b
    return sig * sig * np.exp(-np.maximum(d, 0.0))


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return [line.strip() for line in r.stdout.strip().splitlines()]
    except Exception as e:   # the record says what could not be read
        return [f"nvidia-smi failed: {e}"]


def predict_timed(mm, xp, reps=2):
    """first call warms up (workspaces, module load); the last call is timed, CUDA-event phase times from the library"""
    for _ in range(reps):
        t0 = time.perf_counter()
        mu, var, _ = mm.predict(xp, want_var=True)
        dt = time.perf_counter() - t0
    return mu, var, dt, mm.timings()


def scaling(args, ndev, rec):
    from gpr_sm100a import _ffi
    N, M = args.n, args.m
    x, y, hp = config5_model(N)
    prior = hp[0] ** 2 + hp[-1] ** 2
    xp = np.asfortranarray(np.random.default_rng(7).random((x.shape[0], M)))
    rows, outs = [], {}
    for G in [int(g) for g in args.gpus.split(",")]:
        if G > ndev:
            rows.append({"gpus": G, "skipped": f"the box has {ndev} GPU(s)"})
            continue
        mc = _ffi.MultiContext(list(range(G)), nb=args.nb)
        mm = _ffi.MultiModelHandle(mc, [1, 2], x.shape[0], x, y)
        t0 = time.perf_counter()
        mm.update_cache(hp)
        t_fac = time.perf_counter() - t0
        mu, var, dt, tm = predict_timed(mm, xp)
        flop = M * float(N) ** 2 / G
        row = {"gpus": G, "nb": args.nb, "M": M, "update_cache_s": round(t_fac, 2), "predict_s": round(dt, 3),
               "points_per_s": M / dt, "product_ms": round(tm["pred_trsm"], 1), "tflops_per_rank": flop / (tm["pred_trsm"] * 1e-3) / 1e12,
               "fixup_ms": round(tm["pred_rownorm"], 2), "fixup_GBps": 16.0 * M * N / G / (tm["pred_rownorm"] * 1e-3) / 1e9,
               "kbuild_ms": round(tm["pred_kstar"], 2), "reduce_ms": round(tm["pred_mean"], 2),
               "var_min_over_prior": float(var.min() / prior), "var_max_over_prior": float(var.max() / prior)}
        alpha = mm.fetch(_ffi.FETCH_ALPHA)
        s = np.random.default_rng(1).choice(M, 32, replace=False)
        mref = se_rows(xp[:, s], x, hp) @ alpha
        row["mean_vs_Kalpha_rel"] = float(np.abs(mu[s, 0] - mref).max() / np.abs(mref).max())
        row["var_in_0_prior"] = bool(var.min() >= 0.0 and var.max() <= prior)
        rows.append(row)
        outs[G] = (mu, var)
        print(json.dumps(row), flush=True)
        mm.close(); mc.close()
    done = sorted(outs)
    if len(done) >= 2:
        a, b = outs[done[-1]], outs[done[-2]]
        rec["scaling_agreement"] = {"gpus": done[-2:], "var_abs_over_prior": float(np.abs(a[1] - b[1]).max() / prior),
                                    "mean_rel": float(np.abs(a[0] - b[0]).max() / np.abs(b[0]).max())}
    rec["scaling"] = rows
    return outs


def baseline(args, rec):
    import bench
    from gpr_sm100a import _ffi
    N, M = args.base_n, args.m
    x, y, hp = bench.make_problem(N, 8)
    xp = np.asfortranarray(np.random.default_rng(8).random((8, M)))
    types = [1, 1, 2]
    ctx = _ffi.Context(0)
    m1 = _ffi.ModelHandle(ctx, types, 8, x, y)
    m1.update_cache(hp)
    for _ in range(2):
        t0 = time.perf_counter()
        mu1, var1, _ = m1.predict(xp, want_var=True)
        t1 = time.perf_counter() - t0
    m1.close(); ctx.close()
    mc = _ffi.MultiContext([0], nb=1024)
    mm = _ffi.MultiModelHandle(mc, types, 8, x, y)
    mm.update_cache(hp)
    mu, var, dt, tm = predict_timed(mm, xp)
    mm.close(); mc.close()
    prior = hp[0] ** 2 + hp[9] ** 2 + hp[-1] ** 2          # sigma of both SquaredExp components (D = 8) and sigma_n
    rec["baseline"] = {"N": N, "M": M, "single_gpu_gpr_predict_points_per_s": M / t1, "mgpu_G1_points_per_s": M / dt,
                       "mgpu_G1_phase_ms": {k: round(v, 2) for k, v in tm.items() if k.startswith("pred")},
                       "mgpu_G1_tflops": M * float(N) ** 2 / (tm["pred_trsm"] * 1e-3) / 1e12,
                       "mean_rel_vs_single": float(np.abs(mu - mu1).max() / np.abs(mu1).max()),
                       "var_abs_over_prior_vs_single": float(np.abs(var - var1).max() / prior)}
    print(json.dumps(rec["baseline"]), flush=True)


def dist_worker(out_dir, n, m, nb):
    import torch
    import torch.distributed as dist
    from gpr_sm100a import _ffi, shard
    local = int(os.environ.get("LOCAL_RANK", 0))
    rank = int(os.environ.get("RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    x, y, hp = config5_model(n)
    xp = np.asfortranarray(np.random.default_rng(7).random((x.shape[0], m)))
    dc = shard.dist_context(local, nb=nb)
    mm = _ffi.MultiModelHandle(dc, [1, 2], x.shape[0], x, y)
    mm.update_cache(hp)
    mu, var, dt, tm = predict_timed(mm, xp)
    np.savez(os.path.join(out_dir, f"rank{rank}.npz"), mu=mu, var=var, dt=dt, trsm=tm["pred_trsm"])
    mm.close()
    dist.destroy_process_group()


def nccl_leg(args, ndev, rec, outs):
    if ndev < 2:
        rec["nccl"] = {"skipped": f"the box has {ndev} GPU(s); the transport-2 leg needs >= 2"}
        return
    G = min(ndev, 8)
    with tempfile.TemporaryDirectory() as d:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", f"--nproc_per_node={G}", os.path.abspath(__file__),
               "--dist-worker", d, "--n", str(args.n), "--m", str(args.m), "--nb", str(args.nb)]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            rec["nccl"] = {"gpus": G, "error": r.stderr[-2000:]}
            return
        res = [np.load(os.path.join(d, f"rank{k}.npz")) for k in range(G)]
    same = all(np.array_equal(res[0]["mu"], z["mu"]) and np.array_equal(res[0]["var"], z["var"]) for z in res[1:])
    x, y, hp = config5_model(args.n)
    prior = hp[0] ** 2 + hp[-1] ** 2
    out = {"gpus": G, "identical_across_processes": bool(same), "predict_s": float(max(z["dt"] for z in res)),
           "points_per_s": args.m / float(max(z["dt"] for z in res))}
    if G in outs:
        out["var_abs_over_prior_vs_single_process"] = float(np.abs(res[0]["var"] - outs[G][1]).max() / prior)
    rec["nccl"] = out
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=131072)
    ap.add_argument("--m", type=int, default=16384)
    ap.add_argument("--gpus", default="1,2,4,8")
    ap.add_argument("--nb", type=int, default=2048)
    ap.add_argument("--base-n", type=int, default=32768)
    ap.add_argument("--skip", default="", help="comma list of legs to leave out: scaling, baseline, nccl")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "mgpu_predict_kinv.json"))
    ap.add_argument("--dist-worker", metavar="DIR", default=None)
    args = ap.parse_args()
    if args.dist_worker:
        dist_worker(args.dist_worker, args.n, args.m, args.nb)
        return
    from gpr_sm100a import _ffi
    ndev = _ffi.device_count()
    if ndev < 1:
        sys.exit("no sm_100-class GPU: nothing to measure")
    skip = set(filter(None, args.skip.split(",")))
    rec = {"tool": "tools/mgpu_predict_kinv.py", "card": card(), "devices": ndev, "N": args.n, "M": args.m}
    outs = {} if "scaling" in skip else scaling(args, ndev, rec)
    if "baseline" not in skip:
        baseline(args, rec)
    if "nccl" not in skip:
        nccl_leg(args, ndev, rec, outs)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({"written": args.out}), flush=True)


if __name__ == "__main__":
    main()
