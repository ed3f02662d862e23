"""Box integration on the block-cyclic multi-GPU model (gpr_mgpu_integrate): many boxes per pass over K^-1
(include/gpr_sm100a.h, DESIGN.md 7).

    python tools/mgpu_integrate.py [--n 131072] [--nbox 16384] [--gpus 1,2,4,8] [--nb 2048] [--base-n 32768] [--out FILE]

One JSON record (default profiles/mgpu_integrate.json) with the card name and power limit read in the same call:
  baseline  the benchmark model (bench.py, N = base-n, D = 8) with G = 1 and with every visible GPU: gpr_mgpu_integrate for
            nbox = 1 and nbox boxes in one call, against the single-GPU gpr_integrate looped over the same boxes in the same
            process (every box is run and timed; nothing is extrapolated), and the largest difference between the two.
  config5   config 5's model (N = 131072, D = 16, SquaredExp()+WhiteNoise()) on every GPU count the box has: the same
            timings plus invariants, since the oracle cannot run at this N -- agreement across the GPU counts,
            0 <= var <= k2 (to 1e-9 k2), and Iout against k1^T alpha for 8 boxes (k1 and the product on the host).
A GPU count that does not fit the box, and the one-process-per-GPU (NCCL) transport, are written as "not measured"."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "gaussianprocessregression.jl_b200"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, ROOT)

from mgpu_predict_kinv import card, config5_model   # noqa: E402


def make_boxes(D, nbox, seed):
    """D x nbox boxes with random corners in [0, 1]^D and widths in [0.1, 0.5] per dimension (cell averages over a grid
    are the typical use; random placement keeps every box distinct)"""
    rng = np.random.default_rng(seed)
    a = rng.random((D, nbox)) * 0.8
    return np.asfortranarray(a), np.asfortranarray(a + 0.1 + 0.4 * rng.random((D, nbox)))


def mgpu_timed(mm, a, b):
    """first call warms up (workspaces, module load); the second is timed, with the library's CUDA-event phase times"""
    for _ in range(2):
        t0 = time.perf_counter()
        I, var = mm.integrate(a, b)
        dt = time.perf_counter() - t0
    tm = mm.timings()
    return I, var, dt, {k: round(v, 2) for k, v in tm.items() if k.startswith("pred")}


def k2_of(hp, a, b):
    import gpr_oracle as o
    return np.array([o.antideriv2(hp, a[:, i], b[:, i]) for i in range(a.shape[1])])


def baseline(args, ndev, rec):
    import bench
    from gpr_sm100a import _ffi
    N, D = args.base_n, 8
    x, y, hp = bench.make_problem(N, D)
    types = [1, 1, 2]
    a, b = make_boxes(D, args.nbox, 8)
    ctx = _ffi.Context(0)
    m1 = _ffi.ModelHandle(ctx, types, D, x, y)
    m1.update_cache(hp)
    m1.integrate(a[:, 0], b[:, 0])                        # warm-up
    t0 = time.perf_counter()
    I1 = m1.integrate(a[:, 0], b[:, 0])
    t_one = time.perf_counter() - t0
    Is, vs = np.empty((args.nbox, 1)), np.empty(args.nbox)
    t0 = time.perf_counter()
    for i in range(args.nbox):
        Ii, vi = m1.integrate(a[:, i], b[:, i])
        Is[i], vs[i] = Ii[0], vi[0]
    t_loop = time.perf_counter() - t0
    m1.close(); ctx.close()
    k2 = k2_of(hp, a, b)
    out = {"N": N, "D": D, "nbox": args.nbox, "single_gpu_gpr_integrate_one_box_s": t_one,
           "single_gpu_gpr_integrate_loop_s": t_loop, "single_gpu_boxes_per_s": args.nbox / t_loop, "mgpu": []}
    for G in sorted({1, ndev}):
        mc = _ffi.MultiContext(list(range(G)), nb=1024)
        mm = _ffi.MultiModelHandle(mc, types, D, x, y)
        mm.update_cache(hp)
        J1, w1, dt1, _ = mgpu_timed(mm, a[:, :1], b[:, :1])
        I, var, dt, tm = mgpu_timed(mm, a, b)
        mm.close(); mc.close()
        out["mgpu"].append({"gpus": G, "one_box_s": dt1, "all_boxes_s": dt, "boxes_per_s": args.nbox / dt, "phase_ms": tm,
                            "speedup_over_single_gpu_loop": t_loop / dt,
                            "Iout_rel_vs_single": float(np.abs(I - Is).max() / np.abs(Is).max()),
                            "var_abs_over_k2_vs_single": float((np.abs(var - vs) / k2).max()),
                            "one_box_Iout_rel_vs_single": float(abs(J1[0, 0] - I1[0][0]) / abs(I1[0][0]))})
        print(json.dumps(out["mgpu"][-1]), flush=True)
    out["mgpu"] += [{"gpus": g, "not measured": f"the box has {ndev} GPU(s)"} for g in (2, 4, 8) if g > ndev]
    rec["baseline"] = out


def config5(args, ndev, rec):
    import gpr_oracle as o
    from gpr_sm100a import _ffi
    N = args.n
    x, y, hp = config5_model(N)
    D = x.shape[0]
    a, b = make_boxes(D, args.nbox, 5)
    k2 = k2_of(hp, a, b)
    rows, outs = [], {}
    for G in [int(g) for g in args.gpus.split(",")]:
        if G > ndev:
            rows.append({"gpus": G, "not measured": f"the box has {ndev} GPU(s)"})
            continue
        mc = _ffi.MultiContext(list(range(G)), nb=args.nb)
        mm = _ffi.MultiModelHandle(mc, [1, 2], D, x, y)
        t0 = time.perf_counter()
        mm.update_cache(hp)
        t_fac = time.perf_counter() - t0
        _, _, dt1, _ = mgpu_timed(mm, a[:, :1], b[:, :1])
        I, var, dt, tm = mgpu_timed(mm, a, b)
        alpha = mm.fetch(_ffi.FETCH_ALPHA)
        mm.close(); mc.close()
        s = np.random.default_rng(1).choice(args.nbox, 8, replace=False)
        ref = np.array([o.antideriv(x, hp, a[:, i], b[:, i]) @ alpha for i in s])
        flop = args.nbox * float(N) ** 2 / G
        row = {"gpus": G, "nb": args.nb, "update_cache_s": round(t_fac, 2), "one_box_s": dt1, "all_boxes_s": dt,
               "boxes_per_s": args.nbox / dt, "phase_ms": tm, "tflops_per_rank": flop / (tm["pred_trsm"] * 1e-3) / 1e12,
               "Iout_vs_k1_alpha_rel": float(np.abs(I[s, 0] - ref).max() / np.abs(ref).max()),
               "var_over_k2_min": float((var / k2).min()), "var_over_k2_max": float((var / k2).max()),
               "var_in_0_k2": bool(np.all(var >= -1e-9 * k2) and np.all(var <= k2 * (1 + 1e-9)))}
        rows.append(row)
        outs[G] = (I, var)
        print(json.dumps(row), flush=True)
    done = sorted(outs)
    if len(done) >= 2:
        p, q = outs[done[-1]], outs[done[-2]]
        rec["config5_agreement"] = {"gpus": done[-2:], "Iout_rel": float(np.abs(p[0] - q[0]).max() / np.abs(q[0]).max()),
                                    "var_abs_over_k2": float((np.abs(p[1] - q[1]) / k2).max())}
    else:
        rec["config5_agreement"] = {"not measured": f"needs two GPU counts; the box has {ndev} GPU(s)"}
    rec["config5"] = {"N": N, "D": D, "nbox": args.nbox, "runs": rows}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=131072)
    ap.add_argument("--nbox", type=int, default=16384)
    ap.add_argument("--gpus", default="1,2,4,8")
    ap.add_argument("--nb", type=int, default=2048)
    ap.add_argument("--base-n", type=int, default=32768)
    ap.add_argument("--skip", default="", help="comma list of legs to leave out: baseline, config5")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "mgpu_integrate.json"))
    args = ap.parse_args()
    from gpr_sm100a import _ffi
    ndev = _ffi.device_count()
    if ndev < 1:
        sys.exit("no sm_100-class GPU: nothing to measure")
    skip = set(filter(None, args.skip.split(",")))
    rec = {"tool": "tools/mgpu_integrate.py", "card": card(), "devices": ndev,
           "nccl": {"not measured": "the one-process-per-GPU transport (torchrun) was not run by this tool"}}
    if "baseline" not in skip:
        baseline(args, ndev, rec)
    if "config5" not in skip:
        config5(args, ndev, rec)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({"written": args.out}), flush=True)


if __name__ == "__main__":
    main()
