"""Box integration of many boxes per call on one GPU (gpr_integrate_batch): one triangular solve per tile of boxes
(include/gpr_sm100a.h, DESIGN.md 7).

    python tools/integrate_batch.py [--n 32768] [--nbox 16384] [--loop 512] [--out FILE]

One JSON record (default profiles/integrate_batch.json) with the card name and power limit read in the same call.  On the
benchmark model (bench.py, N = n, D = 8) and nbox random boxes, at the default route ("ozaki" -1) and on the DMMA pipe
("ozaki" 0), all in one process:
  batch     gpr_update_cache without inverse, then gpr_integrate_batch for all boxes (warm-up call, then the timed call) with
            the library's CUDA-event phase times; one box alone through it.
  loop      gpr_integrate over the first `loop` boxes on the same model: the time per box and the total extrapolated to nbox
            boxes (the full loop takes about a minute per route); one box alone.
  mgpu      gpr_mgpu_integrate with G = 1 on the same data, including its gpr_mgpu_update_cache.
  agreement the largest Iout (relative to max|Iout|) and var (over k2 of the box) differences between the three."""
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

from mgpu_integrate import k2_of, make_boxes   # noqa: E402
from mgpu_predict_kinv import card             # noqa: E402


def timed(f, reps=2):
    """the first call warms up (workspaces, module load); the last one is timed"""
    for _ in range(reps):
        t0 = time.perf_counter()
        r = f()
        dt = time.perf_counter() - t0
    return r, dt


def diff(I, v, J, w, k2):
    return {"Iout_rel": float(np.abs(I - J).max() / np.abs(J).max()), "var_abs_over_k2": float((np.abs(v - w) / k2).max())}


def one_route(args, ozaki, x, y, hp, a, b, k2):
    from gpr_sm100a import _ffi
    D, nbox, nl = x.shape[0], a.shape[1], args.loop
    types = [1, 1, 2]
    ctx = _ffi.Context(0)
    ctx.set_option("ozaki", ozaki)
    m = _ffi.ModelHandle(ctx, types, D, x, y)
    t0 = time.perf_counter()
    m.update_cache(hp)
    t_fac = time.perf_counter() - t0
    (I, var), dt = timed(lambda: m.integrate(a, b))
    tm = {k: round(v, 2) for k, v in m.timings().items() if k.startswith("pred")}
    _, dt1 = timed(lambda: m.integrate(a[:, :1], b[:, :1]))
    _, dt1_loop = timed(lambda: m.integrate(a[:, 0], b[:, 0]))
    Il, vl = np.empty((nl, 1)), np.empty(nl)
    t0 = time.perf_counter()
    for i in range(nl):
        Ii, vi = m.integrate(a[:, i], b[:, i])
        Il[i], vl[i] = Ii[0], vi[0]
    t_loop = time.perf_counter() - t0
    digits = m.route()[0]
    m.close(); ctx.close()

    mc = _ffi.MultiContext([0], nb=1024)
    mc.set_option("ozaki", ozaki)
    mm = _ffi.MultiModelHandle(mc, types, D, x, y)
    t0 = time.perf_counter()
    mm.update_cache(hp)
    t_mfac = time.perf_counter() - t0
    (Im, vm), dtm = timed(lambda: mm.integrate(a, b))
    mm.close(); mc.close()

    per_box = t_loop / nl
    rec = {"ozaki": ozaki, "route_digits": digits,
           "batch": {"update_cache_no_inverse_s": t_fac, "all_boxes_s": dt, "boxes_per_s": nbox / dt, "phase_ms": tm,
                     "one_box_s": dt1},
           "loop": {"boxes_run": nl, "per_box_s": per_box, "extrapolated_all_boxes_s": per_box * nbox, "one_box_s": dt1_loop},
           "mgpu_g1": {"update_cache_s": t_mfac, "all_boxes_s": dtm, "boxes_per_s": nbox / dtm},
           "speedup_batch_over_loop": per_box * nbox / dt,
           "agreement": {"batch_vs_loop": diff(I[:nl], var[:nl], Il, vl, k2[:nl]),
                         "batch_vs_mgpu": diff(I, var, Im, vm, k2),
                         "loop_vs_mgpu": diff(Il, vl, Im[:nl], vm[:nl], k2[:nl])}}
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=32768)
    ap.add_argument("--nbox", type=int, default=16384)
    ap.add_argument("--loop", type=int, default=512)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "integrate_batch.json"))
    args = ap.parse_args()
    import bench
    from gpr_sm100a import _ffi
    if _ffi.device_count() < 1:
        sys.exit("no sm_100-class GPU: nothing to measure")
    D = 8
    x, y, hp = bench.make_problem(args.n, D)
    a, b = make_boxes(D, args.nbox, 8)
    k2 = k2_of(hp, a, b)
    rec = {"tool": "tools/integrate_batch.py", "card": card(), "N": args.n, "D": D, "nbox": args.nbox,
           "routes": [one_route(args, oz, x, y, hp, a, b, k2) for oz in (-1, 0)]}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({"written": args.out}), flush=True)


if __name__ == "__main__":
    main()
