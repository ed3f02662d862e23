#!/usr/bin/env python
"""bench.py -- headline benchmark of the GP hot path on B200 (contract: task statement (4), SURVEY.md 8d).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[2], "3-ref" of SURVEY.md 8d): SquaredExp()+SquaredExp()+WhiteNoise() (P = 19),
N = 32768, D = 8, FP64.  One step = one NLML + gradient evaluation (log_loss_grad!, src/cost.jl:60-70) at the
next point of a fixed hyper-parameter trajectory (so nothing can be cached between steps).
  value : evaluations/s with x, y resident in HBM (only hp goes in and F, G come out per step)
  e2e   : the same through the C ABI with HOST buffers: every step re-uploads x, y from pinned host memory
          (gpr_model_set_x/_y), evaluates, and reads F, G back
  N > 1 : the headline metric is replicas only (SURVEY.md 8e): every rank evaluates its own hyper-parameter set, no
          data-path collective.  The SHARDED paths are measured in the same run and reported under `extra`:
            extra.config4 : split predict on the 4096 x 4096 sum-grid (16.8 M points), `e` rows sharded over the ranks
            extra.config5 : ONE factorization distributed block-cyclically over all ranks (one process per GPU, panels
                            over NCCL): N = 65536 for 1-2 GPUs, N = 131072 for 4-8 GPUs (strong scaling of one evaluation)
  --impl reference : the reference-shaped CPU path (oracle/gpr_oracle_big.reference_shaped_eval: materialised K per
          component, dpotrf, dpotrs on the identity, per-hyper-parameter dK + dgemv + ddot) on the host cores: one
          calibration evaluation at N = 16384 (scale <= 8 to the metric's N) + the requested steps at the largest N
          that fits the time budget; ms_per_step is the time actually spent per executed step
  --dump-outputs DIR : after the timed steps, rank 0 writes what its last timed evaluation returned, DIR/F.npy (shape (1,))
          and DIR/G.npy (shape (P,)), float64.  The inputs come from fixed seeds, so two builds run with the same arguments
          can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "gaussianprocessregression.jl_b200"))

METRIC = "NLML+grad evals/s (N=32k,D=8,fp64)"
UNIT = "evals/s"
N_FULL, D_FULL = 32768, 8
WORKLOAD = "3-ref: SquaredExp()+SquaredExp()+WhiteNoise() P=19, N=32768, D=8, one log_loss_grad! per step"


def make_problem(N, D, seed=3003):
    rng = np.random.default_rng(seed)
    x = rng.random((D, N))
    y = np.sin(3 * x).sum(0) + 0.1 * rng.standard_normal(N)
    hp = np.concatenate([[1.0], 0.5 * np.ones(D), [0.5], 2.0 * np.ones(D), [0.1]])
    return x, y, hp


def hp_at(hp0, step, rank=0):
    """Fixed, pre-determined hyper-parameter trajectory (identical work for CPU and GPU arms)."""
    return hp0 * (1.0 + 0.004 * step + 0.01 * rank)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.index, self.rows, self.proc, self.th = index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE, text=True)
        except Exception:
            self.proc = None
            return
        self.th = threading.Thread(target=self._read, daemon=True)
        self.th.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- CPU arm (oracle; checker/baseline only)
COV_REF = ("SquaredExp", "SquaredExp", "WhiteNoise")
MGPU_NB = 2048            # block-column width of the block-cyclic multi-GPU drivers (config 5); GPR_MGPU_NB overrides
CALIBRATION = os.path.join(ROOT, "profiles", "cpu_calibration_r2.json")


def host_info():
    info = {"cores": os.cpu_count() or 1, "ram_gb": None, "blas": None, "blas_threads": None}
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                info["ram_gb"] = round(int(line.split()[1]) / 2 ** 20, 1)
    except Exception:
        pass
    try:
        import threadpoolctl
        for lib in threadpoolctl.threadpool_info():
            if lib.get("user_api") == "blas" and "scipy" in lib.get("filepath", ""):
                info["blas"], info["blas_threads"] = f"{lib.get('internal_api')} {lib.get('version')}", lib.get("num_threads")
    except Exception:
        pass
    return info


class RefArm:
    """The reference's evaluation AS IT EXECUTES IT (oracle/gpr_oracle_big.reference_shaped_eval; src/cost.jl:60-70,
    96-127): one materialised N x N matrix per component, dpotrf, dpotrs, dpotrs on a materialised identity, then per
    hyper-parameter a materialised dK + dgemv + 2 ddot.  BLAS/LAPACK calls use every host thread; the numpy
    element-wise sweeps (covariance build, dK) are single-threaded, as Julia's broadcasts are."""

    def __init__(self):
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import gpr_oracle_big as ob
        self.ob = ob
        self.ws = {}
        # torchrun exports OMP_NUM_THREADS=1 to every rank: the CPU arm must still use every host core (rank 0 is the only rank
        # that runs it), so the BLAS pools are sized explicitly
        try:
            import threadpoolctl
            self._blas_limits = threadpoolctl.threadpool_limits(limits=os.cpu_count() or 1, user_api="blas")
        except Exception:
            self._blas_limits = None

    def run(self, N, step):
        x, y, hp0 = make_problem(N, D_FULL)
        t0 = time.perf_counter()
        F, G, st, ws = self.ob.reference_shaped_eval(COV_REF, np.log(hp_at(hp0, step)), x, y, ws=self.ws.get(N))
        dt = time.perf_counter() - t0
        self.ws = {N: ws}                       # keep one workspace (MllGradCache) alive, like the reference's train loop
        return dt, st, F

    def drop(self):
        self.ws = {}


def fit_cost_model(sizes, times):
    """t(N) = a N^3 + b N^2 (factor / solves vs the N^2 sweeps), least squares in relative error, a, b >= 0."""
    n = np.asarray(sizes, dtype=np.float64)
    t = np.asarray(times, dtype=np.float64)
    A = np.stack([n ** 3 / t, n ** 2 / t], axis=1)
    coef, *_ = np.linalg.lstsq(A, np.ones_like(t), rcond=None)
    a, b = float(coef[0]), float(coef[1])
    if a <= 0 or b < 0:
        a, b = float(np.mean(t / n ** 3)), 0.0
    return a, b


def scale_by_stage(dt, stages, n, n_full=None):
    """Seconds per evaluation at n_full from ONE measured evaluation at n: the factorization and the dpotrs on the identity
    (O(N^3)) grow by (n_full / n)^3, everything else (covariance build, sums, per-hyper-parameter dK sweeps: O(N^2)) by
    (n_full / n)^2.  Grounded in the measured stage times instead of a two-term fit, which on these hosts assigns most of the
    N = 16384 time to the N^2 term and under-predicts the cubic stages."""
    n_full = n_full or N_FULL
    cubic = float(stages.get("potrf", 0.0) + stages.get("potrs_identity", 0.0))
    cubic = min(cubic, dt)
    r = n_full / n
    return cubic * r ** 3 + (dt - cubic) * r ** 2


def reference_measurement(steps, warmup, budget_s, n_cal_max=16384, log=None):
    """Times the reference-shaped CPU evaluation.  (1) probes at N = 2048 and 4096; (2) ONE calibration evaluation at the
    largest N <= n_cal_max whose predicted time fits 0.6 of the budget and whose (nk + 3) N^2 workspace fits the
    host RAM -- the value reported for N = 32768 is that measurement scaled by the fitted model, scale <= 8 when
    N_cal = 16384; (3) `warmup` + `steps` real evaluations at the largest N whose predicted total fits the rest of the
    budget: ms_per_step is their mean wall time, exactly what was executed."""
    say = log or (lambda *a: None)
    arm = RefArm()
    hi = host_info()
    t_start = time.perf_counter()
    meas = {}
    arm.run(1024, 0)                                        # spin up the BLAS thread pool
    for n in (2048, 4096):
        meas[n] = arm.run(n, 0)[0]
        say(f"probe N={n}: {meas[n]:.2f} s")
    a, b = fit_cost_model(list(meas), list(meas.values()))
    pred = lambda n: a * n ** 3 + b * n ** 2
    ram = hi["ram_gb"] or 16.0
    n_cal, cal_stages = None, None
    # calibration: N = 16384 first (scale <= 8 by construction); then, with the fit refined by that measurement, the
    # metric's own N = 32768 if its predicted time fits a third of the budget and its 43 GB workspace fits the host RAM
    for cand in (16384, 32768):
        if cand > n_cal_max or 5 * 8 * cand ** 2 / 2 ** 30 > 0.8 * ram or pred(cand) > 0.6 * budget_s:
            if n_cal is None and cand == 16384:
                for small in (12288, 8192):
                    if pred(small) <= 0.6 * budget_s:
                        cand = small
                        break
                else:
                    break
            else:
                break
        dt, st, _ = arm.run(cand, 0)
        meas[cand] = dt
        n_cal, cal_stages = cand, st
        say(f"calibration N={cand}: {dt:.1f} s {st}")
        a, b = fit_cost_model(list(meas), list(meas.values()))
        arm.drop()
        if cand < 16384:
            break
    arm.drop()
    left = budget_s - (time.perf_counter() - t_start)
    n_step = 2048
    for cand in (16384, 12288, 8192, 6144, 4096, 3072):
        if (cand in meas or 5 * 8 * cand ** 2 / 2 ** 30 <= 0.8 * ram) and (steps + warmup) * (meas.get(cand) or pred(cand)) <= left:
            n_step = cand
            break
    ts, F, st_sum = [], None, {}
    for sidx in range(warmup + steps):
        dt, st, F = arm.run(n_step, sidx)
        if sidx >= warmup:
            ts.append(dt)
            for k, v in st.items():
                st_sum[k] = st_sum.get(k, 0.0) + v / steps
    t_step = float(np.mean(ts))
    meas_all = dict(meas)
    if n_step not in meas or n_step != n_cal:
        meas_all[n_step] = t_step
    a, b = fit_cost_model(list(meas_all), list(meas_all.values()))
    # the figure for N = 32768 comes from the largest size that actually ran (the calibration evaluation, or the timed steps when
    # they ran at a larger N), scaled stage by stage
    if n_cal is not None and n_cal >= n_step:
        n_base, t_base, base_st = n_cal, meas[n_cal], cal_stages
    else:
        n_base, t_base, base_st = n_step, t_step, st_sum
        cal_stages = st_sum
    t_full = scale_by_stage(t_base, base_st, n_base) if n_base != N_FULL else t_base
    scale = t_full / t_base
    meas_all[n_base] = t_base
    return {"t_full": t_full, "n_base": n_base, "t_base": meas_all[n_base], "scale": scale, "n_step": n_step, "t_step": t_step,
            "measured": {str(k): round(v, 3) for k, v in sorted(meas_all.items())}, "fit": {"a_N3": a, "b_N2": b},
            "calibration_stages_s": {k: round(v, 2) for k, v in (cal_stages or {}).items()}, "host": hi, "F_last": F}


FULL_SIZE_NOTE = ("; the same path MEASURED at N=32768 on this pool's host (profiles/cpu_reference_n32768_box_r2q.json, GPR_REF_NCAL=32768): "
                  "402 s per evaluation -- OpenBLAS dpotrf fails there (info != 0 on an SPD matrix), so the factor and the solves go "
                  "through the blocked work-around of oracle/gpr_oracle_big.py and are slower than a working LAPACK; the scaled "
                  "figure above is therefore the conservative (faster-CPU) baseline")


def describe(m):
    h = m["host"]
    return (f"reference-shaped CPU path (oracle/gpr_oracle_big.reference_shaped_eval: per-component K, dpotrf, dpotrs on the identity, "
            f"per-hp dK + dgemv + ddot) on {h['cores']} host cores, {h['blas']} with {h['blas_threads']} threads for BLAS/LAPACK "
            f"(numpy element-wise sweeps single-threaded), {h['ram_gb']} GB RAM available; measured s/eval {m['measured']}; "
            f"value = measured {m['t_base']:.1f} s at N={m['n_base']} x {m['scale']:.2f} (stage-wise: measured dpotrf + dpotrs-on-identity "
            f"seconds x (32768/N)^3, the remaining N^2 sweeps x (32768/N)^2) = {m['t_full']:.0f} s per evaluation at N=32768"
            + (" -- scaled, not run at full size" if m["n_base"] != N_FULL else "") + FULL_SIZE_NOTE)


def cpu_baseline(budget_s=30.0):
    """cpu_baseline leg of the default run: ONE evaluation of the reference-shaped CPU path at N = 16384 (about 25 s on the
    pool's 16-core host; N = 8192 if the host has under 16 GB free or the N = 4096 probe predicts more than 2 x budget_s),
    scaled stage-wise to N = 32768 (scale <= 8).  The committed full --impl reference record is quoted beside it."""
    arm = RefArm()
    hi = host_info()
    arm.run(1024, 0)
    meas = {4096: arm.run(4096, 0)[0]}
    ram = hi["ram_gb"] or 16.0
    n_base = 16384
    if 5 * 8 * n_base ** 2 / 2 ** 30 > 0.8 * ram or meas[4096] * 64 > 4 * budget_s:
        n_base = 8192
    dt, st, _ = arm.run(n_base, 0)
    arm.drop()
    meas[n_base] = dt
    t_full = scale_by_stage(dt, st, n_base)
    scale = t_full / dt
    sample = (f"reference-shaped CPU path (oracle/gpr_oracle_big.reference_shaped_eval: per-component K, dpotrf, dpotrs on the identity, "
              f"per-hp dK + dgemv + ddot) on {hi['cores']} host cores ({hi['blas']}, {hi['blas_threads']} BLAS threads; numpy sweeps "
              f"single-threaded), ONE evaluation at N={n_base}: {dt:.1f} s (stages {({k: round(v, 2) for k, v in st.items()})}); scaled "
              f"x{scale:.2f} to N=32768 stage-wise (dpotrf + dpotrs-on-identity x (32768/N)^3, the N^2 sweeps x (32768/N)^2) = {t_full:.0f} s"
              + FULL_SIZE_NOTE)
    out = {"value": 1.0 / t_full, "unit": UNIT, "cores": hi["cores"], "kind": "port", "sample": sample, "sample_N": n_base, "scale": scale,
           "stages_s": {k: round(v, 3) for k, v in st.items()}}
    try:
        cal = json.load(open(CALIBRATION))
        out["calibrated"] = {"value": cal.get("value"), "sample_N": cal.get("sample_N"), "scale": cal.get("scale"),
                             "measured_s_per_eval": cal.get("measured_s_per_eval"),
                             "source": "profiles/cpu_calibration_r2.json (bench.py --impl reference on this pool's host, committed)"}
    except Exception:
        pass
    return out


def run_reference(args, rank, world):
    if rank != 0:
        return
    budget = float(os.environ.get("GPR_REF_BUDGET_S", "300"))         # whole run: probes + one N = 16384 calibration + warmup + steps
    n_cal_max = int(os.environ.get("GPR_REF_NCAL", "16384"))          # 32768: also measure the metric's own size (~7 min more)
    m = reference_measurement(args.steps, args.warmup, budget, n_cal_max, log=lambda s: print("[reference]", s, file=sys.stderr, flush=True))
    value = 1.0 / m["t_full"]
    base = {"value": value, "unit": UNIT, "cores": m["host"]["cores"], "kind": "port", "sample": describe(m),
            "sample_N": m["n_base"], "scale": m["scale"]}
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": m["t_step"] * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "timing": f"host wall clock; ms_per_step = mean wall time of the {args.steps} executed steps, each one real evaluation at "
                                 f"N={m['n_step']} (the largest size at which warmup+steps fit the time budget); value = the largest measured size "
                                 f"(N={m['n_base']}, {m['t_base']:.1f} s) scaled x{m['scale']:.2f} to N=32768",
                       "step_N": m["n_step"], "sample_N": m["n_base"], "scale": m["scale"], "same_config": m["n_base"] == N_FULL},
            "cpu_baseline": base, "reference_detail": {k: m[k] for k in ("measured", "fit", "calibration_stages_s", "host", "n_step", "t_step")},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- GPU arm
def measure_fp64_peak(torch, n=8192):
    """cuBLAS DGEMM through torch.matmul: the FP64 denominator (MEASURED_PEAKS.json has no FP64 figure)."""
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    for _ in range(3):
        a @ b
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(6):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); a @ b; e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(40):
        a @ b
    e1.record()
    torch.cuda.synchronize()
    sustained = e0.elapsed_time(e1) / 40
    del a, b
    torch.cuda.empty_cache()
    return 2 * n ** 3 / best / 1e9, 2 * n ** 3 / sustained / 1e9


def predict_extras(args, mh, hp0, N, D):
    """Secondary metric of BASELINE.json: predictive points/s (general test points, mean + diagonal variance and mean only)."""
    extra = {}
    M = 16384
    xp = np.asfortranarray(np.random.default_rng(4004).random((D, M)))
    mh.update_cache(hp0)
    mh.predict(xp, want_var=True)
    t0 = time.perf_counter()
    mu, var, _ = mh.predict(xp, want_var=True)
    dt = time.perf_counter() - t0
    tp = mh.timings()
    extra["predict_points_per_s"] = M / dt
    extra["predict_var_tflops"] = M * float(N) ** 2 / dt / 1e12
    extra["predict_stage_ms"] = {k: round(v, 3) for k, v in tp.items() if k.startswith("pred")}
    # the two streaming kernels (K* . wt and row norms of V) read 8*M*N bytes each
    hbm = 6478.9
    try:
        hbm = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        pass
    # streams of the prediction: the K* tile is written once (8*M*N bytes) and V = K* U^-1 is read once for the row
    # norms; mu = K* wt is reduced inside the K* build (no separate stream since round 1c)
    extra["predict_stream_gbs"] = {"kstar_build_write": 8.0 * M * N / tp["pred_kstar"] / 1e6, "rownorm_v": 8.0 * M * N / tp["pred_rownorm"] / 1e6,
                                   "mean": "fused into the K* build", "hbm_peak_gbs": hbm}
    mh.predict(xp, want_var=False)
    t0 = time.perf_counter()
    mh.predict(xp, want_var=False)
    extra["predict_mean_only_points_per_s"] = M / (time.perf_counter() - t0)
    extra["predict_config"] = f"mean+diag variance, M={M} general test points, host in/out, N={N}"
    return extra


def config4_split_predict(torch, dist, _ffi, ctx, rank, world, nvar_rows=64):
    """BASELINE.json config 4 (SURVEY.md 8d): posterior mean for all ne x nq = 16.8 M sum-grid points and the variance of
    `nvar_rows` e rows per rank through gpr_split_predict (src/split_predict.jl:10-53), N = 32768 training points, the `e`
    rows in contiguous blocks per rank (independent units: no data-path collective).  Timed on the device side of each
    call (barrier + synchronize on both sides, max over ranks)."""
    from gpr_sm100a import shard
    N, D, ne, nq = N_FULL, D_FULL, 4096, 4096
    x, y, hp = make_problem(N, D)
    rng = np.random.default_rng(4004)
    xe, xq = np.asfortranarray(0.5 * rng.random((D, ne))), np.asfortranarray(0.5 * rng.random((D, nq)))
    mh = _ffi.ModelHandle(ctx, [1, 1, 2], D, x, y)
    mh.update_cache(hp)
    lo, hi = shard.block_range(ne, rank, world)
    xe_blk = np.asfortranarray(xe[:, lo:hi])
    nv = min(nvar_rows, hi - lo)

    def sync():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    # warm-up at full size into the caller-owned result array (the reference's split predict! writes in place): device workspaces
    # and the host pages exist before the timed call -- a fresh 134 MB array costs 35-500 ms of first-touch faults under the copy
    mean = np.zeros((hi - lo, nq), order="F")
    mh.split_predict(xe_blk, xq, var_range=None, want_var=False, mean_out=mean)
    sync()
    t0 = time.perf_counter()
    mh.split_predict(xe_blk, xq, var_range=None, want_var=False, mean_out=mean)
    sync()
    t_mean = time.perf_counter() - t0
    tm = mh.timings()
    t0 = time.perf_counter()
    _, var = mh.split_predict(xe_blk[:, :nv], xq, var_range=(1, nv), want_var=True)
    sync()
    t_var = time.perf_counter() - t0
    tv = mh.timings()
    if dist is not None:
        tt = torch.tensor([t_mean, t_var], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_mean, t_var = float(tt[0]), float(tt[1])
    out = None
    if rank == 0:
        worst_mu = worst_var = 0.0
        for e in (0, nv // 2, nv - 1):             # split path vs the dense path of the library on explicit points
            pts = np.asfortranarray(xe_blk[:, e:e + 1] + xq[:, :512])
            mu_d, var_d, _ = mh.predict(pts, want_var=True)
            worst_mu = max(worst_mu, float(np.abs(mu_d[:, 0] - mean[e, :512]).max()))
            worst_var = max(worst_var, float(np.abs(var_d - var[e * nq:e * nq + 512]).max()))
        M = ne * nq
        nvp = world * nv * nq
        out = {"workload": f"split predict, N={N}, ne=nq={ne} (M={M}), e rows sharded over {world} rank(s); variance of {nv} e rows per rank",
               "mean_ms_all_points": t_mean * 1e3, "mean_points_per_s": M / t_mean, "mean_tflops": 2.0 * 2 * ne * nq * N / t_mean / 1e12,
               "mean_stage_ms_rank0": {k: round(v, 2) for k, v in tm.items() if k.startswith("split") and v > 0},
               "var_points": nvp, "var_s": t_var, "var_points_per_s": nvp / t_var, "var_tflops_aggregate": nvp * float(N) ** 2 / t_var / 1e12,
               "var_stage_ms_rank0": {k: round(v, 2) for k, v in tv.items() if k.startswith("pred") and v > 0},
               "parity_split_vs_dense": {"max_abs_mean_diff": worst_mu, "max_abs_var_diff": worst_var, "rows": 3, "points_per_row": 512},
               "timing": "host clock around each C-ABI call (host xe/xq in, mean/var out), barrier + synchronize on both sides, max over ranks"}
    mh.close()
    return out


def config5_distributed(torch, dist, _ffi, rank, world, local_rank, n_override=None, evals=1):
    """BASELINE.json config 5 (SURVEY.md 8d/8e): ONE NLML + gradient evaluation of SquaredExp()+WhiteNoise(), D = 16,
    with K / U / K^-1 block-cyclic over all ranks (csrc/dist_blocked.hpp; one process per GPU, panels travel by
    ncclBroadcast / ncclAllGather, the P + 3 partial sums by ncclAllReduce).  N = 65536 on 1-2 GPUs, 131072 on 4-8
    (the 137 GB covariance of the full configuration needs >= 4 GPUs next to the out-of-place workspaces).
    Reports per-phase milliseconds, TFLOP/s per GPU, |K alpha - y| on sampled columns; reference: src/cost.jl:96-127."""
    from gpr_sm100a import shard
    N = n_override or (65536 if world <= 2 else 131072)
    D = 16
    rng = np.random.default_rng(5005)
    x = np.asfortranarray(rng.random((D, N)))
    y = np.sin(3 * x).sum(0) + 0.1 * rng.standard_normal(N)
    hp = np.concatenate([[1.0], 0.4 * np.ones(D), [0.1]])
    nb = int(os.environ.get("GPR_MGPU_NB", str(MGPU_NB)))
    mc = shard.dist_context(device=local_rank, nb=nb) if world > 1 else _ffi.MultiContext([local_rank], nb=nb)
    mm = _ffi.MultiModelHandle(mc, [1, 2], D, x, y)
    mm.nlml_grad(hp * 0.99)                                     # warm-up evaluation
    ts, F, G, tm = [], None, None, None
    for _ in range(evals):
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        t0 = time.perf_counter()
        F, G = mm.nlml_grad(hp)
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
        tm = mm.timings()
    t = min(ts)
    if dist is not None:
        tt = torch.tensor([t], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t = float(tt[0])
    alpha = mm.fetch(_ffi.FETCH_ALPHA)
    out = None
    if rank == 0:
        cols = np.random.default_rng(1).choice(N, 32, replace=False)
        sig, ell, sn = hp[0], hp[1:-1], hp[-1]
        xs = x * ell[:, None]
        Kc = sig * sig * np.exp(-((xs[:, :, None] - xs[:, None, cols]) ** 2).sum(0))
        Kc[cols, np.arange(32)] += 1e-8 + sn * sn
        resid = float(np.abs(Kc.T @ alpha - y[cols]).max() / np.abs(y).max())
        dense_ms = tm["potrf"] + tm["trtri"] + tm["lauum"]
        out = {"workload": f"one NLML+gradient, SquaredExp()+WhiteNoise() P=18, N={N}, D=16, block-cyclic over {world} rank(s), nb={nb}",
               "transport": "NCCL (one process per GPU)" if world > 1 else "single rank",
               "s_per_eval": t, "evals_per_s": 1.0 / t, "phase_ms": {k: round(v, 1) for k, v in tm.items() if v > 0 and not k.startswith("pred")},
               "dense_tflops_aggregate": float(N) ** 3 / (dense_ms * 1e-3) / 1e12, "dense_tflops_per_gpu": float(N) ** 3 / (dense_ms * 1e-3) / 1e12 / world,
               "phase_tflops_per_gpu": {k: float(N) ** 3 / 3 / (tm[k] * 1e-3) / 1e12 / world for k in ("potrf", "trtri", "lauum")},
               "limiter": max(("potrf", "trtri", "lauum"), key=lambda k: tm[k]),
               "F": F, "G_norm": float(np.linalg.norm(G)), "resid_K_alpha_minus_y": resid,
               "timing": "host clock around gpr_mgpu_nlml_grad after a barrier, max over ranks; phases: CUDA events of rank 0"}
    mm.close()
    mc.close()
    return out


def config5_single_process(_ffi, world, n_override=None):
    """Config 5 through the single-process multi-device context (transport 0: NVLink peer memory, copy-engine prefetch)."""
    N = n_override or (65536 if world <= 2 else 131072)
    D = 16
    rng = np.random.default_rng(5005)
    x = np.asfortranarray(rng.random((D, N)))
    y = np.sin(3 * x).sum(0) + 0.1 * rng.standard_normal(N)
    hp = np.concatenate([[1.0], 0.4 * np.ones(D), [0.1]])
    nb = int(os.environ.get("GPR_MGPU_NB", str(MGPU_NB)))
    mc = _ffi.MultiContext(list(range(world)), nb=nb)
    mm = _ffi.MultiModelHandle(mc, [1, 2], D, x, y)
    mm.nlml_grad(hp * 0.99)
    t0 = time.perf_counter()
    F, G = mm.nlml_grad(hp)
    t = time.perf_counter() - t0
    tm = mm.timings()
    dense_ms = tm["potrf"] + tm["trtri"] + tm["lauum"]
    out = {"workload": f"one NLML+gradient, N={N}, D=16, block-cyclic over {world} GPUs driven by one process (peer memory over NVLink), nb={nb}",
           "s_per_eval": t, "evals_per_s": 1.0 / t, "phase_ms": {k: round(v, 1) for k, v in tm.items() if v > 0 and not k.startswith("pred")},
           "dense_tflops_aggregate": float(N) ** 3 / (dense_ms * 1e-3) / 1e12, "dense_tflops_per_gpu": float(N) ** 3 / (dense_ms * 1e-3) / 1e12 / world,
           "limiter": max(("potrf", "trtri", "lauum"), key=lambda k: tm[k]), "F": F, "G_norm": float(np.linalg.norm(G))}
    mm.close()
    mc.close()
    return out


def config3_ext_and_training(_ffi, ctx, steps=2):
    """Config 3 as BASELINE.json words it: SquaredExp()+Matern52()+WhiteNoise() (3-ext; Matern-5/2 is an extension, parity
    unpinned) evaluations/s, and a free-running L-BFGS training run of 3-ref at N = 32768 (src/train.jl:47-56: log-space
    fg! closure over one cache, host optimiser)."""
    import scipy.optimize as so
    x, y, hp0 = make_problem(N_FULL, D_FULL)
    out = {}
    mh = _ffi.ModelHandle(ctx, [1, 3, 2], D_FULL, x, y)
    mh.nlml_grad(np.log(hp0), log_scale=True)
    ev = 0.0
    for sidx in range(steps):
        mh.nlml_grad(np.log(hp_at(hp0, sidx + 1)), log_scale=True)
        ev += mh.timings()["eval"]
    out["config3_ext"] = {"workload": "SquaredExp()+Matern52()+WhiteNoise() P=19, N=32768, D=8 (extension: parity vs own oracle only)",
                          "evals_per_s": steps / (ev * 1e-3), "ms_per_eval": ev / steps}
    mh.close()
    mh = _ffi.ModelHandle(ctx, [1, 1, 2], D_FULL, x, y)
    trace = []

    def fg(v):
        F, G = mh.nlml_grad(v, log_scale=True)
        trace.append(F)
        return F, G

    t0 = time.perf_counter()
    res = so.minimize(fg, np.log(hp0), jac=True, method="L-BFGS-B", options={"maxiter": 4, "maxfun": 8})
    dt = time.perf_counter() - t0
    out["train_free_running"] = {"workload": "L-BFGS-B from the benchmark hp, 3-ref, N=32768 (src/train.jl:47-56), maxiter 4",
                                 "iterations": int(res.nit), "evaluations": len(trace), "seconds": dt, "evals_per_s": len(trace) / dt,
                                 "F_start": trace[0], "F_end": float(res.fun)}
    mh.close()
    return out


def dump_outputs(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def run_gpu(args, rank, world, local_rank):
    import torch
    import gpr_sm100a as g
    from gpr_sm100a import _ffi

    torch.cuda.set_device(local_rank)
    dist = None
    cpu_group = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        cpu_group = dist.new_group(backend="gloo")     # host-side barrier: an NCCL barrier would spin on the waiting ranks' SMs

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    N, D = args.n, D_FULL
    x, y, hp0 = make_problem(N, D)
    P = len(hp0)
    ctx = g.Context(local_rank)
    cov = g.SquaredExp() + g.SquaredExp() + g.WhiteNoise()
    # host buffers of the e2e arm live in pinned memory
    xh = torch.empty((N, D), dtype=torch.float64).pin_memory()
    yh = torch.empty((N,), dtype=torch.float64).pin_memory()
    xh.numpy()[...] = x.T                     # (N, D) C-order == (D, N) column major
    yh.numpy()[...] = y
    x_f = xh.numpy().T                         # F-contiguous (D, N) view of the pinned buffer
    y_f = yh.numpy()
    mh = _ffi.ModelHandle(ctx, [1, 1, 2], D, x_f, y_f)

    fp64_burst = fp64_sust = None
    if rank == 0:
        fp64_burst, fp64_sust = measure_fp64_peak(torch)

    def step(s):
        return mh.nlml_grad(np.log(hp_at(hp0, s, rank)), log_scale=True)

    for s in range(args.warmup):
        step(s)
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    l0 = ctx.launch_count()
    stage = {}
    t0 = time.perf_counter()
    for s in range(args.steps):
        F, G = step(args.warmup + s)
        for k, v in mh.timings().items():     # CUDA events recorded by the library on ITS stream (torch.cuda.Event cannot see it)
            stage[k] = stage.get(k, 0.0) + v
    barrier()
    t_wall = time.perf_counter() - t0
    launches = ctx.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"F": [F], "G": G})
    mh_route = mh.route()                     # product engine of the timed steps (digits of the INT8 route, 0 = DMMA)
    # device time of the K timed steps: event pair around every evaluation on the library stream, summed; max over ranks
    t_loc = stage["eval"] * 1e-3
    t_max = t_loc
    if dist is not None:
        tt = torch.tensor([t_loc, t_wall], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_max, t_wall = float(tt[0].item()), float(tt[1].item())
    value = world * args.steps / t_max

    # end-to-end through the C ABI with host buffers
    def e2e_step(s):
        mh.set_x(x_f)
        mh.set_y(y_f)
        return mh.nlml_grad(np.log(hp_at(hp0, s, rank)), log_scale=True)

    e2e_step(1000)
    barrier()
    t0 = time.perf_counter()
    for s in range(args.steps):
        F2, G2 = e2e_step(2000 + s)
    barrier()
    t_e = time.perf_counter() - t0
    if dist is not None:
        tt = torch.tensor([t_e], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_e = float(tt.item())
    e2e = {"value": world * args.steps / t_e, "unit": UNIT, "h2d_bytes_per_step": 8 * (D * N + N + P), "d2h_bytes_per_step": 8 * (P + 1)}

    # the same evaluation with every FP64 product on the DMMA pipe (INT8-tensor-core route off), for the record
    dmma_only = None
    if rank == 0:
        ctx.set_option("ozaki", 0)
        mh.nlml_grad(np.log(hp_at(hp0, 500, rank)), log_scale=True)
        Fd, Gd = mh.nlml_grad(np.log(hp_at(hp0, args.warmup + args.steps - 1, rank)), log_scale=True)
        td = mh.timings()
        dmma_only = {"ms_per_eval": td["eval"], "evals_per_s": 1e3 / td["eval"], "stage_ms": {k: round(td[k], 2) for k in ("potrf", "trtri", "lauum")},
                     "F": Fd, "relF_vs_default_route": abs(Fd - F) / abs(F),
                     "relG_vs_default_route": float((np.abs(Gd - G) / np.maximum(np.abs(G), 1e-8 * np.linalg.norm(G))).max())}
        ctx.set_option("ozaki", -1)
    # secondary single-GPU numbers that need the headline model (rank 0 only), then free it for the sharded extras
    pred_extra = predict_extras(args, mh, hp0, N, D) if (rank == 0 and not args.no_predict) else {}
    gemm_ms = None
    if rank == 0:
        rng = np.random.default_rng(0)
        A = np.asfortranarray(rng.standard_normal((4096, 4096)))
        _, gemm_ms = _ffi.dbg_dgemm(ctx, "T", "N", 1.0, A, A, 0.0, np.zeros((4096, 4096), order="F"), reps=6)
    mh.close()
    sharded = {}
    if not args.no_sharded:
        sharded["config4"] = config4_split_predict(torch, dist, _ffi, ctx, rank, world)
        sharded["config5"] = config5_distributed(torch, dist, _ffi, rank, world, local_rank, n_override=args.config5_n)
        if world > 1:
            # the same factorization driven by ONE process over all GPUs of the node (gpr_mgpu_create: panels move as
            # peer-memory reads / copy-engine transfers over NVLink, next-step panels prefetched on a side queue) -- the
            # transport a single-process Julia host would use; rank 0 runs it, the other ranks wait
            single = None
            torch.cuda.synchronize()
            dist.barrier(group=cpu_group)              # every rank has released its GPU memory and is idle
            if rank == 0:
                single = config5_single_process(_ffi, world, n_override=args.config5_n)
            dist.barrier(group=cpu_group)              # the waiting ranks block on the host, their GPUs stay free
            sharded["config5_single_process"] = single
        if args.config5_base and world == 1:
            sharded["config5_base_1gpu_n131072"] = config5_distributed(torch, dist, _ffi, rank, world, local_rank, n_override=131072)
        if rank == 0 and world == 1 and N == N_FULL:
            sharded.update(config3_ext_and_training(_ffi, ctx))

    if rank != 0:
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return

    K = args.steps
    ms = {k: v / K for k, v in stage.items()}
    flops_factor_inverse = float(N) ** 3                                # N^3/3 potrf + 2N^3/3 trtri+lauum
    t_dense = (ms["potrf"] + ms["trtri"] + ms["lauum"]) * 1e-3
    achieved = flops_factor_inverse / t_dense / 1e12
    gemm_tf = 2 * 4096 ** 3 / gemm_ms / 1e9

    # secondary metrics of BASELINE.json: Cholesky TFLOP/s, predict points/s
    extra = {"cholesky_tflops": N ** 3 / 3 / ms["potrf"] / 1e9, "inverse_tflops": 2 * N ** 3 / 3 / (ms["trtri"] + ms["lauum"]) / 1e9,
             "stage_ms_per_step": {k: round(v, 3) for k, v in ms.items() if v > 0 and not k.startswith("pred")}}
    extra["dmma_only"] = dmma_only
    extra.update(pred_extra)
    extra.update(sharded)

    hp_peak = None
    try:
        hp_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    # DRAM traffic of the dominant kernel per step: from the committed ncu capture of this command (profiles/), GB
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "dram_traffic.json")))
        if N == tj.get("N"):
            traffic = tj["dgemm128_dram_gb_per_eval"]
    except Exception:
        pass
    # INT8-tensor-core route, isolated: FP64-equivalent rate of one 8192^3 product incl. the digit extraction
    oz_tf, oz9_tf = None, None
    try:
        An = np.asfortranarray(np.random.default_rng(1).standard_normal((8192, 8192)))
        _, oz_ms = _ffi.dbg_ozaki_dgemm(ctx, 1.0, An, An, 0.0, np.zeros((8192, 8192), order="F"), S=8, reps=4)
        oz_tf = 2 * 8192 ** 3 / oz_ms / 1e9
        _, oz9_ms = _ffi.dbg_ozaki_dgemm(ctx, 1.0, An, An, 0.0, np.zeros((8192, 8192), order="F"), S=9, flags=0, reps=4)
        oz9_tf = 2 * 8192 ** 3 / oz9_ms / 1e9
        del An
    except Exception:
        pass
    # which engine the step ran on (gpr_model_route): 8 / 9 digits = INT8 tensor cores, 0 = FP64 DMMA pipe
    try:
        digits, digits_inv = mh_route
    except Exception:
        digits, digits_inv = 0, 0
    bf16_sust = (hp_peak or {}).get("bf16_tflops_sustained") or (hp_peak or {}).get("bf16_tflops")
    bf16_src = "MEASURED_PEAKS.json bf16_tflops_sustained (the kernels are timed inside a long step)"
    if not bf16_sust:
        bf16_sust, bf16_src = 1590.0, "fallback of /opt/skills/guides/B200_PROFILING.md (1.59 PFLOP/s bf16): of fallback"
    common = {"traffic": traffic,
              "traffic_unit": "GB of DRAM read+write by all product kernels (INT8 GEMMs, digit extraction, DMMA GEMMs) of one step (ncu launch list, profiles/dram_traffic.json)",
              "fp64_dgemm_roof_tflops": fp64_sust, "frac_of_fp64_dgemm_roof": achieved / fp64_sust,
              "fp64_dgemm_roof_source": f"cuBLAS DGEMM 8192^3 via torch.matmul, sustained {fp64_sust:.1f} / burst {fp64_burst:.1f} TFLOP/s measured in this run "
                                        "(MEASURED_PEAKS.json holds no FP64 figure" + (f"; its HBM copy figure is {hp_peak.get('hbm_gbs')} GB/s)" if hp_peak else ")"),
              "dmma_kernel_isolated_tflops": gemm_tf, "dmma_kernel_isolated_frac": gemm_tf / fp64_burst}
    if digits > 0:
        # dominant kernels: oz_gemm_kernel<8> (potrf, trtri) and oz_gemm_win_kernel (the inverse's W^T W) on the INT8 tensor pipe.  Their
        # roof in FP64-equivalent TFLOP/s = INT8 rate of the pipe / integer products per FP64 product, with the INT8 rate taken as
        # twice the bf16 rate the driver measured (kind::i8 has twice the MACs of kind::f16 on this part; MEASURED_PEAKS.json has no INT8 line)
        prods = (36.0 * 2 + (45.0 if digits_inv == 9 else 36.0 if digits_inv == 8 else 0.0)) / (3.0 if digits_inv else 2.0)
        peak_eq = 2.0 * bf16_sust / prods
        if digits_inv:
            ach = achieved
            what = "N^3 FP64-equivalent flop / (potrf + trtri + lauum) CUDA-event ms"
        else:   # lauum on the DMMA pipe: the roofline of the INT8 kernels covers potrf + trtri only
            ach = 2.0 * float(N) ** 3 / 3.0 / ((ms["potrf"] + ms["trtri"]) * 1e-3) / 1e12
            what = "2 N^3 / 3 FP64-equivalent flop / (potrf + trtri) CUDA-event ms (lauum ran on the DMMA pipe)"
        roofline = {"bound": "tensor", "achieved": ach, "peak": peak_eq, "unit": "TFLOP/s", "frac": ach / peak_eq,
                    "note": f"FP64-equivalent TFLOP/s.  achieved = {what}: every launch of the phases (INT8 products, digit extraction, the products below "
                            "1024 on the DMMA pipe, leaf kernels), i.e. the in-situ rate.  peak = INT8 tensor-pipe rate / integer products per FP64 product "
                            f"= 2 x {bf16_sust:.1f} TFLOP/s bf16 ({bf16_src}) / {prods:.1f} (36 for the 8-digit products of potrf and trtri, 45 for the "
                            "9-digit W^T W of the inverse, weighted by flops).  The FP64 pipe's own roof (cuBLAS DGEMM, measured in this run) and the ratio "
                            "to it are given beside it: the step runs ABOVE the FP64 roof because it does not use the FP64 pipe for its large products; "
                            "extra.dmma_only holds the same step on the DMMA pipe alone",
                    "kernel": "oz_gemm_kernel<8> + oz_gemm_win_kernel (tcgen05.mma kind::i8, TMEM accumulators; csrc/ozaki_i8.cuh) inside blocked potrf + trtri + lauum",
                    "int8_route": {"digits": digits, "digits_inverse": digits_inv, "integer_products_per_fp64_product": prods,
                                   "achieved_int8_pops_in_situ": ach * prods / 1e3, "int8_peak_pops_from_measured_bf16": 2e-3 * bf16_sust,
                                   "int8_peak_pops_nominal": 4.5,
                                   "kernel_isolated_fp64_equivalent_tflops_8192": oz_tf, "kernel_isolated_fp64_equivalent_tflops_8192_nine_digits": oz9_tf,
                                   "kernel_isolated_int8_pops": (oz_tf * 36 / 1e3) if oz_tf else None,
                                   "kernel_isolated_int8_pops_nine_digits": (oz9_tf * 45 / 1e3) if oz9_tf else None,
                                   "kernel_isolated_frac": (oz_tf * 36 / (2.0 * bf16_sust)) if oz_tf else None,
                                   "ncu": "profiles/ozaki_ncu_full_r2t.md: tensor-core pipe 94 % busy (sm__pipe_tc_cycles_active) in oz_gemm_kernel<8>; 94.7 % "
                                          "and 93 % of the L2 -> SM fill rate in the d = 6..10 window of the nine-digit product"}}
    else:
        roofline = {"bound": "tensor", "achieved": achieved, "peak": fp64_sust, "unit": "TFLOP/s", "frac": achieved / fp64_sust,
                    "note": "achieved = N^3 flop / (potrf + trtri + lauum) CUDA-event ms on the FP64 DMMA pipe; peak = cuBLAS DGEMM measured in this run",
                    "kernel": "dgemm128_tma_kernel (DMMA.8x8x4, TMA-fed) inside blocked potrf + trtri + lauum"}
    roofline.update(common)

    base = None
    if world == 1 and not args.no_cpu:
        base = cpu_baseline(budget_s=30.0)

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": t_max / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD if N == N_FULL else WORKLOAD.replace("N=32768", f"N={N}"),
                       "parallelism": "replicas only (one hyper-parameter set per GPU, no data-path collective)" if world > 1 else "1 GPU",
                       "l2": "inputs larger than L2 (K is 8.6 GB per evaluation); no explicit flush needed",
                       "arithmetic": ("FP64 in, FP64 out; products with M, N, K >= 1024 are formed from exact int8 digit products on the INT8 tensor "
                                      f"cores ({digits} seven-bit digits per operand, {digits_inv} for the inverse's W^T W; error <= 2^-56 of the operand row "
                                      "maxima, parity vs the oracle unchanged), everything else on the FP64 DMMA pipe") if digits > 0 else
                                     "FP64 throughout (DMMA pipe): the condition-number gate kept the INT8 route off for this model",
                       "timing": "CUDA events on the library stream around every evaluation (hp upload .. F, G read back), summed over the K "
                                 "steps, max over ranks; barrier + torch.cuda.synchronize on both sides; wall clock reported beside it"},
            "wall_ms_per_step": t_wall / args.steps * 1e3,
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": base,
            "extra": extra, "F_last": F, "G_norm_last": float(np.linalg.norm(G))}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=N_FULL, help="training-set size (default: the metric's N=32768)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-predict", action="store_true", help="skip the secondary predict metric")
    ap.add_argument("--no-sharded", action="store_true", help="skip the sharded extras (config 4 / config 5 / 3-ext / training)")
    ap.add_argument("--config5-n", type=int, default=None, help="override N of the config-5 extra (default 65536 for 1-2 GPUs, 131072 for 4-8)")
    ap.add_argument("--config5-base", action="store_true", help="1 GPU only: also run config 5 at N = 131072 in place on one GPU (strong-scaling base, ~2.5 min)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write F and G of the last timed evaluation (rank 0) to DIR/F.npy and DIR/G.npy, float64")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the GPU path (--impl b200)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_gpu(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
