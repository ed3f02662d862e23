"""Generates tests/golden/*.npz from the CPU oracle (oracle/gpr_oracle.py) with fixed seeds.

The reference (Julia) cannot run in this image and ships no golden vectors of its own (SURVEY.md 8c), so
these fixtures freeze the oracle that was pinned against the reference's identity tests (tests/test_oracle.py).
They serve two purposes: (1) `pytest -m "not gpu"` detects any drift of the oracle, (2) `pytest -m gpu`
compares the CUDA path with committed numbers, not only with an oracle evaluated on the GPU box.

    python tests/golden/make_golden.py
"""
import os
import sys
import zipfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(HERE)), "oracle"))
import gpr_oracle as o  # noqa: E402

CASES = {
    # name: (cov, D, N, M, ny, train_axis, ne, nq, seed)
    "se_noise_d2": ((o.SE, o.NOISE), 2, 96, 40, 1, 1, 6, 9, 101),
    "se_se_noise_d8": ((o.SE, o.SE, o.NOISE), 8, 150, 70, 1, 1, 7, 5, 202),
    "noise_mid_d3_ny3": ((o.SE, o.NOISE, o.SE), 3, 131, 33, 3, 2, 5, 4, 303),
    "se_plain_d1": (o.SE, 1, 64, 50, 1, 1, 4, 8, 404),
    "se_matern_noise_d4": ((o.SE, o.MATERN52, o.NOISE), 4, 120, 30, 1, 1, 5, 5, 505),   # extension: parity unpinned
}


def make(name):
    cov, D, N, M, ny, ta, ne, nq, seed = CASES[name]
    rng = np.random.default_rng(seed)
    x = rng.random((D, N))
    y = np.sin(3 * x).sum(0) + 0.1 * rng.standard_normal(N)
    if ny > 1:
        y = np.stack([(0.5 + 0.4 * k) * y + 0.05 * rng.standard_normal(N) for k in range(ny)], axis=1)
    xp = rng.random((D, M))
    xe, xq = 0.5 * rng.random((D, ne)), 0.5 * rng.random((D, nq))
    hp = 0.4 + 0.8 * rng.random(o.dim_hp(cov, D))
    ks = o.as_list(cov)
    if o.NOISE in ks:   # keep K well conditioned (SURVEY.md M8)
        dims = [o.dim_hp(k, D) for k in ks]
        hp[int(np.cumsum(dims)[ks.index(o.NOISE)]) - 1] = 0.15
    if not o.is_composed(cov):   # jitter-only model: short length scale keeps cond(K) moderate
        hp = np.array([0.9] + [14.0] * D)
    out = dict(x=x, y=y, xp=xp, xe=xe, xq=xq, hp=hp, train_axis=ta)
    out["K_self"] = o.kernel(cov, hp, x)
    out["K_cross"] = o.kernel(cov, hp, x, xp, same=False) if o.is_composed(cov) else o.kernel_single(cov, hp, x, xp, False)
    md = o.GPRModel(cov, hp, x, y, train_axis=ta)
    tc = o.MllGradCache(md)
    F, G = o.loss_grad(hp, md, tc)
    out.update(F=F, G=G, U=tc.kchol_base, alpha=tc.alpha, Kinv=tc.Kinv)
    Fl, Gl = o.log_loss_grad(np.log(hp), md)
    out.update(G_log=Gl)
    for i in sorted({1, 2, len(hp) - 1, len(hp)}):     # a few hyper-parameters keep the fixtures small
        dK = o.grad_kernel(cov, i, hp, x)
        out[f"dK_{i}"] = np.array([dK[1]]) if isinstance(dK, tuple) else dK
    pc = o.GPRPredictCache(md)
    mu, var = o.predict(md, xp, diagonal_var=True, pc=pc)
    _, Sig = o.predict(md, xp, pc=pc)
    out.update(pred_mean=mu, pred_var=var, pred_cov=Sig, wt=pc.wt)
    out["pred_mean_same_x"] = o.predict_mean(md, x, pc=pc, same=True)
    if ny == 1:
        cm = o.Cmap(xe, xq)
        A, B, C = o.split_kernel(cov, hp, cm, x)
        smu, svar = o.split_predict(md, cm, var_range=(1, 3), pc=pc)
        _, svar_all = o.split_predict(md, cm, var_range=(1, ne), pc=pc)
        out.update(split_A=A, split_B=B, split_C=C, split_mean=smu, split_var=svar, split_var_all=svar_all)
    out["cond"] = np.linalg.cond(out["K_self"])
    return out


def save(path, arrays):
    """np.savez_compressed with LZMA in place of deflate (np.load reads both): se_se_noise_d8 stays under 1 MB."""
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_LZMA) as z:
        for key, val in arrays.items():
            with z.open(key + ".npy", "w") as f:
                np.lib.format.write_array(f, np.asanyarray(val), allow_pickle=False)


if __name__ == "__main__":
    for name in CASES:
        d = make(name)
        save(os.path.join(HERE, name + ".npz"), d)
        print(name, "cond(K) = %.2e" % d["cond"], "F =", d["F"])
