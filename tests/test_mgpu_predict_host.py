"""CPU check of the block-cyclic prediction driver (gpr::DistPredict, csrc/dist_blocked.hpp) on simulated ranks with the
plain-loop backend (tests/hostlogic/dist_predict.cpp): the explicit-inverse quadratic form and the mean against numpy.
The CUDA library instantiates the same template."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import gpr_oracle as o

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def hp_lib(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("hlp") / "libdist_predict_test.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", out,
                           os.path.join(HERE, "hostlogic", "dist_predict.cpp")])
    L = ctypes.CDLL(out)
    L.hl_dist_predict.restype = ctypes.c_longlong
    return L


def dp(a):
    return None if a is None else a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def run(L, K, Y, Kt, nb, G, tile, want_var=True, dense=False):
    N, ny = Y.shape
    M = Kt.shape[1]
    K, Y, Kt = (np.asfortranarray(a, dtype=np.float64) for a in (K, Y, Kt))
    mean = np.empty((M, ny), order="F")
    quad = np.empty(M) if want_var else None
    XX = np.empty((M, M), order="F") if dense else None
    sums = ctypes.c_longlong(0)
    info = L.hl_dist_predict(dp(K), ctypes.c_int64(N), ctypes.c_int64(nb), G, dp(Y), ny, dp(Kt), ctypes.c_int64(M),
                             ctypes.c_int64(tile), dp(mean), dp(quad), dp(XX), ctypes.byref(sums))
    assert info == 0
    return mean, quad, XX, sums.value


def model(N, M, D, ny, seed, same_x=False):
    rng = np.random.default_rng(seed)
    cov = (o.SE, o.NOISE)
    hp = np.concatenate([[1.0], 0.8 + 0.4 * rng.random(D), [0.1]])
    x = rng.random((D, N))
    xp = x if same_x else rng.random((D, M))
    y = np.stack([np.sin(3 * x).sum(0) * (0.5 + 0.3 * k) for k in range(ny)], axis=1)
    K = o.kernel(cov, hp, x)
    Kt = o.kernel(cov, hp, xp, x, same=same_x).T          # K(x, xp): training index fastest
    return K, y, Kt


def check(K, Y, Kt, mean, quad, XX):
    Kinv = np.linalg.inv(K)
    S = Kt.T @ Kinv @ Kt
    mref = Kt.T @ Kinv @ Y
    scale = np.abs(mref).max()
    assert np.abs(mean - mref).max() <= 1e-9 * scale
    if quad is not None:
        assert np.abs(quad - np.diag(S)).max() <= 1e-9 * np.abs(np.diag(S)).max()
    if XX is not None:
        assert np.abs(XX - S).max() <= 1e-9 * np.abs(S).max()


@pytest.mark.parametrize("G", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("nb", [128, 256])
def test_dist_predict_rank_counts(hp_lib, G, nb):
    """N = 700 is no multiple of nb; at nb = 256 (3 blocks) G = 4, 5 leave ranks without a block.  M = 300 in tiles of 128."""
    K, Y, Kt = model(700, 300, 3, 1, 10 * G + nb)
    mean, quad, _, sums = run(hp_lib, K, Y, Kt, nb, G, 128)
    assert sums == 3
    check(K, Y, Kt, mean, quad, None)


@pytest.mark.parametrize("G", [1, 3, 5])
def test_dist_predict_dense(hp_lib, G):
    K, Y, Kt = model(300, 200, 2, 1, G)
    mean, quad, XX, sums = run(hp_lib, K, Y, Kt, 128, G, 200, dense=True)
    assert sums == 1
    check(K, Y, Kt, mean, quad, XX)


def test_dist_predict_matrix_y(hp_lib):
    """ny = 3 (the mean covers every column; train_axis only selects the training column of the loss)"""
    K, Y, Kt = model(500, 260, 4, 3, 7)
    mean, quad, XX, _ = run(hp_lib, K, Y, Kt, 128, 3, 260, dense=True)
    check(K, Y, Kt, mean, quad, XX)


def test_dist_predict_mean_only(hp_lib):
    K, Y, Kt = model(400, 129, 2, 2, 3)
    mean, _, _, _ = run(hp_lib, K, Y, Kt, 128, 2, 128, want_var=False)
    check(K, Y, Kt, mean, None, None)


@pytest.mark.parametrize("G", [2, 4])
def test_dist_predict_same_x(hp_lib, G):
    """xp === x: K(x, xp) carries the jitter on its diagonal; the variance is then small and the quadratic form must
    resolve it (posterior variance = prior - quad, compared as such)."""
    K, Y, Kt = model(384, 384, 3, 1, G, same_x=True)
    mean, quad, XX, _ = run(hp_lib, K, Y, Kt, 128, G, 384, dense=True)
    check(K, Y, Kt, mean, quad, XX)
    prior = 1.0 + 0.01
    vref = prior - np.diag(Kt.T @ np.linalg.solve(K, Kt))
    assert np.abs((prior - quad) - vref).max() <= 1e-9 * prior
