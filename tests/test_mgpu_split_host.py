"""CPU check of the split-prediction drivers of the block-cyclic model (csrc/dist_blocked.hpp: split_slab, DistSplitMean,
DistPredict with quad_only) on simulated ranks with the plain-loop backend (tests/hostlogic/dist_split.cpp), against numpy.
The CUDA library instantiates the same templates."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import gpr_oracle as o

HERE = os.path.dirname(os.path.abspath(__file__))
_i64 = ctypes.c_int64


@pytest.fixture(scope="module")
def hs_lib(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("hls") / "libdist_split_test.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", out,
                           os.path.join(HERE, "hostlogic", "dist_split.cpp")])
    L = ctypes.CDLL(out)
    L.hl_split_mean.restype = ctypes.c_longlong
    L.hl_split_var.restype = ctypes.c_longlong
    return L


def dp(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def rup(v, m=128):
    return (v + m - 1) // m * m


def slabs(L, cols, G):
    out = []
    for r in range(G):
        q0, qn = _i64(0), _i64(0)
        L.hl_split_slab(_i64(cols), G, r, ctypes.byref(q0), ctypes.byref(qn))
        out.append((q0.value, qn.value))
    return out


@pytest.mark.parametrize("G", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("cols", [128, 256, 640, 1024, 4096])
def test_slab_partition(hs_lib, G, cols):
    """Every column of the chunk exactly once, contiguous slabs of whole 128-column tiles in rank order, widths within one
    tile of each other; with fewer tiles than ranks the last ranks get none."""
    s = slabs(hs_lib, cols, G)
    pos = 0
    for q0, qn in s:
        assert q0 % 128 == 0 and qn % 128 == 0 and qn >= 0
        if qn:
            assert q0 == pos
        pos += qn
    assert pos == cols
    widths = [qn for _, qn in s]
    assert max(widths) - min(widths) <= 128
    tiles = cols // 128
    assert sum(1 for w in widths if w == 0) == max(0, G - tiles)


def split_operands(ne, nq, N, Np, nk, seed):
    """Padded A (nep x nqp x nk), B^T (Np x nep x nk), C (Np x nqp x nk), alpha (Np): zero outside the valid ranges, as built"""
    rng = np.random.default_rng(seed)
    nep, nqp = rup(ne), rup(nq)
    A = np.zeros((nep, nqp, nk), order="F")
    Bt = np.zeros((Np, nep, nk), order="F")
    Cc = np.zeros((Np, nqp, nk), order="F")
    A[:ne, :nq] = rng.random((ne, nq, nk))
    Bt[:N, :ne] = rng.random((N, ne, nk))
    Cc[:N, :nq] = rng.random((N, nq, nk))
    alpha = np.zeros(Np)
    alpha[:N] = rng.standard_normal(N)
    return A, Bt, Cc, alpha


@pytest.mark.parametrize("G,ne,nq,N,slab", [(1, 130, 300, 200, 128), (2, 100, 300, 200, 128), (3, 257, 700, 300, 256),
                                            (4, 64, 200, 150, 128), (5, 129, 384, 128, 1024), (3, 50, 1000, 260, 384)])
def test_split_mean_chunks(hs_lib, G, ne, nq, N, slab):
    """ne, nq no multiples of 128; nq < 128 G leaves ranks without a slab (G = 4, 5); slab 128 forces several chunks."""
    nk = 2
    Np = rup(N, 256)   # the training padding of the distributed model (nb = 256)
    A, Bt, Cc, alpha = split_operands(ne, nq, N, Np, nk, 31 * G + ne)
    Cw = np.asfortranarray(alpha[:, None, None] * Cc)
    nep, nqp = A.shape[0], A.shape[1]
    mean = np.full((nep, nqp), np.nan, order="F")
    sums = hs_lib.hl_split_mean(G, nk, _i64(Np), _i64(nep), _i64(nqp), dp(Bt), dp(A), dp(Cw), _i64(slab), dp(mean))
    cols = min(nqp, slab * G)
    assert sums == -(-nqp // cols)
    ref = sum(A[:, :, k] * (Bt[:, :, k].T @ np.diag(alpha) @ Cc[:, :, k]) for k in range(nk))
    assert np.abs(mean - ref).max() <= 1e-12 * np.abs(ref).max()
    assert np.all(mean[ne:] == 0) and np.all(mean[:, nq:] == 0)


@pytest.mark.parametrize("G,nb,ne,nq,N,e_lo,e_hi,mt", [(1, 128, 5, 130, 300, 1, 3, 512), (3, 128, 7, 100, 300, 2, 6, 256),
                                                      (2, 256, 4, 260, 500, 1, 4, 1024), (5, 256, 3, 40, 600, 3, 3, 128),
                                                      (3, 128, 6, 300, 400, 2, 5, 128), (2, 128, 4, 400, 300, 1, 4, 256)])
def test_split_var_rows_quad_only(hs_lib, G, nb, ne, nq, N, e_lo, e_hi, mt):
    """The var_range rows as ordinary test points: DistPredict with quad_only gives diag(Kt^T K^-1 Kt) and sums one tile per
    call (nothing else written).  Tiles of mt points: several rows per tile when a whole row fits, else one row and a slab of
    its q columns (mt = 128, 256 below nqp); at nb = 256, N = 600 G = 5 leaves ranks without a block."""
    rng = np.random.default_rng(G + 10 * nb + N)
    D, nk = 3, 2
    x = rng.random((D, N))
    hp = np.concatenate([[1.0], 0.8 + 0.4 * rng.random(D), [0.1]])
    K = np.asfortranarray(o.kernel((o.SE, o.NOISE), hp, x))
    Np = rup(N, nb)
    A, Bt, Cu, _ = split_operands(ne, nq, N, Np, nk, N + 3)
    nqp, erows = A.shape[1], e_hi - e_lo + 1
    quad = np.full(ne * nq, -7.0)
    tiles = hs_lib.hl_split_var(dp(K), _i64(N), _i64(nb), G, _i64(ne), _i64(nq), nk, dp(A), dp(Bt), dp(Cu), _i64(e_lo), _i64(e_hi),
                                _i64(mt), dp(quad))
    w = min(nqp, mt)
    assert tiles == -(-nqp // w) * -(-erows // min(erows, max(1, mt // w)))
    Kinv = np.linalg.inv(K)
    q2 = quad.reshape(ne, nq)
    for e in range(ne):
        if not (e_lo - 1 <= e < e_hi):
            assert np.all(q2[e] == -7.0)
            continue
        Kt = sum(A[e, :nq, k][None, :] * Bt[:N, e, k][:, None] * Cu[:N, :nq, k] for k in range(nk))   # N x nq
        ref = np.einsum("sq,st,tq->q", Kt, Kinv, Kt)
        assert np.abs(q2[e] - ref).max() <= 1e-9 * np.abs(ref).max()
