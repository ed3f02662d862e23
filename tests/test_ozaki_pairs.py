"""The INT8 product kernels as CTA pairs (csrc/ozaki_i8.cuh, tcgen05 cta_group::2, launch flag 2048 / context option "ozaki_pair")
return the same bits as the single-CTA kernels: the integer accumulation is exact and the epilogue's order is unchanged, so any
difference is a fault of the pair protocol (which CTA loads which half of op(B), which tiles a pair skips, the ghost CTA of an odd
row-tile count), not rounding."""
import importlib.util
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
PAIR = 2048

# (S, M, N, K, flags, beta, shared operands)
CASES = [
    (8, 512, 384, 1024, 0, 0.0, False),        # single pass, even row tiles, M != N
    (8, 384, 512, 1024, 0, 1.0, False),        # odd row tiles: the last pair's second CTA is a ghost
    (7, 640, 256, 512, 0, 1.0, False),
    (6, 256, 640, 768, 0, 0.0, False),
    (8, 640, 640, 640, 1, 0.0, True),          # upper only: a pair straddling the diagonal keeps its lower CTA as a ghost
    (8, 512, 512, 512, 2, 1.0, False),         # K-from-N: both CTAs share the column tile's first k-tile
    (8, 640, 640, 640, 3, 0.0, True),          # upper + K-from-N with shared planes (lauum's form)
    (8, 512, 640, 1024, 64, 1.0, False),       # skip tile (0,0): the leader of the first pair computes and stores nothing
    (8, 384, 384, 384, 1 | 64, 0.0, True),
    (8, 512, 384, 1024, 512, 0.0, False),      # 8-digit two windows
    (8, 640, 512, 2048, 512, 1.0, False),
    (8, 640, 640, 640, 512 | 3, 1.0, True),
    (8, 512, 512, 512, 512 | 64, 0.0, False),
    (9, 640, 640, 1024, 0, 0.0, True),         # nine digits: 96-wide tiles, the last one partial
    (9, 384, 640, 512, 0, 1.0, False),
    (9, 640, 640, 640, 3, 0.0, True),
    (9, 640, 640, 640, 1, 1.0, False),
]


@pytest.mark.parametrize("S,M,N,K,flags,beta,shared", CASES, ids=[f"S{c[0]}-{c[1]}x{c[2]}x{c[3]}-f{c[4]}-b{int(c[5])}{'-sh' if c[6] else ''}" for c in CASES])
def test_pair_kernels_bit_identical(gpr, S, M, N, K, flags, beta, shared):
    from gpr_sm100a import _ffi
    rng = np.random.default_rng(1000 * S + M + N + K + flags)
    A = np.asfortranarray(rng.standard_normal((K, M)) * np.exp(rng.uniform(-8, 0, (K, M))))
    B = A if shared else np.asfortranarray(rng.standard_normal((K, N)))
    C0 = np.asfortranarray(rng.standard_normal((M, N)))
    ctx = gpr.Context(0)
    try:
        C1, _ = _ffi.dbg_ozaki_dgemm(ctx, -1.0, A, B, beta, C0, S=S, flags=flags)
        C2, _ = _ffi.dbg_ozaki_dgemm(ctx, -1.0, A, B, beta, C0, S=S, flags=flags | PAIR)
    finally:
        ctx.close()
    assert np.all(np.isfinite(C1))
    assert not np.array_equal(C1, C0)
    assert np.array_equal(C1, C2), f"max |diff| {np.abs(C1 - C2).max():.3e}"


def test_pair_route_same_bits_on_a_model(gpr):
    """The automatic route of an N = 8192 model (config 2 of the goldens: 8 digits for potrf / trtri, 9 for the inverse's W^T W)
    returns the same F and G bits with "ozaki_pair" = 0 and 1."""
    from gpr_sm100a import _ffi
    spec = importlib.util.spec_from_file_location("mg2", os.path.join(HERE, "golden", "make_golden_config2.py"))
    mg2 = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg2)
    x, y, sets = mg2.inputs()
    hp = sets["A"]
    ctx = gpr.Context(0)
    try:
        out = {}
        for pair in (0, 1):
            ctx.set_option("ozaki_pair", pair)
            mh = _ffi.ModelHandle(ctx, [1, 2], x.shape[0], np.asfortranarray(x), y)
            F, G = mh.nlml_grad(hp)
            out[pair] = (F, G.copy(), mh.route())
            mh.close()
    finally:
        ctx.close()
    assert out[0][2] == out[1][2] and out[0][2][0] > 0, out[0][2]      # the INT8 route was taken both times
    assert out[0][0] == out[1][0]
    assert np.array_equal(out[0][1], out[1][1])
