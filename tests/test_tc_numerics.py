"""CPU emulation of the operand split the tcgen05 GEMM uses, to pin the precision claim made in csrc/gemm_tc.cu
(3xTF32: hi*hi + lo*hi + hi*lo) independently of any GPU: with exact accumulation the split product must reproduce the
fp32 product far inside the 1e-5 parity budget, and a plain single-TF32 product must NOT (which is why the split exists).
The tensor core's truncating fp32 accumulate is a separate, measured effect (gemm_tc.cu header)."""
import numpy as np


def tf32_rna(x):
    """cvt.rna.tf32.f32: keep 10 mantissa bits, round to nearest, ties away from zero (sign-magnitude add)."""
    u = np.asarray(x, dtype=np.float32).view(np.uint32)
    return ((u + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)


def _case(seed, M, N, K, wscale):
    g = np.random.default_rng(seed)
    a = (g.standard_normal((M, K)) * wscale).astype(np.float32)     # weights ~ U(-1/sqrt(H), 1/sqrt(H)) scale
    b = np.tanh(g.standard_normal((N, K))).astype(np.float32)      # states in (-1, 1)
    return a, b, a.astype(np.float64) @ b.astype(np.float64).T


def test_rounding_helpers_are_what_the_ptx_conversions_do():
    x = np.float32(1.0) + np.float32(2.0 ** -11)                    # exactly half an ulp of tf32 above 1.0
    assert tf32_rna(x) == np.float32(1.0 + 2.0 ** -10)              # ties away from zero
    assert tf32_rna(-x) == np.float32(-(1.0 + 2.0 ** -10))
    v = np.float32(0.123456789)
    assert abs(tf32_rna(v) - v) <= abs(v) * 2.0 ** -11


def test_3xtf32_split_reproduces_the_fp32_product_and_single_tf32_does_not():
    a, b, exact = _case(0, 96, 16, 1024, 0.06)
    ah, bh = tf32_rna(a), tf32_rna(b)
    al, bl = a - ah, b - bh                                          # exact in fp32
    assert np.all(al.astype(np.float64) + ah == a) and np.all(bl.astype(np.float64) + bh == b)
    d64 = lambda x, y: x.astype(np.float64) @ y.astype(np.float64).T  # noqa: E731
    split = d64(ah, bh) + d64(al, bh) + d64(ah, bl)
    single = d64(ah, bh)
    scale = np.abs(exact).max()
    assert np.abs(split - exact).max() / scale < 5e-7               # dropped lo*lo ~ 2^-22
    assert np.abs(single - exact).max() / scale > 2e-5              # plain TF32 misses the 1e-5 budget

