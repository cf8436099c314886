"""Numerical model of the fp32-faithful tensor-core scheme (DESIGN.md section 3), checked on the CPU.

The 1x1 convs run on fp16 tensor cores as  Ah*Bh + Al*Bh + Ah*Bl  with fp32 accumulation, where
(hi, lo) are fp16 pairs of power-of-two-scaled operands.  This test emulates that arithmetic with numpy
(fp16 operands, exact fp16xfp16 products, fp32 accumulation) and pins the properties the kernels rely on:
  * the truncation split used in the prologue (hi = mantissa-masked value, lo = fp16(s - hi)) carries
    ~22 significant bits and hi is exactly representable in fp16 for |s| <= 16384,
  * the 3-pass contraction is ~1000x more accurate than a single fp16 pass (SURVEY F5) and within the
    same order as a plain fp32 dot product,
  * the chosen scales (activations * 64, weights * 2^k with max|w*2^k| in [8192, 16384)) stay inside fp16 range.
"""
import numpy as np
import pytest

from oracle import unit_parity as U
from oracle.split_model import error_ratios, split_round, split_trunc


def dot32(a16, b16):
    """fp16 x fp16 products are exact in fp32; accumulate in fp32 (order as numpy's pairwise sum)."""
    return (a16.astype(np.float32) * b16.astype(np.float32)).sum(axis=-1, dtype=np.float32)


def test_three_pass_split_is_fp32_faithful():
    rng = np.random.default_rng(0)
    K, M, N = 512, 256, 64
    a = np.clip(rng.standard_normal((M, K)) * 2.0, -256, 256).astype(np.float32)          # post-activation range
    w = rng.standard_normal((N, K)).astype(np.float32)
    w /= np.sqrt((w * w).sum(1, keepdims=True))                                            # unit-L2 rows (export style)
    exact = a.astype(np.float64) @ w.astype(np.float64).T
    k2 = int(np.floor(np.log2(16384.0 / np.abs(w).max())))
    a_s, w_s = a * np.float32(64.0), w * np.float32(2.0 ** k2)
    assert np.abs(a_s).max() <= 16384 and 8192 <= np.abs(w_s).max() < 16384
    ah, al = split_trunc(a_s)
    assert np.array_equal(ah.astype(np.float32), (a_s.view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32))
    wh, wl = split_round(w_s)
    inv = np.float32(1.0 / (64.0 * 2.0 ** k2))
    main = np.stack([dot32(ah[:, None, :], wh[None, :, :])])[0]
    corr = dot32(al[:, None, :], wh[None, :, :]) + dot32(ah[:, None, :], wl[None, :, :])
    three = (main + corr) * inv
    one = main * inv
    fp32 = (a[:, None, :] * w[None, :, :]).sum(-1, dtype=np.float32)
    e3 = np.abs(three - exact).max()
    e1 = np.abs(one - exact).max()
    e32 = np.abs(fp32 - exact).max()
    scale = np.abs(exact).max()
    assert e3 < 5e-6 * scale                     # ~fp32 level
    assert e3 < 20 * max(e32, 1e-7 * scale)      # same order as a plain fp32 dot product
    assert e1 > 100 * e3                         # the single fp16 pass is orders of magnitude worse


def test_truncation_split_keeps_22_bits():
    """|hi + lo - s| <= 2^-22 |s|, floored by half an fp16 subnormal ulp (2^-25 in SCALED units, i.e. 5e-10 of an
    activation): tiny values lose relative, never absolute, precision."""
    rng = np.random.default_rng(1)
    s = (rng.standard_normal(100000) * 300).astype(np.float32)
    s = np.clip(s, -16384, 16384)
    hi, lo = split_trunc(s)
    rec = hi.astype(np.float64) + lo.astype(np.float64)
    err = np.abs(rec - s.astype(np.float64))
    assert np.all(err <= np.maximum(2.0 ** -22 * np.abs(s), 2.0 ** -25))


@pytest.fixture(scope="module")
def modelled_ratios():
    """{path: (least, worst) ratio} of a contraction's max-abs error to that of torch's CPU float32 1x1 convolution, over
    K = 64 .. 512 (the layers' Cin) and three seeds."""
    worst = {}
    for K in (64, 128, 256, 512):
        for seed in range(3):
            for path, r in error_ratios(K, seed).items():
                worst.setdefault(path, []).append(r)
    return {path: (min(rs), max(rs)) for path, rs in worst.items()}


def test_launch_parity_multiples_follow_the_model(modelled_ratios):
    """tests/test_launch_parity_gpu.py bounds each launch by MULT[path] x the unit's float32 error.  The multiples were set
    at 2x the worst modelled ratio; 1.5x is required here because the float32 reference's reduction order depends on the
    CPU.  The 3-pass bar stays far below what a single fp16 pass reaches."""
    print({path: "%.2f .. %.2f" % r for path, r in modelled_ratios.items()})
    for path in ("simt", "tc", "tc_fast"):
        assert U.MULT[path] >= 1.5 * modelled_ratios[path][1], path
    assert U.MULT["tc"] <= 3 * modelled_ratios["tc"][1]                 # ... and not much more
    assert modelled_ratios["tc_fast"][0] > 50 * U.MULT["tc"]
