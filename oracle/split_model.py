"""numpy model of the tensor-core 1x1 contraction (DESIGN.md section 3).  TEST INFRASTRUCTURE ONLY.

The 1x1 convs run on fp16 tensor cores as  Ah*Bh + Al*Bh + Ah*Bl  with fp32 accumulation, where (hi, lo) are fp16
pairs of power-of-two-scaled operands: activations * 64, split by truncation in the kernel's prologue; weights * 2^k
(max |w * 2^k| in [8192, 16384)), split by rounding on the host.  `tc_fast` runs the Ah*Bh pass alone.

fp16 x fp16 products are exact in fp32, so a float32 matrix product of the fp16 operands emulates one pass.
"""
from __future__ import annotations

import numpy as np

ACT_SCALE = 64.0
TERMS_3PASS = ("hh", "lh", "hl")   # Ah*Bh, Al*Bh, Ah*Bl
TERMS_1PASS = ("hh",)


def split_trunc(s):
    """Prologue split (sepconv_stages.cuh split_pack2): hi32 = s with the low 13 mantissa bits cleared, hi = fp16(hi32),
    lo = fp16(s - hi32).  hi == hi32 except below the fp16 normal range (|s| < 2^-14, an activation below 1e-6)."""
    s = np.asarray(s, dtype=np.float32)
    hi32 = (s.view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)
    hi = hi32.astype(np.float16)
    lo = (s - hi32).astype(np.float16)
    return hi, lo


def split_round(s):
    """Host-side weight split (migan_abi.cu pack_sepconv): hi = fp16(s), lo = fp16(s - hi)."""
    s = np.asarray(s, dtype=np.float32)
    hi = s.astype(np.float16)
    lo = (s - hi.astype(np.float32)).astype(np.float16)
    return hi, lo


def weight_shift(w) -> int:
    """k of the weight scale 2^k: max |w * 2^k| in [8192, 16384)."""
    return int(np.floor(np.log2(16384.0 / np.abs(w).max())))


def tc_matmul(a, w, terms=TERMS_3PASS):
    """a [M, K] float32 activations, w [N, K] float32 weights -> a @ w.T [M, N] float32 as the tensor-core kernel
    forms it from the listed terms.  terms=TERMS_1PASS is the single fp16 pass (rounded operands, no correction)."""
    a = np.asarray(a, dtype=np.float32)
    w = np.asarray(w, dtype=np.float32)
    k2 = weight_shift(w)
    a_s, w_s = a * np.float32(ACT_SCALE), w * np.float32(2.0 ** k2)
    if tuple(terms) == TERMS_1PASS:
        ah, al = a_s.astype(np.float16), None
    else:
        ah, al = split_trunc(a_s)
    wh, wl = split_round(w_s)
    ops = {"hh": (ah, wh), "lh": (al, wh), "hl": (ah, wl)}
    acc = np.zeros((a.shape[0], w.shape[0]), dtype=np.float32)
    for t in terms:
        x, y = ops[t]
        acc += x.astype(np.float32) @ y.astype(np.float32).T
    return acc * np.float32(1.0 / (ACT_SCALE * 2.0 ** k2))


def sequential_fp32_matmul(a, w):
    """a @ w.T accumulated one k at a time in fp32, as a CUDA-core kernel's FMA chain does."""
    a = np.asarray(a, dtype=np.float32)
    w = np.asarray(w, dtype=np.float32)
    acc = np.zeros((a.shape[0], w.shape[0]), dtype=np.float32)
    for k in range(a.shape[1]):
        acc += np.outer(a[:, k], w[:, k]).astype(np.float32)
    return acc


def operands(K: int, seed: int, M: int = 4096, N: int = 256):
    """Post-activation activations (clamped to +-256) and unit-L2-norm weight rows (export style)."""
    rng = np.random.default_rng(seed)
    a = np.clip(rng.standard_normal((M, K)) * 2.0, -256, 256).astype(np.float32)
    w = rng.standard_normal((N, K)).astype(np.float32)
    w /= np.sqrt((w * w).sum(1, keepdims=True))
    return a, w


def error_ratios(K: int, seed: int = 0):
    """Max-abs errors against float64 of the 3-pass, the 1-pass and the sequential-fp32 contraction, each over the
    max-abs error of torch's CPU float32 1x1 convolution -- the float32 evaluation oracle/unit_parity.py bounds launches
    by.  Its blocked reduction is up to ~2x more accurate than a BLAS product or an FMA chain at K >= 256, so the M x N
    sample must be about as large as a layer's for the maxima to compare like for like."""
    import torch
    import torch.nn.functional as F

    a, w = operands(K, seed)
    exact = a.astype(np.float64) @ w.astype(np.float64).T
    conv = F.conv2d(torch.from_numpy(np.ascontiguousarray(a.T)).reshape(1, K, -1, 1), torch.from_numpy(w)[:, :, None, None])
    err = lambda y: np.abs(np.asarray(y, dtype=np.float64) - exact).max()
    e32 = err(conv[0, :, :, 0].T.numpy())
    return {"tc": err(tc_matmul(a, w)) / e32, "tc_fast": err(tc_matmul(a, w, TERMS_1PASS)) / e32,
            "simt": err(sequential_fp32_matmul(a, w)) / e32}
