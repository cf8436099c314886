"""CPU oracle for the MI-GAN generator forward pass.  TEST INFRASTRUCTURE ONLY.

This file is the *checker*, never the product: only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline / ``--impl reference``
legs may import it.  Nothing under ``mi-gan_b200/`` imports it.

It restates, as plain functions over a ``state_dict`` (no ``nn.Module``), the
algorithm of the reference file ``lib/model_zoo/migan_inference.py`` (all
``file:line`` citations below are relative to the reference checkout).  The
arithmetic is expressed with the same torch CPU primitives the reference uses
(``F.conv2d`` / ``F.leaky_relu`` / ``F.pad`` / nearest up-sampling), so on the same
host it reproduces the reference bit for bit; that is also what makes it a fair
CPU baseline ("port") on a box where the reference checkout is absent.

Parity pin: ``tests/golden/make_golden.py`` imports the real reference in the
build container, loads the same seeded ``state_dict`` into it and asserts this
oracle matches it exactly (max-abs 0.0) at R=64/256/512; the outputs are committed
under ``tests/golden/`` and re-checked by ``tests/test_oracle.py`` on every run.
The reference repository ships no tests, golden tensors or weights of its own
(SURVEY.md F4), so real-checkpoint parity is unpinned; seeded export-style
weights (SURVEY.md section 8c) are the pin.
"""
from __future__ import annotations

import math
from collections import OrderedDict
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch
import torch.nn.functional as F

SQRT2 = float(np.sqrt(2))  # migan_inference.py:14-15 uses np.sqrt(2)


# --------------------------------------------------------------------------- #
# Architecture bookkeeping (migan_inference.py:214-233, 329-345)
# --------------------------------------------------------------------------- #
def channels(res: int, ch_base: int = 32768, ch_max: int = 512) -> int:
    """min(ch_base // res, ch_max) -- migan_inference.py:222-223, 342-343."""
    return min(ch_base // res, ch_max)


def check_resolution(resolution: int) -> int:
    """Power-of-two check, raises ValueError like migan_inference.py:214-216."""
    log2res = int(np.log2(resolution))
    if 2 ** log2res != resolution:
        raise ValueError
    return log2res


def encode_res(resolution: int) -> List[int]:
    """[R, R/2, ..., 4] -- migan_inference.py:217."""
    log2res = check_resolution(resolution)
    return [2 ** i for i in range(log2res, 1, -1)]


def block_res(resolution: int) -> List[int]:
    """[4, 8, ..., R] -- migan_inference.py:332."""
    log2res = check_resolution(resolution)
    return [2 ** i for i in range(2, log2res + 1)]


def setup_filter(f, normalize=True, flip_filter=False, gain=1.0) -> torch.Tensor:
    """Outer-product FIR prototype -- migan_inference.py:31-55 (non-separable branch,
    which is the one a 4-tap prototype takes: numel < 8)."""
    f = torch.as_tensor(f, dtype=torch.float32)
    if f.ndim == 0:
        f = f[None]
    if f.ndim == 1:
        f = torch.outer(f, f)
    if normalize:
        f = f / f.sum()
    if flip_filter:
        f = f.flip([0, 1])
    f = f * (gain ** (f.ndim / 2))
    return f


# --------------------------------------------------------------------------- #
# state_dict layout (SURVEY.md section 8b; verified against the reference by make_golden.py)
# --------------------------------------------------------------------------- #
def _sepconv_keys(prefix, cin, cout, *, res=None, noise=False, down=False, up=False):
    """Key order of SeparableConv2d: parameters first (noise_strength is registered
    last in the ctor but nn.Module lists own params before child params), then
    buffers -- what the reference's state_dict() produces (make_golden.py asserts it)."""
    out = []
    if noise:
        out.append((prefix + "noise_strength", ()))
        out.append((prefix + "noise_const", (res, res)))
    out.append((prefix + "conv1.weight", (cin, 1, 3, 3)))
    out.append((prefix + "conv1.bias", (cin,)))
    out.append((prefix + "conv2.weight", (cout, cin, 1, 1)))
    if down:
        out.append((prefix + "downsample.filter.weight", (cin, 1, 4, 4)))
    if up:
        out.append((prefix + "upsample.filter_const", (1, 1, res, res)))
        out.append((prefix + "upsample.filter.weight", (cout, 1, 4, 4)))
    return out


def state_dict_spec(resolution: int) -> "OrderedDict[str, Tuple[int, ...]]":
    """Ordered {key: shape} of Generator(resolution).state_dict()
    (ctor order synthesis then encoder, migan_inference.py:359-360)."""
    spec = []
    bres = block_res(resolution)
    c4 = channels(4)
    p = "synthesis.b4."
    spec += _sepconv_keys(p + "conv1.", c4, c4)
    spec += _sepconv_keys(p + "conv2.", c4, c4)
    spec += [(p + "torgb.weight", (3, c4, 1, 1)), (p + "torgb.bias", (3,))]
    for ri, rj in zip(bres[:-1], bres[1:]):
        ci, cj = channels(ri), channels(rj)
        p = "synthesis.b%d." % rj
        spec += _sepconv_keys(p + "conv1.", ci, cj, res=rj, noise=True, up=True)
        spec += _sepconv_keys(p + "conv2.", cj, cj, res=rj, noise=True)
        spec += [(p + "torgb.weight", (3, cj, 1, 1)), (p + "torgb.bias", (3,))]
        spec += [(p + "upsample.filter_const", (1, 1, rj, rj)),
                 (p + "upsample.filter.weight", (3, 1, 4, 4))]
    eres = encode_res(resolution)
    for idx, (ri, rj) in enumerate(zip(eres[:-1], eres[1:])):
        ci, cj = channels(ri), channels(rj)
        p = "encoder.b%d." % ri
        if idx == 0:
            spec += [(p + "fromrgb.weight", (ci, 4, 1, 1)), (p + "fromrgb.bias", (ci,))]
        spec += _sepconv_keys(p + "conv1.", ci, ci)
        spec += _sepconv_keys(p + "conv2.", ci, cj, down=True)
    c = channels(eres[-1])
    spec += _sepconv_keys("encoder.b4.conv1.", c, c)
    spec += _sepconv_keys("encoder.b4.conv2.", c, c)
    return OrderedDict(spec)


def make_state_dict(resolution: int, seed: int = 1, *, style: str = "export") -> "OrderedDict[str, torch.Tensor]":
    """Seeded weights with the statistics of a released checkpoint (SURVEY.md 8c).

    style="export": every conv weight (depthwise 3x3, 1x1, fromrgb, torgb) is randn
    normalised to unit L2 norm per output channel -- what
    scripts/export_inference_model.py:26 produces; biases ~ 0.1 randn;
    noise_strength ~ 0.1 randn (ctor default 0 would leave the noise path untested,
    migan_inference.py:150); noise_const ~ randn (ctor :149); FIR taps and
    filter_const at their constructor values (:71-72, :83-85, :95-96).
    style="default": like torch's default Conv2d init scale (small outputs).
    """
    g = torch.Generator().manual_seed(seed)
    sd = OrderedDict()
    f_down = setup_filter([1, 3, 3, 1], gain=1)
    f_up = setup_filter([1, 3, 3, 1], gain=4)
    for key, shape in state_dict_spec(resolution).items():
        if key.endswith("filter.weight"):
            f = f_down if "downsample" in key else f_up
            t = f.repeat(shape[0], 1, 1, 1).clone()
        elif key.endswith("filter_const"):
            w = torch.tensor([[1.0, 0.0], [0.0, 0.0]])
            t = w.repeat(1, 1, shape[2] // 2, shape[3] // 2).clone()
        elif key.endswith("noise_const"):
            t = torch.randn(shape, generator=g)
        elif key.endswith("noise_strength"):
            t = 0.1 * torch.randn(shape, generator=g)
        elif key.endswith(".bias"):
            t = 0.1 * torch.randn(shape, generator=g)
        elif key.endswith(".weight"):
            t = torch.randn(shape, generator=g)
            if style == "export":
                n = t.flatten(1).square().sum(1).add(1e-8).rsqrt()
                t = t * n.view(-1, 1, 1, 1)
            else:
                fan_in = shape[1] * shape[2] * shape[3]
                t = t / math.sqrt(3.0 * fan_in)
        else:  # pragma: no cover
            raise KeyError(key)
        sd[key] = t.contiguous()
    return sd


def make_input(resolution: int, n: int, seed: int = 1234, *, hole: float = 0.4) -> torch.Tensor:
    """Synthetic generator input in the callers' convention:
    x = cat([mask - 0.5, img * mask], 1), mask 1=known / 0=hole, img in [-1, 1]
    (scripts/demo.py:56-66; scripts/evaluate_fid_lpips.py:155-161).  Masks are
    blocky random holes (8x8 cells) so that both hole interiors and edges occur."""
    g = torch.Generator().manual_seed(seed)
    img = torch.rand(n, 3, resolution, resolution, generator=g) * 2 - 1
    cells = max(resolution // 8, 1)
    coarse = (torch.rand(n, 1, cells, cells, generator=g) > hole).float()
    mask = F.interpolate(coarse, size=(resolution, resolution), mode="nearest")
    return torch.cat([mask - 0.5, img * mask], dim=1).contiguous()


# --------------------------------------------------------------------------- #
# The forward pass, restated
# --------------------------------------------------------------------------- #
def lrelu_agc(x: torch.Tensor, alpha=0.2, gain=SQRT2, clamp=256.0) -> torch.Tensor:
    """leaky_relu -> * sqrt(2) -> clamp(+-256) -- migan_inference.py:20-28 with the
    defaults every block uses (:179, :210, :255, :289, :325)."""
    x = F.leaky_relu(x, negative_slope=alpha)
    if gain != 1:
        x = x * gain
    if clamp is not None:
        x = x.clamp(-clamp, clamp)
    return x


def downsample2d(x: torch.Tensor, taps: torch.Tensor) -> torch.Tensor:
    """Depthwise 4x4, stride 2, pad 1 -- migan_inference.py:62-76."""
    return F.conv2d(x, taps, stride=2, padding=1, groups=x.shape[1])


def upsample2d(x: torch.Tensor, taps: torch.Tensor, filter_const: torch.Tensor) -> torch.Tensor:
    """nearest x2 -> * filter_const (zero insertion) -> pad (2,1,2,1) -> depthwise 4x4
    -- migan_inference.py:98-103."""
    x = F.interpolate(x, scale_factor=2, mode="nearest")
    x = x * filter_const
    x = F.pad(x, (2, 1, 2, 1))
    return F.conv2d(x, taps, groups=x.shape[1])


def _tap(taps, name: str, x: torch.Tensor, record: bool = True) -> torch.Tensor:
    """Named intermediate of the forward.  ``taps`` is None, a dict that collects the intermediates (names ``record=False``
    leave out), or an object whose ``visit(name, x)`` returns the tensor the forward continues from
    (``oracle/unit_parity.py`` continues from tensors a kernel produced)."""
    if taps is None:
        return x
    visit = getattr(taps, "visit", None)
    if visit is not None:
        return visit(name, x)
    if record:
        taps[name] = x
    return x


def separable_conv2d(sd: Dict[str, torch.Tensor], p: str, x: torch.Tensor,
                     taps: Optional[dict] = None) -> torch.Tensor:
    """SeparableConv2d.forward -- migan_inference.py:154-170.  Which optional stages
    run is decided by which keys exist under prefix ``p``."""
    x = F.conv2d(x, sd[p + "conv1.weight"], sd[p + "conv1.bias"], padding=1, groups=x.shape[1])
    x = lrelu_agc(x)
    x = _tap(taps, p + "dw_act", x)
    if (p + "downsample.filter.weight") in sd:
        x = downsample2d(x, sd[p + "downsample.filter.weight"])
        x = _tap(taps, p + "down", x)
    x = F.conv2d(x, sd[p + "conv2.weight"])
    x = _tap(taps, p + "pw", x)
    if (p + "upsample.filter.weight") in sd:
        x = upsample2d(x, sd[p + "upsample.filter.weight"], sd[p + "upsample.filter_const"])
    if (p + "noise_const") in sd:
        x = x + sd[p + "noise_const"] * sd[p + "noise_strength"]
    x = lrelu_agc(x)
    return _tap(taps, p + "out", x)


def encoder_forward(sd, x_in: torch.Tensor, resolution: int, taps=None):
    """Encoder.forward / EncoderBlock.forward -- migan_inference.py:235-246, 192-200."""
    feats = {}
    x = None
    eres = encode_res(resolution)
    for idx, res in enumerate(eres[:-1]):
        p = "encoder.b%d." % res
        if idx == 0:  # only the first block has fromrgb (:225-228)
            y = F.conv2d(x_in, sd[p + "fromrgb.weight"], sd[p + "fromrgb.bias"])
            y = lrelu_agc(y)
            x = y if x is None else x + y
            x = _tap(taps, p + "fromrgb", x)
        feat = separable_conv2d(sd, p + "conv1.", x, taps)
        x = separable_conv2d(sd, p + "conv2.", feat, taps)
        feats[res] = feat
    feat = separable_conv2d(sd, "encoder.b4.conv1.", x, taps)
    x = separable_conv2d(sd, "encoder.b4.conv2.", feat, taps)
    feats[4] = feat
    return x, feats


def synthesis_forward(sd, x: torch.Tensor, feats, resolution: int, taps=None) -> torch.Tensor:
    """Synthesis.forward -- migan_inference.py:347-352; blocks :270-279 and :303-315."""
    p = "synthesis.b4."
    x = separable_conv2d(sd, p + "conv1.", x, taps)
    x = _tap(taps, p + "conv1.out_skip", x + feats[4], record=False)
    x = separable_conv2d(sd, p + "conv2.", x, taps)
    img = F.conv2d(x, sd[p + "torgb.weight"], sd[p + "torgb.bias"])
    img = _tap(taps, p + "img", img)
    for res in block_res(resolution)[1:]:
        p = "synthesis.b%d." % res
        x = separable_conv2d(sd, p + "conv1.", x, taps)
        x = x + feats[res]            # skip is added AFTER the activation (:304-305)
        x = _tap(taps, p + "conv1.out_skip", x, record=False)
        x = separable_conv2d(sd, p + "conv2.", x, taps)
        img = upsample2d(img, sd[p + "upsample.filter.weight"], sd[p + "upsample.filter_const"])
        img = img + F.conv2d(x, sd[p + "torgb.weight"], sd[p + "torgb.bias"])
        img = _tap(taps, p + "img", img)
    return img


@torch.no_grad()
def generator_forward(sd: Dict[str, torch.Tensor], x: torch.Tensor, resolution: int,
                      taps: Optional[dict] = None, dtype=torch.float32) -> torch.Tensor:
    """Generator.forward(x[N,4,R,R]) -> img[N,3,R,R] -- migan_inference.py:362-369."""
    if x.dim() != 4 or x.shape[1] != 4 or x.shape[2] != resolution or x.shape[3] != resolution:
        raise ValueError("expected x of shape [N,4,%d,%d], got %s" % (resolution, resolution, tuple(x.shape)))
    if dtype != torch.float32:
        sd = {k: v.to(dtype) for k, v in sd.items()}
        x = x.to(dtype)
    x4, feats = encoder_forward(sd, x, resolution, taps)
    for r, f in feats.items():
        _tap(taps, "feat%d" % r, f)
    return synthesis_forward(sd, x4, feats, resolution, taps)


# --------------------------------------------------------------------------- #
# Op-level oracles (torch_utils/ops) -- used by the standalone upfirdn2d / bias_act kernels
# --------------------------------------------------------------------------- #
def upfirdn2d_ref(x, f, up=1, down=1, padding=(0, 0, 0, 0), flip_filter=False, gain=1.0):
    """torch_utils/ops/upfirdn2d.py:169-208 (_upfirdn2d_ref), 2-D (non-separable) filters
    and 1-D separable filters.  padding = (padx0, padx1, pady0, pady1)."""
    n, c, h, w = x.shape
    upx = upy = up
    downx = downy = down
    if isinstance(up, (tuple, list)):
        upx, upy = up
    if isinstance(down, (tuple, list)):
        downx, downy = down
    if isinstance(padding, int):
        padding = (padding,) * 4
    if len(padding) == 2:
        padding = (padding[0], padding[0], padding[1], padding[1])
    padx0, padx1, pady0, pady1 = padding
    if f is None:
        f = torch.ones([1, 1], dtype=torch.float32)
    x = x.reshape(n, c, h, 1, w, 1)
    x = F.pad(x, [0, upx - 1, 0, 0, 0, upy - 1])
    x = x.reshape(n, c, h * upy, w * upx)
    x = F.pad(x, [max(padx0, 0), max(padx1, 0), max(pady0, 0), max(pady1, 0)])
    x = x[:, :, max(-pady0, 0): x.shape[2] - max(-pady1, 0), max(-padx0, 0): x.shape[3] - max(-padx1, 0)]
    f = f * (gain ** (f.ndim / 2))
    f = f.to(x.dtype)
    if not flip_filter:
        f = f.flip(list(range(f.ndim)))
    f = f[None, None].repeat([c, 1] + [1] * f.ndim)
    if f.ndim == 4:
        x = F.conv2d(x, f, groups=c)
    else:
        x = F.conv2d(x, f.unsqueeze(2), groups=c)
        x = F.conv2d(x, f.unsqueeze(3), groups=c)
    return x[:, :, ::downy, ::downx]


_ACT = {  # torch_utils/ops/bias_act.py:22-32 : name -> (func, def_alpha, def_gain, cuda_idx)
    "linear": (lambda x, a: x, 0.0, 1.0, 1),
    "relu": (lambda x, a: F.relu(x), 0.0, SQRT2, 2),
    "lrelu": (lambda x, a: F.leaky_relu(x, a), 0.2, SQRT2, 3),
    "tanh": (lambda x, a: torch.tanh(x), 0.0, 1.0, 4),
    "sigmoid": (lambda x, a: torch.sigmoid(x), 0.0, 1.0, 5),
    "elu": (lambda x, a: F.elu(x), 0.0, 1.0, 6),
    "selu": (lambda x, a: F.selu(x), 0.0, 1.0, 7),
    "softplus": (lambda x, a: F.softplus(x), 0.0, 1.0, 8),
    "swish": (lambda x, a: torch.sigmoid(x) * x, 0.0, SQRT2, 9),
}


def bias_act_ref(x, b=None, dim=1, act="linear", alpha=None, gain=None, clamp=None):
    """torch_utils/ops/bias_act.py:94-123 (_bias_act_ref)."""
    func, def_alpha, def_gain, _ = _ACT[act]
    alpha = float(def_alpha if alpha is None else alpha)
    gain = float(def_gain if gain is None else gain)
    clamp = float(-1 if clamp is None else clamp)
    if b is not None:
        x = x + b.reshape([-1 if i == dim else 1 for i in range(x.ndim)])
    x = func(x, alpha)
    if gain != 1:
        x = x * gain
    if clamp >= 0:
        x = x.clamp(-clamp, clamp)
    return x
