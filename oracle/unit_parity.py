"""Launch-by-launch parity of the generator against float64.  TEST INFRASTRUCTURE ONLY.

A *unit* is the work between two tensors a device plan materialises (its debug taps, `Generator.tap_names()`).  The
walker restates the forward with the oracle's building blocks and, wherever the device provided a tensor, records what
float64 arithmetic computes there from the device's own predecessors and then continues from the device tensor.  Each
unit is therefore judged alone, with no error carried in from upstream launches, and no table of which launch fuses what
is needed: a fused launch simply provides fewer tensors.

Bars come from a model, not from a run: the same walk in float32 (CPU) gives each unit's plain-fp32 error against
float64, floored at FLOOR_ULPS fp32 ulps of the unit's largest value; the device's error may be MULT[path] times that.
The multiples are twice the worst ratio oracle/split_model.py models for one contraction at K = 64 .. 512
(tests/test_split_precision.py pins the derivation); the model's float32 reference is the same torch CPU convolution:
  simt     sequential fp32 FMA chains: modelled ratio <= 4.8                       -> 10
  tc       3-pass fp16 hi/lo split, fp32 accumulation: modelled ratio <= 2.9       -> 6
  tc_fast  one fp16 pass: modelled ratio 650 .. 1360                               -> 3000
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, List

import torch

from . import migan_oracle as O

FLOOR_ULPS = 2.0
MULT = {"simt": 10.0, "tc": 6.0, "tc_fast": 3000.0}


class _Substitute:
    """Tap visitor for `migan_oracle.generator_forward`: continues the forward from the given tensors."""

    def __init__(self, given: Dict[str, torch.Tensor], dtype):
        self.given, self.dtype = given, dtype
        self.computed: Dict[str, torch.Tensor] = {}
        self.gemm: Dict[str, bool] = {}
        self._gemm = False

    def visit(self, name: str, x: torch.Tensor) -> torch.Tensor:
        if name.endswith(".pw"):
            self._gemm = True            # a 1x1 contraction ran since the last given tensor
        t = self.given.get(name)
        if t is None:
            return x
        self.computed[name] = x
        self.gemm[name] = self._gemm
        self._gemm = False
        return t.to(self.dtype)


def walk(sd, x: torch.Tensor, resolution: int, given: Dict[str, torch.Tensor], dtype=torch.float64) -> _Substitute:
    """Forward in `dtype`, continuing from `given` ({tap name: NCHW tensor of the images in x}) wherever it has a tensor."""
    sub = _Substitute(given, dtype)
    O.generator_forward(sd, x, resolution, taps=sub, dtype=dtype)
    return sub


def fp32_ulp(v: float) -> float:
    return 2.0 ** (math.floor(math.log2(v)) - 23) if v > 0 else 2.0 ** -149


@dataclass
class Unit:
    name: str
    err: float        # max |device - float64|
    ref_err: float    # max |float32 - float64|, floored at FLOOR_ULPS ulps of `scale`
    scale: float      # max |float64|
    gemm: bool        # the unit contains a 1x1 contraction

    @property
    def ratio(self) -> float:
        return self.err / self.ref_err


def unit_errors(sd, x: torch.Tensor, resolution: int, given: Dict[str, torch.Tensor]) -> List[Unit]:
    """One Unit per given tensor, in the order given.  A tensor the forward never produces raises KeyError; a non-finite
    device value gives err = inf."""
    w64 = walk(sd, x, resolution, given, torch.float64)
    w32 = walk(sd, x, resolution, given, torch.float32)
    unknown = [k for k in given if k not in w64.computed]
    if unknown:
        raise KeyError("the forward produces no tensor named %s" % unknown)
    units = []
    for name, dev in given.items():
        ref = w64.computed[name]
        if dev.shape != ref.shape:
            raise ValueError("%s: device shape %s, reference %s" % (name, tuple(dev.shape), tuple(ref.shape)))
        dev = dev.double()
        err = float((dev - ref).abs().max()) if bool(torch.isfinite(dev).all()) else math.inf
        scale = float(ref.abs().max())
        e32 = float((w32.computed[name].double() - ref).abs().max())
        units.append(Unit(name, err, max(e32, FLOOR_ULPS * fp32_ulp(scale)), scale, w64.gemm[name]))
    return units


def failures(units: List[Unit], mult: float) -> List[Unit]:
    return [u for u in units if not u.err <= mult * u.ref_err]


def report(units: List[Unit]) -> str:
    worst = max(units, key=lambda u: u.ratio)
    return "%d units, worst ratio %.2f at %s (err %.3e, fp32 %.3e, scale %.3g)" % (
        len(units), worst.ratio, worst.name, worst.err, worst.ref_err, worst.scale)
