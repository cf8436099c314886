"""The launch-by-launch float64 walker (oracle/unit_parity.py) on the CPU: it accepts the oracle's own float32
intermediates, and its `tc` bar names the one unit whose 1x1 contraction was replaced by a numpy emulation of a broken
tensor-core kernel (a single fp16 pass, or the 3-pass split without its Al*Bh correction) while a faithful 3-pass
emulation passes.  tests/test_launch_parity_gpu.py applies the same walker to the device's tensors."""
import math

import numpy as np
import pytest
import torch

from oracle import migan_oracle as O
from oracle import split_model as S
from oracle import unit_parity as U

R, N = 16, 2


@pytest.fixture(scope="module")
def oracle_run():
    sd = O.make_state_dict(R, seed=1)
    x = O.make_input(R, N, seed=3)
    taps = {}
    O.generator_forward(sd, x, R, taps=taps)
    return sd, x, taps


def coarse_layout(sd, taps):
    """What a fused tensor-core plan materialises: the stem, each layer's final output (the raw 1x1 output of up-sampling
    layers) and each level's image."""
    given = {}
    for name, t in taps.items():
        p = name.rsplit(".", 1)[0] + "."
        if name.endswith(".fromrgb") or name.endswith(".img"):
            given[name] = t
        elif name.endswith(".pw") and (p + "upsample.filter.weight") in sd:
            given[name] = t
        elif name.endswith(".out") and (p + "upsample.filter.weight") not in sd:
            given[name] = t
    return given


def test_oracle_intermediates_pass(oracle_run):
    sd, x, taps = oracle_run
    for given in (coarse_layout(sd, taps), {k: v for k, v in taps.items() if not k.startswith("feat")}):
        units = U.unit_errors(sd, x, R, given)
        assert [u.name for u in units] == list(given)
        assert not U.failures(units, 1.0), U.report(units)       # the float32 walk recomputes them exactly
        assert sum(u.gemm for u in units) == sum(k.endswith(".pw") for k in taps)


class _BrokenContraction:
    """Tap visitor: the oracle forward with layer p's 1x1 contraction computed by the tensor-core model from `terms`, as
    a kernel with that defect would run it; every intermediate downstream follows from the broken one."""

    def __init__(self, sd, p, terms):
        self.w = sd[p + "conv2.weight"][:, :, 0, 0].numpy()
        self.p, self.terms, self.taps = p, terms, {}

    def visit(self, name, x):
        if name in (self.p + "dw_act", self.p + "down"):
            self.a = x
        elif name == self.p + "pw":
            n, k, h, w = self.a.shape
            y = S.tc_matmul(self.a.permute(0, 2, 3, 1).reshape(-1, k).numpy(), self.w, self.terms)
            x = torch.from_numpy(y).reshape(n, h, w, -1).permute(0, 3, 1, 2).contiguous()
        self.taps[name] = x
        return x


def planted(sd, x, p, terms):
    broken = _BrokenContraction(sd, p, terms)
    O.generator_forward(sd, x, R, taps=broken)
    unit = p + ("pw" if (p + "upsample.filter.weight") in sd else "out")
    return coarse_layout(sd, broken.taps), unit


@pytest.mark.parametrize("layer", ["encoder.b16.conv2.", "encoder.b4.conv1.", "synthesis.b16.conv1.", "synthesis.b16.conv2."])
def test_tc_bar_names_a_broken_contraction(oracle_run, layer):
    sd, x, taps = oracle_run
    given, name = planted(sd, x, layer, S.TERMS_3PASS)
    units = U.unit_errors(sd, x, R, given)
    assert not U.failures(units, U.MULT["tc"]), U.report(units)             # the faithful split is inside the bar
    for terms in (S.TERMS_1PASS, ("hh", "hl")):                             # single fp16 pass; Al*Bh dropped
        given, name = planted(sd, x, layer, terms)
        units = U.unit_errors(sd, x, R, given)
        assert [u.name for u in U.failures(units, U.MULT["tc"])] == [name], (terms, U.report(units))
        if terms == S.TERMS_1PASS:
            assert not U.failures(units, U.MULT["tc_fast"]), U.report(units)


def test_missing_and_unknown_tensors(oracle_run):
    sd, x, taps = oracle_run
    given = coarse_layout(sd, taps)
    given["synthesis.b8.img"] = torch.full_like(given["synthesis.b8.img"], math.nan)   # a tap that never fired
    bad = U.failures(U.unit_errors(sd, x, R, given), 1e9)
    assert bad[0].name == "synthesis.b8.img" and bad[0].err == math.inf     # (and every unit that reads it)
    given = coarse_layout(sd, taps)
    given["synthesis.b8.conv2.noise"] = given["synthesis.b8.img"]
    with pytest.raises(KeyError):
        U.unit_errors(sd, x, R, given)


def test_default_oracle_unchanged_by_the_hook(oracle_run):
    """generator_forward without taps and with a dict of taps computes the same bits (tests/golden pins the former)."""
    sd, x, taps = oracle_run
    assert torch.equal(O.generator_forward(sd, x, R), O.generator_forward(sd, x, R, taps={}))
    assert not any(k.endswith("out_skip") for k in taps)
    assert np.isfinite(sum(float(t.abs().sum()) for t in taps.values()))
