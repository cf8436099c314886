"""Every launch of the shipped plan against float64, one unit at a time -- needs a B200.

A unit is the work between two tensors the plan materialises (its taps): on `tc` a down layer is dw3x3_down plus the
SPLIT contraction, the STEM unit starts from x, a fused UP unit reads the previous layer's raw 1x1 output, the encoder
feature and the lower image, and the top level ends at y.  oracle/unit_parity.py evaluates each unit in float64 from
the device's own inputs, so an error cannot hide in what upstream launches did, and bounds the device's error by a
modelled multiple of the same unit's plain-fp32 error (tests/test_split_precision.py derives the multiples).

Shapes are chosen from the planner arithmetic at 148 SMs so that different kernels run:
  R=512 N=1 / N=32   64-channel levels (n_tile 64, resident B, STEM and UP prologues at Cin 64); the 16..64^2 levels take
                     narrow N tiles at N=1 and wide ones at N=32
  R=256 N=33         a partial batch tile at 4^2 (8 images per tile);  R=64 N=5: at 8^2 (2 per tile)
  R=8/16/32 N=3      linear SPLIT tiles below 16^2, the unfused stem and torgb
Only the first and last image of a large batch are compared (images are independent), which bounds the CPU work.

The scheduling switches (reserved SMs for a concurrent collective, programmatic dependent launch off) change only which
CTA runs which tile and when a kernel may start, so their outputs must be bit-identical to the default plan's.
"""
import os
import subprocess
import sys

import pytest
import torch

import migan_b200
from oracle import migan_oracle as O
from oracle import unit_parity as U

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SHAPES = [(512, 1), (512, 32), (256, 33), (64, 5), (8, 3), (16, 3), (32, 3)]
FAST_SHAPES = [(512, 1), (256, 33)]


def make_model(R, path):
    sd = O.make_state_dict(R, seed=1)
    g = migan_b200.Generator(R, path=path)
    g.load_state_dict(sd)
    return g.to("cuda:0").eval(), sd


def picked(N):
    return list(range(N)) if N <= 5 else [0, N - 1]


def launch_units(path, R, N):
    """Run the plan once per tap and judge every tapped tensor of the picked images against float64."""
    g, sd = make_model(R, path)
    x = O.make_input(R, N, seed=R + N)
    xd, pick = x.to("cuda:0"), picked(N)
    names = g.tap_names()
    given = {}
    for name, shape in names:
        assert name not in given, "tap %s listed twice" % name
        _, t = g.forward_with_tap(xd, name, shape)      # NaN where the tap did not fire
        given[name] = t[pick].cpu()
    units = U.unit_errors(sd, x[pick], R, given)
    assert [u.name for u in units] == [n for n, _ in names]
    return units


@pytest.mark.parametrize("path", ["simt", "tc"])
@pytest.mark.parametrize("R,N", SHAPES)
def test_every_launch_matches_float64(cuda_device, path, R, N):
    units = launch_units(path, R, N)
    print("launch parity path=%s R=%d N=%d: %s" % (path, R, N, U.report(units)))
    bad = U.failures(units, U.MULT[path])
    assert not bad, "units over %g x their fp32 error: %s" % (
        U.MULT[path], ["%s ratio %.1f" % (u.name, u.ratio) for u in bad[:8]])


@pytest.mark.parametrize("R,N", FAST_SHAPES)
def test_tc_fast_launches_within_single_pass_bound(cuda_device, R, N):
    """tc_fast stays within its single-pass bound, and fails the 3-pass bar on every unit that contains a 1x1 contraction:
    the `tc` bar would notice one launch dropping its correction passes."""
    units = launch_units("tc_fast", R, N)
    print("launch parity path=tc_fast R=%d N=%d: %s" % (R, N, U.report(units)))
    bad = U.failures(units, U.MULT["tc_fast"])
    assert not bad, ["%s ratio %.1f" % (u.name, u.ratio) for u in bad[:8]]
    gemm = [u for u in units if u.gemm]
    assert len(gemm) >= 10
    slipped = [u for u in gemm if u.err <= U.MULT["tc"] * u.ref_err]
    assert not slipped, "single-pass units inside the 3-pass bar: %s" % ["%s ratio %.1f" % (u.name, u.ratio) for u in slipped]


SCHED_SHAPES = [(512, 32), (256, 1)]


def _scheduling_input(R, N):
    return O.make_input(R, N, seed=500 + N)


def test_reserved_sms_are_bit_identical(cuda_device, monkeypatch):
    """MIGAN_TC_RESERVE_SMS (set by parallel.configure_overlap for NCCL runs) shrinks every persistent tensor-core grid."""
    cap = torch.cuda.get_device_properties(cuda_device).multi_processor_count // 2
    for R, N in SCHED_SHAPES:
        x = _scheduling_input(R, N).to(cuda_device)
        monkeypatch.delenv("MIGAN_TC_RESERVE_SMS", raising=False)
        want = make_model(R, "tc")[0](x)
        for reserve in (12, cap):
            monkeypatch.setenv("MIGAN_TC_RESERVE_SMS", str(reserve))
            g, _ = make_model(R, "tc")                   # read when the plan is built: a fresh generator
            assert torch.equal(g(x), want), "R=%d N=%d reserve=%d differs from the full grid" % (R, N, reserve)


_PDL_CHILD = r"""
import sys
sys.path.insert(0, sys.argv[1])
import torch
import migan_b200
from oracle import migan_oracle as O
out = {}
for path in ("simt", "tc"):
    for R, N in %r:
        g = migan_b200.Generator(R, path=path)
        g.load_state_dict(O.make_state_dict(R, seed=1))
        g = g.to("cuda:0").eval()
        out["%%s/%%d/%%d" %% (path, R, N)] = g(O.make_input(R, N, seed=500 + N).to("cuda:0")).cpu()
torch.save(out, sys.argv[2])
""" % (SCHED_SHAPES,)


def test_serialised_launches_are_bit_identical(cuda_device, tmp_path):
    """MIGAN_PDL=0 drops the programmatic-dependent-launch attribute: every kernel then starts after its predecessor has
    finished.  The default relies on each kernel waiting (griddepcontrol.wait) before it reads what any earlier launch
    wrote.  The switch is read once per process, so the serialised run is a child process."""
    dst = tmp_path / "pdl0.pt"
    child = subprocess.run([sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", _PDL_CHILD, ROOT, str(dst)],
                           env=dict(os.environ, MIGAN_PDL="0"), capture_output=True, text=True, timeout=900)
    assert child.returncode == 0, child.stderr[-3000:]
    serial = torch.load(dst)
    for path in ("simt", "tc"):
        for R, N in SCHED_SHAPES:
            got = make_model(R, path)[0](_scheduling_input(R, N).to(cuda_device)).cpu()
            assert torch.equal(got, serial["%s/%d/%d" % (path, R, N)]), "path=%s R=%d N=%d: PDL changes the output" % (path, R, N)
