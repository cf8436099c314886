"""Training snapshot -> inference weights on the B200 (SURVEY.md 8(f) row f3, scripts/export_inference_model.py:17-85):
`migan_b200.export.reparam_filter` / `copy_weights` against oracle/export_oracle.py (pinned to the reference's own
`get_source_w` by tests/test_host.py through tests/golden/scripts.npz).  The source here is a module tree with the training
generator's attribute layout (lib/model_zoo/migan.py) built from plain containers -- the reference is absent on the GPU box.
Bar: relative error < 1e-6 per filter (fp64 sum of squares vs torch's fp32 tree), and the exported generator's forward
equals the oracle's forward on the oracle-exported weights within the generator's own tolerance."""
import pytest
import torch
import torch.nn as nn

import migan_b200
from migan_b200 import arch, export
from oracle import export_oracle as E
from oracle import migan_oracle as O

pytestmark = pytest.mark.gpu


class TrainConv(nn.Module):
    def __init__(self, shape, k, g, bias=True, noise_res=None):
        super().__init__()
        self.reparametrize, self.num_reparam_tensors = k > 1, k
        if k > 1:
            for i in range(k):
                setattr(self, "w%d" % i, nn.Parameter(torch.randn(shape, generator=g)))
        else:
            self.weight = nn.Parameter(torch.randn(shape, generator=g))
        self.bias = nn.Parameter(0.2 * torch.randn(shape[0], generator=g)) if bias else None
        if noise_res:
            self.register_buffer("noise_const", torch.randn(noise_res, noise_res, generator=g))
            self.noise_strength = nn.Parameter(torch.tensor(0.3))


def training_like(R, k, seed):
    """encoder.b{res}.{fromrgb, conv1, conv2} / synthesis.b{res}.{conv1, conv2, torgb}, each conv{1,2} a separable pair
    (conv1 depthwise 3x3, conv2 1x1), shapes taken from the inference generator's own state entries."""
    g = torch.Generator().manual_seed(seed)
    shapes = {key: shape for key, shape, _ in arch.state_entries(R)}
    root = nn.Module()
    for side in ("encoder", "synthesis"):
        blocks = nn.Module()
        for res in [2 ** i for i in range(2, R.bit_length())]:
            blk = nn.Module()
            for name in ("conv1", "conv2"):
                sep = nn.Module()
                p = "%s.b%d.%s." % (side, res, name)
                noise = shapes.get(p + "noise_const")
                sep.conv1 = TrainConv(shapes[p + "conv1.weight"], k, g, bias=(p + "conv1.bias") in shapes)
                sep.conv2 = TrainConv(shapes[p + "conv2.weight"], k, g, bias=(p + "conv2.bias") in shapes, noise_res=noise[-1] if noise else None)
                setattr(blk, name, sep)
            for head in ("fromrgb", "torgb"):
                p = "%s.b%d.%s." % (side, res, head)
                if p + "weight" in shapes:
                    setattr(blk, head, TrainConv(shapes[p + "weight"], k, g, bias=(p + "bias") in shapes))
            setattr(blocks, "b%d" % res, blk)
        setattr(root, side, blocks)
    return root


def _rel_err(got, want):
    return float(((got - want).abs().amax(dim=(1, 2, 3)) / want.abs().amax(dim=(1, 2, 3))).max())


def test_reparam_filter_matches_oracle(cuda_device):
    g = torch.Generator().manual_seed(3)
    for shape, k in (((64, 1, 3, 3), 9), ((128, 64, 1, 1), 9), ((3, 512, 1, 1), 1), ((512, 512, 1, 1), 4), ((512, 1, 3, 3), 16)):
        ws = [torch.randn(shape, generator=g) * (0.5 + i) for i in range(k)]
        got = export.reparam_filter([w.to(cuda_device) for w in ws]).cpu()
        assert _rel_err(got, E.merged_filter(ws)) < 1e-6, (shape, k)
    with pytest.raises(RuntimeError):
        export.reparam_filter([torch.randn(4, 1, 3, 3)])                       # CPU tensor: no CPU path
    with pytest.raises(RuntimeError):
        export.reparam_filter([torch.randn(4, 1, 3, 3, device=cuda_device)] * 17)


@pytest.mark.parametrize("R,k", [(64, 9), (128, 1)])
def test_copy_weights_exports_a_working_generator(cuda_device, R, k):
    src = training_like(R, k, seed=R + k)
    dest = migan_b200.Generator(R)
    export.copy_weights(src, dest, resolution=R, device=cuda_device)
    sd = {key: v.detach().cpu() for key, v in dest.state_dict().items()}
    # every filter against the oracle's expression on the same source tensors; biases / noise taken over unchanged
    for key, want_shape, _ in arch.state_entries(R):
        assert tuple(sd[key].shape) == tuple(want_shape), key
        parts = key.split(".")
        if key.endswith(".weight") and "filter" not in key:
            conv = src
            for a in parts[:-1]:
                conv = getattr(conv, a)
            ws = [getattr(conv, "w%d" % i).detach() for i in range(k)] if k > 1 else [conv.weight.detach()]
            assert _rel_err(sd[key], E.merged_filter(ws)) < 1e-6, key
        elif key.endswith(".bias"):
            conv = src
            for a in parts[:-1]:
                conv = getattr(conv, a)
            assert torch.equal(sd[key], conv.bias.detach()), key
        elif key.endswith("noise_strength") or key.endswith("noise_const"):
            sep = src
            for a in parts[:-1]:
                sep = getattr(sep, a)
            assert torch.equal(sd[key], getattr(sep.conv2, parts[-1]).detach()), key
    # the exported generator runs, and agrees with the oracle forward on its own state_dict
    dest = dest.to(cuda_device).eval()
    x = O.make_input(R, 2)
    y = dest(x.to(cuda_device)).cpu()
    y_or = O.generator_forward(sd, x, R)
    assert float((y - y_or).abs().max()) < 1e-3 * max(1.0, float(y_or.abs().max()))
    full = export.export_state_dict(src, R, device=cuda_device)
    assert list(full.keys()) == [key for key, _, _ in arch.state_entries(R)] and all(not v.is_cuda for v in full.values())
