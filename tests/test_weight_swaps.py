"""The generator re-uploads its weights after every kind of edit a caller makes: `export.copy_weights` and other
parameter / buffer assignments, `p.data = t`, in-place edits and `.to()`.  `_state_version()` is the per-call check; the
CPU test pins that it moves after each edit, the GPU tests that the forward then computes with the new weights."""
import numpy as np
import pytest
import torch
import torch.nn as nn

import migan_b200
from migan_b200 import export
from oracle import migan_oracle as O
from oracle import prepost_oracle as P

R = 16     # CPU test
RG = 64    # GPU tests


def test_state_version_follows_every_edit():
    g = migan_b200.Generator(R)
    g.load_state_dict(O.make_state_dict(R, seed=1))
    v = g._state_version()
    assert g._state_version() == v                                   # nothing changed: same version

    def moved(what):
        nonlocal v
        w = g._state_version()
        assert w != v, "version unchanged after " + what
        assert g._state_version() == w, "version unstable after " + what
        v = w

    conv = g.encoder.b16.conv1.conv2
    conv.weight = nn.Parameter(conv.weight.detach().clone())
    moved("Parameter replacement")
    with torch.no_grad():
        conv.weight.mul_(2.0)
    moved("an in-place edit of the replacing Parameter")
    g.synthesis.b16.conv1.noise_const = torch.randn(R, R)
    moved("buffer replacement")
    g.synthesis.b16.conv1.noise_const.add_(1.0)
    moved("an in-place edit of the replacing buffer")
    conv.weight.data = torch.randn_like(conv.weight)
    moved("p.data = t")
    with torch.no_grad():
        g.synthesis.b8.torgb.bias.zero_()
    moved("an in-place edit under no_grad")
    g.to(torch.float64)
    moved(".to()")
    g.to(torch.float32)
    moved(".to()")
    other = migan_b200.Generator(R)
    other.encoder.b16.conv1.conv2.weight = nn.Parameter(torch.zeros(512, 512, 1, 1))
    assert g._state_version() == v                                   # another generator's edits are not this one's


def _source(seed):
    from test_export_gpu import training_like                        # training-graph attribute layout
    return training_like(RG, 1, seed=seed)


def _edits(device):
    """(description, edit) pairs; each edit changes the output."""
    def copy_from(seed):
        return lambda g: export.copy_weights(_source(seed), g, resolution=RG, device=device)

    def new_param(g):
        w = g.encoder.b16.conv1.conv2.weight
        g.encoder.b16.conv1.conv2.weight = nn.Parameter(w.detach().flip(0).clone())

    def new_noise(g):
        c = g.synthesis.b16.conv2.noise_const
        g.synthesis.b16.conv2.noise_const = torch.randn(c.shape, generator=torch.Generator().manual_seed(4)).to(c.device)
    return [("copy_weights", copy_from(21)), ("copy_weights again", copy_from(22)),
            ("nn.Parameter", new_param), ("noise_const", new_noise)]


def _fresh(g):
    f = migan_b200.Generator(RG, path=g.path)
    f.load_state_dict(g.state_dict())
    return f.to(next(g.parameters()).device).eval()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [8, 1])                                # plain launch sequence; CUDA-graph replay
def test_forward_follows_weight_edits(cuda_device, n):
    g = migan_b200.Generator(RG, path="tc")
    g.load_state_dict(O.make_state_dict(RG, seed=1))
    g = g.to(cuda_device).eval()
    assert n > g.graph_max_batch if n == 8 else n <= g.graph_max_batch
    x = O.make_input(RG, n, seed=7)
    xd = x.to(cuda_device)
    prev = g(xd)
    for what, edit in _edits(cuda_device):
        edit(g)
        y = g(xd)
        assert not torch.equal(y, prev), "output unchanged after " + what
        assert torch.equal(y, _fresh(g)(xd)), what
        sd = {k: v.detach().cpu() for k, v in g.state_dict().items()}
        assert float((y.cpu() - O.generator_forward(sd, x, RG)).abs().max()) < 1e-3, what
        prev = y


@pytest.mark.gpu
def test_forward_u8_follows_weight_edits(cuda_device):
    g = migan_b200.Generator(RG, path="tc")
    g.load_state_dict(O.make_state_dict(RG, seed=1))
    g = g.to(cuda_device).eval()
    rng = np.random.RandomState(5)
    img = torch.from_numpy(rng.randint(0, 256, size=(2, RG, RG, 3), dtype=np.uint8))
    mask = torch.from_numpy(((rng.rand(2, RG, RG) > 0.4) * 255).astype(np.uint8))
    prev = g.forward_u8(img, mask).clone()
    for what, edit in _edits(cuda_device):
        edit(g)
        out = g.forward_u8(img, mask).clone()
        assert not torch.equal(out, prev), "output unchanged after " + what
        assert torch.equal(out, _fresh(g).forward_u8(img, mask)), what
        sd = {k: v.detach().cpu() for k, v in g.state_dict().items()}
        want = torch.from_numpy(P.postprocess(O.generator_forward(sd, P.preprocess(img.numpy(), mask.numpy()), RG),
                                              img.numpy(), mask.numpy()))
        assert int((out.int() - want.int()).abs().max()) <= 1, what          # a value on a uint8 boundary may round over
        prev = out
