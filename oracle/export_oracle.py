"""CPU oracle for the training-snapshot -> inference-weights transformation (SURVEY.md 8(f) row f3).  TEST INFRASTRUCTURE ONLY.

Restates `get_source_w` of scripts/export_inference_model.py:18-27 on plain tensors, with the same torch expressions:
the re-parameterised tensors are summed in order and divided by sqrt(k), then every output filter is scaled to unit L2 norm.
Pinned against the reference function itself through tests/golden/scripts.npz (tests/golden/make_golden_scripts.py runs
the reference's `copy_weights` on the reference's training Generator filled by `seeded_source`)."""
import numpy as np
import torch


def seeded_source(names, shapes, seed):
    """Stand-in training weights for the tensors `copy_weights` reads, drawn in the given order: N(0, 1) filters and
    noise planes, 0.2 N(0, 1) biases, noise strengths 0.3."""
    g = torch.Generator().manual_seed(seed)
    out = {}
    for name, shape in zip(names, shapes):
        if name.endswith("noise_strength"):
            out[name] = torch.full(shape, 0.3)
        elif name.endswith("bias"):
            out[name] = 0.2 * torch.randn(shape, generator=g)
        else:
            out[name] = torch.randn(shape, generator=g)
    return out


def attribute_kind(v):
    """What `copy_weights` learns from reading an attribute of its `dest`: None, a module, a tensor, or a flag's value."""
    if v is None:
        return "None"
    if isinstance(v, bool):
        return str(v)
    if isinstance(v, torch.nn.Module):
        return "module"
    if isinstance(v, torch.Tensor):
        return "tensor"
    return type(v).__name__


def merged_filter(ws):
    """ws: list of k tensors [cout, cin/groups, kh, kw] (k = 1: a plain `weight`)."""
    w = ws[0]
    if len(ws) > 1:
        for t in ws[1:]:                                   # :20-22
            w = w + t
        w = w / np.sqrt(len(ws))                           # :23
    return w * (w.square().sum(dim=[1, 2, 3]) + 1e-8).rsqrt().reshape(-1, 1, 1, 1)   # :26
