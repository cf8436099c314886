"""Pin what the reference's scripts do with this package's classes: write tests/golden/scripts.npz.

Needs a checkout of the reference:   MIGAN_REF=/path/to/MI-GAN python tests/golden/make_golden_scripts.py

1. scripts/export_inference_model.py `copy_weights(source, dest, resolution)`: the reference's training Generator
   (lib/model_zoo/migan.py, R = 64, nine re-parameterisation tensors per convolution) gets the tensors of
   oracle/export_oracle.seeded_source in place of every tensor `copy_weights` reads, then is exported into the reference's
   inference Generator.  Stored: the names / shapes / seed of those tensors (tests/test_host.py regenerates them), every
   attribute `copy_weights` reads on its `dest` with the answer it gets (`fromrgb is None`, `bias is None`, `use_noise`, ...)
   and every assignment it makes with the source it comes from, in order, the exported state_dict's keys with a seeded sample of the elements of every entry, and a seeded sample of the
   training graph's output on oracle make_input(64, 2) (the reference's train == inference pin, export_inference_model.py:149-151).
2. scripts/demo.py:95-100: the state_dict keys of the Co-Mod-GAN generator built at 256 with num_ws = 14.
"""
import os
import sys
import warnings

import re

import numpy as np
import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ["MIGAN_REF"]
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)

from oracle import export_oracle as E  # noqa: E402
from oracle import migan_oracle as O  # noqa: E402

R, SRC_SEED, SAMPLE_SEED = 64, 11, 12
SAMPLE = 32               # elements stored per state_dict entry


class Recorder:
    """Stands in for a module tree and logs, by dotted path, every attribute read through it and every assignment."""

    def __init__(self, obj, path, log, side):
        object.__setattr__(self, "_rec", (obj, path, log, side))

    def __getattr__(self, name):
        obj, path, log, side = self._rec
        v = getattr(obj, name)
        log.append((side, "get", path + name, v))
        return Recorder(v, path + name + ".", log, side) if isinstance(v, nn.Module) else v

    def __setattr__(self, name, value):
        obj, path, log, side = self._rec
        value = value._rec[0] if isinstance(value, Recorder) else value
        log.append((side, "set", path + name, value))
        setattr(obj, name, value)


def trace_copy_weights(copy_weights, src, dest):
    """Run `copy_weights(src, dest)`; return its reads and writes on `dest`.  A write's source is the last source attribute
    read before it: a filter of a training conv (`get_source_w` reads `reparametrize`, `num_reparam_tensors`, `w{i}` or `weight`) or a tensor taken over."""
    log, trace, last = [], [], None
    copy_weights(Recorder(src, "", log, "src"), Recorder(dest, "", log, "dest"), resolution=R)
    for side, op, path, v in log:
        if side == "src":
            last = path
        elif op == "get":
            trace.append(("get", path, E.attribute_kind(v)))
        elif isinstance(v, nn.Module):
            trace.append(("set", path, "block"))
        else:
            conv, leaf = last.rsplit(".", 1)
            how = "filter:" + conv if re.fullmatch(r"w\d+|weight|reparametrize|num_reparam_tensors", leaf) else "take:" + last
            trace.append(("set", path, "%s:%s" % (type(v).__name__, how)))
    return trace


def main():
    warnings.filterwarnings("ignore")
    from lib.model_zoo import comodgan as ref_cm
    from lib.model_zoo import migan as M
    from lib.model_zoo import migan_inference as ref_inf
    from scripts import export_inference_model as exp

    torch.manual_seed(0)
    src = M.Generator(M.Encoder(resolution=R, ic_n=4, depthwise=True, reparametrize=True, num_reparam_tensors=9),
                      M.Synthesis(resolution=R, depthwise=True, reparametrize=True, num_reparam_tensors=9)).eval()
    params = dict(src.named_parameters())
    read = [(k, v) for k, v in src.state_dict().items() if k in params or k.endswith("noise_const")]
    names, shapes = [k for k, _ in read], [tuple(v.shape) for _, v in read]
    seeded = E.seeded_source(names, shapes, SRC_SEED)
    with torch.no_grad():
        for k, v in src.state_dict().items():
            if k in seeded:
                v.copy_(seeded[k])

    dest = ref_inf.Generator(resolution=R).eval()
    trace = trace_copy_weights(exp.copy_weights, src, dest)
    sd = dest.state_dict()
    for op, path, info in trace:                  # every write is explained by its recorded source
        if op == "set" and info != "block":
            kind, how, from_path = info.split(":")
            want = E.merged_filter(_filters(src, from_path)) if how == "filter" else src.get_parameter(from_path) \
                if from_path in params else src.get_buffer(from_path)
            assert torch.equal(sd[path], want.detach()) and kind in ("Parameter", "Tensor"), path
    rng = np.random.default_rng(SAMPLE_SEED)
    out = {}
    for k, v in sd.items():
        flat = v.detach().reshape(-1).numpy()
        idx = np.sort(rng.choice(flat.size, min(flat.size, SAMPLE), replace=False)).astype(np.int32)
        out["idx." + k], out["val." + k] = idx, flat[idx]

    x = O.make_input(R, 2)
    with torch.no_grad():
        y = src(x, noise_mode="const").reshape(-1)
    y_idx = np.sort(rng.choice(y.numel(), 512, replace=False)).astype(np.int32)
    y_or = O.generator_forward({k: v.detach() for k, v in sd.items()}, x, R)
    print("training graph vs oracle on the exported weights: max-abs %.3e" % float((y - y_or.reshape(-1)).abs().max()))

    cm = ref_cm.Generator(ref_cm.Mapping(num_ws=14), ref_cm.Encoder(resolution=256), ref_cm.Synthesis(resolution=256))
    np.savez_compressed(
        os.path.join(HERE, "scripts.npz"), resolution=R, src_seed=SRC_SEED, src_names=np.array(names),
        src_ndim=np.array([len(s) for s in shapes]), src_shapes=np.array([list(s) + [0] * (4 - len(s)) for s in shapes]),
        src_is_param=np.array([k in params for k in names]),
        trace_op=np.array([t[0] for t in trace]), trace_path=np.array([t[1] for t in trace]),
        trace_info=np.array([t[2] for t in trace]), dest_keys=np.array(list(sd.keys())), y_idx=y_idx, y_val=y[y_idx].numpy(),
        comodgan256_keys=np.array(list(cm.state_dict().keys())), **out)
    print("written", os.path.join(HERE, "scripts.npz"))


def _filters(src, conv):
    m = src.get_submodule(conv)
    return [getattr(m, "w%d" % i).detach() for i in range(m.num_reparam_tensors)] if m.reparametrize else [m.weight.detach()]


if __name__ == "__main__":
    main()
