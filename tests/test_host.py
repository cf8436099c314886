"""Host-side logic and the C-ABI surface, no GPU needed."""
import ctypes
import os
import re
import subprocess
import sys

import pytest
import torch

import migan_b200
from migan_b200 import _abi, arch
from oracle import migan_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol(lib):
    header = open(os.path.join(ROOT, "include", "migan_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b((?:migan|b200)_[a-z0-9_]+)\s*\(", header))
    bound = {name for name, _, _ in _abi.SYMBOLS}
    assert declared == bound, declared ^ bound
    for name in declared:
        assert hasattr(lib, name)
    assert b"sm_100a" in lib.migan_version()


@pytest.mark.parametrize("R", [8, 64, 256, 512])
def test_state_dict_layout_matches_reference_order(lib, R):
    """Python module, C registry and the oracle spec (checked against the real reference by
    make_golden.py with strict=True) all agree on names, order and shapes."""
    spec = O.state_dict_spec(R)
    g = migan_b200.Generator(R)
    sd = g.state_dict()
    assert list(sd.keys()) == list(spec.keys())
    assert all(tuple(sd[k].shape) == tuple(spec[k]) for k in spec)
    h = ctypes.c_void_p()
    _abi.check(lib.migan_create(R, -1, ctypes.byref(h)))
    try:
        assert lib.migan_num_weights(h) == len(spec)
        for i, (k, shape) in enumerate(spec.items()):
            nm, nd, sh = ctypes.c_char_p(), ctypes.c_int(), (ctypes.c_int64 * 4)()
            _abi.check(lib.migan_weight_info(h, i, ctypes.byref(nm), ctypes.byref(nd), sh))
            assert nm.value.decode() == k and tuple(sh[: nd.value]) == tuple(shape)
        assert lib.migan_workspace_bytes(h, 2) > lib.migan_workspace_bytes(h, 1) > 0
    finally:
        lib.migan_destroy(h)


def test_param_vs_buffer_split_and_attribute_paths():
    g = migan_b200.Generator(256)
    assert sum(p.numel() for p in g.parameters()) == 5943617      # SURVEY.md section 6
    bufs = dict(g.named_buffers())
    assert "synthesis.b64.conv1.noise_const" in bufs and "synthesis.b64.upsample.filter_const" in bufs
    assert g.encoder.b256.fromrgb.weight.shape == (128, 4, 1, 1)
    assert g.synthesis.b8.conv1.use_noise and not g.synthesis.b4.conv2.use_noise
    assert g.encoder.b64.conv2.downsample.filter.weight.shape == (512, 1, 4, 4)
    # a reference state_dict (seeded stand-in) loads strictly
    g.load_state_dict(O.make_state_dict(256), strict=True)


def test_constructor_and_cpu_errors(lib):
    with pytest.raises(ValueError):
        migan_b200.Generator(96)          # reference raises ValueError (migan_inference.py:215-216)
    g = migan_b200.Generator(64)
    with pytest.raises(RuntimeError, match="no CPU"):
        g(torch.zeros(1, 4, 64, 64))
    h = ctypes.c_void_p()
    assert lib.migan_create(96, -1, ctypes.byref(h)) == _abi.ERR_INVALID
    assert b"power of two" in lib.migan_last_error()
    _abi.check(lib.migan_create(64, -1, ctypes.byref(h)))
    w = torch.zeros(7)
    assert lib.migan_set_weight(h, b"no.such.key", w.data_ptr(), 7) == _abi.ERR_INVALID
    assert lib.migan_set_weight(h, b"encoder.b64.fromrgb.bias", w.data_ptr(), 7) == _abi.ERR_INVALID
    assert lib.migan_finalize_weights(h) == _abi.ERR_CUDA        # description-only context cannot compute
    lib.migan_destroy(h)


def test_no_cuda_device_fails_loudly(lib):
    """Run in a child process with no CUDA device visible (CUDA_VISIBLE_DEVICES empty), so that it holds on a GPU machine too."""
    code = ("import ctypes, sys; sys.path.insert(0, %r); from migan_b200 import _abi; lib = _abi.load(); h = ctypes.c_void_p(); "
            "print(lib.migan_create(64, 0, ctypes.byref(h))); print(lib.migan_last_error().decode())" % ROOT)
    child = subprocess.run([sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code],
                           env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True, timeout=300)
    assert child.returncode == 0, child.stderr[-2000:]
    rc, msg = child.stdout.strip().split("\n", 1)
    assert int(rc) == _abi.ERR_CUDA
    assert "no CPU path" in msg


def test_product_does_not_import_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's checker / CPU legs may touch oracle/: not the package, not tools/."""
    for top in ("mi-gan_b200", "tools", "include"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, top)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h", ".sh")):
                    src = open(os.path.join(dirpath, f)).read()
                    assert "import oracle" not in src and "from oracle" not in src, f


def test_arch_helpers():
    assert arch.encoder_resolutions(256) == [256, 128, 64, 32, 16, 8, 4]
    assert arch.synthesis_resolutions(64) == [4, 8, 16, 32, 64]
    assert [arch.nf(r) for r in (512, 256, 128, 64, 4)] == [64, 128, 256, 512, 512]


# --------------------------------------------------------------------------- #
# Co-Mod-GAN boundary (include/comodgan_b200.h, migan_b200.comodgan)
# --------------------------------------------------------------------------- #
def test_library_exports_every_comodgan_symbol(lib):
    header = open(os.path.join(ROOT, "include", "comodgan_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b((?:comodgan|b200)_[a-z0-9_]+)\s*\(", header))
    bound = {name for name, _, _ in _abi.COMOD_SYMBOLS}
    assert declared == bound, declared ^ bound
    for name in declared:
        assert hasattr(lib, name)


@pytest.mark.parametrize("R", [16, 256, 512])
def test_comodgan_state_dict_layout_matches_reference_order(lib, R):
    """Python modules, C registry and the oracle spec (checked against the real reference by
    make_golden_comodgan.py with strict=True) agree on names, order and shapes."""
    from migan_b200 import comodgan
    from oracle import comodgan_oracle as C
    spec = C.state_dict_spec(R)
    g = comodgan.Generator(comodgan.Mapping(num_ws=C.num_ws(R)), comodgan.Encoder(resolution=R),
                           comodgan.Synthesis(resolution=R))
    sd = g.state_dict()
    assert list(sd.keys()) == list(spec.keys())
    for k, shape in spec.items():
        assert tuple(sd[k].shape) == tuple(shape), k
    params = {k for k, _ in g.named_parameters()}
    assert "mapping.w_avg" not in params and "synthesis.b4.conv.noise_const" not in params
    assert "synthesis.b4.conv.noise_strength" in params and "encoder.b4.fc.weight" in params
    g.load_state_dict(C.make_state_dict(R) if R == 16 else sd, strict=True)
    assert g.num_ws == C.num_ws(R) and g.img_resolution == R and g.z_dim == 512


def test_comodgan_constructor_and_cpu_errors(lib):
    from migan_b200 import comodgan
    with pytest.raises(ValueError):
        comodgan.Encoder(resolution=48)
    with pytest.raises(ValueError):     # num_ws mismatch (stylegan.py:580-581)
        comodgan.Generator(comodgan.Mapping(num_ws=16), comodgan.Encoder(resolution=256), comodgan.Synthesis(resolution=256))
    g = comodgan.Generator(comodgan.Mapping(num_ws=6), comodgan.Encoder(resolution=16), comodgan.Synthesis(resolution=16))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        g(torch.zeros(1, 4, 16, 16))
    with pytest.raises(RuntimeError, match="shape"):
        g(torch.zeros(1, 3, 16, 16))
    h = ctypes.c_void_p()
    assert lib.comodgan_create(16, -1, ctypes.byref(h)) == 0
    assert lib.comodgan_finalize_weights(h) != 0        # no device, no weights: fails loudly
    lib.comodgan_destroy(h)


def _scripts_golden():
    """What the reference's scripts did with these classes (tests/golden/make_golden_scripts.py)."""
    import numpy as np
    return np.load(os.path.join(ROOT, "tests", "golden", "scripts.npz"))


def test_dropin_rebinds_reference_modules(lib, monkeypatch, tmp_path):
    """python -m migan_b200.dropin scripts.demo ...: the reference's import sites (scripts/demo.py:15-21) resolve to the
    B200 classes without editing any reference file.  Stand-in modules take the place of the reference's
    lib.model_zoo.migan_inference / lib.model_zoo.comodgan; the Co-Mod-GAN built through the rebound names has the
    state_dict keys of the reference's own construction (scripts/demo.py:95-100, stored)."""
    import importlib
    (tmp_path / "lib" / "model_zoo").mkdir(parents=True)
    (tmp_path / "lib" / "__init__.py").write_text("")
    (tmp_path / "lib" / "model_zoo" / "__init__.py").write_text("")
    (tmp_path / "lib" / "model_zoo" / "migan_inference.py").write_text("class Generator:\n    pass\n")
    (tmp_path / "lib" / "model_zoo" / "comodgan.py").write_text("".join("class %s:\n    pass\n" % n for n in ("Generator", "Mapping", "Encoder", "Synthesis")))
    monkeypatch.syspath_prepend(str(tmp_path))
    from migan_b200 import comodgan, dropin
    try:
        ref_mi = importlib.import_module("lib.model_zoo.migan_inference")
        ref_cm = importlib.import_module("lib.model_zoo.comodgan")
        saved = (ref_mi.Generator, ref_cm.Generator)
        dropin.install()
        assert ref_mi.Generator is migan_b200.Generator and ref_mi.ReferenceGenerator is saved[0]
        assert ref_cm.Generator is comodgan.Generator and ref_cm.ReferenceGenerator is saved[1]
        assert (ref_cm.Mapping, ref_cm.Encoder, ref_cm.Synthesis) == (comodgan.Mapping, comodgan.Encoder, comodgan.Synthesis)
        model = ref_cm.Generator(ref_cm.Mapping(num_ws=14), ref_cm.Encoder(resolution=256), ref_cm.Synthesis(resolution=256))
        assert list(model.state_dict().keys()) == [str(k) for k in _scripts_golden()["comodgan256_keys"]]
    finally:
        for name in ("lib.model_zoo.comodgan", "lib.model_zoo.migan_inference", "lib.model_zoo", "lib"):
            sys.modules.pop(name, None)


def _export_source(z):
    """The training generator's tensors that the reference's `copy_weights` read, regenerated from the stored names,
    shapes and seed (training parameters as nn.Parameter, noise planes as plain buffers)."""
    from oracle import export_oracle as E
    names = [str(n) for n in z["src_names"]]
    shapes = [tuple(int(d) for d in s[:n]) for s, n in zip(z["src_shapes"], z["src_ndim"])]
    src = E.seeded_source(names, shapes, int(z["src_seed"]))
    return {k: (torch.nn.Parameter(v) if p else v) for (k, v), p in zip(src.items(), z["src_is_param"])}


def _source_filters(src, conv):
    """[w0 .. w{k-1}] of a re-parameterised training conv, [weight] of a plain one."""
    ws = [src["%s.w%d" % (conv, i)] for i in range(16) if "%s.w%d" % (conv, i) in src]
    return [w.detach() for w in (ws or [src[conv + ".weight"]])]


def _sample(t, z, key):
    return t.detach().reshape(-1)[torch.from_numpy(z["idx." + key]).long()]


def test_reference_export_script_accepts_b200_generator(lib):
    """scripts/export_inference_model.py:17-85 `copy_weights(source_G, dest)` -- the reference's route from a training
    snapshot (re-parameterised train graph, lib/model_zoo/migan.py) to inference weights -- works with the B200 class as
    `dest`.  The script's run on its own inference Generator is replayed on the B200 Generator from the stored trace:
    every attribute it reads there (`fromrgb is None`, `conv2.bias is None`, `use_noise`, the blocks) must give the
    answer the reference's class gave, and every assignment it made (filters, biases, noise tensors, blocks) is made
    again, with the same source.  The B200 Generator's state_dict then equals what the reference exported (stored
    sample).  Also the reference's behavioural pin: train graph == inference graph (export_inference_model.py:149-151),
    here the stored training-graph output against the oracle."""
    import torch.nn as nn
    from oracle import export_oracle as E
    z = _scripts_golden()
    src, R = _export_source(z), int(z["resolution"])
    mine = migan_b200.Generator(R).eval()
    keys = [str(k) for k in z["dest_keys"]]
    assert list(mine.state_dict().keys()) == keys
    for op, path, info in zip(z["trace_op"], z["trace_path"], z["trace_info"]):
        parent, _, leaf = str(path).rpartition(".")
        node = mine.get_submodule(parent)
        if op == "get":
            assert E.attribute_kind(getattr(node, leaf)) == info, path
            continue
        if info == "block":                                   # setattr(dest.encoder, f"b{res}", dest_module)
            value = getattr(node, leaf)
        else:
            kind, how, from_path = str(info).split(":")
            value = E.merged_filter(_source_filters(src, from_path)) if how == "filter" else src[from_path]
            if kind == "Parameter" and not isinstance(value, nn.Parameter):
                value = nn.Parameter(value)
        setattr(node, leaf, value)
    b = mine.state_dict()
    assert list(b.keys()) == keys
    for key in keys:
        assert torch.equal(_sample(b[key], z, key), torch.from_numpy(z["val." + key])), key
    x = O.make_input(R, 2)
    y_or = O.generator_forward({k: v.detach() for k, v in b.items()}, x, R)
    y_src = torch.from_numpy(z["y_val"])
    assert float((y_or.reshape(-1)[torch.from_numpy(z["y_idx"]).long()] - y_src).abs().max()) < 1e-4   # SURVEY 8c pin (1)


def test_resolutions_above_512_are_rejected_up_front(lib):
    """min(32768 // R, 512) drops below 64 channels for R > 512: not built (no released model); fail at create, not mid-forward.
    A description-only context (device -1: names and shapes) is still available."""
    h = ctypes.c_void_p()
    assert lib.migan_create(1024, 0, ctypes.byref(h)) == 1 and b"64 channels" in lib.migan_last_error()
    assert lib.migan_create(1024, -1, ctypes.byref(h)) == 0
    lib.migan_destroy(h)


def _emul_reparam(ws):
    """The export kernel's functor compiled for the host (tests/emul), on numpy copies of the tensors."""
    import numpy as np
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emul"))
    import build_emul
    emul = ctypes.CDLL(build_emul.build())
    emul.b200_reparam_filter.restype = ctypes.c_int
    emul.b200_reparam_filter.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p]
    arrs = [np.ascontiguousarray(w.detach().numpy(), dtype=np.float32) for w in ws]
    out = np.empty_like(arrs[0])
    ptrs = (ctypes.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])
    assert emul.b200_reparam_filter(ctypes.cast(ptrs, ctypes.c_void_p), len(arrs), arrs[0].shape[0], arrs[0][0].size,
                                    out.ctypes.data_as(ctypes.c_void_p), None) == 0
    return torch.from_numpy(out)


def test_export_kernel_matches_oracle_in_emulation():
    """csrc/reparam.cu (host-emulation build) against oracle/export_oracle.merged_filter: depthwise 3x3, 1x1 and k = 1 / 9 tensors.
    Bar: relative error < 1e-6 of the filter's largest tap (the sum of squares is accumulated in fp64 instead of torch's fp32 tree)."""
    from oracle import export_oracle as E
    g = torch.Generator().manual_seed(3)
    for shape, k in (((64, 1, 3, 3), 9), ((128, 64, 1, 1), 9), ((3, 512, 1, 1), 1), ((512, 512, 1, 1), 4), ((64, 4, 1, 1), 1)):
        ws = [torch.randn(shape, generator=g) * (0.5 + i) for i in range(k)]
        got, want = _emul_reparam(ws), E.merged_filter(ws)
        assert got.shape == want.shape
        err = (got - want).abs().amax(dim=(1, 2, 3)) / want.abs().amax(dim=(1, 2, 3))
        assert float(err.max()) < 1e-6, (shape, k, float(err.max()))
        assert torch.allclose(got.flatten(1).square().sum(1), torch.ones(shape[0]), atol=1e-5)   # unit L2 filters


def test_export_matches_reference_copy_weights():
    """oracle/export_oracle.merged_filter == the reference's `get_source_w` (through its effect: `copy_weights` into the
    reference's inference Generator, stored sample), and the export kernel (emulation) reproduces every filter of that
    state_dict."""
    from oracle import export_oracle as E
    z = _scripts_golden()
    src = _export_source(z)
    checked = 0
    for key, info in zip(z["trace_path"], z["trace_info"]):     # the filters copy_weights wrote, with their training convs
        if not str(info).startswith("Parameter:filter:"):
            continue
        key, ws = str(key), _source_filters(src, str(info).rsplit(":", 1)[1])
        want = E.merged_filter(ws)
        assert torch.equal(_sample(want, z, key), torch.from_numpy(z["val." + key])), key   # the oracle IS the reference expression
        got = _emul_reparam(ws)
        assert float(((got - want).abs().amax(dim=(1, 2, 3)) / want.abs().amax(dim=(1, 2, 3))).max()) < 1e-6
        checked += 1
    assert checked == 46      # 5 levels x 2 sides x 4 convolutions + 1 fromrgb + 5 torgb
