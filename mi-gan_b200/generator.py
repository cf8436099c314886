"""`Generator(resolution).forward(x[N,4,R,R]) -> img[N,3,R,R]` on B200.

Drop-in for `lib.model_zoo.migan_inference.Generator` (reference
lib/model_zoo/migan_inference.py:355-369): same constructor, same `state_dict` keys /
shapes / order (so `load_state_dict(torch.load(path))` of a released checkpoint works,
scripts/demo.py:110), same attribute paths (`encoder.b256.conv1.conv2.weight`,
`synthesis.b64.conv1.noise_const`, `.use_noise`, used by scripts/export_inference_model.py:35-83),
same forward signature and output layout (fresh contiguous NCHW fp32 tensor on x.device).

The module holds only parameters; all arithmetic happens in the C-ABI library
(`include/migan_b200.h`) through ctypes.  PyTorch is used for device memory and the current
stream, nothing else.  There is no CPU path: a CPU tensor raises RuntimeError.
"""
from __future__ import annotations

import ctypes
import math
import os
from typing import Dict, Optional

import torch
import torch.nn as nn

from . import _abi, arch


# Bumped whenever a parameter, buffer or sub-module of any generator tree is assigned, registered or deleted: the tensor
# list a Generator collected for its per-call weight check is stale after that (Generator._state_version).
_tree_edits = [0]


class _Tracked(nn.Module):
    def __setattr__(self, name, value):
        if value is None or isinstance(value, (torch.Tensor, nn.Module)):
            _tree_edits[0] += 1
        super().__setattr__(name, value)

    def __delattr__(self, name):
        _tree_edits[0] += 1
        super().__delattr__(name)

    def register_parameter(self, name, param):
        _tree_edits[0] += 1
        super().register_parameter(name, param)

    def register_buffer(self, name, tensor, persistent=True):
        _tree_edits[0] += 1
        super().register_buffer(name, tensor, persistent)

    def add_module(self, name, module):
        _tree_edits[0] += 1
        super().add_module(name, module)


class _Node(_Tracked):
    """Parameter container: one level of the reference's attribute tree."""

    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError("migan_b200 sub-modules are parameter containers; call Generator.forward")


def _fir(gain: float) -> torch.Tensor:
    f = torch.tensor(arch.FIR_PROTOTYPE, dtype=torch.float32)
    f = torch.outer(f, f)
    f = f / f.sum()
    return f * gain  # 2-D filter: gain ** (ndim / 2) == gain (migan_inference.py:53)


def _initial_value(key: str, shape) -> torch.Tensor:
    """Constructor-time values with the reference's statistics (nn.Conv2d default init,
    FIR taps / filter_const / noise buffers as at migan_inference.py:71-72, :83-85, :95-96, :149-150)."""
    if key.endswith("filter.weight"):
        return _fir(1.0 if "downsample" in key else 4.0).repeat(shape[0], 1, 1, 1)
    if key.endswith("filter_const"):
        return torch.tensor([[1.0, 0.0], [0.0, 0.0]]).repeat(1, 1, shape[2] // 2, shape[3] // 2)
    if key.endswith("noise_const"):
        return torch.randn(shape)
    if key.endswith("noise_strength"):
        return torch.zeros(shape)
    if key.endswith(".weight"):
        w = torch.empty(shape)
        nn.init.kaiming_uniform_(w, a=math.sqrt(5))
        return w
    if key.endswith(".bias"):
        # fan_in of the matching weight: depthwise 3x3 -> 9, fromrgb -> 4, torgb -> C
        fan_in = 9 if ".conv1.bias" in key else (4 if "fromrgb" in key else arch.CH_MAX)
        bound = 1.0 / math.sqrt(fan_in)
        return torch.empty(shape).uniform_(-bound, bound)
    raise KeyError(key)


class _Engine:
    """One C context per (module, device): uploaded weights + cached workspaces."""

    def __init__(self, resolution: int, device: torch.device):
        self.lib = _abi.load()
        self.device = device
        self.handle = ctypes.c_void_p()
        _abi.check(self.lib.migan_create(resolution, device.index if device.index is not None else torch.cuda.current_device(),
                                         ctypes.byref(self.handle)))
        self.weights_version = None
        self.workspaces: Dict[int, torch.Tensor] = {}

    def close(self):
        if self.handle:
            self.lib.migan_destroy(self.handle)
            self.handle = ctypes.c_void_p()

    def __del__(self):  # best effort
        try:
            self.close()
        except Exception:
            pass

    def upload(self, state: Dict[str, torch.Tensor], version) -> None:
        for key, t in state.items():
            h = t.detach().to(device="cpu", dtype=torch.float32).contiguous()
            _abi.check(self.lib.migan_set_weight(self.handle, key.encode(), h.data_ptr(), h.numel()))
        _abi.check(self.lib.migan_finalize_weights(self.handle))
        self.weights_version = version

    def workspace(self, n: int, host_staging=False):
        """host_staging: False (device forward), True (host-buffer call: two staging slots) or "graph" (captured forward:
        one staging slot)."""
        key = (n, host_staging)
        ws = self.workspaces.get(key)
        if ws is None:
            nbytes = self.lib.migan_workspace_bytes(self.handle, n)
            if host_staging == "graph":
                nbytes += self.lib.migan_graph_staging_bytes(self.handle, n)
            elif host_staging:
                nbytes += self.lib.migan_host_staging_bytes(self.handle, n)
            raw = torch.empty(nbytes + 1024, dtype=torch.uint8, device=self.device)
            off = (-raw.data_ptr()) % 1024
            ws = raw[off:off + nbytes]
            if any(k[0] != n for k in self.workspaces):
                # copies enqueued by forward_host(wait=False) may still be using a staging area that is about to be released
                _abi.check(self.lib.migan_host_wait(self.handle))
            self.workspaces = {k: v for k, v in self.workspaces.items() if k[0] == n}  # keep one batch size
            self.workspaces[key] = ws
        return ws


class Generator(_Tracked):
    """MI-GAN inference generator, B200-native.  See module docstring.

    The weights are uploaded to the device on the first forward and again whenever they change: after `load_state_dict`,
    `.to()`, an assignment of a parameter, buffer or sub-module anywhere in the tree (`export.copy_weights` does this),
    `p.data = t`, and in-place edits of a parameter or buffer (`p.mul_(2)` under `torch.no_grad()`, `p.copy_(t)`).
    In-place writes through `.data` (`p.data.mul_(2)`, `p.data[0] = 1`) bypass the tensors' version counters and go unseen:
    follow them with `load_state_dict(self.state_dict())`."""

    def __init__(self, resolution: int = 256, path: Optional[str] = None):
        super().__init__()
        arch.log2_resolution(resolution)  # ValueError for non powers of two (reference :214-216)
        self.resolution = resolution
        self.path = path  # None -> $MIGAN_B200_PATH -> "tc"
        # batches up to this size go through the CUDA-graph replay of the forward (0 disables it)
        self.graph_max_batch = int(os.environ.get("MIGAN_GRAPH_MAX_N", "4"))
        for key, shape, kind in arch.state_entries(resolution):
            *mods, leaf = key.split(".")
            node = self
            for m in mods:
                if not hasattr(node, m):
                    node.add_module(m, _Node())
                node = getattr(node, m)
            value = _initial_value(key, shape)
            if kind == arch.PARAM:
                node.register_parameter(leaf, nn.Parameter(value))
            else:
                node.register_buffer(leaf, value)
        # attributes the reference's export script reads (scripts/export_inference_model.py:35-83)
        for m in self.modules():
            if hasattr(m, "conv1") and hasattr(m, "conv2") and hasattr(m.conv2, "weight") and hasattr(m.conv1, "bias"):
                m.use_noise = hasattr(m, "noise_const")
                m.conv2.register_parameter("bias", None)      # nn.Conv2d(..., bias=False) of migan_inference.py:136
        for blk in self.encoder.children():                   # EncoderBlock.fromrgb is None except in the first block (:176-186)
            if not hasattr(blk, "fromrgb"):
                blk.fromrgb = None
        self._engines: Dict[torch.device, _Engine] = {}

    def __getstate__(self):  # engines hold C handles: never pickled / deep-copied
        state = self.__dict__.copy()
        state["_engines"] = {}
        state["_state_tensors"] = None
        return state

    # -- plumbing ---------------------------------------------------------------------
    def _path_id(self) -> int:
        name = self.path or os.environ.get("MIGAN_B200_PATH", "tc")
        if name not in _abi.PATHS:
            raise ValueError("unknown path %r (expected one of %s)" % (name, sorted(_abi.PATHS)))
        return _abi.PATHS[name]

    def _state_version(self):
        # Cheap per-call check that the uploaded weights are still current.  The tensor list is collected again only after
        # load_state_dict / .to() / .cuda() or an edit of some generator tree (_tree_edits); the epoch counts the times it
        # came out different.  The cache holds the listed tensors, so `is` compares them exactly.  Each call sums version
        # counters (in-place edits) and reads data pointers (`p.data = t` changes neither the tree nor the version).
        d = self.__dict__
        tensors = d.get("_state_tensors")
        if tensors is None or d.get("_state_edits") != _tree_edits[0]:
            edits = _tree_edits[0]
            fresh = tuple(self.state_dict(keep_vars=True).values())
            if tensors is None or len(fresh) != len(tensors) or any(a is not b for a, b in zip(fresh, tensors)):
                d["_state_epoch"] = d.get("_state_epoch", 0) + 1
            d["_state_tensors"], d["_state_edits"], tensors = fresh, edits, fresh
        return (d["_state_epoch"], sum(t._version for t in tensors), tuple(t.data_ptr() for t in tensors))

    def _apply(self, fn, *args, **kwargs):
        self.__dict__["_state_tensors"] = None
        return super()._apply(fn, *args, **kwargs)

    def load_state_dict(self, *args, **kwargs):
        self.__dict__["_state_tensors"] = None
        return super().load_state_dict(*args, **kwargs)

    def _engine(self, device: torch.device) -> _Engine:
        eng = self._engines.get(device)
        if eng is None:
            eng = _Engine(self.resolution, device)
            self._engines[device] = eng
        version = self._state_version()
        if eng.weights_version != version:
            eng.upload(self.state_dict(keep_vars=True), version)
        return eng

    def _validate(self, x: torch.Tensor) -> torch.Tensor:
        if not isinstance(x, torch.Tensor):
            raise TypeError("x must be a torch.Tensor")
        r = self.resolution
        if x.dim() != 4 or x.shape[1] != 4 or x.shape[2] != r or x.shape[3] != r:
            raise RuntimeError("expected x of shape [N, 4, %d, %d] (mask-0.5, img*mask), got %s" % (r, r, tuple(x.shape)))
        if not x.is_cuda:
            raise RuntimeError("migan_b200.Generator runs on B200 (sm_100a) only; got a %s tensor. "
                               "There is no CPU fallback (the CPU oracle lives in oracle/ for tests)." % x.device)
        if x.dtype != torch.float32:
            raise RuntimeError("expected float32 input, got %s" % x.dtype)
        p = next(self.parameters())
        if p.device != x.device:
            raise RuntimeError("input is on %s but the module parameters are on %s" % (x.device, p.device))
        if x.shape[0] == 0:
            raise RuntimeError("empty batch")
        return x.contiguous()

    # -- the hot path -----------------------------------------------------------------
    @torch.no_grad()
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """x: 4-channel mask+rgb input (migan_inference.py:362-369)."""
        x = self._validate(x)
        n = x.shape[0]
        with torch.cuda.device(x.device):
            eng = self._engine(x.device)
            y = torch.empty((n, 3, self.resolution, self.resolution), dtype=torch.float32, device=x.device)
            stream = torch.cuda.current_stream(x.device).cuda_stream
            if n <= self.graph_max_batch:
                # small batches (the demo runs batch 1) are launch-bound: replay the captured launch sequence
                ws = eng.workspace(n, "graph")
                _abi.check(eng.lib.migan_forward_graph(eng.handle, x.data_ptr(), y.data_ptr(), n, ws.data_ptr(), ws.numel(),
                                                       self._path_id(), stream))
            else:
                ws = eng.workspace(n)
                _abi.check(eng.lib.migan_forward(eng.handle, x.data_ptr(), y.data_ptr(), n, ws.data_ptr(), ws.numel(),
                                                 self._path_id(), stream))
        return y

    @torch.no_grad()
    def forward_host(self, x_host: torch.Tensor, out: Optional[torch.Tensor] = None, wait: bool = True) -> torch.Tensor:
        """End-to-end call with HOST tensors (pinned for full speed): H2D, forward, D2H, sync --
        what scripts/demo.py:131-136 does around the reference model.  With wait=False the call only
        enqueues (serving loop: submit batches back to back, then `host_wait()`); `out` is valid after the wait."""
        r = self.resolution
        if x_host.is_cuda or x_host.dtype != torch.float32 or x_host.dim() != 4 or tuple(x_host.shape[1:]) != (4, r, r):
            raise RuntimeError("forward_host expects a CPU float32 tensor of shape [N, 4, %d, %d]" % (r, r))
        x_host = x_host.contiguous()
        n = x_host.shape[0]
        if n == 0:
            raise RuntimeError("empty batch")
        device = next(self.parameters()).device
        if device.type != "cuda":
            raise RuntimeError("module parameters must be on a CUDA device (call .to('cuda')); there is no CPU path")
        if out is None:
            out = torch.empty((n, 3, r, r), dtype=torch.float32, pin_memory=True)
        if out.is_cuda or out.dtype != torch.float32 or tuple(out.shape) != (n, 3, r, r) or not out.is_contiguous():
            raise RuntimeError("out must be a contiguous CPU float32 tensor of shape [N, 3, %d, %d]" % (r, r))
        with torch.cuda.device(device):
            eng = self._engine(device)
            ws = eng.workspace(n, host_staging=True)
            stream = torch.cuda.current_stream(device).cuda_stream
            fn = eng.lib.migan_forward_host if wait else eng.lib.migan_forward_host_async
            _abi.check(fn(eng.handle, x_host.data_ptr(), out.data_ptr(), n, ws.data_ptr(), ws.numel(), self._path_id(), stream))
        return out

    @torch.no_grad()
    def forward_u8(self, img_u8: torch.Tensor, mask_u8: torch.Tensor, out: Optional[torch.Tensor] = None,
                   wait: bool = True) -> torch.Tensor:
        """uint8 request path (scripts/demo.py:56-66 + :131-142 in one call): img_u8 [N,R,R,3] RGB and mask_u8 [N,R,R]
        (255 = known) are HOST uint8 tensors (pinned for full speed); returns the composed uint8 image [N,R,R,3] on the
        host: known pixels of img, generated pixels elsewhere.  Pre/post-processing run as CUDA kernels around the forward,
        so 7 bytes per pixel cross PCIe instead of 28.  wait=False only enqueues (serving loop: submit requests back to back, then
        `host_wait()`; the copies of request t+1 / t-1 run under the kernels of request t)."""
        r = self.resolution
        if img_u8.is_cuda or mask_u8.is_cuda or img_u8.dtype != torch.uint8 or mask_u8.dtype != torch.uint8:
            raise RuntimeError("forward_u8 expects CPU uint8 tensors")
        if img_u8.dim() != 4 or tuple(img_u8.shape[1:]) != (r, r, 3) or tuple(mask_u8.shape) != (img_u8.shape[0], r, r):
            raise RuntimeError("forward_u8 expects img [N, %d, %d, 3] and mask [N, %d, %d]" % (r, r, r, r))
        img_u8, mask_u8 = img_u8.contiguous(), mask_u8.contiguous()
        n = img_u8.shape[0]
        if n == 0:
            raise RuntimeError("empty batch")
        device = next(self.parameters()).device
        if device.type != "cuda":
            raise RuntimeError("module parameters must be on a CUDA device (call .to('cuda')); there is no CPU path")
        if out is None:
            out = torch.empty((n, r, r, 3), dtype=torch.uint8, pin_memory=True)
        if out.is_cuda or out.dtype != torch.uint8 or tuple(out.shape) != (n, r, r, 3) or not out.is_contiguous():
            raise RuntimeError("out must be a contiguous CPU uint8 tensor of shape [N, %d, %d, 3]" % (r, r))
        with torch.cuda.device(device):
            eng = self._engine(device)
            nbytes = eng.lib.migan_workspace_bytes(eng.handle, n) + eng.lib.migan_u8_staging_bytes(eng.handle, n)
            ws = eng.workspaces.get((n, "u8"))
            if ws is None:
                raw = torch.empty(nbytes + 1024, dtype=torch.uint8, device=device)
                off = (-raw.data_ptr()) % 1024
                ws = raw[off:off + nbytes]
                if any(k[0] != n for k in eng.workspaces):
                    _abi.check(eng.lib.migan_host_wait(eng.handle))
                eng.workspaces = {k: v for k, v in eng.workspaces.items() if k[0] == n}
                eng.workspaces[(n, "u8")] = ws
            stream = torch.cuda.current_stream(device).cuda_stream
            fn = eng.lib.migan_forward_u8 if wait else eng.lib.migan_forward_u8_async
            _abi.check(fn(eng.handle, img_u8.data_ptr(), mask_u8.data_ptr(), out.data_ptr(), n,
                          ws.data_ptr(), ws.numel(), self._path_id(), stream))
        return out

    def host_wait(self) -> None:
        """Block until every batch enqueued with forward_host(wait=False) has landed in its output tensor."""
        for eng in self._engines.values():
            _abi.check(eng.lib.migan_host_wait(eng.handle))

    def from_img_mask(self, img: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
        """Convenience stem of the callers (scripts/demo.py:56-66): img in [-1,1], mask 1 = known."""
        return self.forward(torch.cat([mask - 0.5, img * mask], dim=1))

    # -- test / profiling helpers -----------------------------------------------------
    def last_launch_count(self, device=None) -> int:
        eng = next(iter(self._engines.values())) if device is None else self._engines[torch.device(device)]
        return int(eng.lib.migan_last_launch_count(eng.handle))

    def set_profiling(self, enable: bool, device=None) -> None:
        """Bracket every kernel launch of subsequent forwards with CUDA events (roofline reports)."""
        eng = self._engine(next(self.parameters()).device if device is None else torch.device(device))
        _abi.check(eng.lib.migan_set_profiling(eng.handle, int(bool(enable))))

    def profile_steps(self, device=None):
        """[(label, ms, algorithmic_bytes, flops)] of the most recent profiled forward."""
        eng = self._engine(next(self.parameters()).device if device is None else torch.device(device))
        out = []
        label, ms = ctypes.c_char_p(), ctypes.c_float()
        nbytes, flops = ctypes.c_double(), ctypes.c_double()
        for i in range(eng.lib.migan_profile_num_steps(eng.handle)):
            _abi.check(eng.lib.migan_profile_step(eng.handle, i, ctypes.byref(label), ctypes.byref(ms),
                                                  ctypes.byref(nbytes), ctypes.byref(flops)))
            out.append((label.value.decode(), float(ms.value), float(nbytes.value), float(flops.value)))
        return out

    def tap_names(self, device=None):
        """[(name, (C, H, W))] of the intermediates `forward_with_tap` can return on the current path."""
        eng = self._engine(next(self.parameters()).device if device is None else torch.device(device))
        out, i = [], 0
        name = ctypes.c_char_p()
        shape = (ctypes.c_int * 3)()
        while eng.lib.migan_tap_info(eng.handle, self._path_id(), i, ctypes.byref(name), shape) == 0:
            out.append((name.value.decode(), (shape[0], shape[1], shape[2])))
            i += 1
        return out

    @torch.no_grad()
    def forward_with_tap(self, x: torch.Tensor, tap: str, shape) -> (torch.Tensor, torch.Tensor):
        """Run forward and also return the named intermediate as NCHW (debug / parity tests).  The intermediate is NaN
        where the forward did not write it (a name the plan does not produce)."""
        x = self._validate(x)
        eng = self._engine(x.device)
        buf = torch.full((x.shape[0],) + tuple(shape), float("nan"), dtype=torch.float32, device=x.device)
        _abi.check(eng.lib.migan_set_tap(eng.handle, tap.encode(), buf.data_ptr()))
        try:
            y = self.forward(x)
        finally:
            eng.lib.migan_set_tap(eng.handle, None, None)
        return y, buf
