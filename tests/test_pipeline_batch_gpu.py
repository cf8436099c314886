"""Batched crop pipeline on the B200: `MIGAN_Pipeline.forward_batch` and the `b200_pipeline_batch_*` entry points under it.

Bars: with the generator's output given, every stage is BIT-EXACT against the reference's vectors (tests/golden/pipeline.npz)
and against the oracle on large ragged batches; the device crop-window kernel reproduces the 300 pinned windows; end to end
the batch equals the requests run one by one through `pipe(image, mask)` (byte for byte when the generator is batch-invariant,
otherwise the end-to-end bar of tests/test_pipeline_gpu.py); the call does not wait for the GPU."""
import ctypes
import os
import sys
import time

import numpy as np
import pytest
import torch

from migan_b200 import _abi, synthetic
from migan_b200.pipeline import MIGAN_Pipeline
from oracle import pipeline_oracle as PO

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import make_golden_pipeline as MG  # noqa: E402  (case table + seeded inputs only; main() needs the reference)

pytestmark = pytest.mark.gpu
GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "pipeline.npz"))


class GivenOutput(torch.nn.Module):
    """Stands in for the generator: records the model input, returns a fixed y."""

    def __init__(self, y):
        super().__init__()
        self.y, self.x = y, None

    def forward(self, x):
        self.x = x.clone()
        return self.y


_PIPES = {}


def _pipe(res, pad, device):
    if res not in _PIPES:
        _PIPES[res] = MIGAN_Pipeline(synthetic.export_style_state_dict(res, seed=11), res, padding=pad, device=device)
    p = _PIPES[res]
    p.padding = pad
    return p


def _with_output(pipe, y, fn):
    real = pipe.model
    try:
        pipe.model = GivenOutput(y)
        return fn(), pipe.model.x
    finally:
        pipe.model = real


def test_golden_cases_as_one_ragged_batch(cuda_device):
    cases = [c for c in MG.CASES if c[1] == 64]
    pipe = _pipe(64, 16, cuda_device)
    images = [MG.case_inputs(c)[0].to(cuda_device) for c in cases]
    masks = [MG.case_inputs(c)[1].to(cuda_device) for c in cases]
    ptrs = [im.data_ptr() for im in images]
    y = torch.from_numpy(np.concatenate([GOLD["y_" + c[0]] for c in cases])).to(cuda_device)
    out, x = _with_output(pipe, y, lambda: pipe.forward_batch(images, masks))
    assert [o.data_ptr() for o in out] == ptrs                                 # in place
    boxes = pipe.last_boxes.cpu().numpy()
    for i, c in enumerate(cases):
        assert tuple(boxes[i]) == tuple(GOLD["box_" + c[0]]), c[0]
        assert torch.equal(x[i:i + 1].cpu(), torch.from_numpy(GOLD["x_" + c[0]])), c[0]
        assert np.array_equal(out[i].cpu().numpy(), GOLD["final_" + c[0]]), c[0]


def test_r256_as_batch_of_one(cuda_device):
    case = [c for c in MG.CASES if c[0] == "r256"][0]
    pipe = _pipe(256, 128, cuda_device)
    image, mask = MG.case_inputs(case)
    img = image.to(cuda_device)
    y = torch.from_numpy(GOLD["y_r256"]).to(cuda_device)
    out, x = _with_output(pipe, y, lambda: pipe.forward_batch([img], [mask.to(cuda_device)]))
    assert tuple(pipe.last_boxes[0].tolist()) == tuple(int(v) for v in GOLD["box_r256"])
    assert torch.equal(x.cpu(), torch.from_numpy(GOLD["x_r256"]))
    assert np.array_equal(out[0].cpu().numpy(), GOLD["final_r256"])


def _bbox_masks():
    rng = np.random.RandomState(5)                     # the `bbox_cases` masks, drawn as make_golden_pipeline.py drew them
    for t in range(300):
        H, W = int(rng.randint(8, 400)), int(rng.randint(8, 400))
        mask = np.full((H, W), 255, np.uint8)
        for _ in range(int(rng.randint(0, 3))):
            a, b = sorted(rng.randint(0, H, 2)); c, d = sorted(rng.randint(0, W, 2))
            mask[a:b + 1, c:d + 1] = rng.choice([0, 0, 128, 254])
        pad = int(rng.choice([0, 5, 16, 128]))
        yield t, mask, pad


def test_device_crop_windows_of_pinned_masks(cuda_device):
    """The device hole-extent kernel + box step on the 300 pinned masks, batches grouped by padding.  Each mask starts at a
    different byte offset, so the unaligned head / tail of the 16-byte loads is exercised too."""
    lib = _abi.load()
    table = GOLD["bbox_cases"]
    groups = {}
    for t, mask, pad in _bbox_masks():
        groups.setdefault(pad, []).append((t, mask))
    seen = 0
    stream = torch.cuda.current_stream(cuda_device).cuda_stream
    for pad, items in groups.items():
        for s in range(0, len(items), _abi.PIPE_BATCH_MAX):
            chunk = items[s:s + _abi.PIPE_BATCH_MAX]
            keep = []
            reqs = (_abi.PipeReq * len(chunk))()
            for i, (t, mask) in enumerate(chunk):
                H, W = mask.shape
                buf = torch.empty(H * W + 16, dtype=torch.uint8, device=cuda_device)
                m = buf[t % 16:t % 16 + H * W].view(H, W)
                m.copy_(torch.from_numpy(mask))
                img = torch.zeros(3, H, W, dtype=torch.uint8, device=cuda_device)
                keep += [buf, img]
                reqs[i] = _abi.PipeReq(img.data_ptr(), m.data_ptr(), H, W, H, W)
            preqs = ctypes.cast(reqs, ctypes.c_void_p)
            nbytes = lib.b200_pipeline_batch_scratch_bytes(preqs, len(chunk), 64)
            scratch = torch.empty(nbytes, dtype=torch.uint8, device=cuda_device)
            boxes = torch.full((len(chunk), 4), -1, dtype=torch.int32, device=cuda_device)
            _abi.check(lib.b200_pipeline_batch_boxes(preqs, len(chunk), 64, pad, boxes.data_ptr(), scratch.data_ptr(), nbytes, stream))
            for (t, _), b in zip(chunk, boxes.cpu().numpy()):
                assert tuple(int(v) for v in b) == tuple(int(v) for v in table[t][3:]), t
                seen += 1
    assert seen == 300


def _ragged(rng, sizes, hole_frac=4, mask_sizes=None):
    images, masks = [], []
    for k, (H, W) in enumerate(sizes):
        MH, MW = (mask_sizes or {}).get(k, (H, W))
        images.append(torch.from_numpy(rng.randint(0, 256, size=(1, 3, H, W), dtype=np.uint8)))
        m = torch.full((1, 1, MH, MW), 255, dtype=torch.uint8)
        a = int(rng.randint(0, MH - MH // hole_frac)); c = int(rng.randint(0, MW - MW // hole_frac))
        m[:, :, a:a + max(1, MH // hole_frac), c:c + max(1, MW // hole_frac)] = 0
        masks.append(m)
    return images, masks


def test_large_ragged_batch_against_oracle(cuda_device):
    rng = np.random.RandomState(2024)
    g = torch.Generator().manual_seed(2025)
    pipe = _pipe(64, 16, cuda_device)
    sizes = [(2160, 3840), (1080, 1920), (257, 255), (65, 1000), (1100, 90), (512, 512)]
    images, masks = _ragged(rng, sizes, mask_sizes={3: (33, 500), 5: (300, 301)})
    pipe.padding = 128
    y = torch.randn(len(sizes), 3, 64, 64, generator=g)
    dev_imgs = [im.to(cuda_device) for im in images]
    out, x = _with_output(pipe, y.to(cuda_device), lambda: pipe.forward_batch(dev_imgs, [m.to(cuda_device) for m in masks]))
    boxes = pipe.last_boxes.cpu().numpy()
    for i in range(len(sizes)):
        taps = {}
        want = PO.forward(lambda _x: y[i:i + 1], images[i].clone(), masks[i], 64, 128, taps)
        got = out[i].cpu()
        assert tuple(int(v) for v in boxes[i]) == taps["box"], i
        assert torch.equal(x[i:i + 1].cpu(), taps["x"]), i
        assert torch.equal(got, want), (i, int((got != want).sum()))
        x0, x1, y0, y1 = taps["box"]
        outside = torch.ones_like(got, dtype=torch.bool)
        outside[:, :, y0:y1, x0:x1] = False
        assert torch.equal(got[outside], images[i][outside]), i


def test_end_to_end_against_sequential_requests(cuda_device):
    res = 256
    batch_pipe = MIGAN_Pipeline(synthetic.export_style_state_dict(res, seed=3), res, padding=128, device=cuda_device)
    seq_pipe = MIGAN_Pipeline(synthetic.export_style_state_dict(res, seed=3), res, padding=128, device=cuda_device)
    rng = np.random.RandomState(31)
    sizes = [(300, 420), (1080, 1920), (256, 256), (97, 513), (720, 1280), (513, 97), (400, 300), (2160, 3840)]
    images, masks = _ragged(rng, sizes, mask_sizes={6: (200, 150)})
    dev_imgs = [im.to(cuda_device) for im in images]
    dev_masks = [m.to(cuda_device) for m in masks]
    batch_pipe.forward_batch(dev_imgs, dev_masks)
    # Is the generator batch-invariant?  Same x through batch N and through N batches of one.
    xs = torch.randn(len(sizes), 4, res, res, generator=torch.Generator().manual_seed(5)).to(cuda_device)
    y_all = batch_pipe.model(xs)
    y_one = torch.cat([seq_pipe.model(xs[i:i + 1]) for i in range(len(sizes))])
    invariant = torch.equal(y_all, y_one)
    print("generator batch-invariant (batch %d vs batches of 1): %s, max-abs %.3e" % (
        len(sizes), invariant, float((y_all - y_one).abs().max())))
    boxes = batch_pipe.last_boxes.cpu().tolist()
    for i in range(len(sizes)):
        one = seq_pipe(images[i].clone().to(cuda_device), masks[i].to(cuda_device))
        assert list(seq_pipe.last_box) == boxes[i], i
        got, want = dev_imgs[i].cpu(), one.cpu()
        if invariant:
            assert torch.equal(got, want), (i, int((got != want).sum()))
        else:
            x0, x1, y0, y1 = boxes[i]
            diff = (got.int() - want.int()).abs()
            assert int(diff.max()) <= 1, (i, int(diff.max()))
            assert float((diff[:, :, y0:y1, x0:x1] > 0).float().mean()) < 0.02, i
            outside = torch.ones_like(got, dtype=torch.bool)
            outside[:, :, y0:y1, x0:x1] = False
            assert torch.equal(got[outside], images[i][outside]), i


def test_no_host_synchronisation(cuda_device):
    pipe = MIGAN_Pipeline(synthetic.export_style_state_dict(64, seed=4), 64, padding=16, device=cuda_device)
    rng = np.random.RandomState(8)
    sizes = [(1080, 1920), (300, 200), (64, 64), (513, 777), (2160, 3840), (90, 1000)]
    images, masks = _ragged(rng, sizes, mask_sizes={1: (150, 100)})
    dev_masks = [m.to(cuda_device) for m in masks]
    warm = [im.to(cuda_device) for im in images]
    pipe.forward_batch(warm, dev_masks)                                 # warm-up at the same shapes
    expect = [w.clone() for w in warm]
    dev_imgs = [im.to(cuda_device) for im in images]
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream(cuda_device)
    t0 = time.perf_counter()
    torch.cuda._sleep(int(100e-3 * torch.cuda.get_device_properties(cuda_device).clock_rate * 1e3))   # ~100 ms of spinning
    pipe.forward_batch(dev_imgs, dev_masks)
    returned = time.perf_counter() - t0
    busy = not stream.query()
    torch.cuda.synchronize()
    slept = time.perf_counter() - t0
    print("forward_batch returned after %.1f ms of a %.1f ms sleep" % (returned * 1e3, slept * 1e3))
    assert busy, "the stream was idle when forward_batch returned: the call waited for the GPU"
    assert returned < 0.5 * slept, (returned, slept)
    for a, b in zip(dev_imgs, expect):
        assert torch.equal(a, b)


def test_argument_checks(cuda_device):
    pipe = _pipe(64, 16, cuda_device)
    img = torch.zeros(3, 40, 50, dtype=torch.uint8, device=cuda_device)
    mask = torch.full((40, 50), 255, dtype=torch.uint8, device=cuda_device)
    with pytest.raises(RuntimeError):
        pipe.forward_batch([img, img.clone()], [mask])
    with pytest.raises(RuntimeError):
        pipe.forward_batch([], [])
    with pytest.raises(RuntimeError):
        pipe.forward_batch([img.float()], [mask])
    with pytest.raises(RuntimeError):
        pipe.forward_batch([img[:2]], [mask])
    with pytest.raises(RuntimeError):
        pipe.forward_batch([torch.zeros(3, 2, 50, dtype=torch.uint8, device=cuda_device)], [mask])


def test_images_on_two_devices(cuda_device):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible CUDA devices")
    pipe = _pipe(64, 16, cuda_device)
    img = torch.zeros(3, 40, 50, dtype=torch.uint8, device=cuda_device)
    mask = torch.full((40, 50), 255, dtype=torch.uint8, device=cuda_device)
    with pytest.raises(RuntimeError):
        pipe.forward_batch([img, img.to("cuda:1")], [mask, mask])
