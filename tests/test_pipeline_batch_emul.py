"""CPU checks of the batched crop pipeline (`b200_pipeline_batch_*`, mi-gan_b200/csrc/pipeline.cu) through the emulation build
(test infrastructure: the batched kernel functors run as host loops; the device hole-extent reduction, which uses warp
collectives, is replaced there by a host loop, and everything after it -- extents -> crop window -- is the shared code):

* the six resolution-64 requests of tests/golden/pipeline.npz as ONE ragged batch: crop windows, every row of x and every final
  image equal the reference's vectors bit for bit;
* random ragged batches (odd sizes, holes at the borders, masks at another size, random y) equal the single-request kernels
  per request bit for bit, and the oracle;
* the crop windows of the 300 pinned random masks (`bbox_cases`), run as batches grouped by padding.
"""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "emul"))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))

from oracle import pipeline_oracle as PO  # noqa: E402
from migan_b200 import _abi, ops  # noqa: E402
import build_emul  # noqa: E402
import make_golden_pipeline as MG  # noqa: E402  (case table + seeded inputs; its main() needs the reference and is not run here)

GOLD = np.load(os.path.join(ROOT, "tests", "golden", "pipeline.npz"))
BATCH_SYMBOLS = [s for s in _abi.SYMBOLS if s[0].startswith("b200_pipeline_batch_")]
PIPE_SYMBOLS = [s for s in _abi.SYMBOLS if s[0] in ("b200_pipeline_scratch_bytes", "b200_resize_nearest_u8", "b200_hole_flags",
                                                    "migan_crop_box", "b200_pipeline_preprocess", "b200_pipeline_postprocess")]


@pytest.fixture(scope="module")
def emul():
    return _abi.bind(ctypes.CDLL(build_emul.build()), BATCH_SYMBOLS)


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _aligned(nbytes):
    raw = np.empty(nbytes + 256, np.uint8)
    return raw[(-raw.ctypes.data) % 256:][:nbytes]


def _reqs(images, masks):
    reqs = (_abi.PipeReq * len(images))()
    for i, (im, m) in enumerate(zip(images, masks)):
        reqs[i] = _abi.PipeReq(im.ctypes.data, m.ctypes.data, im.shape[1], im.shape[2], m.shape[0], m.shape[1])
    return ctypes.cast(reqs, ctypes.c_void_p), reqs


def run_batch(lib, images, masks, res, pad, y):
    """images: list of uint8 [3,H,W] (updated in place), masks: list of uint8 [h,w], y: float32 [n,3,res,res].
    Returns (boxes [n,4], x [n,4,res,res])."""
    n = len(images)
    preqs, keep = _reqs(images, masks)
    nbytes = lib.b200_pipeline_batch_scratch_bytes(preqs, n, res)
    scratch = _aligned(nbytes)
    boxes = np.full((n, 4), -1, np.int32)
    x = np.full((n, 4, res, res), np.nan, np.float32)
    assert lib.b200_pipeline_batch_boxes(preqs, n, res, pad, _ptr(boxes), _ptr(scratch), nbytes, None) == 0
    assert lib.b200_pipeline_batch_preprocess(preqs, n, res, _ptr(boxes), _ptr(x), _ptr(scratch), nbytes, None) == 0
    k = np.ascontiguousarray(ops.feather_kernel().numpy())
    yy = np.ascontiguousarray(y, np.float32)
    assert lib.b200_pipeline_batch_postprocess(_ptr(yy), preqs, n, res, _ptr(boxes), _ptr(k), _ptr(scratch), nbytes, None) == 0
    del keep
    return boxes, x


def run_single(lib, image, mask, res, pad, y):
    """One request through the single-request entry points (image [1,3,H,W] updated in place)."""
    image = np.ascontiguousarray(image[0]); mask = np.ascontiguousarray(mask[0, 0])
    H, W = image.shape[1], image.shape[2]
    if mask.shape != (H, W):
        m2 = np.empty((H, W), np.uint8)
        assert lib.b200_resize_nearest_u8(_ptr(mask), mask.shape[0], mask.shape[1], _ptr(m2), H, W, None) == 0
        mask = m2
    flags = np.empty(W + H, np.uint8)
    assert lib.b200_hole_flags(_ptr(mask), H, W, _ptr(flags), None) == 0
    box = np.zeros(4, np.int32)
    assert lib.migan_crop_box(_ptr(flags), H, W, res, pad, _ptr(box)) == 0
    nbytes = lib.b200_pipeline_scratch_bytes(H, W, res)
    scratch = _aligned(nbytes)
    x = np.empty((1, 4, res, res), np.float32)
    assert lib.b200_pipeline_preprocess(_ptr(image), _ptr(mask), H, W, _ptr(box), res, _ptr(x), _ptr(scratch), nbytes, None) == 0
    k = np.ascontiguousarray(ops.feather_kernel().numpy())
    yy = np.ascontiguousarray(y)
    assert lib.b200_pipeline_postprocess(_ptr(yy), _ptr(image), _ptr(mask), H, W, _ptr(box), res, _ptr(k), _ptr(scratch), nbytes, None) == 0
    return tuple(int(v) for v in box), x, image[None]


CASES64 = [c for c in MG.CASES if c[1] == 64 and c[2] == 16]


def test_golden_cases_as_one_ragged_batch(emul):
    assert [c[0] for c in CASES64] == ["down", "corner", "up", "mixed", "maskres", "nohole"]
    images, masks = [], []
    for case in CASES64:
        image, mask = MG.case_inputs(case)
        images.append(np.ascontiguousarray(image[0].numpy()))
        masks.append(np.ascontiguousarray(mask[0, 0].numpy()))
    y = np.concatenate([GOLD["y_" + c[0]] for c in CASES64])
    boxes, x = run_batch(emul, images, masks, 64, 16, y)
    for i, case in enumerate(CASES64):
        tag = case[0]
        assert tuple(boxes[i]) == tuple(GOLD["box_" + tag]), tag
        assert np.array_equal(x[i:i + 1], GOLD["x_" + tag]), (tag, int((x[i:i + 1] != GOLD["x_" + tag]).sum()))
        want = GOLD["final_" + tag][0]
        assert np.array_equal(images[i], want), (tag, int((images[i] != want).sum()))


def random_request(rng, H, W, mask_size=None):
    # holes are 0: with partial values (128, 254) torch's convolution in the oracle and the kernels' fp64 tap sum can round
    # the blend weight apart on rare pixels, for the single-request kernels as well; the golden cases cover such values
    image = rng.randint(0, 256, size=(1, 3, H, W), dtype=np.uint8)
    MH, MW = mask_size or (H, W)
    mask = np.full((1, 1, MH, MW), 255, np.uint8)
    kind = rng.randint(0, 4)
    if kind == 0:                                              # hole touching the top-left border
        mask[:, :, :rng.randint(1, MH // 2 + 1), :rng.randint(1, MW // 2 + 1)] = 0
    elif kind == 1:                                            # hole touching the bottom-right border
        mask[:, :, MH - rng.randint(1, MH // 2 + 1):, MW - rng.randint(1, MW // 2 + 1):] = 0
    elif kind == 2:                                            # interior hole
        a, b = sorted(rng.randint(0, MH, 2)); c, d = sorted(rng.randint(0, MW, 2))
        mask[:, :, a:b + 1, c:d + 1] = 0
    return torch.from_numpy(image), torch.from_numpy(mask)     # kind 3: no hole


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_random_ragged_batches_match_oracle(emul, seed):
    """Per request: bit for bit the single-request kernels (b200_pipeline_preprocess / _postprocess), and the oracle's crop
    window and x.  The final image equals the oracle's except where the single-request kernels differ from it too: on rare
    pixels torch's fp32 convolution in the oracle and the kernels' fp64 tap sum round the blend weight to neighbouring floats
    (one uint8 level; seed 1 has one such pixel)."""
    single = _abi.bind(ctypes.CDLL(build_emul.build()), PIPE_SYMBOLS)
    rng = np.random.RandomState(300 + seed)
    g = torch.Generator().manual_seed(400 + seed)
    res, pad = [(32, 8), (64, 0), (32, 40)][seed]
    n = 5
    reqs = []
    for i in range(n):
        H, W = int(rng.randint(3, 230)), int(rng.randint(3, 230))
        other = rng.rand() < 0.4
        reqs.append(random_request(rng, H, W, (int(rng.randint(2, 120)), int(rng.randint(2, 120))) if other else None))
    y = torch.randn(n, 3, res, res, generator=g)
    images = [np.ascontiguousarray(im[0].numpy().copy()) for im, _ in reqs]
    masks = [np.ascontiguousarray(m[0, 0].numpy()) for _, m in reqs]
    boxes, x = run_batch(emul, images, masks, res, pad, y.numpy())
    for i, (image, mask) in enumerate(reqs):
        taps = {}
        want = PO.forward(lambda _x: y[i:i + 1], image.clone(), mask, res, pad, taps)[0].numpy()
        box1, x1, final1 = run_single(single, image.numpy().copy(), mask.numpy(), res, pad, y[i:i + 1].numpy())
        assert tuple(int(v) for v in boxes[i]) == taps["box"] == box1, (seed, i)
        assert np.array_equal(x[i:i + 1], taps["x"].numpy()) and np.array_equal(x[i:i + 1], x1), (seed, i)
        assert np.array_equal(images[i], final1[0]), (seed, i, int((images[i] != final1[0]).sum()))
        off = images[i] != want
        assert np.array_equal(off, final1[0] != want), (seed, i)
        assert int(np.abs(images[i].astype(int) - want.astype(int)).max()) <= 1 and int(off.sum()) <= 1, (seed, i, int(off.sum()))


def random_bbox_masks():
    """The masks of the `bbox_cases` table (seed 5), drawn exactly as make_golden_pipeline.py drew them."""
    rng = np.random.RandomState(5)
    for t in range(300):
        H, W = int(rng.randint(8, 400)), int(rng.randint(8, 400))
        mask = np.full((H, W), 255, np.uint8)
        for _ in range(int(rng.randint(0, 3))):
            a, b = sorted(rng.randint(0, H, 2)); c, d = sorted(rng.randint(0, W, 2))
            mask[a:b + 1, c:d + 1] = rng.choice([0, 0, 128, 254])
        pad = int(rng.choice([0, 5, 16, 128]))
        yield t, mask, pad


def test_crop_windows_of_pinned_masks(emul):
    """The 300 `bbox_cases` masks (seed 5), batches grouped by padding."""
    table = GOLD["bbox_cases"]
    groups = {}
    for t, mask, pad in random_bbox_masks():
        groups.setdefault(pad, []).append((t, np.ascontiguousarray(mask)))
    seen = 0
    for pad, items in groups.items():
        for s in range(0, len(items), _abi.PIPE_BATCH_MAX):
            chunk = items[s:s + _abi.PIPE_BATCH_MAX]
            masks = [m for _, m in chunk]
            images = [np.zeros((3,) + m.shape, np.uint8) for m in masks]
            preqs, keep = _reqs(images, masks)
            nbytes = emul.b200_pipeline_batch_scratch_bytes(preqs, len(chunk), 64)
            scratch = _aligned(nbytes)
            boxes = np.full((len(chunk), 4), -1, np.int32)
            assert emul.b200_pipeline_batch_boxes(preqs, len(chunk), 64, pad, _ptr(boxes), _ptr(scratch), nbytes, None) == 0
            for (t, _), b in zip(chunk, boxes):
                assert tuple(int(v) for v in b) == tuple(int(v) for v in table[t][3:]), t
                seen += 1
    assert seen == 300
