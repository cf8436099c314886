"""`MIGAN_Pipeline`: the arbitrary-resolution crop pipeline of the deployed (ONNX) form, scripts/create_onnx_pipeline.py:121-264.

Same constructor and call as the reference class:

    pipe = MIGAN_Pipeline(model_path, resolution, padding=128, device="cuda")
    result = pipe(image, mask)       # image (1,3,H,W) uint8, mask (1,1,h,w) uint8 (255 = known); image is updated in place

What happens per request (all on the GPU, kernels in csrc/pipeline.cu behind include/migan_b200.h):
mask -> image size (nearest) -> hole flags per column / row -> [4 ints to the host] crop window (`get_masked_bbox`
arithmetic) -> crop resized to the model resolution (anti-aliased bilinear, bit-identical to torchvision's tensor resize on the
CPU) and turned into the generator input -> `Generator.forward` (the captured CUDA graph at batch 1) -> output mapped to
[0, 255], resized to the crop, blended into the image under the feathered mask.  The one host round trip is the crop
window: the sizes of everything after it depend on it.  There is no CPU path.

    pipe.forward_batch([image_i ...], [mask_i ...])   # any sizes; crop windows stay on the device (pipe.last_boxes)

serves many requests at once: the crop windows are reduced on the device and every later stage reads them from there, with
grids sized for a crop as large as its image, so the call never waits for the GPU and the generator runs once at batch N.
"""
from __future__ import annotations

import ctypes
from typing import List, Optional, Tuple, Union

import torch

from . import _abi, ops
from .generator import Generator


class MIGAN_Pipeline(torch.nn.Module):
    """Drop-in for scripts/create_onnx_pipeline.py:MIGAN_Pipeline.  `model_path`: a state_dict file written by the reference's
    export script (`torch.load`-able), a state_dict, or a ready `migan_b200.Generator`."""

    def __init__(self, model_path, resolution: int, padding: int = 128, device: Union[str, torch.device] = "cuda"):
        super().__init__()
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("migan_b200.MIGAN_Pipeline runs on a CUDA device (there is no CPU path); got %s" % device)
        if isinstance(model_path, Generator):
            if model_path.resolution != resolution:
                raise RuntimeError("generator resolution %d != pipeline resolution %d" % (model_path.resolution, resolution))
            self.model = model_path
        else:
            self.model = Generator(resolution=resolution)
            sd = model_path if isinstance(model_path, dict) else torch.load(model_path, map_location="cpu")
            self.model.load_state_dict(sd)
        self.model = self.model.to(device).eval()
        self.register_buffer("gaussian_kernel", ops.feather_kernel(5, 1.0))     # GaussianSmoothing(1, 5, 1.0), :127-128
        self._k25 = ops.feather_kernel(5, 1.0).contiguous()                     # host copy handed to the C ABI
        self.res = int(resolution)
        self.padding = int(padding)
        self.device_ = device
        self._scratch = None
        self._bscratch = None                                                   # forward_batch's, laid out per call by the C side
        self.last_box: Tuple[int, int, int, int] = (0, 0, 0, 0)
        self.last_boxes: Optional[torch.Tensor] = None                          # forward_batch's crop windows, on the device

    # -- stages (each a call into the C ABI) ------------------------------------------------------------------------
    def get_masked_bbox(self, mask: torch.Tensor) -> Tuple[int, int, int, int]:
        """(x_min, x_max, y_min, y_max) of the crop window for a uint8 CUDA mask [..., H, W] (:133-227)."""
        lib = _abi.load()
        H, W = int(mask.shape[-2]), int(mask.shape[-1])
        mask = mask.reshape(H, W).contiguous()
        flags = torch.empty(W + H, dtype=torch.uint8, device=mask.device)
        with torch.cuda.device(mask.device):
            _abi.check(lib.b200_hole_flags(mask.data_ptr(), H, W, flags.data_ptr(), ops._stream(mask)))
        flags_h = flags.cpu()                                     # the one synchronisation of a request
        box = (ctypes.c_int * 4)()
        _abi.check(lib.migan_crop_box(flags_h.data_ptr(), H, W, self.res, int(self.padding), ctypes.cast(box, ctypes.c_void_p)))
        return int(box[0]), int(box[1]), int(box[2]), int(box[3])

    def _scratch_for(self, H: int, W: int, device) -> torch.Tensor:
        need = int(_abi.load().b200_pipeline_scratch_bytes(H, W, self.res))
        if self._scratch is None or self._scratch.numel() < need or self._scratch.device != device:
            self._scratch = torch.empty(need, dtype=torch.uint8, device=device)
        return self._scratch

    def _one(self, image: torch.Tensor, mask: torch.Tensor) -> None:
        """image [3,H,W] uint8 CUDA contiguous (updated in place), mask [h,w] uint8 CUDA."""
        lib = _abi.load()
        H, W = int(image.shape[1]), int(image.shape[2])
        if H < 3 or W < 3:
            raise RuntimeError("image of %d x %d: the feathering needs at least 3 x 3 pixels" % (H, W))
        stream = ops._stream(image)
        with torch.cuda.device(image.device):
            if tuple(mask.shape) != (H, W):                       # :255
                m2 = torch.empty((H, W), dtype=torch.uint8, device=image.device)
                _abi.check(lib.b200_resize_nearest_u8(mask.data_ptr(), int(mask.shape[0]), int(mask.shape[1]), m2.data_ptr(), H, W, stream))
                mask = m2
            x0, x1, y0, y1 = self.get_masked_bbox(mask)
            self.last_box = (x0, x1, y0, y1)
            box = (ctypes.c_int * 4)(x0, x1, y0, y1)
            pbox = ctypes.cast(box, ctypes.c_void_p)
            scratch = self._scratch_for(H, W, image.device)
            x = torch.empty((1, 4, self.res, self.res), dtype=torch.float32, device=image.device)
            _abi.check(lib.b200_pipeline_preprocess(image.data_ptr(), mask.data_ptr(), H, W, pbox, self.res, x.data_ptr(),
                                                    scratch.data_ptr(), scratch.numel(), stream))
            y = self.model(x)
            _abi.check(lib.b200_pipeline_postprocess(y.data_ptr(), image.data_ptr(), mask.data_ptr(), H, W, pbox, self.res,
                                                     self._k25.data_ptr(), scratch.data_ptr(), scratch.numel(), stream))

    @torch.no_grad()
    def forward(self, image: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
        """image: (N,3,H,W) uint8, mask: (N,1,h,w) uint8 (255 = known).  The image is updated in place and returned (like the
        reference, whose deployed form takes N = 1; N > 1 runs the requests one after the other, each with its own crop)."""
        if image.dtype != torch.uint8 or mask.dtype != torch.uint8:
            raise RuntimeError("MIGAN_Pipeline expects uint8 image and mask")
        if image.dim() != 4 or image.shape[1] != 3 or mask.dim() != 4 or mask.shape[1] != 1 or mask.shape[0] != image.shape[0]:
            raise RuntimeError("MIGAN_Pipeline expects image (N,3,H,W) and mask (N,1,h,w)")
        img_d = image if (image.is_cuda and image.is_contiguous()) else image.to(self.device_).contiguous()
        mask_d = mask.to(img_d.device).contiguous()
        for i in range(img_d.shape[0]):
            self._one(img_d[i], mask_d[i, 0])
        if img_d is not image:
            image.copy_(img_d)
        return image

    # -- batched requests ---------------------------------------------------------------------------------------------
    def _batch_scratch(self, nbytes: int, device) -> torch.Tensor:
        if self._bscratch is None or self._bscratch.numel() < nbytes or self._bscratch.device != device:
            self._bscratch = torch.empty(nbytes, dtype=torch.uint8, device=device)
        return self._bscratch

    @torch.no_grad()
    def forward_batch(self, images: List[torch.Tensor], masks: List[torch.Tensor]) -> List[torch.Tensor]:
        """Many requests of any sizes in one call.  images[i]: uint8 (3,H_i,W_i) or (1,3,H_i,W_i); masks[i]: uint8 (h_i,w_i),
        (1,h_i,w_i) or (1,1,h_i,w_i), 255 = known.  Each image is updated in place; the list is returned.

        The crop windows are found on the device and left there: `self.last_boxes` (int32 [N,4] = x_min, x_max, y_min, y_max).
        For device-resident contiguous inputs the call never waits for the GPU: a fixed number of launches per stage for the
        whole batch plus ONE generator forward at batch N (lists longer than MIGAN_PIPE_BATCH_MAX = 64 go in calls of 64).
        CPU or non-contiguous inputs are copied to the device and back, like `forward`."""
        if not isinstance(images, (list, tuple)) or not isinstance(masks, (list, tuple)):
            raise RuntimeError("forward_batch expects a list of images and a list of masks")
        if len(images) != len(masks):
            raise RuntimeError("forward_batch: %d images but %d masks" % (len(images), len(masks)))
        if len(images) == 0:
            raise RuntimeError("forward_batch: empty batch")
        devices = set()
        imgs, msks = [], []
        for i, (image, mask) in enumerate(zip(images, masks)):
            if image.dtype != torch.uint8 or mask.dtype != torch.uint8:
                raise RuntimeError("forward_batch: request %d: expected uint8 image and mask" % i)
            img = image[0] if image.dim() == 4 and image.shape[0] == 1 else image
            if img.dim() != 3 or img.shape[0] != 3:
                raise RuntimeError("forward_batch: request %d: image must be (3,H,W) or (1,3,H,W), got %s" % (i, tuple(image.shape)))
            if img.shape[1] < 3 or img.shape[2] < 3:
                raise RuntimeError("forward_batch: request %d: image of %d x %d (the feathering needs at least 3 x 3)" % (i, img.shape[1], img.shape[2]))
            if mask.dim() < 2 or mask.dim() > 4 or any(int(s) != 1 for s in mask.shape[:-2]) or mask.shape[-2] < 1 or mask.shape[-1] < 1:
                raise RuntimeError("forward_batch: request %d: mask must be (h,w), (1,h,w) or (1,1,h,w), got %s" % (i, tuple(mask.shape)))
            if image.is_cuda:
                devices.add(image.device)
            imgs.append(img)
            msks.append(mask.reshape(mask.shape[-2], mask.shape[-1]))
        if len(devices) > 1:
            raise RuntimeError("forward_batch: images on several devices %s" % sorted(str(d) for d in devices))
        device = devices.pop() if devices else self.device_
        work = [im if (im.is_cuda and im.is_contiguous()) else im.to(device).contiguous() for im in imgs]
        work_m = [m if (m.is_cuda and m.device == device and m.is_contiguous()) else m.to(device).contiguous() for m in msks]
        lib = _abi.load()
        stream = torch.cuda.current_stream(device).cuda_stream
        boxes = []
        with torch.cuda.device(device):
            for s in range(0, len(work), _abi.PIPE_BATCH_MAX):
                boxes.append(self._batch(lib, work[s:s + _abi.PIPE_BATCH_MAX], work_m[s:s + _abi.PIPE_BATCH_MAX], device, stream))
        self.last_boxes = boxes[0] if len(boxes) == 1 else torch.cat(boxes)
        for src, dst in zip(work, imgs):
            if src is not dst:
                dst.copy_(src)
        return list(images)

    def _batch(self, lib, imgs, msks, device, stream) -> torch.Tensor:
        n = len(imgs)
        reqs = (_abi.PipeReq * n)()
        for i, (im, m) in enumerate(zip(imgs, msks)):
            reqs[i] = _abi.PipeReq(im.data_ptr(), m.data_ptr(), int(im.shape[1]), int(im.shape[2]), int(m.shape[0]), int(m.shape[1]))
        preqs = ctypes.cast(reqs, ctypes.c_void_p)
        need = int(lib.b200_pipeline_batch_scratch_bytes(preqs, n, self.res))
        scratch = self._batch_scratch(need, device)
        boxes = torch.empty((n, 4), dtype=torch.int32, device=device)
        x = torch.empty((n, 4, self.res, self.res), dtype=torch.float32, device=device)
        _abi.check(lib.b200_pipeline_batch_boxes(preqs, n, self.res, int(self.padding), boxes.data_ptr(), scratch.data_ptr(),
                                                 scratch.numel(), stream))
        _abi.check(lib.b200_pipeline_batch_preprocess(preqs, n, self.res, boxes.data_ptr(), x.data_ptr(), scratch.data_ptr(),
                                                      scratch.numel(), stream))
        y = self.model(x)
        if tuple(y.shape) != (n, 3, self.res, self.res) or y.dtype != torch.float32 or y.device != device:
            raise RuntimeError("generator returned %s %s on %s, expected float32 (%d,3,%d,%d) on %s" % (
                tuple(y.shape), y.dtype, y.device, n, self.res, self.res, device))
        y = y.contiguous()
        _abi.check(lib.b200_pipeline_batch_postprocess(y.data_ptr(), preqs, n, self.res, boxes.data_ptr(), self._k25.data_ptr(),
                                                       scratch.data_ptr(), scratch.numel(), stream))
        return boxes
