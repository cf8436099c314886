/* migan_b200.h -- C ABI of the B200-native MI-GAN generator forward.
 *
 * The shared library (mi-gan_b200/lib/libmigan_b200.so, built by __graft_entry__.build())
 * exports exactly the entry points declared here: plain pointers and sizes, no torch types.
 * Each one replaces a reference interface, cited as file:line in /root/reference:
 *
 *   migan_create / migan_destroy      Generator.__init__            lib/model_zoo/migan_inference.py:355-360
 *   migan_set_weight / _finalize      nn.Module.load_state_dict as used by scripts/demo.py:110
 *                                     (key names + shapes = the reference state_dict, SURVEY.md 8b)
 *   migan_forward                     Generator.forward(x)          lib/model_zoo/migan_inference.py:362-369
 *   migan_forward_host                scripts/demo.py:131-136 (x.to(device) -> model(x) -> .cpu())
 *   migan_forward_u8, b200_pre/postprocess_u8   scripts/demo.py:56-66 (preprocess) and :135-142 (uint8 + mask composite)
 *   b200_upfirdn2d                    _plugin.upfirdn2d(...)        torch_utils/ops/upfirdn2d.cpp:16-94
 *   b200_bias_act                     _plugin.bias_act(...)         torch_utils/ops/bias_act.cpp:32-90 (grad == 0)
 *   b200_conv1x1_nhwc                 the F.conv2d of conv2d_resample's 1x1 branches  torch_utils/ops/conv2d_resample.py:106-116
 *
 * Conventions: every function returns 0 on success and a non-zero code on failure, after
 * which migan_last_error() describes the failure (thread-local string).  All device pointers
 * are fp32, 16-byte aligned, on the device the context was created for; `stream` is a
 * cudaStream_t passed as void* (NULL = legacy default stream).  Nothing here falls back to
 * the CPU: without a CUDA device every compute entry point fails with MIGAN_ERR_CUDA.
 */
#ifndef MIGAN_B200_H_
#define MIGAN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MIGAN_OK 0
#define MIGAN_ERR_INVALID 1   /* bad argument (shape, resolution, null pointer, unknown key) */
#define MIGAN_ERR_CUDA 2      /* a CUDA runtime/driver call or kernel launch failed */
#define MIGAN_ERR_STATE 3     /* call order (e.g. forward before weights are finalized) */
#define MIGAN_ERR_WORKSPACE 4 /* workspace too small or misaligned */

/* Contraction engine for the 1x1 pointwise convs. */
#define MIGAN_PATH_SIMT 0     /* fp32 CUDA-core FMA (bring-up / cross-check path) */
#define MIGAN_PATH_TC 1       /* tcgen05 tensor cores, fp16 hi/lo 3-pass split, fp32 accumulate (fp32-faithful) */
#define MIGAN_PATH_TC_FAST 2  /* tcgen05, single fp16 pass (stated lower accuracy, see DESIGN.md) */

typedef struct migan_ctx migan_ctx;

const char* migan_last_error(void);
const char* migan_version(void);

/* Generator(resolution): resolution must be a power of two >= 8 (reference raises ValueError
 * otherwise, migan_inference.py:214-216).  `device` is a CUDA ordinal. */
int migan_create(int resolution, int device, migan_ctx** out);
int migan_destroy(migan_ctx* ctx);

/* Number of state_dict entries the context expects and their names/shapes, in the reference's
 * own state_dict order (154 keys @256, 177 @512). */
int migan_num_weights(const migan_ctx* ctx);
int migan_weight_info(const migan_ctx* ctx, int index, const char** name, int* ndim, int64_t shape[4]);

/* Copy one state_dict tensor (HOST pointer, fp32, contiguous, reference layout OIHW etc.).
 * Unknown names or wrong element counts fail with MIGAN_ERR_INVALID. */
int migan_set_weight(migan_ctx* ctx, const char* name, const float* host_data, int64_t numel);
/* Validate that every key was provided (and that filter_const is the zero-insertion pattern the
 * kernels implement), repack for the kernels (NHWC tap-major depthwise weights, K-major fp16
 * hi/lo pointwise weights, pre-multiplied noise) and upload.  Synchronous. */
int migan_finalize_weights(migan_ctx* ctx);

/* Scratch memory the caller must provide to migan_forward for a batch of n images. */
size_t migan_workspace_bytes(const migan_ctx* ctx, int n);

/* y[n,3,R,R] = Generator.forward(x[n,4,R,R]); x, y, workspace are DEVICE pointers (NCHW fp32,
 * contiguous).  Asynchronous on `stream`. */
int migan_forward(migan_ctx* ctx, const float* x, float* y, int n,
                  void* workspace, size_t workspace_bytes, int path, void* stream);

/* Latency form for small batches (the reference's primary caller runs batch 1: scripts/demo.py:125-142): the launch
 * sequence of one forward is captured ONCE into a CUDA graph that works on fixed staging buffers at the end of the
 * workspace, and replayed per call between two device-to-device copies (x in, y out) -- 3 submissions instead of ~50.
 * Same contract as migan_forward (DEVICE x / y, asynchronous on `stream`); the graph is rebuilt when n, path, the
 * workspace or the weights change.  workspace_bytes must be >= migan_workspace_bytes(n) + migan_graph_staging_bytes(n). */
size_t migan_graph_staging_bytes(const migan_ctx* ctx, int n);
int migan_forward_graph(migan_ctx* ctx, const float* x, float* y, int n,
                        void* workspace, size_t workspace_bytes, int path, void* stream);

/* Same with HOST x / y (pinned for full speed): H2D copy, forward, D2H copy; y_host is complete on return.
 * The batch is split into two micro-batches whose copies overlap the kernels (three streams).  The device
 * staging buffers (two slots) live at the end of the workspace:
 * workspace_bytes must be >= migan_workspace_bytes(n) + migan_host_staging_bytes(n). */
size_t migan_host_staging_bytes(const migan_ctx* ctx, int n);
int migan_forward_host(migan_ctx* ctx, const float* x_host, float* y_host, int n,
                       void* workspace, size_t workspace_bytes, int path, void* stream);
/* Serving form: enqueue only.  Consecutive calls alternate between the two staging slots, so the copies of
 * batch t+1 overlap the kernels and the copy-out of batch t (the batch is not split here: the overlap is across calls); migan_host_wait() blocks until every enqueued
 * batch has landed in its y_host.  x_host / y_host must stay valid (and unmodified) until then. */
int migan_forward_host_async(migan_ctx* ctx, const float* x_host, float* y_host, int n,
                             void* workspace, size_t workspace_bytes, int path, void* stream);
int migan_host_wait(migan_ctx* ctx);

/* uint8 request path (the callers' pre/post-processing fused around the forward, scripts/demo.py:56-66 and :135-142):
 * img_host u8 [n,R,R,3] (RGB, HWC), mask_host u8 [n,R,R] (255 = known pixel, anything else = hole) ->
 * out_host u8 [n,R,R,3] = known pixels of img, generated pixels elsewhere.  7 bytes per pixel cross PCIe instead of 28.
 * workspace_bytes must be >= migan_workspace_bytes(n) + migan_u8_staging_bytes(n) (two staging slots).
 * migan_forward_u8 is synchronous (out_host complete on return); migan_forward_u8_async only enqueues -- consecutive calls
 * alternate between the slots so that the copies of request t+1 / t-1 run under the kernels of request t, and
 * migan_host_wait() blocks until every enqueued request has landed (buffers must stay valid and unmodified until then). */
size_t migan_u8_staging_bytes(const migan_ctx* ctx, int n);
int migan_forward_u8(migan_ctx* ctx, const uint8_t* img_host, const uint8_t* mask_host, uint8_t* out_host, int n,
                     void* workspace, size_t workspace_bytes, int path, void* stream);
int migan_forward_u8_async(migan_ctx* ctx, const uint8_t* img_host, const uint8_t* mask_host, uint8_t* out_host, int n,
                           void* workspace, size_t workspace_bytes, int path, void* stream);
/* The two kernels on their own (DEVICE pointers): x[n,4,r,r] = cat([mask-0.5, img*mask]) and the composite of y[n,3,r,r]. */
int b200_preprocess_u8(const uint8_t* img_hwc, const uint8_t* mask_hw, float* x_nchw, int n, int r, void* stream);
int b200_postprocess_u8(const float* y_nchw, const uint8_t* img_hwc, const uint8_t* mask_hw, uint8_t* out_hwc, int n, int r,
                        void* stream);

/* Feathered composite of the deployed (ONNX) pipeline, scripts/create_onnx_pipeline.py:233-245, for a crop at the model
 * resolution (DEVICE pointers, NCHW like the pipeline): blend weight = 5x5 smoothing (reflect border) of the 3x3 max-pooled
 * mask / 255; out = clamp(image * w + ((y*0.5+0.5)*255).clamp(0,255) * (1 - w), 0, 255) -> uint8.  k25 = the 25 smoothing
 * taps on the HOST (the GaussianSmoothing buffer of :66-88; migan_b200.ops.feather_kernel() builds it the same way). */
int b200_feather_composite(const float* y_nchw, const uint8_t* image_nchw, const uint8_t* mask_n1hw, uint8_t* out_nchw,
                           int n, int H, int W, const float* k25_host, void* stream);

/* Arbitrary-resolution crop pipeline of the deployed (ONNX) form, scripts/create_onnx_pipeline.py:121-264 (MIGAN_Pipeline):
 * the caller's image u8 [3,H,W] and mask u8 [H,W] (255 = known) stay at their own size; the hole's bounding box is padded,
 * squared and clipped into a crop window, the crop is resized to the model resolution for the generator and the result is
 * resized back and blended into the image with a feathered mask.  The stages (DEVICE pointers unless noted):
 *   b200_resize_nearest_u8    mask at another size -> image size (tvF.resize NEAREST, :255)
 *   b200_hole_flags           flags[x] / flags[W + y] = column x / row y contains a value < 255 (:144-149); copy them to the host
 *   migan_crop_box            HOST arithmetic of get_masked_bbox (:151-227) -> box = {x_min, x_max, y_min, y_max}
 *   b200_pipeline_preprocess  crop -> anti-aliased bilinear resize, round -> x[4,res,res] = cat([m/255-0.5, (v*2/255-1)*m/255]) (:229-236)
 *   b200_pipeline_postprocess y[3,res,res] -> [0,255] -> anti-aliased bilinear resize to the crop -> feathered blend (3x3 max-pool,
 *                             5x5 smoothing with the 25 HOST taps k25, reflect border) written into image[crop] in place (:238-262)
 * The resize reproduces what torchvision's tensor `resize` computes on the CPU (ATen's separable anti-aliased filter, fp32
 * fused multiply-adds, width pass first) bit for bit; a pass whose size does not change is the identity.
 * scratch: b200_pipeline_scratch_bytes(H, W, res) bytes of device memory, shared by the two stages. */
size_t b200_pipeline_scratch_bytes(int H, int W, int res);
int b200_resize_nearest_u8(const uint8_t* in_hw, int H, int W, uint8_t* out_hw, int out_h, int out_w, void* stream);
int b200_hole_flags(const uint8_t* mask_hw, int H, int W, uint8_t* flags_w_plus_h, void* stream);
int migan_crop_box(const uint8_t* flags_host, int H, int W, int resolution, int padding, int* box4_host);
int b200_pipeline_preprocess(const uint8_t* image_chw, const uint8_t* mask_hw, int H, int W, const int* box4_host, int resolution,
                             float* x_nchw, void* scratch, size_t scratch_bytes, void* stream);
int b200_pipeline_postprocess(const float* y_nchw, uint8_t* image_chw, const uint8_t* mask_hw, int H, int W, const int* box4_host,
                              int resolution, const float* k25_host, void* scratch, size_t scratch_bytes, void* stream);

/* Batched crop pipeline: n requests of any sizes in one call, crop windows found on the device.  Request i is image_chw u8
 * [3,H,W] (updated in place) and mask_hw u8 [mask_h,mask_w] (255 = known), DEVICE pointers; the table itself is a HOST
 * array of at most MIGAN_PIPE_BATCH_MAX entries, passed to the kernels by value (no staging copy, no host wait).  H, W >= 3.
 * Every stage is a fixed number of launches for the whole batch, sized on the host for crops as large as their images; the
 * kernels read the actual windows from boxes (DEVICE int32 [n][4] = {x_min, x_max, y_min, y_max}), which the host never reads:
 *   b200_pipeline_batch_boxes       masks at another size -> image size (nearest); hole extents of every mask in one pass
 *                                   (16-byte loads, warp reductions, atomics); extents -> crop windows (the arithmetic of
 *                                   migan_crop_box) -> boxes.  3 launches, 4 when some mask needs resizing.
 *   b200_pipeline_batch_preprocess  weight tables, width pass, height pass fused with round + normalisation -> row i of
 *                                   x[n,4,res,res].  3 launches.
 *   [generator forward at batch n: y[n,3,res,res]]
 *   b200_pipeline_batch_postprocess weight tables, width pass of y, height pass fused into the feathered blend -> image[crop].
 *                                   3 launches.
 * Results equal b200_pipeline_preprocess / _postprocess per request bit for bit.  scratch: b200_pipeline_batch_scratch_bytes
 * bytes of device memory (16-byte aligned), the same area for the three calls of a batch (the resized masks live there). */
#define MIGAN_PIPE_BATCH_MAX 64
typedef struct migan_pipe_req {
    uint8_t* image_chw;
    const uint8_t* mask_hw;
    int H, W;
    int mask_h, mask_w;
} migan_pipe_req;
size_t b200_pipeline_batch_scratch_bytes(const migan_pipe_req* reqs_host, int n, int resolution);
int b200_pipeline_batch_boxes(const migan_pipe_req* reqs_host, int n, int resolution, int padding, int* boxes_dev,
                              void* scratch, size_t scratch_bytes, void* stream);
int b200_pipeline_batch_preprocess(const migan_pipe_req* reqs_host, int n, int resolution, const int* boxes_dev, float* x_nchw,
                                   void* scratch, size_t scratch_bytes, void* stream);
int b200_pipeline_batch_postprocess(const float* y_nchw, const migan_pipe_req* reqs_host, int n, int resolution, const int* boxes_dev,
                                    const float* k25_host, void* scratch, size_t scratch_bytes, void* stream);

/* Training snapshot -> inference filter, scripts/export_inference_model.py:18-27 (`get_source_w`): out[cout][fan] =
 * v * rsqrt(sum_fan v^2 + 1e-8) with v = (w_0 + ... + w_{k-1}) / sqrt(k) for a re-parameterised layer (k tensors) or v = w_0
 * (k = 1).  w_dev: HOST array of k DEVICE pointers to [cout][fan] fp32 tensors (fan = cin/groups * kh * kw); out: device.
 * Agrees with the reference's CPU result to a few ulp (the sum of squares is accumulated in fp64). */
int b200_reparam_filter(const float* const* w_dev, int k, int cout, int64_t fan, float* out, void* stream);

/* Stream memory operations for multi-GPU signalling (mi-gan_b200/parallel.py): the stream waits until the 32-bit word at a
 * DEVICE address reaches `value` (cyclic comparison (int32)(*addr - value) >= 0), or writes `value` to it, in stream order.
 * Executed by the stream's front end: no kernel, no SM.  b200_stream_memops_available() is 1 when the driver offers them. */
int b200_stream_memops_available(void);
int b200_stream_wait_value32(void* stream, void* addr, uint32_t value);
int b200_stream_write_value32(void* stream, void* addr, uint32_t value);
/* cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, stream): one copy-engine transfer between any two mapped device
 * addresses (local or a peer's), enqueued on `stream` of the CURRENT device and nothing else (no cross-device event exchange). */
int b200_memcpy_async(void* dst, const void* src, size_t bytes, void* stream);
/* cudaDeviceEnablePeerAccess(peer_device) for the CURRENT device (already enabled is not an error): copies between the two
 * devices' memory then go directly over NVLink instead of being staged. */
int b200_enable_peer_access(int peer_device);

/* Kernels launched by the most recent migan_forward on this context. */
int migan_last_launch_count(const migan_ctx* ctx);

/* Per-launch timing for roofline reports: when enabled, every kernel launch of subsequent
 * forwards is bracketed by cudaEvents on the launching stream.  migan_profile_step returns, for
 * step `index` of the current plan, its label ("<state_dict prefix><kernel>"), the duration of
 * its most recent launch (synchronizes on its end event), and its algorithmic bytes / flops
 * (own inputs read once + output written once; SURVEY.md section 8d). */
int migan_set_profiling(migan_ctx* ctx, int enable);
int migan_profile_num_steps(const migan_ctx* ctx);
int migan_profile_step(migan_ctx* ctx, int index, const char** label, float* ms, double* alg_bytes, double* flops);

/* Debug/test tap: during the next forwards, copy the named intermediate (converted to NCHW
 * fp32) into `dst` (device pointer, large enough).  name == NULL clears the tap.  Names follow
 * the oracle's tap names (oracle/migan_oracle.py), e.g. "encoder.b256.conv1.out". */
int migan_set_tap(migan_ctx* ctx, const char* name, float* dst);
/* Enumerate tap names produced by a forward on `path` (index from 0; returns MIGAN_ERR_INVALID
 * past the end).  shape = {C, H, W} of one image. */
int migan_tap_info(const migan_ctx* ctx, int path, int index, const char** name, int shape[3]);

/* Debug: every pipeline wait inside the tcgen05 kernel is bounded (seconds of wall-clock time); a wait that gives up records
 * (wait code | parity << 12 | block << 16) in a host-mapped word and traps.  Returns that record for `device` (0: none). */
int migan_debug_tc_timeout(int device);

/* upfirdn2d(x[n,c,h,w], f[fh,fw]) -> y[n,c,oh,ow], oh = (h*upy + pady0 + pady1 - fh + downy) / downy
 * (upfirdn2d.cpp:32-33).  f == NULL means the 1x1 identity filter.  Device pointers. */
int b200_upfirdn2d(const float* x, const float* f, float* y, int n, int c, int h, int w, int fh, int fw,
                   int upx, int upy, int downx, int downy, int padx0, int padx1, int pady0, int pady1,
                   int flip_filter, float gain, void* stream);

/* 1x1 convolution on channels-last data: y[p][o] = sum_i x[p][i] * w_t[i][o]  (fp32 CUDA-core GEMM;
 * the conv inside conv2d_resample's 1x1 branches, torch_utils/ops/conv2d_resample.py:106-116).
 * cin % 16 == 0, cout % 64 == 0. */
int b200_conv1x1_nhwc(const float* x, const float* w_t, float* y, int64_t pixels, int cin, int cout, void* stream);

/* bias_act forward: y = clamp(gain * act(x + b)), b indexed along the dimension whose stride is
 * step_b and size size_b (bias_act.cpp:72-73: (xi / stepB) % sizeB); b == NULL: no bias.
 * act: 1 linear 2 relu 3 lrelu 4 tanh 5 sigmoid 6 elu 7 selu 8 softplus 9 swish (bias_act.py:22-32);
 * clamp < 0 disables clamping. */
int b200_bias_act(const float* x, const float* b, float* y, int64_t numel, int64_t step_b, int size_b,
                  int act, float alpha, float gain, float clamp, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MIGAN_B200_H_ */
