// Internal launcher interface between the plan executor (migan_abi.cu) and the kernels.
// Activations are NHWC fp32 in HBM ([n, H, W, C], C a multiple of 4, 16-byte aligned);
// the RGB image path is planar NCHW fp32 ([n, 3, r, r]) so the last level is the output.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>

#include "../../include/migan_b200.h"

namespace migan {

// Per-device one-time setup (dynamic shared memory opt-in); called by migan_create.
cudaError_t configure_elementwise();
cudaError_t configure_sepconv_tc();

// ---- CUDA-core kernels (elementwise.cu) ---------------------------------------------
// fromrgb 1x1 (4 -> C0) + bias + lrelu_agc;  x NCHW [n,4,H,W] -> out NHWC [n,H,W,C0]
cudaError_t launch_stem(const float* x_nchw, const float* w, const float* b, float* out,
                        int n, int H, int W, int C0, cudaStream_t s);
// depthwise 3x3 (pad 1) + bias + lrelu_agc, NHWC -> NHWC.  w9 is tap-major [9][C].
// Writes fp32 (out, if non-null) and/or the scaled fp16 hi/lo split (out_hi/out_lo, if non-null).
cudaError_t launch_dw3x3(const float* in, const float* w9, const float* bias, float* out, __half* out_hi, __half* out_lo,
                         int n, int H, int W, int C, cudaStream_t s);
// depthwise 3x3 + bias + lrelu_agc, then 4x4 FIR stride 2 pad 1 (taps fir16 [16][C]).
// Writes fp32 [n,H/2,W/2,C] to out_f32 (if non-null) and/or the scaled fp16 hi/lo split
// (if out_hi non-null) that the tcgen05 GEMM consumes directly through TMA.
cudaError_t launch_dw3x3_down(const float* in, const float* w9, const float* bias, const float* fir16,
                              float* out_f32, __half* out_hi, __half* out_lo,
                              int n, int H, int W, int C, cudaStream_t s);
// Same stage specialised for the tensor-core feed (pre-split fp16 hi/lo output only): w9s / biass are the taps and bias
// pre-multiplied by kActSplitScale * sqrt(2); C in {64, 128, 256, 512}.
cudaError_t launch_dw3x3_down_split(const float* in, const float* w9s, const float* biass, const float* fir16,
                                    __half* out_hi, __half* out_lo, int n, int H, int W, int C, cudaStream_t s);
// TMA-staged variant (W/2 >= 16): a producer warp streams the input rows of a (64-channel, 36-column) slab into a shared-memory
// ring with cp.async.bulk.tensor (out-of-image rows / columns arrive zero-filled), so the row walk never waits on global
// memory.  `desc` = 128-byte CUtensorMap of the input made by make_down_tensor_map (host, once per plan).
struct alignas(64) DownTensorMap { unsigned char bytes[128]; };
const char* make_down_tensor_map(DownTensorMap* desc, const float* in, int n, int H, int W, int C);   // sepconv_tc.cu (driver entry point lives there)
cudaError_t launch_dw3x3_down_tma(const DownTensorMap& desc, const float* w9s, const float* biass, const float* fir16,
                                  __half* out_hi, __half* out_lo, int n, int H, int W, int C, cudaStream_t s);
// 2x polyphase FIR up-sampling of the raw 1x1-conv output + noise + lrelu_agc + skip add.
// t [n,h,w,C] -> out [n,2h,2w,C]; fir16 [16][C] (gain included); noise [2h*2w] (already
// multiplied by noise_strength) or null; skip [n,2h,2w,C] or null (added AFTER the activation).
cudaError_t launch_up2(const float* t, const float* fir16, const float* noise, const float* skip,
                       float* out, int n, int h, int w, int C, cudaStream_t s);
// img_out[n,3,r,r] = up2(img_lo[n,3,r/2,r/2]) + torgb(x[n,r,r,C]) + b;  img_lo may be null (b4).
cudaError_t launch_torgb(const float* x, const float* w, const float* b, const float* img_lo,
                         const float* fir16x3, float* img_out, int n, int r, int C, cudaStream_t s);
cudaError_t launch_add(float* x, const float* y, int64_t numel, cudaStream_t s);
cudaError_t launch_nhwc_to_nchw(const float* in, float* out, int n, int H, int W, int C, cudaStream_t s);
cudaError_t launch_split_f16(const float* in, __half* hi, __half* lo, float scale, int64_t numel, cudaStream_t s);

// ---- fp32 CUDA-core GEMM for the 1x1 conv (gemm_simt.cu) ----------------------------
// out[p][n] = epilogue( sum_k A[p][k] * Bt[k][n] ), A [P][K], Bt [K][N], out [P][N].
// epilogue: + noise[p % HW] (if noise) then lrelu_agc (if act).
cudaError_t launch_pw_gemm_simt(const float* A, const float* Bt, float* out, int64_t P, int K, int N,
                                const float* noise, int HW, int act, cudaStream_t s);

// ---- standalone ops (ops.cu) ---------------------------------------------------------
cudaError_t launch_upfirdn2d(const float* x, const float* f, float* y, int n, int c, int h, int w,
                             int fh, int fw, int upx, int upy, int downx, int downy,
                             int padx0, int padx1, int pady0, int pady1, int flip, float gain,
                             int oh, int ow, cudaStream_t s);
cudaError_t launch_bias_act(const float* x, const float* b, float* y, int64_t numel, int64_t step_b, int size_b,
                            int act, float alpha, float gain, float clamp, cudaStream_t s);

// ---- uint8 pre/post-processing (prepost.cu): demo.py:56-66 and :135-142 around the forward ------
// feathered composite of the ONNX pipeline (create_onnx_pipeline.py:233-245): NCHW uint8 image / mask, 25 smoothing taps (host array)
int launch_feather_composite(const float* y_nchw, const uint8_t* img_nchw, const uint8_t* mask_n1hw, uint8_t* out_nchw, int n, int H, int W,
                             const float* k25_host, cudaStream_t s);
int launch_preprocess_u8(const uint8_t* img_hwc, const uint8_t* mask_hw, float* x_nchw, int n, int r, cudaStream_t s);
int launch_postprocess_u8(const float* y_nchw, const uint8_t* img_hwc, const uint8_t* mask_hw, uint8_t* out_hwc, int n, int r,
                          cudaStream_t s);


// ---- arbitrary-resolution crop pipeline (pipeline.cu): scripts/create_onnx_pipeline.py:121-264 ------
size_t pipeline_scratch_bytes(int H, int W, int res);
int launch_resize_nearest_u8(const uint8_t* in, int H, int W, uint8_t* out, int oh, int ow, cudaStream_t s);
int launch_hole_flags(const uint8_t* mask, int H, int W, uint8_t* flags, cudaStream_t s);
void crop_box_from_flags(const uint8_t* flags_host, int H, int W, int res, int padding, int* box4);
int launch_pipeline_preprocess(const uint8_t* image, const uint8_t* mask, int H, int W, const int* box, int res, float* x,
                               void* scratch, cudaStream_t s);
int launch_pipeline_postprocess(const float* y, uint8_t* image, const uint8_t* mask, int H, int W, const int* box, int res,
                                const float* k25_host, void* scratch, cudaStream_t s);
// batched form (migan_pipe_req of include/migan_b200.h; boxes on the device)
size_t pipeline_batch_scratch_bytes(const migan_pipe_req* reqs, int n, int res);
int launch_pipeline_batch_boxes(const migan_pipe_req* reqs, int n, int res, int padding, int* boxes, void* scratch, cudaStream_t s);
int launch_pipeline_batch_preprocess(const migan_pipe_req* reqs, int n, int res, const int* boxes, float* x, void* scratch, cudaStream_t s);
int launch_pipeline_batch_postprocess(const float* y, const migan_pipe_req* reqs, int n, int res, const int* boxes,
                                      const float* k25_host, void* scratch, cudaStream_t s);


// ---- training snapshot -> inference filters (reparam.cu): scripts/export_inference_model.py:18-27 ------
int launch_reparam_filter(const float* const* w_dev, int k, int cout, int64_t fan, float* out, cudaStream_t s);

}  // namespace migan
