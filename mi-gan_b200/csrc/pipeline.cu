// Arbitrary-resolution crop pipeline around the generator: the deployed (ONNX) form of the reference,
// scripts/create_onnx_pipeline.py:121-264 (MIGAN_Pipeline), SURVEY.md 8(f) row f4.
//
//   mask (any size) --nearest--> image size                                                   (:255)
//   columns / rows that contain a hole (value < 255) -> flags -> [host] crop window            (:133-227, migan_crop_box)
//   crop --anti-aliased bilinear, round--> res x res uint8 -> x = cat([m/255 - 0.5, (v*2/255-1) * m/255])   (:229-236)
//   [generator forward]
//   y -> ((y*0.5+0.5)*255).clamp(0,255) --anti-aliased bilinear--> crop size -> feathered blend -> image[crop]  (:238-262)
//
// The resize is what torchvision's tensor `resize` lowers to: ATen's separable anti-aliased bilinear filter
// (aten/src/ATen/native/cpu/UpSampleKernel.cpp: HelperInterpBase::_compute_indices_min_size_weights_aa and
// basic_loop_aa_*): width pass, then height pass, each output = sum_j src[xmin + j] * w[j] accumulated left to
// right with fused multiply-adds in fp32; the weight table is evaluated exactly like the C++ (float scale / support /
// centre, the filter argument through double, w / total).  A pass whose size does not change is the identity there;
// here it runs with the table {xmin = i, 1 tap, w = 1}, which is the same value bit for bit.
// Item kernels (comod_kernels.cuh style): the emulation build runs the very same functors on the CPU against the oracle.
//
// Batched form (second half of the file): N requests of different sizes in one call, crop windows found on the device.
// Every stage is one launch for the whole batch; a block finds its request in a per-request block prefix table and walks
// the request's ACTUAL items (sizes read from the device box) in a grid-stride loop, the grid being sized on the host for
// the worst case (a crop is never larger than its image).  The per-value arithmetic is the helpers below, shared with the
// single-request functors.
#include "comod_kernels.cuh"
#include "../../include/migan_b200.h"

#ifdef MIGAN_EMULATE
#include <cmath>
#define PL_MUL(a, b) ((a) * (b))
#define PL_ADD(a, b) ((a) + (b))
#define PL_DIV(a, b) ((a) / (b))
#define PL_FMA(a, b, c) fmaf((a), (b), (c))
#define PL_RINT(a) rintf(a)
#define PL_D inline
#else
#include "kernels.h"
#define PL_MUL(a, b) __fmul_rn((a), (b))
#define PL_ADD(a, b) __fadd_rn((a), (b))
#define PL_DIV(a, b) __fdiv_rn((a), (b))
#define PL_FMA(a, b, c) __fmaf_rn((a), (b), (c))
#define PL_RINT(a) rintf(a)
#define PL_D __device__ __forceinline__
#endif

namespace comod {

// torch's mode='nearest' source index (ATen/native/UpSample.h nearest_neighbor_compute_source_index)
PL_D int nearest_src(int dst, int in_size, int out_size) {
    if (in_size == out_size) return dst;
    const float scale = PL_DIV((float)in_size, (float)out_size);
    const int s = (int)floorf(PL_MUL((float)dst, scale));
    return s < in_size - 1 ? s : in_size - 1;
}

// max_interp_size of _compute_index_ranges_weights (antialias branch): the taps of one output, on host and device
CK_HD int aa_maxk(int in_size, int out_size) {
    if (in_size == out_size) return 1;
    const float scale = (float)in_size / (float)out_size;
    const float support = scale >= 1.0f ? scale : 1.f;
    return (int)ceilf(support) * 2 + 1;
}

CK_HD int pl_imin(int a, int b) { return a < b ? a : b; }
CK_HD int pl_imax(int a, int b) { return a > b ? a : b; }

// Arithmetic of get_masked_bbox (:151-227) after the reduction: the hole's extents (x_min = W, x_max = 0, y_min = H,
// y_max = 0 when there is no hole) -> padded, squared, clipped crop window box = {x_min, x_max, y_min, y_max}.
CK_HD void crop_box_from_extents(int x_min, int x_max, int y_min, int y_max, int H, int W, int res, int padding, int* box) {
    x_min = pl_imin(x_min, x_max); x_max = pl_imax(x_min, x_max);
    y_min = pl_imin(y_min, y_max); y_max = pl_imax(y_min, y_max);
    const int cnt_x = (x_min + x_max) / 2, cnt_y = (y_min + y_max) / 2;      // non-negative: floor division == truncation
    int crop = pl_imax(x_max - x_min, y_max - y_min) + padding * 2;
    crop = pl_imax(crop, res);
    const int off = crop / 2;
    x_min = pl_imax(cnt_x - off, 0); x_max = pl_imin(cnt_x + off, W);
    y_min = pl_imax(cnt_y - off, 0); y_max = pl_imin(cnt_y + off, H);
    const int x_ex = pl_imax(crop - (x_max - x_min), 0), y_ex = pl_imax(crop - (y_max - y_min), 0);
    x_min = pl_imax(x_min - x_ex, 0); x_max = pl_imin(x_max + x_ex, W);
    y_min = pl_imax(y_min - y_ex, 0); y_max = pl_imin(y_max + y_ex, H);
    box[0] = x_min; box[1] = x_max; box[2] = y_min; box[3] = y_max;
}

// ---- per-value bodies, shared by the single-request functors and the batched ones ------------------------------------
PL_D void nearest_u8_item(const uint8_t* in, int H, int W, uint8_t* out, int oh, int ow, int64_t i) {   // i < oh*ow
    const int y = (int)(i / ow), x = (int)(i - (int64_t)y * ow);
    out[i] = in[(int64_t)nearest_src(y, H, oh) * W + nearest_src(x, W, ow)];
}

// One axis of the anti-aliased bilinear filter: for output index i the first source index, the tap count and the taps.
struct AaTable { int* xmin; int* xsize; float* w; int maxk; };

PL_D void aa_weights_item(const AaTable& t, int in_size, int out_size, int64_t i) {   // i < out_size
    float* w = t.w + i * t.maxk;
    if (in_size == out_size) {                          // the reference skips this pass: identity table
        t.xmin[i] = (int)i; t.xsize[i] = 1; w[0] = 1.f;
        for (int j = 1; j < t.maxk; ++j) w[j] = 0.f;
        return;
    }
    const float scale = PL_DIV((float)in_size, (float)out_size);           // area_pixel_compute_scale<float>
    const bool down = scale >= 1.0f;
    const float support = down ? scale : 1.f;                              // (interp_size * 0.5) * scale, interp_size = 2
    const float invscale = down ? (float)(1.0 / (double)scale) : 1.f;
    const float center = (float)((double)scale * ((double)i + 0.5));
    int lo = (int)((double)PL_ADD(center, -support) + 0.5);
    if (lo < 0) lo = 0;
    int hi = (int)((double)PL_ADD(center, support) + 0.5);
    if (hi > in_size) hi = in_size;
    int n = hi - lo;
    n = n < 0 ? 0 : (n > t.maxk ? t.maxk : n);
    float total = 0.f;
    for (int j = 0; j < n; ++j) {
        float a = (float)(((double)PL_ADD((float)(j + lo), -center) + 0.5) * (double)invscale);
        a = fabsf(a);
        const float v = a < 1.0f ? PL_ADD(1.f, -a) : 0.f;                  // aa_filter (triangle)
        w[j] = v;
        total = PL_ADD(total, v);
    }
    if (total != 0.f)
        for (int j = 0; j < n; ++j) w[j] = PL_DIV(w[j], total);
    for (int j = n; j < t.maxk; ++j) w[j] = 0.f;
    t.xmin[i] = lo; t.xsize[i] = n;
}

// Width pass.  SRC = 0: uint8 planes of the image crop; SRC = 1: generator output y mapped to [0, 255] on load (:239).
template <int SRC>
PL_D float aa_load(const void* src, int64_t o) {
    if (SRC == 0) return (float)static_cast<const uint8_t*>(src)[o];
    float g = PL_MUL(PL_ADD(PL_MUL(static_cast<const float*>(src)[o], 0.5f), 0.5f), 255.f);       // ((y * 0.5 + 0.5) * 255)
    return fminf(fmaxf(g, 0.f), 255.f);                                                           // .clamp(0, 255)
}
template <int SRC>   // i < C * rows * ow -> out [C][rows][ow]
PL_D void resize_width_item(const void* src, int64_t plane_stride, int row_stride, const AaTable& t, float* out, int rows, int ow,
                            int64_t i) {
    const int x = (int)(i % ow); int64_t r = i / ow;
    const int y = (int)(r % rows); const int c = (int)(r / rows);
    const int64_t base = c * plane_stride + (int64_t)y * row_stride + t.xmin[x];
    const float* w = t.w + (int64_t)x * t.maxk;
    float acc = PL_MUL(aa_load<SRC>(src, base), w[0]);
    for (int j = 1; j < t.xsize[x]; ++j) acc = PL_FMA(aa_load<SRC>(src, base + j), w[j], acc);
    out[i] = acc;
}

// Height pass, one output: taps down column x of one plane [ih][ow].
PL_D float aa_col(const float* plane, const AaTable& t, int y, int ow, int x) {
    const float* p = plane + (int64_t)t.xmin[y] * ow + x;
    const float* w = t.w + (int64_t)y * t.maxk;
    float acc = PL_MUL(p[0], w[0]);
    for (int j = 1; j < t.xsize[y]; ++j) acc = PL_FMA(p[(int64_t)j * ow], w[j], acc);
    return acc;
}

// Height pass of the image crop fused with the rest of MIGAN_Pipeline.preprocess (:229-236): round to uint8, nearest
// mask, normalise, x = cat([mask - 0.5, image * mask]).  in = width-pass output [3][hc][res]; i < res * res.
PL_D void preprocess_item(const float* in, const AaTable& t, const uint8_t* mask, int mask_row_stride, int hc, int wc, int res,
                          float* x, int64_t i) {
    const int ox = (int)(i % res), oy = (int)(i / res);
    const int64_t plane = (int64_t)res * res;
    const float m = PL_DIV((float)mask[(int64_t)nearest_src(oy, hc, res) * mask_row_stride + nearest_src(ox, wc, res)], 255.f);
    x[i] = PL_ADD(m, -0.5f);
    for (int c = 0; c < 3; ++c) {
        const float acc = aa_col(in + (int64_t)c * hc * res, t, oy, res, ox);
        const float v = (float)(uint8_t)PL_RINT(acc);                                        // round(), .to(uint8)
        const float n = PL_ADD(PL_DIV(PL_MUL(v, 2.f), 255.f), -1.f);                         // image * 2 / 255 - 1
        x[(c + 1) * plane + i] = PL_MUL(n, m);
    }
}

// Feathered blend of the resized generator output into the crop, in place (:241-248, :262).  Same arithmetic as FeatherK
// (prepost.cu) on a window of the full image: max-pool and reflect padding act at the CROP border, like the reference,
// which slices the crop before post-processing.  G: g(c, h, w, i) = resized generator output of channel c at (h, w).
template <class G>
PL_D void feather_item(const G& g, uint8_t* img, const uint8_t* mask, int64_t img_plane, int W, int hc, int wc, const float* k,
                       int64_t i) {   // i < hc * wc
    const int h = (int)(i / wc), w = (int)(i - (int64_t)h * wc);
    double acc = 0.0;
    for (int dy = -2; dy <= 2; ++dy) {
        int yy = h + dy;
        yy = yy < 0 ? -yy : (yy >= hc ? 2 * hc - 2 - yy : yy);
        for (int dx = -2; dx <= 2; ++dx) {
            int xx = w + dx;
            xx = xx < 0 ? -xx : (xx >= wc ? 2 * wc - 2 - xx : xx);
            int mx = 0;
            for (int a = -1; a <= 1; ++a) {
                const int y2 = yy + a;
                if (y2 < 0 || y2 >= hc) continue;
                for (int b = -1; b <= 1; ++b) {
                    const int x2 = xx + b;
                    if (x2 < 0 || x2 >= wc) continue;
                    const int v = mask[(int64_t)y2 * W + x2];
                    mx = v > mx ? v : mx;
                }
            }
            acc += (double)k[(dy + 2) * 5 + (dx + 2)] * (double)mx;
        }
    }
    const float wgt = PL_DIV((float)acc, 255.f);
    const float inv = PL_ADD(1.f, -wgt);
    for (int c = 0; c < 3; ++c) {
        uint8_t* px = img + c * img_plane + (int64_t)h * W + w;
        const float v = PL_ADD(PL_MUL((float)*px, wgt), PL_MUL(g(c, h, w, i), inv));
        *px = (uint8_t)fminf(fmaxf(v, 0.f), 255.f);
    }
}

// ---- single-request functors -------------------------------------------------------------------------------------------
struct NearestU8K {    // items = oh*ow: one uint8 plane [H][W] -> [oh][ow]
    const uint8_t* in; uint8_t* out; int H, W, oh, ow;
    PL_D void operator()(int64_t i) const { nearest_u8_item(in, H, W, out, oh, ow, i); }
};

struct HoleFlagsK {    // items = W + H: flags[x] = column x contains a value < 255, flags[W + y] likewise for row y  (:144-149)
    const uint8_t* mask; uint8_t* flags; int H, W;
    PL_D void operator()(int64_t i) const {
        uint8_t f = 0;
        if (i < W) { for (int y = 0; y < H && !f; ++y) f = mask[(int64_t)y * W + i] < 255; }
        else { const uint8_t* r = mask + (i - W) * (int64_t)W; for (int x = 0; x < W && !f; ++x) f = r[x] < 255; }
        flags[i] = f;
    }
};

struct AaWeightsK {    // items = out_size
    AaTable t; int in_size, out_size;
    PL_D void operator()(int64_t i) const { aa_weights_item(t, in_size, out_size, i); }
};

template <int SRC>
struct ResizeWidthK {  // items = C * rows * ow -> tmp [C][rows][ow]
    const void* src; int64_t plane_stride; int row_stride; AaTable t; float* out; int rows, ow;
    PL_D void operator()(int64_t i) const { resize_width_item<SRC>(src, plane_stride, row_stride, t, out, rows, ow, i); }
};

struct ResizeHeightK { // items = C * oh * ow: tmp [C][ih][ow] -> out [C][oh][ow]
    const float* in; AaTable t; float* out; int ih, oh, ow;
    PL_D void operator()(int64_t i) const {
        const int x = (int)(i % ow); int64_t r = i / ow;
        const int y = (int)(r % oh); const int c = (int)(r / oh);
        out[i] = aa_col(in + (int64_t)c * ih * ow, t, y, ow, x);
    }
};

struct PreprocessK {   // items = res * res
    const float* in; AaTable t; const uint8_t* mask; int mask_row_stride; int hc, wc, res; float* x;
    PL_D void operator()(int64_t i) const { preprocess_item(in, t, mask, mask_row_stride, hc, wc, res, x, i); }
};

struct PlaneG {        // resized generator output held in [3][hc][wc]
    const float* g; int64_t plane;
    PL_D float operator()(int c, int, int, int64_t i) const { return g[c * plane + i]; }
};

struct FeatherCropK {  // items = hc * wc
    const float* g; uint8_t* img; const uint8_t* mask; int64_t img_plane; int W; int hc, wc; float k[25];
    PL_D void operator()(int64_t i) const { feather_item(PlaneG{g, (int64_t)hc * wc}, img, mask, img_plane, W, hc, wc, k, i); }
};

// ---- batched functors ----------------------------------------------------------------------------------------------
// One request of a batch as the kernels see it (laid out on the host by migan::batch_layout).  Its scratch region starts
// at byte `scratch`: the resized mask (when the caller's mask is at another size), then a phase area shared by the
// preprocess tables + width-pass output and, after the generator, the postprocess tables + width-pass output.
struct PipeReq {
    uint8_t* image; const uint8_t* mask_in; uint8_t* mask;      // mask: the H x W mask (mask_in itself, or its copy in scratch)
    int64_t scratch, o_phase;                                   // byte offsets: region in the scratch, phase area in the region
    int H, W, mh, mw;
    int o_th, o_tmp, o_th2, o_tmp2;                             // in the phase area: height table / width-pass output, pre and post
};
// The table travels by value as a kernel parameter: no staging copy, nothing for the host to wait on.
struct PipeBatch {
    PipeReq r[MIGAN_PIPE_BATCH_MAX];
    int n, res;
    unsigned char* scratch;
    const int* boxes;
};

PL_D void box_of(const PipeBatch& b, int r, int& x0, int& y0, int& wc, int& hc) {
    const int* q = b.boxes + 4 * r;
    x0 = q[0]; wc = q[1] - q[0]; y0 = q[2]; hc = q[3] - q[2];
}
PL_D unsigned char* phase_of(const PipeBatch& b, int r) { return b.scratch + b.r[r].scratch + b.r[r].o_phase; }
inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }
PL_D AaTable table_at(unsigned char* p, int in_size, int out_size) {    // same carving as the single-request take_table
    AaTable t;
    t.maxk = aa_maxk(in_size, out_size);
    t.xmin = reinterpret_cast<int*>(p);
    t.xsize = t.xmin + out_size;
    t.w = reinterpret_cast<float*>(p + (((size_t)out_size * 2 * sizeof(int) + 255) & ~(size_t)255));
    return t;
}

// Each batched functor: worst(r) = items of request r for a crop as large as the image (host, sizes the grid),
// items(r) = its actual items (device, from the box), operator()(r, j) = item j of request r.
struct NearestBatchK {     // masks at another size -> image size
    PipeBatch b;
    int64_t worst(int r) const { const PipeReq& q = b.r[r]; return (q.mh != q.H || q.mw != q.W) ? (int64_t)q.H * q.W : 0; }
    PL_D int64_t items(int r) const { const PipeReq& q = b.r[r]; return (q.mh != q.H || q.mw != q.W) ? (int64_t)q.H * q.W : 0; }
    PL_D void operator()(int r, int64_t j) const { const PipeReq& q = b.r[r]; nearest_u8_item(q.mask_in, q.mh, q.mw, q.mask, q.H, q.W, j); }
};

struct PreTablesK {        // width table (wc -> res), then height table (hc -> res)
    PipeBatch b;
    int64_t worst(int) const { return 2 * (int64_t)b.res; }
    PL_D int64_t items(int) const { return 2 * (int64_t)b.res; }
    PL_D void operator()(int r, int64_t j) const {
        int x0, y0, wc, hc; box_of(b, r, x0, y0, wc, hc);
        unsigned char* p = phase_of(b, r);
        if (j < b.res) aa_weights_item(table_at(p, wc, b.res), wc, b.res, j);
        else aa_weights_item(table_at(p + b.r[r].o_th, hc, b.res), hc, b.res, j - b.res);
    }
};

struct PreWidthK {         // crop [3][hc][wc] -> [3][hc][res]
    PipeBatch b;
    int64_t worst(int r) const { return 3 * (int64_t)b.r[r].H * b.res; }
    PL_D int64_t items(int r) const { int x0, y0, wc, hc; box_of(b, r, x0, y0, wc, hc); return 3 * (int64_t)hc * b.res; }
    PL_D void operator()(int r, int64_t j) const {
        const PipeReq& q = b.r[r];
        int x0, y0, wc, hc; box_of(b, r, x0, y0, wc, hc);
        unsigned char* p = phase_of(b, r);
        resize_width_item<0>(q.image + (int64_t)y0 * q.W + x0, (int64_t)q.H * q.W, q.W, table_at(p, wc, b.res),
                             reinterpret_cast<float*>(p + q.o_tmp), hc, b.res, j);
    }
};

struct PreprocessBatchK {  // height pass + round + normalise -> row r of x[N,4,res,res]
    PipeBatch b; float* x;
    int64_t worst(int) const { return (int64_t)b.res * b.res; }
    PL_D int64_t items(int) const { return (int64_t)b.res * b.res; }
    PL_D void operator()(int r, int64_t j) const {
        const PipeReq& q = b.r[r];
        int x0, y0, wc, hc; box_of(b, r, x0, y0, wc, hc);
        unsigned char* p = phase_of(b, r);
        preprocess_item(reinterpret_cast<const float*>(p + q.o_tmp), table_at(p + q.o_th, hc, b.res), q.mask + (int64_t)y0 * q.W + x0,
                        q.W, hc, wc, b.res, x + (int64_t)r * 4 * b.res * b.res, j);
    }
};

struct PostTablesK {       // width table (res -> wc), then height table (res -> hc)
    PipeBatch b;
    int64_t worst(int r) const { return (int64_t)b.r[r].W + b.r[r].H; }
    PL_D int64_t items(int r) const { int x0, y0, wc, hc; box_of(b, r, x0, y0, wc, hc); return (int64_t)wc + hc; }
    PL_D void operator()(int r, int64_t j) const {
        int x0, y0, wc, hc; box_of(b, r, x0, y0, wc, hc);
        unsigned char* p = phase_of(b, r);
        if (j < wc) aa_weights_item(table_at(p, b.res, wc), b.res, wc, j);
        else aa_weights_item(table_at(p + b.r[r].o_th2, b.res, hc), b.res, hc, j - wc);
    }
};

struct PostWidthK {        // y[r] [3][res][res] -> [0,255] -> [3][res][wc]
    PipeBatch b; const float* y;
    int64_t worst(int r) const { return 3 * (int64_t)b.res * b.r[r].W; }
    PL_D int64_t items(int r) const { int x0, y0, wc, hc; box_of(b, r, x0, y0, wc, hc); return 3 * (int64_t)b.res * wc; }
    PL_D void operator()(int r, int64_t j) const {
        int x0, y0, wc, hc; box_of(b, r, x0, y0, wc, hc);
        unsigned char* p = phase_of(b, r);
        const int64_t plane = (int64_t)b.res * b.res;
        resize_width_item<1>(y + (int64_t)r * 3 * plane, plane, b.res, table_at(p, b.res, wc),
                             reinterpret_cast<float*>(p + b.r[r].o_tmp2), b.res, wc, j);
    }
};

struct ColG {              // height pass evaluated where the blend needs it: no [3][hc][wc] buffer
    const float* tmp; AaTable t; int res, wc;
    PL_D float operator()(int c, int h, int w, int64_t) const { return aa_col(tmp + (int64_t)c * res * wc, t, h, wc, w); }
};

struct PostBlendK {        // height pass fused into the feathered blend, written into image[crop]
    PipeBatch b; float k[25];
    int64_t worst(int r) const { return (int64_t)b.r[r].H * b.r[r].W; }
    PL_D int64_t items(int r) const { int x0, y0, wc, hc; box_of(b, r, x0, y0, wc, hc); return (int64_t)hc * wc; }
    PL_D void operator()(int r, int64_t j) const {
        const PipeReq& q = b.r[r];
        int x0, y0, wc, hc; box_of(b, r, x0, y0, wc, hc);
        unsigned char* p = phase_of(b, r);
        const ColG g{reinterpret_cast<const float*>(p + q.o_tmp2), table_at(p + q.o_th2, b.res, hc), b.res, wc};
        const int64_t o = (int64_t)y0 * q.W + x0;
        feather_item(g, q.image + o, q.mask + o, (int64_t)q.H * q.W, q.W, hc, wc, k, j);
    }
};

struct ExtentsInitK {      // items = n: no hole yet = (W, 0, H, 0), the flag scan's starting values
    PipeBatch b; int* ext;
    PL_D void operator()(int64_t r) const { int* e = ext + 4 * r; e[0] = b.r[r].W; e[1] = 0; e[2] = b.r[r].H; e[3] = 0; }
};

struct BoxFromExtentsK {   // items = n
    PipeBatch b; const int* ext; int* boxes; int padding;
    PL_D void operator()(int64_t r) const {
        const int* e = ext + 4 * r;
        crop_box_from_extents(e[0], e[1], e[2], e[3], b.r[r].H, b.r[r].W, b.res, padding, boxes + 4 * r);
    }
};

// ---- the batched launcher: one launch per stage for the whole batch -------------------------------------------------
constexpr int kBatchBlocksMax = 1024;      // blocks per request; larger crops loop (grid stride)
struct BatchGrid { int blk[MIGAN_PIPE_BATCH_MAX + 1]; };   // request r owns blocks [blk[r], blk[r+1])

#ifdef MIGAN_EMULATE
template <class F>
inline int pl_batch_launch(const F& f, int n, ck_stream_t) {
    for (int r = 0; r < n; ++r) {
        const int64_t items = f.items(r);
#pragma omp parallel for schedule(static)
        for (int64_t j = 0; j < items; ++j) f(r, j);
    }
    return 0;
}
#else
__device__ __forceinline__ int request_of(const BatchGrid& g, int n, int block) {   // last r with blk[r] <= block
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (g.blk[mid] <= block) lo = mid; else hi = mid - 1;
    }
    return lo;
}
template <class F>
__global__ void __launch_bounds__(256) pl_batch_kernel(const F f, const BatchGrid g, const int n) {
    const int r = request_of(g, n, blockIdx.x);
    const int64_t items = f.items(r);
    const int64_t step = (int64_t)(g.blk[r + 1] - g.blk[r]) * 256;
    for (int64_t j = (int64_t)(blockIdx.x - g.blk[r]) * 256 + threadIdx.x; j < items; j += step) f(r, j);
}
template <class F>
inline cudaError_t pl_batch_launch(const F& f, int n, ck_stream_t s) {
    BatchGrid g;
    g.blk[0] = 0;
    for (int r = 0; r < n; ++r) {
        int64_t blocks = (f.worst(r) + 255) / 256;
        blocks = blocks > kBatchBlocksMax ? kBatchBlocksMax : blocks;
        g.blk[r + 1] = g.blk[r] + (int)blocks;
    }
    if (g.blk[n] == 0) return cudaSuccess;
    pl_batch_kernel<F><<<g.blk[n], 256, 0, s>>>(f, g, n);
    return cudaGetLastError();
}

// Extents of the hole pixels (value < 255) of every request's mask, one pass over the bytes: 16-byte loads, per-thread
// min / max, warp shuffles, one set of four atomics per block that saw a hole.  Uses warp collectives: GPU only (the
// emulation build reduces on the host and shares only the arithmetic after the reduction).
constexpr int kExtentBlocksMax = 512;
__device__ __forceinline__ void note_hole(int64_t p, int W, int& x_min, int& x_max, int& y_min, int& y_max) {
    const int y = (int)(p / W), x = (int)(p - (int64_t)y * W);
    x_min = min(x_min, x); x_max = max(x_max, x); y_min = min(y_min, y); y_max = max(y_max, y);
}
__global__ void __launch_bounds__(256) hole_extents_kernel(const PipeBatch b, const BatchGrid g, int* ext) {
    const int r = request_of(g, b.n, blockIdx.x);
    const PipeReq& q = b.r[r];
    const int W = q.W, H = q.H;
    const int64_t bytes = (int64_t)H * W;
    const uint8_t* m = q.mask;
    int x_min = W, x_max = 0, y_min = H, y_max = 0;
    const int head = (int)min((int64_t)((16 - ((uintptr_t)m & 15)) & 15), bytes);
    const int64_t nvec = (bytes - head) >> 4;
    const uint4* v = reinterpret_cast<const uint4*>(m + head);
    const int64_t step = (int64_t)(g.blk[r + 1] - g.blk[r]) * 256;
    for (int64_t k = (int64_t)(blockIdx.x - g.blk[r]) * 256 + threadIdx.x; k < nvec; k += step) {
        const uint4 u = __ldg(v + k);
        if ((u.x & u.y & u.z & u.w) == 0xffffffffu) continue;            // 16 known pixels
        const uint32_t w4[4] = {u.x, u.y, u.z, u.w};
        const int64_t p0 = head + k * 16;
        int y = (int)(p0 / W), x = (int)(p0 - (int64_t)y * W);
#pragma unroll
        for (int e = 0; e < 16; ++e) {
            if (((w4[e >> 2] >> ((e & 3) * 8)) & 0xff) != 0xff) {
                x_min = min(x_min, x); x_max = max(x_max, x); y_min = min(y_min, y); y_max = max(y_max, y);
            }
            if (++x == W) { x = 0; ++y; }
        }
    }
    if (blockIdx.x == g.blk[r]) {                                        // unaligned head and tail bytes
        const int64_t tail0 = head + nvec * 16;
        for (int64_t p = threadIdx.x; p < head + (bytes - tail0); p += 256) {
            const int64_t o = p < head ? p : tail0 + (p - head);
            if (m[o] != 255) note_hole(o, W, x_min, x_max, y_min, y_max);
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        x_min = min(x_min, __shfl_xor_sync(0xffffffffu, x_min, d)); x_max = max(x_max, __shfl_xor_sync(0xffffffffu, x_max, d));
        y_min = min(y_min, __shfl_xor_sync(0xffffffffu, y_min, d)); y_max = max(y_max, __shfl_xor_sync(0xffffffffu, y_max, d));
    }
    __shared__ int part[8][4];
    const int warp = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) { part[warp][0] = x_min; part[warp][1] = x_max; part[warp][2] = y_min; part[warp][3] = y_max; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < 8; ++i) {
            x_min = min(x_min, part[i][0]); x_max = max(x_max, part[i][1]); y_min = min(y_min, part[i][2]); y_max = max(y_max, part[i][3]);
        }
        if (y_min < H) {                                                 // this block saw a hole
            int* e = ext + 4 * r;
            atomicMin(e + 0, x_min); atomicMax(e + 1, x_max); atomicMin(e + 2, y_min); atomicMax(e + 3, y_max);
        }
    }
}
#endif

}  // namespace comod

namespace migan {

namespace {

using comod::aa_maxk;
using comod::align256;
inline size_t table_bytes(int in_size, int out_size) {
    return align256((size_t)out_size * 2 * sizeof(int)) + align256((size_t)out_size * aa_maxk(in_size, out_size) * sizeof(float));
}
// carve one axis table out of the scratch area
inline comod::AaTable take_table(unsigned char*& p, int in_size, int out_size) {
    comod::AaTable t;
    t.maxk = aa_maxk(in_size, out_size);
    t.xmin = reinterpret_cast<int*>(p);
    t.xsize = t.xmin + out_size;
    p += align256((size_t)out_size * 2 * sizeof(int));
    t.w = reinterpret_cast<float*>(p);
    p += align256((size_t)out_size * t.maxk * sizeof(float));
    return t;
}

}  // namespace

size_t pipeline_scratch_bytes(int H, int W, int res) {
    // the crop is at most the whole image: pre = tables (H -> res, W -> res) + [3][H][res]; post = tables (res -> H, res -> W)
    // + [3][res][W] + [3][H][W]; the two phases reuse the same area
    const size_t pre = table_bytes(H, res) + table_bytes(W, res) + align256((size_t)3 * H * res * sizeof(float));
    const size_t post = table_bytes(res, H) + table_bytes(res, W) + align256((size_t)3 * res * W * sizeof(float)) +
                        align256((size_t)3 * H * W * sizeof(float));
    return (pre > post ? pre : post) + 1024;
}

int launch_resize_nearest_u8(const uint8_t* in, int H, int W, uint8_t* out, int oh, int ow, ck_stream_t s) {
    comod::NearestU8K k{in, out, H, W, oh, ow};
    return (int)comod::ck_launch(k, (int64_t)oh * ow, s);
}

int launch_hole_flags(const uint8_t* mask, int H, int W, uint8_t* flags, ck_stream_t s) {
    comod::HoleFlagsK k{mask, flags, H, W};
    return (int)comod::ck_launch(k, (int64_t)W + H, s);
}

// Host arithmetic of get_masked_bbox (:151-227) on the hole flags (flags[x] for columns, flags[W + y] for rows).
void crop_box_from_flags(const uint8_t* flags, int H, int W, int res, int padding, int* box) {
    int x_min = W, x_max = 0, y_min = H, y_max = 0;
    for (int x = 0; x < W; ++x) if (flags[x]) { x_min = comod::pl_imin(x_min, x); x_max = comod::pl_imax(x_max, x); }
    for (int y = 0; y < H; ++y) if (flags[W + y]) { y_min = comod::pl_imin(y_min, y); y_max = comod::pl_imax(y_max, y); }
    comod::crop_box_from_extents(x_min, x_max, y_min, y_max, H, W, res, padding, box);
}

int launch_pipeline_preprocess(const uint8_t* image, const uint8_t* mask, int H, int W, const int* box, int res, float* x,
                               void* scratch, ck_stream_t s) {
    const int x0 = box[0], x1 = box[1], y0 = box[2], y1 = box[3];
    const int wc = x1 - x0, hc = y1 - y0;
    unsigned char* p = static_cast<unsigned char*>(scratch);
    comod::AaTable tw = take_table(p, wc, res), th = take_table(p, hc, res);
    float* tmp = reinterpret_cast<float*>(p);                                   // [3][hc][res]
    int e;
    if ((e = (int)comod::ck_launch(comod::AaWeightsK{tw, wc, res}, res, s))) return e;
    if ((e = (int)comod::ck_launch(comod::AaWeightsK{th, hc, res}, res, s))) return e;
    comod::ResizeWidthK<0> kw{image + (int64_t)y0 * W + x0, (int64_t)H * W, W, tw, tmp, hc, res};
    if ((e = (int)comod::ck_launch(kw, (int64_t)3 * hc * res, s))) return e;
    comod::PreprocessK kp{tmp, th, mask + (int64_t)y0 * W + x0, W, hc, wc, res, x};
    return (int)comod::ck_launch(kp, (int64_t)res * res, s);
}

int launch_pipeline_postprocess(const float* y, uint8_t* image, const uint8_t* mask, int H, int W, const int* box, int res,
                                const float* k25_host, void* scratch, ck_stream_t s) {
    const int x0 = box[0], x1 = box[1], y0 = box[2], y1 = box[3];
    const int wc = x1 - x0, hc = y1 - y0;
    unsigned char* p = static_cast<unsigned char*>(scratch);
    comod::AaTable tw = take_table(p, res, wc), th = take_table(p, res, hc);
    float* tmp = reinterpret_cast<float*>(p);                                   // [3][res][wc]
    p += align256((size_t)3 * res * wc * sizeof(float));
    float* g = reinterpret_cast<float*>(p);                                     // [3][hc][wc]
    int e;
    if ((e = (int)comod::ck_launch(comod::AaWeightsK{tw, res, wc}, wc, s))) return e;
    if ((e = (int)comod::ck_launch(comod::AaWeightsK{th, res, hc}, hc, s))) return e;
    comod::ResizeWidthK<1> kw{y, (int64_t)res * res, res, tw, tmp, res, wc};
    if ((e = (int)comod::ck_launch(kw, (int64_t)3 * res * wc, s))) return e;
    comod::ResizeHeightK kh{tmp, th, g, res, hc, wc};
    if ((e = (int)comod::ck_launch(kh, (int64_t)3 * hc * wc, s))) return e;
    comod::FeatherCropK kf{g, image + (int64_t)y0 * W + x0, mask + (int64_t)y0 * W + x0, (int64_t)H * W, W, hc, wc, {0}};
    for (int i = 0; i < 25; ++i) kf.k[i] = k25_host[i];
    return (int)comod::ck_launch(kf, (int64_t)hc * wc, s);
}

// ---- batched crop pipeline ------------------------------------------------------------------------------------------
// Scratch layout: the [n][4] extents, then one region per request (comod::PipeReq).  Every bound is the crop's worst case:
// wc lies in [min(res, W), W] (get_masked_bbox widens a clipped window back to min(crop, W), crop >= res), and the taps
// per output grow with the in / out ratio, with 3 for any up-sampling.  Returns the total bytes; fills `b` when given.
size_t batch_layout(const migan_pipe_req* reqs, int n, int res, void* scratch, comod::PipeBatch* b) {
    size_t off = align256((size_t)n * 4 * sizeof(int));
    for (int r = 0; r < n; ++r) {
        const int H = reqs[r].H, W = reqs[r].W;
        const bool resized = reqs[r].mask_h != H || reqs[r].mask_w != W;
        auto table = [](int out, int maxk) { return align256((size_t)out * 2 * sizeof(int)) + align256((size_t)out * maxk * sizeof(float)); };
        const int kpw = comod::pl_imax(3, aa_maxk(W, res)), kph = comod::pl_imax(3, aa_maxk(H, res));
        const int kqw = comod::pl_imax(3, aa_maxk(res, comod::pl_imin(res, W))), kqh = comod::pl_imax(3, aa_maxk(res, comod::pl_imin(res, H)));
        comod::PipeReq q;
        q.image = reqs[r].image_chw; q.mask_in = reqs[r].mask_hw;
        q.H = H; q.W = W; q.mh = reqs[r].mask_h; q.mw = reqs[r].mask_w;
        q.scratch = (int64_t)off;
        q.o_phase = resized ? (int64_t)align256((size_t)H * W) : 0;
        q.mask = resized ? static_cast<uint8_t*>(scratch) + off : const_cast<uint8_t*>(reqs[r].mask_hw);
        q.o_th = (int)table(res, kpw);
        q.o_tmp = q.o_th + (int)table(res, kph);
        const size_t pre = (size_t)q.o_tmp + align256((size_t)3 * H * res * sizeof(float));
        q.o_th2 = (int)table(W, kqw);
        q.o_tmp2 = q.o_th2 + (int)table(H, kqh);
        const size_t post = (size_t)q.o_tmp2 + align256((size_t)3 * res * W * sizeof(float));
        off += (size_t)q.o_phase + (pre > post ? pre : post);
        if (b) b->r[r] = q;
    }
    if (b) { b->n = n; b->res = res; b->scratch = static_cast<unsigned char*>(scratch); b->boxes = nullptr; }
    return off;
}

size_t pipeline_batch_scratch_bytes(const migan_pipe_req* reqs, int n, int res) { return batch_layout(reqs, n, res, nullptr, nullptr); }

int launch_pipeline_batch_boxes(const migan_pipe_req* reqs, int n, int res, int padding, int* boxes, void* scratch, ck_stream_t s) {
    comod::PipeBatch b;
    batch_layout(reqs, n, res, scratch, &b);
    int* ext = static_cast<int*>(scratch);
    int e;
    if ((e = (int)comod::pl_batch_launch(comod::NearestBatchK{b}, n, s))) return e;
    if ((e = (int)comod::ck_launch(comod::ExtentsInitK{b, ext}, n, s))) return e;
#ifdef MIGAN_EMULATE
    for (int r = 0; r < n; ++r) {                        // the reduction on the host; the box arithmetic below is shared
        const comod::PipeReq& q = b.r[r];
        int* x = ext + 4 * r;
        for (int y = 0; y < q.H; ++y)
            for (int xx = 0; xx < q.W; ++xx)
                if (q.mask[(int64_t)y * q.W + xx] < 255) {
                    x[0] = comod::pl_imin(x[0], xx); x[1] = comod::pl_imax(x[1], xx);
                    x[2] = comod::pl_imin(x[2], y); x[3] = comod::pl_imax(x[3], y);
                }
    }
#else
    {
        comod::BatchGrid g;
        g.blk[0] = 0;
        for (int r = 0; r < n; ++r) {
            int64_t blocks = ((int64_t)reqs[r].H * reqs[r].W / 16 + 255) / 256;
            blocks = blocks < 1 ? 1 : (blocks > comod::kExtentBlocksMax ? comod::kExtentBlocksMax : blocks);
            g.blk[r + 1] = g.blk[r] + (int)blocks;
        }
        comod::hole_extents_kernel<<<g.blk[n], 256, 0, s>>>(b, g, ext);
        if ((e = (int)cudaGetLastError())) return e;
    }
#endif
    return (int)comod::ck_launch(comod::BoxFromExtentsK{b, ext, boxes, padding}, n, s);
}

int launch_pipeline_batch_preprocess(const migan_pipe_req* reqs, int n, int res, const int* boxes, float* x, void* scratch,
                                     ck_stream_t s) {
    comod::PipeBatch b;
    batch_layout(reqs, n, res, scratch, &b);
    b.boxes = boxes;
    int e;
    if ((e = (int)comod::pl_batch_launch(comod::PreTablesK{b}, n, s))) return e;
    if ((e = (int)comod::pl_batch_launch(comod::PreWidthK{b}, n, s))) return e;
    return (int)comod::pl_batch_launch(comod::PreprocessBatchK{b, x}, n, s);
}

int launch_pipeline_batch_postprocess(const float* y, const migan_pipe_req* reqs, int n, int res, const int* boxes,
                                      const float* k25_host, void* scratch, ck_stream_t s) {
    comod::PipeBatch b;
    batch_layout(reqs, n, res, scratch, &b);
    b.boxes = boxes;
    int e;
    if ((e = (int)comod::pl_batch_launch(comod::PostTablesK{b}, n, s))) return e;
    if ((e = (int)comod::pl_batch_launch(comod::PostWidthK{b, y}, n, s))) return e;
    comod::PostBlendK kb{b, {0}};
    for (int i = 0; i < 25; ++i) kb.k[i] = k25_host[i];
    return (int)comod::pl_batch_launch(kb, n, s);
}

}  // namespace migan

#ifdef MIGAN_EMULATE   // the product's extern "C" wrappers (argument checks, error strings) live in migan_abi.cu
namespace migan {
size_t pipeline_scratch_bytes(int H, int W, int res);
}
extern "C" size_t b200_pipeline_scratch_bytes(int H, int W, int res) { return migan::pipeline_scratch_bytes(H, W, res); }
extern "C" int b200_resize_nearest_u8(const uint8_t* in, int H, int W, uint8_t* out, int oh, int ow, void* s) {
    return migan::launch_resize_nearest_u8(in, H, W, out, oh, ow, s);
}
extern "C" int b200_hole_flags(const uint8_t* mask, int H, int W, uint8_t* flags, void* s) { return migan::launch_hole_flags(mask, H, W, flags, s); }
extern "C" int migan_crop_box(const uint8_t* flags, int H, int W, int res, int padding, int* box) {
    migan::crop_box_from_flags(flags, H, W, res, padding, box);
    return 0;
}
extern "C" int b200_pipeline_preprocess(const uint8_t* image, const uint8_t* mask, int H, int W, const int* box, int res, float* x,
                                        void* scratch, size_t, void* s) {
    return migan::launch_pipeline_preprocess(image, mask, H, W, box, res, x, scratch, s);
}
extern "C" int b200_pipeline_postprocess(const float* y, uint8_t* image, const uint8_t* mask, int H, int W, const int* box, int res,
                                         const float* k25, void* scratch, size_t, void* s) {
    return migan::launch_pipeline_postprocess(y, image, mask, H, W, box, res, k25, scratch, s);
}
extern "C" size_t b200_pipeline_batch_scratch_bytes(const migan_pipe_req* reqs, int n, int res) {
    return migan::pipeline_batch_scratch_bytes(reqs, n, res);
}
extern "C" int b200_pipeline_batch_boxes(const migan_pipe_req* reqs, int n, int res, int padding, int* boxes, void* scratch, size_t, void* s) {
    return migan::launch_pipeline_batch_boxes(reqs, n, res, padding, boxes, scratch, s);
}
extern "C" int b200_pipeline_batch_preprocess(const migan_pipe_req* reqs, int n, int res, const int* boxes, float* x, void* scratch, size_t,
                                              void* s) {
    return migan::launch_pipeline_batch_preprocess(reqs, n, res, boxes, x, scratch, s);
}
extern "C" int b200_pipeline_batch_postprocess(const float* y, const migan_pipe_req* reqs, int n, int res, const int* boxes, const float* k25,
                                               void* scratch, size_t, void* s) {
    return migan::launch_pipeline_batch_postprocess(y, reqs, n, res, boxes, k25, scratch, s);
}
#endif
