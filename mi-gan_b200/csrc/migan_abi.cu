// C ABI + host runtime of the B200-native MI-GAN generator (include/migan_b200.h).
//
// Host side of the hot path: weight registry in the reference's state_dict layout, one-time
// repacking for the kernels, a per-batch-size execution plan (a flat list of kernel launches
// with every pointer / tensor map resolved) and the launcher.  Replaces the module tree of
// lib/model_zoo/migan_inference.py:173-369 (EncoderBlock / Encoder / SynthesisBlock* /
// Synthesis / Generator): the control flow of those forward() methods is the plan below.
#include <cuda_runtime.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <array>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../../include/migan_b200.h"
#include "kernels.h"
#include "sepconv_tc.h"

namespace {

thread_local std::string g_last_error;

int fail(int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

#define CUDA_TRY(expr)                                                                        \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess)                                                                \
            return fail(MIGAN_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

inline int channels(int res) { return std::min(32768 / res, 512); }  // migan_inference.py:222-223
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct WeightSpec {
    std::string name;
    int ndim;
    int64_t shape[4];
    int64_t numel() const {
        int64_t n = 1;
        for (int i = 0; i < ndim; ++i) n *= shape[i];
        return n;
    }
};

// One SeparableConv2d (migan_inference.py:106-170), packed for the kernels.
struct SepConv {
    std::string p;  // state_dict prefix, e.g. "encoder.b256.conv2."
    int cin = 0, cout = 0;
    int res_in = 0;   // spatial size the depthwise conv runs at
    int res_pw = 0;   // spatial size the 1x1 conv runs at (res_in / 2 if down)
    int res_out = 0;  // output spatial size (2 * res_pw if up)
    bool down = false, up = false, noise = false;
    // device pointers into the weight arena
    float* w9 = nullptr;      // [9][cin]   depthwise taps, tap-major
    float* bias = nullptr;    // [cin]
    float* w9_tc = nullptr;   // same, pre-multiplied by kActSplitScale * sqrt(2) for the tcgen05 prologue
    float* bias_tc = nullptr;
    float* pw_t = nullptr;    // [cin][cout] fp32 (CUDA-core GEMM)
    __half* pw_hi = nullptr;  // [cout][cin] fp16 hi part of w * 2^k   (tcgen05, K-major)
    __half* pw_lo = nullptr;  // [cout][cin] fp16 lo part
    float tc_inv_scale = 1.f; // 1 / (kActSplitScale * 2^k)
    float* fir16 = nullptr;   // [16][cin] (down) or [16][cout] (up), tap-major
    float* noise_dev = nullptr;  // [res_out^2] = noise_const * noise_strength
    // fused up-sampling prologue of the NEXT layer (sepconv_tc SEPCONV_SRC_UP): needs channel-uniform FIR taps
    bool up_uniform = false;
    float up_taps_s2[16] = {0};      // taps * sqrt(2)
    float* noise_s2_dev = nullptr;   // noise * sqrt(2)
};

struct ToRgb {
    std::string p;  // "synthesis.b64."
    int c = 0, res = 0;
    bool has_up = false;
    float* w = nullptr;    // [3][c]
    float* b = nullptr;    // [3]
    float* fir = nullptr;  // [16][3]
};

enum StepKind { K_STEM, K_DW, K_DWDOWN, K_GEMM_SIMT, K_SEPCONV_TC, K_UP2, K_TORGB, K_ADD };

constexpr int PTR_X = 1, PTR_Y = 2;  // flags: operand is the caller's x / y

struct Step {
    StepKind kind;
    const SepConv* L = nullptr;
    const ToRgb* T = nullptr;
    const float* in = nullptr;
    const float* aux = nullptr;  // skip tensor / low-res image / noise
    const float* aux2 = nullptr; // fused up-sampling prologue: the low-resolution raw tensor
    bool fused_stem = false, fused_up = false;
    float* out = nullptr;
    __half* hi = nullptr;
    __half* lo = nullptr;
    int io_flags = 0;
    int n = 0, H = 0, W = 0, C = 0;  // meaning depends on kind (input dims)
    int act = 0;
    bool want_f32 = false;
    migan::SepconvTcArgs tc;  // resolved tcgen05 launch (tensor maps, tiling)
    migan::DownTensorMap down_map;   // K_DWDOWN on the TMA-staged kernel: tensor map of the input
    bool down_tma = false;
    // roofline bookkeeping: algorithmic bytes = own input(s) read once + output written once
    std::string label;
    double alg_bytes = 0, flops = 0;
    // tap (debug): tensor produced by this step
    std::string tap;
    const float* tap_src = nullptr;
    int tapC = 0, tapH = 0, tapW = 0;
    bool tap_planar = false;
    int tap_flags = 0;
    // second tap (fused torgb: the image produced by the same launch)
    std::string tap2;
    const float* tap2_src = nullptr;
    int tap2C = 0, tap2H = 0, tap2W = 0, tap2_flags = 0;
};

struct Plan {
    int n = 0, path = -1;
    void* ws = nullptr;
    std::vector<Step> steps;
};

}  // namespace

struct migan_ctx {
    int resolution = 0, device = 0;
    std::vector<WeightSpec> specs;
    std::map<std::string, int> spec_index;
    std::vector<std::vector<float>> host;  // host copies, by spec index
    std::vector<bool> provided;
    bool finalized = false;

    std::vector<int> enc_res;  // R .. 4
    std::vector<int> syn_res;  // 4 .. R
    // encoder
    float* fromrgb_w = nullptr;  // [C0][4]
    float* fromrgb_b = nullptr;
    float* fromrgb_w_s2 = nullptr;  // * sqrt(2): stem recomputed in the prologue of encoder.b{R}.conv1
    float* fromrgb_b_s2 = nullptr;
    std::vector<SepConv> enc1, enc2;  // per enc_res entry
    // synthesis
    std::vector<SepConv> syn1, syn2;  // per syn_res entry
    std::vector<ToRgb> torgb;
    void* arena = nullptr;

    Plan plan;
    int last_launches = 0;
    std::string tap_name;
    float* tap_dst = nullptr;
    bool profiling = false;
    std::vector<cudaEvent_t> events;  // 2 per step of the current plan
    // host-buffer pipeline (migan_forward_host): copy streams + events, created on first use
    cudaStream_t s_in = nullptr, s_out = nullptr;
    std::vector<cudaEvent_t> host_events;
    cudaEvent_t slot_compute_done[2] = {nullptr, nullptr}, slot_out_done[2] = {nullptr, nullptr};
    bool slot_used[2] = {false, false};
    const void* slot_base[2] = {nullptr, nullptr};   // staging memory each slot last used (re-ordered after the caller's stream when it changes)
    unsigned host_calls = 0;
    // uint8 request pipeline (migan_forward_u8 / _async): its own two staging slots and events
    cudaEvent_t u8_in[2] = {nullptr, nullptr}, u8_compute_done[2] = {nullptr, nullptr}, u8_out_done[2] = {nullptr, nullptr}, u8_start = nullptr;
    bool u8_used[2] = {false, false};
    const void* u8_base[2] = {nullptr, nullptr};
    unsigned u8_calls = 0;
    // captured forward (migan_forward_graph): valid for one (n, path, workspace)
    cudaGraphExec_t graph_exec = nullptr;
    cudaStream_t s_cap = nullptr;
    int graph_n = 0, graph_path = -1, graph_launches = 0;
    void* graph_ws = nullptr;
    int tap_cache_path = -1;          // tap enumeration cache (migan_tap_info)
    std::vector<std::pair<std::string, std::array<int, 3>>> tap_cache;
};

namespace {

void add_spec(migan_ctx* c, const std::string& name, std::initializer_list<int64_t> shape) {
    WeightSpec s;
    s.name = name;
    s.ndim = (int)shape.size();
    int i = 0;
    for (int64_t d : shape) s.shape[i++] = d;
    for (; i < 4; ++i) s.shape[i] = 1;
    c->spec_index[name] = (int)c->specs.size();
    c->specs.push_back(s);
}

// Key order = the reference state_dict (own params, own buffers, then children; SURVEY.md 8b).
void add_sepconv_specs(migan_ctx* c, const SepConv& L) {
    if (L.noise) {
        add_spec(c, L.p + "noise_strength", {});
        add_spec(c, L.p + "noise_const", {L.res_out, L.res_out});
    }
    add_spec(c, L.p + "conv1.weight", {L.cin, 1, 3, 3});
    add_spec(c, L.p + "conv1.bias", {L.cin});
    add_spec(c, L.p + "conv2.weight", {L.cout, L.cin, 1, 1});
    if (L.down) add_spec(c, L.p + "downsample.filter.weight", {L.cin, 1, 4, 4});
    if (L.up) {
        add_spec(c, L.p + "upsample.filter_const", {1, 1, L.res_out, L.res_out});
        add_spec(c, L.p + "upsample.filter.weight", {L.cout, 1, 4, 4});
    }
}

SepConv make_sepconv(const std::string& p, int cin, int cout, int res_in, bool down, bool up, bool noise) {
    SepConv L;
    L.p = p; L.cin = cin; L.cout = cout; L.res_in = res_in;
    L.down = down; L.up = up; L.noise = noise;
    L.res_pw = down ? res_in / 2 : res_in;
    L.res_out = up ? L.res_pw * 2 : L.res_pw;
    return L;
}

const std::vector<float>& W(const migan_ctx* c, const std::string& name) {
    return c->host[c->spec_index.at(name)];
}

// Bump allocator over a host staging image of the device weight arena.
struct ArenaBuilder {
    std::vector<unsigned char> bytes;
    size_t alloc(size_t n) {
        size_t off = align_up(bytes.size(), 256);
        bytes.resize(off + n, 0);
        return off;
    }
};

}  // namespace

extern "C" {

const char* migan_last_error(void) { return g_last_error.c_str(); }
const char* migan_version(void) { return "migan_b200 0.1 (sm_100a)"; }

int migan_create(int resolution, int device, migan_ctx** out) {
    if (!out) return fail(MIGAN_ERR_INVALID, "out is null");
    *out = nullptr;
    int log2res = 0;
    while ((1 << (log2res + 1)) <= resolution) ++log2res;
    if (resolution < 8 || (1 << log2res) != resolution || resolution > 4096)
        return fail(MIGAN_ERR_INVALID, "resolution must be a power of two in [8, 4096], got %d", resolution);
    if (device >= 0 && channels(resolution) < 64)
        return fail(MIGAN_ERR_INVALID, "resolution %d has %d-channel levels; the kernels are built for >= 64 channels per level "
                    "(resolutions up to 512, i.e. every released MI-GAN model)", resolution, channels(resolution));
    std::unique_ptr<migan_ctx> c(new migan_ctx);
    c->resolution = resolution;
    c->device = device;
    for (int i = log2res; i >= 2; --i) c->enc_res.push_back(1 << i);
    for (int i = 2; i <= log2res; ++i) c->syn_res.push_back(1 << i);

    // synthesis first, then encoder (ctor order migan_inference.py:359-360)
    const int c4 = channels(4);
    c->syn1.push_back(make_sepconv("synthesis.b4.conv1.", c4, c4, 4, false, false, false));
    c->syn2.push_back(make_sepconv("synthesis.b4.conv2.", c4, c4, 4, false, false, false));
    for (size_t i = 1; i < c->syn_res.size(); ++i) {
        const int rj = c->syn_res[i], ri = c->syn_res[i - 1];
        const std::string p = "synthesis.b" + std::to_string(rj) + ".";
        c->syn1.push_back(make_sepconv(p + "conv1.", channels(ri), channels(rj), ri, false, true, true));
        c->syn2.push_back(make_sepconv(p + "conv2.", channels(rj), channels(rj), rj, false, false, true));
    }
    for (size_t i = 0; i < c->syn_res.size(); ++i) {
        const int r = c->syn_res[i];
        const std::string p = "synthesis.b" + std::to_string(r) + ".";
        add_sepconv_specs(c.get(), c->syn1[i]);
        add_sepconv_specs(c.get(), c->syn2[i]);
        add_spec(c.get(), p + "torgb.weight", {3, channels(r), 1, 1});
        add_spec(c.get(), p + "torgb.bias", {3});
        ToRgb t;
        t.p = p; t.c = channels(r); t.res = r; t.has_up = (i > 0);
        if (t.has_up) {
            add_spec(c.get(), p + "upsample.filter_const", {1, 1, r, r});
            add_spec(c.get(), p + "upsample.filter.weight", {3, 1, 4, 4});
        }
        c->torgb.push_back(t);
    }
    for (size_t i = 0; i < c->enc_res.size(); ++i) {
        const int r = c->enc_res[i];
        const std::string p = "encoder.b" + std::to_string(r) + ".";
        const bool last = (i + 1 == c->enc_res.size());
        const int ci = channels(r), cj = last ? ci : channels(c->enc_res[i + 1]);
        if (i == 0) {
            add_spec(c.get(), p + "fromrgb.weight", {ci, 4, 1, 1});
            add_spec(c.get(), p + "fromrgb.bias", {ci});
        }
        c->enc1.push_back(make_sepconv(p + "conv1.", ci, ci, r, false, false, false));
        c->enc2.push_back(make_sepconv(p + "conv2.", ci, cj, r, !last, false, false));
        add_sepconv_specs(c.get(), c->enc1.back());
        add_sepconv_specs(c.get(), c->enc2.back());
    }
    c->host.resize(c->specs.size());
    c->provided.assign(c->specs.size(), false);

    if (device >= 0) {
        int ndev = 0;
        cudaError_t e = cudaGetDeviceCount(&ndev);
        if (e != cudaSuccess || device >= ndev) {
            (void)cudaGetLastError();
            return fail(MIGAN_ERR_CUDA, "CUDA device %d not available (%s; %d devices): this library has no CPU path",
                        device, cudaGetErrorString(e), ndev);
        }
        CUDA_TRY(cudaSetDevice(device));
        cudaDeviceProp prop;
        CUDA_TRY(cudaGetDeviceProperties(&prop, device));
        if (prop.major != 10)
            return fail(MIGAN_ERR_CUDA, "device %d is sm_%d%d; this build targets sm_100a (B200) only", device, prop.major, prop.minor);
        CUDA_TRY(migan::configure_elementwise());
        CUDA_TRY(migan::configure_sepconv_tc());
    }  // device < 0: description-only context (weight registry / workspace sizes), cannot compute
    *out = c.release();
    return MIGAN_OK;
}

int migan_destroy(migan_ctx* ctx) {
    if (!ctx) return MIGAN_OK;
    for (cudaEvent_t e : ctx->events) cudaEventDestroy(e);
    for (cudaEvent_t e : ctx->host_events) cudaEventDestroy(e);
    for (int i = 0; i < 2; ++i) {
        if (ctx->slot_compute_done[i]) cudaEventDestroy(ctx->slot_compute_done[i]);
        if (ctx->slot_out_done[i]) cudaEventDestroy(ctx->slot_out_done[i]);
    }
    for (int i = 0; i < 2; ++i) {
        if (ctx->u8_in[i]) cudaEventDestroy(ctx->u8_in[i]);
        if (ctx->u8_compute_done[i]) cudaEventDestroy(ctx->u8_compute_done[i]);
        if (ctx->u8_out_done[i]) cudaEventDestroy(ctx->u8_out_done[i]);
    }
    if (ctx->u8_start) cudaEventDestroy(ctx->u8_start);
    if (ctx->graph_exec) cudaGraphExecDestroy(ctx->graph_exec);
    if (ctx->s_cap) cudaStreamDestroy(ctx->s_cap);
    if (ctx->s_in) cudaStreamDestroy(ctx->s_in);
    if (ctx->s_out) cudaStreamDestroy(ctx->s_out);
    if (ctx->arena && ctx->device >= 0) {
        cudaSetDevice(ctx->device);
        cudaFree(ctx->arena);
    }
    delete ctx;
    return MIGAN_OK;
}

int migan_num_weights(const migan_ctx* ctx) { return ctx ? (int)ctx->specs.size() : 0; }

int migan_weight_info(const migan_ctx* ctx, int index, const char** name, int* ndim, int64_t shape[4]) {
    if (!ctx || index < 0 || index >= (int)ctx->specs.size()) return fail(MIGAN_ERR_INVALID, "bad weight index %d", index);
    const WeightSpec& s = ctx->specs[index];
    if (name) *name = s.name.c_str();
    if (ndim) *ndim = s.ndim;
    if (shape)
        for (int i = 0; i < 4; ++i) shape[i] = s.shape[i];
    return MIGAN_OK;
}

int migan_set_weight(migan_ctx* ctx, const char* name, const float* host_data, int64_t numel) {
    if (!ctx || !name || !host_data) return fail(MIGAN_ERR_INVALID, "null argument");
    auto it = ctx->spec_index.find(name);
    if (it == ctx->spec_index.end()) return fail(MIGAN_ERR_INVALID, "unexpected key '%s' for resolution %d", name, ctx->resolution);
    const WeightSpec& s = ctx->specs[it->second];
    if (s.numel() != numel)
        return fail(MIGAN_ERR_INVALID, "size mismatch for '%s': expected %lld elements, got %lld", name, (long long)s.numel(), (long long)numel);
    ctx->host[it->second].assign(host_data, host_data + numel);
    ctx->provided[it->second] = true;
    ctx->finalized = false;
    return MIGAN_OK;
}

static int pack_sepconv(migan_ctx* ctx, SepConv& L, ArenaBuilder& ab, std::vector<std::pair<void**, size_t>>& fix) {
    const int cin = L.cin, cout = L.cout;
    {   // depthwise taps [cin,1,3,3] -> [9][cin]
        const std::vector<float>& w = W(ctx, L.p + "conv1.weight");
        size_t off = ab.alloc(sizeof(float) * 9 * cin);
        float* d = reinterpret_cast<float*>(ab.bytes.data() + off);
        for (int c = 0; c < cin; ++c)
            for (int t = 0; t < 9; ++t) d[t * cin + c] = w[c * 9 + t];
        fix.push_back({reinterpret_cast<void**>(&L.w9), off});
    }
    {
        const std::vector<float>& b = W(ctx, L.p + "conv1.bias");
        size_t off = ab.alloc(sizeof(float) * cin);
        memcpy(ab.bytes.data() + off, b.data(), sizeof(float) * cin);
        fix.push_back({reinterpret_cast<void**>(&L.bias), off});
    }
    {   // tcgen05 prologue: activation gain and fp16-split scale folded into the depthwise taps
        const float S = 64.0f /* kActSplitScale */ * 1.41421356237309515f;
        const std::vector<float>& w = W(ctx, L.p + "conv1.weight");
        const std::vector<float>& b = W(ctx, L.p + "conv1.bias");
        size_t off = ab.alloc(sizeof(float) * 9 * cin);
        float* d = reinterpret_cast<float*>(ab.bytes.data() + off);
        for (int c = 0; c < cin; ++c)
            for (int t = 0; t < 9; ++t) d[t * cin + c] = w[c * 9 + t] * S;
        fix.push_back({reinterpret_cast<void**>(&L.w9_tc), off});
        size_t offb = ab.alloc(sizeof(float) * cin);
        float* db = reinterpret_cast<float*>(ab.bytes.data() + offb);
        for (int c = 0; c < cin; ++c) db[c] = b[c] * S;
        fix.push_back({reinterpret_cast<void**>(&L.bias_tc), offb});
    }
    {   // pointwise [cout,cin,1,1] -> fp32 [cin][cout] and fp16 hi/lo [cout][cin]
        const std::vector<float>& w = W(ctx, L.p + "conv2.weight");
        size_t off = ab.alloc(sizeof(float) * cin * cout);
        float* d = reinterpret_cast<float*>(ab.bytes.data() + off);
        float maxabs = 0.f;
        for (int o = 0; o < cout; ++o)
            for (int k = 0; k < cin; ++k) {
                d[(size_t)k * cout + o] = w[(size_t)o * cin + k];
                if (std::isfinite(w[(size_t)o * cin + k])) maxabs = std::max(maxabs, std::fabs(w[(size_t)o * cin + k]));
            }
        fix.push_back({reinterpret_cast<void**>(&L.pw_t), off});
        // power-of-two scale so the largest weight lands in [8192, 16384): hi and lo both stay
        // well inside fp16's normal range, and the scale is undone exactly in the epilogue.
        int k2 = 0;
        if (maxabs > 0.f) k2 = (int)std::floor(std::log2(16384.0 / (double)maxabs));
        k2 = std::max(-14, std::min(24, k2));
        const float wscale = std::ldexp(1.0f, k2);
        L.tc_inv_scale = 1.0f / (wscale * 64.0f /* kActSplitScale */);
        size_t off_hi = ab.alloc(sizeof(__half) * cin * cout);
        size_t off_lo = ab.alloc(sizeof(__half) * cin * cout);
        __half* hi = reinterpret_cast<__half*>(ab.bytes.data() + off_hi);
        __half* lo = reinterpret_cast<__half*>(ab.bytes.data() + off_lo);
        for (size_t i = 0; i < (size_t)cin * cout; ++i) {
            const float s = w[i] * wscale;
            const __half h = __float2half_rn(s);
            hi[i] = h;
            lo[i] = __float2half_rn(s - __half2float(h));
        }
        fix.push_back({reinterpret_cast<void**>(&L.pw_hi), off_hi});
        fix.push_back({reinterpret_cast<void**>(&L.pw_lo), off_lo});
    }
    if (L.down || L.up) {
        const int cf = L.down ? cin : cout;
        const std::vector<float>& f = W(ctx, L.p + (L.down ? "downsample.filter.weight" : "upsample.filter.weight"));
        size_t off = ab.alloc(sizeof(float) * 16 * cf);
        float* d = reinterpret_cast<float*>(ab.bytes.data() + off);
        for (int c = 0; c < cf; ++c)
            for (int t = 0; t < 16; ++t) d[t * cf + c] = f[c * 16 + t];
        fix.push_back({reinterpret_cast<void**>(&L.fir16), off});
        if (L.up) {   // the fused prologue keeps the 16 taps in registers: they must not depend on the channel
            L.up_uniform = true;
            for (int c = 1; c < cf && L.up_uniform; ++c)
                for (int t = 0; t < 16; ++t)
                    if (f[c * 16 + t] != f[t]) { L.up_uniform = false; break; }
            for (int t = 0; t < 16; ++t) L.up_taps_s2[t] = f[t] * 1.41421356237309515f;
        }
    }
    if (L.up) {
        // The kernels implement zero insertion; check filter_const is that pattern (migan_inference.py:83-85).
        const std::vector<float>& fc = W(ctx, L.p + "upsample.filter_const");
        const int r = L.res_out;
        for (int y = 0; y < r; ++y)
            for (int x = 0; x < r; ++x) {
                const float want = ((y | x) & 1) ? 0.f : 1.f;
                if (fc[(size_t)y * r + x] != want)
                    return fail(MIGAN_ERR_INVALID, "%supsample.filter_const is not the zero-insertion pattern at (%d,%d)", L.p.c_str(), y, x);
            }
    }
    if (L.noise) {
        const std::vector<float>& nc = W(ctx, L.p + "noise_const");
        const float ns = W(ctx, L.p + "noise_strength")[0];
        size_t off = ab.alloc(sizeof(float) * nc.size());
        float* d = reinterpret_cast<float*>(ab.bytes.data() + off);
        for (size_t i = 0; i < nc.size(); ++i) d[i] = nc[i] * ns;  // migan_inference.py:166
        fix.push_back({reinterpret_cast<void**>(&L.noise_dev), off});
        if (L.up) {
            size_t off2 = ab.alloc(sizeof(float) * nc.size());
            float* d2 = reinterpret_cast<float*>(ab.bytes.data() + off2);
            for (size_t i = 0; i < nc.size(); ++i) d2[i] = nc[i] * ns * 1.41421356237309515f;
            fix.push_back({reinterpret_cast<void**>(&L.noise_s2_dev), off2});
        }
    }
    return MIGAN_OK;
}

int migan_finalize_weights(migan_ctx* ctx) {
    if (!ctx) return fail(MIGAN_ERR_INVALID, "null ctx");
    if (ctx->device < 0) return fail(MIGAN_ERR_CUDA, "context was created without a CUDA device: this library has no CPU path");
    for (size_t i = 0; i < ctx->specs.size(); ++i)
        if (!ctx->provided[i]) return fail(MIGAN_ERR_STATE, "missing key '%s'", ctx->specs[i].name.c_str());
    ArenaBuilder ab;
    std::vector<std::pair<void**, size_t>> fix;
    {
        const std::string p = "encoder.b" + std::to_string(ctx->resolution) + ".fromrgb.";
        const std::vector<float>& w = W(ctx, p + "weight");
        const std::vector<float>& b = W(ctx, p + "bias");
        size_t ow = ab.alloc(sizeof(float) * w.size());
        memcpy(ab.bytes.data() + ow, w.data(), sizeof(float) * w.size());
        size_t ob = ab.alloc(sizeof(float) * b.size());
        memcpy(ab.bytes.data() + ob, b.data(), sizeof(float) * b.size());
        fix.push_back({reinterpret_cast<void**>(&ctx->fromrgb_w), ow});
        fix.push_back({reinterpret_cast<void**>(&ctx->fromrgb_b), ob});
        size_t ow2 = ab.alloc(sizeof(float) * w.size()), ob2 = ab.alloc(sizeof(float) * b.size());
        float* dw2 = reinterpret_cast<float*>(ab.bytes.data() + ow2);
        float* db2 = reinterpret_cast<float*>(ab.bytes.data() + ob2);
        for (size_t i = 0; i < w.size(); ++i) dw2[i] = w[i] * 1.41421356237309515f;
        for (size_t i = 0; i < b.size(); ++i) db2[i] = b[i] * 1.41421356237309515f;
        fix.push_back({reinterpret_cast<void**>(&ctx->fromrgb_w_s2), ow2});
        fix.push_back({reinterpret_cast<void**>(&ctx->fromrgb_b_s2), ob2});
    }
    for (auto* vec : {&ctx->enc1, &ctx->enc2, &ctx->syn1, &ctx->syn2})
        for (SepConv& L : *vec) {
            int rc = pack_sepconv(ctx, L, ab, fix);
            if (rc) return rc;
        }
    for (ToRgb& t : ctx->torgb) {
        const std::vector<float>& w = W(ctx, t.p + "torgb.weight");
        const std::vector<float>& b = W(ctx, t.p + "torgb.bias");
        size_t ow = ab.alloc(sizeof(float) * w.size());
        memcpy(ab.bytes.data() + ow, w.data(), sizeof(float) * w.size());
        size_t ob = ab.alloc(sizeof(float) * 4);
        memcpy(ab.bytes.data() + ob, b.data(), sizeof(float) * 3);
        fix.push_back({reinterpret_cast<void**>(&t.w), ow});
        fix.push_back({reinterpret_cast<void**>(&t.b), ob});
        if (t.has_up) {
            const std::vector<float>& fc = W(ctx, t.p + "upsample.filter_const");
            for (int y = 0; y < t.res; ++y)
                for (int x = 0; x < t.res; ++x)
                    if (fc[(size_t)y * t.res + x] != (((y | x) & 1) ? 0.f : 1.f))
                        return fail(MIGAN_ERR_INVALID, "%supsample.filter_const is not the zero-insertion pattern", t.p.c_str());
            const std::vector<float>& f = W(ctx, t.p + "upsample.filter.weight");
            size_t of = ab.alloc(sizeof(float) * 48);
            float* d = reinterpret_cast<float*>(ab.bytes.data() + of);
            for (int c = 0; c < 3; ++c)
                for (int k = 0; k < 16; ++k) d[k * 3 + c] = f[c * 16 + k];
            fix.push_back({reinterpret_cast<void**>(&t.fir), of});
        }
    }
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (ctx->arena) {
        CUDA_TRY(cudaDeviceSynchronize());
        CUDA_TRY(cudaFree(ctx->arena));
        ctx->arena = nullptr;
    }
    CUDA_TRY(cudaMalloc(&ctx->arena, ab.bytes.size()));
    CUDA_TRY(cudaMemcpy(ctx->arena, ab.bytes.data(), ab.bytes.size(), cudaMemcpyHostToDevice));
    for (auto& f : fix) *f.first = static_cast<unsigned char*>(ctx->arena) + f.second;
    ctx->plan = Plan();  // pointers changed
    if (ctx->graph_exec) { cudaGraphExecDestroy(ctx->graph_exec); ctx->graph_exec = nullptr; }
    ctx->finalized = true;
    return MIGAN_OK;
}

// ---- workspace layout -------------------------------------------------------------------
//   feats[r]  n * r^2 * ch(r) fp32, one per encoder resolution (the decoder skip inputs)
//   S0..S2    three rotating scratch tensors of n * R^2 * ch(R) fp32 (largest activation)
//   IMG0/1    ping-pong planar RGB images n * 3 * R^2 fp32
static size_t feat_bytes(int n, int r) { return align_up((size_t)n * r * r * channels(r) * sizeof(float), 1024); }
static size_t scratch_bytes(const migan_ctx* c, int n) {
    return align_up((size_t)n * c->resolution * c->resolution * channels(c->resolution) * sizeof(float), 1024);
}
static size_t img_bytes(const migan_ctx* c, int n) {
    return align_up((size_t)n * 3 * c->resolution * c->resolution * sizeof(float), 1024);
}

size_t migan_workspace_bytes(const migan_ctx* ctx, int n) {
    if (!ctx || n <= 0) return 0;
    size_t total = 0;
    for (int r : ctx->enc_res) total += feat_bytes(n, r);
    total += 3 * scratch_bytes(ctx, n) + 2 * img_bytes(ctx, n);
    return total;
}

size_t migan_host_staging_bytes(const migan_ctx* ctx, int n) {
    if (!ctx || n <= 0) return 0;
    const size_t px = (size_t)n * ctx->resolution * ctx->resolution * sizeof(float);
    return 2 * (align_up(4 * px, 1024) + align_up(3 * px, 1024));   // two slots: consecutive calls overlap
}

}  // extern "C"

namespace {

// What the tensor-core kernel's prologue rebuilds on chip instead of reading it from HBM (sepconv_tc.h SepconvSource).
struct Fuse {
    bool stem = false;              // input = fromrgb(x): the stem tensor never exists (encoder.b{R}.conv1)
    const SepConv* up = nullptr;    // input = lrelu_agc(up2(up_t) + noise) + skip, `up` = the preceding up-sampling layer
    const float* up_t = nullptr;    // its raw low-resolution 1x1 output
    bool defer_up = false;          // this layer IS the up-sampling layer: emit only the raw 1x1 conv
};

struct PlanBuilder {
    migan_ctx* c;
    int n, path;
    unsigned char* base;
    std::map<int, float*> feat;
    float* S[3];
    float* IMG[2];
    std::vector<Step> steps;

    int other(int a, int b = -1) const {
        for (int i = 0; i < 3; ++i)
            if (i != a && i != b) return i;
        return 0;
    }
    void set_tap(Step& s, const std::string& name, const float* src, int C, int H, int W, bool planar = false, int flags = 0) {
        s.tap = name; s.tap_src = src; s.tapC = C; s.tapH = H; s.tapW = W; s.tap_planar = planar; s.tap_flags = flags;
    }

    static bool down_tma_enabled() {    // MIGAN_DOWN_TMA=0: register-streaming kernel (A/B measurements)
        const char* e = getenv("MIGAN_DOWN_TMA");
        return !e || atoi(e) != 0;
    }
    static int fuse_mask_dw() {         // MIGAN_FUSE bit 2: run the depthwise stage of the small Cout = 512 levels (res <= 32) inside the
        return fuse_mask() & 4;         // tensor-core kernel (its prologue repeats per N tile, which is cheap there) instead of as its own launch
    }
    static int fuse_mask() {            // MIGAN_FUSE bit 0: UP, bit 1: STEM, bit 2: small-level depthwise (debug / A-B measurements; default all on)
        const char* e = getenv("MIGAN_FUSE");
        return e ? atoi(e) : 7;
    }

    // Emit one SeparableConv2d reading `in` (NHWC [n,res_in,res_in,cin]); `skip` is added after the
    // final activation (decoder conv1, migan_inference.py:304-305).  Returns the output pointer.
    // in_idx: scratch index holding `in` (or -1 if it is a feat buffer); out_fixed: write there if non-null.
    int emit_sepconv(const SepConv& L, const float* in, int in_idx, float* out_fixed, const float* skip, int& out_idx, float*& out_ptr,
                     const migan::SepconvTcRgb* rgb = nullptr, const std::string& rgb_tap = std::string(), int rgb_flags = 0,
                     const Fuse& fuse = Fuse()) {
        const int t1 = other(in_idx), t2 = other(in_idx, t1);
        const bool tc = (path != MIGAN_PATH_SIMT);
        const float* gemm_in = nullptr;
        __half *ghi = nullptr, *glo = nullptr;
        bool presplit = L.down;
        if (L.down) {
            Step s; s.kind = K_DWDOWN; s.L = &L; s.in = in; s.n = n; s.H = L.res_in; s.W = L.res_in; s.C = L.cin;
            if (tc) {
                s.hi = reinterpret_cast<__half*>(S[t1]);
                s.lo = s.hi + (size_t)n * L.res_pw * L.res_pw * L.cin;
                ghi = s.hi; glo = s.lo;
                if (L.res_pw >= 16 && down_tma_enabled()) {   // rows staged through shared memory by TMA (elementwise.cu)
                    if (const char* err = migan::make_down_tensor_map(&s.down_map, in, n, L.res_in, L.res_in, L.cin))
                        return fail(MIGAN_ERR_CUDA, "tensor map for %sdownsample failed: %s", L.p.c_str(), err);
                    s.down_tma = true;
                }
            } else {
                s.out = S[t1]; gemm_in = S[t1];
                set_tap(s, L.p + "down", S[t1], L.cin, L.res_pw, L.res_pw);
            }
            steps.push_back(s);
        } else if (!tc) {
            Step s; s.kind = K_DW; s.L = &L; s.in = in; s.out = S[t1]; s.n = n; s.H = L.res_in; s.W = L.res_in; s.C = L.cin;
            set_tap(s, L.p + "dw_act", S[t1], L.cin, L.res_in, L.res_in);
            steps.push_back(s);
            gemm_in = S[t1];
        } else if (L.cout >= 512 && !rgb && (L.res_in >= 64 || fuse_mask_dw() == 0)) {
            // Cout spans 4 accumulator regions: a fused prologue would re-run the depthwise stage, so run it once as its
            // own kernel and hand the GEMM a pre-split operand (these layers are small: res <= 64)
            Step s; s.kind = K_DW; s.L = &L; s.in = in; s.n = n; s.H = L.res_in; s.W = L.res_in; s.C = L.cin;
            s.hi = reinterpret_cast<__half*>(S[t1]);
            s.lo = s.hi + (size_t)n * L.res_in * L.res_in * L.cin;
            ghi = s.hi; glo = s.lo;
            steps.push_back(s);
            presplit = true;
        }
        // 1x1 conv at res_pw
        float* pw_out;
        int pw_idx;
        const bool raw = L.up;  // up layers: noise/act happen after the FIR (K_UP2, or the next layer's fused prologue)
        if (raw) { pw_out = S[t2]; pw_idx = t2; }
        else if (out_fixed) { pw_out = out_fixed; pw_idx = -1; }
        else { pw_out = S[t2]; pw_idx = t2; }
        {
            Step s; s.L = &L; s.n = n; s.H = L.res_pw; s.W = L.res_pw; s.C = L.cin; s.out = pw_out;
            s.act = raw ? 0 : 1;
            s.aux = (!raw && L.noise) ? L.noise_dev : nullptr;
            if (tc) {
                s.kind = K_SEPCONV_TC;
                s.in = presplit ? nullptr : in;  // pre-split A operand from K_DWDOWN / K_DW
                s.hi = ghi; s.lo = glo;
                migan::SepconvTcDesc d;
                d.passes = (path == MIGAN_PATH_TC_FAST) ? 1 : 3;
                d.source = presplit ? migan::SEPCONV_SRC_SPLIT : migan::SEPCONV_SRC_NHWC;
                d.in_f32 = s.in; d.a_hi = ghi; d.a_lo = glo;
                d.w9 = L.w9_tc; d.bias = L.bias_tc; d.w_hi = L.pw_hi; d.w_lo = L.pw_lo; d.inv_scale = L.tc_inv_scale;
                d.noise = s.aux; d.out = pw_out; d.n = n; d.res = L.res_pw; d.cin = L.cin; d.cout = L.cout; d.act = s.act; d.rgb = rgb;
                if (fuse.stem) {
                    d.source = migan::SEPCONV_SRC_STEM; d.in_f32 = nullptr;
                    d.stem_w = c->fromrgb_w_s2; d.stem_b = c->fromrgb_b_s2;
                    s.in = nullptr; s.io_flags |= PTR_X; s.fused_stem = true;
                } else if (fuse.up) {
                    d.source = migan::SEPCONV_SRC_UP;      // d.in_f32 = `in` = the encoder feature (skip tensor)
                    d.up_t = fuse.up_t;
                    d.up_noise = fuse.up->noise ? fuse.up->noise_s2_dev : nullptr;
                    memcpy(d.up_taps, fuse.up->up_taps_s2, sizeof(d.up_taps));
                    s.aux2 = fuse.up_t; s.fused_up = true;
                }
                const char* err = migan::sepconv_tc_plan_ex(&s.tc, d);
                if (rgb) {
                    s.io_flags |= rgb_flags;
                    s.tap2 = rgb_tap; s.tap2_src = rgb->img_out; s.tap2C = 3; s.tap2H = L.res_pw; s.tap2W = L.res_pw; s.tap2_flags = rgb_flags;
                }
                if (err) return fail(MIGAN_ERR_CUDA, "tcgen05 plan for %s failed: %s", L.p.c_str(), err);
            } else {
                s.kind = K_GEMM_SIMT; s.in = gemm_in;
            }
            if (!(rgb && !rgb->store_out)) set_tap(s, L.p + (raw ? "pw" : "out"), pw_out, L.cout, L.res_pw, L.res_pw);
            steps.push_back(s);
        }
        out_ptr = pw_out; out_idx = pw_idx;
        if (L.up && fuse.defer_up) return MIGAN_OK;   // FIR + noise + activation + skip happen in the next layer's prologue
        if (L.up) {
            float* up_out; int up_idx;
            if (out_fixed) { up_out = out_fixed; up_idx = -1; }
            else { up_idx = other(pw_idx); up_out = S[up_idx]; }
            Step s; s.kind = K_UP2; s.L = &L; s.in = pw_out; s.out = up_out; s.aux = skip;
            s.n = n; s.H = L.res_pw; s.W = L.res_pw; s.C = L.cout;
            set_tap(s, L.p + (skip ? "out_skip" : "out"), up_out, L.cout, L.res_out, L.res_out);
            steps.push_back(s);
            out_ptr = up_out; out_idx = up_idx;
        } else if (skip) {
            Step s; s.kind = K_ADD; s.out = pw_out; s.aux = skip; s.n = n; s.H = L.res_out; s.W = L.res_out; s.C = L.cout;
            set_tap(s, L.p + "out_skip", pw_out, L.cout, L.res_out, L.res_out);
            steps.push_back(s);
        }
        return MIGAN_OK;
    }

    int build() {
        size_t off = 0;
        for (int r : c->enc_res) { feat[r] = reinterpret_cast<float*>(base + off); off += feat_bytes(n, r); }
        for (int i = 0; i < 3; ++i) { S[i] = reinterpret_cast<float*>(base + off); off += scratch_bytes(c, n); }
        for (int i = 0; i < 2; ++i) { IMG[i] = reinterpret_cast<float*>(base + off); off += img_bytes(c, n); }
        const int R = c->resolution;
        const bool tcp = (path != MIGAN_PATH_SIMT);
        const int fm = fuse_mask();
        // ---- encoder (migan_inference.py:235-246) ----
        // The stem (fromrgb + activation, :193-196) is recomputed inside encoder.b{R}.conv1's prologue when that layer runs
        // on the fused tensor-core kernel with 8 x 16 tiles; otherwise it is its own kernel.
        const bool fuse_stem = tcp && (fm & 2) && R >= 16 && channels(R) < 512;
        if (!fuse_stem) {
            Step s; s.kind = K_STEM; s.io_flags = PTR_X; s.out = S[0]; s.n = n; s.H = R; s.W = R; s.C = channels(R);
            set_tap(s, "encoder.b" + std::to_string(R) + ".fromrgb", S[0], channels(R), R, R);
            steps.push_back(s);
        }
        const float* cur = S[0];
        int cur_idx = 0;
        for (size_t i = 0; i < c->enc_res.size(); ++i) {
            const int r = c->enc_res[i];
            int oi; float* op;
            Fuse f1;
            f1.stem = (i == 0 && fuse_stem);
            int rc = emit_sepconv(c->enc1[i], cur, cur_idx, feat[r], nullptr, oi, op, nullptr, std::string(), 0, f1);  // feat = conv1(x)
            if (rc) return rc;
            rc = emit_sepconv(c->enc2[i], feat[r], -1, nullptr, nullptr, oi, op);      // x = conv2(feat)
            if (rc) return rc;
            cur = op; cur_idx = oi;
        }
        // ---- synthesis (migan_inference.py:347-352) ----
        int img_cur = -1;
        for (size_t i = 0; i < c->syn_res.size(); ++i) {
            const int r = c->syn_res[i];
            int oi; float* op;
            const bool last = (i + 1 == c->syn_res.size());
            const int img_next = (img_cur < 0) ? 0 : 1 - img_cur;
            const float* img_lo = (img_cur >= 0) ? IMG[img_cur] : nullptr;
            float* img_out = last ? nullptr : IMG[img_next];      // last level: the caller's y (bound at launch)
            const ToRgb& T = c->torgb[i];
            const bool fuse_rgb = tcp && channels(r) <= 256;   // all output channels of a pixel tile in one CTA (two N halves at 256)
            // conv1's FIR + noise + activation + skip can be rebuilt in conv2's prologue (the up-sampled tensor then never
            // exists in HBM) when conv2 runs its depthwise stage in the tensor-core kernel with 8 x 16 tiles.
            const SepConv& L1 = c->syn1[i];
            const bool fuse_up = tcp && (fm & 1) && L1.up && L1.up_uniform && r >= 16 && (channels(r) < 512 || fuse_rgb);
            Fuse f1; f1.defer_up = fuse_up;
            int rc = emit_sepconv(L1, cur, cur_idx, nullptr, feat[r], oi, op, nullptr, std::string(), 0, f1);  // x = conv1(x) + enc_feat
            if (rc) return rc;
            cur = op; cur_idx = oi;
            Fuse f2;
            const float* in2 = cur;
            if (fuse_up) { f2.up = &L1; f2.up_t = cur; in2 = feat[r]; }   // scratch bookkeeping still protects `cur` (= t)
            if (fuse_rgb) {
                migan::SepconvTcRgb rgb;
                rgb.w = T.w; rgb.b = T.b; rgb.fir = T.fir; rgb.img_lo = img_lo; rgb.img_out = img_out; rgb.store_out = last ? 0 : 1;
                rc = emit_sepconv(c->syn2[i], in2, cur_idx, nullptr, nullptr, oi, op, &rgb, T.p + "img", last ? PTR_Y : 0, f2);
                if (rc) return rc;
                cur = op; cur_idx = oi;
            } else {
                rc = emit_sepconv(c->syn2[i], in2, cur_idx, nullptr, nullptr, oi, op, nullptr, std::string(), 0, f2);
                if (rc) return rc;
                cur = op; cur_idx = oi;
                Step s; s.kind = K_TORGB; s.T = &T; s.in = cur; s.n = n; s.H = r; s.W = r; s.C = channels(r);
                s.aux = img_lo;
                if (last) { s.io_flags = PTR_Y; s.out = nullptr; }
                else s.out = img_out;
                set_tap(s, T.p + "img", s.out, 3, r, r, true, last ? PTR_Y : 0);
                steps.push_back(s);
            }
            img_cur = img_next;
        }
        annotate();
        return MIGAN_OK;
    }

    static const char* kernel_name(StepKind k) {
        switch (k) {
            case K_STEM: return "stem_fromrgb";
            case K_DW: return "dw3x3_act";
            case K_DWDOWN: return "dw3x3_down";
            case K_GEMM_SIMT: return "pw_gemm_simt";
            case K_SEPCONV_TC: return "sepconv_tc";
            case K_UP2: return "up2_noise_act_skip";
            case K_TORGB: return "torgb_img";
            case K_ADD: return "add_inplace";
        }
        return "?";
    }

    void annotate() {
        for (Step& s : steps) {
            const double px = (double)s.n * s.H * s.W, f = sizeof(float);
            switch (s.kind) {
                case K_STEM: s.alg_bytes = px * (4 + s.C) * f; s.flops = px * s.C * 8; break;
                case K_DW: s.alg_bytes = px * s.C * 2 * f; s.flops = px * s.C * 18; break;
                case K_DWDOWN: s.alg_bytes = px * s.C * 1.25 * f; s.flops = px * s.C * (18 + 8); break;
                case K_GEMM_SIMT: s.alg_bytes = px * (s.L->cin + s.L->cout) * f; s.flops = px * 2.0 * s.L->cin * s.L->cout; break;
                case K_SEPCONV_TC:
                    s.alg_bytes = px * (s.L->cin + s.L->cout) * f;
                    s.flops = px * (2.0 * s.L->cin * s.L->cout + ((s.in || s.fused_stem) ? 18.0 * s.L->cin : 0.0));
                    if (s.fused_stem) { s.alg_bytes = px * (4 + s.L->cout) * f; s.flops += px * s.L->cin * 8.0; }
                    if (s.fused_up) { s.alg_bytes += px * 0.25 * s.L->cin * f; s.flops += px * s.L->cin * 8.0; }   // + the low-res tensor
                    if (!s.tap2.empty()) {   // fused torgb: + image in/out, - feature map if it is not stored
                        s.alg_bytes += px * 3.75 * f;
                        s.flops += px * s.L->cout * 6;
                        if (s.tap.empty()) s.alg_bytes -= px * s.L->cout * f;
                    }
                    break;
                case K_UP2: s.alg_bytes = px * s.C * f * (1 + 4 + (s.aux ? 4 : 0)); s.flops = px * 4 * s.C * 8; break;
                case K_TORGB: s.alg_bytes = px * (s.C + 3 + (s.aux ? 0.75 : 0)) * f; s.flops = px * s.C * 6; break;
                case K_ADD: s.alg_bytes = px * s.C * 3 * f; s.flops = px * s.C; break;
            }
            s.label = (s.L ? s.L->p : s.T ? s.T->p + "torgb." : std::string("encoder.fromrgb.")) + kernel_name(s.kind);
        }
    }
};

int build_plan(migan_ctx* ctx, int n, int path, void* ws) {
    PlanBuilder pb;
    pb.c = ctx; pb.n = n; pb.path = path; pb.base = static_cast<unsigned char*>(ws);
    int rc = pb.build();
    if (rc) return rc;
    ctx->plan.n = n; ctx->plan.path = path; ctx->plan.ws = ws;
    ctx->plan.steps.swap(pb.steps);
    return MIGAN_OK;
}

int run_step(migan_ctx* ctx, Step& s, const float* x, float* y, cudaStream_t st) {
    const float* in = (s.io_flags & PTR_X) ? x : s.in;
    float* out = (s.io_flags & PTR_Y) ? y : s.out;
    cudaError_t e = cudaSuccess;
    switch (s.kind) {
        case K_STEM:
            e = migan::launch_stem(in, ctx->fromrgb_w, ctx->fromrgb_b, out, s.n, s.H, s.W, s.C, st);
            break;
        case K_DW:
            e = migan::launch_dw3x3(in, s.L->w9, s.L->bias, s.out, s.hi, s.lo, s.n, s.H, s.W, s.C, st);
            break;
        case K_DWDOWN:
            if (s.down_tma)
                e = migan::launch_dw3x3_down_tma(s.down_map, s.L->w9_tc, s.L->bias_tc, s.L->fir16, s.hi, s.lo, s.n, s.H, s.W, s.C, st);
            else if (s.hi && !s.out && s.W >= 8)   // tensor-core feed: specialised kernel on the pre-scaled tap table
                e = migan::launch_dw3x3_down_split(in, s.L->w9_tc, s.L->bias_tc, s.L->fir16, s.hi, s.lo, s.n, s.H, s.W, s.C, st);
            else
                e = migan::launch_dw3x3_down(in, s.L->w9, s.L->bias, s.L->fir16, s.out, s.hi, s.lo, s.n, s.H, s.W, s.C, st);
            break;
        case K_GEMM_SIMT:
            e = migan::launch_pw_gemm_simt(in, s.L->pw_t, out, (int64_t)s.n * s.H * s.W, s.L->cin, s.L->cout,
                                           s.aux, s.H * s.W, s.act, st);
            break;
        case K_SEPCONV_TC:
            e = migan::launch_sepconv_tc(s.tc, st, (s.io_flags & PTR_Y) ? y : nullptr, s.fused_stem ? x : nullptr);
            break;
        case K_UP2:
            e = migan::launch_up2(in, s.L->fir16, s.L->noise ? s.L->noise_dev : nullptr, s.aux, out, s.n, s.H, s.W, s.C, st);
            break;
        case K_TORGB:
            e = migan::launch_torgb(in, s.T->w, s.T->b, s.aux, s.T->fir, out, s.n, s.H, s.C, st);
            break;
        case K_ADD:
            e = migan::launch_add(out, s.aux, (int64_t)s.n * s.H * s.W * s.C, st);
            break;
    }
    if (e != cudaSuccess)   // asynchronous failures of EARLIER launches surface here too: the pipeline-timeout record names the wait
        return fail(MIGAN_ERR_CUDA, "kernel launch (step %s) failed: %s [tcgen05 pipeline timeout record 0x%x]", s.label.c_str(),
                    cudaGetErrorString(e), (unsigned)migan::sepconv_tc_timeout_record(ctx->device));
    ctx->last_launches++;
    if (ctx->tap_dst && !s.tap.empty() && s.tap == ctx->tap_name) {
        const float* src = (s.tap_flags & PTR_Y) ? y : s.tap_src;
        if (s.tap_planar)
            e = cudaMemcpyAsync(ctx->tap_dst, src, sizeof(float) * (size_t)s.n * s.tapC * s.tapH * s.tapW, cudaMemcpyDeviceToDevice, st);
        else
            e = migan::launch_nhwc_to_nchw(src, ctx->tap_dst, s.n, s.tapH, s.tapW, s.tapC, st);
        if (e != cudaSuccess) return fail(MIGAN_ERR_CUDA, "tap copy failed: %s", cudaGetErrorString(e));
    }
    if (ctx->tap_dst && !s.tap2.empty() && s.tap2 == ctx->tap_name) {
        const float* src = (s.tap2_flags & PTR_Y) ? y : s.tap2_src;
        e = cudaMemcpyAsync(ctx->tap_dst, src, sizeof(float) * (size_t)s.n * s.tap2C * s.tap2H * s.tap2W, cudaMemcpyDeviceToDevice, st);
        if (e != cudaSuccess) return fail(MIGAN_ERR_CUDA, "tap copy failed: %s", cudaGetErrorString(e));
    }
    return MIGAN_OK;
}

}  // namespace

extern "C" {

int migan_forward(migan_ctx* ctx, const float* x, float* y, int n, void* workspace, size_t workspace_bytes,
                  int path, void* stream) {
    if (!ctx || !x || !y || !workspace) return fail(MIGAN_ERR_INVALID, "null argument");
    if (!ctx->finalized) return fail(MIGAN_ERR_STATE, "weights not finalized (call migan_finalize_weights)");
    if (n <= 0) return fail(MIGAN_ERR_INVALID, "batch size must be positive, got %d", n);
    if (path != MIGAN_PATH_SIMT && path != MIGAN_PATH_TC && path != MIGAN_PATH_TC_FAST)
        return fail(MIGAN_ERR_INVALID, "unknown path %d", path);
    if (workspace_bytes < migan_workspace_bytes(ctx, n))
        return fail(MIGAN_ERR_WORKSPACE, "workspace too small: %zu < %zu bytes", workspace_bytes, migan_workspace_bytes(ctx, n));
    if ((reinterpret_cast<uintptr_t>(workspace) & 1023) || (reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(y) & 15))
        return fail(MIGAN_ERR_WORKSPACE, "workspace must be 1024-byte aligned, x / y 16-byte aligned");
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (ctx->plan.n != n || ctx->plan.path != path || ctx->plan.ws != workspace) {
        int rc = build_plan(ctx, n, path, workspace);
        if (rc) return rc;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ctx->last_launches = 0;
    if (ctx->profiling) {
        while (ctx->events.size() < 2 * ctx->plan.steps.size()) {
            cudaEvent_t e;
            CUDA_TRY(cudaEventCreate(&e));
            ctx->events.push_back(e);
        }
    }
    size_t i = 0;
    for (Step& s : ctx->plan.steps) {
        if (ctx->profiling) CUDA_TRY(cudaEventRecord(ctx->events[2 * i], st));
        int rc = run_step(ctx, s, x, y, st);
        if (rc) return rc;
        if (ctx->profiling) CUDA_TRY(cudaEventRecord(ctx->events[2 * i + 1], st));
        ++i;
    }
    return MIGAN_OK;
}

size_t migan_graph_staging_bytes(const migan_ctx* ctx, int n) {
    if (!ctx || n <= 0) return 0;
    const size_t px = (size_t)n * ctx->resolution * ctx->resolution * sizeof(float);
    return align_up(4 * px, 1024) + align_up(3 * px, 1024);
}

int migan_forward_graph(migan_ctx* ctx, const float* x, float* y, int n, void* workspace, size_t workspace_bytes,
                        int path, void* stream) {
    if (!ctx || !x || !y || !workspace) return fail(MIGAN_ERR_INVALID, "null argument");
    if (n <= 0) return fail(MIGAN_ERR_INVALID, "batch size must be positive, got %d", n);
    const size_t ws = migan_workspace_bytes(ctx, n);
    if (workspace_bytes < ws + migan_graph_staging_bytes(ctx, n))
        return fail(MIGAN_ERR_WORKSPACE, "workspace too small for the graph staging buffers: %zu < %zu bytes", workspace_bytes,
                    ws + migan_graph_staging_bytes(ctx, n));
    const size_t px = (size_t)n * ctx->resolution * ctx->resolution * sizeof(float);
    float* xg = reinterpret_cast<float*>(static_cast<unsigned char*>(workspace) + ws);
    float* yg = reinterpret_cast<float*>(static_cast<unsigned char*>(workspace) + ws + align_up(4 * px, 1024));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (!ctx->graph_exec || ctx->graph_n != n || ctx->graph_path != path || ctx->graph_ws != workspace || ctx->profiling || ctx->tap_dst) {
        if (ctx->graph_exec) { cudaGraphExecDestroy(ctx->graph_exec); ctx->graph_exec = nullptr; }
        if (ctx->profiling || ctx->tap_dst) {   // per-launch events / taps need the plain launch sequence
            CUDA_TRY(cudaMemcpyAsync(xg, x, 4 * px, cudaMemcpyDeviceToDevice, st));
            if (int rc = migan_forward(ctx, xg, yg, n, workspace, ws, path, stream)) return rc;
            CUDA_TRY(cudaMemcpyAsync(y, yg, 3 * px, cudaMemcpyDeviceToDevice, st));
            return MIGAN_OK;
        }
        // one plain run first: validates the arguments, builds the plan and binds the stem's tensor map to xg outside the capture
        CUDA_TRY(cudaMemcpyAsync(xg, x, 4 * px, cudaMemcpyDeviceToDevice, st));
        if (int rc = migan_forward(ctx, xg, yg, n, workspace, ws, path, stream)) return rc;
        // capture on a private stream: the caller's stream may be the legacy default stream, which cannot be captured
        if (!ctx->s_cap) CUDA_TRY(cudaStreamCreateWithFlags(&ctx->s_cap, cudaStreamNonBlocking));
        CUDA_TRY(cudaStreamBeginCapture(ctx->s_cap, cudaStreamCaptureModeThreadLocal));
        const int rc = migan_forward(ctx, xg, yg, n, workspace, ws, path, ctx->s_cap);
        cudaGraph_t graph = nullptr;
        const cudaError_t ce = cudaStreamEndCapture(ctx->s_cap, &graph);
        if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
        if (ce != cudaSuccess) { if (graph) cudaGraphDestroy(graph); return fail(MIGAN_ERR_CUDA, "stream capture failed: %s", cudaGetErrorString(ce)); }
        const cudaError_t ie = cudaGraphInstantiate(&ctx->graph_exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ie != cudaSuccess) { ctx->graph_exec = nullptr; return fail(MIGAN_ERR_CUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ie)); }
        ctx->graph_n = n; ctx->graph_path = path; ctx->graph_ws = workspace; ctx->graph_launches = ctx->last_launches;
    }
    CUDA_TRY(cudaMemcpyAsync(xg, x, 4 * px, cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(cudaGraphLaunch(ctx->graph_exec, st));
    CUDA_TRY(cudaMemcpyAsync(y, yg, 3 * px, cudaMemcpyDeviceToDevice, st));
    ctx->last_launches = ctx->graph_launches;
    return MIGAN_OK;
}

int migan_set_profiling(migan_ctx* ctx, int enable) {
    if (!ctx) return fail(MIGAN_ERR_INVALID, "null ctx");
    ctx->profiling = enable != 0;
    return MIGAN_OK;
}

int migan_profile_num_steps(const migan_ctx* ctx) { return ctx ? (int)ctx->plan.steps.size() : 0; }

int migan_profile_step(migan_ctx* ctx, int index, const char** label, float* ms, double* alg_bytes, double* flops) {
    if (!ctx || index < 0 || index >= (int)ctx->plan.steps.size()) return fail(MIGAN_ERR_INVALID, "bad step index %d", index);
    const Step& s = ctx->plan.steps[index];
    if (label) *label = s.label.c_str();
    if (alg_bytes) *alg_bytes = s.alg_bytes;
    if (flops) *flops = s.flops;
    if (ms) {
        *ms = 0.f;
        if (ctx->events.size() >= 2 * (size_t)index + 2) {
            CUDA_TRY(cudaEventSynchronize(ctx->events[2 * index + 1]));
            CUDA_TRY(cudaEventElapsedTime(ms, ctx->events[2 * index], ctx->events[2 * index + 1]));
        }
    }
    return MIGAN_OK;
}

// Enqueue H2D -> forward -> D2H for one host batch without waiting for it.  Two staging slots alternate, so the
// copies of call c+1 overlap the kernels / copy-out of call c (a serving loop submits batches back to back and
// collects them with migan_host_wait).  Within a call the batch is split into micro-batches for the same reason.
static int forward_host_enqueue(migan_ctx* ctx, const float* x_host, float* y_host, int n, void* workspace,
                                size_t workspace_bytes, int path, void* stream, int* slot_out) {
    if (!ctx || !x_host || !y_host || !workspace) return fail(MIGAN_ERR_INVALID, "null argument");
    if (n <= 0) return fail(MIGAN_ERR_INVALID, "batch size must be positive, got %d", n);
    const size_t ws = migan_workspace_bytes(ctx, n);
    if (workspace_bytes < ws + migan_host_staging_bytes(ctx, n))
        return fail(MIGAN_ERR_WORKSPACE, "workspace too small for host staging: %zu < %zu bytes", workspace_bytes,
                    ws + migan_host_staging_bytes(ctx, n));
    const size_t px = (size_t)n * ctx->resolution * ctx->resolution * sizeof(float);
    const size_t slot_bytes = align_up(4 * px, 1024) + align_up(3 * px, 1024);
    const int slot = (int)(ctx->host_calls++ & 1);
    unsigned char* sbase = static_cast<unsigned char*>(workspace) + ws + slot * slot_bytes;
    float* xd = reinterpret_cast<float*>(sbase);
    float* yd = reinterpret_cast<float*>(sbase + align_up(4 * px, 1024));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CUDA_TRY(cudaSetDevice(ctx->device));
    // Micro-batch pipeline: H2D of micro-batch k+1 and D2H of k-1 overlap the kernels of k (three streams).
    // The small-resolution layers cost a fixed ~0.4 ms per forward, so the split is kept coarse.
    // Synchronous call (one batch, then wait): split it so the copies of one half overlap the kernels of the other
    // (measured at 512x512, n = 32: M = 1 / 2 / 4 / 8 -> 1770 / 1926 / 1896 / 1678 img/s).  Enqueue-only call: consecutive
    // batches already overlap through the two staging slots (H2D of batch t+1 and D2H of batch t-1 run under the kernels of
    // batch t), so the batch stays whole and does not pay the fixed per-forward cost of the small layers twice.
    int M = (slot_out != nullptr && n >= 8 && n % 2 == 0) ? 2 : 1;
    if (const char* e = getenv("MIGAN_HOST_PIPELINE")) {
        const int v = atoi(e);
        if (v >= 1 && n % v == 0) M = v;
    }
    if (!ctx->s_in) {
        CUDA_TRY(cudaStreamCreateWithFlags(&ctx->s_in, cudaStreamNonBlocking));
        CUDA_TRY(cudaStreamCreateWithFlags(&ctx->s_out, cudaStreamNonBlocking));
        for (int i = 0; i < 2; ++i) {
            CUDA_TRY(cudaEventCreateWithFlags(&ctx->slot_compute_done[i], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&ctx->slot_out_done[i], cudaEventDisableTiming));
        }
    }
    while ((int)ctx->host_events.size() < 2 * (2 * M + 1)) {
        cudaEvent_t e;
        CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ctx->host_events.push_back(e);
    }
    cudaEvent_t* ev = ctx->host_events.data() + slot * (2 * M + 1);   // per-slot events: [in_k, c_k] x M, start
    cudaEvent_t ev_start = ev[2 * M];
    const int m = n / M;
    const size_t xs = (size_t)m * 4 * ctx->resolution * ctx->resolution, ys = (size_t)m * 3 * ctx->resolution * ctx->resolution;
    // In steady state the copy-in stream does NOT wait for the caller's stream: x_host is host memory (valid from the call
    // on) and the only device hazard -- the staging slot still being read by the forward that used it two calls ago -- is
    // covered by slot_compute_done below.  Waiting on `stream` here would serialise the H2D of batch t+1 behind the kernels
    // of batch t, which is exactly the overlap the two slots exist for.
    // The FIRST use of a staging area is different: the memory may have just been handed over by a stream-ordered
    // allocator (torch's caching allocator assumes same-stream reuse), so work still pending on the caller's stream may be
    // using it.  Order both copy streams after the caller's stream once, whenever a slot sees new memory.
    if (!ctx->slot_used[slot] || ctx->slot_base[slot] != sbase) {
        CUDA_TRY(cudaEventRecord(ev_start, st));
        CUDA_TRY(cudaStreamWaitEvent(ctx->s_in, ev_start, 0));
        CUDA_TRY(cudaStreamWaitEvent(ctx->s_out, ev_start, 0));
        ctx->slot_base[slot] = sbase;
    }
    if (ctx->slot_used[slot]) {
        CUDA_TRY(cudaStreamWaitEvent(ctx->s_in, ctx->slot_compute_done[slot], 0));   // xd[slot] free again
        CUDA_TRY(cudaStreamWaitEvent(st, ctx->slot_out_done[slot], 0));              // yd[slot] copied out
    }
    for (int k = 0; k < M; ++k) {
        CUDA_TRY(cudaMemcpyAsync(xd + k * xs, x_host + k * xs, xs * sizeof(float), cudaMemcpyHostToDevice, ctx->s_in));
        CUDA_TRY(cudaEventRecord(ev[2 * k], ctx->s_in));
    }
    int launches = 0;
    for (int k = 0; k < M; ++k) {
        CUDA_TRY(cudaStreamWaitEvent(st, ev[2 * k], 0));
        int rc = migan_forward(ctx, xd + k * xs, yd + k * ys, m, workspace, ws, path, stream);
        if (rc) return rc;
        launches += ctx->last_launches;
        CUDA_TRY(cudaEventRecord(ev[2 * k + 1], st));
        CUDA_TRY(cudaStreamWaitEvent(ctx->s_out, ev[2 * k + 1], 0));
        CUDA_TRY(cudaMemcpyAsync(y_host + k * ys, yd + k * ys, ys * sizeof(float), cudaMemcpyDeviceToHost, ctx->s_out));
    }
    ctx->last_launches = launches;
    CUDA_TRY(cudaEventRecord(ctx->slot_compute_done[slot], st));
    CUDA_TRY(cudaEventRecord(ctx->slot_out_done[slot], ctx->s_out));
    ctx->slot_used[slot] = true;
    if (slot_out) *slot_out = slot;
    return MIGAN_OK;
}

int migan_forward_host(migan_ctx* ctx, const float* x_host, float* y_host, int n, void* workspace,
                       size_t workspace_bytes, int path, void* stream) {
    int slot = 0;
    int rc = forward_host_enqueue(ctx, x_host, y_host, n, workspace, workspace_bytes, path, stream, &slot);
    if (rc) return rc;
    CUDA_TRY(cudaEventSynchronize(ctx->slot_out_done[slot]));   // y_host is complete on return
    return MIGAN_OK;
}

int migan_forward_host_async(migan_ctx* ctx, const float* x_host, float* y_host, int n, void* workspace,
                             size_t workspace_bytes, int path, void* stream) {
    return forward_host_enqueue(ctx, x_host, y_host, n, workspace, workspace_bytes, path, stream, nullptr);
}

static size_t u8_slot_bytes(const migan_ctx* ctx, int n) {
    const size_t px = (size_t)n * ctx->resolution * ctx->resolution;
    return align_up(4 * px * sizeof(float), 1024) + align_up(3 * px * sizeof(float), 1024) + 2 * align_up(3 * px, 1024) + align_up(px, 1024);
}

size_t migan_u8_staging_bytes(const migan_ctx* ctx, int n) {
    if (!ctx || n <= 0) return 0;
    return 2 * u8_slot_bytes(ctx, n);     // two slots: consecutive calls overlap
}

// Enqueue H2D(img, mask) -> preprocess -> forward -> postprocess -> D2H(out) for one uint8 request batch.  Same three-stream,
// two-slot scheme as the fp32 host call: the copies of call c+1 / c-1 run under the kernels of call c.
static int forward_u8_enqueue(migan_ctx* ctx, const uint8_t* img_host, const uint8_t* mask_host, uint8_t* out_host, int n,
                              void* workspace, size_t workspace_bytes, int path, void* stream, int* slot_out) {
    if (!ctx || !img_host || !mask_host || !out_host || !workspace) return fail(MIGAN_ERR_INVALID, "null argument");
    if (n <= 0) return fail(MIGAN_ERR_INVALID, "batch size must be positive, got %d", n);
    const size_t ws = migan_workspace_bytes(ctx, n);
    if (workspace_bytes < ws + migan_u8_staging_bytes(ctx, n))
        return fail(MIGAN_ERR_WORKSPACE, "workspace too small for uint8 staging: %zu < %zu bytes", workspace_bytes,
                    ws + migan_u8_staging_bytes(ctx, n));
    const int R = ctx->resolution;
    const size_t px = (size_t)n * R * R;
    const int slot = (int)(ctx->u8_calls++ & 1);
    unsigned char* sbase = static_cast<unsigned char*>(workspace) + ws + slot * u8_slot_bytes(ctx, n);
    unsigned char* b = sbase;
    float* xd = reinterpret_cast<float*>(b);               b += align_up(4 * px * sizeof(float), 1024);
    float* yd = reinterpret_cast<float*>(b);               b += align_up(3 * px * sizeof(float), 1024);
    uint8_t* img_d = b;                                     b += align_up(3 * px, 1024);
    uint8_t* out_d = b;                                     b += align_up(3 * px, 1024);
    uint8_t* mask_d = b;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (!ctx->s_in) {
        CUDA_TRY(cudaStreamCreateWithFlags(&ctx->s_in, cudaStreamNonBlocking));
        CUDA_TRY(cudaStreamCreateWithFlags(&ctx->s_out, cudaStreamNonBlocking));
        for (int i = 0; i < 2; ++i) {
            CUDA_TRY(cudaEventCreateWithFlags(&ctx->slot_compute_done[i], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&ctx->slot_out_done[i], cudaEventDisableTiming));
        }
    }
    if (!ctx->u8_start) {
        CUDA_TRY(cudaEventCreateWithFlags(&ctx->u8_start, cudaEventDisableTiming));
        for (int i = 0; i < 2; ++i) {
            CUDA_TRY(cudaEventCreateWithFlags(&ctx->u8_in[i], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&ctx->u8_compute_done[i], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&ctx->u8_out_done[i], cudaEventDisableTiming));
        }
    }
    if (!ctx->u8_used[slot] || ctx->u8_base[slot] != sbase) {   // new staging memory: order the copy streams after the caller's stream once
        CUDA_TRY(cudaEventRecord(ctx->u8_start, st));
        CUDA_TRY(cudaStreamWaitEvent(ctx->s_in, ctx->u8_start, 0));
        CUDA_TRY(cudaStreamWaitEvent(ctx->s_out, ctx->u8_start, 0));
        ctx->u8_base[slot] = sbase;
    }
    if (ctx->u8_used[slot]) {
        CUDA_TRY(cudaStreamWaitEvent(ctx->s_in, ctx->u8_compute_done[slot], 0));   // img_d / mask_d of this slot are free again
        CUDA_TRY(cudaStreamWaitEvent(st, ctx->u8_out_done[slot], 0));              // out_d of this slot has been copied out
    }
    CUDA_TRY(cudaMemcpyAsync(img_d, img_host, 3 * px, cudaMemcpyHostToDevice, ctx->s_in));
    CUDA_TRY(cudaMemcpyAsync(mask_d, mask_host, px, cudaMemcpyHostToDevice, ctx->s_in));
    CUDA_TRY(cudaEventRecord(ctx->u8_in[slot], ctx->s_in));
    CUDA_TRY(cudaStreamWaitEvent(st, ctx->u8_in[slot], 0));
    CUDA_TRY((cudaError_t)migan::launch_preprocess_u8(img_d, mask_d, xd, n, R, st));
    if (int rc = migan_forward(ctx, xd, yd, n, workspace, ws, path, stream)) return rc;
    CUDA_TRY((cudaError_t)migan::launch_postprocess_u8(yd, img_d, mask_d, out_d, n, R, st));
    ctx->last_launches += 2;
    CUDA_TRY(cudaEventRecord(ctx->u8_compute_done[slot], st));
    CUDA_TRY(cudaStreamWaitEvent(ctx->s_out, ctx->u8_compute_done[slot], 0));
    CUDA_TRY(cudaMemcpyAsync(out_host, out_d, 3 * px, cudaMemcpyDeviceToHost, ctx->s_out));
    CUDA_TRY(cudaEventRecord(ctx->u8_out_done[slot], ctx->s_out));
    ctx->u8_used[slot] = true;
    if (slot_out) *slot_out = slot;
    return MIGAN_OK;
}

int migan_forward_u8(migan_ctx* ctx, const uint8_t* img_host, const uint8_t* mask_host, uint8_t* out_host, int n,
                     void* workspace, size_t workspace_bytes, int path, void* stream) {
    int slot = 0;
    if (int rc = forward_u8_enqueue(ctx, img_host, mask_host, out_host, n, workspace, workspace_bytes, path, stream, &slot)) return rc;
    CUDA_TRY(cudaEventSynchronize(ctx->u8_out_done[slot]));   // out_host is complete on return
    return MIGAN_OK;
}

int migan_forward_u8_async(migan_ctx* ctx, const uint8_t* img_host, const uint8_t* mask_host, uint8_t* out_host, int n,
                           void* workspace, size_t workspace_bytes, int path, void* stream) {
    return forward_u8_enqueue(ctx, img_host, mask_host, out_host, n, workspace, workspace_bytes, path, stream, nullptr);
}

int b200_preprocess_u8(const uint8_t* img, const uint8_t* mask, float* x, int n, int r, void* stream) {
    if (!img || !mask || !x || n <= 0 || r <= 0) return fail(MIGAN_ERR_INVALID, "preprocess_u8: bad arguments");
    CUDA_TRY((cudaError_t)migan::launch_preprocess_u8(img, mask, x, n, r, static_cast<cudaStream_t>(stream)));
    return MIGAN_OK;
}

int b200_postprocess_u8(const float* y, const uint8_t* img, const uint8_t* mask, uint8_t* out, int n, int r, void* stream) {
    if (!y || !img || !mask || !out || n <= 0 || r <= 0) return fail(MIGAN_ERR_INVALID, "postprocess_u8: bad arguments");
    CUDA_TRY((cudaError_t)migan::launch_postprocess_u8(y, img, mask, out, n, r, static_cast<cudaStream_t>(stream)));
    return MIGAN_OK;
}

int b200_feather_composite(const float* y, const uint8_t* img, const uint8_t* mask, uint8_t* out, int n, int H, int W,
                           const float* k25, void* stream) {
    if (!y || !img || !mask || !out || !k25) return fail(MIGAN_ERR_INVALID, "feather_composite: null argument");
    if (n <= 0 || H < 3 || W < 3) return fail(MIGAN_ERR_INVALID, "feather_composite: need n >= 1 and H, W >= 3 (reflect padding of 2), got %d x %d x %d", n, H, W);
    CUDA_TRY((cudaError_t)migan::launch_feather_composite(y, img, mask, out, n, H, W, k25, static_cast<cudaStream_t>(stream)));
    return MIGAN_OK;
}

// ---- stream memory operations (multi-GPU signalling without a kernel) ----------------------------------------------------
// cuStreamWaitValue32 / cuStreamWriteValue32 through the runtime's driver entry points (the library has no libcuda link
// dependency).  A wait is executed by the stream's front end: no SM is occupied while a rank waits for its peers.
typedef int (*StreamMemOp32Fn)(cudaStream_t, unsigned long long, unsigned int, unsigned int);
static StreamMemOp32Fn stream_memop(const char* name) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint(name, &ptr, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) return nullptr;
    return reinterpret_cast<StreamMemOp32Fn>(ptr);
}

int b200_stream_memops_available(void) {
    static const int ok = (stream_memop("cuStreamWaitValue32") && stream_memop("cuStreamWriteValue32")) ? 1 : 0;
    return ok;
}

int b200_stream_wait_value32(void* stream, void* addr, uint32_t value) {
    static const StreamMemOp32Fn fn = stream_memop("cuStreamWaitValue32");
    if (!fn) return fail(MIGAN_ERR_CUDA, "cuStreamWaitValue32 entry point not available");
    if (!addr) return fail(MIGAN_ERR_INVALID, "stream_wait_value32: null address");
    const int r = fn(static_cast<cudaStream_t>(stream), (unsigned long long)(uintptr_t)addr, value, 0u /* CU_STREAM_WAIT_VALUE_GEQ: (int32)(*addr - value) >= 0 */);
    if (r != 0) return fail(MIGAN_ERR_CUDA, "cuStreamWaitValue32 failed with CUresult %d", r);
    return MIGAN_OK;
}

int b200_stream_write_value32(void* stream, void* addr, uint32_t value) {
    static const StreamMemOp32Fn fn = stream_memop("cuStreamWriteValue32");
    if (!fn) return fail(MIGAN_ERR_CUDA, "cuStreamWriteValue32 entry point not available");
    if (!addr) return fail(MIGAN_ERR_INVALID, "stream_write_value32: null address");
    const int r = fn(static_cast<cudaStream_t>(stream), (unsigned long long)(uintptr_t)addr, value, 0u);
    if (r != 0) return fail(MIGAN_ERR_CUDA, "cuStreamWriteValue32 failed with CUresult %d", r);
    return MIGAN_OK;
}

// ---- training snapshot -> inference filters (scripts/export_inference_model.py:18-27), kernel in reparam.cu ----
int b200_reparam_filter(const float* const* w_dev, int k, int cout, int64_t fan, float* out, void* stream) {
    if (!w_dev || !out) return fail(MIGAN_ERR_INVALID, "reparam_filter: null argument");
    if (k < 1 || k > 16) return fail(MIGAN_ERR_INVALID, "reparam_filter: %d tensors (1 .. 16 supported)", k);
    if (cout < 1 || fan < 1) return fail(MIGAN_ERR_INVALID, "reparam_filter: bad shape %d x %lld", cout, (long long)fan);
    for (int j = 0; j < k; ++j)
        if (!w_dev[j]) return fail(MIGAN_ERR_INVALID, "reparam_filter: tensor %d is null", j);
    CUDA_TRY((cudaError_t)migan::launch_reparam_filter(w_dev, k, cout, fan, out, static_cast<cudaStream_t>(stream)));
    return MIGAN_OK;
}

int b200_enable_peer_access(int peer_device) {
    const cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return MIGAN_OK; }
    if (e != cudaSuccess) { cudaGetLastError(); return fail(MIGAN_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d): %s", peer_device, cudaGetErrorString(e)); }
    return MIGAN_OK;
}

int b200_memcpy_async(void* dst, const void* src, size_t bytes, void* stream) {
    if (!dst || !src) return fail(MIGAN_ERR_INVALID, "memcpy_async: null argument");
    CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, static_cast<cudaStream_t>(stream)));
    return MIGAN_OK;
}

// ---- arbitrary-resolution crop pipeline (scripts/create_onnx_pipeline.py:121-264), kernels in pipeline.cu ----
size_t b200_pipeline_scratch_bytes(int H, int W, int res) {
    if (H < 1 || W < 1 || res < 1) return 0;
    return migan::pipeline_scratch_bytes(H, W, res);
}

int b200_resize_nearest_u8(const uint8_t* in, int H, int W, uint8_t* out, int oh, int ow, void* stream) {
    if (!in || !out) return fail(MIGAN_ERR_INVALID, "resize_nearest_u8: null argument");
    if (H < 1 || W < 1 || oh < 1 || ow < 1) return fail(MIGAN_ERR_INVALID, "resize_nearest_u8: bad size %d x %d -> %d x %d", H, W, oh, ow);
    CUDA_TRY((cudaError_t)migan::launch_resize_nearest_u8(in, H, W, out, oh, ow, static_cast<cudaStream_t>(stream)));
    return MIGAN_OK;
}

int b200_hole_flags(const uint8_t* mask, int H, int W, uint8_t* flags, void* stream) {
    if (!mask || !flags) return fail(MIGAN_ERR_INVALID, "hole_flags: null argument");
    if (H < 1 || W < 1) return fail(MIGAN_ERR_INVALID, "hole_flags: bad size %d x %d", H, W);
    CUDA_TRY((cudaError_t)migan::launch_hole_flags(mask, H, W, flags, static_cast<cudaStream_t>(stream)));
    return MIGAN_OK;
}

int migan_crop_box(const uint8_t* flags_host, int H, int W, int res, int padding, int* box4) {
    if (!flags_host || !box4) return fail(MIGAN_ERR_INVALID, "crop_box: null argument");
    if (H < 1 || W < 1 || res < 1 || padding < 0) return fail(MIGAN_ERR_INVALID, "crop_box: bad arguments (%d x %d, resolution %d, padding %d)", H, W, res, padding);
    migan::crop_box_from_flags(flags_host, H, W, res, padding, box4);
    return MIGAN_OK;
}

static int check_box(const char* who, int H, int W, const int* box) {
    if (!box) return fail(MIGAN_ERR_INVALID, "%s: null crop window", who);
    if (box[0] < 0 || box[1] > W || box[2] < 0 || box[3] > H || box[1] - box[0] < 3 || box[3] - box[2] < 3)
        return fail(MIGAN_ERR_INVALID, "%s: crop window x[%d,%d) y[%d,%d) must lie inside the %d x %d image and be at least 3 x 3",
                    who, box[0], box[1], box[2], box[3], H, W);
    return MIGAN_OK;
}

int b200_pipeline_preprocess(const uint8_t* image, const uint8_t* mask, int H, int W, const int* box, int res, float* x,
                             void* scratch, size_t scratch_bytes, void* stream) {
    if (!image || !mask || !x || !scratch) return fail(MIGAN_ERR_INVALID, "pipeline_preprocess: null argument");
    if (int rc = check_box("pipeline_preprocess", H, W, box)) return rc;
    if (res < 1) return fail(MIGAN_ERR_INVALID, "pipeline_preprocess: bad resolution %d", res);
    if (scratch_bytes < migan::pipeline_scratch_bytes(H, W, res))
        return fail(MIGAN_ERR_WORKSPACE, "pipeline_preprocess: scratch of %zu bytes, need %zu", scratch_bytes, migan::pipeline_scratch_bytes(H, W, res));
    CUDA_TRY((cudaError_t)migan::launch_pipeline_preprocess(image, mask, H, W, box, res, x, scratch, static_cast<cudaStream_t>(stream)));
    return MIGAN_OK;
}

int b200_pipeline_postprocess(const float* y, uint8_t* image, const uint8_t* mask, int H, int W, const int* box, int res,
                              const float* k25, void* scratch, size_t scratch_bytes, void* stream) {
    if (!y || !image || !mask || !k25 || !scratch) return fail(MIGAN_ERR_INVALID, "pipeline_postprocess: null argument");
    if (int rc = check_box("pipeline_postprocess", H, W, box)) return rc;
    if (res < 1) return fail(MIGAN_ERR_INVALID, "pipeline_postprocess: bad resolution %d", res);
    if (scratch_bytes < migan::pipeline_scratch_bytes(H, W, res))
        return fail(MIGAN_ERR_WORKSPACE, "pipeline_postprocess: scratch of %zu bytes, need %zu", scratch_bytes, migan::pipeline_scratch_bytes(H, W, res));
    CUDA_TRY((cudaError_t)migan::launch_pipeline_postprocess(y, image, mask, H, W, box, res, k25, scratch, static_cast<cudaStream_t>(stream)));
    return MIGAN_OK;
}

static int check_batch(const char* who, const migan_pipe_req* reqs, int n, int res, const void* scratch, size_t scratch_bytes) {
    if (!reqs || !scratch) return fail(MIGAN_ERR_INVALID, "%s: null argument", who);
    if (n < 1 || n > MIGAN_PIPE_BATCH_MAX) return fail(MIGAN_ERR_INVALID, "%s: %d requests (1 to %d per call)", who, n, MIGAN_PIPE_BATCH_MAX);
    if (res < 3) return fail(MIGAN_ERR_INVALID, "%s: bad resolution %d", who, res);
    for (int i = 0; i < n; ++i) {
        const migan_pipe_req& q = reqs[i];
        if (!q.image_chw || !q.mask_hw) return fail(MIGAN_ERR_INVALID, "%s: request %d: null image or mask", who, i);
        if (q.H < 3 || q.W < 3 || q.mask_h < 1 || q.mask_w < 1 || (int64_t)q.H * q.W >= ((int64_t)1 << 31))
            return fail(MIGAN_ERR_INVALID, "%s: request %d: image %d x %d (at least 3 x 3, under 2^31 pixels), mask %d x %d", who, i,
                        q.H, q.W, q.mask_h, q.mask_w);
    }
    if (reinterpret_cast<uintptr_t>(scratch) % 16) return fail(MIGAN_ERR_WORKSPACE, "%s: scratch is not 16-byte aligned", who);
    const size_t need = migan::pipeline_batch_scratch_bytes(reqs, n, res);
    if (scratch_bytes < need) return fail(MIGAN_ERR_WORKSPACE, "%s: scratch of %zu bytes, need %zu", who, scratch_bytes, need);
    return MIGAN_OK;
}

size_t b200_pipeline_batch_scratch_bytes(const migan_pipe_req* reqs, int n, int res) {
    if (!reqs || n < 1 || n > MIGAN_PIPE_BATCH_MAX || res < 1) return 0;
    return migan::pipeline_batch_scratch_bytes(reqs, n, res);
}

int b200_pipeline_batch_boxes(const migan_pipe_req* reqs, int n, int res, int padding, int* boxes, void* scratch, size_t scratch_bytes,
                              void* stream) {
    if (int rc = check_batch("pipeline_batch_boxes", reqs, n, res, scratch, scratch_bytes)) return rc;
    if (!boxes || padding < 0) return fail(MIGAN_ERR_INVALID, "pipeline_batch_boxes: null boxes or padding %d < 0", padding);
    CUDA_TRY((cudaError_t)migan::launch_pipeline_batch_boxes(reqs, n, res, padding, boxes, scratch, static_cast<cudaStream_t>(stream)));
    return MIGAN_OK;
}

int b200_pipeline_batch_preprocess(const migan_pipe_req* reqs, int n, int res, const int* boxes, float* x, void* scratch,
                                   size_t scratch_bytes, void* stream) {
    if (int rc = check_batch("pipeline_batch_preprocess", reqs, n, res, scratch, scratch_bytes)) return rc;
    if (!boxes || !x) return fail(MIGAN_ERR_INVALID, "pipeline_batch_preprocess: null argument");
    CUDA_TRY((cudaError_t)migan::launch_pipeline_batch_preprocess(reqs, n, res, boxes, x, scratch, static_cast<cudaStream_t>(stream)));
    return MIGAN_OK;
}

int b200_pipeline_batch_postprocess(const float* y, const migan_pipe_req* reqs, int n, int res, const int* boxes, const float* k25,
                                    void* scratch, size_t scratch_bytes, void* stream) {
    if (int rc = check_batch("pipeline_batch_postprocess", reqs, n, res, scratch, scratch_bytes)) return rc;
    if (!y || !boxes || !k25) return fail(MIGAN_ERR_INVALID, "pipeline_batch_postprocess: null argument");
    CUDA_TRY((cudaError_t)migan::launch_pipeline_batch_postprocess(y, reqs, n, res, boxes, k25, scratch, static_cast<cudaStream_t>(stream)));
    return MIGAN_OK;
}

int migan_host_wait(migan_ctx* ctx) {
    if (!ctx) return fail(MIGAN_ERR_INVALID, "null ctx");
    if (!ctx->s_out) return MIGAN_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    CUDA_TRY(cudaStreamSynchronize(ctx->s_out));
    return MIGAN_OK;
}

int migan_last_launch_count(const migan_ctx* ctx) { return ctx ? ctx->last_launches : 0; }

int migan_set_tap(migan_ctx* ctx, const char* name, float* dst) {
    if (!ctx) return fail(MIGAN_ERR_INVALID, "null ctx");
    if (!name) { ctx->tap_name.clear(); ctx->tap_dst = nullptr; return MIGAN_OK; }
    ctx->tap_name = name;
    ctx->tap_dst = dst;
    return MIGAN_OK;
}

int migan_tap_info(const migan_ctx* ctx, int path, int index, const char** name, int shape[3]) {
    if (!ctx) return fail(MIGAN_ERR_INVALID, "null ctx");
    // Build a throw-away plan for n = 1 on a fake base (no kernels are launched; tc plans need
    // finalized weights only for pointers, which are not dereferenced here).
    migan_ctx* mctx = const_cast<migan_ctx*>(ctx);
    auto& cache = mctx->tap_cache;
    if (mctx->tap_cache_path != path) {
        // Build a throw-away plan for n = 1 on a fake base address (nothing is launched; tensor maps are
        // only encoded, never dereferenced).
        PlanBuilder pb;
        pb.c = const_cast<migan_ctx*>(ctx); pb.n = 1; pb.path = path;
        pb.base = reinterpret_cast<unsigned char*>(uintptr_t(1) << 30);
        int rc = pb.build();
        if (rc) return rc;
        cache.clear();
        for (Step& s : pb.steps) {
            if (!s.tap.empty()) cache.push_back({s.tap, {s.tapC, s.tapH, s.tapW}});
            if (!s.tap2.empty()) cache.push_back({s.tap2, {s.tap2C, s.tap2H, s.tap2W}});
        }
        mctx->tap_cache_path = path;
    }
    if (index < 0 || index >= (int)cache.size()) return MIGAN_ERR_INVALID;
    if (name) *name = cache[index].first.c_str();
    if (shape) { shape[0] = cache[index].second[0]; shape[1] = cache[index].second[1]; shape[2] = cache[index].second[2]; }
    return MIGAN_OK;
}

int migan_debug_tc_timeout(int device) { return migan::sepconv_tc_timeout_record(device); }

int b200_upfirdn2d(const float* x, const float* f, float* y, int n, int c, int h, int w, int fh, int fw,
                   int upx, int upy, int downx, int downy, int padx0, int padx1, int pady0, int pady1,
                   int flip_filter, float gain, void* stream) {
    if (!x || !y) return fail(MIGAN_ERR_INVALID, "null tensor");
    if (n < 0 || c < 0 || h < 1 || w < 1) return fail(MIGAN_ERR_INVALID, "bad input shape [%d,%d,%d,%d]", n, c, h, w);
    if (upx < 1 || upy < 1 || downx < 1 || downy < 1) return fail(MIGAN_ERR_INVALID, "up/down factors must be >= 1");
    static const float one = 1.0f;
    static thread_local float* d_one = nullptr;
    if (!f) {
        if (!d_one) {
            CUDA_TRY(cudaMalloc(&d_one, sizeof(float)));
            CUDA_TRY(cudaMemcpy(d_one, &one, sizeof(float), cudaMemcpyHostToDevice));
        }
        f = d_one; fh = 1; fw = 1;
    }
    if (fh < 1 || fw < 1 || fh * fw > 1024) return fail(MIGAN_ERR_INVALID, "filter must have 1..1024 taps, got %dx%d", fh, fw);
    const int ow = (w * upx + padx0 + padx1 - fw + downx) / downx;  // upfirdn2d.cpp:32-33
    const int oh = (h * upy + pady0 + pady1 - fh + downy) / downy;
    if (ow < 1 || oh < 1) return fail(MIGAN_ERR_INVALID, "output size must be >= 1, got %dx%d", oh, ow);
    cudaError_t e = migan::launch_upfirdn2d(x, f, y, n, c, h, w, fh, fw, upx, upy, downx, downy, padx0, padx1, pady0, pady1,
                                            flip_filter, gain, oh, ow, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(MIGAN_ERR_CUDA, "upfirdn2d launch failed: %s", cudaGetErrorString(e));
    return MIGAN_OK;
}

int b200_conv1x1_nhwc(const float* x, const float* w_t, float* y, int64_t pixels, int cin, int cout, void* stream) {
    if (pixels < 0 || (pixels > 0 && (!x || !w_t || !y))) return fail(MIGAN_ERR_INVALID, "null tensor");
    if (cin % 16 != 0 || cout % 64 != 0 || cin < 16 || cout < 64)
        return fail(MIGAN_ERR_INVALID, "conv1x1: cin must be a multiple of 16 and cout of 64, got %d -> %d", cin, cout);
    if (pixels == 0) return MIGAN_OK;
    cudaError_t e = migan::launch_pw_gemm_simt(x, w_t, y, pixels, cin, cout, nullptr, 1, 0, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(MIGAN_ERR_CUDA, "conv1x1 launch failed: %s", cudaGetErrorString(e));
    return MIGAN_OK;
}

int b200_bias_act(const float* x, const float* b, float* y, int64_t numel, int64_t step_b, int size_b,
                  int act, float alpha, float gain, float clamp, void* stream) {
    if (numel < 0 || (numel > 0 && (!x || !y))) return fail(MIGAN_ERR_INVALID, "null tensor");
    if (act < 1 || act > 9) return fail(MIGAN_ERR_INVALID, "act must be in 1..9, got %d", act);
    if (b && (step_b < 1 || size_b < 1)) return fail(MIGAN_ERR_INVALID, "bad bias stride/size");
    cudaError_t e = migan::launch_bias_act(x, b, y, numel, step_b, size_b, act, alpha, gain, clamp, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(MIGAN_ERR_CUDA, "bias_act launch failed: %s", cudaGetErrorString(e));
    return MIGAN_OK;
}

}  // extern "C"
