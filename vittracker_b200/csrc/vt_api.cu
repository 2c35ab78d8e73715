// C-ABI layer of libvittrack_b200.so: handle, weight ingestion (power-of-two rebalancing of scale between layers, BN folding into the
// fp32 layouts; each tensor-core weight blob is packed by the file of the kernel that reads it),
// workspace, and the entry points declared in include/vittrack_b200.h.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <omp.h>
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "../../include/vittrack_b200.h"
#include "vt_internal.h"

using namespace vt;
static_assert(vt::VT_TRACK_NUMERIC_RANGE_ == VT_TRACK_NUMERIC_RANGE, "status code shared with the kernels");
static_assert(vt::VT_TRACK_BAD_SLOT_ == VT_TRACK_BAD_SLOT, "status code shared with the kernels");
static_assert(vt::kNz * 4 == 256 && VT_TRACK_RECORD_HEADER_BYTES % 16 == 0, "record layout: 64 + 256 C bytes, 16-byte vectors");

namespace {

thread_local std::string g_create_error;

struct HostTensor {
    std::vector<float> data;
    std::vector<int64_t> shape;
};
using TensorMap = std::map<std::string, HostTensor>;

}  // namespace

struct VtContext {
    VtConfig cfg;
    std::string err;
    TensorMap tensors;
    bool finalized = false;
    bool tracks_ready = false;
    int score_terms = 1;              // split terms of the tensor-core blocks' q k^T (vt_finalize_weights: score_terms)
    uint64_t fingerprint = 0;         // of the weights finalised last (vt_weights_fingerprint)
    int64_t launches = 0;

    float* d_weights = nullptr;       // packed model
    size_t weights_floats = 0;
    ModelW mw{};

    int chunk = 0;
    int num_sms = 148;
    // chunk workspace
    float* d_scratch = nullptr;       // stem intermediates (fp32 NCHW)
    void* d_taps = nullptr;           // per-track tap tables of the fused crop gather
    uint8_t* d_planes = nullptr;      // tensor-core operand images of conv3 / conv4 (zero rows must stay zero); null in SIMT mode
    float* d_tokz = nullptr;          // [chunk][64][48]   (vt_forward only)
    float* d_tokx = nullptr;          // [max_tracks][256][48]
    float* d_tok = nullptr;           // [max_tracks][320][48]
    // per-track state
    double* d_state = nullptr;        // [max_tracks][4]
    float* d_tmpl = nullptr;          // [max_tracks][64][48] cached template tokens (+pos)
    int32_t* d_status = nullptr;      // [max_tracks] crop status of the current call (by track for a range call, by item for a slot list)
    uint32_t* d_claim = nullptr;      // [max_tracks] slot-list deduplication (vt_slots.cu), all 0xffffffff between calls
    int32_t* d_eff = nullptr;         // [max_tracks] effective slot per item of the current slot-list call
    float* d_maps = nullptr;          // [max_tracks][1280] score | size | offset of the last step
    int32_t* d_surf_rect = nullptr;   // [max_tracks][4] bounding rectangle per surface (vt_yuv420_crops_to_surface_rgb), empty between calls
    uint32_t* d_surf_done = nullptr;  // [max_tracks] conversion CTAs of the surface counted in, 0 between calls
    int last_first = 0, last_n = 0;
    // range fallback (vt_set_range_fallback): the flagged items of a tensor-core step, recomputed on the fp32 kernels
    bool fallback = false;
    int64_t* fallback_counter = nullptr;  // the caller's device counter (nullable)
    void* d_fallback = nullptr;           // every array of `fb`, one allocation
    RangeFallback fb{};
    // generic-configuration path (every configuration other than vit_48_h32; vt_generic.cu)
    bool generic = false;
    GenModelW gw{};
    GenWork gws{};
    float* d_gwork = nullptr;
    // optional per-stage timing (vt_profile_*)
    struct ProfRec { int stage; int items; cudaEvent_t a, b; };
    bool profiling = false;
    std::vector<ProfRec> prof;
    std::vector<cudaEvent_t> evpool;
};

namespace {

int fail(VtHandle h, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h) h->err = buf; else g_create_error = buf;
    return code;
}

#define VT_CUDA(h, expr)                                                                         \
    do {                                                                                         \
        cudaError_t e__ = (expr);                                                                \
        if (e__ != cudaSuccess) return fail(h, VT_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(e__)); \
    } while (0)

const char* kTowers[3] = {"ctr", "offset", "size"};
std::string stem_prefix(int l) { return "patch_embed.net." + std::to_string(2 * l) + "."; }
std::string head_prefix(int layer, int tower) { return "box_head.conv" + std::to_string(layer + 1) + "_" + kTowers[tower] + "."; }

// Every tensor of the reference's state_dict for configuration c: name -> shape.  tracker.output_window is optional (the window is
// computed when the tracker's own tensor was not handed over).
std::map<std::string, std::vector<int64_t>> tensor_table(const VtConfig& c) {
    const int64_t C = c.embed_dim, hc = c.head_channels, hid = (int64_t)c.mlp_ratio * C;
    std::map<std::string, std::vector<int64_t>> t;
    t["pos_embed_z"] = {1, 64, C};
    t["pos_embed_x"] = {1, 256, C};
    t["norm.weight"] = {C};
    t["norm.bias"] = {C};
    t["tracker.output_window"] = {1, 1, 16, 16};
    const int64_t ch[5] = {3, C / 8, C / 4, C / 2, C};
    for (int l = 0; l < 4; ++l) {
        const std::string p = stem_prefix(l);
        t[p + "c.weight"] = {ch[l + 1], ch[l], 3, 3};
        for (const char* leaf : {"bn.weight", "bn.bias", "bn.running_mean", "bn.running_var"}) t[p + leaf] = {ch[l + 1]};
    }
    for (int b = 0; b < c.depth; ++b) {
        const std::string p = "blocks." + std::to_string(b) + ".";
        for (const char* leaf : {"norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias", "attn.proj.bias", "mlp.fc2.bias"}) t[p + leaf] = {C};
        t[p + "attn.qkv.weight"] = {3 * C, C};
        t[p + "attn.qkv.bias"] = {3 * C};
        t[p + "attn.proj.weight"] = {C, C};
        t[p + "mlp.fc1.weight"] = {hid, C};
        t[p + "mlp.fc1.bias"] = {hid};
        t[p + "mlp.fc2.weight"] = {C, hid};
    }
    const int64_t hch[5] = {C, hc, hc / 2, hc / 4, hc / 8}, outs[3] = {1, 2, 2};
    for (int k = 0; k < 3; ++k) {
        for (int i = 0; i < 4; ++i) {
            const std::string p = head_prefix(i, k);
            t[p + "0.weight"] = {hch[i + 1], hch[i], 3, 3};
            for (const char* leaf : {"0.bias", "1.weight", "1.bias", "1.running_mean", "1.running_var"}) t[p + leaf] = {hch[i + 1]};
        }
        const std::string p = std::string("box_head.conv5_") + kTowers[k] + ".";
        t[p + "weight"] = {outs[k], hch[4], 1, 1};
        t[p + "bias"] = {outs[k]};
    }
    return t;
}

// First step of finalisation: every tensor of the table that is not optional must have been set.  Past it, every lookup succeeds.
int check_missing(VtHandle h) {
    std::string missing;
    for (const auto& e : tensor_table(h->cfg))
        if (e.first != "tracker.output_window" && !h->tensors.count(e.first) && missing.size() < 300) missing += e.first + " ";
    return missing.empty() ? VT_OK : fail(h, VT_ERR_WEIGHTS, "missing tensors: %s", missing.c_str());
}

const float* tensor(const TensorMap& ts, const std::string& name) { return ts.at(name).data.data(); }

BlockTensors block_tensors(const TensorMap& ts, int b) {
    const std::string p = "blocks." + std::to_string(b) + ".";
    return {tensor(ts, p + "norm1.weight"), tensor(ts, p + "norm1.bias"), tensor(ts, p + "attn.qkv.weight"), tensor(ts, p + "attn.qkv.bias"),
            tensor(ts, p + "attn.proj.weight"), tensor(ts, p + "attn.proj.bias"), tensor(ts, p + "norm2.weight"), tensor(ts, p + "norm2.bias"),
            tensor(ts, p + "mlp.fc1.weight"), tensor(ts, p + "mlp.fc1.bias"), tensor(ts, p + "mlp.fc2.weight"), tensor(ts, p + "mlp.fc2.bias")};
}

// Conv2d (with its bias when `conv_bias`) and BatchNorm2d (eval) folded in float64 (Conv2d_BN.fuse vit_dist.py:22-33; head conv + bias
// -> BN, head.py:16-21): w [co][ci][3][3] in the conv's order, b [co]; co and ci are the conv weight's stored shape.
struct FoldedConv {
    int co, ci;
    std::vector<float> w, b;
};
FoldedConv fold_conv_bn(const TensorMap& ts, const std::string& conv, const std::string& bn, bool conv_bias) {
    const HostTensor& wt = ts.at(conv + "weight");
    const float *w = wt.data.data(), *cb = conv_bias ? tensor(ts, conv + "bias") : nullptr;
    const float *g = tensor(ts, bn + "weight"), *b = tensor(ts, bn + "bias"), *m = tensor(ts, bn + "running_mean"), *v = tensor(ts, bn + "running_var");
    FoldedConv f{(int)wt.shape[0], (int)wt.shape[1], std::vector<float>(wt.data.size()), std::vector<float>(wt.shape[0])};
    const size_t kn = wt.data.size() / f.co;                                  // ci * 9 weights per output channel
    for (int co = 0; co < f.co; ++co) {
        const double s = (double)g[co] / sqrt((double)v[co] + 1e-5);         // BatchNorm2d's default eps
        f.b[co] = (float)(((cb ? (double)cb[co] : 0.0) - (double)m[co]) * s + (double)b[co]);
        for (size_t k = 0; k < kn; ++k) f.w[co * kn + k] = (float)((double)w[co * kn + k] * s);
    }
    return f;
}

// Nearest integer to log2(v / unit), as v's exponent plus a function of its mantissa alone: octave(v * 2^k, unit) == octave(v, unit) + k
// exactly.  0 for a v that is zero or not finite.
int octave(double v, double unit) {
    if (!(v > 0.0) || !std::isfinite(v)) return 0;
    int e = 0;
    const double m = frexp(v, &e);
    return e + (int)lround(log2(m / unit));
}

// Power-of-two rebalancing of the model's scale, on the copy of the tensors that finalisation packs.  A checkpoint may split scale freely
// between a LayerNorm or BatchNorm affine and the next layer's weights, between the q and k rows of a block's qkv, or between its v rows
// and the output projection: the model is the same, but the tensor-core paths split each operand into fp16 hi + lo, which keeps its
// ~22 bits only while both halves are normal fp16 numbers.  Each producer -> consumer pair below moves 2^-p onto the factor its statistic
// reads and 2^p onto the other, p = octave(statistic): the operands come out near the magnitudes of a random-init model whatever the
// checkpoint's split.  Properties that the tests rely on (tests/test_scale_invariance.py):
// - multiplying by a power of two is exact, and so is the rewrite as a whole: the fp32 layers keep their bits, and no kernel changes;
// - scaling a pair's factors by 2^-k and 2^k shifts its p by exactly k, so the packed weights are the same bits.  For that, each
//   statistic reads only tensors that no other pair rescales (qkv.weight is shared by three pairs: the q / k statistic is a ratio of
//   its rows, which ln1's uniform scale leaves alone);
// - p = 0 for random-init weights, so such a model packs exactly the tensors it was handed.
// Returns the final LayerNorm's p: its output, the tokens_norm tap, is scaled back by 2^p.
int rebalance(const VtConfig& c, TensorMap& ts) {
    const size_t C = c.embed_dim;
    auto amax = [&](const std::string& name, size_t first = 0, size_t count = 0) {
        const std::vector<float>& d = ts.at(name).data;
        double m = 0.0;
        for (size_t i = first, end = count ? first + count : d.size(); i < end; ++i) m = fmax(m, fabs((double)d[i]));
        return m;
    };
    auto scale = [&](const std::string& name, int p, size_t first = 0, size_t count = 0) {
        std::vector<float>& d = ts.at(name).data;
        for (size_t i = first, end = count ? first + count : d.size(); i < end; ++i) d[i] = ldexpf(d[i], p);
    };
    // a LayerNorm / BatchNorm affine (weight and bias): its output is about as large as the larger of the two
    auto affine_to = [&](const std::string& norm, const std::vector<std::string>& consumers) {
        const int p = octave(fmax(amax(norm + "weight"), amax(norm + "bias")), 1.0);
        scale(norm + "weight", -p);
        scale(norm + "bias", -p);
        for (const std::string& w : consumers) scale(w, p);
        return p;
    };
    for (int b = 0; b < c.depth; ++b) {
        const std::string p = "blocks." + std::to_string(b) + ".", qkv = p + "attn.qkv.";
        const int pqk = octave(sqrt(amax(qkv + "weight", 0, C * C) / amax(qkv + "weight", C * C, C * C)), 1.0);
        const int pv = octave(amax(p + "attn.proj.weight"), 1.0 / sqrt((double)C));     // random-init Linear weights: |w| < C^-1/2
        affine_to(p + "norm1.", {qkv + "weight"});
        affine_to(p + "norm2.", {p + "mlp.fc1.weight"});
        scale(qkv + "weight", -pqk, 0, C * C);   scale(qkv + "bias", -pqk, 0, C);
        scale(qkv + "weight", pqk, C * C, C * C); scale(qkv + "bias", pqk, C, C);
        scale(qkv + "weight", pv, 2 * C * C, C * C); scale(qkv + "bias", pv, 2 * C, C);
        scale(p + "attn.proj.weight", -pv);
    }
    std::vector<std::string> conv1;
    for (int t = 0; t < 3; ++t) conv1.push_back(head_prefix(0, t) + "0.weight");
    const int pnorm = affine_to("norm.", conv1);
    for (int t = 0; t < 3; ++t)
        for (int i = 0; i < 4; ++i)
            affine_to(head_prefix(i, t) + "1.", {i < 3 ? head_prefix(i + 1, t) + "0.weight" : std::string("box_head.conv5_") + kTowers[t] + ".weight"});
    return pnorm;
}

// Upper bound on the spectral norm of W [rows][cols]: ||W||_2^2 = lambda_max(W^T W) <= ||(W^T W)^32||_F^(1/32), at most 48^(1/64) ~ 6 %
// above it for a 48-column W.  The powers are taken by squaring, renormalised at every step.
double spectral_norm_bound(const float* W, int rows, int cols) {
    std::vector<double> m((size_t)cols * cols, 0.0), t(m.size());
    for (int r = 0; r < rows; ++r)
        for (int i = 0; i < cols; ++i)
            for (int j = 0; j < cols; ++j) m[(size_t)i * cols + j] += (double)W[(size_t)r * cols + i] * W[(size_t)r * cols + j];
    auto frob = [&]() { double s = 0.0; for (double v : m) s += v * v; return sqrt(s); };
    double log_scale = 0.0;                       // (W^T W)^(2^s) = m * exp(log_scale)
    for (int s = 0; s < 5; ++s) {
        const double f = frob();
        if (!(f > 0.0) || !std::isfinite(f)) return f > 0.0 ? INFINITY : 0.0;
        for (double& v : m) v /= f;
        for (int i = 0; i < cols; ++i)
            for (int j = 0; j < cols; ++j) {
                double a = 0.0;
                for (int k = 0; k < cols; ++k) a += m[(size_t)i * cols + k] * m[(size_t)k * cols + j];
                t[(size_t)i * cols + j] = a;
            }
        m.swap(t);
        log_scale = 2.0 * (log_scale + log(f));
    }
    return exp((log(frob()) + log_scale) / 64.0);
}

// Split terms of the tensor-core blocks' scores q k^T (vt_block_tc.cu: kScoresTerms).  The single pass rounds q and k to fp16, so its
// error grows with |q||k|.  Each block bounds |q . k| / sqrt(C) from its weights alone: norm1's output has norm at most
// R = sqrt(C) max|gamma| + ||beta||, so |q| <= ||W_q||_2 R + ||b_q|| and |k| likewise.  Random-init weights stay below 20
// (tests/test_trained_weights.py); above kSharpScores the handle takes the three-term pass whatever blocks_impl asked for.
constexpr double kSharpScores = 512.0;

int score_terms(const VtConfig& c, const TensorMap& ts) {
    if (c.blocks_impl == VT_BLOCKS_TCGEN05_3TERM) return 3;
    const size_t C = c.embed_dim;
    for (int b = 0; b < c.depth; ++b) {
        const std::string p = "blocks." + std::to_string(b) + ".";
        const std::vector<float>& g = ts.at(p + "norm1.weight").data;
        const std::vector<float>& be = ts.at(p + "norm1.bias").data;
        const std::vector<float>& w = ts.at(p + "attn.qkv.weight").data;
        const std::vector<float>& bias = ts.at(p + "attn.qkv.bias").data;
        double gmax = 0.0, bn = 0.0, bq = 0.0, bk = 0.0;
        for (size_t i = 0; i < C; ++i) {
            gmax = fmax(gmax, fabs((double)g[i]));
            bn += (double)be[i] * be[i];
            bq += (double)bias[i] * bias[i];
            bk += (double)bias[C + i] * bias[C + i];
        }
        const double R = sqrt((double)C) * gmax + sqrt(bn);
        const double q = spectral_norm_bound(w.data(), (int)C, (int)C) * R + sqrt(bq);
        const double k = spectral_norm_bound(w.data() + C * C, (int)C, (int)C) * R + sqrt(bk);
        if (!(q * k / sqrt((double)C) <= kSharpScores)) return 3;
    }
    return 1;
}

// FNV-1a 64 over 8-byte little-endian words of a byte stream, the last word zero-padded (the weights fingerprint of the header).
// Word-wise rather than byte-wise: one multiply per 8 bytes.
struct WordFnv {
    uint64_t h = 0xcbf29ce484222325ull;
    uint8_t tail[8];
    size_t nt = 0;
    void word(uint64_t w) { h = (h ^ w) * 0x100000001b3ull; }
    void bytes(const void* p, size_t n) {
        const uint8_t* b = static_cast<const uint8_t*>(p);
        while (nt && n) { tail[nt++] = *b++; --n; if (nt == 8) { uint64_t w; memcpy(&w, tail, 8); word(w); nt = 0; } }
        for (; n >= 8; b += 8, n -= 8) { uint64_t w; memcpy(&w, b, 8); word(w); }
        while (n) { tail[nt++] = *b++; --n; }
    }
    template <typename T> void put(T v) { bytes(&v, sizeof v); }
    uint64_t finish() {
        if (nt) { memset(tail + nt, 0, 8 - nt); uint64_t w; memcpy(&w, tail, 8); word(w); nt = 0; }
        return h;
    }
};

// The template route of the fingerprint: which kernels compute a handle's template tokens.  vit_48_h32 crops and runs the template stem
// on the fp32 CUDA-core kernels for every blocks_impl (launch_crop_stem takes the tensor-core branch for the search crop only); the
// generic stem follows GenModelW's GEMM route.
int32_t template_route(VtHandle h) {
    if (!h->generic) return 0;
    return h->gw.fp32_only ? 1 : h->gw.use_img ? 3 : 2;
}

uint64_t weights_fingerprint(VtHandle h) {
    static const char kVersion[] = "vittrack_b200 weights v1";
    WordFnv f;
    f.bytes(kVersion, sizeof kVersion - 1);
    const VtConfig& c = h->cfg;
    for (int32_t v : {c.embed_dim, c.num_heads, c.depth, c.mlp_ratio, c.head_channels, c.stride, c.template_size, c.search_size}) f.put(v);
    f.put(c.template_factor);
    f.put(c.search_factor);
    f.put(template_route(h));
    for (const auto& e : h->tensors) {                 // std::map: ascending byte-wise name order
        f.bytes(e.first.c_str(), e.first.size() + 1);
        f.put((int32_t)e.second.shape.size());
        for (int64_t d : e.second.shape) f.put(d);
        f.bytes(e.second.data.data(), e.second.data.size() * sizeof(float));
    }
    return f.finish();
}

// The packed weights: one fp32 buffer of 16-byte aligned slots.  slot() allocates one for the ModelW / GenModelW member that will
// point at it and returns its host offset; upload_weights() points every such member into the device buffer.
struct Packer {
    std::vector<float> buf;
    std::vector<std::pair<const float**, size_t>> fslots;
    std::vector<std::pair<const uint8_t**, size_t>> bslots;
    size_t alloc(size_t n) {
        const size_t off = buf.size();
        buf.resize(off + (n + 3) / 4 * 4, 0.f);
        return off;
    }
    size_t slot(const float*& member, size_t n) { fslots.push_back({&member, alloc(n)}); return fslots.back().second; }
    size_t slot(const uint8_t*& member, size_t n) { bslots.push_back({&member, alloc(n)}); return bslots.back().second; }
    size_t put(const float*& member, const float* src, size_t n) {
        const size_t o = slot(member, n);
        memcpy(&buf[o], src, n * sizeof(float));
        return o;
    }
    uint8_t* bytes(size_t o) { return reinterpret_cast<uint8_t*>(&buf[o]); }
};

// The packed weights -> h->d_weights (reallocated when it has grown), then every slot's member -> its place there; returns once the
// copy is done, as pk is the caller's local
int upload_weights(VtHandle h, const Packer& pk, cudaStream_t st) {
    if (h->d_weights && h->weights_floats < pk.buf.size()) { cudaFree(h->d_weights); h->d_weights = nullptr; }
    if (!h->d_weights) {
        VT_CUDA(h, cudaMalloc((void**)&h->d_weights, pk.buf.size() * sizeof(float)));
        h->weights_floats = pk.buf.size();
    }
    VT_CUDA(h, cudaMemcpyAsync(h->d_weights, pk.buf.data(), pk.buf.size() * sizeof(float), cudaMemcpyHostToDevice, st));
    VT_CUDA(h, cudaStreamSynchronize(st));
    for (const auto& e : pk.fslots) *e.first = h->d_weights + e.second;
    for (const auto& e : pk.bslots) *e.first = reinterpret_cast<const uint8_t*>(h->d_weights + e.second);
    return VT_OK;
}

void free_all(VtHandle h) {
    for (auto& r : h->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    for (auto e : h->evpool) cudaEventDestroy(e);
    cudaFree(h->d_weights); cudaFree(h->d_planes); cudaFree(h->d_scratch); cudaFree(h->d_taps); cudaFree(h->d_tokz);
    cudaFree(h->d_tokx); cudaFree(h->d_tok); cudaFree(h->d_state); cudaFree(h->d_tmpl);
    cudaFree(h->d_status); cudaFree(h->d_claim); cudaFree(h->d_eff); cudaFree(h->d_maps); cudaFree(h->d_gwork); cudaFree(h->d_fallback);
    cudaFree(h->d_surf_rect); cudaFree(h->d_surf_done);
}

int check_ready(VtHandle h, bool need_tracks) {
    if (!h) return VT_ERR_INVALID_ARG;
    if (!h->finalized) return fail(h, VT_ERR_STATE, "weights not finalised: call vt_set_tensor for every tensor, then vt_finalize_weights");
    if (need_tracks && !h->tracks_ready) return fail(h, VT_ERR_STATE, "tracks not initialised: call vt_tracks_init first");
    return VT_OK;
}

// Tracks [first, first + n) lie in [lo, lo + count): no intermediate overflows, whatever int32 values a caller passes.
bool tracks_in(int first, int n, int lo, int count) { return n >= 0 && first >= lo && first - lo <= count - n; }

int check_tracks(VtHandle h, const char* where, int first, int n) {
    if (tracks_in(first, n, 0, h->cfg.max_tracks)) return VT_OK;
    return fail(h, VT_ERR_INVALID_ARG, "%s: tracks [%d, %lld) exceed max_tracks %d", where, first, (long long)first + n, h->cfg.max_tracks);
}

int check_yuv_format(VtHandle h, const char* where, int format) {
    if (format == VT_FRAME_NV12 || format == VT_FRAME_I420) return VT_OK;
    return fail(h, VT_ERR_INVALID_ARG, "%s: unknown format %d", where, format);
}

// The checks every entry point that enqueues work starts with, in this order: a null handle; readiness (`need`); n < 0, or with
// `range` tracks [first, first + n) outside max_tracks (a slot list passes first = 0); an empty batch, a successful no-op whose
// pointers may be null (kEmpty); a null `required` pointer.  VT_ENTER returns on anything but VT_OK.
enum Need { kHandle, kWeights, kTracks };
constexpr int kEmpty = 1;
int enter(VtHandle h, const char* where, Need need, int first, int n, bool range, std::initializer_list<const void*> required) {
    if (!h) return VT_ERR_INVALID_ARG;
    if (need != kHandle)
        if (const int rc = check_ready(h, need == kTracks)) return rc;
    if (range) {
        if (const int rc = check_tracks(h, where, first, n)) return rc;
    } else if (n < 0) {
        return fail(h, VT_ERR_INVALID_ARG, "%s: negative n", where);
    }
    if (n == 0) return kEmpty;
    for (const void* p : required)
        if (!p) return fail(h, VT_ERR_INVALID_ARG, "%s: null pointer", where);
    return VT_OK;
}

// Returns the prologue's status, or VT_OK for an empty batch; past it the handle's device is current until the entry point returns.
#define VT_ENTER(h, prologue)                                           \
    if (const int rc__ = (prologue)) return rc__ == kEmpty ? VT_OK : rc__; \
    DeviceGuard dg__((h)->cfg.device);                                  \
    VT_CUDA(h, dg__.err)

int launch_fail(VtHandle h, int k, const char* where) {
    if (k == -2) return fail(h, VT_ERR_UNSUPPORTED, "%s: blocks_impl %d is not available in this build", where, h->cfg.blocks_impl);
    return fail(h, VT_ERR_CUDA, "%s: kernel launch failed: %s", where, cudaGetErrorString(cudaGetLastError()));
}

cudaEvent_t get_event(VtHandle h) {
    if (!h->evpool.empty()) { cudaEvent_t e = h->evpool.back(); h->evpool.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}

// Launch one pipeline stage; when profiling is on, bracket it with events on the launching stream.  kNoStage: the slot-list
// bookkeeping of vt_slots.cu, counted as launches but not as a stage, so that a stage's items stay the number of tracks it processed.
constexpr int kNoStage = -1;
#define VT_LAUNCH(h, stage, items, st, where, expr)                               \
    do {                                                                          \
        const bool prof__ = (h)->profiling && (stage) >= 0;                       \
        cudaEvent_t ea__ = nullptr, eb__ = nullptr;                               \
        if (prof__) { ea__ = get_event(h); eb__ = get_event(h); cudaEventRecord(ea__, st); } \
        const int k__ = (expr);                                                   \
        if (k__ < 0) return launch_fail(h, k__, where);                           \
        (h)->launches += k__;                                                     \
        if (prof__) { cudaEventRecord(eb__, st); (h)->prof.push_back({stage, items, ea__, eb__}); } \
    } while (0)

int run_blocks(VtHandle h, const float* tokz, int zs, const int32_t* zslots, const float* tokx, int xs, float* out, int n, float* taps,
               size_t tap_stride, cudaStream_t st) {
    if (h->cfg.blocks_impl == VT_BLOCKS_SIMT_FP32)
        return launch_blocks_simt(tokz, zs, zslots, tokx, xs, out, n, h->mw, taps, tap_stride, st);
    return launch_blocks_tc(tokz, zs, zslots, tokx, xs, out, n, h->mw, taps, tap_stride, h->num_sms, h->score_terms, st);
}


// HeadArgs of a forward pass over rows [first, first + m) of the caller's output arrays (each nullable)
HeadArgs forward_head_args(int first, int m, float* pred_boxes, float* score_map, float* size_map, float* offset_map) {
    HeadArgs a{};
    a.n = m;
    a.pred_boxes = pred_boxes ? pred_boxes + (size_t)first * 4 : nullptr;
    a.score_map = score_map ? score_map + (size_t)first * 256 : nullptr;
    a.size_map = size_map ? size_map + (size_t)first * 512 : nullptr;
    a.offset_map = offset_map ? offset_map + (size_t)first * 512 : nullptr;
    return a;
}

// The maps of the last tracking step from track `first` on: kept planar per array, score [max_tracks][256] | size [max_tracks][512] |
// offset [max_tracks][512]
struct LastMaps { float *score, *size, *offset; };
LastMaps last_maps(VtHandle h, int first) {
    const size_t mt = h->cfg.max_tracks;
    return {h->d_maps + (size_t)first * 256, h->d_maps + mt * 256 + (size_t)first * 512, h->d_maps + mt * 768 + (size_t)first * 512};
}

// HeadArgs of a tracking step over items [c0, c0 + m); frame_hw, out_boxes and out_detail are the step's arrays.  Range step
// (slots == NULL): item i is track first + i.  Slot list (first == 0): item i is track slots[i]; maps and status stay by item.
HeadArgs track_head_args(VtHandle h, int first, const int32_t* slots, int c0, int m, const int32_t* frame_hw, double* out_boxes,
                         double* out_detail, int update_state) {
    const int t0 = first + c0;
    const LastMaps maps = last_maps(h, t0);
    HeadArgs a{};
    a.n = m;
    a.score_map = maps.score; a.size_map = maps.size; a.offset_map = maps.offset;
    a.state = h->d_state + (size_t)(slots ? 0 : t0) * 4;
    a.slots = slots ? slots + c0 : nullptr;
    a.frame_hw = frame_hw + 2 * c0;
    a.status = h->d_status + t0;
    a.out_boxes = out_boxes + (size_t)c0 * 5;
    a.out_detail = out_detail ? out_detail + (size_t)c0 * 8 : nullptr;
    a.update_state = update_state;
    a.search_factor = h->cfg.search_factor;
    return a;
}

// Hann window (hann.py:6-16; the tracker's own tensor when it was handed over) and normalisation table (data_utils.py:8-14)
void fill_hann_and_lut(const TensorMap& ts, float* hann, float* lut) {
    auto it = ts.find("tracker.output_window");
    if (it != ts.end()) {
        memcpy(hann, it->second.data.data(), 256 * sizeof(float));
    } else {
        float w1[16];
        const float step = (float)(2.0 * M_PI / 17.0);
        for (int k = 0; k < 16; ++k) w1[k] = 0.5f * (1.f - cosf(step * (float)(k + 1)));
        for (int y = 0; y < 16; ++y)
            for (int x = 0; x < 16; ++x) hann[y * 16 + x] = w1[y] * w1[x];
    }
    const float mean[3] = {0.485f, 0.456f, 0.406f}, stdv[3] = {0.229f, 0.224f, 0.225f};
    for (int c = 0; c < 3; ++c)
        for (int v = 0; v < 256; ++v) {
            volatile float a = (float)v / 255.0f;        // (x / 255.0) - mean) / std, each step rounded to fp32
            volatile float d = a - mean[c];
            volatile float r = d / stdv[c];
            lut[c * 256 + v] = r;
        }
}

// Weights of the generic path: the reference's own layouts ([out][in]; conv [cout][ky][kx][cin]) with BatchNorm(eval) folded.
int finalize_generic(VtHandle h, const TensorMap& ts, int pnorm, cudaStream_t st) {
    const int C = h->cfg.embed_dim, hc = h->cfg.head_channels, hid = h->cfg.mlp_ratio * C;
    GenModelW& g = h->gw;
    g.norm_tap_scale = ldexpf(1.f, pnorm);
    Packer pk;
    // split images of the folded convolutions whose K = 9 cin is a whole number of 32-wide panels, packed after the fp32 weights
    struct ConvImg { const uint8_t** img; size_t w; int co, ci; };
    std::vector<ConvImg> imgs;
    auto want_img = [&](const uint8_t*& img, size_t w, int co, int ci) { if (g.use_img && ci % 32 == 0) imgs.push_back({&img, w, co, ci}); };
    auto conv_rows = [&](const FoldedConv& f, size_t ow, size_t ob) {          // -> [co][(ky, kx, ci)] at ow, bias at ob
        for (int co = 0; co < f.co; ++co) {
            pk.buf[ob + co] = f.b[co];
            for (int ci = 0; ci < f.ci; ++ci)
                for (int k = 0; k < 9; ++k) pk.buf[ow + ((size_t)co * 9 + k) * f.ci + ci] = f.w[((size_t)co * f.ci + ci) * 9 + k];
        }
    };
    for (int l = 0; l < 4; ++l) {
        const FoldedConv f = fold_conv_bn(ts, stem_prefix(l) + "c.", stem_prefix(l) + "bn.", false);
        const size_t ow = pk.slot(g.stem_w[l], f.w.size()), ob = pk.slot(g.stem_b[l], f.co);
        conv_rows(f, ow, ob);
        want_img(g.istem_w[l], ow, f.co, f.ci);
    }
    for (int b = 0; b < h->cfg.depth; ++b) {
        const BlockTensors t = block_tensors(ts, b);
        GenBlockW& B = g.blk[b];
        pk.put(B.ln1g, t.ln1_g, C); pk.put(B.ln1b, t.ln1_b, C);
        pk.put(B.wqkv, t.wqkv, (size_t)3 * C * C); pk.put(B.bqkv, t.bqkv, (size_t)3 * C);
        pk.put(B.wproj, t.wproj, (size_t)C * C); pk.put(B.bproj, t.bproj, C);
        pk.put(B.ln2g, t.ln2_g, C); pk.put(B.ln2b, t.ln2_b, C);
        pk.put(B.wfc1, t.wfc1, (size_t)hid * C); pk.put(B.bfc1, t.bfc1, hid);
        pk.put(B.wfc2, t.wfc2, (size_t)C * hid); pk.put(B.bfc2, t.bfc2, C);
    }
    // split images of the blocks' Linear weights for the bulk-copy GEMM (same bytes as the fp32 matrices)
    for (int b = 0; b < h->cfg.depth && g.use_img; ++b) {
        const BlockTensors t = block_tensors(ts, b);
        GenBlockW& B = g.blk[b];
        const struct { const uint8_t*& img; const float* w; int n, k; } lin[4] = {
            {B.iwqkv, t.wqkv, 3 * C, C}, {B.iwproj, t.wproj, C, C}, {B.iwfc1, t.wfc1, hid, C}, {B.iwfc2, t.wfc2, C, hid}};
        for (const auto& L : lin) {
            const size_t o = pk.slot(L.img, gen_img_bytes(L.n, L.k) / 4);
            gen_pack_weight_image(L.w, L.n, L.k, pk.bytes(o));
        }
    }
    pk.put(g.norm_g, tensor(ts, "norm.weight"), C); pk.put(g.norm_b, tensor(ts, "norm.bias"), C);
    pk.put(g.pos_z, tensor(ts, "pos_embed_z"), (size_t)kNz * C); pk.put(g.pos_x, tensor(ts, "pos_embed_x"), (size_t)kNx * C);
    // head: layer 1 merged over the towers (ctr | offset | size), layers 2-4 per tower, conv5 rows ctr, off x, off y, size w, size h
    const size_t w1 = pk.slot(g.head_w1, (size_t)3 * hc * 9 * C), b1 = pk.slot(g.head_b1, (size_t)3 * hc);
    want_img(g.ihead_w1, w1, 3 * hc, C);
    for (int t = 0; t < 3; ++t)
        for (int i = 0; i < 4; ++i) {
            const FoldedConv f = fold_conv_bn(ts, head_prefix(i, t) + "0.", head_prefix(i, t) + "1.", true);
            if (i == 0) {      // the merged layer's rows of this tower (the tower's own layer-1 slot is not read)
                const size_t ow = pk.alloc(f.w.size()), ob = pk.alloc(f.co);
                conv_rows(f, ow, ob);
                conv_rows(f, w1 + (size_t)t * hc * 9 * C, b1 + (size_t)t * hc);
                continue;
            }
            const size_t ow = pk.slot(g.head_w[t][i - 1], f.w.size()), ob = pk.slot(g.head_b[t][i - 1], f.co);
            conv_rows(f, ow, ob);
            want_img(g.ihead_w[t][i - 1], ow, f.co, f.ci);
        }
    const int c5 = hc / 8, row0[3] = {0, 1, 3}, outs[3] = {1, 2, 2};
    const size_t w5 = pk.slot(g.head_w5, (size_t)5 * c5), b5 = pk.slot(g.head_b5, 5);
    for (int t = 0; t < 3; ++t) {
        const std::string p = std::string("box_head.conv5_") + kTowers[t] + ".";
        const float *w = tensor(ts, p + "weight"), *b = tensor(ts, p + "bias");
        for (int o = 0; o < outs[t]; ++o) {
            pk.buf[b5 + row0[t] + o] = b[o];
            for (int k = 0; k < c5; ++k) pk.buf[w5 + (size_t)(row0[t] + o) * c5 + k] = w[(size_t)o * c5 + k];
        }
    }
    const size_t hann = pk.slot(g.hann, 256), lut = pk.slot(h->mw.lut, 768);         // the crop kernel reads the table through ModelW
    fill_hann_and_lut(ts, &pk.buf[hann], &pk.buf[lut]);
    for (const ConvImg& c : imgs) {
        const size_t o = pk.slot(*c.img, gen_img_bytes(c.co, 9 * c.ci) / 4);       // (allocating moves pk.buf: index, hold no pointer)
        gen_pack_weight_image(&pk.buf[c.w], c.co, 9 * c.ci, pk.bytes(o));
    }
    if (const int rc = upload_weights(h, pk, st)) return rc;
    h->finalized = true;
    return VT_OK;
}

// Host rows -> device, the part of a frame upload that scales with its size.  `runs` are packed back to back into the pinned
// `staging` and cross the link into `dev` at the same offsets; dev == NULL: packed only (the caller copies from `staging`).
// Packing is a plain memory copy: a single thread moves ~25 GB/s, a few OpenMP threads (the runtime's pool stays warm between
// frames) ~45 GB/s, the link 55 GB/s.  The rows go in up to four pieces of >= 384 KB, so that a piece crosses the link while the
// next one is packed.  A strided host -> device copy runs at half the link's rate (the DMA engine walks the rows), a contiguous one
// at all of it: each piece crosses in one copy.
struct PackRun {
    const uint8_t* src;
    size_t pitch, bytes;       // `rows` rows of `bytes` bytes, `pitch` apart
    int rows;
};

cudaError_t pack_upload(const PackRun* runs, int nruns, uint8_t* staging, uint8_t* dev, cudaStream_t st) {
    int rows = 0;
    size_t total = 0;
    for (int k = 0; k < nruns; ++k) { rows += runs[k].rows; total += (size_t)runs[k].rows * runs[k].bytes; }
    auto offset_of = [&](int row) {            // packed byte offset of global row `row`
        size_t off = 0;
        for (int k = 0; k < nruns && row > 0; ++k) {
            const int m = row < runs[k].rows ? row : runs[k].rows;
            off += (size_t)m * runs[k].bytes;
            row -= m;
        }
        return off;
    };
    int pieces = (int)(total / (384u << 10));
    pieces = pieces < 1 ? 1 : pieces > 4 ? 4 : pieces;
    if (!dev) pieces = 1;
    const int cap = omp_get_max_threads() < 8 ? omp_get_max_threads() : 8;
    cudaError_t e = cudaSuccess;
    for (int p = 0; p < pieces && e == cudaSuccess; ++p) {
        const int r0 = (int)((long long)rows * p / pieces), r1 = (int)((long long)rows * (p + 1) / pieces);
        const size_t off = offset_of(r0), len = offset_of(r1) - off;
        int nt = (int)(len / (96u << 10));
        nt = nt < 1 ? 1 : nt > cap ? cap : nt;
        size_t base = 0;
        for (int k = 0, g0 = 0; k < nruns; g0 += runs[k].rows, base += (size_t)runs[k].rows * runs[k].bytes, ++k) {
            const int a = (r0 > g0 ? r0 : g0) - g0, b = (r1 < g0 + runs[k].rows ? r1 : g0 + runs[k].rows) - g0;
            const PackRun& R = runs[k];
            uint8_t* out = staging + base;
            if (a >= b) continue;
            if (nt == 1) {
                for (int i = a; i < b; ++i) memcpy(out + (size_t)i * R.bytes, R.src + (size_t)i * R.pitch, R.bytes);
            } else {
#pragma omp parallel for num_threads(nt) schedule(static)
                for (int i = a; i < b; ++i) memcpy(out + (size_t)i * R.bytes, R.src + (size_t)i * R.pitch, R.bytes);
            }
        }
        if (dev) e = cudaMemcpyAsync(dev + off, staging + off, len, cudaMemcpyHostToDevice, st);
    }
    return e;
}


// vt_tracks_init over items [0, n): item i initialises track first + i (slots == NULL), or track slots[i] (first == 0; slots resolved,
// a negative entry initialises nothing).  A range init writes the template tokens, status and state in place; a slot list stages the
// chunk's tokens and statuses by item and scatters them.
int tracks_init(VtHandle h, const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw, const double* boxes_xywh,
                int first, const int32_t* slots, int n, int32_t* out_status, cudaStream_t st) {
    const int C = h->cfg.embed_dim;
    const size_t row = (size_t)kNz * C;
    for (int c0 = 0; c0 < n; c0 += h->chunk) {
        const int m = (n - c0 < h->chunk) ? n - c0 : h->chunk;
        int32_t* status = h->d_status + first + c0;
        float* tok = slots ? (h->generic ? h->gws.tokz : h->d_tokz) : h->d_tmpl + (size_t)(first + c0) * row;
        if (h->generic) {
            VT_LAUNCH(h, VT_STAGE_CROP, m, st, "vt_tracks_init/crop",
                      launch_crop_normalize(frames, frame_offsets + c0, frame_hw + 2 * c0, boxes_xywh + 4 * c0, nullptr, h->cfg.template_factor, kTz, m,
                                            h->mw.lut, h->gws.crop, nullptr, nullptr, nullptr, status, st));
            VT_LAUNCH(h, VT_STAGE_STEM, m, st, "vt_tracks_init/stem", gen_launch_stem(h->gws.crop, kTz, m, h->gw, h->gws, tok, kNz, 0, st));
        } else {
            VT_LAUNCH(h, VT_STAGE_STEM, m, st, "vt_tracks_init/crop+stem",
                      launch_crop_stem(frames, frame_offsets + c0, frame_hw + 2 * c0, boxes_xywh + 4 * c0, nullptr, h->cfg.template_factor, kTz, m,
                                       h->mw, h->d_scratch, tok, kNz, 0, status, h->d_planes, h->chunk, h->d_taps, st));
        }
        if (slots)
            VT_LAUNCH(h, kNoStage, m, st, "vt_tracks_init_slots/scatter",
                      launch_scatter_init(tok, h->d_tmpl, row, boxes_xywh + 4 * c0, h->d_state, status, out_status ? out_status + c0 : nullptr,
                                          slots + c0, m, st));
    }
    if (!slots) {
        VT_CUDA(h, cudaMemcpyAsync(h->d_state + (size_t)first * 4, boxes_xywh, (size_t)n * 4 * sizeof(double), cudaMemcpyDeviceToDevice, st));
        if (out_status) VT_CUDA(h, cudaMemcpyAsync(out_status, h->d_status + first, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
    }
    h->tracks_ready = true;
    return VT_OK;
}

// Range fallback of a tensor-core step over items [0, n) (arguments as tracks_step's): the items the step flagged VT_TRACK_NUMERIC_RANGE
// are compacted on the device and run through the chain a VT_BLOCKS_SIMT_FP32 handle's step runs (fp32 crop + stem per chunk, fp32
// blocks, CUDA-core head) as a slot list, then scattered back to their item positions.  The host does not learn how many there are:
// every launch is sized for n items, and the kernels work only on the items below the device count.  Stages are profiled with 0 items, so
// that the per-stage item counts stay those of the tensor-core pass.
int range_fallback(VtHandle h, const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw, int first, const int32_t* slots,
                   int n, double* out_boxes, double* out_detail, int update_state, cudaStream_t st);

// vt_tracks_step over items [0, n): item i steps track first + i (slots == NULL), or track slots[i] (first == 0; slots resolved).  The
// state and template pointers start at track `first`; crop status and maps are kept at [first + i], i.e. by item for a slot list.
int tracks_step(VtHandle h, const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw, int first, const int32_t* slots,
                int n, double* out_boxes, double* out_detail, int update_state, cudaStream_t st) {
    const double* state = h->d_state + (size_t)first * 4;
    auto state_at = [&](int c0) { return slots ? state : state + (size_t)c0 * 4; };       // state row of the chunk's first item
    auto slots_at = [&](int c0) { return slots ? slots + c0 : nullptr; };
    if (h->generic) {
        // every stage runs per chunk: crop -> stem into the chunk's token buffer, cached template tokens copied in front
        const int C = h->cfg.embed_dim;
        const float* tmpl = h->d_tmpl + (size_t)first * kNz * C;
        for (int c0 = 0; c0 < n; c0 += h->chunk) {
            const int m = (n - c0 < h->chunk) ? n - c0 : h->chunk;
            VT_LAUNCH(h, VT_STAGE_CROP, m, st, "vt_tracks_step/crop",
                      launch_crop_normalize(frames, frame_offsets + c0, frame_hw + 2 * c0, state_at(c0), slots_at(c0), h->cfg.search_factor, kSx, m,
                                            h->mw.lut, h->gws.crop, nullptr, nullptr, nullptr, h->d_status + first + c0, st));
            if (slots)
                VT_LAUNCH(h, kNoStage, m, st, "vt_tracks_step_slots/gather",
                          launch_gather_rows(tmpl, (size_t)kNz * C, h->gws.tok, (size_t)kN * C, (size_t)kNz * C, slots + c0, m, st));
            else
                VT_CUDA(h, cudaMemcpy2DAsync(h->gws.tok, (size_t)kN * C * sizeof(float), tmpl + (size_t)c0 * kNz * C, (size_t)kNz * C * sizeof(float),
                                             (size_t)kNz * C * sizeof(float), m, cudaMemcpyDeviceToDevice, st));
            VT_LAUNCH(h, VT_STAGE_STEM, m, st, "vt_tracks_step/stem", gen_launch_stem(h->gws.crop, kSx, m, h->gw, h->gws, h->gws.tok, kN, kNz, st));
            const HeadArgs a = track_head_args(h, first, slots, c0, m, frame_hw, out_boxes, out_detail, update_state);
            VT_LAUNCH(h, VT_STAGE_BLOCKS, m, st, "vt_tracks_step/blocks+head", gen_launch_blocks_head(h->gws.tok, m, h->gw, h->gws, a, nullptr, 0, st));
        }
        h->last_first = first; h->last_n = n;
        return VT_OK;
    }
    // crop + stem run per chunk (their intermediates are large); blocks + head run once over all n tracks
    for (int c0 = 0; c0 < n; c0 += h->chunk) {
        const int m = (n - c0 < h->chunk) ? n - c0 : h->chunk;
        VT_LAUNCH(h, VT_STAGE_STEM, m, st, "vt_tracks_step/crop+stem",
                  launch_crop_stem(frames, frame_offsets + c0, frame_hw + 2 * c0, state_at(c0), slots_at(c0), h->cfg.search_factor, kSx, m,
                                   h->mw, h->d_scratch, h->d_tokx + (size_t)c0 * kNx * kC, kNx, 0, h->d_status + first + c0,
                                   h->d_planes, h->chunk, h->d_taps, st));
    }
    {
        const int m = n;
        VT_LAUNCH(h, VT_STAGE_BLOCKS, m, st, "vt_tracks_step/blocks",
                  run_blocks(h, h->d_tmpl + (size_t)first * kNz * kC, kNz, slots, h->d_tokx, kNx, h->d_tok, m, nullptr, 0, st));
        HeadArgs a = track_head_args(h, first, slots, 0, m, frame_hw, out_boxes, out_detail, update_state);
        a.tokens = h->d_tok;
        a.use_tc = h->cfg.blocks_impl != VT_BLOCKS_SIMT_FP32;
        VT_LAUNCH(h, VT_STAGE_HEAD, m, st, "vt_tracks_step/head", launch_head(a, h->mw, st));
    }
    h->last_first = first; h->last_n = n;
    return h->fallback ? range_fallback(h, frames, frame_offsets, frame_hw, first, slots, n, out_boxes, out_detail, update_state, st) : VT_OK;
}

int range_fallback(VtHandle h, const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw, int first, const int32_t* slots,
                   int n, double* out_boxes, double* out_detail, int update_state, cudaStream_t st) {
    const RangeFallback& fb = h->fb;
    VT_LAUNCH(h, VT_STAGE_HEAD, 0, st, "vt_tracks_step/fallback compact",
              launch_fallback_compact(out_boxes, h->d_status + first, slots, first, frame_offsets, frame_hw, n, h->chunk, fb,
                                      h->fallback_counter, st));
    for (int c0 = 0; c0 < n; c0 += h->chunk) {
        const int m = (n - c0 < h->chunk) ? n - c0 : h->chunk;
        VT_LAUNCH(h, VT_STAGE_STEM, 0, st, "vt_tracks_step/fallback crop+stem",
                  launch_crop_stem(frames, fb.frame_off + c0, fb.frame_hw + 2 * c0, h->d_state, fb.slot + c0, h->cfg.search_factor, kSx, m,
                                   h->mw, h->d_scratch, h->d_tokx + (size_t)c0 * kNx * kC, kNx, 0, nullptr, nullptr, 0, h->d_taps, st,
                                   fb.count + 1 + c0 / h->chunk));
    }
    VT_LAUNCH(h, VT_STAGE_BLOCKS, 0, st, "vt_tracks_step/fallback blocks",
              launch_blocks_simt(h->d_tmpl, kNz, fb.slot, h->d_tokx, kNx, h->d_tok, n, h->mw, nullptr, 0, st, fb.count));
    const size_t mt = h->cfg.max_tracks;
    HeadArgs a{};
    a.tokens = h->d_tok;
    a.n = n;
    a.score_map = fb.maps; a.size_map = fb.maps + mt * 256; a.offset_map = fb.maps + mt * 768;
    a.state = h->d_state;
    a.slots = fb.slot;
    a.frame_hw = fb.frame_hw;
    a.status = nullptr;               // crop status 0 (compaction rule): the head recomputes the same geometry from the state
    a.out_boxes = fb.boxes;
    a.out_detail = fb.detail;
    a.update_state = update_state;
    a.search_factor = h->cfg.search_factor;
    a.use_tc = 0;
    VT_LAUNCH(h, VT_STAGE_HEAD, 0, st, "vt_tracks_step/fallback head", launch_head(a, h->mw, st, fb.count));
    const LastMaps maps = last_maps(h, first);
    VT_LAUNCH(h, VT_STAGE_HEAD, 0, st, "vt_tracks_step/fallback scatter",
              launch_fallback_scatter(fb, h->cfg.max_tracks, out_boxes, out_detail, maps.score, maps.size, maps.offset, n, st));
    return VT_OK;
}

int64_t record_bytes(VtHandle h) { return VT_TRACK_RECORD_HEADER_BYTES + (int64_t)256 * h->cfg.embed_dim; }

// The entry points below come in pairs: a range call over tracks [first, first + n) (slots == NULL) and its _slots twin (list, first
// == 0), in which item i works on track slots[i].  Each pair is one checked function.  Only a list requires `slots`: a range call
// repeats another required pointer in its place.

// vt_tracks_init / vt_tracks_init_slots; an empty init still makes the handle ready to step.
int init_call(VtHandle h, const char* where, bool list, const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw,
              const double* boxes_xywh, int first, const int32_t* slots, int n, int32_t* out_status, void* stream) {
    const int rc = enter(h, where, kWeights, first, n, true, {frames, frame_offsets, frame_hw, boxes_xywh, list ? (const void*)slots : frames});
    if (rc == kEmpty) h->tracks_ready = true;
    VT_ENTER(h, rc);
    cudaStream_t st = (cudaStream_t)stream;
    if (list) VT_LAUNCH(h, kNoStage, n, st, where, launch_resolve_slots(slots, n, h->cfg.max_tracks, h->d_claim, h->d_eff, st));
    return tracks_init(h, frames, frame_offsets, frame_hw, boxes_xywh, first, list ? h->d_eff : nullptr, n, out_status, st);
}

// vt_tracks_step / vt_tracks_step_slots
int step_call(VtHandle h, const char* where, bool list, const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw,
              int first, const int32_t* slots, int n, double* out_boxes, double* out_detail, int update_state, void* stream) {
    VT_ENTER(h, enter(h, where, kTracks, first, n, true, {frames, frame_offsets, frame_hw, out_boxes, list ? (const void*)slots : frames}));
    cudaStream_t st = (cudaStream_t)stream;
    if (list) VT_LAUNCH(h, kNoStage, n, st, where, launch_resolve_slots(slots, n, h->cfg.max_tracks, h->d_claim, h->d_eff, st));
    return tracks_step(h, frames, frame_offsets, frame_hw, first, list ? h->d_eff : nullptr, n, out_boxes, out_detail, update_state, st);
}

// vt_tracks_export (records written) and vt_tracks_import (records read), with their _slots twins.  An import makes the handle ready
// to step, as an init does.
int records_call(VtHandle h, const char* where, bool do_export, bool list, uint8_t* records, int first, const int32_t* slots, int n,
                 int32_t* out_status, void* stream) {
    VT_ENTER(h, enter(h, where, kWeights, first, n, true, {records, list ? (const void*)slots : records}));
    if (reinterpret_cast<uintptr_t>(records) % 16) return fail(h, VT_ERR_INVALID_ARG, "%s: records must be 16-byte aligned", where);
    cudaStream_t st = (cudaStream_t)stream;
    const RecordArgs a{h->d_state, h->d_tmpl, h->cfg.embed_dim, first, h->cfg.max_tracks, slots, h->d_claim, out_status, h->fingerprint};
    if (list) VT_LAUNCH(h, kNoStage, n, st, where, launch_claim_slots(slots, n, h->cfg.max_tracks, h->d_claim, st));
    if (do_export) {
        VT_LAUNCH(h, kNoStage, n, st, where, launch_tracks_export(a, records, n, st));
    } else {
        VT_LAUNCH(h, kNoStage, n, st, where, launch_tracks_import(a, records, n, st));
        h->tracks_ready = true;
    }
    return VT_OK;
}

}  // namespace

extern "C" {

int vt_abi_version(void) { return VT_ABI_VERSION; }

const char* vt_last_error(VtHandle h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int vt_create(const VtConfig* cfg, VtHandle* out) {
    if (!cfg || !out) return fail(nullptr, VT_ERR_INVALID_ARG, "vt_create: null argument");
    *out = nullptr;
    const bool fast = cfg->embed_dim == kC && cfg->num_heads == 1 && cfg->depth == kDepth && cfg->head_channels == kHeadC;
    if (cfg->mlp_ratio != 4 || cfg->stride != 16 || cfg->template_size != kTz || cfg->search_size != kSx)
        return fail(nullptr, VT_ERR_UNSUPPORTED,
                    "unsupported configuration (this build needs mlp_ratio=4, stride=16, template 128, search 256)");
    if (!fast && (cfg->embed_dim < 8 || cfg->embed_dim % 8 != 0 || cfg->num_heads < 1 || cfg->embed_dim % cfg->num_heads != 0 ||
                  cfg->depth < 1 || cfg->depth > kGenMaxDepth || cfg->head_channels < 8 || cfg->head_channels % 8 != 0))
        return fail(nullptr, VT_ERR_UNSUPPORTED,
                    "unsupported configuration (embed_dim and head_channels must be multiples of 8, embed_dim divisible by "
                    "num_heads, 1 <= depth <= %d)", kGenMaxDepth);
    if (cfg->max_tracks < 1 || !(cfg->template_factor > 0) || !(cfg->search_factor > 0))
        return fail(nullptr, VT_ERR_INVALID_ARG, "vt_create: max_tracks >= 1 and positive crop factors required");
    if (cfg->blocks_impl != VT_BLOCKS_SIMT_FP32 && cfg->blocks_impl != VT_BLOCKS_TCGEN05 && cfg->blocks_impl != VT_BLOCKS_TCGEN05_3TERM)
        return fail(nullptr, VT_ERR_INVALID_ARG, "vt_create: unknown blocks_impl %d", cfg->blocks_impl);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(nullptr, VT_ERR_NO_DEVICE, "no CUDA device: libvittrack_b200 has no CPU fallback");
    }
    if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, VT_ERR_INVALID_ARG, "vt_create: device %d out of range", cfg->device);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess) return fail(nullptr, VT_ERR_CUDA, "cudaGetDeviceProperties failed");
    if (prop.major < 10) return fail(nullptr, VT_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", cfg->device, prop.major, prop.minor);

    VtHandle h = new VtContext();
    h->cfg = *cfg;
    h->num_sms = prop.multiProcessorCount;
    h->generic = !fast;
    h->chunk = cfg->chunk_tracks > 0 ? cfg->chunk_tracks : (fast ? 1024 : 64);        // generic path: ~46 MB of workspace per track at C = 768
    if (h->chunk > cfg->max_tracks) h->chunk = cfg->max_tracks;
    DeviceGuard dg(cfg->device);                 // the caller's current device is restored on return
    if (dg.err != cudaSuccess) { delete h; return fail(nullptr, VT_ERR_CUDA, "cudaSetDevice failed"); }
    const size_t ch = h->chunk, mt = cfg->max_tracks, Cd = cfg->embed_dim;
    cudaError_t e = cudaSuccess;
    auto A = [&](void** p, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc(p, bytes); };
    if (fast) {
        A((void**)&h->d_scratch, ch * stem_scratch_floats(kSx) * sizeof(float));
        A((void**)&h->d_taps, crop_taps_bytes((int)ch));
        if (cfg->blocks_impl != VT_BLOCKS_SIMT_FP32) {
            const size_t pb = ch * tc_planes_bytes_per_track();
            A((void**)&h->d_planes, pb);
            if (e == cudaSuccess) e = cudaMemset(h->d_planes, 0, pb);
        }
        A((void**)&h->d_tokz, ch * kNz * kC * sizeof(float));
        A((void**)&h->d_tokx, mt * kNx * kC * sizeof(float));     // whole-step buffers: blocks + head run once per step
        A((void**)&h->d_tok, mt * kN * kC * sizeof(float));
    } else {
        h->gw.C = cfg->embed_dim; h->gw.heads = cfg->num_heads; h->gw.depth = cfg->depth; h->gw.hc = cfg->head_channels;
        h->gw.use_img = (cfg->blocks_impl != VT_BLOCKS_SIMT_FP32 && cfg->embed_dim % 128 == 0) ? 1 : 0;
        h->gw.fp32_only = cfg->blocks_impl == VT_BLOCKS_SIMT_FP32 ? 1 : 0;
        size_t off[kGenWorkSlots];
        const size_t tot = gen_work_floats(h->gw, h->chunk, off);
        A((void**)&h->d_gwork, tot * sizeof(float));
        if (e == cudaSuccess) e = cudaMemset(h->d_gwork, 0, tot * sizeof(float));      // padding rows of the split images are read (and ignored)
        float** members[kGenWorkSlots] = {&h->gws.crop, &h->gws.col, &h->gws.act1, &h->gws.act2, &h->gws.act3, &h->gws.tokz, &h->gws.tok, &h->gws.ln,
                                          &h->gws.qkv, &h->gws.scores, &h->gws.attn, &h->gws.hid, &h->gws.t1, &h->gws.t2, &h->gws.t3, &h->gws.t4, &h->gws.raw5,
                                          &h->gws.img_ln, &h->gws.img_attn, &h->gws.img_hid};
        for (int i = 0; i < kGenWorkSlots; ++i) *members[i] = h->d_gwork ? h->d_gwork + off[i] : nullptr;
        h->gws.chunk = h->chunk;
    }
    A((void**)&h->d_state, mt * 4 * sizeof(double));
    A((void**)&h->d_tmpl, mt * kNz * Cd * sizeof(float));
    A((void**)&h->d_status, mt * sizeof(int32_t));
    A((void**)&h->d_claim, mt * sizeof(uint32_t));
    A((void**)&h->d_eff, mt * sizeof(int32_t));
    A((void**)&h->d_maps, mt * 1280 * sizeof(float));
    A((void**)&h->d_surf_rect, mt * 4 * sizeof(int32_t));
    A((void**)&h->d_surf_done, mt * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMemset(h->d_state, 0, mt * 4 * sizeof(double));
    if (e == cudaSuccess) e = cudaMemset(h->d_tmpl, 0, mt * kNz * Cd * sizeof(float));     // never-initialised slots export zeros, not stale memory
    if (e == cudaSuccess) e = cudaMemset(h->d_status, 0, mt * sizeof(int32_t));
    if (e == cudaSuccess) e = cudaMemset(h->d_claim, 0xff, mt * sizeof(uint32_t));
    if (e == cudaSuccess) {                                                                  // empty rectangles: {INT32_MAX, INT32_MAX, 0, 0}
        std::vector<int32_t> empty(mt * 4, 0);
        for (size_t s = 0; s < mt; ++s) empty[4 * s] = empty[4 * s + 1] = 0x7fffffff;
        e = cudaMemcpy(h->d_surf_rect, empty.data(), mt * 4 * sizeof(int32_t), cudaMemcpyHostToDevice);
    }
    if (e == cudaSuccess) e = cudaMemset(h->d_surf_done, 0, mt * sizeof(uint32_t));
    if (e != cudaSuccess) {
        fail(nullptr, VT_ERR_CUDA, "vt_create: device allocation failed: %s", cudaGetErrorString(e));
        free_all(h); delete h;
        return VT_ERR_CUDA;
    }
    *out = h;
    return VT_OK;
}

int vt_destroy(VtHandle h) {
    if (!h) return VT_ERR_INVALID_ARG;
    DeviceGuard dg(h->cfg.device);
    free_all(h);                                 // cudaFree waits for work that still uses the allocation
    delete h;
    return VT_OK;
}

int vt_set_tensor(VtHandle h, const char* name, const float* data_host, const int64_t* shape, int32_t ndim) {
    if (!h || !name || ndim < 0 || ndim > 8 || (ndim > 0 && !shape)) return h ? fail(h, VT_ERR_INVALID_ARG, "vt_set_tensor: bad argument") : VT_ERR_INVALID_ARG;
    const std::string nm(name);
    const char* nbt = "num_batches_tracked";
    if (nm.size() >= strlen(nbt) && nm.compare(nm.size() - strlen(nbt), strlen(nbt), nbt) == 0) return VT_OK;   // accepted, unused in eval
    const auto table = tensor_table(h->cfg);
    const auto it = table.find(nm);
    if (it == table.end()) return fail(h, VT_ERR_WEIGHTS, "unknown tensor '%s' (ignored, as load_state_dict(strict=False) would)", name);
    if (!data_host) return fail(h, VT_ERR_INVALID_ARG, "vt_set_tensor: null data for '%s'", name);
    const std::vector<int64_t>& want = it->second;
    std::vector<int64_t> got(shape, shape + ndim);
    if (got != want) {
        std::string g, w;
        for (auto v : got) g += std::to_string(v) + ",";
        for (auto v : want) w += std::to_string(v) + ",";
        return fail(h, VT_ERR_WEIGHTS, "tensor '%s': shape (%s) does not match expected (%s)", name, g.c_str(), w.c_str());
    }
    size_t n = 1;
    for (auto v : got) n *= (size_t)v;
    HostTensor& t = h->tensors[nm];
    t.shape = got;
    t.data.assign(data_host, data_host + n);
    h->finalized = false;
    return VT_OK;
}

int vt_finalize_weights(VtHandle h, void* stream) {
    if (!h) return VT_ERR_INVALID_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    DeviceGuard dg(h->cfg.device);
    VT_CUDA(h, dg.err);
    if (const int rc = check_missing(h)) return rc;
    h->fingerprint = weights_fingerprint(h);
    TensorMap ts = h->tensors;          // rebalanced on a copy: finalising again starts from the tensors as they were set
    const int pnorm = rebalance(h->cfg, ts);
    if (h->generic) return finalize_generic(h, ts, pnorm, st);
    h->score_terms = score_terms(h->cfg, ts);
    Packer pk;
    ModelW& m = h->mw;
    m.norm_tap_scale = ldexpf(1.f, pnorm);

    // ---- stem: BN folded, [co][ci][3][3] -> [ci][ky][kx][co]
    size_t stem_w[4], stem_b[4];
    for (int l = 0; l < 4; ++l) {
        const FoldedConv f = fold_conv_bn(ts, stem_prefix(l) + "c.", stem_prefix(l) + "bn.", false);
        stem_w[l] = pk.slot(m.stem[l].w, f.w.size());
        stem_b[l] = pk.put(m.stem[l].b, f.b.data(), f.co);
        for (int co = 0; co < f.co; ++co)
            for (int ci = 0; ci < f.ci; ++ci)
                for (int k = 0; k < 9; ++k) pk.buf[stem_w[l] + ((size_t)ci * 9 + k) * f.co + co] = f.w[((size_t)co * f.ci + ci) * 9 + k];
    }
    // ---- stem conv2 / conv3 / conv4 for the tensor cores: fp16 hi | lo weight blobs in the kernels' K-step order (vt_stem_tc.cu)
    {
        const int lcin[3] = {6, 12, 24}, lcch[3] = {kConv2Cch, kConv3Cch, kConv4Cch}, lcout[3] = {12, 24, 48}, lnpad[3] = {16, 32, 48};
        for (int i = 0; i < 3; ++i) {
            const size_t bytes = stem_tc_weight_bytes(i);
            const size_t w = pk.slot(m.stem_tc_w[i], bytes / 4), b = pk.slot(m.stem_tc_b[i], lnpad[i]);
            for (int co = 0; co < lcout[i]; ++co) pk.buf[b + co] = pk.buf[stem_b[i + 1] + co];
            stem_tc_pack_weights(lcin[i], lcch[i], lcout[i], lnpad[i], &pk.buf[stem_w[i + 1]], pk.bytes(w), pk.bytes(w) + bytes / 2);
        }
    }
    // ---- stem conv1 for the fused tensor-core front (vt_stem_fused.cu): pixel normalisation folded into the weights / border-variant biases
    const size_t s1_w = pk.slot(m.stem1_tc_w, kStem1TcWBytes / 4), s1_p = pk.slot(m.stem1_tc_par, kStem1TcParFloats);
    stem1_tc_pack(&pk.buf[stem_w[0]], &pk.buf[stem_b[0]], pk.bytes(s1_w), &pk.buf[s1_p]);
    // ---- blocks: Linear weights [out][in] -> K-major [in][out]
    auto transp = [&](size_t o, const float* src, int rows_out, int cols_in) {     // src [out][in] -> dst [in][out]
        for (int r = 0; r < rows_out; ++r)
            for (int c = 0; c < cols_in; ++c) pk.buf[o + (size_t)c * rows_out + r] = src[(size_t)r * cols_in + c];
    };
    for (int b = 0; b < kDepth; ++b) {
        const BlockTensors t = block_tensors(ts, b);
        BlockW& B = m.blk[b];
        pk.put(B.ln1_g, t.ln1_g, kC); pk.put(B.ln1_b, t.ln1_b, kC);
        transp(pk.slot(B.wqkv, kC * 3 * kC), t.wqkv, 3 * kC, kC);
        pk.put(B.bqkv, t.bqkv, 3 * kC);
        transp(pk.slot(B.wproj, kC * kC), t.wproj, kC, kC);
        pk.put(B.bproj, t.bproj, kC);
        pk.put(B.ln2_g, t.ln2_g, kC); pk.put(B.ln2_b, t.ln2_b, kC);
        transp(pk.slot(B.wfc1, kC * kHid), t.wfc1, kHid, kC);
        pk.put(B.bfc1, t.bfc1, kHid);
        transp(pk.slot(B.wfc2, kHid * kC), t.wfc2, kC, kHid);
        pk.put(B.bfc2, t.bfc2, kC);
    }
    // ---- the same blocks for the tensor cores (vt_block_tc.cu)
    for (int b = 0; b < kDepth; ++b) {
        const size_t wa = pk.slot(m.tc[b].wa, kTcWaBytes / 4), wb = pk.slot(m.tc[b].wb, kTcWbBytes / 4), par = pk.slot(m.tc[b].par, kTcParFloats);
        block_tc_pack(block_tensors(ts, b), pk.bytes(wa), pk.bytes(wb), &pk.buf[par]);
    }
    pk.put(m.norm_g, tensor(ts, "norm.weight"), kC); pk.put(m.norm_b, tensor(ts, "norm.bias"), kC);
    pk.put(m.pos_z, tensor(ts, "pos_embed_z"), kNz * kC); pk.put(m.pos_x, tensor(ts, "pos_embed_x"), kNx * kC);

    // ---- head: conv(+bias) -> BN folded; layer i weights laid out [ci][k][tower][co_t]
    const float** head_w[4] = {&m.head.w1, &m.head.w2, &m.head.w3, &m.head.w4};
    const float** head_b[4] = {&m.head.b1, &m.head.b2, &m.head.b3, &m.head.b4};
    size_t hw[4];
    for (int i = 0; i < 4; ++i) {
        FoldedConv f[3];
        for (int t = 0; t < 3; ++t) f[t] = fold_conv_bn(ts, head_prefix(i, t) + "0.", head_prefix(i, t) + "1.", true);
        const int ci_n = f[0].ci, co_n = f[0].co;
        hw[i] = pk.slot(*head_w[i], (size_t)ci_n * 9 * 3 * co_n);
        const size_t hb = pk.slot(*head_b[i], 3 * co_n);
        for (int t = 0; t < 3; ++t)
            for (int co = 0; co < co_n; ++co) {
                pk.buf[hb + t * co_n + co] = f[t].b[co];
                for (int ci = 0; ci < ci_n; ++ci)
                    for (int k = 0; k < 9; ++k)
                        pk.buf[hw[i] + (((size_t)ci * 9 + k) * 3 + t) * co_n + co] = f[t].w[((size_t)co * ci_n + ci) * 9 + k];
            }
    }
    // head conv1 - conv3 for the tensor cores (vt_head.cu)
    const size_t htc1 = pk.slot(m.head_tc_w1, head_tc_weight_bytes(0) / 4), htc2 = pk.slot(m.head_tc_w2, head_tc_weight_bytes(1) / 4),
                 htc3 = pk.slot(m.head_tc_w3, head_tc_weight_bytes(2) / 4);
    head_tc_pack(&pk.buf[hw[0]], &pk.buf[hw[1]], &pk.buf[hw[2]], pk.bytes(htc1), pk.bytes(htc2), pk.bytes(htc3));
    const size_t w5 = pk.slot(m.head.w5, 3 * 4 * 2), b5 = pk.slot(m.head.b5, 3 * 2);
    for (int t = 0; t < 3; ++t) {
        const std::string p = std::string("box_head.conv5_") + kTowers[t] + ".";
        const float *w = tensor(ts, p + "weight"), *b = tensor(ts, p + "bias");
        for (int o = 0; o < (t == 0 ? 1 : 2); ++o) {
            pk.buf[b5 + t * 2 + o] = b[o];
            for (int c = 0; c < 4; ++c) pk.buf[w5 + (t * 4 + c) * 2 + o] = w[o * 4 + c];
        }
    }
    // ---- Hann window (hann.py:6-16) and normalisation table (data_utils.py:8-14) -----------------
    const size_t hann = pk.slot(m.hann, 256), lut = pk.slot(m.lut, 768);
    fill_hann_and_lut(ts, &pk.buf[hann], &pk.buf[lut]);
    if (const int rc = upload_weights(h, pk, st)) return rc;
    h->finalized = true;
    return VT_OK;
}

int vt_crop_normalize(VtHandle h, const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw,
                      const double* boxes_xywh, double factor, int32_t out_size, int32_t n, float* out_nchw,
                      uint8_t* out_u8_hwc, uint8_t* out_mask, double* out_resize_factor, int32_t* out_status,
                      void* stream) {
    VT_ENTER(h, enter(h, "vt_crop_normalize", kWeights, 0, n, false, {frames, frame_offsets, frame_hw, boxes_xywh, out_nchw}));
    if (out_size != 128 && out_size != 256) return fail(h, VT_ERR_UNSUPPORTED, "vt_crop_normalize: out_size must be 128 or 256");
    if (!(factor > 0)) return fail(h, VT_ERR_INVALID_ARG, "vt_crop_normalize: factor must be positive");
    cudaStream_t st = (cudaStream_t)stream;
    VT_LAUNCH(h, kNoStage, n, st, "vt_crop_normalize",
              launch_crop_normalize(frames, frame_offsets, frame_hw, boxes_xywh, nullptr, factor, out_size, n, h->mw.lut, out_nchw,
                                    out_u8_hwc, out_mask, out_resize_factor, out_status, st));
    return VT_OK;
}

int vt_forward(VtHandle h, const float* z, const float* x, int32_t n, float* pred_boxes, float* score_map,
               float* size_map, float* offset_map, float* taps, void* stream) {
    VT_ENTER(h, enter(h, "vt_forward", kWeights, 0, n, false, {z, x}));
    cudaStream_t st = (cudaStream_t)stream;
    if (h->generic) {
        const int C = h->cfg.embed_dim;
        const size_t gtap = (size_t)n * kN * C;
        for (int first = 0; first < n; first += h->chunk) {
            const int m = (n - first < h->chunk) ? n - first : h->chunk;
            VT_LAUNCH(h, VT_STAGE_STEM, m, st, "vt_forward/stem(z)", gen_launch_stem(z + (size_t)first * 3 * kTz * kTz, kTz, m, h->gw, h->gws, h->gws.tok, kN, 0, st));
            VT_LAUNCH(h, VT_STAGE_STEM, m, st, "vt_forward/stem(x)", gen_launch_stem(x + (size_t)first * 3 * kSx * kSx, kSx, m, h->gw, h->gws, h->gws.tok, kN, kNz, st));
            const HeadArgs a = forward_head_args(first, m, pred_boxes, score_map, size_map, offset_map);
            VT_LAUNCH(h, VT_STAGE_BLOCKS, m, st, "vt_forward/blocks+head",
                      gen_launch_blocks_head(h->gws.tok, m, h->gw, h->gws, a, taps ? taps + (size_t)first * kN * C : nullptr, gtap, st));
        }
        return VT_OK;
    }
    const size_t tap_stride = (size_t)n * kN * kC;
    for (int first = 0; first < n; first += h->chunk) {
        const int m = (n - first < h->chunk) ? n - first : h->chunk;
        VT_LAUNCH(h, VT_STAGE_STEM, m, st, "vt_forward/stem(z)", launch_stem(z + (size_t)first * 3 * kTz * kTz, kTz, m, h->mw, h->d_scratch, h->d_tokz, kNz, 0, h->d_planes, h->chunk, st));
        VT_LAUNCH(h, VT_STAGE_STEM, m, st, "vt_forward/stem(x)", launch_stem(x + (size_t)first * 3 * kSx * kSx, kSx, m, h->mw, h->d_scratch, h->d_tokx, kNx, 0, h->d_planes, h->chunk, st));
        VT_LAUNCH(h, VT_STAGE_BLOCKS, m, st, "vt_forward/blocks", run_blocks(h, h->d_tokz, kNz, nullptr, h->d_tokx, kNx, h->d_tok, m,
                                                      taps ? taps + (size_t)first * kN * kC : nullptr, tap_stride, st));
        HeadArgs a = forward_head_args(first, m, pred_boxes, score_map, size_map, offset_map);
        a.tokens = h->d_tok;
        a.tokens_norm = taps ? taps + (size_t)(kDepth + 1) * tap_stride + (size_t)first * kN * kC : nullptr;
        a.use_tc = h->cfg.blocks_impl != VT_BLOCKS_SIMT_FP32;
        VT_LAUNCH(h, VT_STAGE_HEAD, m, st, "vt_forward/head", launch_head(a, h->mw, st));
    }
    return VT_OK;
}

int vt_cal_bbox(VtHandle h, const float* score, const float* size_map, const float* offset_map, int32_t n,
                float* boxes, void* stream) {
    VT_ENTER(h, enter(h, "vt_cal_bbox", kHandle, 0, n, false, {score, size_map, offset_map, boxes}));
    cudaStream_t st = (cudaStream_t)stream;
    VT_LAUNCH(h, kNoStage, n, st, "vt_cal_bbox", launch_cal_bbox(score, size_map, offset_map, n, boxes, st));
    return VT_OK;
}

int vt_tracks_init(VtHandle h, const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw,
                   const double* boxes_xywh, int32_t first, int32_t n, int32_t* out_status, void* stream) {
    return init_call(h, "vt_tracks_init", false, frames, frame_offsets, frame_hw, boxes_xywh, first, nullptr, n, out_status, stream);
}

int vt_tracks_init_slots(VtHandle h, const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw,
                         const double* boxes_xywh, const int32_t* slots, int32_t n, int32_t* out_status, void* stream) {
    return init_call(h, "vt_tracks_init_slots", true, frames, frame_offsets, frame_hw, boxes_xywh, 0, slots, n, out_status, stream);
}

int vt_tracks_step(VtHandle h, const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw,
                   int32_t first, int32_t n, double* out_boxes, double* out_detail, int32_t update_state, void* stream) {
    return step_call(h, "vt_tracks_step", false, frames, frame_offsets, frame_hw, first, nullptr, n, out_boxes, out_detail, update_state, stream);
}

int vt_tracks_step_slots(VtHandle h, const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw,
                         const int32_t* slots, int32_t n, double* out_boxes, double* out_detail, int32_t update_state, void* stream) {
    return step_call(h, "vt_tracks_step_slots", true, frames, frame_offsets, frame_hw, 0, slots, n, out_boxes, out_detail, update_state, stream);
}

int vt_set_range_fallback(VtHandle h, int32_t enable, int64_t* counter_dev) {
    if (!h) return VT_ERR_INVALID_ARG;
    if (h->generic) return fail(h, VT_ERR_UNSUPPORTED, "vt_set_range_fallback: only the vit_48_h32 configuration has the fp32 step chain it needs");
    if (h->cfg.blocks_impl == VT_BLOCKS_SIMT_FP32) return VT_OK;        // no fp16 operands: nothing is ever flagged for range
    if (enable && !h->d_fallback) {
        DeviceGuard dg(h->cfg.device);
        VT_CUDA(h, dg.err);
        const size_t mt = h->cfg.max_tracks, chunks = (mt + h->chunk - 1) / h->chunk;
        size_t off = 0;
        auto carve = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
        const size_t o_count = carve((1 + chunks) * 4), o_item = carve(mt * 4), o_slot = carve(mt * 4), o_off = carve(mt * 8),
                     o_hw = carve(mt * 8), o_boxes = carve(mt * 5 * 8), o_detail = carve(mt * 8 * 8), o_maps = carve(mt * 1280 * 4);
        VT_CUDA(h, cudaMalloc(&h->d_fallback, off));
        uint8_t* b = static_cast<uint8_t*>(h->d_fallback);
        h->fb = RangeFallback{reinterpret_cast<int32_t*>(b + o_count), reinterpret_cast<int32_t*>(b + o_item), reinterpret_cast<int32_t*>(b + o_slot),
                              reinterpret_cast<int64_t*>(b + o_off), reinterpret_cast<int32_t*>(b + o_hw), reinterpret_cast<double*>(b + o_boxes),
                              reinterpret_cast<double*>(b + o_detail), reinterpret_cast<float*>(b + o_maps)};
    }
    h->fallback = enable != 0;
    h->fallback_counter = enable ? counter_dev : nullptr;
    return VT_OK;
}

int vt_weights_fingerprint(VtHandle h, uint64_t* out_host) {
    if (const int rc = check_ready(h, false)) return rc;
    if (!out_host) return fail(h, VT_ERR_INVALID_ARG, "vt_weights_fingerprint: null pointer");
    *out_host = h->fingerprint;
    return VT_OK;
}

int vt_track_record_bytes(VtHandle h, int64_t* out_host) {
    if (!h) return VT_ERR_INVALID_ARG;
    if (!out_host) return fail(h, VT_ERR_INVALID_ARG, "vt_track_record_bytes: null pointer");
    *out_host = record_bytes(h);
    return VT_OK;
}

int vt_tracks_export(VtHandle h, int32_t first, int32_t n, uint8_t* records, void* stream) {
    return records_call(h, "vt_tracks_export", true, false, records, first, nullptr, n, nullptr, stream);
}

int vt_tracks_export_slots(VtHandle h, const int32_t* slots, int32_t n, uint8_t* records, int32_t* out_status, void* stream) {
    return records_call(h, "vt_tracks_export_slots", true, true, records, 0, slots, n, out_status, stream);
}

int vt_tracks_import(VtHandle h, const uint8_t* records, int32_t first, int32_t n, int32_t* out_status, void* stream) {
    return records_call(h, "vt_tracks_import", false, false, const_cast<uint8_t*>(records), first, nullptr, n, out_status, stream);
}

int vt_tracks_import_slots(VtHandle h, const uint8_t* records, const int32_t* slots, int32_t n, int32_t* out_status, void* stream) {
    return records_call(h, "vt_tracks_import_slots", false, true, const_cast<uint8_t*>(records), 0, slots, n, out_status, stream);
}

int vt_tracks_get_state(VtHandle h, double* boxes_xywh, int32_t first, int32_t n, void* stream) {
    VT_ENTER(h, enter(h, "vt_tracks_get_state", kHandle, first, n, true, {boxes_xywh}));
    VT_CUDA(h, cudaMemcpyAsync(boxes_xywh, h->d_state + (size_t)first * 4, (size_t)n * 4 * sizeof(double), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return VT_OK;
}

int vt_tracks_set_state(VtHandle h, const double* boxes_xywh, int32_t first, int32_t n, void* stream) {
    VT_ENTER(h, enter(h, "vt_tracks_set_state", kHandle, first, n, true, {boxes_xywh}));
    VT_CUDA(h, cudaMemcpyAsync(h->d_state + (size_t)first * 4, boxes_xywh, (size_t)n * 4 * sizeof(double), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return VT_OK;
}

int vt_tracks_last_maps(VtHandle h, int32_t first, int32_t n, float* score_map, float* size_map, float* offset_map, void* stream) {
    if (h && !tracks_in(first, n, h->last_first, h->last_n))
        return fail(h, VT_ERR_STATE, "vt_tracks_last_maps: tracks [%d, %lld) were not part of the last step", first, (long long)first + n);
    VT_ENTER(h, enter(h, "vt_tracks_last_maps", kHandle, first, n, false, {}));
    cudaStream_t st = (cudaStream_t)stream;
    const LastMaps maps = last_maps(h, first);
    if (score_map) VT_CUDA(h, cudaMemcpyAsync(score_map, maps.score, (size_t)n * 256 * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (size_map) VT_CUDA(h, cudaMemcpyAsync(size_map, maps.size, (size_t)n * 512 * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (offset_map) VT_CUDA(h, cudaMemcpyAsync(offset_map, maps.offset, (size_t)n * 512 * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return VT_OK;
}

int vt_upload_frame_rect(const uint8_t* image, int32_t H, int32_t W, int32_t y0, int32_t y1, int32_t x0, int32_t x1, uint8_t* staging,
                         uint8_t* staging_dev, uint8_t* frame_dev, void* stream) {
    if (!image || !staging || !frame_dev || H <= 0 || W <= 0 || y0 < 0 || y1 > H || y0 >= y1 || x0 < 0 || x1 > W || x0 >= x1) return VT_ERR_INVALID_ARG;
    const size_t pitch = (size_t)W * 3, wb = (size_t)(x1 - x0) * 3;
    const int rows = y1 - y0;
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t* dst = frame_dev + (size_t)y0 * pitch + (size_t)x0 * 3;
    const bool direct = wb == pitch;                       // full rows: the packed layout is the frame's
    const PackRun run{image + (size_t)y0 * pitch + (size_t)x0 * 3, pitch, wb, rows};
    cudaError_t e = pack_upload(&run, 1, staging, direct ? dst : staging_dev, st);
    if (e == cudaSuccess && !direct)
        e = staging_dev ? cudaMemcpy2DAsync(dst, pitch, staging_dev, wb, wb, (size_t)rows, cudaMemcpyDeviceToDevice, st)
                        : cudaMemcpy2DAsync(dst, pitch, staging, wb, wb, (size_t)rows, cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return VT_ERR_CUDA;
    }
    return VT_OK;
}

int vt_upload_yuv420_rect(VtHandle h, int32_t format, const uint8_t* image, int32_t H, int32_t W, int32_t y0, int32_t y1,
                          int32_t x0, int32_t x1, uint8_t* staging, uint8_t* staging_dev, uint8_t* frame_rgb_dev, void* stream) {
    VT_ENTER(h, enter(h, "vt_upload_yuv420_rect", kHandle, 0, 1, false, {image, staging, staging_dev, frame_rgb_dev}));      // one frame
    if (const int rc = check_yuv_format(h, "vt_upload_yuv420_rect", format)) return rc;
    if (H < 2 || W < 2 || (H & 1) || (W & 1)) return fail(h, VT_ERR_INVALID_ARG, "vt_upload_yuv420_rect: frame %d x %d: H and W must be even and positive", H, W);
    if (y0 < 0 || y1 > H || y0 >= y1 || x0 < 0 || x1 > W || x0 >= x1)
        return fail(h, VT_ERR_INVALID_ARG, "vt_upload_yuv420_rect: rectangle [%d, %d) x [%d, %d) is empty or leaves the %d x %d frame", y0, y1, x0, x1, H, W);
    // widen to even bounds: a 2x2 block shares one chroma sample
    y0 &= ~1; x0 &= ~1; y1 = (y1 + 1) & ~1; x1 = (x1 + 1) & ~1;
    const int rows = y1 - y0, cols = x1 - x0;
    const uint8_t* chroma = image + (size_t)H * W;
    PackRun runs[3];
    int nruns = 0;
    runs[nruns++] = {image + (size_t)y0 * W + x0, (size_t)W, (size_t)cols, rows};
    if (format == VT_FRAME_NV12) {
        runs[nruns++] = {chroma + (size_t)(y0 / 2) * W + x0, (size_t)W, (size_t)cols, rows / 2};
    } else {
        const size_t cw = (size_t)W / 2;
        runs[nruns++] = {chroma + (size_t)(y0 / 2) * cw + x0 / 2, cw, (size_t)cols / 2, rows / 2};
        runs[nruns++] = {chroma + (size_t)(H / 2) * cw + (size_t)(y0 / 2) * cw + x0 / 2, cw, (size_t)cols / 2, rows / 2};
    }
    cudaStream_t st = (cudaStream_t)stream;
    VT_CUDA(h, pack_upload(runs, nruns, staging, staging_dev, st));
    YuvDesc d{};
    d.y = staging_dev;
    d.u = staging_dev + (size_t)rows * cols;
    d.y_pitch = cols;
    d.c_pitch = format == VT_FRAME_NV12 ? cols : cols / 2;
    d.v = d.u + (size_t)(rows / 2) * (cols / 2);
    d.dst = frame_rgb_dev + ((size_t)y0 * W + x0) * 3;
    d.dst_pitch = (int64_t)W * 3;
    d.w = cols; d.h = rows;
    VT_LAUNCH(h, kNoStage, 1, st, "vt_upload_yuv420_rect", launch_yuv420_rect(format, d, h->num_sms, st));
    return VT_OK;
}

int vt_yuv420_to_rgb(VtHandle h, int32_t format, const uint8_t* src, const int64_t* src_offsets, const int32_t* frame_hw,
                     uint8_t* dst, const int64_t* dst_offsets, int32_t n, void* stream) {
    VT_ENTER(h, enter(h, "vt_yuv420_to_rgb", kHandle, 0, n, false, {src, src_offsets, frame_hw, dst, dst_offsets}));
    if (const int rc = check_yuv_format(h, "vt_yuv420_to_rgb", format)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    VT_LAUNCH(h, kNoStage, n, st, "vt_yuv420_to_rgb", launch_yuv420_to_rgb(format, src, src_offsets, frame_hw, dst, dst_offsets, n, h->num_sms, st));
    return VT_OK;
}

int vt_yuv420_crop_to_rgb(VtHandle h, int32_t format, const uint64_t* planes, const int32_t* pitches, const int32_t* frame_hw,
                          const double* boxes_xywh, double factor, int32_t first, int32_t n, uint8_t* dst, const int64_t* dst_offsets,
                          void* stream) {
    const char* where = "vt_yuv420_crop_to_rgb";
    VT_ENTER(h, enter(h, where, kHandle, 0, n, false, {planes, pitches, frame_hw, dst, dst_offsets}));
    if (const int rc = check_yuv_format(h, where, format)) return rc;
    if (!(factor > 0)) return fail(h, VT_ERR_INVALID_ARG, "%s: factor must be positive", where);
    if (const int rc = boxes_xywh ? VT_OK : check_tracks(h, where, first, n)) return rc;       // the boxes are the tracks' state
    const double* boxes = boxes_xywh ? boxes_xywh : h->d_state + (size_t)first * 4;
    cudaStream_t st = (cudaStream_t)stream;
    VT_LAUNCH(h, kNoStage, n, st, where, launch_yuv420_crop_to_rgb(format, planes, pitches, frame_hw, boxes, factor, dst, dst_offsets, n, h->num_sms, st));
    return VT_OK;
}

int vt_yuv420_crops_to_surface_rgb(VtHandle h, int32_t format, const uint64_t* planes, const int32_t* pitches, const int32_t* frame_hw,
                                   int32_t m, const int32_t* item_surface, const double* boxes_xywh, const int32_t* slots, double factor,
                                   int32_t first, int32_t n, uint8_t* dst, const int64_t* dst_offsets, void* stream) {
    const char* where = "vt_yuv420_crops_to_surface_rgb";
    VT_ENTER(h, enter(h, where, kHandle, 0, n, false, {planes, pitches, frame_hw, item_surface, dst, dst_offsets}));
    if (const int rc = check_yuv_format(h, where, format)) return rc;
    if (!(factor > 0)) return fail(h, VT_ERR_INVALID_ARG, "%s: factor must be positive", where);
    if (m < 0 || m > h->cfg.max_tracks) return fail(h, VT_ERR_INVALID_ARG, "%s: %d surfaces outside [0, max_tracks %d]", where, m, h->cfg.max_tracks);
    if (const int rc = boxes_xywh || slots ? VT_OK : check_tracks(h, where, first, n)) return rc;      // the state, by range
    if (slots) first = 0;
    cudaStream_t st = (cudaStream_t)stream;
    const YuvSurfaceArgs a{planes, pitches, frame_hw, m, item_surface, boxes_xywh, h->d_state, slots, h->d_claim, first, h->cfg.max_tracks,
                           factor, dst, dst_offsets, h->d_surf_rect, h->d_surf_done};
    if (slots) VT_LAUNCH(h, kNoStage, n, st, where, launch_claim_slots(slots, n, h->cfg.max_tracks, h->d_claim, st));
    VT_LAUNCH(h, kNoStage, n, st, where, launch_yuv420_crops_to_surface_rgb(format, a, n, h->num_sms, st));
    return VT_OK;
}

int64_t vt_launch_count(VtHandle h) { return h ? h->launches : 0; }

int vt_profile_enable(VtHandle h, int32_t enable) {
    if (!h) return VT_ERR_INVALID_ARG;
    h->profiling = enable != 0;
    return VT_OK;
}

int vt_profile_read(VtHandle h, double* stage_ms, int64_t* stage_launches, int64_t* stage_items) {
    if (!h || !stage_ms || !stage_launches || !stage_items) return h ? fail(h, VT_ERR_INVALID_ARG, "vt_profile_read: null pointer") : VT_ERR_INVALID_ARG;
    for (int i = 0; i < VT_NUM_STAGES; ++i) { stage_ms[i] = 0.0; stage_launches[i] = 0; stage_items[i] = 0; }
    for (auto& r : h->prof) {
        VT_CUDA(h, cudaEventSynchronize(r.b));
        float ms = 0.f;
        VT_CUDA(h, cudaEventElapsedTime(&ms, r.a, r.b));
        if (r.stage >= 0 && r.stage < VT_NUM_STAGES) { stage_ms[r.stage] += ms; stage_launches[r.stage] += 1; stage_items[r.stage] += r.items; }
        h->evpool.push_back(r.a); h->evpool.push_back(r.b);
    }
    h->prof.clear();
    return VT_OK;
}

// Development aid (not part of the documented ABI): which profiled stage launches have started / finished.  Non-blocking, meant to be
// called from a watchdog thread while the owning thread is stuck in a synchronisation.  out[i] = stage * 4 + (started ? 1 : 0) + (finished ? 2 : 0).
int vt_debug_pending(VtHandle h, int32_t* out, int32_t cap) {
    if (!h || !out) return -1;
    int k = 0;
    for (auto& r : h->prof) {
        if (k >= cap) break;
        out[k++] = r.stage * 4 + (cudaEventQuery(r.a) == cudaSuccess ? 1 : 0) + (cudaEventQuery(r.b) == cudaSuccess ? 2 : 0);
    }
    return k;
}

}  // extern "C"
