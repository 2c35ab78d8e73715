// C-ABI layer of libvittrack_b200.so: handle, weight ingestion (BN folding into the fp32 layouts; each tensor-core weight blob is packed
// by the file of the kernel that reads it),
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

namespace {

thread_local std::string g_create_error;

struct HostTensor {
    std::vector<float> data;
    std::vector<int64_t> shape;
};

}  // namespace

struct VtContext {
    VtConfig cfg;
    std::string err;
    std::map<std::string, HostTensor> tensors;
    bool finalized = false;
    bool tracks_ready = false;
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
    int32_t* d_status = nullptr;      // [max_tracks]
    float* d_maps = nullptr;          // [max_tracks][1280] score | size | offset of the last step
    int last_first = 0, last_n = 0;
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

bool expected_shape(const VtConfig& c, const std::string& name, std::vector<int64_t>& shp) {
    const int C = c.embed_dim, hc = c.head_channels;
    char buf[128];
    if (name == "pos_embed_z") { shp = {1, 64, C}; return true; }
    if (name == "pos_embed_x") { shp = {1, 256, C}; return true; }
    if (name == "norm.weight" || name == "norm.bias") { shp = {C}; return true; }
    if (name == "tracker.output_window") { shp = {1, 1, 16, 16}; return true; }
    const int ch[5] = {3, C / 8, C / 4, C / 2, C};
    for (int i = 0; i < 4; ++i) {
        snprintf(buf, sizeof buf, "patch_embed.net.%d.", 2 * i);
        if (name.rfind(buf, 0) == 0) {
            const std::string leaf = name.substr(strlen(buf));
            if (leaf == "c.weight") { shp = {ch[i + 1], ch[i], 3, 3}; return true; }
            if (leaf == "bn.weight" || leaf == "bn.bias" || leaf == "bn.running_mean" || leaf == "bn.running_var") { shp = {ch[i + 1]}; return true; }
            return false;
        }
    }
    for (int b = 0; b < c.depth; ++b) {
        snprintf(buf, sizeof buf, "blocks.%d.", b);
        if (name.rfind(buf, 0) == 0) {
            const std::string leaf = name.substr(strlen(buf));
            const int hid = c.mlp_ratio * C;
            if (leaf == "norm1.weight" || leaf == "norm1.bias" || leaf == "norm2.weight" || leaf == "norm2.bias") { shp = {C}; return true; }
            if (leaf == "attn.qkv.weight") { shp = {3 * C, C}; return true; }
            if (leaf == "attn.qkv.bias") { shp = {3 * C}; return true; }
            if (leaf == "attn.proj.weight") { shp = {C, C}; return true; }
            if (leaf == "attn.proj.bias") { shp = {C}; return true; }
            if (leaf == "mlp.fc1.weight") { shp = {hid, C}; return true; }
            if (leaf == "mlp.fc1.bias") { shp = {hid}; return true; }
            if (leaf == "mlp.fc2.weight") { shp = {C, hid}; return true; }
            if (leaf == "mlp.fc2.bias") { shp = {C}; return true; }
            return false;
        }
    }
    const int hch[5] = {C, hc, hc / 2, hc / 4, hc / 8};
    const int outs[3] = {1, 2, 2};
    for (int t = 0; t < 3; ++t) {
        for (int i = 0; i < 4; ++i) {
            snprintf(buf, sizeof buf, "box_head.conv%d_%s.", i + 1, kTowers[t]);
            if (name.rfind(buf, 0) == 0) {
                const std::string leaf = name.substr(strlen(buf));
                if (leaf == "0.weight") { shp = {hch[i + 1], hch[i], 3, 3}; return true; }
                if (leaf == "0.bias" || leaf == "1.weight" || leaf == "1.bias" || leaf == "1.running_mean" || leaf == "1.running_var") { shp = {hch[i + 1]}; return true; }
                return false;
            }
        }
        snprintf(buf, sizeof buf, "box_head.conv5_%s.", kTowers[t]);
        if (name.rfind(buf, 0) == 0) {
            const std::string leaf = name.substr(strlen(buf));
            if (leaf == "weight") { shp = {outs[t], hch[4], 1, 1}; return true; }
            if (leaf == "bias") { shp = {outs[t]}; return true; }
            return false;
        }
    }
    return false;
}

struct Packer {
    std::vector<float> buf;
    size_t alloc(size_t n) {                     // 16-byte aligned slots
        const size_t off = buf.size();
        buf.resize(off + (n + 3) / 4 * 4, 0.f);
        return off;
    }
};

// Tensor lookup of the finalisers: a tensor that was never set yields null and is listed in `missing`
struct TensorLookup {
    VtHandle h;
    std::string missing;
    const float* operator()(const std::string& n) {
        auto it = h->tensors.find(n);
        if (it == h->tensors.end()) { if (missing.size() < 300) missing += n + " "; return nullptr; }
        return it->second.data.data();
    }
};

// The packed weights -> h->d_weights (reallocated when it has grown); returns once the copy is done, as pk is the caller's local
int upload_weights(VtHandle h, const Packer& pk, cudaStream_t st) {
    if (h->d_weights && h->weights_floats < pk.buf.size()) { cudaFree(h->d_weights); h->d_weights = nullptr; }
    if (!h->d_weights) {
        VT_CUDA(h, cudaMalloc((void**)&h->d_weights, pk.buf.size() * sizeof(float)));
        h->weights_floats = pk.buf.size();
    }
    VT_CUDA(h, cudaMemcpyAsync(h->d_weights, pk.buf.data(), pk.buf.size() * sizeof(float), cudaMemcpyHostToDevice, st));
    VT_CUDA(h, cudaStreamSynchronize(st));
    return VT_OK;
}

void free_all(VtHandle h) {
    for (auto& r : h->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    for (auto e : h->evpool) cudaEventDestroy(e);
    cudaFree(h->d_weights); cudaFree(h->d_planes); cudaFree(h->d_scratch); cudaFree(h->d_taps); cudaFree(h->d_tokz);
    cudaFree(h->d_tokx); cudaFree(h->d_tok); cudaFree(h->d_state); cudaFree(h->d_tmpl);
    cudaFree(h->d_status); cudaFree(h->d_maps); cudaFree(h->d_gwork);
}

int check_ready(VtHandle h, bool need_tracks) {
    if (!h) return VT_ERR_INVALID_ARG;
    if (!h->finalized) return fail(h, VT_ERR_STATE, "weights not finalised: call vt_set_tensor for every tensor, then vt_finalize_weights");
    if (need_tracks && !h->tracks_ready) return fail(h, VT_ERR_STATE, "tracks not initialised: call vt_tracks_init first");
    return VT_OK;
}

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

// Launch one pipeline stage; when profiling is on, bracket it with events on the launching stream.
#define VT_LAUNCH(h, stage, items, st, where, expr)                               \
    do {                                                                          \
        cudaEvent_t ea__ = nullptr, eb__ = nullptr;                               \
        if ((h)->profiling) { ea__ = get_event(h); eb__ = get_event(h); cudaEventRecord(ea__, st); } \
        const int k__ = (expr);                                                   \
        if (k__ < 0) return launch_fail(h, k__, where);                           \
        (h)->launches += k__;                                                     \
        if ((h)->profiling) { cudaEventRecord(eb__, st); (h)->prof.push_back({stage, items, ea__, eb__}); } \
    } while (0)

int run_blocks(VtHandle h, const float* tokz, int zs, const float* tokx, int xs, float* out, int n, float* taps,
               size_t tap_stride, cudaStream_t st) {
    if (h->cfg.blocks_impl == VT_BLOCKS_SIMT_FP32)
        return launch_blocks_simt(tokz, zs, tokx, xs, out, n, h->mw, taps, tap_stride, st);
    return launch_blocks_tc(tokz, zs, tokx, xs, out, n, h->mw, taps, tap_stride, h->num_sms, h->cfg.blocks_impl == VT_BLOCKS_TCGEN05_3TERM ? 3 : 1, st);
}


// Hann window (hann.py:6-16; the tracker's own tensor when it was handed over) and normalisation table (data_utils.py:8-14)
void fill_hann_and_lut(VtHandle h, float* hann, float* lut) {
    auto it = h->tensors.find("tracker.output_window");
    if (it != h->tensors.end()) {
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

// Weights of the generic path: the reference's own layouts ([out][in]; conv [cout][ky][kx][cin]) with BatchNorm(eval) folded
// in float64 (Conv2d_BN.fuse vit_dist.py:22-33; head conv + bias -> BN, head.py:16-21).
int finalize_generic(VtHandle h, cudaStream_t st) {
    const VtConfig& c = h->cfg;
    const int C = c.embed_dim, hc = c.head_channels, hid = c.mlp_ratio * C;
    TensorLookup T{h};
    Packer pk;
    auto put = [&](const float* src, size_t n) { const size_t o = pk.alloc(n); if (src) memcpy(&pk.buf[o], src, n * sizeof(float)); return o; };
    const double eps = 1e-5;
    // conv [co][ci][3][3] (+ optional conv bias) with BN -> [co][(ky, kx, ci)], bias
    auto fold_conv = [&](const float* w, const float* cb, const float* g, const float* b, const float* m, const float* v, int co_n, int ci_n,
                         size_t& ow, size_t& ob) {
        ow = pk.alloc((size_t)co_n * 9 * ci_n); ob = pk.alloc(co_n);
        if (!(w && g && b && m && v)) return;
        for (int co = 0; co < co_n; ++co) {
            const double sc = (double)g[co] / sqrt((double)v[co] + eps);
            pk.buf[ob + co] = (float)((((cb ? (double)cb[co] : 0.0) - (double)m[co]) * sc) + (double)b[co]);
            for (int ci = 0; ci < ci_n; ++ci)
                for (int k = 0; k < 9; ++k)
                    pk.buf[ow + ((size_t)co * 9 + k) * ci_n + ci] = (float)((double)w[((size_t)co * ci_n + ci) * 9 + k] * sc);
        }
    };
    const int ch[5] = {3, C / 8, C / 4, C / 2, C};
    size_t sw[4], sb[4];
    for (int l = 0; l < 4; ++l) {
        const std::string p = "patch_embed.net." + std::to_string(2 * l) + ".";
        fold_conv(T(p + "c.weight"), nullptr, T(p + "bn.weight"), T(p + "bn.bias"), T(p + "bn.running_mean"), T(p + "bn.running_var"), ch[l + 1], ch[l], sw[l], sb[l]);
    }
    struct BO { size_t v[12]; };
    std::vector<BO> bo(c.depth);
    for (int b = 0; b < c.depth; ++b) {
        const std::string p = "blocks." + std::to_string(b) + ".";
        const char* names[12] = {"norm1.weight", "norm1.bias", "attn.qkv.weight", "attn.qkv.bias", "attn.proj.weight", "attn.proj.bias",
                                 "norm2.weight", "norm2.bias", "mlp.fc1.weight", "mlp.fc1.bias", "mlp.fc2.weight", "mlp.fc2.bias"};
        const size_t cnt[12] = {(size_t)C, (size_t)C, (size_t)3 * C * C, (size_t)3 * C, (size_t)C * C, (size_t)C,
                                (size_t)C, (size_t)C, (size_t)hid * C, (size_t)hid, (size_t)C * hid, (size_t)C};
        for (int i = 0; i < 12; ++i) bo[b].v[i] = put(T(p + names[i]), cnt[i]);
    }
    // split images of the blocks' Linear weights for the bulk-copy GEMM (same bytes as the fp32 matrices; packed on a few host threads)
    struct IO { size_t v[4]; };
    std::vector<IO> io(c.depth);
    if (h->gw.use_img) {
        const int wi[4] = {2, 4, 8, 10};                                       // qkv, proj, fc1, fc2 in `names`
        const int wn[4] = {3 * C, C, hid, C}, wk[4] = {C, C, C, hid};
        for (int b = 0; b < c.depth; ++b)
            for (int j = 0; j < 4; ++j) io[b].v[j] = pk.alloc(gen_img_bytes(wn[j], wk[j]) / 4);
        if (T.missing.empty())
            for (int b = 0; b < c.depth; ++b)
                for (int j = 0; j < 4; ++j)
                    gen_pack_weight_image(&pk.buf[bo[b].v[wi[j]]], wn[j], wk[j], reinterpret_cast<uint8_t*>(&pk.buf[io[b].v[j]]));
    }
    const size_t o_ng = put(T("norm.weight"), C), o_nb = put(T("norm.bias"), C);
    const size_t o_pz = put(T("pos_embed_z"), (size_t)kNz * C), o_px = put(T("pos_embed_x"), (size_t)kNx * C);
    // head: layer 1 merged over the towers (ctr | offset | size), layers 2-4 per tower, conv5 rows ctr, off x, off y, size w, size h
    const int hch[5] = {C, hc, hc / 2, hc / 4, hc / 8};
    const size_t o_w1 = pk.alloc((size_t)3 * hc * 9 * C), o_b1 = pk.alloc((size_t)3 * hc);
    size_t hw[3][3], hb[3][3];
    for (int t = 0; t < 3; ++t) {
        for (int i = 0; i < 4; ++i) {
            const std::string p = std::string("box_head.conv") + std::to_string(i + 1) + "_" + kTowers[t] + ".";
            size_t ow, ob;
            fold_conv(T(p + "0.weight"), T(p + "0.bias"), T(p + "1.weight"), T(p + "1.bias"), T(p + "1.running_mean"), T(p + "1.running_var"),
                      hch[i + 1], hch[i], ow, ob);
            if (i == 0) {       // copy into the merged layer (alloc moves pk.buf: index, do not hold pointers)
                for (size_t k = 0; k < (size_t)hc * 9 * C; ++k) pk.buf[o_w1 + (size_t)t * hc * 9 * C + k] = pk.buf[ow + k];
                for (int k = 0; k < hc; ++k) pk.buf[o_b1 + (size_t)t * hc + k] = pk.buf[ob + k];
            } else { hw[t][i - 1] = ow; hb[t][i - 1] = ob; }
        }
    }
    const size_t o_w5 = pk.alloc((size_t)5 * hch[4]), o_b5 = pk.alloc(5);
    {
        const int row0[3] = {0, 1, 3}, outs[3] = {1, 2, 2};
        for (int t = 0; t < 3; ++t) {
            const std::string p = std::string("box_head.conv5_") + kTowers[t] + ".";
            const float *w = T(p + "weight"), *b = T(p + "bias");
            if (!(w && b)) continue;
            for (int o = 0; o < outs[t]; ++o) {
                pk.buf[o_b5 + row0[t] + o] = b[o];
                for (int k = 0; k < hch[4]; ++k) pk.buf[o_w5 + (size_t)(row0[t] + o) * hch[4] + k] = w[(size_t)o * hch[4] + k];
            }
        }
    }
    if (!T.missing.empty()) return fail(h, VT_ERR_WEIGHTS, "missing tensors: %s", T.missing.c_str());
    const size_t o_hann = pk.alloc(256), o_lut = pk.alloc(768);
    fill_hann_and_lut(h, &pk.buf[o_hann], &pk.buf[o_lut]);
    // split images of the folded convolution weights (K = 9 cin must be a whole number of 32-wide panels)
    size_t isw[4] = {0, 0, 0, 0}, ihw1 = 0, ihw[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
    auto conv_img = [&](size_t w_off, int co_n, int ci_n) -> size_t {
        if (!h->gw.use_img || ci_n % 32 != 0) return 0;
        const size_t o = pk.alloc(gen_img_bytes(co_n, 9 * ci_n) / 4);
        gen_pack_weight_image(&pk.buf[w_off], co_n, 9 * ci_n, reinterpret_cast<uint8_t*>(&pk.buf[o]));
        return o;
    };
    for (int l = 1; l < 4; ++l) isw[l] = conv_img(sw[l], ch[l + 1], ch[l]);
    ihw1 = conv_img(o_w1, 3 * hc, C);
    for (int t = 0; t < 3; ++t)
        for (int l = 0; l < 3; ++l) ihw[t][l] = conv_img(hw[t][l], hch[l + 2], hch[l + 1]);

    if (const int rc = upload_weights(h, pk, st)) return rc;
    const float* base = h->d_weights;
    GenModelW& g = h->gw;
    for (int l = 0; l < 4; ++l) { g.stem_w[l] = base + sw[l]; g.stem_b[l] = base + sb[l]; }
    for (int b = 0; b < c.depth; ++b) {
        const float* q[12];
        for (int i = 0; i < 12; ++i) q[i] = base + bo[b].v[i];
        g.blk[b] = GenBlockW{q[0], q[1], q[2], q[3], q[4], q[5], q[6], q[7], q[8], q[9], q[10], q[11], nullptr, nullptr, nullptr, nullptr};
        if (g.use_img) {
            const uint8_t* ib[4];
            for (int j = 0; j < 4; ++j) ib[j] = reinterpret_cast<const uint8_t*>(base + io[b].v[j]);
            g.blk[b].iwqkv = ib[0]; g.blk[b].iwproj = ib[1]; g.blk[b].iwfc1 = ib[2]; g.blk[b].iwfc2 = ib[3];
        }
    }
    g.norm_g = base + o_ng; g.norm_b = base + o_nb; g.pos_z = base + o_pz; g.pos_x = base + o_px;
    g.head_w1 = base + o_w1; g.head_b1 = base + o_b1;
    for (int t = 0; t < 3; ++t)
        for (int l = 0; l < 3; ++l) { g.head_w[t][l] = base + hw[t][l]; g.head_b[t][l] = base + hb[t][l]; }
    g.head_w5 = base + o_w5; g.head_b5 = base + o_b5;
    g.hann = base + o_hann;
    auto imgp = [&](size_t o) { return o ? reinterpret_cast<const uint8_t*>(base + o) : nullptr; };
    for (int l = 0; l < 4; ++l) g.istem_w[l] = imgp(isw[l]);
    g.ihead_w1 = imgp(ihw1);
    for (int t = 0; t < 3; ++t)
        for (int l = 0; l < 3; ++l) g.ihead_w[t][l] = imgp(ihw[t][l]);
    h->mw.hann = base + o_hann; h->mw.lut = base + o_lut;         // the crop kernel reads the table through ModelW
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
    A((void**)&h->d_maps, mt * 1280 * sizeof(float));
    if (e == cudaSuccess) e = cudaMemset(h->d_state, 0, mt * 4 * sizeof(double));
    if (e == cudaSuccess) e = cudaMemset(h->d_status, 0, mt * sizeof(int32_t));
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
    std::vector<int64_t> want;
    if (!expected_shape(h->cfg, nm, want)) return fail(h, VT_ERR_WEIGHTS, "unknown tensor '%s' (ignored, as load_state_dict(strict=False) would)", name);
    if (!data_host) return fail(h, VT_ERR_INVALID_ARG, "vt_set_tensor: null data for '%s'", name);
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
    if (h->generic) return finalize_generic(h, st);
    TensorLookup T{h};
    Packer pk;
    auto slot = [&](size_t n) { return pk.alloc(n); };
    const double eps = 1e-5;     // BatchNorm2d default eps

    // ---- stem: fold BN (Conv2d_BN.fuse, vit_dist.py:22-33), repack [co][ci][3][3] -> [ci][ky][kx][co]
    const int ch[5] = {3, 6, 12, 24, 48};
    size_t stem_w[4], stem_b[4];
    for (int l = 0; l < 4; ++l) {
        const std::string p = "patch_embed.net." + std::to_string(2 * l) + ".";
        const float *w = T(p + "c.weight"), *g = T(p + "bn.weight"), *b = T(p + "bn.bias"), *m = T(p + "bn.running_mean"), *v = T(p + "bn.running_var");
        const int ci_n = ch[l], co_n = ch[l + 1];
        stem_w[l] = slot((size_t)ci_n * 9 * co_n);
        stem_b[l] = slot(co_n);
        if (!(w && g && b && m && v)) continue;
        for (int co = 0; co < co_n; ++co) {
            const double s = (double)g[co] / sqrt((double)v[co] + eps);
            pk.buf[stem_b[l] + co] = (float)((double)b[co] - (double)m[co] * s);
            for (int ci = 0; ci < ci_n; ++ci)
                for (int k = 0; k < 9; ++k)
                    pk.buf[stem_w[l] + ((size_t)ci * 9 + k) * co_n + co] = (float)((double)w[((size_t)co * ci_n + ci) * 9 + k] * s);
        }
    }
    // ---- stem conv3 / conv4 for the tensor cores: fp16 hi | lo weight blobs in the kernels' K-step order (vt_stem_tc.cu)
    size_t stc_w[3], stc_b[3];
    {
        const int lcin[3] = {6, 12, 24}, lcch[3] = {kConv2Cch, kConv3Cch, kConv4Cch}, lcout[3] = {12, 24, 48}, lnpad[3] = {16, 32, 48};
        for (int i = 0; i < 3; ++i) {
            const int l = 1 + i;
            const size_t bytes = stem_tc_weight_bytes(i);
            stc_w[i] = slot(bytes / 4);
            stc_b[i] = slot(lnpad[i]);
            uint8_t* hi8 = reinterpret_cast<uint8_t*>(&pk.buf[stc_w[i]]);
            for (int co = 0; co < lcout[i]; ++co) pk.buf[stc_b[i] + co] = pk.buf[stem_b[l] + co];
            stem_tc_pack_weights(lcin[i], lcch[i], lcout[i], lnpad[i], &pk.buf[stem_w[l]], hi8, hi8 + bytes / 2);
        }
    }
    // ---- stem conv1 for the fused tensor-core front (vt_stem_fused.cu): pixel normalisation folded into the weights / border-variant biases
    const size_t s1_w = slot(kStem1TcWBytes / 4), s1_p = slot(kStem1TcParFloats);
    stem1_tc_pack(&pk.buf[stem_w[0]], &pk.buf[stem_b[0]], reinterpret_cast<uint8_t*>(&pk.buf[s1_w]), &pk.buf[s1_p]);
    // ---- blocks: Linear weights [out][in] -> K-major [in][out]
    struct BOff { size_t ln1g, ln1b, wqkv, bqkv, wproj, bproj, ln2g, ln2b, wfc1, bfc1, wfc2, bfc2; } bo[kDepth];
    BlockTensors bt[kDepth];
    auto copyv = [&](size_t o, const float* src, size_t n) { if (src) memcpy(&pk.buf[o], src, n * sizeof(float)); };
    auto transp = [&](size_t o, const float* src, int rows_out, int cols_in) {     // src [out][in] -> dst [in][out]
        if (!src) return;
        for (int r = 0; r < rows_out; ++r)
            for (int c = 0; c < cols_in; ++c) pk.buf[o + (size_t)c * rows_out + r] = src[(size_t)r * cols_in + c];
    };
    for (int b = 0; b < kDepth; ++b) {
        const std::string p = "blocks." + std::to_string(b) + ".";
        BlockTensors& t = bt[b];
        t = {T(p + "norm1.weight"), T(p + "norm1.bias"), T(p + "attn.qkv.weight"), T(p + "attn.qkv.bias"), T(p + "attn.proj.weight"),
             T(p + "attn.proj.bias"), T(p + "norm2.weight"), T(p + "norm2.bias"), T(p + "mlp.fc1.weight"), T(p + "mlp.fc1.bias"),
             T(p + "mlp.fc2.weight"), T(p + "mlp.fc2.bias")};
        bo[b].ln1g = slot(kC); copyv(bo[b].ln1g, t.ln1_g, kC);
        bo[b].ln1b = slot(kC); copyv(bo[b].ln1b, t.ln1_b, kC);
        bo[b].wqkv = slot(kC * 3 * kC); transp(bo[b].wqkv, t.wqkv, 3 * kC, kC);
        bo[b].bqkv = slot(3 * kC); copyv(bo[b].bqkv, t.bqkv, 3 * kC);
        bo[b].wproj = slot(kC * kC); transp(bo[b].wproj, t.wproj, kC, kC);
        bo[b].bproj = slot(kC); copyv(bo[b].bproj, t.bproj, kC);
        bo[b].ln2g = slot(kC); copyv(bo[b].ln2g, t.ln2_g, kC);
        bo[b].ln2b = slot(kC); copyv(bo[b].ln2b, t.ln2_b, kC);
        bo[b].wfc1 = slot(kC * kHid); transp(bo[b].wfc1, t.wfc1, kHid, kC);
        bo[b].bfc1 = slot(kHid); copyv(bo[b].bfc1, t.bfc1, kHid);
        bo[b].wfc2 = slot(kHid * kC); transp(bo[b].wfc2, t.wfc2, kC, kHid);
        bo[b].bfc2 = slot(kC); copyv(bo[b].bfc2, t.bfc2, kC);
    }
    // ---- the same blocks for the tensor cores (vt_block_tc.cu), packed only when every tensor looked up so far is present
    size_t tc_wa[kDepth], tc_wb[kDepth], tc_par[kDepth];
    for (int b = 0; b < kDepth; ++b) {
        tc_wa[b] = slot(kTcWaBytes / 4); tc_wb[b] = slot(kTcWbBytes / 4); tc_par[b] = slot(kTcParFloats);
        if (T.missing.empty())
            block_tc_pack(bt[b], reinterpret_cast<uint8_t*>(&pk.buf[tc_wa[b]]), reinterpret_cast<uint8_t*>(&pk.buf[tc_wb[b]]), &pk.buf[tc_par[b]]);
    }
    const size_t o_ng = slot(kC), o_nb = slot(kC), o_pz = slot(kNz * kC), o_px = slot(kNx * kC);
    copyv(o_ng, T("norm.weight"), kC); copyv(o_nb, T("norm.bias"), kC);
    copyv(o_pz, T("pos_embed_z"), kNz * kC); copyv(o_px, T("pos_embed_x"), kNx * kC);

    // ---- head: conv(+bias) -> BN folded; layer i weights laid out [ci][k][tower][co_t]
    const int hch[5] = {kC, kHeadC, kHeadC / 2, kHeadC / 4, kHeadC / 8};
    size_t hw[5], hb[5];
    for (int i = 0; i < 4; ++i) {
        const int ci_n = hch[i], co_n = hch[i + 1];
        hw[i] = slot((size_t)ci_n * 9 * 3 * co_n);
        hb[i] = slot(3 * co_n);
        for (int t = 0; t < 3; ++t) {
            const std::string p = std::string("box_head.conv") + std::to_string(i + 1) + "_" + kTowers[t] + ".";
            const float *w = T(p + "0.weight"), *cb = T(p + "0.bias"), *g = T(p + "1.weight"), *b = T(p + "1.bias"), *m = T(p + "1.running_mean"), *v = T(p + "1.running_var");
            if (!(w && cb && g && b && m && v)) continue;
            for (int co = 0; co < co_n; ++co) {
                const double s = (double)g[co] / sqrt((double)v[co] + eps);
                pk.buf[hb[i] + t * co_n + co] = (float)(((double)cb[co] - (double)m[co]) * s + (double)b[co]);
                for (int ci = 0; ci < ci_n; ++ci)
                    for (int k = 0; k < 9; ++k)
                        pk.buf[hw[i] + (((size_t)ci * 9 + k) * 3 + t) * co_n + co] = (float)((double)w[((size_t)co * ci_n + ci) * 9 + k] * s);
            }
        }
    }
    // head conv1 - conv3 for the tensor cores (vt_head.cu)
    size_t o_htc[3];
    for (int i = 0; i < 3; ++i) o_htc[i] = slot(head_tc_weight_bytes(i) / 4);
    head_tc_pack(&pk.buf[hw[0]], &pk.buf[hw[1]], &pk.buf[hw[2]], reinterpret_cast<uint8_t*>(&pk.buf[o_htc[0]]),
                 reinterpret_cast<uint8_t*>(&pk.buf[o_htc[1]]), reinterpret_cast<uint8_t*>(&pk.buf[o_htc[2]]));
    hw[4] = slot(3 * 4 * 2); hb[4] = slot(3 * 2);
    for (int t = 0; t < 3; ++t) {
        const std::string p = std::string("box_head.conv5_") + kTowers[t] + ".";
        const float *w = T(p + "weight"), *b = T(p + "bias");
        if (!(w && b)) continue;
        const int outs = t == 0 ? 1 : 2;
        for (int o = 0; o < outs; ++o) {
            pk.buf[hb[4] + t * 2 + o] = b[o];
            for (int c = 0; c < 4; ++c) pk.buf[hw[4] + (t * 4 + c) * 2 + o] = w[o * 4 + c];
        }
    }
    if (!T.missing.empty()) return fail(h, VT_ERR_WEIGHTS, "missing tensors: %s", T.missing.c_str());

    // ---- Hann window (hann.py:6-16) and normalisation table (data_utils.py:8-14) -----------------
    const size_t o_hann = slot(256), o_lut = slot(768);
    fill_hann_and_lut(h, &pk.buf[o_hann], &pk.buf[o_lut]);

    if (const int rc = upload_weights(h, pk, st)) return rc;
    const float* base = h->d_weights;
    ModelW& m = h->mw;
    for (int l = 0; l < 4; ++l) { m.stem[l].w = base + stem_w[l]; m.stem[l].b = base + stem_b[l]; }
    for (int b = 0; b < kDepth; ++b) {
        BlockW& B = m.blk[b];
        B.ln1_g = base + bo[b].ln1g; B.ln1_b = base + bo[b].ln1b; B.wqkv = base + bo[b].wqkv; B.bqkv = base + bo[b].bqkv;
        B.wproj = base + bo[b].wproj; B.bproj = base + bo[b].bproj; B.ln2_g = base + bo[b].ln2g; B.ln2_b = base + bo[b].ln2b;
        B.wfc1 = base + bo[b].wfc1; B.bfc1 = base + bo[b].bfc1; B.wfc2 = base + bo[b].wfc2; B.bfc2 = base + bo[b].bfc2;
        m.tc[b].wa = reinterpret_cast<const uint8_t*>(base + tc_wa[b]);
        m.tc[b].wb = reinterpret_cast<const uint8_t*>(base + tc_wb[b]);
        m.tc[b].par = base + tc_par[b];
    }
    m.norm_g = base + o_ng; m.norm_b = base + o_nb; m.pos_z = base + o_pz; m.pos_x = base + o_px;
    m.head.w1 = base + hw[0]; m.head.b1 = base + hb[0]; m.head.w2 = base + hw[1]; m.head.b2 = base + hb[1];
    m.head.w3 = base + hw[2]; m.head.b3 = base + hb[2]; m.head.w4 = base + hw[3]; m.head.b4 = base + hb[3];
    m.head.w5 = base + hw[4]; m.head.b5 = base + hb[4];
    m.head_tc_w1 = reinterpret_cast<const uint8_t*>(base + o_htc[0]);
    m.head_tc_w2 = reinterpret_cast<const uint8_t*>(base + o_htc[1]);
    m.head_tc_w3 = reinterpret_cast<const uint8_t*>(base + o_htc[2]);
    for (int i = 0; i < 3; ++i) { m.stem_tc_w[i] = reinterpret_cast<const uint8_t*>(base + stc_w[i]); m.stem_tc_b[i] = base + stc_b[i]; }
    m.stem1_tc_w = reinterpret_cast<const uint8_t*>(base + s1_w); m.stem1_tc_par = base + s1_p;
    m.hann = base + o_hann; m.lut = base + o_lut;
    h->finalized = true;
    return VT_OK;
}

int vt_crop_normalize(VtHandle h, const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw,
                      const double* boxes_xywh, double factor, int32_t out_size, int32_t n, float* out_nchw,
                      uint8_t* out_u8_hwc, uint8_t* out_mask, double* out_resize_factor, int32_t* out_status,
                      void* stream) {
    int rc = check_ready(h, false);
    if (rc) return rc;
    if (n == 0) return VT_OK;                      // an empty batch is a no-op (its pointers may be null)
    if (!frames || !frame_offsets || !frame_hw || !boxes_xywh || !out_nchw || n < 0) return fail(h, VT_ERR_INVALID_ARG, "vt_crop_normalize: null pointer or negative n");
    if (out_size != 128 && out_size != 256) return fail(h, VT_ERR_UNSUPPORTED, "vt_crop_normalize: out_size must be 128 or 256");
    if (!(factor > 0)) return fail(h, VT_ERR_INVALID_ARG, "vt_crop_normalize: factor must be positive");
    DeviceGuard dg(h->cfg.device);
    VT_CUDA(h, dg.err);
    const int k = launch_crop_normalize(frames, frame_offsets, frame_hw, boxes_xywh, factor, out_size, n, h->mw.lut, out_nchw,
                                        out_u8_hwc, out_mask, out_resize_factor, out_status, (cudaStream_t)stream);
    if (k < 0) return fail(h, VT_ERR_CUDA, "crop kernel launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    h->launches += k;
    return VT_OK;
}

int vt_forward(VtHandle h, const float* z, const float* x, int32_t n, float* pred_boxes, float* score_map,
               float* size_map, float* offset_map, float* taps, void* stream) {
    int rc = check_ready(h, false);
    if (rc) return rc;
    if (n == 0) return VT_OK;
    if (!z || !x || n < 0) return fail(h, VT_ERR_INVALID_ARG, "vt_forward: null input or negative n");
    cudaStream_t st = (cudaStream_t)stream;
    DeviceGuard dg(h->cfg.device);
    VT_CUDA(h, dg.err);
    if (h->generic) {
        const int C = h->cfg.embed_dim;
        const size_t gtap = (size_t)n * kN * C;
        for (int first = 0; first < n; first += h->chunk) {
            const int m = (n - first < h->chunk) ? n - first : h->chunk;
            VT_LAUNCH(h, VT_STAGE_STEM, m, st, "vt_forward/stem(z)", gen_launch_stem(z + (size_t)first * 3 * kTz * kTz, kTz, m, h->gw, h->gws, h->gws.tok, kN, 0, st));
            VT_LAUNCH(h, VT_STAGE_STEM, m, st, "vt_forward/stem(x)", gen_launch_stem(x + (size_t)first * 3 * kSx * kSx, kSx, m, h->gw, h->gws, h->gws.tok, kN, kNz, st));
            HeadArgs a{};
            a.n = m;
            a.pred_boxes = pred_boxes ? pred_boxes + (size_t)first * 4 : nullptr;
            a.score_map = score_map ? score_map + (size_t)first * 256 : nullptr;
            a.size_map = size_map ? size_map + (size_t)first * 512 : nullptr;
            a.offset_map = offset_map ? offset_map + (size_t)first * 512 : nullptr;
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
        VT_LAUNCH(h, VT_STAGE_BLOCKS, m, st, "vt_forward/blocks", run_blocks(h, h->d_tokz, kNz, h->d_tokx, kNx, h->d_tok, m,
                                                      taps ? taps + (size_t)first * kN * kC : nullptr, tap_stride, st));
        HeadArgs a{};
        a.tokens = h->d_tok; a.n = m;
        a.pred_boxes = pred_boxes ? pred_boxes + (size_t)first * 4 : nullptr;
        a.score_map = score_map ? score_map + (size_t)first * 256 : nullptr;
        a.size_map = size_map ? size_map + (size_t)first * 512 : nullptr;
        a.offset_map = offset_map ? offset_map + (size_t)first * 512 : nullptr;
        a.tokens_norm = taps ? taps + (size_t)(kDepth + 1) * tap_stride + (size_t)first * kN * kC : nullptr;
        a.use_tc = h->cfg.blocks_impl != VT_BLOCKS_SIMT_FP32;
        VT_LAUNCH(h, VT_STAGE_HEAD, m, st, "vt_forward/head", launch_head(a, h->mw, st));
    }
    return VT_OK;
}

int vt_cal_bbox(VtHandle h, const float* score, const float* size_map, const float* offset_map, int32_t n,
                float* boxes, void* stream) {
    if (!h) return VT_ERR_INVALID_ARG;
    if (!score || !size_map || !offset_map || !boxes || n < 0) return fail(h, VT_ERR_INVALID_ARG, "vt_cal_bbox: null pointer or negative n");
    DeviceGuard dg(h->cfg.device);
    VT_CUDA(h, dg.err);
    const int k = launch_cal_bbox(score, size_map, offset_map, n, boxes, (cudaStream_t)stream);
    if (k < 0) return fail(h, VT_ERR_CUDA, "cal_bbox launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    h->launches += k;
    return VT_OK;
}

int vt_tracks_init(VtHandle h, const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw,
                   const double* boxes_xywh, int32_t first, int32_t n, int32_t* out_status, void* stream) {
    int rc = check_ready(h, false);
    if (rc) return rc;
    if (n == 0) { h->tracks_ready = true; return VT_OK; }
    if (!frames || !frame_offsets || !frame_hw || !boxes_xywh) return fail(h, VT_ERR_INVALID_ARG, "vt_tracks_init: null pointer");
    if (first < 0 || n < 0 || first + n > h->cfg.max_tracks) return fail(h, VT_ERR_INVALID_ARG, "vt_tracks_init: tracks [%d, %d) exceed max_tracks %d", first, first + n, h->cfg.max_tracks);
    cudaStream_t st = (cudaStream_t)stream;
    DeviceGuard dg(h->cfg.device);
    VT_CUDA(h, dg.err);
    for (int c0 = 0; c0 < n && h->generic; c0 += h->chunk) {
        const int m = (n - c0 < h->chunk) ? n - c0 : h->chunk;
        VT_LAUNCH(h, VT_STAGE_CROP, m, st, "vt_tracks_init/crop",
                  launch_crop_normalize(frames, frame_offsets + c0, frame_hw + 2 * c0, boxes_xywh + 4 * c0, h->cfg.template_factor, kTz, m, h->mw.lut,
                                        h->gws.crop, nullptr, nullptr, nullptr, h->d_status + first + c0, st));
        VT_LAUNCH(h, VT_STAGE_STEM, m, st, "vt_tracks_init/stem",
                  gen_launch_stem(h->gws.crop, kTz, m, h->gw, h->gws, h->d_tmpl + (size_t)(first + c0) * kNz * h->cfg.embed_dim, kNz, 0, st));
    }
    for (int c0 = 0; c0 < n && !h->generic; c0 += h->chunk) {
        const int m = (n - c0 < h->chunk) ? n - c0 : h->chunk;
        VT_LAUNCH(h, VT_STAGE_STEM, m, st, "vt_tracks_init/crop+stem",
                  launch_crop_stem(frames, frame_offsets + c0, frame_hw + 2 * c0, boxes_xywh + 4 * c0, h->cfg.template_factor, kTz, m,
                                   h->mw, h->d_scratch, h->d_tmpl + (size_t)(first + c0) * kNz * kC, kNz, 0, h->d_status + first + c0,
                                   h->d_planes, h->chunk, h->d_taps, st));
    }
    VT_CUDA(h, cudaMemcpyAsync(h->d_state + (size_t)first * 4, boxes_xywh, (size_t)n * 4 * sizeof(double), cudaMemcpyDeviceToDevice, st));
    if (out_status) VT_CUDA(h, cudaMemcpyAsync(out_status, h->d_status + first, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
    h->tracks_ready = true;
    return VT_OK;
}

int vt_tracks_step(VtHandle h, const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw,
                   int32_t first, int32_t n, double* out_boxes, double* out_detail, int32_t update_state, void* stream) {
    int rc = check_ready(h, true);
    if (rc) return rc;
    if (n == 0) return VT_OK;
    if (!frames || !frame_offsets || !frame_hw || !out_boxes) return fail(h, VT_ERR_INVALID_ARG, "vt_tracks_step: null pointer");
    if (first < 0 || n < 0 || first + n > h->cfg.max_tracks) return fail(h, VT_ERR_INVALID_ARG, "vt_tracks_step: tracks [%d, %d) exceed max_tracks %d", first, first + n, h->cfg.max_tracks);
    cudaStream_t st = (cudaStream_t)stream;
    DeviceGuard dg(h->cfg.device);
    VT_CUDA(h, dg.err);
    if (h->generic) {
        // every stage runs per chunk: crop -> stem into the chunk's token buffer, cached template tokens copied in front
        const int C = h->cfg.embed_dim;
        for (int c0 = 0; c0 < n; c0 += h->chunk) {
            const int m = (n - c0 < h->chunk) ? n - c0 : h->chunk;
            const int t0 = first + c0;
            VT_LAUNCH(h, VT_STAGE_CROP, m, st, "vt_tracks_step/crop",
                      launch_crop_normalize(frames, frame_offsets + c0, frame_hw + 2 * c0, h->d_state + (size_t)t0 * 4, h->cfg.search_factor, kSx, m,
                                            h->mw.lut, h->gws.crop, nullptr, nullptr, nullptr, h->d_status + t0, st));
            VT_CUDA(h, cudaMemcpy2DAsync(h->gws.tok, (size_t)kN * C * sizeof(float), h->d_tmpl + (size_t)t0 * kNz * C, (size_t)kNz * C * sizeof(float),
                                         (size_t)kNz * C * sizeof(float), m, cudaMemcpyDeviceToDevice, st));
            VT_LAUNCH(h, VT_STAGE_STEM, m, st, "vt_tracks_step/stem", gen_launch_stem(h->gws.crop, kSx, m, h->gw, h->gws, h->gws.tok, kN, kNz, st));
            HeadArgs a{};
            a.n = m;
            a.score_map = h->d_maps + (size_t)t0 * 256;
            a.size_map = h->d_maps + (size_t)h->cfg.max_tracks * 256 + (size_t)t0 * 512;
            a.offset_map = h->d_maps + (size_t)h->cfg.max_tracks * 768 + (size_t)t0 * 512;
            a.state = h->d_state + (size_t)t0 * 4;
            a.frame_hw = frame_hw + 2 * c0;
            a.status = h->d_status + t0;
            a.out_boxes = out_boxes + (size_t)c0 * 5;
            a.out_detail = out_detail ? out_detail + (size_t)c0 * 8 : nullptr;
            a.update_state = update_state;
            a.search_factor = h->cfg.search_factor;
            VT_LAUNCH(h, VT_STAGE_BLOCKS, m, st, "vt_tracks_step/blocks+head", gen_launch_blocks_head(h->gws.tok, m, h->gw, h->gws, a, nullptr, 0, st));
        }
        h->last_first = first; h->last_n = n;
        return VT_OK;
    }
    // crop + stem run per chunk (their intermediates are large); blocks + head run once over all n tracks
    for (int c0 = 0; c0 < n; c0 += h->chunk) {
        const int m = (n - c0 < h->chunk) ? n - c0 : h->chunk;
        const int t0 = first + c0;
        VT_LAUNCH(h, VT_STAGE_STEM, m, st, "vt_tracks_step/crop+stem",
                  launch_crop_stem(frames, frame_offsets + c0, frame_hw + 2 * c0, h->d_state + (size_t)t0 * 4, h->cfg.search_factor, kSx, m,
                                   h->mw, h->d_scratch, h->d_tokx + (size_t)c0 * kNx * kC, kNx, 0, h->d_status + t0,
                                   h->d_planes, h->chunk, h->d_taps, st));
    }
    {
        const int m = n;
        VT_LAUNCH(h, VT_STAGE_BLOCKS, m, st, "vt_tracks_step/blocks",
                  run_blocks(h, h->d_tmpl + (size_t)first * kNz * kC, kNz, h->d_tokx, kNx, h->d_tok, m, nullptr, 0, st));
        HeadArgs a{};
        a.tokens = h->d_tok; a.n = m;
        // maps of the last step are kept planar per array: score [max][256] | size [max][512] | offset [max][512]
        a.score_map = h->d_maps + (size_t)first * 256;
        a.size_map = h->d_maps + (size_t)h->cfg.max_tracks * 256 + (size_t)first * 512;
        a.offset_map = h->d_maps + (size_t)h->cfg.max_tracks * 768 + (size_t)first * 512;
        a.state = h->d_state + (size_t)first * 4;
        a.frame_hw = frame_hw;
        a.status = h->d_status + first;
        a.out_boxes = out_boxes;
        a.out_detail = out_detail;
        a.update_state = update_state;
        a.search_factor = h->cfg.search_factor;
        a.use_tc = h->cfg.blocks_impl != VT_BLOCKS_SIMT_FP32;
        VT_LAUNCH(h, VT_STAGE_HEAD, m, st, "vt_tracks_step/head", launch_head(a, h->mw, st));
    }
    h->last_first = first; h->last_n = n;
    return VT_OK;
}

int vt_tracks_get_state(VtHandle h, double* boxes_xywh, int32_t first, int32_t n, void* stream) {
    if (!h) return VT_ERR_INVALID_ARG;
    if (!boxes_xywh || first < 0 || n < 0 || first + n > h->cfg.max_tracks) return fail(h, VT_ERR_INVALID_ARG, "vt_tracks_get_state: bad range");
    VT_CUDA(h, cudaMemcpyAsync(boxes_xywh, h->d_state + (size_t)first * 4, (size_t)n * 4 * sizeof(double), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return VT_OK;
}

int vt_tracks_set_state(VtHandle h, const double* boxes_xywh, int32_t first, int32_t n, void* stream) {
    if (!h) return VT_ERR_INVALID_ARG;
    if (!boxes_xywh || first < 0 || n < 0 || first + n > h->cfg.max_tracks) return fail(h, VT_ERR_INVALID_ARG, "vt_tracks_set_state: bad range");
    VT_CUDA(h, cudaMemcpyAsync(h->d_state + (size_t)first * 4, boxes_xywh, (size_t)n * 4 * sizeof(double), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return VT_OK;
}

int vt_tracks_last_maps(VtHandle h, int32_t first, int32_t n, float* score_map, float* size_map, float* offset_map, void* stream) {
    if (!h) return VT_ERR_INVALID_ARG;
    if (first < h->last_first || n < 0 || first + n > h->last_first + h->last_n) return fail(h, VT_ERR_STATE, "vt_tracks_last_maps: tracks [%d, %d) were not part of the last step", first, first + n);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t mt = h->cfg.max_tracks;
    if (score_map) VT_CUDA(h, cudaMemcpyAsync(score_map, h->d_maps + (size_t)first * 256, (size_t)n * 256 * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (size_map) VT_CUDA(h, cudaMemcpyAsync(size_map, h->d_maps + mt * 256 + (size_t)first * 512, (size_t)n * 512 * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (offset_map) VT_CUDA(h, cudaMemcpyAsync(offset_map, h->d_maps + mt * 768 + (size_t)first * 512, (size_t)n * 512 * sizeof(float), cudaMemcpyDeviceToDevice, st));
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
    if (!h) return VT_ERR_INVALID_ARG;
    if (format != VT_FRAME_NV12 && format != VT_FRAME_I420) return fail(h, VT_ERR_INVALID_ARG, "vt_upload_yuv420_rect: unknown format %d", format);
    if (!image || !staging || !staging_dev || !frame_rgb_dev) return fail(h, VT_ERR_INVALID_ARG, "vt_upload_yuv420_rect: null pointer");
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
    DeviceGuard dg(h->cfg.device);
    VT_CUDA(h, dg.err);
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
    const int k = launch_yuv420_rect(format, d, h->num_sms, st);
    if (k < 0) return fail(h, VT_ERR_CUDA, "vt_upload_yuv420_rect: kernel launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    h->launches += k;
    return VT_OK;
}

int vt_yuv420_to_rgb(VtHandle h, int32_t format, const uint8_t* src, const int64_t* src_offsets, const int32_t* frame_hw,
                     uint8_t* dst, const int64_t* dst_offsets, int32_t n, void* stream) {
    if (!h) return VT_ERR_INVALID_ARG;
    if (format != VT_FRAME_NV12 && format != VT_FRAME_I420) return fail(h, VT_ERR_INVALID_ARG, "vt_yuv420_to_rgb: unknown format %d", format);
    if (n < 0) return fail(h, VT_ERR_INVALID_ARG, "vt_yuv420_to_rgb: negative n");
    if (n == 0) return VT_OK;
    if (!src || !src_offsets || !frame_hw || !dst || !dst_offsets) return fail(h, VT_ERR_INVALID_ARG, "vt_yuv420_to_rgb: null pointer");
    DeviceGuard dg(h->cfg.device);
    VT_CUDA(h, dg.err);
    const int k = launch_yuv420_to_rgb(format, src, src_offsets, frame_hw, dst, dst_offsets, n, h->num_sms, (cudaStream_t)stream);
    if (k < 0) return fail(h, VT_ERR_CUDA, "vt_yuv420_to_rgb: kernel launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    h->launches += k;
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
