// K4 + K5: final LayerNorm on the search tokens, CENTER head (three conv towers) and the tracker's
// post-processing, one CTA per track with every activation resident in shared memory.
//   forward_head        lib/models/vit_dist/vit_dist.py:94,122-153
//   CenterPredictor     lib/models/layers/head.py:98-201 (conv+bias -> BN(eval) -> ReLU x4, conv1x1,
//                       sigmoid+clamp on ctr/size, raw offset; BN folded at weight-pack time)
//   cal_bbox            lib/models/layers/head.py:142-160 (first arg-max wins)
//   track() epilogue    lib/test/tracker/vit_dist.py:103-111,147-156 + lib/utils/box_ops.py:97-106
// The three towers' first convolutions share their input and are merged into one 48->96 layer whose
// 166 KB of weights are streamed through a double-buffered cp.async ring; later layers reuse the ring.
//
// head_tc_kernel runs the first two convolution layers (48 -> 96 merged and 32 -> 16 per tower, 92 % of the head's
// FLOPs) on the tcgen05 tensor cores instead: the LayerNorm output is written to shared memory as fp16 hi/lo in 8-channel chunks
// [chunk][row 0..17][x 0..15][8] (a zero row above and below), which a no-swizzle K-major UMMA descriptor can
// address for any vertical tap by moving its start row.  Horizontal taps are not gathered at all: for each kx
// one accumulator T_kx[y][x'] = sum_{ky,ci} in[y+ky-1][x'][ci] W[ci][ky][kx][co] is built in TMEM over the
// UNSHIFTED columns, and the epilogue adds T_0[y][x-1] + T_1[y][x] + T_2[y][x+1] with warp shuffles (a
// warp's 32 TMEM lanes are two complete image rows).  Products are hi*hi + lo*hi + hi*lo as in the blocks.
// head_tc_kernel is PERSISTENT (one CTA per SM walks over tracks: TMEM and the bias block are set up once, the mbarriers are
// re-initialised per track); a track's 256 search tokens arrive with one bulk copy - the next track's while the current one runs
// its last layers - and are normalised out of shared memory.
#include "vt_geom.cuh"
#include "vt_internal.h"
#include "vt_tc.cuh"
#include "vt_decode.cuh"

namespace vt {

#ifdef VT_HEAD_TRACE
__device__ long long g_head_trace[32];
#define HEAD_TRACE(i) do { if (blockIdx.x == 0 && threadIdx.x == 0) g_head_trace[i] = clock64(); } while (0)
#define HEAD_TRACE_NS(i) do { if (blockIdx.x == 0 && threadIdx.x == 0) { long long t__; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t__)); g_head_trace[i] = t__; } } while (0)
extern "C" int vt_head_trace_read(long long* host) { cudaDeviceSynchronize(); return (int)cudaMemcpyFromSymbol(host, g_head_trace, sizeof(long long) * 32); }
#else
#define HEAD_TRACE(i) do {} while (0)
#define HEAD_TRACE_NS(i) do {} while (0)
#endif

// max that keeps NaN (fmaxf returns the other operand): the ReLUs and the running maximum of the tensor-core epilogues must not
// squash a NaN born from an overflowed fp16 operand or weight into a plausible number - the range guard has to see it
__device__ __forceinline__ float max_nan(float a, float b) {
    float r;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return r;
}

constexpr int kHeadThreads = 256;
constexpr int kPlane = 18 * 18;                      // zero-bordered 16x16 plane
constexpr int kWChunk = 3456;                        // floats per streamed weight chunk
constexpr int kOffFeat = 0;                          // [48][324]  feat, later conv2 output
constexpr int kOffOut1 = kOffFeat + 48 * kPlane;     // [96][324]  conv1 output, later conv3/conv4 outputs
constexpr int kOffW = kOffOut1 + 96 * kPlane;        // 2 x kWChunk
constexpr int kOffBias = kOffW + 2 * kWChunk;        // b1[96] b2[48] b3[24] b4[12] w5[24] b5[6] -> 256
constexpr int kOffMaps = kOffBias + 256;             // score[256] size[2][256] offset[2][256] resp[256]
constexpr int kOffRed = kOffMaps + 6 * 256;          // reduction scratch (32 floats)
constexpr int kHeadFloats = kOffRed + 32;
constexpr size_t kHeadSmemBytes = (size_t)kHeadFloats * sizeof(float);
static_assert(kHeadSmemBytes <= 227 * 1024, "head smem");

// ---- tensor-core head (head_tc_kernel): shared-memory plan, byte offsets ---------------------------------------
//   R0   conv1 A operand: LayerNorm output, fp16 hi | lo, [chunk 0..5][row 0..17][x 0..15][8 ch]; later conv2's weights
//   RING conv1 weight pieces (5 x 9216 B ring, refilled two pieces behind the issue point); later the cp.async ring of the CUDA-core layers
//   R1   first the staged search tokens (48 KB, bulk copy); then conv2 A operand: conv1 output (96 ch = 12 chunks), same chunk-image layout, hi | lo;
//        later the zero-bordered fp32 planes of conv2 / conv3 / conv4 outputs
constexpr int kTcAChunk = 18 * 16 * 16;                 // bytes of one 8-channel chunk image: 18 rows x 16 px x 16 B
constexpr int kT_R0 = 0, kT_R0Bytes = 2 * 6 * kTcAChunk;                   // 55296
constexpr int kT_Ring = kT_R0 + kT_R0Bytes, kT_PieceBytes = 2 * 2 * 144 * 16;  // piece (h, ky, K step): hi | lo, N = 144 (kx, co), K = 16 -> 9216
constexpr int kT_RingSlots = 5;                          // conv1 weight pieces in flight: 4 x 432 cycles of MMA cover an L2 round trip
constexpr int kT_R1 = kT_Ring + kT_RingSlots * kT_PieceBytes, kT_R1Half = 12 * kTcAChunk; // 55296 per precision
constexpr int kT_W3 = kT_Ring + 2 * kWChunk * 4;        // conv3's weights: the ring's tail (the CUDA-core layer's cp.async ring keeps the head of it)
constexpr int kT_Out3 = kT_R0, kT_Out4 = kT_Out3 + 24 * kPlane * 4;     // zero-bordered fp32 planes of conv3 / conv4 outputs (conv2's weights are dead by then)
constexpr int kT_Bias = kT_R1 + 2 * kT_R1Half;
constexpr int kT_Maps = kT_Bias + 256 * 4;
constexpr int kT_Red = kT_Maps + 6 * 256 * 4;
constexpr int kT_Bar = kT_Red + 32 * 4;                 // loaded[slots], consumed[slots], acc_ready, w2_loaded, acc2_ready, tmem base
constexpr size_t kHeadTcSmemBytes = kT_Bar + (2 * kT_RingSlots + 9) * 8;
constexpr int kT_TokBytes = 256 * kC * 4;               // a track's search tokens, staged in R1 (dead until conv1's first epilogue) for the LayerNorm
static_assert(kT_TokBytes <= 2 * kT_R1Half, "token staging");
constexpr int kT_Issue1 = 2, kT_Issue2 = 6;             // warps issuing conv1's (one per M tile) and conv2's (one per tower x M tile) MMAs
// conv2 / conv3 weights: one blob per tower, hi | lo halves, each K-major [k/8][n][8] (head_tc_pack)
constexpr int kT_W2Half = 12 * 48 * 16;                  // conv2: [12 chunks][n = kx*16 + co][8], k = ky*32 + ci
constexpr int kT_W2Tower = 2 * kT_W2Half, kT_W2Bytes = 3 * kT_W2Tower;
constexpr int kT_W3Half = 6 * 32 * 16;                   // conv3: [6 chunks][n = kx*8 + co, 32 (24 used)][8], k = ky*16 + ci
constexpr int kT_W3Tower = 2 * kT_W3Half, kT_W3Bytes = 3 * kT_W3Tower;
static_assert(kT_W2Bytes <= kT_R0Bytes && kT_Out4 + 12 * kPlane * 4 <= kT_R0 + kT_R0Bytes && kT_W3 + kT_W3Bytes <= kT_R1 && kT_W3 % 128 == 0, "head tc smem plan");
static_assert(kHeadTcSmemBytes <= 227 * 1024 && kT_Bar % 8 == 0 && kT_R1 % 128 == 0, "head smem (tc)");

__device__ __forceinline__ void cp_async16(float* dst_smem, const float* src_gmem) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst_smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(src_gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// One 3x3 / stride 1 / pad 1 layer on a 16x16 map.  Thread = 4 horizontally adjacent pixels x QT output
// channels of group g (g = tower when TOWER_IN, else an arbitrary slice of the merged output axis).
// Weights are streamed from global memory in chunks of CI_CHUNK input channels: [ci][ky*3+kx][NG*QT].
template <int CIN, int QT, int NG, bool TOWER_IN, int CI_CHUNK>
__device__ __forceinline__ void head_conv(const float* in, float* outp, const float* __restrict__ wg,
                                          const float* bias, float* wbuf) {
    constexpr int kCout = NG * QT;
    constexpr int kChunkFloats = CI_CHUNK * 9 * kCout;
    constexpr int kChunks = CIN / CI_CHUNK;
    static_assert(kChunkFloats <= kWChunk && kChunkFloats % 4 == 0 && CIN % CI_CHUNK == 0, "chunking");
    const int tid = threadIdx.x;
    const int pg = tid & 63, g = tid >> 6;
    const bool active = g < NG;
    const int y = pg >> 2, x0 = (pg & 3) * 4;
    const float* inb = in + (TOWER_IN && active ? g * CIN * kPlane : 0) + y * 18 + x0;

    float acc[4][QT];
#pragma unroll
    for (int q = 0; q < QT; ++q) {
        const float b = active ? bias[g * QT + q] : 0.f;
#pragma unroll
        for (int p = 0; p < 4; ++p) acc[p][q] = b;
    }
    auto issue = [&](int c) {
        float* dst = wbuf + (c & 1) * kWChunk;
        const float* src = wg + (size_t)c * kChunkFloats;
        for (int i = tid * 4; i < kChunkFloats; i += kHeadThreads * 4) cp_async16(dst + i, src + i);
        cp_async_commit();
    };
    issue(0);
#pragma unroll 1
    for (int c = 0; c < kChunks; ++c) {
        if (c + 1 < kChunks) { issue(c + 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
        __syncthreads();
        if (active) {
            const float* wc = wbuf + (c & 1) * kWChunk + g * QT;
#pragma unroll 1
            for (int cl = 0; cl < CI_CHUNK; ++cl) {
                const float* ip = inb + (c * CI_CHUNK + cl) * kPlane;
#pragma unroll
                for (int ky = 0; ky < 3; ++ky) {
                    float xi[6];
#pragma unroll
                    for (int j = 0; j < 6; ++j) xi[j] = ip[ky * 18 + j];
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx) {
                        const float* wp = wc + (cl * 9 + ky * 3 + kx) * kCout;
                        float wv[QT];
#pragma unroll
                        for (int q = 0; q < QT; q += 4) {
                            const float4 t = *reinterpret_cast<const float4*>(wp + q);
                            wv[q] = t.x; wv[q + 1] = t.y; wv[q + 2] = t.z; wv[q + 3] = t.w;
                        }
#pragma unroll
                        for (int p = 0; p < 4; ++p)
#pragma unroll
                            for (int q = 0; q < QT; ++q) acc[p][q] = fmaf(xi[p + kx], wv[q], acc[p][q]);
                    }
                }
            }
        }
        __syncthreads();
    }
    if (active) {
#pragma unroll
        for (int q = 0; q < QT; ++q) {
            float* op = outp + (g * QT + q) * kPlane + (y + 1) * 18 + x0 + 1;
#pragma unroll
            for (int p = 0; p < 4; ++p) op[p] = fmaxf(acc[p][q], 0.f);          // ReLU
        }
    }
    __syncthreads();
}

// Final LayerNorm of one token row (vit_dist.py:94); optionally stores the normalised row (tokens_norm tap, scaled back to the model's
// LayerNorm by w.norm_tap_scale).
// `bad` is raised when the row holds a non-finite value (an fp16-range overflow anywhere upstream on the tensor-core path ends as
// inf / NaN in the residual stream: K / V' / q / P poison every query row of their track, the MLP its own row) or when the
// normalised row itself would not fit the fp16 operand range.
// `staged`: the row in shared memory (head_tc_kernel stages a track's search tokens with one bulk copy); null = read it from global memory.
__device__ __forceinline__ void head_norm_row(const HeadArgs& a, const ModelW& w, int trk, int row, float (&y)[kC], int& bad,
                                              const float* staged = nullptr) {
    float x[kC];
    if (staged) {
#pragma unroll
        for (int k = 0; k < kC; k += 4) {
            const float4 v = *reinterpret_cast<const float4*>(staged + k);
            x[k] = v.x; x[k + 1] = v.y; x[k + 2] = v.z; x[k + 3] = v.w;
        }
    } else {
        const float* src = a.tokens + ((size_t)trk * kN + row) * kC;
#pragma unroll
        for (int k = 0; k < kC; k += 4) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(src + k));
            x[k] = v.x; x[k + 1] = v.y; x[k + 2] = v.z; x[k + 3] = v.w;
        }
    }
    float mean = 0.f;
#pragma unroll
    for (int k = 0; k < kC; ++k) mean += x[k];
    mean *= (1.f / kC);
    float var = 0.f;
#pragma unroll
    for (int k = 0; k < kC; ++k) { const float d = x[k] - mean; var = fmaf(d, d, var); }
    const float rstd = rsqrtf(var * (1.f / kC) + kLnEps);
#pragma unroll
    for (int k = 0; k < kC; ++k) y[k] = (x[k] - mean) * rstd * __ldg(w.norm_g + k) + __ldg(w.norm_b + k);
    float ymax = 0.f;
#pragma unroll
    for (int k = 0; k < kC; ++k) ymax = fmaxf(ymax, fabsf(y[k]));
    bad |= (!(var < INFINITY) ? 1 : 0) | (!(ymax < kF16Max) ? 2 : 0);     // bit 0: non-finite input, bit 1: fp16 operand range (NaN compares false)
    if (a.tokens_norm) {
        float* t = a.tokens_norm + ((size_t)trk * kN + row) * kC;
#pragma unroll
        for (int k = 0; k < kC; k += 4)
            *reinterpret_cast<float4*>(t + k) = make_float4(y[k] * w.norm_tap_scale, y[k + 1] * w.norm_tap_scale, y[k + 2] * w.norm_tap_scale,
                                                            y[k + 3] * w.norm_tap_scale);
    }
}

// conv5 (1x1) + sigmoid/clamp, raw and Hann-weighted arg-max, box decode, state update (thread = pixel).
// out4: [3 towers][4][324] zero-bordered planes; sb: bias block (w5 at +180, b5 at +204).
__device__ __forceinline__ void head_finish(const HeadArgs& a, const ModelW& w, int trk, const float* out4, const float* sb,
                                            float* maps, float* red, uint32_t tmem_to_free, int bad) {
    const int tid = threadIdx.x;
    HEAD_TRACE(5);
    // ---- conv5 (1x1) + sigmoid/clamp: thread = pixel ---------------------------------------------
    float* m_score = maps; float* m_size = maps + 256; float* m_off = maps + 768; float* m_resp = maps + 1280;
    {
        const int py = tid >> 4, px = tid & 15;
        const float* ip = out4 + (py + 1) * 18 + px + 1;
        const float* w5 = sb + 180; const float* b5 = sb + 204;
        float o[3][2];
#pragma unroll
        for (int t = 0; t < 3; ++t) {
            o[t][0] = b5[t * 2]; o[t][1] = b5[t * 2 + 1];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const float v = ip[(t * 4 + c) * kPlane];
                o[t][0] = fmaf(v, w5[(t * 4 + c) * 2], o[t][0]);
                o[t][1] = fmaf(v, w5[(t * 4 + c) * 2 + 1], o[t][1]);
            }
        }
        const float sc = sigmoid_clamp(o[0][0]);
        const float sw = sigmoid_clamp(o[2][0]), sh = sigmoid_clamp(o[2][1]);
        m_score[tid] = sc; m_size[tid] = sw; m_size[256 + tid] = sh;
        m_off[tid] = o[1][0]; m_off[256 + tid] = o[1][1];
        m_resp[tid] = __ldg(w.hann + tid) * sc;                               // output_window * score_map
        if (a.score_map) a.score_map[(size_t)trk * 256 + tid] = sc;
        if (a.size_map) { a.size_map[(size_t)trk * 512 + tid] = sw; a.size_map[(size_t)trk * 512 + 256 + tid] = sh; }
        if (a.offset_map) { a.offset_map[(size_t)trk * 512 + tid] = o[1][0]; a.offset_map[(size_t)trk * 512 + 256 + tid] = o[1][1]; }
    }
    const int any_bad = __syncthreads_or(bad | (a.state && item_slot(a.slots, trk) < 0));
    if (any_bad) {
        // never a silent wrong answer: the maps of a track whose activations left the representable range are NaN (ReLU and the
        // sigmoid would otherwise squash inf / NaN into plausible numbers), and the tracker output carries VT_TRACK_NUMERIC_RANGE
        const float qnan = __int_as_float(0x7fc00000);
        if (a.score_map) a.score_map[(size_t)trk * 256 + tid] = qnan;
        if (a.size_map) { a.size_map[(size_t)trk * 512 + tid] = qnan; a.size_map[(size_t)trk * 512 + 256 + tid] = qnan; }
        if (a.offset_map) { a.offset_map[(size_t)trk * 512 + tid] = qnan; a.offset_map[(size_t)trk * 512 + 256 + tid] = qnan; }
    }

    // ---- cal_bbox on the raw score (forward's pred_boxes) and on the windowed response (tracker) ----
    float raw_max, win_max; int raw_idx, win_idx;
    decode_argmax(m_score, m_resp, red, raw_max, raw_idx, win_max, win_idx);
    HEAD_TRACE(6);
    if (tmem_to_free != 0xffffffffu && tid < 32) tc::tmem_dealloc(tmem_to_free, 512);     // all TMEM reads ended before the barriers above
    if (tid == 0) decode_box(a, trk, m_size, m_off, raw_max, raw_idx, win_max, win_idx, any_bad ? VT_TRACK_NUMERIC_RANGE_ : 0);
    HEAD_TRACE(7);
}

// Track trk on the CUDA cores.
__device__ __forceinline__ void head_track(const HeadArgs& a, const ModelW& w, int trk) {
    extern __shared__ __align__(128) float smem[];
    float* feat = smem + kOffFeat;
    float* out1 = smem + kOffOut1;
    float* wbuf = smem + kOffW;
    float* sb = smem + kOffBias;
    float* maps = smem + kOffMaps;
    float* red = smem + kOffRed;
    const int tid = threadIdx.x;
    int bad = 0;

    HEAD_TRACE(0);
    // zero the activation planes once: layer outputs only ever write interiors, borders stay zero
    for (int i = tid * 4; i < kOffW; i += kHeadThreads * 4) *reinterpret_cast<float4*>(smem + i) = make_float4(0.f, 0.f, 0.f, 0.f);
    if (tid < 96) sb[tid] = w.head.b1[tid];
    if (tid < 48) sb[96 + tid] = w.head.b2[tid];
    if (tid < 24) sb[144 + tid] = w.head.b3[tid];
    if (tid < 12) sb[168 + tid] = w.head.b4[tid];
    if (tid < 24) sb[180 + tid] = w.head.w5[tid];
    if (tid < 6) sb[204 + tid] = w.head.b5[tid];
    __syncthreads();

    // ---- final LayerNorm (vit_dist.py:94) on search token `tid`; tokens -> (C,16,16) (vit_dist.py:126-129)
    {
        float y[kC];
        int flags = 0, unused = 0;
        head_norm_row(a, w, trk, kNz + tid, y, flags);
        bad = flags & 1;                             // fp32 path: only non-finite inputs are flagged
        const int py = tid >> 4, px = tid & 15;
#pragma unroll
        for (int k = 0; k < kC; ++k) feat[k * kPlane + (py + 1) * 18 + px + 1] = y[k];
        if (a.tokens_norm && tid < kNz) { float yz[kC]; head_norm_row(a, w, trk, tid, yz, unused); }
    }
    __syncthreads();

    HEAD_TRACE(1);
    // ---- conv towers ---------------------------------------------------------------------------
    head_conv<48, 24, 4, false, 4>(feat, out1, w.head.w1, sb, wbuf);               // 48 -> 3x32 (merged)
    HEAD_TRACE(2);
    float* out2 = feat;                                                            // [3][16] planes
    head_conv<32, 16, 3, true, 8>(out1, out2, w.head.w2, sb + 96, wbuf);           // 32 -> 16 per tower
    HEAD_TRACE(3);
    float* out3 = out1;                                                            // [3][8] planes
    head_conv<16, 8, 3, true, 16>(out2, out3, w.head.w3, sb + 144, wbuf);          // 16 -> 8
    HEAD_TRACE(4);
    float* out4 = out1 + 24 * kPlane;                                              // [3][4] planes
    head_conv<8, 4, 3, true, 8>(out3, out4, w.head.w4, sb + 168, wbuf);            // 8 -> 4

    head_finish(a, w, trk, out4, sb, maps, red, 0xffffffffu, bad);
}

// Track blockIdx.x; COUNTED (the range fallback of vt_api.cu): tracks blockIdx.x, blockIdx.x + gridDim.x, ... below *count.
template <bool COUNTED>
__global__ void __launch_bounds__(kHeadThreads, 1) head_kernel(HeadArgs a, ModelW w, const int32_t* __restrict__ count) {
    if constexpr (COUNTED) {
        for (int trk = blockIdx.x; trk < *count; trk += gridDim.x) {
            head_track(a, w, trk);
            __syncthreads();                                 // the next track clears shared memory
        }
    } else {
        head_track(a, w, blockIdx.x);
    }
}

// Tensor-core head: conv1 (48 -> 96 merged) and conv2 (32 -> 16 per tower) on tcgen05, conv3-5 on CUDA cores.
__global__ void __launch_bounds__(kHeadThreads, 1) head_tc_kernel(HeadArgs a, ModelW w) {
    extern __shared__ __align__(128) float smem[];
    uint8_t* sm8 = reinterpret_cast<uint8_t*>(smem);
    float* sb = reinterpret_cast<float*>(sm8 + kT_Bias);
    float* maps = reinterpret_cast<float*>(sm8 + kT_Maps);
    float* red = reinterpret_cast<float*>(sm8 + kT_Red);
    float* wbuf = reinterpret_cast<float*>(sm8 + kT_Ring);
    uint64_t* bar_loaded = reinterpret_cast<uint64_t*>(sm8 + kT_Bar);      // [kT_RingSlots]
    uint64_t* bar_consumed = bar_loaded + kT_RingSlots;                    // [kT_RingSlots]
    uint64_t* bar_acc = bar_loaded + 2 * kT_RingSlots;
    uint64_t* bar_w2 = bar_acc + 1;
    uint64_t* bar_acc2 = bar_acc + 2;
    uint64_t* bar_w3 = bar_acc + 3;
    uint64_t* bar_acc3 = bar_acc + 4;
    uint32_t* tc_tmem = reinterpret_cast<uint32_t*>(bar_acc + 5);
    uint64_t* bar_tok = bar_acc + 6;
    uint64_t* bar_w2t = bar_acc + 7;        // [2] conv2's weights of towers 1 and 2 (tower 0: bar_w2), so that a tower starts when ITS weights are in
    const int tid = threadIdx.x, warp = tid >> 5;
    const int py = tid >> 4, px = tid & 15;

    // ---- once per CTA: the bias block, the TMEM allocation.  The kernel is PERSISTENT (one CTA per SM walks over tracks): a CTA per
    // track costs ~3 us of hand-over per track (tear-down, launch, cold prologue) against 21 us of work.
    // bias block b1[96] b2[48] b3[24] b4[12] w5[24] b5[6]: ONE load per thread (six load -> store pairs in a row cost six L2 round trips)
    if (tid < 210) {
        const float* p = tid < 96 ? w.head.b1 + tid : tid < 144 ? w.head.b2 + (tid - 96) : tid < 168 ? w.head.b3 + (tid - 144)
                         : tid < 180 ? w.head.b4 + (tid - 168) : tid < 204 ? w.head.w5 + (tid - 180) : w.head.b5 + (tid - 204);
        sb[tid] = __ldg(p);
    }
    if (warp == 0) tc::tmem_alloc(tc_tmem, 512);
    // A track's 256 search tokens (48 KB, contiguous) come in with ONE bulk copy into the place of conv1's output image (dead from the
    // end of conv3's MMAs to conv1's first epilogue): read row by row from global memory (a thread per token, 192-byte stride between
    // lanes) they cost every load 32 sectors and the LayerNorm 8 k cycles.  The first track's copy starts here, track i + 1's when
    // conv3 of track i has read its operands; bar_tok is used once per track (phase = track parity).
    if (tid == 0) {
        tc::mbar_init(bar_tok, 1);
        tc::mbar_fence_init();
        if ((int)blockIdx.x < a.n) {
            tc::mbar_arrive_expect_tx(bar_tok, kT_TokBytes);
            tc::bulk_g2s(sm8 + kT_R1, a.tokens + ((size_t)blockIdx.x * kN + kNz) * kC, kT_TokBytes, bar_tok);
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tbase = __shfl_sync(0xffffffffu, *tc_tmem, 0);
    const uint32_t sbase = tc::smem_u32(smem);
    const uint32_t lane_addr = (uint32_t)(32 * (warp & 3)) << 16;
    const int tile = warp >> 2;                                            // epilogue: pixel = tid, M tile = warp / 4

    HEAD_TRACE_NS(28);
    HEAD_TRACE(30);
#pragma unroll 1
    for (int trk = blockIdx.x, iter = 0; trk < a.n; trk += gridDim.x, ++iter) {
    int bad = 0;                 // fp16 operand range guard (see head_norm_row); OR-reduced over the CTA in head_finish
    float vmax = 0.f;            // largest value this thread hands to a tensor-core operand image

    HEAD_TRACE(0);
    // Every other barrier starts a track in phase 0: they are re-initialised per track (all of the previous track's waits are over and
    // every asynchronous arrival has landed - the CTA barrier that ended it came after the last tcgen05.commit was waited for).
    // zero rows 0 and 17 of conv1's chunk images (the vertical zero padding); conv2's / conv3's images - the staging area now - get theirs
    // while conv1's first MMAs run
    for (int i = tid; i < 12 * 2 * 16; i += kHeadThreads) {
        const int cimg = i / 32, rsel = (i / 16) & 1, q = i & 15;          // 12 chunk images (hi and lo), row 0 / 17, 16 px
        *reinterpret_cast<float4*>(sm8 + kT_R0 + cimg * kTcAChunk + (rsel ? 17 * 256 : 0) + q * 16) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    HEAD_TRACE(20);
    HEAD_TRACE(21);
    if (tid == 32) {
        uint64_t* all[] = {bar_acc, bar_w2, bar_acc2, bar_w3, bar_acc3, bar_w2t, bar_w2t + 1};
        if (iter > 0) {
            for (int i = 0; i < kT_RingSlots; ++i) { tc::mbar_inval(bar_loaded + i); tc::mbar_inval(bar_consumed + i); }
            for (uint64_t* b : all) tc::mbar_inval(b);
        }
        for (int i = 0; i < kT_RingSlots; ++i) { tc::mbar_init(bar_loaded + i, 1); tc::mbar_init(bar_consumed + i, kT_Issue1); }
        tc::mbar_init(bar_acc, kT_Issue1);
        tc::mbar_init(bar_w2, 1);
        tc::mbar_init(bar_w2t, 1);
        tc::mbar_init(bar_w2t + 1, 1);
        tc::mbar_init(bar_acc2, kT_Issue2);
        tc::mbar_init(bar_w3, 1);
        tc::mbar_init(bar_acc3, kT_Issue2);
        tc::mbar_fence_init();
    }
    tc::fence_async_smem();
    __syncthreads();
    HEAD_TRACE(10);
    // the first conv1 weight pieces stream in underneath the LayerNorm
    if (warp == 0) {
#pragma unroll
        for (int p = 0; p < kT_RingSlots; ++p)
            tc::bulk_g2s_elect(sm8 + kT_Ring + p * kT_PieceBytes, w.head_tc_w1 + (size_t)p * kT_PieceBytes, kT_PieceBytes, bar_loaded + p);
    }
    // ---- final LayerNorm -> conv1's operand image (fp16 hi | lo, 8-channel chunks) ----------------------------------
    {
        float y[kC];
        tc::mbar_wait(bar_tok, iter & 1);
        head_norm_row(a, w, trk, kNz + tid, y, bad, reinterpret_cast<const float*>(sm8 + kT_R1) + tid * kC);
        uint8_t* ab = sm8 + kT_R0 + ((py + 1) * 16 + px) * 16;
#pragma unroll
        for (int c = 0; c < 6; ++c) {
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) tc::split_pack2(y[8 * c + 2 * j], y[8 * c + 2 * j + 1], hi[j], lo[j]);
            *reinterpret_cast<uint4*>(ab + c * kTcAChunk) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<uint4*>(ab + (6 + c) * kTcAChunk) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        }
        if (a.tokens_norm && tid < kNz) { float yz[kC]; int unused = 0; head_norm_row(a, w, trk, tid, yz, unused); }
    }
    HEAD_TRACE(11);
    tc::fence_async_smem();
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    HEAD_TRACE(1);

    // ---- conv1: 18 weight pieces p = (h * 3 + ky) * 3 + ks through the ring; D(tile, kx) = columns (tile * 3 + kx) * 48 ----
    {
        const uint32_t id144 = tc::instr_desc_f16(128, 144, false);
        auto load_piece = [&](int p) {
            tc::bulk_g2s_elect(sm8 + kT_Ring + (p % kT_RingSlots) * kT_PieceBytes, w.head_tc_w1 + (size_t)p * kT_PieceBytes, kT_PieceBytes,
                               bar_loaded + p % kT_RingSlots);
        };
#pragma unroll 1
        for (int h = 0; h < 2; ++h) {
            // A single warp issues a 48-column tcgen05.mma every ~35 cycles (descriptor transfers to uniform registers), the tensor
            // pipe needs 24: one issuing warp per M tile (on different schedulers) keeps the pipe fed.  Warp 0 also streams the pieces.
            if (warp < kT_Issue1) {              // convergent: every lane runs the program, one elected lane issues
                const int tl = warp;
#pragma unroll 1
                for (int q = 0; q < 9; ++q) {
                    const int p = 9 * h + q, ky = q / 3, ks = q % 3;
                    // refill: the slot of piece p - 2 (both tiles' MMAs on it have had a piece's time to complete - waiting for piece p - 1
                    // instead would hold this warp, and with it this tile's share of the tensor pipe, until the MMAs it just issued are done)
                    if (warp == 0 && p >= 2 && p - 2 + kT_RingSlots < 18) {
                        tc::mbar_wait(bar_consumed + (p - 2) % kT_RingSlots, ((p - 2) / kT_RingSlots) & 1);
                        load_piece(p - 2 + kT_RingSlots);
                    }
                    tc::mbar_wait(bar_loaded + p % kT_RingSlots, (p / kT_RingSlots) & 1);
                    tc::tc_fence_after();
                    // one N = 144 MMA per product: the piece holds all three horizontal taps, the three per-kx accumulators are adjacent
                    // TMEM columns - the A operand (4 KB of shared-memory reads per MMA, the bound of these small-N MMAs) is read once
                    const uint32_t wb = sbase + kT_Ring + (p % kT_RingSlots) * kT_PieceBytes;
                    const uint32_t d = tbase + tl * 144;
                    const uint32_t aoff = kT_R0 + (2 * ks) * kTcAChunk + (8 * tl + ky) * 256;
                    const uint64_t ah = tc::smem_desc(sbase + aoff, kTcAChunk, 128);
                    const uint64_t al = tc::smem_desc(sbase + aoff + 6 * kTcAChunk, kTcAChunk, 128);
                    const uint64_t bh = tc::smem_desc(wb, 144 * 16, 128);
                    const uint64_t bl = tc::smem_desc(wb + kT_PieceBytes / 2, 144 * 16, 128);
                    tc::mma_ss_elect(d, ah, bh, id144, q != 0);
                    tc::mma_ss_elect(d, al, bh, id144, 1);
                    tc::mma_ss_elect(d, ah, bl, id144, 1);
                    tc::mma_commit_elect(bar_consumed + p % kT_RingSlots);
                }
                tc::mma_commit_elect(bar_acc);
            }
            if (h == 0 && warp >= kT_Issue1) {       // rows 0 and 17 of conv2's / conv3's 24 chunk images, while the tensor pipe works
                for (int i = tid - 32 * kT_Issue1; i < 24 * 2 * 16; i += kHeadThreads - 32 * kT_Issue1) {
                    const int cimg = i / 32, rsel = (i / 16) & 1, q = i & 15;
                    *reinterpret_cast<float4*>(sm8 + kT_R1 + cimg * kTcAChunk + (rsel ? 17 * 256 : 0) + q * 16) = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
            tc::mbar_wait(bar_acc, h);
            tc::tc_fence_after();
            HEAD_TRACE(12 + 3 * h);
            if (h == 1 && warp == 0) {           // conv1's operand and weight ring are dead: conv2's and conv3's weights stream into their place
                tc::bulk_g2s_elect(sm8 + kT_R0, w.head_tc_w2, kT_W2Tower, bar_w2);
                tc::bulk_g2s_elect(sm8 + kT_R0 + kT_W2Tower, w.head_tc_w2 + kT_W2Tower, kT_W2Tower, bar_w2t);
                tc::bulk_g2s_elect(sm8 + kT_R0 + 2 * kT_W2Tower, w.head_tc_w2 + 2 * kT_W2Tower, kT_W2Tower, bar_w2t + 1);
                tc::bulk_g2s_elect(sm8 + kT_W3, w.head_tc_w3, kT_W3Bytes, bar_w3);
            }
            // epilogue: combine the three horizontal taps, bias, ReLU -> conv2's operand image (channels 48 h ..)
            {
                const uint32_t ta = tbase + lane_addr + tile * 144;
                uint8_t* ob = sm8 + kT_R1 + ((py + 1) * 16 + px) * 16;
#pragma unroll 1
                for (int c0 = 0; c0 < 48; c0 += 16) {
                    uint32_t r0[16], r1[16], r2[16];
                    tc::tmem_ld16(ta + c0, r0);
                    tc::tmem_ld16(ta + 48 + c0, r1);
                    tc::tmem_ld16(ta + 96 + c0, r2);
                    tc::tc_wait_ld();
                    float v[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        float t0 = __shfl_up_sync(0xffffffffu, __uint_as_float(r0[j]), 1);     // T_0[y][x-1]
                        float t2 = __shfl_down_sync(0xffffffffu, __uint_as_float(r2[j]), 1);   // T_2[y][x+1]
                        if (px == 0) t0 = 0.f;
                        if (px == 15) t2 = 0.f;
                        v[j] = max_nan((t0 + __uint_as_float(r1[j])) + t2 + sb[h * 48 + c0 + j], 0.f);
                        vmax = max_nan(vmax, v[j]);
                    }
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        uint32_t hi[4], lo[4];
#pragma unroll
                        for (int j = 0; j < 4; ++j) tc::split_pack2(v[8 * c + 2 * j], v[8 * c + 2 * j + 1], hi[j], lo[j]);
                        const int chunk = (h * 48 + c0) / 8 + c;
                        *reinterpret_cast<uint4*>(ob + chunk * kTcAChunk) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                        *reinterpret_cast<uint4*>(ob + kT_R1Half + chunk * kTcAChunk) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                    }
                }
            }
            HEAD_TRACE(13 + 3 * h);
            tc::fence_async_smem();
            tc::tc_fence_before();
            __syncthreads();
            tc::tc_fence_after();
        }
    }
    HEAD_TRACE(2);

    // ---- conv2 (per tower 32 -> 16): D(tower, tile, kx) = columns ((tower * 2 + tile) * 3 + kx) * 16 ----------------------
    if (warp < kT_Issue2) {                      // one issuing warp per (tower, M tile); N = 48 = the three horizontal taps side by side
        const uint32_t id48 = tc::instr_desc_f16(128, 48, false);
        const int tw = warp >> 1, tl = warp & 1;
        tc::mbar_wait(tw == 0 ? bar_w2 : bar_w2t + (tw - 1), 0);
        tc::tc_fence_after();
        const uint32_t d = tbase + (tw * 2 + tl) * 48;
        const uint32_t wb = sbase + kT_R0 + tw * kT_W2Tower;
#pragma unroll
        for (int ky = 0; ky < 3; ++ky)
#pragma unroll
            for (int kp = 0; kp < 2; ++kp) {
                const uint32_t aoff = kT_R1 + (4 * tw + 2 * kp) * kTcAChunk + (8 * tl + ky) * 256;
                const uint64_t ah = tc::smem_desc(sbase + aoff, kTcAChunk, 128);
                const uint64_t al = tc::smem_desc(sbase + aoff + kT_R1Half, kTcAChunk, 128);
                const uint64_t bh = tc::smem_desc(wb + (ky * 4 + 2 * kp) * 768, 768, 128);
                const uint64_t bl = tc::smem_desc(wb + kT_W2Half + (ky * 4 + 2 * kp) * 768, 768, 128);
                tc::mma_ss_elect(d, ah, bh, id48, (ky | kp) != 0);
                tc::mma_ss_elect(d, al, bh, id48, 1);
                tc::mma_ss_elect(d, ah, bl, id48, 1);
            }
        tc::mma_commit_elect(bar_acc2);
    }
    tc::mbar_wait(bar_acc2, 0);
    tc::tc_fence_after();
    HEAD_TRACE(18);
    // conv2's weights are dead: their place becomes the zero-bordered fp32 planes of conv3's / conv4's outputs
    for (int i = tid * 4; i < (24 + 12) * kPlane; i += kHeadThreads * 4)
        *reinterpret_cast<float4*>(sm8 + kT_Out3 + i * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
    float* out3 = reinterpret_cast<float*>(sm8 + kT_Out3);
    float* out4 = reinterpret_cast<float*>(sm8 + kT_Out4);
    // conv2's epilogue -> conv3's operand image: tower tw's 16 channels = chunk images 2 tw, 2 tw + 1 of R1 (hi | lo), whose zero rows
    // 0 and 17 were never written
    {
        uint8_t* ob = sm8 + kT_R1 + ((py + 1) * 16 + px) * 16;
#pragma unroll 1
        for (int tw = 0; tw < 3; ++tw) {
            const uint32_t ta = tbase + lane_addr + ((tw * 2 + tile) * 3) * 16;
            uint32_t r0[16], r1[16], r2[16];
            tc::tmem_ld16(ta, r0);
            tc::tmem_ld16(ta + 16, r1);
            tc::tmem_ld16(ta + 32, r2);
            tc::tc_wait_ld();
            float v[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                float t0 = __shfl_up_sync(0xffffffffu, __uint_as_float(r0[j]), 1);
                float t2 = __shfl_down_sync(0xffffffffu, __uint_as_float(r2[j]), 1);
                if (px == 0) t0 = 0.f;
                if (px == 15) t2 = 0.f;
                v[j] = max_nan((t0 + __uint_as_float(r1[j])) + t2 + sb[96 + tw * 16 + j], 0.f);
                vmax = max_nan(vmax, v[j]);
            }
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                uint32_t hi[4], lo[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) tc::split_pack2(v[8 * c + 2 * j], v[8 * c + 2 * j + 1], hi[j], lo[j]);
                *reinterpret_cast<uint4*>(ob + (2 * tw + c) * kTcAChunk) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                *reinterpret_cast<uint4*>(ob + kT_R1Half + (2 * tw + c) * kTcAChunk) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
            }
        }
    }
    tc::fence_async_smem();
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    HEAD_TRACE(3);

    // ---- conv3 (per tower 16 -> 8): N = 32 = three horizontal taps x 8 channels (+ 8 padding); D(tower, tile) = columns 288 + (tower * 2 + tile) * 32 ----
    if (warp < kT_Issue2) {
        const uint32_t id32 = tc::instr_desc_f16(128, 32, false);
        const int tw = warp >> 1, tl = warp & 1;
        tc::mbar_wait(bar_w3, 0);
        tc::tc_fence_after();
        const uint32_t d = tbase + 288 + (tw * 2 + tl) * 32;
        const uint32_t wb = sbase + kT_W3 + tw * kT_W3Tower;
#pragma unroll
        for (int ky = 0; ky < 3; ++ky) {
            const uint32_t aoff = kT_R1 + (2 * tw) * kTcAChunk + (8 * tl + ky) * 256;
            const uint64_t ah = tc::smem_desc(sbase + aoff, kTcAChunk, 128);
            const uint64_t al = tc::smem_desc(sbase + aoff + kT_R1Half, kTcAChunk, 128);
            const uint64_t bh = tc::smem_desc(wb + (ky * 2) * 512, 512, 128);
            const uint64_t bl = tc::smem_desc(wb + kT_W3Half + (ky * 2) * 512, 512, 128);
            tc::mma_ss_elect(d, ah, bh, id32, ky != 0);
            tc::mma_ss_elect(d, al, bh, id32, 1);
            tc::mma_ss_elect(d, ah, bl, id32, 1);
        }
        tc::mma_commit_elect(bar_acc3);
    }
    tc::mbar_wait(bar_acc3, 0);
    tc::tc_fence_after();
    if (tid == 0 && trk + (int)gridDim.x < a.n) {          // conv3 has read its operands: the next track's tokens may land in their place
        tc::mbar_arrive_expect_tx(bar_tok, kT_TokBytes);
        tc::bulk_g2s(sm8 + kT_R1, a.tokens + ((size_t)(trk + gridDim.x) * kN + kNz) * kC, kT_TokBytes, bar_tok);
    }
    {
        float* op = out3 + (py + 1) * 18 + px + 1;
#pragma unroll 1
        for (int tw = 0; tw < 3; ++tw) {
            const uint32_t ta = tbase + lane_addr + 288 + (tw * 2 + tile) * 32;
            uint32_t r0[8], r1[8], r2[8];
            tc::tmem_ld8(ta, r0);
            tc::tmem_ld8(ta + 8, r1);
            tc::tmem_ld8(ta + 16, r2);
            tc::tc_wait_ld();
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float t0 = __shfl_up_sync(0xffffffffu, __uint_as_float(r0[j]), 1);
                float t2 = __shfl_down_sync(0xffffffffu, __uint_as_float(r2[j]), 1);
                if (px == 0) t0 = 0.f;
                if (px == 15) t2 = 0.f;
                const float o3 = max_nan((t0 + __uint_as_float(r1[j])) + t2 + sb[144 + tw * 8 + j], 0.f);
                op[(tw * 8 + j) * kPlane] = o3;
                vmax = max_nan(vmax, o3 < INFINITY ? 0.f : o3);          // conv3's operands were fp16 too: a non-finite result (inf or NaN) is an overflow
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    HEAD_TRACE(4);
    head_conv<8, 4, 3, true, 8>(out3, out4, w.head.w4, sb + 168, wbuf);            // 8 -> 4
    bad |= !(vmax < kF16Max);
    head_finish(a, w, trk, out4, sb, maps, red, 0xffffffffu, bad);
    // end of the track: every thread is past its last read of the planes, the maps and TMEM; the next track's bulk copies (async proxy)
    // overwrite regions this one wrote through the generic proxy
    tc::fence_async_smem();
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    HEAD_TRACE(8);
    }
    HEAD_TRACE_NS(29);
    HEAD_TRACE(31);
    if (warp == 0) tc::tmem_dealloc(tbase, 512);
}

int launch_head(const HeadArgs& a, const ModelW& w, cudaStream_t st, const int32_t* count) {
    if (a.n <= 0) return 0;
    static DeviceOnce once_simt, once_tc, once_counted;
    if (!ensure_dyn_smem(once_simt, head_kernel<false>, kHeadSmemBytes) || !ensure_dyn_smem(once_tc, head_tc_kernel, kHeadTcSmemBytes)) return -1;
    if (count) {
        if (!ensure_dyn_smem(once_counted, head_kernel<true>, kHeadSmemBytes)) return -1;
        head_kernel<true><<<counted_rows(a.n, 1, 1), kHeadThreads, kHeadSmemBytes, st>>>(a, w, count);
        return cudaGetLastError() == cudaSuccess ? 1 : -1;
    }
    if (a.use_tc) {
        static int sms[kMaxDevices] = {};
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return -1;
        if (sms[dev] == 0 && cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1;
        head_tc_kernel<<<a.n < sms[dev] ? a.n : sms[dev], kHeadThreads, kHeadTcSmemBytes, st>>>(a, w);      // persistent: one CTA (220 KB) per SM
    }
    else head_kernel<false><<<a.n, kHeadThreads, kHeadSmemBytes, st>>>(a, w, nullptr);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

size_t head_tc_weight_bytes(int layer) { return layer == 0 ? (size_t)18 * kT_PieceBytes : layer == 1 ? kT_W2Bytes : kT_W3Bytes; }

// Host side: the folded fp32 weights (HeadW: w1 [ci][ky*3+kx][96], w2 [ci][ky*3+kx][tower][16], w3 [ci][ky*3+kx][tower][8]) -> the
// fp16 hi | lo blobs head_tc_kernel reads.
void head_tc_pack(const float* w1, const float* w2, const float* w3, uint8_t* blob1, uint8_t* blob2, uint8_t* blob3) {
    // conv1: piece p = (h * 3 + ky) * 3 + ks holds one K step (input channels 16 ks .. 16 ks + 15) of vertical tap ky for ALL three
    // horizontal taps: B[n = kx * 48 + (co - 48 h)][k = ci], [hi | lo] x [chunk 2][n 144][8] - one N = 144 MMA feeds the three
    // per-kx accumulators (adjacent TMEM columns) from a single read of the A operand
    for (int h = 0; h < 2; ++h)
        for (int ky = 0; ky < 3; ++ky)
            for (int ks = 0; ks < 3; ++ks) {
                uint8_t* piece = blob1 + (size_t)((h * 3 + ky) * 3 + ks) * kT_PieceBytes;
                for (int kx = 0; kx < 3; ++kx)
                    for (int n = 0; n < 48; ++n)
                        for (int e = 0; e < 16; ++e)
                            tc::put_kmajor_f16(piece, piece + kT_PieceBytes / 2, 144, kx * 48 + n, e,
                                               w1[((size_t)(16 * ks + e) * 9 + ky * 3 + kx) * 96 + h * 48 + n]);
            }
    // conv2 / conv3, one blob per tower t: B[n = kx * co_n + co][k = ky * ci_n + ci], N = npad
    auto towers = [](uint8_t* blob, int tower_bytes, int ci_n, int co_n, int npad, const float* wf) {
        for (int t = 0; t < 3; ++t)
            for (int kx = 0; kx < 3; ++kx)
                for (int n = 0; n < co_n; ++n)
                    for (int ky = 0; ky < 3; ++ky)
                        for (int ci = 0; ci < ci_n; ++ci)
                            tc::put_kmajor_f16(blob + t * tower_bytes, blob + t * tower_bytes + tower_bytes / 2, npad, kx * co_n + n, ky * ci_n + ci,
                                               wf[(((size_t)ci * 9 + ky * 3 + kx) * 3 + t) * co_n + n]);
    };
    towers(blob2, kT_W2Tower, 32, 16, 48, w2);
    memset(blob3, 0, kT_W3Bytes);                        // conv3's output columns 24..31 are padding
    towers(blob3, kT_W3Tower, 16, 8, 32, w3);
}

// box_head.cal_bbox(score, size_map, offset_map) on caller-provided maps (head.py:142-160).
__global__ void __launch_bounds__(256) cal_bbox_kernel(const float* __restrict__ score, const float* __restrict__ size_map,
                                                      const float* __restrict__ offset_map, float* __restrict__ boxes) {
    __shared__ float red[32];
    const int trk = blockIdx.x, tid = threadIdx.x;
    float best; int idx;
    block_argmax256(score[(size_t)trk * 256 + tid], tid, red, best, idx);
    if (tid == 0) {
        const float* sz = size_map + (size_t)trk * 512;
        const float* of = offset_map + (size_t)trk * 512;
        float* pb = boxes + (size_t)trk * 4;
        pb[0] = ((float)(idx & 15) + of[idx]) / 16.f;
        pb[1] = ((float)(idx >> 4) + of[256 + idx]) / 16.f;
        pb[2] = sz[idx];
        pb[3] = sz[256 + idx];
    }
}

int launch_cal_bbox(const float* score, const float* size_map, const float* offset_map, int n, float* boxes,
                    cudaStream_t st) {
    if (n <= 0) return 0;
    cal_bbox_kernel<<<n, 256, 0, st>>>(score, size_map, offset_map, boxes);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

}  // namespace vt
