// K2: LeViT-style conv stem - 4x [conv3x3 stride 2 pad 1 (no bias) + BatchNorm(eval)], Hardswish
// after the first three (lib/models/vit_dist/vit_dist.py:10-54), BN folded into the convolution
// at weight-pack time, fp32 direct convolution on CUDA cores.
//
// One templated tile kernel serves all four layers.  A CTA stages a (2*TH+1) x (2*TW+1) x CIN
// input tile in shared memory with even and odd columns de-interleaved, so that the stride-2 reads
// of a warp (lanes = consecutive output columns) are stride-1 and bank-conflict free.  Weights sit
// in shared memory as [cin][ky][kx][cout]; a thread owns P output pixels x QG output channels and
// reads its weights with broadcast vector loads.  The last layer writes tokens (row = y*16+x,
// token-major [token][48]) with the positional embedding added (vit_dist.py:53,81-82).
#include <type_traits>

#include "vt_geom.cuh"
#include "vt_internal.h"
#include "vt_taps.cuh"
#include "vt_tc.cuh"

namespace vt {

// cp.async of BYTES (4 or 16) bytes; when !valid nothing is read and the destination is zero-filled
template <int BYTES>
__device__ __forceinline__ void cp_async(float* dst_smem, const float* src_gmem, bool valid) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst_smem);
    const int sz = valid ? BYTES : 0;
    if (BYTES == 16)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(d), "l"(src_gmem), "r"(sz) : "memory");
    else
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(d), "l"(src_gmem), "r"(sz) : "memory");
}

template <int CIN, int COUT, int QG, int P, int TW, int TH>
struct ConvCfg {
    static constexpr int kPixGroups = TW * TH / P;
    static constexpr int kChGroups = COUT / QG;
    static constexpr int kThreads = kPixGroups * kChGroups;
    static constexpr int kInRows = 2 * TH + 1;
    // One tile row holds input columns 2*tx0-1 .. 2*tx0+2*TW-1 de-interleaved by parity:
    //   [0] pad | [1 .. TW+1] even-slot columns E[0..TW] | [TW+2 .. 2TW+1] odd-slot columns O[0..TW-1]
    // (tile column c = input column - (2*tx0-1); even c -> E[c/2], odd c -> O[c/2]).  The pad keeps the
    // 8-byte stores of the staging loop aligned; output pixel x reads E[x], O[x], E[x+1]: stride-1 per lane.
    static constexpr int kEOff = 1;
    static constexpr int kOOff = TW + 2;
    static constexpr int kPitchRaw = 2 * TW + 2;
    // TW == 16: two output rows share a warp -> row pitch must be == 8 (mod 16) to stay conflict free
    static constexpr int kPitch = (TW == 32) ? kPitchRaw : ((kPitchRaw - 8 + 15) / 16 * 16 + 8);
    static constexpr int kChunks = TW / 2 + 1;               // aligned float4 chunks per tile row
    static constexpr int kTileFloats = (CIN * kInRows * kPitch + 3) / 4 * 4;   // keeps the weights 16-byte aligned
    static constexpr int kWFloats = (CIN * 9 * COUT + 3) / 4 * 4;      // copied in 16-byte pieces (packed slots are padded alike)
    static constexpr size_t kSmemBytes = (size_t)(kTileFloats + kWFloats + COUT) * sizeof(float);
    static_assert(kPixGroups % 32 == 0, "channel group must be warp uniform");
    static_assert(32 % TW == 0 && (TW == 16 || TW == 32), "tile width");
    static_assert(COUT % QG == 0 && QG % 2 == 0, "channel grouping");
    static_assert(kPitch % 2 == 0 && kOOff % 2 == 0, "8-byte aligned odd-slot stores");
};

// sm_100 packed fp32 FMA (SASS FFMA2): two independent IEEE fmaf in one issue slot - bit-identical to two scalar FFMA
__device__ __forceinline__ uint64_t pack_f32x2(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ uint64_t ffma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}

__device__ __forceinline__ uint64_t fmul2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uint64_t fadd2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}

// Preprocessor.process (lib/test/tracker/data_utils.py:8-14) on a uint8 pixel value without a table:  ((v / 255) - mean) / std, every
// step rounded to fp32.  Both divisions are by constants and take the same form as div6_exact -  q = a r;  q' = fma(fma(-d, q, a), r, q)
// with r = fl(1 / d)  - which equals the IEEE quotient for each of the 256 pixel values and each of the three channels (checked
// exhaustively in exact rational arithmetic: tools/norm_exact_check.py; the table of vt_api.cu fill_hann_and_lut holds the same bits).
// Three table loads per pixel, each scattered over eight cache lines, were 44 % of the kernel's global-load sectors.
struct NormConst {
    static constexpr float kR255 = 1.0f / 255.0f;
    __device__ static constexpr float mean(int ch) { return ch == 0 ? 0.485f : ch == 1 ? 0.456f : 0.406f; }
    __device__ static constexpr float stdv(int ch) { return ch == 0 ? 0.229f : ch == 1 ? 0.224f : 0.225f; }
    __device__ static constexpr float rstd(int ch) { return ch == 0 ? 1.0f / 0.229f : ch == 1 ? 1.0f / 0.224f : 1.0f / 0.225f; }
};
template <int CH>
__device__ __forceinline__ float normalize_px(int v) {                     // 0 <= v <= 255
    const float a = __int_as_float(0x4b000000 | v) - 8388608.f;            // exact int -> float
    const float q = __fmul_rn(a, NormConst::kR255);
    const float x = __fmaf_rn(__fmaf_rn(-255.f, q, a), NormConst::kR255, q);
    const float y = __fadd_rn(x, -NormConst::mean(CH));
    const float z = __fmul_rn(y, NormConst::rstd(CH));
    return __fmaf_rn(__fmaf_rn(-NormConst::stdv(CH), z, y), NormConst::rstd(CH), z);
}
template <int CH>
__device__ __forceinline__ void normalize_px2(int v0, int v1, float& o0, float& o1) {      // two pixels per issue slot
    const uint64_t a = fadd2(pack_f32x2(__int_as_float(0x4b000000 | v0), __int_as_float(0x4b000000 | v1)), pack_f32x2(-8388608.f, -8388608.f));
    const uint64_t r = pack_f32x2(NormConst::kR255, NormConst::kR255), rs = pack_f32x2(NormConst::rstd(CH), NormConst::rstd(CH));
    const uint64_t q = fmul2(a, r);
    const uint64_t x = ffma2(ffma2(pack_f32x2(-255.f, -255.f), q, a), r, q);
    const uint64_t y = fadd2(x, pack_f32x2(-NormConst::mean(CH), -NormConst::mean(CH)));
    const uint64_t z = fmul2(y, rs);
    const uint64_t o = ffma2(ffma2(pack_f32x2(-NormConst::stdv(CH), -NormConst::stdv(CH)), z, y), rs, z);
    asm("mov.b64 {%0, %1}, %2;" : "=f"(o0), "=f"(o1) : "l"(o));
}

// Accumulate and store: the tile / weights / bias are in shared memory (see ConvCfg for the tile layout).
// PAIRED: the weights sit in shared memory duplicated, [cin][ky][kx][cout] of float2 {w, w}, and two output pixels of a
// thread share one packed FMA (the accumulation order of every output is unchanged, so the results are too).
template <int CIN, int COUT, int QG, int P, int TW, int TH, bool HSWISH, bool TOKENS, int TCOUT_CCH = 0, bool PAIRED = false>
__device__ __forceinline__ void conv_compute(const float* tile, const float* ws, const float* bs, int tx0, int ty0, int Hout,
                                             int Wout, int b, float* __restrict__ out, const float* __restrict__ pos,
                                             int tok_stride_rows, int tok_off) {
    using K = ConvCfg<CIN, COUT, QG, P, TW, TH>;
    const int tid = threadIdx.x;
    const int cg = tid / K::kPixGroups;                 // warp-uniform channel group
    const int pg = tid % K::kPixGroups;
    const int lane = pg & 31, wq = pg >> 5;
    constexpr int kRowsPerWarp = 32 / TW;
    const int lx = lane % TW;
    int ly[P];
#pragma unroll
    for (int p = 0; p < P; ++p) ly[p] = (wq * P + p) * kRowsPerWarp + lane / TW;

    float acc[P][QG];
    if constexpr (PAIRED) {
        static_assert(!PAIRED || (P % 2 == 0 && QG % 2 == 0), "pixel pairs, channel pairs per 16-byte weight load");
        uint64_t acc2[P / 2][QG];
#pragma unroll
        for (int pp = 0; pp < P / 2; ++pp)
#pragma unroll
            for (int q = 0; q < QG; ++q) acc2[pp][q] = pack_f32x2(bs[cg * QG + q], bs[cg * QG + q]);
#pragma unroll 1
        for (int ci = 0; ci < CIN; ++ci) {
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
                uint64_t x2[P / 2][3];
#pragma unroll
                for (int pp = 0; pp < P / 2; ++pp) {
                    const float* r0 = tile + (ci * K::kInRows + 2 * ly[2 * pp] + ky) * K::kPitch;
                    const float* r1 = tile + (ci * K::kInRows + 2 * ly[2 * pp + 1] + ky) * K::kPitch;
                    x2[pp][0] = pack_f32x2(r0[K::kEOff + lx], r1[K::kEOff + lx]);
                    x2[pp][1] = pack_f32x2(r0[K::kOOff + lx], r1[K::kOOff + lx]);
                    x2[pp][2] = pack_f32x2(r0[K::kEOff + lx + 1], r1[K::kEOff + lx + 1]);
                }
#pragma unroll
                for (int kx = 0; kx < 3; ++kx) {
                    const ulonglong2* wp = reinterpret_cast<const ulonglong2*>(ws) + ((((ci * 3 + ky) * 3 + kx) * COUT + cg * QG) >> 1);
#pragma unroll
                    for (int q = 0; q < QG; q += 2) {
                        const ulonglong2 w2 = wp[q >> 1];                      // {w[q], w[q]}, {w[q+1], w[q+1]}
#pragma unroll
                        for (int pp = 0; pp < P / 2; ++pp) {
                            acc2[pp][q] = ffma2(x2[pp][kx], w2.x, acc2[pp][q]);
                            acc2[pp][q + 1] = ffma2(x2[pp][kx], w2.y, acc2[pp][q + 1]);
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int pp = 0; pp < P / 2; ++pp) {
            float h[2 * QG];                                               // the pixel pair's values, still register pairs
#pragma unroll
            for (int q = 0; q < QG; ++q) {
                h[2 * q] = __uint_as_float((uint32_t)acc2[pp][q]);
                h[2 * q + 1] = __uint_as_float((uint32_t)(acc2[pp][q] >> 32));
            }
            if (HSWISH) hardswish_exact_n<2 * QG>(h);                      // x * relu6(x + 3) / 6
#pragma unroll
            for (int q = 0; q < QG; ++q) {
                acc[2 * pp][q] = h[2 * q];
                acc[2 * pp + 1][q] = h[2 * q + 1];
            }
        }
    } else {
#pragma unroll
    for (int p = 0; p < P; ++p)
#pragma unroll
        for (int q = 0; q < QG; ++q) acc[p][q] = bs[cg * QG + q];

#pragma unroll 1
    for (int ci = 0; ci < CIN; ++ci) {
#pragma unroll
        for (int ky = 0; ky < 3; ++ky) {
            float xin[P][3];
#pragma unroll
            for (int p = 0; p < P; ++p) {
                const float* row = tile + (ci * K::kInRows + 2 * ly[p] + ky) * K::kPitch;
                xin[p][0] = row[K::kEOff + lx];          // tile col 2x   (even slot x)
                xin[p][1] = row[K::kOOff + lx];          // tile col 2x+1 (odd slot x)
                xin[p][2] = row[K::kEOff + lx + 1];      // tile col 2x+2 (even slot x+1)
            }
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
                const float* wp = ws + ((ci * 3 + ky) * 3 + kx) * COUT + cg * QG;
                float wv[QG];
                if constexpr (QG % 4 == 0 && (COUT % 4) == 0) {
#pragma unroll
                    for (int q = 0; q < QG; q += 4) {
                        const float4 t = *reinterpret_cast<const float4*>(wp + q);
                        wv[q] = t.x; wv[q + 1] = t.y; wv[q + 2] = t.z; wv[q + 3] = t.w;
                    }
                } else {
#pragma unroll
                    for (int q = 0; q < QG; q += 2) {
                        const float2 t = *reinterpret_cast<const float2*>(wp + q);
                        wv[q] = t.x; wv[q + 1] = t.y;
                    }
                }
#pragma unroll
                for (int p = 0; p < P; ++p)
#pragma unroll
                    for (int q = 0; q < QG; ++q) acc[p][q] = fmaf(xin[p][kx], wv[q], acc[p][q]);
            }
        }
    }
    }

    const int ox = tx0 + lx;
#pragma unroll
    for (int p = 0; p < P; ++p) {
        const int oy = ty0 + ly[p];
        if (ox >= Wout || oy >= Hout) continue;
        if (HSWISH && !PAIRED) hardswish_exact_n<QG>(acc[p]);              // x * relu6(x + 3) / 6
        if (TCOUT_CCH > 0) {
            // the next layer runs on the tensor cores: write its operand image (fp16 hi | lo, 8-channel chunks, parity planes)
            static_assert(TCOUT_CCH == 0 || QG == COUT, "thread must own every channel of the pixel");
            uint8_t* ob = reinterpret_cast<uint8_t*>(out) + (size_t)b * tc_planes_bytes(TCOUT_CCH, Wout / 2);
#pragma unroll
            for (int c = 0; c < TCOUT_CCH; ++c) {
                uint32_t hi[4], lo[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float v0 = (8 * c + 2 * j < COUT) ? acc[p][(8 * c + 2 * j) % QG] : 0.f;
                    const float v1 = (8 * c + 2 * j + 1 < COUT) ? acc[p][(8 * c + 2 * j + 1) % QG] : 0.f;
                    tc::split_pack2(v0, v1, hi[j], lo[j]);
                }
                *reinterpret_cast<uint4*>(ob + tc_planes_offset(0, oy, ox, c, TCOUT_CCH, Wout / 2)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                *reinterpret_cast<uint4*>(ob + tc_planes_offset(1, oy, ox, c, TCOUT_CCH, Wout / 2)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
            }
        } else if (TOKENS) {
            const int t = oy * Wout + ox;
            float* o = out + ((size_t)b * tok_stride_rows + tok_off + t) * COUT + cg * QG;
            const float* pe = pos + (size_t)t * COUT + cg * QG;
#pragma unroll
            for (int q = 0; q < QG; q += 4) {
                const float4 e = *reinterpret_cast<const float4*>(pe + q);
                float4 r = make_float4(acc[p][q] + e.x, acc[p][q + 1] + e.y, acc[p][q + 2] + e.z, acc[p][q + 3] + e.w);
                *reinterpret_cast<float4*>(o + q) = r;
            }
        } else {
#pragma unroll
            for (int q = 0; q < QG; ++q)
                out[(((size_t)b * COUT + cg * QG + q) * Hout + oy) * Wout + ox] = acc[p][q];
        }
    }
}

template <int CIN, int COUT, int QG, int P, int TW, int TH, bool HSWISH, bool TOKENS, int TCOUT_CCH = 0>
__global__ void __launch_bounds__(ConvCfg<CIN, COUT, QG, P, TW, TH>::kThreads)
conv3x3s2_kernel(const float* __restrict__ in, int Hin, int Win, const float* __restrict__ wg,
                 const float* __restrict__ bg, float* __restrict__ out, const float* __restrict__ pos,
                 int tok_stride_rows, int tok_off) {
    using K = ConvCfg<CIN, COUT, QG, P, TW, TH>;
    extern __shared__ __align__(16) float smem[];
    float* tile = smem;
    float* ws = smem + K::kTileFloats;
    float* bs = ws + K::kWFloats;

    const int Hout = Hin >> 1, Wout = Win >> 1;
    const int tiles_x = (Wout + TW - 1) / TW;
    const int tx0 = (blockIdx.x % tiles_x) * TW;
    const int ty0 = (blockIdx.x / tiles_x) * TH;
    const int b = blockIdx.y;
    const int tid = threadIdx.x;

    // weights / bias / input tile are staged with cp.async: every load is in flight at once (the tile
    // fill was latency-bound as a loop of dependent ld.global + st.shared); padding is zero-filled
    for (int i = tid * 4; i < K::kWFloats; i += K::kThreads * 4) cp_async<16>(ws + i, wg + i, true);
    if (tid < COUT) cp_async<4>(bs + tid, bg + tid, true);

    // Input tile: aligned float4 loads (chunk j of a row covers input columns 2*tx0-4+4j .. +3), several
    // in flight per thread, de-interleaved in registers.  Win is a multiple of 4, so a chunk is entirely
    // inside or outside the image; outside (and rows outside) is the convolution's zero padding.
    {
        const float* inb = in + (size_t)b * CIN * Hin * Win;
        const int gx0 = 2 * tx0 - 4, iy0 = 2 * ty0 - 1;
        constexpr int kItems = CIN * K::kInRows * K::kChunks;
        constexpr int kBatch = 4;
#pragma unroll 1
        for (int i0 = tid; i0 < kItems; i0 += kBatch * K::kThreads) {
            float4 v[kBatch];
            int dst[kBatch], jj[kBatch];
#pragma unroll
            for (int u = 0; u < kBatch; ++u) {
                const int i = i0 + u * K::kThreads;
                const int j = i % K::kChunks;
                const int rr = i / K::kChunks;                // ci * kInRows + r
                const int r = rr % K::kInRows;
                const int ci = rr / K::kInRows;
                const int gx = gx0 + 4 * j, gy = iy0 + r;
                v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                jj[u] = j;
                dst[u] = (i < kItems) ? rr * K::kPitch : -1;
                if (i < kItems && gx >= 0 && gx < Win && gy >= 0 && gy < Hin)
                    v[u] = __ldg(reinterpret_cast<const float4*>(inb + ((size_t)ci * Hin + gy) * Win + gx));
            }
#pragma unroll
            for (int u = 0; u < kBatch; ++u) {
                if (dst[u] < 0) continue;
                float* row = tile + dst[u];
                const int j = jj[u];
                if (j == 0) {
                    row[K::kEOff] = v[u].w;                                              // c = 0 -> E[0]
                } else {
                    // c = 4j-3 (odd) 4j-2 (even) 4j-1 (odd) 4j (even) -> O[2j-2], E[2j-1], O[2j-1], E[2j]
                    *reinterpret_cast<float2*>(row + K::kOOff + 2 * j - 2) = make_float2(v[u].x, v[u].z);
                    *reinterpret_cast<float2*>(row + K::kEOff + 2 * j - 1) = make_float2(v[u].y, v[u].w);
                }
            }
        }
    }
    asm volatile("cp.async.commit_group;\n" ::: "memory");
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");
    __syncthreads();

    conv_compute<CIN, COUT, QG, P, TW, TH, HSWISH, TOKENS, TCOUT_CCH>(tile, ws, bs, tx0, ty0, Hout, Wout, b, out, pos, tok_stride_rows, tok_off);
}

// ---------------------------------------------------------------------------------------------------
// Fused K1 + first stem layer: the 65 x 65 x 3 input tile of conv1 is gathered straight from the raw
// uint8 frame (crop + zero pad + OpenCV-exact fixed-point bilinear + normalisation LUT, exactly the
// arithmetic of crop_normalize_kernel in vt_crop.cu), so the normalised 3 x S x S crop is never
// written to or re-read from HBM.  Column / row taps are computed once per CTA (float64 geometry).
// ---------------------------------------------------------------------------------------------------
using Conv1Cfg = ConvCfg<3, 6, 6, 4, 32, 32>;
constexpr int kCc1Threads = Conv1Cfg::kThreads;                         // 256
constexpr int kCc1TileSide = 2 * 32 + 1;                                // 65 resized-crop pixels per side
constexpr int kCc1WFloats = 2 * Conv1Cfg::kWFloats;                    // conv1 weights duplicated {w, w} for the packed FMAs
constexpr size_t kCc1SmemBytes = Conv1Cfg::kSmemBytes + Conv1Cfg::kWFloats * sizeof(float) + 64 + 2 * 80 * sizeof(int4);     // 4 CTAs / SM

template <int S>
__global__ void __launch_bounds__(kCc1Threads, 4)
crop_conv1_kernel(const uint8_t* __restrict__ frames, const int64_t* __restrict__ frame_offsets,
                  const int4* __restrict__ taps, const float* __restrict__ wg,
                  const float* __restrict__ bg, float* __restrict__ out) {
    using K = Conv1Cfg;
    extern __shared__ __align__(16) float smem[];
    float* tile = smem;
    float* ws = smem + K::kTileFloats;
    float* bs = ws + kCc1WFloats;
    int4* s_col = reinterpret_cast<int4*>(smem + ((K::kTileFloats + kCc1WFloats + 6 + 3) / 4 * 4));
    int4* s_row = s_col + 80;

    constexpr int Hout = S / 2;
    constexpr int tiles_x = Hout / 32;
    const int tx0 = (blockIdx.x % tiles_x) * 32;
    const int ty0 = (blockIdx.x / tiles_x) * 32;
    const int item = blockIdx.y;
    const int tid = threadIdx.x;

    if (tid < 3 * 9 * 6) {                                                 // weights as {w, w} pairs (conv_compute PAIRED)
        const float wv = __ldg(wg + tid);
        reinterpret_cast<float2*>(ws)[tid] = make_float2(wv, wv);
    }
    if (tid < 6) cp_async<4>(bs + tid, bg + tid, true);
    asm volatile("cp.async.commit_group;\n" ::: "memory");

    // this tile's 65 column and 65 row records of the per-track tap tables (crop_taps_kernel)
    if (tid < kCc1TileSide) s_col[tid] = __ldg(taps + ((size_t)item * 2 + 0) * kTapPitch + 2 * tx0 + tid);
    else if (tid >= 128 && tid < 128 + kCc1TileSide) s_row[tid - 128] = __ldg(taps + ((size_t)item * 2 + 1) * kTapPitch + 2 * ty0 + tid - 128);
    __syncthreads();

    const uint8_t* __restrict__ im = frames + frame_offsets[item];
    // One resized-crop pixel (3 channels) of tile position (r, c): 2x2 source taps, 11-bit fixed point exactly as
    // cv::resize (HResize then VResizeLinear 8U), then the normalisation (normalize_px).  Each tap row is read as three aligned
    // 32-bit words covering the pair's six bytes (R0 G0 B0 R1 G1 B1), realigned with funnel shifts; a channel's
    // horizontal pass is one byte permute + one two-way dot product with the packed weights.
    // kB tile rows of one column per batch, in three explicit phases so that every global load of the batch is in
    // flight before its first use: (1) 6 word loads per row, (2) fixed-point bilinear + normalisation, (3) tile stores.
    // Branch-free: padding positions read offset 0 with weight 0 and are zeroed at the end.
    auto gather_col = [&](auto kb_tag, int r_first, int r_step, int n_batches, const int4 ct, int slot) {
        constexpr int kB = decltype(kb_tag)::value;
        const unsigned wx = (unsigned)ct.y;
        const uint8_t* __restrict__ colp = im + ct.x;                     // this thread's column; row offsets are unsigned 32-bit (< 2^31)
#pragma unroll 1
        for (int rb = 0; rb < n_batches; ++rb) {
            uint32_t wd[kB][6];
            unsigned sh[kB][2];
            int bz[kB];
            bool outside[kB];
#pragma unroll
            for (int k = 0; k < kB; ++k) {
                const int4 rt = s_row[r_first + (rb * kB + k) * r_step];
                const uintptr_t q0 = reinterpret_cast<uintptr_t>(colp + (unsigned)rt.x);
                const uintptr_t q1 = reinterpret_cast<uintptr_t>(colp + (unsigned)rt.y);
                const uint32_t* p0 = reinterpret_cast<const uint32_t*>(q0 & ~static_cast<uintptr_t>(3));
                const uint32_t* p1 = reinterpret_cast<const uint32_t*>(q1 & ~static_cast<uintptr_t>(3));
                wd[k][0] = __ldg(p0); wd[k][1] = __ldg(p0 + 1); wd[k][2] = __ldg(p0 + 2);
                wd[k][3] = __ldg(p1); wd[k][4] = __ldg(p1 + 1); wd[k][5] = __ldg(p1 + 2);
                sh[k][0] = (unsigned)q0 << 3; sh[k][1] = (unsigned)q1 << 3;           // the funnel shift takes the amount mod 32 = 8 * (q & 3)
                bz[k] = rt.z;
                outside[k] = ((ct.w | rt.w) & 1) != 0;
            }
            float val[kB][3];
            int px[kB][3];
#pragma unroll
            for (int k = 0; k < kB; ++k) {
                const uint32_t u0 = __funnelshift_r(wd[k][0], wd[k][1], sh[k][0]), u1 = __funnelshift_r(wd[k][1], wd[k][2], sh[k][0]);   // R0 G0 B0 R1 | G1 B1 . .
                const uint32_t t0 = __funnelshift_r(wd[k][3], wd[k][4], sh[k][1]), t1 = __funnelshift_r(wd[k][4], wd[k][5], sh[k][1]);
                const int b0 = bz[k] & 0xffff, b1 = (unsigned)bz[k] >> 16;
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) {
                    const unsigned sel = ch == 0 ? 0x0030u : ch == 1 ? 0x0041u : 0x0052u;             // (first, second) pixel's byte
                    const int h0 = (int)__dp2a_lo(wx, __byte_perm(u0, u1, sel), 0u);
                    const int h1 = (int)__dp2a_lo(wx, __byte_perm(t0, t1, sel), 0u);
                    px[k][ch] = (((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2;       // always in [0, 255]
                }
            }
            // normalisation in registers (no table loads), two rows per packed operation
#pragma unroll
            for (int k = 0; k + 1 < kB; k += 2) {
                normalize_px2<0>(px[k][0], px[k + 1][0], val[k][0], val[k + 1][0]);
                normalize_px2<1>(px[k][1], px[k + 1][1], val[k][1], val[k + 1][1]);
                normalize_px2<2>(px[k][2], px[k + 1][2], val[k][2], val[k + 1][2]);
            }
            if constexpr (kB % 2 == 1) {
                val[kB - 1][0] = normalize_px<0>(px[kB - 1][0]);
                val[kB - 1][1] = normalize_px<1>(px[kB - 1][1]);
                val[kB - 1][2] = normalize_px<2>(px[kB - 1][2]);
            }
#pragma unroll
            for (int k = 0; k < kB; ++k) {
                float* dst = tile + (r_first + (rb * kB + k) * r_step) * K::kPitch + slot;
                dst[0] = outside[k] ? 0.f : val[k][0];
                dst[K::kInRows * K::kPitch] = outside[k] ? 0.f : val[k][1];
                dst[2 * K::kInRows * K::kPitch] = outside[k] ? 0.f : val[k][2];
            }
        }
    };
    {
        // threads own a fixed column (taps in registers) and walk down rows 0..63 in 4 row phases; row 64 and column 64
        // (the tile's halo) are 129 single pixels
        const int c = tid & 63;
        gather_col(std::integral_constant<int, 4>{}, tid >> 6, 4, 4, s_col[c], (c & 1) ? (K::kOOff + (c >> 1)) : (K::kEOff + (c >> 1)));
        if (tid < 64) gather_col(std::integral_constant<int, 1>{}, 64, 0, 1, s_col[tid], (tid & 1) ? (K::kOOff + (tid >> 1)) : (K::kEOff + (tid >> 1)));
        else if (tid < 129) gather_col(std::integral_constant<int, 1>{}, tid - 64, 0, 1, s_col[64], K::kEOff + 32);
    }
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");
    __syncthreads();
    conv_compute<3, 6, 6, 4, 32, 32, true, false, 0, true>(tile, ws, bs, tx0, ty0, Hout, Hout, item, out, nullptr, 0, 0);
}

template <int CIN, int COUT, int QG, int P, int TW, int TH, bool HSWISH, bool TOKENS, int TCOUT_CCH = 0>
static int run_conv(const float* in, int Hin, int n, const StemLayerW& w, float* out, const float* pos,
                    int tok_stride_rows, int tok_off, cudaStream_t st) {
    using K = ConvCfg<CIN, COUT, QG, P, TW, TH>;
    auto kern = conv3x3s2_kernel<CIN, COUT, QG, P, TW, TH, HSWISH, TOKENS, TCOUT_CCH>;
    static DeviceOnce once;
    if (!ensure_dyn_smem(once, kern, K::kSmemBytes)) return -1;
    const int Hout = Hin / 2;
    const int tiles = ((Hout + TW - 1) / TW) * ((Hout + TH - 1) / TH);
    int launched = 0;
    for (int first = 0; first < n; first += 32768) {
        const int m = min(32768, n - first);
        dim3 grid(tiles, m);
        const float* inp = in + (size_t)first * CIN * Hin * Hin;
        float* o = TCOUT_CCH > 0 ? reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(out) + (size_t)first * tc_planes_bytes(TCOUT_CCH, Hout / 2))
                   : TOKENS ? out + (size_t)first * tok_stride_rows * COUT : out + (size_t)first * COUT * Hout * Hout;
        kern<<<grid, K::kThreads, K::kSmemBytes, st>>>(inp, Hin, Hin, w.w, w.b, o, pos, tok_stride_rows, tok_off);
        ++launched;
    }
    return cudaGetLastError() == cudaSuccess ? launched : -1;
}

size_t stem_scratch_floats(int S) {
    // conv1 out 6 x S/2 x S/2, conv2 out 12 x S/4 x S/4, conv3 out 24 x S/8 x S/8
    return (size_t)6 * (S / 2) * (S / 2) + (size_t)12 * (S / 4) * (S / 4) + (size_t)24 * (S / 8) * (S / 8);
}

size_t crop_taps_bytes(int n) { return (size_t)n * 2 * kTapPitch * sizeof(int4) + 256; }      // + the fused front's work counter

template <int S>
static int run_crop_conv1(const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw, const double* boxes,
                          double factor, int n, const ModelW& w, float* out, int32_t* out_status, int4* taps, cudaStream_t st) {
    auto kern = crop_conv1_kernel<S>;
    static DeviceOnce once;
    if (!ensure_dyn_smem(once, kern, kCc1SmemBytes)) return -1;
    constexpr int tiles = (S / 64) * (S / 64);
    crop_taps_kernel<S><<<n, 288, 0, st>>>(frame_hw, boxes, factor, taps, out_status, nullptr, 0);
    int launched = 1;
    for (int first = 0; first < n; first += 32768) {
        const int m = min(32768, n - first);
        kern<<<dim3(tiles, m), kCc1Threads, kCc1SmemBytes, st>>>(frames, frame_offsets + first, taps + (size_t)first * 2 * kTapPitch,
                                                                 w.stem[0].w, w.stem[0].b, out + (size_t)first * 6 * (S / 2) * (S / 2));
        ++launched;
    }
    return cudaGetLastError() == cudaSuccess ? launched : -1;
}

// Crop + stem straight from raw frames (fused first layer); same outputs as launch_crop_normalize + launch_stem.
int launch_crop_stem(const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw, const double* boxes,
                     double factor, int S, int n, const ModelW& w, float* scratch, float* tokens, int tok_stride_rows,
                     int tok_off, int32_t* out_status, uint8_t* planes, int plane_tracks, void* tap_tables, cudaStream_t st) {
    if (n <= 0) return 0;
    int4* taps = reinterpret_cast<int4*>(tap_tables);
    float* a1 = scratch;
    float* a2 = a1 + (size_t)n * 6 * (S / 2) * (S / 2);
    float* a3 = a2 + (size_t)n * 12 * (S / 4) * (S / 4);
    const float* pos = (S == kSx) ? w.pos_x : w.pos_z;
    int total = 0, r;
    if (planes && S == kSx && n <= plane_tracks) {
        // search branch: crop + conv1 + conv2 in one tcgen05 kernel (vt_stem_fused.cu), then layers 3-4 on tcgen05.  The planes
        // buffer keeps conv2's operand image first (launch_stem writes it), so conv3's image starts after it.
        uint8_t* planes3 = planes + (size_t)plane_tracks * tc_planes_bytes(kConv2Cch, kConv2Wout);
        uint8_t* planes4 = planes3 + (size_t)plane_tracks * tc_planes_bytes(kConv3Cch, kConv3Wout);
        if ((r = launch_crop_stem12_fused(frames, frame_offsets, frame_hw, boxes, factor, n, w, out_status, tap_tables, planes3, st)) < 0) return r;
        total += r;
        if ((r = launch_stem34_tc(planes3, n, w, planes4, tokens, tok_stride_rows, tok_off, st)) < 0) return r;
        return total + r;
    }
    if (S == 256) r = run_crop_conv1<256>(frames, frame_offsets, frame_hw, boxes, factor, n, w, a1, out_status, taps, st);
    else if (S == 128) r = run_crop_conv1<128>(frames, frame_offsets, frame_hw, boxes, factor, n, w, a1, out_status, taps, st);
    else return -1;
    if (r < 0) return r;
    total += r;
    if ((r = run_conv<6, 12, 12, 2, 32, 16, true, false>(a1, S / 2, n, w.stem[1], a2, nullptr, 0, 0, st)) < 0) return r;
    total += r;
    if ((r = run_conv<12, 24, 12, 2, 32, 8, true, false>(a2, S / 4, n, w.stem[2], a3, nullptr, 0, 0, st)) < 0) return r;
    total += r;
    if ((r = run_conv<24, 48, 12, 4, 16, 16, false, true>(a3, S / 8, n, w.stem[3], tokens, pos, tok_stride_rows, tok_off, st)) < 0) return r;
    total += r;
    return total;
}

int launch_stem(const float* img, int S, int n, const ModelW& w, float* scratch, float* tokens,
                int tok_stride_rows, int tok_off, uint8_t* planes, int plane_tracks, cudaStream_t st) {
    if (n <= 0) return 0;
    float* a1 = scratch;
    float* a2 = a1 + (size_t)n * 6 * (S / 2) * (S / 2);
    float* a3 = a2 + (size_t)n * 12 * (S / 4) * (S / 4);
    const float* pos = (S == kSx) ? w.pos_x : w.pos_z;
    int total = 0, r;
    //                CIN COUT QG P  TW  TH  hswish tokens
    if (planes && S == kSx && n <= plane_tracks) {
        // search branch: conv1 writes conv2's tensor-core operand image; layers 2-4 run on tcgen05
        uint8_t* planes2 = planes;
        uint8_t* planes3 = planes2 + (size_t)plane_tracks * tc_planes_bytes(kConv2Cch, kConv2Wout);
        uint8_t* planes4 = planes3 + (size_t)plane_tracks * tc_planes_bytes(kConv3Cch, kConv3Wout);
        if ((r = run_conv<3, 6, 6, 4, 32, 32, true, false, kConv2Cch>(img, S, n, w.stem[0], reinterpret_cast<float*>(planes2), nullptr, 0, 0, st)) < 0) return r;
        total += r;
        if ((r = launch_stem234_tc(planes2, n, w, planes3, planes4, tokens, tok_stride_rows, tok_off, st)) < 0) return r;
        return total + r;
    }
    if ((r = run_conv<3, 6, 6, 4, 32, 32, true, false>(img, S, n, w.stem[0], a1, nullptr, 0, 0, st)) < 0) return r;
    total += r;
    if ((r = run_conv<6, 12, 12, 2, 32, 16, true, false>(a1, S / 2, n, w.stem[1], a2, nullptr, 0, 0, st)) < 0) return r;
    total += r;
    if ((r = run_conv<12, 24, 12, 2, 32, 8, true, false>(a2, S / 4, n, w.stem[2], a3, nullptr, 0, 0, st)) < 0) return r;
    total += r;
    if ((r = run_conv<24, 48, 12, 4, 16, 16, false, true>(a3, S / 8, n, w.stem[3], tokens, pos, tok_stride_rows, tok_off, st)) < 0) return r;
    total += r;
    return total;
}

}  // namespace vt
