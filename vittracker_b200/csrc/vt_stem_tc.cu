// Stem layers 2, 3 and 4 (conv3x3 stride 2 pad 1 + folded BN [+ Hardswish], lib/models/vit_dist/vit_dist.py:36-54)
// on the tcgen05 tensor cores, for the search branch (S = 256).
//
// A stride-2 convolution reads in[2oy+ky-1][2ox+kx-1].  Its input arrives as a "plane image" (vt_internal.h,
// tc_planes_offset) that the PRODUCING layer's epilogue wrote: fp16 hi / lo, 8-channel chunks, split by (row
// parity, column parity) into four planes P[rp][cp][r][c] = in[2r+rp][2c+cp] with pitch exactly W_out.  The
// 128 output pixels of an M tile are then 128 consecutive 16-byte rows of any plane, so a no-swizzle K-major
// UMMA descriptor addresses tap (ky, kx) by picking the plane (rp = ky odd ? 0 : 1, cp = kx odd ? 0 : 1) and
// a start row, and staging a band of 8 output rows is a handful of cp.async.bulk copies - no instructions.
// The kx = 0 taps need column index ox-1: they accumulate UNSHIFTED into a second TMEM accumulator T_B that
// the epilogue shifts by one TMEM lane with a warp shuffle (a warp's 32 lanes are whole image rows - or, at W_out = 64,
// half a row, the value crossing the middle going through shared memory; the value entering at ox = 0 is the zero padding).  Products are hi*hi + lo*hi + hi*lo, fp32 accumulation.
#include <string.h>

#include "vt_internal.h"
#include "vt_stem_tc.cuh"
#include "vt_tc.cuh"

namespace vt {

using namespace tc;

// Optional cycle trace of the control warp and of one epilogue thread of CTA 0 of the conv4 instantiation (development aid):
// -DVT_CONV_TRACE, read back with vt_conv_trace_read().
#ifdef VT_CONV_TRACE
__device__ long long g_conv_trace[3][2048];
__device__ int g_conv_trace_n[3];
#define CONV_TRACE(side, on)                                                                                     \
    do {                                                                                                         \
        if ((on) && blockIdx.x == 0 && lane == 0) { int k__ = g_conv_trace_n[side]; if (k__ < 2048) { g_conv_trace[side][k__] = clock64(); g_conv_trace_n[side] = k__ + 1; } } \
    } while (0)
extern "C" int vt_conv_trace_read(long long* host, int* n) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(n, g_conv_trace_n, 3 * sizeof(int));
    cudaMemcpyFromSymbol(host, g_conv_trace, sizeof(long long) * 3 * 2048);
    int zero[3] = {0, 0, 0};
    cudaMemcpyToSymbol(g_conv_trace_n, zero, sizeof zero);
    return 0;
}
#else
#define CONV_TRACE(side, on) do {} while (0)
#endif

// Persistent: a CTA walks over work items (track, band of BR output rows).  in: plane images [n][tc_planes_bytes(CCH, WOUT)];
// wt: packed fp16 hi|lo weight blob in K-step order (loaded once per CTA); bias fp32 [COUT].  OUT_PLANES: write the next
// layer's plane image (NEXT_CCH chunks, WOUT/2 wide), else tokens [n][tok_stride_rows][COUT] + positional embedding.
// Warp 17 = bulk copies (one stage ahead), warp 16 = single-thread MMA issue, warps 0-7 / 8-15 = the
// epilogue groups of accumulator set 0 / 1; two A stages in shared memory and two accumulator sets in TMEM, handed over
// through mbarriers.
template <int CCH, int COUT, int NPAD, int WOUT, int BR, bool HSWISH, bool OUT_PLANES, int NEXT_CCH>
__global__ void __launch_bounds__(576)
conv_s2_tc_kernel(const uint8_t* __restrict__ in, const uint8_t* __restrict__ wt, const float* __restrict__ bias,
                  void* __restrict__ outp, const float* __restrict__ pos, int tok_stride_rows, int tok_off, int n_items) {
    using K = TcConv<CCH, COUT, NPAD, WOUT, BR>;
    constexpr int kBands = WOUT / BR;
    extern __shared__ __align__(128) uint8_t smem_tc[];
    uint8_t* sW = smem_tc + K::kOffW;
    float* sBias = reinterpret_cast<float*>(smem_tc + K::kOffBias);
    float* sXchg = reinterpret_cast<float*>(smem_tc + K::kOffXchg);
    uint64_t* bar_w = reinterpret_cast<uint64_t*>(smem_tc + K::kOffBar);
    uint64_t* bar_full = bar_w + 1;      // [2] A stage landed                    (one expect_tx arrival for the stage's copies)
    uint64_t* bar_afree = bar_w + 3;     // [2] A stage consumed by the MMAs      (tcgen05.commit)
    uint64_t* bar_tfull = bar_w + 5;     // [2] accumulators complete             (tcgen05.commit)
    uint64_t* bar_tfree = bar_w + 7;     // [2] accumulators read by the epilogue (8 warp arrivals)
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bar_w + 9);
    const int tid = threadIdx.x, lane = tid & 31;
    const int wid = tid >> 5;                    // 0-15 epilogue, 16 MMA issue, 17 bulk copies
    const int warp = wid & 7, group = wid >> 3;  // epilogue warp within its group; group = accumulator set it serves

    if (wid == 16) tmem_alloc(s_tmem, K::kTmemCols);
    if (tid == 0) {
        mbar_init(bar_w, 1);
        for (int i = 0; i < 2; ++i) { mbar_init(bar_full + i, 1); mbar_init(bar_afree + i, 1); mbar_init(bar_tfull + i, 1); mbar_init(bar_tfree + i, 8); }
        mbar_fence_init();
    }
    if (tid < NPAD) sBias[tid] = tid < COUT ? __ldg(bias + tid) : 0.f;
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tbase = __shfl_sync(0xffffffffu, *s_tmem, 0);

    if (wid == 17) {
        // ---- producer warp: the bulk copies of every item, one stage ahead of the MMAs.  A stage's 8 - 24 copies are started by ONE warp
        // instruction (a copy per lane) behind a single arming of the barrier, and by a warp of their own: issued one after the other
        // between the MMAs they cost the control warp ~200 cycles each - more than half of an item's time in conv4.
        static_assert(K::kCopies <= 32, "one copy per lane");
        bulk_g2s_elect(sW, wt, K::kWBytes, bar_w);
        int it = 0;
#pragma unroll 1
        for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
            const int st = it & 1;
            CONV_TRACE(2, CCH == 3);
            if (it >= 2) mbar_wait(bar_afree + st, ((it - 2) >> 1) & 1);                // the stage's previous user's MMAs are done
            CONV_TRACE(2, CCH == 3);
            const int b = item / kBands, oy0 = (item % kBands) * K::kBR;     // plane rows [oy0, oy0 + BR + 1) of every (precision, plane, chunk)
            const uint8_t* inr = in + (size_t)b * tc_planes_bytes(CCH, WOUT) + (size_t)oy0 * WOUT * 16;
            uint8_t* sA = smem_tc + K::kOffA + st * K::kStageBytes;
            mbar_arrive_expect_tx_elect(bar_full + st, K::kCopies * K::kChunkBytes);
            __syncwarp();
            if (lane < K::kCopies) {
                const int chunk = lane % CCH, plane = (lane / CCH) & 3, prec = lane / (4 * CCH);
                const size_t src = ((size_t)(prec * 4 + plane) * CCH + chunk) * (WOUT + 1) * WOUT * 16;
                bulk_g2s(sA + prec * K::kABytes + (plane * CCH + chunk) * K::kChunkBytes, inr + src, K::kChunkBytes, bar_full + st);
            }
            __syncwarp();
            CONV_TRACE(2, CCH == 3);
        }
    } else if (wid == 16) {          // MMA warp; convergent, the elected lane issues MMAs and commits
        const uint32_t sbase = smem_u32(smem_tc);
        const uint32_t idesc = instr_desc_f16(128, NPAD, false);
        mbar_wait(bar_w, 0);
        int it = 0;
#pragma unroll 1
        for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
            const int st = it & 1;
            const uint32_t ph = (it >> 1) & 1;
            CONV_TRACE(0, CCH == 3);
            mbar_wait(bar_full + st, ph);
            CONV_TRACE(0, CCH == 3);
            if (it >= 2) mbar_wait(bar_tfree + st, ((it - 2) >> 1) & 1);                // accumulator set st has been read
            tc_fence_after();
            CONV_TRACE(0, CCH == 3);
            const uint32_t abase = sbase + K::kOffA + st * K::kStageBytes;
#pragma unroll 1
            for (int tile = 0; tile < K::kTiles; ++tile) {          // rolled: the descriptors are affine in `tile`
#pragma unroll
                for (int acc = 0; acc < 2; ++acc) {                             // 0: T_A (kx = 1, 2)   1: T_B (kx = 0, shifted later)
                    const uint32_t d = tbase + st * K::kAccCols + (tile * 2 + acc) * NPAD;
                    const int nsteps = acc == 0 ? K::kStepsA : K::kStepsB;
#pragma unroll
                    for (int s2 = 0; s2 < nsteps; ++s2) {
                        int tap0, ch0, tap1, ch1; bool zero1;
                        tcs_step(CCH, acc, s2, tap0, ch0, tap1, ch1, zero1);
                        int ky, kx, p0, r0, p1, r1;
                        tcs_tap(acc, tap0, ky, kx); tcs_tap_pos(ky, kx, p0, r0);
                        tcs_tap(acc, tap1, ky, kx); tcs_tap_pos(ky, kx, p1, r1);
                        const uint32_t a0 = (p0 * CCH + ch0) * K::kChunkBytes + (tile * K::kRowsPerTile + r0) * WOUT * 16;
                        const uint32_t a1 = (p1 * CCH + ch1) * K::kChunkBytes + (tile * K::kRowsPerTile + r1) * WOUT * 16;
                        const uint32_t lbo = zero1 ? 16 : a1 - a0;              // > 0 by construction of the schedule; zero weights: any finite data
                                                                                // inside the CTA's shared memory (one pixel further: at most 16 bytes into the next region)
                        const uint64_t ah = smem_desc(abase + a0, lbo, 128);
                        const uint64_t al = smem_desc(abase + K::kABytes + a0, lbo, 128);
                        const uint32_t boff = ((acc == 0 ? 0 : K::kStepsA) + s2) * 2 * NPAD * 16;
                        const uint64_t bh = smem_desc(sbase + K::kOffW + boff, NPAD * 16, 128);
                        const uint64_t bl = smem_desc(sbase + K::kOffW + K::kWPrecBytes + boff, NPAD * 16, 128);
                        mma_ss_elect(d, ah, bh, idesc, s2 > 0 ? 1u : 0u);
                        mma_ss_elect(d, al, bh, idesc, 1u);
                        mma_ss_elect(d, ah, bl, idesc, 1u);
                    }
                }
            }
            mma_commit_elect(bar_afree + st);
            mma_commit_elect(bar_tfull + st);
            CONV_TRACE(0, CCH == 3);
        }
        __syncwarp();
    } else {
        // ---- epilogue: 8 warps = 2 (tile or channel half) x 4 TMEM lane quarters; thread -> one output pixel ------------------
        constexpr int kPasses = (K::kTiles >= 2) ? K::kTiles / 2 : 1;           // two tiles per pass, or one tile split by channels
        constexpr int kChPerThread = (K::kTiles >= 2) ? NPAD : NPAD / 2;
        static_assert(kChPerThread % 8 == 0 && (K::kTiles == 1 || K::kTiles % 2 == 0), "epilogue split");
        constexpr bool kSplitRows = WOUT > 32;                                  // TMEM lane quarter (= warp) shorter than an image row
        static_assert(!kSplitRows || (WOUT == 64 && K::kTiles >= 2 && kPasses * (kChPerThread / 8) <= 4), "row split");
        const int chb = (K::kTiles >= 2) ? 0 : (warp >> 2) * kChPerThread;
        const int r = 32 * (warp & 3) + lane;                                   // row of the M tile = TMEM lane
        int it = 0;
#pragma unroll 1
        for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
            const int st = it & 1;
            if (st != group) continue;                                          // the other group's accumulator set
            const int b = item / kBands, oy0 = (item % kBands) * K::kBR;
            CONV_TRACE(1, CCH == 3 && wid == 0);
            mbar_wait(bar_tfull + st, (it >> 1) & 1);
            tc_fence_after();
            CONV_TRACE(1, CCH == 3 && wid == 0);
#pragma unroll 1
            for (int pass = 0; pass < kPasses; ++pass) {
                const int tile = (K::kTiles >= 2) ? 2 * pass + (warp >> 2) : 0;
                const int oy = oy0 + tile * K::kRowsPerTile + r / WOUT, ox = r % WOUT;
                const uint32_t ta = tbase + ((uint32_t)(32 * (warp & 3)) << 16) + st * K::kAccCols + tile * 2 * NPAD + chb;
#pragma unroll 1
                for (int c0 = 0; c0 < kChPerThread; c0 += 8) {
                    uint32_t ra[8], rb[8];
                    tmem_ld8(ta + c0, ra);
                    tmem_ld8(ta + NPAD + c0, rb);
                    tc_wait_ld();
                    float* xs = sXchg + ((((group * 4 + pass * (kChPerThread / 8) + c0 / 8) * 2 + (warp >> 2)) * 2 + ((warp & 3) >> 1)) * 8);
                    if constexpr (kSplitRows) {
                        // an image row spans two warps: column 31's T_B crosses to column 32 through shared memory
                        if (lane == 31 && !(warp & 1)) {
#pragma unroll
                            for (int j = 0; j < 8; ++j) xs[j] = __uint_as_float(rb[j]);
                        }
                        asm volatile("bar.sync %0, 256;" ::"r"(1 + group) : "memory");
                    }
                    float v[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        float tb = __shfl_up_sync(0xffffffffu, __uint_as_float(rb[j]), 1);     // T_B[oy][ox-1]
                        if constexpr (kSplitRows) {
                            if (lane == 0 && (warp & 1)) tb = xs[j];
                        }
                        if (ox == 0) tb = 0.f;
                        v[j] = __uint_as_float(ra[j]) + tb + sBias[chb + c0 + j];
                    }
                    if (HSWISH) hardswish_n<8>(v);
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        if (chb + c0 + j >= COUT) v[j] = 0.f;                           // padding channels stay exactly zero
                    if (chb + c0 >= COUT) continue;
                    if (OUT_PLANES) {
                        // this layer's output pixel (oy, ox) is the next layer's input pixel: 8 channels = one chunk, hi | lo
                        uint32_t hi[4], lo[4];
#pragma unroll
                        for (int j = 0; j < 4; ++j) split_pack2(v[2 * j], v[2 * j + 1], hi[j], lo[j]);
                        uint8_t* ob = reinterpret_cast<uint8_t*>(outp) + (size_t)b * tc_planes_bytes(NEXT_CCH, WOUT / 2);
                        const int chunk = (chb + c0) / 8;
                        *reinterpret_cast<uint4*>(ob + tc_planes_offset(0, oy, ox, chunk, NEXT_CCH, WOUT / 2)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                        *reinterpret_cast<uint4*>(ob + tc_planes_offset(1, oy, ox, chunk, NEXT_CCH, WOUT / 2)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                    } else {
                        const int tok = oy * WOUT + ox;
                        float* o = reinterpret_cast<float*>(outp) + ((size_t)b * tok_stride_rows + tok_off + tok) * COUT + chb + c0;
                        const float* pe = pos + (size_t)tok * COUT + chb + c0;
                        const float4 e0 = __ldg(reinterpret_cast<const float4*>(pe)), e1 = __ldg(reinterpret_cast<const float4*>(pe + 4));
                        *reinterpret_cast<float4*>(o) = make_float4(v[0] + e0.x, v[1] + e0.y, v[2] + e0.z, v[3] + e0.w);
                        *reinterpret_cast<float4*>(o + 4) = make_float4(v[4] + e1.x, v[5] + e1.y, v[6] + e1.z, v[7] + e1.w);
                    }
                }
            }
            // the row-split exchange slots are reused by the next item: every epilogue warp is past its reads
            if constexpr (kSplitRows) asm volatile("bar.sync %0, 256;" ::"r"(1 + group) : "memory");
            CONV_TRACE(1, CCH == 3 && wid == 0);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_tfree + st);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (wid == 16) tmem_dealloc(tbase, K::kTmemCols);
}

template <int CCH, int COUT, int NPAD, int WOUT, int BR, bool HSWISH, bool OUT_PLANES, int NEXT_CCH>
static int run_tc_conv(const uint8_t* in, int n, const uint8_t* wt, const float* bias, void* out, const float* pos,
                       int tok_stride_rows, int tok_off, cudaStream_t st) {
    using K = TcConv<CCH, COUT, NPAD, WOUT, BR>;
    auto kern = conv_s2_tc_kernel<CCH, COUT, NPAD, WOUT, BR, HSWISH, OUT_PLANES, NEXT_CCH>;
    static int grid_caps[kMaxDevices] = {};                          // per device ordinal: the opt-in and the SM count are per device
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return -1;
    if (grid_caps[dev] == 0) {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, K::kSmemBytes) != cudaSuccess) return -1;
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1;
        grid_caps[dev] = sms * resident_ctas_per_sm(kern, K::kThreads, K::kSmemBytes, K::kTmemCols, dev);
    }
    const int grid_cap = grid_caps[dev];
    const long long items = (long long)n * (WOUT / K::kBR);
    if (items > 0x7fffffffLL) return -1;
    const int grid = items < grid_cap ? (int)items : grid_cap;
    kern<<<grid, K::kThreads, K::kSmemBytes, st>>>(in, wt, bias, out, pos, tok_stride_rows, tok_off, (int)items);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

// Search-branch layers on the tensor cores: conv2 (6 -> 12, 128x128 -> 64x64), conv3 (12 -> 24, -> 32x32), both with
// Hardswish and writing the next layer's operand image, and conv4 (24 -> 48, -> 16x16) writing tokens + pos-embed.
int launch_stem234_tc(const uint8_t* planes2, int n, const ModelW& w, uint8_t* planes3, uint8_t* planes4, float* tokens,
                      int tok_stride_rows, int tok_off, cudaStream_t st) {
    int total = 0, r;
    if ((r = run_tc_conv<kConv2Cch, 12, 16, kConv2Wout, kConv2BR, true, true, kConv3Cch>(planes2, n, w.stem_tc_w[0], w.stem_tc_b[0], planes3,
                                                                               nullptr, 0, 0, st)) < 0) return r;
    total += r;
    if ((r = run_tc_conv<kConv3Cch, 24, 32, kConv3Wout, kConv3BR, true, true, kConv4Cch>(planes3, n, w.stem_tc_w[1], w.stem_tc_b[1], planes4,
                                                                               nullptr, 0, 0, st)) < 0) return r;
    total += r;
    if ((r = run_tc_conv<kConv4Cch, 48, 48, kConv4Wout, 8, false, false, 1>(planes4, n, w.stem_tc_w[2], w.stem_tc_b[2], tokens, w.pos_x,
                                                                          tok_stride_rows, tok_off, st)) < 0) return r;
    total += r;
    return total;
}

int launch_stem34_tc(const uint8_t* planes3, int n, const ModelW& w, uint8_t* planes4, float* tokens, int tok_stride_rows, int tok_off,
                     cudaStream_t st) {
    int total = 0, r;
    if ((r = run_tc_conv<kConv3Cch, 24, 32, kConv3Wout, kConv3BR, true, true, kConv4Cch>(planes3, n, w.stem_tc_w[1], w.stem_tc_b[1], planes4,
                                                                               nullptr, 0, 0, st)) < 0) return r;
    total += r;
    if ((r = run_tc_conv<kConv4Cch, 48, 48, kConv4Wout, 8, false, false, 1>(planes4, n, w.stem_tc_w[2], w.stem_tc_b[2], tokens, w.pos_x,
                                                                          tok_stride_rows, tok_off, st)) < 0) return r;
    return total + r;
}

size_t stem_tc_weight_bytes(int layer) {      // layer 0: conv2, 1: conv3, 2: conv4
    return layer == 0 ? (size_t)TcConv<kConv2Cch, 12, 16, kConv2Wout, kConv2BR>::kWBytes
           : layer == 1 ? (size_t)TcConv<kConv3Cch, 24, 32, kConv3Wout, kConv3BR>::kWBytes : (size_t)TcConv<kConv4Cch, 48, 48, kConv4Wout, 8>::kWBytes;
}

// Host side of the K-step schedule: weight blob of one layer (fp16 hi | lo), `wf` = folded weights [ci][ky][kx][cout].
void stem_tc_pack_weights(int cin, int cch, int cout, int npad, const float* wf, uint8_t* hi8, uint8_t* lo8) {
    int slot = 0;
    for (int acc = 0; acc < 2; ++acc)
        for (int s = 0; s < tcs_nsteps(cch, acc); ++s, ++slot) {
            int tap[2], ch[2]; bool zero1;
            tcs_step(cch, acc, s, tap[0], ch[0], tap[1], ch[1], zero1);
            for (int half = 0; half < 2; ++half) {
                int ky, kx;
                tcs_tap(acc, tap[half], ky, kx);
                for (int n = 0; n < npad; ++n)
                    for (int e = 0; e < 8; ++e) {
                        const int ci = ch[half] * 8 + e;
                        float v = 0.f;
                        if (!(half == 1 && zero1) && ci < cin && n < cout) v = wf[(((size_t)ci * 3 + ky) * 3 + kx) * cout + n];
                        uint16_t h, l;
                        split_f16(v, &h, &l);
                        const size_t off = ((size_t)(slot * 2 + half) * npad + n) * 16 + e * 2;
                        memcpy(hi8 + off, &h, 2);
                        memcpy(lo8 + off, &l, 2);
                    }
            }
        }
}

}  // namespace vt
