// Fused search-branch stem front: sample_target (crop + zero pad + OpenCV-exact bilinear resize) -> Preprocessor (normalisation) ->
// conv1 (3 -> 6, 3x3 s2, BN folded, Hardswish) -> conv2 (6 -> 12, 3x3 s2, BN folded, Hardswish) in ONE kernel, both convolutions on the
// tcgen05 tensor cores, nothing but the raw uint8 frame read and conv3's operand image written.
//   lib/train/data/processing_utils.py:12-79, lib/test/tracker/data_utils.py:6-17, lib/models/vit_dist/vit_dist.py:10-54
//
// Why conv1 can run on the tensor cores exactly: the resized crop is uint8, and an integer 0..255 is exact in fp16.  The normalisation
// ((p / 255) - mean) / std is affine per channel, so it folds into the weights and the bias:
//     sum_taps w * ((p / 255 - mean) / std)  =  sum_taps (w / (255 std)) * p  -  sum_taps w * mean / std
// The A operand is the crop itself (fp16, exact), the B operand the folded weights as fp16 hi + lo (scaled by a power of two so that
// both halves are normal numbers), accumulation fp32 in TMEM.  Zero padding of the CONVOLUTION contributes 0 to the first sum because
// the padded pixel is 0; its share of the second sum is left out of the bias: four bias variants (interior, top row, left column,
// corner).  Zero padding of the CROP (pixels outside the frame) is pixel value 0, as in the reference, and needs nothing special.
//
// Work item = (track, band of kBR2 = 4 conv2 output rows).  Per item, with 512 threads:
//   1. gather: the band needs resized-crop rows 4 oy0 - 3 .. 4 oy0 + 4 kBR2 - 1; a thread owns one PAIR of adjacent columns (2x, 2x + 1)
//      and walks down the rows (same integer arithmetic as crop_conv1_kernel: aligned word loads, funnel shifts, byte permute + dp2a,
//      11-bit fixed point).  The six bytes of the pair become six fp16 = one 16-byte K chunk {R G B R G B 0 0} - one STS.128.  A row is
//      stored as a zero chunk followed by its 128 pair chunks.
//   2. conv1: an M = 128 tile is one conv1 output row; tap ky is the row slot 2r + ky.  Taps kx = 1, 2 are the two pixels of chunk x, tap
//      kx = 0 is the second pixel of chunk x - 1: a second MMA whose A operand starts one chunk EARLIER (the zero chunk feeds x = 0)
//      accumulates it into the same columns - no shifted accumulator, no shuffles.  hi and lo weights sit side by side on the N axis
//      (N = 16: columns 0..5 | 8..13), so a K step is one MMA per variant: 4 MMAs per output row.
//   3. epilogue 1: (hi + lo) * 2^-s + bias variant, Hardswish, fp16 hi/lo split -> conv2's parity-plane operand image in shared memory.
//   4. conv2 + epilogue 2: as conv_s2_tc_kernel (vt_stem_tc.cu), reading that image; writes conv3's operand image to global memory.
#include <math.h>
#include <string.h>

#include "vt_geom.cuh"
#include "vt_internal.h"
#include "vt_stem_tc.cuh"
#include "vt_taps.cuh"
#include "vt_tc.cuh"

namespace vt {

using namespace tc;

// Optional cycle trace of one worker thread of CTA 0 (development aid): -DVT_FUSED_TRACE, read back with vt_fused_trace_read().
#ifdef VT_FUSED_TRACE
__device__ long long g_fused_trace[8192];
__device__ int g_fused_trace_n;
__device__ long long g_fused_cta[1024][4];      // per CTA: globaltimer at kernel entry, loop start, loop end; SM id
#define FUSED_TRACE()                                                                                                   \
    do {                                                                                                                \
        if (blockIdx.x == 0 && threadIdx.x == 511) { int k__ = g_fused_trace_n; if (k__ < 8192) { g_fused_trace[k__] = clock64(); g_fused_trace_n = k__ + 1; } } \
    } while (0)
#else
#define FUSED_TRACE() do {} while (0)
#endif

namespace {

constexpr int kFThreads = 512;
constexpr int kIPitch = 129 * 16;              // one resized-crop row in shared memory: a zero chunk + 128 pixel-pair chunks of 16 bytes

struct Fused {
    static constexpr int kBR2 = 4;                                // conv2 output rows of a band
    using C2 = TcConv<kConv2Cch, 12, 16, kConv2Wout, kBR2>;      // conv2: band geometry (A operand planes) and weight blob
    static constexpr int kBands = kConv2Wout / kBR2;
    static constexpr int kUnitBands = 4;                          // consecutive bands of one track a CTA takes at a time (work unit), at most
    static constexpr int kIRows = 4 * kBR2 + 3;                   // resized-crop rows of a band
    static constexpr int kA1Rows = 2 * kBR2 + 1;                  // conv1 output rows of a band
    static constexpr int kOffI = 0;
    static constexpr int kIBytes = (kIRows * kIPitch + 16 + 127) / 128 * 128;     // + one trailing zero chunk
    static constexpr int kOffA1 = kOffI + kIBytes;
    static constexpr int kOffW1 = kOffA1 + 2 * C2::kABytes;       // hi | lo planes
    static constexpr int kOffW2 = kOffW1 + kStem1TcWBytes;
    static constexpr int kOffPar = kOffW2 + C2::kWBytes;          // conv1: bias[4][8], 2^-s (40 floats); conv2: bias[16]
    static constexpr int kOffXchg = kOffPar + (kStem1TcParFloats + 16) * 4;
    static constexpr int kPasses = (C2::kTiles + 1) / 2;
    static constexpr int kXchgFloats = kPasses * 2 * 2 * 2 * 8;   // [pass][tile of the pair][channel half][image row of the tile][8]
    static constexpr int kOffBar = (kOffXchg + kXchgFloats * 4 + 7) / 8 * 8;
    static constexpr int kSmemBytes = kOffBar + 4 * 8;            // bar1, bar2, TMEM base, next item [2]
    static_assert(kBands % kUnitBands == 0 && kUnitBands >= 2, "work units");
    static constexpr int kCol2 = kA1Rows * 16;                    // conv2's accumulators follow conv1's
    static constexpr int kCols = kCol2 + C2::kTiles * 32;
    static constexpr int kTmemCols = kCols <= 128 ? 128 : kCols <= 256 ? 256 : 512;
    static constexpr int kCtasPerSm = (2 * kSmemBytes <= 220 * 1024 && kTmemCols <= 256) ? 2 : 1;
    static_assert(kOffA1 % 128 == 0 && kOffW1 % 128 == 0 && kOffW2 % 128 == 0 && kCols <= 512 && C2::kTiles % 2 == 0 && kSmemBytes <= 227 * 1024, "layout");
};

// One resized-crop pixel (3 channels) from its 2 x 2 source taps, exactly cv::resize's 8U bilinear (HResize: 11-bit weights, then
// VResizeLinear: ((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2) - the arithmetic of crop_conv1_kernel /
// crop_normalize_kernel - with 0x6400 added: the result is the bit pattern of the fp16 number 1024 + v.
// wd: three aligned words per tap row covering the pixel pair's six bytes; sh: byte misalignment * 8; b0 / b1: the row weights.
// One permute serves two channels: R0 R1 G0 G1 in one word feeds dp2a.lo (red) and dp2a.hi (green).  (tools/ubench/gather_arith.cu: this
// arrangement costs 44 issue cycles per pixel and warp against 49 with a permute per channel; multiply-high forms of the vertical
// pass - (b * (h >> 4)) >> 16 == hi32((h & ~15) * (b << 12)) - are slower, 52 - 69: IMAD.HI is not a full-rate instruction.)
__device__ __forceinline__ void bilinear_px3(const uint32_t (&wd)[6], unsigned sh0, unsigned sh1, unsigned wx, int b0, int b1, int (&px)[3]) {
    const uint32_t u0 = __funnelshift_r(wd[0], wd[1], sh0), u1 = __funnelshift_r(wd[1], wd[2], sh0);   // R0 G0 B0 R1 | G1 B1 . .
    const uint32_t t0 = __funnelshift_r(wd[3], wd[4], sh1), t1 = __funnelshift_r(wd[4], wd[5], sh1);
    const uint32_t urg = __byte_perm(u0, u1, 0x4130), ubb = __byte_perm(u0, u1, 0x0052);                // R0 R1 G0 G1 | B0 B1 . .
    const uint32_t trg = __byte_perm(t0, t1, 0x4130), tbb = __byte_perm(t0, t1, 0x0052);
    const int h0[3] = {(int)__dp2a_lo(wx, urg, 0u), (int)__dp2a_hi(wx, urg, 0u), (int)__dp2a_lo(wx, ubb, 0u)};
    const int h1[3] = {(int)__dp2a_lo(wx, trg, 0u), (int)__dp2a_hi(wx, trg, 0u), (int)__dp2a_lo(wx, tbb, 0u)};
#pragma unroll
    for (int ch = 0; ch < 3; ++ch)
        px[ch] = (((b0 * (h0[ch] >> 4)) >> 16) + ((b1 * (h1[ch] >> 4)) >> 16) + (2 + (0x6400 << 2))) >> 2;   // v + 0x6400, v in [0, 255]
}
// two values (each 0x6400 + v) -> packed fp16 {v_lo, v_hi}: (1024 + v) - 1024 is exact
__device__ __forceinline__ uint32_t pack_u8_f16x2(int a, int b) {
    const uint32_t w = __byte_perm((uint32_t)a, (uint32_t)b, 0x5410);
    const __half2 r = __hsub2(*reinterpret_cast<const __half2*>(&w), __half2(__ushort_as_half(0x6400), __ushort_as_half(0x6400)));
    return *reinterpret_cast<const uint32_t*>(&r);
}

}  // namespace

__global__ void __launch_bounds__(kFThreads, Fused::kCtasPerSm)
stem12_fused_kernel(const uint8_t* __restrict__ frames, const int64_t* __restrict__ frame_offsets, const int4* __restrict__ taps,
                    const uint8_t* __restrict__ w1g, const float* __restrict__ par1g, const uint8_t* __restrict__ w2g,
                    const float* __restrict__ bias2g, uint8_t* __restrict__ planes3, int n_units, int n_big, int unit_bands,
                    int* __restrict__ work_counter) {
    using F = Fused;
    using C2 = F::C2;
    extern __shared__ __align__(128) uint8_t sm[];
#ifdef VT_FUSED_TRACE
    if (threadIdx.x == 0 && blockIdx.x < 1024) {
        long long t; unsigned smid;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        g_fused_cta[blockIdx.x][0] = t; g_fused_cta[blockIdx.x][3] = smid;
    }
#endif
    float* sPar = reinterpret_cast<float*>(sm + F::kOffPar);
    float* sB2 = sPar + kStem1TcParFloats;
    float* sXchg = reinterpret_cast<float*>(sm + F::kOffXchg);
    uint64_t* bar1 = reinterpret_cast<uint64_t*>(sm + F::kOffBar);
    uint64_t* bar2 = bar1 + 1;
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bar1 + 2);
    volatile int* s_next = reinterpret_cast<volatile int*>(bar1 + 3);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    // one-off: the zero chunks of the row slots (the whole region is cleared; data chunks are rewritten per item), weights, parameters
    for (int i = tid * 16; i < F::kIBytes; i += kFThreads * 16) *reinterpret_cast<uint4*>(sm + F::kOffI + i) = make_uint4(0, 0, 0, 0);
    for (int i = tid * 16; i < kStem1TcWBytes; i += kFThreads * 16) *reinterpret_cast<uint4*>(sm + F::kOffW1 + i) = __ldg(reinterpret_cast<const uint4*>(w1g + i));
    for (int i = tid * 16; i < C2::kWBytes; i += kFThreads * 16) *reinterpret_cast<uint4*>(sm + F::kOffW2 + i) = __ldg(reinterpret_cast<const uint4*>(w2g + i));
    if (tid < kStem1TcParFloats) sPar[tid] = __ldg(par1g + tid);
    if (tid < 16) sB2[tid] = tid < 12 ? __ldg(bias2g + tid) : 0.f;
    if (warp == 0) tmem_alloc(s_tmem, F::kTmemCols);
    if (tid == 32) {
        mbar_init(bar1, 1);
        mbar_init(bar2, 1);
        mbar_fence_init();
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tbase = __shfl_sync(0xffffffffu, *s_tmem, 0);
    const uint32_t sbase = smem_u32(sm);
    const float inv_scale = sPar[32];

    // reuse: the item is the band below the one whose rows are in the slots - its first three rows are that band's last three
    auto gather = [&](int item, bool reuse) {
        const int b = item / F::kBands, oy0 = (item % F::kBands) * F::kBR2;
        const int i0 = 4 * oy0 - 3;                                   // resized-crop row held by slot 0
        const uint8_t* __restrict__ im = frames + frame_offsets[b];
        const int4* __restrict__ tcol = taps + (size_t)b * 2 * kTapPitch + 1;    // record of resized-crop column d at [d]
        const int4* __restrict__ trow = tcol + kTapPitch;
        // ---- 1. gather: thread = pixel-pair column x, rows slot = s0 + ph + 4 j (j = 0 .. 4).  The rows go through two register sets as a
        // rolling pipeline - the loads of row j + 2 are issued as soon as row j has been consumed - so a thread always has one row of taps
        // in flight while it does the arithmetic of the other, instead of waiting out a full memory round trip per batch.
        {
            const int x = tid & 127, ph = tid >> 7;
            const int4 c0 = __ldg(tcol + 2 * x), c1 = __ldg(tcol + 2 * x + 1);
            // byte offsets are taken from the frame's word-aligned base: address = one wide multiply-add, misalignment = the offset's low bits
            const unsigned mis = (unsigned)(reinterpret_cast<uintptr_t>(im) & 3u);
            const uint32_t* __restrict__ imw = reinterpret_cast<const uint32_t*>(im - mis);
            const unsigned colx[2] = {(unsigned)c0.x + mis, (unsigned)c1.x + mis};
            const unsigned wx0 = (unsigned)c0.y, wx1 = (unsigned)c1.y;
            uint8_t* dst = sm + F::kOffI + 16 * (x + 1);
            if (reuse && ph > 0)      // slot 15 + ph moves to slot ph - 1; the same thread rewrites slot 15 + ph afterwards (program order)
                *reinterpret_cast<uint4*>(dst + (ph - 1) * kIPitch) = *reinterpret_cast<const uint4*>(dst + (15 + ph) * kIPitch);
            struct Row {
                uint32_t wd[2][6];
                unsigned sh[2][2];
                unsigned bz;
            };
            auto live = [&](int slot) { return slot < F::kIRows && i0 + slot >= 0; };     // warp-uniform
            auto load = [&](Row& r, int slot) {
                if (live(slot)) {
                    const int4 rt = __ldg(trow + i0 + slot);
                    r.bz = (unsigned)rt.z;
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const unsigned q0 = colx[j] + (unsigned)rt.x, q1 = colx[j] + (unsigned)rt.y;
                        const uint32_t* p0 = imw + (q0 >> 2);
                        const uint32_t* p1 = imw + (q1 >> 2);
                        // the pair's six bytes reach into the third word only when they start at byte 3 of the first: that load is predicated
                        // per lane (a quarter of the lanes on average - fewer sectors through L1, the front's busiest unit)
                        r.wd[j][0] = __ldg(p0); r.wd[j][1] = __ldg(p0 + 1); r.wd[j][2] = 0u;
                        r.wd[j][3] = __ldg(p1); r.wd[j][4] = __ldg(p1 + 1); r.wd[j][5] = 0u;
                        if ((q0 & 3u) == 3u) r.wd[j][2] = __ldg(p0 + 2);
                        if ((q1 & 3u) == 3u) r.wd[j][5] = __ldg(p1 + 2);
                        r.sh[j][0] = q0 << 3; r.sh[j][1] = q1 << 3;                       // the funnel shift takes the amount mod 32
                    }
                }
            };
            auto finish = [&](const Row& r, int slot) {
                if (live(slot)) {
                    int pa[3], pb[3];
                    const int b0 = (int)(r.bz & 0xffffu), b1 = (int)(r.bz >> 16);
                    bilinear_px3(r.wd[0], r.sh[0][0], r.sh[0][1], wx0, b0, b1, pa);
                    bilinear_px3(r.wd[1], r.sh[1][0], r.sh[1][1], wx1, b0, b1, pb);
                    *reinterpret_cast<uint4*>(dst + slot * kIPitch) =
                        make_uint4(pack_u8_f16x2(pa[0], pa[1]), pack_u8_f16x2(pa[2], pb[0]), pack_u8_f16x2(pb[1], pb[2]), 0u);
                } else if (slot < F::kIRows && i0 + slot == -1) {
                    *reinterpret_cast<uint4*>(dst + slot * kIPitch) = make_uint4(0u, 0u, 0u, 0u);         // the convolution's zero row above the crop
                }
            };
            static_assert(F::kIRows <= 20, "five rows per thread");
            const int s0 = (reuse ? 3 : 0) + ph;
            Row ra, rb;
            load(ra, s0);
            load(rb, s0 + 4);
            finish(ra, s0);
            load(ra, s0 + 8);
            finish(rb, s0 + 4);
            load(rb, s0 + 12);
            finish(ra, s0 + 8);
            load(ra, s0 + 16);
            finish(rb, s0 + 12);
            finish(ra, s0 + 16);
        }
    };
    // The tap records of a later item, pulled into L1 one phase ahead: the gather's first two loads (column record, row record) head a
    // dependent chain (record -> pixel addresses -> pixels) that every warp of the CTA walks at the same time.
    auto prefetch_taps = [&](int item) {
        if (tid >= 32 && tid < 72) {
            const int b = item / F::kBands, oy0 = (item % F::kBands) * F::kBR2;
            const int4* tcol = taps + (size_t)b * 2 * kTapPitch;
            const int l = tid - 32;
            const int4* p = l < 34 ? tcol + 8 * l : tcol + kTapPitch + max(4 * oy0 - 3, 0) + 8 * (l - 34);
            asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
        }
    };
    auto issue_conv1 = [&](int item) {
        const int oy0 = (item % F::kBands) * F::kBR2;
        // ---- 2. conv1: per output row r (y = 2 oy0 - 1 + r) four MMAs into columns [16 r, 16 r + 16)
        if (warp == 0) {                     // convergent; one elected lane issues
            const uint32_t idesc1 = instr_desc_f16(128, 16, false);
#pragma unroll 1
            for (int r = (oy0 == 0 ? 1 : 0); r < F::kA1Rows; ++r) {
                const uint32_t row0 = sbase + F::kOffI + (2 * r) * kIPitch;        // slot of tap ky = 0 (resized-crop row 2 y - 1)
                const uint32_t d = tbase + r * 16;
#pragma unroll
                for (int v = 0; v < 2; ++v)                                        // 0: taps kx = 1, 2 (chunk x)   1: tap kx = 0 (chunk x - 1)
#pragma unroll
                    for (int ks = 0; ks < 2; ++ks) {                               // 0: rows ky = 0 | 1   1: row ky = 2 | zero weights
                        const uint32_t a = row0 + (ks ? 2 * kIPitch : 0) + (v ? 0 : 16);
                        const uint64_t ad = smem_desc(a, ks ? 16 : kIPitch, 128);
                        const uint64_t bd = smem_desc(sbase + F::kOffW1 + (v * 2 + ks) * 512, 16 * 16, 128);
                        mma_ss_elect(d, ad, bd, idesc1, (v | ks) != 0 ? 1u : 0u);
                    }
            }
            mma_commit_elect(bar1);
        }
    };
    auto epilogue1 = [&](int item) {
        const int oy0 = (item % F::kBands) * F::kBR2;
        // ---- 3. epilogue 1: thread = (pixel x = TMEM lane, row group); -> conv2's operand image (parity planes, fp16 hi | lo)
        {
            const int q = warp & 3, g = warp >> 2;
            const int x = 32 * q + lane;
#pragma unroll 1
            for (int r = g; r < F::kA1Rows; r += 4) {
                const int y = 2 * oy0 - 1 + r;
                if (y < 0) continue;                                               // conv2's zero row above the image: cleared below
                uint32_t acc[16];
                tmem_ld16(tbase + ((uint32_t)(32 * q) << 16) + r * 16, acc);
                tc_wait_ld();
                const float* bv = sPar + 8 * ((y == 0 ? 2 : 0) + (x == 0 ? 1 : 0));
                float v[6];
#pragma unroll
                for (int c = 0; c < 6; ++c) v[c] = fmaf(__uint_as_float(acc[c]) + __uint_as_float(acc[8 + c]), inv_scale, bv[c]);
                hardswish_n<6>(v);
                uint32_t hi[4], lo[4];
#pragma unroll
                for (int j = 0; j < 3; ++j) split_pack2(v[2 * j], v[2 * j + 1], hi[j], lo[j]);
                hi[3] = 0u; lo[3] = 0u;
                const int off = ((y & 1) * 2 + (x & 1)) * C2::kChunkBytes + (((y >> 1) - (oy0 - 1)) * 64 + (x >> 1)) * 16;
                *reinterpret_cast<uint4*>(sm + F::kOffA1 + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                *reinterpret_cast<uint4*>(sm + F::kOffA1 + C2::kABytes + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
            }
            if (oy0 == 0 && tid < 256) {     // band row 0 of the odd-row planes = conv1 output row -1: zero (64 px x 16 B per plane and precision)
                const int prec = tid >> 7, plane = 2 + ((tid >> 6) & 1), px = tid & 63;
                *reinterpret_cast<uint4*>(sm + F::kOffA1 + prec * C2::kABytes + plane * C2::kChunkBytes + px * 16) = make_uint4(0u, 0u, 0u, 0u);
            }
        }
    };
    auto issue_conv2 = [&]() {
        // ---- 4. conv2 (6 -> 12): the K-step schedule of vt_stem_tc.cuh over the operand image in shared memory
        if (warp == 0) {
            const uint32_t idesc2 = instr_desc_f16(128, 16, false);
            const uint32_t abase = sbase + F::kOffA1;
#pragma unroll 1
            for (int tile = 0; tile < C2::kTiles; ++tile) {
#pragma unroll
                for (int acc = 0; acc < 2; ++acc) {                                 // 0: T_A (kx = 1, 2)   1: T_B (kx = 0, shifted by the epilogue)
                    const uint32_t d = tbase + F::kCol2 + (tile * 2 + acc) * 16;
                    const int nsteps = acc == 0 ? C2::kStepsA : C2::kStepsB;
#pragma unroll
                    for (int s2 = 0; s2 < nsteps; ++s2) {
                        int tap0, ch0, tap1, ch1; bool zero1;
                        tcs_step(kConv2Cch, acc, s2, tap0, ch0, tap1, ch1, zero1);
                        int ky, kx, p0, r0, p1, r1;
                        tcs_tap(acc, tap0, ky, kx); tcs_tap_pos(ky, kx, p0, r0);
                        tcs_tap(acc, tap1, ky, kx); tcs_tap_pos(ky, kx, p1, r1);
                        const uint32_t a0 = (p0 * kConv2Cch + ch0) * C2::kChunkBytes + (tile * C2::kRowsPerTile + r0) * kConv2Wout * 16;
                        const uint32_t a1 = (p1 * kConv2Cch + ch1) * C2::kChunkBytes + (tile * C2::kRowsPerTile + r1) * kConv2Wout * 16;
                        const uint32_t lbo = zero1 ? 16 : a1 - a0;
                        const uint64_t ah = smem_desc(abase + a0, lbo, 128);
                        const uint64_t al = smem_desc(abase + C2::kABytes + a0, lbo, 128);
                        const uint32_t boff = ((acc == 0 ? 0 : C2::kStepsA) + s2) * 2 * 16 * 16;
                        const uint64_t bh = smem_desc(sbase + F::kOffW2 + boff, 16 * 16, 128);
                        const uint64_t bl = smem_desc(sbase + F::kOffW2 + C2::kWPrecBytes + boff, 16 * 16, 128);
                        mma_ss_elect(d, ah, bh, idesc2, s2 > 0 ? 1u : 0u);
                        mma_ss_elect(d, al, bh, idesc2, 1u);
                        mma_ss_elect(d, ah, bl, idesc2, 1u);
                    }
                }
            }
            mma_commit_elect(bar2);
        }
    };
    auto epilogue2 = [&](int item) {
        const int b = item / F::kBands, oy0 = (item % F::kBands) * F::kBR2;
        // ---- 5. epilogue 2: 16 warps = (channel half) x (tile of a pair) x (TMEM lane quarter); thread = one output pixel x 8 channels
        {
            const int q = warp & 3, tsel = (warp >> 2) & 1, half = warp >> 3;
            const int rr = 32 * q + lane;                                           // row of the M tile
            const int ox = rr & 63;
            uint8_t* ob = planes3 + (size_t)b * tc_planes_bytes(kConv3Cch, kConv3Wout);
            uint32_t ra[F::kPasses][8], rb[F::kPasses][8];
#pragma unroll
            for (int pass = 0; pass < F::kPasses; ++pass) {
                const int tile = 2 * pass + tsel;
                const uint32_t ta = tbase + ((uint32_t)(32 * q) << 16) + F::kCol2 + tile * 32 + 8 * half;
                tmem_ld8(ta, ra[pass]);
                tmem_ld8(ta + 16, rb[pass]);
            }
            tc_wait_ld();
            // an image row (64 px) spans two warps: column 31's T_B crosses to column 32 through shared memory
#pragma unroll
            for (int pass = 0; pass < F::kPasses; ++pass) {
                if (lane == 31 && !(q & 1)) {
                    float* xs = sXchg + ((((pass * 2 + tsel) * 2 + half) * 2 + (q >> 1)) * 8);
#pragma unroll
                    for (int j = 0; j < 8; ++j) xs[j] = __uint_as_float(rb[pass][j]);
                }
            }
            // only the two warps that share the image row meet here (named barriers 1 .. 8, 64 threads each), not the CTA
            asm volatile("bar.sync %0, 64;" ::"r"(1 + ((half * 2 + tsel) * 2 + (q >> 1))) : "memory");
#pragma unroll
            for (int pass = 0; pass < F::kPasses; ++pass) {
                const int tile = 2 * pass + tsel;
                const int oy = oy0 + tile * 2 + (rr >> 6);
                const float* xs = sXchg + ((((pass * 2 + tsel) * 2 + half) * 2 + (q >> 1)) * 8);
                float v[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    float tb = __shfl_up_sync(0xffffffffu, __uint_as_float(rb[pass][j]), 1);      // T_B[oy][ox - 1]
                    if (lane == 0 && (q & 1)) tb = xs[j];
                    if (ox == 0) tb = 0.f;
                    v[j] = __uint_as_float(ra[pass][j]) + tb + sB2[8 * half + j];
                }
                hardswish_n<8>(v);
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    if (8 * half + j >= 12) v[j] = 0.f;                             // padding channels stay exactly zero
                uint32_t hi[4], lo[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) split_pack2(v[2 * j], v[2 * j + 1], hi[j], lo[j]);
                *reinterpret_cast<uint4*>(ob + tc_planes_offset(0, oy, ox, half, kConv3Cch, kConv3Wout)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                *reinterpret_cast<uint4*>(ob + tc_planes_offset(1, oy, ox, half, kConv3Cch, kConv3Wout)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
            }
        }
    };
    // Software pipeline over the CTA's items: the tensor pipe's latency never sits on the critical path - conv1's MMAs of item i run under
    // epilogue 2 of item i - 1, conv2's MMAs of item i under the gather of item i + 1.
    //   every thread:  G(i) | S | [conv1(i) issued] E2(i-1) wait1 E1(i) | S | [conv2(i) issued] G(i+1) | S | ...
    // Hazards (program order per thread + the two barriers): conv2's accumulators of i - 1 are read (E2) before the barrier that precedes
    // conv2(i); conv1's accumulators are read (E1) before the barrier that precedes conv1(i + 1); the row slots are rewritten (G(i + 1)) after
    // every thread has waited for conv1(i); the plane image is rewritten (E1(i + 1)) after every thread has waited for conv2(i).
    // Work distribution: a unit = consecutive bands of one track (the row reuse above works inside a unit): the first n_big units have
    // unit_bands bands, the remaining ones a single band - the queue ends in small pieces, so that the last CTA finishes one band, not one
    // unit, after the others.  CTAs take their first unit by index and every further one from a global counter (crop_taps_kernel resets
    // it to gridDim.x): items differ in cost with the crop's scale and position, and a static round-robin leaves the slowest CTA 10 %
    // behind the mean.  The successor of the NEXT item is fetched by one thread during the gather phase, so the atomic's round trip is
    // never waited for.
    int unit_last = -1;                              // last item of the unit the newest item belongs to (meaningful in thread 480)
    auto unit_first = [&](int u) -> int {
        if (u >= n_units) return -1;
        if (u < n_big) { unit_last = (u + 1) * unit_bands - 1; return u * unit_bands; }
        unit_last = n_big * unit_bands + (u - n_big);
        return unit_last;
    };
    auto successor = [&](int x) -> int {
        if (x < 0) return -1;
        if (x < unit_last) return x + 1;
        return unit_first(atomicAdd(work_counter, 1));
    };
    int it = 0, prev = -1;
    int item = unit_first((int)blockIdx.x);
#ifdef VT_FUSED_TRACE
    if (threadIdx.x == 0 && blockIdx.x < 1024) { long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); g_fused_cta[blockIdx.x][1] = t; }
#endif
    if (tid == 480) s_next[0] = successor(item);
    if (item >= 0) gather(item, false);
#pragma unroll 1
    for (; item >= 0; ++it) {
        FUSED_TRACE();
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
        FUSED_TRACE();
        const int nxt = s_next[it & 1];
        issue_conv1(item);
        if (nxt >= 0) prefetch_taps(nxt);
        if (prev >= 0) {
            mbar_wait(bar2, (it - 1) & 1);
            tc_fence_after();
            FUSED_TRACE();
            epilogue2(prev);
        } else {
            FUSED_TRACE();
        }
        FUSED_TRACE();
        mbar_wait(bar1, it & 1);
        tc_fence_after();
        FUSED_TRACE();
        epilogue1(item);
        FUSED_TRACE();
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
        FUSED_TRACE();
        issue_conv2();
        if (tid == 480) s_next[(it + 1) & 1] = successor(nxt);
        if (nxt >= 0) gather(nxt, nxt == item + 1 && nxt % F::kBands != 0);
        FUSED_TRACE();
        prev = item;
        item = nxt;
    }
    if (prev >= 0) {
        mbar_wait(bar2, (it - 1) & 1);
        tc_fence_after();
        epilogue2(prev);
    }
#ifdef VT_FUSED_TRACE
    if (threadIdx.x == 0 && blockIdx.x < 1024) { long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); g_fused_cta[blockIdx.x][2] = t; }
#endif
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tbase, F::kTmemCols);
}

// Search crop of n tracks straight from the raw frames -> conv3's operand image (planes3): tap tables + the fused kernel.
// tap_tables: crop_taps_bytes(n) bytes; the fused kernel's work counter sits behind the n tables.
int launch_crop_stem12_fused(const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw, const double* boxes,
                             const int32_t* slots, double factor, int n, const ModelW& w, int32_t* out_status, void* tap_tables, uint8_t* planes3, cudaStream_t st) {
    if (n <= 0) return 0;
    using F = Fused;
    auto kern = stem12_fused_kernel;
    static int grid_caps[kMaxDevices] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return -1;
    if (grid_caps[dev] == 0) {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, F::kSmemBytes) != cudaSuccess) return -1;
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1;
        grid_caps[dev] = sms * resident_ctas_per_sm(kern, kFThreads, F::kSmemBytes, F::kTmemCols, dev);
    }
    // few tracks (the batch-1 latency path): single bands, so that a track spreads over kBands CTAs instead of kBands / kUnitBands
    const int unit_bands = (long long)n * (F::kBands / F::kUnitBands) >= 2LL * grid_caps[dev] ? F::kUnitBands : 1;
    const long long bands = (long long)n * F::kBands;
    if (bands > 0x7fffffffLL) return -1;
    // the last sixteenth of the bands (at least two rounds of the grid) is handed out band by band
    long long small = bands / 16;
    if (small < 2LL * grid_caps[dev]) small = 2LL * grid_caps[dev];
    if (small > bands || unit_bands == 1) small = bands;
    const int n_big = (int)((bands - small) / unit_bands);
    const int n_units = n_big + (int)(bands - (long long)n_big * unit_bands);
    const int grid = n_units < grid_caps[dev] ? n_units : grid_caps[dev];
    int4* taps = reinterpret_cast<int4*>(tap_tables);
    int* work_counter = reinterpret_cast<int*>(taps + (size_t)n * 2 * kTapPitch);
    crop_taps_kernel<kSx><<<n, 288, 0, st>>>(frame_hw, boxes, slots, factor, taps, out_status, work_counter, grid, nullptr);
    if (cudaGetLastError() != cudaSuccess) return -1;
    kern<<<grid, kFThreads, F::kSmemBytes, st>>>(frames, frame_offsets, taps, w.stem1_tc_w, w.stem1_tc_par, w.stem_tc_w[0], w.stem_tc_b[0],
                                                 planes3, n_units, n_big, unit_bands, work_counter);
    return cudaGetLastError() == cudaSuccess ? 2 : -1;
}

// Host side: conv1's folded weights [ci][ky][kx][co] (BatchNorm folded, fp32) + bias -> the kernel's operands.
//   blob [variant 2][K step 2] x 512 bytes: B[n][k] as [chunk 2][n 16][8] fp16; n = co (hi) | 8 + co (lo); chunk = resized-crop row
//   (K step 0: ky = 0 | ky = 1; K step 1: ky = 2 | zeros); k = 3 * pixel + ci over the chunk's two pixels.
//   variant 0: pixel 0 -> kx = 1, pixel 1 -> kx = 2;  variant 1 (A operand one chunk earlier): pixel 1 -> kx = 0.
//   par: bias[4][8] (variant = 2 * (y == 0) + (x == 0): taps in the convolution's zero padding left out), par[32] = 2^-s.
void stem1_tc_pack(const float* wf, const float* bf, uint8_t* blob, float* par) {
    const double mean[3] = {0.485, 0.456, 0.406}, stdv[3] = {0.229, 0.224, 0.225};
    auto W = [&](int ci, int ky, int kx, int co) { return (double)wf[(((size_t)ci * 3 + ky) * 3 + kx) * 6 + co]; };
    double maxabs = 0.0;
    for (int ci = 0; ci < 3; ++ci)
        for (int t = 0; t < 9; ++t)
            for (int co = 0; co < 6; ++co) {
                const double v = fabs(W(ci, t / 3, t % 3, co) / (255.0 * stdv[ci]));
                if (v > maxabs) maxabs = v;
            }
    int e = 0;
    if (maxabs > 0.0) frexp(maxabs, &e);                 // maxabs = m * 2^e, m in [0.5, 1)
    const int s = 14 - e;                                // scaled maximum in [2^13, 2^14): hi and lo are both normal fp16 numbers
    const double scale = ldexp(1.0, s);
    memset(blob, 0, kStem1TcWBytes);
    for (int v = 0; v < 2; ++v)
        for (int ks = 0; ks < 2; ++ks)
            for (int c = 0; c < 2; ++c) {
                const int ky = ks == 0 ? c : (c == 0 ? 2 : -1);
                if (ky < 0) continue;
                for (int co = 0; co < 6; ++co)
                    for (int k = 0; k < 6; ++k) {
                        const int pix = k / 3, ci = k % 3;
                        int kx;
                        if (v == 0) kx = 1 + pix; else { if (pix == 0) continue; kx = 0; }
                        const float val = (float)(W(ci, ky, kx, co) / (255.0 * stdv[ci]) * scale);
                        uint16_t h, l;
                        split_f16(val, &h, &l);
                        uint8_t* base = blob + (v * 2 + ks) * 512 + c * 256 + k * 2;
                        memcpy(base + co * 16, &h, 2);
                        memcpy(base + (8 + co) * 16, &l, 2);
                    }
            }
    for (int var = 0; var < 4; ++var)
        for (int co = 0; co < 8; ++co) {
            double acc = co < 6 ? (double)bf[co] : 0.0;
            for (int ci = 0; ci < 3 && co < 6; ++ci)
                for (int ky = 0; ky < 3; ++ky)
                    for (int kx = 0; kx < 3; ++kx) {
                        if ((var & 2) && ky == 0) continue;          // top row: the taps above the crop are zero padding
                        if ((var & 1) && kx == 0) continue;          // left column
                        acc -= W(ci, ky, kx, co) * mean[ci] / stdv[ci];
                    }
            par[var * 8 + co] = (float)acc;
        }
    par[32] = (float)ldexp(1.0, -s);
    for (int i = 33; i < kStem1TcParFloats; ++i) par[i] = 0.f;
}

#ifdef VT_FUSED_TRACE
extern "C" int vt_fused_trace_read(long long* host, int* n) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(n, g_fused_trace_n, sizeof(int));
    cudaMemcpyFromSymbol(host, g_fused_trace, sizeof(long long) * 8192);
    cudaMemcpyFromSymbol(host + 8192, g_fused_cta, sizeof(long long) * 4096);
    int zero = 0;
    cudaMemcpyToSymbol(g_fused_trace_n, &zero, sizeof zero);
    return 0;
}
#endif

}  // namespace vt

// Development aid (not part of the ABI): what the occupancy API answers for the fused kernel on the current device.
extern "C" int vt_debug_fused_occupancy(int* out) {
    using F = vt::Fused;
    auto kern = vt::stem12_fused_kernel;
    int a = -1, b = -1, c = -1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&a, kern, vt::kFThreads, F::kSmemBytes);
    cudaError_t e1 = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, F::kSmemBytes);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, kern, vt::kFThreads, F::kSmemBytes);
    cudaError_t e2 = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&c, kern, vt::kFThreads, F::kSmemBytes);
    cudaFuncAttributes fa;
    cudaFuncGetAttributes(&fa, kern);
    out[0] = a; out[1] = b; out[2] = c; out[3] = (int)e1; out[4] = (int)e2; out[5] = fa.numRegs; out[6] = (int)fa.sharedSizeBytes;
    out[7] = F::kSmemBytes; out[8] = fa.maxDynamicSharedSizeBytes; out[9] = fa.preferredShmemCarveout;
    return 0;
}
