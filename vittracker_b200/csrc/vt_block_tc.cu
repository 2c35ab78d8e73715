// K3 (tensor-core variant): the three ViT blocks on tcgen05 tensor cores with TMEM accumulators.
//   x = x + proj(softmax((q*48^-0.5) k^T) v),  [q;k;v] = qkv(LN(x));   x = x + fc2(GELU_erf(fc1(LN(x))))
// (lib/models/vit_dist/vit_dist.py:84,88-89; timm Block restated at tracking/onnxexport.py:126-225)
//
// One persistent CTA per SM walks over tracks.  A track's 320 tokens form three M=128 row tiles
// (the third is half padding).  Every contraction is a chain of tcgen05.mma (kind::f16, M=128,
// fp32 accumulate in TMEM) whose A operand is read FROM TMEM and whose B operand (weights, K, V) is
// read from shared memory through no-swizzle UMMA descriptors:
//   - the epilogue threads read an accumulator row with tcgen05.ld (TMEM lane = token row), apply
//     bias / LayerNorm / softmax / GELU in fp32, split the result into fp16 hi + lo and write it back
//     to TMEM with tcgen05.st as the A operand of the next contraction (P overwrites S in place);
//   - every product is evaluated as hi*hi + lo*hi + hi*lo (three MMAs per K step into one
//     accumulator), which keeps ~22 mantissa bits on the operands: single-pass fp16/bf16/TF32
//     inputs flip the Hann-weighted arg-max the tracker depends on (SURVEY 7.2);
//   - softmax row statistics are thread-local (one row per TMEM lane); the 48 / 192 / 320 columns of
//     a row are shared by kNS warps (column groups) that exchange partial sums through smem.
// Warp roles: warps 0 .. 4 kNS - 1 = epilogue (lane quarter = warp % 4, column group = warp / 4),
// the last warp = control (bulk weight loads + single-thread MMA issue).  Control and epilogue ping-pong
// through two mbarriers (`go`: operands ready, one arrival per epilogue warp; `done`: tcgen05.commit).
//
// Algorithmic work per track: 112.07 MFLOP (SURVEY 8d); issued MMA work is 3x that (split) x 1.2
// (padding of the third tile).
#include <vector>

#include "vt_internal.h"
#include "vt_tc.cuh"

namespace vt {

using namespace tc;

// Optional per-step cycle trace of CTA 0 (development aid): -DVT_TC_TRACE, read back with vt_tc_trace_read().
#ifdef VT_TC_TRACE
__device__ long long g_tc_trace[2][4096];
__device__ int g_tc_trace_n[2];
#define TC_TRACE(side)                                                                      \
    do {                                                                                    \
        if (blockIdx.x == 0) { int k__ = g_tc_trace_n[side]; if (k__ < 4096) { g_tc_trace[side][k__] = clock64(); g_tc_trace_n[side] = k__ + 1; } } \
    } while (0)
#else
#define TC_TRACE(side) do {} while (0)
#endif

namespace {

// Epilogue warps: lane quarter = warp % 4 (TMEM lanes 32q .. 32q+31 = token rows), column group = warp / 4.
// kNS column groups share the columns of a row; more groups = more warps in flight to hide TMEM / MUFU latency.
constexpr int kNS = 6;
// Split terms of the score contraction S = q k^T:  3 = hi*hi + lo*hi + hi*lo (as every other contraction), 2 = without hi*lo (K at fp16),
// 1 = hi*hi only (single-pass fp16).  The per-contraction precision budget (tools/precision_budget.py, profiles/r02_precision_budget*.json:
// oracle-side emulation of this kernel's operand rounding on 3 x 10^4 frames, two weight sets) shows the scores are the one contraction whose
// low-order terms do not reach the arg-max: S feeds a softmax (a perturbation of S scales P by 1 + dS, and the row normalisation removes
// its common part), |dS| ~ 2^-12 |q||k| / sqrt(48) ~ 1e-5 here.  Dropping either term of q k^T: 0 flips, score-map error 1e-6 (the noise
// floor of the three-term scheme is 8e-7); every other contraction flips the arg-max when it loses a term (errors 2e-5 .. 1.5e-4).
// That budget is measured on the specified workload (random-init weights: |S| < 1).  A trained checkpoint has sharper attention - larger
// |q||k| and the same RELATIVE operand error - so the kernel is compiled in both forms and the handle chooses: VT_BLOCKS_TCGEN05 (single
// pass, the default) or VT_BLOCKS_TCGEN05_3TERM (blocks_impl = "tcgen05_3term": three terms everywhere, ~9 % slower blocks).
constexpr int kEpiWarps = 4 * kNS;
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kTcThreads = kEpiThreads + 32;   // + the control warp
constexpr int kCW = kC / kNS;                  // residual / LayerNorm columns per thread (8)
constexpr int kQW = 3 * kC / kNS;              // QKV output columns per thread (24)
constexpr int kHW = kHid / kNS;                // hidden columns per thread (32)

// ---- TMEM columns --------------------------------------------------------------------------------
constexpr uint32_t kColBig = 0;        // [0,320): QKV out (2 buffers of 144 at 0 / 160), S -> P, fc1 out -> GELU operand
constexpr uint32_t kColOut = 320;      // [320,368): free during attention (O' accumulates in the q slots); part of H_B in the MLP phase
constexpr uint32_t kColOpa = 368;      // [368,512): three 48-column A-operand slots (hi 24 | lo 24), one per row tile
// MLP phase (the attention regions are dead by then): two fc1-output / GELU-operand buffers and two fc2 outputs, so
// that the GELU of one row tile overlaps the MMAs of the others.  H_B / Y_A / Y_B alias the A-operand slots; the
// control program orders every aliasing write after the MMA that last read the slot.
constexpr uint32_t kColHA = 0, kColHB = 192;       // 192 columns each
constexpr uint32_t kColYA = 384, kColYB = 432;     // 48 columns each

// ---- one block's weight blobs (block_tc_pack), byte offsets: fp16 hi | lo halves, UMMA no-swizzle K-major [k/8][n][8] ------------
//   wa: [Wq; Wk; Wproj Wv] (N 144, K 48) hi | lo           wb: W1 (N 192, K 48) hi | lo, then W2 (N 48, K 192) hi | lo
constexpr int kWaLo = 3 * kC * kC * 2;                    // 13824
constexpr int kWbW1Lo = kHid * kC * 2;                    // 18432
constexpr int kWbW2Hi = 2 * kWbW1Lo;                      // 36864 = W1 hi | lo
constexpr int kWbW2Lo = kWbW2Hi + kC * kHid * 2;          // 55296
static_assert(kTcWaBytes == 2 * kWaLo && kTcWbBytes == kWbW2Lo + kC * kHid * 2, "block weight blobs");

// ---- shared memory (bytes) -------------------------------------------------------------------------
constexpr int kSmWa = 0;                                  // Wqkv hi|lo, Wproj hi|lo (bulk copied per block)
constexpr int kSmX = kSmWa + kTcWaBytes;                  // attention: K hi|lo, V hi|lo ; MLP: W1 hi|lo, W2 hi|lo
constexpr int kKBytes = kN * kC * 2;                      // 30720 per precision
constexpr int kSmKhi = kSmX, kSmKlo = kSmX + kKBytes, kSmVhi = kSmX + 2 * kKBytes, kSmVlo = kSmX + 3 * kKBytes;
constexpr int kSmW2hi = kSmX, kSmW2lo = kSmX + (kWbW2Lo - kWbW2Hi);   // W2 hi|lo overlays K (streamed in once attention is over)
constexpr int kSmW1 = kSmX + 4 * kKBytes;                 // W1 hi|lo in its own region: prefetched during attention
constexpr int kSmW1hi = kSmW1, kSmW1lo = kSmW1 + kWbW1Lo;
constexpr int kSmPar = kSmW1 + kWbW2Hi;                   // fp32 parameters of all blocks
constexpr int kSmRed = kSmPar + kDepth * kTcParFloats * 4;   // 6 arrays x kNS column groups x 128 rows fp32
constexpr int kSmBar = kSmRed + 6 * kNS * 128 * 4;        // mbarriers
constexpr int kSmTmem = kSmBar + 20 * 8;
static_assert(kSmTmem + 16 <= 227 * 1024, "shared memory");
constexpr int kTcSmemBytes = kSmTmem + 16;
static_assert(kTcWbBytes - kWbW2Hi <= 4 * kKBytes, "W2 overlays the K/V region");
static_assert(kSmBar % 8 == 0 && kSmX % 128 == 0, "alignment");

// parameter offsets inside one block's fp32 parameter vector
constexpr int kPLn1g = 0, kPLn1b = 48, kPBqkv = 96, kPBproj = 240, kPLn2g = 288, kPLn2b = 336, kPBfc1 = 384, kPBfc2 = 576;
static_assert(kPBfc2 + kC == kTcParFloats, "parameter vector");

__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory"); }

struct Epi {
    uint32_t tbase;        // TMEM base address
    uint32_t lane_addr;    // (32 * quarter) << 16
    int q, s, lane, row;   // lane quarter, column group, lane, row inside the tile (32q + lane)
    float* red;            // [4][kNS][128]
    uint64_t *mb_go, *mb_done;
    uint32_t done_ph;

    __device__ __forceinline__ bool active(int t) const { return !(t == 2 && q >= 2); }    // rows 320..383 are padding
    __device__ __forceinline__ uint32_t taddr(uint32_t col) const { return tbase + lane_addr + col; }

    // operands written (TMEM and/or smem): publish to the control thread
    __device__ __forceinline__ void signal(uint64_t* bar, bool wrote_smem) {
        tc_wait_st();
        if (wrote_smem) fence_async_smem();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar);
    }
    __device__ __forceinline__ void signal_go(bool wrote_smem) { signal(mb_go, wrote_smem); }
    __device__ __forceinline__ void wait_bar(uint64_t* bar, uint32_t& ph) {
        if (threadIdx.x == 0) TC_TRACE(1);
        mbar_wait(bar, ph);
        ph ^= 1;
        tc_fence_after();
        if (threadIdx.x == 0) TC_TRACE(1);
    }
    __device__ __forceinline__ void wait_done() {
        if (threadIdx.x == 0) TC_TRACE(1);
        mbar_wait(mb_done, done_ph);
        done_ph ^= 1;
        tc_fence_after();
        if (threadIdx.x == 0) TC_TRACE(1);
    }

    // sum over the 48 columns of a row (kNS column groups) of a per-thread partial; `arr` selects the scratch array
    __device__ __forceinline__ float row_sum(float partial, int arr) {
        float* r = red + arr * (kNS * 128);
        r[s * 128 + row] = partial;
        epi_bar();
        float t = r[row];
#pragma unroll
        for (int g = 1; g < kNS; ++g) t += r[g * 128 + row];
        return t;
    }

    // LayerNorm of a 48-wide row held as kNS x kCW values
    __device__ __forceinline__ void ln(const float (&v)[kCW], const float* g, const float* b, float (&y)[kCW]) {
        float sum = 0.f;
#pragma unroll
        for (int i = 0; i < kCW; ++i) sum += v[i];
        const float mean = row_sum(sum, 0) * (1.f / 48.f);
        float var = 0.f;
#pragma unroll
        for (int i = 0; i < kCW; ++i) { const float d = v[i] - mean; var = fmaf(d, d, var); }
        const float rstd = rsqrtf(row_sum(var, 1) * (1.f / 48.f) + kLnEps);
#pragma unroll
        for (int i = 0; i < kCW; ++i) y[i] = (v[i] - mean) * rstd * g[kCW * s + i] + b[kCW * s + i];
    }

    // write this thread's K-elements [kCW s, kCW s + kCW) of row `row` into A-operand slot t (hi cols, then lo cols at +24)
    __device__ __forceinline__ void store_opa(int t, const float (&y)[kCW]) {
        uint32_t hi[kCW / 2], lo[kCW / 2];
#pragma unroll
        for (int j = 0; j < kCW / 2; ++j) split_pack2(y[2 * j], y[2 * j + 1], hi[j], lo[j]);
        tmem_st<kCW / 2>(taddr(kColOpa + 48 * t + (kCW / 2) * s), hi);
        tmem_st<kCW / 2>(taddr(kColOpa + 48 * t + 24 + (kCW / 2) * s), lo);
    }
};

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// sm_100's packed fp32 arithmetic (fma / mul / add .f32x2, SASS FFMA2 / FMUL2 / FADD2): two independent IEEE operations per issue slot.
__device__ __forceinline__ uint64_t f2pack(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void f2unpack(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t f2bcast(float c) { return f2pack(c, c); }
__device__ __forceinline__ uint64_t f2fma(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ uint64_t f2mul(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uint64_t f2add(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
// GELU(v) = 0.5 v (1 + erf(v / sqrt 2)) with erf from Abramowitz & Stegun 7.1.26 (|abs err| <= 1.5e-7): with x = |v| / sqrt 2,
// t = 1 / (1 + p x), erf(x) = 1 - P(t) t exp(-x^2), both signs of v collapse to
//     GELU(v) = max(v, 0) - |v| (P(t) / 2) t exp(-v^2 / 2)
// - no cancellation against 1, one reciprocal, one exponential, and the 1/2, 1/sqrt 2 and log2(e) folded into constants
// (erff's two branch-selected polynomials were ~30 % of this kernel's CUDA-core instructions).
// Two GELUs at once in packed arithmetic: 19 issue slots per pair instead of 28 for two scalar evaluations.  The polynomial carries the
// minus sign of the last product in its coefficients (-P(t) / 2), which is exact.
__device__ __forceinline__ void gelu_erf2(uint64_t v, float& h0, float& h1) {
    float v0, v1;
    f2unpack(v, v0, v1);
    const uint64_t av = f2pack(fabsf(v0), fabsf(v1));
    float d0, d1;
    f2unpack(f2fma(f2bcast(0.3275911f * 0.70710678118654752f), av, f2bcast(1.f)), d0, d1);
    const uint64_t t = f2pack(rcp_approx(d0), rcp_approx(d1));
    uint64_t p = f2fma(f2bcast(-0.5f * 1.061405429f), t, f2bcast(0.5f * 1.453152027f));       // -P(t) / 2
    p = f2fma(p, t, f2bcast(-0.5f * 1.421413741f));
    p = f2fma(p, t, f2bcast(0.5f * 0.284496736f));
    p = f2fma(p, t, f2bcast(-0.5f * 0.254829592f));
    float w0, w1;
    f2unpack(f2mul(v, f2mul(f2bcast(-0.5f * 1.4426950408889634f), v)), w0, w1);
    const uint64_t e = f2pack(ex2_approx(w0), ex2_approx(w1));
    f2unpack(f2fma(f2mul(av, f2mul(p, t)), e, f2pack(fmaxf(v0, 0.f), fmaxf(v1, 0.f))), h0, h1);
}

}  // namespace

template <int kScoresTerms>
__global__ void __launch_bounds__(kTcThreads, 1)
blocks_tc_kernel(const float* __restrict__ tok_z, int z_stride_rows, const float* __restrict__ tok_x, int x_stride_rows,
                 float* __restrict__ out, int n, ModelW w, float* __restrict__ taps, size_t tap_stride) {
    extern __shared__ __align__(128) uint8_t smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    float* s_par = reinterpret_cast<float*>(smem + kSmPar);
    float* s_red = reinterpret_cast<float*>(smem + kSmRed);
    uint64_t* mb_go = reinterpret_cast<uint64_t*>(smem + kSmBar);
    uint64_t* mb_done = mb_go + 1;
    uint64_t* mb_wa = mb_go + 2;
    uint64_t* mb_wb = mb_go + 3;
    uint64_t* mb_h = mb_go + 4;        // [2] fc1 output ready in H_A / H_B          (tcgen05.commit)
    uint64_t* mb_y = mb_go + 6;        // [2] fc2 output ready in Y_A / Y_B          (tcgen05.commit)
    uint64_t* mb_g = mb_go + 8;        // [2] GELU operand written in H_A / H_B      (one arrival per epilogue warp)
    uint64_t* mb_yfree = mb_go + 10;   // Y_A has been read, may be overwritten      (one arrival per epilogue warp)
    uint64_t* mb_w1 = mb_go + 11;      // W1 landed in shared memory
    uint64_t* mb_qd = mb_go + 12;      // [2] QKV output of a tile ready in buffer 0 / 1     (tcgen05.commit)
    uint64_t* mb_pa = mb_go + 15;      // first part of P (keys 0..159) written            (one arrival per epilogue warp)
    uint64_t* mb_qf = mb_go + 14;      // QKV buffer 0 has been read (tile 0's epilogue)     (one arrival per epilogue warp)
    // LayerNorm-1 operand of tile t written: one barrier PER TILE.  The three hand-overs follow each other without the epilogue warps
    // ever waiting for the control warp in between, so on a shared barrier two phases can complete before a late control warp (cold
    // weight load, preempted issue) has looked at the first - and a parity wait cannot tell "two phases ago" from "not yet" (deadlock
    // seen under ncu's cache-flushed launches).  Every other barrier's next completion depends on its waiters having seen the last one.
    uint64_t* mb_l1 = mb_go + 16;      // [3]                                              (one arrival per epilogue warp)
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + kSmTmem);

    if (warp == kEpiWarps) tmem_alloc(s_tmem, 512);
    if (tid == 0) {
        mbar_init(mb_go, kEpiWarps);
        mbar_init(mb_done, 1);
        mbar_init(mb_wa, 1);
        mbar_init(mb_wb, 1);
        mbar_init(mb_w1, 1);
        mbar_init(mb_qd, 1); mbar_init(mb_qd + 1, 1);
        mbar_init(mb_qf, kEpiWarps);
        mbar_init(mb_pa, kEpiWarps);
        for (int t = 0; t < 3; ++t) mbar_init(mb_l1 + t, kEpiWarps);
        mbar_init(mb_h, 1); mbar_init(mb_h + 1, 1);
        mbar_init(mb_y, 1); mbar_init(mb_y + 1, 1);
        mbar_init(mb_g, kEpiWarps); mbar_init(mb_g + 1, kEpiWarps);
        mbar_init(mb_yfree, kEpiWarps);
        mbar_fence_init();
    }
    for (int i = tid; i < kDepth * kTcParFloats; i += kTcThreads) s_par[i] = __ldg(w.tc[i / kTcParFloats].par + i % kTcParFloats);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tbase = __shfl_sync(0xffffffffu, *s_tmem, 0);       // provably warp-uniform
    const uint32_t sbase = smem_u32(smem);

    if (warp == kEpiWarps) {
        // =========================== control: weight loads + MMA issue (one thread) ===========================
        {   // the whole warp runs this program convergently; MMA / commit / bulk copy are done by one elected lane
            uint32_t go_ph = 0, wa_ph = 0, wb_ph = 0, w1_ph = 0;
            const uint32_t id48 = instr_desc_f16(128, 48, false), id48mn = instr_desc_f16(128, 48, true);
            const uint32_t id144 = instr_desc_f16(128, 144, false), id160 = instr_desc_f16(128, 160, false);
            const uint32_t id192 = instr_desc_f16(128, 192, false);
            auto wait_go = [&]() { TC_TRACE(0); mbar_wait(mb_go, go_ph); go_ph ^= 1; tc_fence_after(); TC_TRACE(0); };
            auto load_wa = [&](int blk) { bulk_g2s_elect(smem + kSmWa, w.tc[blk].wa, kTcWaBytes, mb_wa); };
            auto load_w1 = [&](int blk) { bulk_g2s_elect(smem + kSmW1, w.tc[blk].wb, kWbW2Hi, mb_w1); };
            auto load_w2 = [&](int blk) { bulk_g2s_elect(smem + kSmX, w.tc[blk].wb + kWbW2Hi, kTcWbBytes - kWbW2Hi, mb_wb); };
            // D[d_col] = A(opa slot t, K = 48) x B^T, B K-major [k/8][N][8] at byte offsets b_hi / b_lo
            auto gemm_k48 = [&](int t, uint32_t d_col, uint32_t b_hi, uint32_t b_lo, int N, uint32_t idesc) {
                const uint32_t a = tbase + kColOpa + 48 * t;
#pragma unroll
                for (int ks = 0; ks < 3; ++ks) {
                    const uint64_t bh = smem_desc(sbase + b_hi + ks * 2 * N * 16, N * 16, 128);
                    const uint64_t bl = smem_desc(sbase + b_lo + ks * 2 * N * 16, N * 16, 128);
                    mma_ts_elect(tbase + d_col, a + 8 * ks, bh, idesc, ks > 0);           // hi * hi
                    mma_ts_elect(tbase + d_col, a + 24 + 8 * ks, bh, idesc, true);        // lo * hi
                    mma_ts_elect(tbase + d_col, a + 8 * ks, bl, idesc, true);             // hi * lo
                }
            };
            auto qkv = [&](int t, uint32_t d_col) { gemm_k48(t, d_col, kSmWa, kSmWa + kWaLo, 144, id144); };
            auto fc1 = [&](int t, uint32_t h_col) { gemm_k48(t, h_col, kSmW1hi, kSmW1lo, 192, id192); };
            // S = q k^T over 320 keys as two N = 160 halves; K operand K-major [k/8][320][8]
            auto scores_half = [&](int t, int half) {
                const uint32_t a = tbase + kColOpa + 48 * t;
                const uint32_t d = tbase + kColBig + 160 * half;
#pragma unroll
                for (int ks = 0; ks < 3; ++ks) {
                    const uint32_t off = ks * 2 * (kN * 16) + half * 160 * 16;
                    const uint64_t bh = smem_desc(sbase + kSmKhi + off, kN * 16, 128);
                    const uint64_t bl = smem_desc(sbase + kSmKlo + off, kN * 16, 128);
                    mma_ts_elect(d, a + 8 * ks, bh, id160, ks > 0);                               // q_hi k_hi
                    if (kScoresTerms >= 2) mma_ts_elect(d, a + 24 + 8 * ks, bh, id160, true);     // q_lo k_hi
                    if (kScoresTerms >= 3) mma_ts_elect(d, a + 8 * ks, bl, id160, true);          // q_hi k_lo
                }
            };
            // O' = P V' accumulated in the tile's (now dead) q slot: P in TMEM (16-key group g: hi cols 16g.., lo cols 16g+8..),
            // V' = V Wproj^T MN-major [f/8][key/8][key%8][f%8]; key groups [g0, g1)
            auto pv = [&](int t, int g0, int g1) {
                const uint32_t d = tbase + kColOpa + 48 * t;
#pragma unroll 5
                for (int g = g0; g < g1; ++g) {
                    const uint32_t a = tbase + kColBig + 16 * g;
                    const uint64_t bh = smem_desc(sbase + kSmVhi + g * 256, 128, (kN / 8) * 128);
                    const uint64_t bl = smem_desc(sbase + kSmVlo + g * 256, 128, (kN / 8) * 128);
                    mma_ts_elect(d, a, bh, id48mn, g > 0);
                    mma_ts_elect(d, a + 8, bh, id48mn, true);
                    mma_ts_elect(d, a, bl, id48mn, true);
                }
            };
            // y = gelu(h) W2^T: operand in TMEM (16-wide group g: hi 16g.., lo 16g+8..), W2 K-major [k/8][48][8], K = 192
            auto fc2 = [&](uint32_t h_col, uint32_t y_col) {
#pragma unroll 4
                for (int g = 0; g < kHid / 16; ++g) {
                    const uint32_t a = tbase + h_col + 16 * g;
                    const uint64_t bh = smem_desc(sbase + kSmW2hi + g * 2 * 48 * 16, 48 * 16, 128);
                    const uint64_t bl = smem_desc(sbase + kSmW2lo + g * 2 * 48 * 16, 48 * 16, 128);
                    mma_ts_elect(tbase + y_col, a, bh, id48, g > 0);
                    mma_ts_elect(tbase + y_col, a + 8, bh, id48, true);
                    mma_ts_elect(tbase + y_col, a, bl, id48, true);
                }
            };
            uint32_t h_ph[2] = {0, 0}, y_ph[2] = {0, 0}, g_ph[2] = {0, 0}, yfree_ph = 0, qf_ph = 0, pa_ph = 0, l1_ph[3] = {0, 0, 0};
            auto wait_on = [&](uint64_t* bar, uint32_t& ph) { TC_TRACE(0); mbar_wait(bar, ph); ph ^= 1; tc_fence_after(); TC_TRACE(0); };
            bool first = true;
            for (int trk = blockIdx.x; trk < n; trk += gridDim.x) {
                const bool last_track = trk + (int)gridDim.x >= n;
                for (int blk = 0; blk < kDepth; ++blk) {
                    if (first) { load_wa(0); load_w1(0); first = false; }
                    // QKV per tile, overlapped with the LayerNorms / epilogues of the other tiles (two output buffers)
                    wait_on(mb_l1, l1_ph[0]);                                    // 1a: LN1 operand of tile 0
                    mbar_wait(mb_wa, wa_ph); wa_ph ^= 1;
                    qkv(0, kColBig); mma_commit_elect(mb_qd);
                    wait_on(mb_l1 + 1, l1_ph[1]); qkv(1, kColBig + 160); mma_commit_elect(mb_qd + 1);     // 1b
                    wait_on(mb_l1 + 2, l1_ph[2]);                                // 1c: LN1 operand of tile 2
                    wait_on(mb_qf, qf_ph);                                       // 2: tile 0's QKV output has been read
                    qkv(2, kColBig); mma_commit_elect(mb_qd);
                    wait_go(); scores_half(0, 0); scores_half(0, 1); mma_commit_elect(mb_done);     // 3: K, V' complete
                    // per tile: the softmax publishes P in two parts (keys 0..159 first); P V' of a part and the next tile's scores
                    // over the same columns are issued behind it, in that order, while the epilogue warps go on with the other part
#pragma unroll
                    for (int t = 0; t < 3; ++t) {
                        wait_on(mb_pa, pa_ph);                                   // 4a: P(t), key groups 0..9 (at least)
                        pv(t, 0, 10);
                        if (t < 2) scores_half(t + 1, 0);
                        wait_go();                                               // 4b: all of P(t)
                        pv(t, 10, 20);
                        if (t < 2) scores_half(t + 1, 1);
                        mma_commit_elect(mb_done);
                    }
                    wait_go(); load_w2(blk);                                     // 7: attention output + LN2 of every tile done; K/V' dead
                    if (!(last_track && blk == kDepth - 1)) load_wa((blk + 1) % kDepth);
                    mbar_wait(mb_w1, w1_ph); w1_ph ^= 1;                         // W1 was prefetched during attention
                    // ---- MLP, pipelined over row tiles (tile 0 -> H_A/Y_A, tile 1 -> H_B/Y_B, tile 2 -> H_A/Y_A) ----
                    // (issuing fc1 of tile 0 ahead of step 7, behind P V'(2), saves one MMA round trip but hangs under ncu's serialised
                    // launches - cause not understood, see DESIGN.md; the conservative order stays)
                    fc1(0, kColHA); mma_commit_elect(mb_h);
                    wait_on(mb_h, h_ph[0]);                                      // H_B aliases operand slot 0: fc1(0) must be done
                    fc1(1, kColHB); mma_commit_elect(mb_h + 1);
                    wait_on(mb_g, g_ph[0]);                                      // GELU(0) operand in H_A
                    wait_on(mb_h + 1, h_ph[1]);                                  // Y_A aliases operand slots 0/1: fc1(1) must be done
                    mbar_wait(mb_wb, wb_ph); wb_ph ^= 1;                         // W2 landed
                    fc2(kColHA, kColYA); mma_commit_elect(mb_y);
                    wait_on(mb_y, y_ph[0]);                                      // fc2(0) has read H_A
                    fc1(2, kColHA); mma_commit_elect(mb_h);
                    wait_on(mb_g + 1, g_ph[1]);                                  // GELU(1) operand in H_B
                    wait_on(mb_h, h_ph[0]);                                      // Y_B aliases operand slot 2: fc1(2) must be done
                    if (!(last_track && blk == kDepth - 1)) load_w1((blk + 1) % kDepth);   // W1 dead -> the next block's streams in
                    fc2(kColHB, kColYB); mma_commit_elect(mb_y + 1);
                    wait_on(mb_g, g_ph[0]);                                      // GELU(2) operand in H_A
                    wait_on(mb_yfree, yfree_ph);                                 // Y_A (tile 0) has been consumed
                    fc2(kColHA, kColYA); mma_commit_elect(mb_y);
                    wait_on(mb_y + 1, y_ph[1]);                                  // keep this side's phase bits in step
                    wait_on(mb_y, y_ph[0]);
                }
            }
        }
        __syncwarp();        // reconverge the control warp before the CTA-wide barrier below
    } else {
        // ======================================= epilogue warps ===========================================
        Epi e;
        e.tbase = tbase; e.q = warp & 3; e.s = warp >> 2; e.lane = lane; e.row = 32 * e.q + lane;
        e.lane_addr = (uint32_t)(32 * e.q) << 16;
        e.red = s_red; e.mb_go = mb_go; e.mb_done = mb_done; e.done_ph = 0;
        const int s = e.s, row = e.row;
        const float scale = 0.14433756729740643f;                 // 48 ** -0.5
        const float kLog2e = 1.4426950408889634f;
        uint32_t h_ph[2] = {0, 0}, y_ph[2] = {0, 0}, qd_ph[2] = {0, 0};
        // QKV epilogue: which of q / K / V this column group handles, and where inside its 48 columns
        const int qkv_part = (s * kQW) / 48, qkv_off = (s * kQW) % 48;

        for (int trk = blockIdx.x; trk < n; trk += gridDim.x) {
            // residual slice x[t][kCW]: tile t, row 128 t + row, columns [kCW s, kCW s + kCW)
            float x[3][kCW];
#pragma unroll
            for (int t = 0; t < 3; ++t) {
                const int r = 128 * t + row;
                const float* src = nullptr;
                if (r < kNz) src = tok_z + ((size_t)trk * z_stride_rows + r) * kC + kCW * s;
                else if (r < kN) src = tok_x + ((size_t)trk * x_stride_rows + (r - kNz)) * kC + kCW * s;
#pragma unroll
                for (int i = 0; i < kCW; i += 4) {
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (src) v = __ldg(reinterpret_cast<const float4*>(src + i));
                    x[t][i] = v.x; x[t][i + 1] = v.y; x[t][i + 2] = v.z; x[t][i + 3] = v.w;
                }
                if (taps && r < kN) {
                    float* tp = taps + ((size_t)trk * kN + r) * kC + kCW * s;
#pragma unroll
                    for (int i = 0; i < kCW; i += 4) *reinterpret_cast<float4*>(tp + i) = make_float4(x[t][i], x[t][i + 1], x[t][i + 2], x[t][i + 3]);
                }
            }

#pragma unroll 1
            for (int blk = 0; blk < kDepth; ++blk) {
                const float* par = s_par + blk * kTcParFloats;

#pragma unroll
                for (int t = 0; t < 3; ++t) {      // LayerNorm 1 -> the tiles' A-operand slots; each tile's QKV GEMM starts at once
                    float y[kCW];
                    e.ln(x[t], par + kPLn1g, par + kPLn1b, y);
                    if (e.active(t)) e.store_opa(t, y);
                    e.signal(mb_l1 + t, false); // -> 1a, 1b, 1c
                }

                // ---- QKV epilogue: a column group handles kQW of the 144 output columns: part 0 -> q (scaled) into the
                //      tile's A slot, part 1 -> K rows, part 2 -> V rows (shared memory, UMMA layouts)
                auto epi_qkv = [&](int t, uint32_t col) {
                    if (!e.active(t)) return;
                    float v[kQW];
                    {
                        uint32_t r[kQW / 8][8];
#pragma unroll
                        for (int c = 0; c < kQW / 8; ++c) tmem_ld8(e.taddr(col + kQW * s + 8 * c), r[c]);
                        tc_wait_ld();
#pragma unroll
                        for (int c = 0; c < kQW / 8; ++c)
#pragma unroll
                            for (int j = 0; j < 8; ++j) v[8 * c + j] = __uint_as_float(r[c][j]) + par[kPBqkv + kQW * s + 8 * c + j];
                    }
                    const int key = 128 * t + row;
                    if (qkv_part == 0) {
#pragma unroll
                        for (int c = 0; c < kQW / 2; c += 4) {
                            uint32_t hi[4], lo[4];
#pragma unroll
                            for (int j = 0; j < 4; ++j) split_pack2(v[2 * (c + j)] * scale, v[2 * (c + j) + 1] * scale, hi[j], lo[j]);
                            tmem_st4(e.taddr(kColOpa + 48 * t + qkv_off / 2 + c), hi);
                            if (kScoresTerms >= 2) tmem_st4(e.taddr(kColOpa + 48 * t + 24 + qkv_off / 2 + c), lo);
                        }
                    } else {
                        // K: K-major [k/8][key][8]   V: MN-major [f/8][key/8][key%8][f%8]  (both: chunk * 320*16 + key*16)
                        uint8_t* hi_base = smem + (qkv_part == 1 ? kSmKhi : kSmVhi) + key * 16 + (qkv_off / 8) * (kN * 16);
                        uint8_t* lo_base = smem + (qkv_part == 1 ? kSmKlo : kSmVlo) + key * 16 + (qkv_off / 8) * (kN * 16);
#pragma unroll
                        for (int c = 0; c < kQW / 8; ++c) {
                            uint32_t hi[4], lo[4];
#pragma unroll
                            for (int j = 0; j < 4; ++j) split_pack2(v[8 * c + 2 * j], v[8 * c + 2 * j + 1], hi[j], lo[j]);
                            *reinterpret_cast<uint4*>(hi_base + c * (kN * 16)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                            if (qkv_part == 2 || kScoresTerms >= 3)                    // K's low-order half is read by the q_hi k_lo term only
                                *reinterpret_cast<uint4*>(lo_base + c * (kN * 16)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                        }
                    }
                };
                e.wait_bar(mb_qd, qd_ph[0]);      epi_qkv(0, kColBig);        e.signal(mb_qf, true);     // -> 2 (buffer 0 free)
                e.wait_bar(mb_qd + 1, qd_ph[1]);  epi_qkv(1, kColBig + 160);
                e.wait_bar(mb_qd, qd_ph[0]);      epi_qkv(2, kColBig);        e.signal_go(true);         // -> 3

                // ---- attention per tile -------------------------------------------------------------------
                auto softmax = [&](int t) {
                    // the 20 groups of 16 score columns are dealt round-robin: column group s owns groups s, s + kNS, ...  After
                    // kRoundsA rounds every group of keys 0..159 is done and is published on its own barrier, so that the tensor
                    // pipe starts P V' (and the next tile's scores over those columns) while the remaining rounds are computed.
                    // TMEM loads are software pipelined (the next group is in flight while one is processed).
                    constexpr int kRounds = (20 + kNS - 1) / kNS;          // 4
                    constexpr int kRoundsA = (10 + kNS - 1) / kNS;         // 2: rounds that cover key groups 0..9
                    const int my_groups = (20 - s + kNS - 1) / kNS;
                    const uint32_t a0 = e.taddr(kColBig + 16 * s);
                    float m = -INFINITY;
                    if (e.active(t)) {
#pragma unroll
                        for (int k = 0; k < kRounds; ++k) {
                            if (k < my_groups) {
                                uint32_t r[16];
                                tmem_ld16(a0 + 16 * kNS * k, r);
                                tc_wait_ld();
#pragma unroll
                                for (int j = 0; j < 16; ++j) m = fmaxf(m, __uint_as_float(r[j]));
                            }
                        }
                    }
                    // row maxima: two arrays alternating with the tile.  softmax(t + 1) may start once S(t + 1) is complete, which the control warp
                    // commits only after every epilogue warp has arrived at the end of softmax(t) - an ordering through mbarriers and
                    // tcgen05.commit that is real but invisible to compute-sanitizer's racecheck; with one array per tile parity the write below
                    // is also separated from the previous reads of the same array by bar.sync's (epi_out), which the tool does see
                    float* rm = e.red + ((t & 1) ? 5 : 2) * (kNS * 128);
                    rm[s * 128 + row] = m;
                    epi_bar();
                    m = rm[row];
#pragma unroll
                    for (int g = 1; g < kNS; ++g) m = fmaxf(m, rm[g * 128 + row]);
                    float l = 0.f;
                    const float mb = m * kLog2e;
#pragma unroll
                    for (int k = 0; k < kRounds; ++k) {
                        if (e.active(t) && k < my_groups) {
                            uint32_t r[16];
                            tmem_ld16(a0 + 16 * kNS * k, r);
                            tc_wait_ld();
                            uint32_t hi[8], lo[8];
                            // packed fp32 (FFMA2 / FADD2): two running sums, two keys per issue slot
                            uint64_t l2 = 0ull;
                            const uint64_t nmb2 = f2bcast(-mb);
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                float a0, a1;
                                f2unpack(f2fma(f2pack(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1])), f2bcast(kLog2e), nmb2), a0, a1);
                                const float p0 = ex2_approx(a0), p1 = ex2_approx(a1);
                                l2 = f2add(l2, f2pack(p0, p1));
                                split_pack2(p0, p1, hi[j], lo[j]);
                            }
                            float l0, l1;
                            f2unpack(l2, l0, l1);
                            l += l0 + l1;
                            tmem_st8(a0 + 16 * kNS * k, hi);       // P overwrites S in place: [hi x8 | lo x8] per 16 keys
                            tmem_st8(a0 + 16 * kNS * k + 8, lo);
                        }
                        if (k == kRoundsA - 1) e.signal(mb_pa, false);           // -> 4a
                    }
                    e.red[(3 + (t & 1)) * (kNS * 128) + s * 128 + row] = l;     // summed in epi_out(t)
                    e.signal_go(false);                                          // -> 4b
                };
                // attention output of tile t: x += (P V')/l + bproj (V' carries the output projection), then LayerNorm 2 -> A slot.
                // O' sits in the tile's own slot: every thread reads its columns before the LayerNorm barriers, writes after.
                auto epi_out = [&](int t) {
                    epi_bar();                               // partial row sums of softmax(t) are visible
                    const float* rl = e.red + (3 + (t & 1)) * (kNS * 128);
                    float lsum = rl[row];
#pragma unroll
                    for (int g = 1; g < kNS; ++g) lsum += rl[g * 128 + row];
                    const float inv = 1.f / lsum;
                    if (e.active(t)) {
                        uint32_t r[kCW];
                        tmem_ld<kCW>(e.taddr(kColOpa + 48 * t + kCW * s), r);
                        tc_wait_ld();
#pragma unroll
                        for (int j = 0; j < kCW; ++j) x[t][j] += fmaf(__uint_as_float(r[j]), inv, par[kPBproj + kCW * s + j]);
                    }
                    float y[kCW];
                    e.ln(x[t], par + kPLn2g, par + kPLn2b, y);
                    if (e.active(t)) e.store_opa(t, y);
                };
                e.wait_done(); softmax(0);
                e.wait_done(); softmax(1); epi_out(0);        // epi_out overlaps P V' (1) and S(2)
                e.wait_done(); softmax(2); epi_out(1);
                e.wait_done(); epi_out(2); e.signal_go(false);                    // -> 7

                // ---- MLP per tile -------------------------------------------------------------------------
                auto gelu = [&](int t, uint32_t h_col) {
                    if (!e.active(t)) return;
                    const uint32_t a0 = e.taddr(h_col + kHW * s);                 // group s owns hidden columns [kHW s, kHW s + kHW)
#pragma unroll
                    for (int g = 0; g < kHW / 16; ++g) {
                        uint32_t r[16];
                        tmem_ld16(a0 + 16 * g, r);
                        tc_wait_ld();
                        uint32_t hi[8], lo[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            float h0, h1;
                            gelu_erf2(f2add(f2pack(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1])),
                                            f2pack(par[kPBfc1 + kHW * s + 16 * g + 2 * j], par[kPBfc1 + kHW * s + 16 * g + 2 * j + 1])), h0, h1);
                            split_pack2(h0, h1, hi[j], lo[j]);
                        }
                        tmem_st8(a0 + 16 * g, hi);
                        tmem_st8(a0 + 16 * g + 8, lo);
                    }
                };
                auto epi_fc2 = [&](int t, uint32_t y_col) {
                    if (!e.active(t)) return;
                    uint32_t r[kCW];
                    tmem_ld<kCW>(e.taddr(y_col + kCW * s), r);
                    tc_wait_ld();
#pragma unroll
                    for (int j = 0; j < kCW; ++j) x[t][j] += __uint_as_float(r[j]) + par[kPBfc2 + kCW * s + j];
                    const int rr = 128 * t + row;
                    if (taps && rr < kN) {
                        float* tp = taps + (size_t)(blk + 1) * tap_stride + ((size_t)trk * kN + rr) * kC + kCW * s;
#pragma unroll
                        for (int i = 0; i < kCW; i += 4) *reinterpret_cast<float4*>(tp + i) = make_float4(x[t][i], x[t][i + 1], x[t][i + 2], x[t][i + 3]);
                    }
                    if (blk == kDepth - 1 && rr < kN) {
                        float* dst = out + ((size_t)trk * kN + rr) * kC + kCW * s;
#pragma unroll
                        for (int i = 0; i < kCW; i += 4) *reinterpret_cast<float4*>(dst + i) = make_float4(x[t][i], x[t][i + 1], x[t][i + 2], x[t][i + 3]);
                    }
                };
                // MLP, pipelined over row tiles: the tensor pipe runs fc1 / fc2 of the other tiles during each GELU
                e.wait_bar(mb_h, h_ph[0]);      gelu(0, kColHA);     e.signal(mb_g, false);
                e.wait_bar(mb_h + 1, h_ph[1]);  gelu(1, kColHB);     e.signal(mb_g + 1, false);
                e.wait_bar(mb_y, y_ph[0]);      epi_fc2(0, kColYA);  e.signal(mb_yfree, false);
                e.wait_bar(mb_h, h_ph[0]);      gelu(2, kColHA);     e.signal(mb_g, false);
                e.wait_bar(mb_y + 1, y_ph[1]);  epi_fc2(1, kColYB);
                e.wait_bar(mb_y, y_ph[0]);      epi_fc2(2, kColYA);
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == kEpiWarps) tmem_dealloc(tbase, 512);
}

#ifdef VT_TC_WATCHDOG
extern "C" int vt_tc_watchdog_read(int* rec, int* n) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(n, tc::g_wd_n, sizeof(int));
    cudaMemcpyFromSymbol(rec, tc::g_wd_rec, sizeof(int) * 256 * 6);
    return 0;
}
#endif

#ifdef VT_TC_TRACE
extern "C" int vt_tc_trace_read(long long* host, int* n) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(n, g_tc_trace_n, 2 * sizeof(int));
    cudaMemcpyFromSymbol(host, g_tc_trace, sizeof(long long) * 2 * 4096);
    int zero[2] = {0, 0};
    cudaMemcpyToSymbol(g_tc_trace_n, zero, sizeof zero);
    return 0;
}
#endif

int launch_blocks_tc(const float* tok_z, int z_stride_rows, const float* tok_x, int x_stride_rows, float* out, int n,
                     const ModelW& w, float* taps, size_t tap_stride, int num_sms, int scores_terms, cudaStream_t st) {
    if (n <= 0) return 0;
    static DeviceOnce once1, once3;
    if (!ensure_dyn_smem(once1, blocks_tc_kernel<1>, kTcSmemBytes) || !ensure_dyn_smem(once3, blocks_tc_kernel<3>, kTcSmemBytes)) return -1;
    const int grid = n < num_sms ? n : num_sms;
    if (scores_terms == 1) blocks_tc_kernel<1><<<grid, kTcThreads, kTcSmemBytes, st>>>(tok_z, z_stride_rows, tok_x, x_stride_rows, out, n, w, taps, tap_stride);
    else blocks_tc_kernel<3><<<grid, kTcThreads, kTcSmemBytes, st>>>(tok_z, z_stride_rows, tok_x, x_stride_rows, out, n, w, taps, tap_stride);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

// Host side: one block's checkpoint tensors -> its blobs wa, wb and parameter vector par (layouts above).
// The attention output projection is folded into the value projection: (P V) Wp^T = P (V Wp^T), V Wp^T = LN(x) (Wp Wv)^T + Wp bv
// (products accumulated in float64; the kernel then needs no separate proj GEMM).
void block_tc_pack(const BlockTensors& t, uint8_t* wa, uint8_t* wb, float* par) {
    auto pack_kmajor = [](uint8_t* dst_hi, uint8_t* dst_lo, const float* W, int N, int K) {     // W: [N][K] (torch Linear weight)
        for (int n = 0; n < N; ++n)
            for (int k = 0; k < K; ++k) put_kmajor_f16(dst_hi, dst_lo, N, n, k, W[(size_t)n * K + k]);
    };
    std::vector<float> wf(t.wqkv, t.wqkv + 3 * kC * kC), bvp(kC);
    for (int o = 0; o < kC; ++o) {
        for (int i = 0; i < kC; ++i) {
            double acc = 0.0;
            for (int j = 0; j < kC; ++j) acc += (double)t.wproj[o * kC + j] * (double)t.wqkv[(2 * kC + j) * kC + i];
            wf[(2 * kC + o) * kC + i] = (float)acc;
        }
        double accb = 0.0;
        for (int j = 0; j < kC; ++j) accb += (double)t.wproj[o * kC + j] * (double)t.bqkv[2 * kC + j];
        bvp[o] = (float)accb;
    }
    pack_kmajor(wa, wa + kWaLo, wf.data(), 3 * kC, kC);
    pack_kmajor(wb, wb + kWbW1Lo, t.wfc1, kHid, kC);
    pack_kmajor(wb + kWbW2Hi, wb + kWbW2Lo, t.wfc2, kC, kHid);
    auto put = [&](int o, const float* src, int n) { memcpy(par + o, src, n * sizeof(float)); };
    put(kPLn1g, t.ln1_g, kC);
    put(kPLn1b, t.ln1_b, kC);
    put(kPBqkv, t.bqkv, 2 * kC);                     // bq, bk
    put(kPBqkv + 2 * kC, bvp.data(), kC);            // bias of the folded value projection
    put(kPBproj, t.bproj, kC);
    put(kPLn2g, t.ln2_g, kC);
    put(kPLn2b, t.ln2_b, kC);
    put(kPBfc1, t.bfc1, kHid);
    put(kPBfc2, t.bfc2, kC);
}

}  // namespace vt
