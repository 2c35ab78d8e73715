// Shared by the tensor-core stem kernels (vt_stem_tc.cu, vt_stem_fused.cu) and the host weight packer: the K-step schedule of a
// 3x3 stride-2 convolution over a parity-plane operand image, and the shared-memory geometry of one band of output rows.
#pragma once
#include "vt_internal.h"
#include "vt_tc.cuh"

namespace vt {

// ---- K-step schedule shared by the device issue loop and the host weight packer -------------------------------
// Accumulator 0 (T_A) sums taps (ky, kx in {1,2}), accumulator 1 (T_B) taps (ky, kx = 0).  A K step covers two
// 8-channel chunks: chunks (2j, 2j+1) of one tap, and - when the chunk count is odd - the last chunks of two taps
// paired (lower shared-memory address first; a tap left alone is paired with itself against zero weights).
__host__ __device__ inline int tcs_ntaps(int acc) { return acc == 0 ? 6 : 3; }
__host__ __device__ inline void tcs_tap(int acc, int tap, int& ky, int& kx) {
    ky = acc == 0 ? tap / 2 : tap;
    kx = acc == 0 ? 1 + (tap & 1) : 0;
}
// position of a tap's operand inside the band image, in units that order addresses: plane index and first row
__host__ __device__ inline void tcs_tap_pos(int ky, int kx, int& plane, int& row0) {
    plane = ((ky == 1) ? 0 : 2) + ((kx == 1) ? 0 : 1);
    row0 = (ky == 0) ? 0 : 1;
}
__host__ __device__ inline int tcs_nsteps(int cch, int acc) {
    const int t = tcs_ntaps(acc);
    return t * (cch / 2) + ((cch & 1) ? (t + 1) / 2 : 0);
}
// K step s of accumulator acc -> the two (tap, chunk) halves; zero1 = second half multiplies zero weights
__host__ __device__ inline void tcs_step(int cch, int acc, int s, int& tap0, int& ch0, int& tap1, int& ch1, bool& zero1) {
    const int t = tcs_ntaps(acc), per = cch / 2;
    zero1 = false;
    if (s < t * per) { tap0 = tap1 = s / per; ch0 = 2 * (s % per); ch1 = ch0 + 1; return; }
    const int p = s - t * per;
    int a = 2 * p, b = 2 * p + 1;
    ch0 = ch1 = cch - 1;
    if (b >= t) { tap0 = tap1 = a; zero1 = true; return; }
    int ky, kx, pa, ra, pb, rb;
    tcs_tap(acc, a, ky, kx); tcs_tap_pos(ky, kx, pa, ra);
    tcs_tap(acc, b, ky, kx); tcs_tap_pos(ky, kx, pb, rb);
    if (pa > pb || (pa == pb && ra > rb)) { const int tmp = a; a = b; b = tmp; }
    tap0 = a; tap1 = b;
}

constexpr int kConv2BR = 4, kConv3BR = 4;     // output rows per CTA

template <int CCH, int COUT, int NPAD, int WOUT, int BR>
struct TcConv {
    static constexpr int kBR = BR;                              // output rows per CTA (smaller band = more CTAs per SM, more halo)
    static constexpr int kRowsPerTile = 128 / WOUT;
    static constexpr int kTiles = kBR / kRowsPerTile;            // M tiles per CTA
    static constexpr int kPlaneRows = kBR + 1;                   // band row 0 <-> plane row oy0 - 1
    static constexpr int kChunkBytes = kPlaneRows * WOUT * 16;
    static constexpr int kPlaneBytes = CCH * kChunkBytes;
    static constexpr int kABytes = 4 * kPlaneBytes;              // one precision
    static constexpr int kStepsA = 6 * (CCH / 2) + ((CCH & 1) ? 3 : 0), kStepsB = 3 * (CCH / 2) + ((CCH & 1) ? 2 : 0);
    static constexpr int kWPrecBytes = (kStepsA + kStepsB) * 2 * NPAD * 16;   // one precision, two 8-wide chunks per K step
    static constexpr int kWBytes = 2 * kWPrecBytes;
    static constexpr int kStages = 2;                            // A operand stages (bulk copies of item i+1 overlap MMA + epilogue of item i)
    static constexpr int kStageBytes = 2 * kABytes;              // hi | lo
    static constexpr int kOffA = 0;
    static constexpr int kOffW = kStages * kStageBytes;
    static constexpr int kOffBias = kOffW + kWBytes;
    static constexpr int kOffXchg = kOffBias + NPAD * 4;         // row-split exchange (WOUT = 64 only): [tile pair or chunk][2][2][8] floats
    static constexpr int kXchgFloats = 2 * 4 * 2 * 2 * 8;         // per epilogue group
    static constexpr int kOffBar = kOffXchg + kXchgFloats * 4;   // w, full[2], afree[2], tfull[2], tfree[2], tmem base
    static constexpr int kSmemBytes = kOffBar + 10 * 8;
    static constexpr int kCopies = 2 * 4 * CCH;                  // bulk copies per band: (precision, plane, chunk)
    static constexpr int kAccCols = kTiles * 2 * NPAD;           // TMEM columns of one item's accumulators (T_A | T_B per tile)
    static constexpr int kTmemCols = (2 * kAccCols <= 32) ? 32 : (2 * kAccCols <= 64) ? 64 : (2 * kAccCols <= 128) ? 128 : (2 * kAccCols <= 256) ? 256 : 512;
    static constexpr int kThreads = 576;                         // 2 x 8 epilogue warps (one group per accumulator set) + MMA warp + copy warp
    static_assert(NPAD % 16 == 0 && NPAD >= COUT && 128 % WOUT == 0 && kBR % kRowsPerTile == 0, "shape");
    static_assert(kOffBar % 8 == 0 && kOffW % 128 == 0 && kStageBytes % 128 == 0 && 2 * kAccCols <= 512, "alignment");
};

}  // namespace vt
