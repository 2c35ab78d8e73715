// K1: fused crop + zero-pad + OpenCV-exact u8 bilinear resize + normalise, straight from raw uint8
// frames in HBM.  Replaces sample_target (lib/train/data/processing_utils.py:12-71: numpy slice,
// cv.copyMakeBorder, cv.resize) + Preprocessor.process (lib/test/tracker/data_utils.py:11-17).
// The padded crop is never materialised: every output pixel gathers its 2x2 source taps.
//
// Bound: HBM.  Algorithmic bytes per item: 3*min(crop^2, 4*S^2) source bytes + 12*S^2 written.
#include "vt_geom.cuh"
#include "vt_internal.h"

namespace vt {

constexpr int kCropThreads = 256;
constexpr int kCropRows = 8;      // output rows per CTA

// One CTA = kCropRows output rows of one item.  Thread -> output column (S == 256) or
// (row parity, column) (S == 128).  Per-column taps are computed once per thread and reused for
// every row; per-row taps are warp-uniform.
template <int S>
__global__ void __launch_bounds__(kCropThreads)
crop_normalize_kernel(const uint8_t* __restrict__ frames, const int64_t* __restrict__ frame_offsets,
                      const int32_t* __restrict__ frame_hw, const double* __restrict__ boxes, const int32_t* __restrict__ slots, double factor,
                      const float* __restrict__ lut, float* __restrict__ out_nchw,
                      uint8_t* __restrict__ out_u8, uint8_t* __restrict__ out_mask,
                      double* __restrict__ out_rf, int32_t* __restrict__ out_status) {
    __shared__ float s_lut[3 * 256];
    for (int i = threadIdx.x; i < 3 * 256; i += kCropThreads) s_lut[i] = lut[i];

    const int item = blockIdx.y;
    const int H = frame_hw[2 * item], W = frame_hw[2 * item + 1];
    const int slot = item_slot(slots, item);
    const double* bx = boxes + 4 * (size_t)(slot < 0 ? 0 : slot);
    const CropGeom g = slot < 0 ? CropGeom{0, 0, 0, VT_TRACK_BAD_SLOT_, 0.0} : crop_geometry(bx[0], bx[1], bx[2], bx[3], factor, S, H, W);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        if (out_rf) out_rf[item] = g.resize_factor;
        if (out_status) out_status[item] = g.status;
    }
    __syncthreads();

    constexpr int kRowsPerPass = kCropThreads / S;            // 1 (S=256) or 2 (S=128)
    const int col = threadIdx.x % S;
    const int rsub = threadIdx.x / S;
    const int row_base = blockIdx.x * kCropRows;
    const size_t plane = (size_t)S * S;
    float* o_f = out_nchw + (size_t)item * 3 * plane;

    if (g.status != 0) {     // failed item: deterministic zeros
        for (int r = rsub; r < kCropRows; r += kRowsPerPass) {
            const int oy = row_base + r;
            const size_t p = (size_t)oy * S + col;
            o_f[p] = 0.f; o_f[plane + p] = 0.f; o_f[2 * plane + p] = 0.f;
            if (out_u8) { uint8_t* q = out_u8 + ((size_t)item * plane + p) * 3; q[0] = q[1] = q[2] = 0; }
            if (out_mask) out_mask[(size_t)item * plane + p] = 1;
        }
        return;
    }

    const uint8_t* __restrict__ im = frames + frame_offsets[item];
    const double scale = resize_scale(S, g.crop_sz);

    int sx0, sx1, a0, a1; bool wx0, wx1;
    tap_x(col, scale, g.crop_sz, sx0, sx1, a0, a1, wx0, wx1);
    const int ix0 = g.x1 + sx0, ix1 = g.x1 + sx1;
    const bool vx0 = ix0 >= 0 && ix0 <= W - 2;
    const bool vx1 = ix1 >= 0 && ix1 <= W - 2;
    const bool padx = (!vx0 && wx0) || (!vx1 && wx1);
    const size_t rowb = (size_t)W * 3;

#pragma unroll
    for (int r = rsub; r < kCropRows; r += kRowsPerPass) {
        const int oy = row_base + r;
        int r0, r1, b0, b1; bool wy0, wy1;
        tap_y(oy, scale, g.crop_sz, r0, r1, b0, b1, wy0, wy1);
        const int iy0 = g.y1 + r0, iy1 = g.y1 + r1;
        const bool vy0 = iy0 >= 0 && iy0 <= H - 2;
        const bool vy1 = iy1 >= 0 && iy1 <= H - 2;

        int p00[3] = {0, 0, 0}, p01[3] = {0, 0, 0}, p10[3] = {0, 0, 0}, p11[3] = {0, 0, 0};
        if (vy0) {
            const uint8_t* rp = im + (size_t)iy0 * rowb;
            if (vx0) { const uint8_t* q = rp + (size_t)ix0 * 3; p00[0] = __ldg(q); p00[1] = __ldg(q + 1); p00[2] = __ldg(q + 2); }
            if (vx1) { const uint8_t* q = rp + (size_t)ix1 * 3; p01[0] = __ldg(q); p01[1] = __ldg(q + 1); p01[2] = __ldg(q + 2); }
        }
        if (vy1) {
            const uint8_t* rp = im + (size_t)iy1 * rowb;
            if (vx0) { const uint8_t* q = rp + (size_t)ix0 * 3; p10[0] = __ldg(q); p10[1] = __ldg(q + 1); p10[2] = __ldg(q + 2); }
            if (vx1) { const uint8_t* q = rp + (size_t)ix1 * 3; p11[0] = __ldg(q); p11[1] = __ldg(q + 1); p11[2] = __ldg(q + 2); }
        }
        const size_t p = (size_t)oy * S + col;
        uint8_t v8[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const int h0 = p00[c] * a0 + p01[c] * a1;            // HResize (int32, 11-bit coefficients)
            const int h1 = p10[c] * a0 + p11[c] * a1;
            int v = (((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2;   // VResizeLinear 8U
            v = min(max(v, 0), 255);
            v8[c] = (uint8_t)v;
            o_f[c * plane + p] = s_lut[c * 256 + v];
        }
        if (out_u8) { uint8_t* q = out_u8 + ((size_t)item * plane + p) * 3; q[0] = v8[0]; q[1] = v8[1]; q[2] = v8[2]; }
        if (out_mask) {
            const bool pady = (!vy0 && wy0) || (!vy1 && wy1);
            out_mask[(size_t)item * plane + p] = (padx || pady) ? 1 : 0;
        }
    }
}

int launch_crop_normalize(const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw,
                          const double* boxes, const int32_t* slots, double factor, int S, int n, const float* lut,
                          float* out_nchw, uint8_t* out_u8, uint8_t* out_mask, double* out_rf,
                          int32_t* out_status, cudaStream_t st) {
    if (n <= 0) return 0;
    int launched = 0;
    // gridDim.y is limited to 65535: split very large batches
    for (int first = 0; first < n; first += 32768) {
        const int m = min(32768, n - first);
        dim3 grid(S / kCropRows, m);
        const size_t plane = (size_t)S * S;
        float* o = out_nchw + (size_t)first * 3 * plane;
        uint8_t* u = out_u8 ? out_u8 + (size_t)first * 3 * plane : nullptr;
        uint8_t* mk = out_mask ? out_mask + (size_t)first * plane : nullptr;
        double* rf = out_rf ? out_rf + first : nullptr;
        int32_t* stt = out_status ? out_status + first : nullptr;
        const double* bx = slots ? boxes : boxes + 4 * first;
        const int32_t* sl = slots ? slots + first : nullptr;
        if (S == 256)
            crop_normalize_kernel<256><<<grid, kCropThreads, 0, st>>>(frames, frame_offsets + first, frame_hw + 2 * first,
                                                                     bx, sl, factor, lut, o, u, mk, rf, stt);
        else if (S == 128)
            crop_normalize_kernel<128><<<grid, kCropThreads, 0, st>>>(frames, frame_offsets + first, frame_hw + 2 * first,
                                                                     bx, sl, factor, lut, o, u, mk, rf, stt);
        else
            return -1;
        ++launched;
    }
    return cudaGetLastError() == cudaSuccess ? launched : -1;
}

}  // namespace vt
