// Per-track tap tables of the fused crop gathers (vt_stem.cu: crop + conv1 on CUDA cores; vt_stem_fused.cu: crop + conv1 + conv2 on tcgen05).
#pragma once
#include "vt_geom.cuh"
#include "vt_internal.h"

namespace vt {

// Per-track tap tables of the fused gather, computed once per track (float64 geometry + the resize taps) instead of by
// every tile's CTA: taps[item][0][d + 1] = column record of resized-crop column d, taps[item][1][d + 1] = row record,
// d = -1 .. S - 1.  Columns: the two horizontal taps of cv::resize are the same or adjacent source pixels, so a column is
// one PAIR of adjacent pixels (.x = byte offset of the first, .y = weights first | second << 16; a tap that is padding
// or clamped away has weight 0 - a zero pixel and a zero weight give the same products - and the pair is anchored on a
// tap that is inside the image, so the six bytes read always are).  Rows: .x/.y = byte offsets of the two tap rows
// (0 when the row is padding), .z = weights lo | hi << 16.  .w = 1 when the position is outside the resized crop
// (= the convolution's zero padding, which is 0.0f and not the normalised pixel 0).
// The box of item i is track item_slot(slots, i) of `boxes`; a bad slot gives status VT_TRACK_BAD_SLOT and empty tables.
// `work_counter` (may be null) is the consumer kernel's dynamic work counter: block 0 resets it to `work_counter0` on the way.
// COUNTED: only items below *count are processed (the range fallback of vt_api.cu, whose item count is known on the device only);
// the uncounted instantiation, which the fused tensor-core front launches, does not read `count`.
constexpr int kTapPitch = 264;
template <int S, bool COUNTED = false>
__global__ void __launch_bounds__(288)
crop_taps_kernel(const int32_t* __restrict__ frame_hw, const double* __restrict__ boxes, const int32_t* __restrict__ slots, double factor,
                 int4* __restrict__ taps,
                 int32_t* __restrict__ out_status, int* __restrict__ work_counter, int work_counter0, const int32_t* __restrict__ count) {
    __shared__ CropGeom sg;
    __shared__ double s_scale;
    const int item = blockIdx.x, tid = threadIdx.x;
    if (COUNTED && item >= *count) return;
    const int H = frame_hw[2 * item], W = frame_hw[2 * item + 1];
    if (item == 0 && tid == 287 && work_counter) *work_counter = work_counter0;
    if (tid == 0) {
        const int slot = item_slot(slots, item);
        if (slot < 0) {
            sg = CropGeom{0, 0, 0, VT_TRACK_BAD_SLOT_, 0.0};
            s_scale = 0.0;
        } else {
            const double* bx = boxes + 4 * (size_t)slot;
            sg = crop_geometry(bx[0], bx[1], bx[2], bx[3], factor, S, H, W);
            s_scale = resize_scale(S, sg.crop_sz);
        }
        if (out_status) out_status[item] = sg.status;
    }
    __syncthreads();
    const CropGeom g = sg;
    const double scale = s_scale;
    if (tid > S) return;
    const int d = tid - 1;
    // Padding rows are read with weight 0 (branch-free gather); they read the crop's first in-image row rather than row 0 of the frame, so
    // that a track never touches frame rows outside [max(0, y1), min(H, y1 + crop_sz)) - callers may upload only those rows.
    const int anchor = g.status == 0 ? min(max(g.y1, 0), max(H - 2, 0)) * W * 3 : 0;
    int4 tc = make_int4(0, 0, 0, 1), tr = make_int4(anchor, anchor, 0, 1);
    if (d >= 0 && g.status == 0) {
        {
            int s0, s1, a0, a1; bool w0, w1;
            tap_x(d, scale, g.crop_sz, s0, s1, a0, a1, w0, w1);
            const int ix0 = g.x1 + s0, ix1 = g.x1 + s1;
            if (!(ix0 >= 0 && ix0 <= W - 2)) a0 = 0;
            if (!(ix1 >= 0 && ix1 <= W - 2) || ix1 == ix0) a1 = 0;      // s1 == s0 only where cv::resize clamps, and there a1 == 0
            if (a0 != 0) tc = make_int4(ix0 * 3, a0 | (a1 << 16), 0, 0);
            else if (a1 != 0) tc = make_int4(ix1 * 3, a1, 0, 0);
            else tc = make_int4(0, 0, 0, 0);
        }
        {
            int r0, r1, b0, b1; bool w0, w1;
            tap_y(d, scale, g.crop_sz, r0, r1, b0, b1, w0, w1);
            const int iy0 = g.y1 + r0, iy1 = g.y1 + r1;
            const bool v0 = iy0 >= 0 && iy0 <= H - 2, v1 = iy1 >= 0 && iy1 <= H - 2;
            tr = make_int4(v0 ? iy0 * W * 3 : anchor, v1 ? iy1 * W * 3 : anchor, (v0 ? b0 : 0) | ((v1 ? b1 : 0) << 16), 0);
        }
    }
    taps[((size_t)item * 2 + 0) * kTapPitch + tid] = tc;
    taps[((size_t)item * 2 + 1) * kTapPitch + tid] = tr;
}

}  // namespace vt
