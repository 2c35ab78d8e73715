// Post-processing shared by the fused head kernels (vt_head.cu) and the generic path (vt_generic.cu):
//   cal_bbox            lib/models/layers/head.py:142-160 (first arg-max wins)
//   track() epilogue    lib/test/tracker/vit_dist.py:103-111,147-156 + lib/utils/box_ops.py:97-106
#pragma once
#include "vt_geom.cuh"
#include "vt_internal.h"

namespace vt {

// arg-max with first-index tie-break over 256 values (one per thread); result broadcast to all threads.
__device__ __forceinline__ void block_argmax256(float v, int idx, float* red, float& best, int& best_idx) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, v, o);
        const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
        if (ov > v || (ov == v && oi < idx)) { v = ov; idx = oi; }
    }
    __syncthreads();
    if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5] = v; red[8 + (threadIdx.x >> 5)] = __int_as_float(idx); }
    __syncthreads();
    best = red[0]; best_idx = __float_as_int(red[8]);
#pragma unroll
    for (int k = 1; k < 8; ++k) {
        const float ov = red[k]; const int oi = __float_as_int(red[8 + k]);
        if (ov > best || (ov == best && oi < best_idx)) { best = ov; best_idx = oi; }
    }
}

__device__ __forceinline__ float sigmoid_clamp(float v) {
    const float s = 1.f / (1.f + expf(-v));
    return fminf(fmaxf(s, 1e-4f), 0.9999f);               // torch.clamp(x.sigmoid_(), 1e-4, 1 - 1e-4)
}

// Raw and Hann-weighted arg-max of one track's maps (256 threads, thread = pixel); results broadcast to all threads.
__device__ __forceinline__ void decode_argmax(const float* m_score, const float* m_resp, float* red, float& raw_max, int& raw_idx,
                                              float& win_max, int& win_idx) {
    block_argmax256(m_score[threadIdx.x], threadIdx.x, red, raw_max, raw_idx);
    block_argmax256(m_resp[threadIdx.x], threadIdx.x, red, win_max, win_idx);
}

// One thread: forward's pred_boxes from the raw arg-max; the tracker's box from the windowed arg-max mapped back to the
// frame, clipped, and written to out_boxes / out_detail / state.  m_size: [2][256], m_off: [2][256].
// numeric_status: 0, or VT_TRACK_NUMERIC_RANGE when the track's activations left the representable range (result withheld).
__device__ __forceinline__ void decode_box(const HeadArgs& a, int trk, const float* m_size, const float* m_off, float raw_max,
                                           int raw_idx, float win_max, int win_idx, int numeric_status = 0) {
    if (a.pred_boxes) {
        float* pb = a.pred_boxes + (size_t)trk * 4;
        const float qnan = __int_as_float(0x7fc00000);
        pb[0] = numeric_status ? qnan : ((float)(raw_idx & 15) + m_off[raw_idx]) / 16.f;
        pb[1] = numeric_status ? qnan : ((float)(raw_idx >> 4) + m_off[256 + raw_idx]) / 16.f;
        pb[2] = numeric_status ? qnan : m_size[raw_idx];
        pb[3] = numeric_status ? qnan : m_size[256 + raw_idx];
    }
    if (a.state) {
        double* ob = a.out_boxes + (size_t)trk * 5;
        double* od = a.out_detail ? a.out_detail + (size_t)trk * 8 : nullptr;
        const int slot = item_slot(a.slots, trk);
        if (slot < 0) {               // bad slot-list entry: no state to read or write
            ob[0] = ob[1] = ob[2] = ob[3] = 0.0; ob[4] = -1.0;
            if (od) { od[0] = od[1] = od[2] = od[3] = od[4] = 0.0; od[5] = -1.0; od[6] = (double)VT_TRACK_BAD_SLOT_; od[7] = 0.0; }
            return;
        }
        double* st = a.state + (size_t)slot * 4;
        const double sx = st[0], sy = st[1], sw = st[2], sh = st[3];
        const int H = a.frame_hw[2 * trk], W = a.frame_hw[2 * trk + 1];
        const CropGeom g = crop_geometry(sx, sy, sw, sh, a.search_factor, kSx, H, W);
        int status = a.status ? a.status[trk] : g.status;
        if (status == 0) status = numeric_status;
        if (status != 0) {            // the reference raises here; keep the state and flag the track
            ob[0] = sx; ob[1] = sy; ob[2] = sw; ob[3] = sh; ob[4] = -1.0;
            if (od) { od[0] = od[1] = od[2] = od[3] = 0.0; od[4] = g.resize_factor; od[5] = -1.0; od[6] = (double)status; od[7] = 0.0; }
            return;
        }
        // pred_box = (pred_boxes.mean(0) * search_size / resize_factor).tolist()   (fp32 on the device)
        const float rf32 = (float)g.resize_factor;
        const float bx = ((float)(win_idx & 15) + m_off[win_idx]) / 16.f;
        const float by = ((float)(win_idx >> 4) + m_off[256 + win_idx]) / 16.f;
        const float pcx = __fdiv_rn(__fmul_rn(bx, 256.f), rf32);
        const float pcy = __fdiv_rn(__fmul_rn(by, 256.f), rf32);
        const float pw = __fdiv_rn(__fmul_rn(m_size[win_idx], 256.f), rf32);
        const float ph = __fdiv_rn(__fmul_rn(m_size[256 + win_idx], 256.f), rf32);
        // map_box_back (float64, Python semantics)
        const double cx_prev = __dadd_rn(sx, __dmul_rn(0.5, sw)), cy_prev = __dadd_rn(sy, __dmul_rn(0.5, sh));
        const double half_side = __ddiv_rn(__dmul_rn(0.5, (double)kSx), g.resize_factor);
        const double cx_real = __dadd_rn((double)pcx, __dsub_rn(cx_prev, half_side));
        const double cy_real = __dadd_rn((double)pcy, __dsub_rn(cy_prev, half_side));
        double x1 = __dsub_rn(cx_real, __dmul_rn(0.5, (double)pw));
        double y1 = __dsub_rn(cy_real, __dmul_rn(0.5, (double)ph));
        double bw = (double)pw, bh = (double)ph;
        // clip_box(box, H, W, margin=10)
        double x2 = __dadd_rn(x1, bw), y2 = __dadd_rn(y1, bh);
        x1 = fmin(fmax(0.0, x1), (double)(W - 10));
        x2 = fmin(fmax(10.0, x2), (double)W);
        y1 = fmin(fmax(0.0, y1), (double)(H - 10));
        y2 = fmin(fmax(10.0, y2), (double)H);
        bw = fmax(10.0, __dsub_rn(x2, x1));
        bh = fmax(10.0, __dsub_rn(y2, y1));
        ob[0] = x1; ob[1] = y1; ob[2] = bw; ob[3] = bh; ob[4] = (double)raw_max;
        if (od) {
            od[0] = (double)pcx; od[1] = (double)pcy; od[2] = (double)pw; od[3] = (double)ph;
            od[4] = g.resize_factor; od[5] = (double)win_idx; od[6] = 0.0; od[7] = (double)win_max;
        }
        if (a.update_state) { st[0] = x1; st[1] = y1; st[2] = bw; st[3] = bh; }
    }
}

}  // namespace vt
