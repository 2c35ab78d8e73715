// Slot lists of vt_tracks_init_slots / vt_tracks_step_slots: the caller's list -> one effective slot per item, and the row copies
// between item-ordered workspace and slot-addressed track state.  Nothing here synchronises with the host or allocates, so the calls
// that use it can be captured in a CUDA graph and replayed with new contents in the slot buffer.
#include "vt_internal.h"

namespace vt {

constexpr int kSlotThreads = 256;

// Every valid entry offers its item index for its slot; the lowest index (the first occurrence) wins.
__global__ void claim_slots_kernel(const int32_t* __restrict__ slots, int n, int max_tracks, uint32_t* __restrict__ claim) {
    const int i = blockIdx.x * kSlotThreads + threadIdx.x;
    if (i >= n) return;
    const int s = slots[i];
    if (s >= 0 && s < max_tracks) atomicMin(claim + s, (uint32_t)i);
}

// The winner of each slot reads its own index back and then releases the claim (resolve_slot).
__global__ void resolve_slots_kernel(const int32_t* __restrict__ slots, int n, int max_tracks, uint32_t* __restrict__ claim,
                                     int32_t* __restrict__ eff) {
    const int i = blockIdx.x * kSlotThreads + threadIdx.x;
    if (i >= n) return;
    eff[i] = resolve_slot(slots, i, max_tracks, claim);
}

int launch_claim_slots(const int32_t* slots, int n, int max_tracks, uint32_t* claim, cudaStream_t st) {
    if (n <= 0) return 0;
    claim_slots_kernel<<<(n + kSlotThreads - 1) / kSlotThreads, kSlotThreads, 0, st>>>(slots, n, max_tracks, claim);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

int launch_resolve_slots(const int32_t* slots, int n, int max_tracks, uint32_t* claim, int32_t* eff, cudaStream_t st) {
    if (n <= 0) return 0;
    const int grid = (n + kSlotThreads - 1) / kSlotThreads;
    claim_slots_kernel<<<grid, kSlotThreads, 0, st>>>(slots, n, max_tracks, claim);
    resolve_slots_kernel<<<grid, kSlotThreads, 0, st>>>(slots, n, max_tracks, claim, eff);
    return cudaGetLastError() == cudaSuccess ? 2 : -1;
}

// One CTA per item.
__global__ void gather_rows_kernel(const float* __restrict__ src, size_t src_stride, float* __restrict__ dst, size_t dst_stride,
                                   size_t row, const int32_t* __restrict__ eff) {
    const int i = blockIdx.x, s = eff[i];
    float* d = dst + (size_t)i * dst_stride;
    const float* q = src + (size_t)(s < 0 ? 0 : s) * src_stride;
    for (size_t k = threadIdx.x; k < row; k += kSlotThreads) d[k] = s < 0 ? 0.f : q[k];
}

int launch_gather_rows(const float* src, size_t src_stride, float* dst, size_t dst_stride, size_t row, const int32_t* eff, int n,
                       cudaStream_t st) {
    if (n <= 0) return 0;
    gather_rows_kernel<<<n, kSlotThreads, 0, st>>>(src, src_stride, dst, dst_stride, row, eff);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

// One CTA per item.
__global__ void scatter_init_kernel(const float* __restrict__ tok, float* __restrict__ tmpl, size_t row, const double* __restrict__ boxes,
                                    double* __restrict__ state, const int32_t* __restrict__ status, int32_t* __restrict__ out_status,
                                    const int32_t* __restrict__ eff) {
    const int i = blockIdx.x, s = eff[i];
    if (threadIdx.x == 0 && out_status) out_status[i] = s < 0 ? VT_TRACK_BAD_SLOT_ : status[i];
    if (s < 0) return;
    if (threadIdx.x < 4) state[(size_t)s * 4 + threadIdx.x] = boxes[(size_t)i * 4 + threadIdx.x];
    const float* q = tok + (size_t)i * row;
    float* d = tmpl + (size_t)s * row;
    for (size_t k = threadIdx.x; k < row; k += kSlotThreads) d[k] = q[k];
}

int launch_scatter_init(const float* tok, float* tmpl, size_t row, const double* boxes, double* state, const int32_t* status,
                        int32_t* out_status, const int32_t* eff, int n, cudaStream_t st) {
    if (n <= 0) return 0;
    scatter_init_kernel<<<n, kSlotThreads, 0, st>>>(tok, tmpl, row, boxes, state, status, out_status, eff);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

// Range fallback: one CTA walks the items in tiles of 1024 and appends the flagged ones in item order (ballot + per-warp counts).  A
// real confidence is a clamped sigmoid in [1e-4, 0.9999], so -1 marks a withheld result; crop status 0 and a valid slot leave
// VT_TRACK_NUMERIC_RANGE as its only cause.
constexpr int kCompactThreads = 1024;
__global__ void __launch_bounds__(kCompactThreads)
fallback_compact_kernel(const double* __restrict__ out_boxes, const int32_t* __restrict__ status, const int32_t* __restrict__ eff, int first,
                        const int64_t* __restrict__ frame_offsets, const int32_t* __restrict__ frame_hw, int n, int chunk, RangeFallback fb,
                        int64_t* __restrict__ counter) {
    __shared__ int warp_n[kCompactThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int base = 0;
    for (int i0 = 0; i0 < n; i0 += kCompactThreads) {
        const int i = i0 + (int)threadIdx.x;
        int slot = -1;
        bool flagged = false;
        if (i < n) {
            slot = eff ? eff[i] : first + i;
            flagged = slot >= 0 && status[i] == 0 && out_boxes[(size_t)i * 5 + 4] == -1.0;
        }
        const unsigned b = __ballot_sync(0xffffffffu, flagged);
        if (lane == 0) warp_n[warp] = __popc(b);
        __syncthreads();
        int before = 0, tile = 0;
        for (int k = 0; k < kCompactThreads / 32; ++k) {
            const int c = warp_n[k];
            before += k < warp ? c : 0;
            tile += c;
        }
        if (flagged) {
            const int j = base + before + __popc(b & ((1u << lane) - 1u));
            fb.item[j] = i;
            fb.slot[j] = slot;
            fb.frame_off[j] = frame_offsets[i];
            fb.frame_hw[2 * j] = frame_hw[2 * i];
            fb.frame_hw[2 * j + 1] = frame_hw[2 * i + 1];
        }
        base += tile;
        __syncthreads();                                  // warp_n is rewritten by the next tile
    }
    if (threadIdx.x == 0) {
        fb.count[0] = base;
        for (int k = 0; k * chunk < n; ++k) fb.count[1 + k] = min(max(base - k * chunk, 0), chunk);
        if (counter) *counter += base;
    }
}

int launch_fallback_compact(const double* out_boxes, const int32_t* status, const int32_t* eff, int first, const int64_t* frame_offsets,
                            const int32_t* frame_hw, int n, int chunk, const RangeFallback& fb, int64_t* counter, cudaStream_t st) {
    if (n <= 0) return 0;
    fallback_compact_kernel<<<1, kCompactThreads, 0, st>>>(out_boxes, status, eff, first, frame_offsets, frame_hw, n, chunk, fb, counter);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

// Entries blockIdx.x, blockIdx.x + gridDim.x, ... below the count.
__global__ void fallback_scatter_kernel(RangeFallback fb, int max_tracks, double* __restrict__ out_boxes, double* __restrict__ out_detail,
                                        float* __restrict__ score, float* __restrict__ size, float* __restrict__ offset) {
    const int t = threadIdx.x;
    for (int j = blockIdx.x; j < fb.count[0]; j += gridDim.x) {
        const int i = fb.item[j];
        if (t < 5) out_boxes[(size_t)i * 5 + t] = fb.boxes[(size_t)j * 5 + t];
        if (out_detail && t < 8) out_detail[(size_t)i * 8 + t] = fb.detail[(size_t)j * 8 + t];
        const float* s_score = fb.maps + (size_t)j * 256;
        const float* s_size = fb.maps + (size_t)max_tracks * 256 + (size_t)j * 512;
        const float* s_off = fb.maps + (size_t)max_tracks * 768 + (size_t)j * 512;
        score[(size_t)i * 256 + t] = s_score[t];
        size[(size_t)i * 512 + t] = s_size[t];
        size[(size_t)i * 512 + 256 + t] = s_size[256 + t];
        offset[(size_t)i * 512 + t] = s_off[t];
        offset[(size_t)i * 512 + 256 + t] = s_off[256 + t];
    }
}

int launch_fallback_scatter(const RangeFallback& fb, int max_tracks, double* out_boxes, double* out_detail, float* score, float* size,
                            float* offset, int n, cudaStream_t st) {
    if (n <= 0) return 0;
    static_assert(kSlotThreads == 256, "one thread per map pixel");
    fallback_scatter_kernel<<<counted_rows(n, 1), kSlotThreads, 0, st>>>(fb, max_tracks, out_boxes, out_detail, score, size, offset);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

}  // namespace vt
