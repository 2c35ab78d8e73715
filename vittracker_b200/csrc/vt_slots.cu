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

// The winner of each slot reads its own index back and then releases the claim.  A losing item reads the winner's index or the
// released value, neither of which is its own, so the release needs no ordering against it.
__global__ void resolve_slots_kernel(const int32_t* __restrict__ slots, int n, int max_tracks, uint32_t* __restrict__ claim,
                                     int32_t* __restrict__ eff) {
    const int i = blockIdx.x * kSlotThreads + threadIdx.x;
    if (i >= n) return;
    const int s = slots[i];
    int e = -1;
    if (s >= 0 && s < max_tracks && claim[s] == (uint32_t)i) {
        e = s;
        claim[s] = 0xffffffffu;
    }
    eff[i] = e;
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

}  // namespace vt
