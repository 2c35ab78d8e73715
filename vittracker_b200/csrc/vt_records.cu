// Track records (include/vittrack_b200.h, vt_tracks_export / vt_tracks_import): one CTA per item copies a track's box and template
// tokens between the handle's state and a self-checking byte image, with 16-byte vector accesses.  The payload checksum is a sum mod
// 2^64, so the CTA reduces it in any order with the same bits.  Nothing here synchronises with the host or allocates.
#include "../../include/vittrack_b200.h"
#include "vt_internal.h"

namespace vt {

constexpr int kRecThreads = 256;
constexpr int kRecRows = kNz;                          // template token rows of a record
constexpr uint64_t kGolden = 0x9E3779B97F4A7C15ull;

__device__ __forceinline__ uint64_t splitmix64(uint64_t z) {
    z += kGolden;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// Checksum terms of payload vector v (words 2v and 2v + 1).
__device__ __forceinline__ uint64_t vec_terms(uint4 x, int v) {
    const uint64_t w0 = (uint64_t)x.x | ((uint64_t)x.y << 32), w1 = (uint64_t)x.z | ((uint64_t)x.w << 32);
    return splitmix64(w0 + (uint64_t)(2 * v) * kGolden) + splitmix64(w1 + (uint64_t)(2 * v + 1) * kGolden);
}

// Sum over the CTA; the result is valid in thread 0.
__device__ __forceinline__ uint64_t cta_sum(uint64_t s, uint64_t* red) {
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    s = 0;
    if (threadIdx.x == 0)
        for (int w = 0; w < kRecThreads / 32; ++w) s += red[w];
    return s;
}

__device__ __forceinline__ int item_track(const RecordArgs& a, int i) {
    return a.slots ? resolve_slot(a.slots, i, a.max_tracks, a.claim) : a.first + i;
}

// Payload vector v of track s: the box (v < 2) or the template tokens.
__device__ __forceinline__ uint4* payload_vec(const RecordArgs& a, int s, int v) {
    return v < 2 ? reinterpret_cast<uint4*>(a.state + (size_t)s * 4) + v
                 : reinterpret_cast<uint4*>(a.tmpl + (size_t)s * kRecRows * a.C) + (v - 2);
}

__global__ void __launch_bounds__(kRecThreads) tracks_export_kernel(RecordArgs a, uint8_t* __restrict__ records) {
    __shared__ int s_track;
    __shared__ uint64_t red[kRecThreads / 32];
    const int i = blockIdx.x;
    const size_t R = VT_TRACK_RECORD_HEADER_BYTES + (size_t)256 * a.C;
    uint4* rec = reinterpret_cast<uint4*>(records + (size_t)i * R);
    if (threadIdx.x == 0) s_track = item_track(a, i);
    __syncthreads();
    const int s = s_track;
    if (threadIdx.x == 0 && a.out_status) a.out_status[i] = s < 0 ? VT_TRACK_BAD_SLOT : VT_TRACK_OK;
    const int nvec = 2 + 16 * a.C;                     // payload: 32 bytes of box + 256 C bytes of tokens
    if (s < 0) {                                       // an all-zero record: magic 0 can never be imported
        for (int v = threadIdx.x; v < 2 + nvec; v += kRecThreads) rec[v] = make_uint4(0, 0, 0, 0);
        return;
    }
    uint64_t sum = 0;
    for (int v = threadIdx.x; v < nvec; v += kRecThreads) {
        const uint4 x = *payload_vec(a, s, v);
        rec[2 + v] = x;
        sum += vec_terms(x, v);
    }
    sum = cta_sum(sum, red);
    if (threadIdx.x == 0) {
        rec[0] = make_uint4(VT_TRACK_RECORD_MAGIC, VT_TRACK_RECORD_VERSION, (uint32_t)a.fingerprint, (uint32_t)(a.fingerprint >> 32));
        rec[1] = make_uint4((uint32_t)a.C, (uint32_t)kRecRows, (uint32_t)sum, (uint32_t)(sum >> 32));
    }
}

// Every check completes before the first write: a rejected record leaves the slot's bytes as they were.
__global__ void __launch_bounds__(kRecThreads) tracks_import_kernel(RecordArgs a, const uint8_t* __restrict__ records) {
    __shared__ int s_track, s_ok;
    __shared__ uint64_t red[kRecThreads / 32];
    const int i = blockIdx.x;
    const size_t R = VT_TRACK_RECORD_HEADER_BYTES + (size_t)256 * a.C;
    const uint4* rec = reinterpret_cast<const uint4*>(records + (size_t)i * R);
    if (threadIdx.x == 0) {
        const int s = item_track(a, i);
        s_track = s;
        if (s >= 0) {
            const uint4 h0 = rec[0], h1 = rec[1];
            const double* box = reinterpret_cast<const double*>(rec + 2);
            const uint64_t fp = (uint64_t)h0.z | ((uint64_t)h0.w << 32);
            bool ok = h0.x == VT_TRACK_RECORD_MAGIC && h0.y == VT_TRACK_RECORD_VERSION && fp == a.fingerprint && h1.x == (uint32_t)a.C &&
                      h1.y == (uint32_t)kRecRows;
            for (int k = 0; k < 4; ++k) ok = ok && isfinite(box[k]);
            s_ok = ok;
        }
    }
    __syncthreads();
    const int s = s_track;
    if (s < 0) {
        if (threadIdx.x == 0 && a.out_status) a.out_status[i] = VT_TRACK_BAD_SLOT;
        return;
    }
    // a record whose C differs from the handle's is rejected above; its payload is still read at this handle's size, which lies inside
    // the n records of R bytes the caller passed
    const int nvec = 2 + 16 * a.C;
    uint64_t sum = 0;
    for (int v = threadIdx.x; v < nvec; v += kRecThreads) sum += vec_terms(rec[2 + v], v);
    sum = cta_sum(sum, red);
    if (threadIdx.x == 0) {
        const uint4 h1 = rec[1];
        const int ok = s_ok && sum == ((uint64_t)h1.z | ((uint64_t)h1.w << 32));
        s_ok = ok;
        if (a.out_status) a.out_status[i] = ok ? VT_TRACK_OK : VT_TRACK_BAD_RECORD;
    }
    __syncthreads();
    if (!s_ok) return;
    for (int v = threadIdx.x; v < nvec; v += kRecThreads) *payload_vec(a, s, v) = rec[2 + v];
}

int launch_tracks_export(const RecordArgs& a, uint8_t* records, int n, cudaStream_t st) {
    if (n <= 0) return 0;
    tracks_export_kernel<<<n, kRecThreads, 0, st>>>(a, records);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

int launch_tracks_import(const RecordArgs& a, const uint8_t* records, int n, cudaStream_t st) {
    if (n <= 0) return 0;
    tracks_import_kernel<<<n, kRecThreads, 0, st>>>(a, records);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

}  // namespace vt
