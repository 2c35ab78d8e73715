// YUV 4:2:0 (NV12 / I420) -> packed RGB, bit-exact with OpenCV's cvtColor(COLOR_YUV2RGB_NV12 / _I420)
// (modules/imgproc/src/color_yuv.simd.hpp, OpenCV 4.13.0): integer arithmetic with 20 fractional bits,
//     y = max(0, Y - 16) * 1220542
//     R = sat_u8((y + 2^19 + 1673527 (V - 128)) >> 20)
//     G = sat_u8((y + 2^19 -  852492 (V - 128) - 409993 (U - 128)) >> 20)
//     B = sat_u8((y + 2^19 + 2116026 (U - 128)) >> 20)
// and every 2x2 luma block uses its one chroma sample (no interpolation).  Every term fits in int32.
//
// It writes the RGB frames the tracking kernels read; they are unchanged.  Bound: HBM, 1.5 bytes read and 3 written per pixel.
//
// One work unit = one chroma row (two luma rows) x kSegPx columns of one item; a thread converts a run of two 2x2 blocks (one
// chroma load feeds four pixels).  Sources and destinations may sit at any byte offset: loads are aligned words joined with a
// funnel shift (only words that hold a wanted byte are read), and each output row segment is assembled in shared memory and
// written as aligned words plus single head / tail bytes, so no byte outside the item is touched.
#include "vt_internal.h"

namespace vt {

constexpr int kYuvThreads = 64;
constexpr int kYuvPx = 4;                                 // pixels of a row per thread: two 2x2 blocks
constexpr int kSegPx = kYuvThreads * kYuvPx;              // 256 columns per unit
constexpr int kRowWords = kSegPx * 3 / 4 + 1;             // one spare word: the funnel shift reads one past the end

struct YuvBatch {                                         // whole frames: descriptors are formed on the device
    const uint8_t* src;
    const int64_t* src_off;                               // null: the kernel converts `one` instead
    const int32_t* hw;
    uint8_t* dst;
    const int64_t* dst_off;
};

// nbytes (1..4) bytes at p, little-endian in the low bytes; reads only the aligned words that hold one of them
__device__ __forceinline__ uint32_t load_bytes(const uint8_t* p, int nbytes) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const uint32_t* w = reinterpret_cast<const uint32_t*>(a & ~uintptr_t(3));
    const int sh = (int)(a & 3);
    const uint32_t w0 = __ldg(w);
    const uint32_t w1 = sh + nbytes > 4 ? __ldg(w + 1) : 0u;
    return __funnelshift_r(w0, w1, 8 * sh);
}

__device__ __forceinline__ uint32_t sat_u8(int v) { return (uint32_t)min(max(v >> 20, 0), 255); }

template <int Layout>
__device__ __forceinline__ bool make_desc(const YuvBatch& b, const YuvDesc& one, int item, YuvDesc& d) {
    if (b.src_off == nullptr) { d = one; return true; }
    const int H = b.hw[2 * item], W = b.hw[2 * item + 1];
    if (H < 2 || W < 2 || (H & 1) || (W & 1)) return false;
    d.y = b.src + b.src_off[item];
    d.u = d.y + (int64_t)H * W;
    d.v = Layout == kYuvI420 ? d.u + (int64_t)(H / 2) * (W / 2) : d.u;
    d.dst = b.dst + b.dst_off[item];
    d.y_pitch = W;
    d.c_pitch = Layout == kYuvI420 ? W / 2 : W;
    d.dst_pitch = (int64_t)W * 3;
    d.w = W; d.h = H;
    return true;
}

template <int Layout>
__global__ void __launch_bounds__(kYuvThreads)
yuv420_to_rgb_kernel(YuvBatch b, YuvDesc one) {
    __shared__ uint32_t s_row[2][kRowWords];
    YuvDesc d;
    if (!make_desc<Layout>(b, one, blockIdx.y, d)) return;
    const int t = threadIdx.x;
    const int nseg = (d.w + kSegPx - 1) / kSegPx;
    const int units = (d.h / 2) * nseg;
    for (int u = blockIdx.x; u < units; u += gridDim.x) {
        const int r = u / nseg, x0 = (u - r * nseg) * kSegPx;
        const int seg_w = min(kSegPx, d.w - x0);
        const int nb = min(max((seg_w - kYuvPx * t) / 2, 0), 2);       // 2x2 blocks of this thread: 0, 1 or 2
        if (nb > 0) {
            const int px = x0 + kYuvPx * t;
            const uint8_t* yr = d.y + (int64_t)(2 * r) * d.y_pitch + px;
            const uint32_t y0 = load_bytes(yr, 2 * nb), y1 = load_bytes(yr + d.y_pitch, 2 * nb);
            uint32_t uu, vv;                                              // U / V of block j in byte j
            if (Layout == kYuvNV12) {
                const uint32_t c = load_bytes(d.u + (int64_t)r * d.c_pitch + px, 2 * nb);     // U0 V0 U1 V1
                uu = __byte_perm(c, 0, 0x4420);
                vv = __byte_perm(c, 0, 0x4431);
            } else {
                uu = load_bytes(d.u + (int64_t)r * d.c_pitch + px / 2, nb);
                vv = load_bytes(d.v + (int64_t)r * d.c_pitch + px / 2, nb);
            }
            uint32_t rgb[2][3];                                           // per row: 12 bytes, R G B of four pixels
#pragma unroll
            for (int row = 0; row < 2; ++row) {
                const uint32_t yw = row ? y1 : y0;
                uint32_t bytes[12];
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const int U = (int)((uu >> (8 * j)) & 255) - 128, V = (int)((vv >> (8 * j)) & 255) - 128;
                    const int ruv = (1 << 19) + 1673527 * V;
                    const int guv = (1 << 19) - 852492 * V - 409993 * U;
                    const int buv = (1 << 19) + 2116026 * U;
#pragma unroll
                    for (int k = 0; k < 2; ++k) {
                        const int Y = (int)((yw >> (16 * j + 8 * k)) & 255);
                        const int yy = max(0, Y - 16) * 1220542;
                        bytes[6 * j + 3 * k + 0] = sat_u8(yy + ruv);
                        bytes[6 * j + 3 * k + 1] = sat_u8(yy + guv);
                        bytes[6 * j + 3 * k + 2] = sat_u8(yy + buv);
                    }
                }
#pragma unroll
                for (int w = 0; w < 3; ++w)
                    rgb[row][w] = bytes[4 * w] | (bytes[4 * w + 1] << 8) | (bytes[4 * w + 2] << 16) | (bytes[4 * w + 3] << 24);
            }
#pragma unroll
            for (int row = 0; row < 2; ++row)
#pragma unroll
                for (int w = 0; w < 3; ++w) s_row[row][3 * t + w] = rgb[row][w];
        }
        __syncthreads();
        const int L = seg_w * 3;
#pragma unroll
        for (int row = 0; row < 2; ++row) {
            uint8_t* D = d.dst + (int64_t)(2 * r + row) * d.dst_pitch + (int64_t)x0 * 3;
            const int head = min((int)((4 - (reinterpret_cast<uintptr_t>(D) & 3)) & 3), L);
            const int nw = (L - head) >> 2, tail = (L - head) & 3;
            uint32_t* Dw = reinterpret_cast<uint32_t*>(D + head);
            for (int k = t; k < nw; k += kYuvThreads) {
                const int s = head + 4 * k;
                Dw[k] = __funnelshift_r(s_row[row][s >> 2], s_row[row][(s >> 2) + 1], 8 * (s & 3));
            }
            const uint8_t* sb = reinterpret_cast<const uint8_t*>(s_row[row]);
            if (t < head) D[t] = sb[t];
            else if (t >= 4 && t - 4 < tail) D[head + 4 * nw + t - 4] = sb[head + 4 * nw + t - 4];
        }
        __syncthreads();
    }
}

namespace {

int launch(int format, const YuvBatch& b, const YuvDesc& one, dim3 grid, cudaStream_t st) {
    if (format == kYuvNV12) yuv420_to_rgb_kernel<kYuvNV12><<<grid, kYuvThreads, 0, st>>>(b, one);
    else if (format == kYuvI420) yuv420_to_rgb_kernel<kYuvI420><<<grid, kYuvThreads, 0, st>>>(b, one);
    else return -1;
    return cudaPeekAtLastError() == cudaSuccess ? 1 : -1;
}

}  // namespace

int launch_yuv420_to_rgb(int format, const uint8_t* src, const int64_t* src_offsets, const int32_t* frame_hw, uint8_t* dst,
                         const int64_t* dst_offsets, int n, int num_sms, cudaStream_t st) {
    if (n <= 0) return 0;
    // frame sizes live on the device: a fixed number of CTAs per frame, each striding over that frame's units (enough for a few
    // resident waves of 64-thread CTAs over the whole batch)
    const int per_item = max(1, min(4096, num_sms * 32 * 2 / min(n, 32768)));
    int launched = 0;
    for (int first = 0; first < n; first += 32768) {                      // gridDim.y is limited to 65535
        const int m = min(32768, n - first);
        const YuvBatch b{src, src_offsets + first, frame_hw + 2 * first, dst, dst_offsets + first};
        const int k = launch(format, b, YuvDesc{}, dim3(per_item, m), st);
        if (k < 0) return k;
        launched += k;
    }
    return launched;
}

int launch_yuv420_rect(int format, const YuvDesc& d, int num_sms, cudaStream_t st) {
    const int units = (d.h / 2) * ((d.w + kSegPx - 1) / kSegPx);
    if (units <= 0) return 0;
    const YuvBatch b{nullptr, nullptr, nullptr, nullptr, nullptr};
    return launch(format, b, d, dim3(min(units, num_sms * 32), 1), st);
}

}  // namespace vt
