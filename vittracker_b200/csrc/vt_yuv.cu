// YUV 4:2:0 (NV12 / I420) -> packed RGB, bit-exact with OpenCV's cvtColor(COLOR_YUV2RGB_NV12 / _I420)
// (modules/imgproc/src/color_yuv.simd.hpp, OpenCV 4.13.0): integer arithmetic with 20 fractional bits,
//     y = max(0, Y - 16) * 1220542
//     R = sat_u8((y + 2^19 + 1673527 (V - 128)) >> 20)
//     G = sat_u8((y + 2^19 -  852492 (V - 128) - 409993 (U - 128)) >> 20)
//     B = sat_u8((y + 2^19 + 2116026 (U - 128)) >> 20)
// and every 2x2 luma block uses its one chroma sample (no interpolation).  Every term fits in int32.
//
// It writes the RGB frames the tracking kernels read; they are unchanged.  Bound: HBM, 1.5 bytes read and 3 written per pixel.
// Three callers: whole contiguous frames, one packed rectangle (the host upload), and per item only the rectangle its crop reads, from
// pitched planes (decoder surfaces), with the rectangle computed on the device from the box (yuv420_crop_to_rgb_kernel).
//
// One work unit = one chroma row (two luma rows) x kSegPx columns of one item; a thread converts a run of two 2x2 blocks (one
// chroma load feeds four pixels).  Sources and destinations may sit at any byte offset: loads are aligned words joined with a
// funnel shift (only words that hold a wanted byte are read), and each output row segment is assembled in shared memory and
// written as aligned words plus single head / tail bytes, so no byte outside the item is touched.
#include "vt_geom.cuh"
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

// The rectangle of a crop (vt_yuv420_crop_to_rgb, vt_yuv420_crops_to_surface_rgb): the box's crop geometry, computed by the code the
// crop kernels run, gives rows [max(0, y1), min(H, y1 + crop_sz)) x columns [max(0, x1 - 1), min(W, x1 + crop_sz + 1)) (sequences.py
// crop_rect), widened to even bounds (tracker.py even_rect): rows [r.y0, r.y1) x columns [r.x0, r.x1).  False: nothing to write
// (degenerate crop, odd or tiny frame, a pitch below its row's width); the box is read only for a well-formed frame.
struct EvenRect { int y0, x0, y1, x1; };

template <int Layout>
__device__ __forceinline__ bool crop_even_rect(const double* bx, double factor, int H, int W, int yp, int cp, EvenRect& r) {
    if (H < 2 || W < 2 || (H & 1) || (W & 1) || yp < W || cp < (Layout == kYuvI420 ? W / 2 : W)) return false;
    const CropGeom g = crop_geometry(bx[0], bx[1], bx[2], bx[3], factor, 1, H, W);
    if (g.status != 0) return false;
    const long long y0 = max(0, g.y1), y1 = min((long long)H, (long long)g.y1 + g.crop_sz);
    const long long x0 = max(0, g.x1 - 1), x1 = min((long long)W, (long long)g.x1 + g.crop_sz + 1);
    if (y1 <= y0 || x1 <= x0) return false;
    r.y0 = (int)y0 & ~1; r.y1 = min(H, (int)(y1 + 1) & ~1); r.x0 = (int)x0 & ~1; r.x1 = min(W, (int)(x1 + 1) & ~1);
    return true;
}

// The descriptor of the even rectangle r inside one picture's planes p (Y, U or UV, V) and its W-wide RGB frame at dst.
template <int Layout>
__device__ __forceinline__ void rect_desc(const uint64_t* p, int yp, int cp, int W, uint8_t* dst, const EvenRect& r, YuvDesc& d) {
    d.y = reinterpret_cast<const uint8_t*>(p[0]) + (int64_t)r.y0 * yp + r.x0;
    d.u = reinterpret_cast<const uint8_t*>(p[1]) + (int64_t)(r.y0 / 2) * cp + (Layout == kYuvI420 ? r.x0 / 2 : r.x0);
    d.v = Layout == kYuvI420 ? reinterpret_cast<const uint8_t*>(p[2]) + (int64_t)(r.y0 / 2) * cp + r.x0 / 2 : d.u;
    d.dst = dst + ((int64_t)r.y0 * W + r.x0) * 3;
    d.y_pitch = yp;
    d.c_pitch = cp;
    d.dst_pitch = (int64_t)W * 3;
    d.w = r.x1 - r.x0; d.h = r.y1 - r.y0;
}

struct YuvCropBatch {
    const uint64_t* planes;                               // [n][3] Y, U (NV12: UV), V
    const int32_t* pitches;                               // [n][2] luma, chroma
    const int32_t* hw;
    const double* boxes;                                  // [n][4]
    double factor;
    uint8_t* dst;
    const int64_t* dst_off;
};

template <int Layout>
__device__ __forceinline__ bool make_crop_desc(const YuvCropBatch& b, int item, YuvDesc& d) {
    const int W = b.hw[2 * item + 1], yp = b.pitches[2 * item], cp = b.pitches[2 * item + 1];
    EvenRect r;
    if (!crop_even_rect<Layout>(b.boxes + 4 * item, b.factor, b.hw[2 * item], W, yp, cp, r)) return false;
    rect_desc<Layout>(b.planes + 3 * item, yp, cp, W, b.dst + b.dst_off[item], r, d);
    return true;
}

// The CTA's share of the item d (units blockIdx.x, blockIdx.x + gridDim.x, ...); no byte outside d's rectangle is written.
template <int Layout>
__device__ __forceinline__ void convert_units(const YuvDesc& d, uint32_t (&s_row)[2][kRowWords]) {
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

template <int Layout>
__global__ void __launch_bounds__(kYuvThreads)
yuv420_to_rgb_kernel(YuvBatch b, YuvDesc one) {
    __shared__ uint32_t s_row[2][kRowWords];
    YuvDesc d;
    if (!make_desc<Layout>(b, one, blockIdx.y, d)) return;
    convert_units<Layout>(d, s_row);
}

// CTAs of an item whose rectangle has fewer units than blockIdx.x exit at once.
template <int Layout>
__global__ void __launch_bounds__(kYuvThreads)
yuv420_crop_to_rgb_kernel(YuvCropBatch b) {
    __shared__ uint32_t s_row[2][kRowWords];
    YuvDesc d;
    if (!make_crop_desc<Layout>(b, blockIdx.y, d)) return;
    convert_units<Layout>(d, s_row);
}

// Shared surfaces (vt_yuv420_crops_to_surface_rgb): pass 1 folds every valid item's rectangle into its surface's bounding rectangle,
// pass 2 converts each surface's bounding rectangle once into the surface's own RGB frame.  An item's crop reads only its own
// rectangle, which lies inside the bounding one, so every track reads the bytes the per-item path would have written for it.
constexpr int kUnionThreads = 256;
constexpr EvenRect kEmptyRect{0x7fffffff, 0x7fffffff, 0, 0};          // also the state of the scratch between calls

// One thread per item.  Every item of a slot list resolves its entry (the winner releases its claim) before anything may skip it.
template <int Layout>
__global__ void __launch_bounds__(kUnionThreads)
yuv420_surface_union_kernel(YuvSurfaceArgs a, int n) {
    const int i = blockIdx.x * kUnionThreads + threadIdx.x;
    if (i >= n) return;
    const int slot = a.slots ? resolve_slot(a.slots, i, a.max_tracks, a.claim) : a.first + i;
    const int s = a.item_surface[i];
    if (slot < 0 || s < 0 || s >= a.m) return;
    const double* bx = a.boxes ? a.boxes + 4 * i : a.state + 4 * (int64_t)slot;
    EvenRect r;
    if (!crop_even_rect<Layout>(bx, a.factor, a.hw[2 * s], a.hw[2 * s + 1], a.pitches[2 * s], a.pitches[2 * s + 1], r)) return;
    int* u = a.rect + 4 * s;                                         // y0, x0: minima; y1, x1: maxima
    atomicMin(u, r.y0);
    atomicMin(u + 1, r.x0);
    atomicMax(u + 2, r.y1);
    atomicMax(u + 3, r.x1);
}

// gridDim.x CTAs per surface (blockIdx.y).  Each CTA reads the bounding rectangle, then counts itself in; the last one to do so empties
// the scratch for the next call.  A surface without a valid item has an empty rectangle: nothing is written.
template <int Layout>
__global__ void __launch_bounds__(kYuvThreads)
yuv420_surface_to_rgb_kernel(YuvSurfaceArgs a, int s0) {
    __shared__ uint32_t s_row[2][kRowWords];
    __shared__ EvenRect s_rect;
    const int s = s0 + blockIdx.y;
    if (threadIdx.x == 0) {
        int* u = a.rect + 4 * s;
        s_rect = EvenRect{u[0], u[1], u[2], u[3]};
        __threadfence();                                              // the read above is complete before this CTA is counted
        if (atomicAdd(a.done + s, 1u) == gridDim.x - 1) {
            u[0] = kEmptyRect.y0; u[1] = kEmptyRect.x0; u[2] = kEmptyRect.y1; u[3] = kEmptyRect.x1;
            a.done[s] = 0;
        }
    }
    __syncthreads();
    const EvenRect r = s_rect;
    if (r.y1 <= r.y0) return;
    const int W = a.hw[2 * s + 1];
    YuvDesc d;
    rect_desc<Layout>(a.planes + 3 * s, a.pitches[2 * s], a.pitches[2 * s + 1], W, a.dst + a.dst_off[s], r, d);
    convert_units<Layout>(d, s_row);
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

int launch_yuv420_crop_to_rgb(int format, const uint64_t* planes, const int32_t* pitches, const int32_t* frame_hw, const double* boxes,
                              double factor, uint8_t* dst, const int64_t* dst_offsets, int n, int num_sms, cudaStream_t st) {
    if (n <= 0) return 0;
    // the rectangles are known on the device only: a fixed number of CTAs per item, as for whole frames, sized for a search crop
    // (a 400 x 402 rectangle of a 100 x 100 box is ~400 units)
    const int per_item = max(1, min(256, num_sms * 32 * 2 / min(n, 32768)));
    int launched = 0;
    for (int first = 0; first < n; first += 32768) {
        const int m = min(32768, n - first);
        const YuvCropBatch b{planes + 3 * first, pitches + 2 * first, frame_hw + 2 * first, boxes + 4 * first, factor, dst,
                             dst_offsets + first};
        const dim3 grid(per_item, m);
        if (format == kYuvNV12) yuv420_crop_to_rgb_kernel<kYuvNV12><<<grid, kYuvThreads, 0, st>>>(b);
        else if (format == kYuvI420) yuv420_crop_to_rgb_kernel<kYuvI420><<<grid, kYuvThreads, 0, st>>>(b);
        else return -1;
        if (cudaPeekAtLastError() != cudaSuccess) return -1;
        ++launched;
    }
    return launched;
}

template <int Layout>
int launch_surfaces(const YuvSurfaceArgs& a, int n, int num_sms, cudaStream_t st) {
    yuv420_surface_union_kernel<Layout><<<(n + kUnionThreads - 1) / kUnionThreads, kUnionThreads, 0, st>>>(a, n);
    if (cudaPeekAtLastError() != cudaSuccess) return -1;
    // a bounding rectangle can be a whole frame: a fixed number of CTAs per surface, as for whole frames
    const int per_surface = max(1, min(4096, num_sms * 32 * 2 / min(max(a.m, 1), 32768)));
    int launched = 1;
    for (int s0 = 0; s0 < a.m; s0 += 32768) {                              // gridDim.y is limited to 65535
        yuv420_surface_to_rgb_kernel<Layout><<<dim3(per_surface, min(32768, a.m - s0)), kYuvThreads, 0, st>>>(a, s0);
        if (cudaPeekAtLastError() != cudaSuccess) return -1;
        ++launched;
    }
    return launched;
}

int launch_yuv420_crops_to_surface_rgb(int format, const YuvSurfaceArgs& a, int n, int num_sms, cudaStream_t st) {
    if (n <= 0) return 0;
    if (format == kYuvNV12) return launch_surfaces<kYuvNV12>(a, n, num_sms, st);
    if (format == kYuvI420) return launch_surfaces<kYuvI420>(a, n, num_sms, st);
    return -1;
}

}  // namespace vt
