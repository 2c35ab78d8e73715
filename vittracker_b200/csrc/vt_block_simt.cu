// K3 (fp32 CUDA-core variant): the three pre-norm ViT blocks of OstrackDist.forward
// (lib/models/vit_dist/vit_dist.py:84,88-89; timm Block restated at tracking/onnxexport.py:126-225):
//   x = x + proj(softmax((q*48^-0.5) k^T) v),  [q;k;v] = qkv(LN(x));   x = x + fc2(GELU_erf(fc1(LN(x))))
// One CTA per track, one thread per token (320 threads).  A token's residual row stays in registers
// across all three blocks; K and V rows live in shared memory and are read with warp-broadcast
// vector loads; weights are staged per phase in shared memory.  This is the numerically plain fp32
// implementation used for bring-up and as the "exact" mode; the tensor-core kernel lives in
// vt_block_tc.cu.
#include "vt_internal.h"

namespace vt {

constexpr int kBlkThreads = kN;        // 320
constexpr int kKvPitch = 100;          // floats per K|V row: 48 K + 48 V + 4 pad (conflict-free float4 row stores)
// phase A region: wqkv[48][144] | bqkv[144] | ln1_g[48] | ln1_b[48]
constexpr int kOffWqkv = 0, kOffBqkv = 6912, kOffLn1g = 7056, kOffLn1b = 7104, kAFloats = 7152;
// phase B region (overlays K/V): wproj[48][48] | bproj | ln2_g | ln2_b | wfc1[48][192] | bfc1[192] | wfc2[192][48] | bfc2
constexpr int kOffWproj = 0, kOffBproj = 2304, kOffLn2g = 2352, kOffLn2b = 2400, kOffWfc1 = 2448,
              kOffBfc1 = 11664, kOffWfc2 = 11856, kOffBfc2 = 21072, kBFloats = 21120;
constexpr int kKvFloats = kN * kKvPitch;   // 32000
static_assert(kBFloats <= kKvFloats, "phase-B weights must fit in the K/V region");
constexpr size_t kBlkSmemBytes = (size_t)(kAFloats + kKvFloats) * sizeof(float);

__device__ __forceinline__ void coop_copy(float* dst, const float* __restrict__ src, int n) {
    for (int i = threadIdx.x * 4; i < n; i += kBlkThreads * 4)
        *reinterpret_cast<float4*>(dst + i) = __ldg(reinterpret_cast<const float4*>(src + i));
}

__device__ __forceinline__ void layer_norm48(const float (&x)[kC], const float* g, const float* b, float (&y)[kC]) {
    float mean = 0.f;
#pragma unroll
    for (int k = 0; k < kC; ++k) mean += x[k];
    mean *= (1.f / kC);
    float var = 0.f;
#pragma unroll
    for (int k = 0; k < kC; ++k) { const float d = x[k] - mean; var = fmaf(d, d, var); }
    const float rstd = rsqrtf(var * (1.f / kC) + kLnEps);
#pragma unroll
    for (int k = 0; k < kC; ++k) y[k] = (x[k] - mean) * rstd * g[k] + b[k];
}

// acc[0..47] = bias[0..47] + sum_k in[k] * W[k][col0 + n],  W row pitch = ldw (weights broadcast from smem)
template <int K>
__device__ __forceinline__ void matvec48(const float (&in)[K], const float* W, int ldw, const float* bias,
                                         float (&acc)[kC]) {
#pragma unroll
    for (int n = 0; n < kC; n += 4) {
        const float4 b4 = *reinterpret_cast<const float4*>(bias + n);
        acc[n] = b4.x; acc[n + 1] = b4.y; acc[n + 2] = b4.z; acc[n + 3] = b4.w;
    }
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const float a = in[k];
#pragma unroll
        for (int n = 0; n < kC; n += 4) {
            const float4 w4 = *reinterpret_cast<const float4*>(W + k * ldw + n);
            acc[n] = fmaf(a, w4.x, acc[n]);
            acc[n + 1] = fmaf(a, w4.y, acc[n + 1]);
            acc[n + 2] = fmaf(a, w4.z, acc[n + 2]);
            acc[n + 3] = fmaf(a, w4.w, acc[n + 3]);
        }
    }
}

// Track trk.
__device__ __forceinline__ void blocks_simt_track(const float* __restrict__ tok_z, int z_stride_rows, const int32_t* __restrict__ z_slots,
                                                  const float* __restrict__ tok_x, int x_stride_rows, float* __restrict__ out, const ModelW& w,
                                                  float* __restrict__ taps, size_t tap_stride, int trk) {
    extern __shared__ __align__(16) float smem[];
    float* sA = smem;
    float* sKV = smem + kAFloats;
    const int i = threadIdx.x;

    // residual row of token i: template tokens first (vit_dist.py:84)
    float x[kC];
    {
        const float* src = (i < kNz) ? tok_z + ((size_t)max(item_slot(z_slots, trk), 0) * z_stride_rows + i) * kC
                                     : tok_x + ((size_t)trk * x_stride_rows + (i - kNz)) * kC;
#pragma unroll
        for (int k = 0; k < kC; k += 4) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(src + k));
            x[k] = v.x; x[k + 1] = v.y; x[k + 2] = v.z; x[k + 3] = v.w;
        }
    }
    if (taps) {
        float* t = taps + ((size_t)trk * kN + i) * kC;
#pragma unroll
        for (int k = 0; k < kC; k += 4) *reinterpret_cast<float4*>(t + k) = make_float4(x[k], x[k + 1], x[k + 2], x[k + 3]);
    }

    const float scale = 0.14433756729740643f;     // 48 ** -0.5 rounded to fp32 (q * self.scale)

#pragma unroll 1
    for (int blk = 0; blk < kDepth; ++blk) {
        const BlockW& bw = w.blk[blk];
        // ---- phase A: stage qkv weights --------------------------------------------------------
        __syncthreads();                                   // previous block finished with smem
        coop_copy(sA + kOffWqkv, bw.wqkv, 6912);
        coop_copy(sA + kOffBqkv, bw.bqkv, 144);
        coop_copy(sA + kOffLn1g, bw.ln1_g, 48);
        coop_copy(sA + kOffLn1b, bw.ln1_b, 48);
        __syncthreads();

        float q[kC];
        {
            float h[kC];
            layer_norm48(x, sA + kOffLn1g, sA + kOffLn1b, h);
            float acc[kC];
            matvec48<kC>(h, sA + kOffWqkv + 48, 144, sA + kOffBqkv + 48, acc);        // K
#pragma unroll
            for (int n = 0; n < kC; n += 4)
                *reinterpret_cast<float4*>(sKV + i * kKvPitch + n) = make_float4(acc[n], acc[n + 1], acc[n + 2], acc[n + 3]);
            matvec48<kC>(h, sA + kOffWqkv + 96, 144, sA + kOffBqkv + 96, acc);        // V
#pragma unroll
            for (int n = 0; n < kC; n += 4)
                *reinterpret_cast<float4*>(sKV + i * kKvPitch + 48 + n) = make_float4(acc[n], acc[n + 1], acc[n + 2], acc[n + 3]);
            matvec48<kC>(h, sA + kOffWqkv, 144, sA + kOffBqkv, q);                    // Q
#pragma unroll
            for (int n = 0; n < kC; ++n) q[n] *= scale;
        }
        __syncthreads();

        // ---- attention over all 320 keys, online softmax in chunks of 8 keys --------------------
        float o[kC];
#pragma unroll
        for (int n = 0; n < kC; ++n) o[n] = 0.f;
        float m = -INFINITY, l = 0.f;
#pragma unroll 1
        for (int j0 = 0; j0 < kN; j0 += 8) {
            float s[8];
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                const float* kr = sKV + (j0 + t) * kKvPitch;
                float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
                for (int n = 0; n < kC; n += 4) {
                    const float4 k4 = *reinterpret_cast<const float4*>(kr + n);
                    a0 = fmaf(q[n], k4.x, a0); a1 = fmaf(q[n + 1], k4.y, a1);
                    a2 = fmaf(q[n + 2], k4.z, a2); a3 = fmaf(q[n + 3], k4.w, a3);
                }
                s[t] = (a0 + a1) + (a2 + a3);
            }
            float mc = s[0];
#pragma unroll
            for (int t = 1; t < 8; ++t) mc = fmaxf(mc, s[t]);
            const float mn = fmaxf(m, mc);
            const float corr = expf(m - mn);             // exp(-inf) = 0 on the first chunk
            l *= corr;
#pragma unroll
            for (int n = 0; n < kC; ++n) o[n] *= corr;
            m = mn;
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                const float p = expf(s[t] - m);
                l += p;
                const float* vr = sKV + (j0 + t) * kKvPitch + 48;
#pragma unroll
                for (int n = 0; n < kC; n += 4) {
                    const float4 v4 = *reinterpret_cast<const float4*>(vr + n);
                    o[n] = fmaf(p, v4.x, o[n]); o[n + 1] = fmaf(p, v4.y, o[n + 1]);
                    o[n + 2] = fmaf(p, v4.z, o[n + 2]); o[n + 3] = fmaf(p, v4.w, o[n + 3]);
                }
            }
        }
        {
            const float inv = 1.f / l;
#pragma unroll
            for (int n = 0; n < kC; ++n) o[n] *= inv;
        }
        __syncthreads();                                   // everyone done reading K/V

        // ---- phase B: stage proj + MLP weights over the K/V region ------------------------------
        float* sB = sKV;
        coop_copy(sB + kOffWproj, bw.wproj, 2304);
        coop_copy(sB + kOffBproj, bw.bproj, 48);
        coop_copy(sB + kOffLn2g, bw.ln2_g, 48);
        coop_copy(sB + kOffLn2b, bw.ln2_b, 48);
        coop_copy(sB + kOffWfc1, bw.wfc1, 9216);
        coop_copy(sB + kOffBfc1, bw.bfc1, 192);
        coop_copy(sB + kOffWfc2, bw.wfc2, 9216);
        coop_copy(sB + kOffBfc2, bw.bfc2, 48);
        __syncthreads();

        {
            float acc[kC];
            matvec48<kC>(o, sB + kOffWproj, 48, sB + kOffBproj, acc);
#pragma unroll
            for (int n = 0; n < kC; ++n) x[n] += acc[n];
        }
        {
            float h[kC];
            layer_norm48(x, sB + kOffLn2g, sB + kOffLn2b, h);
            float y[kC];
#pragma unroll
            for (int n = 0; n < kC; n += 4) {
                const float4 b4 = *reinterpret_cast<const float4*>(sB + kOffBfc2 + n);
                y[n] = b4.x; y[n + 1] = b4.y; y[n + 2] = b4.z; y[n + 3] = b4.w;
            }
#pragma unroll 1
            for (int c = 0; c < kHid / kC; ++c) {
                float hc[kC];
                matvec48<kC>(h, sB + kOffWfc1 + c * kC, kHid, sB + kOffBfc1 + c * kC, hc);
#pragma unroll
                for (int n = 0; n < kC; ++n) hc[n] = 0.5f * hc[n] * (1.f + erff(hc[n] * 0.70710678118654752f));
                const float* W2 = sB + kOffWfc2 + c * kC * kC;
#pragma unroll
                for (int k = 0; k < kC; ++k) {
                    const float a = hc[k];
#pragma unroll
                    for (int n = 0; n < kC; n += 4) {
                        const float4 w4 = *reinterpret_cast<const float4*>(W2 + k * kC + n);
                        y[n] = fmaf(a, w4.x, y[n]); y[n + 1] = fmaf(a, w4.y, y[n + 1]);
                        y[n + 2] = fmaf(a, w4.z, y[n + 2]); y[n + 3] = fmaf(a, w4.w, y[n + 3]);
                    }
                }
            }
#pragma unroll
            for (int n = 0; n < kC; ++n) x[n] += y[n];
        }
        if (taps) {
            float* t = taps + (size_t)(blk + 1) * tap_stride + ((size_t)trk * kN + i) * kC;
#pragma unroll
            for (int k = 0; k < kC; k += 4) *reinterpret_cast<float4*>(t + k) = make_float4(x[k], x[k + 1], x[k + 2], x[k + 3]);
        }
    }
    float* dst = out + ((size_t)trk * kN + i) * kC;
#pragma unroll
    for (int k = 0; k < kC; k += 4) *reinterpret_cast<float4*>(dst + k) = make_float4(x[k], x[k + 1], x[k + 2], x[k + 3]);
}

// Track blockIdx.x; COUNTED (the range fallback of vt_api.cu, whose item count is known on the device only): tracks blockIdx.x,
// blockIdx.x + gridDim.x, ... below *count.
template <bool COUNTED>
__global__ void __launch_bounds__(kBlkThreads, 1)
blocks_simt_kernel(const float* __restrict__ tok_z, int z_stride_rows, const int32_t* __restrict__ z_slots, const float* __restrict__ tok_x,
                   int x_stride_rows, float* __restrict__ out, ModelW w, float* __restrict__ taps,
                   size_t tap_stride, const int32_t* __restrict__ count) {
    if constexpr (COUNTED) {
        for (int trk = blockIdx.x; trk < *count; trk += gridDim.x) {
            blocks_simt_track(tok_z, z_stride_rows, z_slots, tok_x, x_stride_rows, out, w, taps, tap_stride, trk);
            __syncthreads();                                 // the next track restages shared memory
        }
    } else {
        blocks_simt_track(tok_z, z_stride_rows, z_slots, tok_x, x_stride_rows, out, w, taps, tap_stride, blockIdx.x);
    }
}

int launch_blocks_simt(const float* tok_z, int z_stride_rows, const int32_t* z_slots, const float* tok_x, int x_stride_rows,
                       float* out, int n, const ModelW& w, float* taps, size_t tap_stride, cudaStream_t st, const int32_t* count) {
    if (n <= 0) return 0;
    static DeviceOnce once, once_counted;
    if (count) {
        if (!ensure_dyn_smem(once_counted, blocks_simt_kernel<true>, kBlkSmemBytes)) return -1;
        blocks_simt_kernel<true><<<counted_rows(n, 1, 1), kBlkThreads, kBlkSmemBytes, st>>>(tok_z, z_stride_rows, z_slots, tok_x, x_stride_rows, out, w,
                                                                                            taps, tap_stride, count);
        return cudaGetLastError() == cudaSuccess ? 1 : -1;
    }
    if (!ensure_dyn_smem(once, blocks_simt_kernel<false>, kBlkSmemBytes)) return -1;
    blocks_simt_kernel<false><<<n, kBlkThreads, kBlkSmemBytes, st>>>(tok_z, z_stride_rows, z_slots, tok_x, x_stride_rows, out, w, taps, tap_stride, nullptr);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

}  // namespace vt
