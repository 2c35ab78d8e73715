// Generic-configuration path: OstrackDist.forward for ANY member of the vit_dist family (embed dim C, heads, depth,
// head width), used for every configuration other than vit_48_h32 - in particular the widest one (C = 768, 12 heads,
// depth 12, head 256; BASELINE configs[4]).  Same arithmetic as the reference graph:
//   LevitPatchEmbedding   lib/models/vit_dist/vit_dist.py:10-54   conv3x3 s2 + BN(eval, folded) [+ Hardswish] x4
//   OstrackDist.forward   lib/models/vit_dist/vit_dist.py:77-100  pos-embed add, cat(z, x), blocks, LayerNorm
//   timm Block            tracking/onnxexport.py:126-225          LN -> qkv -> MHSA (h heads) -> proj, LN -> fc1 -> GELU -> fc2
//   CenterPredictor       lib/models/layers/head.py:98-201        three conv towers, sigmoid / clamp
// Convolutions are im2col (NHWC, k = (ky, kx, ci)) + one tiled GEMM with a fused bias / activation / residual epilogue;
// attention is two batched GEMMs (batch = track x head) around a row softmax.  The decode is the code the fused head
// kernels use (vt_decode.cuh).  This path favours coverage over speed; the tuned kernels are vit_48_h32's.
// Precision: under blocks_impl "simt" (GenModelW::fp32_only) every GEMM runs on the fp32 CUDA-core kernel (sgemm_kernel).  Otherwise
// the GEMMs whose shapes allow it run on the tensor cores with fp16 hi / lo operand splits (three products: hi*hi + lo*hi + hi*lo),
// gemm_tc_kernel converting fp32 operands per tile and, for C a multiple of 128, gemm_img_kernel reading pre-split images; the rest
// stays on sgemm_kernel.  tests/test_generic_edges.py maps which configuration reaches which kernel.
#include <stdlib.h>
#include <string.h>

#include <thread>
#include <vector>

#include <cuda_fp16.h>

#include "vt_decode.cuh"
#include "vt_internal.h"
#include "vt_tc.cuh"

namespace vt {

namespace {

enum { ACT_NONE = 0, ACT_RELU = 1, ACT_HSWISH = 2, ACT_GELU = 3 };

struct GemmArgs {
    const float* A; const float* B; float* C; const float* bias; const float* R;
    int M, N, K;
    int lda, ldb, ldc, ldr;
    // batch z -> (z / nh, z % nh); element offset of each operand = (z / nh) * s?1 + (z % nh) * s?2
    int nh;
    long long sa1, sa2, sb1, sb2, sc1, sc2, sr1, sr2;
    int rmod;            // > 0: residual row = m % rmod (broadcast over groups of rows, e.g. the positional embedding)
    float alpha;
    int act;
    // optional: write the result as the split image of a matrix with img_K columns instead of C (tensor-core kernel only):
    // element (m, n) of batch z lands at image row z1 * img_rows1 + m, column z2 * img_cols2 + n
    uint8_t* Cimg; int img_K; long long img_rows1; int img_cols2;
    int tile_y0, z0;     // row tile and batch index of blockIdx.y = 0 / blockIdx.z = 0 (launch_pieces)
};

constexpr int kBM = 64, kBN = 64, kBK = 16;

// C[m][n] = act(alpha * sum_k A[m][k] * B(n, k) + bias[n]) + R[m][n];  B(n, k) = B[n * ldb + k] (NN = false) or B[k * ldb + n]
template <bool NN>
__global__ void __launch_bounds__(256) sgemm_kernel(GemmArgs g) {
    __shared__ float As[kBK][kBM + 4];
    __shared__ float Bs[kBK][kBN + 4];
    const int z = blockIdx.z + g.z0, z1 = z / g.nh, z2 = z % g.nh;
    const float* A = g.A + z1 * g.sa1 + z2 * g.sa2;
    const float* B = g.B + z1 * g.sb1 + z2 * g.sb2;
    float* C = g.C + z1 * g.sc1 + z2 * g.sc2;
    const float* R = g.R ? g.R + z1 * g.sr1 + z2 * g.sr2 : nullptr;
    const int m0 = (blockIdx.y + g.tile_y0) * kBM, n0 = blockIdx.x * kBN;
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (int k0 = 0; k0 < g.K; k0 += kBK) {
        {   // A tile: 64 rows x 16 k; thread -> row tid / 4, k (tid % 4) * 4 .. + 3
            const int r = tid >> 2, c = (tid & 3) * 4;
            const int m = m0 + r;
            const float* ap = A + (size_t)m * g.lda + k0 + c;
#pragma unroll
            for (int i = 0; i < 4; ++i) As[c + i][r] = (m < g.M && k0 + c + i < g.K) ? __ldg(ap + i) : 0.f;
        }
        if (!NN) {
            const int r = tid >> 2, c = (tid & 3) * 4;
            const int n = n0 + r;
            const float* bp = B + (size_t)n * g.ldb + k0 + c;
#pragma unroll
            for (int i = 0; i < 4; ++i) Bs[c + i][r] = (n < g.N && k0 + c + i < g.K) ? __ldg(bp + i) : 0.f;
        } else {
            const int kr = tid >> 4, c = (tid & 15) * 4;
            const float* bp = B + (size_t)(k0 + kr) * g.ldb + n0 + c;
#pragma unroll
            for (int i = 0; i < 4; ++i) Bs[kr][c + i] = (k0 + kr < g.K && n0 + c + i < g.N) ? __ldg(bp + i) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < kBK; ++k) {
            const float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
        if (m >= g.M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n >= g.N) continue;
            float v = acc[i][j] * g.alpha;
            if (g.bias) v += __ldg(g.bias + n);
            if (g.act == ACT_RELU) v = v < 0.f ? 0.f : v;      // NaN stays NaN (fmaxf would squash it): the range guard in gen_decode_kernel relies on it
            else if (g.act == ACT_HSWISH) v = hardswish_exact(v);
            else if (g.act == ACT_GELU) v = 0.5f * v * (1.f + erff(v * 0.70710678118654752f));
            if (R) v += R[(size_t)(g.rmod > 0 ? m % g.rmod : m) * g.ldr + n];
            C[(size_t)m * g.ldc + n] = v;
        }
    }
}

// ---- tcgen05 GEMM of the generic path: C = act(A B^T + bias) + R with fp32 operands in global memory ------------------------
// A [M][K] and B [N][K] row-major (torch Linear / flattened conv weight).  A CTA owns a 128 x 128 output tile; four producer
// warps turn 128 x 32 fp32 panels of A and B into fp16 hi | lo images in shared memory (no-swizzle K-major UMMA layout
// [k/8][row][8]: a thread owns one row, so its 16-byte stores are conflict free), one thread issues hi*hi + lo*hi + hi*lo
// tcgen05.mma (M = N = 128, K = 16) into a 128-column fp32 accumulator in TMEM, and the producer warps run the epilogue
// (bias / ReLU / Hardswish / GELU / residual, thread = output row).  kTcStages panels are in flight behind mbarriers.
constexpr int kTcBM = 128, kTcBN = 128, kTcBK = 32, kTcStages = 3;
constexpr int kTcPanel = kTcBM * kTcBK * 2;                 // one operand, one precision: 8192 B
constexpr int kTcStageBytes = 4 * kTcPanel;                 // A hi | A lo | B hi | B lo
constexpr int kTcGemmSmem = kTcStages * kTcStageBytes + 2 * kTcStages * 8 + 8 + 16;      // 2 CTAs per SM
constexpr int kTcGemmThreads = 9 * 32;                      // warps 0-3: A rows, 4-7: B rows (all eight: epilogue), 8: MMA issue

__device__ __forceinline__ void gen_split8(const float4& u, const float4& v, uint4& hi, uint4& lo) {
    tc::split_pack2(u.x, u.y, hi.x, lo.x);
    tc::split_pack2(u.z, u.w, hi.y, lo.y);
    tc::split_pack2(v.x, v.y, hi.z, lo.z);
    tc::split_pack2(v.z, v.w, hi.w, lo.w);
}

template <bool NN>
__global__ void __launch_bounds__(kTcGemmThreads) gemm_tc_kernel(GemmArgs g) {
    extern __shared__ __align__(128) uint8_t gsm[];
    uint64_t* bar_full = reinterpret_cast<uint64_t*>(gsm + kTcStages * kTcStageBytes);     // [stages] panels written (256 arrivals)
    uint64_t* bar_empty = bar_full + kTcStages;                                            // [stages] panels consumed (tcgen05.commit)
    uint64_t* bar_acc = bar_empty + kTcStages;
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bar_acc + 1);
    const int tid = threadIdx.x, warp = tid >> 5;
    const int z = blockIdx.z + g.z0, z1 = z / g.nh, z2 = z % g.nh;
    const float* A = g.A + z1 * g.sa1 + z2 * g.sa2;
    const float* B = g.B + z1 * g.sb1 + z2 * g.sb2;
    float* C = g.C + z1 * g.sc1 + z2 * g.sc2;
    const float* R = g.R ? g.R + z1 * g.sr1 + z2 * g.sr2 : nullptr;
    const int m0 = (blockIdx.y + g.tile_y0) * kTcBM, n0 = blockIdx.x * kTcBN;
    const int ksteps = (g.K + kTcBK - 1) / kTcBK;

    if (warp == 8) tc::tmem_alloc(s_tmem, 128);
    if (tid == 0) {
        for (int i = 0; i < kTcStages; ++i) { tc::mbar_init(bar_full + i, 256); tc::mbar_init(bar_empty + i, 1); }
        tc::mbar_init(bar_acc, 1);
        tc::mbar_fence_init();
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tbase = __shfl_sync(0xffffffffu, *s_tmem, 0);

    if (warp < 8) {
        // ---- producers: thread = one row of the A panel (warps 0-3) or of the B panel (warps 4-7) ----
        const int op = warp >> 2, rloc = tid & 127;
        const int row = (op == 0 ? m0 : n0) + rloc;
        const float* src0 = (op == 0 ? A + (size_t)row * g.lda : B + (size_t)row * g.ldb);
        const bool valid = row < (op == 0 ? g.M : g.N);
#pragma unroll 1
        for (int ks = 0; ks < ksteps; ++ks) {
            const int st = ks % kTcStages;
            const int k0 = ks * kTcBK;
            float4 v[8];
            if (NN && op == 1) {
                // B[k][n]: a warp reads 32 consecutive n of one k row per load (coalesced); the thread still owns operand row n
                const float* bp = B + (size_t)k0 * g.ldb + row;
                float* vf = reinterpret_cast<float*>(v);
#pragma unroll
                for (int j = 0; j < 32; ++j) vf[j] = (valid && k0 + j < g.K) ? __ldg(bp + (size_t)j * g.ldb) : 0.f;
            } else {
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    v[j] = (valid && k0 + 4 * j < g.K) ? __ldg(reinterpret_cast<const float4*>(src0 + k0 + 4 * j)) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            if (ks >= kTcStages) tc::mbar_wait(bar_empty + st, ((ks / kTcStages) - 1) & 1);
            uint8_t* sp = gsm + st * kTcStageBytes + (2 * op) * kTcPanel + rloc * 16;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                uint4 hi, lo;
                gen_split8(v[2 * c], v[2 * c + 1], hi, lo);
                *reinterpret_cast<uint4*>(sp + c * (kTcBM * 16)) = hi;
                *reinterpret_cast<uint4*>(sp + kTcPanel + c * (kTcBM * 16)) = lo;
            }
            tc::fence_async_smem();
            tc::mbar_arrive(bar_full + st);
        }
        // ---- epilogue: thread = output row (TMEM lane 32 (warp % 4) + lane), warps 0-3 columns 0-63, warps 4-7 columns 64-127 ----
        tc::mbar_wait(bar_acc, 0);
        tc::tc_fence_after();
        const int m = m0 + 32 * (warp & 3) + (tid & 31);
        const uint32_t ta = tbase + ((uint32_t)(32 * (warp & 3)) << 16);
#pragma unroll 1
        for (int c0 = 64 * op; c0 < 64 * op + 64; c0 += 16) {
            if (n0 + c0 >= g.N) break;
            uint32_t r[16];
            tc::tmem_ld16(ta + c0, r);
            tc::tc_wait_ld();
            if (m >= g.M) continue;
            if (g.Cimg) {             // plain product (no bias / activation on this route) as a split image: 16 columns = two 8-wide chunks
                const long long ir = (long long)z1 * g.img_rows1 + m;
                const int ic = z2 * g.img_cols2 + n0 + c0;
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    if (n0 + c0 + 8 * c >= g.N) break;
                    uint32_t hi[4], lo[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        tc::split_pack2(__uint_as_float(r[8 * c + 2 * j]) * g.alpha, __uint_as_float(r[8 * c + 2 * j + 1]) * g.alpha, hi[j], lo[j]);
                    *reinterpret_cast<uint4*>(g.Cimg + gen_img_offset(ir, ic / 8 + c, g.img_K, 0)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                    *reinterpret_cast<uint4*>(g.Cimg + gen_img_offset(ir, ic / 8 + c, g.img_K, 1)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                }
                continue;
            }
            float* cp = C + (size_t)m * g.ldc + n0 + c0;
            const float* rp = R ? R + (size_t)(g.rmod > 0 ? m % g.rmod : m) * g.ldr + n0 + c0 : nullptr;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                if (n0 + c0 + j >= g.N) break;
                float v = __uint_as_float(r[j]) * g.alpha;
                if (g.bias) v += __ldg(g.bias + n0 + c0 + j);
                if (g.act == ACT_RELU) v = v < 0.f ? 0.f : v;      // NaN stays NaN (fmaxf would squash it): the range guard in gen_decode_kernel relies on it
                else if (g.act == ACT_HSWISH) v = hardswish_exact(v);
                else if (g.act == ACT_GELU) v = 0.5f * v * (1.f + erff(v * 0.70710678118654752f));
                if (rp) v += rp[j];
                cp[j] = v;
            }
        }
    } else {
        // ---- MMA issue: the warp runs convergently, one elected lane issues ----
        const uint32_t sbase = tc::smem_u32(gsm);
        const uint32_t idesc = tc::instr_desc_f16(128, kTcBN, false);
#pragma unroll 1
        for (int ks = 0; ks < ksteps; ++ks) {
            const int st = ks % kTcStages;
            tc::mbar_wait(bar_full + st, (ks / kTcStages) & 1);
            tc::tc_fence_after();
            const uint32_t pa = sbase + st * kTcStageBytes;
#pragma unroll
            for (int kk = 0; kk < kTcBK / 16; ++kk) {
                const uint32_t off = kk * 2 * (kTcBM * 16);
                const uint64_t ah = tc::smem_desc(pa + off, kTcBM * 16, 128), al = tc::smem_desc(pa + kTcPanel + off, kTcBM * 16, 128);
                const uint64_t bh = tc::smem_desc(pa + 2 * kTcPanel + off, kTcBN * 16, 128), bl = tc::smem_desc(pa + 3 * kTcPanel + off, kTcBN * 16, 128);
                tc::mma_ss_elect(tbase, ah, bh, idesc, (ks | kk) != 0 ? 1u : 0u);
                tc::mma_ss_elect(tbase, al, bh, idesc, 1u);
                tc::mma_ss_elect(tbase, ah, bl, idesc, 1u);
            }
            tc::mma_commit_elect(bar_empty + st);
        }
        tc::mma_commit_elect(bar_acc);
        __syncwarp();
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 8) tc::tmem_dealloc(tbase, 128);
}

bool gemm_tc_ok(const GemmArgs& g, bool nn) {
    auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    if (!(g.K % 8 == 0 && g.K >= 64 && g.N >= 64 && g.M >= 128 && g.lda % 4 == 0 && al16(g.A) && g.sa1 % 4 == 0 && g.sa2 % 4 == 0)) return false;
    return nn || (g.ldb % 4 == 0 && al16(g.B) && g.sb1 % 4 == 0 && g.sb2 % 4 == 0);     // B[k][n] is read with scalar loads
}

// gridDim.y and gridDim.z are limited to 65535 (stem conv1 of the search crop has 256 row tiles per track): a launch takes at most
// that many row tiles and batch entries, and the kernels add tile_y0 / z0.  Every output element is computed by the same thread
// arithmetic whatever the piece, so the split changes no bit.  Returns the number of launches.
constexpr int kMaxGridYZ = 65535;
template <typename Launch>
int launch_pieces(GemmArgs g, int tiles_x, int tiles_y, int batch, Launch launch) {
    int launched = 0;
    for (g.z0 = 0; g.z0 < batch; g.z0 += kMaxGridYZ)
        for (g.tile_y0 = 0; g.tile_y0 < tiles_y; g.tile_y0 += kMaxGridYZ, ++launched)
            launch(g, dim3(tiles_x, min(kMaxGridYZ, tiles_y - g.tile_y0), min(kMaxGridYZ, batch - g.z0)));
    return cudaGetLastError() == cudaSuccess ? launched : -1;
}

template <bool NN>
int launch_gemm_tc(const GemmArgs& g, int batch, cudaStream_t st) {
    static DeviceOnce once;
    if (!ensure_dyn_smem(once, gemm_tc_kernel<NN>, kTcGemmSmem)) return -1;
    return launch_pieces(g, (g.N + kTcBN - 1) / kTcBN, (g.M + kTcBM - 1) / kTcBM, batch,
                         [&](const GemmArgs& p, dim3 grid) { gemm_tc_kernel<NN><<<grid, kTcGemmThreads, kTcGemmSmem, st>>>(p); });
}

// ---- split-image GEMM: C = act(A B^T + bias) + R with BOTH operands already in the tensor cores' shared-memory layout -------------------
// A: image of [M][K] activations (written by layernorm_img_kernel or by a producing GEMM's epilogue), B: image of a [N][K] Linear weight
// (packed once at vt_finalize_weights).  A pipeline stage is two 16 KB bulk copies (cp.async.bulk, one per operand) completing on an
// mbarrier - no thread touches the operands; one warp issues the copies, one the MMAs (hi*hi + lo*hi + hi*lo, M = N = 128, K = 16), eight
// warps run the epilogue.  Output: fp32 row-major (bias / activation / residual) and / or the split image of the result for the next GEMM.
// Against gemm_tc_kernel this removes the fp32 -> fp16 hi/lo conversion of both operands from every tile of every GEMM (the A panel was
// re-converted once per 128 output columns: 18 times for the QKV projection at C = 768).
struct ImgGemmArgs {
    const uint8_t* A; const uint8_t* B;
    int M, N, K;
    float* C; int ldc;
    const float* bias; const float* R; int ldr;
    int act;
    uint8_t* Cimg;          // image of the result (K' = N), or null
    int rmod;               // > 0: residual row = m % rmod (the positional embedding, broadcast over tracks)
    int c_group, c_stride;  // c_group > 0: output row of m = (m / c_group) * c_stride + m % c_group (tokens of a track inside [320][C])
    int tile_y0;            // row tile of blockIdx.y = 0 (run_gemm_img splits the grid like launch_pieces)
};
constexpr int kIgStages = 3;
constexpr int kIgStageBytes = 2 * kImgBlockBytes;                                   // A block | B block
constexpr int kIgSmem = kIgStages * kIgStageBytes + (2 * kIgStages + 1) * 8 + 16;   // 2 CTAs per SM
constexpr int kIgThreads = 10 * 32;                                                 // warps 0-7 epilogue, 8 bulk copies, 9 MMA issue

__global__ void __launch_bounds__(kIgThreads) gemm_img_kernel(ImgGemmArgs g) {
    extern __shared__ __align__(128) uint8_t gsm[];
    uint64_t* bar_full = reinterpret_cast<uint64_t*>(gsm + kIgStages * kIgStageBytes);
    uint64_t* bar_empty = bar_full + kIgStages;
    uint64_t* bar_acc = bar_empty + kIgStages;
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bar_acc + 1);
    const int tid = threadIdx.x, warp = tid >> 5;
    const int ty = blockIdx.y + g.tile_y0, m0 = ty * 128, n0 = blockIdx.x * 128;
    const int ksteps = g.K / 32;
    if (warp == 9) tc::tmem_alloc(s_tmem, 128);
    if (tid == 0) {
        for (int i = 0; i < kIgStages; ++i) { tc::mbar_init(bar_full + i, 2); tc::mbar_init(bar_empty + i, 1); }
        tc::mbar_init(bar_acc, 1);
        tc::mbar_fence_init();
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tbase = __shfl_sync(0xffffffffu, *s_tmem, 0);

    if (warp == 8) {
        // ---- bulk copies: block (row tile, K panel) of each operand, kIgStages in flight ----
        const uint8_t* ab = g.A + (size_t)ty * ksteps * kImgBlockBytes;
        const uint8_t* bb = g.B + (size_t)blockIdx.x * ksteps * kImgBlockBytes;
#pragma unroll 1
        for (int ks = 0; ks < ksteps; ++ks) {
            const int st = ks % kIgStages;
            if (ks >= kIgStages) tc::mbar_wait(bar_empty + st, ((ks / kIgStages) - 1) & 1);
            uint8_t* sp = gsm + st * kIgStageBytes;
            tc::bulk_g2s_elect(sp, ab + (size_t)ks * kImgBlockBytes, kImgBlockBytes, bar_full + st);
            tc::bulk_g2s_elect(sp + kImgBlockBytes, bb + (size_t)ks * kImgBlockBytes, kImgBlockBytes, bar_full + st);
        }
        __syncwarp();
    } else if (warp == 9) {
        // ---- MMA issue ----
        const uint32_t sbase = tc::smem_u32(gsm);
        const uint32_t idesc = tc::instr_desc_f16(128, 128, false);
#pragma unroll 1
        for (int ks = 0; ks < ksteps; ++ks) {
            const int st = ks % kIgStages;
            tc::mbar_wait(bar_full + st, (ks / kIgStages) & 1);
            tc::tc_fence_after();
            const uint32_t pa = sbase + st * kIgStageBytes, pb = pa + kImgBlockBytes;
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
                const uint32_t off = kk * 2 * 2048;
                const uint64_t ah = tc::smem_desc(pa + off, 2048, 128), al = tc::smem_desc(pa + 8192 + off, 2048, 128);
                const uint64_t bh = tc::smem_desc(pb + off, 2048, 128), bl = tc::smem_desc(pb + 8192 + off, 2048, 128);
                tc::mma_ss_elect(tbase, ah, bh, idesc, (ks | kk) != 0 ? 1u : 0u);
                tc::mma_ss_elect(tbase, al, bh, idesc, 1u);
                tc::mma_ss_elect(tbase, ah, bl, idesc, 1u);
            }
            tc::mma_commit_elect(bar_empty + st);
        }
        tc::mma_commit_elect(bar_acc);
        __syncwarp();
    } else {
        // ---- epilogue: thread = output row (TMEM lane), warps 0-3 columns 0-63, warps 4-7 columns 64-127 ----
        tc::mbar_wait(bar_acc, 0);
        tc::tc_fence_after();
        const int half = warp >> 2;
        const int m = m0 + 32 * (warp & 3) + (tid & 31);
        const uint32_t ta = tbase + ((uint32_t)(32 * (warp & 3)) << 16);
#pragma unroll 1
        for (int c0 = 64 * half; c0 < 64 * half + 64; c0 += 16) {
            uint32_t r[16];
            tc::tmem_ld16(ta + c0, r);
            tc::tc_wait_ld();
            if (m >= g.M) continue;
            if (n0 + c0 >= g.N) break;                       // N is a multiple of 16 (tail tile of a 128-column grid)
            float v[16];
            const float* rp = g.R ? g.R + (size_t)(g.rmod > 0 ? m % g.rmod : m) * g.ldr + n0 + c0 : nullptr;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                float x = __uint_as_float(r[j]);
                if (g.bias) x += __ldg(g.bias + n0 + c0 + j);
                if (g.act == ACT_RELU) x = x < 0.f ? 0.f : x;
                else if (g.act == ACT_HSWISH) x = hardswish_exact(x);
                else if (g.act == ACT_GELU) x = 0.5f * x * (1.f + erff(x * 0.70710678118654752f));
                if (rp) x += rp[j];
                v[j] = x;
            }
            if (g.C) {
                const size_t orow = g.c_group > 0 ? (size_t)(m / g.c_group) * g.c_stride + m % g.c_group : (size_t)m;
                float4* cp = reinterpret_cast<float4*>(g.C + orow * g.ldc + n0 + c0);
#pragma unroll
                for (int j = 0; j < 4; ++j) cp[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            }
            if (g.Cimg) {
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    uint32_t hi[4], lo[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) tc::split_pack2(v[8 * c + 2 * j], v[8 * c + 2 * j + 1], hi[j], lo[j]);
                    *reinterpret_cast<uint4*>(g.Cimg + gen_img_offset(m, (n0 + c0) / 8 + c, g.N, 0)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                    *reinterpret_cast<uint4*>(g.Cimg + gen_img_offset(m, (n0 + c0) / 8 + c, g.N, 1)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                }
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 9) tc::tmem_dealloc(tbase, 128);
}

int run_gemm_img(const ImgGemmArgs& g0, cudaStream_t st) {
    if (g0.M <= 0) return 0;
    if (g0.N % 16 != 0 || g0.K % 32 != 0 || (g0.C && (g0.ldc % 4 != 0)) || (g0.Cimg && g0.N % 32 != 0)) return -1;
    static DeviceOnce once;
    if (!ensure_dyn_smem(once, gemm_img_kernel, kIgSmem)) return -1;
    const int tiles_y = (g0.M + 127) / 128;
    int launched = 0;
    ImgGemmArgs g = g0;
    for (g.tile_y0 = 0; g.tile_y0 < tiles_y; g.tile_y0 += kMaxGridYZ, ++launched)
        gemm_img_kernel<<<dim3((g.N + 127) / 128, min(kMaxGridYZ, tiles_y - g.tile_y0)), kIgThreads, kIgSmem, st>>>(g);
    return cudaGetLastError() == cudaSuccess ? launched : -1;
}

// LayerNorm over the last dim C (eps 1e-5), one warp per row (same arithmetic as layernorm_kernel), result written as a split image
__global__ void __launch_bounds__(256) layernorm_img_kernel(const float* __restrict__ in, uint8_t* __restrict__ img, const float* __restrict__ g,
                                                           const float* __restrict__ b, int rows, int C) {
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= rows) return;
    const float* x = in + (size_t)row * C;
    float s = 0.f;
    for (int c = lane; c < C; c += 32) s += x[c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float mean = s / (float)C;
    float v = 0.f;
    for (int c = lane; c < C; c += 32) { const float d = x[c] - mean; v = fmaf(d, d, v); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const float rstd = rsqrtf(v / (float)C + kLnEps);
    for (int c8 = lane; c8 < C / 8; c8 += 32) {
        const float4 x0 = *reinterpret_cast<const float4*>(x + 8 * c8), x1 = *reinterpret_cast<const float4*>(x + 8 * c8 + 4);
        const float4 g0 = __ldg(reinterpret_cast<const float4*>(g + 8 * c8)), g1 = __ldg(reinterpret_cast<const float4*>(g + 8 * c8 + 4));
        const float4 b0 = __ldg(reinterpret_cast<const float4*>(b + 8 * c8)), b1 = __ldg(reinterpret_cast<const float4*>(b + 8 * c8 + 4));
        const float y[8] = {(x0.x - mean) * rstd * g0.x + b0.x, (x0.y - mean) * rstd * g0.y + b0.y, (x0.z - mean) * rstd * g0.z + b0.z,
                            (x0.w - mean) * rstd * g0.w + b0.w, (x1.x - mean) * rstd * g1.x + b1.x, (x1.y - mean) * rstd * g1.y + b1.y,
                            (x1.z - mean) * rstd * g1.z + b1.z, (x1.w - mean) * rstd * g1.w + b1.w};
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) tc::split_pack2(y[2 * j], y[2 * j + 1], hi[j], lo[j]);
        *reinterpret_cast<uint4*>(img + gen_img_offset(row, c8, C, 0)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4*>(img + gen_img_offset(row, c8, C, 1)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    }
}

// fp32 rows [rows][K] (K a multiple of 8) -> split image, thread = (row, 8-wide chunk)
__global__ void __launch_bounds__(256) rows_img_kernel(const float* __restrict__ in, uint8_t* __restrict__ img, long long rows, int K) {
    const int chunks = K / 8;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < rows * chunks; i += (long long)gridDim.x * 256) {
        const long long row = i / chunks;
        const int kc = (int)(i % chunks);
        const float4* p = reinterpret_cast<const float4*>(in + row * K + 8 * kc);
        uint4 hi, lo;
        gen_split8(p[0], p[1], hi, lo);
        *reinterpret_cast<uint4*>(img + gen_img_offset(row, kc, K, 0)) = hi;
        *reinterpret_cast<uint4*>(img + gen_img_offset(row, kc, K, 1)) = lo;
    }
}

int run_gemm(const GemmArgs& g, int batch, bool nn, const GenModelW& w, cudaStream_t st);

}  // namespace

// Host: W[N][K] fp32 (torch Linear weight) -> split image (rows padded to 128 with zeros).  A few threads: 10^8 elements at C = 768.
void gen_pack_weight_image(const float* w, int N, int K, uint8_t* img) {
    const size_t bytes = gen_img_bytes(N, K);
    memset(img, 0, bytes);
    auto work = [&](int n_lo, int n_hi) {
        for (int n = n_lo; n < n_hi; ++n)
            for (int k = 0; k < K; ++k) {
                uint16_t hi, lo;
                tc::split_f16(w[(size_t)n * K + k], &hi, &lo);
                const size_t off = gen_img_offset(n, k / 8, K, 0) + (k % 8) * 2;
                memcpy(img + off, &hi, 2);
                memcpy(img + off + 8192, &lo, 2);
            }
    };
    const int nt = 8;
    std::vector<std::thread> th;
    for (int t = 0; t < nt; ++t) th.emplace_back(work, (int)((long long)N * t / nt), (int)((long long)N * (t + 1) / nt));
    for (auto& t : th) t.join();
}

namespace {

// w.fp32_only (blocks_impl "simt"): every GEMM on the fp32 CUDA-core kernel, no fp16 operand anywhere
int run_gemm(const GemmArgs& g, int batch, bool nn, const GenModelW& w, cudaStream_t st) {
    if (g.M <= 0 || g.N <= 0 || batch <= 0) return 0;
    if (!w.fp32_only && gemm_tc_ok(g, nn)) return nn ? launch_gemm_tc<true>(g, batch, st) : launch_gemm_tc<false>(g, batch, st);
    if (g.Cimg) return -1;                      // the image epilogue exists on the tensor-core kernel only
    return launch_pieces(g, (g.N + kBN - 1) / kBN, (g.M + kBM - 1) / kBM, batch, [&](const GemmArgs& p, dim3 grid) {
        if (nn) sgemm_kernel<true><<<grid, 256, 0, st>>>(p);
        else sgemm_kernel<false><<<grid, 256, 0, st>>>(p);
    });
}

GemmArgs gemm_args(const float* A, int lda, const float* B, int ldb, float* C, int ldc, int M, int N, int K, const float* bias, int act) {
    GemmArgs g{};
    g.A = A; g.B = B; g.C = C; g.bias = bias; g.R = nullptr;
    g.M = M; g.N = N; g.K = K; g.lda = lda; g.ldb = ldb; g.ldc = ldc; g.ldr = 0;
    g.nh = 1; g.alpha = 1.f; g.act = act; g.rmod = 0;
    return g;
}

// 3x3 patches, pad 1: out[(b * Ho + oy) * Wo + ox][(ky * 3 + kx) * Cin + ci] = in(b, stride * oy + ky - 1, stride * ox + kx - 1, ci)
//   NCHW: in[((b * Cin + ci) * H + y) * W + x]      NHWC: in[b * bstride + (y * W + x) * ld + choff + ci]
template <bool NCHW>
__global__ void __launch_bounds__(256) im2col3x3_kernel(const float* __restrict__ in, long long bstride, int ld, int choff, int Cin,
                                                       int H, int W, int stride, int Ho, int Wo, float* __restrict__ out, long long total) {
    const int K = 9 * Cin;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
        const int k = (int)(i % K);
        const long long row = i / K;
        const int ci = k % Cin, tap = k / Cin, ky = tap / 3, kx = tap % 3;
        const int ox = (int)(row % Wo), oy = (int)((row / Wo) % Ho);
        const long long b = row / ((long long)Wo * Ho);
        const int y = stride * oy + ky - 1, x = stride * ox + kx - 1;
        float v = 0.f;
        if (y >= 0 && y < H && x >= 0 && x < W)
            v = NCHW ? __ldg(in + ((b * Cin + ci) * H + y) * W + x) : __ldg(in + b * bstride + ((long long)y * W + x) * ld + choff + ci);
        out[i] = v;
    }
}

// The same patches written as the split image of the [rows][9 Cin] matrix (NHWC input, Cin a multiple of 8: a chunk of 8 consecutive k is
// 8 consecutive channels of one tap): thread = (row, chunk), two 16-byte loads, one 16-byte store per precision.
__global__ void __launch_bounds__(256) im2col3x3_img_kernel(const float* __restrict__ in, long long bstride, int ld, int choff, int Cin, int H, int W,
                                                           int stride, int Ho, int Wo, uint8_t* __restrict__ img, long long rows) {
    const int K = 9 * Cin, chunks = K / 8, cpt = Cin / 8;
    const long long total = (rows + 127) / 128 * 128 * chunks;         // the index space covers whole 128-row tiles; rows beyond `rows` are skipped
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
        // consecutive threads = consecutive rows of one chunk: the image stores of a warp are contiguous
        const long long row = (i / (128LL * chunks)) * 128 + (i % 128);
        const int kc = (int)((i / 128) % chunks);
        if (row >= rows) continue;
        const int tap = kc / cpt, ci = (kc % cpt) * 8, ky = tap / 3, kx = tap % 3;
        const int ox = (int)(row % Wo), oy = (int)((row / Wo) % Ho);
        const long long b = row / ((long long)Wo * Ho);
        const int y = stride * oy + ky - 1, x = stride * ox + kx - 1;
        float4 v0 = make_float4(0.f, 0.f, 0.f, 0.f), v1 = v0;
        if (y >= 0 && y < H && x >= 0 && x < W) {
            const float* p = in + b * bstride + ((long long)y * W + x) * ld + choff + ci;
            v0 = __ldg(reinterpret_cast<const float4*>(p));
            v1 = __ldg(reinterpret_cast<const float4*>(p + 4));
        }
        uint4 hi, lo;
        gen_split8(v0, v1, hi, lo);
        *reinterpret_cast<uint4*>(img + gen_img_offset(row, kc, K, 0)) = hi;
        *reinterpret_cast<uint4*>(img + gen_img_offset(row, kc, K, 1)) = lo;
    }
}

int run_im2col_img(const float* in, long long bstride, int ld, int choff, int Cin, int H, int stride, int n, uint8_t* img, cudaStream_t st) {
    const int Ho = (H + 2 - 3) / stride + 1;
    const long long rows = (long long)n * Ho * Ho, total = (rows + 127) / 128 * 128 * (9 * Cin / 8);
    if (rows <= 0) return 0;
    const int blocks = (int)((total + 255) / 256 < 148 * 32 ? (total + 255) / 256 : 148 * 32);
    im2col3x3_img_kernel<<<blocks, 256, 0, st>>>(in, bstride, ld, choff, Cin, H, H, stride, Ho, Ho, img, rows);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

int run_im2col(bool nchw, const float* in, long long bstride, int ld, int choff, int Cin, int H, int stride, int n, float* out, cudaStream_t st) {
    const int Ho = (H + 2 - 3) / stride + 1;
    const long long total = (long long)n * Ho * Ho * 9 * Cin;
    if (total <= 0) return 0;
    const int blocks = (int)((total + 255) / 256 < 148 * 32 ? (total + 255) / 256 : 148 * 32);
    if (nchw) im2col3x3_kernel<true><<<blocks, 256, 0, st>>>(in, bstride, ld, choff, Cin, H, H, stride, Ho, Ho, out, total);
    else im2col3x3_kernel<false><<<blocks, 256, 0, st>>>(in, bstride, ld, choff, Cin, H, H, stride, Ho, Ho, out, total);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

// LayerNorm over the last dim C (eps 1e-5), one warp per row; two passes over the row (mean, then variance) like torch
__global__ void __launch_bounds__(256) layernorm_kernel(const float* __restrict__ in, float* __restrict__ out, const float* __restrict__ g,
                                                       const float* __restrict__ b, int rows, int C) {
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= rows) return;
    const float* x = in + (size_t)row * C;
    float s = 0.f;
    for (int c = lane; c < C; c += 32) s += x[c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float mean = s / (float)C;
    float v = 0.f;
    for (int c = lane; c < C; c += 32) { const float d = x[c] - mean; v = fmaf(d, d, v); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const float rstd = rsqrtf(v / (float)C + kLnEps);
    float* y = out + (size_t)row * C;
    for (int c = lane; c < C; c += 32) y[c] = (x[c] - mean) * rstd * __ldg(g + c) + __ldg(b + c);
}

// softmax over rows of `cols` values in place, one warp per row
__global__ void __launch_bounds__(256) softmax_rows_kernel(float* __restrict__ s, long long rows, int cols) {
    const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    float* x = s + row * cols;
    float m = -INFINITY;
    for (int c = lane; c < cols; c += 32) m = fmaxf(m, x[c]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float l = 0.f;
    for (int c = lane; c < cols; c += 32) { const float e = expf(x[c] - m); x[c] = e; l += e; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
    const float inv = 1.f / l;
    for (int c = lane; c < cols; c += 32) x[c] *= inv;
}

// out = in * s: the final LayerNorm's tap, scaled back to the model's LayerNorm (GenModelW::norm_tap_scale)
__global__ void __launch_bounds__(256) scale_copy_kernel(const float* __restrict__ in, float* __restrict__ out, long long n, float s) {
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) out[i] = in[i] * s;
}

// raw conv5 outputs [n][256][5] (ctr, offset x, offset y, size w, size h) -> maps, arg-max, boxes, tracker state
// Range guard: the tensor-core GEMMs take fp16 hi + lo operands, so an activation beyond fp16 range becomes inf and then inf / NaN
// downstream.  Two chokepoints catch every such track: the final LayerNorm's output row (`ln_x`, first element: a non-finite input
// makes the whole row NaN) for everything up to the blocks, and the raw conv5 outputs for the head (its ReLUs keep NaN).
__global__ void __launch_bounds__(256) gen_decode_kernel(const float* __restrict__ raw5, HeadArgs a, const float* __restrict__ hann,
                                                        const float* __restrict__ ln_x, int C) {
    __shared__ float maps[6 * 256];
    __shared__ float red[32];
    const int trk = blockIdx.x, tid = threadIdx.x;
    float* m_score = maps; float* m_size = maps + 256; float* m_off = maps + 768; float* m_resp = maps + 1280;
    const float* r = raw5 + ((size_t)trk * 256 + tid) * 5;
    const float sc = sigmoid_clamp(r[0]), sw = sigmoid_clamp(r[3]), sh = sigmoid_clamp(r[4]);
    const float ox = r[1], oy = r[2];
    int bad = 0;
#pragma unroll
    for (int k = 0; k < 5; ++k) bad |= !(fabsf(r[k]) < INFINITY);
    bad |= !(fabsf(__ldg(ln_x + ((size_t)trk * kN + kNz + tid) * C)) < INFINITY);
    m_score[tid] = sc; m_size[tid] = sw; m_size[256 + tid] = sh; m_off[tid] = ox; m_off[256 + tid] = oy;
    m_resp[tid] = __ldg(hann + tid) * sc;
    if (a.score_map) a.score_map[(size_t)trk * 256 + tid] = sc;
    if (a.size_map) { a.size_map[(size_t)trk * 512 + tid] = sw; a.size_map[(size_t)trk * 512 + 256 + tid] = sh; }
    if (a.offset_map) { a.offset_map[(size_t)trk * 512 + tid] = ox; a.offset_map[(size_t)trk * 512 + 256 + tid] = oy; }
    const int any_bad = __syncthreads_or(bad | (a.state && item_slot(a.slots, trk) < 0));
    if (any_bad) {                                   // never a silent wrong answer (see head_finish in vt_head.cu)
        const float qnan = __int_as_float(0x7fc00000);
        if (a.score_map) a.score_map[(size_t)trk * 256 + tid] = qnan;
        if (a.size_map) { a.size_map[(size_t)trk * 512 + tid] = qnan; a.size_map[(size_t)trk * 512 + 256 + tid] = qnan; }
        if (a.offset_map) { a.offset_map[(size_t)trk * 512 + tid] = qnan; a.offset_map[(size_t)trk * 512 + 256 + tid] = qnan; }
    }
    float raw_max, win_max; int raw_idx, win_idx;
    decode_argmax(m_score, m_resp, red, raw_max, raw_idx, win_max, win_idx);
    if (tid == 0) decode_box(a, trk, m_size, m_off, raw_max, raw_idx, win_max, win_idx, any_bad ? VT_TRACK_NUMERIC_RANGE_ : 0);
}

#define GEN_TRY(expr)                      \
    do {                                   \
        const int r__ = (expr);            \
        if (r__ < 0) return r__;           \
        total += r__;                      \
    } while (0)

}  // namespace

// workspace plan for `chunk` tracks; offsets[i] in floats, order = the pointer members of GenWork
size_t gen_work_floats(const GenModelW& w, int chunk, size_t* off) {
    const size_t C = w.C, hc = w.hc, n = chunk;
    const size_t img_rows = ((n * kN + 127) / 128) * 128;
    const size_t sizes[kGenWorkSlots] = {
        n * 3 * kSx * kSx,                                    // crop
        n * 4096 * 9 * (C / 8) > n * 256 * 9 * C ? n * 4096 * 9 * (C / 8) : n * 256 * 9 * C,   // col (largest: conv2 or head conv1; conv1 is 16384 x 27)
        n * 16384 * (C / 8), n * 4096 * (C / 4), n * 1024 * (C / 2),              // act1..3
        n * kNz * C, n * kN * C, n * kN * C, n * kN * 3 * C,                    // tokz, tok, ln, qkv
        n * w.heads * (size_t)kN * kN, n * kN * C, n * kN * 4 * C,              // scores, attn, hid
        n * 256 * 3 * hc, n * 256 * 3 * (hc / 2), n * 256 * 3 * (hc / 4), n * 256 * 3 * (hc / 8), n * 256 * 5,    // t1..t4, raw5
        w.use_img ? img_rows * C : 0, w.use_img ? img_rows * C : 0, w.use_img ? img_rows * 4 * C : 0};           // split images: 4 bytes per element
    size_t tot = 0;
    for (int i = 0; i < kGenWorkSlots; ++i) {
        size_t s = sizes[i];
        if (i == 1 && s < n * 16384 * 27) s = n * 16384 * 27;
        off[i] = tot;
        tot += (s + 63) / 64 * 64;
    }
    return tot;
}

int gen_launch_stem(const float* img, int S, int n, const GenModelW& w, const GenWork& ws, float* tokens, int tok_stride_rows,
                    int tok_off, cudaStream_t st) {
    if (n <= 0) return 0;
    int total = 0;
    const int C = w.C;
    const int ch[5] = {3, C / 8, C / 4, C / 2, C};
    float* acts[3] = {ws.act1, ws.act2, ws.act3};
    int H = S;
    for (int l = 0; l < 4; ++l) {
        const int Ho = H / 2, K = 9 * ch[l];
        if (l > 0 && w.istem_w[l]) {
            // patches written as a split image, weights pre-split: the bulk-copy GEMM (no per-tile operand conversion)
            uint8_t* col_img = reinterpret_cast<uint8_t*>(ws.col);
            GEN_TRY(run_im2col_img(acts[l - 1], (long long)H * H * ch[l], ch[l], 0, ch[l], H, 2, n, col_img, st));
            ImgGemmArgs g{};
            g.A = col_img; g.B = w.istem_w[l]; g.M = n * Ho * Ho; g.N = ch[l + 1]; g.K = K; g.bias = w.stem_b[l];
            if (l < 3) { g.C = acts[l]; g.ldc = ch[l + 1]; g.act = ACT_HSWISH; }
            else {
                g.C = tokens + (size_t)tok_off * C; g.ldc = C; g.act = ACT_NONE;
                g.R = (S == kSx) ? w.pos_x : w.pos_z; g.ldr = C; g.rmod = Ho * Ho;
                g.c_group = Ho * Ho; g.c_stride = tok_stride_rows;
            }
            GEN_TRY(run_gemm_img(g, st));
            H = Ho;
            continue;
        }
        if (l == 0) GEN_TRY(run_im2col(true, img, 0, 0, 0, 3, H, 2, n, ws.col, st));
        else GEN_TRY(run_im2col(false, acts[l - 1], (long long)H * H * ch[l], ch[l], 0, ch[l], H, 2, n, ws.col, st));
        if (l < 3) {
            GemmArgs g = gemm_args(ws.col, K, w.stem_w[l], K, acts[l], ch[l + 1], n * Ho * Ho, ch[l + 1], K, w.stem_b[l], ACT_HSWISH);
            GEN_TRY(run_gemm(g, 1, false, w, st));
        } else {
            // last layer: one GEMM per track (batch), rows = tokens, + positional embedding (broadcast residual)
            GemmArgs g = gemm_args(ws.col, K, w.stem_w[l], K, tokens + (size_t)tok_off * C, C, Ho * Ho, C, K, w.stem_b[l], ACT_NONE);
            g.sa1 = (long long)Ho * Ho * K; g.sc1 = (long long)tok_stride_rows * C;
            g.R = (S == kSx) ? w.pos_x : w.pos_z; g.ldr = C;
            GEN_TRY(run_gemm(g, n, false, w, st));
        }
        H = Ho;
    }
    return total;
}

int gen_launch_blocks_head(float* tokens, int n, const GenModelW& w, const GenWork& ws, const HeadArgs& a, float* taps,
                           size_t tap_stride, cudaStream_t st) {
    if (n <= 0) return 0;
    int total = 0;
    const int C = w.C, hd = C / w.heads, rows = n * kN;
    const size_t tok_bytes = (size_t)rows * C * sizeof(float);
    auto ln = [&](const float* in, float* out, const float* g, const float* b) {
        layernorm_kernel<<<(rows + 7) / 8, 256, 0, st>>>(in, out, g, b, rows, C);
        return cudaGetLastError() == cudaSuccess ? 1 : -1;
    };
    if (taps && cudaMemcpyAsync(taps, tokens, tok_bytes, cudaMemcpyDeviceToDevice, st) != cudaSuccess) return -1;
    uint8_t* img_ln = reinterpret_cast<uint8_t*>(ws.img_ln);
    uint8_t* img_attn = reinterpret_cast<uint8_t*>(ws.img_attn);
    uint8_t* img_hid = reinterpret_cast<uint8_t*>(ws.img_hid);
    auto ln_img = [&](const float* in, const float* g, const float* b) {
        layernorm_img_kernel<<<(rows + 7) / 8, 256, 0, st>>>(in, img_ln, g, b, rows, C);
        return cudaGetLastError() == cudaSuccess ? 1 : -1;
    };
    auto lin = [&](const uint8_t* a_img, const uint8_t* w_img, int N, int K, float* out, const float* bias, int act, const float* resid, uint8_t* out_img) {
        ImgGemmArgs g{};
        g.A = a_img; g.B = w_img; g.M = rows; g.N = N; g.K = K; g.C = out; g.ldc = N; g.bias = bias; g.R = resid; g.ldr = N; g.act = act; g.Cimg = out_img;
        return run_gemm_img(g, st);
    };
    for (int b = 0; b < w.depth; ++b) {
        const GenBlockW& B = w.blk[b];
        if (w.use_img) {
            // Linear layers on the split-image GEMM: LayerNorm and the producing epilogues write the next GEMM's A operand in its
            // shared-memory layout; the attention products (6 % of the block's FLOPs) stay on the converting kernel
            GEN_TRY(ln_img(tokens, B.ln1g, B.ln1b));
            GEN_TRY(lin(img_ln, B.iwqkv, 3 * C, C, ws.qkv, B.bqkv, ACT_NONE, nullptr, nullptr));
            {
                GemmArgs g = gemm_args(ws.qkv, 3 * C, ws.qkv + C, 3 * C, ws.scores, kN, kN, kN, hd, nullptr, ACT_NONE);
                g.nh = w.heads;
                g.sa1 = g.sb1 = (long long)kN * 3 * C; g.sa2 = g.sb2 = hd;
                g.sc1 = (long long)w.heads * kN * kN; g.sc2 = (long long)kN * kN;
                g.alpha = 1.f / sqrtf((float)hd);
                GEN_TRY(run_gemm(g, n * w.heads, false, w, st));
            }
            {
                const long long srows = (long long)n * w.heads * kN;
                softmax_rows_kernel<<<(unsigned)((srows + 7) / 8), 256, 0, st>>>(ws.scores, srows, kN);
                if (cudaGetLastError() != cudaSuccess) return -1;
                ++total;
            }
            {   // attn = P V straight into the image that the output projection reads
                GemmArgs g = gemm_args(ws.scores, kN, ws.qkv + 2 * C, 3 * C, ws.attn, C, kN, hd, kN, nullptr, ACT_NONE);
                g.nh = w.heads;
                g.sa1 = (long long)w.heads * kN * kN; g.sa2 = (long long)kN * kN;
                g.sb1 = (long long)kN * 3 * C; g.sb2 = hd;
                g.sc1 = (long long)kN * C; g.sc2 = hd;
                if (gemm_tc_ok(g, true) && hd % 8 == 0) {          // the image epilogue writes whole 8-column chunks of one head
                    g.Cimg = img_attn; g.img_K = C; g.img_rows1 = kN; g.img_cols2 = hd;
                    GEN_TRY(run_gemm(g, n * w.heads, true, w, st));
                } else {                                            // head width < 64: fp32 P V, then the image
                    GEN_TRY(run_gemm(g, n * w.heads, true, w, st));
                    const long long chunks = (long long)rows * (C / 8);
                    rows_img_kernel<<<(int)((chunks + 255) / 256 < 148 * 32 ? (chunks + 255) / 256 : 148 * 32), 256, 0, st>>>(ws.attn, img_attn, rows, C);
                    if (cudaGetLastError() != cudaSuccess) return -1;
                    ++total;
                }
            }
            GEN_TRY(lin(img_attn, B.iwproj, C, C, tokens, B.bproj, ACT_NONE, tokens, nullptr));
            GEN_TRY(ln_img(tokens, B.ln2g, B.ln2b));
            GEN_TRY(lin(img_ln, B.iwfc1, 4 * C, C, nullptr, B.bfc1, ACT_GELU, nullptr, img_hid));
            GEN_TRY(lin(img_hid, B.iwfc2, C, 4 * C, tokens, B.bfc2, ACT_NONE, tokens, nullptr));
            if (taps && cudaMemcpyAsync(taps + (size_t)(b + 1) * tap_stride, tokens, tok_bytes, cudaMemcpyDeviceToDevice, st) != cudaSuccess) return -1;
            continue;
        }
        GEN_TRY(ln(tokens, ws.ln, B.ln1g, B.ln1b));
        GEN_TRY(run_gemm(gemm_args(ws.ln, C, B.wqkv, C, ws.qkv, 3 * C, rows, 3 * C, C, B.bqkv, ACT_NONE), 1, false, w, st));
        {   // scores[b][h] = (q k^T) * hd^-0.5, batch = track x head
            GemmArgs g = gemm_args(ws.qkv, 3 * C, ws.qkv + C, 3 * C, ws.scores, kN, kN, kN, hd, nullptr, ACT_NONE);
            g.nh = w.heads;
            g.sa1 = g.sb1 = (long long)kN * 3 * C; g.sa2 = g.sb2 = hd;
            g.sc1 = (long long)w.heads * kN * kN; g.sc2 = (long long)kN * kN;
            g.alpha = 1.f / sqrtf((float)hd);
            GEN_TRY(run_gemm(g, n * w.heads, false, w, st));
        }
        {
            const long long srows = (long long)n * w.heads * kN;
            softmax_rows_kernel<<<(unsigned)((srows + 7) / 8), 256, 0, st>>>(ws.scores, srows, kN);
            if (cudaGetLastError() != cudaSuccess) return -1;
            ++total;
        }
        {   // attn[b][:, h] = P V, V = qkv[..., 2C + h hd ...] as [key][hd]
            GemmArgs g = gemm_args(ws.scores, kN, ws.qkv + 2 * C, 3 * C, ws.attn, C, kN, hd, kN, nullptr, ACT_NONE);
            g.nh = w.heads;
            g.sa1 = (long long)w.heads * kN * kN; g.sa2 = (long long)kN * kN;
            g.sb1 = (long long)kN * 3 * C; g.sb2 = hd;
            g.sc1 = (long long)kN * C; g.sc2 = hd;
            GEN_TRY(run_gemm(g, n * w.heads, true, w, st));
        }
        {   // x = x + proj(attn)
            GemmArgs g = gemm_args(ws.attn, C, B.wproj, C, tokens, C, rows, C, C, B.bproj, ACT_NONE);
            g.R = tokens; g.ldr = C;
            GEN_TRY(run_gemm(g, 1, false, w, st));
        }
        GEN_TRY(ln(tokens, ws.ln, B.ln2g, B.ln2b));
        GEN_TRY(run_gemm(gemm_args(ws.ln, C, B.wfc1, C, ws.hid, 4 * C, rows, 4 * C, C, B.bfc1, ACT_GELU), 1, false, w, st));
        {
            GemmArgs g = gemm_args(ws.hid, 4 * C, B.wfc2, 4 * C, tokens, C, rows, C, 4 * C, B.bfc2, ACT_NONE);
            g.R = tokens; g.ldr = C;
            GEN_TRY(run_gemm(g, 1, false, w, st));
        }
        if (taps && cudaMemcpyAsync(taps + (size_t)(b + 1) * tap_stride, tokens, tok_bytes, cudaMemcpyDeviceToDevice, st) != cudaSuccess) return -1;
    }
    GEN_TRY(ln(tokens, ws.ln, w.norm_g, w.norm_b));
    if (taps) {
        const long long m = (long long)rows * C;
        scale_copy_kernel<<<(int)((m + 255) / 256 < 148 * 32 ? (m + 255) / 256 : 148 * 32), 256, 0, st>>>(ws.ln, taps + (size_t)(w.depth + 1) * tap_stride,
                                                                                                           m, w.norm_tap_scale);
        if (cudaGetLastError() != cudaSuccess) return -1;
        ++total;
    }

    // ---- CENTER head on the 16 x 16 search feature map (tokens 64..319 of every track, NHWC) ----
    const int hc = w.hc, prow = n * 256;
    const int co[5] = {C, hc, hc / 2, hc / 4, hc / 8};
    uint8_t* col_img = reinterpret_cast<uint8_t*>(ws.col);
    auto conv_img = [&](const float* in, long long bstride, int ld, int choff, int ci, const uint8_t* wimg, const float* bias, float* out, int ldo, int cn) {
        int r = run_im2col_img(in, bstride, ld, choff, ci, kFeat, 1, n, col_img, st);
        if (r < 0) return r;
        ImgGemmArgs g{};
        g.A = col_img; g.B = wimg; g.M = prow; g.N = cn; g.K = 9 * ci; g.C = out; g.ldc = ldo; g.bias = bias; g.act = ACT_RELU;
        const int r2 = run_gemm_img(g, st);
        return r2 < 0 ? r2 : r + r2;
    };
    if (w.ihead_w1 && (3 * hc) % 16 == 0) GEN_TRY(conv_img(ws.ln + (size_t)kNz * C, (long long)kN * C, C, 0, C, w.ihead_w1, w.head_b1, ws.t1, 3 * hc, 3 * hc));
    else {
        GEN_TRY(run_im2col(false, ws.ln + (size_t)kNz * C, (long long)kN * C, C, 0, C, kFeat, 1, n, ws.col, st));
        GEN_TRY(run_gemm(gemm_args(ws.col, 9 * C, w.head_w1, 9 * C, ws.t1, 3 * hc, prow, 3 * hc, 9 * C, w.head_b1, ACT_RELU), 1, false, w, st));
    }
    float* tbuf[4] = {ws.t1, ws.t2, ws.t3, ws.t4};
    for (int l = 1; l < 4; ++l)
        for (int t = 0; t < 3; ++t) {
            const int ci = co[l], cn = co[l + 1];
            if (w.ihead_w[t][l - 1] && cn % 16 == 0) {
                GEN_TRY(conv_img(tbuf[l - 1], (long long)256 * 3 * ci, 3 * ci, t * ci, ci, w.ihead_w[t][l - 1], w.head_b[t][l - 1], tbuf[l] + t * cn, 3 * cn, cn));
                continue;
            }
            GEN_TRY(run_im2col(false, tbuf[l - 1], (long long)256 * 3 * ci, 3 * ci, t * ci, ci, kFeat, 1, n, ws.col, st));
            GEN_TRY(run_gemm(gemm_args(ws.col, 9 * ci, w.head_w[t][l - 1], 9 * ci, tbuf[l] + t * cn, 3 * cn, prow, cn, 9 * ci, w.head_b[t][l - 1], ACT_RELU), 1, false, w, st));
        }
    {   // conv5 (1x1): tower t -> its columns of raw5 (ctr 0 | offset 1, 2 | size 3, 4)
        const int c4 = co[4];
        const int col0[3] = {0, 1, 3}, outs[3] = {1, 2, 2};
        for (int t = 0; t < 3; ++t)
            GEN_TRY(run_gemm(gemm_args(ws.t4 + t * c4, 3 * c4, w.head_w5 + (size_t)col0[t] * c4, c4, ws.raw5 + col0[t], 5, prow, outs[t], c4,
                                       w.head_b5 + col0[t], ACT_NONE), 1, false, w, st));
    }
    gen_decode_kernel<<<n, 256, 0, st>>>(ws.raw5, a, w.hann, ws.ln, C);
    if (cudaGetLastError() != cudaSuccess) return -1;
    return total + 1;
}

}  // namespace vt
