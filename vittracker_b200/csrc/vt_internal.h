// Internal declarations shared by the kernels and the C-ABI layer of libvittrack_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace vt {

// ---- vit_48_h32_noKD dimensions (experiments/vit_dist/vit_48_h32_noKD.yaml) -------------------
constexpr int kC = 48;          // embed dim
constexpr int kNz = 64;         // template tokens (128/16)^2
constexpr int kNx = 256;        // search tokens   (256/16)^2
constexpr int kN = kNz + kNx;   // 320
constexpr int kHid = 192;       // MLP hidden
constexpr int kDepth = 3;
constexpr int kFeat = 16;       // search feature map side
constexpr int kHeadC = 32;      // head tower width
constexpr int kTz = 128;        // template crop side
constexpr int kSx = 256;        // search crop side
constexpr float kLnEps = 1e-5f;
constexpr float kF16Max = 65504.f;           // largest finite fp16: operands of the tensor-core path are fp16 hi + lo
constexpr int VT_TRACK_NUMERIC_RANGE_ = 3;    // == VT_TRACK_NUMERIC_RANGE of include/vittrack_b200.h
constexpr int VT_TRACK_BAD_SLOT_ = 4;         // == VT_TRACK_BAD_SLOT

#ifdef __CUDACC__
// Hardswish exactly as PyTorch evaluates it, x * relu6(x + 3) / 6 (vit_dist.py:41, torch.nn.Hardswish): the product is rounded to fp32 and
// then DIVIDED by 6, correctly rounded.  The division is  q = p r;  q' = fma(fma(-6, q, p), r, q)  with r = fl(1/6): checked over all 2^32
// bit patterns (tools/div6_check.cu) to equal IEEE p / 6.f for every |p| >= 2^-125; below that (subnormal quotients, signed zeros - a
// negative x <= -3 gives p = -0) the IEEE division runs.  4 instructions instead of the ~12 + slow path of a general fp32 division.
__device__ __forceinline__ float div6_exact(float p) {
    const float r = 0.16666667163372039794921875f;
    const float q = __fmul_rn(p, r);
    const float fast = __fmaf_rn(__fmaf_rn(-6.f, q, p), r, q);
    return fabsf(p) >= 1e-36f ? fast : __fdiv_rn(p, 6.f);
}
__device__ __forceinline__ float hardswish_exact(float x) { return div6_exact(__fmul_rn(x, fminf(fmaxf(x + 3.f, 0.f), 6.f))); }

// The same function over N values (N even) with sm_100's packed fp32 arithmetic (add / mul / fma .f32x2: two independent IEEE operations
// per issue slot, SASS FADD2 / FMUL2 / FFMA2) and ONE branch: the fast quotient keeps the sign of a zero product through an OR with the
// product's sign bit (p = -0 for every x <= -3), and the products that need the IEEE division (0 < |p| < 1e-36) only raise a flag; the
// division then runs for the whole group, out of line.  Bit-identical to hardswish_exact per element.
template <int N>
__device__ __forceinline__ void hardswish_exact_n(float (&v)[N]) {
    static_assert(N % 2 == 0, "pairs");
    const uint64_t k3 = 0x4040000040400000ull, kr = 0x3e2aaaab3e2aaaabull, km6 = 0xc0c00000c0c00000ull;   // {3, 3}, {fl(1/6)} x 2, {-6, -6}
    float p[N];
    bool slow = false;
#pragma unroll
    for (int i = 0; i < N; i += 2) {
        uint64_t x, t, pp, q, e, f;
        float t0, t1;
        asm("mov.b64 %0, {%1, %2};" : "=l"(x) : "f"(v[i]), "f"(v[i + 1]));
        asm("add.rn.f32x2 %0, %1, %2;" : "=l"(t) : "l"(x), "l"(k3));
        asm("mov.b64 {%0, %1}, %2;" : "=f"(t0), "=f"(t1) : "l"(t));
        t0 = fminf(fmaxf(t0, 0.f), 6.f);
        t1 = fminf(fmaxf(t1, 0.f), 6.f);
        asm("mov.b64 %0, {%1, %2};" : "=l"(t) : "f"(t0), "f"(t1));
        asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(pp) : "l"(x), "l"(t));
        asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(q) : "l"(pp), "l"(kr));
        asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(e) : "l"(km6), "l"(q), "l"(pp));
        asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(f) : "l"(e), "l"(kr), "l"(q));
        const uint32_t p0 = (uint32_t)pp, p1 = (uint32_t)(pp >> 32);
        p[i] = __uint_as_float(p0);
        p[i + 1] = __uint_as_float(p1);
        v[i] = __uint_as_float((uint32_t)f | (p0 & 0x80000000u));
        v[i + 1] = __uint_as_float((uint32_t)(f >> 32) | (p1 & 0x80000000u));
        // 0 < |p| < 1e-36f (bits 0x03aa2425): shift the sign out, map zero above everything
        slow |= (2u * p0 - 1u) < (2u * 0x03aa2425u - 1u);
        slow |= (2u * p1 - 1u) < (2u * 0x03aa2425u - 1u);
    }
    if (__builtin_expect(slow, 0)) {
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = __fdiv_rn(p[i], 6.f);
    }
}

// Hardswish of the tensor-core stem's epilogues: x * relu6(x + 3) * fl(1/6) - within one ulp of the exactly rounded quotient above (the
// three-term fp16 products these epilogues follow carry 2^-22 already), at a third of the instructions: no correction step, no sign
// fix-up, no branch.
template <int N>
__device__ __forceinline__ void hardswish_n(float (&v)[N]) {
    static_assert(N % 2 == 0, "pairs");
    const uint64_t k3 = 0x4040000040400000ull, kr = 0x3e2aaaab3e2aaaabull;   // {3, 3}, {fl(1/6)} x 2
#pragma unroll
    for (int i = 0; i < N; i += 2) {
        uint64_t x, t, pp;
        float t0, t1;
        asm("mov.b64 %0, {%1, %2};" : "=l"(x) : "f"(v[i]), "f"(v[i + 1]));
        asm("add.rn.f32x2 %0, %1, %2;" : "=l"(t) : "l"(x), "l"(k3));
        asm("mov.b64 {%0, %1}, %2;" : "=f"(t0), "=f"(t1) : "l"(t));
        t0 = fminf(fmaxf(t0, 0.f), 6.f);
        t1 = fminf(fmaxf(t1, 0.f), 6.f);
        asm("mov.b64 %0, {%1, %2};" : "=l"(t) : "f"(t0), "f"(t1));
        asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(pp) : "l"(x), "l"(t));
        asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(pp) : "l"(pp), "l"(kr));
        asm("mov.b64 {%0, %1}, %2;" : "=f"(v[i]), "=f"(v[i + 1]) : "l"(pp));
    }
}
#endif

// ---- packed weights (device, fp32) --------------------------------------------------------------
struct StemLayerW {          // conv3x3 s2 p1 with BN folded
    const float* w;          // [cin][3][3][cout]
    const float* b;          // [cout]
};

struct BlockW {              // timm Block, weights stored K-major ("transposed": [in][out])
    const float *ln1_g, *ln1_b;
    const float *wqkv, *bqkv;      // [48][144], [144]
    const float *wproj, *bproj;    // [48][48], [48]
    const float *ln2_g, *ln2_b;
    const float *wfc1, *bfc1;      // [48][192], [192]
    const float *wfc2, *bfc2;      // [192][48], [48]
};

struct HeadW {               // CENTER head, BN folded, towers ordered ctr, offset, size
    const float *w1, *b1;    // [48][9][96], [96]      (3 towers x 32 merged on the output axis)
    const float *w2, *b2;    // [32][9][3][16], [48]
    const float *w3, *b3;    // [16][9][3][8],  [24]
    const float *w4, *b4;    // [8][9][3][4],   [12]
    const float *w5, *b5;    // [3][4][2] (ctr uses column 0), [3][2]
};

// Tensor-core block kernel operands (vt_block_tc.cu: block_tc_pack): fp16 hi/lo split weights in the UMMA
// no-swizzle K-major layout [k/8][n][8], one bulk-copyable blob per phase, plus fp32 parameters.
constexpr int kTcWaBytes = 2 * (144 * 48 * 2);                         // [Wq; Wk; Wproj Wv] hi|lo = 27648 (the output projection is folded into V)
constexpr int kTcWbBytes = 2 * (192 * 48 * 2) + 2 * (48 * 192 * 2);     // W1 hi|lo, W2 hi|lo     = 73728
constexpr int kStem1TcWBytes = 4 * 512;     // fused stem, conv1 on tcgen05 (vt_stem_fused.cu): [variant 2][K step 2] x (2 chunks x 16 n x 16 B)
constexpr int kStem1TcParFloats = 40;       // bias[4 border variants][8], 2^-s at [32]
constexpr int kTcParFloats = 624;   // ln1_g 48 | ln1_b 48 | bq 48 | bk 48 | Wproj bv 48 | bproj 48 | ln2_g 48 | ln2_b 48 | bfc1 192 | bfc2 48
struct BlockTcW {
    const uint8_t* wa;     // kTcWaBytes
    const uint8_t* wb;     // kTcWbBytes
    const float* par;      // kTcParFloats
};
// One ViT block's tensors as the checkpoint holds them (host memory; Linear weights [out][in])
struct BlockTensors { const float *ln1_g, *ln1_b, *wqkv, *bqkv, *wproj, *bproj, *ln2_g, *ln2_b, *wfc1, *bfc1, *wfc2, *bfc2; };
void block_tc_pack(const BlockTensors& t, uint8_t* wa, uint8_t* wb, float* par);

struct ModelW {
    StemLayerW stem[4];
    BlockW blk[kDepth];
    BlockTcW tc[kDepth];
    const float *norm_g, *norm_b;
    float norm_tap_scale;          // 2^p: the final LayerNorm runs on weights rebalanced by 2^-p (vt_api.cu: rebalance); its tap is scaled back
    const float *pos_z, *pos_x;    // [64][48], [256][48]
    HeadW head;
    const uint8_t* stem_tc_w[3];   // stem conv2 / conv3 / conv4 for tcgen05 (vt_stem_tc.cu): fp16 hi | lo blobs in K-step order
    const float* stem_tc_b[3];     // biases
    const uint8_t* stem1_tc_w;     // stem conv1 for tcgen05 with the pixel normalisation folded in (vt_stem_fused.cu: stem1_tc_pack)
    const float* stem1_tc_par;     // its border-variant biases and scale
    const uint8_t* head_tc_w1;     // head conv1 for tcgen05: 18 pieces (half h, ky, K step) x [hi | lo] x K-major [2 chunks][n = kx*48 + co][8]
    const uint8_t* head_tc_w3;     // head conv3 for tcgen05: 3 blobs (tower) x [hi | lo] x K-major [k/8][n = kx*8 + co, 32][8], k = ky*16 + ci
    const uint8_t* head_tc_w2;     // head conv2 for tcgen05: 3 blobs (tower) x [hi | lo] x K-major [k/8][n = kx*16 + co][8], k = ky*32 + ci
    const float* hann;             // [256] fp32 window (lib/test/utils/hann.py)
    const float* lut;              // [3][256] normalisation table ((v/255 - mean)/std)
};

// ---- tensor-core operand image ("planes") of a stride-2 conv input, written by the producing layer --------
// in[gy][gx][ci] (gy, gx in [0, 2*Wout)) is stored as fp16 hi / lo in 8-channel chunks, split by row / column parity:
//   byte offset = ((((prec * 4 + (gy&1)*2 + (gx&1)) * CCH + ci/8) * (Wout + 1) + (gy>>1) + 1) * Wout + (gx>>1)) * 16 + (ci%8)*2
// Row 0 of every plane is the zero padding above the image (kept zero: nobody writes it).
__host__ __device__ constexpr size_t tc_planes_bytes(int cch, int wout) { return (size_t)2 * 4 * cch * (wout + 1) * wout * 16; }
__host__ __device__ inline size_t tc_planes_offset(int prec, int gy, int gx, int chunk, int cch, int wout) {
    return ((((size_t)(prec * 4 + (gy & 1) * 2 + (gx & 1)) * cch + chunk) * (wout + 1) + (gy >> 1) + 1) * wout + (gx >> 1)) * 16;
}
constexpr int kConv2Cch = 1, kConv2Wout = 64;     // conv2 input:  6 channels -> 1 chunk, 128x128 -> planes of 65 x 64
constexpr int kConv3Cch = 2, kConv3Wout = 32;     // conv3 input: 12 channels -> 2 chunks, 64x64 -> planes of 33 x 32
constexpr int kConv4Cch = 3, kConv4Wout = 16;     // conv4 input: 24 channels -> 3 chunks, 32x32 -> planes of 17 x 16

// ---- per-device one-off kernel configuration ------------------------------------------------------
// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) applies to the CURRENT device only, and one process may hold handles on
// several GPUs (VtConfig.device): every launcher keeps one flag per device ordinal instead of one per process.
constexpr int kMaxDevices = 64;
struct DeviceOnce {
    bool done[kMaxDevices] = {};
    // returns the current device ordinal if its flag is still clear (the caller configures, then calls set()), -1 if already
    // configured, -2 on a CUDA error; ordinals beyond the table are configured on every launch
    int pending() const {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return -2;
        return (dev >= 0 && dev < kMaxDevices && done[dev]) ? -1 : dev;
    }
    void set(int dev) { if (dev >= 0 && dev < kMaxDevices) done[dev] = true; }
};
template <typename Kern>
inline bool ensure_dyn_smem(DeviceOnce& once, Kern kern, size_t bytes) {
    const int dev = once.pending();
    if (dev == -1) return true;
    if (dev == -2) return false;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess) return false;
    once.set(dev);
    return true;
}

// Resident CTAs per SM of a persistent kernel, from the kernel's own resource use and the device limits (registers are allocated per
// warp in units of 256; 1 KB of shared memory per CTA is reserved by the driver; TMEM has 512 columns per SM).  Computed by hand:
// cudaOccupancyMaxActiveBlocksPerMultiprocessor answers 1 for these kernels on this driver although two (or more) CTAs are resident
// (Nsight Compute's launch limits agree with the arithmetic below) - and a persistent grid sized from it ran one CTA per SM.
template <typename Kern>
inline int resident_ctas_per_sm(Kern kern, int threads, size_t dyn_smem, int tmem_cols, int dev) {
    cudaFuncAttributes fa;
    if (cudaFuncGetAttributes(&fa, kern) != cudaSuccess) return 1;
    int regs_sm = 65536, smem_sm = 233472, thr_sm = 2048, blk_sm = 32;
    cudaDeviceGetAttribute(&regs_sm, cudaDevAttrMaxRegistersPerMultiprocessor, dev);
    cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev);
    cudaDeviceGetAttribute(&thr_sm, cudaDevAttrMaxThreadsPerMultiProcessor, dev);
    cudaDeviceGetAttribute(&blk_sm, cudaDevAttrMaxBlocksPerMultiprocessor, dev);
    const int warps = (threads + 31) / 32;
    const int regs_warp = (fa.numRegs * 32 + 255) / 256 * 256;
    int k = blk_sm;
    if (regs_warp > 0) k = min(k, regs_sm / (regs_warp * warps));
    k = min(k, (int)(smem_sm / (dyn_smem + fa.sharedSizeBytes + 1024)));
    k = min(k, thr_sm / (warps * 32));
    if (tmem_cols > 0) k = min(k, 512 / tmem_cols);
    return k < 1 ? 1 : k;
}

// RAII: make `device` current for the duration of a C-ABI call and restore the caller's device afterwards (the host
// language's runtime - PyTorch - keeps its own notion of the current device).
struct DeviceGuard {
    int prev = -1;
    cudaError_t err = cudaSuccess;
    explicit DeviceGuard(int device) {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != device) err = cudaSetDevice(device); else if (err == cudaSuccess) prev = -1;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};

// Grid rows of a kernel that strides over a device-side item count (the range fallback of vt_api.cu), `tiles` CTAs per item: about
// ctas_per_sm CTAs per SM in all (a grid that costs little when the count is 0), at least 1 and at most n.
inline int counted_rows(int n, int tiles, int ctas_per_sm = 4) {
    static int sms[kMaxDevices] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) dev = -1;
    int s = dev >= 0 ? sms[dev] : 0;
    if (s == 0) {
        if (cudaDeviceGetAttribute(&s, cudaDevAttrMultiProcessorCount, dev < 0 ? 0 : dev) != cudaSuccess || s <= 0) s = 148;
        if (dev >= 0) sms[dev] = s;
    }
    const int rows = ctas_per_sm * s / tiles;
    return rows < 1 ? 1 : rows > n ? n : rows;
}

// ---- kernel launchers (each returns the number of kernels it launched, or <0 on a CUDA error) -----
// YUV 4:2:0 -> RGB (vt_yuv.cu).  One work item: an even w x h image whose luma rows are y_pitch apart and whose chroma rows
// (one per two luma rows) are c_pitch apart; NV12 reads interleaved U V pairs at u, I420 reads U at u and V at v.
constexpr int kYuvNV12 = 1, kYuvI420 = 2;
struct YuvDesc {
    const uint8_t* y;
    const uint8_t* u;
    const uint8_t* v;
    uint8_t* dst;                  // w x h x 3 RGB, rows dst_pitch apart
    int64_t y_pitch, c_pitch, dst_pitch;
    int32_t w, h;
};
// n whole frames laid out as cv2.cvtColor takes them ((H*3/2) x W, pitch W); items whose H or W is odd or < 2 are skipped.
int launch_yuv420_to_rgb(int format, const uint8_t* src, const int64_t* src_offsets, const int32_t* frame_hw, uint8_t* dst,
                         const int64_t* dst_offsets, int n, int num_sms, cudaStream_t st);
int launch_yuv420_rect(int format, const YuvDesc& d, int num_sms, cudaStream_t st);
// Per item, only the even-widened rectangle the crop of boxes[i] (factor) reads, from pitched planes (planes [n][3] device addresses
// Y, U or UV, V; pitches [n][2] luma, chroma) into the H x W x 3 frame at dst + dst_offsets[i]; degenerate crops, odd or tiny sizes
// and pitches below the row width are skipped.
int launch_yuv420_crop_to_rgb(int format, const uint64_t* planes, const int32_t* pitches, const int32_t* frame_hw, const double* boxes,
                              double factor, uint8_t* dst, const int64_t* dst_offsets, int n, int num_sms, cudaStream_t st);
// Shared surfaces: items [0, n) on m surfaces.  Item i's box is boxes[i], or the state of track slots[i] / first + i; it is skipped for a
// surface index outside [0, m), a bad slot (outside [0, max_tracks) or repeating an earlier item's: the list is claimed first, with
// launch_claim_slots) or a rectangle launch_yuv420_crop_to_rgb would skip.  Each surface's frame at dst + dst_off[s] gets the bounding
// rectangle of its valid items' rectangles.  rect [m][4] int32 (y0, x0: minima; y1, x1: maxima) and done [m] are the handle's scratch,
// empty between calls ({INT32_MAX, INT32_MAX, 0, 0} and 0).  Launches: one union pass, then one conversion per 32768 surfaces.
struct YuvSurfaceArgs {
    const uint64_t* planes;                               // [m][3] Y, U (NV12: UV), V
    const int32_t* pitches;                               // [m][2] luma, chroma
    const int32_t* hw;                                    // [m][2]
    int m;
    const int32_t* item_surface;                          // [n]
    const double* boxes;                                  // [n][4] or null: the state
    const double* state;                                  // [max_tracks][4]
    const int32_t* slots;                                 // [n] or null: tracks first + i
    uint32_t* claim;
    int first, max_tracks;
    double factor;
    uint8_t* dst;
    const int64_t* dst_off;                               // [m]
    int32_t* rect;
    uint32_t* done;
};
int launch_yuv420_crops_to_surface_rgb(int format, const YuvSurfaceArgs& a, int n, int num_sms, cudaStream_t st);

// Slot lists (the vt_tracks_*_slots entry points): a kernel that reads per-track state takes `slots` (nullable).  Item i reads the
// state of track slots[i], or of track i of the pre-offset state pointer when slots == NULL (the range calls); a negative slot is a
// bad entry (VT_TRACK_BAD_SLOT): its state is not read or written.
__host__ __device__ inline int item_slot(const int32_t* slots, int item) { return slots ? slots[item] : item; }

int launch_crop_normalize(const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw,
                          const double* boxes, const int32_t* slots, double factor, int S, int n, const float* lut,
                          float* out_nchw, uint8_t* out_u8, uint8_t* out_mask, double* out_rf,
                          int32_t* out_status, cudaStream_t st);

// Stem on `n` images of side S (128 or 256): in NCHW fp32 -> tokens[(b*tok_stride) + tok_off + t][48] (+pos).
// scratch must hold n * stem_scratch_floats(S) floats and be zero-initialised once (the tensor-core path keeps zero rows in it).
size_t stem_scratch_floats(int S);
// planes (tensor-core path only): zero-initialised buffer of plane_tracks * tc_planes_bytes_per_track() bytes
int launch_stem(const float* img, int S, int n, const ModelW& w, float* scratch, float* tokens,
                int tok_stride_rows, int tok_off, uint8_t* planes, int plane_tracks, cudaStream_t st);
// Search-branch conv2 + conv3 + conv4 on the tensor cores, for launch_stem: planes2 is conv2's operand image (written by conv1), planes3
// and planes4 receive conv3's and conv4's
int launch_stem234_tc(const uint8_t* planes2, int n, const ModelW& w, uint8_t* planes3, uint8_t* planes4, float* tokens,
                      int tok_stride_rows, int tok_off, cudaStream_t st);
__host__ __device__ constexpr size_t tc_planes_bytes_per_track() {
    return tc_planes_bytes(kConv2Cch, kConv2Wout) + tc_planes_bytes(kConv3Cch, kConv3Wout) + tc_planes_bytes(kConv4Cch, kConv4Wout);
}
// conv3 + conv4 only (the fused front kernel has written planes3)
int launch_stem34_tc(const uint8_t* planes3, int n, const ModelW& w, uint8_t* planes4, float* tokens, int tok_stride_rows, int tok_off,
                     cudaStream_t st);
// Fused front of the search-branch stem (vt_stem_fused.cu): tap tables + crop gather -> conv1 -> conv2 on tcgen05 -> planes3
int launch_crop_stem12_fused(const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw, const double* boxes,
                             const int32_t* slots, double factor, int n, const ModelW& w, int32_t* out_status, void* tap_tables, uint8_t* planes3, cudaStream_t st);
void stem1_tc_pack(const float* wf, const float* bf, uint8_t* blob, float* par);
size_t stem_tc_weight_bytes(int layer);
void stem_tc_pack_weights(int cin, int cch, int cout, int npad, const float* wf, uint8_t* hi8, uint8_t* lo8);

// Crop + stem straight from raw uint8 frames (the first conv layer gathers its tile from the frame).
// count (device, nullable): only items below *count are processed; given, the stem runs on the fp32 CUDA-core kernels whatever `planes`.
int launch_crop_stem(const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw, const double* boxes,
                     const int32_t* slots, double factor, int S, int n, const ModelW& w, float* scratch, float* tokens, int tok_stride_rows,
                     int tok_off, int32_t* out_status, uint8_t* planes, int plane_tracks, void* tap_tables, cudaStream_t st,
                     const int32_t* count = nullptr);
size_t crop_taps_bytes(int n);      // size of the tap-table buffer launch_crop_stem needs for n tracks

// ViT blocks (fp32 SIMT): tokens_z [n][64][48] (stride z_stride rows per track; item i reads row block item_slot(z_slots, i), a negative
// slot reads block 0), tokens_x likewise (by item); in place
// result written to out [n][320][48]; taps (or null) receives [depth][n][320][48].  count (device, nullable): only items below *count.
int launch_blocks_simt(const float* tok_z, int z_stride_rows, const int32_t* z_slots, const float* tok_x, int x_stride_rows,
                       float* out, int n, const ModelW& w, float* taps, size_t tap_stride, cudaStream_t st, const int32_t* count = nullptr);

// ViT blocks on the tcgen05 tensor cores (fp16 hi/lo split operands, fp32 accumulation in TMEM).
int launch_blocks_tc(const float* tok_z, int z_stride_rows, const int32_t* z_slots, const float* tok_x, int x_stride_rows,
                     float* out, int n, const ModelW& w, float* taps, size_t tap_stride, int num_sms, int scores_terms, cudaStream_t st);

struct HeadArgs {
    const float* tokens;      // [n][320][48] block output (pre final-norm)
    int n;
    // forward outputs (nullable)
    float *pred_boxes, *score_map, *size_map, *offset_map;   // [n][4], [n][256], [n][2][256], [n][2][256]
    float* tokens_norm;       // [n][320][48] tap (nullable)
    // tracker outputs (nullable as a group: enabled when state != nullptr)
    double* state;            // [n][4] previous boxes, updated in place when update_state; item i's is row item_slot(slots, i)
    const int32_t* slots;     // [n] or null (see item_slot); a negative slot: maps NaN, status VT_TRACK_BAD_SLOT, state untouched
    const int32_t* frame_hw;  // [n][2]
    const int32_t* status;    // [n] VT_TRACK_* from the crop stage (nullable)
    double* out_boxes;        // [n][5]
    double* out_detail;       // [n][8] (nullable)
    int update_state;
    double search_factor;
    int use_tc;               // first (48 -> 96) convolution on the tcgen05 tensor cores
};
// count (device, nullable; CUDA-core head only, use_tc == 0): only items below *count are processed.
int launch_head(const HeadArgs& a, const ModelW& w, cudaStream_t st, const int32_t* count = nullptr);
// Weights of the tensor-core head (vt_head.cu): blob sizes (0: conv1, 1: conv2, 2: conv3) and the host packer that fills them from
// the folded HeadW layouts w1, w2, w3.
size_t head_tc_weight_bytes(int layer);
void head_tc_pack(const float* w1, const float* w2, const float* w3, uint8_t* blob1, uint8_t* blob2, uint8_t* blob3);

int launch_cal_bbox(const float* score, const float* size_map, const float* offset_map, int n, float* boxes,
                    cudaStream_t st);

// ---- generic-configuration path (vt_generic.cu): any embed dim / heads / depth / head width of the vit_dist family ----
// (BASELINE configs[4]: the widest config, C = 768, 12 heads, depth 12, head 256).  im2col + tiled GEMM (fp32 CUDA cores, or
// tensor cores with fp16 hi / lo splits unless fp32_only) with fused bias / activation / residual epilogues, LayerNorm, softmax,
// and the shared decode.  Activations are NHWC
// (= token-major), weights keep the reference's [out][in] layout (conv: [cout][ky][kx][cin], BN folded).
constexpr int kGenMaxDepth = 32;
struct GenBlockW {
    const float *ln1g, *ln1b, *wqkv, *bqkv, *wproj, *bproj, *ln2g, *ln2b, *wfc1, *bfc1, *wfc2, *bfc2;
    const uint8_t *iwqkv, *iwproj, *iwfc1, *iwfc2;           // split images of the four Linear weights (GenModelW::use_img), else null
};
// "Split image" of a K-major GEMM operand X[rows][K] (vt_generic.cu, gemm_img_kernel): fp16 hi | lo in the UMMA no-swizzle layout, one
// contiguous 16 KB block per (128-row tile, 32-wide K panel) so that a pipeline stage is ONE bulk copy per operand:
//   byte offset of (r, k, prec) = (((r / 128) * (K / 32) + k / 32) * 2 + prec) * 8192 + ((k / 8) % 4) * 2048 + (r % 128) * 16 + (k % 8) * 2
constexpr int kImgBlockBytes = 2 * 4 * 128 * 16;
__host__ __device__ inline size_t gen_img_bytes(long long rows, int K) { return (size_t)((rows + 127) / 128) * (K / 32) * kImgBlockBytes; }
__host__ __device__ inline size_t gen_img_offset(long long r, int kchunk, int K, int prec) {      // kchunk = k / 8
    return (((size_t)(r >> 7) * (K >> 5) + (kchunk >> 2)) * 2 + prec) * 8192 + (size_t)(kchunk & 3) * 2048 + (size_t)(r & 127) * 16;
}
void gen_pack_weight_image(const float* w, int N, int K, uint8_t* img);     // host: W[N][K] fp32 -> split image
struct GenModelW {
    int C, heads, depth, hc;
    int use_img;                                             // Linear layers of the blocks on the split-image GEMM (C % 128 == 0)
    int fp32_only;                                           // blocks_impl "simt": every GEMM on the fp32 CUDA-core kernel
    const float* stem_w[4]; const float* stem_b[4];          // [cout][9 cin], [cout]
    GenBlockW blk[kGenMaxDepth];
    const float *norm_g, *norm_b, *pos_z, *pos_x;
    float norm_tap_scale;                                    // as ModelW::norm_tap_scale
    const float* head_w1; const float* head_b1;              // three towers merged: [3 hc][9 C], [3 hc]  (ctr | offset | size)
    const float* head_w[3][3]; const float* head_b[3][3];    // [tower][layer 2..4]: [co][9 ci], [co]
    const float* head_w5; const float* head_b5;              // [5][hc / 8] rows ctr, offset x, offset y, size w, size h; [5]
    const float* hann;
    // split images of the convolution weights ([cout][9 cin] as a [N][K] matrix) for the layers whose cin is a multiple of 32, else null
    const uint8_t* istem_w[4]; const uint8_t* ihead_w1; const uint8_t* ihead_w[3][3];
};
struct GenWork {             // device scratch for `chunk` tracks
    int chunk;
    float *crop, *col, *act1, *act2, *act3, *tokz, *tok, *ln, *qkv, *scores, *attn, *hid, *t1, *t2, *t3, *t4, *raw5;
    float *img_ln, *img_attn, *img_hid;                      // split images (bytes = 4 per element, rows padded to 128) when use_img
};
constexpr int kGenWorkSlots = 20;
size_t gen_work_floats(const GenModelW& w, int chunk, size_t* offsets /*[kGenWorkSlots]*/);
// Stem of n images (NCHW fp32, side S) -> tokens[(b * tok_stride_rows + tok_off + t)][C] (+ pos)
int gen_launch_stem(const float* img, int S, int n, const GenModelW& w, const GenWork& ws, float* tokens, int tok_stride_rows,
                    int tok_off, cudaStream_t st);
// Blocks (in place on tokens [n][320][C]) + final LayerNorm (-> ws.ln) + head + decode.  taps: [depth + 2][n][320][C] or null.
int gen_launch_blocks_head(float* tokens, int n, const GenModelW& w, const GenWork& ws, const HeadArgs& a, float* taps,
                           size_t tap_stride, cudaStream_t st);

// ---- slot lists (vt_slots.cu) ---------------------------------------------------------------------
// slots [n] as the caller gave them -> eff [n]: the slot, or -1 for an entry outside [0, max_tracks) or repeating an earlier item's.
// claim: [max_tracks] uint32, all 0xffffffff between calls (the second kernel restores what the first changed).
int launch_resolve_slots(const int32_t* slots, int n, int max_tracks, uint32_t* claim, int32_t* eff, cudaStream_t st);
// Its first kernel alone: every valid entry claims its slot.  A kernel that runs next on the stream resolves item i with resolve_slot.
int launch_claim_slots(const int32_t* slots, int n, int max_tracks, uint32_t* claim, cudaStream_t st);
#ifdef __CUDACC__
// Item i's effective slot after the claim, or -1; the winner releases its claim.  A losing item reads the winner's index or the released
// value, neither of which is its own, so the release needs no ordering against it.
__device__ __forceinline__ int resolve_slot(const int32_t* slots, int i, int max_tracks, uint32_t* claim) {
    const int s = slots[i];
    if (s >= 0 && s < max_tracks && claim[s] == (uint32_t)i) {
        claim[s] = 0xffffffffu;
        return s;
    }
    return -1;
}
#endif
// Gather: dst + i * dst_stride <- src + eff[i] * src_stride, `row` floats (zeros for eff[i] < 0).
int launch_gather_rows(const float* src, size_t src_stride, float* dst, size_t dst_stride, size_t row, const int32_t* eff, int n,
                       cudaStream_t st);
// Template scatter of vt_tracks_init_slots: for eff[i] >= 0, tmpl + eff[i] * row <- tok + i * row, state[eff[i]] <- boxes[i]; out_status[i]
// (nullable) <- status[i], or VT_TRACK_BAD_SLOT for eff[i] < 0.
int launch_scatter_init(const float* tok, float* tmpl, size_t row, const double* boxes, double* state, const int32_t* status,
                        int32_t* out_status, const int32_t* eff, int n, cudaStream_t st);

// ---- track records (vt_tracks_export* / vt_tracks_import*; vt_records.cu) ------------------------------------------------
// Item i of n works on track first + i (slots == NULL), or on slots[i] resolved against `claim` after launch_claim_slots (first == 0).
// state [max_tracks][4] and tmpl [max_tracks][64][C] are the handle's; records [n][64 + 256 C] (16-byte aligned); out_status nullable.
struct RecordArgs {
    double* state;
    float* tmpl;
    int C, first, max_tracks;
    const int32_t* slots;
    uint32_t* claim;
    int32_t* out_status;
    uint64_t fingerprint;     // the handle's: written by export, required by import
};
int launch_tracks_export(const RecordArgs& a, uint8_t* records, int n, cudaStream_t st);
int launch_tracks_import(const RecordArgs& a, const uint8_t* records, int n, cudaStream_t st);

// ---- range fallback (vt_set_range_fallback; vt_slots.cu) ------------------------------------------------
// The items of a tensor-core step that ended with VT_TRACK_NUMERIC_RANGE, compacted in item order, and the fp32 pass's rows for them.
struct RangeFallback {
    int32_t* count;        // [1 + chunks]: [0] flagged items of the step, [1 + k] of them in chunk k (items [k chunk, (k + 1) chunk))
    int32_t* item;         // [max_tracks] item index of compacted entry j
    int32_t* slot;         // [max_tracks] its track slot
    int64_t* frame_off;    // [max_tracks] its frame offset
    int32_t* frame_hw;     // [max_tracks][2]
    double* boxes;         // [max_tracks][5] the fp32 pass's out_boxes rows
    double* detail;        // [max_tracks][8] ... out_detail rows
    float* maps;           // score [max_tracks][256] | size [max_tracks][512] | offset [max_tracks][512] ... maps
};
// Finds the flagged items of a step over n items: out_boxes[i][4] == -1, crop status[i] == 0 (status by item) and a valid slot (slot
// first + i, or eff[i] >= 0 when eff is given).  Writes fb's per-item arrays and counts, and adds the count to *counter (nullable).
int launch_fallback_compact(const double* out_boxes, const int32_t* status, const int32_t* eff, int first, const int64_t* frame_offsets,
                            const int32_t* frame_hw, int n, int chunk, const RangeFallback& fb, int64_t* counter, cudaStream_t st);
// Writes entry j < count[0] of the fp32 pass back to item fb.item[j]: out_boxes, out_detail (nullable) and the maps at score / size /
// offset (the step's planar map rows from its first item, max_tracks rows per array in fb.maps).
int launch_fallback_scatter(const RangeFallback& fb, int max_tracks, double* out_boxes, double* out_detail, float* score, float* size,
                            float* offset, int n, cudaStream_t st);

}  // namespace vt
