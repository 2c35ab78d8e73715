/*
 * vittrack_b200.h - C ABI of libvittrack_b200.so
 *
 * B200-native (sm_100a) implementation of VitTracker's per-frame inference hot path
 * (tracker "vit_dist", config vit_48_h32_noKD).  The reference is pure Python; these entry
 * points are what a binding for that path would call instead of the PyTorch/OpenCV code
 * cited next to each function (paths relative to the reference repository root).
 *
 * Conventions
 *   - C linkage, plain pointers and sizes, no C++/torch types.
 *   - Every function returns VT_OK (0) or a negative VtStatus; vt_last_error() gives the text.
 *   - Unless a parameter says "host", data pointers are DEVICE pointers owned by the caller.
 *   - `stream` is a cudaStream_t passed as void*; work is asynchronous with respect to the
 *     host and ordered on that stream.  A handle is not thread-safe.
 *   - No exceptions and no caller-visible allocation cross the ABI; the handle owns its
 *     workspace (allocated in vt_create / grown in vt_reserve).
 *   - There is no CPU fallback: without a CUDA device every compute entry point fails.
 *   - An empty batch (n == 0) is a successful no-op; its data pointers may be null.
 */
#ifndef VITTRACK_B200_H
#define VITTRACK_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VT_ABI_VERSION 1

typedef struct VtContext* VtHandle;

typedef enum VtStatus {
    VT_OK = 0,
    VT_ERR_INVALID_ARG = -1,
    VT_ERR_CUDA = -2,
    VT_ERR_WEIGHTS = -3,        /* unknown / missing / mis-shaped tensor                        */
    VT_ERR_STATE = -4,          /* call order (weights not finalised, tracks not initialised)   */
    VT_ERR_UNSUPPORTED = -5,    /* configuration this build has no kernels for                  */
    VT_ERR_NO_DEVICE = -6
} VtStatus;

/* Per-track status written by the crop stage (processing_utils.py:32-33 raises for the first). */
#define VT_TRACK_OK 0
#define VT_TRACK_TOO_SMALL 1      /* crop_sz < 1: 'Too small bounding box.'                       */
#define VT_TRACK_OUT_OF_DOMAIN 2  /* crop does not overlap the image: undefined in the reference  */
#define VT_TRACK_NUMERIC_RANGE 3  /* an activation was non-finite, or left the fp16 operand range of the
                                   * tensor-core path (|v| >= 65504; operands are fp16 hi + lo): the result is
                                   * withheld (state kept, confidence -1, maps NaN) instead of silently wrong.
                                   * Rerun the track with VT_BLOCKS_SIMT_FP32 (all fp32).                    */

/* Which implementation of the ViT blocks vt_forward / vt_tracks_step use. */
#define VT_BLOCKS_SIMT_FP32 0     /* fp32 CUDA-core kernel: bring-up / exact mode                 */
#define VT_BLOCKS_TCGEN05 1       /* tcgen05 tensor-core kernels: fp16 hi/lo split operands (three products per contraction),
                                   * fp32 accumulation; the attention scores q k^T as a single fp16 pass - the one contraction whose
                                   * low-order terms the measured precision budget (profiles/r02_precision_budget*.json) shows
                                   * never reach the arg-max on the specified (random-init) workload                          */
#define VT_BLOCKS_TCGEN05_3TERM 2 /* the same kernels with three products for q k^T too: for checkpoints with sharp attention
                                   * (large |q||k|), ~9 % slower blocks                                                       */

/* Model / tracker configuration: experiments/vit_dist/vit_48_h32_noKD.yaml:56-64,89-92,
 * lib/config/vit_dist/config.py:27-37, build_ostrack_dist(cfg, depth=3) vit_dist.py:159. */
typedef struct VtConfig {
    int32_t embed_dim;        /* MODEL.BACKBONE.CHANNELS   (48)  */
    int32_t num_heads;        /* MODEL.BACKBONE.HEADS      (1)   */
    int32_t depth;            /* number of ViT blocks      (3)   */
    int32_t mlp_ratio;        /* timm Block default        (4)   */
    int32_t head_channels;    /* MODEL.HEAD.NUM_CHANNELS   (32)  */
    int32_t stride;           /* MODEL.BACKBONE.STRIDE     (16)  */
    int32_t template_size;    /* TEST.TEMPLATE_SIZE        (128) */
    int32_t search_size;      /* TEST.SEARCH_SIZE          (256) */
    double template_factor;   /* TEST.TEMPLATE_FACTOR      (2.0) */
    double search_factor;     /* TEST.SEARCH_FACTOR        (4.0) */
    int32_t max_tracks;       /* capacity of the per-track state (>= 1)                          */
    int32_t chunk_tracks;     /* tracks processed per internal pass (0 = default)                */
    int32_t device;           /* CUDA device ordinal                                             */
    int32_t blocks_impl;      /* VT_BLOCKS_*                                                     */
} VtConfig;

/* ABI version of the loaded library (== VT_ABI_VERSION of the header it was built from). */
int vt_abi_version(void);

/* Text of the last error on this handle (or of the last failed vt_create when h == NULL). */
const char* vt_last_error(VtHandle h);

/* Replaces Vit_dist.__init__ (lib/test/tracker/vit_dist.py:22-51) minus weight loading:
 * validates the configuration, allocates device workspace and per-track state, builds the
 * Hann window (lib/test/utils/hann.py:6-16) and the normalisation table. */
int vt_create(const VtConfig* cfg, VtHandle* out);
int vt_destroy(VtHandle h);

/* Replaces network.load_state_dict(torch.load(ckpt)['net'], strict=False)
 * (lib/test/tracker/vit_dist.py:25).  Call once per state_dict entry with the reference's own
 * key (e.g. "blocks.0.attn.qkv.weight", "patch_embed.net.0.bn.running_var",
 * "box_head.conv1_ctr.0.weight"); `data` is a HOST pointer to contiguous fp32.  Unknown keys
 * return VT_ERR_WEIGHTS and are otherwise ignored ("*.num_batches_tracked" is accepted and
 * dropped).  vt_finalize_weights folds every eval-mode BatchNorm into its convolution
 * (Conv2d_BN.fuse, lib/models/vit_dist/vit_dist.py:22-33; head: conv+bias -> BN,
 * lib/models/layers/head.py:16-21), packs the kernels' layouts and uploads them; it fails if
 * a required tensor was never set. */
int vt_set_tensor(VtHandle h, const char* name, const float* data_host, const int64_t* shape, int32_t ndim);
int vt_finalize_weights(VtHandle h, void* stream);

/* Replaces sample_target(im, box, factor, output_sz) + Preprocessor.process
 * (lib/train/data/processing_utils.py:12-71, lib/test/tracker/data_utils.py:11-17) for n
 * independent (frame, box) pairs, as one gather kernel over raw uint8 frames.
 *   frames        base pointer of uint8 HWC (3-channel) frames
 *   frame_offsets [n] byte offset of item i's frame from `frames`
 *   frame_hw      [n][2] (H, W) of item i's frame
 *   boxes_xywh    [n][4] float64 x, y, w, h (top-left + size, pixels)
 *   out_nchw      [n][3][S][S] fp32  ((v/255 - mean)/std), required
 *   out_u8_hwc    [n][S][S][3] the uint8 crop the reference would have produced (or NULL)
 *   out_mask      [n][S][S] uint8 0/1 attention mask (or NULL)
 *   out_resize_factor [n] float64 S / crop_sz (or NULL)
 *   out_status    [n] VT_TRACK_* (or NULL); failed items produce zeros */
int vt_crop_normalize(VtHandle h, const uint8_t* frames, const int64_t* frame_offsets,
                      const int32_t* frame_hw, const double* boxes_xywh, double factor,
                      int32_t out_size, int32_t n, float* out_nchw, uint8_t* out_u8_hwc,
                      uint8_t* out_mask, double* out_resize_factor, int32_t* out_status,
                      void* stream);

/* Replaces OstrackDist.forward(z, x) in eval mode (lib/models/vit_dist/vit_dist.py:77-100,
 * 122-153): stem on both images, pos-embed add, concat (template first), `depth` ViT blocks,
 * final LayerNorm, CENTER head, cal_bbox on the un-windowed score.
 *   z [n][3][Tz][Tz], x [n][3][Sx][Sx] fp32 normalised
 *   pred_boxes [n][1][4], score_map [n][1][F][F], size_map [n][2][F][F], offset_map [n][2][F][F]
 *   taps (or NULL): [depth+2][n][Nz+Nx][C] tokens after the stem (+pos-embed), after each block
 *   and after the final LayerNorm - debugging / parity aid. */
int vt_forward(VtHandle h, const float* z, const float* x, int32_t n, float* pred_boxes,
               float* score_map, float* size_map, float* offset_map, float* taps, void* stream);

/* Replaces box_head.cal_bbox(score, size_map, offset_map) (lib/models/layers/head.py:142-160),
 * which the tracker calls on the Hann-weighted response (lib/test/tracker/vit_dist.py:105).
 *   boxes [n][4] (cx, cy, w, h) normalised to the search crop. */
int vt_cal_bbox(VtHandle h, const float* score, const float* size_map, const float* offset_map,
                int32_t n, float* boxes, void* stream);

/* Batched tracker state machine: n independent tracks whose state (previous box, cached
 * template tokens) lives on the device.
 *
 * vt_tracks_init replaces Vit_dist.initialize (lib/test/tracker/vit_dist.py:53-74) for tracks
 * [first, first+n): template crop (factor/size from the config), stem, pos-embed; state <- box.
 * The reference keeps the template as pixels and re-runs its stem every frame
 * (vit_dist.py:78); caching the tokens is bit-identical and is what makes a step cheap. */
int vt_tracks_init(VtHandle h, const uint8_t* frames, const int64_t* frame_offsets,
                   const int32_t* frame_hw, const double* boxes_xywh, int32_t first, int32_t n,
                   int32_t* out_status, void* stream);

/* vt_tracks_step replaces Vit_dist.track (lib/test/tracker/vit_dist.py:76-148) for tracks
 * [first, first+n): search crop around the current state, forward, Hann weighting, arg-max,
 * box decode, map_box_back (:150-156), clip_box(margin=10) (lib/utils/box_ops.py:97-106);
 * state <- result.
 *   out_boxes  [n][5] float64: x, y, w, h (frame pixels), confidence (= un-windowed
 *              score_map.max(), vit_dist.py:148)
 *   out_detail [n][8] float64 or NULL: pred cx, cy, w, h (the fp32 `pred_box` of vit_dist.py:
 *              108-109 before map_box_back), resize_factor, arg-max index of the windowed
 *              response, VT_TRACK_* status, windowed maximum
 *   update_state != 0 writes the new box back as the track state (closed loop).
 * Of a track's frame only rows [max(0, y1), min(H, y1 + crop_sz)) are read (crop_sz = ceil(sqrt(w h) search_factor),
 * y1 = round(y + h/2 - crop_sz/2) of its current state): a caller may upload just those rows, and frame_offsets[i]
 * may point before its buffer as long as the rows that are read lie inside it. */
int vt_tracks_step(VtHandle h, const uint8_t* frames, const int64_t* frame_offsets,
                   const int32_t* frame_hw, int32_t first, int32_t n, double* out_boxes,
                   double* out_detail, int32_t update_state, void* stream);

/* Read / overwrite the per-track boxes ([n][4] float64 device pointers). */
int vt_tracks_get_state(VtHandle h, double* boxes_xywh, int32_t first, int32_t n, void* stream);
int vt_tracks_set_state(VtHandle h, const double* boxes_xywh, int32_t first, int32_t n, void* stream);

/* Maps of the most recent vt_tracks_step chunk-by-chunk copy: score [n][F*F], size [n][2][F*F],
 * offset [n][2][F*F] for tracks [first, first+n) of that step (debug / parity aid; any may be
 * NULL). Valid only if the step covered those tracks. */
int vt_tracks_last_maps(VtHandle h, int32_t first, int32_t n, float* score_map, float* size_map,
                        float* offset_map, void* stream);

/* Number of kernels this handle has launched so far (bench.py reports it as gpu_launches). */
int64_t vt_launch_count(VtHandle h);

/* Optional per-stage device timing.  While enabled, every pipeline stage a vt_forward /
 * vt_tracks_init / vt_tracks_step call launches is bracketed by CUDA events on the caller's
 * stream.  vt_profile_read waits for the recorded events, returns per stage the summed device
 * time in milliseconds, the number of bracketed launches and the number of items (tracks) they
 * processed, and clears the record.  Arrays have VT_NUM_STAGES entries indexed by VT_STAGE_*. */
#define VT_STAGE_CROP 0
#define VT_STAGE_STEM 1
#define VT_STAGE_BLOCKS 2
#define VT_STAGE_HEAD 3
#define VT_NUM_STAGES 4
int vt_profile_enable(VtHandle h, int32_t enable);
int vt_profile_read(VtHandle h, double* stage_ms, int64_t* stage_launches, int64_t* stage_items);

/* Host frame -> device frame buffer, only the rectangle a crop reads.  `image` is a host HxWx3 uint8 frame (pageable memory is
 * fine), `frame_dev` the device buffer holding the frame at the same layout (byte offset (y * W + x) * 3), `staging` a pinned host
 * buffer and `staging_dev` a device buffer (may be NULL: one strided host -> device copy instead, at about half the rate) of at
 * least (y1 - y0) * (x1 - x0) * 3 bytes each.  Rows [y0, y1) x columns [x0, x1) are packed into `staging` by a few host threads, cross
 * the link as one contiguous copy and are spread over the frame's rows on the device, all on `stream`.  The rest of `frame_dev` is
 * left as it is: sample_target (lib/train/data/processing_utils.py:34-48) slices im[y1:y2, x1:x2] and reads nothing else, and the
 * crop kernels read nothing else with a non-zero weight (vt_tracks_step's row guarantee, plus columns [x0, x1) and the first two
 * pixels of a row, whose weight is zero).  `staging` and `staging_dev` may be reused once `stream` has passed the copies. */
int vt_upload_frame_rect(const uint8_t* image, int32_t H, int32_t W, int32_t y0, int32_t y1, int32_t x0, int32_t x1,
                         uint8_t* staging, uint8_t* staging_dev, uint8_t* frame_dev, void* stream);

/* YUV 4:2:0 frames, as video decoders hand them out.  Replaces cv2.cvtColor(frame, COLOR_YUV2RGB_NV12 / COLOR_YUV2RGB_I420)
 * in front of sample_target, bit for bit (OpenCV 4.13.0, modules/imgproc/src/color_yuv.simd.hpp, 20 fractional bits):
 *     y = max(0, Y - 16) * 1220542
 *     R = sat_u8((y + (1 << 19) + 1673527 (V - 128)) >> 20)
 *     G = sat_u8((y + (1 << 19) -  852492 (V - 128) - 409993 (U - 128)) >> 20)
 *     B = sat_u8((y + (1 << 19) + 2116026 (U - 128)) >> 20)
 * with one (U, V) sample per 2x2 luma block and no interpolation.  A frame is the array cvtColor takes: uint8 (H*3/2) x W,
 * contiguous, pitch W, H and W even.  NV12: the H x W Y plane, then H/2 rows of W interleaved bytes U V U V ...; I420
 * (yuv420p): the Y plane, then U (H/2 x W/2), then V (H/2 x W/2).  The result is the H x W x 3 RGB frame every other entry
 * point takes; the tracking kernels read it unchanged. */
#define VT_FRAME_NV12 1
#define VT_FRAME_I420 2

/* n whole frames, device -> device.  src + src_offsets[i]: a (H*3/2) x W YUV frame, frame_hw[i] = (H, W) (even);
 * dst + dst_offsets[i]: the H x W x 3 RGB frame the other entry points take.  Arrays are device pointers.  Offsets may be
 * any byte offset.  The sizes are read on the device: an item whose H or W is odd or below 2 is skipped (its destination is
 * not written); a caller that cannot vouch for its sizes checks them on the host.  One kernel launch. */
int vt_yuv420_to_rgb(VtHandle h, int32_t format, const uint8_t* src, const int64_t* src_offsets, const int32_t* frame_hw,
                     uint8_t* dst, const int64_t* dst_offsets, int32_t n, void* stream);

/* The YUV counterpart of vt_upload_frame_rect: rows [y0, y1) x columns [x0, x1) of a host YUV frame (`image`, pageable memory
 * is fine; H and W even), widened to even bounds, are packed (Y rows, then the chroma rows), cross the link as one contiguous
 * copy into staging_dev and are converted straight into frame_rgb_dev at their place in the H x W x 3 frame.  Nothing outside
 * the widened rectangle is written.  `staging` (pinned host) and `staging_dev` (device, required) hold at least
 * rows * cols * 3/2 bytes of the widened rectangle; they may be reused once `stream` has passed the conversion. */
int vt_upload_yuv420_rect(VtHandle h, int32_t format, const uint8_t* image, int32_t H, int32_t W, int32_t y0, int32_t y1,
                          int32_t x0, int32_t x1, uint8_t* staging, uint8_t* staging_dev, uint8_t* frame_rgb_dev, void* stream);

/* Development aid: which profiled stage launches (vt_profile_enable) have started / finished.  Non-blocking;
 * meant for a watchdog thread while the owning thread waits in a synchronisation (tools/hang_probe.py,
 * tests/test_gpu_soak.py).  out[i] = stage * 4 + (started ? 1 : 0) + (finished ? 2 : 0); returns the count. */
int vt_debug_pending(VtHandle h, int32_t* out, int32_t cap);

#ifdef __cplusplus
}
#endif
#endif /* VITTRACK_B200_H */
