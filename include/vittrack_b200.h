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
                                   * vt_set_range_fallback recomputes such tracks on the fp32 kernels within the
                                   * same step call.                                                           */
#define VT_TRACK_BAD_SLOT 4       /* slot outside [0, max_tracks) or named by an earlier item of the same call */
#define VT_TRACK_BAD_RECORD 5     /* vt_tracks_import*: the record failed a check (header, fingerprint, checksum, box); nothing written */

/* Which implementation of the ViT blocks vt_forward / vt_tracks_step use. */
#define VT_BLOCKS_SIMT_FP32 0     /* fp32 CUDA-core kernel: bring-up / exact mode                 */
#define VT_BLOCKS_TCGEN05 1       /* tcgen05 tensor-core kernels: fp16 hi/lo split operands (three products per contraction),
                                   * fp32 accumulation; the attention scores q k^T as a single fp16 pass - the one contraction whose
                                   * low-order terms the measured precision budget (profiles/r02_precision_budget*.json) shows
                                   * never reach the arg-max on the specified (random-init) workload.  Its error grows with
                                   * |q||k|: max |map - float64| (score / offset) over 1024 open-loop 720p tracks, NVIDIA B200 at
                                   * 1000 W (tests/test_trained_weights.py), q and k scaled to a max |logit| of:
                                   *                   random init        4                 16                64
                                   *   single pass     8.8e-7 / 1.4e-5    3.6e-6 / 3.9e-5   4.0e-5 / 5.8e-4   4.2e-4 / 2.9e-3
                                   *   three terms     6.0e-7 / 1.0e-5    6.4e-7 / 1.1e-5   9.0e-7 / 1.5e-5   1.0e-6 / 1.3e-5
                                   * At 64 the single pass moves boxes past the 1e-2 parity bound, so vt_finalize_weights takes the
                                   * three-term pass when a bound on |q.k|/sqrt(C) from the weights alone exceeds 512 (random-init
                                   * weights: < 20)                                                                          */
#define VT_BLOCKS_TCGEN05_3TERM 2 /* the same kernels with three products for q k^T too, whatever the weights: for checkpoints
                                   * with sharp attention (large |q||k|), ~9 % slower blocks                                  */

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

/* The same two calls for any set of tracks: item i works on track slots[i].  `slots` is a DEVICE int32 array of n entries in any
 * order; every other array is per item, in item order, exactly as in vt_tracks_init / vt_tracks_step.  A multi-target caller adds a
 * target by initialising a free slot, retires one by no longer listing it, and steps the live set in one call.
 *   - The list is checked on the device, without a host synchronisation.  An entry outside [0, max_tracks), or equal to the slot
 *     of an earlier item of the same call, is not processed: vt_tracks_init_slots sets out_status[i] = VT_TRACK_BAD_SLOT and writes
 *     no state or template; vt_tracks_step_slots writes out_boxes[i] = (0, 0, 0, 0, -1), out_detail[i] with status
 *     VT_TRACK_BAD_SLOT and arg-max -1, NaN maps, and reads or writes no state.  Among repeated slots the first item wins.
 *   - VT_ERR_INVALID_ARG before any launch for a null handle, n < 0, n > max_tracks, or a null pointer (out_status and out_detail
 *     may be null) when n > 0.  n == 0 is a no-op.  vt_tracks_step_slots before any init returns VT_ERR_STATE.
 *   - No allocation and no host synchronisation: a call can be captured in a CUDA graph and replayed with new contents in `slots`.
 *   - A slot that was never initialised holds the zero box vt_create gave it: stepping it returns VT_TRACK_TOO_SMALL.
 *   - A track's outputs, maps and new state are the same bits whether it is stepped by range or by slot list, in any order and next
 *     to any other items.
 *   - After vt_tracks_step_slots, vt_tracks_last_maps(first, n) addresses item positions [first, first + n) of that call.
 * Cost over the range calls: two small kernels that resolve the list per call, plus per chunk one row-copy kernel (the template
 * scatter of an init; on configurations other than vit_48_h32, the template gather of a step). */
int vt_tracks_init_slots(VtHandle h, const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw,
                         const double* boxes_xywh, const int32_t* slots, int32_t n, int32_t* out_status, void* stream);
int vt_tracks_step_slots(VtHandle h, const uint8_t* frames, const int64_t* frame_offsets, const int32_t* frame_hw,
                         const int32_t* slots, int32_t n, double* out_boxes, double* out_detail, int32_t update_state,
                         void* stream);

/* Range fallback (off by default).  With enable != 0, every item of vt_tracks_step / vt_tracks_step_slots that the tensor-core
 * kernels end with VT_TRACK_NUMERIC_RANGE is recomputed on the fp32 kernels of VT_BLOCKS_SIMT_FP32 before the call returns.
 *   counter_dev  optional DEVICE int64: each step adds the number of items it recomputed (no host synchronisation to read it).
 *                A CUDA graph captured while it is set keeps adding to that address on every replay: it must outlive such graphs.
 * Contract:
 *   1. A recomputed item's out_boxes, out_detail, maps (vt_tracks_last_maps) and new state are, bit for bit, what a
 *      VT_BLOCKS_SIMT_FP32 handle with the same weights, template frame and box, and state gives for that track, for range and
 *      slot-list steps, update_state 0 and 1, in any chunk.
 *   2. An item that is not recomputed is bit-identical to the same handle with the fallback off.
 *   3. An item the fp32 kernels flag too (a non-finite activation) keeps VT_TRACK_NUMERIC_RANGE, with the fp32 pass's outputs.
 *   4. Items with VT_TRACK_TOO_SMALL, VT_TRACK_OUT_OF_DOMAIN or VT_TRACK_BAD_SLOT are never recomputed.
 *   5. The step still allocates nothing and does not synchronise: it can be captured in a CUDA graph, and a replay recomputes
 *      whichever items that replay flags.
 * Detection: an item is recomputed when its confidence is -1 (a real one is a clamped sigmoid in [1e-4, 0.9999]), its crop status
 * is 0 and its slot is valid.  The host never learns how many there are, so the fp32 kernels are launched as for every item of
 * the step and work only on the items below the device count: nine extra launches per step at one chunk (one compaction, five for
 * the fp32 crop + stem, blocks, head, one scatter), five more per further chunk.
 * This call allocates the compacted per-item arrays and output rows (about 5.3 KB per track of max_tracks) the first time it
 * enables the fallback.  VT_ERR_UNSUPPORTED for configurations other than vit_48_h32 (their fp32 route has no device-side item
 * count); a VT_BLOCKS_SIMT_FP32 handle returns VT_OK and changes nothing (it has no fp16 operands). */
int vt_set_range_fallback(VtHandle h, int32_t enable, int64_t* counter_dev);

/* Read / overwrite the per-track boxes ([n][4] float64 device pointers). */
int vt_tracks_get_state(VtHandle h, double* boxes_xywh, int32_t first, int32_t n, void* stream);
int vt_tracks_set_state(VtHandle h, const double* boxes_xywh, int32_t first, int32_t n, void* stream);

/* Track records: a whole track state (box + cached template tokens) as a fixed-size, self-checking byte image, so that a track can
 * be saved, restored, forked, or moved to another slot, handle or GPU and continue bit for bit.  A record is
 * R = VT_TRACK_RECORD_HEADER_BYTES + 256 C bytes (12 352 at C = 48, 196 672 at C = 768), all fields little-endian:
 *   offset  bytes  field
 *        0      4  uint32 VT_TRACK_RECORD_MAGIC
 *        4      4  uint32 VT_TRACK_RECORD_VERSION
 *        8      8  uint64 weights fingerprint of the exporting handle (vt_weights_fingerprint)
 *       16      4  int32  embed_dim C
 *       20      4  int32  template token rows (64)
 *       24      8  uint64 checksum of the payload (below)
 *       32     32  float64 box x, y, w, h (the track state)
 *       64  256 C  float32 template tokens [64][C]: stem output + pos_embed_z, as vt_tracks_init computed them
 * Payload checksum: the payload is bytes [32, R) read as little-endian uint64 words w_0 .. w_{K-1} (K = 4 + 32 C; w_0 .. w_3 the
 * box), and
 *     checksum = sum over k of splitmix64(w_k + k * 0x9E3779B97F4A7C15)  (mod 2^64),
 *     splitmix64(z): z += 0x9E3779B97F4A7C15; z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9; z = (z ^ (z >> 27)) * 0x94D049BB133111EB;
 *                    return z ^ (z >> 31)           (all arithmetic mod 2^64)
 * which depends on every word and its position, and not on the order in which the terms are added.
 * Weights fingerprint, computed on the host by vt_finalize_weights: FNV-1a 64 (offset basis 0xcbf29ce484222325, prime
 * 0x100000001b3) over 8-byte little-endian words of a byte stream (h ^= word; h *= prime), the last word zero-padded:
 *   1. the 24 ASCII bytes "vittrack_b200 weights v1" (no terminator);
 *   2. int32 embed_dim, num_heads, depth, mlp_ratio, head_channels, stride, template_size, search_size, then float64
 *      template_factor, search_factor (max_tracks, chunk_tracks, device and blocks_impl are not hashed);
 *   3. int32 template route: how the handle computes template tokens.  0: vit_48_h32 (fp32 crop + stem on the CUDA cores for every
 *      blocks_impl); other configurations: 1 VT_BLOCKS_SIMT_FP32 (fp32 GEMMs), 2 tensor-core GEMMs, 3 tensor-core split-image GEMMs
 *      (embed_dim % 128 == 0);
 *   4. every tensor the handle holds ("*.num_batches_tracked" is never held; tracker.output_window is
 *      when it was set) in byte-wise ascending name order: the name's bytes and a NUL, int32 ndim, int64 shape[ndim], then the fp32
 *      data exactly as vt_set_tensor received it (before BatchNorm folding or scale rebalancing).
 * Two handles with equal fingerprints compute the same template-token bits from the same frame and box, so a record moves freely
 * between them (e.g. between the VT_BLOCKS_* of vit_48_h32, which share route 0).  Hashing is one multiply per 8 bytes: about
 * 82 ms for the widest configuration's 381 MB on one Intel Xeon core, of the 1.8 s vt_finalize_weights takes there in all. */
#define VT_TRACK_RECORD_MAGIC 0x52545456u     /* "VTTR" as little-endian bytes */
#define VT_TRACK_RECORD_VERSION 1
#define VT_TRACK_RECORD_HEADER_BYTES 64       /* bytes before the template tokens: the fields above and the box */

/* The handle's weights fingerprint (host out_host); VT_ERR_STATE before vt_finalize_weights. */
int vt_weights_fingerprint(VtHandle h, uint64_t* out_host);
/* R, the size of one record of this handle, in bytes (host out_host). */
int vt_track_record_bytes(VtHandle h, int64_t* out_host);
/* Export tracks [first, first + n), or slots[i] for item i, into `records`; import records into tracks [first, first + n) or slots.
 *   - `records` is a DEVICE array of n records R bytes apart, 16-byte aligned.  `slots` and out_status are device int32 [n]; out_status
 *     may be null.  Export's out_status[i] is VT_TRACK_OK or VT_TRACK_BAD_SLOT; import's VT_TRACK_OK, VT_TRACK_BAD_SLOT or
 *     VT_TRACK_BAD_RECORD.
 *   - Export is VT_ERR_STATE before vt_finalize_weights.  A slot that was never initialised exports the zero box of vt_create.
 *   - Import checks every record on the device, without a host synchronisation: magic, version, C, rows, a fingerprint equal to this
 *     handle's, the checksum and a finite box.  A record that fails any check gets VT_TRACK_BAD_RECORD and writes nothing.
 *   - Slot lists are checked as in vt_tracks_init_slots: an entry outside [0, max_tracks) or repeating an earlier item's slot gets
 *     VT_TRACK_BAD_SLOT (which takes precedence over VT_TRACK_BAD_RECORD); the first item wins.  An export item with a bad slot writes
 *     an all-zero record (magic 0: it can never be imported).
 *   - Import writes the state and the template tokens in place (CUDA graphs captured earlier stay valid) and makes the handle ready
 *     to step, as vt_tracks_init does.
 *   - An accepted record continues exactly as the exported track would have: its out_boxes, out_detail, maps and new state are the
 *     same bits, for range and slot-list steps, in any chunk, with the range fallback on or off.
 *   - VT_ERR_INVALID_ARG before any launch for a null handle, n < 0, n > max_tracks, first < 0 or first + n > max_tracks, a null
 *     pointer when n > 0, or a `records` that is not 16-byte aligned.  n == 0 is a no-op.
 *   - No allocation and no host synchronisation: the calls can be captured in a CUDA graph and replayed with new contents in `slots`
 *     and `records`.  One kernel launch per range call, two per slot-list call (the slot claim, then the copy). */
int vt_tracks_export(VtHandle h, int32_t first, int32_t n, uint8_t* records, void* stream);
int vt_tracks_export_slots(VtHandle h, const int32_t* slots, int32_t n, uint8_t* records, int32_t* out_status, void* stream);
int vt_tracks_import(VtHandle h, const uint8_t* records, int32_t first, int32_t n, int32_t* out_status, void* stream);
int vt_tracks_import_slots(VtHandle h, const uint8_t* records, const int32_t* slots, int32_t n, int32_t* out_status, void* stream);

/* Maps of the most recent vt_tracks_step chunk-by-chunk copy: score [n][F*F], size [n][2][F*F],
 * offset [n][2][F*F] for tracks [first, first+n) of that step (debug / parity aid; any may be
 * NULL). Valid only if the step covered those tracks.  After vt_tracks_step_slots: items
 * [first, first+n) of that call. */
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

/* Device-resident YUV surfaces (a hardware decoder's output: pitched planes, the chroma plane wherever the decoder put it),
 * converted only where a crop reads them.  For item i of n:
 *   planes     [n][3] device addresses of the Y plane, the U plane (NV12: the interleaved U V plane) and the V plane (I420; NV12
 *              ignores it).  Any byte alignment.
 *   pitches    [n][2] int32 byte distance between rows of the luma plane and of the chroma plane(s): at least W for luma and for
 *              NV12 chroma, at least W/2 for I420 chroma (U and V share it).
 *   frame_hw   [n][2] int32 (H, W) of the picture (even; a decoder surface's padding rows below H are never read).
 *   boxes_xywh [n][4] float64 boxes, or NULL: the current state of tracks [first, first + n) (what vt_tracks_step will crop).
 *   factor     the crop factor (the configuration's template_factor before vt_tracks_init, search_factor before vt_tracks_step).
 *   dst + dst_offsets[i]: the item's H x W x 3 RGB frame, the one passed to vt_tracks_init / vt_tracks_step afterwards.
 * The box's crop geometry is computed on the device by the code the crop kernels run: crop_sz = ceil(sqrt(w h) factor),
 * x1 = round(x + w/2 - crop_sz/2), y1 = round(y + h/2 - crop_sz/2) (half to even).  Only rows [max(0, y1), min(H, y1 + crop_sz))
 * x columns [max(0, x1 - 1), min(W, x1 + crop_sz + 1)) - what sample_target reads plus one spare column on either side - widened
 * to even bounds (a 2x2 block shares one chroma sample) are read and converted, with the cvtColor arithmetic above, at their place
 * in the RGB frame.  No other byte of dst is written.  Nothing is written for an item whose crop is degenerate (VT_TRACK_TOO_SMALL
 * or VT_TRACK_OUT_OF_DOMAIN), whose H or W is odd or below 2, or whose pitch is below its row width.  The rest of the RGB frame
 * keeps what it held: zero-fill it once (the crop kernels read the first pixels of a row with weight 0).
 * All arrays are device pointers.  No allocation and no host synchronisation: the call can be captured in a CUDA graph.
 * Bad host arguments (format, null pointers, n < 0, factor <= 0, first + n > max_tracks when the state is used) return
 * VT_ERR_INVALID_ARG before any launch.  One kernel launch. */
int vt_yuv420_crop_to_rgb(VtHandle h, int32_t format, const uint64_t* planes, const int32_t* pitches, const int32_t* frame_hw,
                          const double* boxes_xywh, double factor, int32_t first, int32_t n, uint8_t* dst,
                          const int64_t* dst_offsets, void* stream);

/* Several tracks on one surface (many targets in one camera stream): each surface is converted once, into one RGB frame per
 * surface, over the bounding rectangle of the crops of its items.  For m surfaces and n items:
 *   planes, pitches, frame_hw   per surface ([m][3], [m][2], [m][2]), as for vt_yuv420_crop_to_rgb.
 *   dst + dst_offsets[s]        surface s's H x W x 3 RGB frame ([m]); every item on surface s is then initialised or stepped on it.
 *   item_surface [n] int32      the surface of item i.
 *   boxes_xywh   [n][4]         float64 boxes, or NULL: the crop is taken around the track state, of track slots[i] when `slots` is
 *                               given and of track first + i otherwise.
 *   slots        [n] int32      track slots (as vt_tracks_init_slots / vt_tracks_step_slots take them), or NULL; `first` is ignored
 *                               when they are given.
 * Item i's rectangle is the one vt_yuv420_crop_to_rgb converts for its box and factor (the crop's rows and columns plus one spare
 * column on either side, widened to even bounds).  An item is skipped when its surface index is outside [0, m), when `slots` is given
 * and slots[i] is a bad slot as vt_tracks_init_slots defines it (outside [0, max_tracks) or repeating an earlier item's slot), or when
 * vt_yuv420_crop_to_rgb would skip its rectangle (degenerate crop, odd or tiny frame, a pitch below the row width).  Surface s's
 * frame gets the cvtColor bytes of the bounding rectangle of its valid items' rectangles, and no other byte of dst is written; a
 * surface without a valid item is not written at all.  A track's crop reads only its own rectangle, which lies inside the bounding
 * rectangle and holds there the bytes the per-item path writes, so vt_tracks_init / vt_tracks_step on these frames give, bit for
 * bit, what they give on the per-item path's frames.  The bounding rectangle is not the exact union: at worst one whole frame per
 * surface is converted.
 * All arrays are device pointers.  No allocation and no host synchronisation (the handle owns a 16-byte rectangle and a counter per
 * surface, left empty after each call): the call can be captured in a CUDA graph.  Bad host arguments (format, n < 0, m < 0 or
 * m > max_tracks, factor <= 0, first + n > max_tracks when the state is read by range, null pointers when n > 0) return
 * VT_ERR_INVALID_ARG before any launch; n == 0 is a no-op.  Launches: two, three with `slots`. */
int vt_yuv420_crops_to_surface_rgb(VtHandle h, int32_t format, const uint64_t* planes, const int32_t* pitches, const int32_t* frame_hw,
                                   int32_t m, const int32_t* item_surface, const double* boxes_xywh, const int32_t* slots, double factor,
                                   int32_t first, int32_t n, uint8_t* dst, const int64_t* dst_offsets, void* stream);

/* Development aid: which profiled stage launches (vt_profile_enable) have started / finished.  Non-blocking;
 * meant for a watchdog thread while the owning thread waits in a synchronisation (tools/hang_probe.py,
 * tests/test_gpu_soak.py).  out[i] = stage * 4 + (started ? 1 : 0) + (finished ? 2 : 0); returns the count. */
int vt_debug_pending(VtHandle h, int32_t* out, int32_t cap);

#ifdef __cplusplus
}
#endif
#endif /* VITTRACK_B200_H */
