/* fear_b200.h -- C ABI of libfear_b200.so: the B200-native (sm_100a) FEAR-XS per-frame
 * inference hot path (backbone -> pixel-wise correlation -> cls/reg heads -> box decode).
 *
 * The reference (PinataFarms/FEARTracker) is pure Python/PyTorch and has no FFI; these entry
 * points are what a binding for its hot path replaces (file:line relative to the reference):
 *
 *   fear_get_features     FEARNet.get_features            model_training/model/fear_net.py:63-66
 *                         (= Encoder stages 0..17 + AdjustLayer, blocks.py:8-42,75-88)
 *   fear_backbone         FEARNet.feature_extractor       model_training/model/fear_net.py:58-61
 *   fear_head             FEARNet.connector / BoxTower.forward  fear_net.py:76-81, blocks.py:174-194
 *   fear_track            FEARNet.track (+ FEARTracker._postprocess / FEARBoxCoder.decode)
 *                         fear_net.py:90-96, tracker/fear_tracker.py:74-86, dataset/box_coder.py:75-107
 *   fear_forward          FEARNet.forward((template, search))   fear_net.py:83-88
 *   fear_corr_concat_f32  MobileCorrelation.forward front half (matmul + cat)  blocks.py:121-124
 *   fear_corr_nhwc_f32    same contraction on the library's internal channels-last layout
 *   fear_decode           FEARBoxCoder.decode                 dataset/box_coder.py:75-107
 *   fear_pack_weights     load_from_lighting + nn.Module.load_state_dict  utils/torch.py:11-24
 *
 *   fear_head_update      BoxTower.forward(search, kernel, update)   blocks.py:174-179
 *   fear_crop_resize_u8   get_extended_crop (crop + pad + resize)    model_training/utils/utils.py:215-253
 *   fear_track_crops_u8   the same for N tracks at once, context box computed on the device
 *   fear_track_advance    Tracker._rescale_bbox + clamp_bbox of FEARTracker.update, on the device
 *
 * Conventions: every pointer named d_* is a DEVICE pointer owned by the caller (torch keeps
 * ownership); tensors are dense fp32 in the reference's NCHW layout unless stated; `stream`
 * is a cudaStream_t passed as void*.  Hot-path calls are asynchronous on `stream`, never synchronise
 * it and never allocate (workspace is reserved up front by fear_reserve -- the only call besides
 * fear_pack_weights / fear_free that allocates or synchronises; a batch larger than the reservation is
 * processed in chunks; fear_corr_concat_ws_f32 takes its scratch from the caller).  Return 0 on success,
 * a positive cudaError_t or a negative FEAR_E* code otherwise; fear_last_error() gives the message
 * (thread-local).  Handles are not thread-safe: one handle per host thread / stream.  A handle belongs to the
 * device that was current when it was packed; every entry point selects that device for its own duration and
 * restores the caller's current device (several devices per process are fine: call fear_init for each).
 */
#ifndef FEAR_B200_H
#define FEAR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FEAR_ABI_VERSION 1

#define FEAR_EINVAL (-1)    /* bad argument (shape, null pointer, alignment)            */
#define FEAR_ESTATE (-2)    /* handle not initialised / weights not packed              */
#define FEAR_ENOMEM (-3)    /* workspace reservation failed                             */
#define FEAR_ENODEV (-4)    /* no sm_100 device                                         */

#define FEAR_FEAT_CH 256        /* AdjustLayer output channels                          */
#define FEAR_SCORE 16           /* score map side (256 / 16)                            */
#define FEAR_TMPL 8             /* template feature side (128 / 16)                     */
#define FEAR_CORR_CH 64         /* FEAR_TMPL^2 correlation channels                     */

/* One decoded frame (FEARBoxCoder.decode semantics: xywh in float64 like the reference,
 * which promotes to double through its float64 grid; (row, col) = unravel(argmax)). */
typedef struct FearBox {
  double x, y, w, h;
  float score;      /* sigmoid(cls)[row, col]                                           */
  int32_t row, col; /* argmax of sigmoid(cls), first maximum in row-major order         */
  int32_t flat;     /* row * 16 + col                                                   */
} FearBox;

typedef struct FearContext FearContext;

/* Verify `device` is sm_100, initialise the library's per-device state and make it the current device
 * (like torch's .cuda(id)).  Call once per device before packing weights on it; repeated calls are cheap. */
int fear_init(int device);
int fear_abi_version(void);
const char* fear_last_error(void);

/* ---- weights ------------------------------------------------------------------------
 * The library owns the canonical list of (BN-folded) tensors it needs; the host packs them
 * in that order into one fp32 blob.  Names look like "xif4_5.pw.w"; shapes are torch-native
 * ([Cout][Cin] for 1x1, [C][k][k] for depthwise, [16][3][3][3] for the stem). */
int fear_weight_count(void);
const char* fear_weight_name(int i);
int64_t fear_weight_numel(int i);

/* blob: HOST pointer to the packed fp32 tensors; offsets[i] = element offset of tensor i,
 * offsets[n] = total elements; n must equal fear_weight_count().  Creates *handle. */
int fear_pack_weights(const float* blob, const uint64_t* offsets, int n, FearContext** handle);
/* Reserve device workspace for batches up to max_batch search frames (default 1). */
int fear_reserve(FearContext* h, int max_batch);
void fear_free(FearContext* h);

/* ---- hot path -----------------------------------------------------------------------*/
/* img (B,3,H,W) -> feat (B,256,H/16,W/16);  H, W multiples of 16, <= 256. */
int fear_get_features(FearContext* h, const float* d_img, int B, int H, int W, float* d_feat, void* stream);

/* img (B,3,H,W) -> backbone features (B,112,H/16,W/16) before the neck
 * (FEARNet.feature_extractor, fear_net.py:58-61). */
int fear_backbone(FearContext* h, const float* d_img, int B, int H, int W, float* d_feat, void* stream);

/* zfeat (Bz,256,8,8) with Bz == B or 1 (broadcast); xfeat (B,256,16,16)
 * -> bbox (B,4,16,16) = exp(adjust*pred+bias), cls (B,1,16,16) = 0.1*pred (logits). */
int fear_head(FearContext* h, const float* d_zfeat, int Bz, const float* d_xfeat, int B,
              float* d_bbox, float* d_cls, void* stream);

/* BoxTower.forward(search, kernel, update) (blocks.py:174-179): as fear_head, but the CLASSIFICATION branch correlates
 * with the dynamic template d_zupdate (Bu,256,8,8), Bu == B or 1, while the regression branch keeps d_zfeat.
 * d_zupdate == NULL is exactly fear_head. */
int fear_head_update(FearContext* h, const float* d_zfeat, int Bz, const float* d_zupdate, int Bu, const float* d_xfeat,
                     int B, float* d_bbox, float* d_cls, void* stream);

/* search (B,3,256,256) + zfeat (Bz,256,8,8) -> maps and (if non-null) decoded boxes[B].
 * d_bbox / d_cls may be null when only boxes are wanted. */
int fear_track(FearContext* h, const float* d_search, const float* d_zfeat, int Bz, int B,
               float* d_bbox, float* d_cls, FearBox* d_boxes, void* stream);

/* Same as fear_track / fear_get_features but the image is the tracker's raw uint8 RGB crop in HWC layout
 * (B,H,W,3): the ImageNet normalisation of Tracker._preprocess_image (tracker/base_tracker.py:69-81,97-103)
 * is applied inside the stem kernel with the same float32 roundings (bit-identical to host normalisation);
 * the host->device copy is 4x smaller. */
int fear_track_u8(FearContext* h, const uint8_t* d_search_u8, const float* d_zfeat, int Bz, int B,
                  float* d_bbox, float* d_cls, FearBox* d_boxes, void* stream);
int fear_get_features_u8(FearContext* h, const uint8_t* d_img_u8, int B, int H, int W, float* d_feat, void* stream);

/* template (B,3,128,128) + search (B,3,256,256) -> maps (+ boxes). */
int fear_forward(FearContext* h, const float* d_template, const float* d_search, int B,
                 float* d_bbox, float* d_cls, FearBox* d_boxes, void* stream);

/* Host pre-processing of the tracking loop on the device (get_extended_crop, reference
 * model_training/utils/utils.py:215-253 = context crop, constant-colour padding, cv2.resize(INTER_LINEAR) on uint8):
 * d_frame (H,W,3) uint8 RGB stays on the device; d_crop (out_size,out_size,3) uint8 is what fear_track_u8 /
 * fear_get_features_u8 consume.  Bit-identical to OpenCV's 8-bit fixed-point bilinear kernel.  d_params (device,
 * int32, 8 + 6 * out_size entries, so a captured CUDA graph sees per-frame values): [0..3] context x, y, w, h in frame
 * coordinates (may leave the frame), [4..6] padding colour R, G, B, [7] 0, then xofs, xa0, xa1, yofs, ya0, ya1
 * (out_size entries each): per-axis source offset and the two 11-bit coefficients, computed on the host exactly as
 * cv::resize computes them (feartracker_b200.image_ops.resize_tables). */
int fear_crop_resize_u8(const uint8_t* d_frame, int H, int W, const int32_t* d_params, uint8_t* d_crop, int out_size,
                        void* stream);

/* ---- batched tracking loop with device-resident state ---------------------------------
 * One input frame of a step: absolute device pointer, so a captured CUDA graph stays valid whatever buffer the
 * frame sits in. */
typedef struct FearFrame {
  const uint8_t* data; /* DEVICE pointer to (h, w, 3) RGB uint8, row-major                   */
  int32_t h, w;
} FearFrame;

/* Device-resident state of one target (FEARTracker.tracking_state). */
typedef struct FearTrack {
  int32_t x, y, w, h;                    /* current box in frame pixels (tracking_state.bbox)          */
  int32_t cx, cy, cw, ch;                /* context box of the last crop (tracking_state.mapping)      */
  int32_t pad_r, pad_g, pad_b, reserved; /* rint(mean colour of the init frame), clipped to 0..255     */
} FearTrack;

/* For every track n with d_frame_of_track[n] in [0, F): context box of (x, y, w, h) grown by `context` per side
 * (image_ops.context_box), stored into the track's cx..ch, and crop n of d_crops (N, out_size, out_size, 3) cut from
 * frame d_frames[d_frame_of_track[n]] -- bit-identical to fear_crop_resize_u8 with the host's crop_params (and so to
 * cv2).  Tracks with index -1 are skipped (their crop and state are left untouched).  Search crops: out_size 256,
 * context = search_context; template crops: 128, template_bbox_offset. */
int fear_track_crops_u8(const FearFrame* d_frames, int F, const int32_t* d_frame_of_track, FearTrack* d_tracks, int N,
                        int out_size, double context, uint8_t* d_crops, void* stream);
/* For every track n with d_frame_of_track[n] >= 0: box = clamp_bbox(rescale_bbox(d_boxes[n], (cx, cy, cw, ch),
 * instance_size), frame size of d_frames[d_frame_of_track[n]]) bit for bit (image_ops), written into x..h.
 * Frame indices are not bounds-checked here: pass the table fear_track_crops_u8 accepted. */
int fear_track_advance(const FearBox* d_boxes, const FearFrame* d_frames, const int32_t* d_frame_of_track,
                       FearTrack* d_tracks, int N, int instance_size, void* stream);

/* Decode maps produced elsewhere: bbox (B,4,16,16), cls logits (B,1,16,16) -> boxes[B].
 * apply_sigmoid = 0 treats cls as already-activated scores (decode(use_sigmoid=False)). */
int fear_decode(const float* d_bbox, const float* d_cls, int B, int apply_sigmoid, FearBox* d_boxes,
                void* stream);

/* z (Bz,256,64), x (B,256,256)  [= (B,256,16,16)]  ->  out (B,320,256):
 * out[:, :256] = x ; out[b, 256+k, p] = sum_c z[b,c,k] * x[b,c,p].   (blocks.py:121-124)
 * Workspace-free compatibility form: a direct CUDA-core kernel on the reference layouts (one D2D copy + one launch). */
int fear_corr_concat_f32(const float* d_z, int Bz, const float* d_x, int B, float* d_out, void* stream);
/* Same result through the hot path's tcgen05 kernel (layout changes in the caller's scratch: d_workspace must be
 * 1024-byte aligned and hold fear_corr_concat_workspace_bytes(B, Bz) bytes). */
size_t fear_corr_concat_workspace_bytes(int B, int Bz);
int fear_corr_concat_ws_f32(const float* d_z, int Bz, const float* d_x, int B, float* d_out, void* d_workspace,
                            size_t workspace_bytes, void* stream);

/* Channels-last core of the same contraction (the kernel the hot path launches):
 * zt (Bz,64,256) [k][c], cat (B,256,320) [p][c'] whose first 256 channels hold x;
 * writes cat[b, p, 256+k] = sum_c zt[b,k,c] * cat[b,p,c]. */
int fear_corr_nhwc_f32(const float* d_zt, int Bz, float* d_cat, int B, void* stream);

/* ---- introspection (tests / bench) ---------------------------------------------------*/
/* Select a kernel implementation for a stage by name.  Returns FEAR_EINVAL for unknown names.
 * Default = best validated implementation; every alternative is parity-tested against it.
 *   "corr", "pw"   : "auto" | "ffma" | "tcgen05"                  (correlation / 1x1 convs; ffma = CUDA-core baseline)
 *   "dw"           : "auto" | "pixel" | "strip" | "roll" | "tma"  (depthwise)
 *   "fuse_stem"    : "1" (default) stem + xif1_0 in one kernel | "0" four separate kernels
 *   "fuse_irf"     : "1" (default) xif2_0 (expand 1x1 -> depthwise 3x3 s2 -> project 1x1) in ONE tcgen05 kernel, the
 *                    6x expanded tensor never leaves the SM | "0" three kernels
 *   "fuse_dwpw"    : bit mask (default 15): 1 = IRF blocks on 16x16 maps, 4 = also those on 32x32 maps, 2 = head SepConvs run
 *                    their depthwise conv inside the 1x1 GEMM kernel, 8 = the expand-1 blocks (depthwise 3x3 -> 1x1 24 -> 24
 *                    -> + x) run as one CUDA-core kernel; all bit-identical to the two-kernel paths (the depthwise maps are
 *                    never written)
 *   "pw_ts"        : "1" (default) plain 1x1 GEMMs take the activation operand from tensor memory (TS-form MMA) where their
 *                    accumulators leave room for it | "0" both operands in shared memory; bit-identical
 *   "pdl"          : "1" (default) programmatic dependent launch (process-wide) */
int fear_set_option(FearContext* h, const char* key, const char* value);
/* Number of kernels launched by this handle since creation (for bench's gpu_launches). */
int64_t fear_launch_count(const FearContext* h);
/* Changes whenever the handle's workspace pointers or options change (fear_reserve growth, fear_set_option):
 * a CUDA graph captured from calls on this handle is stale once the value differs from the one seen at capture. */
int64_t fear_generation(const FearContext* h);
/* When enabled, every stage of the next calls is bracketed by CUDA events on `stream`;
 * fear_stage_ms returns accumulated milliseconds and launch counts (synchronises events). */
int fear_profile(FearContext* h, int enable);
int fear_stage_count(void);
const char* fear_stage_name(int i);
int fear_stage_ms(FearContext* h, int i, float* ms, int64_t* launches);

/* Debug: run the stem + the first `nblocks` backbone blocks (0..16) on img (B,3,H,W) and return
 * that activation as NCHW; B must not exceed the reserved batch. */
int fear_debug_backbone_prefix(FearContext* h, const float* d_img, int B, int H, int W, int nblocks,
                               float* d_out, void* stream);
/* Debug: copy a head intermediate of the last fear_head / fear_track / fear_forward call as NCHW
 * (B,C,16,16): "search_features" | "cat_cls" | "cat_reg" (320 ch: encode output + correlation) |
 * "cls_dw" | "reg_dw" | "x_reg" | "cls_tower" (256 ch).  (BoxTower.forward's 3rd/4th outputs.) */
int fear_debug_head_tensor(FearContext* h, const char* name, int B, float* d_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FEAR_B200_H */
