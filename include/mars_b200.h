/*
 * mars_b200.h -- additive C-ABI entry points of libmars_b200.so (B200 build).
 *
 * Nothing here changes a signature of the reference API (include/mars_runtime.h,
 * include/mars_math.h, include/nna.h); these functions expose what the reference
 * does not have: an image batch sharded over HBM "slots", device-resident runs,
 * and the YOLO post-process (reference file-static functions) as library calls.
 * Plain pointers and sizes only -- no torch / CUDA types cross this boundary.
 */
#ifndef MARS_B200_H
#define MARS_B200_H

#include "mars_runtime.h"

#ifdef __cplusplus
extern "C" {
#endif

/* det_t of reference src/mars/mars_yolo_test.c:37 (centre box, 24 bytes) */
typedef struct { float x, y, w, h, conf; int32_t cls; } mars_det_t;
/* Detection of reference examples/yolo_detect.cpp:39-43 (corner box, 24 bytes) */
typedef struct { float x0, y0, x1, y1, confidence; int32_t class_id; } mars_box_t;

/* ---- library / device ---------------------------------------------------- */
const char *mars_b200_version(void);
/* number of visible CUDA devices, or <0 (MARS_ERR_NNA_INIT_FAILED) without a driver */
int mars_b200_device_count(void);
/* select the device used by subsequent mars_load_* calls (default: MARS_DEVICE env or 0) */
int mars_b200_set_device(int ordinal);
/* arena bytes for subsequent loads; 0 = the reference's 8 MiB literal
 * (src/mars/mars_runtime.c:209).  Also settable with MARS_ARENA_BYTES. */
void mars_b200_set_arena_bytes(size_t bytes);
/* last diagnostic of the calling thread's most recent failing call */
const char *mars_b200_last_error(void);

/* ---- whole-arena mirror control (strict drop-in / tests) ---------------- */
/* copy the host mirror (ddr_base) of image slot `slot` to the device arena / back.
 * mars_run() itself only moves the work buffers holding model inputs / outputs. */
mars_error_t mars_b200_arena_upload(mars_model_t *m, int slot);
mars_error_t mars_b200_arena_download(mars_model_t *m, int slot, void *host_dst, size_t bytes);
/* zero every work buffer of every slot (the reference never clears them; parity
 * protocol = zero at load, then compare run k against run k) */
mars_error_t mars_b200_arena_clear(mars_model_t *m);
/* run a single layer on slot 0 (per-layer parity tests; mirrors oracle_ref_run_layer) */
mars_error_t mars_b200_run_layer(mars_model_t *m, uint32_t layer);
/* per-layer schedule summary as text: kernel kind, hazard class, fusion decision */
size_t mars_b200_describe(mars_model_t *m, char *dst, size_t cap);
/* 0 = exact direct kernels only; 1 = + tcgen05 convolutions and vectorised memory-bound kernels,
 * one device op per layer (per-layer semantics kept); 2 = + SIGMOID/MUL folded into conv epilogues (whole arena
 * still byte-identical to the reference's); 3 = + stores that no later layer, no later run and no output
 * buffer can observe are dropped from fused epilogues (default; every model OUTPUT stays bit-exact) */
void mars_b200_set_opt_level(mars_model_t *m, int level);
/* 0 = reference semantics (DEPTHWISE_CONV2D is a no-op, src/mars/mars_runtime.c:1168-1170),
 * 1 = restated depthwise convolution (parity unpinned; see DESIGN.md) */
void mars_b200_set_depthwise_mode(mars_model_t *m, int mode);
/* strict mode (also MARS_STRICT=1): when a convolution cannot be planned on the tensor-core kernel the library normally
 * recompiles the whole model on the exact direct kernels (correct, ~100x slower) and says so on stderr; in strict mode the
 * call that compiles the model (mars_load_*, mars_b200_set_batch, ...) fails with MARS_ERR_LAYER_FAILED instead */
void mars_b200_set_strict(int on);
/* float32 convolutions (reference conv2d_float32_mxu, src/mars/mxu_conv.c:673-710): 2 (default; also MARS_F32_MODE) = tcgen05
 * kind::tf32 with a hi/lo operand split, three MMAs per k-step (fp32-grade products, results within ~1e-6 relative of the
 * reference's sequential fp32 sum); 1 = plain tf32 (operands rounded to 10 mantissa bits, ~5e-4 per product); 0 = the
 * exact-order fp32 kernel, bit-identical to the reference (the control) */
void mars_b200_set_f32_mode(mars_model_t *m, int mode);

/* ---- image batch ---------------------------------------------------------- */
/* allocate `capacity` image slots (each = one set of work buffers; weights shared) */
mars_error_t mars_b200_set_batch(mars_model_t *m, int capacity);
int mars_b200_get_batch(mars_model_t *m);
/* bytes of one image's input tensor 0 / output tensor 0 (numel * elem size) */
size_t mars_b200_input_bytes(mars_model_t *m);
size_t mars_b200_output_bytes(mars_model_t *m);
/* host -> slots [first, first+n): n inputs, `stride` bytes apart in host memory */
mars_error_t mars_b200_upload_inputs(mars_model_t *m, int first, int n, const void *host, size_t stride);
/* Pre-processing in front of mars_run (what the reference's caller does on the CPU, src/mars/mars_yolo_test.c:40-77 and
 * :157-165): n RGB8 frames of w x h pixels in host memory, frame_stride bytes apart, are letterboxed on the GPU into input
 * tensor 0 of slots [first, first+n): stbir_resize_uint8 (include/stb/stb_image_resize.h) semantics bit for bit, gray border
 * -17, px - 128, NCHW or NHWC as the tensor's format field says.  Replaces load_image + mars_b200_upload_inputs. */
mars_error_t mars_b200_preprocess_batch(mars_model_t *m, int first, int n, const uint8_t *frames, size_t frame_stride, int w, int h);
/* one RGB8 frame: h rows of w pixels, rows row_stride bytes apart (0 = w * 3) */
typedef struct { const uint8_t *rgb; int32_t w, h; size_t row_stride; } mars_b200_frame_t;
/* The same pre-processing for a batch of frames of any mix of sizes and row pitches, in one pass on the device; each slot's
 * tensor is byte-identical to mars_b200_letterbox of its frame alone.  Host memory; synchronous like
 * mars_b200_preprocess_batch; records each slot's frame size for the letterbox inverse (mars_b200_set_frame_size).
 * Every frame is checked first -- rgb not NULL, w, h > 0, row_stride 0 or >= w * 3, a letterbox at least one pixel wide and
 * tall -- and a rejected call writes no slot; mars_b200_last_error names the frame. */
mars_error_t mars_b200_preprocess_frames(mars_model_t *m, int first, int n, const mars_b200_frame_t *frames);
/* the same with rgb = device addresses on the model's device (e.g. a hardware decoder's output), read in place: enqueued on
 * mars_b200_compute_stream(m) and returns.  The frames must be complete before that stream reaches the launches and stay
 * valid until it has passed them; the table itself may be reused as soon as the call returns. */
mars_error_t mars_b200_preprocess_frames_device(mars_model_t *m, int first, int n, const mars_b200_frame_t *frames);
/* YUV -> RGB conversion of an NV12 frame (16.16 fixed point, no chroma interpolation: the U,V pair of a 2 x 2 block serves
 * all four pixels; mars_b200_yuv_coefficients), chosen per frame */
enum { MARS_B200_YUV_BT601_LIMITED = 0, MARS_B200_YUV_BT709_LIMITED = 1, MARS_B200_YUV_BT601_FULL = 2, MARS_B200_YUV_BT709_FULL = 3 };
/* one NV12 frame (a hardware video decoder's or a camera ISP's output): h rows of w luma bytes (y_stride apart, 0 = w), then
 * ceil(h/2) rows of ceil(w/2) interleaved U,V pairs (uv_stride apart, 0 = 2 * ceil(w/2)); the planes may sit in one allocation
 * (e.g. uv = y + pitch * aligned height) or two.  colour = MARS_B200_YUV_* */
typedef struct { const uint8_t *y, *uv; int32_t w, h; size_t y_stride, uv_stride; int32_t colour; } mars_b200_nv12_frame_t;
/* mars_b200_preprocess_frames from NV12 frames: each slot's tensor is byte-identical to that of the RGB8 frame the conversion
 * gives, letterboxed by mars_b200_preprocess_frames.  The conversion happens where the resize reads each source pixel; no RGB
 * copy is made.  Every frame is checked first -- y and uv not NULL, w, h > 0, y_stride 0 or >= w, uv_stride 0 or
 * >= 2 * ceil(w/2), colour a MARS_B200_YUV_* value, a letterbox at least one pixel wide and tall -- and a rejected call writes
 * no slot; mars_b200_last_error names the frame.  Host memory, synchronous; records each slot's frame size. */
mars_error_t mars_b200_preprocess_frames_nv12(mars_model_t *m, int first, int n, const mars_b200_nv12_frame_t *frames);
/* the same with both planes in device memory of the model's device (e.g. an NVDEC surface), read in place: enqueued on
 * mars_b200_compute_stream(m), as mars_b200_preprocess_frames_device */
mars_error_t mars_b200_preprocess_frames_nv12_device(mars_model_t *m, int first, int n, const mars_b200_nv12_frame_t *frames);
/* host half, no GPU needed: out[6] = y0, cy, crv, cgu, cgv, cbu of a colour variant, with R = clamp((cy (Y - y0) + crv (V - 128)
 * + 32768) >> 16), G = clamp((cy (Y - y0) - cgu (U - 128) - cgv (V - 128) + 32768) >> 16), B = clamp((cy (Y - y0) + cbu (U - 128)
 * + 32768) >> 16).  Returns 0, or -1 for an unknown variant. */
int mars_b200_yuv_coefficients(int colour, int32_t *out);
/* slots -> host: output tensor 0 of n images */
mars_error_t mars_b200_download_outputs(mars_model_t *m, int first, int n, void *host, size_t stride);
/* run all layers for slots [first, first+n) with inputs already resident in HBM */
mars_error_t mars_b200_run_resident(mars_model_t *m, int first, int n);
/* decode + NMS on the device for slots [first, first+n); results stay resident */
mars_error_t mars_b200_detect_resident(mars_model_t *m, int first, int n, float nms_thresh);
/* copy the detections of slots [first, first+n) to the host:
 * dets[n][maxd] (maxd <= 1000), counts[n] */
mars_error_t mars_b200_download_detections(mars_model_t *m, int first, int n, mars_det_t *dets, int32_t *counts, int maxd);
/* end to end from host buffers: H2D, all layers, decode, NMS, D2H (pipelined in chunks) */
mars_error_t mars_b200_detect_batch(mars_model_t *m, int n, const void *inputs, size_t in_stride,
                                    mars_det_t *dets, int32_t *counts, int maxd, float nms_thresh);
/* asynchronous form: queue a batch of up to capacity/2 images on half `pool` (0 or 1) of the slot pool and return;
 * mars_b200_wait_batch(pool) blocks until its detections are in dets/counts.  Submitting to one half while the other
 * computes overlaps the host->device copy and the read-back with the kernels.  Buffers must stay valid (pinned memory,
 * e.g. nna_malloc, for true overlap) until the wait returns. */
mars_error_t mars_b200_submit_batch(mars_model_t *m, int pool, int n, const void *inputs, size_t in_stride,
                                    mars_det_t *dets, int32_t *counts, int maxd, float nms_thresh);
mars_error_t mars_b200_wait_batch(mars_model_t *m, int pool);
/* the same without the YOLO post-process: output tensor 0 of every image is read back (out_stride bytes apart); waited for
 * with mars_b200_wait_batch like a detection batch */
mars_error_t mars_b200_submit_run_batch(mars_model_t *m, int pool, int n, const void *inputs, size_t in_stride, void *outputs, size_t out_stride);
/* end to end from host buffers returning raw output tensor 0 per image */
mars_error_t mars_b200_run_batch(mars_model_t *m, int n, const void *inputs, size_t in_stride,
                                 void *outputs, size_t out_stride);
/* run all layers, then (with_detect) decode + NMS, as ONE device-timed region */
mars_error_t mars_b200_step_resident(mars_model_t *m, int first, int n, float nms_thresh, int with_detect);
/* the same step without the host synchronisation: returns once the work is enqueued on the model's compute stream
 * (mars_b200_compute_stream); the caller orders its own work behind it there -- e.g. the NCCL gather of the records -- and waits itself */
mars_error_t mars_b200_enqueue_step_resident(mars_model_t *m, int first, int n, float nms_thresh, int with_detect);
/* device addresses of the resident detection records, for a device-side gather (NCCL):
 * dets = mars_det_t[capacity][*stride_dets], counts = int32[capacity] */
void mars_b200_detections_device(mars_model_t *m, void **dets, void **counts, int *stride_dets);

/* ---- YOLOv5 Detect heads on the batched path ------------------------------------------------------------------------------ */
/* A compiler-emitted YOLOv5 .mars file keeps only the three raw head convolutions of its Detect block; output0 then holds stale
 * bytes (the Split / Pow / Constant nodes are dropped).  These calls decode the heads inside the program instead: right after each
 * head conv the anchor grid of examples/yolo_detect.cpp:176-181 (mgk-decompiler/test_yolo_inference.py:136-202) turns it into
 * corner-box candidates (at most 1000 per image over the three levels), then the corner NMS of examples/yolo_detect.cpp:152-173
 * and, for slots with a frame size, the letterbox inverse of :208-227 give mars_box_t records. */
/* host only: tensor ids (mars_tensor_t.id) of the outputs of the three CONV2D layers of a YOLOv5 Detect block, stride 8 / 16 / 32
 * (int8, 3 (5 + nc) channels, NCHW [1,C,gh,gw] or NHWC [1,gh,gw,C], input size / grid in {8, 16, 32}).  Returns 3, or 0 without heads */
int mars_b200_find_yolo_heads(const void *data, size_t size, uint32_t *tensor_ids, int cap);
/* decode these heads (level 0, 1, 2 = stride 8, 16, 32) inside every run; tensor_ids = NULL: mars_b200_find_yolo_heads, n = 0: off
 * (the default; the program is then the one without heads).  MARS_ERR_INVALID_TENSOR (mars_b200_last_error) when a tensor is not a
 * conv output, has the wrong channel count or grid, a scale <= 0, or the heads are not produced in level order.  Recompiles and
 * drops captured graphs like mars_b200_set_opt_level. */
mars_error_t mars_b200_set_yolo_heads(mars_model_t *m, const uint32_t *tensor_ids, int n, float conf_thresh);
/* NanoDet GFL heads (this library's decode; the reference has no NanoDet code).  A GFL head is the int8 output of the 1x1 conv
 * NanoDet shares between classification and regression, NCHW [1,C,gh,gw] or NHWC [1,gh,gw,C] with C = nc + 4 (reg_max + 1): nc
 * class logits, then the distributions of the left, top, right and bottom distances, reg_max + 1 bins each.  Level k has stride
 * 8 << k; 3 levels (NanoDet-m) or 4 (NanoDet-Plus).  Per cell: score = max over classes of sigmoid (label = the first class with
 * that score), a candidate when score > conf_thresh; each distance is the expectation of the softmax of its bins, times the
 * stride; the box is (cx - l, cy - t, cx + r, cy + b) clipped to the input, cx = (x + 0.5) * stride with
 * MARS_B200_GFL_CENTRE_HALF (NanoDet-m), x * stride with MARS_B200_GFL_CENTRE_CORNER (NanoDet-Plus).  Every operation is one
 * float32 rounding, exponentials come from host-built tables: the result is bit-exact to the C statement.  Candidates (at most
 * 1000 per image, in (level, y, x) order) then go through the same corner NMS and letterbox inverse as the YOLOv5 heads, so
 * every heads entry point below serves a model with GFL heads set. */
#define MARS_B200_GFL_CENTRE_HALF 0
#define MARS_B200_GFL_CENTRE_CORNER 1
/* host only: tensor ids of the GFL head convs in stride order: per stride 8 / 16 / 32 / 64 the last 1x1 CONV2D without activation
 * and without a compute reader that has nc + 4 (reg_max + 1) channels.  Returns 3 or 4, or 0 when the strides are not 8, 16, 32
 * (, 64) */
int mars_b200_find_gfl_heads(const void *data, size_t size, int nc, int reg_max, uint32_t *tensor_ids, int cap);
/* decode these heads (n = 3 or 4, level k = stride 8 << k) inside every run, replacing YOLO heads if set; tensor_ids = NULL (n != 0):
 * mars_b200_find_gfl_heads; n = 0: off.  MARS_ERR_INVALID_TENSOR (mars_b200_last_error) when a tensor is not an int8 4-D conv
 * output, has the wrong channel count or grid, a scale <= 0 or not finite, lives in the weight blob, or the heads are not produced
 * in level order; when nc < 1, reg_max is outside 1..16, centre is unknown or conf_thresh is not finite.  Recompiles and drops
 * captured graphs only when something changed. */
mars_error_t mars_b200_set_gfl_heads(mars_model_t *m, const uint32_t *tensor_ids, int n, int nc, int reg_max, int centre,
                                     float conf_thresh);
/* original frame size of slots [first, first+n) for the letterbox inverse (0 x 0: keep network coordinates, the default).
 * mars_b200_preprocess_batch and the frames calls record it as well. */
mars_error_t mars_b200_set_frame_size(mars_model_t *m, int first, int n, int w, int h);
/* corner NMS + letterbox inverse on the candidates of the last pass of slots [first, first+n); results stay resident */
mars_error_t mars_b200_detect_heads_resident(mars_model_t *m, int first, int n, float nms_thresh);
/* all layers (with the head decodes), NMS and the letterbox inverse as one device-timed region; a CUDA graph from the second call on */
mars_error_t mars_b200_step_heads_resident(mars_model_t *m, int first, int n, float nms_thresh);
mars_error_t mars_b200_enqueue_step_heads_resident(mars_model_t *m, int first, int n, float nms_thresh);
/* mars_b200_submit_batch with the heads decode: boxes[n][maxd], counts[n]; waited for with mars_b200_wait_batch */
mars_error_t mars_b200_submit_heads_batch(mars_model_t *m, int pool, int n, const void *inputs, size_t in_stride, mars_box_t *boxes,
                                          int32_t *counts, int maxd, float nms_thresh);
/* mars_b200_submit_heads_batch from n host frames (mars_b200_preprocess_frames): H2D of each frame on the copy stream, the
 * letterbox, layers, heads, NMS and the letterbox inverse on the compute stream, D2H of the boxes -- in each frame's own
 * coordinates.  The frames, boxes and counts must stay valid until mars_b200_wait_batch(pool) returns; the frames must be
 * pinned (e.g. nna_malloc) for their upload to overlap the kernels.  Each pool keeps device staging for its frames and
 * pinned staging for its descriptor table, sized by the largest batch so far: a batch that needs more grows it, which waits
 * for the device once. */
mars_error_t mars_b200_submit_frames_heads_batch(mars_model_t *m, int pool, int n, const mars_b200_frame_t *frames,
                                                 mars_box_t *boxes, int32_t *counts, int maxd, float nms_thresh);
/* the same from n host NV12 frames (mars_b200_preprocess_frames_nv12): both planes of each frame are uploaded on the copy
 * stream -- half the bytes of the RGB8 frame -- and converted inside the letterbox */
mars_error_t mars_b200_submit_frames_nv12_heads_batch(mars_model_t *m, int pool, int n, const mars_b200_nv12_frame_t *frames,
                                                      mars_box_t *boxes, int32_t *counts, int maxd, float nms_thresh);
/* kept boxes of slots [first, first+n): boxes[n][maxd] (maxd <= 1000), counts[n] */
mars_error_t mars_b200_download_boxes(mars_model_t *m, int first, int n, mars_box_t *boxes, int32_t *counts, int maxd);

/* ---- tiled (sliced) detection on high-resolution frames --------------------------------------------------------------------
 * A 3840x2160 frame fitted whole into a 640x640 input is shrunk 6 times; small objects vanish.  These calls letterbox regions of
 * interest of the frames -- typically overlapping tiles, plus the whole frame -- into one slot each, run the heads step on the
 * slots, shift each region's kept boxes back into its frame and merge them per frame with the corner NMS of
 * examples/yolo_detect.cpp:152-173.  Tiling and the merge are this library's additions (the reference has neither); the merge's
 * NMS is the reference's nms.  Regions of one frame are contiguous in the region table; their order fixes the order in which
 * their boxes are concatenated for the merge. */
/* one region of interest of frame `frame` (an index into the call's frame table): the w x h pixels at (x, y) */
typedef struct { int32_t frame, x, y, w, h; } mars_b200_roi_t;
/* host only, no GPU: the tile grid of a w x h frame.  Along x the step is tile_w - overlap_w; there is one column when
 * w <= tile_w, else ceil((w - tile_w) / step) + 1; column i starts at min(i * step, w - tile_w) (the last is flush with the right
 * edge) and is min(tile_w, w) wide.  The same along y.  Tiles in row-major order; with_full and more than one tile: the whole
 * frame comes first as one more region.  Returns the count (when it exceeds cap nothing is written), or -1 for non-positive
 * sizes, a negative overlap or an overlap not smaller than its tile.  3840x2160, 640x640 tiles, overlap 128: 8 x 4 = 32 tiles. */
int mars_b200_tile_rois(int frame, int w, int h, int tile_w, int tile_h, int overlap_w, int overlap_h, int with_full,
                        mars_b200_roi_t *out, int cap);
/* Letterboxes region r of rois into input tensor 0 of slot first + r: byte-identical to mars_b200_letterbox of the cropped frame
 * frame[y:y+h, x:x+w] (for NV12, of the same crop of the RGB8 frame the conversion gives; chroma comes from the frame's own 2 x 2
 * blocks, so odd origins are exact).  Each slot records the region's size as its frame size, so the letterbox inverse gives
 * boxes in region coordinates.  Each frame is uploaded once, however many regions it has.  Every frame and region is checked
 * first -- the frame checks of mars_b200_preprocess_frames, frame in [0, n_frames) and not decreasing, x, y >= 0, w, h > 0,
 * inside its frame, a letterbox at least one pixel wide and tall, n_rois slots in range -- and a rejected call writes no slot;
 * mars_b200_last_error names the frame or region.  Host RGB8 frames, synchronous. */
mars_error_t mars_b200_preprocess_rois(mars_model_t *m, int first, int n_frames, const mars_b200_frame_t *frames, int n_rois,
                                       const mars_b200_roi_t *rois);
/* the same from NV12 frames in device memory of the model's device, read in place: enqueued on mars_b200_compute_stream(m) */
mars_error_t mars_b200_preprocess_rois_nv12_device(mars_model_t *m, int first, int n_frames, const mars_b200_nv12_frame_t *frames,
                                                   int n_rois, const mars_b200_roi_t *rois);
/* After a heads step on slots [first, first+n_rois) (mars_b200_step_heads_resident or the enqueue form): for each frame f the
 * kept boxes of its regions' slots, in region order and each slot's kept order, shifted into frame coordinates (x + (float)roi.x,
 * y + (float)roi.y), capped at the first 1000 by descending confidence (ties in that order), then the corner NMS (same class,
 * IoU > merge_thresh) -> frame record first + f (mars_b200_download_frame_boxes).  The slots' own boxes stay as they are.
 * Enqueued on mars_b200_compute_stream(m). */
mars_error_t mars_b200_merge_rois_resident(mars_model_t *m, int first, int n_frames, int n_rois, const mars_b200_roi_t *rois,
                                           float merge_thresh);
/* merged boxes of frame records [first, first+n): boxes[n][maxd] (maxd <= 1000), counts[n] */
mars_error_t mars_b200_download_frame_boxes(mars_model_t *m, int first, int n, mars_box_t *boxes, int32_t *counts, int maxd);
/* The whole flow on one pool: the n_frames host frames uploaded once each and the region and merge tables in one pinned upload,
 * on the copy stream; then on the compute stream the letterbox of n_rois slots, the (graphed) heads step on them and the merge;
 * then the D2H of the n_frames frame records.  boxes[n_frames][maxd], counts[n_frames], in frame coordinates; waited for with
 * mars_b200_wait_batch.  n_rois and n_frames must fit half the slot pool.  Nothing returns to the host in between. */
mars_error_t mars_b200_submit_rois_heads_batch(mars_model_t *m, int pool, int n_frames, const mars_b200_frame_t *frames, int n_rois,
                                               const mars_b200_roi_t *rois, mars_box_t *boxes, int32_t *counts, int maxd,
                                               float nms_thresh, float merge_thresh);
/* the same from host NV12 frames (both planes uploaded, converted inside the letterbox) */
mars_error_t mars_b200_submit_rois_nv12_heads_batch(mars_model_t *m, int pool, int n_frames, const mars_b200_nv12_frame_t *frames,
                                                    int n_rois, const mars_b200_roi_t *rois, mars_box_t *boxes, int32_t *counts,
                                                    int maxd, float nms_thresh, float merge_thresh);

/* ---- multi-object tracking of camera streams -------------------------------------------------------------------------------
 * A tracker per camera stream whose state stays on the device: after a heads step, one CTA per stream turns the frame's kept
 * corner boxes into tracked boxes with persistent IDs.  The schedule is ByteTrack's (Zhang et al., ECCV 2022): high-score
 * detections (conf > high_thresh) are matched first to the Tracked and Lost tracks predicted by ByteTrack's Kalman filter, with
 * similarity IoU * conf; low-score detections (low_thresh < conf < high_thresh) then keep the still unmatched Tracked tracks
 * alive, with similarity IoU; the high-score detections left over are matched to the unconfirmed tracks (born on an earlier frame
 * but not yet matched again), and the rest with conf >= new_thresh start tracks.  Matching is greedy under a strict total order
 * -- the admissible pair (similarity > gate, both unused, equal classes with class_aware) with the largest similarity first,
 * ties by the smaller track_id, then the smaller detection index -- where ByteTrack solves an optimal assignment.  A track lost
 * for more than max_lost frames is removed; an unconfirmed track that misses once is removed.  All arithmetic is float32 with
 * one rounding per operation: the results are bit-exact to the C statement of the definition (tests/track_oracle.c).  Boxes with
 * a non-finite value or a non-positive width or height are ignored.  Track IDs start at 1 per stream. */
#define MARS_B200_MAX_TRACKS 256
/* one tracked object of a frame: the filter's box after this frame's update, and the confidence, class and index (in the frame's
 * kept boxes) of the detection it was matched to (32 bytes) */
typedef struct { float x0, y0, x1, y1, confidence; int32_t class_id, track_id, det_index; } mars_b200_track_box_t;
typedef struct {
    float high_thresh, low_thresh, new_thresh; /* detection classes and the birth threshold */
    float sim_high, sim_low, sim_unconfirmed;  /* gates of the three matchings, in [0, 1) */
    int32_t max_lost, class_aware;             /* frames a lost track survives (>= 0); 1: only equal classes match */
} mars_b200_track_params_t;
#define MARS_B200_TRACK_PARAMS_DEFAULT {0.5f, 0.1f, 0.6f, 0.2f, 0.5f, 0.3f, 30, 0}
/* tracker state for n_streams streams, all reset (frame 0, next ID 1); n_streams = 0 frees it; p = NULL: the defaults.
 * MARS_ERR_INVALID_TENSOR when a parameter is not finite, low_thresh < 0 or > high_thresh, a gate is outside [0, 1), max_lost < 0 or
 * class_aware is not 0 or 1.  Waits for the compute stream. */
mars_error_t mars_b200_set_tracking(mars_model_t *m, int n_streams, const mars_b200_track_params_t *p);
/* streams [first_stream, first_stream + n) start over (frame 0, next ID 1); enqueued on the compute stream */
mars_error_t mars_b200_reset_tracks(mars_model_t *m, int first_stream, int n);
/* after a heads step on slots [first, first+n): the kept boxes of slot first + i are the next frame of stream streams[i]; its
 * tracked boxes go to track record first + i (mars_b200_download_tracks).  Enqueued on the compute stream.  Every call checks
 * first that tracking is set, the slots are in range, heads are configured and every stream id is in [0, n_streams) and named
 * once; a rejected call changes no stream (mars_b200_last_error names the entry). */
mars_error_t mars_b200_track_resident(mars_model_t *m, int first, int n, const int32_t *streams);
/* tracked boxes of track records [first, first+n): out[n][maxd] (maxd <= 256), counts[n] */
mars_error_t mars_b200_download_tracks(mars_model_t *m, int first, int n, mars_b200_track_box_t *out, int32_t *counts, int maxd);
/* the same kernel on detections from the host: entry i is the next frame of stream streams[i], with counts[i] (0..min(box_stride,
 * 1000)) boxes at boxes + i * box_stride; out[n][maxd], out_counts[n].  Synchronous; needs no heads and no slots. */
mars_error_t mars_b200_track_boxes(mars_model_t *m, int n, const int32_t *streams, const mars_box_t *boxes, const int32_t *counts,
                                   int box_stride, mars_b200_track_box_t *out, int32_t *out_counts, int maxd);
/* mars_b200_submit_frames_heads_batch followed by the tracker on the pool's slots (frame i = the next frame of stream streams[i]):
 * out[n][maxd] tracked boxes in frame coordinates and counts[n] are read back instead of the boxes; waited for with
 * mars_b200_wait_batch.  The stream table travels in the pool's pinned upload.  Both pools use the compute stream, so the track
 * kernels run in submit order and a stream may appear in consecutive submits on alternating pools. */
mars_error_t mars_b200_submit_frames_track_batch(mars_model_t *m, int pool, int n, const mars_b200_frame_t *frames, const int32_t *streams,
                                                 mars_b200_track_box_t *out, int32_t *counts, int maxd, float nms_thresh);
mars_error_t mars_b200_submit_frames_nv12_track_batch(mars_model_t *m, int pool, int n, const mars_b200_nv12_frame_t *frames,
                                                      const int32_t *streams, mars_b200_track_box_t *out, int32_t *counts, int maxd,
                                                      float nms_thresh);

/* ---- zones and counting lines on tracked streams ----------------------------------------------------------------------------
 * Line-crossing counts, zone occupancy and enter / dwell / exit events per tracker stream, computed on the device right after the
 * tracker, with the per-track state in HBM.  This is the library's own definition; the C statement is tests/zones_oracle.c and
 * the device equals it byte for byte.
 *
 * Geometry is set per tracker stream (mars_b200_set_zones), in the coordinates of the tracked boxes: frame coordinates for slots
 * with a frame size, network coordinates otherwise.  A zone is a polygon of 3..16 vertices with a class (-1: any), an anchor and
 * min_dwell (frames; 0: no dwell events).  A line is a directed segment (x0, y0) -> (x1, y1) with distinct ends, a class and an
 * anchor.  A track is "shown" in a frame when the tracker outputs it in that frame (Tracked and confirmed); its anchor is taken
 * from its tracked box (mars_b200_track_box_t after this frame's update):
 *   MARS_B200_ANCHOR_BOTTOM  ((x0 + x1) * 0.5f, y1)        MARS_B200_ANCHOR_CENTRE  ((x0 + x1) * 0.5f, (y0 + y1) * 0.5f)
 * All arithmetic is float32, one rounding per operation, in the order written.  A class matches when the geometry's class is -1
 * or equals the track's class in this frame.
 *   inside(P, px, py) (crossing number, even-odd): for i = 0 .. n-1 and j = (i + n - 1) mod n, toggle when (yi > py) != (yj > py)
 *     and px < xi + ((xj - xi) * (py - yi)) / (yj - yi).
 *   side(L, px, py): the sign (+1, -1, 0) of (x1 - x0) * (py - y0) - (y1 - y0) * (px - x0); +1 is the right-hand side walking
 *     from end 0 to end 1 on screen (y down).
 *   crossing: per (track, line) sigma is the last non-zero side seen at a shown frame (0: none yet).  At a shown frame with anchor
 *     q, the track shown before with anchor p, a crossing counts when side(q) != 0, sigma == -side(q), the class matches, and the
 *     step meets the closed segment: o_a = (qx - px) * (ay - py) - (qy - py) * (ax - px) and o_b (the same with end b) are not both
 *     > 0 and not both < 0.  A crossing to +1 is CROSS_POS, to -1 CROSS_NEG.  Then sigma = side(q) when that is non-zero, whatever
 *     the class.  So walking around a line's end never counts, stopping on the line and going on counts once, and a crossing made
 *     during a lost gap counts when the track is shown again.  There is no debouncing: a track jittering over a line counts each
 *     crossing.
 *   zones: membership is evaluated at shown frames only: inside(anchor) and the class matches.  A track not shown in a frame
 *     (Lost, or not confirmed yet) keeps its state.  ENTER: inside now and not at the previous shown frame (value 1 at the track's
 *     first shown frame since the stream's analytics started, else 0); the entry frame is recorded.  DWELL: once per stay, at the
 *     first shown frame with frame - entry + 1 >= min_dwell > 0 (value: that number).  EXIT: inside before, shown outside now
 *     (value frame - entry).  GONE: the tracker removed a track that was inside (value frame - entry, the last class known); its
 *     analytics state is then dropped.
 *   occupancy of a zone: the tracks shown in the frame that are inside it.  Line totals: CROSS_POS and CROSS_NEG counts since
 *     mars_b200_set_zones or mars_b200_reset_tracks on that stream.
 *   events of a frame in order: ascending track_id (removed tracks included); within a track its crossings in line order, then its
 *     zone events in zone order; within a zone ENTER before DWELL (both in one frame when min_dwell == 1).  The first
 *     MARS_B200_MAX_ZONE_EVENTS are written; n_events is the full count.  A crossing's value is the line's total of that
 *     direction after it; GONE, EXIT, ENTER and DWELL have index = the zone, crossings index = the line.
 * `frame` of a record is the tracker's frame number of the stream.  A record of a stream without geometry has its frame number,
 * zeros and no events. */
#define MARS_B200_MAX_ZONES 8
#define MARS_B200_MAX_ZONE_VERTS 16
#define MARS_B200_MAX_LINES 8
#define MARS_B200_MAX_ZONE_EVENTS 128
enum { MARS_B200_ANCHOR_BOTTOM = 0, MARS_B200_ANCHOR_CENTRE = 1 };
enum { MARS_B200_ZONE_ENTER = 0, MARS_B200_ZONE_DWELL = 1, MARS_B200_ZONE_EXIT = 2, MARS_B200_ZONE_GONE = 3, MARS_B200_CROSS_POS = 4,
       MARS_B200_CROSS_NEG = 5 };
typedef struct {
    float x[MARS_B200_MAX_ZONE_VERTS], y[MARS_B200_MAX_ZONE_VERTS]; /* vertices 0 .. n_verts-1 */
    int32_t n_verts, class_id, anchor, min_dwell;
} mars_b200_zone_t; /* 144 bytes */
typedef struct { float x0, y0, x1, y1; int32_t class_id, anchor; } mars_b200_line_t; /* 24 bytes */
typedef struct { int32_t track_id, class_id; int16_t kind, index; int32_t value; } mars_b200_zone_event_t; /* 16 bytes */
typedef struct {
    int32_t frame, n_events;
    int32_t occupancy[MARS_B200_MAX_ZONES];                      /* this frame */
    int32_t crossed_pos[MARS_B200_MAX_LINES], crossed_neg[MARS_B200_MAX_LINES]; /* line totals after this frame */
    mars_b200_zone_event_t events[MARS_B200_MAX_ZONE_EVENTS];
} mars_b200_zone_frame_t; /* 2152 bytes */
/* geometry of tracker stream `stream`; its analytics state and line totals start over.  n_zones = n_lines = 0 switches the stream
 * off.  Needs tracking set (mars_b200_set_tracking, which drops all geometry); waits for the compute stream.  Everything is checked
 * first (stream in range, counts within the limits, 3..16 vertices, finite coordinates, class_id >= -1, a known anchor, min_dwell >=
 * 0, distinct line ends): a rejected call changes nothing and mars_b200_last_error names the zone or line and the field.  While any
 * stream has geometry, every tracker call (resident, host boxes, submits) runs the analytics after the tracker, so each stream's
 * analytics see every frame; mars_b200_reset_tracks clears the analytics state and totals of its streams, not their geometry. */
mars_error_t mars_b200_set_zones(mars_model_t *m, int stream, const mars_b200_zone_t *zones, int n_zones, const mars_b200_line_t *lines,
                                 int n_lines);
/* zone records of track records [first, first+n), as the last mars_b200_track_resident or track submit on those slots wrote them.
 * Those calls write the records only while some stream has geometry (so that, with none, they launch what they launched before
 * zones existed); a slot not written since keeps its earlier record, or zeros from mars_b200_set_batch */
mars_error_t mars_b200_download_zones(mars_model_t *m, int first, int n, mars_b200_zone_frame_t *out);
/* mars_b200_track_boxes, plus zone_out[n] (NULL: none): the analytics run in this call even when no stream has geometry */
mars_error_t mars_b200_track_boxes_zones(mars_model_t *m, int n, const int32_t *streams, const mars_box_t *boxes, const int32_t *counts,
                                         int box_stride, mars_b200_track_box_t *out, int32_t *out_counts, int maxd,
                                         mars_b200_zone_frame_t *zone_out);
/* mars_b200_submit_frames[_nv12]_track_batch, plus zones[n]: the zone record of every frame, in the same read-back (waited for with
 * mars_b200_wait_batch) */
mars_error_t mars_b200_submit_frames_zones_batch(mars_model_t *m, int pool, int n, const mars_b200_frame_t *frames, const int32_t *streams,
                                                 mars_b200_track_box_t *out, int32_t *counts, int maxd, mars_b200_zone_frame_t *zones,
                                                 float nms_thresh);
mars_error_t mars_b200_submit_frames_nv12_zones_batch(mars_model_t *m, int pool, int n, const mars_b200_nv12_frame_t *frames,
                                                      const int32_t *streams, mars_b200_track_box_t *out, int32_t *counts, int maxd,
                                                      mars_b200_zone_frame_t *zones, float nms_thresh);

/* ---- several GPUs of one box behind one call (batch sharded over the devices, no inter-GPU traffic on the path) ---------- */
typedef struct mars_b200_group mars_b200_group_t;
/* one replica of the model per device (devices = NULL: ordinals 0 .. n_devices-1), `per_gpu_batch` image slots each */
mars_error_t mars_b200_group_load(const void *data, size_t size, const int *devices, int n_devices, int per_gpu_batch, mars_b200_group_t **out);
void mars_b200_group_free(mars_b200_group_t *g);
int mars_b200_group_size(mars_b200_group_t *g);
/* the replica on the i-th device of the group (for per-device settings: opt level, f32 mode, ...) */
mars_model_t *mars_b200_group_model(mars_b200_group_t *g, int i);
/* mars_b200_detect_batch over the whole group: image b runs on GPU b / ceil(n / G), one host thread per GPU; dets[n][maxd] and
 * counts[n] are filled directly by every GPU's read-back (the single-process form of the detection gather) */
mars_error_t mars_b200_group_detect_batch(mars_b200_group_t *g, int n, const void *inputs, size_t in_stride, mars_det_t *dets, int32_t *counts,
                                          int maxd, float nms_thresh);

/* ---- introspection (tests, bench) ----------------------------------------- */
/* record CUDA events around every device op of full passes; read back with mars_b200_op_info */
void mars_b200_set_profile(mars_model_t *m, int on);
int mars_b200_num_ops(mars_model_t *m);
/* info[0..12] = kind, layer, impl, mode, ic, oc, oh, ow, kh, kw, fused_layers, ih, iw */
int mars_b200_op_info(mars_model_t *m, int op, int32_t *info, double *ms, uint64_t *calls, uint64_t *flat_n);
/* out5 = weights_size, buffer_size, num_buffers, slot_stride, arena_size */
void mars_b200_geometry(mars_model_t *m, size_t *out5);
/* arena offset of tensor table entry `index` (reference planner, src/mars/mars_runtime.c:248-337) */
size_t mars_b200_tensor_offset(mars_model_t *m, uint32_t index);

/* the CUDA stream (cudaStream_t) the model's kernels run on; work enqueued there by the caller (e.g. an NCCL gather of the
 * resident detection records) is ordered between the batches */
void *mars_b200_compute_stream(mars_model_t *m);
/* kernels launched by this model since load (the bench's gpu_launches claim) */
uint64_t mars_b200_launch_count(mars_model_t *m);
/* CUDA-event time of the last mars_b200_run_resident / detect_resident, milliseconds */
float mars_b200_last_gpu_ms(mars_model_t *m);

/* ---- YOLO pre-process on host buffers ------------------------------------ */
/* load_image of reference src/mars/mars_yolo_test.c:40-77 without the file decode: rgb = h x w x 3 bytes in,
 * out = tw x th x 3 int8 (three planes, or interleaved when nhwc != 0).  Returns 0 on success, -1 on failure. */
int mars_b200_letterbox(const uint8_t *rgb, int w, int h, int tw, int th, int nhwc, int8_t *out);
/* load_and_preprocess_image of reference examples/yolo_detect.cpp:72-130 without the file decode: the same resize into an
 * RGBA uint8 frame, out = tw x th x 4 bytes (the reference fixes 640 x 640): 114 everywhere outside the image (alpha
 * included), R, G, B, 0 inside.  Returns 0 on success, -1 on failure. */
int mars_b200_letterbox_rgba(const uint8_t *rgb, int w, int h, int tw, int th, uint8_t *out);
/* host half of the above (no GPU needed): the (source sample, coefficient) taps each of the out_size output samples of one
 * axis sums, in the order stbir_resize_uint8 adds them.  start[out_size + 1]; returns the tap count (> cap: nothing copied). */
int mars_b200_resize_taps(int in_size, int out_size, int32_t *start, int32_t *src, float *w, int cap);

/* ---- planner (host half, no GPU needed) ----------------------------------- */
/* What the library would do with a .mars blob: the compiled op list at `opt_level` (0 exact kernels ... 3 default), one line per
 * device op with its kernel choice and the fused / linked / forwarded / elided output streams, written to dst (NUL terminated,
 * truncated to cap).  arena_bytes = 0: the reference's 8 MiB (src/mars/mars_runtime.c:209).  Returns the full length, 0 on error. */
size_t mars_b200_plan_describe(const void *data, size_t size, size_t arena_bytes, int opt_level, char *dst, size_t cap);

/* ---- conv requantisation in integers (host half, no GPU needed) ----------- */
/* The tcgen05 conv epilogue replaces the float requantisation of reference src/mars/mxu_conv.c:663-666,
 * r = clamp((int32)(fl((float)t * scale) +- 0.5f)), by clamp(floor((t * m + c) / 2^(32 + s))) when integers (m, s, c) exist that
 * reproduce it for EVERY |t| <= tmax (t = accumulator + bias).  Returns 1 and fills m / s / c, or 0 when no such triple exists
 * (the layer then keeps a float variant).  Exposed so that the CPU test suite can check the fit by brute force. */
int mars_b200_requant_fit(float scale, long long tmax, int *m, int *s, long long *c);
/* the reference's requantisation of one value, restated (what the fit is checked against) */
int mars_b200_requant_ref(int t, float scale);
/* the requantisation variant the tcgen05 conv epilogue takes for conv scale `scale` and bound = max over output channels of
 * 128 * sum |w| + |bias| (read as int32): 3 integer form, 2 float half-up, 1 float with a fast conversion, 0 general float with the
 * x86 overflow rule.  A compiled model reports the variant of each such layer as " rq=N" in mars_b200_describe. */
int mars_b200_requant_variant(float scale, long long bound);

/* ---- NNA-native tensor layouts (SURVEY 8f4) -------------------------------- */
/* The layouts behind the format tags MARS_FORMAT_NMHWSOIB2 / MARS_FORMAT_NDHWC32 (reference include/mars.h:46-56), which the
 * reference's compiler can emit and its runtime only sizes (src/mars/mars_runtime.c:93-110):
 *   NMHWSOIB2 weights  [ceil(Co/32)][ceil(Ci/32)][KH][KW][32 out][32 in], 1024-byte blocks, absent channels zero
 *                      (packer: mars-compiler/src/mars_format.rs:436-470; unpackers: mgk-decompiler/mgk_decompiler.py:530-540,
 *                      mgk-decompiler/scripts/extract_weights_nmhwsoib2.py:52-80)
 *   NDHWC32 features   [N][ceil(C/32)][H][W][32], absent channels zero (mars-compiler/src/mars_format.rs:490-531)
 * Byte permutations on the device; host-buffer forms (copy in, convert, copy out) and device-resident forms (`stream` is a
 * cudaStream_t or NULL; the NDHWC32 buffer must be 16-byte aligned).  All return 0 on success, -1 on error
 * (mars_b200_last_error); the size helpers return 0 for non-positive dimensions. */
size_t mars_b200_nmhwsoib2_size(int out_ch, int in_ch, int kh, int kw);            /* mars_format.rs:472-476 */
size_t mars_b200_ndhwc32_size(int batch, int channels, int height, int width);     /* mars_format.rs:485-488 */
int mars_b200_pack_weights_nmhwsoib2(const int8_t *oihw, int out_ch, int in_ch, int kh, int kw, uint8_t *packed);
int mars_b200_unpack_weights_nmhwsoib2(const uint8_t *packed, int out_ch, int in_ch, int kh, int kw, int8_t *oihw);
int mars_b200_nchw_to_ndhwc32(const uint8_t *nchw, int batch, int channels, int height, int width, uint8_t *out);
int mars_b200_ndhwc32_to_nchw(const uint8_t *native, int batch, int channels, int height, int width, uint8_t *nchw);
int mars_b200_pack_weights_nmhwsoib2_device(const int8_t *d_oihw, int out_ch, int in_ch, int kh, int kw, uint8_t *d_packed, void *stream);
int mars_b200_unpack_weights_nmhwsoib2_device(const uint8_t *d_packed, int out_ch, int in_ch, int kh, int kw, int8_t *d_oihw, void *stream);
int mars_b200_nchw_to_ndhwc32_device(const uint8_t *d_nchw, int batch, int channels, int height, int width, uint8_t *d_out, void *stream);
int mars_b200_ndhwc32_to_nchw_device(const uint8_t *d_native, int batch, int channels, int height, int width, uint8_t *d_nchw, void *stream);

/* ---- YOLO post-process on host buffers ----------------------------------- */
/* parse_output of reference src/mars/mars_yolo_test.c:80-104 (conf threshold 0.25) */
int mars_yolo_parse_output(const int8_t *data, int npred, float scale, mars_det_t *dets, int maxd);
/* nms of reference src/mars/mars_yolo_test.c:107-130 (exchange sort + greedy, centre boxes) */
int mars_yolo_nms(mars_det_t *dets, int n, float thresh);
/* nms of reference examples/yolo_detect.cpp:152-173 (corner boxes; ties keep input order) */
int mars_yolo_nms_boxes(mars_box_t *dets, int n, float thresh);
/* scale_detections of reference examples/yolo_detect.cpp:208-227 */
void mars_yolo_scale_detections(mars_box_t *dets, int n, int orig_w, int orig_h, int net_w, int net_h);
/* anchor-grid decode (formula: mgk-decompiler/test_yolo_inference.py:136-202, anchors
 * examples/yolo_detect.cpp:176-181).  head = int8 [3,gh,gw,85]; appends after `cnt`. */
int mars_yolo_decode_anchor_grid(const int8_t *head, int gh, int gw, float scale, int level,
                                 float conf_thresh, mars_box_t *dets, int cnt, int maxd);
/* the GFL decode of mars_b200_set_gfl_heads on one head: head = int8 [gh][gw][nc + 4 (reg_max + 1)] dequantised with `scale`,
 * level stride `stride`, boxes clipped to net_w x net_h; appends after `cnt`, at most maxd in all.  Returns the new count */
int mars_b200_decode_gfl(const int8_t *head, int gh, int gw, int nc, int reg_max, float scale, int stride, int centre, int net_w,
                         int net_h, float conf_thresh, mars_box_t *dets, int cnt, int maxd);

#ifdef __cplusplus
}
#endif
#endif /* MARS_B200_H */
