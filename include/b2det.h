/*
 * b2det -- C ABI of the B200-native tile-detection engine.
 *
 * This is the drop-in boundary for the one hot path of
 * jacgeborys/aerial_image_recognition (SURVEY.md section 8b).  The reference has no
 * FFI of its own: its hot path is Python calling into the onnxruntime / OpenCV /
 * Pillow wheels.  Each entry point below therefore cites the *Python call site* it
 * replaces (file:line relative to the reference root); the ctypes binding a
 * maintainer would add is shown in INTEGRATION.md and shipped as
 * aerial_image_recognition_b200/_lib.py.
 *
 * Conventions: plain C, no C++ or torch types.  Every function returns 0 on success
 * and a negative code on failure; b2d_last_error() gives the message (thread-local).
 * Pointers named *_dev are CUDA device pointers on the engine's device, *_host are
 * host pointers.  `stream` is a cudaStream_t passed as void*.  An engine belongs to
 * one GPU and one owner thread (the reference issues all inference from one thread,
 * SURVEY.md section 8b "Threading").
 */
#ifndef B2DET_H
#define B2DET_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2D_VERSION 101

typedef struct b2d_engine b2d_engine;

/* ---- records ------------------------------------------------------------------------- */

/* One candidate / detection in model-input pixel space (32 bytes). */
typedef struct b2d_det {
    float cx, cy, w, h;   /* box centre and size, input pixels (reference rows cols 0-3)   */
    float conf;           /* reference rows col 4 (v7: objectness; v8 adapter: max class)  */
    int32_t cls;          /* best class (v8) / 0                                           */
    int32_t tile;         /* index of the tile inside the batch                            */
    int32_t anchor;       /* row index inside the tile's output (stable tie-break key)     */
} b2d_det;

/* One georeferenced detection (40 bytes). */
typedef struct b2d_geodet {
    double x, y;          /* lon/lat, or CRS metres for the affine form                    */
    float conf;
    float x_img, y_img;   /* SimpleDetector's 'image' {x,y} (simple_detector.py:490-491)   */
    float x_yolo, y_yolo; /* SimpleDetector's 'yolo'  {x,y} (simple_detector.py:500)       */
    int32_t tile;
} b2d_geodet;

/* One oriented detection of a yolov8m-obb engine in model-input pixel space (36 bytes): Ultralytics' regularized
 * rotated box (w >= h, theta in [0, pi), radians, the rotation of the w side from +x towards +y).                       */
typedef struct b2d_obb {
    float cx, cy, w, h, theta;
    float conf;           /* best class score                                              */
    int32_t cls;
    int32_t tile;
    int32_t anchor;       /* anchor index inside the tile (stable tie-break key)          */
} b2d_obb;

/* One georeferenced oriented detection (104 bytes): centre and the four corners (Ultralytics xywhr2xyxyxyxy order:
 * c+v1+v2, c+v1-v2, c-v1-v2, c-v1+v2 with v1 along w, v2 along h) in lon/lat or CRS units, box size in the
 * georeferenced form's pixels (bounds: crop pixels; affine: source-window pixels).                                     */
typedef struct b2d_geoobb {
    double x, y;
    double corners[8];    /* x0, y0, x1, y1, x2, y2, x3, y3                                */
    float conf, w, h, theta;
    int32_t cls;
    int32_t tile;
} b2d_geoobb;

/* ---- enums ----------------------------------------------------------------------------- */
enum { B2D_ACT_NONE = 0, B2D_ACT_SILU = 1 };
enum { B2D_CONV_AUTO = 0, B2D_CONV_TCGEN05 = 1 };   /* one backend: a shape the tensor-core kernels cannot run fails b2d_plan_finalize */
/* resize modes of b2d_preprocess */
enum {
    B2D_RESIZE_IDENTITY = 0,     /* input already model-sized (BASELINE configs C2/C3)            */
    B2D_RESIZE_CV2_LINEAR = 1,   /* cv2.resize(img,(640,640))      -- _script/gpu_handler.py:74-76 */
    B2D_RESIZE_PIL_BICUBIC = 2,  /* PIL Image.resize((640,640))    -- simple_detector.py:463, :655 */
    B2D_RESIZE_LETTERBOX = 3     /* Ultralytics LetterBox, pad 114 -- x_arch/02_analyze_images:1 (cell 6) */
};
enum { B2D_OUT_BF16_NHWC4 = 0, B2D_OUT_F32_NCHW = 1, B2D_OUT_U8_NHWC = 2, B2D_OUT_F16_NHWC4 = 3 };
/* head kinds: v8 DFL boxes, v7 anchor boxes, v8 oriented boxes (DFL distances + one angle logit per anchor, Ultralytics >= 8.1
 * OBB head; the angle logit is the fp32 channel (64 + nc + 3) / 4 * 4 of the head map, the first 16-byte-aligned one after the
 * 64 DFL logits and the nc class logits)                                                                                   */
enum { B2D_HEAD_V8_DFL = 0, B2D_HEAD_V7_ANCHOR = 1, B2D_HEAD_V8_OBB = 2 };
/* georeferencing forms */
enum {
    B2D_GEO_BOUNDS = 0,      /* simple_detector.py:487-494 : params = west,east,south,north,crop_size   */
    B2D_GEO_GPUHANDLER = 1,  /* _script/gpu_handler.py:182-190 : params = lon_min,lat_min,lon_max,lat_max */
    B2D_GEO_AFFINE = 2,      /* x_arch/02_analyze_images:1 (cell 6) pixel_to_geo: params = gt[6], win_x, win_y,
                                pad_x, pad_y, gain, w0, h0 (letterbox undo = Ultralytics scale_boxes) */
    B2D_GEO_TENSOR_F32 = 3   /* _script/gpu_handler.py:243-253 (_process_tensors): the float32 CUDA-tensor form of the
                                test-time-augmentation path; params = lon_min,lat_min,lon_max,lat_max           */
};
enum { B2D_COLOUR_RGB2LAB = 0, B2D_COLOUR_LAB2RGB = 1 };
#define B2D_GEO_PARAMS 16    /* doubles per tile in every form */

/* ---- engine lifetime ------------------------------------------------------------------- */
/* Replaces ort.InferenceSession(...) at _script/gpu_handler.py:61-65 and
 * simple_detector.py:39-46.  Fails (does not fall back) when no sm_100 device exists. */
int b2d_create(int device, int max_batch, b2d_engine** out);
void b2d_destroy(b2d_engine* e);
const char* b2d_last_error(void);
int b2d_version(void);
int b2d_device_sm_count(b2d_engine* e);
/* Storage format of activations and weights (accumulation is fp32 either way; head maps stay fp32).
 * B2D_PREC_BF16 is the default and the configuration BASELINE.json is quoted on; B2D_PREC_FP16 keeps three
 * more mantissa bits per stored activation (same tensor-core rate) for callers that want to sit closer to
 * the reference's fp32 onnxruntime results.  B2D_PREC_FP16X2 stores every activation as an fp16 high part plus an
 * fp16 low part (~22 mantissa bits; weights as fp16, exact for bf16-representable weights): the same kernels with
 * K doubled, about half the throughput, results within 1e-3 on scores / 0.5 px on boxes of an fp32 runtime
 * (tests/test_gpu_parity.py).  Call right after b2d_create, before any b2d_plan_*.                         */
enum { B2D_PREC_BF16 = 0, B2D_PREC_FP16 = 1, B2D_PREC_FP16X2 = 2 };
int b2d_set_precision(b2d_engine* e, int precision);
int b2d_get_precision(b2d_engine* e);

/* ---- plan building: the graph onnxruntime would have read from the .onnx file ---------- */
/* Buffers are NHWC; id 0 must be the network input [max_batch, H, W, 4], 16-bit, holding RAW pixel values 0..255
 * (exact in bf16 and fp16): the reference's `/ 255.0` is applied to the fp32 accumulator of the convolutions that
 * read buffer 0.                                                                          */
int b2d_plan_buffer(b2d_engine* e, int h, int w, int c, int is_f32);
/* weight_host: fp32 [cout][cin][k][k] (deploy form, BN folded); bias_host: fp32 [cout].  */
int b2d_plan_conv(b2d_engine* e, int src, int src_c0, int cin, int dst, int dst_c0, int cout,
                  int k, int stride, int act, const float* weight_host, const float* bias_host,
                  int res, int res_c0, int impl);
int b2d_plan_dwconv(b2d_engine* e, int src, int src_c0, int dst, int dst_c0, int c, int act,
                    const float* weight_host, const float* bias_host);
int b2d_plan_maxpool(b2d_engine* e, int src, int src_c0, int dst, int dst_c0, int c, int k, int stride);
int b2d_plan_upsample2x(b2d_engine* e, int src, int src_c0, int dst, int dst_c0, int c);
/* head level: fp32 buffer `buf` [.,hw,hw,c]; anchors_px: 6 floats (v7) or NULL (v8, v8 OBB).
 * An engine planned with B2D_HEAD_V8_OBB levels answers only the *_obb stage entry points below, any other engine only
 * the axis-aligned ones; a call of the other family fails with a message.                   */
int b2d_plan_head_level(b2d_engine* e, int kind, int buf, int stride, int nc, const float* anchors_px);
int b2d_plan_finalize(b2d_engine* e);
void* b2d_buffer_ptr(b2d_engine* e, int buf);
size_t b2d_buffer_bytes(b2d_engine* e, int buf);
int b2d_num_anchors(b2d_engine* e);
int b2d_num_kernels_per_forward(b2d_engine* e);

/* ---- stages ---------------------------------------------------------------------------- */
/* Resize + normalise + layout.  Replaces simple_detector.py:463-467, :655-659 and
 * _script/gpu_handler.py:67-92 (and the BGR variant :142-149 via `bgr`).
 * src_dev: n images uint8 HWC RGB, row pitch `pitch` bytes, image stride `img_stride`.
 * out_kind B2D_OUT_F32_NCHW is the tensor the reference builds (pixel / 255.0f, IEEE division, CHW);
 * B2D_OUT_U8_NHWC the resized image; B2D_OUT_BF16_NHWC4 / B2D_OUT_F16_NHWC4 the engine's network-input format (raw
 * pixel values, see b2d_plan_buffer).  dst_dev == NULL writes the engine's own input buffer.  */
int b2d_preprocess(b2d_engine* e, const uint8_t* src_dev, int n, int h, int w, int pitch,
                   long long img_stride, int mode, int bgr, int out_kind, void* dst_dev, void* stream);

/* Load the tensor the reference hands to session.run -- float32 [n,3,H,W] in [0,1], RGB
 * (simple_detector.py:466-467, :474) -- into the engine's input buffer.  The network input is 8-bit: every value is
 * mapped back to the pixel it came from (rint(x * 255), exact for every u8 / 255.0f the reference produces).   */
int b2d_set_input_f32(b2d_engine* e, const float* src_dev, int n, void* stream);

/* The network: replaces session.run at simple_detector.py:474, :666 and
 * _script/gpu_handler.py:165.  Reads buffer 0, leaves raw head maps in the head buffers.   */
int b2d_forward(b2d_engine* e, int n, void* stream);

/* Dense decode to the layout the reference indexes: rows_dev fp32 [n][A][6]
 * (cx,cy,w,h,conf,cls) -- outputs[0][0] at simple_detector.py:479 (v7: in-graph decode,
 * conf = objectness; v8: DFL decode, conf = max class, an adapter -- SURVEY.md section 8b).         */
int b2d_decode_rows(b2d_engine* e, int n, float* rows_dev, void* stream);

/* Fused decode + confidence filter + compaction (+ IoU-NMS when iou_thr > 0).
 *  - reference filter: `rows[:,4] >= thr` (inclusive=1), simple_detector.py:480, output in
 *    row order; top_k > 0 keeps the k best per tile (gpu_handler.py:173);
 *  - iou_thr > 0: Ultralytics NMS [EXT] (class-offset boxes, suppress iff IoU > thr, at most
 *    max_det per tile, output in descending confidence); like Ultralytics' max_nms, only the
 *    30000 best candidates of a tile enter the NMS.
 * Order: descending confidence as floats compare (+0.0 and -0.0 equal), equal confidences in
 * ascending anchor (row) order.  Every passing row is a candidate: a tile of more than 65536
 * rows is refused, never truncated.
 * dets_dev: [n][cap]; counts_dev: int32 [n] (number written per tile, <= cap).               */
int b2d_postprocess(b2d_engine* e, int n, float conf_thr, int inclusive, float iou_thr, int top_k,
                    int max_det, b2d_det* dets_dev, int32_t* counts_dev, int cap, void* stream);

/* Same as above but from caller-supplied rows [n][A][ncol>=6] (tests; YOLOv7-style graphs
 * whose decode is in the exported model).                                                    */
int b2d_postprocess_rows(b2d_engine* e, const float* rows_dev, int n, int num_rows, int ncol,
                         float conf_thr, int inclusive, float iou_thr, int top_k, int max_det,
                         b2d_det* dets_dev, int32_t* counts_dev, int cap, void* stream);

/* The whole device-resident path in one call (SURVEY.md section 8b "b2d_infer_tiles"): b2d_preprocess into the engine's
 * input buffer, b2d_forward, b2d_postprocess.  Arguments as in those three.                                    */
int b2d_infer_tiles(b2d_engine* e, const uint8_t* src_dev, int n, int h, int w, int pitch, long long img_stride, int mode, int bgr,
                    float conf_thr, int inclusive, float iou_thr, int top_k, int max_det, b2d_det* dets_dev,
                    int32_t* counts_dev, int cap, void* stream);

/* The same from HOST buffers to HOST buffers -- what GPUHandler.process_batch / SimpleDetector.detect_batch do with the
 * images they are handed (gpu_handler.py:151-213, simple_detector.py:648-677): n tiles uint8 [n][h][w][3] (any n; pinned
 * memory lets the copies overlap), params_host double [n][B2D_GEO_PARAMS] for b2d_georef in `geo_mode`; results
 * out_host [n][cap] records and counts_host [n].  Chunks of max_batch tiles are double-buffered: the next chunk's
 * host->device copy runs on the engine's copy stream while the current chunk computes.  Returns after the results
 * have landed in host memory.                                                                                    */
int b2d_detect_host(b2d_engine* e, const uint8_t* tiles_host, int n, int h, int w, int mode, int bgr, float conf_thr,
                    int inclusive, float iou_thr, int top_k, int max_det, int geo_mode, const double* params_host,
                    b2d_geodet* out_host, int32_t* counts_host, int cap, void* stream);

/* Pixel -> CRS.  params_dev: double [n][B2D_GEO_PARAMS] per tile.  fp64, no FMA contraction.
 * Replaces simple_detector.py:484-502, gpu_handler.py:178-190, pixel_to_geo.                 */
int b2d_georef(b2d_engine* e, const b2d_det* dets_dev, const int32_t* counts_dev, int n, int cap,
               int mode, const double* params_dev, b2d_geodet* out_dev, void* stream);

/* ---- oriented boxes (engines planned with B2D_HEAD_V8_OBB) --------------------------------
 * Ultralytics >= 8.1 OBB semantics [EXT]: decode theta = (sigmoid(z) - 0.25) pi and dist2rbox; rotated NMS =
 * non_max_suppression(rotated=True): class-offset boxes (+7680 cls), descending confidence, keep j iff
 * ProbIoU(i, j) < iou_thr for EVERY earlier i ("fast NMS": a suppressed box still suppresses), at most max_det
 * (<= 30000 candidates enter); results regularized (regularize_rboxes).                                        */
/* Dense decode: rows_dev fp32 [n][A][7] = cx, cy, w, h, conf (max class), cls, theta (not regularized).            */
int b2d_decode_rows_obb(b2d_engine* e, int n, float* rows_dev, void* stream);
/* Decode + filter + (iou_thr > 0) rotated NMS, arguments as b2d_postprocess; dets_dev: b2d_obb [n][cap].          */
int b2d_postprocess_obb(b2d_engine* e, int n, float conf_thr, int inclusive, float iou_thr, int top_k,
                        int max_det, b2d_obb* dets_dev, int32_t* counts_dev, int cap, void* stream);
/* Georeference centre and corners, arguments as b2d_georef; modes B2D_GEO_BOUNDS (per-point interpolation) and
 * B2D_GEO_AFFINE (letterbox undone on centre and size, no clipping; fp32 corners; window offset + geotransform
 * in fp64).  The other two forms are refused.                                                                   */
int b2d_georef_obb(b2d_engine* e, const b2d_obb* dets_dev, const int32_t* counts_dev, int n, int cap,
                   int mode, const double* params_dev, b2d_geoobb* out_dev, void* stream);

/* Mosaic-wide merge of oriented boxes from overlapping windows: Ultralytics' DOTA slice merge (obb/val.py, nms_rotated
 * ProbIoU "fast NMS" on boxes shifted into the full-image frame), over all windows at once.  dets_dev b2d_obb [n][cap] with
 * counts_dev int32 [n] (b2d_postprocess_obb), params_dev double [n][B2D_GEO_PARAMS] in the B2D_GEO_AFFINE form of each window;
 * record (r, s) is row r, slot s.  keep_dev uint8 [n][cap].  The rule:
 *  1. frame: cx' = (cx - pad_x) / gain, cy' likewise, w' = w / gain, h' likewise, in fp32, theta unchanged;
 *     X = (double)cx' + win_x, Y likewise, in fp64 -- b2d_georef_obb's B2D_GEO_AFFINE arithmetic, so merged boxes and
 *     georeferenced footprints are in one frame;
 *  2. eligible iff s < counts[r] and conf > conf_thr (strict); an ineligible record is never kept and suppresses nothing;
 *  3. priority: confidence descending as floats compare (+0.0 == -0.0), ties to the lower row, then the lower slot;
 *  4. record j is suppressed iff an eligible record i of higher priority and the same class (no class offset) has
 *     ProbIoU(i, j) >= iou_thr, with i as batch_probiou's obb1, centre difference dx = (float)(X_i - X_j) (dy likewise)
 *     and each box's Gaussian from (w', h', theta) as in b2d_postprocess_obb; a suppressed record still suppresses;
 *  5. keep = eligible and not suppressed.
 * The result equals the all-pairs evaluation of this rule, degenerate and non-finite boxes included (DESIGN.md section 6).
 * iou_thr must lie in (0, 1) and n * cap must fit an int32.                                                           */
int b2d_mosaic_nms_obb(b2d_engine* e, const b2d_obb* dets_dev, const int32_t* counts_dev, const double* params_dev, int n, int cap,
                       float conf_thr, float iou_thr, uint8_t* keep_dev, void* stream);

/* Greedy centre-distance dedup in a metric CRS.  Replaces SimpleDetector._remove_duplicates
 * (simple_detector.py:558-596, inclusive=1) and ResultsManager.remove_duplicates
 * (_script/utils.py:229-256, inclusive=0).  Priority = conf desc, then tiebreak_dev asc
 * (int64 per detection; NULL = input index, i.e. Python's stable sort at :565).
 * keep_dev: uint8 [count].                                                                    */
int b2d_dedup(b2d_engine* e, const double* x_dev, const double* y_dev, const float* conf_dev,
              const long long* tiebreak_dev, int count, double thr, int inclusive, uint8_t* keep_dev, void* stream);

/* Multi-GPU seam support (no reference counterpart: the reference is single-process).  On entry
 * flag_dev[i] != 0 marks detections within `thr` of another shard's coverage; on exit the flag is
 * closed under the "within thr" relation, so unflagged detections can be deduplicated locally and
 * only flagged ones need to be exchanged.                                                        */
int b2d_seam_closure(b2d_engine* e, const double* x_dev, const double* y_dev, int count, double thr,
                     int inclusive, uint8_t* flag_dev, void* stream);

/* WGS84 lon/lat -> UTM metres (replaces pyproj at simple_detector.py:551-556).              */
int b2d_utm_forward(b2d_engine* e, const double* lon_dev, const double* lat_dev, int count,
                    int zone, int north, double* x_dev, double* y_dev, void* stream);

/* Cut model-sized windows out of a device-resident mosaic (sliding window of
 * x_arch/02_analyze_images:1 (cell 6)); out-of-mosaic pixels are filled with `fill`.
 * origins_dev: int32 [n][4] = (x0, y0, w0, h0): the clipped window is centred in the tile
 * as Ultralytics LetterBox does, no resampling.  dst: uint8 [n][win][win][3].                */
int b2d_cut_windows(b2d_engine* e, const uint8_t* mosaic_dev, int mh, int mw, long long pitch,
                    const int32_t* origins_dev, int n, int win, int fill, uint8_t* dst_dev, void* stream);

/* Windows of any size `win`, resampled from the mosaic straight into an imgsz x imgsz canvas (imgsz = the
 * engine's input side) in one launch: Ultralytics LetterBox with one gain g = imgsz / win for every window,
 * new_w = max(1, rint(w0 g)), left = rint((imgsz - new_w) / 2 - 0.1) (same for h / top), cv2 INTER_LINEAR from
 * w0 x h0 to new_w x new_h, the rest `fill`.  At g = 1 the bytes equal b2d_cut_windows'.  origins_dev as there;
 * `bgr` swaps R and B.  out_kind B2D_OUT_U8_NHWC: dst uint8 [n][imgsz][imgsz][3].  B2D_OUT_BF16_NHWC4 (or
 * B2D_OUT_F16_NHWC4) with dst_dev == NULL writes the engine's own input buffer (raw pixel values, n <= max_batch).
 * The origins stay on the device, so they are not checked here: a window with w0 or h0 outside 1..win, or one
 * reaching outside the mosaic, comes out as a canvas of `fill` (Engine.resize_windows refuses them).            */
int b2d_resize_windows(b2d_engine* e, const uint8_t* mosaic_dev, int mh, int mw, long long pitch,
                       const int32_t* origins_dev, int n, int win, int fill, int bgr, int out_kind, void* dst_dev,
                       void* stream);

/* Host-only: the integer coefficient table one axis of b2d_preprocess uses (mode PIL_BICUBIC or
 * CV2_LINEAR).  bounds_out int32 [out][2], coef_out int32 [out][ksize]; pass NULLs to query ksize. */
int b2d_resize_table(int mode, int in_size, int out_size, int32_t* bounds_out, int32_t* coef_out, int* ksize_out);

/* ---- test-time-augmentation variants (SURVEY.md section 8f-4) -------------------------------
 * The reference builds five views of every tile (_script/gpu_handler.py:94-140; the archived set at
 * gpu_handler_archive.py:67-122 has eight), runs the network on each, scales the confidences per view
 * (:274-283) and keeps `conf > thr` (:238).  The views are uint8 RGB images [n][h][w][3], contiguous, on the
 * device; each result is bit-identical to the OpenCV / Pillow call it replaces.  dst may equal src.      */

/* cv2.cvtColor(img, COLOR_RGB2LAB) -> cv2.createCLAHE(clip_limit, (tiles_x, tiles_y)).apply(L) -> cv2.merge ->
 * cv2.cvtColor(COLOR_LAB2RGB): gpu_handler.py:104-110 (3.0, 8x8), :128-136 (4.0, 4x4),
 * gpu_handler_archive.py:100-117.                                                                           */
int b2d_tta_clahe(b2d_engine* e, const uint8_t* src_dev, int n, int h, int w, double clip_limit, int tiles_x, int tiles_y,
                  uint8_t* dst_dev, void* stream);
/* dst[i] = lut[src[i]] over n images of img_bytes bytes; lut_dev: uint8 [256], or [n][256] when per_image.  PIL
 * ImageEnhance.Brightness(img).enhance(f) (gpu_handler.py:113-115) and the gamma curve
 * (np.power(img / 255.0, 1 / gamma) * 255).astype(uint8) (:118-121) are such tables (host side: tta.py).   */
int b2d_tta_lut(b2d_engine* e, const uint8_t* src_dev, int n, long long img_bytes, const uint8_t* lut_dev, int per_image,
                uint8_t* dst_dev, void* stream);
/* PIL ImageEnhance.Contrast(img).enhance(factor) (gpu_handler_archive.py:82): grey mean of each image
 * (ITU-R 601-2 luma, rounded), then Image.blend(mean, image, factor).                                       */
int b2d_tta_contrast(b2d_engine* e, const uint8_t* src_dev, int n, int h, int w, float factor, uint8_t* dst_dev, void* stream);
/* The 8-bit colour conversions on their own (cv2.cvtColor COLOR_RGB2LAB / COLOR_LAB2RGB), npix pixels.      */
int b2d_colour_convert(b2d_engine* e, const uint8_t* src_dev, long long npix, int code, uint8_t* dst_dev, void* stream);
/* `boxes[:, 4] *= conf_adjustment` before the threshold (gpu_handler.py:236-238): every later b2d_postprocess /
 * b2d_postprocess_rows multiplies the confidence by `scale` (float32) first.  1.0 (the default) is exact.    */
int b2d_set_conf_scale(b2d_engine* e, float scale);

/* Segmentation head (BASELINE config C5, "ramp XUnet 256": the reference holds only the blob's name,
 * /root/reference/.MISSING_LARGE_BLOBS:3; [EXT] ramp post-processes its 4-class softmax output with a per-pixel argmax).
 * Reads the fp32 NHWC logits of planned buffer `buf` ([n, H, W, c], the first `nc` channels), writes the class with the largest
 * logit (first maximum wins) as uint8 [n, H, W] and, if conf_dev is not NULL, its softmax probability as float32 [n, H, W].  */
int b2d_segment(b2d_engine* e, int buf, int n, int nc, uint8_t* labels_dev, float* conf_dev, void* stream);

/* Debug / test hooks ---------------------------------------------------------------------- */
/* Run a single planned op (index in plan order) -- used by the per-layer parity tests.      */
int b2d_run_op(b2d_engine* e, int op_index, int n, void* stream);
int b2d_num_ops(b2d_engine* e);
/* b2d_forward runs a depthwise 3x3 and the 1x1 conv that is its only consumer (Ultralytics 8.3.x cls branch, the convs inside
 * `session.run`, _script/gpu_handler.py:165) as one kernel; b2d_run_op still runs the two ops separately.
 * b2d_fused_with_next: 1 if op i starts such a pair, 0 if not, -1 on a bad index.  b2d_run_op_fused runs the pair kernel.   */
int b2d_fused_with_next(b2d_engine* e, int op_index);
int b2d_run_op_fused(b2d_engine* e, int op_index, int n, void* stream);
/* Describe op i: writes a short text (kernel, tile shape, stages) into buf.                 */
int b2d_describe_op(b2d_engine* e, int op_index, char* buf, int buflen);

#ifdef __cplusplus
}
#endif
#endif /* B2DET_H */
