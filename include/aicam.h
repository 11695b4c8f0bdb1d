/* aicam.h - C ABI of the B200-native AI-Camera hot path (YOLOv8 detect -> DeepSORT track).
 *
 * The reference (abdur75648/AI-Camera) is pure Python and has no FFI; its only native seam
 * is the TensorRT engine object.  Each entry point below names the reference interface it
 * replaces (paths relative to the reference repository root).  All functions:
 *   - return 0 (AICAM_OK) or a negative AICAM_ERR_* code; aicam_last_error() gives the text;
 *   - never throw and never exit;
 *   - take raw DEVICE pointers unless a parameter is marked "host";
 *   - are asynchronous on the given cudaStream_t (passed as void*; NULL = default stream)
 *     and do not synchronise unless documented, like TRTEngine.infer
 *     (src/trt_utils/trt_engine.py:188-201);
 *   - allocate nothing on the hot path: engines and trackers own their workspaces, sized at
 *     create time; callers own every I/O buffer.
 * A handle is bound to one CUDA device and is not thread-safe (one per GPU, as the
 * reference keeps one engine per process).
 */
#ifndef AICAM_H_
#define AICAM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AICAM_OK 0
#define AICAM_ERR_INVALID_ARG (-1)
#define AICAM_ERR_CUDA (-2)
#define AICAM_ERR_IO (-3)          /* blob missing/corrupt: FileNotFoundError/RuntimeError in trt_engine.py:46-60 */
#define AICAM_ERR_CAPACITY (-4)    /* batch / crops / tracks exceed what the handle was created for */
#define AICAM_ERR_UNSUPPORTED (-5)

#define AICAM_KIND_YOLOV8 1
#define AICAM_KIND_REID 2

#define AICAM_YOLO_INPUT 640       /* src/config.py:16 */
#define AICAM_REID_H 128           /* src/config.py:32 */
#define AICAM_REID_W 64
#define AICAM_HEAD_DFL 64          /* 4 sides x 16 DFL bins */

typedef struct aicam_engine aicam_engine;
typedef struct aicam_tracker aicam_tracker;

int aicam_version(void);
const char* aicam_last_error(void);
/* Number of kernels this library has launched in the calling process (all handles). */
uint64_t aicam_launch_count(void);
/* Profiling of the convolution kernel (the dominant kernel of the path): while enabled, every
 * conv launch is bracketed by CUDA events on its own stream.  aicam_profile_conv synchronises,
 * returns the summed kernel time and the number of launches since the last call, and resets.
 * Not for use under CUDA-graph capture. */
int aicam_profile_enable(int on);
int aicam_profile_conv(double* total_ms, uint64_t* launches);
/* Debug: in-graph timeline of the window-convolution launches.  op 1: start with room for `capacity` launches (each
 * later launch - also inside a CUDA-graph capture - gets a record its CTA 0 stamps with the GPU's global timer at entry,
 * when its dependency on the previous kernel has resolved, and at exit); op 2: copy the records to host_out
 * ([n][4] int64: entry ns, dependency ns, exit ns, tag = cout * 1e6 + cin * 1e3 + input height), returns n; op 0: stop. */
int aicam_debug_timeline(int op, long long* host_out, int capacity);

/* ------------------------------------------------------------------------------------------
 * Engine: replaces TRTEngine (src/trt_utils/trt_engine.py:15-216): __init__/_init_engine
 * (deserialize_cuda_engine, :45-60) -> aicam_engine_create on a flat ".aicw" weight blob;
 * get_input_details/get_output_details (:212-216) -> aicam_engine_io_count / aicam_engine_io_info;
 * infer (:151-203) -> aicam_nchw_to_nhwc4 + aicam_yolo_detect (network, decode and NMS; the pieces
 * aicam_yolo_forward + aicam_decode_nms remain) for the detector engine (whose ONNX embeds the NMS), aicam_nchw_to_nhwc4 + aicam_reid_forward for the ReID engine.
 * ---------------------------------------------------------------------------------------- */
int aicam_engine_create(const char* blob_path, int device, int max_batch, aicam_engine** out);
void aicam_engine_destroy(aicam_engine* e);
int aicam_engine_kind(const aicam_engine* e);        /* AICAM_KIND_* */
int aicam_engine_max_batch(const aicam_engine* e);
int aicam_engine_num_classes(const aicam_engine* e); /* yolov8: nc; reid: feature dim */
int aicam_engine_num_anchors(const aicam_engine* e); /* yolov8: 8400 at 640x640 */
double aicam_engine_flops_per_item(const aicam_engine* e); /* 2*MACs per frame / per crop */
int aicam_engine_num_launches(const aicam_engine* e);      /* kernels per forward */
/* The engine's bindings as TRTEngine.get_input_details / get_output_details report them
 * (TensorInfo(name, dtype, shape, is_dynamic), trt_engine.py:11,212-216).  topk: the K the caller
 * runs aicam_decode_nms with (the detector's post-NMS outputs are [1][K]...); -1 in shape = dynamic. */
#define AICAM_DTYPE_F32 0
#define AICAM_DTYPE_I32 1
typedef struct {
  char name[32];
  int dtype;      /* AICAM_DTYPE_* */
  int ndim;
  int shape[4];
  int is_dynamic;
} aicam_tensor_info;
int aicam_engine_io_count(const aicam_engine* e, int is_output);
int aicam_engine_io_info(const aicam_engine* e, int is_output, int index, int topk, aicam_tensor_info* info);
/* Overwrite a bias vector by blob tensor name (host float32 in); used to calibrate the
 * synthetic detector/ReID heads.  aicam_engine_get_bias reads it back (host out).
 * The bias of most layers is passed to the kernels as a launch argument: a change takes effect
 * at the next launch and is NOT seen by CUDA graphs captured earlier. */
int aicam_engine_set_bias(aicam_engine* e, const char* name, const float* host, int n);
int aicam_engine_get_bias(aicam_engine* e, const char* name, float* host, int n);

/* YOLOv8 forward (the engine body behind yolo_detector.py:97).
 *   in_nhwc4 : bf16 [batch][640][640][4]  (RGB in [0,1] + one zero channel), from aicam_preprocess
 *   head     : fp32 [batch][num_anchors][64 + nc]  raw DFL logits + class logits, anchors
 *              level-major (strides 8,16,32) then row-major */
int aicam_yolo_forward(aicam_engine* e, const void* in_nhwc4, int batch, float* head, void* stream);
/* Same network, input already space-to-depth as aicam_preprocess format 2 writes it:
 * bf16 [batch][320][320][16] = 2x2 pixel blocks [row parity][column parity][R, G, B, 0].  The 3x3 stride-2
 * stem runs as a 2x2 window over these blocks; aicam_yolo_forward repacks an NHWC4 input into this
 * layout first.  aicam_engine_accepts_s2d: 1 when the engine was built with that stem, 2 when it also has the
 * stem over 4x4 pixel blocks (yolov8n; aicam_preprocess format 3, taken by aicam_yolo_detect with in_is_s2d = 2). */
int aicam_yolo_forward_s2d(aicam_engine* e, const void* in_s2d16, int batch, float* head, void* stream);
int aicam_engine_accepts_s2d(const aicam_engine* e);

/* ReID forward (the engine body behind reid_model.py:115).
 *   crops_nhwc4 : bf16 [n][128][64][4] ImageNet-normalised RGB (+ zero channel), from aicam_reid_crops
 *   feats       : fp32 [n][512], L2-normalised
 *   n_dev       : optional device i32[1]: when not NULL the number of crops is read on the
 *                 device (clamped to n, which then is the capacity, n <= max_batch), so that
 *                 the whole frame step needs no host synchronisation (the reference syncs at
 *                 reid_model.py:126) */
int aicam_reid_forward(aicam_engine* e, const void* crops_nhwc4, int n, const int32_t* n_dev,
                       float* feats, void* stream);
/* Same network, crops already NHWC8 (aicam_reid_crops format 2: bf16 [n][128][64][8] = R, G, B + five zero
 * channels, one pixel = one 16-byte K chunk of the fused stem); n is the capacity, the count is read from n_dev.
 * aicam_engine_accepts_nhwc8: 1 when the engine was built with the fused stem. */
int aicam_reid_forward_nhwc8(aicam_engine* e, const void* crops_nhwc8, int n, const int32_t* n_dev,
                             float* feats, void* stream);
int aicam_engine_accepts_nhwc8(const aicam_engine* e);

/* Reference-layout converters used by the TRTEngine-shaped facade:
 * fp32 NCHW [n][3][h][w] -> bf16 NHWC4 [n][h][w][4]. */
int aicam_nchw_to_nhwc4(const float* in, int n, int h, int w, void* out_nhwc4, void* stream);

/* One convolution (+bias, activation, residual) on NHWC bf16 - the operator both engines are
 * built from; exposed for parity tests.  weights_oihw/bias are HOST float32. */
typedef struct {
  int batch, h, w, cin, cout, ksize, stride;
  int act;        /* 0 none, 1 SiLU, 2 ReLU */
  int res_mode;   /* 0 none, 1 act(conv)+res, 2 act(conv+res) */
  int out_f32;    /* 0: bf16 output, 1: fp32 output */
  /* optional device i32[1], as the engines pass it to every layer: when not NULL, aicam_conv2d[_padded] read the
   * number of images on the device (clamped to batch, which then is the capacity the launch is planned for); the
   * images below that count neither read nor write the images at or past it.  NULL: all batch images.
   * aicam_conv2d_bench ignores it. */
  const int32_t* n_dev;
} aicam_conv_desc;
int aicam_conv2d(const aicam_conv_desc* d, const void* in_nhwc, const float* weights_oihw,
                 const float* bias, const void* res_nhwc, void* out_nhwc, void* stream);
/* The same operator over zero-bordered ("padded") tensors.  in_pad / out_pad give the border kind of the input /
 * of the output and residual:
 *   1  symmetric: [batch][h + 2][w + 2][c], a one-pixel border of zeros all round, interior at (1, 1);
 *   2  shared:    [batch][h + 1][w + 1][c], interior at (0, 0), one zero column x = w and one zero row y = h: in the
 *                 flat raster of all pixels the column is the right border of its row and the left border of the
 *                 next, the row the bottom border of its image and the top border of the next (what precedes the
 *                 first image is read as zeros).  This is the layout the ReID engine keeps its trunk in.
 * The border of the output must be zero already; kernels write only zeros there.  The 3x3 stride-1 layers then run
 * over one flat raster of padded pixels (csrc/conv_win.cu mode 4, csrc/conv_pair.cu).
 * Supported: 3x3 stride 1 with in_pad = out_pad != 0; any stride-2 layer with either. */
int aicam_conv2d_padded(const aicam_conv_desc* d, const void* in_nhwc, const float* weights_oihw,
                        const float* bias, const void* res_nhwc, void* out_nhwc, int in_pad, int out_pad,
                        void* stream);
/* Micro-benchmark of the same operator on device-resident random data: `iters` launches
 * bracketed by CUDA events on `stream`; returns the mean kernel time in milliseconds. */
int aicam_conv2d_bench(const aicam_conv_desc* d, int iters, double* mean_ms, void* stream);
/* The fused ReID stem on its own (test entry): Conv3x3(3->64, s1, p1) + bias + ReLU + MaxPool(3, s2, p1),
 * the first two layers of the ReID engine (reid_model.py:115).
 *   in_nhwc4 : bf16 [n][h][w][4] (h, w even)   weights_oihw : fp32 host [64][3][3][3]   bias : fp32 host [64]
 *   out      : bf16 [n][h/2][w/2][64] */
int aicam_reid_stem_pool(const void* in_nhwc4, int n, int h, int w, const float* weights_oihw,
                         const float* bias, void* out, void* stream);

/* ------------------------------------------------------------------------------------------
 * Preprocessing: replaces image_processing.letterbox + preprocess_yolo_input
 * (src/utils/image_processing.py:7-102, called at yolo_detector.py:86) and the H2D copy of
 * the fp32 tensor (yolo_detector.py:91).
 *   frames : u8 [batch][h][w][3] BGR
 *   format 0: out = fp32 [batch][3][640][640] RGB/255 (the reference tensor, bit-exact)
 *   format 1: out = bf16 [batch][640][640][4] (what aicam_yolo_forward consumes)
 *   format 2: out = bf16 [batch][320][320][16], the same values space-to-depth: 2x2 pixel blocks
 *             [row parity][column parity][R, G, B, 0] (what aicam_yolo_forward_s2d consumes)
 *   format 3: out = bf16 [batch][160][160][64], the format-2 blocks grouped 2x2 once more: 4x4 pixel blocks
 *             [block row parity][block column parity][row parity][column parity][R, G, B, 0] (aicam_yolo_detect
 *             with in_is_s2d = 2, engines for which aicam_engine_accepts_s2d returns 2: a 64-channel block is one
 *             128-byte tensor-copy request where four 16-channel blocks are four)
 * meta (host out, may be NULL): ratio, pad_w, pad_h as the reference returns them. */
typedef struct {
  double ratio, pad_w, pad_h;
} aicam_letterbox;
int aicam_letterbox_params(int h, int w, aicam_letterbox* meta);
int aicam_preprocess(const uint8_t* frames, int batch, int h, int w, int format, void* out,
                     void* stream);
/* The same from NV12 frames (u8 [batch][h * 3 / 2][w]: Y plane, then the interleaved U, V plane; h, w even):
 * the surface format of hardware video decoders, 1.5 bytes per pixel instead of 3.  Where the reference's
 * loop receives BGR from cv2.VideoCapture.read() (src/aicamera_tracker.py:170), the decoder underneath
 * converted exactly such a surface; here that conversion (OpenCV's COLOR_YUV2BGR_NV12: BT.601, 20-bit fixed
 * point) is applied per fetched pixel, so the output equals aicam_preprocess on the converted BGR frame bit
 * for bit.  aicam_nv12_to_bgr makes that BGR frame (u8 [batch][h][w][3]). */
int aicam_preprocess_nv12(const uint8_t* frames_nv12, int batch, int h, int w, int format, void* out,
                          void* stream);
int aicam_nv12_to_bgr(const uint8_t* frames_nv12, int batch, int h, int w, uint8_t* frames_bgr,
                      void* stream);

/* ------------------------------------------------------------------------------------------
 * Frame table: one descriptor per stream, so that one batched step can take frames of different sizes, row pitches and
 * surface formats (a camera fleet mixes 4K, 1080p, 720p and 540p; decoders hand out one pitched surface per stream).
 * The table entry points below (aicam_preprocess_table, aicam_yolo_detect_table, aicam_reid_crops_table) take the
 * batch from the table; frame n of the batch is descriptor n of the last aicam_frame_table_set.
 *   data   : BGR: h rows of 3w bytes, `pitch` bytes apart;  NV12: the luma plane, h rows of w bytes, `pitch` apart
 *   chroma : NV12: the interleaved U, V plane, h/2 rows of w bytes, `pitch` apart (any allocation);  NULL for BGR
 *   kind   : 0 BGR, 1 NV12 (one table may mix them)
 * The caller guarantees that `data` spans h * pitch bytes and `chroma` (h/2) * pitch bytes, and that the frames stay
 * valid while work that reads the table is in flight.
 * aicam_frame_table_create: capacity = the most frames one set may hold; (max_h, max_w) = the largest frame size it may
 *   hold.  The launch configuration of every table entry point depends only on the count of the last set and on this
 *   bound, never on the frame sizes, and the kernels read everything else from the table on the device: a step
 *   captured into a CUDA graph stays valid when aicam_frame_table_set changes pointers, pitches, kinds and sizes
 *   (within the bound, same count) between replays.
 * aicam_frame_table_set: validates every descriptor on the host and launches nothing on error: null plane pointer,
 *   h or w <= 0, a kind other than 0 / 1, odd NV12 sizes, pitch < row bytes (AICAM_ERR_INVALID_ARG); n > capacity or a
 *   frame beyond the bound (AICAM_ERR_CAPACITY).  It resolves each frame's letterbox geometry (the first sight of a
 *   frame size allocates and uploads its coefficient table, as aicam_preprocess does), then copies the records to the
 *   device with one asynchronous copy on `stream` from pinned staging (two buffers used alternately; a set waits for
 *   the copy out of the buffer it reuses).  Not capturable; everything that reads the table is. */
typedef struct aicam_frame_table aicam_frame_table;
typedef struct {
  const uint8_t* data;
  const uint8_t* chroma;
  int h, w, pitch;
  int kind;
} aicam_frame_desc;
int aicam_frame_table_create(int device, int capacity, int max_h, int max_w, aicam_frame_table** out);
void aicam_frame_table_destroy(aicam_frame_table* t);
int aicam_frame_table_set(aicam_frame_table* t, const aicam_frame_desc* host_descs, int n, void* stream);
/* Presence: a camera fleet mixes frame rates, drops frames and has streams that end or reconnect, so a step need not
 * have a frame for every stream.  aicam_frame_table_set_present is aicam_frame_table_set with a host mask:
 * present_host[i] == 0 marks frame i ABSENT - its descriptor is neither read nor validated (NULL pointers are fine);
 * present_host == NULL means every frame is present, which is exactly aicam_frame_table_set (same validation, same
 * error codes, nothing launched on error).  The present frames are packed to the front of the network batch: present
 * frame i takes packed slot p(i), the number of present frames before it (p(i) = i when all are present).
 * aicam_frame_table_present: device i32[capacity], 1 for a present frame of the last set, 0 otherwise; the pointer is
 * stable for the table's lifetime, so a captured aicam_tracker_step_present can read it.  Launch configurations of the
 * table entry points still depend only on the set's count and the size bound: a captured step stays valid when the
 * presence pattern changes between replays, and absent frames cost no launch. */
int aicam_frame_table_set_present(aicam_frame_table* t, const aicam_frame_desc* host_descs, const uint8_t* present_host, int n,
                                  void* stream);
const int32_t* aicam_frame_table_present(const aicam_frame_table* t);
/* Per-stream detection and filter settings: a camera fleet mixes scenes that want different thresholds and tracked
 * classes (a parking camera tracks vehicles, a corridor camera people; a far-field camera needs a lower confidence
 * threshold), so each table entry may carry its own:
 *   score_thr, iou_thr   : aicam_yolo_detect_table's NMS score and IoU thresholds (aicam_nms_params) for the entry
 *   min_confidence       : aicam_reid_crops_table's confidence filter for the entry
 *   class_mask_lo / hi   : its class mask (bit c = COCO class c is tracked)
 * aicam_frame_table_set_filters (host only, launches nothing) stores host[0 .. n) in the table; every following
 * aicam_frame_table_set[_present] resolves entry i < n into its device record, in that set's single copy, so the settings
 * take effect with the next set and a captured step follows them.  Entries at or beyond n, and every entry after a call
 * with host == NULL or n == 0 (which clears the settings), use the arguments passed to the entry points, as before.
 * Entry i's results then equal the uniform entry points (batch 1) called with its settings.  AICAM_ERR_CAPACITY when
 * n > capacity; AICAM_ERR_INVALID_ARG for a threshold that is not finite or not in [0, 1]; on an error nothing is stored. */
typedef struct {
  float score_thr, iou_thr, min_confidence;
  int reserved;
  uint64_t class_mask_lo, class_mask_hi;
} aicam_stream_filter;
int aicam_frame_table_set_filters(aicam_frame_table* t, const aicam_stream_filter* host, int n);
/* Per-stream regions: where in its frame a stream tracks (a door camera whose top third shows a street, a parking camera
 * facing a screen or a poster).  Each entry may carry up to AICAM_REGION_MAX_POLYGONS polygons of 3 to
 * AICAM_COUNT_MAX_VERTICES integer frame-pixel vertices (|v| <= AICAM_COUNT_MAX_COORD), each an include (kind 0) or an
 * exclude (kind 1) polygon.  aicam_reid_crops_table then keeps a detection only when, besides passing the entry's
 * confidence and class filter, its anchor is inside at least one include polygon (or the entry has none) and inside no
 * exclude polygon.  A detection that fails is treated as if detect() had not returned it: no det_index entry, no crop,
 * no part in tracking; the crop rows of the others stay in scan order.
 *   anchor  the bottom centre of boxes_orig's (x1, y1, x2, y2), doubled: PX = floor(x1 + x2) with the sum rounded to
 *           float32, PY = floor(2 * y2), each clamped to +-2^24 (as counting's anchor)
 *   inside  counting's zone test: even-odd rule, half-open edges, exact int64 arithmetic on doubled vertices
 * aicam_frame_table_set_regions: entry indices_host[i] takes host[i] (i < n, host arrays); the other entries keep
 *   theirs and n_polygons == 0 clears an entry.  The whole call is validated first; AICAM_ERR_INVALID_ARG (nothing
 *   stored, copied or launched) for an index outside 0..capacity-1, n_polygons outside 0..8, a kind other than 0 / 1, a
 *   vertex count outside 3..32 or a coordinate beyond AICAM_COUNT_MAX_COORD.  On success it copies the table's region
 *   block (capacity records) to the device with one asynchronous copy on `stream` from pinned staging.  Not capturable;
 *   captured steps read the block, so they follow its changes, absent or not.
 * Once any entry of the table has had polygons, aicam_reid_crops_table makes one more launch (the region test, one CTA
 * per entry) before its filter, whatever the regions are later; a step captured before that does not include it, so
 * capture again after the first region.  With regions, stride_k is limited to 1024 (AICAM_ERR_CAPACITY). */
#define AICAM_REGION_MAX_POLYGONS 8
typedef struct {
  int32_t n_polygons;
  int32_t kind[AICAM_REGION_MAX_POLYGONS];        /* 0 include, 1 exclude */
  int32_t n_vertices[AICAM_REGION_MAX_POLYGONS];
  int32_t xy[AICAM_REGION_MAX_POLYGONS][32][2];   /* 32 = AICAM_COUNT_MAX_VERTICES */
} aicam_stream_region;
int aicam_frame_table_set_regions(aicam_frame_table* t, const int32_t* indices_host, const aicam_stream_region* host, int n,
                                  void* stream);
/* aicam_preprocess / aicam_preprocess_nv12 over a frame table (formats 0-3): present frame i's slice of `out` is slice p(i)
 * (packed, see above; slice i when all frames are present) and equals the uniform entry on that frame alone; slices past
 * the present count are not written.  Frames whose geometry is a pure decimation (1080p) and whose planes, pitch and row
 * bytes are multiples of 16 take the row-staged path, all others the per-pixel path: at most one launch each. */
int aicam_preprocess_table(const aicam_frame_table* t, int format, void* out, void* stream);

/* ------------------------------------------------------------------------------------------
 * Detection post-processing: the decode + NMS the reference's engine embeds (it returns
 * num_dets/bboxes/scores/labels, yolo_detector.py:49-54,108-112) and the part of
 * YOLODetector.detect after the engine (yolo_detector.py:107-149, scale_bboxes
 * image_processing.py:141-183).
 *   head        : fp32 [batch][anchors][64+nc], any nc >= 1 (rows need not be 16-byte aligned)
 *   num_dets    : i32 [batch]
 *   boxes_lb    : fp32 [batch][topk][4] xyxy in letterbox pixels (engine output)
 *   boxes_orig  : fp32 [batch][topk][4] xyxy in frame pixels, clipped (detect() output), may be NULL
 *   scores      : fp32 [batch][topk]       labels : i32 [batch][topk]
 * Entries past num_dets[b] are zero.  Order: score descending, anchor index ascending. */
typedef struct {
  float score_thr;   /* src/config.py:17 */
  float iou_thr;     /* src/config.py:18 */
  int topk;          /* <= 1024 */
  int max_candidates;/* multiple of 32 in 32..2048: pre-NMS candidates kept per frame */
  int frame_h, frame_w; /* for boxes_orig */
} aicam_nms_params;
int aicam_decode_nms(const float* head, int batch, int anchors, int nc, const aicam_nms_params* p,
                     int32_t* num_dets, float* boxes_lb, float* boxes_orig, float* scores,
                     int32_t* labels, void* workspace, size_t workspace_bytes, void* stream);
size_t aicam_decode_nms_workspace(int batch, int anchors, const aicam_nms_params* p);
/* Decode only: per-anchor boxes [batch][anchors][4], best score, best label. */
int aicam_decode(const float* head, int batch, int anchors, int nc, float* boxes, float* scores,
                 int32_t* labels, void* stream);
/* NMS only, on caller-provided per-anchor boxes/scores/labels (bit-exact parity entry). */
int aicam_nms(const float* boxes, const float* scores, const int32_t* labels, int batch, int anchors,
              const aicam_nms_params* p, int32_t* num_dets, float* boxes_lb, float* boxes_orig,
              float* out_scores, int32_t* out_labels, int32_t* keep_index, void* workspace,
              size_t workspace_bytes, void* stream);
/* The whole engine call of YOLODetector.detect (yolo_detector.py:97: network + embedded decode + NMS) in one
 * entry: aicam_yolo_forward[_s2d] + aicam_decode_nms, with the decode FUSED into the epilogues of the six 1x1
 * Detect-head layers when aicam_engine_fused_decode(e) is 1 - the fp32 head tensor (310 MB per 64 frames,
 * written once and read once) then never exists and `head` may be NULL; otherwise `head` is the scratch
 * tensor [batch][anchors][64 + nc].  in: the aicam_preprocess output of format 1 + in_is_s2d (0: NHWC4, 1: 2x2 blocks,
 * 2: 4x4 blocks - only when aicam_engine_accepts_s2d(e) returns 2).
 * workspace: aicam_decode_nms_workspace bytes.  Results as aicam_decode_nms (same arithmetic, same order). */
int aicam_yolo_detect(aicam_engine* e, const void* in, int in_is_s2d, int batch, const aicam_nms_params* p,
                      float* head, int32_t* num_dets, float* boxes_lb, float* boxes_orig, float* scores,
                      int32_t* labels, void* workspace, size_t workspace_bytes, void* stream);
int aicam_engine_fused_decode(const aicam_engine* e);
/* aicam_yolo_detect over a frame table (in = aicam_preprocess_table output): the outputs have one row per table entry
 * (the table's count), and boxes_orig un-letterboxes each frame with its own ratio, pad and size (p->frame_h / frame_w
 * are ignored).  Present frame n's results equal aicam_yolo_detect with batch 1 on that frame.  The network runs over the
 * packed present frames only, their count read on the device (none present: it launches as usual and does nothing); an
 * absent frame's row has num_dets = 0 and zero entries. */
int aicam_yolo_detect_table(aicam_engine* e, const void* in, int in_is_s2d, const aicam_frame_table* t,
                            const aicam_nms_params* p, float* head, int32_t* num_dets, float* boxes_lb, float* boxes_orig,
                            float* scores, int32_t* labels, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * ReID crops: replaces DeepSORT.update steps 1-2 (class/confidence filter,
 * src/tracker/deepsort_tracker.py:88-101), _extract_image_crops (:143-159),
 * preprocess_reid_input (image_processing.py:105-138) and the batch concat + H2D
 * (reid_model.py:83-101).
 *   frames : u8 [batch][h][w][3] BGR;  boxes fp32 [batch][stride_k][4] xyxy frame px
 *   det_index : i32 [batch][stride_k]  out: indices (into the frame's detections) that pass
 *               the filter, in order; det_count i32 [batch]
 *   crop_slot : i32 [batch][stride_k]  out: row in `crops` of the filtered detection's crop,
 *               or -1 when the crop rectangle is empty (feature None, :155-158)
 *   crops     : format 0: fp32 [max_crops][3][128][64] (reference tensor, bit-exact)
 *               format 1: bf16 [max_crops][128][64][4]
 *               format 2: bf16 [max_crops][128][64][8] (what aicam_reid_forward_nhwc8 consumes)
 *   crop_rect : i32 [max_crops][5] out: frame index, x1, y1, x2, y2 (int()-truncated, clamped)
 *   crop_count: i32 [2]: [0] = crops written this call (<= max_crops; crops beyond the capacity are
 *               dropped and their crop_slot is -1); [1] = high-water mark of the crops WANTED
 *               (un-clamped) since the caller last zeroed it: [1] > max_crops means some detection
 *               lost its feature to the capacity, which the reference never does
 * class_mask_lo/hi: bit c set = COCO class c is tracked (src/config.py:53 -> ids 0,2,3,5,7). */
int aicam_reid_crops(const uint8_t* frames, int batch, int h, int w, const float* boxes,
                     const float* scores, const int32_t* labels, const int32_t* num_dets,
                     int stride_k, float min_confidence, uint64_t class_mask_lo,
                     uint64_t class_mask_hi, int format, int max_crops, int32_t* det_index,
                     int32_t* det_count, int32_t* crop_slot, int32_t* crop_rect, void* crops,
                     int32_t* crop_count, void* stream);
/* The same with NV12 frames (see aicam_preprocess_nv12): crops equal those of the converted BGR frame. */
int aicam_reid_crops_nv12(const uint8_t* frames_nv12, int batch, int h, int w, const float* boxes,
                          const float* scores, const int32_t* labels, const int32_t* num_dets,
                          int stride_k, float min_confidence, uint64_t class_mask_lo,
                          uint64_t class_mask_hi, int format, int max_crops, int32_t* det_index,
                          int32_t* det_count, int32_t* crop_slot, int32_t* crop_rect, void* crops,
                          int32_t* crop_count, void* stream);
/* The same over a frame table (any mix of sizes, pitches, BGR and NV12): the batch is the table's count, boxes are
 * clamped to each frame's own size, crop_rect's frame index is the table index.  An absent frame gets det_count 0
 * whatever num_dets says for it.  A crop loads whole 32-bit words of its
 * rows only when its frame's planes are 4-byte aligned and h * pitch ((h/2) * pitch) is a multiple of 4. */
int aicam_reid_crops_table(const aicam_frame_table* t, const float* boxes, const float* scores, const int32_t* labels,
                           const int32_t* num_dets, int stride_k, float min_confidence, uint64_t class_mask_lo,
                           uint64_t class_mask_hi, int format, int max_crops, int32_t* det_index, int32_t* det_count,
                           int32_t* crop_slot, int32_t* crop_rect, void* crops, int32_t* crop_count, void* stream);

/* ------------------------------------------------------------------------------------------
 * Tracker: replaces TrackerCore / Track / KalmanFilter / matching / linear_assignment
 * (all modules under src/tracker/core/) and the formatting loop of DeepSORT.update
 * (deepsort_tracker.py:123-141).  One handle holds n_streams independent trackers, each
 * with its own id counter starting at 1 (track.py:21 is a process-global; one reference
 * process per stream gives the same ids).
 * ---------------------------------------------------------------------------------------- */
typedef struct {
  int n_streams;
  int max_tracks;          /* live tracks per stream (capacity) */
  int max_dets;            /* filtered detections per frame per stream (capacity) */
  int feature_dim;         /* 512; AICAM_ERR_CAPACITY when the appearance kernel's 16 * feature_dim + 128 floats of
                              shared memory exceed what a block may opt in to (feature_dim <= 3624 at 227 KB) */
  double max_cosine_distance; /* src/config.py:23 (a Python float: kept as double so that
                                 max_distance + 1e-5 rounds as in linear_assignment.py:58) */
  double max_iou_distance;    /* src/config.py:26 */
  int max_age;               /* src/config.py:27 */
  int n_init;                /* src/config.py:28 */
  int nn_budget;             /* src/config.py:29 */
  int device;
} aicam_tracker_config;
int aicam_tracker_create(const aicam_tracker_config* cfg, aicam_tracker** out);
void aicam_tracker_destroy(aicam_tracker* t);
int aicam_tracker_reset(aicam_tracker* t, void* stream);
/* Reset the streams whose entry of the device mask i32[n_streams] is non-zero: each becomes what a freshly created
 * tracker's stream is (no tracks, ids from 1, no overflow flags); every other stream is untouched.  One kernel launch,
 * capturable, so a slot can be handed to another camera or clip while the other streams keep their tracks. */
int aicam_tracker_reset_streams(aicam_tracker* t, const int32_t* mask, void* stream);
/* Per-stream association settings (DeepSORT's max_cosine_distance, max_iou_distance, max_age, n_init; the doubles are
 * kept for the reason given in aicam_tracker_config).  aicam_tracker_create gives every stream the values of its config;
 * aicam_tracker_set_stream_assoc gives stream indices_host[i] the values host[i] (i < n, host arrays) and copies the
 * stream table to the device with one asynchronous copy on `stream` from pinned staging.  Not capturable; captured steps
 * read the table, so they follow its changes from the next step on.  As in the reference, where these are attributes of
 * one process's tracker: the cascade depth is the stream's current max_age, while each track keeps the n_init and
 * max_age that applied when it was created, for its confirmation and its deletion.  A reset keeps the settings.
 * AICAM_ERR_INVALID_ARG (nothing copied) for max_age outside 1..255, n_init < 1, a distance that is negative or not
 * finite, or an index outside 0..n_streams-1. */
typedef struct {
  double max_cosine_distance, max_iou_distance;
  int max_age, n_init;
} aicam_stream_assoc;
int aicam_tracker_set_stream_assoc(aicam_tracker* t, const int32_t* indices_host, const aicam_stream_assoc* host, int n,
                                   void* stream);

/* One frame for every stream: predict, cascade + IoU matching, update, initiate, prune,
 * format.  Inputs describe, per stream b, the detections of the frame (as returned by
 * detect()/aicam_decode_nms) and which of them reach the tracker:
 *   boxes fp32 [n_streams][stride_k][4], scores fp32 [..][stride_k], labels i32 [..][stride_k]
 *   det_index/det_count/crop_slot as written by aicam_reid_crops
 *   feats fp32 [rows][feature_dim] indexed by crop_slot; NULL = the frame has no features at all
 *         (every appearance cost is INFTY_COST, nothing is appended to the galleries)
 * Outputs (device):
 *   out_tracks i32 [n_streams][max_tracks][6] = x1,y1,x2,y2,track_id,class_id (rounded half-even)
 *   out_conf   fp32 [n_streams][max_tracks]     out_count i32 [n_streams]
 * in the reference's order (track list order, confirmed and updated this frame only). */
int aicam_tracker_step(aicam_tracker* t, const float* boxes, const float* scores,
                       const int32_t* labels, int stride_k, const int32_t* det_index,
                       const int32_t* det_count, const int32_t* crop_slot, const float* feats,
                       int32_t* out_tracks, float* out_conf, int32_t* out_count, void* stream);
/* aicam_tracker_step with a device i32[n_streams] presence mask (e.g. aicam_frame_table_present); NULL = every stream is
 * present, which is exactly aicam_tracker_step.  An absent stream is treated as if its reference process had not been
 * called for this frame: its state (tracks, Kalman state, age, time_since_update, galleries, free slots, id counter,
 * overflow flags) does not change bit for bit - no predict, no aging - and out_count is 0 for it; its detection inputs
 * are not read.  Aging tracks through a dropped frame (predict with no detections) is a different policy, not this one.
 * The launches are those of aicam_tracker_step whatever the mask, so a captured step follows presence changes. */
int aicam_tracker_step_present(aicam_tracker* t, const float* boxes, const float* scores, const int32_t* labels, int stride_k,
                               const int32_t* det_index, const int32_t* det_count, const int32_t* crop_slot, const float* feats,
                               const int32_t* present, int32_t* out_tracks, float* out_conf, int32_t* out_count, void* stream);

/* Snapshot of the live tracks of one stream in track-list order (host out; synchronises):
 *   ints  [n][7]  = track_id, state(1 tentative, 2 confirmed), hits, age, time_since_update,
 *                   class_id, gallery size
 *   floats[n][25] = mean[8], covariance blocks a[4] b[4] c[4] d[4], confidence
 * returns n (>= 0) or a negative error. */
int aicam_tracker_snapshot(aicam_tracker* t, int stream_index, int32_t* ints, float* floats,
                           int capacity);
/* Parity probe of the appearance cost (K8, matching.py:109-217) and the Mahalanobis gate (K9,
 * linear_assignment.py:160-212); changes no tracker state.  For every live track of every stream, in
 * track-list order (k < n_tracks[s]), against every filtered detection d < det_count[s]:
 *   app_cost [n_streams][max_tracks][max_dets]  min over the gallery of max(0, 1 - cosine), 1e5 for
 *            tentative tracks, empty galleries or detections without a feature
 *   gate_d2  [n_streams][max_tracks][max_dets]  squared Mahalanobis distance to the PREDICTED state
 *   track_ids [n_streams][max_tracks], n_tracks [n_streams]
 * Call it with the inputs of the next aicam_tracker_step. */
int aicam_tracker_cost_probe(aicam_tracker* t, const float* boxes, int stride_k, const int32_t* det_index,
                             const int32_t* det_count, const int32_t* crop_slot, const float* feats,
                             float* app_cost, float* gate_d2, int32_t* track_ids, int32_t* n_tracks,
                             void* stream);
/* Sticky per-stream overflow flags since the last reset (host out i32[n_streams]):
 * bit 0 = track capacity exceeded, bit 1 = detection capacity exceeded. */
int aicam_tracker_overflow(aicam_tracker* t, int32_t* flags_host);
/* Device i32[n_streams][max_tracks]: row n < out_count[s] of the last step's out_tracks came from tracker slot
 * row_slots[s][n].  A live track keeps its slot; live tracks of a stream have distinct slots.  Stable for the tracker's
 * lifetime (aicam_counter_step reads it). */
const int32_t* aicam_tracker_row_slots(const aicam_tracker* t);

/* ------------------------------------------------------------------------------------------
 * Counting: line crossings and zone entries per stream, on the tracker's reported rows, in one capturable launch after
 * the tracker step (what a camera-fleet operator does with the tracks: people through a door, cars over a stop line,
 * objects in a loading bay).  All geometry is exact integer arithmetic:
 *   anchor   the bottom centre of a row x1,y1,x2,y2 held doubled, P = (x1 + x2, 2 * y2), each coordinate clamped to
 *            [-2^24, 2^24]; line and zone coordinates are integer frame pixels, |v| <= 2^20, doubled to match
 *   state    per (stream, tracker slot): track id, last reported anchor, bit set of the zones the track is in; a row whose
 *            id differs from its slot's stored id is the track's first report
 *   line A->B: side(P) = +1 if (Bx-Ax)*(Py-Ay) - (By-Ay)*(Px-Ax) > 0, else -1 (a point on the line is on the -1 side).
 *            A report moving a track from P0 (its last reported anchor) to P1 crosses when side(P0) != side(P1) and A, B
 *            are not strictly on the same side of the line P0P1.  -1 -> +1 is "in" (on screen, y down: from the left of
 *            A->B to its right), +1 -> -1 "out".  Every crossing counts; a first report never crosses.
 *   zone     a polygon of 3..AICAM_COUNT_MAX_VERTICES vertices, even-odd rule with half-open edges: edge (xi,yi)->(xj,yj)
 *            counts when (yi > Py) != (yj > Py) and P is strictly left of the edge at Py (int64, no division).  A report
 *            inside a zone the track was not in is an entry (a first report inside included), a report outside a zone
 *            it was in an exit.  A track deleted inside a zone makes no exit; a track not reported at a step (missed,
 *            tentative) keeps its bits.
 *   classes  each line and zone counts only rows whose class is in its 80-bit mask (lo, hi as aicam_stream_filter);
 *            membership bits are kept for every row.
 * ---------------------------------------------------------------------------------------- */
#define AICAM_COUNT_MAX_LINES 16
#define AICAM_COUNT_MAX_ZONES 16
#define AICAM_COUNT_MAX_VERTICES 32
#define AICAM_COUNT_CLASSES 80
#define AICAM_COUNT_MAX_COORD (1 << 20)
typedef struct aicam_counter aicam_counter;
typedef struct {
  int32_t n_lines, n_zones;
  int32_t line[AICAM_COUNT_MAX_LINES][4];                          /* ax, ay, bx, by */
  uint64_t line_class_mask[AICAM_COUNT_MAX_LINES][2];              /* lo, hi */
  int32_t zone_n[AICAM_COUNT_MAX_ZONES];                           /* vertex count */
  int32_t zone_xy[AICAM_COUNT_MAX_ZONES][AICAM_COUNT_MAX_VERTICES][2];
  uint64_t zone_class_mask[AICAM_COUNT_MAX_ZONES][2];
} aicam_stream_counting;
/* Device outputs, stable for the counter's lifetime; entries of streams present at the last step:
 *   line_counts i64 [S][MAX_LINES][2][80]  cumulative in / out per class     zone_counts i64 [S][MAX_ZONES][2][80]
 *   occupancy   i32 [S][MAX_ZONES][80]     rows of the last step inside      cumulative entries / exits per class
 *   row_zones   u32 [S][max_tracks]        zone bits of row n of out_tracks (bit z = zone z)
 *   events      i32 [S][max_events][4]     (kind, index, track id, class): kind 0 line in, 1 line out, 2 zone entry,
 *               3 zone exit; one per counted crossing, entry or exit of the last step, ordered by row, then lines by
 *               index, then zones by index
 *   event_count i32 [S]                    events of the last step (at most max_events) */
typedef struct {
  int64_t* line_counts;
  int64_t* zone_counts;
  int32_t* occupancy;
  uint32_t* row_zones;
  int32_t* events;
  int32_t* event_count;
} aicam_counter_output;
/* n_streams and max_tracks as the tracker whose rows it counts; max_events >= 1 per stream and step.  Every stream starts
 * with no lines and zones and no state. */
int aicam_counter_create(int device, int n_streams, int max_tracks, int max_events, aicam_counter** out);
void aicam_counter_destroy(aicam_counter* c);
/* Stream indices_host[i] takes the geometry host[i] (host arrays, i < n): validated as a whole first - counts over the
 * maxima, a zone of fewer than 3 vertices, a zero-length line, a coordinate beyond AICAM_COUNT_MAX_COORD, an index outside
 * 0..n_streams-1 are AICAM_ERR_INVALID_ARG and nothing is copied or launched.  Then one asynchronous copy on `stream` from
 * pinned staging and the masked reset of those streams (as aicam_counter_reset_streams).  Not capturable; captured steps
 * read the table, so they follow its changes.  Once dwell is set, the reset restarts their dwell state too (one more
 * launch; their dwell settings are kept). */
int aicam_counter_set_streams(aicam_counter* c, const int32_t* indices_host, const aicam_stream_counting* host, int n,
                              void* stream);
/* One launch, capturable, no host synchronisation: counts the rows out_tracks i32 [S][max_tracks][6] / out_count i32 [S]
 * of a tracker step whose slots are row_slot (aicam_tracker_row_slots).  present: device i32[S] as for
 * aicam_tracker_step_present, NULL = every stream; an absent stream changes no state, counter, occupancy or row_zones
 * entry, and its event_count is 0.  Counters are integer atomics: the result does not depend on the order of the rows.
 * Events beyond max_events are dropped and set the stream's sticky overflow flag; the counters stay exact. */
int aicam_counter_step(aicam_counter* c, const int32_t* out_tracks, const int32_t* out_count, const int32_t* row_slot,
                       const int32_t* present, void* stream);
/* Zero the counters, occupancy and overflow flag of the streams whose entry of the device mask i32[S] is non-zero and
 * forget their tracks (each track's next report is a first report); one launch, capturable.  It must accompany every
 * aicam_tracker_reset_streams of a stream: ids restart at 1 there, and a new track could otherwise continue an old one.
 * Once dwell is set, a second launch restarts the dwell state of those streams (clock, visits, counters, overflow flag;
 * their dwell settings are kept). */
int aicam_counter_reset_streams(aicam_counter* c, const int32_t* mask, void* stream);
int aicam_counter_outputs(const aicam_counter* c, aicam_counter_output* out);
/* Sticky per-stream event-overflow flags since the stream's last reset (host out i32[S]); synchronises. */
int aicam_counter_overflow(aicam_counter* c, int32_t* flags_host);

/* ------------------------------------------------------------------------------------------
 * Dwell: how long tracks stay in the counting zones of a stream, and loitering alerts, in one more capturable launch
 * after aicam_counter_step (queue wait at a checkout, a vehicle's time in a loading bay, someone staying too long by a
 * door).  Integer rules, on counting's zone membership and class masks:
 *   clock    each stream with dwell enabled has a frame clock f: the number of present steps of the stream since its
 *            dwell state last started, this step included (1 at the first).  The state starts when dwell is enabled for
 *            the stream and again at aicam_counter_set_streams / aicam_counter_reset_streams of it.  An absent step does
 *            not advance the clock and changes nothing.  All times are in the stream's own frames (a stream present at
 *            every other step of a 30 fps fleet counts 15 per second); int32: 2^31 present steps.
 *   state    per (stream, tracker slot): track id, a bit set of the zones with an open visit, a bit set of the visits
 *            already alerted, entry[16] (the clock at each open visit's entry).  A row whose id differs from its slot's
 *            stored id is a first report: the visits still open from the slot's previous occupant are dropped without
 *            being counted (as counting makes no exit for a track deleted inside a zone).  A row without a valid slot is
 *            a first report and keeps no state.
 *   per row and zone z < n_zones, with in = bit z of the row's row_zones entry:
 *            class not in the zone's class mask: the visit state of z is left as it is; the row reports -1 for z.
 *            in, no open visit: a visit opens, entry = f.
 *            not in, open visit: it closes with duration d = f - entry (>= 1): visits[z][cls] += 1,
 *              frames_total[z][cls] += d, frames_max[z][cls] = max(.., d), and a visit event.
 *            in, open visit, loiter_frames[z] = L > 0, f - entry >= L, not yet alerted: a loiter event, and the visit is
 *              alerted (once per visit, at its first report at or past L; L = 0: no alerts).
 *   A track not reported at a step (missed, tentative) keeps its open visits, and their clock keeps running.
 * ---------------------------------------------------------------------------------------- */
#define AICAM_DWELL_MAX_LOITER (1 << 30)
typedef struct {
  int32_t enabled;                                  /* 0 or 1 */
  int32_t loiter_frames[AICAM_COUNT_MAX_ZONES];     /* 0..AICAM_DWELL_MAX_LOITER; 0 = no alerts */
} aicam_stream_dwell;
/* Device outputs, stable for the counter's lifetime once dwell is set; entries of enabled streams present at the last
 * dwell step:
 *   visits, frames_total, frames_max  i64 [S][MAX_ZONES][80]  completed visits per zone and class since the stream's
 *                                                             dwell state last started, their summed and largest
 *                                                             durations in frames
 *   row_dwell         i32 [S][max_tracks][MAX_ZONES]  frames since entry of row n's open visit in zone z (0 at the
 *                                                     entry step), -1 otherwise; aligned with out_tracks
 *   events            i32 [S][max_events][5]  (kind, zone, track id, class, frames): kind 0 visit completed (frames =
 *                                             its duration), 1 loiter (frames = f - entry); ordered by row, then zone
 *   event_count       i32 [S]                 events of the last step (at most max_events; 0 for a disabled or absent
 *                                             stream) */
typedef struct {
  int64_t* visits;
  int64_t* frames_total;
  int64_t* frames_max;
  int32_t* row_dwell;
  int32_t* events;
  int32_t* event_count;
} aicam_counter_dwell_output;
/* Stream indices_host[i] takes the dwell settings host[i] (host arrays, i < n): validated as a whole first - enabled
 * not 0 or 1, loiter_frames outside 0..AICAM_DWELL_MAX_LOITER, an index outside 0..n_streams-1 are AICAM_ERR_INVALID_ARG
 * and nothing is allocated, copied or launched.  The first valid call allocates the dwell buffers (a counter that never
 * sets dwell allocates and launches nothing more).  Then one asynchronous copy on `stream` from pinned staging; a stream
 * that goes from disabled to enabled starts its dwell state (one launch), an enabled stream whose thresholds change keeps
 * it.  Not capturable; captured dwell steps read the settings, so they follow their changes. */
int aicam_counter_set_dwell(aicam_counter* c, const int32_t* indices_host, const aicam_stream_dwell* host, int n,
                            void* stream);
/* One launch, capturable, no host synchronisation: the dwell step of the rows aicam_counter_step has just counted, with
 * the same out_tracks, out_count, row_slot and present, on the same stream after it (it reads the counter's row_zones
 * and zone class masks).  Disabled and absent streams change nothing.  Events beyond max_events are dropped and set the
 * stream's sticky dwell-overflow flag; the counters stay exact.  AICAM_ERR_INVALID_ARG before aicam_counter_set_dwell. */
int aicam_counter_dwell_step(aicam_counter* c, const int32_t* out_tracks, const int32_t* out_count, const int32_t* row_slot,
                             const int32_t* present, void* stream);
/* AICAM_ERR_INVALID_ARG before aicam_counter_set_dwell. */
int aicam_counter_dwell_outputs(const aicam_counter* c, aicam_counter_dwell_output* out);
/* Sticky per-stream dwell event-overflow flags since the stream's dwell state last started (host out i32[S], all 0
 * before aicam_counter_set_dwell); synchronises. */
int aicam_counter_dwell_overflow(aicam_counter* c, int32_t* flags_host);

/* Stand-alone pieces of the association, exposed for bit-exact parity tests. */
/* scipy.optimize.linear_sum_assignment (linear_assignment.py:62) on `count` fp32 cost
 * matrices [count][nr][nc]; col_for_row i32 [count][nr] (-1 = unassigned). */
int aicam_lsap(const float* cost, int count, int nr, int nc, int32_t* col_for_row, void* stream);
/* KalmanFilter.gating_distance (kalman_filter.py:206-249): state fp32 [n][24] (mean8+cov16),
 * meas fp32 [n][m][4] -> d2 fp32 [n][m]. */
int aicam_kf_gating(const float* state, const float* meas, int n, int m, float* d2, void* stream);

/* ------------------------------------------------------------------------------------------
 * Overlay (SURVEY 8f, N3): replaces the drawing loop of src/utils/visualization.py (draw_tracks :72-124,
 * draw_detections :9-69, draw_fps :127-167, draw_info_panel :170-227: cv2.rectangle / cv2.putText on a host
 * copy of every frame, called from src/aicamera_tracker.py:211-225) on frames that stay in device memory.
 * frames_bgr u8 [batch][h][w][3], drawn in place.  Frame n's items are items[item_start[n] .. item_start[n + 1])
 * (both device arrays), drawn IN ORDER like the sequential cv2 calls:
 *   type 0  cv2.rectangle(.., (x1, y1), (x2, y2), color, 2): the 3-pixel band around the rectangle minus its
 *           four outer corner pixels (what OpenCV's thick-line rasteriser fills), clipped to the frame
 *   type 1  cv2.rectangle(.., color, -1): the inclusive filled rectangle
 *   type 2  decal `slot` of the atlas (u8 [slots][slot_h][slot_w][8]: B0 B1 B2 0 A0 A1 A2 0 per pixel), its
 *           first pixel at (x1, y1), (x2, y2) = the used (width, height): frame = B + (frame * A + 127) / 255 per
 *           channel; (B, A) = (0, 255) leaves a pixel untouched.  ai-camera_b200/visualization.py builds decals
 *           of anti-aliased text by running cv2.putText itself on a black and a white canvas.
 * color = b | g << 8 | r << 16. */
typedef struct {
  int32_t type, x1, y1, x2, y2, color, slot, reserved;
} aicam_overlay_item;
int aicam_overlay_draw(uint8_t* frames_bgr, int batch, int h, int w, const aicam_overlay_item* items,
                       const int32_t* item_start, const uint8_t* atlas, int slot_w, int slot_h, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AICAM_H_ */
