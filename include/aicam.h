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
/* A chain of 2-5 stride-1 convolutions (1x1 / 3x3, pad k/2) fused into ONE kernel launch (csrc/conv_chain.cu): the
 * Bottleneck pairs and C2f tails of the detector's backbone / neck and the 3x3 -> 3x3 -> 1x1 branches of its Detect
 * head, which the reference's TensorRT engine also fuses behind src/detector/yolo_detector.py:97.  Intermediate
 * activations stay in shared memory; only the last stage's output is stored.  Exposed for parity tests.
 *   buffer 0 = the input tensor (bf16 NHWC [batch][h][w][in_c]); buffer i >= 1 = the output of stage i - 1.
 *   A stage reads the concatenation of nsrc (1 or 2) channel ranges [src_coff, src_coff + src_c) of earlier
 *   buffers (multiples of 16 channels; cin = their sum) and may add a residual: channels
 *   [res_coff, res_coff + cout) of buffer res_buf at the same pixel (res_mode as in aicam_conv_desc).
 *   weights_oihw[s] / bias[s]: HOST fp32 [cout][cin][k][k] / [cout].   out: bf16 or fp32 NHWC [batch][h][w][cout_last].
 * Returns AICAM_ERR_UNSUPPORTED when the chain does not fit the kernel (the engine then runs the layers one by one). */
typedef struct {
  int cin, cout, ksize;
  int act;        /* 0 none, 1 SiLU, 2 ReLU */
  int nsrc;
  int src_buf[2], src_coff[2], src_c[2];
  int res_buf, res_coff, res_mode;
} aicam_chain_stage;
typedef struct {
  int batch, h, w, in_c;
  int nstages;
  aicam_chain_stage st[5];
  int out_f32;
} aicam_chain_desc;
int aicam_conv_chain(const aicam_chain_desc* d, const void* in_nhwc, const float* const* weights_oihw,
                     const float* const* bias, void* out_nhwc, void* stream);
/* Micro-benchmark of one such chain on device-resident pseudo-random data (like aicam_conv2d_bench). */
int aicam_conv_chain_bench(const aicam_chain_desc* d, int iters, double* mean_ms, void* stream);
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
 *   head        : fp32 [batch][anchors][64+nc]
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
  int feature_dim;         /* 512 */
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
