// K3/K4: Detect-head decode, candidate selection, class-aware bitmask NMS, and the
// post-processing of YOLODetector.detect.
//
// In the reference, decode + NMS run inside the TensorRT engine, which returns
// num_dets/bboxes/scores/labels (/root/reference/src/detector/yolo_detector.py:49-54,108-112);
// detect() then filters by confidence and un-letterboxes (yolo_detector.py:125-149,
// src/utils/image_processing.py:141-183).  The semantics implemented here are the ones the
// oracle defines (oracle/detect_post.py, DESIGN.md):
//   decode  DFL softmax-expectation per side, xyxy = (ax-l, ay-t, ax+r, ay+b)*stride,
//           score = sigmoid(best class logit), lowest class index on ties
//   select  score >= score_thr, the max_candidates best by (score desc, anchor asc)
//   NMS     greedy, class-aware, IoU > iou_thr (strict) suppresses, at most topk keeps
//   IoU     fp32, every operation rounded (this file is compiled with --fmad=false):
//           inter / ((area_a + area_b) - inter)
// NMS is a bitmask kernel, one CTA per frame: (1) bitonic sort of the 64-bit keys
// (~score bits, anchor) in shared memory, (2) all threads fill the suppression bit matrix
// mask[i][j/32] for j > i, (3) one warp scans it, keeping its "removed" bitmap in registers.
#include "common.cuh"
#include "frame_table.cuh"

namespace aicam {

extern void count_launch();
void letterbox_geometry(int h, int w, double* r, int* new_h, int* new_w, double* dw, double* dh, int* top, int* left);

namespace {

constexpr int NMS_THREADS = 1024;
constexpr int MAX_CAND = 2048;
constexpr int MAX_SORT = 16384;

// ---- decode: four threads per anchor ---------------------------------------------------------
// Thread k of an anchor owns DFL side k (l, t, r, b: 16 logits = four 16-byte loads) and a quarter of the
// class logits; a warp reads 8 consecutive head rows (8 x 576 B, every sector fully used).  The softmax
// expectation is a register loop (no shuffles); two shuffle rounds merge the class argmax
// (lowest index on ties) and gather the four distances.
// VEC: every head row starts on a 16-byte boundary (64 + nc a multiple of 4, head 16-byte aligned) and the logits are
// read as float4; otherwise (nc = 1, 2, 3, 601, ...) every logit is a scalar load.
template <bool VEC>
__global__ void __launch_bounds__(256) decode_kernel(const float* __restrict__ head, int anchors, int nc, int total,
                                                     float* __restrict__ boxes, float* __restrict__ scores,
                                                     int* __restrict__ labels) {
  const long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  const int k = static_cast<int>(t & 3);
  const int gw_raw = static_cast<int>(t >> 2);
  const bool live = gw_raw < total;
  const int gw = live ? gw_raw : total - 1;  // tail lanes recompute the last anchor (the shuffles need a full warp)
  const float* row = head + static_cast<long long>(gw) * (AICAM_HEAD_DFL + nc);
  float v[16];
  if (VEC) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 q = __ldg(reinterpret_cast<const float4*>(row + 16 * k) + i);
      v[4 * i] = q.x; v[4 * i + 1] = q.y; v[4 * i + 2] = q.z; v[4 * i + 3] = q.w;
    }
  } else {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __ldg(row + 16 * k + i);
  }
  float m = v[0];
#pragma unroll
  for (int i = 1; i < 16; ++i) m = fmaxf(m, v[i]);
  float s = 0.0f, ws = 0.0f;
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const float e = expf(v[i] - m);
    s += e;
    ws += e * static_cast<float>(i);
  }
  const float dist = ws / s;
  // best class of my quarter (ascending scan with a strict compare keeps the lowest index on ties)
  const int per = ((nc + 3) / 4 + 3) / 4 * 4;
  const int c_lo = min(nc, k * per), c_hi = min(nc, c_lo + per);
  float best = -INFINITY;
  int bi = 0x7fffffff;
  const float* cls = row + AICAM_HEAD_DFL;
  if (VEC) {
    for (int c = c_lo; c < c_hi; c += 4) {
      const float4 q = __ldg(reinterpret_cast<const float4*>(cls + c));
      if (q.x > best) { best = q.x; bi = c; }
      if (q.y > best) { best = q.y; bi = c + 1; }
      if (q.z > best) { best = q.z; bi = c + 2; }
      if (q.w > best) { best = q.w; bi = c + 3; }
    }
  } else {
    for (int c = c_lo; c < c_hi; ++c) {
      const float q = __ldg(cls + c);
      if (q > best) { best = q; bi = c; }
    }
  }
#pragma unroll
  for (int o = 1; o <= 2; o <<= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
  }
  const int base = threadIdx.x & 28;  // lane of side 0 of my anchor
  const float l = __shfl_sync(0xffffffffu, dist, base), tt = __shfl_sync(0xffffffffu, dist, base + 1);
  const float r = __shfl_sync(0xffffffffu, dist, base + 2), b = __shfl_sync(0xffffffffu, dist, base + 3);
  if (k == 0 && live) {
    // anchor geometry for a 640x640 input: levels of 80^2, 40^2, 20^2 cells
    int idx = gw % anchors, gridw = AICAM_YOLO_INPUT / 8;
    float stride = 8.0f;
    if (idx >= gridw * gridw) {
      idx -= gridw * gridw; gridw = AICAM_YOLO_INPUT / 16; stride = 16.0f;
      if (idx >= gridw * gridw) { idx -= gridw * gridw; gridw = AICAM_YOLO_INPUT / 32; stride = 32.0f; }
    }
    const float ax = static_cast<float>(idx % gridw) + 0.5f, ay = static_cast<float>(idx / gridw) + 0.5f;
    float4 box = make_float4((ax - l) * stride, (ay - tt) * stride, (ax + r) * stride, (ay + b) * stride);
    reinterpret_cast<float4*>(boxes)[gw] = box;
    scores[gw] = 1.0f / (1.0f + expf(-best));
    labels[gw] = bi;
  }
}

// ---- select + sort + bitmask NMS: one CTA per frame -----------------------------------------
struct NmsArgs {
  const float* boxes;    // [batch][anchors][4]
  const float* scores;   // [batch][anchors]
  const int* labels;     // [batch][anchors]
  int anchors;
  float score_thr, iou_thr;
  int topk, max_cand;
  float pad_w, pad_h, ratio, frame_w, frame_h;
  int* num_dets;
  float* boxes_lb;
  float* boxes_orig;
  float* out_scores;
  int* out_labels;
  int* keep_index;
  uint32_t* mask_ws;     // [batch][max_cand][max_cand/32]
  const FrameRec* recs;  // frame table: per-frame un-letterboxing (pad_w .. frame_h above unused) and packed slot; null: one
                         // geometry, frame b at b
};

__device__ __forceinline__ bool iou_gt(const float4& a, const float4& b, float thr) {
  const float iw = fmaxf(0.0f, fminf(a.z, b.z) - fmaxf(a.x, b.x));
  const float ih = fmaxf(0.0f, fminf(a.w, b.w) - fmaxf(a.y, b.y));
  const float inter = iw * ih;
  const float area_a = (a.z - a.x) * (a.w - a.y);
  const float area_b = (b.z - b.x) * (b.w - b.y);
  const float uni = (area_a + area_b) - inter;
  const float iou = uni > 0.0f ? __fdiv_rn(inter, uni) : 0.0f;
  return iou > thr;
}

__global__ void __launch_bounds__(NMS_THREADS) nms_kernel(const NmsArgs p) {
  extern __shared__ __align__(16) uint8_t sm[];
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(sm);                 // MAX_SORT x 8
  float4* cbox = reinterpret_cast<float4*>(sm + static_cast<size_t>(MAX_SORT) * 8);    // MAX_CAND x 16
  int* clab = reinterpret_cast<int*>(cbox + MAX_CAND);                                 // MAX_CAND x 4
  int* keep = clab + MAX_CAND;                                                         // MAX_CAND x 4
  __shared__ int s_count, s_kept;
  const int b = blockIdx.x, tid = threadIdx.x;
  // frame table: CTA b is table entry b, whose network outputs sit at its packed slot; an absent entry (slot -1) reports no
  // detections and a zeroed row (the whole CTA leaves before the first barrier)
  const int slot = p.recs ? p.recs[b].slot : b;
  if (slot < 0) {
    const long long ob = static_cast<long long>(b) * p.topk;
    for (int r = tid; r < p.topk; r += NMS_THREADS) {
      reinterpret_cast<float4*>(p.boxes_lb)[ob + r] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (p.boxes_orig) reinterpret_cast<float4*>(p.boxes_orig)[ob + r] = make_float4(0.f, 0.f, 0.f, 0.f);
      p.out_scores[ob + r] = 0.f;
      p.out_labels[ob + r] = 0;
      if (p.keep_index) p.keep_index[ob + r] = -1;
    }
    if (tid == 0) p.num_dets[b] = 0;
    return;
  }
  // thresholds: the entry's own when the table carries settings for it (aicam_frame_table_set_filters)
  float score_thr = p.score_thr, iou_thr = p.iou_thr;
  if (p.recs && p.recs[b].filt) { score_thr = p.recs[b].score_thr; iou_thr = p.recs[b].iou_thr; }
  const float* scores = p.scores + static_cast<long long>(slot) * p.anchors;
  if (tid == 0) { s_count = 0; s_kept = 0; }
  __syncthreads();
  for (int a = tid; a < p.anchors; a += NMS_THREADS) {
    const float s = __ldg(scores + a);
    if (s >= score_thr) {
      const int pos = atomicAdd(&s_count, 1);
      keys[pos] = (static_cast<unsigned long long>(~__float_as_uint(s)) << 32) | static_cast<unsigned>(a);
    }
  }
  __syncthreads();
  const int count = s_count;
  int nsort = 32;
  while (nsort < count) nsort <<= 1;
  for (int i = count + tid; i < nsort; i += NMS_THREADS) keys[i] = ~0ull;
  __syncthreads();
  for (int k = 2; k <= nsort; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = tid; i < nsort; i += NMS_THREADS) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const unsigned long long x = keys[i], y = keys[ixj];
          const bool up = (i & k) == 0;
          if ((x > y) == up) { keys[i] = y; keys[ixj] = x; }
        }
      }
      __syncthreads();
    }
  }
  const int n = min(count, p.max_cand);
  const float4* gboxes = reinterpret_cast<const float4*>(p.boxes) + static_cast<long long>(slot) * p.anchors;
  const int* glabels = p.labels + static_cast<long long>(slot) * p.anchors;
  for (int i = tid; i < n; i += NMS_THREADS) {
    const int a = static_cast<int>(keys[i] & 0xffffffffu);
    cbox[i] = __ldg(gboxes + a);
    clab[i] = __ldg(glabels + a);
  }
  __syncthreads();
  const int words = (n + 31) >> 5;
  uint32_t* mask = p.mask_ws + static_cast<long long>(b) * p.max_cand * (p.max_cand / 32);
  for (int idx = tid; idx < n * words; idx += NMS_THREADS) {
    const int i = idx / words, wj = idx - i * words;
    uint32_t bits = 0;
    if (32 * wj + 31 > i) {
      const float4 bi = cbox[i];
      const int li = clab[i];
      const int j0 = 32 * wj;
      const int jend = min(32, n - j0);
      for (int jj = 0; jj < jend; ++jj) {
        const int j = j0 + jj;
        if (j > i && clab[j] == li && iou_gt(cbox[j], bi, iou_thr)) bits |= 1u << jj;
      }
    }
    mask[idx] = bits;
  }
  __syncthreads();
  if (tid < 32) {
    uint32_t removed[MAX_CAND / 32 / 32] = {0};  // lane l owns words l, l+32
    int kept = 0;
    for (int i = 0; i < n && kept < p.topk; ++i) {
      const int w = i >> 5;
      uint32_t word = 0;
#pragma unroll
      for (int k = 0; k < MAX_CAND / 32 / 32; ++k)
        if ((w >> 5) == k) word = removed[k];
      word = __shfl_sync(0xffffffffu, word, w & 31);
      if (!((word >> (i & 31)) & 1u)) {
        if (tid == 0) keep[kept] = i;
        ++kept;
#pragma unroll
        for (int k = 0; k < MAX_CAND / 32 / 32; ++k) {
          const int wi = tid + 32 * k;
          if (wi < words) removed[k] |= mask[i * words + wi];
        }
      }
    }
    if (tid == 0) s_kept = kept;
  }
  __syncthreads();
  const int kept = s_kept;
  const long long ob = static_cast<long long>(b) * p.topk;
  float pad_w = p.pad_w, pad_h = p.pad_h, ratio = p.ratio, frame_w = p.frame_w, frame_h = p.frame_h;
  if (p.recs) {
    const FrameRec& g = p.recs[b];
    pad_w = g.pad_w; pad_h = g.pad_h; ratio = g.ratio; frame_w = static_cast<float>(g.w); frame_h = static_cast<float>(g.h);
  }
  for (int r = tid; r < p.topk; r += NMS_THREADS) {
    float4 bx = make_float4(0.f, 0.f, 0.f, 0.f), bo = bx;
    float sc = 0.f;
    int lb = 0, ki = -1;
    if (r < kept) {
      const int i = keep[r];
      bx = cbox[i];
      lb = clab[i];
      ki = static_cast<int>(keys[i] & 0xffffffffu);
      sc = __uint_as_float(~static_cast<uint32_t>(keys[i] >> 32));
      // scale_bboxes (image_processing.py:162-181): subtract pad, divide by ratio, clip
      bo.x = fminf(fmaxf(__fdiv_rn(bx.x - pad_w, ratio), 0.0f), frame_w);
      bo.y = fminf(fmaxf(__fdiv_rn(bx.y - pad_h, ratio), 0.0f), frame_h);
      bo.z = fminf(fmaxf(__fdiv_rn(bx.z - pad_w, ratio), 0.0f), frame_w);
      bo.w = fminf(fmaxf(__fdiv_rn(bx.w - pad_h, ratio), 0.0f), frame_h);
    }
    reinterpret_cast<float4*>(p.boxes_lb)[ob + r] = bx;
    if (p.boxes_orig) reinterpret_cast<float4*>(p.boxes_orig)[ob + r] = bo;
    p.out_scores[ob + r] = sc;
    p.out_labels[ob + r] = lb;
    if (p.keep_index) p.keep_index[ob + r] = ki;
  }
  if (tid == 0) p.num_dets[b] = kept;
}

constexpr size_t NMS_SMEM = static_cast<size_t>(MAX_SORT) * 8 + static_cast<size_t>(MAX_CAND) * (16 + 4 + 4);

int check_params(const aicam_nms_params* p, int anchors) {
  if (!p) return fail(AICAM_ERR_INVALID_ARG, "nms: null params");
  if (p->topk <= 0 || p->topk > 1024) return fail(AICAM_ERR_INVALID_ARG, "nms: topk must be in 1..1024");
  if (p->max_candidates <= 0 || p->max_candidates > MAX_CAND || p->max_candidates % 32)
    return fail(AICAM_ERR_INVALID_ARG, "nms: max_candidates must be a multiple of 32 in 32..2048");
  if (anchors <= 0 || anchors > MAX_SORT) return fail(AICAM_ERR_INVALID_ARG, "nms: anchors must be in 1..16384");
  return AICAM_OK;
}

size_t dense_bytes(int batch, int anchors) { return static_cast<size_t>(batch) * anchors * (16 + 4 + 4); }
size_t mask_bytes(int batch, const aicam_nms_params* p) {
  return static_cast<size_t>(batch) * p->max_candidates * (p->max_candidates / 32) * 4;
}

int launch_nms(const float* boxes, const float* scores, const int* labels, int batch, int anchors,
               const aicam_nms_params* p, int* num_dets, float* boxes_lb, float* boxes_orig, float* out_scores,
               int* out_labels, int* keep_index, uint32_t* mask_ws, cudaStream_t stream, const FrameRec* recs) {
  NmsArgs a;
  a.boxes = boxes; a.scores = scores; a.labels = labels; a.anchors = anchors;
  a.score_thr = p->score_thr; a.iou_thr = p->iou_thr; a.topk = p->topk; a.max_cand = p->max_candidates;
  double r = 1.0, dw = 0.0, dh = 0.0;
  int nh, nw, top, left;
  if (p->frame_h > 0 && p->frame_w > 0) letterbox_geometry(p->frame_h, p->frame_w, &r, &nh, &nw, &dw, &dh, &top, &left);
  a.pad_w = static_cast<float>(dw); a.pad_h = static_cast<float>(dh); a.ratio = static_cast<float>(r);
  a.frame_w = static_cast<float>(p->frame_w); a.frame_h = static_cast<float>(p->frame_h);
  a.num_dets = num_dets; a.boxes_lb = boxes_lb; a.boxes_orig = (recs || (p->frame_h > 0 && p->frame_w > 0)) ? boxes_orig : nullptr;
  a.recs = recs;
  a.out_scores = out_scores; a.out_labels = out_labels; a.keep_index = keep_index; a.mask_ws = mask_ws;
  if (int rc = ensure_dynamic_smem(nms_kernel, NMS_SMEM)) return rc;
  nms_kernel<<<batch, NMS_THREADS, NMS_SMEM, stream>>>(a);
  count_launch();
  return last_launch("nms_kernel");
}

}  // namespace

// aicam_nms / aicam_decode_nms; recs: per-frame un-letterboxing from a frame table (aicam_yolo_detect_table), or null
int nms_impl(const float* boxes, const float* scores, const int32_t* labels, int batch, int anchors, const aicam_nms_params* p,
             int32_t* num_dets, float* boxes_lb, float* boxes_orig, float* out_scores, int32_t* out_labels, int32_t* keep_index,
             void* workspace, size_t workspace_bytes, void* stream, const FrameRec* recs) {
  if (int rc = check_params(p, anchors)) return rc;
  if (!boxes || !scores || !labels || !num_dets || !boxes_lb || !out_scores || !out_labels || batch < 0)
    return fail(AICAM_ERR_INVALID_ARG, "nms: null argument");
  if (batch == 0) return AICAM_OK;
  if (!workspace || workspace_bytes < mask_bytes(batch, p)) return fail(AICAM_ERR_CAPACITY, "nms: workspace too small");
  return launch_nms(boxes, scores, labels, batch, anchors, p, num_dets, boxes_lb, boxes_orig, out_scores, out_labels,
                    keep_index, static_cast<uint32_t*>(workspace), static_cast<cudaStream_t>(stream), recs);
}

int decode_nms_impl(const float* head, int batch, int anchors, int nc, const aicam_nms_params* p, int32_t* num_dets,
                    float* boxes_lb, float* boxes_orig, float* scores, int32_t* labels, void* workspace,
                    size_t workspace_bytes, void* stream, const FrameRec* recs) {
  if (int rc = check_params(p, anchors)) return rc;
  if (batch == 0) return AICAM_OK;
  if (!workspace || workspace_bytes < aicam_decode_nms_workspace(batch, anchors, p))
    return fail(AICAM_ERR_CAPACITY, "decode_nms: workspace too small");
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  float* dboxes = reinterpret_cast<float*>(ws);
  float* dscores = reinterpret_cast<float*>(ws + static_cast<size_t>(batch) * anchors * 16);
  int* dlabels = reinterpret_cast<int*>(ws + static_cast<size_t>(batch) * anchors * 20);
  uint32_t* mask = reinterpret_cast<uint32_t*>(ws + (dense_bytes(batch, anchors) + 255) / 256 * 256);
  if (int rc = aicam_decode(head, batch, anchors, nc, dboxes, dscores, dlabels, stream)) return rc;
  return launch_nms(dboxes, dscores, dlabels, batch, anchors, p, num_dets, boxes_lb, boxes_orig, scores, labels, nullptr,
                    mask, static_cast<cudaStream_t>(stream), recs);
}

}  // namespace aicam

using namespace aicam;

extern "C" {

size_t aicam_decode_nms_workspace(int batch, int anchors, const aicam_nms_params* p) {
  if (!p || batch <= 0 || anchors <= 0) return 0;
  return dense_bytes(batch, anchors) + mask_bytes(batch, p) + 256;
}

int aicam_decode(const float* head, int batch, int anchors, int nc, float* boxes, float* scores, int32_t* labels,
                 void* stream) {
  if (!head || !boxes || !scores || !labels || batch < 0 || nc < 1) return fail(AICAM_ERR_INVALID_ARG, "decode: bad arguments");
  if (anchors != 8400) return fail(AICAM_ERR_UNSUPPORTED, "decode: only the 640x640 anchor grid (8400) is supported");
  if (batch == 0) return AICAM_OK;
  const int total = batch * anchors;
  const bool vec = (AICAM_HEAD_DFL + nc) % 4 == 0 && reinterpret_cast<uintptr_t>(head) % 16 == 0;
  const int grid = cdiv(total * 4, 256);
  if (vec) decode_kernel<true><<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(head, anchors, nc, total, boxes, scores, labels);
  else decode_kernel<false><<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(head, anchors, nc, total, boxes, scores, labels);
  count_launch();
  return last_launch("decode_kernel");
}

int aicam_nms(const float* boxes, const float* scores, const int32_t* labels, int batch, int anchors,
              const aicam_nms_params* p, int32_t* num_dets, float* boxes_lb, float* boxes_orig, float* out_scores,
              int32_t* out_labels, int32_t* keep_index, void* workspace, size_t workspace_bytes, void* stream) {
  return nms_impl(boxes, scores, labels, batch, anchors, p, num_dets, boxes_lb, boxes_orig, out_scores, out_labels, keep_index,
                  workspace, workspace_bytes, stream, nullptr);
}

int aicam_decode_nms(const float* head, int batch, int anchors, int nc, const aicam_nms_params* p, int32_t* num_dets,
                     float* boxes_lb, float* boxes_orig, float* scores, int32_t* labels, void* workspace,
                     size_t workspace_bytes, void* stream) {
  return decode_nms_impl(head, batch, anchors, nc, p, num_dets, boxes_lb, boxes_orig, scores, labels, workspace, workspace_bytes,
                         stream, nullptr);
}

}  // extern "C"
