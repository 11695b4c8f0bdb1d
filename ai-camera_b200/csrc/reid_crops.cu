// K5: detection filter + ROI crop / resize / normalise of every tracked detection of every
// stream into one batched ReID input tensor.
//
// Replaces DeepSORT.update steps 1-2 (confidence/class filter,
// /root/reference/src/tracker/deepsort_tracker.py:88-101), _extract_image_crops (:143-159,
// int() truncation + clamp; empty rectangle -> no feature), preprocess_reid_input
// (src/utils/image_processing.py:105-138: cv2.resize INTER_LINEAR to 64x128, BGR->RGB,
// (x/255 - mean)/std, CHW) and the concat + H2D of src/tracker/reid_model.py:83-101.
//
// The resize is OpenCV's fixed-point bilinear (see preprocess.cu), evaluated per crop: the
// coefficient tables depend on the crop size, so each CTA derives them in shared memory with
// the same double -> float -> 11-bit rounding steps (explicit _rn intrinsics; the file is also
// compiled with --fmad=false), then every thread interpolates its pixels.  Result: the uint8
// resized crop, and therefore the float tensor, equals the reference's bit for bit.
// HBM-bound: reads ~crop bytes, writes 128*64*8 B (NHWC4 bf16) or 128*64*16 B (NHWC8, what the fused ReID stem reads) per crop.
#include "common.cuh"
#include "frame_src.cuh"
#include "frame_table.cuh"
#include "polygon.cuh"

namespace aicam {

extern void count_launch();

namespace {

constexpr int RH = AICAM_REID_H, RW = AICAM_REID_W;

// One block, one WARP per frame: stable filter of the frame's detections (ballot compaction, lanes over
// detections), crop rectangles, and (via a block-wide exclusive scan over frames) deterministic crop rows.
__global__ void __launch_bounds__(1024) filter_kernel(const float* __restrict__ boxes, const float* __restrict__ scores,
                                                      const int* __restrict__ labels, const int* __restrict__ num_dets,
                                                      int batch, int stride_k, int h, int w, float min_conf,
                                                      unsigned long long mask_lo, unsigned long long mask_hi,
                                                      int max_crops, int* __restrict__ det_index,
                                                      int* __restrict__ det_count, int* __restrict__ crop_slot,
                                                      int* __restrict__ crop_rect, int* __restrict__ crop_count,
                                                      const FrameRec* __restrict__ recs,  // frame table: per-frame (w, h)
                                                                                          // and presence; or null
                                                      const unsigned* __restrict__ region_keep,  // region_kernel's bits,
                                                      const aicam_stream_region* __restrict__ regions) {  // or null
  __shared__ int s_scan[32];  // valid crops per frame of the current group of 32 frames, then their exclusive scan
  __shared__ int s_base;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const unsigned lt = (1u << lane) - 1u;
  if (threadIdx.x == 0) s_base = 0;
  __syncthreads();
  for (int b0 = 0; b0 < batch; b0 += 32) {
    const int b = b0 + warp;
    const int fw = recs && b < batch ? recs[b].w : w, fh = recs && b < batch ? recs[b].h : h;
    int nvalid = 0, nkeep = 0;
    if (b < batch) {
      // an absent frame of a table keeps no detection whatever num_dets says, so no crop reads its (unset) descriptor
      const int n = recs && recs[b].slot < 0 ? 0 : min(num_dets[b], stride_k);
      const long long fo = static_cast<long long>(b) * stride_k;
      // the entry's own confidence and class mask when the table carries settings for it
      float mc = min_conf;
      unsigned long long mlo = mask_lo, mhi = mask_hi;
      if (recs && recs[b].filt) { mc = recs[b].min_conf; mlo = recs[b].mask_lo; mhi = recs[b].mask_hi; }
      // the entry's region test (region_kernel) when it has polygons
      const unsigned* rk = region_keep && regions[b].n_polygons > 0 ? region_keep + static_cast<long long>(b) * 32 : nullptr;
      for (int i0 = 0; i0 < n; i0 += 32) {
        const int i = i0 + lane;
        bool keep = false, ok = false;
        if (i < n) {
          const int cls = labels[fo + i];
          const bool tracked = cls >= 0 && cls < 128 && (((cls < 64 ? mlo >> cls : mhi >> (cls - 64)) & 1ull) != 0);
          keep = scores[fo + i] >= mc && tracked && (!rk || ((rk[i >> 5] >> (i & 31)) & 1u));
          if (keep) {
            const float4 bx = reinterpret_cast<const float4*>(boxes)[fo + i];
            const int x1 = max(0, static_cast<int>(bx.x)), y1 = max(0, static_cast<int>(bx.y));
            const int x2 = min(fw, static_cast<int>(bx.z)), y2 = min(fh, static_cast<int>(bx.w));
            ok = x1 < x2 && y1 < y2;
          }
        }
        const unsigned km = __ballot_sync(0xffffffffu, keep), vm = __ballot_sync(0xffffffffu, ok);
        if (keep) {
          const int k = nkeep + __popc(km & lt);
          det_index[fo + k] = i;
          // provisional: local crop ordinal or -1; rebased after the scan
          crop_slot[fo + k] = ok ? nvalid + __popc(vm & lt) : -1;
        }
        nkeep += __popc(km);
        nvalid += __popc(vm);
      }
      if (lane == 0) det_count[b] = nkeep;
    }
    if (lane == 0) s_scan[warp] = nvalid;
    __syncthreads();
    if (warp == 0) {  // exclusive scan of the group's 32 counts
      const int v = s_scan[lane];
      int incl = v;
      for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += u;
      }
      s_scan[lane] = s_base + incl - v;
      __syncwarp();
      if (lane == 31) s_base += incl;
    }
    __syncthreads();
    if (b < batch) {
      const int base = s_scan[warp];
      const long long fo = static_cast<long long>(b) * stride_k;
      for (int k = lane; k < nkeep; k += 32) {  // (my own writes of det_index / crop_slot: same warp, ordered by the barriers)
        const int local = crop_slot[fo + k];
        if (local < 0) continue;
        const int slot = base + local;
        if (slot < max_crops) {
          const float4 bx = reinterpret_cast<const float4*>(boxes)[fo + det_index[fo + k]];
          crop_slot[fo + k] = slot;
          crop_rect[slot * 5 + 0] = b;
          crop_rect[slot * 5 + 1] = max(0, static_cast<int>(bx.x));
          crop_rect[slot * 5 + 2] = max(0, static_cast<int>(bx.y));
          crop_rect[slot * 5 + 3] = min(fw, static_cast<int>(bx.z));
          crop_rect[slot * 5 + 4] = min(fh, static_cast<int>(bx.w));
        } else {
          crop_slot[fo + k] = -1;
        }
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    crop_count[0] = min(s_base, max_crops);
    // high-water mark of the crops WANTED (un-clamped): > max_crops means detections lost their feature to the
    // capacity (the reference always extracts one); sticky until the caller zeroes it
    if (s_base > crop_count[1]) crop_count[1] = s_base;
  }
}

// The per-entry region test of aicam_frame_table_set_regions: one CTA per table entry, the entry's polygons in shared
// memory, threads over its (detection, polygon) pairs.  Writes one keep bit per detection (bit i of word i / 32 of the
// entry's 32 words); filter_kernel reads them for entries with polygons only, so absent entries and entries without
// polygons leave at once.  The anchor is the only float arithmetic: one float32 sum (no contraction: --fmad=false) and
// two floors; the test itself is counting's exact integer in_zone (polygon.cuh).
constexpr int REGION_THREADS = 256;

__global__ void __launch_bounds__(REGION_THREADS) region_kernel(const FrameRec* __restrict__ recs,
                                                                const aicam_stream_region* __restrict__ regions,
                                                                const float* __restrict__ boxes,
                                                                const int* __restrict__ num_dets, int stride_k,
                                                                unsigned* __restrict__ keep) {
  __shared__ __align__(16) aicam_stream_region g;
  __shared__ unsigned hits[1024];  // per detection: bit p = inside polygon p
  const int b = blockIdx.x, tid = threadIdx.x;
  if (recs[b].slot < 0 || regions[b].n_polygons <= 0) return;
  {
    const int* src = reinterpret_cast<const int*>(regions + b);
    int* dst = reinterpret_cast<int*>(&g);
    for (int i = tid; i < static_cast<int>(sizeof(aicam_stream_region) / 4); i += REGION_THREADS) dst[i] = src[i];
  }
  const int n = min(num_dets[b], stride_k);
  for (int i = tid; i < n; i += REGION_THREADS) hits[i] = 0u;
  __syncthreads();
  const int np = g.n_polygons;
  const long long fo = static_cast<long long>(b) * stride_k;
  for (int q = tid; q < n * np; q += REGION_THREADS) {
    const int i = q / np, p = q - i * np;
    const float4 bx = reinterpret_cast<const float4*>(boxes)[fo + i];
    const long long px = clamp_anchor(__float2ll_rd(__fadd_rn(bx.x, bx.z)));
    const long long py = clamp_anchor(__float2ll_rd(__fmul_rn(2.0f, bx.w)));
    if (in_zone(g.xy[p], g.n_vertices[p], px, py)) atomicOr(&hits[i], 1u << p);
  }
  __syncthreads();
  unsigned inc = 0u, exc = 0u;
  for (int p = 0; p < np; ++p) (g.kind[p] ? exc : inc) |= 1u << p;
  for (int i0 = tid & ~31; i0 < n; i0 += REGION_THREADS) {  // whole warps: one ballot per 32 detections
    const int i = i0 + (tid & 31);
    const unsigned h = i < n ? hits[i] : 0u;
    const bool k = i < n && (inc == 0u || (h & inc) != 0u) && (h & exc) == 0u;
    const unsigned w = __ballot_sync(0xffffffffu, k);
    if ((tid & 31) == 0) keep[static_cast<long long>(b) * 32 + (i0 >> 5)] = w;
  }
}

// cv2 linear-resize tables for one axis, one entry per thread
__device__ __forceinline__ void axis_entry(int src, int dst, int d, bool horizontal, int* i0, int* i1, int* w0, int* w1) {
  const double scale = __ddiv_rn(1.0, __ddiv_rn(static_cast<double>(dst), static_cast<double>(src)));
  float f = __double2float_rn(__dsub_rn(__dmul_rn(static_cast<double>(d) + 0.5, scale), 0.5));
  int s = __float2int_rd(f);
  f = __fsub_rn(f, static_cast<float>(s));
  if (horizontal) {
    if (s < 0) { f = 0.0f; s = 0; }
    if (s >= src - 1) { f = 0.0f; s = src - 1; }
    *i0 = s;
    *i1 = min(s + 1, src - 1);
  } else {
    *i0 = min(max(s, 0), src - 1);
    *i1 = min(max(s + 1, 0), src - 1);
  }
  *w0 = __float2int_rn(__fmul_rn(__fsub_rn(1.0f, f), 2048.0f));
  *w1 = __float2int_rn(__fmul_rn(f, 2048.0f));
}

// a / b correctly rounded, given rcp = RN(1 / b): quotient estimate, exact remainder, one correction - three
// instructions instead of the generic IEEE division sequence.  Equal to __fdiv_rn(a, b) on every input this kernel can
// produce: v / 255 for the 256 byte values and (v / 255 - mean) / std for the 3 x 256 (channel, value) pairs were checked
// exhaustively with exact rational arithmetic, and tests/test_gpu_crops.py compares whole crops with the oracle bit for
// bit.  Explicit fmaf: this file is compiled with --fmad=false.
__device__ __forceinline__ float div_exact(float a, float b, float rcp) {
  const float q = __fmul_rn(a, rcp);
  return fmaf(fmaf(-b, q, a), rcp, q);
}

// One output pixel from its (up to) four source taps, normalised and stored.  tap(r, i, v): BGR of tap column i (0: sx0,
// 1: sx1) of source row r (0: sy0, 1: sy1).
template <int FORMAT, typename Tap>
__device__ __forceinline__ void crop_pixel(int mode, int a0, int a1, int b0, int b1, Tap tap, void* __restrict__ out, int slot, int p) {
  int v[3];
  if (mode == 2) {
    tap(0, 0, v);
  } else if (mode == 1) {
    int p00[3], p01[3], p10[3], p11[3];
    tap(0, 0, p00); tap(0, 1, p01); tap(1, 0, p10); tap(1, 1, p11);
#pragma unroll
    for (int c = 0; c < 3; ++c) v[c] = (p00[c] + p01[c] + p10[c] + p11[c] + 2) >> 2;
  } else {
    // taps with a zero weight are not fetched
    int p00[3] = {0, 0, 0}, p01[3] = {0, 0, 0}, p10[3] = {0, 0, 0}, p11[3] = {0, 0, 0};
    if (b0 != 0) {
      tap(0, 0, p00);
      if (a1 != 0) tap(0, 1, p01);
    }
    if (b1 != 0) {
      tap(1, 0, p10);
      if (a1 != 0) tap(1, 1, p11);
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const int h0 = p00[c] * a0 + p01[c] * a1, h1 = p10[c] * a0 + p11[c] * a1;
      const int o = (((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2;
      v[c] = min(max(o, 0), 255);
    }
  }
  const float mean[3] = {0.485f, 0.456f, 0.406f}, stdv[3] = {0.229f, 0.224f, 0.225f};
  const float rstd[3] = {0x1.1779dap+2f, 0x1.1db6dap+2f, 0x1.1c71c8p+2f};  // RN(1 / std)
  float rgb[3];
#pragma unroll
  for (int c = 0; c < 3; ++c)  // BGR -> RGB, (x/255 - mean)/std in float32
    rgb[c] = div_exact(__fsub_rn(div_exact(static_cast<float>(v[2 - c]), 255.0f, 0x1.010102p-8f), mean[c]), stdv[c], rstd[c]);
  if (FORMAT == 0) {
    float* o = static_cast<float*>(out) + static_cast<long long>(slot) * 3 * RH * RW + p;
    o[0] = rgb[0]; o[RH * RW] = rgb[1]; o[2 * RH * RW] = rgb[2];
  } else if (FORMAT == 1) {
    uint2 q;
    q.x = pack_bf16x2(rgb[0], rgb[1]);
    q.y = pack_bf16x2(rgb[2], 0.0f);
    reinterpret_cast<uint2*>(out)[static_cast<long long>(slot) * RH * RW + p] = q;
  } else {  // NHWC8: one pixel = one 16-byte K chunk of the fused ReID stem (stem_pool.cu)
    reinterpret_cast<uint4*>(out)[static_cast<long long>(slot) * RH * RW + p] =
        make_uint4(pack_bf16x2(rgb[0], rgb[1]), pack_bf16x2(rgb[2], 0.0f), 0u, 0u);
  }
}

// Crops up to CROP_STAGE_W pixels wide are resized from shared memory: one WARP per output row brings the row's two
// source-row segments in with coalesced 32-bit loads (aligned words covering the segment, ONE pass: a BGR segment of 168
// pixels is 128 words = four per lane), then every lane interpolates two output pixels from there - the direct path
// issues up to twelve scattered byte loads per output pixel.  Wider crops keep the direct path: staging them takes
// several dependent passes per row and measured slower than the direct path's independent loads (B200, 64 streams:
// 130 us against 83 us per ~1 100 crops when every crop up to 512 pixels wide was staged).
constexpr int CROP_STAGE_W = 168;
constexpr int CROP_SEG = CROP_STAGE_W * 3 + 16;  // bytes of one staged segment (BGR row; NV12: luma + chroma halves)
constexpr int CROP_WARPS = 8;

// Row addresses of the frame sources (frame_src.cuh) for the staged path: BGR / luma row y, and the chroma row of row y.
__device__ __forceinline__ const uint8_t* src_row(const FrameSrc<0>& s, int y) { return s.f + static_cast<long long>(y) * s.w * 3; }
__device__ __forceinline__ const uint8_t* src_row(const FrameSrc<1>& s, int y) { return s.f + static_cast<long long>(y) * s.w; }
__device__ __forceinline__ const uint8_t* src_row(const FrameSrc<2>& s, int y) { return s.f + static_cast<long long>(y) * s.pitch; }
__device__ __forceinline__ const uint8_t* src_row(const FrameSrc<3>& s, int y) { return s.f + static_cast<long long>(y) * s.pitch; }
__device__ __forceinline__ const uint8_t* src_crow(const FrameSrc<0>& s, int y) { return nullptr; }
__device__ __forceinline__ const uint8_t* src_crow(const FrameSrc<1>& s, int y) {
  return s.f + static_cast<long long>(s.h) * s.w + static_cast<long long>(y >> 1) * s.w;
}
__device__ __forceinline__ const uint8_t* src_crow(const FrameSrc<2>& s, int y) { return nullptr; }
__device__ __forceinline__ const uint8_t* src_crow(const FrameSrc<3>& s, int y) { return s.c + static_cast<long long>(y >> 1) * s.pitch; }

// (Staging: the aligned 32-bit words that cover a byte segment [p, p + n) are loaded with coalesced __ldg, WPP words per lane, and
//  written to 4-byte aligned shared memory; shift = p & 3 is where the segment starts there.  The caller passes frame_words only
//  when no such word crosses the end of the frame's planes.)
// One crop (slot) of the rectangle (x1, y1, cw, ch) of `src`; tx / ty / seg: the CTA's shared memory.
template <int FORMAT, int SRC>
__device__ __forceinline__ void crop_body(const FrameSrc<SRC>& src, bool frame_words, int x1, int y1, int cw, int ch,
                                          int (&tx)[4][RW], int (&ty)[4][RH], uint8_t (&seg)[CROP_WARPS][2][CROP_SEG],
                                          void* __restrict__ out, int slot) {
  constexpr bool NV = (SRC & 1) != 0;
  const int mode = (cw == RW && ch == RH) ? 2 : ((cw == 2 * RW && ch == 2 * RH) ? 1 : 0);
  {
    const int t = threadIdx.x;
    if (mode == 0) {
      if (t < RW) axis_entry(cw, RW, t, true, &tx[0][t], &tx[1][t], &tx[2][t], &tx[3][t]);
      else if (t < RW + RH) axis_entry(ch, RH, t - RW, false, &ty[0][t - RW], &ty[1][t - RW], &ty[2][t - RW], &ty[3][t - RW]);
    } else {  // exact 2x (box average of 2x2) / copy: the taps as tables too
      const int f = mode == 1 ? 2 : 1;
      if (t < RW) { tx[0][t] = f * t; tx[1][t] = f * t + (f - 1); tx[2][t] = 0; tx[3][t] = 0; }
      else if (t < RW + RH) { const int u = t - RW; ty[0][u] = f * u; ty[1][u] = f * u + (f - 1); ty[2][u] = 0; ty[3][u] = 0; }
    }
  }
  __syncthreads();
  const bool staged = cw <= CROP_STAGE_W && frame_words;
  if (!staged) {
    for (int p = threadIdx.x; p < RH * RW; p += blockDim.x) {
      const int oy = p / RW, ox = p - oy * RW;
      const int sx[2] = {x1 + tx[0][ox], x1 + tx[1][ox]}, sy[2] = {y1 + ty[0][oy], y1 + ty[1][oy]};
      crop_pixel<FORMAT>(mode, tx[2][ox], tx[3][ox], ty[2][oy], ty[3][oy],
                         [&](int r, int i, int (&v)[3]) { src.pix(sy[r], sx[i], v); }, out, slot, p);
    }
    return;
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int lsx[RW / 32][2], la[RW / 32][2];  // this lane's columns never change: taps (relative to the crop) and weights
#pragma unroll
  for (int k = 0; k < RW / 32; ++k) {
    lsx[k][0] = tx[0][lane + 32 * k]; lsx[k][1] = tx[1][lane + 32 * k];
    la[k][0] = tx[2][lane + 32 * k]; la[k][1] = tx[3][lane + 32 * k];
  }
  // Software pipeline over the warp's rows: the words of row i + CROP_WARPS are requested (into registers) right after row i's
  // have been written to shared memory, so their memory round trip overlaps the interpolation of row i (a row used to cost one
  // exposed round trip, 16 of them in series per warp).  Measured per 1 024 crops, filter + crops: 95 -> 71 us (NV12 114 -> 95);
  // two rows ahead measured no better (73 us).  One pass per row: staged segments are at most 128 (BGR) / 64 (NV12) words.
  constexpr int NSEG = NV ? 4 : 2, WPP = NV ? 2 : 4;
  struct RowFetch {
    uint32_t v[NSEG][WPP];
    int nwords[NSEG], shift[NSEG];
  };
  auto fetch = [&](int oy, RowFetch& f) {
    const int sy[2] = {y1 + ty[0][oy], y1 + ty[1][oy]};
    const int b0 = ty[2][oy], b1 = ty[3][oy];
    // which of the two source rows the row's pixels read (crop_pixel skips taps with a zero weight)
    const bool need[2] = {mode != 0 || b0 != 0, mode == 1 || (mode == 0 && b1 != 0)};
    const uint8_t* ps[NSEG];
    int ns[NSEG];
    if (!NV) {
      ps[0] = src_row(src, sy[0]) + x1 * 3; ps[1] = src_row(src, sy[1]) + x1 * 3;
      ns[0] = need[0] ? cw * 3 : 0; ns[1] = need[1] ? cw * 3 : 0;
    } else {  // luma segments, then the chroma pairs of columns x1 & ~1 .. (even start: U first)
      const int cn = ((x1 + cw + 1) & ~1) - (x1 & ~1);
      ps[0] = src_row(src, sy[0]) + x1; ps[1] = src_row(src, sy[1]) + x1;
      ps[NSEG - 2] = src_crow(src, sy[0]) + (x1 & ~1); ps[NSEG - 1] = src_crow(src, sy[1]) + (x1 & ~1);
      ns[0] = need[0] ? cw : 0; ns[1] = need[1] ? cw : 0; ns[NSEG - 2] = need[0] ? cn : 0; ns[NSEG - 1] = need[1] ? cn : 0;
    }
#pragma unroll
    for (int q = 0; q < NSEG; ++q) {
      f.shift[q] = static_cast<int>(reinterpret_cast<uintptr_t>(ps[q]) & 3);
      const uint32_t* pa = reinterpret_cast<const uint32_t*>(ps[q] - f.shift[q]);
      f.nwords[q] = ns[q] > 0 ? (f.shift[q] + ns[q] + 3) >> 2 : 0;
#pragma unroll
      for (int j = 0; j < WPP; ++j) {
        const int i = lane + 32 * j;
        f.v[q][j] = i < f.nwords[q] ? __ldg(pa + i) : 0u;
      }
    }
  };
  RowFetch cur;
  if (warp < RH) fetch(warp, cur);
  for (int oy = warp; oy < RH; oy += CROP_WARPS) {
    const int b0 = ty[2][oy], b1 = ty[3][oy];
    int shift[2] = {cur.shift[0], cur.shift[1]}, cshift[2] = {0, 0};
    if (NV) { cshift[0] = cur.shift[NSEG - 2]; cshift[1] = cur.shift[NSEG - 1]; }
    __syncwarp();  // the previous row's taps have been read
    {
      uint8_t* const ds[4] = {seg[warp][0], seg[warp][1], seg[warp][0] + CROP_SEG / 2, seg[warp][1] + CROP_SEG / 2};
#pragma unroll
      for (int q = 0; q < NSEG; ++q)
#pragma unroll
        for (int j = 0; j < WPP; ++j) {
          const int i = lane + 32 * j;
          if (i < cur.nwords[q]) reinterpret_cast<uint32_t*>(ds[q])[i] = cur.v[q][j];
        }
    }
    if (oy + CROP_WARPS < RH) fetch(oy + CROP_WARPS, cur);  // in flight while this row is interpolated
    __syncwarp();
#pragma unroll
    for (int k = 0; k < RW / 32; ++k) {
      const int ox = lane + 32 * k;
      const int sx[2] = {lsx[k][0], lsx[k][1]};
      crop_pixel<FORMAT>(mode, la[k][0], la[k][1], b0, b1,
                         [&](int r, int i, int (&v)[3]) {
                           if (!NV) {
                             const uint8_t* q = seg[warp][r] + shift[r] + sx[i] * 3;
                             v[0] = q[0]; v[1] = q[1]; v[2] = q[2];
                           } else {
                             const uint8_t* c = seg[warp][r] + CROP_SEG / 2 + cshift[r] + (((x1 + sx[i]) & ~1) - (x1 & ~1));
                             yuv_to_bgr_601(seg[warp][r][shift[r] + sx[i]], c[0], c[1], v);
                           }
                         },
                         out, slot, oy * RW + ox);
    }
  }
}


template <int FORMAT, int SRC>
__global__ void __launch_bounds__(32 * CROP_WARPS) crop_kernel(const uint8_t* __restrict__ frames, int batch, int h, int w,
                                                               const int* __restrict__ crop_rect,
                                                               const int* __restrict__ crop_count, void* __restrict__ out) {
  const int slot = blockIdx.x;
  if (slot >= *crop_count) return;
  __shared__ int tx[4][RW];
  __shared__ int ty[4][RH];
  __shared__ __align__(16) uint8_t seg[CROP_WARPS][2][CROP_SEG];
  const int b = crop_rect[slot * 5], x1 = crop_rect[slot * 5 + 1], y1 = crop_rect[slot * 5 + 2];
  const int cw = crop_rect[slot * 5 + 3] - x1, ch = crop_rect[slot * 5 + 4] - y1;
  // the frame batch is a multiple of 4 bytes long and 4-byte aligned: no word crosses its end
  const bool words = (reinterpret_cast<uintptr_t>(frames) & 3) == 0 && ((static_cast<long long>(batch) * FrameSrc<SRC>::frame_bytes(h, w)) & 3) == 0;
  crop_body<FORMAT>(FrameSrc<SRC>{frames + b * FrameSrc<SRC>::frame_bytes(h, w), h, w}, words, x1, y1, cw, ch, tx, ty, seg, out, slot);
}

// The crops over a frame table: each crop reads its frame's record (any size, pitch, BGR or NV12).  Whole words are loaded
// only from frames whose planes allow it (FrameRec::crop_staged); a crop at the last row of a separately allocated frame
// would otherwise read past the allocation.
template <int FORMAT>
__global__ void __launch_bounds__(32 * CROP_WARPS) crop_table_kernel(const FrameRec* __restrict__ recs, const int* __restrict__ crop_rect,
                                                                     const int* __restrict__ crop_count, void* __restrict__ out) {
  const int slot = blockIdx.x;
  if (slot >= *crop_count) return;
  __shared__ int tx[4][RW];
  __shared__ int ty[4][RH];
  __shared__ __align__(16) uint8_t seg[CROP_WARPS][2][CROP_SEG];
  const int b = crop_rect[slot * 5], x1 = crop_rect[slot * 5 + 1], y1 = crop_rect[slot * 5 + 2];
  const int cw = crop_rect[slot * 5 + 3] - x1, ch = crop_rect[slot * 5 + 4] - y1;
  const FrameRec& r = recs[b];
  if (r.kind == 0)
    crop_body<FORMAT>(FrameSrc<2>{r.data, r.pitch}, r.crop_staged != 0, x1, y1, cw, ch, tx, ty, seg, out, slot);
  else
    crop_body<FORMAT>(FrameSrc<3>{r.data, r.chroma, r.pitch}, r.crop_staged != 0, x1, y1, cw, ch, tx, ty, seg, out, slot);
}

}  // namespace
}  // namespace aicam

using namespace aicam;

namespace aicam {
namespace {
template <int SRC>
int reid_crops_impl(const uint8_t* frames, int batch, int h, int w, const float* boxes, const float* scores,
                    const int32_t* labels, const int32_t* num_dets, int stride_k, float min_confidence,
                    uint64_t class_mask_lo, uint64_t class_mask_hi, int format, int max_crops,
                    int32_t* det_index, int32_t* det_count, int32_t* crop_slot, int32_t* crop_rect,
                    void* crops, int32_t* crop_count, void* stream) {
  if (!boxes || !scores || !labels || !num_dets || !det_index || !det_count || !crop_slot || !crop_rect || !crop_count)
    return fail(AICAM_ERR_INVALID_ARG, "reid_crops: null argument");
  if (batch < 0 || stride_k <= 0 || h <= 0 || w <= 0 || max_crops < 0 || (format < 0 || format > 2))
    return fail(AICAM_ERR_INVALID_ARG, "reid_crops: bad shape arguments");
  if (reinterpret_cast<uintptr_t>(boxes) % 16) return fail(AICAM_ERR_INVALID_ARG, "reid_crops: boxes must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  filter_kernel<<<1, 1024, 0, st>>>(boxes, scores, labels, num_dets, batch, stride_k, h, w, min_confidence,
                                    class_mask_lo, class_mask_hi, max_crops, det_index, det_count, crop_slot, crop_rect,
                                    crop_count, nullptr, nullptr, nullptr);
  count_launch();
  if (int rc = last_launch("filter_kernel")) return rc;
  if (max_crops == 0 || !frames || !crops) return AICAM_OK;  // filter only
  if (format == 0)
    crop_kernel<0, SRC><<<max_crops, 32 * CROP_WARPS, 0, st>>>(frames, batch, h, w, crop_rect, crop_count, crops);
  else if (format == 1)
    crop_kernel<1, SRC><<<max_crops, 32 * CROP_WARPS, 0, st>>>(frames, batch, h, w, crop_rect, crop_count, crops);
  else
    crop_kernel<2, SRC><<<max_crops, 32 * CROP_WARPS, 0, st>>>(frames, batch, h, w, crop_rect, crop_count, crops);
  count_launch();
  return last_launch("crop_kernel");
}
}  // namespace
}  // namespace aicam

extern "C" int aicam_reid_crops(const uint8_t* frames, int batch, int h, int w, const float* boxes, const float* scores,
                                const int32_t* labels, const int32_t* num_dets, int stride_k, float min_confidence,
                                uint64_t class_mask_lo, uint64_t class_mask_hi, int format, int max_crops,
                                int32_t* det_index, int32_t* det_count, int32_t* crop_slot, int32_t* crop_rect,
                                void* crops, int32_t* crop_count, void* stream) {
  return reid_crops_impl<0>(frames, batch, h, w, boxes, scores, labels, num_dets, stride_k, min_confidence, class_mask_lo,
                            class_mask_hi, format, max_crops, det_index, det_count, crop_slot, crop_rect, crops, crop_count, stream);
}

extern "C" int aicam_reid_crops_nv12(const uint8_t* frames_nv12, int batch, int h, int w, const float* boxes, const float* scores,
                                     const int32_t* labels, const int32_t* num_dets, int stride_k, float min_confidence,
                                     uint64_t class_mask_lo, uint64_t class_mask_hi, int format, int max_crops,
                                     int32_t* det_index, int32_t* det_count, int32_t* crop_slot, int32_t* crop_rect,
                                     void* crops, int32_t* crop_count, void* stream) {
  if (h % 2 || w % 2) return fail(AICAM_ERR_INVALID_ARG, "reid_crops_nv12: NV12 frames have even height and width");
  return reid_crops_impl<1>(frames_nv12, batch, h, w, boxes, scores, labels, num_dets, stride_k, min_confidence, class_mask_lo,
                            class_mask_hi, format, max_crops, det_index, det_count, crop_slot, crop_rect, crops, crop_count, stream);
}

extern "C" int aicam_reid_crops_table(const aicam_frame_table* t, const float* boxes, const float* scores, const int32_t* labels,
                                      const int32_t* num_dets, int stride_k, float min_confidence, uint64_t class_mask_lo,
                                      uint64_t class_mask_hi, int format, int max_crops, int32_t* det_index, int32_t* det_count,
                                      int32_t* crop_slot, int32_t* crop_rect, void* crops, int32_t* crop_count, void* stream) {
  if (!t || !boxes || !scores || !labels || !num_dets || !det_index || !det_count || !crop_slot || !crop_rect || !crop_count)
    return fail(AICAM_ERR_INVALID_ARG, "reid_crops_table: null argument");
  if (stride_k <= 0 || max_crops < 0 || (format < 0 || format > 2))
    return fail(AICAM_ERR_INVALID_ARG, "reid_crops_table: bad shape arguments");
  if (reinterpret_cast<uintptr_t>(boxes) % 16) return fail(AICAM_ERR_INVALID_ARG, "reid_crops_table: boxes must be 16-byte aligned");
  if (t->region_test && stride_k > 1024)
    return fail(AICAM_ERR_CAPACITY, "reid_crops_table: the region test takes at most 1024 detections per frame (stride_k)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (t->region_test && t->n > 0) {
    region_kernel<<<t->n, REGION_THREADS, 0, st>>>(t->recs(), t->regions_dev, boxes, num_dets, stride_k, t->region_keep);
    count_launch();
    if (int rc = last_launch("region_kernel")) return rc;
  }
  const bool regions = t->region_test && t->n > 0;
  filter_kernel<<<1, 1024, 0, st>>>(boxes, scores, labels, num_dets, t->n, stride_k, 0, 0, min_confidence, class_mask_lo,
                                    class_mask_hi, max_crops, det_index, det_count, crop_slot, crop_rect, crop_count, t->recs(),
                                    regions ? t->region_keep : nullptr, regions ? t->regions_dev : nullptr);
  count_launch();
  if (int rc = last_launch("filter_kernel (table)")) return rc;
  if (max_crops == 0 || !crops) return AICAM_OK;  // filter only
  if (format == 0)
    crop_table_kernel<0><<<max_crops, 32 * CROP_WARPS, 0, st>>>(t->recs(), crop_rect, crop_count, crops);
  else if (format == 1)
    crop_table_kernel<1><<<max_crops, 32 * CROP_WARPS, 0, st>>>(t->recs(), crop_rect, crop_count, crops);
  else
    crop_table_kernel<2><<<max_crops, 32 * CROP_WARPS, 0, st>>>(t->recs(), crop_rect, crop_count, crops);
  count_launch();
  return last_launch("crop_table_kernel");
}

// NV12 -> packed BGR (cv2.cvtColor(.., COLOR_YUV2BGR_NV12)): the frames the NV12 entry points see, as the reference's
// decoder would have handed them out; for parity tests and for callers that keep a BGR copy.
namespace aicam {
namespace {
__global__ void __launch_bounds__(256) nv12_to_bgr_kernel(const uint8_t* __restrict__ nv12, int h, int w, uint8_t* __restrict__ bgr,
                                                          long long total) {
  const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;  // one thread per 2 horizontal pixels
  if (idx >= total) return;
  const int xp = static_cast<int>(idx % (w / 2));
  const long long t = idx / (w / 2);
  const int y = static_cast<int>(t % h);
  const long long n = t / h;
  const uint8_t* f = nv12 + n * FrameSrc<1>::frame_bytes(h, w);
  const uint8_t* c = f + static_cast<long long>(h) * w + static_cast<long long>(y >> 1) * w + 2 * xp;
  const int u = __ldg(c), v = __ldg(c + 1);
  int p0[3], p1[3];
  yuv_to_bgr_601(__ldg(f + static_cast<long long>(y) * w + 2 * xp), u, v, p0);
  yuv_to_bgr_601(__ldg(f + static_cast<long long>(y) * w + 2 * xp + 1), u, v, p1);
  uint8_t* o = bgr + ((n * h + y) * w + 2 * xp) * 3;
  o[0] = p0[0]; o[1] = p0[1]; o[2] = p0[2]; o[3] = p1[0]; o[4] = p1[1]; o[5] = p1[2];
}
}  // namespace
}  // namespace aicam

extern "C" int aicam_nv12_to_bgr(const uint8_t* frames_nv12, int batch, int h, int w, uint8_t* frames_bgr, void* stream) {
  if (!frames_nv12 || !frames_bgr || batch < 0 || h <= 0 || w <= 0 || h % 2 || w % 2)
    return fail(AICAM_ERR_INVALID_ARG, "nv12_to_bgr: bad arguments (NV12 frames have even height and width)");
  if (batch == 0) return AICAM_OK;
  const long long total = static_cast<long long>(batch) * h * (w / 2);
  nv12_to_bgr_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(frames_nv12, h, w, frames_bgr, total);
  count_launch();
  return last_launch("nv12_to_bgr_kernel");
}
