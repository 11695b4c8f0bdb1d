// K1: fused letterbox-resize / BGR->RGB / normalise / layout kernel.
//
// Replaces, per frame, image_processing.letterbox (cv2.resize INTER_LINEAR + copyMakeBorder
// 114, /root/reference/src/utils/image_processing.py:7-70), preprocess_yolo_input (BGR->RGB,
// HWC->CHW, /255, :73-102) and the 4.9 MB H2D copy of the float tensor
// (src/detector/yolo_detector.py:91).
//
// Bit-exactness: cv2.resize on uint8 is fixed point (11-bit coefficients, horizontal pass in
// int32, vertical pass (((b0*(r0>>4))>>16) + ((b1*(r1>>4))>>16) + 2) >> 2, exact-2x shortcut to
// the 2x2 box average).  The coefficient tables are computed on the HOST with the same
// double/float arithmetic OpenCV uses and cached per frame size; the kernel evaluates the
// integer formula, so the uint8 letterboxed image - and therefore the float tensor - equals
// the reference's bit for bit.  Taps with a zero weight are not loaded: for 1080p (exact 3:1)
// the kernel touches one source pixel per output pixel, 360 of the 1080 rows.
//
// Pure-decimation geometries (1080p -> 640 x 360 is exactly 3:1) take a row-staged path: bulk copies of each touched
// source row into a shared-memory ring, byte picks from there (preprocess_pairs_kernel).
//
// HBM-bound.  Algorithmic bytes per 1080p frame: 360 rows x 5760 B read + 640*640*8 B written
// (NHWC4 bf16) = 5 350 400 B   (format 0, fp32 NCHW: 2 073 600 + 4 915 200 B).
#include <cmath>
#include <cstdlib>
#include <map>
#include <mutex>
#include <vector>

#include "common.cuh"
#include "frame_src.cuh"
#include "frame_table.cuh"
#include "tc_ptx.cuh"

namespace aicam {

extern void count_launch();

namespace {

constexpr int S = AICAM_YOLO_INPUT;

struct Geometry {
  int decimate;  // every output pixel is exactly ONE source pixel (integer-ratio resize or copy): row-staged fast path
  int mode;  // 0 bilinear, 1 exact 2x box average, 2 copy
  int new_h, new_w, top, left;
  // device tables: x: sx0, sx1, a0, a1 (new_w each); y: sy0, sy1, b0, b1 (new_h each)
  int* tab;
};

struct GeoKey {
  int device, h, w;
  bool operator<(const GeoKey& o) const {
    return device != o.device ? device < o.device : (h != o.h ? h < o.h : w < o.w);
  }
};

std::map<GeoKey, Geometry> g_geo;
std::mutex g_geo_mutex;

int cv_round_coef(float v) { return static_cast<int>(std::nearbyintf(v * 2048.0f)); }

void axis_tables(int src, int dst, bool horizontal, std::vector<int>& i0, std::vector<int>& i1,
                 std::vector<int>& w0, std::vector<int>& w1) {
  const double scale = 1.0 / (static_cast<double>(dst) / static_cast<double>(src));
  for (int d = 0; d < dst; ++d) {
    float f = static_cast<float>((d + 0.5) * scale - 0.5);
    int s = static_cast<int>(std::floor(f));
    f -= static_cast<float>(s);
    if (horizontal) {
      if (s < 0) { f = 0.0f; s = 0; }
      if (s >= src - 1) { f = 0.0f; s = src - 1; }
      i0[d] = s;
      i1[d] = std::min(s + 1, src - 1);
    } else {
      i0[d] = std::min(std::max(s, 0), src - 1);
      i1[d] = std::min(std::max(s + 1, 0), src - 1);
    }
    w0[d] = cv_round_coef(1.0f - f);
    w1[d] = cv_round_coef(f);
  }
}

}  // namespace

void letterbox_geometry(int h, int w, double* r, int* new_h, int* new_w, double* dw, double* dh, int* top, int* left) {
  const double rh = std::min(static_cast<double>(S) / h, 1.0), rw = std::min(static_cast<double>(S) / w, 1.0);
  *r = std::min(rh, rw);
  *new_h = static_cast<int>(std::nearbyint(h * *r));  // python round(): half to even
  *new_w = static_cast<int>(std::nearbyint(w * *r));
  *dw = (S - *new_w) / 2.0;
  *dh = (S - *new_h) / 2.0;
  *top = static_cast<int>(std::nearbyint(*dh - 0.1));
  *left = static_cast<int>(std::nearbyint(*dw - 0.1));
}

namespace {

int get_geometry(int h, int w, Geometry* out) {
  int device = 0;
  AICAM_CUDA_OK(cudaGetDevice(&device));
  std::lock_guard<std::mutex> lock(g_geo_mutex);
  GeoKey key{device, h, w};
  auto it = g_geo.find(key);
  if (it != g_geo.end()) {
    *out = it->second;
    return AICAM_OK;
  }
  Geometry g;
  double r, dw, dh;
  letterbox_geometry(h, w, &r, &g.new_h, &g.new_w, &dw, &dh, &g.top, &g.left);
  if (g.new_h <= 0 || g.new_w <= 0 || g.new_h > S || g.new_w > S)
    return fail(AICAM_ERR_INVALID_ARG, "preprocess: frame size not supported");
  g.mode = (g.new_h == h && g.new_w == w) ? 2 : ((h == 2 * g.new_h && w == 2 * g.new_w) ? 1 : 0);
  std::vector<int> x0(g.new_w), x1(g.new_w), a0(g.new_w), a1(g.new_w), y0(g.new_h), y1(g.new_h), b0(g.new_h),
      b1(g.new_h);
  axis_tables(w, g.new_w, true, x0, x1, a0, a1);
  axis_tables(h, g.new_h, false, y0, y1, b0, b1);
  // pure decimation: all second taps have weight 0 (e.g. 1080p -> 640 x 360 is exactly 3:1, the bilinear sample
  // point falls on a source pixel centre), so cv2's fixed-point formula returns the source byte itself
  g.decimate = g.mode != 1;
  for (int d = 0; d < g.new_w && g.decimate; ++d) g.decimate = (a1[d] == 0 && a0[d] == 2048) || g.mode == 2;
  for (int d = 0; d < g.new_h && g.decimate; ++d) g.decimate = (b1[d] == 0 && b0[d] == 2048) || g.mode == 2;
  if (g.mode == 2) {  // copy: identity tables
    for (int d = 0; d < g.new_w; ++d) x0[d] = d;
    for (int d = 0; d < g.new_h; ++d) y0[d] = d;
  }
  std::vector<int> tab;
  for (auto* v : {&x0, &x1, &a0, &a1}) tab.insert(tab.end(), v->begin(), v->end());
  for (auto* v : {&y0, &y1, &b0, &b1}) tab.insert(tab.end(), v->begin(), v->end());
  AICAM_CUDA_OK(cudaMalloc(&g.tab, tab.size() * sizeof(int)));
  AICAM_CUDA_OK(cudaMemcpy(g.tab, tab.data(), tab.size() * sizeof(int), cudaMemcpyHostToDevice));
  g_geo[key] = g;
  *out = g;
  return AICAM_OK;
}

}  // namespace

int k1_geometry(int h, int w, int* decimate, int* mode, int* new_h, int* new_w, int* top, int* left, const int** tab) {
  Geometry g;
  if (int rc = get_geometry(h, w, &g)) return rc;
  *decimate = g.decimate; *mode = g.mode; *new_h = g.new_h; *new_w = g.new_w; *top = g.top; *left = g.left; *tab = g.tab;
  return AICAM_OK;
}

namespace {

constexpr int PIX = 4;  // output pixels per thread (consecutive x)

// float(v) / 255.0f, correctly rounded, for an integer 0 <= v <= 255: q = v * RN(1/255), one exact remainder, one
// correction (three instructions instead of the generic IEEE division sequence).  Equal to __fdiv_rn(v, 255.0f) for all
// 256 inputs (checked exhaustively with exact rational arithmetic; tests/test_gpu_preprocess.py compares every value
// with the oracle).  Explicit fmaf: this file is compiled with --fmad=false.
__device__ __forceinline__ float byte_to_unit(int v) {
  const float a = static_cast<float>(v);
  const float rcp = 0x1.010102p-8f;  // RN(1 / 255)
  const float q = a * rcp;
  return fmaf(fmaf(-255.0f, q, a), rcp, q);
}

// Output pixels 4 xg .. 4 xg + 3 of row y of frame n, read from `src` through the frame's letterbox geometry.
template <int FORMAT, typename Src>
__device__ __forceinline__ void preprocess_pixels(const Src& src, int mode, int new_h, int new_w, int top, int left,
                                                  const int* __restrict__ tab, void* __restrict__ out, int n, int y, int xg) {
  const int dy = y - top;
  const bool row_in = dy >= 0 && dy < new_h;
  const int* tx = tab;
  const int* ty = tab + 4 * new_w;
  int sy0 = 0, sy1 = 0, b0 = 0, b1 = 0;
  if (row_in) {
    sy0 = __ldg(ty + dy); sy1 = __ldg(ty + new_h + dy);
    b0 = __ldg(ty + 2 * new_h + dy); b1 = __ldg(ty + 3 * new_h + dy);
  }
  float rgb[PIX][3];
#pragma unroll
  for (int p = 0; p < PIX; ++p) {
    const int x = xg * PIX + p;
    const int dx = x - left;
    int v[3] = {114, 114, 114};  // BGR pad colour (image_processing.py:10)
    if (row_in && dx >= 0 && dx < new_w) {
      if (mode == 2) {
        src.pix(dy, dx, v);
      } else if (mode == 1) {
        int p00[3], p01[3], p10[3], p11[3];
        src.pix(2 * dy, 2 * dx, p00); src.pix(2 * dy, 2 * dx + 1, p01);
        src.pix(2 * dy + 1, 2 * dx, p10); src.pix(2 * dy + 1, 2 * dx + 1, p11);
#pragma unroll
        for (int c = 0; c < 3; ++c) v[c] = (p00[c] + p01[c] + p10[c] + p11[c] + 2) >> 2;
      } else {
        const int sx0 = __ldg(tx + dx), sx1 = __ldg(tx + new_w + dx);
        const int a0 = __ldg(tx + 2 * new_w + dx), a1 = __ldg(tx + 3 * new_w + dx);
        // taps with a zero weight are not fetched
        int p00[3] = {0, 0, 0}, p01[3] = {0, 0, 0}, p10[3] = {0, 0, 0}, p11[3] = {0, 0, 0};
        if (b0 != 0) {
          src.pix(sy0, sx0, p00);
          if (a1 != 0) src.pix(sy0, sx1, p01);
        }
        if (b1 != 0) {
          src.pix(sy1, sx0, p10);
          if (a1 != 0) src.pix(sy1, sx1, p11);
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const int h0 = p00[c] * a0 + p01[c] * a1, h1 = p10[c] * a0 + p11[c] * a1;
          int o = (((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2;
          v[c] = min(max(o, 0), 255);
        }
      }
    }
    // BGR -> RGB, /255 in float32 exactly as ndarray.astype(float32) / 255.0
    rgb[p][0] = byte_to_unit(v[2]);
    rgb[p][1] = byte_to_unit(v[1]);
    rgb[p][2] = byte_to_unit(v[0]);
  }
  if (FORMAT == 0) {
    float* o = static_cast<float*>(out) + static_cast<long long>(n) * 3 * S * S + static_cast<long long>(y) * S + xg * PIX;
#pragma unroll
    for (int c = 0; c < 3; ++c)
      *reinterpret_cast<float4*>(o + static_cast<long long>(c) * S * S) =
          make_float4(rgb[0][c], rgb[1][c], rgb[2][c], rgb[3][c]);
  } else {
    uint4 q0, q1;
    q0.x = pack_bf16x2(rgb[0][0], rgb[0][1]); q0.y = pack_bf16x2(rgb[0][2], 0.0f);
    q0.z = pack_bf16x2(rgb[1][0], rgb[1][1]); q0.w = pack_bf16x2(rgb[1][2], 0.0f);
    q1.x = pack_bf16x2(rgb[2][0], rgb[2][1]); q1.y = pack_bf16x2(rgb[2][2], 0.0f);
    q1.z = pack_bf16x2(rgb[3][0], rgb[3][1]); q1.w = pack_bf16x2(rgb[3][2], 0.0f);
    if (FORMAT == 1) {
      uint4* o = reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(out) +
                                          ((static_cast<long long>(n) * S + y) * S + xg * PIX) * 4);
      o[0] = q0;
      o[1] = q1;
    } else if (FORMAT == 2) {
      // space-to-depth: 2x2 pixel block (Y, X) = 16 channels [row parity][column parity][RGB0]; this thread
      // holds columns 4 xg .. 4 xg + 3 of row y = blocks X = 2 xg, 2 xg + 1, row parity y & 1
      uint4* o = reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(out) +
                                          ((static_cast<long long>(n) * (S / 2) + (y >> 1)) * (S / 2) + 2 * xg) * 16 + (y & 1) * 8);
      o[0] = q0;
      o[2] = q1;
    } else {
      // two levels of space-to-depth: 4x4 pixel block (Y, X) = 64 channels [2x2 sub-block (by, bx)][row parity][column
      // parity][RGB0] - the format-2 blocks grouped 2x2 once more; this thread holds row y of block X = xg
      uint4* o = reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(out) +
                                          ((static_cast<long long>(n) * (S / 4) + (y >> 2)) * (S / 4) + xg) * 64);
      const int by = (y >> 1) & 1, py = y & 1;
      o[by * 4 + py] = q0;
      o[by * 4 + 2 + py] = q1;
    }
  }
}

template <int FORMAT, int SRC>
__global__ void __launch_bounds__(256) preprocess_kernel(const uint8_t* __restrict__ frames, int h, int w, int mode,
                                                         int new_h, int new_w, int top, int left,
                                                         const int* __restrict__ tab, void* __restrict__ out,
                                                         long long total) {
  const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (idx >= total) return;
  const int xg = static_cast<int>(idx % (S / PIX));
  long long t = idx / (S / PIX);
  const int y = static_cast<int>(t % S);
  const int n = static_cast<int>(t / S);
  const FrameSrc<SRC> src{frames + n * FrameSrc<SRC>::frame_bytes(h, w), h, w};
  preprocess_pixels<FORMAT>(src, mode, new_h, new_w, top, left, tab, out, n, y, xg);
}

// The per-pixel path over a frame table: the frames of the table's per-pixel list (frame_table.cuh), any size, pitch and
// kind, each written at its packed slot (absent frames are on no list).  The grid is sized from the table's capacity and walks the list with a grid-stride loop; the list's length is read
// on the device, so a captured launch stays valid when the table is set to other frames.
template <int FORMAT>
__global__ void __launch_bounds__(256) preprocess_table_kernel(const int* __restrict__ counts, const int* __restrict__ list,
                                                               const FrameRec* __restrict__ recs, void* __restrict__ out) {
  const long long total = static_cast<long long>(counts[2]) * S * (S / PIX);
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int xg = static_cast<int>(idx % (S / PIX));
    const long long t = idx / (S / PIX);
    const int y = static_cast<int>(t % S);
    const FrameRec& r = recs[list[t / S]];
    if (r.kind == 0)
      preprocess_pixels<FORMAT>(FrameSrc<2>{r.data, r.pitch}, r.mode, r.new_h, r.new_w, r.top, r.left, r.tab, out, r.slot, y, xg);
    else
      preprocess_pixels<FORMAT>(FrameSrc<3>{r.data, r.chroma, r.pitch}, r.mode, r.new_h, r.new_w, r.top, r.left, r.tab, out, r.slot, y, xg);
  }
}

// Row-staged fast path for pure decimation (Geometry::decimate).  Persistent CTAs, each walking output-row PAIRS
// (y, y + 1 with y even: the two rows of a space-to-depth block row); the touched source rows of a pair are brought into
// a K1_STAGES-deep shared-memory ring by bulk copies (cp.async.bulk, completion counted on an mbarrier) issued by one
// thread up to K1_STAGES - 1 pairs ahead, so every SM keeps tens of KB of reads in flight without any thread waiting on
// a load; every byte of a touched row is fetched, one pixel in `ratio` is used (the algorithmic traffic in the header).
// Each thread then picks the bytes of its four pixels of both rows from shared memory and writes 64 contiguous bytes
// (format 2: two whole 2x2 blocks) or 32 per row (format 1).  Rows of the letterbox border issue no loads.
constexpr int K1_STAGES = 4;

// The frame an output-row pair of the row-staged path belongs to, and where its source rows are.
struct PairFrame {
  const uint8_t* data;    // BGR rows / NV12 luma rows, `pitch` bytes apart
  const uint8_t* chroma;  // NV12 chroma rows, `pitch` bytes apart
  int pitch, w, nv12, new_h, new_w, top, left, n;
  const int* tab;
};

// TABLE: the pairs are those of the frames on the table's row-staged list (frame_table.cuh), each with its own geometry and
// written at its packed slot, and the count is read on the device; the frame arguments are then unused and a ring stage holds two rows of stage_row bytes.
// Each CTA then walks one contiguous, even-aligned run of pairs, so that its frame - and the geometry it loads from the table,
// three dependent loads - changes at most a few times per CTA instead of at every pair.
template <int FORMAT, int SRC, bool TABLE = false>
__global__ void __launch_bounds__(S / PIX) preprocess_pairs_kernel(const uint8_t* __restrict__ frames, int h, int w, int new_h,
                                                                   int new_w, int top, int left, const int* __restrict__ tab,
                                                                   void* __restrict__ out, int n_pairs, int stages,
                                                                   const int* __restrict__ t_counts = nullptr,
                                                                   const int* __restrict__ t_list = nullptr,
                                                                   const FrameRec* __restrict__ t_recs = nullptr,
                                                                   int stage_row = 0) {
  extern __shared__ __align__(128) uint8_t sm_rows[];
  __shared__ __align__(8) uint64_t full_bar[K1_STAGES];
  const int row_bytes = TABLE ? stage_row : (SRC == 0 ? w * 3 : 2 * w);  // one staged source row: BGR, or the luma row followed by its chroma row
  const int stage_bytes = 2 * row_bytes;
  if (TABLE) n_pairs = t_counts[1] * (S / 2);
  const int tid = threadIdx.x;
  if (tid == 0) {
    for (int k = 0; k < stages; ++k) ptx::mbar_init(smem_u32(&full_bar[k]), 1);
    ptx::mbar_init_fence();
  }
  __syncthreads();
  auto frame_of = [&](int pair) -> PairFrame {
    PairFrame g;
    if (TABLE) {
      const FrameRec& r = t_recs[t_list[pair / (S / 2)]];
      g.n = r.slot;  // the packed network slot of the (present) frame
      g.data = r.data; g.chroma = r.chroma; g.pitch = r.pitch; g.w = r.w; g.nv12 = r.kind;
      g.new_h = r.new_h; g.new_w = r.new_w; g.top = r.top; g.left = r.left; g.tab = r.tab;
    } else {
      g.n = pair / (S / 2);
      g.data = frames + g.n * FrameSrc<SRC>::frame_bytes(h, w);
      g.chroma = g.data + static_cast<long long>(h) * w;
      g.pitch = SRC == 0 ? 3 * w : w; g.w = w; g.nv12 = SRC;
      g.new_h = new_h; g.new_w = new_w; g.top = top; g.left = left; g.tab = tab;
    }
    return g;
  };
  // Over a table the geometry of a pair's frame is reloaded only when the frame changes (list position k); on the uniform
  // path it is arithmetic.  One copy for thread 0's refills (which run ahead), one for the pair being computed.
  PairFrame ig, g;
  int ik = -1, gk = -1;
  auto issue = [&](int pair, int stage) {  // thread 0: the source rows of one output-row pair -> ring stage
    if (!TABLE || pair / (S / 2) != ik) {
      ik = pair / (S / 2);
      ig = frame_of(pair);
    }
    const int y0 = (pair - (pair / (S / 2)) * (S / 2)) * 2;
    const int* ty = ig.tab + 4 * ig.new_w;
    const uint32_t bar = smem_u32(&full_bar[stage]);
    const int fetch = ig.nv12 ? 2 * ig.w : 3 * ig.w;
    int sy[2];
    uint32_t bytes = 0;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int dy = y0 + r - ig.top;
      sy[r] = (dy >= 0 && dy < ig.new_h) ? __ldg(ty + dy) : -1;
      if (sy[r] >= 0) bytes += fetch;
    }
    ptx::mbar_arrive_expect_tx(bar, bytes);  // (a border pair completes the phase with no bytes)
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      if (sy[r] < 0) continue;
      const uint32_t dst = smem_u32(sm_rows + static_cast<size_t>(stage) * stage_bytes + r * row_bytes);
      if (!ig.nv12) {
        ptx::bulk_g2s(dst, ig.data + static_cast<long long>(sy[r]) * ig.pitch, fetch, bar);
      } else {
        ptx::bulk_g2s(dst, ig.data + static_cast<long long>(sy[r]) * ig.pitch, ig.w, bar);
        ptx::bulk_g2s(dst + ig.w, ig.chroma + static_cast<long long>(sy[r] >> 1) * ig.pitch, ig.w, bar);
      }
    }
  };
  // k-th item of this CTA: output-row pairs are handed out two at a time (n_pairs is even), so the four rows of a 4x4 pixel block
  // (format 3: the two 64-byte halves of a 128-byte block) are written by the same threads in consecutive iterations
  long long run_begin = 0, run_end = 0;  // TABLE: this CTA's pairs (run lengths even: pair parity = item parity)
  if (TABLE) {
    const int run = (n_pairs + 2 * static_cast<int>(gridDim.x) - 1) / (2 * static_cast<int>(gridDim.x)) * 2;
    run_begin = static_cast<long long>(blockIdx.x) * run;
    run_end = min(static_cast<long long>(n_pairs), run_begin + run);
  }
  auto pair_of = [&](int k) -> long long {
    if (TABLE) return run_begin + k < run_end ? run_begin + k : n_pairs;
    return 2 * (blockIdx.x + static_cast<long long>(k >> 1) * gridDim.x) + (k & 1);
  };
  if (tid == 0)
    for (int k = 0; k < stages; ++k) {
      const long long pair = pair_of(k);
      if (pair < n_pairs) issue(static_cast<int>(pair), k);
    }
  // the four source columns of this thread (for one geometry: fixed on the uniform path, per frame over a table)
  const int xg = tid;
  int sx[PIX];
  if (!TABLE) {
#pragma unroll
    for (int p = 0; p < PIX; ++p) {
      const int dx = xg * PIX + p - left;
      sx[p] = (dx >= 0 && dx < new_w) ? __ldg(tab + dx) : -1;
    }
  }
  for (int it = 0;; ++it) {
    const long long pair_l = pair_of(it);
    if (pair_l >= n_pairs) break;
    const int pair = static_cast<int>(pair_l);
    const int stage = it % stages;
    if (!TABLE || pair / (S / 2) != gk) {
      gk = pair / (S / 2);
      g = frame_of(pair);
      if (TABLE) {
#pragma unroll
        for (int p = 0; p < PIX; ++p) {
          const int dx = xg * PIX + p - g.left;
          sx[p] = (dx >= 0 && dx < g.new_w) ? __ldg(g.tab + dx) : -1;
        }
      }
    }
    const int n = g.n, y0 = (pair - (pair / (S / 2)) * (S / 2)) * 2;
    ptx::mbar_wait(smem_u32(&full_bar[stage]), (it / stages) & 1);
    uint4 q[2][2];
    float pl[2][PIX][3];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int dy = y0 + r - g.top;
      const bool row_in = dy >= 0 && dy < g.new_h;
      const uint8_t* srow = sm_rows + static_cast<size_t>(stage) * stage_bytes + r * row_bytes;
      float rgb[PIX][3];
#pragma unroll
      for (int p = 0; p < PIX; ++p) {
        int v0 = 114, v1 = 114, v2 = 114;  // BGR pad colour (image_processing.py:10)
        if (row_in && sx[p] >= 0) {
          if (!g.nv12) {
            const uint8_t* sp = srow + sx[p] * 3;
            v0 = sp[0]; v1 = sp[1]; v2 = sp[2];
          } else {
            int bgr[3];
            yuv_to_bgr_601(srow[sx[p]], srow[g.w + (sx[p] & ~1)], srow[g.w + (sx[p] & ~1) + 1], bgr);
            v0 = bgr[0]; v1 = bgr[1]; v2 = bgr[2];
          }
        }
        // BGR -> RGB, /255 in float32 exactly as ndarray.astype(float32) / 255.0
        rgb[p][0] = byte_to_unit(v2);
        rgb[p][1] = byte_to_unit(v1);
        rgb[p][2] = byte_to_unit(v0);
      }
      if (FORMAT == 0) {
#pragma unroll
        for (int p = 0; p < PIX; ++p)
#pragma unroll
          for (int c = 0; c < 3; ++c) pl[r][p][c] = rgb[p][c];
      } else {
        q[r][0].x = pack_bf16x2(rgb[0][0], rgb[0][1]); q[r][0].y = pack_bf16x2(rgb[0][2], 0.0f);
        q[r][0].z = pack_bf16x2(rgb[1][0], rgb[1][1]); q[r][0].w = pack_bf16x2(rgb[1][2], 0.0f);
        q[r][1].x = pack_bf16x2(rgb[2][0], rgb[2][1]); q[r][1].y = pack_bf16x2(rgb[2][2], 0.0f);
        q[r][1].z = pack_bf16x2(rgb[3][0], rgb[3][1]); q[r][1].w = pack_bf16x2(rgb[3][2], 0.0f);
      }
    }
    __syncthreads();  // the stage has been read by everyone: refill it
    if (tid == 0) {
      const long long next = pair_of(it + stages);
      if (next < n_pairs) issue(static_cast<int>(next), stage);
    }
    if (FORMAT == 0) {
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        float* o = static_cast<float*>(out) + static_cast<long long>(n) * 3 * S * S + static_cast<long long>(y0 + r) * S + xg * PIX;
#pragma unroll
        for (int c = 0; c < 3; ++c)
          *reinterpret_cast<float4*>(o + static_cast<long long>(c) * S * S) = make_float4(pl[r][0][c], pl[r][1][c], pl[r][2][c], pl[r][3][c]);
      }
    } else if (FORMAT == 1) {
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        uint4* o = reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(out) + ((static_cast<long long>(n) * S + y0 + r) * S + xg * PIX) * 4);
        o[0] = q[r][0];
        o[1] = q[r][1];
      }
    } else if (FORMAT == 2) {
      // space-to-depth: 2x2 pixel block (Y, X) = 16 channels [row parity][column parity][RGB0]; this thread holds
      // columns 4 xg .. 4 xg + 3 of both rows = the whole blocks X = 2 xg and 2 xg + 1 of block row y0 / 2
      uint4* o = reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(out) +
                                          ((static_cast<long long>(n) * (S / 2) + (y0 >> 1)) * (S / 2) + 2 * xg) * 16);
      o[0] = q[0][0];
      o[1] = q[1][0];
      o[2] = q[0][1];
      o[3] = q[1][1];
    } else {
      // 4x4 pixel blocks of 64 channels (format 3): these 64 bytes are sub-block row by = it & 1 of block (y0 / 4, xg).  The two
      // iterations of a block row leave their halves in a shared-memory image of the row's 160 blocks (20 KB, contiguous in the
      // tensor; 16-byte chunks XOR-swizzled by the block index so that neither side has bank conflicts), which the CTA then
      // writes with fully coalesced 16-byte stores - lanes 128 bytes apart measured 86 us per 64 frames instead of 74
      uint4* os = reinterpret_cast<uint4*>(sm_rows + static_cast<size_t>(stages) * stage_bytes);
      const int by = it & 1, sw = xg & 7;
      os[xg * 8 + ((by * 4 + 0) ^ sw)] = q[0][0];
      os[xg * 8 + ((by * 4 + 1) ^ sw)] = q[1][0];
      os[xg * 8 + ((by * 4 + 2) ^ sw)] = q[0][1];
      os[xg * 8 + ((by * 4 + 3) ^ sw)] = q[1][1];
      if (by) {
        __syncthreads();
        uint4* o = reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(out) + (static_cast<long long>(n) * (S / 4) + (y0 >> 2)) * (S / 4) * 64);
#pragma unroll
        for (int c = tid; c < (S / 4) * 8; c += S / PIX) {
          const int b = c >> 3;
          o[c] = os[b * 8 + ((c & 7) ^ (b & 7))];
        }
      }
    }
  }
}

}  // namespace

}  // namespace aicam

using namespace aicam;

namespace aicam {
namespace {
template <int SRC>
int preprocess_impl(const uint8_t* frames, int batch, int h, int w, int format, void* out, void* stream);
}
}  // namespace aicam

extern "C" {

int aicam_letterbox_params(int h, int w, aicam_letterbox* meta) {
  if (!meta || h <= 0 || w <= 0) return fail(AICAM_ERR_INVALID_ARG, "letterbox_params: bad arguments");
  int nh, nw, top, left;
  letterbox_geometry(h, w, &meta->ratio, &nh, &nw, &meta->pad_w, &meta->pad_h, &top, &left);
  return AICAM_OK;
}

int aicam_preprocess(const uint8_t* frames, int batch, int h, int w, int format, void* out, void* stream) {
  return preprocess_impl<0>(frames, batch, h, w, format, out, stream);
}

int aicam_preprocess_nv12(const uint8_t* frames_nv12, int batch, int h, int w, int format, void* out, void* stream) {
  if (h % 2 || w % 2) return fail(AICAM_ERR_INVALID_ARG, "preprocess_nv12: NV12 frames have even height and width");
  return preprocess_impl<1>(frames_nv12, batch, h, w, format, out, stream);
}

int aicam_preprocess_table(const aicam_frame_table* t, int format, void* out, void* stream) {
  if (!t || !out) return fail(AICAM_ERR_INVALID_ARG, "preprocess_table: null argument");
  if (format < 0 || format > 3) return fail(AICAM_ERR_INVALID_ARG, "preprocess_table: format must be 0, 1, 2 or 3");
  const int n = t->n;
  if (n == 0) return AICAM_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // Row-staged path: the ring is sized from the table's width bound, the grid from n; the kernel reads how many frames take it.
  const size_t stage_bytes = 2 * static_cast<size_t>(t->stage_row());
  if (t->ring_fits()) {  // (the condition under which aicam_frame_table_set puts frames on this path)
    int stages = K1_STAGES * stage_bytes <= K1_SMEM_LIMIT / 2 ? K1_STAGES : 2;
    if (format == 3) stages = 2;  // as aicam_preprocess
    const size_t smem = stages * stage_bytes + (format == 3 ? K1_BLOCK_ROW_IMAGE : 0);
    auto kernel = format == 0 ? preprocess_pairs_kernel<0, 0, true>
                              : (format == 1 ? preprocess_pairs_kernel<1, 0, true>
                                             : (format == 2 ? preprocess_pairs_kernel<2, 0, true> : preprocess_pairs_kernel<3, 0, true>));
    if (smem > 48 * 1024) {
      if (int rc = ensure_dynamic_smem(kernel, K1_SMEM_LIMIT)) return rc;
    }
    const int per_sm = static_cast<int>(std::max<size_t>(1, std::min<size_t>(8, K1_SMEM_LIMIT / (smem + 1024))));
    const unsigned grid = static_cast<unsigned>(std::min<long long>(static_cast<long long>(n) * (S / 4), static_cast<long long>(current_num_sms()) * per_sm));
    kernel<<<grid, S / PIX, smem, st>>>(nullptr, 0, 0, 0, 0, 0, 0, nullptr, out, 0, stages, t->counts(), t->lists(), t->recs(),
                                        t->stage_row());
    count_launch();
    if (int rc = last_launch("preprocess_pairs_kernel (table)")) return rc;
  }
  // Per-pixel path for every other frame.
  auto kernel = format == 0 ? preprocess_table_kernel<0>
                            : (format == 1 ? preprocess_table_kernel<1> : (format == 2 ? preprocess_table_kernel<2> : preprocess_table_kernel<3>));
  const long long total = static_cast<long long>(n) * S * (S / PIX);
  const unsigned blocks = static_cast<unsigned>(std::min<long long>((total + 255) / 256, static_cast<long long>(current_num_sms()) * 8));
  kernel<<<blocks, 256, 0, st>>>(t->counts(), t->lists() + t->capacity, t->recs(), out);
  count_launch();
  return last_launch("preprocess_table_kernel");
}

}  // extern "C"

namespace aicam {
namespace {
template <int SRC>
int preprocess_impl(const uint8_t* frames, int batch, int h, int w, int format, void* out, void* stream) {
  if (!frames || !out || batch < 0 || h <= 0 || w <= 0) return fail(AICAM_ERR_INVALID_ARG, "preprocess: bad arguments");
  if (format < 0 || format > 3) return fail(AICAM_ERR_INVALID_ARG, "preprocess: format must be 0, 1, 2 or 3");
  if (batch == 0) return AICAM_OK;
  Geometry g;
  if (int rc = get_geometry(h, w, &g)) return rc;
  const long long total = static_cast<long long>(batch) * S * (S / PIX);
  const unsigned blocks = static_cast<unsigned>((total + 255) / 256);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  static const bool no_fast = getenv("AICAM_PREPROCESS_GENERIC") != nullptr;
  const int row_bytes = SRC == 0 ? w * 3 : w;  // bytes of one bulk copy (NV12: the luma row; its chroma row has as many)
  const size_t stage_bytes = 2 * (SRC == 0 ? static_cast<size_t>(w) * 3 : static_cast<size_t>(w) * 2);
  if (g.decimate && !no_fast && row_bytes % 16 == 0 && reinterpret_cast<uintptr_t>(frames) % 16 == 0 &&
      FrameSrc<SRC>::frame_bytes(h, w) % 16 == 0 && (static_cast<long long>(h) * w) % 16 == 0 && 2 * stage_bytes <= 200 * 1024) {
    const int n_pairs = batch * (S / 2);
    int stages = K1_STAGES * stage_bytes <= 100 * 1024 ? K1_STAGES : 2;
    if (format == 3) stages = 2;  // with the 20 KB block-row image, two stages keep four CTAs per SM: measured 63 us per 64 frames against 70 with four
    const size_t smem = stages * stage_bytes + (format == 3 ? static_cast<size_t>(S / 4) * 128 : 0);  // + the block-row image of format 3
    auto kernel = format == 0 ? preprocess_pairs_kernel<0, SRC>
                              : (format == 1 ? preprocess_pairs_kernel<1, SRC> : (format == 2 ? preprocess_pairs_kernel<2, SRC> : preprocess_pairs_kernel<3, SRC>));
    if (smem > 48 * 1024) {
      if (int rc = ensure_dynamic_smem(kernel, 200 * 1024)) return rc;
    }
    const int per_sm = static_cast<int>(std::max<size_t>(1, std::min<size_t>(8, (200 * 1024) / (smem + 1024))));
    const unsigned grid = static_cast<unsigned>(std::min<long long>(n_pairs / 2, static_cast<long long>(current_num_sms()) * per_sm));
    kernel<<<grid, S / PIX, smem, st>>>(frames, h, w, g.new_h, g.new_w, g.top, g.left, g.tab, out, n_pairs, stages, nullptr, nullptr,
                                        nullptr, 0);
    count_launch();
    return last_launch("preprocess_pairs_kernel");
  }
  auto kernel = format == 0 ? preprocess_kernel<0, SRC>
                            : (format == 1 ? preprocess_kernel<1, SRC> : (format == 2 ? preprocess_kernel<2, SRC> : preprocess_kernel<3, SRC>));
  kernel<<<blocks, 256, 0, st>>>(frames, h, w, g.mode, g.new_h, g.new_w, g.top, g.left, g.tab, out, total);
  count_launch();
  return last_launch("preprocess_kernel");
}
}  // namespace
}  // namespace aicam
