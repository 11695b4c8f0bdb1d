// K7-K12: the whole DeepSORT association on device, one CTA per video stream.
//
// Replaces /root/reference/src/tracker/core/ (kalman_filter.py, track.py, detection.py,
// matching.py, linear_assignment.py, tracker_core.py) and the formatting loop of
// DeepSORT.update (src/tracker/deepsort_tracker.py:123-141).
//
// Bit-exactness.  The reference tracker is float32 end to end and its Kalman algebra only
// ever touches four 2x2 blocks of the covariance, so every BLAS/LAPACK call reduces to a
// fixed sequence of correctly rounded float32 operations (oracle/kalman.py, SURVEY.md
// Appendix C).  This file spells those sequences out and is compiled with --fmad=false, so
// no product-sum is contracted.  The assignment follows scipy's rectangular LSAP step by
// step in float64 (oracle/lsap.py, SURVEY.md Appendix B): the column scan is spread over
// one warp (small problems) or the whole CTA, and the (value, first position, last unassigned
// position) reduction reproduces the sequential tie rule exactly.  The only value that is NOT
// bit-reproducible is the cosine distance (a BLAS sgemm in the reference): parity there is
// a tolerance, and assignments are bit-exact given the same cost matrix.
//
// State layout in HBM (struct of arrays, per stream, indexed by a track SLOT):
//   mean[S][T][8] cov[S][T][16] f32 | id/state/hits/age/tsu/class[S][T] i32 | conf[S][T] f32
//   gallery[S][T][G][F] f32 (L2-normalised at insert; ring buffer: head, count)
//   order[S][T]: slots of the live tracks in creation order (the reference's track list)
//   free_slots[S][T] stack, next_id[S]
//   row_slot[S][T]: the slot behind each row of out_tracks of the last step (what aicam_counter_step keys its state by)
//   trk_n_init/trk_max_age[S][T] i32: the n_init / max_age a track was created with (track.py keeps them per track)
//   assoc[S]: each stream's association settings (aicam_tracker_set_stream_assoc), read once per step by its CTA
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "common.cuh"
#include "staging.cuh"

namespace aicam {

extern void count_launch();

// appearance_tf32.cu: K8 of crowded frames on the tensor cores (TF32x3)
struct AppearanceTf32;
bool appearance_tf32_eligible(int S, int F, int G, int D);
int appearance_tf32_create(AppearanceTf32** out, int S, int T, int D, int F, int G, const float* gal_hi, const float* gal_lo,
                           const float* feat_hi, const float* feat_lo);
void appearance_tf32_destroy(AppearanceTf32* p);
int launch_appearance_tf32(const AppearanceTf32* p, int S, int T, int D, int F, int G, int min_dets, const int* n_tracks,
                           const int* order, const int* state, const int* gal_count, const int* det_count, const int* crop_slot,
                           int stride_k, const int* present, float* app_cost,
                           cudaStream_t stream);

namespace {

constexpr int TENTATIVE = 1, CONFIRMED = 2, DELETED = 3;  // track.py:10-14
constexpr float INFTY_COST = 1e5f;                         // linear_assignment.py:9
constexpr float CHI2_GATE = 9.487729036781154f;            // kalman_filter.py:16, compared in float32
constexpr int ASSOC_THREADS = 256;

// one stream's association settings: the thresholds as the reference compares them (float32 of the Python float) and the
// clamps of linear_assignment.py:58 (max_distance + 1e-5 rounded from double), the cascade depth and the confirmation count
struct AssocRec {
  float thr_cos, clamp_cos, thr_iou, clamp_iou;
  int max_age, n_init;
};

AssocRec resolve_assoc(const aicam_stream_assoc& a) {
  return AssocRec{static_cast<float>(a.max_cosine_distance), static_cast<float>(a.max_cosine_distance + 1e-5),
                  static_cast<float>(a.max_iou_distance), static_cast<float>(a.max_iou_distance + 1e-5), a.max_age, a.n_init};
}

struct Dev {
  int S, T, D, F, G;
  const AssocRec* assoc;  // [S]
  int* trk_n_init; int* trk_max_age;
  float* mean; float* cov;
  int* track_id; int* state; int* hits; int* age; int* tsu; int* cls; float* conf;
  int* gal_count; int* gal_head; float* gallery;
  int* order; int* n_tracks; int* free_slots; int* n_free; int* next_id; int* overflow;
  int* row_slot;    // [S][T]: tracker slot of each reported row of the last step (aicam_tracker_row_slots)
  float* app_cost;  // [S][T][D] by (slot, det)
  float* cost_ws;   // [S][T*D]
  float* featn;     // [S][D][F]
  // TF32 split copies (x = hi + lo, hi exactly representable with a 10-bit mantissa) of the gallery and of the
  // normalised detection features: the operands of appearance_tf32.cu; null when that path is not in use
  float* gal_hi; float* gal_lo; float* featn_hi; float* featn_lo;
};

__device__ __forceinline__ float tf32_hi(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u); }

// ---- float32 building blocks (oracle/kalman.py) ------------------------------------------------
__device__ __forceinline__ float sq_via_double(float x) {
  const double d = static_cast<double>(x);
  return static_cast<float>(d * d);
}
__device__ __forceinline__ float c_wp() { return static_cast<float>(1.0 / 20); }
__device__ __forceinline__ float c_wv() { return static_cast<float>(1.0 / 160); }
__device__ __forceinline__ float c_wp2() { return static_cast<float>(2 * (1.0 / 20)); }
__device__ __forceinline__ float c_wv10() { return static_cast<float>(10 * (1.0 / 160)); }
__device__ __forceinline__ float c_sq_1e2() { return static_cast<float>(1e-2 * 1e-2); }
__device__ __forceinline__ float c_sq_1e5() { return static_cast<float>(1e-5 * 1e-5); }
__device__ __forceinline__ float c_sq_1e1() { return static_cast<float>(1e-1 * 1e-1); }

// kalman_filter.py:55-83
__device__ void kf_initiate(const float z[4], float* mean, float* cov) {
  for (int i = 0; i < 4; ++i) { mean[i] = z[i]; mean[4 + i] = 0.0f; }
  const float sp = sq_via_double(c_wp2() * z[3]);
  const float sv = sq_via_double(c_wv10() * z[3]);
  for (int i = 0; i < 4; ++i) {
    cov[i] = (i == 2) ? c_sq_1e2() : sp;
    cov[4 + i] = 0.0f;
    cov[8 + i] = 0.0f;
    cov[12 + i] = (i == 2) ? c_sq_1e5() : sv;
  }
}

// kalman_filter.py:85-120  (P' = F (P F^T) + Q)
__device__ void kf_predict(float* mean, float* cov) {
  const float h = mean[3];
  const float sp = sq_via_double(c_wp() * h);
  const float sv = sq_via_double(c_wv() * h);
  for (int i = 0; i < 4; ++i) {
    const float a = cov[i], b = cov[4 + i], c = cov[8 + i], d = cov[12 + i];
    const float qp = (i == 2) ? c_sq_1e2() : sp;
    const float qv = (i == 2) ? c_sq_1e5() : sv;
    mean[i] = mean[i] + mean[4 + i];
    const float y00 = a + b;
    const float y10 = c + d;
    cov[i] = (y00 + y10) + qp;
    cov[4 + i] = b + d;
    cov[8 + i] = y10;
    cov[12 + i] = d + qv;
  }
}

// diagonal of S = H P H^T + R, kalman_filter.py:122-151
__device__ __forceinline__ float kf_innov(const float* mean, const float* cov, int i) {
  const float r = (i == 2) ? c_sq_1e1() : sq_via_double(c_wp() * mean[3]);
  return cov[i] + r;
}

// kalman_filter.py:206-249; n_meas selects the OpenBLAS path the reference takes
__device__ float kf_gating(const float* mean, const float* cov, const float z[4], int n_meas) {
  float q[4];
  for (int i = 0; i < 4; ++i) {
    const float L = sqrtf(kf_innov(mean, cov, i));
    const float delta = z[i] - mean[i];
    const float y = (n_meas >= 2) ? delta * (1.0f / L) : delta / L;
    q[i] = y * y;
  }
  return ((q[0] + q[1]) + q[2]) + q[3];
}

// kalman_filter.py:153-204
__device__ void kf_update(float* mean, float* cov, const float z[4]) {
  float nm[8], nc[16];
  for (int i = 0; i < 4; ++i) {
    const float a = cov[i], b = cov[4 + i], c = cov[8 + i], d = cov[12 + i];
    const float s = kf_innov(mean, cov, i);
    const float inv = 1.0f / sqrtf(s);
    const float k0 = (a * inv) * inv;
    const float k1 = (c * inv) * inv;
    const float e = z[i] - mean[i];
    nm[i] = mean[i] + k0 * e;
    nm[4 + i] = mean[4 + i] + k1 * e;
    const float s0 = s * k0, s1 = s * k1;
    nc[i] = a - k0 * s0;
    nc[4 + i] = b - k0 * s1;
    nc[8 + i] = c - k1 * s0;
    nc[12 + i] = d - k1 * s1;
  }
  for (int i = 0; i < 8; ++i) mean[i] = nm[i];
  for (int i = 0; i < 16; ++i) cov[i] = nc[i];
}

// detection.py:36-47
__device__ __forceinline__ void tlwh_to_xyah(const float t[4], float z[4]) {
  z[0] = t[0] + t[2] / 2.0f;
  z[1] = t[1] + t[3] / 2.0f;
  z[2] = t[3] > 0.0f ? t[2] / t[3] : 0.0f;
  z[3] = t[3];
}

// track.py:133-151
__device__ __forceinline__ void mean_to_tlwh(const float* mean, float t[4]) {
  float h = mean[3], w;
  if (h > 0.0f) { w = mean[2] * h; } else { w = 0.0f; h = fmaxf(0.0f, h); }
  t[0] = mean[0] - w / 2.0f;
  t[1] = mean[1] - h / 2.0f;
  t[2] = w;
  t[3] = h;
}

// matching.py:13-54, cost = 1 - IoU (matching.py:104)
__device__ __forceinline__ float iou_cost(const float a[4], const float c[4]) {
  const float abx = a[0] + a[2], aby = a[1] + a[3];
  const float cbx = c[0] + c[2], cby = c[1] + c[3];
  const float tlx = fmaxf(a[0], c[0]), tly = fmaxf(a[1], c[1]);
  const float brx = fminf(abx, cbx), bry = fminf(aby, cby);
  const float iw = fmaxf(0.0f, brx - tlx), ih = fmaxf(0.0f, bry - tly);
  const float inter = iw * ih;
  const float area_a = a[2] * a[3], area_c = c[2] * c[3];
  const float uni = (area_a + area_c) - inter;
  const float iou = inter / fmaxf(uni, 1e-7f);
  return 1.0f - iou;
}

// ---- rectangular LSAP (scipy _lsap) on one warp or on the whole CTA ------------------------------
struct LsapMem {
  double* wmn; int* wf; int* wlu;  // cross-warp reduction slots, [2 parities][4 warps]
  double* u; double* v; double* spc;
  int* path; int* col4row; int* row4col; int* remaining;
  unsigned char* SR; unsigned char* SC;
};
constexpr int LSAP_MAX_WARPS = 4;
constexpr int LSAP_WIDE = 48;  // problems with more columns than this are scanned by LSAP_MAX_WARPS warps

// minimum over the warp of a non-NaN double in two redux.sync steps: the bit pattern is mapped to an unsigned key whose
// order is the order of the values (-0.0 sorts below +0.0; the callers only compare the result with ==, which does not
// tell them apart), high word first, then the low word among the lanes that hold the minimal high word
__device__ __forceinline__ double warp_min_d(double x) {
  unsigned long long b = static_cast<unsigned long long>(__double_as_longlong(x));
  b = (b >> 63) ? ~b : (b | 0x8000000000000000ull);
  const unsigned hi = static_cast<unsigned>(b >> 32), lo = static_cast<unsigned>(b);
  const unsigned mhi = __reduce_min_sync(0xffffffffu, hi);
  const unsigned mlo = __reduce_min_sync(0xffffffffu, hi == mhi ? lo : 0xffffffffu);
  unsigned long long mb = (static_cast<unsigned long long>(mhi) << 32) | mlo;
  mb = (mb >> 63) ? (mb & 0x7fffffffffffffffull) : ~mb;
  return __longlong_as_double(static_cast<long long>(mb));
}

// cost(r, c) = cost[rmap[r] * ld + cmap[c]] (identity maps when null) for r < nr, c < nc.  Writes col_for_row[r] (or -1)
// for r < nr.  Called by the first nw warps of the CTA (tid < 32 nw; nw = 1: warp-synchronous, nw > 1: named barrier 1); every array
// lives in shared memory.  The column scan of the augmenting-path search - scipy's sequential loop over `remaining` - is
// strided over the threads; each keeps (lowest value, first position holding it, last UNASSIGNED position holding it),
// positions packed with their column as (position << 10 | column), and the reduction over lanes and warps reproduces the
// sequential tie rule exactly: the last unassigned column among the minima if there is one, else the first minimum.
// The thread that owns position `index` performs scipy's swap-removal itself, so one barrier per iteration suffices.
__device__ void lsap_cta(const float* cost, int ld, int nr, int nc, const LsapMem& m, int* col_for_row, int tid, int nw,
                         const int* rmap = nullptr, const int* cmap = nullptr) {
  const int nth = nw * 32, lane = tid & 31, warp = tid >> 5;
  auto sync = [&]() {
    if (nw == 1) __syncwarp();
    else asm volatile("bar.sync 1, %0;" ::"r"(nth) : "memory");
  };
  const bool tr = nc < nr;  // scipy transposes so that rows <= cols
  const int R = tr ? nc : nr, C = tr ? nr : nc;
  // element (i, j) of the (possibly transposed) problem
  auto at = [&](int i, int j) {
    const int r = tr ? j : i, c = tr ? i : j;
    return cost[static_cast<long long>(rmap ? rmap[r] : r) * ld + (cmap ? cmap[c] : c)];
  };
  if (R == 1) {
    // One row (a cascade level that holds one track, or one detection left): the search above scans `remaining`, i.e.
    // the columns in DESCENDING order, all of them unassigned, and keeps the last minimum it meets = the minimal cost at
    // the smallest column index; the float64 arithmetic reduces to the cost itself.  Warp 0 finds it with two redux steps.
    if (warp == 0) {
      float best = __int_as_float(0x7f800000);
      int bj = 0x7fffffff;
      for (int j = lane; j < C; j += 32) {
        const float c = at(0, j);
        if (c < best) { best = c; bj = j; }
      }
      unsigned kb = __float_as_uint(best);
      kb = (kb >> 31) ? ~kb : (kb | 0x80000000u);
      const unsigned mk = __reduce_min_sync(0xffffffffu, kb);
      // (== on the values, not on the keys: -0.0f and 0.0f are one minimum)
      const float mv = __uint_as_float((mk >> 31) ? (mk & 0x7fffffffu) : ~mk);
      const int j = __reduce_min_sync(0xffffffffu, best == mv ? bj : 0x7fffffff);
      for (int r = lane; r < nr; r += 32) col_for_row[r] = -1;
      __syncwarp();
      if (lane == 0) col_for_row[tr ? j : 0] = tr ? 0 : j;
      __syncwarp();
    }
    sync();
    return;
  }
  if (C <= 32) {
    // Up to 32 columns: the whole state lives in registers of warp 0 - lane j holds column j (v, shortest path cost,
    // path, row4col, its position in scipy's `remaining` array) and lane i holds row i (u, col4row, SR).  Same search,
    // same float64 arithmetic, same tie rule (positions instead of a scanned array: the swap-removal moves the column at
    // the last position to `index`); no shared-memory traffic but the cost element.
    if (warp == 0) {
      const double inf = __longlong_as_double(0x7ff0000000000000ll);
      const bool is_col = lane < C, is_row = lane < R;
      // loop-invariant half of the element address
      const int fix_c = is_col ? (tr ? (rmap ? rmap[lane] : lane) * ld : (cmap ? cmap[lane] : lane)) : 0;
      double u = 0.0, v = 0.0;
      int col4row = -1, row4col = -1, path = -1;
      for (int cur = 0; cur < R; ++cur) {
        double spc = inf, min_val = 0.0;
        bool SC = false, SR = false;
        int pos = C - 1 - lane, i = cur, num_remaining = C, sink = -1;
        while (sink == -1) {
          if (lane == i) SR = true;
          const double ui = __shfl_sync(0xffffffffu, u, i);
          const int var_i = tr ? (cmap ? cmap[i] : i) : (rmap ? rmap[i] : i) * ld;
          const bool active = is_col && !SC;
          if (active) {
            const double r = ((min_val + static_cast<double>(cost[fix_c + var_i])) - ui) - v;
            if (r < spc) { path = i; spc = r; }
          }
          const double sv = active ? spc : inf;
          const double mn = warp_min_d(sv);
          const bool ismin = active && sv == mn;
          const int f = __reduce_min_sync(0xffffffffu, ismin ? pos : 0x7fffffff);
          const int lu = __reduce_max_sync(0xffffffffu, (ismin && row4col == -1) ? pos : -1);
          const int index = lu >= 0 ? lu : f;
          const int jl = __ffs(__ballot_sync(0xffffffffu, active && pos == index)) - 1;
          const int owner = __shfl_sync(0xffffffffu, row4col, jl);
          min_val = mn;
          if (owner == -1) sink = jl; else i = owner;
          if (active && pos == num_remaining - 1) pos = index;  // remaining[index] = remaining[--num_remaining]
          if (lane == jl) SC = true;
          --num_remaining;
        }
        // dual variables (rows in SR other than cur are assigned: col4row is a lane)
        const double spc_of_mine = __shfl_sync(0xffffffffu, spc, col4row < 0 ? 0 : col4row);
        if (lane == cur) u += min_val;
        else if (is_row && SR) u += min_val - spc_of_mine;
        if (SC) v -= min_val - spc;
        // augment along the path
        for (int j = sink;;) {
          const int ii = __shfl_sync(0xffffffffu, path, j);
          if (lane == j) row4col = ii;
          const int nxt = __shfl_sync(0xffffffffu, col4row, ii);
          if (lane == ii) col4row = j;
          j = nxt;
          if (ii == cur) break;
        }
      }
      for (int r = lane; r < nr; r += 32) col_for_row[r] = -1;
      __syncwarp();
      if (is_row) col_for_row[tr ? col4row : lane] = tr ? lane : col4row;
      __syncwarp();
    }
    sync();
    return;
  }
  for (int i = tid; i < R; i += nth) { m.u[i] = 0.0; m.col4row[i] = -1; }
  for (int j = tid; j < C; j += nth) { m.v[j] = 0.0; m.row4col[j] = -1; m.path[j] = -1; }
  sync();
  const double inf = __longlong_as_double(0x7ff0000000000000ll);
  int par = 0;
  for (int cur = 0; cur < R; ++cur) {
    for (int j = tid; j < C; j += nth) { m.spc[j] = inf; m.SC[j] = 0; m.remaining[j] = C - 1 - j; }
    for (int i = tid; i < R; i += nth) m.SR[i] = 0;
    sync();
    double min_val = 0.0;
    int i = cur, num_remaining = C, sink = -1;
    while (sink == -1) {
      if (tid == 0) m.SR[i] = 1;
      const double ui = m.u[i];
      double lowest = inf;
      int first_key = 0x7fffffff, last_un = -1;
      for (int it = tid; it < num_remaining; it += nth) {
        const int j = m.remaining[it];
        const double r = ((min_val + static_cast<double>(at(i, j))) - ui) - m.v[j];
        double sv = m.spc[j];
        if (r < sv) { m.path[j] = i; m.spc[j] = r; sv = r; }
        const bool unassigned = m.row4col[j] == -1;
        const int key = (it << 10) | j;
        if (sv < lowest) { lowest = sv; first_key = key; last_un = unassigned ? key : -1; }
        else if (sv == lowest && unassigned) { last_un = key; }
      }
      double mn = warp_min_d(lowest);
      int f = __reduce_min_sync(0xffffffffu, lowest == mn ? first_key : 0x7fffffff);
      int lu = __reduce_max_sync(0xffffffffu, lowest == mn ? last_un : -1);
      if (nw > 1) {
        if (lane == 0) { m.wmn[par * LSAP_MAX_WARPS + warp] = mn; m.wf[par * LSAP_MAX_WARPS + warp] = f; m.wlu[par * LSAP_MAX_WARPS + warp] = lu; }
        sync();
        double g = m.wmn[par * LSAP_MAX_WARPS];
        for (int w = 1; w < nw; ++w) g = fmin(g, m.wmn[par * LSAP_MAX_WARPS + w]);
        f = 0x7fffffff; lu = -1;
        for (int w = 0; w < nw; ++w)
          if (m.wmn[par * LSAP_MAX_WARPS + w] == g) { f = min(f, m.wf[par * LSAP_MAX_WARPS + w]); lu = max(lu, m.wlu[par * LSAP_MAX_WARPS + w]); }
        mn = g;
        par ^= 1;
      }
      const int key = lu >= 0 ? lu : f;
      const int index = key >> 10, j = key & 1023;
      min_val = mn;
      const int owner = m.row4col[j];
      if (owner == -1) sink = j; else i = owner;
      // scipy: remaining[index] = remaining[--num_remaining].  Position `index` is scanned by thread index % nth, which
      // does the swap; the moved element was last written before this iteration's barrier
      if (index % nth == tid) m.remaining[index] = m.remaining[num_remaining - 1];
      if (tid == 0) m.SC[j] = 1;
      --num_remaining;
      if (nw == 1) __syncwarp();
    }
    sync();
    if (tid == 0) m.u[cur] += min_val;
    for (int i2 = tid; i2 < R; i2 += nth)
      if (m.SR[i2] && i2 != cur) m.u[i2] += min_val - m.spc[m.col4row[i2]];
    for (int j2 = tid; j2 < C; j2 += nth)
      if (m.SC[j2]) m.v[j2] -= min_val - m.spc[j2];
    sync();
    if (tid == 0) {
      int j = sink;
      for (;;) {
        const int ii = m.path[j];
        m.row4col[j] = ii;
        const int t = m.col4row[ii];
        m.col4row[ii] = j;
        j = t;
        if (ii == cur) break;
      }
    }
    sync();
  }
  for (int r = tid; r < nr; r += nth) col_for_row[r] = -1;
  sync();
  if (tr) { for (int k = tid; k < R; k += nth) col_for_row[m.col4row[k]] = k; }
  else    { for (int k = tid; k < R; k += nth) col_for_row[k] = m.col4row[k]; }
  sync();
}

__host__ __device__ inline int lsap_warps(int nr, int nc) { return (nr > nc ? nr : nc) > LSAP_WIDE ? LSAP_MAX_WARPS : 1; }

__host__ __device__ inline size_t lsap_bytes(int n) {
  return (128 + static_cast<size_t>(n) * (3 * 8 + 4 * 4 + 2) + 64 + 15) / 16 * 16;
}
__device__ inline LsapMem lsap_carve(uint8_t* p, int n) {
  LsapMem m;
  m.wmn = reinterpret_cast<double*>(p); m.wf = reinterpret_cast<int*>(m.wmn + 2 * LSAP_MAX_WARPS); m.wlu = m.wf + 2 * LSAP_MAX_WARPS;
  m.u = reinterpret_cast<double*>(p + 128); m.v = m.u + n; m.spc = m.v + n;
  m.path = reinterpret_cast<int*>(m.spc + n); m.col4row = m.path + n; m.row4col = m.col4row + n;
  m.remaining = m.row4col + n;
  m.SR = reinterpret_cast<unsigned char*>(m.remaining + n); m.SC = m.SR + n;
  return m;
}

// ---- kernels -------------------------------------------------------------------------------------
// detection features -> L2-normalised copies (matching.py:125-130), one block per (det, stream)
__global__ void __launch_bounds__(128) normalize_kernel(Dev t, const int* __restrict__ det_count,
                                                        const int* __restrict__ crop_slot, int stride_k,
                                                        const float* __restrict__ feats, const int* __restrict__ present) {
  const int s = blockIdx.y, d = blockIdx.x;
  if (present && !present[s]) return;  // an absent stream's crop slots are not this step's
  if (d >= min(det_count[s], t.D)) return;
  const int row = crop_slot[static_cast<long long>(s) * stride_k + d];
  if (row < 0) return;
  __shared__ float red[128];
  const float* f = feats + static_cast<long long>(row) * t.F;
  float ss = 0.0f;
  for (int k = threadIdx.x; k < t.F; k += blockDim.x) { const float v = f[k]; ss += v * v; }
  red[threadIdx.x] = ss;
  __syncthreads();
  for (int o = 64; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  const float nrm = fmaxf(sqrtf(red[0]), 1e-7f);
  const long long ob = (static_cast<long long>(s) * t.D + d) * t.F;
  for (int k = threadIdx.x; k < t.F; k += blockDim.x) {
    const float v = f[k] / nrm;
    t.featn[ob + k] = v;
    if (t.featn_hi) {
      const float h = tf32_hi(v);
      t.featn_hi[ob + k] = h;
      t.featn_lo[ob + k] = v - h;
    }
  }
}

// K8: cost[slot][d] = min over the gallery of max(0, 1 - <g, f_d>)  (matching.py:109-217)
// detections per shared-memory tile of the row kernel.  The gallery is re-read (from L2) once per tile; frames with
// more than APP_GEMM_MIN detections take the SGEMM tiling below (crowded scenes, configs[4]: the row kernel measured
// 17 GB of DRAM reads against 1 GB of gallery and was shared-memory-load bound).  A 32-wide tile was measured slower
// on the usual ~17-detection frames (97 vs 70 us per 64 streams: three times the shared memory, a third of the blocks).
constexpr int APP_DT = 16;
constexpr int APP_GEMM_MIN = 48;
// dynamic shared memory of the row kernel: the detection tile and the per-warp minima.  aicam_tracker_create rejects a
// feature_dim for which this exceeds what a block can opt in to.
constexpr size_t appearance_rows_smem(int F) { return (static_cast<size_t>(APP_DT) * F + 8 * APP_DT) * sizeof(float); }
__device__ __forceinline__ void appearance_rows(const Dev& t, const int* __restrict__ det_count,
                                                const int* __restrict__ crop_slot, int stride_k, float* sm_f) {
  // sm_f: [APP_DT][F] detection tile, then [8][APP_DT] per-warp minima
  const int s = blockIdx.y, ti = blockIdx.x;
  if (ti >= t.n_tracks[s]) return;
  const int slot = t.order[static_cast<long long>(s) * t.T + ti];
  const long long ts = static_cast<long long>(s) * t.T + slot;
  if (t.state[ts] != CONFIRMED) return;  // only confirmed tracks enter the appearance cascade
  const int nd = min(det_count[s], t.D);
  const int ng = t.gal_count[ts];
  const float* gal = t.gallery + ts * t.G * t.F;
  float* out = t.app_cost + ts * t.D;
  float* tile = sm_f;
  float* wmin = sm_f + APP_DT * t.F;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int d0 = 0; d0 < nd; d0 += APP_DT) {
    const int dn = min(APP_DT, nd - d0);
    __syncthreads();
    for (int idx = threadIdx.x; idx < dn * t.F; idx += blockDim.x) {
      const int dd = idx / t.F, k = idx - dd * t.F;
      const bool has = crop_slot[static_cast<long long>(s) * stride_k + d0 + dd] >= 0;
      tile[idx] = has ? t.featn[(static_cast<long long>(s) * t.D + d0 + dd) * t.F + k] : 0.0f;
    }
    __syncthreads();
    float best = INFTY_COST;  // lane dd < dn tracks the minimum for detection d0 + dd
    for (int g = warp; g < ng; g += 8) {
      const float* grow = gal + static_cast<long long>(g) * t.F;
      float acc[APP_DT];
#pragma unroll
      for (int dd = 0; dd < APP_DT; ++dd) acc[dd] = 0.0f;
      for (int k = lane; k < t.F; k += 32) {
        const float gv = grow[k];
#pragma unroll
        for (int dd = 0; dd < APP_DT; ++dd) acc[dd] = fmaf(gv, tile[dd * t.F + k], acc[dd]);
      }
#pragma unroll
      for (int dd = 0; dd < APP_DT; ++dd) {
        float v = acc[dd];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == dd) best = fminf(best, fmaxf(1.0f - v, 0.0f));
      }
    }
    if (lane < APP_DT) wmin[warp * APP_DT + lane] = best;
    __syncthreads();
    if (threadIdx.x < dn) {
      float v = INFTY_COST;
      for (int w = 0; w < 8; ++w) v = fminf(v, wmin[w * APP_DT + threadIdx.x]);
      const bool has = crop_slot[static_cast<long long>(s) * stride_k + d0 + threadIdx.x] >= 0;
      out[d0 + threadIdx.x] = (has && ng > 0) ? v : INFTY_COST;
    }
  }
}

// K8 as a register-tiled SGEMM (feature dims that are multiples of 32): a block owns one track; its gallery (<= 128
// rows per pass) meets 64 detections at a time, K in chunks of 32 staged k-major in shared memory; every thread
// accumulates 8 gallery rows x 4 detections (32 FMAs per 12 shared-memory loads).  The gallery is read from DRAM
// once per track (the passes over further detection tiles hit L2) - the one-warp-per-row kernel above re-read it per
// tile and was shared-memory-load bound in crowded scenes (profiles/r1_crowded_scene_tracker.txt).
constexpr int AG_ROWS = 128, AG_DT = 64, AG_KC = 32;
__device__ __forceinline__ void appearance_gemm(const Dev& t, const int* __restrict__ det_count,
                                                const int* __restrict__ crop_slot, int stride_k, float* sm_f) {
  float (*Gs)[AG_ROWS + 4] = reinterpret_cast<float (*)[AG_ROWS + 4]>(sm_f);
  float (*Fs)[AG_DT + 4] = reinterpret_cast<float (*)[AG_DT + 4]>(sm_f + AG_KC * (AG_ROWS + 4));
  float (*wmin)[AG_DT] = reinterpret_cast<float (*)[AG_DT]>(sm_f + AG_KC * (AG_ROWS + 4) + AG_KC * (AG_DT + 4));
  const int s = blockIdx.y, ti = blockIdx.x;
  if (ti >= t.n_tracks[s]) return;
  const int slot = t.order[static_cast<long long>(s) * t.T + ti];
  const long long ts = static_cast<long long>(s) * t.T + slot;
  if (t.state[ts] != CONFIRMED) return;  // only confirmed tracks enter the appearance cascade
  const int nd = min(det_count[s], t.D);
  const int ng = t.gal_count[ts];
  const int F = t.F;
  const float* gal = t.gallery + ts * t.G * F;
  const float* fn = t.featn + static_cast<long long>(s) * t.D * F;
  const int* cs = crop_slot + static_cast<long long>(s) * stride_k;
  float* out = t.app_cost + ts * t.D;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  for (int d0 = 0; d0 < nd; d0 += AG_DT) {
    const int dn = min(AG_DT, nd - d0);
    float best[4] = {INFTY_COST, INFTY_COST, INFTY_COST, INFTY_COST};
    for (int r0 = 0; r0 < ng; r0 += AG_ROWS) {
      const int rn = min(AG_ROWS, ng - r0);
      float acc[8][4];
#pragma unroll
      for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[r][j] = 0.0f;
      for (int k0 = 0; k0 < F; k0 += AG_KC) {
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 4; ++i) {  // gallery chunk: 128 rows x 8 float4
          const int idx = tid + 256 * i, row = idx >> 3, kq = (idx & 7) * 4;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (row < rn) v = __ldg(reinterpret_cast<const float4*>(gal + static_cast<long long>(r0 + row) * F + k0 + kq));
          Gs[kq][row] = v.x; Gs[kq + 1][row] = v.y; Gs[kq + 2][row] = v.z; Gs[kq + 3][row] = v.w;
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {  // detection chunk: 64 detections x 8 float4 (no feature: zeros)
          const int idx = tid + 256 * i, dd = idx >> 3, kq = (idx & 7) * 4;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (dd < dn && cs[d0 + dd] >= 0) v = *reinterpret_cast<const float4*>(fn + static_cast<long long>(d0 + dd) * F + k0 + kq);
          Fs[kq][dd] = v.x; Fs[kq + 1][dd] = v.y; Fs[kq + 2][dd] = v.z; Fs[kq + 3][dd] = v.w;
        }
        __syncthreads();
#pragma unroll 4
        for (int k = 0; k < AG_KC; ++k) {
          float g[8], f[4];
#pragma unroll
          for (int r = 0; r < 8; ++r) g[r] = Gs[k][ty + 16 * r];
#pragma unroll
          for (int j = 0; j < 4; ++j) f[j] = Fs[k][tx + 16 * j];
#pragma unroll
          for (int r = 0; r < 8; ++r)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[r][j] = fmaf(g[r], f[j], acc[r][j]);
        }
      }
#pragma unroll
      for (int r = 0; r < 8; ++r)
        if (ty + 16 * r < rn) {
#pragma unroll
          for (int j = 0; j < 4; ++j) best[j] = fminf(best[j], fmaxf(1.0f - acc[r][j], 0.0f));
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) wmin[ty][tx + 16 * j] = best[j];
    __syncthreads();
    if (tid < dn) {
      float v = INFTY_COST;
#pragma unroll
      for (int w = 0; w < 16; ++w) v = fminf(v, wmin[w][tid]);
      out[d0 + tid] = (cs[d0 + tid] >= 0 && ng > 0) ? v : INFTY_COST;
    }
    __syncthreads();
  }
}

constexpr size_t AG_SMEM = (AG_KC * (AG_ROWS + 4) + AG_KC * (AG_DT + 4) + 16 * AG_DT) * sizeof(float);
// One launch, two tilings: frames with at most APP_GEMM_MIN detections take the row kernel (no padding work), busier
// frames the SGEMM tiling.  The choice is per block from the device-side count.
__global__ void __launch_bounds__(256) appearance_kernel(Dev t, const int* __restrict__ det_count,
                                                         const int* __restrict__ crop_slot, int stride_k, int gemm_ok,
                                                         const int* __restrict__ present) {
  extern __shared__ __align__(16) float sm_f[];
  if (present && !present[blockIdx.y]) return;  // absent stream: nothing of it is read or written
  const bool crowded = min(det_count[blockIdx.y], t.D) > APP_GEMM_MIN;
  if (crowded && gemm_ok == 2) return;  // appearance_tf32_kernel owns this stream's frame
  if (crowded && gemm_ok == 1) appearance_gemm(t, det_count, crop_slot, stride_k, sm_f);
  else appearance_rows(t, det_count, crop_slot, stride_k, sm_f);
}

struct StepIO {
  const float* boxes; const float* scores; const int* labels; int stride_k;
  const int* det_index; const int* det_count; const int* crop_slot;
  int* out_tracks; float* out_conf; int* out_count;
  int cm_in_smem;  // the T x D cost matrix fits in shared memory (else the per-stream global workspace)
  long long* trace;  // debug (AICAM_ASSOC_TRACE): clock64 stamps of stream 0's CTA, see aicam_tracker_destroy
  int has_feats;   // 0: the frame carries no features at all (feats == NULL): every appearance cost is INFTY_COST and
                   // nothing is appended to the galleries, as in the reference when every Detection.feature is None
  const int* present;  // [S] 0: the stream has no frame this step and its state is left as it is; null: all present
};

// one normalised detection feature (and its TF32 split copies) -> a gallery row, by one warp.  Feature rows are 16-byte
// aligned when F is a multiple of 4; all loads are issued before the first store (the compiler cannot hoist them itself:
// the pointers may alias), so a row costs one memory round trip instead of F / 32.
__device__ __forceinline__ void copy_feature_row(const Dev& t, long long go, long long so, int lane) {
  const int F = t.F;
  const int nsrc = t.gal_hi ? 3 : 1;
  for (int a = 0; a < nsrc; ++a) {
    const float* src = (a == 0 ? t.featn : a == 1 ? t.featn_hi : t.featn_lo) + so;
    float* dst = (a == 0 ? t.gallery : a == 1 ? t.gal_hi : t.gal_lo) + go;
    if (F % 128 == 0 && F <= 1024) {
      float4 v[8];
      const int n4 = F / 128;
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (i < n4) v[i] = reinterpret_cast<const float4*>(src)[lane + 32 * i];
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (i < n4) reinterpret_cast<float4*>(dst)[lane + 32 * i] = v[i];
    } else {
      for (int f = lane; f < F; f += 32) dst[f] = src[f];
    }
  }
}

// K7 + K9-K12: predict, cascade, IoU stage, update, initiate, prune, output.  One CTA per stream.
__global__ void __launch_bounds__(ASSOC_THREADS) assoc_kernel(Dev t, StepIO io) {
  extern __shared__ __align__(16) uint8_t smraw[];
  const int s = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int T = t.T, Dm = t.D;
  // shared-memory carve-up
  uint8_t* p = smraw;
  float* d_tlwh = reinterpret_cast<float*>(p); p += sizeof(float) * 4 * Dm;
  float* d_xyah = reinterpret_cast<float*>(p); p += sizeof(float) * 4 * Dm;
  int* U = reinterpret_cast<int*>(p); p += sizeof(int) * Dm;          // unmatched detections, ordered
  int* Utmp = reinterpret_cast<int*>(p); p += sizeof(int) * max(T, Dm);  // (also the costs of a one-column problem)
  int* conf_list = reinterpret_cast<int*>(p); p += sizeof(int) * T;   // order positions of confirmed tracks
  int* tent_list = reinterpret_cast<int*>(p); p += sizeof(int) * T;
  int* L = reinterpret_cast<int*>(p); p += sizeof(int) * T;           // rows of the current problem (order positions)
  int* match = reinterpret_cast<int*>(p); p += sizeof(int) * T;       // by order position: detection or -1
  int* cfr = reinterpret_cast<int*>(p); p += sizeof(int) * T;         // col_for_row of the current LSAP
  int* det_used = reinterpret_cast<int*>(p); p += sizeof(int) * Dm;
  // per-position copies of the track list and of the two fields every serial phase keeps asking for: the
  // single-thread loops below (lists, cascade levels, prune, output) then run on shared-memory latency
  int* ord = reinterpret_cast<int*>(p); p += sizeof(int) * T;        // order[k]: slot of the k-th track
  int* st_state = reinterpret_cast<int*>(p); p += sizeof(int) * T;
  int* st_tsu = reinterpret_cast<int*>(p); p += sizeof(int) * T;
  p = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(p) + 15) & ~static_cast<uintptr_t>(15));
  // predicted (x, y, a, h) and the four position variances per track-list position: all the gate and the IoU cost read
  float4* st_mean4 = reinterpret_cast<float4*>(p); p += sizeof(float4) * T;
  float4* st_cov4 = reinterpret_cast<float4*>(p); p += sizeof(float4) * T;
  int* fstack = reinterpret_cast<int*>(p); p += sizeof(int) * T;     // the stream's free-slot stack (written back at the end)
  int* gpos = reinterpret_cast<int*>(p); p += sizeof(int) * T;       // gallery row a matched track appends to, or -1
  p = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(p) + 15) & ~static_cast<uintptr_t>(15));
  const int nmax = max(T, Dm);
  LsapMem lm = lsap_carve(p, nmax);
  p += lsap_bytes(nmax);
  __shared__ int s_nconf, s_ntent, s_nU, s_nL, s_levels[8], s_nt, s_nfree1;

#define ASSOC_STAMP(i) do { if (io.trace && s == 0 && tid == 0) io.trace[i] = clock64(); } while (0)
  ASSOC_STAMP(0);
  // an absent stream: no predict, no aging, no state change at all - as if its reference process had not been called for
  // this frame; the whole CTA leaves before the first barrier
  if (io.present && !io.present[s]) {
    if (tid == 0) io.out_count[s] = 0;
    return;
  }
  const AssocRec cfg = t.assoc[s];  // the stream's settings of this step (register copies: the fewest spills, DESIGN §3.5)
  const long long sb = static_cast<long long>(s) * T;
  int nt = t.n_tracks[s];
  int nd = io.det_count[s];
  if (nd > Dm) { nd = Dm; if (tid == 0) atomicOr(&t.overflow[s], 2); }
  int* order = t.order + sb;
  const int nfree0 = t.n_free[s];
  for (int k = tid; k < nfree0; k += ASSOC_THREADS) fstack[k] = t.free_slots[sb + k];

  // -- K7 predict (tracker_core.py:44-49, track.py:76-80)
  for (int k = tid; k < nt; k += ASSOC_THREADS) {
    const int slot = order[k];
    const long long ts = sb + slot;
    float mean[8], cov[16];
    for (int i = 0; i < 8; ++i) mean[i] = t.mean[ts * 8 + i];
    for (int i = 0; i < 16; ++i) cov[i] = t.cov[ts * 16 + i];
    kf_predict(mean, cov);
    for (int i = 0; i < 8; ++i) t.mean[ts * 8 + i] = mean[i];
    for (int i = 0; i < 16; ++i) t.cov[ts * 16 + i] = cov[i];
    t.age[ts] += 1;
    const int tsu = t.tsu[ts] + 1;
    t.tsu[ts] = tsu;
    ord[k] = slot;
    st_mean4[k] = make_float4(mean[0], mean[1], mean[2], mean[3]);
    st_cov4[k] = make_float4(cov[0], cov[1], cov[2], cov[3]);
    st_tsu[k] = tsu;
    st_state[k] = t.state[ts];
    match[k] = -1;
  }
  // -- detections (deepsort_tracker.py:180-198, detection.py:15-47)
  for (int k = tid; k < nd; k += ASSOC_THREADS) {
    const long long o = static_cast<long long>(s) * io.stride_k + io.det_index[static_cast<long long>(s) * io.stride_k + k];
    const float4 b = reinterpret_cast<const float4*>(io.boxes)[o];
    float tl[4] = {b.x, b.y, b.z - b.x, b.w - b.y}, z[4];
    tlwh_to_xyah(tl, z);
    for (int i = 0; i < 4; ++i) { d_tlwh[4 * k + i] = tl[i]; d_xyah[4 * k + i] = z[i]; }
    U[k] = k;
    det_used[k] = 0;
  }
  __syncthreads();
  // -- confirmed / tentative lists in track-list order (tracker_core.py:112-117): ballot compaction by warp 0
  if (warp == 0) {
    int nc = 0, nn = 0;
    unsigned lv_bits[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int b0 = 0; b0 < nt; b0 += 32) {
      const int k = b0 + lane;
      const int st = k < nt ? st_state[k] : 0;
      const unsigned bc = __ballot_sync(0xffffffffu, st == CONFIRMED), bt = __ballot_sync(0xffffffffu, st == TENTATIVE);
      const unsigned below = (1u << lane) - 1u;
      if (st == CONFIRMED) {
        conf_list[nc + __popc(bc & below)] = k;
        const int lv = st_tsu[k];
        if (lv >= 1 && lv <= cfg.max_age && lv < 256) lv_bits[lv >> 5] |= 1u << (lv & 31);
      } else if (st == TENTATIVE) {
        tent_list[nn + __popc(bt & below)] = k;
      }
      nc += __popc(bc); nn += __popc(bt);
    }
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      const unsigned all = __reduce_or_sync(0xffffffffu, lv_bits[w]);
      if (lane == 0) s_levels[w] = all;
    }
    if (lane == 0) { s_nconf = nc; s_ntent = nn; s_nU = nd; }
  }
  __syncthreads();
  ASSOC_STAMP(1);

  float* cm = io.cm_in_smem ? reinterpret_cast<float*>(p) : t.cost_ws + static_cast<long long>(s) * T * Dm;
  const int nconf = s_nconf;
  // gated appearance cost of one (track position, detection) pair (linear_assignment.py:160-212: the squared Mahalanobis
  // distance gates with a strict >; n_meas selects the reference's BLAS path, see kf_gating), thresholded (:58)
  auto gated_cost = [&](int pos, int d, int n_meas) {
    float c = io.has_feats ? t.app_cost[(sb + ord[pos]) * Dm + d] : INFTY_COST;
    const float4 m4 = st_mean4[pos], c4 = st_cov4[pos];
    const float mean4[4] = {m4.x, m4.y, m4.z, m4.w}, cov4[4] = {c4.x, c4.y, c4.z, c4.w};
    if (kf_gating(mean4, cov4, d_xyah + 4 * d, n_meas) > CHI2_GATE) c = INFTY_COST;
    return c > cfg.thr_cos ? cfg.clamp_cos : c;
  };
  // unmatched detections keep their order (linear_assignment.py:64-88): in-place compaction of U by warp 0
  auto compact_U = [&](int nU) {
    int n = 0;
    for (int b0 = 0; b0 < nU; b0 += 32) {
      const int j = b0 + lane;
      const int d = j < nU ? U[j] : 0;
      const bool keep = j < nU && !det_used[d];
      const unsigned bal = __ballot_sync(0xffffffffu, keep);
      __syncwarp();
      if (keep) U[n + __popc(bal & ((1u << lane) - 1u))] = d;
      n += __popc(bal);
    }
    __syncwarp();
    if (lane == 0) s_nU = n;
  };
  // -- stage 1: matching cascade over confirmed tracks (linear_assignment.py:91-157).  The cost of every (confirmed
  //    track, detection) pair is computed ONCE, by track-list position; a level's problem is the sub-matrix (rows L,
  //    columns U) read in place through the two index lists.  Levels that hold no track are skipped through the bitmap.
  //    Frames whose problems all fit one warp run the whole cascade on warp 0 without a block barrier.
  for (int idx = tid; idx < nconf * nd; idx += ASSOC_THREADS) {
    const int i = idx / nd, d = idx - i * nd;
    const int pos = conf_list[i];
    cm[pos * nd + d] = gated_cost(pos, d, 2);
  }
  __syncthreads();
  {
    const bool small = max(nconf, nd) <= LSAP_WIDE;
    const int cth = small ? 32 : ASSOC_THREADS;
    auto csync = [&]() { if (small) __syncwarp(); else __syncthreads(); };
    float* colv = reinterpret_cast<float*>(Utmp);  // (a one-column problem's costs: nL <= T floats, see the carve-up)
    if (!small || warp == 0) {
      int level = 0, nU = nd;
      for (;;) {
        for (++level; level <= cfg.max_age; ) {  // next level that holds a confirmed track
          const unsigned wbits = s_levels[level >> 5] >> (level & 31);
          if (wbits) { level += __ffs(wbits) - 1; break; }
          level = (level | 31) + 1;
        }
        if (level > cfg.max_age || nU == 0) break;
        if (warp == 0) {  // L = the level's tracks in track-list order
          int n = 0;
          for (int b0 = 0; b0 < nconf; b0 += 32) {
            const int k = b0 + lane;
            const int pos = k < nconf ? conf_list[k] : 0;
            const bool keep = k < nconf && st_tsu[pos] == level;
            const unsigned bal = __ballot_sync(0xffffffffu, keep);
            if (keep) L[n + __popc(bal & ((1u << lane) - 1u))] = pos;
            n += __popc(bal);
          }
          if (lane == 0) s_nL = n;
        }
        csync();
        const int nL = s_nL;
        const bool one_col = nU == 1;  // the gate's n_meas == 1 form: computed here
        if (one_col) {
          for (int i = tid; i < nL; i += cth) colv[i] = gated_cost(L[i], U[0], 1);
          csync();
        }
        const int nw = small ? 1 : lsap_warps(nL, nU);
        const long long c0 = (io.trace && s == 0 && tid == 0) ? clock64() : 0;
        if (warp < nw) {
          if (one_col) lsap_cta(colv, 1, nL, 1, lm, cfr, tid, nw);
          else lsap_cta(cm, nd, nL, nU, lm, cfr, tid, nw, L, U);
        }
        csync();
        if (io.trace && s == 0 && tid == 0) { io.trace[10] += clock64() - c0; io.trace[11] += 1; io.trace[12] += static_cast<long long>(nL) * 1024 + nU; }
        for (int i = tid; i < nL; i += cth) {  // keep pairs with cost <= max_distance
          const int j = cfr[i];
          if (j < 0) continue;
          const float c = one_col ? colv[i] : cm[L[i] * nd + U[j]];
          if (c <= cfg.thr_cos) { match[L[i]] = U[j]; det_used[U[j]] = 1; }
        }
        csync();
        if (warp == 0) compact_U(nU);
        csync();
        nU = s_nU;
      }
    }
  }
  __syncthreads();
  ASSOC_STAMP(2);
  // -- stage 2: IoU matching (tracker_core.py:138-166)
  if (tid == 0) {
    int n = 0;
    for (int k = 0; k < s_ntent; ++k) L[n++] = tent_list[k];
    for (int k = 0; k < nconf; ++k) {
      const int pos = conf_list[k];
      if (match[pos] < 0 && st_tsu[pos] == 1) L[n++] = pos;
    }
    s_nL = n;
  }
  __syncthreads();
  if (s_nL > 0 && s_nU > 0) {
    const int nL = s_nL, nU = s_nU;
    for (int idx = tid; idx < nL * nU; idx += ASSOC_THREADS) {
      const int i = idx / nU, j = idx - i * nU;
      const float4 m4 = st_mean4[L[i]];
      const float mean4[4] = {m4.x, m4.y, m4.z, m4.w};
      float tl[4];
      mean_to_tlwh(mean4, tl);
      const float c = iou_cost(tl, d_tlwh + 4 * U[j]);
      cm[idx] = c > cfg.thr_iou ? cfg.clamp_iou : c;  // linear_assignment.py:58
    }
    __syncthreads();
    const int nw = lsap_warps(nL, nU);
    const long long c0 = (io.trace && s == 0 && tid == 0) ? clock64() : 0;
    if (warp < nw) lsap_cta(cm, nU, nL, nU, lm, cfr, tid, nw);
    __syncthreads();
    if (io.trace && s == 0 && tid == 0) { io.trace[10] += clock64() - c0; io.trace[11] += 1; io.trace[12] += static_cast<long long>(nL) * 1024 + nU; }
    for (int i = tid; i < nL; i += ASSOC_THREADS) {
      const int j = cfr[i];
      if (j >= 0 && cm[i * nU + j] <= cfg.thr_iou) { match[L[i]] = U[j]; det_used[U[j]] = 1; }
    }
    __syncthreads();
    if (warp == 0) compact_U(nU);
    __syncthreads();
  }
  ASSOC_STAMP(3);

  // -- update matched tracks / mark missed (tracker_core.py:62-68, track.py:82-119): the Kalman update and the scalar
  //    fields one thread per track, then the gallery rows one warp per matched track
  for (int k = tid; k < nt; k += ASSOC_THREADS) {
    const long long ts = sb + ord[k];
    const int d = match[k];
    if (d >= 0) {
      float mean[8], cov[16];
      for (int i = 0; i < 8; ++i) mean[i] = t.mean[ts * 8 + i];
      for (int i = 0; i < 16; ++i) cov[i] = t.cov[ts * 16 + i];
      kf_update(mean, cov, d_xyah + 4 * d);
      for (int i = 0; i < 8; ++i) t.mean[ts * 8 + i] = mean[i];
      for (int i = 0; i < 16; ++i) t.cov[ts * 16 + i] = cov[i];
      const long long o = static_cast<long long>(s) * io.stride_k + io.det_index[static_cast<long long>(s) * io.stride_k + d];
      const int hits = t.hits[ts] + 1;
      t.hits[ts] = hits;
      t.tsu[ts] = 0;
      st_tsu[k] = 0;
      t.conf[ts] = io.scores[o];
      t.cls[ts] = io.labels[o];
      if (st_state[k] == TENTATIVE && hits >= t.trk_n_init[ts]) { t.state[ts] = CONFIRMED; st_state[k] = CONFIRMED; }
      // track.py:70-74: the feature is appended to the gallery, FIFO at the budget (rows copied below, one warp each)
      int gp = -1;
      if (io.has_feats && io.crop_slot[static_cast<long long>(s) * io.stride_k + d] >= 0) {
        const int cnt = t.gal_count[ts], head = t.gal_head[ts];
        gp = cnt < t.G ? (head + cnt) % t.G : head;
        if (cnt < t.G) t.gal_count[ts] = cnt + 1; else t.gal_head[ts] = (head + 1) % t.G;
      }
      gpos[k] = gp;
    } else if (st_state[k] == TENTATIVE || (st_state[k] == CONFIRMED && st_tsu[k] > t.trk_max_age[ts])) {
      t.state[ts] = DELETED;
      st_state[k] = DELETED;
    }
  }
  __syncthreads();
  if (io.has_feats) {
    for (int k = warp; k < nt; k += ASSOC_THREADS / 32) {
      const int d = match[k];
      if (d < 0 || gpos[k] < 0) continue;
      copy_feature_row(t, ((sb + ord[k]) * t.G + gpos[k]) * t.F, (static_cast<long long>(s) * Dm + d) * t.F, lane);
    }
  }
  __syncthreads();
  ASSOC_STAMP(4);
  // -- prune deleted tracks, then initiate one track per unmatched detection in ascending order
  //    (tracker_core.py:70-75, :180-194; ids come from the stream's own counter)
  if (tid == 0) {
    int n = 0;
    int nfree = nfree0;
    for (int k = 0; k < nt; ++k) {
      const int slot = ord[k];
      if (st_state[k] == DELETED) {
        fstack[nfree++] = slot;
      } else {  // compaction in place (n <= k)
        if (n != k) { order[n] = slot; ord[n] = slot; st_state[n] = st_state[k]; st_tsu[n] = st_tsu[k]; }
        ++n;
      }
    }
    const int nU = s_nU;
    int created = 0;
    int next_id = t.next_id[s];
    for (int j = 0; j < nU; ++j) {
      if (nfree == 0) { atomicOr(&t.overflow[s], 1); break; }
      const int slot = fstack[--nfree];
      order[n] = slot; ord[n] = slot; st_state[n] = TENTATIVE; st_tsu[n] = 0;
      ++n;
      Utmp[created++] = slot;
      const long long ts = sb + slot;
      t.track_id[ts] = next_id++;
      t.state[ts] = TENTATIVE;
      t.hits[ts] = 1; t.age[ts] = 1; t.tsu[ts] = 0;
      t.gal_count[ts] = 0; t.gal_head[ts] = 0;
      t.trk_n_init[ts] = cfg.n_init; t.trk_max_age[ts] = cfg.max_age;
    }
    t.next_id[s] = next_id;
    t.n_free[s] = nfree;
    t.n_tracks[s] = n;
    s_nt = n;
    s_nL = created;
    s_nfree1 = nfree;
  }
  __syncthreads();
  // (the stack was worked on in shared memory: write every live entry back, at most T ints)
  for (int k = tid; k < s_nfree1; k += ASSOC_THREADS) t.free_slots[sb + k] = fstack[k];
  for (int j = warp; j < s_nL; j += ASSOC_THREADS / 32) {
    const int d = U[j];
    const long long ts = sb + Utmp[j];
    const int row = io.has_feats ? io.crop_slot[static_cast<long long>(s) * io.stride_k + d] : -1;
    if (row >= 0) {
      copy_feature_row(t, ts * t.G * t.F, (static_cast<long long>(s) * Dm + d) * t.F, lane);
      if (lane == 0) t.gal_count[ts] = 1;
    }
    if (lane == 0) {
      float mean[8], cov[16];
      kf_initiate(d_xyah + 4 * d, mean, cov);
      for (int i = 0; i < 8; ++i) t.mean[ts * 8 + i] = mean[i];
      for (int i = 0; i < 16; ++i) t.cov[ts * 16 + i] = cov[i];
      const long long o = static_cast<long long>(s) * io.stride_k + io.det_index[static_cast<long long>(s) * io.stride_k + d];
      t.conf[ts] = io.scores[o];
      t.cls[ts] = io.labels[o];
    }
  }
  __syncthreads();
  ASSOC_STAMP(5);
  // -- output (deepsort_tracker.py:125-141): confirmed and updated this frame, track-list order
  if (tid == 0) {  // which positions are reported (shared memory only) ...
    int n = 0;
    const int ntn = s_nt;
    for (int k = 0; k < ntn; ++k)
      if (st_state[k] == CONFIRMED && st_tsu[k] == 0) L[n++] = k;
    s_nL = n;
    io.out_count[s] = n;
  }
  __syncthreads();
  for (int n = tid; n < s_nL; n += ASSOC_THREADS) {  // ... and their rows, one thread each
    const int slot = ord[L[n]];
    const long long ts = sb + slot;
    float tl[4];
    mean_to_tlwh(t.mean + ts * 8, tl);
    const float w = tl[2] > 0.0f ? tl[2] : 0.0f, h = tl[3] > 0.0f ? tl[3] : 0.0f;
    int* o = io.out_tracks + (sb + n) * 6;
    o[0] = __float2int_rn(tl[0]);
    o[1] = __float2int_rn(tl[1]);
    o[2] = __float2int_rn(tl[0] + w);
    o[3] = __float2int_rn(tl[1] + h);
    o[4] = t.track_id[ts];
    o[5] = t.cls[ts];
    io.out_conf[sb + n] = t.conf[ts];
    t.row_slot[sb + n] = slot;
  }
  __syncthreads();
  ASSOC_STAMP(6);
  if (io.trace && s == 0 && tid == 0) { io.trace[8] = nt; io.trace[9] = nd; }
#undef ASSOC_STAMP
}

// mask: device i32[S], streams with a zero entry are left as they are; null resets every stream
__global__ void reset_kernel(Dev t, const int* __restrict__ mask) {
  const int s = blockIdx.x;
  if (mask && !mask[s]) return;
  const long long sb = static_cast<long long>(s) * t.T;
  for (int k = threadIdx.x; k < t.T; k += blockDim.x) {
    t.free_slots[sb + k] = t.T - 1 - k;  // slot 0 is popped first
    t.state[sb + k] = DELETED;
    t.gal_count[sb + k] = 0;
    t.gal_head[sb + k] = 0;
  }
  if (threadIdx.x == 0) { t.n_tracks[s] = 0; t.n_free[s] = t.T; t.next_id[s] = 1; t.overflow[s] = 0; }
}

__global__ void lsap_kernel(const float* cost, int nr, int nc, int* col_for_row) {
  extern __shared__ __align__(16) uint8_t smraw[];
  LsapMem m = lsap_carve(smraw, max(nr, nc));
  int* cfr = reinterpret_cast<int*>(smraw + lsap_bytes(max(nr, nc)));
  const int nw = lsap_warps(nr, nc);
  if (static_cast<int>(threadIdx.x) < 32 * nw) lsap_cta(cost + static_cast<long long>(blockIdx.x) * nr * nc, nc, nr, nc, m, cfr, threadIdx.x, nw);
  __syncthreads();
  for (int r = threadIdx.x; r < nr; r += blockDim.x) col_for_row[static_cast<long long>(blockIdx.x) * nr + r] = cfr[r];
}

__global__ void gating_kernel(const float* state, const float* meas, int n, int m, float* d2) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * m) return;
  const int i = idx / m;
  d2[idx] = kf_gating(state + static_cast<long long>(i) * 24, state + static_cast<long long>(i) * 24 + 8,
                      meas + static_cast<long long>(idx) * 4, m);
}

// Parity probe of K8 / K9 (no tracker state is changed): for every live track of every stream, in track-list order,
// the raw appearance cost (appearance_kernel's output: min over the gallery of the clamped cosine distance,
// INFTY_COST for tentative tracks / missing features) and the squared Mahalanobis distance of every filtered
// detection to the track's PREDICTED state (kf_predict applied to a copy) - what linear_assignment.py:160-212 gates
// with.  One block per (track position, stream).
__global__ void __launch_bounds__(128) cost_probe_kernel(Dev t, const float* __restrict__ boxes, int stride_k,
                                                         const int* __restrict__ det_index, const int* __restrict__ det_count,
                                                         float* __restrict__ app_cost, float* __restrict__ gate_d2,
                                                         int* __restrict__ track_ids, int* __restrict__ n_tracks) {
  const int s = blockIdx.y, k = blockIdx.x;
  const int nt = t.n_tracks[s];
  if (k == 0 && threadIdx.x == 0) n_tracks[s] = nt;
  if (k >= nt) return;
  const long long sb = static_cast<long long>(s) * t.T;
  const long long ts = sb + t.order[sb + k];
  float mean[8], cov[16];
  for (int i = 0; i < 8; ++i) mean[i] = t.mean[ts * 8 + i];
  for (int i = 0; i < 16; ++i) cov[i] = t.cov[ts * 16 + i];
  kf_predict(mean, cov);
  const int nd = min(det_count[s], t.D);
  const bool confirmed = t.state[ts] == CONFIRMED;
  if (threadIdx.x == 0) track_ids[sb + k] = t.track_id[ts];
  for (int d = threadIdx.x; d < nd; d += blockDim.x) {
    const long long o = static_cast<long long>(s) * stride_k + det_index[static_cast<long long>(s) * stride_k + d];
    const float4 b = reinterpret_cast<const float4*>(boxes)[o];
    float tl[4] = {b.x, b.y, b.z - b.x, b.w - b.y}, z[4];
    tlwh_to_xyah(tl, z);
    app_cost[(sb + k) * t.D + d] = confirmed ? t.app_cost[ts * t.D + d] : INFTY_COST;
    gate_d2[(sb + k) * t.D + d] = kf_gating(mean, cov, z, nd);
  }
}

constexpr size_t CM_SMEM_LIMIT = 96 * 1024;  // cost matrices up to this size live in shared memory
size_t assoc_smem(int T, int D, int* cm_in_smem = nullptr) {
  const size_t base = sizeof(float) * 8 * D + sizeof(int) * (2 * D + std::max(T, D) + 10 * T) + 32 + 32 * static_cast<size_t>(T) + lsap_bytes(std::max(T, D));
  const size_t cm = sizeof(float) * T * D;
  const bool fits = cm <= CM_SMEM_LIMIT;
  if (cm_in_smem) *cm_in_smem = fits ? 1 : 0;
  return base + (fits ? cm : 0);
}

}  // namespace
}  // namespace aicam

struct aicam_tracker {
  aicam::Dev d;
  aicam_tracker_config cfg;
  std::vector<aicam::AssocRec> assoc;  // host copy of d.assoc
  aicam::AssocRec* assoc_dev = nullptr;
  aicam::PinnedStaging staging;        // of aicam_tracker_set_stream_assoc
  std::vector<void*> allocs;
  aicam::AppearanceTf32* tf = nullptr;  // tensor-core appearance path (frames with more than APP_GEMM_MIN detections)
  long long* trace = nullptr;           // AICAM_ASSOC_TRACE: 16 clock64 slots, printed by aicam_tracker_destroy
};

using namespace aicam;

namespace {
template <typename Tp>
int dev_alloc(aicam_tracker* t, Tp** p, size_t n) {
  void* q = nullptr;
  if (cudaMalloc(&q, n * sizeof(Tp)) != cudaSuccess) return fail(AICAM_ERR_CUDA, "tracker_create: cudaMalloc failed");
  cudaMemset(q, 0, n * sizeof(Tp));
  t->allocs.push_back(q);
  *p = static_cast<Tp*>(q);
  return AICAM_OK;
}

// the host copy of the stream table to the device: one copy from pinned staging
int upload_assoc(aicam_tracker* t, cudaStream_t st) {
  uint8_t* h = nullptr;
  AICAM_CUDA_OK(t->staging.acquire(&h));
  const size_t bytes = t->assoc.size() * sizeof(AssocRec);
  std::memcpy(h, t->assoc.data(), bytes);
  AICAM_CUDA_OK(t->staging.upload(t->assoc_dev, bytes, st));
  return AICAM_OK;
}

int check_assoc(const aicam_stream_assoc& a, const std::string& at) {
  if (a.max_age < 1 || a.max_age > 255 || a.n_init < 1)
    return fail(AICAM_ERR_INVALID_ARG, at + "max_age must be in 1..255 and n_init >= 1");
  if (!std::isfinite(a.max_cosine_distance) || !std::isfinite(a.max_iou_distance) || a.max_cosine_distance < 0 ||
      a.max_iou_distance < 0)
    return fail(AICAM_ERR_INVALID_ARG, at + "distances must be finite and non-negative");
  return AICAM_OK;
}
}  // namespace

namespace {
// K8: L2-normalise the frame's detection features, then the appearance cost of every confirmed track
int launch_appearance(const Dev& d, const AppearanceTf32* tf, const int32_t* det_count, const int32_t* crop_slot, int stride_k,
                      const float* feats, const int32_t* present, cudaStream_t st) {
  normalize_kernel<<<dim3(d.D, d.S), 128, 0, st>>>(d, det_count, crop_slot, stride_k, feats, present);
  count_launch();
  if (int rc = last_launch("normalize_kernel")) return rc;
  // 0: row kernel for every frame; 1: fp32 FFMA tiling for crowded frames; 2: crowded frames are left to the
  // tensor-core kernel launched below (their blocks return at once here)
  const int gemm_ok = tf ? 2 : (d.F % AG_KC == 0 ? 1 : 0);
  const size_t sm = std::max(appearance_rows_smem(d.F), gemm_ok == 1 ? AG_SMEM : size_t(0));
  if (int rc = ensure_dynamic_smem(appearance_kernel, sm)) return rc;
  appearance_kernel<<<dim3(d.T, d.S), 256, sm, st>>>(d, det_count, crop_slot, stride_k, gemm_ok, present);
  count_launch();
  if (int rc = last_launch("appearance_kernel")) return rc;
  if (tf)
    return launch_appearance_tf32(tf, d.S, d.T, d.D, d.F, d.G, APP_GEMM_MIN, d.n_tracks, d.order, d.state, d.gal_count, det_count,
                                  crop_slot, stride_k, present, d.app_cost, st);
  return AICAM_OK;
}
}  // namespace

extern "C" {

int aicam_tracker_create(const aicam_tracker_config* cfg, aicam_tracker** out) {
  if (!cfg || !out) return fail(AICAM_ERR_INVALID_ARG, "tracker_create: null argument");
  *out = nullptr;
  if (cfg->n_streams <= 0 || cfg->max_tracks <= 0 || cfg->max_dets <= 0 || cfg->feature_dim <= 0)
    return fail(AICAM_ERR_INVALID_ARG, "tracker_create: sizes must be positive");
  if (cfg->max_tracks > 1024 || cfg->max_dets > 1024)
    return fail(AICAM_ERR_CAPACITY, "tracker_create: max_tracks and max_dets are limited to 1024");
  if (cfg->nn_budget <= 0)
    return fail(AICAM_ERR_UNSUPPORTED, "tracker_create: nn_budget must be positive (unbounded galleries unsupported)");
  if (cfg->max_age < 1 || cfg->max_age > 255 || cfg->n_init < 1)
    return fail(AICAM_ERR_INVALID_ARG, "tracker_create: max_age must be in 1..255 and n_init >= 1");
  AICAM_CUDA_OK(cudaSetDevice(cfg->device));
  int smem_optin = 0;
  AICAM_CUDA_OK(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, cfg->device));
  if (appearance_rows_smem(cfg->feature_dim) > static_cast<size_t>(smem_optin))
    return fail(AICAM_ERR_CAPACITY, "tracker_create: feature_dim " + std::to_string(cfg->feature_dim) + " needs " +
                                        std::to_string(appearance_rows_smem(cfg->feature_dim)) +
                                        " bytes of shared memory in the appearance kernel, more than the " +
                                        std::to_string(smem_optin) + " a block can use");
  aicam_tracker* t = new aicam_tracker();
  t->cfg = *cfg;
  Dev& d = t->d;
  d.S = cfg->n_streams; d.T = cfg->max_tracks; d.D = cfg->max_dets; d.F = cfg->feature_dim; d.G = cfg->nn_budget;
  t->assoc.assign(d.S, resolve_assoc(aicam_stream_assoc{cfg->max_cosine_distance, cfg->max_iou_distance, cfg->max_age,
                                                         cfg->n_init}));
  const size_t ST = static_cast<size_t>(d.S) * d.T;
  int rc = 0;
  rc |= dev_alloc(t, &d.mean, ST * 8);  rc |= dev_alloc(t, &d.cov, ST * 16);
  rc |= dev_alloc(t, &d.track_id, ST);  rc |= dev_alloc(t, &d.state, ST);  rc |= dev_alloc(t, &d.hits, ST);
  rc |= dev_alloc(t, &d.age, ST);       rc |= dev_alloc(t, &d.tsu, ST);    rc |= dev_alloc(t, &d.cls, ST);
  rc |= dev_alloc(t, &d.conf, ST);      rc |= dev_alloc(t, &d.gal_count, ST); rc |= dev_alloc(t, &d.gal_head, ST);
  rc |= dev_alloc(t, &d.gallery, ST * d.G * d.F);
  rc |= dev_alloc(t, &d.order, ST);     rc |= dev_alloc(t, &d.free_slots, ST);
  rc |= dev_alloc(t, &d.n_tracks, d.S); rc |= dev_alloc(t, &d.n_free, d.S); rc |= dev_alloc(t, &d.next_id, d.S);
  rc |= dev_alloc(t, &d.overflow, d.S);     rc |= dev_alloc(t, &d.row_slot, ST);
  rc |= dev_alloc(t, &t->assoc_dev, d.S); d.assoc = t->assoc_dev;
  rc |= dev_alloc(t, &d.trk_n_init, ST); rc |= dev_alloc(t, &d.trk_max_age, ST);
  if (t->staging.create(d.S * sizeof(AssocRec)) != cudaSuccess) rc |= 1;
  rc |= dev_alloc(t, &d.app_cost, ST * d.D); rc |= dev_alloc(t, &d.cost_ws, ST * d.D);
  rc |= dev_alloc(t, &d.featn, static_cast<size_t>(d.S) * d.D * d.F);
  d.gal_hi = d.gal_lo = d.featn_hi = d.featn_lo = nullptr;
  static const bool no_tf32 = getenv("AICAM_APPEARANCE_NO_TF32") != nullptr;
  // frames can only be crowded when the detection capacity allows it: the split copies cost 2 x the gallery memory
  const bool want_tf = !no_tf32 && d.D > APP_GEMM_MIN && appearance_tf32_eligible(d.S, d.F, d.G, d.D);
  if (want_tf) {
    rc |= dev_alloc(t, &d.gal_hi, ST * d.G * d.F + static_cast<size_t>(128) * d.F);  // (+ slack: the last tile's masked rows)
    rc |= dev_alloc(t, &d.gal_lo, ST * d.G * d.F + static_cast<size_t>(128) * d.F);
    rc |= dev_alloc(t, &d.featn_hi, static_cast<size_t>(d.S) * d.D * d.F);
    rc |= dev_alloc(t, &d.featn_lo, static_cast<size_t>(d.S) * d.D * d.F);
  }
  if (rc) { aicam_tracker_destroy(t); return AICAM_ERR_CUDA; }
  if (want_tf) {
    if (int r3 = appearance_tf32_create(&t->tf, d.S, d.T, d.D, d.F, d.G, d.gal_hi, d.gal_lo, d.featn_hi, d.featn_lo)) {
      aicam_tracker_destroy(t);
      return r3;
    }
  }
  const size_t sm = assoc_smem(d.T, d.D);
  if (sm > 200 * 1024) { aicam_tracker_destroy(t); return fail(AICAM_ERR_CAPACITY, "tracker_create: max_tracks/max_dets need too much shared memory"); }
  // (the > 48 KB opt-ins are made per launch in aicam_tracker_step: a running maximum per device, so that trackers of
  //  different sizes - or on different GPUs - never lower each other's limit)
  if (getenv("AICAM_ASSOC_TRACE")) { if (dev_alloc(t, &t->trace, 16)) { aicam_tracker_destroy(t); return AICAM_ERR_CUDA; } }
  if (int r2 = aicam_tracker_reset(t, nullptr)) { aicam_tracker_destroy(t); return r2; }
  if (int r2 = upload_assoc(t, nullptr)) { aicam_tracker_destroy(t); return r2; }
  AICAM_CUDA_OK(cudaDeviceSynchronize());
  *out = t;
  return AICAM_OK;
}

void aicam_tracker_destroy(aicam_tracker* t) {
  if (!t) return;
  cudaSetDevice(t->cfg.device);
  if (t->trace) {  // phase durations (cycles) of stream 0's CTA in the last step
    long long h[16];
    cudaDeviceSynchronize();
    if (cudaMemcpy(h, t->trace, sizeof(h), cudaMemcpyDeviceToHost) == cudaSuccess)
      fprintf(stderr, "assoc trace (stream 0, last step; cycles): predict+lists %lld cascade %lld iou %lld update %lld prune+initiate %lld "
              "output %lld total %lld | tracks %lld dets %lld | lsap: %lld cycles in %lld solves (sum rows*1024+cols %lld)\n",
              h[1] - h[0], h[2] - h[1], h[3] - h[2], h[4] - h[3], h[5] - h[4], h[6] - h[5], h[6] - h[0], h[8], h[9], h[10], h[11], h[12]);
  }
  t->staging.destroy();
  for (void* p : t->allocs) cudaFree(p);
  if (t->tf) appearance_tf32_destroy(t->tf);
  delete t;
}

int aicam_tracker_reset(aicam_tracker* t, void* stream) {
  if (!t) return fail(AICAM_ERR_INVALID_ARG, "tracker_reset: null handle");
  reset_kernel<<<t->d.S, 128, 0, static_cast<cudaStream_t>(stream)>>>(t->d, nullptr);
  count_launch();
  return last_launch("reset_kernel");
}

int aicam_tracker_reset_streams(aicam_tracker* t, const int32_t* mask, void* stream) {
  if (!t || !mask) return fail(AICAM_ERR_INVALID_ARG, "tracker_reset_streams: null argument");
  reset_kernel<<<t->d.S, 128, 0, static_cast<cudaStream_t>(stream)>>>(t->d, mask);
  count_launch();
  return last_launch("reset_kernel (masked)");
}

int aicam_tracker_set_stream_assoc(aicam_tracker* t, const int32_t* indices_host, const aicam_stream_assoc* host, int n,
                                   void* stream) {
  if (!t || n < 0 || (n > 0 && (!indices_host || !host)))
    return fail(AICAM_ERR_INVALID_ARG, "tracker_set_stream_assoc: null argument or negative count");
  std::vector<AssocRec> next = t->assoc;  // validated as a whole before anything is stored or copied
  for (int i = 0; i < n; ++i) {
    const std::string at = "tracker_set_stream_assoc: entry " + std::to_string(i) + ": ";
    if (indices_host[i] < 0 || indices_host[i] >= t->d.S) return fail(AICAM_ERR_INVALID_ARG, at + "stream index out of range");
    if (int rc = check_assoc(host[i], at)) return rc;
    next[indices_host[i]] = resolve_assoc(host[i]);
  }
  if (n == 0) return AICAM_OK;
  AICAM_CUDA_OK(cudaSetDevice(t->cfg.device));
  t->assoc.swap(next);
  return upload_assoc(t, static_cast<cudaStream_t>(stream));
}

int aicam_tracker_step(aicam_tracker* t, const float* boxes, const float* scores, const int32_t* labels, int stride_k,
                       const int32_t* det_index, const int32_t* det_count, const int32_t* crop_slot, const float* feats,
                       int32_t* out_tracks, float* out_conf, int32_t* out_count, void* stream) {
  return aicam_tracker_step_present(t, boxes, scores, labels, stride_k, det_index, det_count, crop_slot, feats, nullptr, out_tracks,
                                    out_conf, out_count, stream);
}

int aicam_tracker_step_present(aicam_tracker* t, const float* boxes, const float* scores, const int32_t* labels, int stride_k,
                               const int32_t* det_index, const int32_t* det_count, const int32_t* crop_slot, const float* feats,
                               const int32_t* present, int32_t* out_tracks, float* out_conf, int32_t* out_count, void* stream) {
  if (!t || !boxes || !scores || !labels || !det_index || !det_count || !crop_slot || !out_tracks || !out_conf || !out_count)
    return fail(AICAM_ERR_INVALID_ARG, "tracker_step: null argument");
  if (stride_k <= 0) return fail(AICAM_ERR_INVALID_ARG, "tracker_step: stride_k must be positive");
  if (reinterpret_cast<uintptr_t>(boxes) % 16) return fail(AICAM_ERR_INVALID_ARG, "tracker_step: boxes must be 16-byte aligned");
  const Dev& d = t->d;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (feats) {
    if (int rc = launch_appearance(d, t->tf, det_count, crop_slot, stride_k, feats, present, st)) return rc;
  }
  StepIO io{boxes, scores, labels, stride_k, det_index, det_count, crop_slot, out_tracks, out_conf, out_count, 0, t->trace, feats ? 1 : 0,
            present};
  if (t->trace) cudaMemsetAsync(t->trace, 0, sizeof(long long) * 16, st);
  const size_t asm_bytes = assoc_smem(d.T, d.D, &io.cm_in_smem);
  if (int rc = ensure_dynamic_smem(assoc_kernel, asm_bytes)) return rc;
  assoc_kernel<<<d.S, ASSOC_THREADS, asm_bytes, st>>>(d, io);
  count_launch();
  return last_launch("assoc_kernel");
}

int aicam_tracker_cost_probe(aicam_tracker* t, const float* boxes, int stride_k, const int32_t* det_index,
                             const int32_t* det_count, const int32_t* crop_slot, const float* feats, float* app_cost,
                             float* gate_d2, int32_t* track_ids, int32_t* n_tracks, void* stream) {
  if (!t || !boxes || !det_index || !det_count || !crop_slot || !feats || !app_cost || !gate_d2 || !track_ids || !n_tracks)
    return fail(AICAM_ERR_INVALID_ARG, "tracker_cost_probe: null argument");
  if (stride_k <= 0 || reinterpret_cast<uintptr_t>(boxes) % 16)
    return fail(AICAM_ERR_INVALID_ARG, "tracker_cost_probe: stride_k must be positive and boxes 16-byte aligned");
  const Dev& d = t->d;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int rc = launch_appearance(d, t->tf, det_count, crop_slot, stride_k, feats, nullptr, st)) return rc;
  cost_probe_kernel<<<dim3(d.T, d.S), 128, 0, st>>>(d, boxes, stride_k, det_index, det_count, app_cost, gate_d2, track_ids, n_tracks);
  count_launch();
  return last_launch("cost_probe_kernel");
}

int aicam_tracker_snapshot(aicam_tracker* t, int stream_index, int32_t* ints, float* floats, int capacity) {
  if (!t || !ints || !floats || stream_index < 0 || stream_index >= t->d.S)
    return fail(AICAM_ERR_INVALID_ARG, "tracker_snapshot: bad arguments");
  const Dev& d = t->d;
  AICAM_CUDA_OK(cudaSetDevice(t->cfg.device));
  AICAM_CUDA_OK(cudaDeviceSynchronize());
  int n = 0;
  AICAM_CUDA_OK(cudaMemcpy(&n, d.n_tracks + stream_index, sizeof(int), cudaMemcpyDeviceToHost));
  if (n > capacity) return fail(AICAM_ERR_CAPACITY, "tracker_snapshot: capacity too small");
  const size_t T = d.T, sb = static_cast<size_t>(stream_index) * T;
  std::vector<int> order(T), id(T), state(T), hits(T), age(T), tsu(T), cls(T), gc(T);
  std::vector<float> mean(T * 8), cov(T * 16), conf(T);
  auto get = [&](void* dst, const void* src, size_t bytes) { return cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost); };
  AICAM_CUDA_OK(get(order.data(), d.order + sb, T * 4));
  AICAM_CUDA_OK(get(id.data(), d.track_id + sb, T * 4));
  AICAM_CUDA_OK(get(state.data(), d.state + sb, T * 4));
  AICAM_CUDA_OK(get(hits.data(), d.hits + sb, T * 4));
  AICAM_CUDA_OK(get(age.data(), d.age + sb, T * 4));
  AICAM_CUDA_OK(get(tsu.data(), d.tsu + sb, T * 4));
  AICAM_CUDA_OK(get(cls.data(), d.cls + sb, T * 4));
  AICAM_CUDA_OK(get(gc.data(), d.gal_count + sb, T * 4));
  AICAM_CUDA_OK(get(conf.data(), d.conf + sb, T * 4));
  AICAM_CUDA_OK(get(mean.data(), d.mean + sb * 8, T * 8 * 4));
  AICAM_CUDA_OK(get(cov.data(), d.cov + sb * 16, T * 16 * 4));
  for (int k = 0; k < n; ++k) {
    const int sl = order[k];
    int* io = ints + k * 7;
    io[0] = id[sl]; io[1] = state[sl]; io[2] = hits[sl]; io[3] = age[sl]; io[4] = tsu[sl]; io[5] = cls[sl]; io[6] = gc[sl];
    float* fo = floats + k * 25;
    for (int i = 0; i < 8; ++i) fo[i] = mean[sl * 8 + i];
    for (int i = 0; i < 16; ++i) fo[8 + i] = cov[sl * 16 + i];
    fo[24] = conf[sl];
  }
  return n;
}

const int32_t* aicam_tracker_row_slots(const aicam_tracker* t) { return t ? t->d.row_slot : nullptr; }

int aicam_tracker_overflow(aicam_tracker* t, int32_t* flags_host) {
  if (!t || !flags_host) return fail(AICAM_ERR_INVALID_ARG, "tracker_overflow: null argument");
  AICAM_CUDA_OK(cudaSetDevice(t->cfg.device));
  AICAM_CUDA_OK(cudaDeviceSynchronize());
  AICAM_CUDA_OK(cudaMemcpy(flags_host, t->d.overflow, sizeof(int) * t->d.S, cudaMemcpyDeviceToHost));
  return AICAM_OK;
}

int aicam_lsap(const float* cost, int count, int nr, int nc, int32_t* col_for_row, void* stream) {
  if (!cost || !col_for_row || count < 0 || nr <= 0 || nc <= 0 || nr > 1024 || nc > 1024)
    return fail(AICAM_ERR_INVALID_ARG, "lsap: bad arguments (sizes are limited to 1024)");
  if (count == 0) return AICAM_OK;
  const size_t sm = lsap_bytes(std::max(nr, nc)) + sizeof(int) * nr + 16;
  if (int rc = ensure_dynamic_smem(lsap_kernel, sm)) return rc;
  lsap_kernel<<<count, 32 * LSAP_MAX_WARPS, sm, static_cast<cudaStream_t>(stream)>>>(cost, nr, nc, col_for_row);
  count_launch();
  return last_launch("lsap_kernel");
}

int aicam_kf_gating(const float* state, const float* meas, int n, int m, float* d2, void* stream) {
  if (!state || !meas || !d2 || n < 0 || m <= 0) return fail(AICAM_ERR_INVALID_ARG, "kf_gating: bad arguments");
  if (n == 0) return AICAM_OK;
  gating_kernel<<<cdiv(n * m, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(state, meas, n, m, d2);
  count_launch();
  return last_launch("gating_kernel");
}

}  // extern "C"
