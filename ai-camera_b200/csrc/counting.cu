// Line crossings and zone entries per stream on the tracker's reported rows (include/aicam.h, "Counting"), one CTA per
// stream and one thread per row.  Integer arithmetic only (no --fmad entry in build.py: there is no float to contract),
// so the device and oracle/counting.py agree bit for bit.
//
// State in HBM, per (stream, tracker slot): st_id (0 = none; ids start at 1), the last reported doubled anchor
// st_px / st_py, the zone bits st_zones.  Counters are integer atomics, so the result does not depend on the order the
// rows are processed in; events get their offsets from a block scan over per-row event counts, in row order.
#include <cstring>
#include <string>
#include <vector>

#include "common.cuh"
#include "polygon.cuh"
#include "staging.cuh"

namespace aicam {

extern void count_launch();

namespace {

constexpr int COUNT_THREADS = 256;
constexpr int NL = AICAM_COUNT_MAX_LINES, NZ = AICAM_COUNT_MAX_ZONES, NV = AICAM_COUNT_MAX_VERTICES;
constexpr int NCLS = AICAM_COUNT_CLASSES;
constexpr int MAX_EVENTS = 1 << 20;

struct CounterDev {
  int S, T, E;
  const aicam_stream_counting* geom;  // [S]
  const int* set_mask;                // [S], right after geom in one allocation: the streams of the last set call
  int* st_id; int* st_px; int* st_py; unsigned* st_zones;  // [S][T]
  int64_t* line_counts;               // [S][NL][2][NCLS]
  int64_t* zone_counts;               // [S][NZ][2][NCLS]
  int* occupancy;                     // [S][NZ][NCLS]
  unsigned* row_zones;                // [S][T]
  int* events;                        // [S][E][4]
  int* event_count; int* overflow;    // [S]
};

// Dwell (include/aicam.h, "Dwell"): every pointer null until the first aicam_counter_set_dwell.
struct DwellDev {
  const aicam_stream_dwell* cfg;      // [S]
  const int* restart;                 // [S], right after cfg in one allocation: the streams the last set call enabled
  int* clock;                         // [S]
  int* st_id; unsigned* st_bits;      // [S][T]: bits 0..15 open visits, 16..31 alerted visits
  int* st_entry;                      // [S][T][NZ]
  int64_t* visits; int64_t* frames_total; int64_t* frames_max;  // [S][NZ][NCLS]
  int* row_dwell;                     // [S][T][NZ]
  int* events;                        // [S][E][5]
  int* event_count; int* overflow;    // [S]
};

__device__ __forceinline__ bool class_in(const uint64_t* mask, int cls) {
  return cls >= 0 && cls < NCLS && ((cls < 64 ? mask[0] >> cls : mask[1] >> (cls - 64)) & 1ull);
}

// +1 when P is strictly on the positive side of A->B (a point on the line belongs to the -1 side)
__device__ __forceinline__ int line_side(long long ax, long long ay, long long bx, long long by, long long px, long long py) {
  return (bx - ax) * (py - ay) - (by - ay) * (px - ax) > 0 ? 1 : -1;
}

__global__ void __launch_bounds__(COUNT_THREADS) count_kernel(CounterDev c, const int* __restrict__ out_tracks,
                                                              const int* __restrict__ out_count,
                                                              const int* __restrict__ row_slot,
                                                              const int* __restrict__ present) {
  __shared__ __align__(16) aicam_stream_counting g;
  __shared__ int occ[NZ * NCLS];
  __shared__ int warp_sum[COUNT_THREADS / 32];
  const int s = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (present && !present[s]) {  // absent: nothing of the stream changes; no events this step
    if (tid == 0) c.event_count[s] = 0;
    return;
  }
  {
    const int* src = reinterpret_cast<const int*>(c.geom + s);
    int* dst = reinterpret_cast<int*>(&g);
    for (int i = tid; i < static_cast<int>(sizeof(aicam_stream_counting) / 4); i += COUNT_THREADS) dst[i] = src[i];
  }
  for (int i = tid; i < NZ * NCLS; i += COUNT_THREADS) occ[i] = 0;
  __syncthreads();
  const long long sT = static_cast<long long>(s) * c.T;
  const int n = max(0, min(out_count[s], c.T));
  const int nl = g.n_lines, nz = g.n_zones;
  int64_t* lc = c.line_counts + static_cast<long long>(s) * NL * 2 * NCLS;
  int64_t* zc = c.zone_counts + static_cast<long long>(s) * NZ * 2 * NCLS;
  int* ev = c.events + static_cast<long long>(s) * c.E * 4;
  int base = 0;  // events of the rows before this tile (the same value in every thread)
  for (int r0 = 0; r0 < n; r0 += COUNT_THREADS) {
    const int r = r0 + tid;
    unsigned l_in = 0, l_out = 0, z_in = 0, z_out = 0;  // counted crossings / entries / exits, bit = line or zone index
    int id = 0, cls = 0;
    if (r < n) {
      const int* row = out_tracks + (sT + r) * 6;
      id = row[4];
      cls = row[5];
      const long long px = clamp_anchor(static_cast<long long>(row[0]) + row[2]), py = clamp_anchor(2ll * row[3]);
      const int slot = row_slot[sT + r];
      const bool valid = slot >= 0 && slot < c.T;  // (a row without a slot is counted as a first report, keeps no state)
      const long long ss = sT + (valid ? slot : 0);
      const bool first = !valid || c.st_id[ss] != id;
      const long long x0 = first ? 0 : c.st_px[ss], y0 = first ? 0 : c.st_py[ss];
      const unsigned z_prev = first ? 0u : c.st_zones[ss];
      if (!first) {
        for (int l = 0; l < nl; ++l) {
          const long long ax = 2ll * g.line[l][0], ay = 2ll * g.line[l][1], bx = 2ll * g.line[l][2], by = 2ll * g.line[l][3];
          const int s0 = line_side(ax, ay, bx, by, x0, y0), s1 = line_side(ax, ay, bx, by, px, py);
          if (s0 == s1) continue;
          const long long dx = px - x0, dy = py - y0;
          const long long da = dx * (ay - y0) - dy * (ax - x0), db = dx * (by - y0) - dy * (bx - x0);
          if ((da > 0 && db > 0) || (da < 0 && db < 0)) continue;  // A and B strictly on one side of P0P1
          if (!class_in(g.line_class_mask[l], cls)) continue;
          const int dir = s1 > 0 ? 0 : 1;
          if (dir == 0) l_in |= 1u << l; else l_out |= 1u << l;
          atomicAdd(reinterpret_cast<unsigned long long*>(lc + (l * 2 + dir) * NCLS + cls), 1ull);
        }
      }
      unsigned z_now = 0;
      for (int z = 0; z < nz; ++z) {
        const bool inside = in_zone(g.zone_xy[z], g.zone_n[z], px, py);
        if (inside) z_now |= 1u << z;
        if (!class_in(g.zone_class_mask[z], cls)) continue;
        if (inside) atomicAdd(&occ[z * NCLS + cls], 1);
        const bool was = (z_prev >> z) & 1u;
        if (inside == was) continue;
        const int k = inside ? 0 : 1;
        if (inside) z_in |= 1u << z; else z_out |= 1u << z;
        atomicAdd(reinterpret_cast<unsigned long long*>(zc + (z * 2 + k) * NCLS + cls), 1ull);
      }
      c.row_zones[sT + r] = z_now;
      if (valid) { c.st_id[ss] = id; c.st_px[ss] = static_cast<int>(px); c.st_py[ss] = static_cast<int>(py); c.st_zones[ss] = z_now; }
    }
    // block-wide exclusive scan of the per-row event counts: events are laid out in row order
    const int nev = __popc(l_in | l_out) + __popc(z_in | z_out);
    int incl = nev;
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) warp_sum[warp] = incl;
    __syncthreads();
    int before = 0, total = 0;
    for (int w = 0; w < COUNT_THREADS / 32; ++w) {
      const int v = warp_sum[w];
      if (w < warp) before += v;
      total += v;
    }
    int at = base + before + incl - nev;
    for (int l = 0; l < nl && at < c.E; ++l) {
      if (!(((l_in | l_out) >> l) & 1u)) continue;
      *reinterpret_cast<int4*>(ev + 4ll * at) = make_int4((l_in >> l) & 1u ? 0 : 1, l, id, cls);
      ++at;
    }
    for (int z = 0; z < nz && at < c.E; ++z) {
      if (!(((z_in | z_out) >> z) & 1u)) continue;
      *reinterpret_cast<int4*>(ev + 4ll * at) = make_int4((z_in >> z) & 1u ? 2 : 3, z, id, cls);
      ++at;
    }
    base += total;
    __syncthreads();  // (warp_sum is rewritten by the next tile; occ is complete after the last)
  }
  if (tid == 0) {
    c.event_count[s] = min(base, c.E);
    if (base > c.E) c.overflow[s] = 1;
  }
  int* oc = c.occupancy + static_cast<long long>(s) * NZ * NCLS;
  for (int i = tid; i < NZ * NCLS; i += COUNT_THREADS) oc[i] = occ[i];
}

// mask: device i32[S]; streams with a zero entry are left as they are, null resets every stream
__global__ void counter_reset_kernel(CounterDev c, const int* __restrict__ mask) {
  const int s = blockIdx.x;
  if (mask && !mask[s]) return;
  const long long sT = static_cast<long long>(s) * c.T;
  for (int k = threadIdx.x; k < c.T; k += blockDim.x) { c.st_id[sT + k] = 0; c.st_zones[sT + k] = 0u; c.row_zones[sT + k] = 0u; }
  for (int i = threadIdx.x; i < NL * 2 * NCLS; i += blockDim.x) c.line_counts[static_cast<long long>(s) * NL * 2 * NCLS + i] = 0;
  for (int i = threadIdx.x; i < NZ * 2 * NCLS; i += blockDim.x) c.zone_counts[static_cast<long long>(s) * NZ * 2 * NCLS + i] = 0;
  for (int i = threadIdx.x; i < NZ * NCLS; i += blockDim.x) c.occupancy[static_cast<long long>(s) * NZ * NCLS + i] = 0;
  if (threadIdx.x == 0) { c.event_count[s] = 0; c.overflow[s] = 0; }
}

// One CTA per stream, one thread per row, after count_kernel of the same step: reads its row_zones and the zone class
// masks.  Per row the open and alerted bits and entry[16] live in registers (loops over zones fully unrolled); durations
// are added with integer atomics, events laid out in row order by the same block scan as count_kernel.
__global__ void __launch_bounds__(COUNT_THREADS) dwell_kernel(CounterDev c, DwellDev w, const int* __restrict__ out_tracks,
                                                              const int* __restrict__ out_count,
                                                              const int* __restrict__ row_slot,
                                                              const int* __restrict__ present) {
  __shared__ uint64_t zmask[NZ][2];
  __shared__ int loiter[NZ];
  __shared__ int warp_sum[COUNT_THREADS / 32];
  __shared__ int clock_s, nz_s;
  const int s = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if ((present && !present[s]) || !w.cfg[s].enabled) {  // nothing of the stream changes, its clock included
    if (tid == 0) w.event_count[s] = 0;
    return;
  }
  if (tid < NZ) {
    zmask[tid][0] = c.geom[s].zone_class_mask[tid][0];
    zmask[tid][1] = c.geom[s].zone_class_mask[tid][1];
    loiter[tid] = w.cfg[s].loiter_frames[tid];
  }
  if (tid == 0) {
    clock_s = w.clock[s] + 1;
    w.clock[s] = clock_s;
    nz_s = c.geom[s].n_zones;
  }
  __syncthreads();
  const int f = clock_s, nz = nz_s;
  const long long sT = static_cast<long long>(s) * c.T;
  const int n = max(0, min(out_count[s], c.T));
  const long long sz = static_cast<long long>(s) * NZ * NCLS;
  int* ev = w.events + static_cast<long long>(s) * c.E * 5;
  int base = 0;
  for (int r0 = 0; r0 < n; r0 += COUNT_THREADS) {
    const int r = r0 + tid;
    unsigned closed = 0, alert = 0;  // bit z: a visit of zone z completed / alerted at this row
    int id = 0, cls = 0;
    int val[NZ];  // frames since entry (the duration, for a completed visit)
    if (r < n) {
      const int* row = out_tracks + (sT + r) * 6;
      id = row[4];
      cls = row[5];
      const unsigned zb = c.row_zones[sT + r];
      const int slot = row_slot[sT + r];
      const bool valid = slot >= 0 && slot < c.T;  // (a row without a slot is a first report and keeps no state)
      const long long ss = sT + (valid ? slot : 0);
      const bool first = !valid || w.st_id[ss] != id;
      unsigned bits = first ? 0u : w.st_bits[ss];
      int4* ep = reinterpret_cast<int4*>(w.st_entry + ss * NZ);
      int entry[NZ];
#pragma unroll
      for (int q = 0; q < NZ / 4; ++q) {
        const int4 e = first ? make_int4(0, 0, 0, 0) : ep[q];
        entry[4 * q] = e.x; entry[4 * q + 1] = e.y; entry[4 * q + 2] = e.z; entry[4 * q + 3] = e.w;
      }
      unsigned shown = 0;  // zones whose row_dwell entry is val
#pragma unroll
      for (int z = 0; z < NZ; ++z) {
        val[z] = -1;
        if (z >= nz || !class_in(zmask[z], cls)) continue;
        const unsigned ob = 1u << z, ab = 1u << (16 + z);
        if ((zb >> z) & 1u) {
          if (!(bits & ob)) { bits = (bits | ob) & ~ab; entry[z] = f; }
          val[z] = f - entry[z];
          shown |= ob;
          if (loiter[z] > 0 && val[z] >= loiter[z] && !(bits & ab)) { bits |= ab; alert |= ob; }
        } else if (bits & ob) {
          val[z] = f - entry[z];
          bits &= ~(ob | ab);
          closed |= ob;
          const long long k = sz + z * NCLS + cls;
          atomicAdd(reinterpret_cast<unsigned long long*>(w.visits + k), 1ull);
          atomicAdd(reinterpret_cast<unsigned long long*>(w.frames_total + k), static_cast<unsigned long long>(val[z]));
          atomicMax(reinterpret_cast<long long*>(w.frames_max + k), static_cast<long long>(val[z]));
        }
      }
      int4* rd = reinterpret_cast<int4*>(w.row_dwell + (sT + r) * NZ);
#pragma unroll
      for (int q = 0; q < NZ / 4; ++q) {
        int o[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) o[k] = (shown >> (4 * q + k)) & 1u ? val[4 * q + k] : -1;
        rd[q] = make_int4(o[0], o[1], o[2], o[3]);
      }
      if (valid) {
        w.st_id[ss] = id;
        w.st_bits[ss] = bits;
#pragma unroll
        for (int q = 0; q < NZ / 4; ++q)
          ep[q] = make_int4(entry[4 * q], entry[4 * q + 1], entry[4 * q + 2], entry[4 * q + 3]);
      }
    }
    const int nev = __popc(closed | alert);
    int incl = nev;
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) warp_sum[warp] = incl;
    __syncthreads();
    int before = 0, total = 0;
    for (int q = 0; q < COUNT_THREADS / 32; ++q) {
      const int v = warp_sum[q];
      if (q < warp) before += v;
      total += v;
    }
    int at = base + before + incl - nev;
#pragma unroll
    for (int z = 0; z < NZ; ++z) {
      if (!(((closed | alert) >> z) & 1u) || at >= c.E) continue;
      int* e = ev + 5ll * at;
      e[0] = (closed >> z) & 1u ? 0 : 1; e[1] = z; e[2] = id; e[3] = cls; e[4] = val[z];
      ++at;
    }
    base += total;
    __syncthreads();  // (warp_sum is rewritten by the next tile)
  }
  if (tid == 0) {
    w.event_count[s] = min(base, c.E);
    if (base > c.E) w.overflow[s] = 1;
  }
}

// Restart the dwell state of the streams whose mask entry is non-zero (null: every stream); settings are kept.
__global__ void dwell_reset_kernel(CounterDev c, DwellDev w, const int* __restrict__ mask) {
  const int s = blockIdx.x;
  if (mask && !mask[s]) return;
  const long long sT = static_cast<long long>(s) * c.T;
  for (int k = threadIdx.x; k < c.T; k += blockDim.x) { w.st_id[sT + k] = 0; w.st_bits[sT + k] = 0u; }
  for (int k = threadIdx.x; k < c.T * NZ; k += blockDim.x) w.row_dwell[sT * NZ + k] = -1;
  for (int i = threadIdx.x; i < NZ * NCLS; i += blockDim.x) {
    const long long k = static_cast<long long>(s) * NZ * NCLS + i;
    w.visits[k] = 0; w.frames_total[k] = 0; w.frames_max[k] = 0;
  }
  if (threadIdx.x == 0) { w.clock[s] = 0; w.event_count[s] = 0; w.overflow[s] = 0; }
}

bool coord_ok(int32_t v) { return v >= -AICAM_COUNT_MAX_COORD && v <= AICAM_COUNT_MAX_COORD; }
bool mask_ok(const uint64_t* m) { return (m[1] >> (NCLS - 64)) == 0; }

int check_counting(const aicam_stream_counting& g, const std::string& at) {
  if (g.n_lines < 0 || g.n_lines > NL || g.n_zones < 0 || g.n_zones > NZ)
    return fail(AICAM_ERR_INVALID_ARG, at + "n_lines and n_zones must be in 0..16");
  for (int l = 0; l < g.n_lines; ++l) {
    const int32_t* p = g.line[l];
    if (!coord_ok(p[0]) || !coord_ok(p[1]) || !coord_ok(p[2]) || !coord_ok(p[3]))
      return fail(AICAM_ERR_INVALID_ARG, at + "line " + std::to_string(l) + ": coordinate beyond 2^20");
    if (p[0] == p[2] && p[1] == p[3]) return fail(AICAM_ERR_INVALID_ARG, at + "line " + std::to_string(l) + " has zero length");
    if (!mask_ok(g.line_class_mask[l])) return fail(AICAM_ERR_INVALID_ARG, at + "line " + std::to_string(l) + ": class beyond 79");
  }
  for (int z = 0; z < g.n_zones; ++z) {
    if (g.zone_n[z] < 3 || g.zone_n[z] > NV)
      return fail(AICAM_ERR_INVALID_ARG, at + "zone " + std::to_string(z) + " must have 3..32 vertices");
    for (int v = 0; v < g.zone_n[z]; ++v)
      if (!coord_ok(g.zone_xy[z][v][0]) || !coord_ok(g.zone_xy[z][v][1]))
        return fail(AICAM_ERR_INVALID_ARG, at + "zone " + std::to_string(z) + ": coordinate beyond 2^20");
    if (!mask_ok(g.zone_class_mask[z])) return fail(AICAM_ERR_INVALID_ARG, at + "zone " + std::to_string(z) + ": class beyond 79");
  }
  return AICAM_OK;
}

}  // namespace
}  // namespace aicam

struct aicam_counter {
  aicam::CounterDev d;
  int device = 0;
  std::vector<aicam_stream_counting> geom;  // host copy of d.geom
  uint8_t* upload = nullptr;                // device: geom [S] then the set mask i32 [S]
  aicam::PinnedStaging staging;             // of aicam_counter_set_streams
  std::vector<void*> allocs;
  aicam::DwellDev w{};                      // dwell: allocated by the first aicam_counter_set_dwell
  std::vector<aicam_stream_dwell> dwell;    // host copy of w.cfg (empty until then)
  uint8_t* dwell_upload = nullptr;          // device: cfg [S] then the restart mask i32 [S]
  aicam::PinnedStaging dwell_staging;       // of aicam_counter_set_dwell
};

using namespace aicam;

namespace {
size_t upload_bytes(int S) { return static_cast<size_t>(S) * (sizeof(aicam_stream_counting) + sizeof(int32_t)); }

template <typename Tp>
int counter_alloc(aicam_counter* c, Tp** p, size_t n) {
  void* q = nullptr;
  if (cudaMalloc(&q, n * sizeof(Tp)) != cudaSuccess) return fail(AICAM_ERR_CUDA, "counter_create: cudaMalloc failed");
  c->allocs.push_back(q);
  if (cudaMemset(q, 0, n * sizeof(Tp)) != cudaSuccess) return fail(AICAM_ERR_CUDA, "counter_create: cudaMemset failed");
  *p = static_cast<Tp*>(q);
  return AICAM_OK;
}

size_t dwell_upload_bytes(int S) { return static_cast<size_t>(S) * (sizeof(aicam_stream_dwell) + sizeof(int32_t)); }

int launch_dwell_reset(aicam_counter* c, const int32_t* mask, cudaStream_t st) {
  dwell_reset_kernel<<<c->d.S, 256, 0, st>>>(c->d, c->w, mask);
  count_launch();
  return last_launch("dwell_reset_kernel");
}

// (the dwell restart is a launch of its own, made only once dwell is set, so that counting alone launches as before)
int launch_reset(aicam_counter* c, const int32_t* mask, cudaStream_t st) {
  counter_reset_kernel<<<c->d.S, 256, 0, st>>>(c->d, mask);
  count_launch();
  if (int rc = last_launch("counter_reset_kernel")) return rc;
  return c->w.cfg ? launch_dwell_reset(c, mask, st) : AICAM_OK;
}

int dwell_alloc(aicam_counter* c) {
  DwellDev w{};
  const int S = c->d.S;
  const size_t ST = static_cast<size_t>(S) * c->d.T, SZK = static_cast<size_t>(S) * NZ * NCLS;
  int rc = 0;
  rc |= counter_alloc(c, &c->dwell_upload, dwell_upload_bytes(S));
  rc |= counter_alloc(c, &w.clock, S);
  rc |= counter_alloc(c, &w.st_id, ST); rc |= counter_alloc(c, &w.st_bits, ST); rc |= counter_alloc(c, &w.st_entry, ST * NZ);
  rc |= counter_alloc(c, &w.visits, SZK); rc |= counter_alloc(c, &w.frames_total, SZK); rc |= counter_alloc(c, &w.frames_max, SZK);
  rc |= counter_alloc(c, &w.row_dwell, ST * NZ);
  rc |= counter_alloc(c, &w.events, static_cast<size_t>(S) * c->d.E * 5);
  rc |= counter_alloc(c, &w.event_count, S); rc |= counter_alloc(c, &w.overflow, S);
  if (rc) return AICAM_ERR_CUDA;
  if (cudaMemset(w.row_dwell, 0xff, ST * NZ * sizeof(int)) != cudaSuccess)
    return fail(AICAM_ERR_CUDA, "counter_set_dwell: cudaMemset failed");
  if (c->dwell_staging.create(dwell_upload_bytes(S)) != cudaSuccess) {
    c->dwell_staging.destroy();
    return fail(AICAM_ERR_CUDA, "counter_set_dwell: pinned staging failed");
  }
  // (the zeroing above runs on the legacy stream: finish it before work on the caller's stream reads the buffers)
  if (cudaDeviceSynchronize() != cudaSuccess) return fail(AICAM_ERR_CUDA, "counter_set_dwell: synchronise failed");
  w.cfg = reinterpret_cast<const aicam_stream_dwell*>(c->dwell_upload);
  w.restart = reinterpret_cast<const int*>(c->dwell_upload + static_cast<size_t>(S) * sizeof(aicam_stream_dwell));
  c->w = w;
  c->dwell.assign(S, aicam_stream_dwell{});
  return AICAM_OK;
}
}  // namespace

extern "C" {

int aicam_counter_create(int device, int n_streams, int max_tracks, int max_events, aicam_counter** out) {
  if (!out) return fail(AICAM_ERR_INVALID_ARG, "counter_create: null argument");
  *out = nullptr;
  if (n_streams <= 0 || max_tracks <= 0 || max_events <= 0)
    return fail(AICAM_ERR_INVALID_ARG, "counter_create: sizes must be positive");
  if (max_tracks > 1024 || max_events > MAX_EVENTS)
    return fail(AICAM_ERR_CAPACITY, "counter_create: max_tracks is limited to 1024 and max_events to 2^20");
  AICAM_CUDA_OK(cudaSetDevice(device));
  aicam_counter* c = new aicam_counter();
  c->device = device;
  CounterDev& d = c->d;
  d.S = n_streams; d.T = max_tracks; d.E = max_events;
  c->geom.assign(d.S, aicam_stream_counting{});
  const size_t ST = static_cast<size_t>(d.S) * d.T;
  int rc = 0;
  rc |= counter_alloc(c, &c->upload, upload_bytes(d.S));
  rc |= counter_alloc(c, &d.st_id, ST); rc |= counter_alloc(c, &d.st_px, ST); rc |= counter_alloc(c, &d.st_py, ST);
  rc |= counter_alloc(c, &d.st_zones, ST); rc |= counter_alloc(c, &d.row_zones, ST);
  rc |= counter_alloc(c, &d.line_counts, static_cast<size_t>(d.S) * NL * 2 * NCLS);
  rc |= counter_alloc(c, &d.zone_counts, static_cast<size_t>(d.S) * NZ * 2 * NCLS);
  rc |= counter_alloc(c, &d.occupancy, static_cast<size_t>(d.S) * NZ * NCLS);
  rc |= counter_alloc(c, &d.events, static_cast<size_t>(d.S) * d.E * 4);
  rc |= counter_alloc(c, &d.event_count, d.S); rc |= counter_alloc(c, &d.overflow, d.S);
  if (!rc && c->staging.create(upload_bytes(d.S)) != cudaSuccess) rc = fail(AICAM_ERR_CUDA, "counter_create: pinned staging failed");
  if (rc) { aicam_counter_destroy(c); return AICAM_ERR_CUDA; }
  d.geom = reinterpret_cast<const aicam_stream_counting*>(c->upload);
  d.set_mask = reinterpret_cast<const int*>(c->upload + static_cast<size_t>(d.S) * sizeof(aicam_stream_counting));
  if (cudaDeviceSynchronize() != cudaSuccess) { aicam_counter_destroy(c); return fail(AICAM_ERR_CUDA, "counter_create: synchronise failed"); }
  *out = c;
  return AICAM_OK;
}

void aicam_counter_destroy(aicam_counter* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  c->staging.destroy();
  c->dwell_staging.destroy();
  for (void* p : c->allocs) cudaFree(p);
  delete c;
}

int aicam_counter_set_streams(aicam_counter* c, const int32_t* indices_host, const aicam_stream_counting* host, int n,
                              void* stream) {
  if (!c || n < 0 || (n > 0 && (!indices_host || !host)))
    return fail(AICAM_ERR_INVALID_ARG, "counter_set_streams: null argument or negative count");
  std::vector<aicam_stream_counting> next = c->geom;  // validated as a whole before anything is stored or copied
  std::vector<int32_t> mask(c->d.S, 0);
  for (int i = 0; i < n; ++i) {
    const std::string at = "counter_set_streams: entry " + std::to_string(i) + ": ";
    if (indices_host[i] < 0 || indices_host[i] >= c->d.S) return fail(AICAM_ERR_INVALID_ARG, at + "stream index out of range");
    if (int rc = check_counting(host[i], at)) return rc;
    next[indices_host[i]] = host[i];
    mask[indices_host[i]] = 1;
  }
  if (n == 0) return AICAM_OK;
  AICAM_CUDA_OK(cudaSetDevice(c->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* h = nullptr;
  AICAM_CUDA_OK(c->staging.acquire(&h));
  const size_t gbytes = next.size() * sizeof(aicam_stream_counting);
  std::memcpy(h, next.data(), gbytes);
  std::memcpy(h + gbytes, mask.data(), mask.size() * sizeof(int32_t));
  AICAM_CUDA_OK(c->staging.upload(c->upload, upload_bytes(c->d.S), st));
  c->geom.swap(next);
  return launch_reset(c, c->d.set_mask, st);
}

int aicam_counter_step(aicam_counter* c, const int32_t* out_tracks, const int32_t* out_count, const int32_t* row_slot,
                       const int32_t* present, void* stream) {
  if (!c || !out_tracks || !out_count || !row_slot) return fail(AICAM_ERR_INVALID_ARG, "counter_step: null argument");
  count_kernel<<<c->d.S, COUNT_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(c->d, out_tracks, out_count, row_slot, present);
  count_launch();
  return last_launch("count_kernel");
}

int aicam_counter_reset_streams(aicam_counter* c, const int32_t* mask, void* stream) {
  if (!c || !mask) return fail(AICAM_ERR_INVALID_ARG, "counter_reset_streams: null argument");
  return launch_reset(c, mask, static_cast<cudaStream_t>(stream));
}

int aicam_counter_outputs(const aicam_counter* c, aicam_counter_output* out) {
  if (!c || !out) return fail(AICAM_ERR_INVALID_ARG, "counter_outputs: null argument");
  const CounterDev& d = c->d;
  *out = aicam_counter_output{d.line_counts, d.zone_counts, d.occupancy, d.row_zones, d.events, d.event_count};
  return AICAM_OK;
}

int aicam_counter_overflow(aicam_counter* c, int32_t* flags_host) {
  if (!c || !flags_host) return fail(AICAM_ERR_INVALID_ARG, "counter_overflow: null argument");
  AICAM_CUDA_OK(cudaSetDevice(c->device));
  AICAM_CUDA_OK(cudaDeviceSynchronize());
  AICAM_CUDA_OK(cudaMemcpy(flags_host, c->d.overflow, sizeof(int32_t) * c->d.S, cudaMemcpyDeviceToHost));
  return AICAM_OK;
}

int aicam_counter_set_dwell(aicam_counter* c, const int32_t* indices_host, const aicam_stream_dwell* host, int n,
                            void* stream) {
  if (!c || n < 0 || (n > 0 && (!indices_host || !host)))
    return fail(AICAM_ERR_INVALID_ARG, "counter_set_dwell: null argument or negative count");
  const int S = c->d.S;
  // validated as a whole before anything is allocated, stored or copied
  std::vector<aicam_stream_dwell> next = c->dwell.empty() ? std::vector<aicam_stream_dwell>(S, aicam_stream_dwell{}) : c->dwell;
  for (int i = 0; i < n; ++i) {
    const std::string at = "counter_set_dwell: entry " + std::to_string(i) + ": ";
    if (indices_host[i] < 0 || indices_host[i] >= S) return fail(AICAM_ERR_INVALID_ARG, at + "stream index out of range");
    if (host[i].enabled != 0 && host[i].enabled != 1) return fail(AICAM_ERR_INVALID_ARG, at + "enabled must be 0 or 1");
    for (int z = 0; z < NZ; ++z)
      if (host[i].loiter_frames[z] < 0 || host[i].loiter_frames[z] > AICAM_DWELL_MAX_LOITER)
        return fail(AICAM_ERR_INVALID_ARG, at + "loiter_frames[" + std::to_string(z) + "] must be in 0..2^30");
    next[indices_host[i]] = host[i];
  }
  if (n == 0) return AICAM_OK;
  AICAM_CUDA_OK(cudaSetDevice(c->device));
  if (!c->w.cfg)
    if (int rc = dwell_alloc(c)) return rc;
  std::vector<int32_t> restart(S, 0);  // disabled -> enabled: the stream's dwell state starts
  bool any = false;
  for (int k = 0; k < S; ++k) {
    restart[k] = next[k].enabled && !c->dwell[k].enabled;
    any |= restart[k] != 0;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* h = nullptr;
  AICAM_CUDA_OK(c->dwell_staging.acquire(&h));
  const size_t cbytes = next.size() * sizeof(aicam_stream_dwell);
  std::memcpy(h, next.data(), cbytes);
  std::memcpy(h + cbytes, restart.data(), restart.size() * sizeof(int32_t));
  AICAM_CUDA_OK(c->dwell_staging.upload(c->dwell_upload, dwell_upload_bytes(S), st));
  c->dwell.swap(next);
  return any ? launch_dwell_reset(c, c->w.restart, st) : AICAM_OK;
}

int aicam_counter_dwell_step(aicam_counter* c, const int32_t* out_tracks, const int32_t* out_count, const int32_t* row_slot,
                             const int32_t* present, void* stream) {
  if (!c || !out_tracks || !out_count || !row_slot) return fail(AICAM_ERR_INVALID_ARG, "counter_dwell_step: null argument");
  if (!c->w.cfg) return fail(AICAM_ERR_INVALID_ARG, "counter_dwell_step: dwell is not set (aicam_counter_set_dwell)");
  dwell_kernel<<<c->d.S, COUNT_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(c->d, c->w, out_tracks, out_count, row_slot,
                                                                                present);
  count_launch();
  return last_launch("dwell_kernel");
}

int aicam_counter_dwell_outputs(const aicam_counter* c, aicam_counter_dwell_output* out) {
  if (!c || !out) return fail(AICAM_ERR_INVALID_ARG, "counter_dwell_outputs: null argument");
  if (!c->w.cfg) return fail(AICAM_ERR_INVALID_ARG, "counter_dwell_outputs: dwell is not set (aicam_counter_set_dwell)");
  const DwellDev& w = c->w;
  *out = aicam_counter_dwell_output{w.visits, w.frames_total, w.frames_max, w.row_dwell, w.events, w.event_count};
  return AICAM_OK;
}

int aicam_counter_dwell_overflow(aicam_counter* c, int32_t* flags_host) {
  if (!c || !flags_host) return fail(AICAM_ERR_INVALID_ARG, "counter_dwell_overflow: null argument");
  if (!c->w.cfg) {
    std::memset(flags_host, 0, sizeof(int32_t) * c->d.S);
    return AICAM_OK;
  }
  AICAM_CUDA_OK(cudaSetDevice(c->device));
  AICAM_CUDA_OK(cudaDeviceSynchronize());
  AICAM_CUDA_OK(cudaMemcpy(flags_host, c->w.overflow, sizeof(int32_t) * c->d.S, cudaMemcpyDeviceToHost));
  return AICAM_OK;
}

}  // extern "C"
