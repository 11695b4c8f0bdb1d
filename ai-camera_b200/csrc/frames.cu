// The frame table (include/aicam.h, aicam_frame_table_*): per-stream frame descriptors, validated and resolved on the
// host, read on the device by the ragged K1 / detect / K5 entry points and, for presence, by the tracker step.  See frame_table.cuh for the device layout.
#include <algorithm>
#include <cstring>
#include <string>
#include <vector>

#include "frame_table.cuh"

namespace aicam {
void letterbox_geometry(int h, int w, double* r, int* new_h, int* new_w, double* dw, double* dh, int* top, int* left);
}

using namespace aicam;

namespace {

bool aligned(const void* p, uintptr_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }

}  // namespace

extern "C" {

int aicam_frame_table_create(int device, int capacity, int max_h, int max_w, aicam_frame_table** out) {
  if (!out) return fail(AICAM_ERR_INVALID_ARG, "frame_table_create: null out");
  *out = nullptr;
  if (capacity <= 0 || max_h <= 0 || max_w <= 0 || max_h > 32768 || max_w > 32768)
    return fail(AICAM_ERR_INVALID_ARG, "frame_table_create: capacity must be positive and the bound in 1..32768");
  AICAM_CUDA_OK(cudaSetDevice(device));
  aicam_frame_table* t = new aicam_frame_table();
  t->device = device; t->capacity = capacity; t->max_h = max_h; t->max_w = max_w;
  const size_t bytes = frame_table_bytes(capacity);
  cudaError_t e = cudaMalloc(&t->dev, bytes);
  if (e == cudaSuccess) e = t->staging.create(bytes);
  if (e == cudaSuccess) e = cudaMemset(t->dev, 0, bytes);  // count 0 until the first set
  if (e != cudaSuccess) {
    aicam_frame_table_destroy(t);
    return fail(AICAM_ERR_CUDA, std::string("frame_table_create: ") + cudaGetErrorString(e));
  }
  *out = t;
  return AICAM_OK;
}

void aicam_frame_table_destroy(aicam_frame_table* t) {
  if (!t) return;
  cudaSetDevice(t->device);
  t->staging.destroy();
  t->region_staging.destroy();
  if (t->dev) cudaFree(t->dev);
  if (t->regions_dev) cudaFree(t->regions_dev);
  if (t->region_keep) cudaFree(t->region_keep);
  delete t;
}

int aicam_frame_table_set(aicam_frame_table* t, const aicam_frame_desc* descs, int n, void* stream) {
  return aicam_frame_table_set_present(t, descs, nullptr, n, stream);
}

int aicam_frame_table_set_present(aicam_frame_table* t, const aicam_frame_desc* descs, const uint8_t* present_host, int n,
                                  void* stream) {
  auto is_present = [&](int i) { return !present_host || present_host[i] != 0; };
  if (!t || n < 0) return fail(AICAM_ERR_INVALID_ARG, "frame_table_set: null table or descriptors");
  if (!descs)
    for (int i = 0; i < n; ++i)
      if (is_present(i)) return fail(AICAM_ERR_INVALID_ARG, "frame_table_set: null table or descriptors");
  if (n > t->capacity) return fail(AICAM_ERR_CAPACITY, "frame_table_set: more frames than the table's capacity");
  // validate every present descriptor before touching the staging or launching anything (absent ones are not read)
  for (int i = 0; i < n; ++i) {
    if (!is_present(i)) continue;
    const aicam_frame_desc& d = descs[i];
    const std::string at = "frame_table_set: frame " + std::to_string(i) + ": ";
    if (d.kind != 0 && d.kind != 1) return fail(AICAM_ERR_INVALID_ARG, at + "kind must be 0 (BGR) or 1 (NV12)");
    if (!d.data || (d.kind == 1 && !d.chroma)) return fail(AICAM_ERR_INVALID_ARG, at + "null plane pointer");
    if (d.h <= 0 || d.w <= 0) return fail(AICAM_ERR_INVALID_ARG, at + "height and width must be positive");
    if (d.h > t->max_h || d.w > t->max_w) return fail(AICAM_ERR_CAPACITY, at + "frame exceeds the table's size bound");
    if (d.kind == 1 && (d.h % 2 || d.w % 2)) return fail(AICAM_ERR_INVALID_ARG, at + "NV12 frames have even height and width");
    const long long row = d.kind == 0 ? 3LL * d.w : d.w;
    if (d.pitch < row) return fail(AICAM_ERR_INVALID_ARG, at + "pitch is smaller than a row");
  }
  AICAM_CUDA_OK(cudaSetDevice(t->device));
  std::vector<FrameRec> recs(n);
  std::vector<int> ring, pix;
  const bool ring_fits = t->ring_fits();
  int packed = 0;
  for (int i = 0; i < n; ++i) {
    FrameRec& r = recs[i];
    if (!is_present(i)) {  // nothing of the frame is read: no geometry, no list, no slot
      r = FrameRec{};
      r.slot = -1;
      continue;
    }
    const aicam_frame_desc& d = descs[i];
    r.slot = packed++;
    r.data = d.data; r.chroma = d.kind == 1 ? d.chroma : nullptr;
    r.h = d.h; r.w = d.w; r.pitch = d.pitch; r.kind = d.kind;
    int decimate = 0;
    if (int rc = k1_geometry(d.h, d.w, &decimate, &r.mode, &r.new_h, &r.new_w, &r.top, &r.left, &r.tab)) return rc;
    double ratio, dw, dh;
    int nh, nw, top, left;
    letterbox_geometry(d.h, d.w, &ratio, &nh, &nw, &dw, &dh, &top, &left);
    r.ratio = static_cast<float>(ratio); r.pad_w = static_cast<float>(dw); r.pad_h = static_cast<float>(dh);
    // bulk copies move 16-byte multiples between 16-byte aligned addresses
    const int row = d.kind == 0 ? 3 * d.w : d.w;
    r.staged = decimate && ring_fits && aligned(d.data, 16) && d.pitch % 16 == 0 && row % 16 == 0 &&
               (d.kind == 0 || aligned(d.chroma, 16));
    (r.staged ? ring : pix).push_back(i);
    // the staged crop path loads aligned 32-bit words covering a segment: no word may cross the end of a plane
    r.crop_staged = aligned(d.data, 4) && (static_cast<long long>(d.h) * d.pitch) % 4 == 0 &&
                    (d.kind == 0 || (aligned(d.chroma, 4) && (static_cast<long long>(d.h / 2) * d.pitch) % 4 == 0));
  }
  for (int i = 0; i < n && i < static_cast<int>(t->filters.size()); ++i) {  // absent entries carry them too (unread)
    const aicam_stream_filter& f = t->filters[i];
    FrameRec& r = recs[i];
    r.filt = 1;
    r.score_thr = f.score_thr; r.iou_thr = f.iou_thr; r.min_conf = f.min_confidence;
    r.mask_lo = f.class_mask_lo; r.mask_hi = f.class_mask_hi;
  }
  // stage into the pinned buffer whose previous copy has completed
  uint8_t* h = nullptr;
  AICAM_CUDA_OK(t->staging.acquire(&h));
  int* counts = reinterpret_cast<int*>(h);
  counts[0] = n; counts[1] = static_cast<int>(ring.size()); counts[2] = static_cast<int>(pix.size()); counts[3] = packed;
  int* lists = counts + FT_COUNTS;
  std::copy(ring.begin(), ring.end(), lists);
  std::copy(pix.begin(), pix.end(), lists + t->capacity);
  int* present = lists + 2 * t->capacity;
  for (int i = 0; i < t->capacity; ++i) present[i] = i < n && recs[i].slot >= 0 ? 1 : 0;
  if (n) std::memcpy(h + frame_table_recs_offset(t->capacity), recs.data(), n * sizeof(FrameRec));
  AICAM_CUDA_OK(t->staging.upload(t->dev, frame_table_recs_offset(t->capacity) + n * sizeof(FrameRec),
                                   static_cast<cudaStream_t>(stream)));
  t->n = n;
  return AICAM_OK;
}

int aicam_frame_table_set_filters(aicam_frame_table* t, const aicam_stream_filter* host, int n) {
  if (!t || n < 0) return fail(AICAM_ERR_INVALID_ARG, "frame_table_set_filters: null table or negative count");
  if (!host || n == 0) {
    t->filters.clear();
    return AICAM_OK;
  }
  if (n > t->capacity) return fail(AICAM_ERR_CAPACITY, "frame_table_set_filters: more entries than the table's capacity");
  for (int i = 0; i < n; ++i) {
    const aicam_stream_filter& f = host[i];
    for (float v : {f.score_thr, f.iou_thr, f.min_confidence})
      if (!(v >= 0.0f && v <= 1.0f))  // (false for NaN)
        return fail(AICAM_ERR_INVALID_ARG, "frame_table_set_filters: entry " + std::to_string(i) +
                                               ": thresholds must be finite and in [0, 1]");
  }
  t->filters.assign(host, host + n);
  return AICAM_OK;
}

int aicam_frame_table_set_regions(aicam_frame_table* t, const int32_t* indices_host, const aicam_stream_region* host, int n,
                                  void* stream) {
  if (!t || n < 0 || (n > 0 && (!indices_host || !host)))
    return fail(AICAM_ERR_INVALID_ARG, "frame_table_set_regions: null argument or negative count");
  // validated as a whole before anything is stored, allocated or copied
  for (int i = 0; i < n; ++i) {
    const aicam_stream_region& r = host[i];
    const std::string at = "frame_table_set_regions: entry " + std::to_string(i) + ": ";
    if (indices_host[i] < 0 || indices_host[i] >= t->capacity) return fail(AICAM_ERR_INVALID_ARG, at + "index out of range");
    if (r.n_polygons < 0 || r.n_polygons > AICAM_REGION_MAX_POLYGONS)
      return fail(AICAM_ERR_INVALID_ARG, at + "n_polygons must be in 0..8");
    for (int p = 0; p < r.n_polygons; ++p) {
      const std::string pa = at + "polygon " + std::to_string(p) + ": ";
      if (r.kind[p] != 0 && r.kind[p] != 1) return fail(AICAM_ERR_INVALID_ARG, pa + "kind must be 0 (include) or 1 (exclude)");
      if (r.n_vertices[p] < 3 || r.n_vertices[p] > AICAM_COUNT_MAX_VERTICES)
        return fail(AICAM_ERR_INVALID_ARG, pa + "must have 3..32 vertices");
      for (int v = 0; v < r.n_vertices[p]; ++v)
        for (int c = 0; c < 2; ++c)
          if (r.xy[p][v][c] < -AICAM_COUNT_MAX_COORD || r.xy[p][v][c] > AICAM_COUNT_MAX_COORD)
            return fail(AICAM_ERR_INVALID_ARG, pa + "coordinate beyond 2^20");
    }
  }
  if (n == 0) return AICAM_OK;
  AICAM_CUDA_OK(cudaSetDevice(t->device));
  const size_t bytes = static_cast<size_t>(t->capacity) * sizeof(aicam_stream_region);
  if (!t->regions_dev) {
    const size_t keep_bytes = static_cast<size_t>(t->capacity) * (1024 / 8);
    cudaError_t e = cudaMalloc(&t->regions_dev, bytes);
    if (e == cudaSuccess) e = cudaMalloc(&t->region_keep, keep_bytes);
    if (e == cudaSuccess) e = t->region_staging.create(bytes);
    if (e != cudaSuccess) {
      t->region_staging.destroy();
      if (t->regions_dev) cudaFree(t->regions_dev);
      if (t->region_keep) cudaFree(t->region_keep);
      t->regions_dev = nullptr; t->region_keep = nullptr;
      return fail(AICAM_ERR_CUDA, std::string("frame_table_set_regions: ") + cudaGetErrorString(e));
    }
    t->regions.assign(t->capacity, aicam_stream_region{});
  }
  std::vector<aicam_stream_region> next = t->regions;
  bool any = false;
  for (int i = 0; i < n; ++i) {
    next[indices_host[i]] = host[i];
    any |= host[i].n_polygons > 0;
  }
  uint8_t* h = nullptr;
  AICAM_CUDA_OK(t->region_staging.acquire(&h));
  std::memcpy(h, next.data(), bytes);
  AICAM_CUDA_OK(t->region_staging.upload(t->regions_dev, bytes, static_cast<cudaStream_t>(stream)));
  t->regions.swap(next);
  t->region_test |= any;
  return AICAM_OK;
}

const int32_t* aicam_frame_table_present(const aicam_frame_table* t) {
  if (!t) {
    fail(AICAM_ERR_INVALID_ARG, "frame_table_present: null table");
    return nullptr;
  }
  return t->present();
}

}  // extern "C"
