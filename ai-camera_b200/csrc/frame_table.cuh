// The device-side frame table (aicam_frame_table_*, csrc/frames.cu): one record per stream that the ragged entry points
// (aicam_preprocess_table, aicam_yolo_detect_table, aicam_reid_crops_table) read on the device, so that one batched step
// can take frames of different sizes, pitches and surface formats.
//
// Device block layout (one cudaMemcpyAsync per aicam_frame_table_set[_present]):
//   int  counts[4]           n, frames on the row-staged K1 path, frames on the per-pixel K1 path, present frames
//   int  lists[2][capacity]  table indices of the present frames of each K1 path, in table order
//   int  present[capacity]   1: frame i is present, 0: absent (and every entry at or past n)
//   FrameRec recs[capacity]
// The present frames are packed to the front of the network batch: present frame i takes slot p(i), the number of present
// frames before it, and the network runs over counts[3] images, a count it reads on the device.  Only the copy of a set
// writes the block, so kernels that read the count before their grid dependency resolves see the step's value.
#pragma once
#include <cuda_runtime.h>

#include <vector>

#include "common.cuh"
#include "staging.cuh"

namespace aicam {

struct FrameRec {
  const uint8_t* data;    // BGR rows of 3w bytes / NV12 luma rows of w bytes, `pitch` bytes apart
  const uint8_t* chroma;  // NV12: interleaved U, V rows of w bytes, `pitch` apart (h / 2 of them); BGR: null
  int h, w, pitch, kind;  // kind 0 BGR, 1 NV12
  // letterbox geometry of K1 (see Geometry in preprocess.cu)
  int mode, staged, new_h, new_w, top, left;
  const int* tab;
  // the un-letterboxing of detect() (scale_bboxes) as the NMS kernel takes it: float(ratio), float(pad_w), float(pad_h)
  float ratio, pad_w, pad_h;
  int crop_staged;        // K5: whole 32-bit words of the frame's planes can be loaded without leaving them
  int slot;               // packed network slot (K1 output, network outputs), -1 when the frame is absent
  // per-entry detection and filter settings (aicam_frame_table_set_filters): when `filt` is 1 the NMS kernel and K5's filter
  // read these instead of the thresholds and class mask passed to the entry points
  int filt;
  float score_thr, iou_thr, min_conf;
  unsigned long long mask_lo, mask_hi;
};

constexpr int FT_COUNTS = 4;

// Dynamic shared memory the row-staged K1 kernel opts in to, and the block-row image of its format 3 (preprocess.cu).
constexpr size_t K1_SMEM_LIMIT = 200 * 1024;
constexpr size_t K1_BLOCK_ROW_IMAGE = static_cast<size_t>(AICAM_YOLO_INPUT / 4) * 128;

__host__ __device__ inline size_t frame_table_recs_offset(int capacity) {
  return (static_cast<size_t>(FT_COUNTS + 3 * capacity) * sizeof(int) + 15) / 16 * 16;
}
__host__ __device__ inline size_t frame_table_bytes(int capacity) {
  return frame_table_recs_offset(capacity) + static_cast<size_t>(capacity) * sizeof(FrameRec);
}

// K1 geometry of a frame size (preprocess.cu; allocates the coefficient table on the first sight of a size)
int k1_geometry(int h, int w, int* decimate, int* mode, int* new_h, int* new_w, int* top, int* left, const int** tab);

}  // namespace aicam

struct aicam_frame_table {
  int device, capacity, max_h, max_w;
  int n;                  // frames set by the last aicam_frame_table_set[_present], absent ones included
  uint8_t* dev;           // the device block
  aicam::PinnedStaging staging;
  std::vector<aicam_stream_filter> filters;  // of aicam_frame_table_set_filters: entry i < size() carries filters[i]
  // aicam_frame_table_set_regions, allocated by its first call: the host copy of the region block, the device block
  // (capacity records), its own staging (the block is ~2 KB per entry, far larger than the records), and K5's scratch of
  // the region test, one keep bit per detection (capacity x 1024 bits)
  std::vector<aicam_stream_region> regions;
  aicam_stream_region* regions_dev = nullptr;
  unsigned* region_keep = nullptr;
  aicam::PinnedStaging region_staging;
  bool region_test = false;  // some entry has had polygons: aicam_reid_crops_table launches the region test

  const int* counts() const { return reinterpret_cast<const int*>(dev); }
  const int* lists() const { return reinterpret_cast<const int*>(dev) + aicam::FT_COUNTS; }
  const int* present() const { return lists() + 2 * capacity; }
  const aicam::FrameRec* recs() const { return reinterpret_cast<const aicam::FrameRec*>(dev + aicam::frame_table_recs_offset(capacity)); }
  // One row slot of the row-staged K1 ring: the longest staged source row (a BGR row of max_w pixels; an NV12 luma + chroma
  // row is shorter), rounded up to 16 bytes so that every slot, and the format-3 image behind the ring, is a valid 16-byte
  // aligned bulk-copy destination whatever the bound.
  int stage_row() const { return (3 * max_w + 15) / 16 * 16; }
  // Whether the ring fits: its largest configuration is two stages of two rows plus the format-3 image (four stages are
  // used only when they take at most half of the limit).
  bool ring_fits() const { return 4 * static_cast<size_t>(stage_row()) + aicam::K1_BLOCK_ROW_IMAGE <= aicam::K1_SMEM_LIMIT; }
};
