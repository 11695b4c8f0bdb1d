// Frame sources of K1 / K5: where a BGR pixel of a video frame comes from.
//
//   SRC 0  packed BGR uint8 [h][w][3]: what cv2.VideoCapture.read() hands the reference
//          (/root/reference/src/aicamera_tracker.py:170) and what its detect(frame) / update(.., frame) take.
//   SRC 1  NV12 (Y plane [h][w], then interleaved U, V plane [h/2][w]; 1.5 bytes per pixel): what a hardware video
//          decoder emits and what the reference's decoder converts FROM before handing out BGR.  The conversion is
//          OpenCV's COLOR_YUV2BGR_NV12 (ITU-R BT.601, 20-bit fixed point), applied per fetched pixel, so that a kernel
//          reading NV12 produces bit for bit what the same kernel produces from the BGR frame cv2 would have made
//          (oracle/image_ops.py: nv12_to_bgr, verified against cv2 4.13).
#pragma once
#include "common.cuh"

namespace aicam {

__device__ __forceinline__ void yuv_to_bgr_601(int y, int u, int v, int (&bgr)[3]) {
  // OpenCV color_yuv: ITUR_BT_601_CY / CUB / CUG / CVG / CVR, shift 20, rounding constant 1 << 19
  const int yy = max(0, y - 16) * 1220542;
  const int uu = u - 128, vv = v - 128;
  const int b = (yy + (1 << 19) + 2116026 * uu) >> 20;
  const int g = (yy + (1 << 19) - 852492 * vv - 409993 * uu) >> 20;
  const int r = (yy + (1 << 19) + 1673527 * vv) >> 20;
  bgr[0] = min(max(b, 0), 255);
  bgr[1] = min(max(g, 0), 255);
  bgr[2] = min(max(r, 0), 255);
}

template <int SRC>
struct FrameSrc;

template <>
struct FrameSrc<0> {
  const uint8_t* f;  // first byte of the frame
  int h, w;
  static __host__ __device__ long long frame_bytes(int h, int w) { return static_cast<long long>(h) * w * 3; }
  __device__ __forceinline__ void pix(int y, int x, int (&v)[3]) const {
    const uint8_t* s = f + (static_cast<long long>(y) * w + x) * 3;
    v[0] = __ldg(s); v[1] = __ldg(s + 1); v[2] = __ldg(s + 2);
  }
};

template <>
struct FrameSrc<1> {
  const uint8_t* f;
  int h, w;
  static __host__ __device__ long long frame_bytes(int h, int w) { return static_cast<long long>(h) * w * 3 / 2; }
  __device__ __forceinline__ void pix(int y, int x, int (&v)[3]) const {
    const int yy = __ldg(f + static_cast<long long>(y) * w + x);
    const uint8_t* c = f + static_cast<long long>(h) * w + static_cast<long long>(y >> 1) * w + (x & ~1);
    yuv_to_bgr_601(yy, __ldg(c), __ldg(c + 1), v);
  }
};

// Frames of a frame table (frame_table.cuh): rows `pitch` bytes apart, the NV12 chroma plane anywhere.
//   SRC 2  BGR, row y at f + y * pitch
//   SRC 3  NV12, luma row y at f + y * pitch, chroma row y / 2 at c + (y / 2) * pitch
template <>
struct FrameSrc<2> {
  const uint8_t* f;
  int pitch;
  __device__ __forceinline__ void pix(int y, int x, int (&v)[3]) const {
    const uint8_t* s = f + static_cast<long long>(y) * pitch + x * 3;
    v[0] = __ldg(s); v[1] = __ldg(s + 1); v[2] = __ldg(s + 2);
  }
};

template <>
struct FrameSrc<3> {
  const uint8_t* f;
  const uint8_t* c;
  int pitch;
  __device__ __forceinline__ void pix(int y, int x, int (&v)[3]) const {
    const int yy = __ldg(f + static_cast<long long>(y) * pitch + x);
    const uint8_t* cp = c + static_cast<long long>(y >> 1) * pitch + (x & ~1);
    yuv_to_bgr_601(yy, __ldg(cp), __ldg(cp + 1), v);
  }
};

}  // namespace aicam
