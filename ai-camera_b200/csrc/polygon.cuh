// Exact integer point-in-polygon geometry shared by counting (counting.cu) and the per-stream regions of K5
// (reid_crops.cu): doubled coordinates, int64 products, no division, so the device and the oracle (oracle/counting.py,
// oracle/regions.py) agree bit for bit.
#pragma once
#include <stdint.h>

namespace aicam {

constexpr long long ANCHOR_LIMIT = 1ll << 24;  // |anchor coordinate| after clamping: every cross product fits in int64

__device__ __forceinline__ long long clamp_anchor(long long v) {
  return v < -ANCHOR_LIMIT ? -ANCHOR_LIMIT : (v > ANCHOR_LIMIT ? ANCHOR_LIMIT : v);
}

// even-odd rule, half-open edges, doubled coordinates; "strictly left of the edge at py" without division
__device__ inline bool in_zone(const int32_t (*xy)[2], int n, long long px, long long py) {
  bool inside = false;
  for (int i = 0, j = n - 1; i < n; j = i++) {
    const long long xi = 2ll * xy[i][0], yi = 2ll * xy[i][1], xj = 2ll * xy[j][0], yj = 2ll * xy[j][1];
    if ((yi > py) != (yj > py)) {
      const long long dy = yj - yi, lhs = (px - xi) * dy, rhs = (py - yi) * (xj - xi);
      if (dy > 0 ? lhs < rhs : lhs > rhs) inside = !inside;
    }
  }
  return inside;
}

}  // namespace aicam
