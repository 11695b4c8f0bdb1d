// Pinned host staging of the small host-side set calls (aicam_frame_table_set[_present], aicam_tracker_set_stream_assoc):
// two buffers used alternately, each guarded by an event recorded after the copy out of it, so that a call fills one
// buffer while the previous call's copy may still be in flight and waits only for the copy out of the buffer it reuses.
// Every upload is one cudaMemcpyAsync.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace aicam {

struct PinnedStaging {
  uint8_t* host[2] = {nullptr, nullptr};
  cudaEvent_t done[2] = {nullptr, nullptr};
  int next = 0;

  cudaError_t create(size_t bytes) {
    cudaError_t e = cudaSuccess;
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) e = cudaMallocHost(&host[i], bytes);
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) e = cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming);
    return e;
  }
  void destroy() {
    for (int i = 0; i < 2; ++i) {
      if (done[i]) cudaEventSynchronize(done[i]), cudaEventDestroy(done[i]);
      if (host[i]) cudaFreeHost(host[i]);
      done[i] = nullptr; host[i] = nullptr;
    }
  }
  // the buffer the next upload copies from, once the copy out of it has completed
  cudaError_t acquire(uint8_t** out) {
    *out = host[next];
    return cudaEventSynchronize(done[next]);
  }
  // the first `bytes` of the acquired buffer to `dst` on `st`
  cudaError_t upload(void* dst, size_t bytes, cudaStream_t st) {
    cudaError_t e = cudaMemcpyAsync(dst, host[next], bytes, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaEventRecord(done[next], st);
    if (e == cudaSuccess) next ^= 1;
    return e;
  }
};

}  // namespace aicam
