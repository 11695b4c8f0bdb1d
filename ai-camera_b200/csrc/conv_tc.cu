// Implicit-GEMM convolution (+bias, SiLU/ReLU, residual) on tcgen05 tensor cores, sm_100a.
//
// This is the operator behind every Conv+BN+SiLU / C2f / SPPF / Detect layer of YOLOv8 and
// every BasicBlock of the DeepSORT ReID net - the work the reference hands to a TensorRT
// engine (/root/reference/src/trt_utils/trt_engine.py:191, called from
// src/detector/yolo_detector.py:97 and src/tracker/reid_model.py:115).
//
// GEMM view:  D[m][n] = sum_k A[m][k] * B[n][k]
//   m = output pixel (batch, oy, ox) flattened            tile M = 128 (one UMMA, cta_group::1)
//   n = output channel                                    tile N = n_tile (16..128, divides cout_pad)
//   k = (tap, input channel)                              staged 64 at a time (8 x 16-byte chunks)
// Operands are bf16, accumulation is fp32 in TMEM.  Both operands sit in shared memory in the
// canonical K-major NO-SWIZZLE UMMA layout: 8-row x 16-byte core matrices, rows of one chunk
// contiguous:  addr(row, chunk) = chunk * (ROWS*16) + row*16   (SBO = 128 B, LBO = ROWS*16 B).
//
// Warp roles (192 threads):
//   warps 0-3  im2col gather: thread t owns output pixel m0+t and cp.async's its 16-byte
//              channel chunks (zero-filled outside the image) straight into the UMMA layout and
//              signals the stage with cp.async.mbarrier.arrive.noinc (no wait in the thread);
//              afterwards the same warps run the epilogue (TMEM -> registers -> bias/act/
//              residual -> bf16/fp32 NHWC stores); warp w reads TMEM lanes 32w..32w+31.
//   warp 4     allocates TMEM, issues tcgen05.mma (one elected lane), commits to mbarriers.
//   warp 5     streams the packed weights with cp.async.bulk (1-D bulk copy, mbarrier tx).
// Pipeline: 3 shared-memory stages, full/empty mbarriers.  The kernel is persistent: up to 3 CTAs
// per SM each loop over output tiles (TMEM allocation and barrier set-up are paid once; one CTA's
// epilogue overlaps another's main loop); the tile count may come from a device-side batch count.
#include "conv_tc.cuh"

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

namespace aicam {

namespace {

constexpr int TILE_M = 128;
constexpr int STAGES = 3;
constexpr int CHUNKS_PER_STAGE = 8;                 // 8 x 16 B = 64 bf16 of K per stage
// LBO of A: 128 rows x 16 B plus one 16-byte pad, so that the 8 lanes that copy the 8 chunks of
// one pixel (consecutive channels, one 128-byte line) hit 8 different bank groups
constexpr int A_CHUNK_BYTES = TILE_M * 16 + 16;
constexpr int A_STAGE_BYTES = A_CHUNK_BYTES * CHUNKS_PER_STAGE;  // 16.1 KiB
constexpr int SMEM_HEADER = 1024;  // 256 B of barriers + 512 B of per-tile bias (n_tile <= 128 floats)
constexpr int BIAS_OFFSET = 256;
constexpr int NUM_THREADS = 192;

struct ConvKernelArgs {
  const __nv_bfloat16* in;
  long long in_img_stride;
  int in_cstride, in_coff;
  int h, w, ho, wo, howo, m_total;
  int ksize, stride, pad;
  int cin_chunks;   // cin_pad / 8 (0 in stem mode)
  int stem;         // 1: cin_pad == 4, a chunk is two taps of 4 channels
  int taps;
  int q, q_pad;     // real / padded number of 16-byte K chunks
  const __nv_bfloat16* wgt;
  const float* bias;
  int cout, cout_pad, n_tile;
  void* out;
  long long out_img_stride;
  int out_cstride, out_coff, out_f32;
  const __nv_bfloat16* res;
  long long res_img_stride;
  int res_cstride, res_coff, res_mode;
  int act;
  uint32_t idesc;
  uint32_t tmem_cols;
  const int* batch_dev;  // optional: images actually present (device), m_total is the capacity
  int staged;            // 1: epilogue goes through the coalescing shared-memory staging path
  int out_dense, res_dense;  // 1: pixel address = m * cstride (images are contiguous in the buffer)
  int res_stage_off;     // byte offset of the residual staging area in shared memory (0: none)
  long long* trace;      // optional debug buffer: clock64 stamps of CTA 0 (conv2d_bench with AICAM_CONV_TRACE)
};

// ---- PTX wrappers ----------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait with back-off: waiting warps must not steal issue slots from the gather and
// epilogue warps (the kernel is issue-bound), and a protocol bug traps instead of hanging.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  uint32_t spin = 0;
  while (!mbar_try_wait(bar, parity)) {
    __nanosleep(spin < 8 ? 32 : 128);
    if (++spin > (1u << 24)) {
      printf("aicam conv: mbarrier timeout block %d thread %d bar %u parity %u\n", blockIdx.x, threadIdx.x, bar,
             parity);
      __trap();
    }
  }
}
__device__ __forceinline__ void cp_async_16(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_8(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_arrive_noinc(uint32_t bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// K-major: start >> 4 | LBO >> 4 (bits 16..29) | SBO >> 4 (bits 32..45) | version 1 (bit 46)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = static_cast<uint64_t>((addr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= 1ull << 46;
  return d;
}

__device__ __forceinline__ float apply_act(float x, int act) {
  if (act == 1) return x * __frcp_rn(1.0f + __expf(-x));
  if (act == 2) return fmaxf(x, 0.0f);
  return x;
}

__global__ void __launch_bounds__(NUM_THREADS, 3) conv_tc_kernel(const ConvKernelArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t bar_full = smem_base;            // STAGES x 8 B
  const uint32_t bar_empty = smem_base + 64;      // STAGES x 8 B
  const uint32_t bar_tmem_full = smem_base + 128;
  const uint32_t bar_tmem_empty = smem_base + 136;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(smem + 160);
  const uint32_t smem_a = smem_base + SMEM_HEADER;
  const uint32_t b_stage_bytes = static_cast<uint32_t>(a.n_tile) * 16u * CHUNKS_PER_STAGE;
  const uint32_t smem_b = smem_a + STAGES * A_STAGE_BYTES;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_kb = (a.q_pad + CHUNKS_PER_STAGE - 1) / CHUNKS_PER_STAGE;
  int m_total = a.m_total;
  if (a.batch_dev) m_total = min(m_total, __ldg(a.batch_dev) * a.howo);
  const int n_tiles = a.cout_pad / a.n_tile;
  const int total_tiles = ((m_total + TILE_M - 1) / TILE_M) * n_tiles;
  if (static_cast<int>(blockIdx.x) >= total_tiles) return;  // whole CTA: nothing to do

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(bar_full + 8 * s, TILE_M + 1);  // 128 gather threads + the weight loader's expect_tx
      mbar_init(bar_empty + 8 * s, 1);          // one tcgen05.commit
    }
    mbar_init(bar_tmem_full, 1);
    mbar_init(bar_tmem_empty, TILE_M);          // the 128 epilogue threads
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 4) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)),
                 "r"(a.tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  // Persistent loop: CTA b processes tiles b, b + gridDim.x, ...  (n-tile index fastest, so the
  // CTAs that share an A tile run close together).  Pipeline stage/phase counters run on
  // across tiles: g_kb counts K-blocks since kernel start.
  if (warp < 4) {
    const int j = threadIdx.x & 7;    // chunk slot within a K-block
    const int r0 = threadIdx.x >> 3;  // rows r0 + 16 i, i < 8
    const uint32_t dst_thread = j * A_CHUNK_BYTES + r0 * 16;
    const int row = threadIdx.x;      // epilogue: TMEM lane == tile row
    const uint32_t taddr_row = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
    const int esize = a.out_f32 ? 4 : 2;
    const uint32_t pitch = a.n_tile * esize + 16;  // staging row pitch (bytes), conflict-free
    uint8_t* stage_w = smem + SMEM_HEADER + static_cast<size_t>(warp) * 32 * pitch;
    uint8_t* my_stage = stage_w + static_cast<size_t>(lane) * pitch;
    const bool fast = a.staged != 0;
    const int cs_bytes = a.in_cstride * 2;
    float* bias_s = reinterpret_cast<float*>(smem + BIAS_OFFSET);
    const bool res_pref = fast && a.res_mode != 0 && a.res_dense != 0;  // residual tile fetched by cp.async
    const uint32_t rpitch = pitch;                   // residual rows live in the output staging rows
    uint8_t* res_stage = smem + SMEM_HEADER;
    int g_kb = 0;
    int t_iter = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++t_iter) {
      const int m_blk = tile / n_tiles;
      const int n0 = (tile - m_blk * n_tiles) * a.n_tile;
      const int m0 = m_blk * TILE_M;
      if (threadIdx.x < a.n_tile) bias_s[threadIdx.x] = __ldg(a.bias + n0 + threadIdx.x);
      // ---------------------------------------------------------------- im2col gather
      // Thread t copies chunk slot j of every K-block for its 8 rows: the 8 lanes of a quarter
      // warp read the 8 consecutive 16-byte channel chunks of ONE pixel (one 128-byte line).
      // Per row: a byte pointer to tap (0,0) and a 9-bit mask of the taps that are inside the
      // image, so that one copy costs an add, a bit test and two selects.
      const uint8_t* rowptr[8];
      uint32_t tmask[8];
      {
        int m = m0 + r0;
        int n_img = m / a.howo;
        int rem = m - n_img * a.howo;
        int oy = rem / a.wo;
        int ox = rem - oy * a.wo;
  #pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int iy0 = oy * a.stride - a.pad, ix0 = ox * a.stride - a.pad;
          // taps inside the image: 3-bit column mask replicated into the valid filter rows
          uint32_t mk = 0;
          if (m < m_total) {
            uint32_t xm = 0;
  #pragma unroll
            for (int tc = 0; tc < 3; ++tc)
              if (tc < a.ksize && static_cast<unsigned>(ix0 + tc) < static_cast<unsigned>(a.w)) xm |= 1u << tc;
  #pragma unroll
            for (int tr = 0; tr < 3; ++tr)
              if (tr < a.ksize && static_cast<unsigned>(iy0 + tr) < static_cast<unsigned>(a.h)) mk |= xm << (tr * a.ksize);
          }
          tmask[i] = mk;
          rowptr[i] = reinterpret_cast<const uint8_t*>(a.in + a.in_coff) +
                      (static_cast<long long>(n_img) * a.h * a.w + static_cast<long long>(iy0) * a.w + ix0) * cs_bytes;
          // advance 16 output pixels
          m += 16;
          ox += 16;
          while (ox >= a.wo) { ox -= a.wo; if (++oy == a.ho) { oy = 0; ++n_img; } }
        }
      }
      // running position of chunk q = kb * 8 + j in (tap, channel chunk) space
      int tap = 0, tr = 0, tc = 0, c8 = 0;
      if (!a.stem) {
        c8 = j;
        while (c8 >= a.cin_chunks) { c8 -= a.cin_chunks; ++tap; if (++tc == a.ksize) { tc = 0; ++tr; } }
      }
      for (int kb = 0; kb < num_kb; ++kb, ++g_kb) {
        const int s = g_kb % STAGES;
        const int it = g_kb / STAGES;
        mbar_wait(bar_empty + 8 * s, (it & 1) ^ 1);
        if (a.trace && blockIdx.x == 0 && threadIdx.x == 0 && g_kb < 60) a.trace[g_kb * 4 + 0] = clock64();
        const uint32_t dst = smem_a + s * A_STAGE_BYTES + dst_thread;
        const int q = kb * CHUNKS_PER_STAGE + j;
        if (q < a.q_pad) {
          if (!a.stem) {
            const uint32_t bit = (q < a.q) ? (1u << tap) : 0u;
            const int delta = (tr * a.w + tc) * cs_bytes + c8 * 16;
  #pragma unroll
            for (int i = 0; i < 8; ++i) {
              const bool ok = (tmask[i] & bit) != 0;
              const uint8_t* src = ok ? rowptr[i] + delta : reinterpret_cast<const uint8_t*>(a.in);
              cp_async_16(dst + i * 256, src, ok ? 16u : 0u);
            }
            c8 += CHUNKS_PER_STAGE;
            while (c8 >= a.cin_chunks) { c8 -= a.cin_chunks; ++tap; if (++tc == a.ksize) { tc = 0; ++tr; } }
          } else {
  #pragma unroll
            for (int half = 0; half < 2; ++half) {
              const int tp = 2 * q + half;
              const int ttr = tp / 3, ttc = tp - ttr * 3;  // the stem is always 3x3
              const uint32_t bit = (tp < a.taps) ? (1u << tp) : 0u;
              const int delta = (ttr * a.w + ttc) * cs_bytes;
  #pragma unroll
              for (int i = 0; i < 8; ++i) {
                const bool ok = (tmask[i] & bit) != 0;
                const uint8_t* src = ok ? rowptr[i] + delta : reinterpret_cast<const uint8_t*>(a.in);
                cp_async_8(dst + i * 256 + half * 8, src, ok ? 8u : 0u);
              }
            }
          }
        }
        // Arrive on the stage's full barrier when this thread's copies have landed (asynchronous).
        cp_async_arrive_noinc(bar_full + 8 * s);
        if (a.trace && blockIdx.x == 0 && threadIdx.x == 0 && g_kb < 60) a.trace[g_kb * 4 + 1] = clock64();
      }
      const int ncols = min(a.n_tile, a.cout - n0);  // valid output channels of this tile
      // ---------------------------------------------------------------- epilogue
      // TMEM -> registers (thread = row) -> bias / residual / activation -> shared-memory staging
      // (the A stages are free once the accumulator is complete) -> coalesced 16-byte stores.
      mbar_wait(bar_tmem_full, t_iter & 1);
      tc_fence_after();
      if (res_pref) {
        // Residual tile -> staging rows (the A stages are free now): 16-byte chunks, lanes on
        // consecutive chunks of one row (coalesced), all copies of the tile in flight at once;
        // dense tensor => pixel address = m * cstride.
        const int rcpr = (ncols * 2) >> 4;
        int cp2 = 2;
        while (cp2 < rcpr) cp2 <<= 1;               // chunks per row rounded up to a power of two
        const int ch = threadIdx.x & (cp2 - 1);
        const int rstep = TILE_M / cp2;
        for (int rr = threadIdx.x / cp2; rr < TILE_M; rr += rstep) {
          const int mm = m0 + rr;
          if (ch < rcpr && mm < m_total)
            cp_async_16(smem_u32(res_stage + static_cast<size_t>(rr) * rpitch + ch * 16),
                        a.res + static_cast<long long>(mm) * a.res_cstride + a.res_coff + n0 + ch * 8, 16u);
        }
        asm volatile("cp.async.wait_all;" ::: "memory");
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");   // bias_s and the residual tile are visible
      if (a.trace && blockIdx.x == 0 && threadIdx.x == 0 && t_iter < 8) a.trace[240 + t_iter * 4 + 0] = clock64();
      const int m = m0 + row;
      const bool valid = m < m_total;
      long long out_pix, res_pix;
      if (a.out_dense && (a.res_dense || a.res_mode == 0)) {
        out_pix = static_cast<long long>(m) * a.out_cstride + a.out_coff + n0;
        res_pix = static_cast<long long>(m) * a.res_cstride + a.res_coff + n0;
      } else {
        int n_img = 0, rem = 0;
        if (valid) { n_img = m / a.howo; rem = m - n_img * a.howo; }
        out_pix = static_cast<long long>(n_img) * a.out_img_stride + static_cast<long long>(rem) * a.out_cstride +
                  a.out_coff + n0;
        res_pix = static_cast<long long>(n_img) * a.res_img_stride + static_cast<long long>(rem) * a.res_cstride +
                  a.res_coff + n0;
      }
      const int cpr = (ncols * esize) >> 4;          // 16-byte chunks per output row (fast path)
      const uint8_t* my_res = my_stage;
      if (fast && a.res_mode != 0 && !res_pref) {
        const int rcpr = (ncols * 2) >> 4;
        for (int idx = lane; idx < 32 * rcpr; idx += 32) {
          const int rr = idx / rcpr, ch = idx - rr * rcpr;
          const long long rp = __shfl_sync(0xffffffffu, res_pix, rr);
          const int rv = __shfl_sync(0xffffffffu, static_cast<int>(valid), rr);
          if (rv) {
            const uint4 v = __ldg(reinterpret_cast<const uint4*>(a.res + rp) + ch);
            *reinterpret_cast<uint4*>(stage_w + static_cast<size_t>(rr) * pitch + ch * 16) = v;
          }
        }
        __syncwarp();
      }
      for (int c0 = 0; c0 < a.n_tile; c0 += 16) {
        uint32_t v[16];
        tc_ld16(taddr_row + c0, v);
        const int cvalid = min(16, a.cout - (n0 + c0));  // <= 0 when the group is channel padding
        if (!valid || cvalid <= 0) continue;
        float x[16];
        const float4* bp = reinterpret_cast<const float4*>(bias_s + c0);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 b4 = bp[i];
          x[4 * i] = __uint_as_float(v[4 * i]) + b4.x;
          x[4 * i + 1] = __uint_as_float(v[4 * i + 1]) + b4.y;
          x[4 * i + 2] = __uint_as_float(v[4 * i + 2]) + b4.z;
          x[4 * i + 3] = __uint_as_float(v[4 * i + 3]) + b4.w;
        }
        float r[16];
        if (a.res_mode != 0) {
          if (fast) {
            const uint4 q0 = *reinterpret_cast<const uint4*>(my_res + c0 * 2);
            const uint4 q1 = *reinterpret_cast<const uint4*>(my_res + c0 * 2 + 16);
            const uint32_t rw[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i) { r[2 * i] = bf16_lo(rw[i]); r[2 * i + 1] = bf16_hi(rw[i]); }
          } else {
            const __nv_bfloat16* rp = a.res + res_pix + c0;
#pragma unroll
            for (int i = 0; i < 16; ++i) r[i] = i < cvalid ? __bfloat162float(rp[i]) : 0.0f;
          }
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          if (a.res_mode == 2) x[i] += r[i];
          x[i] = apply_act(x[i], a.act);
          if (a.res_mode == 1) x[i] += r[i];
        }
        if (fast) {
          if (a.out_f32) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
              *reinterpret_cast<float4*>(my_stage + c0 * 4 + i * 16) =
                  make_float4(x[4 * i], x[4 * i + 1], x[4 * i + 2], x[4 * i + 3]);
          } else {
            uint4 o0, o1;
            o0.x = pack_bf16x2(x[0], x[1]);   o0.y = pack_bf16x2(x[2], x[3]);
            o0.z = pack_bf16x2(x[4], x[5]);   o0.w = pack_bf16x2(x[6], x[7]);
            o1.x = pack_bf16x2(x[8], x[9]);   o1.y = pack_bf16x2(x[10], x[11]);
            o1.z = pack_bf16x2(x[12], x[13]); o1.w = pack_bf16x2(x[14], x[15]);
            *reinterpret_cast<uint4*>(my_stage + c0 * 2) = o0;
            *reinterpret_cast<uint4*>(my_stage + c0 * 2 + 16) = o1;
          }
        } else if (a.out_f32) {
          float* op = reinterpret_cast<float*>(a.out) + out_pix + c0;
          for (int i = 0; i < cvalid; ++i) op[i] = x[i];
        } else {
          __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(a.out) + out_pix + c0;
          for (int i = 0; i < cvalid; ++i) op[i] = __float2bfloat16_rn(x[i]);
        }
      }
      // the accumulator has been read: the MMA warp may start the next tile
      tc_fence_before();
      mbar_arrive(bar_tmem_empty);
      if (a.trace && blockIdx.x == 0 && threadIdx.x == 0 && t_iter < 8) a.trace[240 + t_iter * 4 + 1] = clock64();
      if (fast) {
        __syncwarp();
        uint8_t* out_bytes = reinterpret_cast<uint8_t*>(a.out);
        int cp2 = 1;
        while (cp2 < cpr) cp2 <<= 1;                 // chunks per row rounded up to a power of two (<= 32)
        const int ch = lane & (cp2 - 1);
        const int rstep = 32 / cp2;
        for (int rr = lane / cp2; rr < 32; rr += rstep) {
          const long long op = __shfl_sync(0xffffffffu, out_pix, rr);
          const int rv = __shfl_sync(0xffffffffu, static_cast<int>(valid), rr);
          if (rv && ch < cpr) {
            const uint4 v = *reinterpret_cast<const uint4*>(stage_w + static_cast<size_t>(rr) * pitch + ch * 16);
            *reinterpret_cast<uint4*>(out_bytes + op * esize + ch * 16) = v;
          }
        }
      }
      // staging rows alias the A stages, bias_s / res_stage are rewritten by the next tile
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (a.trace && blockIdx.x == 0 && threadIdx.x == 0 && t_iter < 8) a.trace[240 + t_iter * 4 + 2] = clock64();
    }
  } else if (warp == 4) {
    // ------------------------------------------------------------------ MMA issuer
    const uint32_t b_chunk_bytes = static_cast<uint32_t>(a.n_tile) * 16u;
    int g_kb = 0, t_iter = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++t_iter) {
      mbar_wait(bar_tmem_empty, (t_iter & 1) ^ 1);  // epilogue of the previous tile has drained TMEM
      tc_fence_after();
      for (int kb = 0; kb < num_kb; ++kb, ++g_kb) {
        const int s = g_kb % STAGES;
        const int it = g_kb / STAGES;
        mbar_wait(bar_full + 8 * s, it & 1);
        tc_fence_after();
        if (a.trace && blockIdx.x == 0 && lane == 0 && g_kb < 60) a.trace[g_kb * 4 + 2] = clock64();
        if (lane == 0) {
          const int nchunks = min(CHUNKS_PER_STAGE, a.q_pad - kb * CHUNKS_PER_STAGE);
          const uint32_t a_stage = smem_a + s * A_STAGE_BYTES;
          const uint32_t b_stage = smem_b + s * b_stage_bytes;
          for (int kk = 0; kk < nchunks / 2; ++kk) {
            const uint64_t da = make_smem_desc(a_stage + kk * 2 * A_CHUNK_BYTES, A_CHUNK_BYTES, 128);
            const uint64_t db = make_smem_desc(b_stage + kk * 2 * b_chunk_bytes, b_chunk_bytes, 128);
            tc_mma_bf16(tmem_base, da, db, a.idesc, (kb | kk) != 0 ? 1u : 0u);
          }
          tc_commit(bar_empty + 8 * s);
          if (kb == num_kb - 1) tc_commit(bar_tmem_full);
          if (a.trace && blockIdx.x == 0 && g_kb < 60) a.trace[g_kb * 4 + 3] = clock64();
        }
        __syncwarp();
      }
    }
    tc_fence_before();
  } else {
    // ------------------------------------------------------------------ weight loader
    if (lane == 0) {
      const uint32_t b_chunk_bytes = static_cast<uint32_t>(a.n_tile) * 16u;
      int g_kb = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int n0 = (tile % n_tiles) * a.n_tile;
        for (int kb = 0; kb < num_kb; ++kb, ++g_kb) {
          const int s = g_kb % STAGES;
          const int it = g_kb / STAGES;
          mbar_wait(bar_empty + 8 * s, (it & 1) ^ 1);
          const int nchunks = min(CHUNKS_PER_STAGE, a.q_pad - kb * CHUNKS_PER_STAGE);
          const uint32_t bar = bar_full + 8 * s;
          const uint32_t dst = smem_b + s * b_stage_bytes;
          mbar_arrive_expect_tx(bar, nchunks * b_chunk_bytes);
          const __nv_bfloat16* src = a.wgt + (static_cast<long long>(kb) * CHUNKS_PER_STAGE * a.cout_pad + n0) * 8;
          if (a.n_tile == a.cout_pad) {
            bulk_g2s(dst, src, nchunks * b_chunk_bytes, bar);
          } else {
            for (int jj = 0; jj < nchunks; ++jj)
              bulk_g2s(dst + jj * b_chunk_bytes, src + static_cast<long long>(jj) * a.cout_pad * 8, b_chunk_bytes, bar);
          }
        }
      }
    }
  }
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(a.tmem_cols) : "memory");
  }
}

inline uint16_t f32_to_bf16_bits(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return static_cast<uint16_t>((u >> 16) | 0x40);
  u += 0x7fffu + ((u >> 16) & 1u);
  return static_cast<uint16_t>(u >> 16);
}

int pick_n_tile(int cout_pad, bool out_f32) {
  // fp32 outputs are staged at 4 bytes per element: keep 128 rows x (n_tile*4 + 16) within the A stages
  for (int nt = out_f32 ? 80 : 128; nt >= 16; nt -= 16)
    if (cout_pad % nt == 0) return nt;
  return 16;
}

}  // namespace

extern void count_launch();
int try_launch_conv_win(const PackedConv& pc, const ConvLaunch& L, cudaStream_t stream);
bool profile_begin(cudaStream_t st, size_t* slot);
void profile_end(cudaStream_t st, size_t slot);

int pack_conv_weights(const float* w, const float* bias, int cout, int cin, int ksize, int stride,
                      PackedConv* out) {
  if (cout <= 0 || cin <= 0 || (ksize != 1 && ksize != 3) || (stride != 1 && stride != 2))
    return fail(AICAM_ERR_INVALID_ARG, "pack_conv_weights: unsupported convolution shape");
  const int taps = ksize * ksize;
  const bool stem = cin <= 4;
  const int cin_pad = stem ? 4 : (cin + 7) / 8 * 8;
  const int k_total = taps * cin_pad;
  const int q = (k_total + 7) / 8;
  const int q_pad = (q + 1) / 2 * 2;
  const int cout_pad = (cout + 15) / 16 * 16;
  std::vector<uint16_t> packed(static_cast<size_t>(q_pad) * cout_pad * 8, 0);
  for (int o = 0; o < cout; ++o)
    for (int t = 0; t < taps; ++t)
      for (int c = 0; c < cin; ++c) {
        const int k = t * cin_pad + c;
        const float v = w[(static_cast<size_t>(o) * cin + c) * taps + t];
        packed[(static_cast<size_t>(k / 8) * cout_pad + o) * 8 + (k % 8)] = f32_to_bf16_bits(v);
      }
  std::vector<float> b(cout_pad, 0.0f);
  for (int o = 0; o < cout; ++o) b[o] = bias ? bias[o] : 0.0f;
  PackedConv p;
  p.cin = cin; p.cin_pad = cin_pad; p.cout = cout; p.ksize = ksize; p.stride = stride; p.q = q; p.q_pad = q_pad;
  AICAM_CUDA_OK(cudaMalloc(&p.w, packed.size() * 2));
  AICAM_CUDA_OK(cudaMalloc(&p.bias, b.size() * 4));
  AICAM_CUDA_OK(cudaMemcpy(p.w, packed.data(), packed.size() * 2, cudaMemcpyHostToDevice));
  AICAM_CUDA_OK(cudaMemcpy(p.bias, b.data(), b.size() * 4, cudaMemcpyHostToDevice));
  p.bias_host = static_cast<float*>(std::malloc(b.size() * 4));
  if (p.bias_host) std::memcpy(p.bias_host, b.data(), b.size() * 4);
  const int nb = cout_pad % 256 == 0 ? 256 : pick_n_tile(cout_pad, false);  // (conv_win.cu takes 256-column tiles when it can)
  if (nb < cout_pad) {  // n-tile-major copy for the streamed-weight window kernel
    std::vector<uint16_t> nt(packed.size());
    for (int qq = 0; qq < q_pad; ++qq)
      for (int o = 0; o < cout_pad; ++o)
        std::memcpy(&nt[((static_cast<size_t>(o / nb) * q_pad + qq) * nb + o % nb) * 8],
                    &packed[(static_cast<size_t>(qq) * cout_pad + o) * 8], 16);
    AICAM_CUDA_OK(cudaMalloc(&p.w_nt, nt.size() * 2));
    AICAM_CUDA_OK(cudaMemcpy(p.w_nt, nt.data(), nt.size() * 2, cudaMemcpyHostToDevice));
    p.nt_block = nb;
  }
  *out = p;
  return AICAM_OK;
}

int pack_conv_weights_s2d(const float* w, const float* bias, int cout, int cin, int c0_pad, PackedConv* out) {
  if (cout <= 0 || cin <= 0 || cin > c0_pad || (c0_pad != 4 && c0_pad != 16))
    return fail(AICAM_ERR_INVALID_ARG, "pack_conv_weights_s2d: unsupported shape");
  // output (oy, ox) reads input (2 oy - 1 + ky, 2 ox - 1 + kx): block row oy - 1 + ty, row parity sy with
  // ky = 0 -> (ty 0, sy 1), ky = 1 -> (ty 1, sy 0), ky = 2 -> (ty 1, sy 1); same along x
  const int cin_pad = 4 * c0_pad;
  const int k_total = 4 * cin_pad;
  const int q = k_total / 8;
  const int cout_pad = (cout + 15) / 16 * 16;
  std::vector<uint16_t> packed(static_cast<size_t>(q) * cout_pad * 8, 0);
  const int t_of[3] = {0, 1, 1}, s_of[3] = {1, 0, 1};
  for (int o = 0; o < cout; ++o)
    for (int ky = 0; ky < 3; ++ky)
      for (int kx = 0; kx < 3; ++kx)
        for (int c = 0; c < cin; ++c) {
          const int tap2 = t_of[ky] * 2 + t_of[kx];
          const int k = tap2 * cin_pad + (s_of[ky] * 2 + s_of[kx]) * c0_pad + c;
          const float v = w[(static_cast<size_t>(o) * cin + c) * 9 + ky * 3 + kx];
          packed[(static_cast<size_t>(k / 8) * cout_pad + o) * 8 + (k % 8)] = f32_to_bf16_bits(v);
        }
  std::vector<float> b(cout_pad, 0.0f);
  for (int o = 0; o < cout; ++o) b[o] = bias ? bias[o] : 0.0f;
  PackedConv p;
  p.cin = cin; p.cin_pad = cin_pad; p.cout = cout; p.ksize = 2; p.stride = 1; p.q = q; p.q_pad = q; p.s2d_c0 = c0_pad;
  AICAM_CUDA_OK(cudaMalloc(&p.w, packed.size() * 2));
  AICAM_CUDA_OK(cudaMalloc(&p.bias, b.size() * 4));
  AICAM_CUDA_OK(cudaMemcpy(p.w, packed.data(), packed.size() * 2, cudaMemcpyHostToDevice));
  AICAM_CUDA_OK(cudaMemcpy(p.bias, b.data(), b.size() * 4, cudaMemcpyHostToDevice));
  p.bias_host = static_cast<float*>(std::malloc(b.size() * 4));
  if (p.bias_host) std::memcpy(p.bias_host, b.data(), b.size() * 4);
  *out = p;
  return AICAM_OK;
}

void free_packed_conv(PackedConv* p) {
  if (p->w) cudaFree(p->w);
  if (p->bias) cudaFree(p->bias);
  if (p->w_nt) cudaFree(p->w_nt);
  if (p->w_pair) cudaFree(p->w_pair);
  std::free(p->bias_host);
  p->bias_host = nullptr;
  p->w_nt = nullptr;
  p->w_pair = nullptr;
  p->w = nullptr;
  p->bias = nullptr;
}

int launch_conv(const PackedConv& pc, const ConvLaunch& L, cudaStream_t stream) {
  if (pc.s2d_c0) {  // space-to-depth layers exist only on the window kernel
    if (L.batch <= 0) return AICAM_OK;
    const int wrc = try_launch_conv_win(pc, L, stream);
    if (wrc < 0) return wrc;
    return wrc == 1 ? AICAM_OK : fail(AICAM_ERR_UNSUPPORTED, "launch_conv: space-to-depth layer not eligible for the window kernel");
  }
  if (L.in_pad || L.out_pad) {  // zero-bordered tensors exist only on the window kernel
    if (L.batch <= 0) return AICAM_OK;
    const int wrc = try_launch_conv_win(pc, L, stream);
    if (wrc < 0) return wrc;
    return wrc == 1 ? AICAM_OK : fail(AICAM_ERR_UNSUPPORTED, "launch_conv: padded layer not eligible for the window kernel");
  }
  ConvKernelArgs a;
  a.in = L.in; a.in_img_stride = L.in_img_stride; a.in_cstride = L.in_cstride; a.in_coff = L.in_coff;
  a.h = L.h; a.w = L.w; a.ho = L.ho; a.wo = L.wo; a.howo = L.ho * L.wo;
  a.m_total = L.batch * a.howo;
  a.ksize = pc.ksize; a.stride = pc.stride; a.pad = pc.ksize / 2;
  a.stem = pc.cin_pad == 4 ? 1 : 0;
  a.cin_chunks = a.stem ? 0 : pc.cin_pad / 8;
  a.taps = pc.ksize * pc.ksize;
  a.q = pc.q; a.q_pad = pc.q_pad;
  a.wgt = pc.w; a.bias = pc.bias;
  a.cout = pc.cout; a.cout_pad = (pc.cout + 15) / 16 * 16;
  a.n_tile = pick_n_tile(a.cout_pad, L.out_f32 != 0);
  a.out = L.out; a.out_img_stride = L.out_img_stride; a.out_cstride = L.out_cstride; a.out_coff = L.out_coff;
  a.out_f32 = L.out_f32;
  a.res = L.res; a.res_img_stride = L.res_img_stride; a.res_cstride = L.res_cstride; a.res_coff = L.res_coff;
  a.res_mode = L.res ? L.res_mode : 0;
  a.act = L.act;
  a.batch_dev = L.batch_dev;
  a.trace = L.trace;
  // instruction descriptor: fp32 accumulate, bf16 A/B, both K-major, N = n_tile, M = 128
  a.idesc = (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(a.n_tile >> 3) << 17) |
            (static_cast<uint32_t>(TILE_M >> 4) << 24);
  uint32_t cols = 32;
  while (cols < static_cast<uint32_t>(a.n_tile)) cols <<= 1;
  a.tmem_cols = cols;
  if (a.m_total <= 0) return AICAM_OK;
  if (L.in_img_stride != static_cast<long long>(L.h) * L.w * L.in_cstride)
    return fail(AICAM_ERR_INVALID_ARG, "launch_conv: input images must be dense NHWC");
  if (static_cast<long long>(L.batch) * L.h * L.w >= (1ll << 31) || static_cast<long long>(L.batch) * a.howo >= (1ll << 31))
    return fail(AICAM_ERR_CAPACITY, "launch_conv: more than 2^31 pixels in one launch");
  {
    // coalesced epilogue needs 16-byte aligned rows and whole 16-byte chunks of valid channels
    const int es = L.out_f32 ? 4 : 2;
    bool ok = (a.cout * es) % 16 == 0 && (static_cast<long long>(L.out_cstride) * es) % 16 == 0 &&
              (static_cast<long long>(L.out_coff) * es) % 16 == 0 && (L.out_img_stride * es) % 16 == 0 &&
              (reinterpret_cast<uintptr_t>(L.out) % 16) == 0 && (a.n_tile * es) % 16 == 0 &&
              128 * (a.n_tile * es + 16) <= STAGES * A_STAGE_BYTES;
    if (a.res_mode)
      ok = ok && L.res_cstride % 8 == 0 && L.res_coff % 8 == 0 && L.res_img_stride % 8 == 0 &&
           (reinterpret_cast<uintptr_t>(L.res) % 16) == 0 && a.cout % 8 == 0 && !L.out_f32;
    a.staged = ok ? 1 : 0;
  }
  a.out_dense = L.out_img_stride == static_cast<long long>(a.howo) * L.out_cstride ? 1 : 0;
  a.res_dense = (a.res_mode == 0 || L.res_img_stride == static_cast<long long>(a.howo) * L.res_cstride) ? 1 : 0;
  if (!a.stem && (L.in_cstride % 8 != 0 || L.in_coff % 8 != 0))
    return fail(AICAM_ERR_INVALID_ARG, "launch_conv: input channel stride/offset must be multiples of 8");
  if (a.stem && (L.in_cstride != 4 || L.in_coff != 0))
    return fail(AICAM_ERR_INVALID_ARG, "launch_conv: stem input must be NHWC4");
  // 3x3 / 1x1 stride-1 layers: patch-based window kernel (conv_win.cu) when the shape is eligible
  {
    const int wrc = try_launch_conv_win(pc, L, stream);
    if (wrc < 0) return wrc;
    if (wrc == 1) return AICAM_OK;
    if (L.out_s2d) return fail(AICAM_ERR_UNSUPPORTED, "launch_conv: space-to-depth output needs the window kernel");
    if (L.decode) return fail(AICAM_ERR_UNSUPPORTED, "launch_conv: the fused Detect decode needs the window kernel");
  }
  size_t smem = SMEM_HEADER + STAGES * (A_STAGE_BYTES + static_cast<size_t>(a.n_tile) * 16 * CHUNKS_PER_STAGE);
  a.res_stage_off = 0;
  if (int rc = ensure_dynamic_smem(conv_tc_kernel, 160 * 1024)) return rc;
  // persistent CTAs: at most 3 resident per SM (registers / shared memory), each loops over tiles
  const int num_sms = current_num_sms();
  const long long tiles = static_cast<long long>(cdiv(a.m_total, TILE_M)) * (a.cout_pad / a.n_tile);
  const int per_sm = static_cast<int>(std::min<size_t>(3, (227 * 1024) / (smem + 1024)));
  dim3 grid(static_cast<unsigned>(std::min<long long>(tiles, static_cast<long long>(num_sms) * std::max(1, per_sm))));
  size_t slot = 0;
  const bool prof = profile_begin(stream, &slot);
  conv_tc_kernel<<<grid, NUM_THREADS, smem, stream>>>(a);
  if (prof) profile_end(stream, slot);
  count_launch();
  return last_launch("conv_tc_kernel");
}

}  // namespace aicam
