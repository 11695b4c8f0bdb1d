// K8 on the tensor cores: the appearance cost of crowded frames as a TF32x3 GEMM on tcgen05 / TMEM / TMA, sm_100a.
//
//   cost[track][det] = min over the track's gallery of max(0, 1 - <g, f_det>)
//   (/root/reference/src/tracker/core/matching.py:109-217: a float32 sgemm per track, then a min over rows)
//
// The reference multiplies float32 features, and parity on the cost is held to 1e-5 (tests/test_gpu_tracker.py), so
// bf16 operands are out.  Every normalised feature x is kept as x = hi + lo with hi = x rounded to the 10-bit TF32
// mantissa (exactly representable, so whatever the tensor core does with the 13 low bits, it reads hi) and
// lo = x - hi (exact in float32); <g, f> ~ <g_hi, f_hi> + <g_hi, f_lo> + <g_lo, f_hi> accumulated in fp32 by three
// kind::tf32 MMAs per K step: relative error ~2^-21, i.e. ~1e-6 on a unit-vector dot product.  The split halves of
// the gallery are written when a feature is inserted (tracker.cu), those of the detections by normalize_kernel.
//
// Work item = (stream, confirmed track, tile of 128 detections).  M = detections (TMEM lanes), N = 112 = the track's
// gallery rows (100 at the reference's budget, + 12 rows that belong to the next slot and are masked), K = 512 in
// 16 slabs of 32 floats (128-byte rows, hardware 128-byte swizzle, both operands K-major straight from TMA).  With
// the detections on the lanes the min over the gallery is a min over accumulator COLUMNS: each epilogue thread
// reduces its own row, no cross-lane traffic.  Persistent CTAs, 3-stage operand ring (60 KB per stage: A hi / lo,
// B hi / lo), double-buffered accumulators (2 x 128 TMEM columns) so that the reduction of item i overlaps the MMAs
// of item i + 1.  Frames with at most APP_TC_MIN detections stay on the row kernel of tracker.cu (no padding work).
//
// Bound: tensor pipe ~ L2 -> SM operand traffic.  Per item 192 MMAs of 128 x 112 x 8; at 16 streams x 300 tracks x
// 300 detections (BASELINE.json configs[4]) 14 400 items ~ 0.6-1.2 ms against ~8 ms for the fp32 FFMA tiling.
#include <cstring>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace aicam {

extern void count_launch();

namespace {

using namespace ptx;

constexpr int TF_THREADS = 192;        // 4 epilogue warps, MMA issuer, TMA producer
constexpr int TF_STAGES = 3;
constexpr int TF_M = 128;              // detections per tile
constexpr int TF_N = 112;              // gallery rows per tile (>= nn_budget, multiple of 16)
constexpr int TF_KS = 32;              // floats per K slab = one 128-byte swizzled row
constexpr uint32_t TF_A_BYTES = TF_M * 128, TF_B_BYTES = TF_N * 128;
constexpr uint32_t TF_STAGE_BYTES = 2 * TF_A_BYTES + 2 * TF_B_BYTES;  // 61 440
constexpr uint32_t TF_OFF_RING = 1024;
constexpr size_t TF_SMEM = TF_OFF_RING + TF_STAGES * TF_STAGE_BYTES;
constexpr float TF_INFTY = 1e5f;

struct TfMaps {
  CUtensorMap g_hi, g_lo, f_hi, f_lo;
};

struct TfArgs {
  int S, T, D, F, G;
  int m_tiles;              // ceil(D / 128)
  int min_dets;             // streams with at most this many detections are left to the row kernel
  const int* n_tracks; const int* order; const int* state; const int* gal_count;
  const int* det_count; const int* crop_slot; int stride_k;
  const int* present;       // [S] 0: the stream is absent this step (no work), or null
  float* app_cost;          // [S][T][D] by (slot, det)
};

__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
      : "memory");
}

// Work enumeration, identical in every role: the crowded streams (a bitmap in shared memory, built once per CTA from
// the device-side detection counts) in ascending order, each contributing n_tracks[s] x ceil(nd / 128) items; item i
// of the concatenation belongs to CTA i mod gridDim.  Tracks that are not confirmed are skipped after one load.
struct Item {
  int s, slot, m, nd, ng;
};
constexpr int TF_MAX_STREAMS = 4096;  // bitmap capacity (512 bytes of shared memory)

template <typename Fn>
__device__ __forceinline__ void for_each_item(const TfArgs& a, const uint32_t* crowded, Fn&& fn) {
  const long long g = gridDim.x;
  long long base = 0;
  for (int w = 0; w < (a.S + 31) / 32; ++w) {
    uint32_t bits = crowded[w];
    while (bits) {
      const int s = w * 32 + __ffs(bits) - 1;
      bits &= bits - 1;
      const int nd = min(__ldg(a.det_count + s), a.D);
      const int mt = (nd + TF_M - 1) / TF_M;
      const int n = __ldg(a.n_tracks + s) * mt;
      long long r = (static_cast<long long>(blockIdx.x) - base % g + g) % g;
      for (; r < n; r += g) {
        Item it;
        it.s = s; it.nd = nd;
        const int ti = static_cast<int>(r) / mt;
        it.m = static_cast<int>(r) - ti * mt;
        it.slot = __ldg(a.order + static_cast<long long>(s) * a.T + ti);
        const long long ts = static_cast<long long>(s) * a.T + it.slot;
        if (__ldg(a.state + ts) != 2) continue;  // only confirmed tracks enter the appearance cascade (tracker_core.py:112-117)
        it.ng = __ldg(a.gal_count + ts);
        fn(it);
      }
      base += n;
    }
  }
}

__global__ void __launch_bounds__(TF_THREADS, 1) appearance_tf32_kernel(const __grid_constant__ TfArgs a,
                                                                        const __grid_constant__ TfMaps maps) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar_full = sbase, bar_empty = sbase + 32, bar_acc_full = sbase + 64, bar_acc_empty = sbase + 80;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(smem + 96);
  uint32_t* crowded = reinterpret_cast<uint32_t*>(smem + 128);  // [TF_MAX_STREAMS / 32]
  __shared__ int s_any;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // streams with more than min_dets detections; an ordinary frame has none and the CTA leaves at once
  if (threadIdx.x == 0) s_any = 0;
  for (int w = threadIdx.x; w < TF_MAX_STREAMS / 32; w += TF_THREADS) crowded[w] = 0;
  __syncthreads();
  for (int s = threadIdx.x; s < a.S; s += TF_THREADS)
    if ((!a.present || __ldg(a.present + s)) && min(__ldg(a.det_count + s), a.D) > a.min_dets) {
      atomicOr(&crowded[s >> 5], 1u << (s & 31));
      s_any = 1;
    }
  __syncthreads();
  if (!s_any) return;

  if (threadIdx.x == 0) {
    for (int s = 0; s < TF_STAGES; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(bar_acc_full + 8 * s, 1);
      mbar_init(bar_acc_empty + 8 * s, 128);
    }
    mbar_init_fence();
  }
  if (warp == 4) tc_alloc(smem_u32(tmem_ptr_smem), 256);
  if (warp == 5 && lane == 0) {
    tma_prefetch_desc(&maps.g_hi); tma_prefetch_desc(&maps.g_lo);
    tma_prefetch_desc(&maps.f_hi); tma_prefetch_desc(&maps.f_lo);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  const int slabs = a.F / TF_KS;

  if (warp < 4) {
    // ============================================================ epilogue: segmented min over accumulator columns
    const uint32_t taddr_lane = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
    int n = 0;
    for_each_item(a, crowded, [&](const Item& it) {
      const int buf = n & 1;
      mbar_wait(bar_acc_full + 8 * buf, (n >> 1) & 1);
      tc_fence_after();
      float best = TF_INFTY;
      const uint32_t taddr = taddr_lane + buf * 128;
#pragma unroll 1
      for (int g = 0; g < TF_N / 16; ++g) {
        if (g * 16 >= it.ng) break;  // (uniform: ng is per item)
        uint32_t v[16];
        tc_ld16_nowait(taddr + g * 16, v);
        tc_ld_wait();
#pragma unroll
        for (int i = 0; i < 16; ++i)
          if (g * 16 + i < it.ng) best = fminf(best, fmaxf(1.0f - __uint_as_float(v[i]), 0.0f));
      }
      tc_fence_before();
      mbar_arrive(bar_acc_empty + 8 * buf);
      const int d = it.m * TF_M + warp * 32 + lane;
      if (d < it.nd) {
        const bool has = __ldg(a.crop_slot + static_cast<long long>(it.s) * a.stride_k + d) >= 0;
        a.app_cost[(static_cast<long long>(it.s) * a.T + it.slot) * a.D + d] = (has && it.ng > 0) ? best : TF_INFTY;
      }
      ++n;
    });
  } else if (warp == 4) {
    // ============================================================ MMA issuer (one lane)
    if (lane == 0) {
      // K-major, 128-byte swizzle: SBO = 8 rows x 128 B, descriptor version 1, layout type 2
      const uint64_t hi_word = static_cast<uint64_t>((1024u >> 4) | (1u << 14) | (2u << 29)) << 32;
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(TF_N >> 3) << 17) |
                             (static_cast<uint32_t>(TF_M >> 4) << 24);
      uint32_t st = 0, ph = 0;
      int n = 0;
      for_each_item(a, crowded, [&](const Item& it) {
        const int buf = n & 1;
        mbar_wait(bar_acc_empty + 8 * buf, ((n >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * 128;
        for (int s = 0; s < slabs; ++s) {
          mbar_wait(bar_full + 8 * st, ph);
          tc_fence_after();
          const uint32_t base = sbase + TF_OFF_RING + st * TF_STAGE_BYTES;
          const uint32_t a_hi = base, a_lo = base + TF_A_BYTES, b_hi = base + 2 * TF_A_BYTES, b_lo = b_hi + TF_B_BYTES;
#pragma unroll
          for (int k = 0; k < TF_KS / 8; ++k) {
            const uint64_t dah = hi_word | (((a_hi >> 4) + 2 * k) & 0x3FFF) | (1ull << 16);
            const uint64_t dal = hi_word | (((a_lo >> 4) + 2 * k) & 0x3FFF) | (1ull << 16);
            const uint64_t dbh = hi_word | (((b_hi >> 4) + 2 * k) & 0x3FFF) | (1ull << 16);
            const uint64_t dbl = hi_word | (((b_lo >> 4) + 2 * k) & 0x3FFF) | (1ull << 16);
            // small terms first: the fp32 accumulator then adds them before the leading product dominates
            mma_tf32(d_tmem, dah, dbl, idesc, (s | k) != 0 ? 1u : 0u);
            mma_tf32(d_tmem, dal, dbh, idesc, 1u);
            mma_tf32(d_tmem, dah, dbh, idesc, 1u);
          }
          tc_commit(bar_empty + 8 * st);
          if (++st == TF_STAGES) { st = 0; ph ^= 1; }
        }
        tc_commit(bar_acc_full + 8 * buf);
        ++n;
      });
      tc_fence_before();
    }
  } else {
    // ============================================================ TMA producer (one lane)
    if (lane == 0) {
      uint32_t st = 0, ph = 1;
      for_each_item(a, crowded, [&](const Item& it) {
        const int row_f = it.s * a.D + it.m * TF_M;
        const int row_g = (it.s * a.T + it.slot) * a.G;
        for (int s = 0; s < slabs; ++s) {
          mbar_wait(bar_empty + 8 * st, ph);
          const uint32_t bar = bar_full + 8 * st;
          const uint32_t base = sbase + TF_OFF_RING + st * TF_STAGE_BYTES;
          mbar_arrive_expect_tx(bar, TF_STAGE_BYTES);
          tma_load_2d(base, &maps.f_hi, bar, s * TF_KS, row_f);
          tma_load_2d(base + TF_A_BYTES, &maps.f_lo, bar, s * TF_KS, row_f);
          tma_load_2d(base + 2 * TF_A_BYTES, &maps.g_hi, bar, s * TF_KS, row_g);
          tma_load_2d(base + 2 * TF_A_BYTES + TF_B_BYTES, &maps.g_lo, bar, s * TF_KS, row_g);
          if (++st == TF_STAGES) { st = 0; ph ^= 1; }
        }
      });
    }
  }
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    tc_dealloc(tmem_base, 256);
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn tf_encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

int encode_rows(CUtensorMap* m, const float* base, long long rows, int F, int box_rows) {
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(F), static_cast<cuuint64_t>(rows)};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(F) * 4};
  const cuuint32_t box[2] = {TF_KS, static_cast<cuuint32_t>(box_rows)};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult cr = tf_encode_tiled()(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return cr == CUDA_SUCCESS ? AICAM_OK : fail(AICAM_ERR_CUDA, "appearance_tf32: cuTensorMapEncodeTiled failed with " + std::to_string(static_cast<int>(cr)));
}

}  // namespace

// The four tensor maps of a tracker's split feature arrays (made once, at tracker creation): opaque to the caller.
struct AppearanceTf32 {
  TfMaps maps;
};

bool appearance_tf32_eligible(int S, int F, int G, int D) {
  return tf_encode_tiled() != nullptr && F % TF_KS == 0 && G <= TF_N && G >= 1 && D >= 1 && S <= TF_MAX_STREAMS;
}

int appearance_tf32_create(AppearanceTf32** out, int S, int T, int D, int F, int G, const float* gal_hi, const float* gal_lo,
                           const float* feat_hi, const float* feat_lo) {
  AppearanceTf32* p = new AppearanceTf32();
  std::memset(&p->maps, 0, sizeof(p->maps));
  int rc = encode_rows(&p->maps.g_hi, gal_hi, static_cast<long long>(S) * T * G, F, TF_N);
  if (!rc) rc = encode_rows(&p->maps.g_lo, gal_lo, static_cast<long long>(S) * T * G, F, TF_N);
  if (!rc) rc = encode_rows(&p->maps.f_hi, feat_hi, static_cast<long long>(S) * D, F, TF_M);
  if (!rc) rc = encode_rows(&p->maps.f_lo, feat_lo, static_cast<long long>(S) * D, F, TF_M);
  if (rc) { delete p; return rc; }
  *out = p;
  return AICAM_OK;
}

void appearance_tf32_destroy(AppearanceTf32* p) { delete p; }

int launch_appearance_tf32(const AppearanceTf32* p, int S, int T, int D, int F, int G, int min_dets, const int* n_tracks,
                           const int* order, const int* state, const int* gal_count, const int* det_count, const int* crop_slot,
                           int stride_k, const int* present, float* app_cost, cudaStream_t stream) {
  TfArgs a;
  a.S = S; a.T = T; a.D = D; a.F = F; a.G = G;
  a.m_tiles = (D + TF_M - 1) / TF_M;
  a.min_dets = min_dets;
  a.n_tracks = n_tracks; a.order = order; a.state = state; a.gal_count = gal_count;
  a.det_count = det_count; a.crop_slot = crop_slot; a.stride_k = stride_k; a.present = present; a.app_cost = app_cost;
  if (int rc = ensure_dynamic_smem(appearance_tf32_kernel, TF_SMEM)) return rc;
  const long long total = static_cast<long long>(S) * T * a.m_tiles;
  const int sms = current_num_sms();
  const unsigned grid = static_cast<unsigned>(total < sms ? total : sms);
  appearance_tf32_kernel<<<grid, TF_THREADS, TF_SMEM, stream>>>(a, p->maps);
  count_launch();
  return last_launch("appearance_tf32_kernel");
}

}  // namespace aicam
