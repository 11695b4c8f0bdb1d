// 3x3 stride-1 convolution over zero-bordered tensors on CTA PAIRS: tcgen05.mma.cta_group::2, sm_100a.
//
// Same operator, same data layout and same flat padded raster as operand mode 4 of conv_win.cu (the 3x3 layers
// of the ReID trunk, /root/reference/src/tracker/reid_model.py:115 -> trt_engine.py:191), different MMA shape.
// With one CTA per MMA a 128 x N x 16 instruction reads 4 KB of A and N * 32 B of B from the CTA's shared memory:
// for N = 64 that is 48 cycles of the 128 B/clk port against 32 tensor-pipe cycles, for N = 128 64 against 64 - the
// port, not the tensor pipe, paces those layers (ncu: tensor pipe 39-43 % / 65-68 % active).  A CTA pair (cluster
// of two, the two SMs of a TPC) issues ONE 256 x N x 16 instruction: each CTA feeds its own 128 rows of A and only
// HALF of B (N / 2 weight columns live in each CTA), so the fetch drops to 40 cycles (N = 64) and 48 (N = 128).
//
//   * tile = 2 x 128 MT consecutive raster positions; CTA rank r of the pair owns rows [(2 pt + r) TM, + TM);
//   * both CTAs run their own patch (A) producer, weight (B) producer for their half of the columns, epilogue
//     and TMA store warp, exactly as in conv_win.cu;
//   * only the leader (rank 0) issues MMAs.  It needs to know that the PEER's operands have landed and that the
//     peer's epilogue has drained the accumulator: the peer's otherwise idle MMA warp relays those three local
//     barriers (patch full, weight full, accumulator empty) to the leader with remote mbarrier arrives, in the
//     same order in which the leader waits for them;
//   * tcgen05.commit.cta_group::2 ... multicast::cluster frees the operand slots and publishes the accumulator
//     in BOTH CTAs.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "conv_tc.cuh"
#include "tc_ptx.cuh"

namespace aicam {

extern void count_launch();
bool profile_begin(cudaStream_t st, size_t* slot);
void profile_end(cudaStream_t st, size_t slot);

namespace {

using namespace ptx;

constexpr int NWG = 4;
constexpr int PAIR_THREADS = (4 * NWG + 4) * 32;
constexpr int MAX_RING = 8;
constexpr uint32_t OFF_RING_A = 1024;  // barriers and the TMEM pointer live below
constexpr size_t SMEM_LIMIT = 227 * 1024;
constexpr uint32_t ROW_BYTES = 128;  // 64-channel slabs
// (filter taps per streamed weight stage - one contiguous bulk copy - are a launch parameter: 3, or 1 for 256-column tiles)

struct PairMaps {
  CUtensorMap in, out, res;
};

struct PairArgs {
  int h, w, hw, rw;           // logical image size, padded pixels per image, padded row pitch
  int lo;                     // offset of the interior inside the padded image (1 symmetric border, 0 shared border)
  int slabs, cin_pad;
  int sa, sb, resident;
  uint32_t patch_bytes, box_bytes, bstage_bytes, wbytes_half;
  int box_rows;
  int n_tile, n_half, cout, n_tiles, tps;
  const __nv_bfloat16* wgt_pair;  // [n-tile][rank][slab][tap][8 K chunks][n_half][8]: the order in which the MMAs consume it
  long long half_elems;           // elements of one rank's weights of one n-tile
  int res_mode;
  int batch;
  const int* batch_dev;
  uint32_t idesc, tmem_cols;
  uint32_t off_w, off_b, off_stage, stage_buf_bytes;
  int nstage, pieces;
  uint32_t piece_off[4];
  uint32_t res_tx_bytes;
  float4 bias4[128];  // the bias, read from the constant bank
  long long* trace;  // debug: clock64 stamps of CTA 0 (AICAM_CONV_TRACE in aicam_conv2d_bench), same slots as conv_win.cu
  int warp_arrive;   // one elected lane per epilogue warp arrives on the mbarriers (default) instead of every thread (conv_win.cu)
};

#define PAIR_TRACE(it, who) do { if (a.trace && blockIdx.x == 0 && (it) < 32) a.trace[(it) * 16 + (who)] = clock64(); } while (0)

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint32_t bar, uint32_t rank) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}" ::"r"(bar),
      "r"(rank)
      : "memory");
}
__device__ __forceinline__ void tc_alloc2(uint32_t smem_dst, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_dealloc2(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// executed by the whole (converged) warp, performed by the lane whose `leader` predicate is set
__device__ __forceinline__ void mma2_issue(bool leader, uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo,
                                           uint32_t b_hi, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "setp.ne.b32 q, %7, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "@q tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %5, p;\n\t}" ::"r"(tmem_d),
      "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate), "r"(static_cast<uint32_t>(leader))
      : "memory");
}
// completion of every MMA issued so far -> one arrival on the barrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void tc_commit2_if(bool leader, uint32_t bar) {
  asm volatile(
      "{\n\t.reg .pred q;\n\t.reg .b16 m;\n\t"
      "setp.ne.b32 q, %1, 0;\n\t"
      "mov.b16 m, 3;\n\t"
      "@q tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], m;\n\t}" ::"r"(bar),
      "r"(static_cast<uint32_t>(leader))
      : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
      "elect.sync rx|px, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, px;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

template <int ACT>
__device__ __forceinline__ float activate(float x) {
  if (ACT == 1) {
    const float h = 0.5f * x;
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
    return fmaf(h, t, h);
  }
  if (ACT == 2) return fmaxf(x, 0.0f);
  return x;
}

// 16 accumulator columns of one row: + bias (+ residual, read from the staging tile itself), activation, bf16, back
// into the staging tile (two 16-byte chunks at swizzled positions o0 / o1)
template <int ACT>
__device__ __forceinline__ void finish16(const uint32_t (&v)[16], const float (&bias)[16], int res_mode, uint8_t* p0, uint8_t* p1) {
  float x[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) x[i] = __uint_as_float(v[i]) + bias[i];
  if (res_mode) {
    const uint4 q0 = *reinterpret_cast<const uint4*>(p0);
    const uint4 q1 = *reinterpret_cast<const uint4*>(p1);
    const uint32_t rw_[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (res_mode == 2) {
        x[2 * i] = activate<ACT>(x[2 * i] + bf16_lo(rw_[i]));
        x[2 * i + 1] = activate<ACT>(x[2 * i + 1] + bf16_hi(rw_[i]));
      } else {
        x[2 * i] = activate<ACT>(x[2 * i]) + bf16_lo(rw_[i]);
        x[2 * i + 1] = activate<ACT>(x[2 * i + 1]) + bf16_hi(rw_[i]);
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < 16; ++i) x[i] = activate<ACT>(x[i]);
  }
  *reinterpret_cast<uint4*>(p0) = make_uint4(pack_bf16x2(x[0], x[1]), pack_bf16x2(x[2], x[3]), pack_bf16x2(x[4], x[5]), pack_bf16x2(x[6], x[7]));
  *reinterpret_cast<uint4*>(p1) =
      make_uint4(pack_bf16x2(x[8], x[9]), pack_bf16x2(x[10], x[11]), pack_bf16x2(x[12], x[13]), pack_bf16x2(x[14], x[15]));
}

template <int MT, int ACT, int TPS>
__global__ void __launch_bounds__(PAIR_THREADS, 1) conv_pair_kernel(const __grid_constant__ PairArgs a,
                                                                    const __grid_constant__ PairMaps maps) {
  constexpr int TM = 128 * MT;
  constexpr int TAPS = 9;
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar_a_full = sbase, bar_a_empty = sbase + 64, bar_b_full = sbase + 128, bar_b_empty = sbase + 192;
  const uint32_t bar_acc_full = sbase + 256, bar_acc_empty = sbase + 272, bar_w_full = sbase + 288;
  const uint32_t bar_res_full = sbase + 296, bar_res_empty = sbase + 312, bar_stage_free = sbase + 328;
  const uint32_t bar_peer_w = sbase + 344;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(smem + 352);
  const uint32_t bar_peer_a = sbase + 384, bar_peer_b = sbase + 448, bar_peer_acc = sbase + 512;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  int batch = a.batch;
  if (a.batch_dev) batch = min(batch, __ldg(a.batch_dev));
  const long long total_rows = static_cast<long long>(batch) * a.hw;
  const int m_tiles = static_cast<int>((total_rows + 2 * TM - 1) / (2 * TM));
  const int pair_tiles = m_tiles * a.n_tiles;  // work items of a pair: (row tile, n-tile), n-tile fastest
  pdl_trigger();
  if (pair >= pair_tiles) return;  // (both CTAs of the pair)

  if (threadIdx.x == 0) {
    for (int s = 0; s < MAX_RING; ++s) {
      mbar_init(bar_a_full + 8 * s, 1); mbar_init(bar_a_empty + 8 * s, 1);
      mbar_init(bar_b_full + 8 * s, 1); mbar_init(bar_b_empty + 8 * s, 1);
      mbar_init(bar_peer_a + 8 * s, 1); mbar_init(bar_peer_b + 8 * s, 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(bar_acc_full + 8 * s, 1); mbar_init(bar_acc_empty + 8 * s, a.warp_arrive ? 4 * NWG : 128 * NWG);
      mbar_init(bar_peer_acc + 8 * s, 1);
      mbar_init(bar_res_full + 8 * s, 1); mbar_init(bar_res_empty + 8 * s, a.warp_arrive ? 4 * NWG : 128 * NWG);
      mbar_init(bar_stage_free + 8 * s, 1);
    }
    mbar_init(bar_w_full, 1);
    mbar_init(bar_peer_w, 1);
    mbar_init_fence();
  }
  if (warp == 4 * NWG) tc_alloc2(smem_u32(tmem_ptr_smem), a.tmem_cols);
  if (warp == 4 * NWG + 1 && lane == 0) tma_prefetch_desc(&maps.in);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // both CTAs: barriers initialised, TMEM allocated
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  const uint32_t acc_cols = static_cast<uint32_t>(MT * a.n_tile);

  if (warp < 4 * NWG) {
    // ================================================================== epilogue (16 warps): TMEM -> staging tile, in place
    constexpr int PARTS = MT == 2 ? 2 : 4;
    const int wg = warp >> 2, wq = warp & 3;
    const int my_j = MT == 2 ? (wg >> 1) : 0;
    const int part = MT == 2 ? (wg & 1) : wg;
    const int r = my_j * 128 + wq * 32 + lane;
    const uint32_t taddr_lane = tmem_base + (static_cast<uint32_t>(wq * 32) << 16);
    const uint32_t ro = static_cast<uint32_t>(r) * 128u;         // my row inside a 64-channel piece (128-byte rows)
    const uint32_t rxor = ((ro >> 7) & 7u) << 4;
    uint8_t* stage0 = smem + a.off_stage;
    const int groups = a.n_tile >> 4;
    const int g_lo = (groups * part) / PARTS, g_hi = (groups * (part + 1)) / PARTS;
    int it = 0;
    for (int pt = pair; pt < pair_tiles; pt += npairs, ++it) {
      const int buf = it & 1;
      const int mt_i = pt / a.n_tiles, n0 = (pt - mt_i * a.n_tiles) * a.n_tile;
      const uint32_t p = (static_cast<uint32_t>(mt_i) * 2 + rank) * TM + r;  // (< 2^31 padded pixels, checked on the host)
      const uint32_t rem = p % static_cast<uint32_t>(a.hw);
      const int yy = static_cast<int>(rem / static_cast<uint32_t>(a.rw)), xx = static_cast<int>(rem) - yy * a.rw;
      const bool zero_row = !(yy >= a.lo && yy < a.lo + a.h && xx >= a.lo && xx < a.lo + a.w);
      if (threadIdx.x == 0) PAIR_TRACE(it, 8);
      mbar_wait(bar_acc_full + 8 * buf, (it >> 1) & 1);
      tc_fence_after();
      if (threadIdx.x == 0) PAIR_TRACE(it, 9);
      const int sbuf = a.nstage == 2 ? (it & 1) : 0;
      const uint32_t spar = a.nstage == 2 ? ((it >> 1) & 1) : (it & 1);
      if (a.res_mode) mbar_wait(bar_res_full + 8 * sbuf, spar);
      if (threadIdx.x == 0) PAIR_TRACE(it, 10);
      const uint32_t taddr = taddr_lane + buf * acc_cols + my_j * a.n_tile;
      uint8_t* stage = stage0 + sbuf * a.stage_buf_bytes;
      bool stage_ok = false;
      for (int g = g_lo; g < g_hi; g += 2) {
        uint32_t v0[16], v1[16];
        const bool two = g + 1 < g_hi;
        __syncwarp();
        tc_ld16_nowait(taddr + g * 16, v0);
        if (two) tc_ld16_nowait(taddr + g * 16 + 16, v1);
        if (!stage_ok) {
          mbar_wait(bar_stage_free + 8 * sbuf, spar ^ 1);
          stage_ok = true;
        }
        tc_ld_wait();
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          if (hh == 1 && !two) break;
          const int c = (g + hh) * 16;
          const uint32_t pc = static_cast<uint32_t>(c >> 6), ch0 = static_cast<uint32_t>(c & 63) * 2;
          uint8_t* p0 = stage + a.piece_off[pc] + ro + (ch0 ^ rxor);
          uint8_t* p1 = stage + a.piece_off[pc] + ro + ((ch0 + 16) ^ rxor);
          if (zero_row) {
            *reinterpret_cast<uint4*>(p0) = make_uint4(0u, 0u, 0u, 0u);
            *reinterpret_cast<uint4*>(p1) = make_uint4(0u, 0u, 0u, 0u);
          } else {
            float bv[16];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float4 b4 = a.bias4[((n0 + c) >> 2) + i];
              bv[4 * i] = b4.x; bv[4 * i + 1] = b4.y; bv[4 * i + 2] = b4.z; bv[4 * i + 3] = b4.w;
            }
            finish16<ACT>(hh ? v1 : v0, bv, a.res_mode, p0, p1);
          }
        }
      }
      if (!stage_ok) mbar_wait(bar_stage_free + 8 * sbuf, spar ^ 1);
      tc_fence_before();
      if (a.warp_arrive) {
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(bar_acc_empty + 8 * buf);
          if (a.res_mode) mbar_arrive(bar_res_empty + 8 * sbuf);
        }
      } else {
        mbar_arrive(bar_acc_empty + 8 * buf);
        if (a.res_mode) mbar_arrive(bar_res_empty + 8 * sbuf);
      }
      if (threadIdx.x == 0) PAIR_TRACE(it, 12);
      fence_proxy_async();
      asm volatile("bar.arrive %0, %1;" ::"r"(2 + (it & 1)), "n"(128 * NWG + 32) : "memory");
    }
  } else if (warp == 4 * NWG) {
    // ================================================================== MMA issuer (leader) / barrier relay (peer)
    const bool elected = elect_one();
    const uint32_t n_sa = a.sa, n_sb = a.sb;
    constexpr int tps = TPS;
    uint32_t sa = 0, pa = 0, sbi = 0, pb = 0;
    if (rank == 0) {
      const uint32_t a_hi = ((8 * ROW_BYTES) >> 4) | (1u << 14) | (2u << 29);  // SBO | version | SWIZZLE_128B
      const uint32_t b_hi = (128u >> 4) | (1u << 14);
      const uint32_t a_ring = sbase + OFF_RING_A, b_ring = sbase + a.off_b, w_base = sbase + a.off_w;
      const uint32_t rw_units = static_cast<uint32_t>(a.rw) * (ROW_BYTES >> 4);
      const uint32_t lbo = static_cast<uint32_t>(a.n_half);  // K-chunk stride of my half of the weights, 16-byte units
      const uint32_t b_k16 = 2 * lbo, b_lo_flags = lbo << 16;
      const uint32_t w_tap = 8u * lbo;  // one (slab, tap) block of my weights: 8 K chunks, 16-byte units
      const uint32_t tmem0 = __shfl_sync(0xffffffffu, tmem_base, 0);
      if (a.resident) {
        mbar_wait(bar_w_full, 0);
        mbar_wait(bar_peer_w, 0);
      }
      int it = 0;
      for (int pt = pair; pt < pair_tiles; pt += npairs, ++it) {
        const int buf = it & 1;
        if (elected) PAIR_TRACE(it, 0);
        mbar_wait(bar_acc_empty + 8 * buf, ((it >> 1) & 1) ^ 1);
        // the relay arrives once per tile AFTER its own wait on the peer's accumulator barrier (which passes freely
        // for the first use of each buffer): its n-th arrival completes phase n
        mbar_wait(bar_peer_acc + 8 * buf, (it >> 1) & 1);
        tc_fence_after();
        if (elected) PAIR_TRACE(it, 1);
        const uint32_t d_tmem = tmem0 + buf * acc_cols;
        for (int s = 0; s < a.slabs; ++s) {
          mbar_wait(bar_a_full + 8 * sa, pa);
          if (elected && s == 0) PAIR_TRACE(it, 13);
          mbar_wait(bar_peer_a + 8 * sa, pa);
          tc_fence_after();
          if (elected && s == 0) PAIR_TRACE(it, 2);
          const uint32_t a_lo0 = ((a_ring + sa * a.patch_bytes) >> 4) + (1u << 16);
          uint32_t w_lo = ((w_base >> 4) + static_cast<uint32_t>(s * TAPS) * w_tap) | b_lo_flags;  // resident: (slab, tap) blocks
#pragma unroll
          for (int t = 0; t < TAPS; ++t) {
            const int dy = t / 3, dx = t - dy * 3;
            const uint32_t a_lo = a_lo0 + dy * rw_units + dx * (ROW_BYTES >> 4);
            uint32_t b_lo;
            if (a.resident) {
              b_lo = w_lo;
              w_lo += w_tap;
            } else {
              if (t % tps == 0) {
                mbar_wait(bar_b_full + 8 * sbi, pb);
                mbar_wait(bar_peer_b + 8 * sbi, pb);
                tc_fence_after();
              }
              b_lo = (((b_ring + sbi * a.bstage_bytes) >> 4) + static_cast<uint32_t>(t % tps) * w_tap) | b_lo_flags;
            }
#pragma unroll
            for (int j = 0; j < MT; ++j)
#pragma unroll
              for (int k = 0; k < 4; ++k)
                mma2_issue(elected, d_tmem + j * a.n_tile, a_lo + j * (128 * ROW_BYTES >> 4) + k * 2, a_hi, b_lo + k * b_k16, b_hi,
                           a.idesc, (s | t | k) != 0 ? 1u : 0u);
            if (!a.resident && t % tps == tps - 1) {
              tc_commit2_if(elected, bar_b_empty + 8 * sbi);
              if (++sbi == n_sb) { sbi = 0; pb ^= 1; }
            }
          }
          tc_commit2_if(elected, bar_a_empty + 8 * sa);
          if (++sa == n_sa) { sa = 0; pa ^= 1; }
        }
        tc_commit2_if(elected, bar_acc_full + 8 * buf);
        if (elected) PAIR_TRACE(it, 3);
      }
      tc_fence_before();
    } else {
      // peer: my operands landed / my accumulator drained -> tell the leader, in the order the leader waits
      if (a.resident) {
        mbar_wait(bar_w_full, 0);
        if (elected) mbar_arrive_remote(bar_peer_w, 0);
      }
      int it = 0;
      for (int pt = pair; pt < pair_tiles; pt += npairs, ++it) {
        const int buf = it & 1;
        mbar_wait(bar_acc_empty + 8 * buf, ((it >> 1) & 1) ^ 1);
        if (elected) mbar_arrive_remote(bar_peer_acc + 8 * buf, 0);
        for (int s = 0; s < a.slabs; ++s) {
          mbar_wait(bar_a_full + 8 * sa, pa);
          if (elected) mbar_arrive_remote(bar_peer_a + 8 * sa, 0);
          if (!a.resident) {
            for (int t = 0; t < TAPS / tps; ++t) {
              mbar_wait(bar_b_full + 8 * sbi, pb);
              if (elected) mbar_arrive_remote(bar_peer_b + 8 * sbi, 0);
              if (++sbi == n_sb) { sbi = 0; pb ^= 1; }
            }
          }
          if (++sa == n_sa) { sa = 0; pa ^= 1; }
        }
      }
    }
  } else if (warp == 4 * NWG + 1) {
    // ================================================================== patch (A) producer, both CTAs
    if (lane == 0) {
      pdl_wait();
      const uint32_t a_ring = sbase + OFF_RING_A;
      uint32_t sa = 0, pa = 1;
      const uint32_t n_sa = a.sa;
      for (int pt = pair; pt < pair_tiles; pt += npairs) {
        const long long p0 = (static_cast<long long>(pt / a.n_tiles) * 2 + rank) * TM;
        const int row0 = static_cast<int>(p0) - (a.rw + 1);
        const int pit = (pt - pair) / npairs;
        for (int s = 0; s < a.slabs; ++s) {
          if (s == 0) PAIR_TRACE(pit, 4);
          mbar_wait(bar_a_empty + 8 * sa, pa);
          if (s == 0) PAIR_TRACE(pit, 5);
          const uint32_t bar = bar_a_full + 8 * sa;
          const uint32_t dst = a_ring + sa * a.patch_bytes;
          mbar_arrive_expect_tx(bar, a.box_bytes);
#pragma unroll
          for (int j = 0; j < MT; ++j) tma_load_2d(dst + j * (a.box_rows * ROW_BYTES), &maps.in, bar, s * 64, row0 + j * a.box_rows);
          if (++sa == n_sa) { sa = 0; pa ^= 1; }
        }
      }
    }
  } else if (warp == 4 * NWG + 2) {
    // ================================================================== weight (B) producer: MY half of the columns
    if (lane == 0) {
      const __nv_bfloat16* wsrc = a.wgt_pair + static_cast<long long>(rank) * a.half_elems;  // (+ 2 half_elems per n-tile)
      if (a.resident) {
        mbar_arrive_expect_tx(bar_w_full, a.wbytes_half);
        const uint8_t* src = reinterpret_cast<const uint8_t*>(wsrc);
        for (uint32_t off = 0; off < a.wbytes_half; off += 16384)
          bulk_g2s(sbase + a.off_w + off, src + off, min(16384u, a.wbytes_half - off), bar_w_full);
      } else {
        const uint32_t b_ring = sbase + a.off_b;
        uint32_t sbi = 0, pb = 1;
        const uint32_t n_sb = a.sb;
        for (int pt = pair; pt < pair_tiles; pt += npairs) {
          const __nv_bfloat16* wnt = wsrc + static_cast<long long>(pt % a.n_tiles) * 2 * a.half_elems;
          for (int s = 0; s < a.slabs; ++s) {
            for (int t = 0; t < TAPS; t += TPS) {
              mbar_wait(bar_b_empty + 8 * sbi, pb);
              const uint32_t bar = bar_b_full + 8 * sbi;
              mbar_arrive_expect_tx(bar, a.bstage_bytes);
              bulk_g2s(b_ring + sbi * a.bstage_bytes, wnt + static_cast<long long>(s * TAPS + t) * 8 * a.n_half * 8, a.bstage_bytes, bar);
              if (++sbi == n_sb) { sbi = 0; pb ^= 1; }
            }
          }
        }
      }
    }
  } else {
    // ================================================================== epilogue I/O warp: residual tile in, finished tile out
    pdl_wait();
    auto load_res = [&](int pt, uint32_t slot, uint32_t phase) {
      const int mt_i = pt / a.n_tiles, n0 = (pt - mt_i * a.n_tiles) * a.n_tile;
      const int cx = static_cast<int>((static_cast<long long>(mt_i) * 2 + rank) * TM);
      mbar_wait(bar_res_empty + 8 * slot, phase ^ 1);
      if (lane == 0) {
        const uint32_t rbar = bar_res_full + 8 * slot;
        const uint32_t rdst = sbase + a.off_stage + slot * a.stage_buf_bytes;
        mbar_arrive_expect_tx(rbar, a.res_tx_bytes);
        for (int q = 0; q < a.pieces; ++q) tma_load_2d(rdst + a.piece_off[q], &maps.res, rbar, n0 + q * 64, cx);
      }
      __syncwarp();
    };
    const int nres = a.res_mode ? a.nstage : 0;
    uint32_t lslot = 0, lphase = 0;
    int ahead = pair;
    for (int k = 0; k < nres && ahead < pair_tiles; ++k, ahead += npairs) {
      load_res(ahead, lslot, lphase);
      if (++lslot == static_cast<uint32_t>(nres)) { lslot = 0; lphase ^= 1; }
    }
    int io_it = 0;
    for (int pt = pair; pt < pair_tiles; pt += npairs, ++io_it) {
      const int mt_i = pt / a.n_tiles, n0 = (pt - mt_i * a.n_tiles) * a.n_tile;
      const int cx = static_cast<int>((static_cast<long long>(mt_i) * 2 + rank) * TM);
      const int sbuf = a.nstage == 2 ? (io_it & 1) : 0;
      const uint32_t src = sbase + a.off_stage + sbuf * a.stage_buf_bytes;
      asm volatile("bar.sync %0, %1;" ::"r"(2 + (io_it & 1)), "n"(128 * NWG + 32) : "memory");
      if (lane == 0) {
        for (int q = 0; q < a.pieces; ++q) tma_store_2d(&maps.out, src + a.piece_off[q], n0 + q * 64, cx);
        bulk_commit();
        bulk_wait_read_all();
        mbar_arrive(bar_stage_free + 8 * sbuf);
      }
      __syncwarp();
      if (nres && ahead < pair_tiles) {
        load_res(ahead, lslot, lphase);
        if (++lslot == static_cast<uint32_t>(nres)) { lslot = 0; lphase ^= 1; }
        ahead += npairs;
      }
    }
    if (lane == 0) bulk_wait_all();
  }
  __syncthreads();
  tc_fence_before();
  cluster_sync_all();  // the peer may still be reading its accumulator / receiving commits until here
  if (warp == 4 * NWG) {
    tc_fence_after();
    tc_dealloc2(tmem_base, a.tmem_cols);
  }
}

typedef void (*PairKernelFn)(const PairArgs, const PairMaps);
template <int MT, int TPS>
PairKernelFn pick_pair(int act) {
  if (act == 1) return conv_pair_kernel<MT, 1, TPS>;
  if (act == 2) return conv_pair_kernel<MT, 2, TPS>;
  return conv_pair_kernel<MT, 0, TPS>;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
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

}  // namespace

// host: [K / 8][cout_pad][8] -> [rank][slab][tap][8 K chunks][cout_pad / 2][8]: each CTA of a pair keeps half of the
// output channels, laid out in the order the MMAs consume them (any run of taps of a slab is one bulk copy)
int pack_pair_weights(PackedConv* pc) {
  const int cout_pad = (pc->cout + 15) / 16 * 16;
  if (pc->w_pair || pc->ksize != 3 || pc->stride != 1 || pc->s2d_c0 || pc->cin_pad % 64 ||
      (cout_pad != 64 && cout_pad != 128 && cout_pad % 256 != 0) || cout_pad > 512 || pc->cout != cout_pad)
    return AICAM_OK;
  const size_t elems = static_cast<size_t>(pc->q_pad) * cout_pad * 8;
  std::vector<uint16_t> src(elems), dst(elems);
  AICAM_CUDA_OK(cudaMemcpy(src.data(), pc->w, elems * 2, cudaMemcpyDeviceToHost));
  const int n_tile = std::min(cout_pad, 256), nh = n_tile / 2, slabs = pc->cin_pad / 64;
  if (pc->q_pad * 8 != 9 * pc->cin_pad) return AICAM_OK;
  for (int sl = 0; sl < slabs; ++sl)
    for (int t = 0; t < 9; ++t)
      for (int c8 = 0; c8 < 8; ++c8) {
        const int q = (t * pc->cin_pad + sl * 64) / 8 + c8;
        for (int o = 0; o < cout_pad; ++o) {
          const int half = o / nh;  // = n-tile * 2 + rank
          std::memcpy(&dst[((((static_cast<size_t>(half) * slabs + sl) * 9 + t) * 8 + c8) * nh + o % nh) * 8],
                      &src[(static_cast<size_t>(q) * cout_pad + o) * 8], 16);
        }
      }
  AICAM_CUDA_OK(cudaMalloc(&pc->w_pair, elems * 2));
  AICAM_CUDA_OK(cudaMemcpy(pc->w_pair, dst.data(), elems * 2, cudaMemcpyHostToDevice));
  return AICAM_OK;
}

// Returns 1 when launched on the pair kernel, 0 when the layer is not eligible, negative on error.
int try_launch_conv_pair(const PackedConv& pc, const ConvLaunch& L, cudaStream_t stream) {
  static const bool enabled = getenv("AICAM_NO_PAIR") == nullptr;
  if (!enabled || !pc.w_pair || !L.in_pad || !L.out_pad || L.out_f32 || L.out_s2d || encode_tiled_fn() == nullptr) return 0;
  const int cout_pad = (pc.cout + 15) / 16 * 16;
  // Measured on B200 (1024 crops, same box, conv_win.cu mode 4 -> pairs): 128 channels 146 -> 135 us; 64 channels
  // 203 -> 190..224 us (the epilogue's shared-memory traffic competes with an operand fetch that now keeps the port 95 %
  // busy); 256 / 512 channels 148 -> 158 us and 197 -> 198 us (the 256-column single-CTA tile is already tensor-bound).
  // So only the 128- and 512-channel layers run on pairs.
  if (cout_pad != 128 && cout_pad != 512) return 0;  // (512 channels: 204 -> 195 us with the deeper weight ring)
  const int n_tile = std::min(cout_pad, 256), n_half = n_tile / 2, n_tiles = cout_pad / n_tile;
  const int tps = n_tile == 256 ? 1 : 3;
  const int res_mode = L.res ? L.res_mode : 0;
  if (L.in_pad != L.out_pad) return 0;
  const int hp = L.h + pad_ext(L.in_pad), wp = L.w + pad_ext(L.in_pad);
  if (L.in_cstride % 8 || L.in_coff % 8 || L.out_cstride % 8 || L.out_coff % 8 || (res_mode && (L.res_cstride % 8 || L.res_coff % 8))) return 0;
  if (L.in_img_stride != static_cast<long long>(hp) * wp * L.in_cstride || L.out_img_stride != static_cast<long long>(hp) * wp * L.out_cstride ||
      (res_mode && L.res_img_stride != static_cast<long long>(hp) * wp * L.res_cstride))
    return 0;
  const long long padded_pixels = static_cast<long long>(L.batch) * hp * wp;
  if (padded_pixels >= (1ll << 31) || L.batch <= 0) return 0;
  const int slabs = pc.cin_pad / 64;
  const size_t wbytes_half = static_cast<size_t>(pc.q_pad) * n_half * 16;
  const bool resident = wbytes_half <= 100 * 1024 && n_tiles == 1;
  const uint32_t bstage = static_cast<uint32_t>(tps) * 8u * n_half * 16u;  // tps taps x one 64-channel slab x my half of the columns
  const int pieces = n_tile / 64;

  // tiling: MT accumulators per CTA; staging = the TMA-epilogue tile (residual finished in place)
  int best_mt = 0, best_sa = 0, best_sb = 0, best_nstage = 0, best_bh = 0;
  for (int mt = 2; mt >= 1; --mt) {
    if (2 * mt * n_tile > 512) continue;
    const int tm = 128 * mt;
    const int bh = ((tm + 2 * wp + 2 + mt - 1) / mt + 7) / 8 * 8;
    if (bh > 256) continue;
    const size_t patch = static_cast<size_t>(mt) * bh * ROW_BYTES;
    const size_t stage_buf = static_cast<size_t>(pieces) * tm * 128;
    const size_t wsm = resident ? (wbytes_half + 1023) / 1024 * 1024 : 0;
    // two staging buffers where they fit (the residual load of tile i + 1 then overlaps the epilogue of tile i),
    // at least two patches and three weight stages in flight
    // (streamed weights: a tile's MMAs outlast the store -> residual-load chain of a single staging buffer, and the
    //  weight ring needs the shared memory more: every stage makes a relay hop through the peer)
    for (int nstage = resident ? 2 : 1; nstage >= 1 && !best_mt; --nstage) {
      const size_t fixed = OFF_RING_A + wsm + nstage * stage_buf + 1024;
      if (fixed + 2 * patch + (resident ? 0 : 3 * static_cast<size_t>(bstage)) > SMEM_LIMIT) continue;
      int sa = 2, sb = resident ? 1 : 3;
      size_t used = fixed + sa * patch + (resident ? 0 : static_cast<size_t>(sb) * bstage);
      if (!resident)
        while (sb < MAX_RING && used + bstage + (sa < 3 ? patch : 0) <= SMEM_LIMIT) { ++sb; used += bstage; }
      while (sa < std::max(3, 2 * slabs) && sa < MAX_RING && used + patch <= SMEM_LIMIT) { ++sa; used += patch; }
      best_mt = mt; best_sa = sa; best_sb = sb; best_nstage = nstage; best_bh = bh;
    }
    if (best_mt) break;
  }
  if (!best_mt) return 0;
  const int mt = best_mt, tm = 128 * mt;
  PairArgs a;
  std::memset(&a, 0, sizeof(a));
  static const bool thread_arrive = getenv("AICAM_WIN_THREAD_ARRIVE") != nullptr;
  a.warp_arrive = thread_arrive ? 0 : 1;
  a.h = L.h; a.w = L.w; a.hw = hp * wp; a.rw = wp; a.lo = pad_lo(L.in_pad);
  a.slabs = slabs; a.cin_pad = pc.cin_pad;
  a.sa = best_sa; a.sb = best_sb; a.resident = resident ? 1 : 0;
  a.box_rows = best_bh;
  a.box_bytes = static_cast<uint32_t>(mt) * best_bh * ROW_BYTES;
  a.patch_bytes = a.box_bytes;
  a.bstage_bytes = bstage; a.wbytes_half = static_cast<uint32_t>(wbytes_half);
  a.n_tile = n_tile; a.n_half = n_half; a.cout = pc.cout; a.n_tiles = n_tiles; a.tps = tps;
  a.wgt_pair = pc.w_pair; a.half_elems = static_cast<long long>(pc.q_pad) * n_half * 8;
  a.res_mode = res_mode;
  if (!pc.bias_host) return 0;
  std::memcpy(a.bias4, pc.bias_host, sizeof(float) * cout_pad);
  a.batch = L.batch; a.batch_dev = L.batch_dev;
  a.trace = L.trace;
  // instruction descriptor: fp32 accumulate, bf16 A / B, K-major, N = n_tile, M = 256 (the pair)
  a.idesc = (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n_tile >> 3) << 17) | (static_cast<uint32_t>(256 >> 4) << 24);
  uint32_t cols = 32;
  while (cols < static_cast<uint32_t>(2 * mt * n_tile)) cols <<= 1;
  a.tmem_cols = cols;
  const uint32_t ring_end = OFF_RING_A + static_cast<uint32_t>(best_sa) * a.patch_bytes;
  a.off_w = ring_end; a.off_b = ring_end;
  a.off_stage = (ring_end + static_cast<uint32_t>(resident ? (wbytes_half + 1023) / 1024 * 1024 : static_cast<size_t>(best_sb) * bstage) + 1023) / 1024 * 1024;
  a.stage_buf_bytes = static_cast<uint32_t>(pieces) * tm * 128;
  a.nstage = best_nstage; a.pieces = pieces;
  for (int q = 0; q < pieces; ++q) a.piece_off[q] = static_cast<uint32_t>(q) * tm * 128;
  a.res_tx_bytes = a.stage_buf_bytes;
  const size_t smem = a.off_stage + static_cast<size_t>(best_nstage) * a.stage_buf_bytes;
  if (smem > SMEM_LIMIT) return 0;

  alignas(64) PairMaps maps;
  std::memset(&maps, 0, sizeof(maps));
  const cuuint32_t estr[2] = {1, 1};
  {
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(pc.cin_pad), static_cast<cuuint64_t>(padded_pixels)};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(L.in_cstride) * 2};
    const cuuint32_t box[2] = {64, static_cast<cuuint32_t>(best_bh)};
    if (encode_tiled_fn()(&maps.in, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<__nv_bfloat16*>(L.in) + L.in_coff, dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return 0;
  }
  {
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(pc.cout), static_cast<cuuint64_t>(padded_pixels)};
    const cuuint32_t box[2] = {64, static_cast<cuuint32_t>(tm)};
    const cuuint64_t os[1] = {static_cast<cuuint64_t>(L.out_cstride) * 2};
    if (encode_tiled_fn()(&maps.out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, static_cast<__nv_bfloat16*>(L.out) + L.out_coff, dims, os, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return 0;
    if (res_mode) {
      const cuuint64_t rs[1] = {static_cast<cuuint64_t>(L.res_cstride) * 2};
      if (encode_tiled_fn()(&maps.res, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<__nv_bfloat16*>(L.res) + L.res_coff, dims, rs, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
        return 0;
    }
  }
  static const bool debug_plan = getenv("AICAM_WIN_DEBUG") != nullptr;
  if (debug_plan)
    fprintf(stderr, "conv_pair: %dx%d c%d->%d mt %d n_tile %d resident %d sa %d sb %d patch %u bstage %u nstage %d smem %zu\n", L.h, L.w,
            pc.cin_pad, pc.cout, mt, n_tile, a.resident, a.sa, a.sb, a.patch_bytes, a.bstage_bytes, a.nstage, smem);
  PairKernelFn kernel = tps == 1 ? pick_pair<1, 1>(L.act) : (mt == 2 ? pick_pair<2, 3>(L.act) : pick_pair<1, 3>(L.act));
  if (int rc = ensure_dynamic_smem(kernel, SMEM_LIMIT)) return rc;  // per (device, instantiation)
  const int num_sms = current_num_sms();
  const long long pair_tiles = (padded_pixels + 2 * tm - 1) / (2 * tm) * n_tiles;
  const unsigned pairs = static_cast<unsigned>(std::min<long long>(pair_tiles, num_sms / 2));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * pairs); cfg.blockDim = dim3(PAIR_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  static const bool no_pdl = getenv("AICAM_NO_PDL") != nullptr;
  cfg.attrs = attr; cfg.numAttrs = no_pdl ? 1 : 2;
  size_t slot = 0;
  const bool prof = profile_begin(stream, &slot);
  const cudaError_t le = cudaLaunchKernelEx(&cfg, kernel, a, maps);
  if (prof) profile_end(stream, slot);
  if (le != cudaSuccess) return fail(AICAM_ERR_CUDA, std::string("conv_pair: launch failed: ") + cudaGetErrorString(le));
  count_launch();
  const int rc = last_launch("conv_pair_kernel");
  return rc ? rc : 1;
}

}  // namespace aicam
