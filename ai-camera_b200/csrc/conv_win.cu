// "Window" convolution on tcgen05 tensor cores: 3x3 / stride 1 / pad 1 and 1x1 / stride 1 layers, sm_100a.
//
// Same operator as conv_tc.cu (the layers the reference hands to its TensorRT engines,
// /root/reference/src/trt_utils/trt_engine.py:191), different data movement.  conv_tc.cu builds an
// im2col A tile per filter tap, so a 3x3 layer pulls every input pixel through L2 nine times and
// re-streams the whole weight tensor for every 128-pixel tile; measured on B200 that traffic
// (~57 B/clk/SM), not the tensor pipe, bounds the small-channel layers.  Here:
//
//   * ONE tiled TMA load per (tile, 64-channel slab) brings a haloed input patch
//     [rows][raster width RW = strip width + 2][slab] into shared memory (hardware 32/64/128-byte
//     swizzle, out-of-image halo pixels zero-filled by the TMA unit = the convolution's padding);
//   * output positions are enumerated in the patch's own raster (row pitch RW), so the A operand of
//     filter tap (dy, dx) is the SAME shared-memory patch read through a UMMA descriptor whose start
//     address is advanced by (dy*RW + dx) pixels: nine taps, zero extra bytes.  The two raster
//     columns per row that have no output pixel produce junk accumulator rows that are never stored;
//   * weights stay resident in shared memory for the life of the persistent CTA when they fit
//     (<= 120 KB, all YOLOv8n 3x3 layers up to 80 channels and the ReID 64-channel stage), otherwise
//     they stream through a 4-deep ring, each block feeding `mt` (1 or 2) 128-row accumulators;
//   * accumulators are double-buffered in TMEM (2 x mt x n_tile columns), so the epilogue of tile i
//     (TMEM -> registers -> bias / residual / activation -> staging -> coalesced 16-byte stores)
//     overlaps the MMAs of tile i+1; the epilogue is warp-local (no block barriers).
//
// Warp roles (608 threads): 0-15 epilogue (four warpgroups split the accumulator columns; TMEM lane
// quarter = warp % 4), 16 MMA issuer (one thread) + TMEM owner, 17 patch (A) producer, 18 weight (B) producer.
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

constexpr int NWG = 4;                          // epilogue warpgroups
constexpr int WIN_THREADS = (4 * NWG + 4) * 32;  // + MMA issuer, patch producer, weight producer, epilogue I/O warp
constexpr int MAX_RING = 8;
constexpr uint32_t OFF_BIAS = 512;      // fp32 bias, <= 512 channels
constexpr uint32_t OFF_ROWOFF = 2560;   // 2 tile parities x (output, residual) x 8 teams x 32 rows x int64 element offsets
constexpr uint32_t OFF_RING_A = 11264;   // 1024-byte aligned: swizzle patterns repeat every 1024 B
constexpr uint32_t OFF_RING_A_EPI = 3072;  // TMA epilogue: no row-offset tables, the operand ring starts right after the bias
constexpr size_t SMEM_LIMIT = 227 * 1024;
constexpr size_t RESIDENT_LIMIT = 120 * 1024;

// tensor maps of one launch: the input (patch / flat / im2col), and for the TMA epilogue the output and the
// residual, one map per channel piece (<= 64 channels = one 128-byte swizzled row)
struct WinMaps {
  CUtensorMap in;
  CUtensorMap out[2];
  CUtensorMap res[2];
};

struct WinArgs {
  int mode;  // 0: 3x3 window over 4-D patches, 1: 1x1 over the flat [pixels][channels] matrix
  int h, w, hw;
  int rw, tw, strips, tstep, tiles_per_strip, tiles_per_img;
  float inv_rw;
  // TMA epilogue (window modes, row-aligned tiles): compact staging tile [th * tw rows][piece channels], swizzled
  int th;                 // raster rows per tile
  int pieces;             // channel pieces of an n-tile: 1 or 2, or four 64-channel pieces (n_tile = 256)
  int piece_ch[4];        // channels per piece: 64 / 32 / 16
  uint32_t piece_off[4];  // byte offset of the piece inside a staging buffer (1024-aligned)
  uint32_t stage_buf_bytes, res_tx_bytes;
  int nres;               // residual staging buffers (TMA-loaded one or two tiles ahead)
  int nstage;             // output staging buffers (2: the store of tile i overlaps the staging of tile i + 1)
  long long* trace;       // debug: clock64 stamps of CTA 0 (AICAM_CONV_TRACE in aicam_conv2d_bench)
  long long* tl;          // debug (aicam_debug_timeline): %globaltimer of CTA 0 at entry / dependency resolved / exit
  int res_direct;  // residual read straight from global in the finish phase (no staging): deep, streamed layers
  int out_s2d;  // window modes: the output is stored space-to-depth: [h/2][w/2][2x2 sub-pixel][out_cstride]
  int flat;  // 1x1 mode: output and residual are dense, pixel p of the batch sits at p * cstride
  int out_pad;   // flat / im2col modes: output (and residual) images carry a zero border: extra rows / columns per image ...
  int out_lo;    // ... and the offset of the interior in it (conv_tc.cuh: pad kinds)
  int in_lo;     // mode 4: offset of the interior inside the padded raster (1 symmetric border, 0 shared border)
  int box_rows;  // mode 4: raster rows per TMA box (a patch is MT boxes)
  int s2d_store;    // TMA epilogue of a space-to-depth output: the tile is stored through a 5-D map (2C, x/2, y&1, y/2, n) whose
                    // box image is the plain compact [y][x][C] staging tile (no swizzle); tile origins and sizes are even
  int epi_alt;      // TMA epilogue, two accumulators per tile, narrow n-tiles: the two column teams take ALTERNATE tiles
                    // (all columns each) instead of half the columns of every tile - each team then has two tile times
                    // for its latency chain (TMEM read -> finish -> staging -> store hand-off)
  int res_inplace;  // TMA epilogue: the residual tile is loaded INTO the output staging buffer and finished in place
                    // (no residual ring): the store of tile i is followed by the residual load of tile i + nstage
  int warp_arrive;  // epilogue -> MMA / I/O hand-offs: one elected lane per warp arrives on the mbarriers (default) instead of every
                    // thread: 32 same-address arrives serialise on the shared-memory port the tensor core reads its operands through
  int pad_store;    // im2col mode, TMA epilogue, zero-bordered output: a tile is whole rows of one image or whole images, stored as ONE 4-D box
                    // (channels, wo, rows, images) into the interiors - the generic epilogue's row-by-row copy-out was half of its tile time
  int img_tile;     // mode 4 on 8-pixel-wide maps of 128 pixels (ReID layer 3): a tile is ONE image's interior - accumulator row 8 y + x - read
                    // through a descriptor whose 8-row groups are a raster row (RW pixels) apart, so the border column and row cost no MMA
                    // rows (84 % -> 100 % useful); stored / residual-loaded as one 4-D box like pad_store
  int ws;           // MMA issue in the weight-stationary form (tcgen05.mma.ws, collector buffers for B)
  int decode;       // generic epilogue of a Detect-head 1x1 layer: decode the staged fp32 rows instead of storing them (ConvLaunch::decode)
  int dec_anchor_base, dec_anchors;
  float dec_stride;
  float* dec_boxes;
  float* dec_scores;
  int* dec_labels;
  int direct_out;  // generic epilogue: every thread stores its finished 32-byte groups straight to global (whole
                   // sectors, no staging tile): deep streamed layers spend the shared memory on operand rings instead
  int mt, tm;
  int slab, slabs, taps, cin_pad;
  int ksize, stride, pad, wo, slabs_per_tap;  // im2col mode: filter geometry, output width, channel slabs per tap
  int resident, sa, sb;
  uint32_t patch_bytes, box_bytes, bstage_bytes, wbytes;
  int n_tile, n_tiles, cout, cout_pad;
  const __nv_bfloat16* wgt;
  const __nv_bfloat16* wgt_nt;  // n-tile-major copy ([n-tile][K chunk][n_tile][8]) or null
  int q_pad;                    // K chunks per n-tile block of wgt_nt
  const float* bias;
  void* out;
  long long out_img_stride;
  int out_cstride, out_coff, out_f32;
  const __nv_bfloat16* res;
  long long res_img_stride;
  int res_cstride, res_coff, res_mode;
  int act;
  int batch;
  const int* batch_dev;
  uint32_t idesc, tmem_cols;
  uint32_t off_w, off_b, off_stage, off_res, stage_pitch, res_pitch;
  float4 bias4[128];  // TMA epilogue: the bias (<= 512 channels) read from the constant bank, not from shared memory
};

__device__ __forceinline__ long long global_timer_ns() {
  long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

__device__ __forceinline__ float silu_fast(float x) {
  // x * sigmoid(x) = h + h * tanh(h), h = x / 2: one MUFU instead of two
  const float h = 0.5f * x;
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}

// tcgen05.mma with the two 64-bit descriptors passed as (lo, hi) halves: the issuing warp only
// ever adds to the low halves (start address >> 4), the high halves are loop constants.  Executed by
// the whole (converged) warp, performed by the lane whose `leader` predicate is set.
__device__ __forceinline__ void mma_issue(bool leader, uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo,
                                          uint32_t b_hi, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "setp.ne.b32 q, %7, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}" ::"r"(tmem_d),
      "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate), "r"(static_cast<uint32_t>(leader))
      : "memory");
}
// Weight-stationary form (tcgen05.mma.ws): the B block (weights of one tap / K step) is kept in collector buffer BUF - COP 0: fill
// (fetch from shared memory and keep), 1: lastuse (take it from the collector: no shared-memory fetch), 2: discard (fetch, do not keep).
// Consecutive MMAs of the accumulators of one tile share their weights, so only the first of them reads B through the port.
template <int COP>
__device__ __forceinline__ void mma_issue_ws(int BUF, bool leader, uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo,
                                             uint32_t b_hi, uint32_t idesc, uint32_t accumulate) {
#define AICAM_WS_ASM(BUFS, OPS)                                                                                        \
  asm volatile(                                                                                                        \
      "{\n\t.reg .pred p, q;\n\t.reg .b64 da, db;\n\t"                                                               \
      "setp.ne.b32 p, %6, 0;\n\t"                                                                                      \
      "setp.ne.b32 q, %7, 0;\n\t"                                                                                      \
      "mov.b64 da, {%1, %2};\n\t"                                                                                      \
      "mov.b64 db, {%3, %4};\n\t"                                                                                      \
      "@q tcgen05.mma.ws.cta_group::1.kind::f16.collector::" BUFS "::" OPS " [%0], da, db, %5, p;\n\t}" ::"r"(tmem_d), \
      "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate), "r"(static_cast<uint32_t>(leader))      \
      : "memory")
#define AICAM_WS_BUF(BUFS)                         \
  do {                                             \
    if (COP == 0) AICAM_WS_ASM(BUFS, "fill");      \
    else if (COP == 1) AICAM_WS_ASM(BUFS, "lastuse"); \
    else AICAM_WS_ASM(BUFS, "discard");            \
  } while (0)
  if (BUF == 0) AICAM_WS_BUF("b0");
  else if (BUF == 1) AICAM_WS_BUF("b1");
  else if (BUF == 2) AICAM_WS_BUF("b2");
  else AICAM_WS_BUF("b3");
#undef AICAM_WS_BUF
#undef AICAM_WS_ASM
}
__device__ __forceinline__ void tc_commit_if(bool leader, uint32_t bar) {
  asm volatile(
      "{\n\t.reg .pred q;\n\t"
      "setp.ne.b32 q, %1, 0;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(bar),
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
  if (ACT == 1) return silu_fast(x);
  if (ACT == 2) return fmaxf(x, 0.0f);
  return x;
}

// One 16-column group of an accumulator row: + bias (+ residual), activation, pack into the staging row.
template <int ACT>
__device__ __forceinline__ void finish_group(const uint32_t (&v)[16], const float* bias, const uint8_t* res_row,
                                             int res_mode, int out_f32, uint8_t* dst, const uint8_t* res_hi = nullptr,
                                             uint8_t* dst_hi = nullptr) {
  // res_hi / dst_hi: address of the second 16-byte chunk when it is not adjacent (swizzled staging)
  if (res_hi == nullptr) res_hi = res_row + 16;
  if (dst_hi == nullptr) dst_hi = dst + 16;
  float x[16];
  const float4* bp = reinterpret_cast<const float4*>(bias);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 b4 = bp[i];
    x[4 * i] = __uint_as_float(v[4 * i]) + b4.x;
    x[4 * i + 1] = __uint_as_float(v[4 * i + 1]) + b4.y;
    x[4 * i + 2] = __uint_as_float(v[4 * i + 2]) + b4.z;
    x[4 * i + 3] = __uint_as_float(v[4 * i + 3]) + b4.w;
  }
  if (res_mode) {
    const uint4 q0v = *reinterpret_cast<const uint4*>(res_row);
    const uint4 q1v = *reinterpret_cast<const uint4*>(res_hi);
    const uint32_t rw_[8] = {q0v.x, q0v.y, q0v.z, q0v.w, q1v.x, q1v.y, q1v.z, q1v.w};
    if (res_mode == 2) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        x[2 * i] = activate<ACT>(x[2 * i] + bf16_lo(rw_[i]));
        x[2 * i + 1] = activate<ACT>(x[2 * i + 1] + bf16_hi(rw_[i]));
      }
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        x[2 * i] = activate<ACT>(x[2 * i]) + bf16_lo(rw_[i]);
        x[2 * i + 1] = activate<ACT>(x[2 * i + 1]) + bf16_hi(rw_[i]);
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < 16; ++i) x[i] = activate<ACT>(x[i]);
  }
  if (out_f32) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
      *reinterpret_cast<float4*>(dst + i * 16) = make_float4(x[4 * i], x[4 * i + 1], x[4 * i + 2], x[4 * i + 3]);
  } else {
    uint4 o0, o1;
    o0.x = pack_bf16x2(x[0], x[1]);   o0.y = pack_bf16x2(x[2], x[3]);
    o0.z = pack_bf16x2(x[4], x[5]);   o0.w = pack_bf16x2(x[6], x[7]);
    o1.x = pack_bf16x2(x[8], x[9]);   o1.y = pack_bf16x2(x[10], x[11]);
    o1.z = pack_bf16x2(x[12], x[13]); o1.w = pack_bf16x2(x[14], x[15]);
    *reinterpret_cast<uint4*>(dst) = o0;
    *reinterpret_cast<uint4*>(dst_hi) = o1;
  }
}

// the same with the bias already in registers and bf16 output (TMA epilogue)
template <int ACT>
__device__ __forceinline__ void finish_group_b(const uint32_t (&v)[16], const float (&b)[16], const uint8_t* res_row, int res_mode,
                                               uint8_t* dst, const uint8_t* res_hi, uint8_t* dst_hi) {
  float x[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) x[i] = __uint_as_float(v[i]) + b[i];
  if (res_mode) {
    const uint4 q0v = *reinterpret_cast<const uint4*>(res_row);
    const uint4 q1v = *reinterpret_cast<const uint4*>(res_hi);
    const uint32_t rw_[8] = {q0v.x, q0v.y, q0v.z, q0v.w, q1v.x, q1v.y, q1v.z, q1v.w};
    if (res_mode == 2) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        x[2 * i] = activate<ACT>(x[2 * i] + bf16_lo(rw_[i]));
        x[2 * i + 1] = activate<ACT>(x[2 * i + 1] + bf16_hi(rw_[i]));
      }
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        x[2 * i] = activate<ACT>(x[2 * i]) + bf16_lo(rw_[i]);
        x[2 * i + 1] = activate<ACT>(x[2 * i + 1]) + bf16_hi(rw_[i]);
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < 16; ++i) x[i] = activate<ACT>(x[i]);
  }
  uint4 o0, o1;
  o0.x = pack_bf16x2(x[0], x[1]);   o0.y = pack_bf16x2(x[2], x[3]);
  o0.z = pack_bf16x2(x[4], x[5]);   o0.w = pack_bf16x2(x[6], x[7]);
  o1.x = pack_bf16x2(x[8], x[9]);   o1.y = pack_bf16x2(x[10], x[11]);
  o1.z = pack_bf16x2(x[12], x[13]); o1.w = pack_bf16x2(x[14], x[15]);
  *reinterpret_cast<uint4*>(dst) = o0;
  *reinterpret_cast<uint4*>(dst_hi) = o1;
}

// Detect-head decode inside the generic epilogue (ConvLaunch::decode) - the arithmetic of decode_kernel (detect_post.cu,
// compiled without FMA contraction: the multiply-add of the DFL expectation is spelled out here).  A 16-column accumulator
// group of the box branch IS one DFL side: the thread that holds it in registers reduces it to the side's expected distance.
__device__ __forceinline__ float dfl_side(const uint32_t (&v)[16], const float* bias) {
  float x[16];
  const float4* bp = reinterpret_cast<const float4*>(bias);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 b4 = bp[i];
    x[4 * i] = __uint_as_float(v[4 * i]) + b4.x;
    x[4 * i + 1] = __uint_as_float(v[4 * i + 1]) + b4.y;
    x[4 * i + 2] = __uint_as_float(v[4 * i + 2]) + b4.z;
    x[4 * i + 3] = __uint_as_float(v[4 * i + 3]) + b4.w;
  }
  float m = x[0];
#pragma unroll
  for (int i = 1; i < 16; ++i) m = fmaxf(m, x[i]);
  float s = 0.0f, ws = 0.0f;
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const float e = expf(x[i] - m);
    s = __fadd_rn(s, e);
    ws = __fadd_rn(ws, __fmul_rn(e, static_cast<float>(i)));
  }
  return __fdiv_rn(ws, s);
}
// class branch: running best logit of an ascending column scan (strict compare: the lowest class index wins ties)
__device__ __forceinline__ void cls_scan(const uint32_t (&v)[16], const float* bias, int c0, int ncols, float& best, int& bi) {
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const float x = __uint_as_float(v[i]) + bias[i];
    if (c0 + i < ncols && x > best) { best = x; bi = c0 + i; }
  }
}

// Tile index -> image, column strip and first raster position (window mode)
struct TilePos {
  int n_img, strip, q0;
};
__device__ __forceinline__ TilePos tile_pos(const WinArgs& a, int mt_idx) {
  TilePos t;
  t.n_img = mt_idx / a.tiles_per_img;
  const int r2 = mt_idx - t.n_img * a.tiles_per_img;
  t.strip = r2 / a.tiles_per_strip;
  t.q0 = (r2 - t.strip * a.tiles_per_strip) * a.tstep;
  return t;
}

// trace slot layout: [tile < 32][16 stamps]; who: 0-3 MMA warp, 4-5 producer, 8-13 epilogue thread 0
#define WIN_TRACE(it, who) do { if (a.trace && blockIdx.x == 0 && (it) < 32) a.trace[(it) * 16 + (who)] = clock64(); } while (0)

// EPIW: bit 0 = TMA epilogue, bit 1 = MMAs issued in the weight-stationary form (64-column tiles of the window modes)
template <int SLAB, int AMODE, int MT, int ACT, int EPIW>
__global__ void __launch_bounds__(WIN_THREADS, 1) conv_win_kernel(const __grid_constant__ WinArgs a, const __grid_constant__ WinMaps maps) {
  constexpr int EPI = EPIW & 1;
  constexpr bool WS = (EPIW & 2) != 0;
  constexpr uint32_t ROW_BYTES = SLAB * 2;
  constexpr int K16S = SLAB / 16;
  constexpr uint32_t LTYPE = SLAB == 64 ? 2u : (SLAB == 32 ? 4u : 6u);
  // 0: 3x3 window patches, 1: flat 1x1, 2: im2col TMA (any 1x1 / 3x3, stride 1 / 2),
  // 3: 2x2 window, pad 1 on the top / left only: a 3x3 stride-2 layer over its space-to-depth input
  //    (2x2 pixel blocks stored as one 4C-channel pixel; weights re-packed by pack_conv_weights_s2d)
  // 4: 3x3 stride 1 over zero-bordered ("padded") tensors: input, output and residual are [batch][h+2][w+2][c] with a
  //    zero border, so the WHOLE batch is one flat raster of padded pixels (row pitch RW = w + 2).  A tile is any TM
  //    consecutive raster positions, its patch the TM + 2 RW + 2 positions around it (one 2-D box per 128 rows, no
  //    per-image halo, no row alignment), tap (dy, dx) the patch shifted by dy RW + dx positions as in mode 0.
  //    Border positions produce junk accumulator rows that are never stored, so the border stays zero.
  constexpr bool WINDOW = AMODE == 0 || AMODE == 3;
  constexpr bool FLATWIN = AMODE == 4;
  constexpr int MODE = WINDOW ? 0 : (FLATWIN ? 1 : AMODE);
  constexpr int KW = AMODE == 3 ? 2 : 3;                        // window width in raster positions
  constexpr int TAPS = (AMODE == 0 || AMODE == 4) ? 9 : (AMODE == 3 ? 4 : 1);   // taps that share one A stage
  constexpr int TM = 128 * MT;
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar_a_full = sbase, bar_a_empty = sbase + 64, bar_b_full = sbase + 128, bar_b_empty = sbase + 192;
  const uint32_t bar_acc_full = sbase + 256, bar_acc_empty = sbase + 272, bar_w_full = sbase + 288;
  const uint32_t bar_res_full = sbase + 296, bar_res_empty = sbase + 312;  // TMA epilogue: residual staging ring
  const uint32_t bar_stage_free = sbase + 328;  // x2, TMA epilogue: the store that used the staging buffer has read it
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(smem + 352);
  float* bias_s = reinterpret_cast<float*>(smem + OFF_BIAS);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  int batch = a.batch;
  if (a.batch_dev) batch = min(batch, __ldg(a.batch_dev));
  long long m_tiles;
  if (MODE == 0) m_tiles = static_cast<long long>(batch) * a.tiles_per_img;
  else if (FLATWIN && a.img_tile) m_tiles = batch;
  else m_tiles = (static_cast<long long>(batch) * a.hw + TM - 1) / TM;
  const int total_tiles = static_cast<int>(m_tiles) * a.n_tiles;
  pdl_trigger();  // the next layer's CTAs may take over each SM as soon as the CTA here exits
  if (a.tl && blockIdx.x == 0 && threadIdx.x == 0) a.tl[0] = global_timer_ns();
  if (static_cast<int>(blockIdx.x) >= total_tiles) return;

  if (threadIdx.x == 0) {
    for (int s = 0; s < MAX_RING; ++s) {
      mbar_init(bar_a_full + 8 * s, 1);
      mbar_init(bar_a_empty + 8 * s, 1);
      mbar_init(bar_b_full + 8 * s, 1);
      mbar_init(bar_b_empty + 8 * s, 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(bar_acc_full + 8 * s, 1);
      mbar_init(bar_acc_empty + 8 * s, (a.epi_alt ? 64 * NWG : 128 * NWG) >> (a.warp_arrive ? 5 : 0));
    }
    mbar_init(bar_w_full, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(bar_res_full + 8 * s, 1);
      mbar_init(bar_res_empty + 8 * s, (a.epi_alt ? 64 * NWG : 128 * NWG) >> (a.warp_arrive ? 5 : 0));
    }
    mbar_init(bar_stage_free, 1);
    mbar_init(bar_stage_free + 8, 1);
    mbar_init_fence();
  }
  if (warp == 4 * NWG) tc_alloc(smem_u32(tmem_ptr_smem), a.tmem_cols);
  if (warp == 4 * NWG + 1 && lane == 0) tma_prefetch_desc(&maps.in);
  for (int i = threadIdx.x; i < a.cout_pad; i += WIN_THREADS) bias_s[i] = __ldg(a.bias + i);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  const uint32_t acc_cols = static_cast<uint32_t>(MT * a.n_tile);

  if (EPI == 1 && warp < 4 * NWG) {
    // ================================================================== epilogue, TMA flavour (16 warps)
    // Row-aligned window tiles: a tile is `th` whole raster rows, so its valid outputs are a th x tw box of
    // the output image.  Each thread finishes its accumulator row (column split as below) into a COMPACT
    // staging tile [y][x < tw][channels] written with the TMA swizzle; one thread then issues a tensor
    // store per channel piece - the hardware drops the box rows / columns that fall outside the image.
    // The residual arrives the same way (a box load issued by the patch producer one or two tiles ahead).
    // No per-row addresses, no validity tables, no copy loops.
    constexpr int PARTS = MT == 2 ? 2 : 4;
    const int wg = warp >> 2, wq = warp & 3;
    const int my_j = MT == 2 ? (wg >> 1) : 0;
    const int part = MT == 2 ? (wg & 1) : wg;
    const int r = my_j * 128 + wq * 32 + lane;  // my position inside the tile (tile-invariant)
    bool valid = true;
    int crow = r;                               // flat / im2col tiles: 128 MT consecutive pixels, already compact
    if (WINDOW) {
      const int y_l = r / a.rw, xp = r - y_l * a.rw;
      valid = r < a.tstep && xp < a.tw;
      crow = y_l * a.tw + xp;                   // my row of the compact tile
    }
    const uint32_t taddr_lane = tmem_base + (static_cast<uint32_t>(wq * 32) << 16);
    // per piece: byte offset of my row and the swizzle XOR of its 16-byte chunks
    uint32_t row_off[4], row_xor[4];
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      const uint32_t pb = static_cast<uint32_t>(a.piece_ch[p]) * 2;
      const uint32_t ro = static_cast<uint32_t>(crow) * pb;
      const uint32_t mask = pb == 128 ? 7u : (pb == 64 ? 3u : 1u);
      row_off[p] = a.piece_off[p] + ro;
      row_xor[p] = a.s2d_store ? 0u : ((ro >> 7) & mask) << 4;
    }
    uint8_t* stage0 = smem + a.off_stage;
    const uint8_t* res_base = smem + (a.res_inplace ? a.off_stage : a.off_res);
    const bool alt = MT == 2 && a.epi_alt != 0;
    const uint32_t hand_off = alt ? 64 * NWG + 32 : 128 * NWG + 32;  // threads on the epilogue -> I/O warp barrier
    int it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      if (alt && (it & 1) != part) continue;  // the other team's tile
      const int buf = it & 1;
      const uint32_t rslot = a.nres == 2 ? (it & 1) : 0, rphase = a.nres == 2 ? ((it >> 1) & 1) : (it & 1);
      const int mt_idx = a.n_tiles == 1 ? tile : tile / a.n_tiles;
      const int n0 = (tile - mt_idx * a.n_tiles) * a.n_tile;
      const int ncols = min(a.n_tile, a.cout - n0);
      const int groups = (ncols + 15) >> 4;
      const int g_lo = alt ? 0 : (groups * part) / PARTS, g_hi = alt ? groups : (groups * (part + 1)) / PARTS;
      if (threadIdx.x == 0) WIN_TRACE(it, 8);
      mbar_wait(bar_acc_full + 8 * buf, (it >> 1) & 1);
      tc_fence_after();
      if (threadIdx.x == 0) WIN_TRACE(it, 9);
      const uint8_t* res_buf = res_base + rslot * a.stage_buf_bytes;
      if (a.res_mode) mbar_wait(bar_res_full + 8 * rslot, rphase);
      if (threadIdx.x == 0) WIN_TRACE(it, 10);
      const uint32_t taddr = taddr_lane + buf * acc_cols + my_j * a.n_tile;
      // staging buffer of this tile and the parity of "its previous store has been read"
      const int sbuf = a.nstage == 2 ? (it & 1) : 0;
      const uint32_t sfree_bar = bar_stage_free + 8 * sbuf;
      const uint32_t sfree_par = (a.nstage == 2 ? ((it >> 1) & 1) : (it & 1)) ^ 1;
      uint8_t* stage = stage0 + sbuf * a.stage_buf_bytes;
      bool stage_ok = false;
      bool zero_row = false;
      if (FLATWIN && !a.img_tile) {  // my raster position of this tile: border positions are stored as zeros (the border stays zero)
        // (32-bit unsigned arithmetic: the host guarantees fewer than 2^31 padded pixels; the 64-bit modulo was 9 % of
        //  the kernel's instructions)
        const uint32_t p = static_cast<uint32_t>(mt_idx) * TM + r;
        const uint32_t rem = p % static_cast<uint32_t>(a.hw);
        const int yy = static_cast<int>(rem / static_cast<uint32_t>(a.rw)), xx = static_cast<int>(rem) - yy * a.rw;
        zero_row = !(yy >= a.in_lo && yy < a.in_lo + a.h && xx >= a.in_lo && xx < a.in_lo + a.w);
      }
      for (int g = g_lo; g < g_hi; g += 2) {
        uint32_t v0[16], v1[16];
        const bool two = g + 1 < g_hi;  // warp-uniform
        __syncwarp();
        tc_ld16_nowait(taddr + g * 16, v0);
        if (two) tc_ld16_nowait(taddr + g * 16 + 16, v1);
        if (!stage_ok) {  // the I/O warp's store of the previous tile has finished reading the staging tile
          mbar_wait(sfree_bar, sfree_par);
          stage_ok = true;
        }
        tc_ld_wait();
        if (valid) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            if (h == 1 && !two) break;
            const int c = (g + h) * 16;                      // first channel of the group inside the n-tile
            const int p = a.pieces > 2 ? (c >> 6) : (c < a.piece_ch[0] ? 0 : 1);  // (more than two pieces: all 64 wide)
            const uint32_t ch0 = static_cast<uint32_t>(a.pieces > 2 ? (c & 63) : c - (p ? a.piece_ch[0] : 0)) * 2;  // byte offset inside the piece row
            const uint32_t o0 = row_off[p] + (ch0 ^ row_xor[p]), o1 = row_off[p] + ((ch0 + 16) ^ row_xor[p]);
            if (FLATWIN && zero_row) {
              *reinterpret_cast<uint4*>(stage + o0) = make_uint4(0u, 0u, 0u, 0u);
              *reinterpret_cast<uint4*>(stage + o1) = make_uint4(0u, 0u, 0u, 0u);
            } else {
              float bv[16];
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float4 b4 = a.bias4[((n0 + c) >> 2) + i];
                bv[4 * i] = b4.x; bv[4 * i + 1] = b4.y; bv[4 * i + 2] = b4.z; bv[4 * i + 3] = b4.w;
              }
              finish_group_b<ACT>(h ? v1 : v0, bv, res_buf + o0, a.res_mode, stage + o0, res_buf + o1, stage + o1);
            }
          }
        }
      }
      if (!stage_ok) mbar_wait(sfree_bar, sfree_par);  // (no column group: keep the phases in step)
      tc_fence_before();
      if (a.warp_arrive) {
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(bar_acc_empty + 8 * buf);
          if (a.res_mode) mbar_arrive(bar_res_empty + 8 * rslot);
        }
      } else {
        mbar_arrive(bar_acc_empty + 8 * buf);
        if (a.res_mode) mbar_arrive(bar_res_empty + 8 * rslot);
      }
      if (threadIdx.x == 0) WIN_TRACE(it, 12);
      fence_proxy_async();  // my staging writes -> visible to the TMA unit
      // hand the tile to the I/O warp: arrive without waiting (it syncs on the same barrier).  Two barrier ids
      // alternate: a thread can be one tile ahead of the I/O warp, never two (the staging-buffer wait above)
      asm volatile("bar.arrive %0, %1;" ::"r"(2 + (it & 1)), "r"(hand_off) : "memory");
      if (threadIdx.x == 0) WIN_TRACE(it, 13);
    }
  } else if (warp < 4 * NWG) {
    // ================================================================== epilogue (16 warps)
    // The PARTS warps {wq + 4 p} that share TMEM lane quarter wq (rows 32 wq .. 32 wq + 31 of a
    // 128-row accumulator) form a team.  TMEM -> staging is split by COLUMNS inside the team (a warp
    // can only read its own lane quarter), the global <-> staging copies are split by ROWS so that
    // every copy instruction moves whole contiguous rows.  Two named barriers per tile keep the team
    // in step.  MT == 1: one team of 4 warps per quarter; MT == 2: two teams of 2 (one per accumulator).
    constexpr int PARTS = MT == 2 ? 2 : 4;
    constexpr int ROWS_PER_WARP = 32 / PARTS;
    const int wg = warp >> 2, wq = warp & 3;
    const int my_j = MT == 2 ? (wg >> 1) : 0;
    const int part = MT == 2 ? (wg & 1) : wg;
    const int row = wq * 32 + lane;          // my accumulator row (TMEM lane)
    const int bar_id = 1 + my_j * 4 + wq;    // named barrier of my team
    const int bar_threads = 32 * PARTS;
    const uint32_t taddr_lane = tmem_base + (static_cast<uint32_t>(wq * 32) << 16);
    const int esize = a.out_f32 ? 4 : 2;
    const uint32_t pitch = a.stage_pitch, rpitch = a.res_pitch;
    uint8_t* stage_q = smem + a.off_stage + static_cast<size_t>(my_j * 128 + wq * 32) * pitch;  // my team's 32 rows
    uint8_t* my_stage = stage_q + static_cast<size_t>(lane) * pitch;
    uint8_t* res_q = smem + a.off_res + static_cast<size_t>(my_j * 128 + wq * 32) * rpitch;
    const uint8_t* my_res = res_q + static_cast<size_t>(lane) * rpitch;
    // element offsets of the team's 32 rows in the output / residual tensors (-1: not stored),
    // double-buffered by tile parity, written by the team's part-0 warp
    long long* rowoff_base = reinterpret_cast<long long*>(smem + OFF_ROWOFF) + (my_j * 4 + wq) * 32;
    uint8_t* out_bytes = reinterpret_cast<uint8_t*>(a.out);
    const long long total_pix = static_cast<long long>(batch) * a.hw;

    // publish where the team's rows of `tile` live (part-0 warp, lane = row)
    auto publish_rows = [&](int tile, int slot) {
      const int mt_idx = a.n_tiles == 1 ? tile : tile / a.n_tiles;
      const int n0 = (tile - mt_idx * a.n_tiles) * a.n_tile;
      bool valid;
      int img, pix;
      if (MODE == 0) {
        const TilePos tp = tile_pos(a, mt_idx);
        const int rel = my_j * 128 + row;
        const int q = tp.q0 + rel;
        const int y = __float2int_rd((static_cast<float>(q) + 0.5f) * a.inv_rw);  // exact: q < 2^18
        const int xp = q - y * a.rw;
        const int x = tp.strip * a.tw + xp;
        valid = rel < a.tstep && y < a.h && xp < a.tw && x < a.w;
        img = tp.n_img;
        pix = a.out_s2d ? (((y >> 1) * (a.w >> 1) + (x >> 1)) << 2) + ((y & 1) << 1) + (x & 1) : y * a.w + x;
      } else {
        const long long p = static_cast<long long>(mt_idx) * TM + my_j * 128 + row;
        valid = p < total_pix;
        if (a.flat) {  // every tensor involved is dense: pixel p of the batch is at p * cstride
          img = 0;
          pix = static_cast<int>(p);
          if (FLATWIN) {  // p runs over the padded raster: only interior positions are outputs
            const int rem = pix - (pix / a.hw) * a.hw;
            const int yy = rem / a.rw, xx = rem - yy * a.rw;
            valid = valid && yy >= a.in_lo && yy < a.in_lo + a.h && xx >= a.in_lo && xx < a.in_lo + a.w;
          }
        } else {
          img = static_cast<int>(p) / a.hw;
          pix = static_cast<int>(p) - img * a.hw;
          if (a.out_pad) {  // zero-bordered output image: (y, x) -> (y + lo, x + lo) of a (wo + border)-wide raster
            const int y = pix / a.wo, x = pix - y * a.wo;
            pix = (y + a.out_lo) * (a.wo + a.out_pad) + x + a.out_lo;
          }
        }
      }
      long long* ro = rowoff_base + slot * (2 * 8 * 32);
      ro[lane] = valid ? img * a.out_img_stride + static_cast<long long>(pix) * a.out_cstride + a.out_coff + n0 : -1;
      if (a.res_mode)
        ro[8 * 32 + lane] = valid ? img * a.res_img_stride + static_cast<long long>(pix) * a.res_cstride + a.res_coff + n0 : -1;
      if (a.decode)  // (never together with a residual) the anchor row the decode phase writes
        ro[8 * 32 + lane] = valid ? (static_cast<long long>(pix) << 32) | static_cast<long long>(img * a.dec_anchors + a.dec_anchor_base + pix) : -1;  // (pixel of the level, anchor row of the batch)
    };
    // per-n-tile constants: column range of the TMEM phase, chunks per row of the copy phases.  With a
    // single n-tile (most layers) they are computed once; otherwise again for every tile.
    struct Cols { int n0, ncols, c_lo, c_hi, cpr, cpr_sh, rcpr, rcpr_sh; };
    auto cols_of = [&](int nt) -> Cols {
      Cols c;
      c.n0 = nt * a.n_tile;
      c.ncols = min(a.n_tile, a.cout - c.n0);
      const int groups = (c.ncols + 15) >> 4;
      c.c_lo = min(c.ncols, ((groups * part) / PARTS) << 4);
      c.c_hi = min(c.ncols, ((groups * (part + 1)) / PARTS) << 4);
      c.cpr = (c.ncols * esize) >> 4;
      c.rcpr = (c.ncols * 2) >> 4;
      c.cpr_sh = 0;
      while ((1 << c.cpr_sh) < c.cpr) ++c.cpr_sh;
      c.rcpr_sh = 0;
      while ((1 << c.rcpr_sh) < c.rcpr) ++c.rcpr_sh;
      return c;
    };
    const bool single_n = a.n_tiles == 1;
    Cols cc = cols_of(single_n ? 0 : static_cast<int>(blockIdx.x) % a.n_tiles);
    const bool res_staged = a.res_mode != 0 && a.res_direct == 0;
    // residual rows [ROWS_PER_WARP * part, +ROWS_PER_WARP) of the team's quarter -> residual staging:
    // 16-byte cp.async, lanes on consecutive chunks of a row (whole rows per instruction)
    auto prefetch_res = [&](const Cols& c, int slot) {
      const int ch = lane & ((1 << c.rcpr_sh) - 1);
      const long long* ro = rowoff_base + slot * (2 * 8 * 32) + 8 * 32;
      for (int rr = lane >> c.rcpr_sh; rr < ROWS_PER_WARP; rr += 32 >> c.rcpr_sh) {
        const int r = part * ROWS_PER_WARP + rr;
        const long long off = ro[r];
        if (off >= 0 && ch < c.rcpr) cp_async_16(smem_u32(res_q + static_cast<size_t>(r) * rpitch + ch * 16), a.res + off + ch * 8);
      }
    };

    if (part == 0) publish_rows(blockIdx.x, 0);
    asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "r"(bar_threads) : "memory");
    pdl_wait();  // residual reads and output stores: only after the previous layer has completed
    if (res_staged) prefetch_res(cc, 0);
    int it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      const int buf = it & 1;
      const Cols c = cc;
      const long long* ro = rowoff_base + buf * (2 * 8 * 32);
      if (threadIdx.x == 0) WIN_TRACE(it, 8);
      mbar_wait(bar_acc_full + 8 * buf, (it >> 1) & 1);
      tc_fence_after();
      if (threadIdx.x == 0) WIN_TRACE(it, 9);
      if (res_staged) cp_async_wait_all();
      // B1: the team's residual rows have landed, its row offsets are published, and every warp of
      // the team is done copying the previous tile out of the staging rows
      asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "r"(bar_threads) : "memory");
      if (threadIdx.x == 0) WIN_TRACE(it, 10);
      const bool valid = ro[lane] >= 0;
      // residual of my row: staged in shared memory, or (deep layers) read from global right here
      const uint8_t* res_row = my_res;
      if (a.res_direct && valid) res_row = reinterpret_cast<const uint8_t*>(a.res + ro[8 * 32 + lane]);
      // ---- TMEM -> registers -> bias / residual / activation -> my staging row (32 columns in flight)
      const uint32_t taddr = taddr_lane + buf * acc_cols + my_j * a.n_tile;
      float dec_best = -INFINITY;
      int dec_bi = 0x7fffffff;
      for (int c0 = c.c_lo; c0 < c.c_hi; c0 += 32) {
        uint32_t v0[16], v1[16];
        const bool two = c0 + 16 < c.c_hi;  // warp-uniform
        __syncwarp();  // tcgen05.ld is warp-collective: reconverge after the per-row predicated body
        tc_ld16_nowait(taddr + c0, v0);
        if (two) tc_ld16_nowait(taddr + c0 + 16, v1);
        tc_ld_wait();
        if (a.decode == 1) {  // box branch: my 16-column groups are DFL sides -> expected distances, slot `side` of my staging row
          reinterpret_cast<float*>(my_stage)[c0 >> 4] = dfl_side(v0, bias_s + c0);
          if (two) reinterpret_cast<float*>(my_stage)[(c0 >> 4) + 1] = dfl_side(v1, bias_s + c0 + 16);
        } else if (a.decode == 2) {
          cls_scan(v0, bias_s + c0, c0, c.ncols, dec_best, dec_bi);
          if (two) cls_scan(v1, bias_s + c0 + 16, c0 + 16, c.ncols, dec_best, dec_bi);
        } else if (valid) {
          uint8_t* dst = a.direct_out ? out_bytes + ro[lane] * esize : my_stage;
          finish_group<ACT>(v0, bias_s + c.n0 + c0, res_row + c0 * 2, a.res_mode, a.out_f32, dst + c0 * esize);
          if (two)
            finish_group<ACT>(v1, bias_s + c.n0 + c0 + 16, res_row + (c0 + 16) * 2, a.res_mode, a.out_f32,
                              dst + (c0 + 16) * esize);
        }
      }
      if (a.decode == 2) {  // my columns' best class -> slot `part` of my staging row
        reinterpret_cast<float*>(my_stage)[2 * part] = dec_best;
        reinterpret_cast<int*>(my_stage)[2 * part + 1] = dec_bi;
      }
      // my part of the accumulator buffer has been read: the MMA thread may reuse it for tile it + 2
      tc_fence_before();
      if (a.warp_arrive) {
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_acc_empty + 8 * buf);
      } else {
        mbar_arrive(bar_acc_empty + 8 * buf);
      }
      if (threadIdx.x == 0) WIN_TRACE(it, 12);
      const int next = tile + static_cast<int>(gridDim.x);
      const bool more = next < total_tiles;
      if (!single_n && more) cc = cols_of(next % a.n_tiles);
      if (part == 0 && more) publish_rows(next, buf ^ 1);
      // B2: the team's staging rows are complete, the residual staging is free, next offsets are published
      asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "r"(bar_threads) : "memory");
      if (threadIdx.x == 0) WIN_TRACE(it, 13);
      if (res_staged && more) prefetch_res(cc, buf ^ 1);
      // ---- staging -> global, rows [ROWS_PER_WARP * part, +ROWS_PER_WARP): whole rows per instruction
      if (a.decode) {
        // the team's part-0 warp (lane = row) gathers what the column teams left in the row's staging slots
        const long long packed = ro[8 * 32 + lane];
        if (part == 0 && packed >= 0) {
          const int gw = static_cast<int>(packed & 0x7fffffff), idx = static_cast<int>(packed >> 32);
          if (a.decode == 1) {
            const float4 d = *reinterpret_cast<const float4*>(my_stage);  // l, t, r, b
            const int gy = idx / a.w, gx = idx - gy * a.w;
            const float ax = static_cast<float>(gx) + 0.5f, ay = static_cast<float>(gy) + 0.5f, st = a.dec_stride;
            reinterpret_cast<float4*>(a.dec_boxes)[gw] =
                make_float4(__fmul_rn(ax - d.x, st), __fmul_rn(ay - d.y, st), __fmul_rn(ax + d.z, st), __fmul_rn(ay + d.w, st));
          } else {
            float best = -INFINITY;
            int bi = 0x7fffffff;
#pragma unroll
            for (int q = 0; q < PARTS; ++q) {  // ascending column ranges: a strict compare keeps the lowest index on ties
              const float ov = reinterpret_cast<const float*>(my_stage)[2 * q];
              const int oi = reinterpret_cast<const int*>(my_stage)[2 * q + 1];
              if (ov > best) { best = ov; bi = oi; }
            }
            a.dec_scores[gw] = __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-best)));
            a.dec_labels[gw] = bi;
          }
        }
      } else if (c.cpr > 0 && !a.direct_out) {
        const int ch = lane & ((1 << c.cpr_sh) - 1);
        for (int rr = lane >> c.cpr_sh; rr < ROWS_PER_WARP; rr += 32 >> c.cpr_sh) {
          const int r = part * ROWS_PER_WARP + rr;
          const long long oo = ro[r];
          if (oo >= 0 && ch < c.cpr) {
            const uint4 val = *reinterpret_cast<const uint4*>(stage_q + static_cast<size_t>(r) * pitch + ch * 16);
            *reinterpret_cast<uint4*>(out_bytes + oo * esize + ch * 16) = val;
          }
        }
      }
    }
  } else if (warp == 4 * NWG) {
    // ================================================================== MMA issuer
    // The whole warp walks the loop convergently, so every descriptor lives in uniform registers;
    // only the tcgen05.mma / tcgen05.commit instructions are predicated on one elected lane.
    {
      const bool leader = elect_one();
      // SBO | version | swizzle; image tiles: consecutive 8-row groups are one raster row apart (the swizzle follows the address bits)
      const uint32_t a_hi = ((((FLATWIN && a.img_tile) ? a.rw : 8) * ROW_BYTES) >> 4) | (1u << 14) | (LTYPE << 29);
      const uint32_t b_hi = (128u >> 4) | (1u << 14);                           // SBO = 128 B, no swizzle
      const uint32_t a_ring = sbase + (EPI ? OFF_RING_A_EPI : OFF_RING_A), b_ring = sbase + a.off_b, w_base = sbase + a.off_w;
      const uint32_t rw_units = static_cast<uint32_t>(a.rw) * (ROW_BYTES >> 4);  // one raster row, in 16-byte units
      const uint32_t lbo = static_cast<uint32_t>(a.resident ? a.cout_pad : a.n_tile);  // K-chunk stride, 16-byte units
      const uint32_t b_k16 = 2 * lbo;
      const uint32_t b_lo_flags = lbo << 16;
      const uint32_t idesc = a.idesc;
      const uint32_t n_tile = static_cast<uint32_t>(a.n_tile);
      const uint32_t tmem0 = __shfl_sync(0xffffffffu, tmem_base, 0);
      uint32_t sa = 0, pa = 0, sbi = 0, pb = 0;  // ring slot / phase parity of the A and B rings
      const uint32_t n_sa = a.sa, n_sb = a.sb;
      int it = 0;
      if (a.resident) mbar_wait(bar_w_full, 0);
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
        const int buf = it & 1;
        uint32_t xp0 = 0;
        if (MODE == 0 && a.tstep % a.rw != 0) {  // row-aligned tiles start at raster column 0
          const int mt_idx = tile / a.n_tiles;
          const int r2 = mt_idx % a.tiles_per_img;
          xp0 = static_cast<uint32_t>(((r2 % a.tiles_per_strip) * a.tstep) % a.rw);
        }
        if (leader) WIN_TRACE(it, 0);
        // the first operand stage usually lands long before the epilogue frees the accumulator: poll it first so
        // that its barrier round trip is off the accumulator -> first MMA path
        mbar_wait(bar_a_full + 8 * sa, pa);
        if (leader) WIN_TRACE(it, 2);
        mbar_wait(bar_acc_empty + 8 * buf, ((it >> 1) & 1) ^ 1);
        tc_fence_after();
        if (leader) WIN_TRACE(it, 1);
        const uint32_t d_tmem = tmem0 + buf * acc_cols;
        for (int s = 0; s < a.slabs; ++s) {
          if (s > 0) {
            mbar_wait(bar_a_full + 8 * sa, pa);
            tc_fence_after();
          }
          // descriptor low word of the patch at raster position xp0: start >> 4 | LBO (unused, 1)
          const uint32_t a_lo0 = ((a_ring + sa * a.patch_bytes) >> 4) + xp0 * (ROW_BYTES >> 4) + (1u << 16);
          uint32_t w_lo = ((w_base >> 4) + static_cast<uint32_t>(s * SLAB >> 3) * lbo) | b_lo_flags;
          const uint32_t w_tap = static_cast<uint32_t>(a.cin_pad >> 3) * lbo;
#pragma unroll
          for (int t = 0; t < TAPS; ++t) {
            const int dy = t / KW, dx = t - dy * KW;  // TAPS == 1: (0, 0)
            const uint32_t a_lo = a_lo0 + dy * rw_units + dx * (ROW_BYTES >> 4);
            uint32_t b_lo;
            if (a.resident) {
              b_lo = w_lo;
              w_lo += w_tap;
            } else {
              mbar_wait(bar_b_full + 8 * sbi, pb);
              tc_fence_after();
              b_lo = ((b_ring + sbi * a.bstage_bytes) >> 4) | b_lo_flags;
            }
            if (WS) {  // weight-stationary: K step outermost, the tile's accumulators share the collected weight block
#pragma unroll
              for (int k = 0; k < K16S; ++k) {
#pragma unroll
                for (int j = 0; j < MT; ++j) {
                  const uint32_t acc = (s | t | k) != 0 ? 1u : 0u;
                  const uint32_t al = a_lo + j * (128 * ROW_BYTES >> 4) + k * 2, bl = b_lo + k * b_k16;
                  if (MT == 1) mma_issue_ws<2>(k & 3, leader, d_tmem, al, a_hi, bl, b_hi, idesc, acc);
                  else if (j == 0) mma_issue_ws<0>(k & 3, leader, d_tmem, al, a_hi, bl, b_hi, idesc, acc);
                  else mma_issue_ws<1>(k & 3, leader, d_tmem + j * n_tile, al, a_hi, bl, b_hi, idesc, acc);
                }
              }
            } else {
#pragma unroll
              for (int j = 0; j < MT; ++j) {
#pragma unroll
                for (int k = 0; k < K16S; ++k)
                  mma_issue(leader, d_tmem + j * n_tile, a_lo + j * (128 * ROW_BYTES >> 4) + k * 2, a_hi, b_lo + k * b_k16, b_hi,
                            idesc, (s | t | k) != 0 ? 1u : 0u);
              }
            }
            if (!a.resident) {
              tc_commit_if(leader, bar_b_empty + 8 * sbi);
              if (++sbi == n_sb) { sbi = 0; pb ^= 1; }
            }
          }
          tc_commit_if(leader, bar_a_empty + 8 * sa);
          if (++sa == n_sa) { sa = 0; pa ^= 1; }
        }
        tc_commit_if(leader, bar_acc_full + 8 * buf);
        if (leader) WIN_TRACE(it, 3);
      }
      tc_fence_before();
    }
  } else if (warp == 4 * NWG + 1) {
    // ================================================================== patch (A) producer
    if (lane == 0) {
      pdl_wait();  // the patches are the previous layer's output
      if (a.tl && blockIdx.x == 0) a.tl[1] = global_timer_ns();
      const uint32_t a_ring = sbase + (EPI ? OFF_RING_A_EPI : OFF_RING_A);
      uint32_t sa = 0, pa = 1;
      const uint32_t n_sa = a.sa;
      const long long total_pix = static_cast<long long>(batch) * a.hw;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int mt_idx = tile / a.n_tiles;
        int n_img = 0, x_start = 0, y_start = 0;
        int cn[MT], cw[MT], chh[MT];  // im2col: base pixel (image, column, row) of each 128-row sub-tile
        uint32_t tx_bytes = a.box_bytes;
        if (MODE == 0) {
          const TilePos tp = tile_pos(a, mt_idx);
          n_img = tp.n_img;
          x_start = tp.strip * a.tw - 1;
          y_start = tp.q0 / a.rw - 1;
        } else if (MODE == 2) {
          tx_bytes = 0;
#pragma unroll
          for (int j = 0; j < MT; ++j) {
            const long long m = static_cast<long long>(mt_idx) * TM + j * 128;
            cn[j] = -1;
            if (m < total_pix) {  // sub-tiles beyond the batch are not loaded (their rows are never stored)
              cn[j] = static_cast<int>(m / a.hw);
              const int rem = static_cast<int>(m - static_cast<long long>(cn[j]) * a.hw);
              const int pr = rem / a.wo;
              cw[j] = (rem - pr * a.wo) * a.stride - a.pad;
              chh[j] = pr * a.stride - a.pad;
              tx_bytes += 128 * ROW_BYTES;
            }
          }
        }
        int tap = 0, sl = 0;  // im2col: virtual slab -> (filter tap, channel slab)
        const int pit = (tile - static_cast<int>(blockIdx.x)) / static_cast<int>(gridDim.x);
        for (int s = 0; s < a.slabs; ++s) {
          if (s == 0) WIN_TRACE(pit, 4);
          mbar_wait(bar_a_empty + 8 * sa, pa);
          if (s == 0) WIN_TRACE(pit, 5);
          const uint32_t bar = bar_a_full + 8 * sa;
          const uint32_t dst = a_ring + sa * a.patch_bytes;
          mbar_arrive_expect_tx(bar, tx_bytes);
          if (MODE == 0) {
            tma_load_4d(dst, &maps.in, bar, s * SLAB, x_start, y_start, n_img);
          } else if (FLATWIN) {
            // negative / past-the-end rows are zero-filled; image tiles start RW + 1 positions before the image's first interior pixel
            const int row0 = a.img_tile ? mt_idx * a.hw + (a.in_lo - 1) * (a.rw + 1) : mt_idx * TM - (a.rw + 1);
#pragma unroll
            for (int j = 0; j < MT; ++j)
              tma_load_2d(dst + j * (a.box_rows * ROW_BYTES), &maps.in, bar, s * SLAB, row0 + j * a.box_rows);
          } else if (MODE == 1) {
            tma_load_2d(dst, &maps.in, bar, s * SLAB, mt_idx * TM);
          } else {
            const int tr = tap / a.ksize, tc = tap - tr * a.ksize;
#pragma unroll
            for (int j = 0; j < MT; ++j)
              if (cn[j] >= 0)
                tma_load_im2col_4d(dst + j * (128 * ROW_BYTES), &maps.in, bar, sl * SLAB, cw[j], chh[j], cn[j],
                                   static_cast<uint16_t>(tc), static_cast<uint16_t>(tr));
            if (++sl == a.slabs_per_tap) { sl = 0; ++tap; }
          }
          if (++sa == n_sa) { sa = 0; pa ^= 1; }
        }
      }
    }
  } else if (warp == 4 * NWG + 2) {
    // ================================================================== weight (B) producer
    if (lane == 0) {
      if (a.resident) {
        mbar_arrive_expect_tx(bar_w_full, a.wbytes);
        const uint8_t* src = reinterpret_cast<const uint8_t*>(a.wgt);
        for (uint32_t off = 0; off < a.wbytes; off += 16384)
          bulk_g2s(sbase + a.off_w + off, src + off, min(16384u, a.wbytes - off), bar_w_full);
      } else {
        const uint32_t b_ring = sbase + a.off_b;
        const uint32_t chunk_bytes = static_cast<uint32_t>(a.n_tile) * 16;
        constexpr int nchunks = SLAB / 8;
        uint32_t sbi = 0, pb = 1;
        const uint32_t n_sb = a.sb;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
          const int n0 = (tile % a.n_tiles) * a.n_tile;
          for (int s = 0; s < a.slabs; ++s) {
            for (int t = 0; t < TAPS; ++t) {
              mbar_wait(bar_b_empty + 8 * sbi, pb);
              const uint32_t bar = bar_b_full + 8 * sbi;
              const uint32_t dst = b_ring + sbi * a.bstage_bytes;
              mbar_arrive_expect_tx(bar, a.bstage_bytes);
              const int chunk0 = (t * a.cin_pad + s * SLAB) >> 3;
              const __nv_bfloat16* src = a.wgt + (static_cast<long long>(chunk0) * a.cout_pad + n0) * 8;
              if (a.n_tile == a.cout_pad) {
                bulk_g2s(dst, src, a.bstage_bytes, bar);
              } else if (a.wgt_nt) {  // the stage is one contiguous run of the n-tile-major copy
                bulk_g2s(dst, a.wgt_nt + (static_cast<long long>(n0 / a.n_tile) * a.q_pad + chunk0) * a.n_tile * 8, a.bstage_bytes, bar);
              } else {
                for (int c = 0; c < nchunks; ++c)
                  bulk_g2s(dst + c * chunk_bytes, src + static_cast<long long>(c) * a.cout_pad * 8, chunk_bytes, bar);
              }
              if (++sbi == n_sb) { sbi = 0; pb ^= 1; }
            }
          }
        }
      }
    }
  } else if (EPI == 1) {
    // ================================================================== epilogue I/O warp (TMA flavour only)
    // Residual boxes are fetched up to `nres` tiles ahead of the epilogue; finished tiles are stored with one
    // tensor store per channel piece.  The epilogue warps never wait for either instruction to issue.
    pdl_wait();  // residual loads / output stores: only after the previous layer has completed
    auto coords = [&](int tile, int& n0, int& cx, int& cy, int& cn) {
      const int mt_idx = a.n_tiles == 1 ? tile : tile / a.n_tiles;
      n0 = (tile - mt_idx * a.n_tiles) * a.n_tile;
      if (WINDOW) {
        const TilePos tp = tile_pos(a, mt_idx);
        cx = tp.strip * a.tw; cy = tp.q0 / a.rw; cn = tp.n_img;
      } else {
        cx = mt_idx * TM; cy = 0; cn = 0;
        if (MODE == 2 && a.pad_store) {  // first pixel of the tile -> (image, row); tiles are whole rows / whole images
          cn = cx / a.hw;
          cy = (cx - cn * a.hw) / a.wo;
          cx = 0;
        }
        if (FLATWIN && a.img_tile) { cn = mt_idx; cy = 0; cx = 0; }
      }
    };
    auto load_res = [&](int tile, uint32_t slot, uint32_t phase) {
      int n0, cx, cy, cn;
      coords(tile, n0, cx, cy, cn);
      mbar_wait(bar_res_empty + 8 * slot, phase ^ 1);
      if (lane == 0) {
        const uint32_t rbar = bar_res_full + 8 * slot;
        const uint32_t rdst = sbase + (a.res_inplace ? a.off_stage : a.off_res) + slot * a.stage_buf_bytes;
        mbar_arrive_expect_tx(rbar, a.res_tx_bytes);
        if (WINDOW) {
          tma_load_4d(rdst + a.piece_off[0], &maps.res[0], rbar, n0, cx, cy, cn);
          if (a.pieces == 2) tma_load_4d(rdst + a.piece_off[1], &maps.res[1], rbar, n0 + a.piece_ch[0], cx, cy, cn);
        } else {
          int pc0 = 0;  // first channel of the piece
          for (int q = 0; q < a.pieces; ++q) {
            if (FLATWIN && a.img_tile) tma_load_4d(rdst + a.piece_off[q], &maps.res[q ? 1 : 0], rbar, n0 + pc0, 0, 0, cn);
            else tma_load_2d(rdst + a.piece_off[q], &maps.res[q ? 1 : 0], rbar, n0 + pc0, cx);
            pc0 += a.piece_ch[q];
          }
        }
      }
      __syncwarp();
    };
    uint32_t lslot = 0, lphase = 0;  // next residual slot to fill
    int ahead = blockIdx.x;          // next tile whose residual is to be fetched
    if (a.res_mode)
      for (int k = 0; k < a.nres && ahead < total_tiles; ++k, ahead += gridDim.x) {
        load_res(ahead, lslot, lphase);
        if (++lslot == static_cast<uint32_t>(a.nres)) { lslot = 0; lphase ^= 1; }
      }
    int io_it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++io_it) {
      int n0, cx, cy, cn;
      coords(tile, n0, cx, cy, cn);
      const int sbuf = a.nstage == 2 ? (io_it & 1) : 0;
      const uint32_t src = sbase + a.off_stage + sbuf * a.stage_buf_bytes;
      asm volatile("bar.sync %0, %1;" ::"r"(2 + (io_it & 1)), "r"((MT == 2 && a.epi_alt) ? 64 * NWG + 32 : 128 * NWG + 32)
                   : "memory");  // every epilogue thread (of the tile's team) has staged its part
      if (lane == 0) {
        const bool two = a.pieces == 2 && n0 + a.piece_ch[0] < a.cout;
        if (WINDOW && a.s2d_store) {
          tma_store_5d(&maps.out[0], src + a.piece_off[0], 0, cx >> 1, 0, cy >> 1, cn);
        } else if (WINDOW) {
          tma_store_4d(&maps.out[0], src + a.piece_off[0], n0, cx, cy, cn);
          if (two) tma_store_4d(&maps.out[1], src + a.piece_off[1], n0 + a.piece_ch[0], cx, cy, cn);
        } else {
          int pc0 = 0;
          for (int q = 0; q < a.pieces && n0 + pc0 < a.cout; ++q) {
            if ((MODE == 2 && a.pad_store) || (FLATWIN && a.img_tile)) tma_store_4d(&maps.out[q ? 1 : 0], src + a.piece_off[q], n0 + pc0, 0, cy, cn);
            else tma_store_2d(&maps.out[q ? 1 : 0], src + a.piece_off[q], n0 + pc0, cx);
            pc0 += a.piece_ch[q];
          }
        }
        bulk_commit();
        bulk_wait_read_all();
        mbar_arrive(bar_stage_free + 8 * sbuf);  // that staging buffer may be overwritten
      }
      __syncwarp();
      // the epilogue has consumed this tile's residual: refill that slot for the tile `nres` ahead
      if (a.res_mode && ahead < total_tiles) {
        load_res(ahead, lslot, lphase);
        if (++lslot == static_cast<uint32_t>(a.nres)) { lslot = 0; lphase ^= 1; }
        ahead += gridDim.x;
      }
    }
    if (lane == 0) bulk_wait_all();
  }
  __syncthreads();
  if (a.tl && blockIdx.x == 0 && threadIdx.x == 0) a.tl[2] = global_timer_ns();
  if (warp == 4 * NWG) {
    tc_fence_after();
    tc_dealloc(tmem_base, a.tmem_cols);
  }
}

typedef void (*WinKernelFn)(const WinArgs, const WinMaps);

template <int SLAB, int AMODE, int MT, int EPI>
WinKernelFn pick_act(int act) {
  if (act == 1) return conv_win_kernel<SLAB, AMODE, MT, 1, EPI>;
  if (act == 2) return conv_win_kernel<SLAB, AMODE, MT, 2, EPI>;
  return conv_win_kernel<SLAB, AMODE, MT, 0, EPI>;
}
template <int SLAB, int AMODE, int EPI>
WinKernelFn pick_mt(int mt, int act) {
  return mt == 2 ? pick_act<SLAB, AMODE, 2, EPI>(act) : pick_act<SLAB, AMODE, 1, EPI>(act);
}
template <int SLAB>
WinKernelFn pick_mode(int mode, int mt, int act, int epi) {
  if (SLAB == 64 && epi == 3) {  // weight-stationary variants exist for the 64-channel-slab window modes only
    if (mode == 0) return pick_mt<64, 0, 3>(mt, act);
    if (mode == 4) return pick_mt<64, 4, 3>(mt, act);
  }
  epi &= 1;
  if (mode == 0) return epi ? pick_mt<SLAB, 0, 1>(mt, act) : pick_mt<SLAB, 0, 0>(mt, act);
  if (mode == 3) return epi ? pick_mt<SLAB, 3, 1>(mt, act) : pick_mt<SLAB, 3, 0>(mt, act);
  if (mode == 4) return epi ? pick_mt<SLAB, 4, 1>(mt, act) : pick_mt<SLAB, 4, 0>(mt, act);
  if (mode == 1) return epi ? pick_mt<SLAB, 1, 1>(mt, act) : pick_mt<SLAB, 1, 0>(mt, act);
  return epi ? pick_mt<SLAB, 2, 1>(mt, act) : pick_mt<SLAB, 2, 0>(mt, act);
}
WinKernelFn pick_kernel(int slab, int mode, int mt, int act, int epi) {
  if (slab == 64) return pick_mode<64>(mode, mt, act, epi);
  if (slab == 32) return pick_mode<32>(mode, mt, act, epi);
  return pick_mode<16>(mode, mt, act, epi);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const int*, const int*, cuuint32_t, cuuint32_t, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeIm2colFn get_encode_im2col() {
  static EncodeIm2colFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeIm2colFn>(p);
  }
  return fn;
}

// 3x3 stride-1 layer over zero-bordered tensors: operand mode 4
inline bool mode_is_flatwin(const PackedConv& pc, const ConvLaunch& L) {
  return L.in_pad && L.out_pad && pc.stride == 1 && pc.ksize == 3 && pc.s2d_c0 == 0;
}

struct WinPlan {
  bool ok = false;
  double cost = 0.0;
  int rw = 0, tw = 0, strips = 1, tstep = 0, tiles_per_strip = 0, mt = 1, bh = 0;
  int sa = 0, sb = 0;
  uint32_t patch_bytes = 0, box_bytes = 0, off_w = 0, off_b = 0, off_stage = 0;
  size_t smem = 0;
  long long tiles = 0;
  uint32_t stage_buf = 0;
  int nres = 0, nstage = 1;
  bool img = false;  // mode 4: one image per tile (WinArgs::img_tile)
};

}  // namespace

// Returns 1 when the layer was launched on the window kernel, 0 when the shape is not eligible
// (the caller falls back to conv_tc_kernel), negative on error.
int try_launch_conv_pair(const PackedConv& pc, const ConvLaunch& L, cudaStream_t stream);
long long* timeline_slot(long long tag);  // api.cu

int try_launch_conv_win(const PackedConv& pc, const ConvLaunch& L, cudaStream_t stream) {
  if (mode_is_flatwin(pc, L) && pc.w_pair) {  // 64 / 128-channel 3x3 layers of a zero-bordered trunk: CTA pairs (conv_pair.cu)
    const int prc = try_launch_conv_pair(pc, L, stream);
    if (prc != 0) return prc;
  }
  static const bool disabled = getenv("AICAM_NO_WIN") != nullptr;
  if (disabled || get_encode_tiled() == nullptr) return 0;
  static const bool no_im2col = getenv("AICAM_WIN_NO_IM2COL") != nullptr;
  const bool s2d = pc.s2d_c0 != 0;  // 3x3 stride-2 layer packed as a 2x2 window over 2x2 input blocks
  if (s2d) {
    // the launch describes the space-to-depth tensor: [batch][h][w][4 c0] dense, output h x w
    if (pc.ksize != 2 || pc.stride != 1 || pc.cin_pad != 4 * pc.s2d_c0 || (pc.cin_pad != 16 && pc.cin_pad != 64) ||
        L.in_cstride != pc.cin_pad || L.in_coff != 0 || L.ho != L.h || L.wo != L.w)
      return fail(AICAM_ERR_INVALID_ARG, "conv_win: space-to-depth layer with an unsupported geometry");
  } else if ((pc.stride != 1 && pc.stride != 2) || (pc.ksize != 1 && pc.ksize != 3) || pc.cin_pad % 16 != 0 || pc.cin_pad == 4) {
    return 0;
  }
  if (L.batch <= 0 || get_encode_im2col() == nullptr) return 0;
  const int es = L.out_f32 ? 4 : 2;
  const int cout_pad = (pc.cout + 15) / 16 * 16;
  if ((pc.cout * es) % 16 != 0 || (static_cast<long long>(L.out_cstride) * es) % 16 != 0 ||
      (static_cast<long long>(L.out_coff) * es) % 16 != 0 || (L.out_img_stride * es) % 16 != 0 ||
      reinterpret_cast<uintptr_t>(L.out) % 16 != 0 || cout_pad > 512)
    return 0;
  const int res_mode = L.res ? L.res_mode : 0;
  if (res_mode && (L.out_f32 || pc.cout % 8 != 0 || L.res_cstride % 8 != 0 || L.res_coff % 8 != 0 || L.res_img_stride % 8 != 0 ||
                   reinterpret_cast<uintptr_t>(L.res) % 16 != 0))
    return 0;
  if (L.in_cstride % 8 != 0 || L.in_coff % 8 != 0 || reinterpret_cast<uintptr_t>(L.in) % 16 != 0) return 0;
  const int ip = L.in_pad ? 1 : 0, opd = L.out_pad ? 1 : 0;
  const int ilo = pad_lo(L.in_pad), iext = pad_ext(L.in_pad), olo = pad_lo(L.out_pad), oext = pad_ext(L.out_pad);
  const int hp = L.h + iext, wp = L.w + iext;  // input image as it lies in memory
  if (L.in_img_stride != static_cast<long long>(hp) * wp * L.in_cstride) return 0;
  if (opd && (L.out_img_stride != static_cast<long long>(L.ho + oext) * (L.wo + oext) * L.out_cstride ||
              (res_mode && L.res_img_stride != static_cast<long long>(L.ho + oext) * (L.wo + oext) * L.res_cstride) || L.out_s2d || s2d))
    return fail(AICAM_ERR_INVALID_ARG, "conv_win: padded output with an inconsistent image stride");
  if (ip && opd && pc.stride == 1 && L.in_pad != L.out_pad)
    return fail(AICAM_ERR_INVALID_ARG, "conv_win: a stride-1 layer over padded tensors needs the same border kind on both sides");
  const long long pixels = static_cast<long long>(L.batch) * L.ho * L.wo;  // output pixels
  const long long padded_pixels = static_cast<long long>(L.batch) * hp * wp;
  if (pixels >= (1ll << 31) || padded_pixels >= (1ll << 31)) return 0;

  // 0: window patches (3x3 stride 1), 1: flat (1x1 stride 1), 2: im2col TMA (stride 2, and 3x3 on maps too
  // small for the window raster)
  int mode = s2d ? 3 : (pc.stride == 1 ? (pc.ksize == 3 ? 0 : 1) : 2);
  if (ip && pc.stride == 1) {
    // stride 1 over a padded input: the flat padded raster (mode 4), output in the same padded geometry
    if (pc.ksize != 3 || !opd || s2d) return fail(AICAM_ERR_UNSUPPORTED, "conv_win: padded input needs a 3x3 stride-1 layer with a padded output, or stride 2");
    mode = 4;
  }
  if (mode == 2 && no_im2col) return 0;
  if (L.out_s2d && mode != 0 && mode != 3) return 0;  // the caller reports the unsupported combination
  bool window = mode == 0 || mode == 3;
  const int kw1 = mode == 3 ? 1 : 2;  // window extent - 1 (both axes)
  const int win_h = L.h, win_w = L.w;  // size of the raster the window slides over
  const int taps = pc.ksize * pc.ksize;
  const int slab = pc.cin_pad % 64 == 0 ? 64 : (pc.cin_pad % 32 == 0 ? 32 : 16);
  const int slabs = pc.cin_pad / slab;
  const uint32_t row_bytes = slab * 2;
  int n_tile = 16;
  for (int nt = L.out_f32 ? 80 : 128; nt >= 16; nt -= 16)
    if (cout_pad % nt == 0) { n_tile = nt; break; }
  // 256-column tiles where the layer is wide enough: one 128 x 256 x 16 MMA reads 12 KB of operands in its 128
  // tensor-pipe cycles (96 at 128 B/clk), a 128 x 128 one reads 8 KB in 64 - the narrower tile is bound by the
  // shared-memory port (measured ~88 cycles per MMA), the wide one by the tensor pipe
  static const bool no_n256 = getenv("AICAM_WIN_NO_N256") != nullptr;
  if (!no_n256 && !L.out_f32 && cout_pad % 256 == 0 && (cout_pad == 256 || pc.nt_block == 256) && (mode == 4 || mode == 2 || mode == 1)) n_tile = 256;
  const int n_tiles = cout_pad / n_tile;
  const size_t wbytes = static_cast<size_t>(pc.q_pad) * cout_pad * 16;
  if (static_cast<size_t>(pc.q_pad) * 8 != static_cast<size_t>(taps) * pc.cin_pad) return 0;
  const bool resident = n_tiles == 1 && wbytes <= RESIDENT_LIMIT;
  if (!resident && slab != 64) return 0;
  const uint32_t bstage_bytes = static_cast<uint32_t>(slab / 8) * n_tile * 16;
  const uint32_t stage_pitch = n_tile * es + 16;
  const uint32_t res_pitch = n_tile * 2 + 16;
  const int sb = resident ? 0 : (n_tile == 256 ? 3 : 4);  // 32 KB stages at 256 columns
  // mode 4 fallback when the TMA epilogue is unavailable: no staging tile, every thread stores its own 32-byte groups
  // (measured: ~15k cycles per 256 x 128 tile, LSU-bound - one sector per lane per instruction)
  static const bool no_tma_epi4 = getenv("AICAM_WIN_NO_TMA_EPI") != nullptr;
  const int nt_rest = n_tile - (n_tile >= 64 ? 64 : (n_tile >= 32 ? 32 : 16));  // the n-tile splits into <= 2 swizzled pieces
  const bool epi4 = mode == 4 && !no_tma_epi4 && !L.out_f32 && pc.cout % 8 == 0 &&
                    (n_tile == 256 || nt_rest == 0 || nt_rest == 64 || nt_rest == 32 || nt_rest == 16);
  const bool direct_out = mode == 4 && !resident && !L.out_f32 && !epi4;
  // streamed (deep-K) layers: the epilogue is a small share of a tile, read the residual from global there
  // instead of spending 70 KB of shared memory that the 256-row tiling needs
  const bool res_staged = res_mode != 0 && resident;
  const size_t fixed_tail = (resident ? (wbytes + 1023) / 1024 * 1024 : static_cast<size_t>(sb) * bstage_bytes);

  // ---- TMA epilogue (window modes, bf16, natural layout): the n-tile splits into one or two channel pieces
  // of 64 / 32 / 16 channels, each a swizzled staging tile with its own output / residual tensor map
  static const bool no_tma_epi = getenv("AICAM_WIN_NO_TMA_EPI") != nullptr;
  int piece_ch[4] = {0, 0, 0, 0};
  if (n_tile == 256) {
    piece_ch[0] = piece_ch[1] = piece_ch[2] = piece_ch[3] = 64;
  } else {
    const int first = n_tile >= 64 ? 64 : (n_tile >= 32 ? 32 : 16);
    const int rest = n_tile - first;
    if (rest == 0 || rest == 64 || rest == 32 || rest == 16) { piece_ch[0] = first; piece_ch[1] = rest; }
  }
  // a space-to-depth output can take the TMA epilogue when the tile is the whole channel width of a dense tensor
  static const bool no_s2d_epi = getenv("AICAM_WIN_NO_S2D_EPI") != nullptr;
  const bool s2d_store = L.out_s2d && !no_s2d_epi && !res_mode && n_tiles == 1 && piece_ch[1] == 0 && piece_ch[0] == pc.cout &&
                         L.out_cstride == pc.cout && L.out_coff == 0 && L.ho % 2 == 0 && L.wo % 2 == 0 && pc.cout * 2 % 16 == 0;
  bool epi = !no_tma_epi && piece_ch[0] != 0 && !L.out_f32 && (!L.out_s2d || s2d_store) && pc.cout % 8 == 0;

  // ---- choose the tiling: strips x (linear | row-aligned) x mt, cheapest estimated time
  WinPlan best;
  const int k16_total = taps * pc.cin_pad / 16;
  bool pad2_failed = false;
  const bool epi_pad2_ok = epi;  // (the static conditions of the TMA epilogue: bf16, channel pieces, cout % 8)
plan:
  best = WinPlan();
  size_t fixed_base = 0;  // set below, once this pass's epilogue flavour is known
  window = mode == 0 || mode == 3;
  // flat / im2col tiles are runs of consecutive output pixels: the store is a 2-D box when pixel p of the batch
  // sits at p * cstride in the output (and residual) tensor
  const bool flat_io = L.out_img_stride == static_cast<long long>(L.ho) * L.wo * L.out_cstride &&
                       (!res_mode || L.res_img_stride == static_cast<long long>(L.ho) * L.wo * L.res_cstride);
  // measured: the TMA epilogue pays off where the epilogue bounds the tile (window modes, small K); deep
  // im2col / flat layers are L2-bound and need the shared memory for deeper operand rings instead
  // (1x1 layers with few input channels are all epilogue: measured 70 -> 50 us on 32 -> 32 @160x160)
  const bool epi_flat = mode == 1 && flat_io && resident && pc.cin_pad <= 128;
  // im2col layers storing into zero-bordered images (the stride-2 entry layers of the ReID trunk and their 1x1 partners): TMA epilogue
  // when the tiles can be whole rows of an image or whole images (checked per tile height below)
  static const bool no_pad_store = getenv("AICAM_WIN_NO_PAD_STORE") != nullptr;
  // (measured in the step: the 1x1 stride-2 partners 59 / 38 / 23 -> 58 / 33 / 19 us; the 3x3 entry layers are bound by operand ingest and
  //  lose a little to the smaller operand ring, so they keep the generic epilogue)
  const bool epi_pad2 = mode == 2 && opd && !res_mode && pc.ksize == 1 && !no_pad_store && !pad2_failed && epi_pad2_ok;
  if (!window && !epi_flat && !epi_pad2) epi = false;
  if (mode == 4) epi = epi4 && piece_ch[0] != 0;  // flat TMA epilogue: border positions are stored as zeros
  else if (opd && !epi_pad2) epi = false;           // (un-padded raster -> padded image: row-by-row offsets, generic epilogue)
  fixed_base = (epi ? OFF_RING_A_EPI : OFF_RING_A) + fixed_tail;
  // 64-column tiles are bound by the shared-memory port (4 KB of A + 2 KB of B per 32-cycle MMA): the weight-stationary MMA form
  // keeps a tile's B block in a collector buffer across the accumulators of the tile
  static const bool no_ws = getenv("AICAM_WIN_NO_WS") != nullptr;
  const bool ws_ok = !no_ws && epi && slab == 64 && n_tile == 64 && (mode == 0 || mode == 4);
  for (int mt = 1; mt <= 2; ++mt) {
    const int tm = 128 * mt;
    if (2 * mt * n_tile > 512) continue;
    if (epi && epi_pad2) {  // tiles = whole output rows of one image, or whole images
      const int hwo = L.ho * L.wo;
      if (!((hwo % tm == 0 && tm % L.wo == 0) || tm % hwo == 0)) continue;
    }
    for (int strips = 1; strips <= (window ? 8 : 1); ++strips) {
      for (int aligned = (epi && window) ? 1 : 0; aligned <= (window ? 1 : 0); ++aligned) {
        WinPlan p;
        p.mt = mt;
        p.strips = strips;
        size_t stage_bytes = direct_out ? 0 : static_cast<size_t>(tm) * (stage_pitch + (res_staged ? res_pitch : 0));
        if (window) {
          p.tw = (win_w + strips - 1) / strips;
          if (s2d_store && epi && (p.tw & 1)) ++p.tw;  // even strip widths: strips start on 2x2 block boundaries
          p.rw = p.tw + kw1;
          if (p.rw > 256 || (strips > 1 && p.tw < 8)) continue;
          if (aligned) {
            int th = tm / p.rw;
            if (s2d_store && epi) th &= ~1;  // whole 2x2 blocks per tile
            if (th < 1) continue;
            p.tstep = th * p.rw;
            p.tiles_per_strip = (win_h + th - 1) / th;
          } else {
            p.tstep = tm;
            p.tiles_per_strip = (win_h * p.rw + tm - 1) / tm;
          }
          const int xp0max = aligned ? 0 : p.rw - 1;
          p.bh = aligned ? p.tstep / p.rw + kw1 : (xp0max + p.tstep - 1 + kw1 * p.rw + kw1) / p.rw + 1;
          if (epi) {
            // compact staging tile(s): output + residual ring, every piece 1024-byte aligned
            const int rows_c = (p.tstep / p.rw) * p.tw;
            size_t buf = 0;
            for (int q = 0; q < 4; ++q)
              if (piece_ch[q]) buf += (static_cast<size_t>(rows_c) * piece_ch[q] * 2 + 1023) / 1024 * 1024;
            p.stage_buf = static_cast<uint32_t>(buf);
            p.nres = res_mode ? 2 : 0;
            p.nstage = 2;
            stage_bytes = buf * (p.nstage + p.nres) + 1024;  // + alignment slack after the weight / B ring
          }
          if (p.bh > 256) continue;
          p.box_bytes = static_cast<uint32_t>(p.bh) * p.rw * row_bytes;
          const uint32_t reach = static_cast<uint32_t>(xp0max + tm + kw1 * p.rw + kw1 + 1) * row_bytes;  // junk rows stay inside the stage
          p.patch_bytes = (std::max(p.box_bytes, reach) + 1023) / 1024 * 1024;
          p.tiles = static_cast<long long>(L.batch) * strips * p.tiles_per_strip;
        } else if (mode == 4) {
          // flat padded raster: MT boxes of `bh` rows cover the tile and the RW + 1 positions either side of it
          p.tw = L.w; p.rw = wp; p.tstep = tm; p.tiles_per_strip = 0;
          p.bh = ((tm + 2 * wp + 2 + mt - 1) / mt + 7) / 8 * 8;
          // 8-pixel-wide maps of 128 pixels (ReID layer 3): one image per tile, its rows picked by the descriptor's group stride
          static const bool no_img_tile = getenv("AICAM_WIN_NO_IMG_TILE") != nullptr;
          p.img = epi && mt == 1 && L.w == 8 && L.h * L.w == 128 && !no_img_tile;
          if (p.img) p.bh = ((L.h - 1) * wp + L.w + 2 * wp + 2 + 7) / 8 * 8;
          if (p.bh > 256) continue;
          p.box_bytes = static_cast<uint32_t>(mt) * p.bh * row_bytes;
          (void)ilo;
          p.patch_bytes = (p.box_bytes + 1023) / 1024 * 1024;
          p.tiles = p.img ? L.batch : (padded_pixels + tm - 1) / tm;
          if (epi) {
            // the residual tile is loaded into the staging buffer and finished in place: no residual ring
            size_t buf = 0;
            for (int q = 0; q < 4; ++q)
              if (piece_ch[q]) buf += (static_cast<size_t>(tm) * piece_ch[q] * 2 + 1023) / 1024 * 1024;
            p.stage_buf = static_cast<uint32_t>(buf);
            p.nstage = 2;
            if (fixed_base + buf * 2 + 1024 + 2 * static_cast<size_t>(p.patch_bytes) > SMEM_LIMIT) p.nstage = 1;
            p.nres = res_mode ? p.nstage : 0;
            stage_bytes = buf * p.nstage + 1024;
          }
        } else {
          p.tw = L.w; p.rw = L.w; p.tstep = tm; p.tiles_per_strip = 0; p.bh = 0;
          p.box_bytes = static_cast<uint32_t>(tm) * row_bytes;
          p.patch_bytes = (p.box_bytes + 1023) / 1024 * 1024;
          p.tiles = (pixels + tm - 1) / tm;
          if (epi) {
            size_t buf = 0;
            for (int q = 0; q < 4; ++q)
              if (piece_ch[q]) buf += (static_cast<size_t>(tm) * piece_ch[q] * 2 + 1023) / 1024 * 1024;
            p.stage_buf = static_cast<uint32_t>(buf);
            p.nres = res_mode ? 2 : 0;
            p.nstage = 2;
            stage_bytes = buf * (p.nstage + p.nres) + 1024;
          }
        }
        size_t fixed = fixed_base + stage_bytes;
        if (epi && mode != 4 && fixed + 3 * static_cast<size_t>(p.patch_bytes) > SMEM_LIMIT) {
          p.nstage = 1;  // single output staging buffer rather than a shallow patch ring
          stage_bytes = static_cast<size_t>(p.stage_buf) * (p.nstage + p.nres) + 1024;
          fixed = fixed_base + stage_bytes;
        }
        if (epi && mode != 4 && p.nres == 2 && fixed + 3 * static_cast<size_t>(p.patch_bytes) > SMEM_LIMIT) {
          p.nres = 1;  // then one residual buffer
          stage_bytes = static_cast<size_t>(p.stage_buf) * (p.nstage + p.nres) + 1024;
          fixed = fixed_base + stage_bytes;
        }
        if (fixed + 2 * static_cast<size_t>(p.patch_bytes) > SMEM_LIMIT) continue;
        p.sa = static_cast<int>(std::min<size_t>(MAX_RING, (SMEM_LIMIT - fixed) / p.patch_bytes));
        // enough patches in flight to cover the HBM latency of a tile, no more
        p.sa = std::min(p.sa, (window || mode == 4) ? std::max(4, 2 * slabs) : 6);
        p.smem = fixed + static_cast<size_t>(p.sa) * p.patch_bytes;
        // estimated cycles per tile: tensor pipe vs L2->SM traffic vs epilogue, plus a fixed hand-off cost
        // one 128 x n_tile x 16 MMA: tensor pipe n_tile / 2 cycles, operand fetch (4 KB + n_tile * 32 B) at 128 B/clk
        // (weight-stationary issue, two accumulators per tile: the second MMA of a pair takes B from the collector - measured on
        //  ReID layer 1: 57 cycles per 128 x 64 x 16 MMA instead of 68, tile of 256 rows 4 500 cycles instead of 2 x 2 790)
        const bool ws_pair = ws_ok && mode == 4 && mt == 2;
        const double mma = static_cast<double>(mt) * k16_total * std::max(n_tile / 2.0, 32.0 + n_tile / (ws_pair ? 8.0 : 4.0));
        const double l2 = (static_cast<double>(p.box_bytes) * slabs * (mode == 2 ? taps : 1) +
                           (resident ? 0.0 : static_cast<double>(wbytes) / n_tiles)) / 48.0;
        const int groups = (n_tile + 15) / 16;
        const int active = mt == 2 ? 2 * std::min(2, groups) : std::min(4, groups);
        // measured on B200 (clock64 traces): TMA epilogue ~35 cycles per column per thread + ~600, generic ~3x that
        const double epi_cyc = epi ? (static_cast<double>(mt) * groups / active) * 550.0 + 600.0
                                   : (static_cast<double>(mt) * groups / active) * 1000.0 + 1700.0;
        double per_tile = std::max(mma, std::max(l2, epi_cyc)) + 250.0;
        // shallow rings serialise producer, MMA and epilogue
        if ((window || (mode == 4 && slabs == 1)) && p.sa < 3 && !(ws_pair && p.sa == 2 && p.nstage == 2)) per_tile *= 1.6;
        if (epi && mode != 4 && res_mode && p.nres < 2) per_tile *= 2.0;  // (mode 4 finishes the residual in place)
        p.cost = static_cast<double>(p.tiles) * n_tiles * per_tile;
        p.ok = true;
        if (!best.ok || p.cost < best.cost) best = p;
      }
    }
  }
  if (epi && mode != 4 && (!best.ok || static_cast<double>(pixels) / (static_cast<double>(best.tiles) * 128 * best.mt) < 0.6)) {
    epi = false;  // row-aligned tiles waste too much here: generic epilogue, linear raster
    goto plan;
  }
  if (mode == 0) {
    // junk raster positions must not eat the gain: tiny feature maps go through im2col loads instead
    const double eff = best.ok ? static_cast<double>(pixels) / (static_cast<double>(best.tiles) * 128 * best.mt) : 0.0;
    if (eff < 0.6) {
      if (no_im2col || L.out_s2d) return 0;
      mode = 2;
      goto plan;
    }
  }
  if (!best.ok && epi && epi_pad2) {  // no tile height fits the image: generic epilogue
    pad2_failed = true;
    epi = false;
    goto plan;
  }
  if (!best.ok) return 0;

  WinArgs a;
  std::memset(&a, 0, sizeof(a));
  a.mode = mode; a.h = win_h; a.w = win_w; a.hw = mode == 4 ? hp * wp : L.ho * L.wo;
  a.ksize = pc.ksize; a.stride = pc.stride; a.pad = pc.ksize / 2 - ilo; a.wo = L.wo; a.slabs_per_tap = slabs;
  a.out_pad = oext; a.out_lo = olo; a.in_lo = ilo; a.box_rows = best.bh; a.direct_out = direct_out ? 1 : 0;
  a.rw = best.rw; a.tw = best.tw; a.strips = best.strips; a.tstep = best.tstep;
  a.tiles_per_strip = best.tiles_per_strip; a.tiles_per_img = best.strips * best.tiles_per_strip;
  a.mt = best.mt; a.tm = 128 * best.mt;
  a.slab = slab; a.slabs = mode == 2 ? taps * slabs : slabs; a.taps = taps; a.cin_pad = pc.cin_pad;
  a.resident = resident ? 1 : 0; a.sa = best.sa; a.sb = resident ? 1 : sb;
  a.patch_bytes = best.patch_bytes; a.box_bytes = best.box_bytes; a.bstage_bytes = bstage_bytes;
  a.wbytes = static_cast<uint32_t>(wbytes);
  a.n_tile = n_tile; a.n_tiles = n_tiles; a.cout = pc.cout; a.cout_pad = cout_pad;
  a.wgt = pc.w; a.bias = pc.bias;
  if (epi) {
    if (!pc.bias_host) return fail(AICAM_ERR_INVALID_ARG, "conv_win: packed layer has no host copy of its bias");
    std::memcpy(a.bias4, pc.bias_host, sizeof(float) * cout_pad);
  }
  a.wgt_nt = (pc.w_nt && pc.nt_block == n_tile) ? pc.w_nt : nullptr; a.q_pad = pc.q_pad;
  a.out = L.out; a.out_img_stride = L.out_img_stride; a.out_cstride = L.out_cstride; a.out_coff = L.out_coff; a.out_f32 = L.out_f32;
  a.res = L.res; a.res_img_stride = L.res_img_stride; a.res_cstride = L.res_cstride; a.res_coff = L.res_coff; a.res_mode = res_mode;
  a.act = L.act;
  a.trace = L.trace;
  a.tl = timeline_slot(pc.cout * 1000000ll + pc.cin_pad * 1000ll + L.h);
  a.out_s2d = (window && L.out_s2d) ? 1 : 0;
  a.s2d_store = (epi && s2d_store) ? 1 : 0;
  a.batch = L.batch; a.batch_dev = L.batch_dev;
  a.idesc = (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n_tile >> 3) << 17) | (static_cast<uint32_t>(128 >> 4) << 24);
  uint32_t cols = 32;
  while (cols < static_cast<uint32_t>(2 * best.mt * n_tile)) cols <<= 1;
  a.tmem_cols = cols;
  const uint32_t ring_a_end = (epi ? OFF_RING_A_EPI : OFF_RING_A) + static_cast<uint32_t>(best.sa) * best.patch_bytes;
  a.off_w = ring_a_end;
  a.off_b = ring_a_end;
  a.off_stage = ring_a_end + static_cast<uint32_t>(resident ? (wbytes + 1023) / 1024 * 1024 : static_cast<size_t>(sb) * bstage_bytes);
  a.stage_pitch = stage_pitch;
  a.res_pitch = res_pitch;
  a.off_res = a.off_stage + a.tm * stage_pitch;
  a.th = window ? best.tstep / best.rw : 0;
  if (epi) {
    a.off_stage = (a.off_stage + 1023) / 1024 * 1024;
    a.nstage = best.nstage;
    a.off_res = a.off_stage + best.nstage * best.stage_buf;
    a.stage_buf_bytes = best.stage_buf;
    a.nres = best.nres;
    a.pieces = piece_ch[2] ? 4 : (piece_ch[1] ? 2 : 1);
    const int rows_c = window ? a.th * best.tw : a.tm;
    uint32_t off = 0;
    a.res_tx_bytes = 0;
    for (int q = 0; q < 4; ++q) {
      a.piece_ch[q] = piece_ch[q];
      a.piece_off[q] = off;
      off += static_cast<uint32_t>((static_cast<size_t>(rows_c) * piece_ch[q] * 2 + 1023) / 1024 * 1024);
      a.res_tx_bytes += static_cast<uint32_t>(rows_c) * piece_ch[q] * 2;
    }
  }
  a.inv_rw = 1.0f / static_cast<float>(best.rw);
  a.flat = (mode != 0 && L.out_img_stride == static_cast<long long>(a.hw) * L.out_cstride &&
            (!res_mode || L.res_img_stride == static_cast<long long>(a.hw) * L.res_cstride)) ? 1 : 0;
  a.res_direct = (!epi && res_mode != 0 && !res_staged) ? 1 : 0;
  a.res_inplace = (epi && mode == 4) ? 1 : 0;
  static const bool no_alt = getenv("AICAM_WIN_NO_EPI_ALT") != nullptr;
  if (L.decode) {
    // the decode phase reads whole fp32 rows of ONE n-tile from the generic epilogue's staging rows
    if (mode != 1 || epi || direct_out || n_tiles != 1 || !L.out_f32 || res_mode || (pc.cout & 3) || (L.decode == 1 && pc.cout != AICAM_HEAD_DFL) ||
        (L.decode == 1 && !L.dec_boxes) || (L.decode == 2 && (!L.dec_scores || !L.dec_labels)) || L.dec_anchors <= 0)
      return fail(AICAM_ERR_UNSUPPORTED, "conv_win: this layer cannot take the fused Detect decode");
    a.decode = L.decode; a.dec_anchor_base = L.dec_anchor_base; a.dec_anchors = L.dec_anchors;
    a.dec_stride = static_cast<float>(AICAM_YOLO_INPUT / L.w);
    a.dec_boxes = L.dec_boxes; a.dec_scores = L.dec_scores; a.dec_labels = L.dec_labels;
    a.flat = 0;  // (image, pixel) per row
  }
  a.ws = (ws_ok && best.mt == 2) ? 1 : 0;
  a.pad_store = (epi && epi_pad2) ? 1 : 0;
  a.img_tile = (mode == 4 && epi && best.img) ? 1 : 0;
  static const bool thread_arrive = getenv("AICAM_WIN_THREAD_ARRIVE") != nullptr;
  a.warp_arrive = thread_arrive ? 0 : 1;
  a.epi_alt = (!no_alt && epi && best.mt == 2 && n_tile <= 32 && best.nstage == 2 && (!res_mode || best.nres == 2) && !a.res_inplace) ? 1 : 0;
  const size_t smem = epi ? a.off_stage + static_cast<size_t>(best.stage_buf) * (best.nstage + (a.res_inplace ? 0 : best.nres))
                          : a.off_stage + (direct_out ? 0 : static_cast<size_t>(a.tm) * (stage_pitch + (res_staged ? res_pitch : 0)));
  if (smem > SMEM_LIMIT) return 0;

  alignas(64) WinMaps maps;
  std::memset(&maps, 0, sizeof(maps));
  CUtensorMap& tmap = maps.in;
  const CUtensorMapSwizzle sw = slab == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : (slab == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
  void* base = const_cast<__nv_bfloat16*>(L.in) + L.in_coff;
  CUresult cr;
  if (window) {
    const cuuint64_t dims[4] = {static_cast<cuuint64_t>(pc.cin_pad), static_cast<cuuint64_t>(L.w), static_cast<cuuint64_t>(L.h),
                                static_cast<cuuint64_t>(L.batch)};
    const cuuint64_t strides[3] = {static_cast<cuuint64_t>(L.in_cstride) * 2, static_cast<cuuint64_t>(L.w) * L.in_cstride * 2,
                                   static_cast<cuuint64_t>(L.h) * L.w * L.in_cstride * 2};
    const cuuint32_t box[4] = {static_cast<cuuint32_t>(slab), static_cast<cuuint32_t>(best.rw), static_cast<cuuint32_t>(best.bh), 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    cr = get_encode_tiled()(&maps.in, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                            CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  } else if (mode == 2) {
    // a padded input already holds its halo: the image is (h + 2) x (w + 2) and base pixels start at (ip - pad)
    const cuuint64_t dims[4] = {static_cast<cuuint64_t>(pc.cin_pad), static_cast<cuuint64_t>(wp), static_cast<cuuint64_t>(hp),
                                static_cast<cuuint64_t>(L.batch)};
    const cuuint64_t strides[3] = {static_cast<cuuint64_t>(L.in_cstride) * 2, static_cast<cuuint64_t>(wp) * L.in_cstride * 2,
                                   static_cast<cuuint64_t>(hp) * wp * L.in_cstride * 2};
    const int pad = pc.ksize / 2;
    const int ihi = iext - ilo;  // border rows / columns after the interior
    const int lower[2] = {ilo - pad, ilo - pad};
    const int upper[2] = {pad - (pc.ksize - 1) - ihi, pad - (pc.ksize - 1) - ihi};
    const cuuint32_t estr[4] = {1, static_cast<cuuint32_t>(pc.stride), static_cast<cuuint32_t>(pc.stride), 1};
    cr = get_encode_im2col()(&maps.in, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, base, dims, strides, lower, upper, static_cast<cuuint32_t>(slab),
                             128, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  } else {
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(pc.cin_pad), static_cast<cuuint64_t>(mode == 4 ? padded_pixels : pixels)};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(L.in_cstride) * 2};
    const cuuint32_t box[2] = {static_cast<cuuint32_t>(slab), static_cast<cuuint32_t>(mode == 4 ? best.bh : a.tm)};
    const cuuint32_t estr[2] = {1, 1};
    cr = get_encode_tiled()(&maps.in, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                            CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  }
  if (cr != CUDA_SUCCESS) {
    if (getenv("AICAM_REQUIRE_WIN")) return fail(AICAM_ERR_CUDA, "conv_win: cuTensorMapEncodeTiled failed with " + std::to_string(static_cast<int>(cr)));
    return 0;
  }

  if (epi) {
    // output / residual boxes: [piece channels][tw columns][th rows][1 image] of the NHWC tensor (channel slice)
    for (int q = 0; q < std::min(a.pieces, 2) && cr == CUDA_SUCCESS; ++q) {  // (pieces beyond the second reuse map 1)
      const int pb = piece_ch[q] * 2;
      const CUtensorMapSwizzle psw = pb == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : (pb == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
      if (a.pad_store || a.img_tile) {
        // interiors of the zero-bordered output images: (channels, wo, ho, batch), rows (wo + border) pixels apart
        const int hwo = L.ho * L.wo;
        const cuuint64_t pd[4] = {static_cast<cuuint64_t>(pc.cout), static_cast<cuuint64_t>(L.wo), static_cast<cuuint64_t>(L.ho),
                                  static_cast<cuuint64_t>(L.batch)};
        const cuuint64_t ps[3] = {static_cast<cuuint64_t>(L.out_cstride) * 2, static_cast<cuuint64_t>(L.wo + oext) * L.out_cstride * 2,
                                  static_cast<cuuint64_t>(L.out_img_stride) * 2};
        const cuuint32_t pbx[4] = {static_cast<cuuint32_t>(piece_ch[q]), static_cast<cuuint32_t>(L.wo),
                                   static_cast<cuuint32_t>(a.tm <= hwo ? a.tm / L.wo : L.ho), static_cast<cuuint32_t>(a.tm <= hwo ? 1 : a.tm / hwo)};
        const cuuint32_t pe[4] = {1, 1, 1, 1};
        __nv_bfloat16* obase = static_cast<__nv_bfloat16*>(L.out) + L.out_coff + static_cast<long long>(olo) * (L.wo + oext + 1) * L.out_cstride;
        cr = get_encode_tiled()(&maps.out[q], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, obase, pd, ps, pbx, pe, CU_TENSOR_MAP_INTERLEAVE_NONE, psw,
                                CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (cr == CUDA_SUCCESS && res_mode) {  // (image tiles: the residual shares the output's zero-bordered layout)
          const cuuint64_t rs[3] = {static_cast<cuuint64_t>(L.res_cstride) * 2, static_cast<cuuint64_t>(L.wo + oext) * L.res_cstride * 2,
                                    static_cast<cuuint64_t>(L.res_img_stride) * 2};
          const __nv_bfloat16* rbase = L.res + L.res_coff + static_cast<long long>(olo) * (L.wo + oext + 1) * L.res_cstride;
          cr = get_encode_tiled()(&maps.res[q], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<__nv_bfloat16*>(rbase), pd, rs, pbx, pe,
                                  CU_TENSOR_MAP_INTERLEAVE_NONE, psw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        }
        continue;
      }
      if (!window) {
        // flat: [piece channels][128 MT pixels] of the [pixels][cstride] matrix
        const cuuint64_t fd[2] = {static_cast<cuuint64_t>(pc.cout), static_cast<cuuint64_t>(mode == 4 ? padded_pixels : pixels)};
        const cuuint32_t fb[2] = {static_cast<cuuint32_t>(piece_ch[q]), static_cast<cuuint32_t>(a.tm)};
        const cuuint32_t fe[2] = {1, 1};
        const cuuint64_t fos[1] = {static_cast<cuuint64_t>(L.out_cstride) * 2};
        cr = get_encode_tiled()(&maps.out[q], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, static_cast<__nv_bfloat16*>(L.out) + L.out_coff, fd, fos, fb, fe,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, psw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (cr == CUDA_SUCCESS && res_mode) {
          const cuuint64_t frs[1] = {static_cast<cuuint64_t>(L.res_cstride) * 2};
          cr = get_encode_tiled()(&maps.res[q], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<__nv_bfloat16*>(L.res) + L.res_coff, fd, frs, fb,
                                  fe, CU_TENSOR_MAP_INTERLEAVE_NONE, psw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        }
        continue;
      }
      if (a.s2d_store) {
        // [n][y/2][x/2][y&1][x&1][C] seen as (2C, x/2, y&1, y/2, n): a (tw x th) tile is the box (2C, tw/2, 2, th/2, 1)
        const cuuint64_t C2 = static_cast<cuuint64_t>(pc.cout) * 2;
        const cuuint64_t d5[5] = {C2, static_cast<cuuint64_t>(L.wo / 2), 2, static_cast<cuuint64_t>(L.ho / 2), static_cast<cuuint64_t>(L.batch)};
        const cuuint64_t s5[4] = {2 * C2 * 2, C2 * 2, static_cast<cuuint64_t>(L.wo / 2) * 2 * C2 * 2,
                                  static_cast<cuuint64_t>(L.out_img_stride) * 2};
        const cuuint32_t b5[5] = {static_cast<cuuint32_t>(C2), static_cast<cuuint32_t>(best.tw / 2), 2, static_cast<cuuint32_t>(a.th / 2), 1};
        const cuuint32_t e5[5] = {1, 1, 1, 1, 1};
        cr = get_encode_tiled()(&maps.out[q], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, static_cast<__nv_bfloat16*>(L.out), d5, s5, b5, e5,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        continue;
      }
      const cuuint32_t box[4] = {static_cast<cuuint32_t>(piece_ch[q]), static_cast<cuuint32_t>(best.tw), static_cast<cuuint32_t>(a.th), 1};
      const cuuint32_t estr[4] = {1, 1, 1, 1};
      const cuuint64_t odims[4] = {static_cast<cuuint64_t>(pc.cout), static_cast<cuuint64_t>(L.wo), static_cast<cuuint64_t>(L.ho),
                                   static_cast<cuuint64_t>(L.batch)};
      const cuuint64_t ostr[3] = {static_cast<cuuint64_t>(L.out_cstride) * 2, static_cast<cuuint64_t>(L.wo) * L.out_cstride * 2,
                                  static_cast<cuuint64_t>(L.out_img_stride) * 2};
      cr = get_encode_tiled()(&maps.out[q], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, static_cast<__nv_bfloat16*>(L.out) + L.out_coff, odims, ostr,
                              box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, psw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (cr == CUDA_SUCCESS && res_mode) {
        const cuuint64_t rstr[3] = {static_cast<cuuint64_t>(L.res_cstride) * 2, static_cast<cuuint64_t>(L.wo) * L.res_cstride * 2,
                                    static_cast<cuuint64_t>(L.res_img_stride) * 2};
        cr = get_encode_tiled()(&maps.res[q], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<__nv_bfloat16*>(L.res) + L.res_coff, odims, rstr,
                                box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, psw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      }
    }
    if (cr != CUDA_SUCCESS)
      return fail(AICAM_ERR_CUDA, "conv_win: cuTensorMapEncodeTiled (epilogue) failed with " + std::to_string(static_cast<int>(cr)));
  }
  static const bool debug_plan = getenv("AICAM_WIN_DEBUG") != nullptr;
  if (debug_plan)
    fprintf(stderr, "conv_win: %dx%d c%d->%d k%d s%d mode %d mt %d n_tile %d x%d slab %d x%d resident %d sa %d sb %d patch %u bstage %u "
            "epi %d direct %d tiles %lld smem %zu\n", L.h, L.w, pc.cin_pad, pc.cout, pc.ksize, pc.stride, mode, best.mt, n_tile, n_tiles,
            slab, slabs, resident ? 1 : 0, a.sa, a.sb, a.patch_bytes, a.bstage_bytes, epi ? 1 : 0, a.direct_out, best.tiles * n_tiles, smem);
  WinKernelFn kernel = pick_kernel(slab, mode, best.mt, L.act, (epi ? 1 : 0) | (a.ws ? 2 : 0));
  if (int rc = ensure_dynamic_smem(kernel, SMEM_LIMIT)) return rc;  // per (device, instantiation)
  const int num_sms = current_num_sms();
  const long long total_tiles = best.tiles * n_tiles;
  dim3 grid(static_cast<unsigned>(std::min<long long>(total_tiles, num_sms)));
  size_t slot = 0;
  const bool prof = profile_begin(stream, &slot);
  {
    // programmatic dependent launch: this layer's prologue (barriers, TMEM, bias, resident weights / first weight
    // stages) overlaps the previous layer's tail; its activation traffic starts after griddepcontrol.wait
    static const bool no_pdl = getenv("AICAM_NO_PDL") != nullptr;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = dim3(WIN_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = no_pdl ? 0 : 1;
    const cudaError_t le = cudaLaunchKernelEx(&cfg, kernel, a, maps);
    if (le != cudaSuccess) return fail(AICAM_ERR_CUDA, std::string("conv_win: launch failed: ") + cudaGetErrorString(le));
  }
  if (prof) profile_end(stream, slot);
  count_launch();
  const int rc = last_launch("conv_win_kernel");
  return rc ? rc : 1;
}

}  // namespace aicam
