// Small NHWC bf16 layers around the convolutions: max-pool (SPPF 5x5 s1, ReID 3x3 s2),
// nearest 2x upsample into a concat slice, global average pool + L2 normalise, and the
// fp32 NCHW -> bf16 NHWC4 converter used by the TRTEngine-shaped facade.
// All are HBM/L2-bound elementwise kernels: 16-byte vector accesses, one 8-channel group
// per thread, consecutive threads on consecutive channel groups (coalesced).
#include "layers.cuh"

namespace aicam {

extern void count_launch();

namespace {

__device__ __forceinline__ uint32_t bf16x2_max(uint32_t a, uint32_t b) {
  __nv_bfloat162 x = *reinterpret_cast<__nv_bfloat162*>(&a);
  __nv_bfloat162 y = *reinterpret_cast<__nv_bfloat162*>(&b);
  __nv_bfloat162 r = __hmax2(x, y);
  return *reinterpret_cast<uint32_t*>(&r);
}

// out[n][oy][ox][coff_out + c] = max over k x k window (pad k/2, -inf padding) of in[..][coff_in + c]
__global__ void maxpool_kernel(const __nv_bfloat16* __restrict__ in, long long in_img_stride, int in_cstride,
                               int in_coff, int h, int w, int c8, int k, int stride, int ho, int wo,
                               __nv_bfloat16* __restrict__ out, long long out_img_stride, int out_cstride,
                               int out_coff, long long total, const int* __restrict__ n_dev) {
  const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (idx >= total) return;
  const int g = static_cast<int>(idx % c8);
  long long p = idx / c8;
  const int ox = static_cast<int>(p % wo); p /= wo;
  const int oy = static_cast<int>(p % ho);
  const int n = static_cast<int>(p / ho);
  if (n_dev && n >= __ldg(n_dev)) return;
  const int pad = k / 2;
  const uint32_t ninf = 0xFF80FF80u;  // two bf16 -inf
  uint4 m = make_uint4(ninf, ninf, ninf, ninf);
  const __nv_bfloat16* base = in + n * in_img_stride + in_coff + g * 8;
  for (int dy = 0; dy < k; ++dy) {
    const int iy = oy * stride - pad + dy;
    if (iy < 0 || iy >= h) continue;
    for (int dx = 0; dx < k; ++dx) {
      const int ix = ox * stride - pad + dx;
      if (ix < 0 || ix >= w) continue;
      const uint4 v = __ldg(reinterpret_cast<const uint4*>(base + (static_cast<long long>(iy) * w + ix) * in_cstride));
      m.x = bf16x2_max(m.x, v.x); m.y = bf16x2_max(m.y, v.y);
      m.z = bf16x2_max(m.z, v.z); m.w = bf16x2_max(m.w, v.w);
    }
  }
  *reinterpret_cast<uint4*>(out + n * out_img_stride + (static_cast<long long>(oy) * wo + ox) * out_cstride +
                            out_coff + g * 8) = m;
}

// SPPF: three chained 5x5 stride-1 max-pools (= windows 5, 9, 13 of the input) in ONE launch.  A block owns one image
// x 32 channels (64-byte runs per pixel): the map lives in shared memory, each pool is a separable row / column max,
// every pooled map is written to its channel slice of the concat buffer and feeds the next pool from shared memory.
__global__ void __launch_bounds__(256) sppf_pool3_kernel(__nv_bfloat16* __restrict__ buf, long long img_stride, int cstride,
                                                         int coff, int h, int w, int hc, const int* __restrict__ n_dev) {
  extern __shared__ __align__(16) uint4 sp[];  // three [h * w][4] tiles
  const int blocks_per_img = hc >> 5;
  const int n = blockIdx.x / blocks_per_img, cb = blockIdx.x - n * blocks_per_img;
  if (n_dev && n >= __ldg(n_dev)) return;
  const int hw = h * w, items = hw * 4;
  uint4* A = sp;
  uint4* T = sp + items;
  uint4* B = sp + 2 * items;
  __nv_bfloat16* base = buf + n * img_stride + coff + cb * 32;
  for (int i = threadIdx.x; i < items; i += blockDim.x)
    A[i] = *reinterpret_cast<const uint4*>(base + static_cast<long long>(i >> 2) * cstride + (i & 3) * 8);
  __syncthreads();
  auto mx = [](uint4 a, uint4 b) {
    return make_uint4(bf16x2_max(a.x, b.x), bf16x2_max(a.y, b.y), bf16x2_max(a.z, b.z), bf16x2_max(a.w, b.w));
  };
  for (int r = 1; r <= 3; ++r) {
    for (int i = threadIdx.x; i < items; i += blockDim.x) {  // row max over x - 2 .. x + 2
      const int px = i >> 2, g = i & 3, y = px / w, x = px - y * w;
      uint4 m = A[i];
      for (int dx = -2; dx <= 2; ++dx)
        if (dx != 0 && x + dx >= 0 && x + dx < w) m = mx(m, A[((px + dx) << 2) + g]);
      T[i] = m;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < items; i += blockDim.x) {  // column max over y - 2 .. y + 2
      const int px = i >> 2, g = i & 3, y = px / w;
      uint4 m = T[i];
      for (int dy = -2; dy <= 2; ++dy)
        if (dy != 0 && y + dy >= 0 && y + dy < h) m = mx(m, T[((px + dy * w) << 2) + g]);
      B[i] = m;
      *reinterpret_cast<uint4*>(base + static_cast<long long>(r) * hc + static_cast<long long>(px) * cstride + g * 8) = m;
    }
    __syncthreads();
    uint4* t2 = A; A = B; B = t2;
  }
}

// nearest-neighbour 2x: one thread per INPUT 16-byte chunk (8 channels of one pixel): one load, four stores
__global__ void __launch_bounds__(256) upsample2x_kernel(const __nv_bfloat16* __restrict__ in, long long in_img_stride, int in_cstride,
                                                         int in_coff, int h, int w, int c8, __nv_bfloat16* __restrict__ out,
                                                         long long out_img_stride, int out_cstride, int out_coff, unsigned total,
                                                         const int* __restrict__ n_dev) {
  const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const unsigned g = idx % c8;
  unsigned p = idx / c8;
  const unsigned x = p % w; p /= w;
  const unsigned y = p % h;
  const unsigned n = p / h;
  if (n_dev && static_cast<int>(n) >= __ldg(n_dev)) return;
  const uint4 v = __ldg(reinterpret_cast<const uint4*>(
      in + n * in_img_stride + (static_cast<long long>(y) * w + x) * in_cstride + in_coff + g * 8));
  __nv_bfloat16* o = out + n * out_img_stride + (static_cast<long long>(2 * y) * 2 * w + 2 * x) * out_cstride + out_coff + g * 8;
  const long long row = static_cast<long long>(2 * w) * out_cstride;
  *reinterpret_cast<uint4*>(o) = v;
  *reinterpret_cast<uint4*>(o + out_cstride) = v;
  *reinterpret_cast<uint4*>(o + row) = v;
  *reinterpret_cast<uint4*>(o + row + out_cstride) = v;
}

// One block per image: mean over hw pixels of each of c channels, then x / ||x||_2 (fp32).  Thread t owns the
// 8-channel group t % (c / 8) (16-byte loads) and every (256 / (c / 8))-th pixel; partial sums meet in shared memory.
__global__ void __launch_bounds__(256) avgpool_l2norm_kernel(const __nv_bfloat16* __restrict__ in, int hw, int hw_div, int c,
                                                             float* __restrict__ out, const int* __restrict__ n_dev) {
  extern __shared__ float red[];  // [256][8] partial sums, then the block reduction of the squared norm
  const int n = blockIdx.x;
  if (n_dev && n >= __ldg(n_dev)) return;
  const int groups = c >> 3;                   // 8-channel groups (<= 256)
  const int lanes = blockDim.x / groups;       // pixel phases per group
  const int g = threadIdx.x % groups, ph = threadIdx.x / groups;
  const __nv_bfloat16* base = in + static_cast<long long>(n) * hw * c + g * 8;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (ph < lanes)
    for (int p = ph; p < hw; p += lanes) {
      const uint4 v = __ldg(reinterpret_cast<const uint4*>(base + static_cast<long long>(p) * c));
      const uint32_t wv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) { acc[2 * i] += bf16_lo(wv[i]); acc[2 * i + 1] += bf16_hi(wv[i]); }
    }
#pragma unroll
  for (int i = 0; i < 8; ++i) red[threadIdx.x * 8 + i] = acc[i];
  __syncthreads();
  float ss = 0.0f;
  for (int ch = threadIdx.x; ch < c; ch += blockDim.x) {  // phases summed in a fixed order: deterministic
    float s = 0.0f;
    for (int q = 0; q < lanes; ++q) s += red[(q * groups + (ch >> 3)) * 8 + (ch & 7)];
    s /= static_cast<float>(hw_div);
    out[static_cast<long long>(n) * c + ch] = s;
    ss += s * s;
  }
  __syncthreads();
  red[threadIdx.x] = ss;
  __syncthreads();
  for (int o = blockDim.x / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  const float inv = 1.0f / sqrtf(red[0]);
  for (int ch = threadIdx.x; ch < c; ch += blockDim.x) out[static_cast<long long>(n) * c + ch] *= inv;
}

__global__ void nchw_to_nhwc4_kernel(const float* __restrict__ in, int hw, __nv_bfloat16* __restrict__ out,
                                     long long total) {
  const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (idx >= total) return;
  const long long n = idx / hw;
  const long long p = idx - n * hw;
  const float* b = in + n * 3 * hw + p;
  uint2 o;
  o.x = pack_bf16x2(b[0], b[hw]);
  o.y = pack_bf16x2(b[2 * static_cast<long long>(hw)], 0.0f);
  reinterpret_cast<uint2*>(out)[idx] = o;
}

// [n][h][w][c] -> [n][h/2][w/2][2x2 sub-pixel][c]: one thread per 16-byte (or, for 4 channels, 8-byte) piece
template <typename V>
__global__ void space_to_depth_kernel(const V* __restrict__ in, V* __restrict__ out, int h, int w, int pieces, long long total,
                                      const int* __restrict__ n_dev) {
  const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (idx >= total) return;
  const int pc = static_cast<int>(idx % pieces);
  long long p = idx / pieces;
  const int x = static_cast<int>(p % w); p /= w;
  const int y = static_cast<int>(p % h);
  const long long n = p / h;
  if (n_dev && n >= __ldg(n_dev)) return;
  const long long dst = (((n * (h >> 1) + (y >> 1)) * (w >> 1) + (x >> 1)) * 4 + ((y & 1) << 1) + (x & 1)) * pieces + pc;
  out[dst] = __ldg(in + idx);
}

}  // namespace

int launch_space_to_depth(const __nv_bfloat16* in, int batch, int h, int w, int c, __nv_bfloat16* out, cudaStream_t stream,
                          const int* n_dev) {
  if ((c != 4 && c % 8) || h % 2 || w % 2) return fail(AICAM_ERR_INVALID_ARG, "space_to_depth: 4 or a multiple of 8 channels, even sizes");
  const int pieces = c == 4 ? 1 : c / 8;
  const long long total = static_cast<long long>(batch) * h * w * pieces;
  if (total == 0) return AICAM_OK;
  const unsigned blocks = static_cast<unsigned>((total + 255) / 256);
  if (c == 4)
    space_to_depth_kernel<uint2><<<blocks, 256, 0, stream>>>(reinterpret_cast<const uint2*>(in), reinterpret_cast<uint2*>(out), h, w, 1, total, n_dev);
  else
    space_to_depth_kernel<uint4><<<blocks, 256, 0, stream>>>(reinterpret_cast<const uint4*>(in), reinterpret_cast<uint4*>(out), h, w, pieces, total, n_dev);
  count_launch();
  return last_launch("space_to_depth_kernel");
}

int launch_maxpool(const __nv_bfloat16* in, long long in_img_stride, int in_cstride, int in_coff, int batch, int h,
                   int w, int c, int k, int stride, __nv_bfloat16* out, long long out_img_stride, int out_cstride,
                   int out_coff, cudaStream_t stream, const int* n_dev) {
  if (c % 8 || in_cstride % 8 || in_coff % 8 || out_cstride % 8 || out_coff % 8)
    return fail(AICAM_ERR_INVALID_ARG, "maxpool: channel counts/offsets must be multiples of 8");
  const int pad = k / 2;
  const int ho = (h + 2 * pad - k) / stride + 1, wo = (w + 2 * pad - k) / stride + 1;
  const long long total = static_cast<long long>(batch) * ho * wo * (c / 8);
  if (total == 0) return AICAM_OK;
  maxpool_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, stream>>>(
      in, in_img_stride, in_cstride, in_coff, h, w, c / 8, k, stride, ho, wo, out, out_img_stride, out_cstride,
      out_coff, total, n_dev);
  count_launch();
  return last_launch("maxpool_kernel");
}

// pools 5 / 9 / 13 of channels [coff, coff + hc) of `buf` into [coff + hc, coff + 4 hc); returns 1 when launched,
// 0 when the shape is not eligible (the caller chains three max-pools instead)
int try_launch_sppf_pool3(__nv_bfloat16* buf, long long img_stride, int cstride, int coff, int batch, int h, int w, int hc,
                          cudaStream_t stream, const int* n_dev) {
  const size_t smem = static_cast<size_t>(3) * h * w * 64;
  if (hc % 32 || cstride % 8 || coff % 8 || smem > 200 * 1024 || batch <= 0) return 0;
  if (ensure_dynamic_smem(sppf_pool3_kernel, 200 * 1024) != AICAM_OK) return 0;
  sppf_pool3_kernel<<<static_cast<unsigned>(batch * (hc / 32)), 256, smem, stream>>>(buf, img_stride, cstride, coff, h, w, hc, n_dev);
  count_launch();
  const int rc = last_launch("sppf_pool3_kernel");
  return rc ? rc : 1;
}

int launch_upsample2x(const __nv_bfloat16* in, long long in_img_stride, int in_cstride, int in_coff, int batch, int h,
                      int w, int c, __nv_bfloat16* out, long long out_img_stride, int out_cstride, int out_coff,
                      cudaStream_t stream, const int* n_dev) {
  if (c % 8 || in_cstride % 8 || in_coff % 8 || out_cstride % 8 || out_coff % 8)
    return fail(AICAM_ERR_INVALID_ARG, "upsample: channel counts/offsets must be multiples of 8");
  const long long total = static_cast<long long>(batch) * h * w * (c / 8);  // input chunks
  if (total == 0) return AICAM_OK;
  if (total >= (1ll << 32)) return fail(AICAM_ERR_CAPACITY, "upsample: tensor too large");
  upsample2x_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, stream>>>(
      in, in_img_stride, in_cstride, in_coff, h, w, c / 8, out, out_img_stride, out_cstride, out_coff, static_cast<unsigned>(total), n_dev);
  count_launch();
  return last_launch("upsample2x_kernel");
}

int launch_avgpool_l2norm(const __nv_bfloat16* in, int batch, int hw, int hw_div, int c, float* out, cudaStream_t stream,
                          const int* n_dev) {
  if (batch == 0) return AICAM_OK;
  if (c % 8 || c > 2048 || 256 % (c / 8 > 256 ? 256 : c / 8))
    return fail(AICAM_ERR_INVALID_ARG, "avgpool_l2norm: channels must be 8 x a divisor of 256");
  if (c / 8 > 256) return fail(AICAM_ERR_INVALID_ARG, "avgpool_l2norm: at most 2048 channels");
  avgpool_l2norm_kernel<<<batch, 256, 256 * 8 * sizeof(float), stream>>>(in, hw, hw_div, c, out, n_dev);
  count_launch();
  return last_launch("avgpool_l2norm_kernel");
}

int launch_nchw_to_nhwc4(const float* in, int n, int h, int w, __nv_bfloat16* out, cudaStream_t stream) {
  const long long total = static_cast<long long>(n) * h * w;
  if (total == 0) return AICAM_OK;
  nchw_to_nhwc4_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, stream>>>(in, h * w, out, total);
  count_launch();
  return last_launch("nchw_to_nhwc4_kernel");
}

}  // namespace aicam
