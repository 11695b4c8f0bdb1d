#pragma once
#include "common.cuh"

namespace aicam {

int launch_maxpool(const __nv_bfloat16* in, long long in_img_stride, int in_cstride, int in_coff, int batch, int h,
                   int w, int c, int k, int stride, __nv_bfloat16* out, long long out_img_stride, int out_cstride,
                   int out_coff, cudaStream_t stream, const int* n_dev = nullptr);
int try_launch_sppf_pool3(__nv_bfloat16* buf, long long img_stride, int cstride, int coff, int batch, int h, int w, int hc,
                          cudaStream_t stream, const int* n_dev = nullptr);
int launch_upsample2x(const __nv_bfloat16* in, long long in_img_stride, int in_cstride, int in_coff, int batch, int h,
                      int w, int c, __nv_bfloat16* out, long long out_img_stride, int out_cstride, int out_coff,
                      cudaStream_t stream, const int* n_dev = nullptr);
// mean over the hw pixels stored per image divided by hw_div (hw > hw_div: zero-bordered images), then L2 normalisation
int launch_avgpool_l2norm(const __nv_bfloat16* in, int batch, int hw, int hw_div, int c, float* out, cudaStream_t stream,
                          const int* n_dev = nullptr);
// bf16 [n][h][w][c] -> [n][h/2][w/2][2x2 sub-pixel][c] (c = 4 or a multiple of 8)
int launch_space_to_depth(const __nv_bfloat16* in, int batch, int h, int w, int c, __nv_bfloat16* out, cudaStream_t stream,
                          const int* n_dev = nullptr);
int launch_nchw_to_nhwc4(const float* in, int n, int h, int w, __nv_bfloat16* out, cudaStream_t stream);

}  // namespace aicam
