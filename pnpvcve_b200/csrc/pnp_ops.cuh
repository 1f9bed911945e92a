// Launchers of the memory-bound kernels in pnp_ops.cu.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace pnp {

struct DynRef;

constexpr int kPackBlockBytes = 8192;

// tensor2img's quantisation of one sample (mmedit/core/misc.py:55-56,69): clamp_(0,1); (v - 0) / (1 - 0); * 255.0;
// numpy round (half to even).  Returns the uint8 value as a float.  Shared by the metrics and the uint8 store of
// conv_last, so that a uint8 frame is exactly what quantising the fp32 frame gives.
__device__ __forceinline__ float quant_u8(float v) {
  v = fminf(fmaxf(v, 0.0f), 1.0f);
  return rintf(__fmul_rn(v, 255.0f));
}

// tm_src / tm_dst: (64, W, H, images) bf16 maps of the source / destination buffer, boxes (64, 10, 10, 1) / (64, 8, 8, 1),
// 128B swizzle, zero fill; table mode: both span the pool that starts at pool_base and the entry's pointers select the
// images
cudaError_t warp_prepare();
cudaError_t launch_mv_warp(const CUtensorMap& tm_src, const CUtensorMap& tm_dst, const void* src, const float* flow_x,
                           const float* flow_y, long long flow_sy, long long flow_sn, void* dst, int N, int H, int W,
                           int* dbg_x0, int* dbg_y0, const DynRef& dyn, const void* pool_base, int use_tma,
                           cudaStream_t stream);
cudaError_t launch_lr_im2col(const float* lr, long long sn, long long sc, long long sy, void* dst, int N,
                             int H, int W, int dst_channels, const DynRef& dyn, cudaStream_t stream);
cudaError_t launch_fetch_pinned(const void* src_dev_view, void* dst, long long bytes, cudaStream_t stream);
cudaError_t launch_pack_mix_blocks(const float* w2, const float* w1x1, int n_blocks, int n_experts, const float* coef,
                                   const float* row_scale, void* dst, long long dst_stride, cudaStream_t stream);
cudaError_t launch_pack_conv3x3_rowstack(const float* w, int n_experts, const float* coef,
                                         const float* row_scale, int out_ch, int in_total, int in_begin,
                                         int in_begin2, int in_count, void* dst, int tap_n, bool flip_ky,
                                         cudaStream_t stream);
cudaError_t launch_pack_rows(const float* w, int rows, int cols, long long row_stride, long long col_stride,
                             void* dst, int row_offset, cudaStream_t stream);
cudaError_t launch_pack_aux(const float* w, int out_ch, int in_total, void* dst, cudaStream_t stream);
cudaError_t launch_caa_heads(const float* base_qp, const float* qp, int frames, const float* b0w,
                             const float* b0b, const float* b2w, const float* b2b, const float* s0w,
                             const float* s2w, int n_experts, int se_hidden, float* experts, float* gamma,
                             cudaStream_t stream);
cudaError_t launch_mix_bias(const float* conv2_bias, long long block_stride, int n_blocks, int n_experts,
                            const float* experts, const float* gamma, int frames, float* out,
                            cudaStream_t stream);

cudaError_t launch_unit_from_u8(const uint8_t* src, long long s_sf, long long s_sc, long long s_sy, float* dst,
                               long long d_sf, long long d_sc, long long d_sy, int F, int H, int W,
                               cudaStream_t stream);

// a_u8 / b_u8: the operand is a uint8 frame (read as is) instead of an fp32 one (quantised with quant_u8)
cudaError_t launch_frame_quality(const void* a, bool a_u8, long long a_sf, long long a_sc, long long a_sy,
                                 const void* b, bool b_u8, long long b_sf, long long b_sc, long long b_sy, int F, int H,
                                 int W, int crop, int ch_first, int n_ch, const double* gauss11,
                                 unsigned long long* sse, double* ssim_sum, int num_sms, cudaStream_t stream);

// window = false: a whole clip (tail must be 0, every negative p_target is an error); true: a frame window with `tail`
// (0 / 1) tail frames after its T frames and p_target -2 for targets before the window
cudaError_t launch_mv_rasterize(const float* rec, const int* frame_off, const int* is_b, const int* p_target,
                                int T, int tail, bool window, int R, int H, int W, unsigned* own_f, unsigned* own_b,
                                unsigned* pmask, float* mvs, float* partitions, int* status, cudaStream_t stream);

}  // namespace pnp
