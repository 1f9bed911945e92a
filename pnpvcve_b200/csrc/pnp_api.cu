// extern "C" surface of libpnpvcve.so (declared in include/pnp_vcve.h).
#include <cmath>
#include <cstddef>
#include <cuda.h>
#include <cuda_runtime.h>
#include <mutex>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/pnp_vcve.h"
#include "pnp_conv.cuh"
#include "pnp_ops.cuh"

namespace {

thread_local char g_err[512] = "";
int g_pair_override = -1;      // pnp_set_pair_mode(): -1 = follow PNP_PAIR

static_assert(sizeof(pnp_dyn_entry) == sizeof(pnp::DynEntry), "launch-table entry layout");

int fail(int code, const char* fmt, const char* detail = "") {
  snprintf(g_err, sizeof(g_err), fmt, detail);
  return code;
}

int cuda_fail(cudaError_t e, const char* where) {
  snprintf(g_err, sizeof(g_err), "%s: %s", where, cudaGetErrorString(e));
  return PNP_ERR_CUDA;
}

struct DeviceInfo {
  bool ok = false;
  int sms = 0;
  int max_pairs = 0;       // CTA pairs (clusters of 2) of the pair conv variants that can be resident at once
  cudaError_t err = cudaSuccess;
};

// One entry per device ordinal, filled exactly once (std::call_once) and read-only afterwards: properties, and the
// shared-memory opt-in of every conv kernel variant (done here so that it never happens inside a stream capture).
DeviceInfo g_dev[64];
std::once_flag g_dev_once[64];

int device_info(DeviceInfo** out) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return cuda_fail(e, "cudaGetDevice");
  if (dev < 0 || dev >= 64) return fail(PNP_ERR_ARG, "device ordinal out of range");
  std::call_once(g_dev_once[dev], [dev]() {
    cudaDeviceProp prop;
    cudaError_t e2 = cudaGetDeviceProperties(&prop, dev);
    if (e2 == cudaSuccess) {
      g_dev[dev].ok = (prop.major == 10);
      g_dev[dev].sms = prop.multiProcessorCount;
      if (g_dev[dev].ok) e2 = pnp::conv_rows_prepare(&g_dev[dev].max_pairs);
      if (g_dev[dev].ok && e2 == cudaSuccess) e2 = pnp::warp_prepare();
    }
    g_dev[dev].err = e2;
  });
  *out = &g_dev[dev];
  if (g_dev[dev].err != cudaSuccess) return cuda_fail(g_dev[dev].err, "device initialisation");
  if (!g_dev[dev].ok) return fail(PNP_ERR_ARCH, "libpnpvcve needs an sm_100 device (B200)");
  return PNP_OK;
}

// Process-wide switches, read ONCE when the library is first used.  Only performance-neutral layout knobs exist in the
// default build; the what-if / trace knobs that make results wrong or write through a pointer taken from the
// environment exist only in PNP_DIAG builds (tools/).
struct Knobs {
  int l2_hints = 0;        // PNP_L2_HINTS=1: evict_first on launch B's dead reads (measured: no effect); 2: residency scheme --
                           // launch A keeps x (evict_last) and streams t (evict_first), launch B streams t and x and
                           // keeps its output for the next launch A; 3: launch A keeps t instead (B's source)
  int par_split = 1;       // PNP_PAR_SPLIT=0: single-role epilogue of block launch A
  int warp_tma = 1;        // PNP_WARP_TMA=0: the warp takes its taps by global gathers only (A/B timing)
  int pair = 0;            // PNP_PAIR=1: CTA-pair (cta_group::2) form of the conv kernel where the shape allows it; 2: also
                           // with a phantom column.  Off by default: measured level in cycles and 3-5 % slower in time
                           // under the power cap (profiles/r02_notes.md); pnp_set_pair_mode() overrides at run time
  int rings_nio = 0, rings_sa = 0;   // PNP_RINGS="<n_io>,<s_a>": shared-memory split override
  int debug_skip = 0;      // PNP_DIAG only
  long long* trace = nullptr;   // PNP_DIAG only
};

const Knobs& knobs() {
  static const Knobs k = []() {
    Knobs v;
    if (const char* e = getenv("PNP_L2_HINTS")) v.l2_hints = atoi(e);
    if (const char* e = getenv("PNP_PAR_SPLIT")) v.par_split = atoi(e) != 0;
    if (const char* e = getenv("PNP_PAIR")) v.pair = atoi(e);
    if (const char* e = getenv("PNP_WARP_TMA")) v.warp_tma = atoi(e) != 0;
    if (const char* e = getenv("PNP_RINGS")) {
      if (sscanf(e, "%d,%d", &v.rings_nio, &v.rings_sa) != 2) v.rings_nio = v.rings_sa = 0;
    }
#ifdef PNP_DIAG
    if (const char* e = getenv("PNP_DEBUG_SKIP")) v.debug_skip = atoi(e);
    if (const char* e = getenv("PNP_TRACE_PTR")) v.trace = reinterpret_cast<long long*>(strtoull(e, nullptr, 10));
#endif
    return v;
  }();
  return k;
}

pnp::DynRef dyn_ref(const pnp_dyn_ref* d) {
  pnp::DynRef r;
  r.table = d ? reinterpret_cast<const pnp::DynEntry*>(d->table) : nullptr;
  r.step = d ? d->step : nullptr;
  r.node = d ? d->node : 0;
  r.stride = d ? d->stride : 0;
  return r;
}

typedef CUresult (*MemsetD32AsyncFn)(CUdeviceptr, unsigned int, size_t, CUstream);

MemsetD32AsyncFn memset32_fn() {
  static MemsetD32AsyncFn fn = []() -> MemsetD32AsyncFn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuMemsetD32Async", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      return reinterpret_cast<MemsetD32AsyncFn>(p);
    return nullptr;
  }();
  return fn;
}

int store_step(int32_t* word, int32_t value, cudaStream_t stream) {
  MemsetD32AsyncFn fn = memset32_fn();
  if (fn == nullptr) return fail(PNP_ERR_CUDA, "cuMemsetD32Async entry point not available");
  CUresult r = fn(reinterpret_cast<CUdeviceptr>(word), static_cast<unsigned int>(value), 1, stream);
  if (r != CUDA_SUCCESS) {
    snprintf(g_err, sizeof(g_err), "cuMemsetD32Async failed with CUresult %d", (int)r);
    return PNP_ERR_CUDA;
  }
  return PNP_OK;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = []() -> EncodeTiledFn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      return reinterpret_cast<EncodeTiledFn>(p);
    return nullptr;
  }();
  return fn;
}

// (64, W, H, N) bf16 NHWC tensor, box (64, box_w, 1, 1), 128-byte swizzle, zero fill out of range.
// spx/sy/sn: element strides between pixels / rows / images (0 = contiguous NHWC).
// ch = 32: a (32, W, H, N) tensor of 64-byte pixels, box (32, box_w, 1, 1), 64-byte swizzle (the LR im2col operand).
int make_map(CUtensorMap* m, const void* base, int N, int H, int W, int box_w, long long spx = 0, long long sy = 0,
             long long sn = 0, int box_h = 1, int ch = 64) {
  EncodeTiledFn fn = encode_fn();
  if (fn == nullptr) return fail(PNP_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  const cuuint64_t px = (cuuint64_t)ch * 2;
  cuuint64_t dims[4] = {(cuuint64_t)ch, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {px, (cuuint64_t)W * px, (cuuint64_t)H * W * px};
  if (spx != 0) {
    strides[0] = (cuuint64_t)spx * 2;
    strides[1] = (cuuint64_t)sy * 2;
    strides[2] = (cuuint64_t)sn * 2;
  }
  cuuint32_t box[4] = {(cuuint32_t)ch, (cuuint32_t)box_w, (cuuint32_t)box_h, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, ch == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(g_err, sizeof(g_err), "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return PNP_ERR_CUDA;
  }
  return PNP_OK;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// pnp_frame_quality / pnp_frame_quality_u8: one implementation, operands fp32 or uint8
int frame_quality(const char* name, const void* a, bool a_u8, int64_t a_sf, int64_t a_sc, int64_t a_sy, const void* b,
                  bool b_u8, int64_t b_sf, int64_t b_sc, int64_t b_sy, int F, int H, int W, int crop_border,
                  unsigned long long* sse, double* ssim_sum, void* stream) {
  if (!a || !b || !sse || !ssim_sum) return fail(PNP_ERR_ARG, "%s: null pointer", name);
  if (F < 1 || crop_border < 0 || H - 2 * crop_border < 11 || W - 2 * crop_border < 11)
    return fail(PNP_ERR_ARG, "%s: the cropped frame must be at least 11 x 11", name);
  if ((long long)F * 3 > 65535) return fail(PNP_ERR_ARG, "%s: at most 21845 frames per call", name);
  DeviceInfo* d;
  int rc = device_info(&d);
  if (rc) return rc;
  // cv2.getGaussianKernel(11, 1.5): exp(-(i-5)^2 / (2 sigma^2)), normalised to sum 1 (float64)
  double g[11], s = 0.0;
  for (int i = 0; i < 11; ++i) {
    g[i] = exp(-((double)(i - 5) * (i - 5)) / (2.0 * 1.5 * 1.5));
    s += g[i];
  }
  for (int i = 0; i < 11; ++i) g[i] /= s;
  const int ch_first = crop_border != 0 ? 2 : 0, n_ch = crop_border != 0 ? 1 : 3;
  cudaError_t e = pnp::launch_frame_quality(a, a_u8, a_sf, a_sc, a_sy, b, b_u8, b_sf, b_sc, b_sy, F, H, W, crop_border,
                                            ch_first, n_ch, g, sse, ssim_sum, d->sms, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? PNP_OK : cuda_fail(e, name);
}

}  // namespace

extern "C" {

static_assert(sizeof(pnp_conv_desc) == 280 && offsetof(pnp_conv_desc, out_spx) == 184 &&
                  offsetof(pnp_conv_desc, img_off) == 224 && offsetof(pnp_conv_desc, dyn) == 232 &&
                  offsetof(pnp_conv_desc, src_images) == 256 && offsetof(pnp_conv_desc, aux_channels) == 272 &&
                  offsetof(pnp_conv_desc, out_u8) == 276,
              "pnp_conv_desc layout is part of the ABI (mirrored by pnpvcve_b200/_lib.py: ConvDesc)");
int pnp_abi_version(void) { return 10; }

const char* pnp_last_error(void) { return g_err; }

int pnp_device_check(void) {
  DeviceInfo* d;
  return device_info(&d);
}

int pnp_device_pairs(void) {
  DeviceInfo* d;
  int rc = device_info(&d);
  return rc ? rc : d->max_pairs;
}

int pnp_set_pair_mode(int mode) {
  const int prev = g_pair_override;
  g_pair_override = mode < 0 ? -1 : (mode > 2 ? 2 : mode);
  return prev;
}

int pnp_graph_begin(void* stream) {
  DeviceInfo* d;
  int rc = device_info(&d);
  if (rc) return rc;
  // relaxed: unrelated CUDA calls of other threads (allocator, copies on other streams) do not invalidate the capture
  cudaError_t e = cudaStreamBeginCapture(static_cast<cudaStream_t>(stream), cudaStreamCaptureModeRelaxed);
  return e == cudaSuccess ? PNP_OK : cuda_fail(e, "pnp_graph_begin");
}

int pnp_graph_end(void* stream, void** graph_exec) {
  if (!graph_exec) return fail(PNP_ERR_ARG, "pnp_graph_end: null output");
  *graph_exec = nullptr;
  cudaGraph_t g = nullptr;
  cudaError_t e = cudaStreamEndCapture(static_cast<cudaStream_t>(stream), &g);
  if (e != cudaSuccess || g == nullptr) {
    if (g) cudaGraphDestroy(g);
    return cuda_fail(e != cudaSuccess ? e : cudaErrorUnknown, "pnp_graph_end: capture");
  }
  cudaGraphExec_t x = nullptr;
  e = cudaGraphInstantiate(&x, g, 0);
  cudaGraphDestroy(g);
  if (e != cudaSuccess) return cuda_fail(e, "pnp_graph_end: instantiate");
  *graph_exec = x;
  return PNP_OK;
}

int pnp_graph_launch(void* graph_exec, int32_t* step_word, int32_t step_value, void* stream) {
  if (!graph_exec) return fail(PNP_ERR_ARG, "pnp_graph_launch: null graph");
  if (step_word) {
    int rc = store_step(step_word, step_value, static_cast<cudaStream_t>(stream));
    if (rc) return rc;
  }
  cudaError_t e = cudaGraphLaunch(static_cast<cudaGraphExec_t>(graph_exec), static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? PNP_OK : cuda_fail(e, "pnp_graph_launch");
}

int pnp_graph_destroy(void* graph_exec) {
  if (!graph_exec) return PNP_OK;
  cudaError_t e = cudaGraphExecDestroy(static_cast<cudaGraphExec_t>(graph_exec));
  return e == cudaSuccess ? PNP_OK : cuda_fail(e, "pnp_graph_destroy");
}

int pnp_set_step(int32_t* step_word, int32_t step_value, void* stream) {
  if (!step_word) return fail(PNP_ERR_ARG, "pnp_set_step: null step word");
  return store_step(step_word, step_value, static_cast<cudaStream_t>(stream));
}

int pnp_fetch_pinned(void* dst, const void* src_pinned, int64_t bytes, void* stream) {
  if (!dst || !src_pinned) return fail(PNP_ERR_ARG, "pnp_fetch_pinned: null pointer");
  if (bytes < 0 || (bytes & 15) || !aligned16(dst) || !aligned16(src_pinned))
    return fail(PNP_ERR_ARG, "pnp_fetch_pinned: size and pointers must be multiples of 16 bytes");
  DeviceInfo* d;
  int rc = device_info(&d);
  if (rc) return rc;
  cudaPointerAttributes at;
  cudaError_t e = cudaPointerGetAttributes(&at, src_pinned);
  if (e != cudaSuccess) return cuda_fail(e, "pnp_fetch_pinned");
  if (at.type != cudaMemoryTypeHost || at.devicePointer == nullptr)
    return fail(PNP_ERR_ARG, "pnp_fetch_pinned: src must be page-locked host memory the device can address");
  e = pnp::launch_fetch_pinned(at.devicePointer, dst, bytes, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? PNP_OK : cuda_fail(e, "pnp_fetch_pinned");
}

int pnp_mv_warp(const void* src, const float* flow_x, const float* flow_y, int64_t flow_row_stride,
                int64_t flow_image_stride, void* dst, int N, int H, int W, int32_t* dbg_x0, int32_t* dbg_y0,
                void* stream) {
  if (!src || !flow_x || !flow_y || !dst) return fail(PNP_ERR_ARG, "pnp_mv_warp: null pointer");
  if (N <= 0 || H < 10 || W < 10) return fail(PNP_ERR_ARG, "pnp_mv_warp: bad shape (images of at least 10 x 10 pixels)");
  if (!aligned16(src) || !aligned16(dst) || src == dst)
    return fail(PNP_ERR_ARG, "pnp_mv_warp: src/dst must be distinct 16-byte aligned buffers");
  if ((dbg_x0 == nullptr) != (dbg_y0 == nullptr) || (dbg_x0 && N != 1))
    return fail(PNP_ERR_ARG, "pnp_mv_warp: dbg outputs come in pairs and need N == 1");
  DeviceInfo* d;
  int rc = device_info(&d);
  if (rc) return rc;
  CUtensorMap tm, tmd;
  if ((rc = make_map(&tm, src, N, H, W, 10, 0, 0, 0, 10))) return rc;
  if ((rc = make_map(&tmd, dst, N, H, W, 8, 0, 0, 0, 8))) return rc;
  cudaError_t e = pnp::launch_mv_warp(tm, tmd, src, flow_x, flow_y, flow_row_stride, flow_image_stride, dst, N, H, W, dbg_x0,
                                      dbg_y0, dyn_ref(nullptr), nullptr, knobs().warp_tma, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? PNP_OK : cuda_fail(e, "pnp_mv_warp");
}

int pnp_mv_warp_dyn(const pnp_dyn_ref* dyn, const void* src_pool, int src_pool_images, int64_t flow_row_stride,
                    int64_t flow_image_stride, int N, int H, int W, void* stream) {
  if (!dyn || !dyn->table || !dyn->step) return fail(PNP_ERR_ARG, "pnp_mv_warp_dyn: null launch table");
  if (N <= 0 || H < 10 || W < 10) return fail(PNP_ERR_ARG, "pnp_mv_warp_dyn: bad shape (images of at least 10 x 10 pixels)");
  if (!src_pool || src_pool_images < N || !aligned16(src_pool))
    return fail(PNP_ERR_ARG, "pnp_mv_warp_dyn: src_pool must be the 16-byte aligned buffer every table entry's src lies in");
  DeviceInfo* d;
  int rc = device_info(&d);
  if (rc) return rc;
  CUtensorMap tm, tmd;
  if ((rc = make_map(&tm, src_pool, src_pool_images, H, W, 10, 0, 0, 0, 10))) return rc;
  if ((rc = make_map(&tmd, src_pool, src_pool_images, H, W, 8, 0, 0, 0, 8))) return rc;
  cudaError_t e = pnp::launch_mv_warp(tm, tmd, nullptr, nullptr, nullptr, flow_row_stride, flow_image_stride, nullptr, N, H, W,
                                      nullptr, nullptr, dyn_ref(dyn), src_pool, knobs().warp_tma,
                                      static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? PNP_OK : cuda_fail(e, "pnp_mv_warp_dyn");
}

int pnp_lr_im2col(const float* lr, int64_t sn, int64_t sc, int64_t sy, void* dst, int N, int H, int W,
                  int dst_channels, void* stream) {
  if (!lr || !dst) return fail(PNP_ERR_ARG, "pnp_lr_im2col: null pointer");
  if (N <= 0 || H <= 0 || W <= 0 || !aligned16(dst) || (dst_channels != 64 && dst_channels != 32))
    return fail(PNP_ERR_ARG, "pnp_lr_im2col: bad argument (dst_channels is 64 or 32)");
  DeviceInfo* d;
  int rc = device_info(&d);
  if (rc) return rc;
  cudaError_t e = pnp::launch_lr_im2col(lr, sn, sc, sy, dst, N, H, W, dst_channels, dyn_ref(nullptr),
                                        static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? PNP_OK : cuda_fail(e, "pnp_lr_im2col");
}

int pnp_lr_im2col_dyn(const pnp_dyn_ref* dyn, int64_t sn, int64_t sc, int64_t sy, int N, int H, int W, int dst_channels,
                      void* stream) {
  if (!dyn || !dyn->table || !dyn->step) return fail(PNP_ERR_ARG, "pnp_lr_im2col_dyn: null launch table");
  if (N <= 0 || H <= 0 || W <= 0 || (dst_channels != 64 && dst_channels != 32))
    return fail(PNP_ERR_ARG, "pnp_lr_im2col_dyn: bad shape (dst_channels is 64 or 32)");
  DeviceInfo* d;
  int rc = device_info(&d);
  if (rc) return rc;
  cudaError_t e = pnp::launch_lr_im2col(nullptr, sn, sc, sy, nullptr, N, H, W, dst_channels, dyn_ref(dyn),
                                        static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? PNP_OK : cuda_fail(e, "pnp_lr_im2col_dyn");
}

int pnp_pack_conv3x3_rowstack(const float* w, int n_experts, const float* coef, const float* row_scale,
                              int out_ch, int in_total, int in_begin, int in_begin2, int in_count, void* dst,
                              int tap_n, int flip_ky, void* stream) {
  if (!w || !dst) return fail(PNP_ERR_ARG, "pnp_pack_conv3x3_rowstack: null pointer");
  if (n_experts < 1 || (coef == nullptr && n_experts != 1) || out_ch < 1 || (tap_n != 64 && tap_n != 16) ||
      out_ch > tap_n || in_count < 1 || in_count > 64 || in_begin < 0 || in_begin + in_count > in_total ||
      (in_begin2 >= 0 && in_begin2 + in_count > in_total) || !aligned16(dst))
    return fail(PNP_ERR_ARG, "pnp_pack_conv3x3_rowstack: bad argument");
  DeviceInfo* d;
  int rc = device_info(&d);
  if (rc) return rc;
  cudaError_t e = pnp::launch_pack_conv3x3_rowstack(w, n_experts, coef, row_scale, out_ch, in_total, in_begin, in_begin2,
                                                    in_count, dst, tap_n, flip_ky != 0, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? PNP_OK : cuda_fail(e, "pnp_pack_conv3x3_rowstack");
}

int pnp_pack_rows(const float* w, int rows, int cols, int64_t row_stride, int64_t col_stride, void* dst,
                  int row_offset, void* stream) {
  if (!w || !dst) return fail(PNP_ERR_ARG, "pnp_pack_rows: null pointer");
  if (rows < 1 || rows > 64 || cols < 1 || cols > 64 || row_offset < 0 || !aligned16(dst))
    return fail(PNP_ERR_ARG, "pnp_pack_rows: bad argument");
  DeviceInfo* d;
  int rc = device_info(&d);
  if (rc) return rc;
  cudaError_t e = pnp::launch_pack_rows(w, rows, cols, row_stride, col_stride, dst, row_offset,
                                        static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? PNP_OK : cuda_fail(e, "pnp_pack_rows");
}

int pnp_pack_aux(const float* w, int out_ch, int in_total, void* dst, void* stream) {
  if (!w || !dst) return fail(PNP_ERR_ARG, "pnp_pack_aux: null pointer");
  if (out_ch < 1 || out_ch > 64 || in_total < 3 || !aligned16(dst))
    return fail(PNP_ERR_ARG, "pnp_pack_aux: bad argument");
  DeviceInfo* d;
  int rc = device_info(&d);
  if (rc) return rc;
  cudaError_t e = pnp::launch_pack_aux(w, out_ch, in_total, dst, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? PNP_OK : cuda_fail(e, "pnp_pack_aux");
}

int pnp_pack_mix_blocks(const float* w2, const float* w1x1, int n_blocks, int n_experts, const float* coef,
                        const float* row_scale, void* dst, int64_t dst_block_stride, void* stream) {
  if (!w2 || !w1x1 || !coef || !row_scale || !dst) return fail(PNP_ERR_ARG, "pnp_pack_mix_blocks: null pointer");
  if (n_blocks < 1 || n_blocks > 65535 || n_experts < 1 || dst_block_stride < 12 * 8192 || (dst_block_stride & 15) ||
      !aligned16(dst))
    return fail(PNP_ERR_ARG, "pnp_pack_mix_blocks: bad argument");
  DeviceInfo* d;
  int rc = device_info(&d);
  if (rc) return rc;
  cudaError_t e = pnp::launch_pack_mix_blocks(w2, w1x1, n_blocks, n_experts, coef, row_scale, dst, dst_block_stride,
                                              static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? PNP_OK : cuda_fail(e, "pnp_pack_mix_blocks");
}

int pnp_caa_heads(const float* base_qp, const float* qp, int frames, const float* base0_w,
                  const float* base0_b, const float* base2_w, const float* base2_b, const float* se0_w,
                  const float* se2_w, int n_experts, int se_hidden, float* experts, float* gamma,
                  void* stream) {
  if (!base_qp || !qp || !base0_w || !base0_b || !base2_w || !base2_b || !se0_w || !se2_w || !experts || !gamma)
    return fail(PNP_ERR_ARG, "pnp_caa_heads: null pointer");
  if (frames < 1 || n_experts < 1 || n_experts > 16 || se_hidden < 1 || se_hidden > 64)
    return fail(PNP_ERR_ARG, "pnp_caa_heads: bad argument");
  DeviceInfo* d;
  int rc = device_info(&d);
  if (rc) return rc;
  cudaError_t e = pnp::launch_caa_heads(base_qp, qp, frames, base0_w, base0_b, base2_w, base2_b, se0_w, se2_w,
                                        n_experts, se_hidden, experts, gamma, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? PNP_OK : cuda_fail(e, "pnp_caa_heads");
}

int pnp_mix_bias(const float* conv2_bias, int n_blocks, int n_experts, const float* experts,
                 const float* gamma, int frames, float* out, void* stream) {
  if (!conv2_bias || !experts || !gamma || !out) return fail(PNP_ERR_ARG, "pnp_mix_bias: null pointer");
  if (n_blocks < 1 || n_blocks > 65535 || n_experts < 1 || frames < 1)
    return fail(PNP_ERR_ARG, "pnp_mix_bias: bad argument");
  DeviceInfo* d;
  int rc = device_info(&d);
  if (rc) return rc;
  cudaError_t e = pnp::launch_mix_bias(conv2_bias, (long long)n_experts * 64, n_blocks, n_experts, experts, gamma,
                                       frames, out, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? PNP_OK : cuda_fail(e, "pnp_mix_bias");
}

int pnp_mv_rasterize(const float* records, const int32_t* frame_offsets, const int32_t* is_b,
                     const int32_t* p_target, int T, int R, int H, int W, uint32_t* owner_fwd,
                     uint32_t* owner_bwd, uint32_t* part_mask, float* mvs, float* partitions,
                     int32_t* status, void* stream) {
  if (!frame_offsets || !is_b || !p_target || !owner_fwd || !owner_bwd || !part_mask || !mvs || !partitions ||
      !status || (R > 0 && !records))
    return fail(PNP_ERR_ARG, "pnp_mv_rasterize: null pointer");
  if (T < 1 || T > 65535 || R < 0 || H < 1 || H > 65535 || W < 1 || (long long)T * H * W >= (1LL << 31))
    return fail(PNP_ERR_ARG, "pnp_mv_rasterize: bad shape");
  DeviceInfo* d;
  int rc = device_info(&d);
  if (rc) return rc;
  cudaError_t e = pnp::launch_mv_rasterize(records, frame_offsets, is_b, p_target, T, 0, false, R, H, W, owner_fwd,
                                           owner_bwd, part_mask, mvs, partitions, status,
                                           static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? PNP_OK : cuda_fail(e, "pnp_mv_rasterize");
}

int pnp_mv_rasterize_window(const float* records, const int32_t* frame_offsets, const int32_t* is_b,
                            const int32_t* p_target, int T, int tail, int R, int H, int W, uint32_t* owner_fwd,
                            uint32_t* owner_bwd, uint32_t* part_mask, float* mvs, float* partitions,
                            int32_t* status, void* stream) {
  if (!frame_offsets || !is_b || !p_target || !owner_fwd || !owner_bwd || !part_mask || !mvs || !partitions ||
      !status || (R > 0 && !records))
    return fail(PNP_ERR_ARG, "pnp_mv_rasterize_window: null pointer");
  if (T < 1 || T > 65535 || (tail != 0 && tail != 1) || R < 0 || H < 1 || H > 65535 || W < 1 ||
      (long long)T * H * W >= (1LL << 31))
    return fail(PNP_ERR_ARG, "pnp_mv_rasterize_window: bad shape");
  DeviceInfo* d;
  int rc = device_info(&d);
  if (rc) return rc;
  cudaError_t e = pnp::launch_mv_rasterize(records, frame_offsets, is_b, p_target, T, tail, true, R, H, W, owner_fwd,
                                           owner_bwd, part_mask, mvs, partitions, status,
                                           static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? PNP_OK : cuda_fail(e, "pnp_mv_rasterize_window");
}

int pnp_frame_quality(const float* a, int64_t a_sf, int64_t a_sc, int64_t a_sy, const float* b, int64_t b_sf,
                      int64_t b_sc, int64_t b_sy, int F, int H, int W, int crop_border, unsigned long long* sse,
                      double* ssim_sum, void* stream) {
  return frame_quality("pnp_frame_quality", a, false, a_sf, a_sc, a_sy, b, false, b_sf, b_sc, b_sy, F, H, W, crop_border,
                       sse, ssim_sum, stream);
}

int pnp_frame_quality_u8(const void* a, int a_is_u8, int64_t a_sf, int64_t a_sc, int64_t a_sy, const void* b,
                         int b_is_u8, int64_t b_sf, int64_t b_sc, int64_t b_sy, int F, int H, int W, int crop_border,
                         unsigned long long* sse, double* ssim_sum, void* stream) {
  return frame_quality("pnp_frame_quality_u8", a, a_is_u8 != 0, a_sf, a_sc, a_sy, b, b_is_u8 != 0, b_sf, b_sc, b_sy, F,
                       H, W, crop_border, sse, ssim_sum, stream);
}

int pnp_unit_from_u8(const uint8_t* src, int64_t s_sf, int64_t s_sc, int64_t s_sy, float* dst, int64_t d_sf,
                     int64_t d_sc, int64_t d_sy, int F, int H, int W, void* stream) {
  if (!src || !dst) return fail(PNP_ERR_ARG, "pnp_unit_from_u8: null pointer");
  if (F < 1 || F > 65535 || H < 1 || H > 21845 || W < 1)
    return fail(PNP_ERR_ARG, "pnp_unit_from_u8: bad shape (1 <= F <= 65535, 1 <= H <= 21845)");
  DeviceInfo* d;
  int rc = device_info(&d);
  if (rc) return rc;
  cudaError_t e = pnp::launch_unit_from_u8(src, s_sf, s_sc, s_sy, dst, d_sf, d_sc, d_sy, F, H, W,
                                           static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? PNP_OK : cuda_fail(e, "pnp_unit_from_u8");
}

int pnp_conv3x3(const pnp_conv_desc* c, void* stream) {
  if (!c) return fail(PNP_ERR_ARG, "pnp_conv3x3: null descriptor");
  const bool table = c->dyn.table != nullptr;
  if (!c->src || (!table && !c->wpack)) return fail(PNP_ERR_ARG, "pnp_conv3x3: null src/wpack");
  if (table && (!c->dyn.step || c->dyn.node < 0 || c->dyn.stride <= c->dyn.node))
    return fail(PNP_ERR_ARG, "pnp_conv3x3: bad launch-table reference");
  // (H >= 8: the bound on commits in flight per accumulator ring, pnp_conv_rows.cu kStepRing, assumes it)
  if (c->N < 1 || c->H < 8 || c->W < 1) return fail(PNP_ERR_ARG, "pnp_conv3x3: bad shape (at least 8 rows)");
  const bool last = (c->mode == PNP_CONV_LAST);
  if (c->mode != PNP_CONV_BF16 && !last) return fail(PNP_ERR_ARG, "pnp_conv3x3: bad mode");
  const bool par = c->par != nullptr;
  if (last) {
    if (!c->lq || !c->outf || c->tap_n != 16 || c->aux || c->idt || par)
      return fail(PNP_ERR_ARG, "pnp_conv3x3: PNP_CONV_LAST needs lq/outf, tap_n=16, no aux/idt/par");
  } else {
    if (!c->out || c->tap_n != 64) return fail(PNP_ERR_ARG, "pnp_conv3x3: PNP_CONV_BF16 needs out and tap_n=64");
    if (c->out == c->src && !table) return fail(PNP_ERR_ARG, "pnp_conv3x3: out must not alias src (halo rows)");
  }
  if ((c->aux != nullptr) != (c->aux_k16 > 0) || c->aux_k16 < 0 || c->aux_k16 > 4)
    return fail(PNP_ERR_ARG, "pnp_conv3x3: aux / aux_k16 mismatch");
  const bool aux32 = c->aux && c->aux_channels == 32;
  if (c->aux && c->aux_channels != 0 && c->aux_channels != 64 && !aux32)
    return fail(PNP_ERR_ARG, "pnp_conv3x3: aux_channels is 64 (or 0) or 32");
  if (aux32 && c->aux_k16 > 2) return fail(PNP_ERR_ARG, "pnp_conv3x3: a 32-channel aux source carries K <= 32");
  if (par && (c->aux || c->idt)) return fail(PNP_ERR_ARG, "pnp_conv3x3: par takes no aux / idt");
  if (c->act < 0 || c->act > 2) return fail(PNP_ERR_ARG, "pnp_conv3x3: bad act");
  const bool strided_out = c->out_spx != 0 || c->out_sy != 0 || c->out_sn != 0;
  if (strided_out && (last || c->out_spx < 64 || c->out_sy < c->out_spx * c->W || (c->N > 1 && c->out_sn < c->out_sy * c->H) ||
                      ((c->out_spx | c->out_sy | c->out_sn) & 7)))
    return fail(PNP_ERR_ARG, "pnp_conv3x3: out strides must be non-overlapping multiples of 8 elements (PNP_CONV_BF16 only)");
  if (c->out_u8 && !last) return fail(PNP_ERR_ARG, "pnp_conv3x3: out_u8 needs PNP_CONV_LAST");
  if (c->lq_up4 && (!last || (c->H & 3) || (c->W & 3)))
    return fail(PNP_ERR_ARG, "pnp_conv3x3: lq_up4 needs PNP_CONV_LAST and H, W multiples of 4");
  if (!aligned16(c->src) || (c->wpack && !aligned16(c->wpack)) || (c->aux && !aligned16(c->aux)) ||
      (c->idt && !aligned16(c->idt)) || (c->out && !aligned16(c->out)))
    return fail(PNP_ERR_ARG, "pnp_conv3x3: pointers must be 16-byte aligned");
  if (c->src_images < 0 || c->aux_images < 0 || c->idt_images < 0 || c->out_images < 0)
    return fail(PNP_ERR_ARG, "pnp_conv3x3: negative image count");
  DeviceInfo* d;
  int rc = device_info(&d);
  if (rc) return rc;
  if (c->per_image && (c->N > d->sms || (!table && !c->img_off)))
    return fail(PNP_ERR_ARG, "pnp_conv3x3: per_image needs img_off and at most one image per SM");

  const Knobs& kn = knobs();
  pnp::ConvParams p;
  memset(&p, 0, sizeof(p));
  auto images = [&](int32_t n) { return n > 0 ? n : c->N; };
  if ((rc = make_map(&p.tm_src, c->src, images(c->src_images), c->H, c->W, pnp::kHaloPx))) return rc;
  if (c->aux && (rc = make_map(&p.tm_aux, c->aux, images(c->aux_images), c->H, c->W, pnp::kTilePx, 0, 0, 0, 1,
                               aux32 ? 32 : 64)))
    return rc;
  if (c->idt && (rc = make_map(&p.tm_id, c->idt, images(c->idt_images), c->H, c->W, pnp::kTilePx))) return rc;
  if (!last && (rc = make_map(&p.tm_out, c->out, images(c->out_images), c->H, c->W, pnp::kTilePx, c->out_spx, c->out_sy,
                              c->out_sn)))
    return rc;
  if (last) p.tm_out = p.tm_src;  // never used; keeps the prefetch harmless
  p.dyn = dyn_ref(&c->dyn);
  p.wpack = c->wpack;
  p.scale = c->scale;
  p.bias = c->bias;
  p.has_bias = c->bias != nullptr;
  p.img_off = c->per_image ? reinterpret_cast<const long long*>(c->img_off) : nullptr;
  p.par = c->par;
  p.has_par = par ? 1 : 0;
  p.par_sn = c->par_sn; p.par_sc = c->par_sc; p.par_sy = c->par_sy;
  p.lq = c->lq;
  p.lq_sn = c->lq_sn; p.lq_sc = c->lq_sc; p.lq_sy = c->lq_sy;
  p.outf = c->outf;
  p.of_sn = c->of_sn; p.of_sc = c->of_sc; p.of_sy = c->of_sy;
  p.out_u8 = c->out_u8 ? 1 : 0;
  p.H = c->H; p.W = c->W; p.N = c->N;
  p.strips = (c->W + pnp::kTilePx - 1) / pnp::kTilePx;
  const long long tiles = (long long)c->N * p.strips * c->H;
  if (tiles > 0x7fffffffLL) return fail(PNP_ERR_ARG, "pnp_conv3x3: too many tiles");
  p.tiles_total = (int)tiles;
  // CTA-pair form (cluster of 2, tcgen05 cta_group::2, see pnp_conv_rows.cu): the two CTAs of a pair walk the same rows
  // of two adjacent (image, strip) columns, so columns are paired up; an odd column count leaves one phantom column
  // (taken only when that wastes < 7 %), and with per-image weights both columns of a pair must belong to one image.
  const long long cols = (long long)c->N * p.strips;
  const int pair_mode = g_pair_override >= 0 ? g_pair_override : kn.pair;
  // (a 32-channel aux source is wired for the single-CTA form only: both forms compute identical values)
  const bool pair_ok = pair_mode != 0 && !last && !aux32 && c->tap_n == 64 && d->max_pairs >= 8 && (!par || kn.par_split) &&
                       (c->per_image ? (p.strips % 2 == 0 && c->N <= d->max_pairs)
                                     : (cols % 2 == 0 || cols >= 15 || pair_mode == 2));
  int grid;
  if (pair_ok) {
    p.pair = 1;
    const int max_pairs = d->max_pairs < d->sms / 2 ? d->max_pairs : d->sms / 2;
    if (c->per_image) {
      const int tiles_img = (p.strips / 2) * c->H;
      int cpi = max_pairs / c->N;
      if (cpi > tiles_img) cpi = tiles_img;
      p.tiles_per_cta = (tiles_img + cpi - 1) / cpi;
      cpi = (tiles_img + p.tiles_per_cta - 1) / p.tiles_per_cta;
      p.cpi = cpi;
      p.tiles_total = tiles_img * c->N;
      grid = 2 * cpi * c->N;
    } else {
      const long long pair_tiles = ((cols + 1) / 2) * c->H;
      p.tiles_total = (int)pair_tiles;
      int clusters = max_pairs < pair_tiles ? max_pairs : (int)pair_tiles;
      p.tiles_per_cta = (p.tiles_total + clusters - 1) / clusters;
      clusters = (p.tiles_total + p.tiles_per_cta - 1) / p.tiles_per_cta;
      grid = 2 * clusters;
    }
  } else if (c->per_image) {
    // CTAs are partitioned by image so that each can hold its image's weights: cpi CTAs walk one image
    const int tiles_img = p.strips * c->H;
    int cpi = d->sms / c->N;
    if (cpi > tiles_img) cpi = tiles_img;
    p.tiles_per_cta = (tiles_img + cpi - 1) / cpi;
    cpi = (tiles_img + p.tiles_per_cta - 1) / p.tiles_per_cta;
    p.cpi = cpi;
    grid = cpi * c->N;
  } else {
    grid = d->sms < p.tiles_total ? d->sms : p.tiles_total;
    p.tiles_per_cta = (p.tiles_total + grid - 1) / grid;
    grid = (p.tiles_total + p.tiles_per_cta - 1) / p.tiles_per_cta;
  }
  p.tap_n = c->tap_n;
  p.aux_k16 = c->aux_k16;
  p.aux_pitch64 = aux32 ? 1 : 0;
  p.has_id = c->idt != nullptr;
  p.act = c->act;
  p.mode = last ? pnp::kModeLast : pnp::kModeBf16;
  p.flip_y = c->flip_y ? 1 : 0;
  p.w_stable = c->wpack_stable ? 1 : 0;
  p.lq_up4 = c->lq_up4 ? 1 : 0;
  p.par_sparse = (par && c->par_sparse) ? 1 : 0;
  // block launch B (identity, bottom-up) reads t and x for the last time
  if (kn.l2_hints && c->idt && c->flip_y) {            // launch B
    p.l2_src = p.l2_idt = 1;
    if (kn.l2_hints >= 2) p.l2_out = 2;
  } else if (kn.l2_hints >= 2 && par) {                // launch A
    p.l2_src = kn.l2_hints == 2 ? 2 : 1;
    p.l2_out = kn.l2_hints == 2 ? 1 : 2;
  }
  p.par_split = (par && kn.par_split) ? 1 : 0;
  p.debug_skip = kn.debug_skip;
  p.trace = kn.trace;
  // shared-memory budget: weights + (aux ring) + staging ring + source-row ring from what is left.
  // With an identity operand the staging ring also prefetches identity tiles (n_io - 2 tiles ahead),
  // so it gets 4 slots as long as 5 source rows (3 in use + 2 in flight) still fit.
  const long long budget = 232448 - 2048;
  // (pair mode: a CTA holds half of the aux / 1x1 block, and the 3x3 weights as two half-sized layouts)
  const long long w_bytes = ((long long)9 * c->tap_n * 128 + (c->aux ? pnp::kWChunkBytes : 0) / (p.pair ? 2 : 1) +
                             (par ? 3 * 64 * 128 : 0) / (p.pair ? 2 : 1) + 1023) & ~1023LL;
  auto fixed_bytes = [&](int n_io) {
    return w_bytes + (c->aux ? 2 * pnp::kTileBytes : 0) + (long long)n_io * pnp::kTileBytes;
  };
  p.n_io = 2;
  if (par) p.n_io = 3;   // the next row's 1x1 blend is parked in its staging slot one row early
  if (c->idt) {
    p.n_io = 4;
    while (p.n_io > 2 && (budget - fixed_bytes(p.n_io)) / pnp::kASlotBytes < 5) --p.n_io;
  }
  long long slots = (budget - fixed_bytes(p.n_io)) / pnp::kASlotBytes;
  const long long max_slots = 6;   // a row lives one step there: 6 = 5 in flight
  if (slots > max_slots) slots = max_slots;
  if (slots < 4) return fail(PNP_ERR_RESOURCE, "pnp_conv3x3: shared-memory budget cannot hold 4 source rows");
  // the MMA thread checks the next step's barriers before the current step is committed; with an identity operand
  // that needs a staging ring of >= 3 slots to stay deadlock free
  if (c->idt && p.n_io < 3)
    return fail(PNP_ERR_RESOURCE, "pnp_conv3x3: idt needs 3 staging slots (drop aux)");
  p.s_a = (int)slots;
  if (kn.rings_nio >= 2 && kn.rings_nio <= pnp::kMaxIoSlots && kn.rings_sa >= 3 && kn.rings_sa <= pnp::kMaxASlots &&
      fixed_bytes(kn.rings_nio) + (long long)kn.rings_sa * pnp::kASlotBytes <= budget && !(c->idt && kn.rings_nio < 3) &&
      !(par && kn.rings_nio < 3)) {
    p.n_io = kn.rings_nio;
    p.s_a = kn.rings_sa;
  }
  cudaError_t e = pnp::launch_conv_rows(p, grid, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? PNP_OK : cuda_fail(e, "pnp_conv3x3");
}

}  // extern "C"
