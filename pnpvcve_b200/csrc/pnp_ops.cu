// Memory-bound kernels of the BAE path: MV-guided warp (K1), LR im2col packing, weight packing with
// expert mixing (K4) and the CAA heads.
#include <cstdlib>

#include "pnp_conv.cuh"
#include "pnp_ops.cuh"
#include "pnp_ptx.cuh"

namespace pnp {

// =====================================================================================
// K1: motion-vector guided bilinear warp.
// Reference: flow_warp (mmedit/models/common/flow_warp.py:6-50) called by VOSAlignment.forward
// (mmedit/models/backbones/sr_backbones/iconvsr_mv.py:17-18) -> F.grid_sample(bilinear, zeros,
// align_corners=True).  The reference normalises x+mv to [-1,1] and ATen un-normalises it again;
// that fp32 round trip is not the identity, so the exact operation sequence is replayed with
// explicitly rounded intrinsics (no FMA contraction) to keep the integer taps bit-exact.
//
// One thread = one pixel x 16 channels (32 bytes): 4 consecutive threads read one 128-byte NHWC
// pixel per tap, a warp writes 1 KB contiguous.
// =====================================================================================
__device__ __forceinline__ float warp_coord(float pos, float mv, float size_m1_div, float size_m1) {
  const float g = __fadd_rn(pos, mv);                                  // grid + flow
  const float nrm = __fsub_rn(__fdiv_rn(__fmul_rn(2.0f, g), size_m1_div), 1.0f);  // 2*g/max(s-1,1) - 1
  return __fmul_rn(__fmul_rn(__fadd_rn(nrm, 1.0f), 0.5f), size_m1);    // ((c+1)/2)*(s-1)
}

// Per-pixel part shared by both tap sources: coordinates (exact reference op order), weights, integer taps.
struct WarpTaps {
  int x0, y0;
  float wnw, wne, wsw, wse;
};
__device__ __forceinline__ WarpTaps warp_taps(float fx, float fy, int x, int y, int H, int W, float& x0f, float& y0f) {
  const float ix = warp_coord((float)x, fx, (float)max(W - 1, 1), (float)(W - 1));
  const float iy = warp_coord((float)y, fy, (float)max(H - 1, 1), (float)(H - 1));
  x0f = floorf(ix);
  y0f = floorf(iy);
  const float x1f = __fadd_rn(x0f, 1.0f), y1f = __fadd_rn(y0f, 1.0f);
  const float wx1 = __fsub_rn(ix, x0f), wx0 = __fsub_rn(x1f, ix);
  const float wy1 = __fsub_rn(iy, y0f), wy0 = __fsub_rn(y1f, iy);
  WarpTaps t;
  t.wnw = __fmul_rn(wx0, wy0);
  t.wne = __fmul_rn(wx1, wy0);
  t.wsw = __fmul_rn(wx0, wy1);
  t.wse = __fmul_rn(wx1, wy1);
  // clamp before the int conversion so huge |mv| cannot overflow; out-of-range taps are dropped
  t.x0 = (int)fminf(fmaxf(x0f, -2.0f), (float)W + 1.0f);
  t.y0 = (int)fminf(fmaxf(y0f, -2.0f), (float)H + 1.0f);
  return t;
}

// nw*wnw + ne*wne + sw*wsw + se*wse in fp32 (FMA chain, like ATen's CUDA grid sampler) of 8 bf16 channels.  The two
// channels of a 32-bit word are blended as one packed fp32 pair (FMUL2 / FFMA2 on sm_100: the same IEEE operations per
// element, half the instructions -- the kernel is bound by instruction issue, not by bytes).
__device__ __forceinline__ uint4 warp_blend(const uint4& va, const uint4& vb, const uint4& vc, const uint4& vd,
                                            const WarpTaps& t) {
  const uint32_t a[4] = {va.x, va.y, va.z, va.w}, b[4] = {vb.x, vb.y, vb.z, vb.w};
  const uint32_t c[4] = {vc.x, vc.y, vc.z, vc.w}, d[4] = {vd.x, vd.y, vd.z, vd.w};
  const float2 wnw = make_float2(t.wnw, t.wnw), wne = make_float2(t.wne, t.wne);
  const float2 wsw = make_float2(t.wsw, t.wsw), wse = make_float2(t.wse, t.wse);
  uint32_t r[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float2 acc = __fmul2_rn(make_float2(bf16_lo(a[j]), bf16_hi(a[j])), wnw);
    acc = __ffma2_rn(make_float2(bf16_lo(b[j]), bf16_hi(b[j])), wne, acc);
    acc = __ffma2_rn(make_float2(bf16_lo(c[j]), bf16_hi(c[j])), wsw, acc);
    acc = __ffma2_rn(make_float2(bf16_lo(d[j]), bf16_hi(d[j])), wse, acc);
    r[j] = pack_bf16x2(acc.x, acc.y);
  }
  return make_uint4(r[0], r[1], r[2], r[3]);
}

// History.  v1 spent ~550 SASS instructions per 48 bytes moved (64-bit index divisions, per-tap rounded mul/add chains)
// and was issue-bound at ~45 % of the HBM roofline.  v2: 2-D grid, 32-bit indexing, 4 threads per pixel x 32 bytes,
// FMA blend, 32 x 8 pixel tiles walked two rows at a time so that the tap row shared by vertically adjacent outputs is
// found in L1: 52.9 us at 720p cold (70 % of the measured HBM rate), still issue bound (ncu: DRAM throughput 38 %,
// issue slots 64 % busy, ~1500 warp instructions per 32 pixels): every tap is a predicated, bounds-checked
// 64-bit-addressed global load and the four threads of a pixel all redo its coordinate arithmetic.
//
// v3 (this kernel): TMA tile staging in both directions, one thread per pixel.  The codec's motion vectors are constant
// over blocks of >= 8 x 8 pixels, so an 8 x 8 output block reads a 9 x 9 source window (10 x 10 with the one-pixel slack
// the reference's fp32 normalise / un-normalise round trip can add).  A CTA owns a 32 x 8 pixel tile = four such blocks,
// 64 threads each.  Every thread computes its pixel's exact integer taps and weights ONCE (motion vectors are call
// inputs, so this runs ahead of griddepcontrol.wait), the block's tap bounding box is reduced with redux.sync, and one
// thread per block issues a (64 ch, 10, 10) TMA box load of that window into 128B-swizzled shared memory --
// out-of-image taps arrive as zeros, which IS grid_sample's padding_mode='zeros'.  The taps are then 16-byte
// shared-memory reads without bounds checks or global address arithmetic (a warp reads 32 window rows whose chunks the
// swizzle spreads over all banks), the blended pixel is parked in a swizzled output tile and leaves by a TMA box store
// (clipped at the image edge).  A block whose taps do not fit a 10 x 10 window (arbitrary per-pixel flow) reads its taps
// with global loads instead, so any flow field gives the reference's result.
constexpr int kWarpWin = 10;                             // staged window: kWarpWin x kWarpWin source pixels
constexpr int kWarpWinBytes = kWarpWin * kWarpWin * 128;   // 12800
constexpr int kWarpWinPitch = 13 * 1024;                 // 1024-aligned slot (the swizzle is a function of address bits)
constexpr int kWarpOutBytes = 64 * 128;                  // one 8 x 8 output block
#ifndef PNP_WARP_BLOCKS
#define PNP_WARP_BLOCKS 1
#endif
constexpr int kWarpBlocks = PNP_WARP_BLOCKS;             // 8 x 8 blocks per CTA (tile 8*kWarpBlocks x 8), 64 threads each
constexpr int kWarpSmem = kWarpBlocks * kWarpWinPitch + 1024;     // the output tile re-uses its block's window slot

__global__ void __launch_bounds__(64 * kWarpBlocks, 14 / kWarpBlocks)     // 14 slots of 13 KB + 1 KB per SM
mv_warp_kernel(const __grid_constant__ CUtensorMap tm_src, const __grid_constant__ CUtensorMap tm_dst,
               const uint4* __restrict__ src, const float* __restrict__ flow_x, const float* __restrict__ flow_y,
               long long flow_sy, long long flow_sn, uint4* __restrict__ dst, int H, int W, int* __restrict__ dbg_x0,
               int* __restrict__ dbg_y0, const DynRef dyn, const uint8_t* pool_base, int use_tma) {
  extern __shared__ uint8_t warp_smem_raw[];
  __shared__ uint64_t bar[kWarpBlocks];
  __shared__ int part[kWarpBlocks][2][4];                // per block and warp: min x0, max x0, min y0, max y0 of the valid pixels
  int img_src = 0, img_dst = 0;                          // first image inside the tensor maps
  if (const DynEntry* e = dyn.entry()) {
    // table mode: p{-, flow_x, flow_y, -}, i{src image, -, -, dst image} inside the pool both maps span.  (Image
    // indices, not pointers: turning a pointer into an image index costs every thread two 64-bit divisions -- and this
    // kernel is bound by instruction issue and latency, not by bytes, once the SM clock is power-capped.)
    flow_x = reinterpret_cast<const float*>(e->p[1]);
    flow_y = reinterpret_cast<const float*>(e->p[2]);
    img_src = e->i[0];
    img_dst = e->i[3];
    src = reinterpret_cast<const uint4*>(pool_base + (long long)img_src * H * W * 128);
    dst = reinterpret_cast<uint4*>(const_cast<uint8_t*>(pool_base) + (long long)img_dst * H * W * 128);
  }
  const uint32_t raw = smem_u32(warp_smem_raw);
  const uint32_t sbase = (raw + 1023u) & ~1023u;
  uint8_t* sgen = warp_smem_raw + (sbase - raw);
  const int tid = threadIdx.x;
  const int b = tid >> 6;                                // this thread's 8 x 8 block (two warps per block)
  const int col = tid & 7, row = (tid >> 3) & 7;         // its pixel inside the block
  if (tid < kWarpBlocks) mbar_init(smem_u32(&bar[tid]), 1);
  if (tid == 0) {
    mbar_fence_init();
    tma_prefetch_desc(&tm_src);
    tma_prefetch_desc(&tm_dst);
  }
  griddep_launch_dependents();
  __syncthreads();
  // blockIdx.z = image of the batch: same-shape clips with their own motion fields
  const int n = blockIdx.z;
  flow_x += (long long)n * flow_sn;
  flow_y += (long long)n * flow_sn;
  const int bx = (blockIdx.x * kWarpBlocks + b) * 8, by = blockIdx.y * 8;
  const int x = bx + col, y = by + row;
  const bool valid = x < W && y < H;
  // ---- the pixel's taps and weights (motion vectors are inputs of the call: no dependence on the previous kernel)
  float fx = 0.f, fy = 0.f;
  if (valid) {
    fx = __ldg(flow_x + (long long)y * flow_sy + x);
    fy = __ldg(flow_y + (long long)y * flow_sy + x);
  }
  float x0f, y0f;
  const WarpTaps t = warp_taps(fx, fy, x, y, H, W, x0f, y0f);
  if (dbg_x0 != nullptr && valid) {
    dbg_x0[y * W + x] = (int)fminf(fmaxf(x0f, -2147483000.0f), 2147483000.0f);
    dbg_y0[y * W + x] = (int)fminf(fmaxf(y0f, -2147483000.0f), 2147483000.0f);
  }
  if (use_tma) {
    const int mnx = __reduce_min_sync(0xffffffffu, valid ? t.x0 : 0x7fffffff);
    const int mxx = __reduce_max_sync(0xffffffffu, valid ? t.x0 : -0x7fffffff);
    const int mny = __reduce_min_sync(0xffffffffu, valid ? t.y0 : 0x7fffffff);
    const int mxy = __reduce_max_sync(0xffffffffu, valid ? t.y0 : -0x7fffffff);
    if ((tid & 31) == 0) {                               // two warps per block: plain stores, combined behind the barrier
      int* pw = part[b][(tid >> 5) & 1];
      pw[0] = mnx;
      pw[1] = mxx;
      pw[2] = mny;
      pw[3] = mxy;
    }
  }
  __syncthreads();
  griddep_wait();                                        // the source features come from the previous kernel
  const bool any = bx < W && by < H;                     // the block has pixels inside the image
  int bx0 = 0, by0 = 0;
  bool staged = false;
  if (use_tma && any) {
    bx0 = min(part[b][0][0], part[b][1][0]);
    by0 = min(part[b][0][2], part[b][1][2]);
    const int bx1 = max(part[b][0][1], part[b][1][1]), by1 = max(part[b][0][3], part[b][1][3]);
    staged = bx0 <= bx1 && bx1 + 2 - bx0 <= kWarpWin && by1 + 2 - by0 <= kWarpWin;
  }
  // ---- one thread per block: stage its tap window (taps x0..x0+1, y0..y0+1 of every pixel) if it fits
  if (staged && (tid & 63) == 0) {
    mbar_arrive_expect_tx(smem_u32(&bar[b]), kWarpWinBytes);
    tma_load_4d(sbase + b * kWarpWinPitch, &tm_src, smem_u32(&bar[b]), 0, bx0, by0, img_src + n);
  }
  // the block's output tile (row = pixel index) takes over its window slot once every thread has read its taps
  uint8_t* const ob = sgen + b * kWarpWinPitch;
  const int p = tid & 63;
  uint4 o[8];
  if (staged) {
    mbar_wait(smem_u32(&bar[b]), 0, 20);
    // (pixels outside the image took no part in the bounding box: their taps may lie outside the window, and their
    // outputs are clipped by the store anyway)
    const int r00 = valid ? (t.y0 - by0) * kWarpWin + (t.x0 - bx0) : 0;          // window row of the north-west tap
    // Rows are 128-byte aligned, so "row + swizzled chunk offset" is (row ^ ((row & 7) << 4)) ^ (chunk << 4): one XOR
    // with an immediate per load.  Chunks are walked in LOGICAL order -- at a fixed logical chunk the lanes' physical
    // chunks differ with their rows, which is what keeps the reads free of bank conflicts (walking physical chunks,
    // tried: every lane on the same four banks, 44 -> 99 us).  Offsets are taken from the 1024-aligned base `sgen`.
    auto rowx = [&](int r) { return ((uint32_t)(b * kWarpWinPitch) + (uint32_t)r * 128u) ^ (((uint32_t)r & 7u) << 4); };
    const uint32_t pa = rowx(r00), pb = rowx(r00 + 1), pc = rowx(r00 + kWarpWin), pd = rowx(r00 + kWarpWin + 1);
    auto lds = [&](uint32_t off) { return *reinterpret_cast<const uint4*>(sgen + off); };
#pragma unroll
    for (int c = 0; c < 8; ++c) o[c] = warp_blend(lds(pa ^ (16 * c)), lds(pb ^ (16 * c)), lds(pc ^ (16 * c)), lds(pd ^ (16 * c)), t);
    named_bar_sync(1 + b, 64);                           // every tap of the block has been read
    {
      const uint32_t orow = (uint32_t)(b * kWarpWinPitch) + (((uint32_t)p * 128u) ^ (((uint32_t)p & 7u) << 4));
#pragma unroll
      for (int c = 0; c < 8; ++c) *reinterpret_cast<uint4*>(sgen + (orow ^ (16 * c))) = o[c];
    }
  } else if (any) {
    // Gather path (the block's taps do not fit one window -- e.g. the reversed P-frame vectors the reference scatters
    // at their target positions, loading_ipb.py:352-356, or any per-pixel flow): four lanes per pixel, 32 bytes each,
    // so that a tap is one full 128-byte line per pixel and neighbouring pixels' lines are found in L1 (the v2
    // scheme).  A warp owns 32 pixels and handles 8 of them per round; the owner lane's taps travel by shuffle.
    const uint4* sp = src + (size_t)n * H * W * 8;
    const int lane = tid & 31, q = lane & 3;
    const uint4 z = make_uint4(0, 0, 0, 0);
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int owner = r * 8 + (lane >> 2);
      WarpTaps u;
      u.x0 = __shfl_sync(0xffffffffu, t.x0, owner);
      u.y0 = __shfl_sync(0xffffffffu, t.y0, owner);
      u.wnw = __shfl_sync(0xffffffffu, t.wnw, owner);
      u.wne = __shfl_sync(0xffffffffu, t.wne, owner);
      u.wsw = __shfl_sync(0xffffffffu, t.wsw, owner);
      u.wse = __shfl_sync(0xffffffffu, t.wse, owner);
      const bool uvalid = __shfl_sync(0xffffffffu, (int)valid, owner) != 0;
      const bool okx0 = uvalid && u.x0 >= 0 && u.x0 < W, okx1 = uvalid && u.x0 + 1 >= 0 && u.x0 + 1 < W;
      const bool oky0 = u.y0 >= 0 && u.y0 < H, oky1 = u.y0 + 1 >= 0 && u.y0 + 1 < H;
      const uint4* t00 = sp + ((long long)u.y0 * W + u.x0) * 8 + q * 2;         // pixel = 8 uint4
      const uint4* t10 = t00 + (size_t)W * 8;
      const int pp = (p & 32) + owner;                     // the pixel's row in the output tile
      const uint32_t orow = (uint32_t)(b * kWarpWinPitch) + (((uint32_t)pp * 128u) ^ (((uint32_t)pp & 7u) << 4));
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const uint4 v = warp_blend((okx0 && oky0) ? __ldg(t00 + h) : z, (okx1 && oky0) ? __ldg(t00 + 8 + h) : z,
                                   (okx0 && oky1) ? __ldg(t10 + h) : z, (okx1 && oky1) ? __ldg(t10 + 8 + h) : z, u);
        *reinterpret_cast<uint4*>(sgen + (orow ^ (16 * (2 * q + h)))) = v;
      }
    }
  }
  // ---- the block's output tile leaves by one TMA store (pixels outside the image are clipped)
  fence_proxy_async_smem();
  named_bar_sync(1 + b, 64);
  if (any && p == 0) {
    tma_store_4d(&tm_dst, smem_u32(ob), 0, bx, by, img_dst + n);
    tma_store_commit();
    tma_store_wait_read<0>();             // shared memory must stay valid until the store has read it
  }
}

cudaError_t warp_prepare() {
  return cudaFuncSetAttribute(mv_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kWarpSmem);
}

cudaError_t launch_mv_warp(const CUtensorMap& tm_src, const CUtensorMap& tm_dst, const void* src, const float* flow_x,
                           const float* flow_y, long long flow_sy, long long flow_sn, void* dst, int N, int H, int W,
                           int* dbg_x0, int* dbg_y0, const DynRef& dyn, const void* pool_base, int use_tma,
                           cudaStream_t stream) {
  if ((long long)H * W >= (1LL << 27) || N > 65535) return cudaErrorInvalidValue;   // 32-bit pixel indexing
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((W + 8 * kWarpBlocks - 1) / (8 * kWarpBlocks), (H + 7) / 8, N);
  cfg.blockDim = dim3(64 * kWarpBlocks);
  cfg.dynamicSmemBytes = kWarpSmem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, mv_warp_kernel, tm_src, tm_dst, reinterpret_cast<const uint4*>(src), flow_x, flow_y,
                            flow_sy, flow_sn, reinterpret_cast<uint4*>(dst), H, W, dbg_x0, dbg_y0, dyn,
                            reinterpret_cast<const uint8_t*>(pool_base), use_tma);
}

// =====================================================================================
// LR frame -> im2col'd bf16 NHWC "aux" operand: channel k = tap*3 + c (27 used, 5 zero pad, the
// upper 32 channels of the 64-channel row are never read).  The 3-channel part of the reference's
// 131/195-channel input conv (basicvsr_net.py:484 on cat([lr, ...]), iconvsr_ipb_par.py:90,125)
// becomes a K=32 centre-tap GEMM.
// =====================================================================================
// One block = a 64 x 4 pixel tile: the 3 x 6 x 66 source window is staged in shared memory with coalesced loads.
constexpr int kI2cW = 64, kI2cH = 4;
__global__ void __launch_bounds__(256)
lr_im2col_kernel(const float* __restrict__ lr, long long sn, long long sc, long long sy, uint4* __restrict__ dst,
                 int N, int H, int W, int px16, const DynRef dyn) {   // px16: 16-byte chunks per destination pixel (8 | 4)
  __shared__ float win[3][kI2cH + 2][kI2cW + 2];
  if (const DynEntry* e = dyn.entry()) {                  // table mode: p{lr, dst}
    lr = reinterpret_cast<const float*>(e->p[0]);
    dst = reinterpret_cast<uint4*>(e->p[1]);
  }
  const int n = blockIdx.z;
  const int x0 = blockIdx.x * kI2cW, y0 = blockIdx.y * kI2cH;
  const float* base = lr + (long long)n * sn;
  for (int i = threadIdx.x; i < 3 * (kI2cH + 2) * (kI2cW + 2); i += 256) {
    const int c = i / ((kI2cH + 2) * (kI2cW + 2));
    const int r = i % ((kI2cH + 2) * (kI2cW + 2));
    const int wy = r / (kI2cW + 2), wx = r % (kI2cW + 2);
    const int yy = y0 + wy - 1, xx = x0 + wx - 1;
    const bool ok = yy >= 0 && yy < H && xx >= 0 && xx < W;
    win[c][wy][wx] = ok ? __ldg(base + (long long)c * sc + (long long)yy * sy + xx) : 0.f;   // zero = conv padding
  }
  __syncthreads();
  // Each thread builds its pixel's 27-entry operand (static indexing) and parks the 64 used bytes in shared memory;
  // the tile then leaves as 16-byte chunks with a quad of lanes per pixel (two full 32-byte sectors per pixel and
  // store instruction).  Measured (tools/im2col_bench.py, 720p, cold): 27.4 us with 27 scalar global loads and
  // per-thread stores, 28.9 with the staged window only, 26.7 like this -- with 128-byte destination pixels the kernel
  // is bound by writing HALF of every 128-byte line (59 MB useful at the DRAM cost of 118 MB); with 64-byte pixels
  // (dst_channels = 32, the conv kernels' SWIZZLE_64B aux path) the stores are contiguous.
  __shared__ uint4 otile[kI2cW * kI2cH][4];
  {
    const int tx = threadIdx.x % kI2cW, ty = threadIdx.x / kI2cW;
    float v[32];
#pragma unroll
    for (int tap = 0; tap < 9; ++tap)
#pragma unroll
      for (int c = 0; c < 3; ++c) v[tap * 3 + c] = win[c][ty + tap / 3][tx + tap % 3];
#pragma unroll
    for (int k = 27; k < 32; ++k) v[k] = 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q)
      otile[threadIdx.x][q] = make_uint4(pack_bf16x2(v[8 * q], v[8 * q + 1]), pack_bf16x2(v[8 * q + 2], v[8 * q + 3]),
                                         pack_bf16x2(v[8 * q + 4], v[8 * q + 5]), pack_bf16x2(v[8 * q + 6], v[8 * q + 7]));
  }
  __syncthreads();
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int item = it * 256 + threadIdx.x;
    const int px = item >> 2, q = item & 3;
    const int x = x0 + px % kI2cW, y = y0 + px / kI2cW;
    if (x < W && y < H) dst[((size_t)((size_t)n * H + y) * W + x) * px16 + q] = otile[px][q];
  }
}

cudaError_t launch_lr_im2col(const float* lr, long long sn, long long sc, long long sy, void* dst, int N,
                             int H, int W, int dst_channels, const DynRef& dyn, cudaStream_t stream) {
  if ((H + kI2cH - 1) / kI2cH > 65535 || N > 65535) return cudaErrorInvalidValue;
  dim3 grid((W + kI2cW - 1) / kI2cW, (H + kI2cH - 1) / kI2cH, N);
  lr_im2col_kernel<<<grid, 256, 0, stream>>>(lr, sn, sc, sy, reinterpret_cast<uint4*>(dst), N, H, W, dst_channels / 8, dyn);
  return cudaGetLastError();
}

// =====================================================================================
// 8-bit frames -> the reference's fp32 lq: RescaleToZeroOne computes img.astype(np.float32) / 255. (normalization.py:
// 93-99), a correctly rounded fp32 division.  Multiplying by fl(1/255) instead differs for 126 of the 256 values, so
// the value table is built with __fdiv_rn.  HBM-bound (3 B in, 12 B out per pixel); kept out of lr_im2col and the
// conv_last epilogue, which read the fp32 frame: what fusing would save is ~14 MB per 720p frame against ~10 GB of
// feature traffic.
// =====================================================================================
constexpr int kU8PerThread = 4;
__global__ void __launch_bounds__(256)
unit_from_u8_kernel(const uint8_t* __restrict__ src, long long s_sf, long long s_sc, long long s_sy,
                    float* __restrict__ dst, long long d_sf, long long d_sc, long long d_sy, int H, int W) {
  __shared__ float lut[256];
  lut[threadIdx.x] = __fdiv_rn((float)threadIdx.x, 255.0f);
  __syncthreads();
  const int f = blockIdx.z, c = blockIdx.y / H, y = blockIdx.y % H;
  const uint8_t* s = src + f * s_sf + c * s_sc + y * s_sy;
  float* d = dst + f * d_sf + c * d_sc + y * d_sy;
  const int x0 = blockIdx.x * (256 * kU8PerThread) + threadIdx.x;
#pragma unroll
  for (int k = 0; k < kU8PerThread; ++k) {
    const int x = x0 + k * 256;
    if (x < W) d[x] = lut[__ldg(s + x)];
  }
}

cudaError_t launch_unit_from_u8(const uint8_t* src, long long s_sf, long long s_sc, long long s_sy, float* dst,
                               long long d_sf, long long d_sc, long long d_sy, int F, int H, int W,
                               cudaStream_t stream) {
  if (3LL * H > 65535 || F > 65535) return cudaErrorInvalidValue;
  dim3 grid((W + 256 * kU8PerThread - 1) / (256 * kU8PerThread), 3 * H, F);
  unit_from_u8_kernel<<<grid, 256, 0, stream>>>(src, s_sf, s_sc, s_sy, dst, d_sf, d_sc, d_sy, H, W);
  return cudaGetLastError();
}

// =====================================================================================
// Launch-table upload without the copy engine: the kernel reads PINNED host memory over the bus itself.  A
// cudaMemcpyAsync of the (small) table queues behind whatever the H2D copy engine is already moving -- with clips
// streaming in (driver.ClipStreamer) that is up to a whole clip, 67 ms at 720p x 100 frames, during which the first
// frame step cannot start (measured: 262 instead of 302 frames/s for such steps, tools/e2e_probe.py).
// =====================================================================================
__global__ void __launch_bounds__(256) fetch_pinned_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, long long n16) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (long long)gridDim.x * blockDim.x)
    dst[i] = src[i];
}

cudaError_t launch_fetch_pinned(const void* src_dev_view, void* dst, long long bytes, cudaStream_t stream) {
  const long long n16 = bytes >> 4;
  long long blocks = (n16 + 255) / 256;
  if (blocks > 592) blocks = 592;
  if (blocks < 1) return cudaSuccess;
  fetch_pinned_kernel<<<(int)blocks, 256, 0, stream>>>(reinterpret_cast<const uint4*>(src_dev_view),
                                                     reinterpret_cast<uint4*>(dst), n16);
  return cudaGetLastError();
}

// =====================================================================================
// K4: weight packing.  Packed operands are 128-byte rows [row = out channel][64 cols = in channel] bf16 with
// the 128B swizzle pre-applied (16-byte column group g of row r is stored at g ^ (r & 7)).
//
// With n_experts > 1 the block is the expert mixture  sum_e coef[e] * w[e]  of
// Dynamic_conv2d_se.forward (sr_backbone_utils.py:198-199), evaluated once per distinct CRF instead
// of once per block per frame.  `in_begin2 >= 0` adds a second input-channel slice (the
// neighbour == key_warp case of iconvsr_ipb_par.py:85-88, where two K slices see the same tensor).
// =====================================================================================
__device__ __forceinline__ size_t packed_offset(int block, int row, int col) {
  return (size_t)block * kPackBlockBytes + (size_t)row * 128 + (size_t)((((col >> 3) ^ (row & 7)) << 4)) +
         (size_t)(col & 7) * 2;
}

// Row-stacked layout of pnp_conv_rows.cu: per dx one block of 3*tap_n rows, sub-block sb = 0,1,2
// holding the weights of ky = 2 - sb (dy = +1, 0, -1); rows are 128-byte, 128B-swizzled.
__global__ void __launch_bounds__(256)
pack_conv3x3_rowstack_kernel(const float* __restrict__ w, int n_experts, const float* __restrict__ coef,
                             const float* __restrict__ row_scale, int out_ch, int in_total, int in_begin,
                             int in_begin2, int in_count, uint8_t* __restrict__ dst, int tap_n, bool flip_ky) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int per_dx = 3 * tap_n * 64;
  if (idx >= 3 * per_dx) return;
  const int dxi = idx / per_dx;
  const int rem = idx - dxi * per_dx;
  const int col = rem & 63, r = rem >> 6;          // r = sb * tap_n + o
  const int sb = r / tap_n, o = r - sb * tap_n;
  const int ky = flip_ky ? sb : 2 - sb, kx = dxi;    // mirrored for bottom-up traversal (flip_y)
  float acc = 0.f;
  if (o < out_ch && col < in_count) {
    const size_t per_expert = (size_t)out_ch * in_total * 9;
    for (int e = 0; e < n_experts; ++e) {
      const float ce = coef ? coef[e] : 1.0f;
      float v = w[e * per_expert + ((size_t)o * in_total + in_begin + col) * 9 + ky * 3 + kx];
      if (in_begin2 >= 0) v += w[e * per_expert + ((size_t)o * in_total + in_begin2 + col) * 9 + ky * 3 + kx];
      acc = fmaf(ce, v, acc);
    }
    if (row_scale) acc *= row_scale[o];
  }
  const size_t off = (size_t)dxi * (3 * tap_n * 128) + (size_t)r * 128 + (size_t)((((col >> 3) ^ (r & 7)) << 4)) +
                     (size_t)(col & 7) * 2;
  *reinterpret_cast<__nv_bfloat16*>(dst + off) = __float2bfloat16_rn(acc);
}

__global__ void __launch_bounds__(256)
pack_rows_kernel(const float* __restrict__ w, int rows, int cols, long long row_stride, long long col_stride,
                 uint8_t* __restrict__ dst, int row_offset) {
  // generic [rows<=64][cols<=64] matrix into rows row_offset.. of a packed block sequence
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 64 * 64) return;
  const int col = idx & 63, row = idx >> 6;
  float v = 0.f;
  if (row < rows && col < cols) v = w[(long long)row * row_stride + (long long)col * col_stride];
  const int r = row_offset + row;
  *reinterpret_cast<__nv_bfloat16*>(dst + packed_offset(r >> 6, r & 63, col)) = __float2bfloat16_rn(v);
}

__global__ void __launch_bounds__(256)
pack_aux_kernel(const float* __restrict__ w, int out_ch, int in_total, uint8_t* __restrict__ dst) {
  // [64 rows][64 cols]: col = tap*3 + c for the first 3 input channels
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 64 * 64) return;
  const int col = idx & 63, row = idx >> 6;
  float v = 0.f;
  if (row < out_ch && col < 27) {
    const int tap = col / 3, c = col - tap * 3;
    v = w[((size_t)row * in_total + c) * 9 + tap];
  }
  *reinterpret_cast<__nv_bfloat16*>(dst + packed_offset(0, row, col)) = __float2bfloat16_rn(v);
}

// All expert-mixed block-launch-A packs of one (CRF, QP) condition in ONE launch: block b of the stack gets
// [row-stacked gamma_o * sum_e a_e W2[b][e] (72 KB)][three 1x1 partition convs as 192 rows (24 KB)] at
// dst + b * dst_stride -- Dynamic_conv2d_se's per-block, per-frame torch.mm (sr_backbone_utils.py:198-208) done
// once per condition for the whole network.
__global__ void __launch_bounds__(256)
pack_mix_blocks_kernel(const float* __restrict__ w2, const float* __restrict__ w1x1, int n_experts,
                       const float* __restrict__ coef, const float* __restrict__ row_scale,
                       uint8_t* __restrict__ dst, long long dst_stride) {
  const int b = blockIdx.y;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  uint8_t* out = dst + (long long)b * dst_stride;
  constexpr int kMain = 9 * 64 * 64, kSide = 3 * 64 * 64;
  if (idx < kMain) {
    const int dxi = idx / (3 * 64 * 64);
    const int rem = idx - dxi * (3 * 64 * 64);
    const int col = rem & 63, r = rem >> 6;
    const int sb = r >> 6, o = r & 63;
    const int ky = 2 - sb, kx = dxi;
    const float* wb = w2 + (size_t)b * n_experts * 64 * 64 * 9;
    float acc = 0.f;
    for (int e = 0; e < n_experts; ++e)
      acc = fmaf(coef[e], wb[(size_t)e * 64 * 64 * 9 + ((size_t)o * 64 + col) * 9 + ky * 3 + kx], acc);
    acc *= row_scale[o];
    const size_t off = (size_t)dxi * (3 * 64 * 128) + (size_t)r * 128 + (size_t)((((col >> 3) ^ (r & 7)) << 4)) +
                       (size_t)(col & 7) * 2;
    *reinterpret_cast<__nv_bfloat16*>(out + off) = __float2bfloat16_rn(acc);
  } else if (idx < kMain + kSide) {
    const int k = idx - kMain;
    const int col = k & 63, r = k >> 6;             // r = class * 64 + out channel
    const float v = w1x1[(size_t)b * kSide + (size_t)r * 64 + col];
    *reinterpret_cast<__nv_bfloat16*>(out + 9 * 64 * 128 + packed_offset(r >> 6, r & 63, col)) = __float2bfloat16_rn(v);
  }
}

cudaError_t launch_pack_mix_blocks(const float* w2, const float* w1x1, int n_blocks, int n_experts, const float* coef,
                                   const float* row_scale, void* dst, long long dst_stride, cudaStream_t stream) {
  dim3 grid((12 * 64 * 64 + 255) / 256, n_blocks);
  pack_mix_blocks_kernel<<<grid, 256, 0, stream>>>(w2, w1x1, n_experts, coef, row_scale, reinterpret_cast<uint8_t*>(dst),
                                                   dst_stride);
  return cudaGetLastError();
}

cudaError_t launch_pack_conv3x3_rowstack(const float* w, int n_experts, const float* coef,
                                         const float* row_scale, int out_ch, int in_total, int in_begin,
                                         int in_begin2, int in_count, void* dst, int tap_n, bool flip_ky,
                                         cudaStream_t stream) {
  const int total = 3 * 3 * tap_n * 64;
  pack_conv3x3_rowstack_kernel<<<(total + 255) / 256, 256, 0, stream>>>(
      w, n_experts, coef, row_scale, out_ch, in_total, in_begin, in_begin2, in_count, reinterpret_cast<uint8_t*>(dst), tap_n, flip_ky);
  return cudaGetLastError();
}

cudaError_t launch_pack_rows(const float* w, int rows, int cols, long long row_stride, long long col_stride,
                             void* dst, int row_offset, cudaStream_t stream) {
  pack_rows_kernel<<<16, 256, 0, stream>>>(w, rows, cols, row_stride, col_stride,
                                           reinterpret_cast<uint8_t*>(dst), row_offset);
  return cudaGetLastError();
}

cudaError_t launch_pack_aux(const float* w, int out_ch, int in_total, void* dst, cudaStream_t stream) {
  pack_aux_kernel<<<16, 256, 0, stream>>>(w, out_ch, in_total, reinterpret_cast<uint8_t*>(dst));
  return cudaGetLastError();
}

// =====================================================================================
// CAA heads (compression-aware adaptation), one thread block per frame:
//   experts = softmax(W2 relu(W1 crf + b1) + b2)            Base_Predictor, domain_aware.py:172-183
//   gamma   = relu6(V2 relu(V1 qp) + 3) / 3                 SEModule/Hsigmoid, domain_aware.py:201-222
// and the per-frame, per-block epilogue bias  gamma * (experts . conv2.bias)
// (sr_backbone_utils.py:200-208), so that the conv kernels only see (scale, bias) vectors.
// =====================================================================================
__global__ void __launch_bounds__(64)
caa_heads_kernel(const float* __restrict__ base_qp, const float* __restrict__ qp, int frames,
                 const float* __restrict__ b0w, const float* __restrict__ b0b, const float* __restrict__ b2w,
                 const float* __restrict__ b2b, const float* __restrict__ s0w, const float* __restrict__ s2w,
                 int n_experts, int se_hidden, float* __restrict__ experts, float* __restrict__ gamma) {
  __shared__ float h[64];
  __shared__ float logit[16];
  const int f = blockIdx.x, tid = threadIdx.x;
  if (f >= frames) return;
  const float crf = base_qp[f], q = qp[f];
  h[tid] = fmaxf(fmaf(b0w[tid], crf, b0b[tid]), 0.f);
  __syncthreads();
  if (tid < n_experts) {
    float a = b2b[tid];
    for (int k = 0; k < 64; ++k) a = fmaf(b2w[tid * 64 + k], h[k], a);
    logit[tid] = a;
  }
  __syncthreads();
  if (tid < n_experts) {
    float m = logit[0];
    for (int e = 1; e < n_experts; ++e) m = fmaxf(m, logit[e]);
    float s = 0.f;
    for (int e = 0; e < n_experts; ++e) s += expf(logit[e] - m);
    experts[(size_t)f * n_experts + tid] = expf(logit[tid] - m) / s;
  }
  float g = 0.f;
  for (int k = 0; k < se_hidden; ++k) g = fmaf(s2w[tid * se_hidden + k], fmaxf(s0w[k] * q, 0.f), g);
  g = fminf(fmaxf(g + 3.0f, 0.f), 6.0f) / 3.0f;
  gamma[(size_t)f * 64 + tid] = g;
}

__global__ void __launch_bounds__(64)
mix_bias_kernel(const float* __restrict__ conv2_bias, long long block_stride, int n_blocks, int n_experts,
                const float* __restrict__ experts, const float* __restrict__ gamma, int frames,
                float* __restrict__ out) {
  // out[f][blk][c] = gamma[f][c] * sum_e experts[f][e] * conv2_bias[blk][e][c]
  const int f = blockIdx.x, blk = blockIdx.y, c = threadIdx.x;
  if (f >= frames) return;
  const float* b = conv2_bias + (long long)blk * block_stride;
  float a = 0.f;
  for (int e = 0; e < n_experts; ++e) a = fmaf(experts[(size_t)f * n_experts + e], b[e * 64 + c], a);
  out[((size_t)f * n_blocks + blk) * 64 + c] = a * gamma[(size_t)f * 64 + c];
}

cudaError_t launch_caa_heads(const float* base_qp, const float* qp, int frames, const float* b0w,
                             const float* b0b, const float* b2w, const float* b2b, const float* s0w,
                             const float* s2w, int n_experts, int se_hidden, float* experts, float* gamma,
                             cudaStream_t stream) {
  caa_heads_kernel<<<frames, 64, 0, stream>>>(base_qp, qp, frames, b0w, b0b, b2w, b2b, s0w, s2w, n_experts,
                                              se_hidden, experts, gamma);
  return cudaGetLastError();
}

cudaError_t launch_mix_bias(const float* conv2_bias, long long block_stride, int n_blocks, int n_experts,
                            const float* experts, const float* gamma, int frames, float* out,
                            cudaStream_t stream) {
  dim3 grid(frames, n_blocks);
  mix_bias_kernel<<<grid, 64, 0, stream>>>(conv2_bias, block_stride, n_blocks, n_experts, experts, gamma,
                                           frames, out);
  return cudaGetLastError();
}

}  // namespace pnp
