// Parameters of the row-stacked tcgen05 implicit-GEMM 3x3 convolution kernel (pnp_conv_rows.cu).
#pragma once
#include <cuda.h>
#include <stdint.h>

namespace pnp {

constexpr int kTilePx = 128;                 // output pixels per UMMA tile (one image-row segment)
constexpr int kHaloPx = kTilePx + 2;         // source pixels staged per row (x halo of 1 each side)
constexpr int kRowBytes = kHaloPx * 128;     // 16640: one staged source row, 64 bf16 per pixel
constexpr int kASlotBytes = 17 * 1024;       // ring slot (1024-aligned, >= kRowBytes)
constexpr int kTileBytes = kTilePx * 128;    // 16384: one 128-pixel x 64-channel bf16 tile
constexpr int kWChunkBytes = 8192;           // one 64(N) x 64(K) bf16 weight block
constexpr int kRowsThreads = 352;            // warp0 TMA producer, warp1 MMA issuer, warps2-9 epilogue, warp10 barrier scout
constexpr int kRowsThreadsPar = 480;         // block launch A: + warps 11-14, the readers of the 1x1 accumulator region
constexpr int kEpilogueWarps = 8;
constexpr int kMaxASlots = 8;
constexpr int kMaxIoSlots = 6;
constexpr int kTmemCols = 512;

enum ConvMode { kModeBf16 = 0, kModeLast = 1 };
enum ConvAct { kActNone = 0, kActLrelu = 1, kActRelu = 2 };

// One entry of a device-resident launch table (include/pnp_vcve.h: pnp_dyn_entry): the operands of a launch that
// change from frame step to frame step.  A kernel launched in table mode reads entry
// table[*step * stride + node]; everything else in its parameters is constant for the clip, so the launch can sit
// in a CUDA graph that is replayed for every frame.
struct DynEntry {
  unsigned long long p[6];
  int i[4];
};
static_assert(sizeof(DynEntry) == 64, "launch-table entry is 64 bytes (ABI)");

struct DynRef {
  const DynEntry* table;   // nullptr: static launch, every operand is in the kernel parameters
  const int* step;
  int node, stride;
  __device__ __forceinline__ const DynEntry* entry() const {
    return table ? table + ((long long)(*step) * stride + node) : nullptr;
  }
};

struct ConvParams {
  CUtensorMap tm_src;   // (64, W, H, images) bf16, box (64,130,1,1), SWIZZLE_128B
  CUtensorMap tm_aux;   // box (64,128,1,1); aux_pitch64: (32,128,1,1), SWIZZLE_64B
  CUtensorMap tm_id;    // box (64,128,1,1)
  CUtensorMap tm_out;   // box (64,128,1,1)
  DynRef dyn;           // table mode: conv entry = p{wpack, bias, par, lq, outf, img_off}, i{src_f, aux_f, idt_f, out_f}
  const void* wpack;    // packed weights, pre-swizzled, in consumption order
  const float* scale;   // [64] per-output-channel scale of the 3x3 accumulator, or null
  const float* bias;    // [64] ([3] in kModeLast), or null
  const long long* img_off;  // per-image (weight byte offset, bias float offset) pairs, or null; needs cpi > 0
  const float* par;     // partition map (n,3,H,W) fp32 view, or null
  long long par_sn, par_sc, par_sy;
  const float* lq;      // kModeLast: (n,3,H,W) fp32 view added to the output
  long long lq_sn, lq_sc, lq_sy;
  float* outf;          // kModeLast: (n,3,H,W) fp32 view -- uint8 with out_u8 (strides then in bytes)
  long long of_sn, of_sc, of_sy;
  int H, W, N, strips;
  int tiles_total, tiles_per_cta;
  int cpi;              // > 0: CTAs per image -- a CTA's tiles never cross an image (per-image weights / bias)
  int has_par;          // 3x3 + three partition 1x1 convs (block launch A)
  int has_bias;
  int tap_n;            // N of one dy sub-block: 64, or 16 for the 64->3 tail
  int aux_k16;          // K/16 of the aux source (centre row only); 0 = no aux
  int aux_pitch64;      // the aux source is a (N,H,W,32) tensor: 64-byte pixels, SWIZZLE_64B tiles of 8 KB (single-CTA form only)
  int has_id;
  int act;
  int mode;
  int flip_y;           // walk the image bottom-up (weights packed with ky mirrored)
  int l2_src, l2_idt, l2_out;   // L2 eviction policy of the src / identity loads and the output stores:
                        // 0 default, 1 evict_first (dead after this access), 2 evict_last (the next launch reads it)
  int par_split;        // partition variant: dedicated reader warps for the 1x1 accumulator region
  int par_sparse;       // partition blend: last non-zero class only, / 255 (the reference's sparse_val eval path)
  int lq_up4;           // kModeLast: lq is the (H/4, W/4) frame, the epilogue adds its x4 bilinear upsampling
  int w_stable;         // weights may be fetched before the previous kernel in the stream has completed
  int pair;             // CTA-pair mode (cluster of 2, tcgen05 cta_group::2): a "tile" below is a PAIR of 128-pixel tiles,
                        // the same row of two adjacent (image, strip) columns; tiles_total / tiles_per_cta / cpi then
                        // count pair-tiles per cluster
  int s_a;              // A ring slots
  int n_io;             // id/out staging slots
  long long* trace;     // PNP_DIAG builds: device buffer for per-tile clock64 stamps of CTA 0
  int debug_skip;       // PNP_DIAG builds: what-if profiling bits (results are WRONG)
  int out_u8;           // kModeLast: store tensor2img's uint8 value of each output sample (quant_u8) instead of fp32
};

// sparse_val eval path of the reference (sr_backbone_utils.py:294-302, basicvsr_net.py:511-514): per class the
// 1x1 result is scattered to the pixels whose mask is non-zero, later classes overwrite earlier ones.  Turns the
// three map values into blend weights: 1/255 for the surviving class, 0 for the others -- the dense blend code
// then computes W_k x * fl(1/255), within one fp32 ulp of the reference's W_k x / 255, and the hot epilogue
// loops stay free of a second code path (a runtime branch with a true division in them cost launch A 45 %).
__device__ __forceinline__ void par_sparse_select(float& p0, float& p1, float& p2) {
  const bool n2 = p2 != 0.f, n1 = p1 != 0.f, n0 = p0 != 0.f;
  const float c = 1.0f / 255.0f;
  p2 = n2 ? c : 0.f;
  p1 = (!n2 && n1) ? c : 0.f;
  p0 = (!n2 && !n1 && n0) ? c : 0.f;
}

// weights packed as [dx][dy sub-block][tap_n rows] (pnp_pack_conv3x3_rowstack)
size_t conv_rows_smem_bytes(const ConvParams& p);
// opt every kernel variant in to 227 KB of shared memory on the current device; max_pairs = CTA pairs (clusters of 2)
// of the pair variants that can be resident at once
cudaError_t conv_rows_prepare(int* max_pairs);
// grid = CTAs (p.pair: 2 x clusters)
cudaError_t launch_conv_rows(const ConvParams& p, int grid, cudaStream_t stream);

}  // namespace pnp
