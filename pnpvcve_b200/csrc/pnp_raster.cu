// On-GPU rasteriser of the codec side information: per-block motion-vector records -> dense
// (T,4,H,W) motion fields and (T,3,H,W) partition maps (SURVEY.md section 8(f), rank 1).
//
// Replaces the per-record Python loop of LoadImageFromFileList_ipb.__call__
// (mmedit/datasets/pipelines/loading_ipb.py:328-369) + RescaleToZeroOne on the partition maps
// (normalization.py:93-99) + FramesToTensor (formating.py:101-138), bit for bit:
//   * ints by truncation (int()), motion/scale as an IEEE fp32 division;
//   * block = numpy slice [c - s//2 : c + s//2) per axis: negative bounds wrap once, then clamp;
//   * records are applied in order, later records overwrite earlier ones (resolved with an atomicMax
//     of the record index per pixel, then one gather pass);
//   * direction<0 -> channels 0,1 of the record's frame; direction>0 on a B frame -> channels 2,3;
//     direction>0 on a non-B frame -> NEGATED into channels 2,3 of the previous non-B frame at the
//     SOURCE block position; direction==0 -> no motion write (the reference's assert is a no-op);
//   * partition channel {256:0,128:1,64:2}[w*h] is set (never cleared) for every record.
// A frame window [a, b) of a clip (pnp_mv_rasterize_window) gives the planes of frames [a, b) of the whole-clip result:
// its table holds the window's records plus the reversed records of the tail frame e (the first non-B frame >= b, the
// only later frame that writes into the window), in clip order, so record-order overwrite and the fill pass's negation
// test hold unchanged.  A tail record makes only its reversed write; a target before the window (p_target -2) is
// skipped.
#include "pnp_ops.cuh"

namespace pnp {

namespace {

__device__ __forceinline__ int floordiv2(int v) { return v >> 1; }   // python // 2 (arithmetic shift)

// numpy slice(a, b) on an axis of length n -> [lo, hi) (empty when hi <= lo)
__device__ __forceinline__ void np_slice(int a, int b, int n, int& lo, int& hi) {
  if (a < 0) a += n;
  if (b < 0) b += n;
  lo = min(max(a, 0), n);
  hi = min(max(b, 0), n);
}

}  // namespace

__global__ void __launch_bounds__(256)
raster_owner_kernel(const float* __restrict__ rec, const int* __restrict__ frame_off, const int* __restrict__ is_b,
                    const int* __restrict__ p_target, int T, int tail, int window, int R, int H, int W,
                    unsigned* __restrict__ own_f, unsigned* __restrict__ own_b, unsigned* __restrict__ pmask,
                    int* __restrict__ status) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= R) return;
  const float* r = rec + (size_t)warp * 10;
  const float direction = r[0];
  const int w = (int)r[1], h = (int)r[2], xs = (int)r[3], ys = (int)r[4], x = (int)r[5], y = (int)r[6];
  // frame of this record: last f with frame_off[f] <= warp
  int f = 0;
  {
    int lo = 0, hi = T + tail;                // frame_off has T+tail+1 entries
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (frame_off[mid] <= warp) lo = mid; else hi = mid;
    }
    f = lo;
  }
  const bool in_tail = f == T;               // the tail frame's own planes lie outside the window
  const size_t plane = (size_t)H * W;
  const unsigned key = (unsigned)warp + 1u;   // global record index + 1: later records win
  // partition: every record, destination block
  int r0, r1, c0, c1;
  np_slice(y - floordiv2(h), y + floordiv2(h), H, r0, r1);
  np_slice(x - floordiv2(w), x + floordiv2(w), W, c0, c1);
  const int area = w * h;
  unsigned pbit = in_tail ? 0u : area == 256 ? 1u : area == 128 ? 2u : area == 64 ? 4u : 0u;
  if (pbit == 0u && !in_tail && lane == 0) atomicOr(status, 1);   // KeyError in the reference
  unsigned* owner = nullptr;
  int tr0 = r0, tr1 = r1, tc0 = c0, tc1 = c1;
  if (direction < 0.f) {
    if (!in_tail) owner = own_f + (size_t)f * plane;
  } else if (direction > 0.f) {
    if (!in_tail && is_b[f]) {                // (the tail frame is non-B)
      owner = own_b + (size_t)f * plane;
    } else {
      const int tgt = p_target[f];
      if (tgt == -2 && window) {
        // target before the window: the write lands outside it
      } else if (tgt < 0) {
        if (lane == 0) atomicOr(status, 2);                  // p_offset unbound / before the clip
      } else {
        owner = own_b + (size_t)tgt * plane;
        np_slice(ys - floordiv2(h), ys + floordiv2(h), H, tr0, tr1);
        np_slice(xs - floordiv2(w), xs + floordiv2(w), W, tc0, tc1);
      }
    }
  }
  // destination block: partition bits (+ motion owner when it is the same block)
  {
    const int bw = max(c1 - c0, 0), bh = max(r1 - r0, 0);
    const bool same = owner != nullptr && tr0 == r0 && tr1 == r1 && tc0 == c0 && tc1 == c1;
    for (int i = lane; i < bw * bh; i += 32) {
      const int yy = r0 + i / bw, xx = c0 + i % bw;
      const size_t p = (size_t)yy * W + xx;
      if (pbit) atomicOr(pmask + (size_t)f * plane + p, pbit);
      if (same) atomicMax(owner + p, key);
    }
    if (same) owner = nullptr;
  }
  if (owner != nullptr) {                                     // reversed P record: source block
    const int bw = max(tc1 - tc0, 0), bh = max(tr1 - tr0, 0);
    for (int i = lane; i < bw * bh; i += 32) {
      const int yy = tr0 + i / bw, xx = tc0 + i % bw;
      atomicMax(owner + (size_t)yy * W + xx, key);
    }
  }
}

__global__ void __launch_bounds__(256)
raster_fill_kernel(const float* __restrict__ rec, const int* __restrict__ frame_off,
                   const unsigned* __restrict__ own_f, const unsigned* __restrict__ own_b,
                   const unsigned* __restrict__ pmask, int H, int W, float* __restrict__ mvs,
                   float* __restrict__ partitions) {
  const int x = blockIdx.x * 256 + threadIdx.x;
  const int y = blockIdx.y;
  const int f = blockIdx.z;
  if (x >= W) return;
  const size_t plane = (size_t)H * W;
  const size_t p = (size_t)y * W + x;
  const unsigned kf = own_f[(size_t)f * plane + p];
  const unsigned kb = own_b[(size_t)f * plane + p];
  float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;
  if (kf) {
    const float* r = rec + (size_t)(kf - 1) * 10;
    v0 = __fdiv_rn(r[7], r[9]);
    v1 = __fdiv_rn(r[8], r[9]);
  }
  if (kb) {
    const float* r = rec + (size_t)(kb - 1) * 10;
    v2 = __fdiv_rn(r[7], r[9]);
    v3 = __fdiv_rn(r[8], r[9]);
    if ((int)(kb - 1) >= frame_off[f + 1]) {   // written by a later P frame: reversed flow
      v2 = -v2;
      v3 = -v3;
    }
  }
  float* m = mvs + (size_t)f * 4 * plane + p;
  m[0] = v0;
  m[plane] = v1;
  m[2 * plane] = v2;
  m[3 * plane] = v3;
  const unsigned pm = pmask[(size_t)f * plane + p];
  const float one = __fdiv_rn(1.0f, 255.0f);   // RescaleToZeroOne: float32(1) / 255
  float* q = partitions + (size_t)f * 3 * plane + p;
  q[0] = (pm & 1u) ? one : 0.f;
  q[plane] = (pm & 2u) ? one : 0.f;
  q[2 * plane] = (pm & 4u) ? one : 0.f;
}

cudaError_t launch_mv_rasterize(const float* rec, const int* frame_off, const int* is_b, const int* p_target,
                                int T, int tail, bool window, int R, int H, int W, unsigned* own_f, unsigned* own_b,
                                unsigned* pmask, float* mvs, float* partitions, int* status, cudaStream_t stream) {
  if (R > 0) {
    const long long threads = (long long)R * 32;
    raster_owner_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(
        rec, frame_off, is_b, p_target, T, tail, window ? 1 : 0, R, H, W, own_f, own_b, pmask, status);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  dim3 grid((W + 255) / 256, H, T);
  raster_fill_kernel<<<grid, 256, 0, stream>>>(rec, frame_off, own_f, own_b, pmask, H, W, mvs, partitions);
  return cudaGetLastError();
}

}  // namespace pnp
