// Row-stacked variant of the tcgen05 3x3 convolution: one source row feeds THREE output rows.
//
// Why (measured, profiles/r01_notes.md): an M=128,K=16 tcgen05.mma costs max(N/2, (4096+32N)/128)
// cycles, so the N=64 MMAs of the tap-major kernel (pnp_conv.cu) are bound by the shared-memory
// operand pipe at 64 % of the tensor peak.  Here the A operand is still "128 pixels of source row r,
// shifted by dx", but B stacks the three dy weight blocks [W(+1,dx); W(0,dx); W(-1,dx)] so a single
// N=192 MMA (~98 cycles instead of 3 x 50) adds row r's contribution to the accumulators of output
// rows r-1, r and r+1 at once.  Accumulators of eight consecutive output rows live in a TMEM ring
// (8 x 64 columns = all 512), each source row is staged in shared memory for exactly one step, and
// an output row is finished -- and handed to the epilogue -- one step after its own source row.
//
// Same reference semantics as pnp_conv.cu (F.conv2d + bias/activation/identity/LR-aux/+lq fused).
//
// kPar (block launch A of ResidualBlockNoBNDynamic_drt, sr_backbone_utils.py:310-311): the three
// partition-modulated 1x1 convs are one extra N=192 MMA group on the centre row into a dedicated
// 192-column TMEM region; the epilogue folds sum_k par_k * conv1x1_k(x) into registers one step
// ahead of the 3x3 result (accumulator ring shrinks to 5 x 64 columns to make room).
//
// kPair (round 2): the same kernel as a CLUSTER OF TWO CTAs issuing tcgen05.mma.cta_group::2 (M = 256).  The two CTAs
// walk the same rows of two adjacent (image, strip) columns in lockstep; every MMA multiplies both CTAs' source rows
// with ONE weight block of which each CTA holds (and fetches from its shared memory) only half of the rows: 56 instead
// of 80 shared-memory cycles per N=192 MMA -- the measured bound of this kernel is the 128 B/clk shared-memory pipe.
// Only the leader (cluster rank 0) runs the MMA issuer and the scout; its "full"/"free" barriers collect the TMA
// completions and the epilogue arrivals of both CTAs, commits are multicast to both.  Accumulator windows that wrap
// the TMEM ring (or are clipped at a segment end) cannot be issued as partial-N MMAs out of an N-split weight block,
// so they run as per-sub-block N=64 MMAs out of a second, per-sub-block-split copy of the weights, chained through the
// A-operand collector (fill/use/lastuse: the A tile is fetched once; tools/umma_collect_bench.cu).
#include <type_traits>

#include "pnp_conv.cuh"
#include "pnp_ops.cuh"
#include "pnp_ptx.cuh"

// Diagnostics (what-if bits, clock traces) exist only in PNP_DIAG builds (PNP_DIAG=1 python -m pnpvcve_b200.build):
// the default library neither reads such knobs nor carries their code.
#ifdef PNP_DIAG
#define PNP_DBG(bit) ((p.debug_skip & (bit)) != 0)
#define PNP_TRACING (p.trace != nullptr)
#else
#define PNP_DBG(bit) false
#define PNP_TRACING false
#endif

namespace pnp {

namespace {

constexpr int kAccRingMax = 8;   // output-row accumulators in TMEM (8 x 64 columns; 5 with kPar)
// Step-completion barriers.  A barrier is re-used every kStepRing steps, so the issuing thread must never commit step
// s + kStepRing before the slowest waiter has looked at step s.  What holds it back is the ACCUMULATOR ring -- it can
// be at most 8 output rows (5 with kPar) ahead of the epilogue -- but steps are not rows: two rows can complete with one
// step (the last two of a segment that ends at the image bottom) and a segment can begin with a step that completes no
// row, so 9 rows in flight span up to 12 steps (H >= 8).  With 8 barriers the CTA whose range ends a few rows into a new
// column (at 720p: CTA 102, 42 + 7 rows) could commit step 50 on the barrier of step 42 while its epilogue was a full
// ring behind and still about to wait for step 42: the phase flips twice, the wait never returns.  Seen once in ~10^6
// launches, reproduced at will under compute-sanitizer (which slows the epilogue); 16 barriers close it.
#ifndef PNP_STEP_RING_LOG2
#define PNP_STEP_RING_LOG2 4     // (3 re-creates the dead-lock for the regression test's own validation)
#endif
constexpr int kStepShift = PNP_STEP_RING_LOG2;
constexpr int kStepRing = 1 << kStepShift;
constexpr int kParCol = 320;     // TMEM column of the partition 1x1 accumulators (3 x 64)

struct RowsLayout {
  uint32_t w, a, aux, io, misc, total;
};

__host__ __device__ inline RowsLayout rows_layout(int w_bytes, int s_a, int has_aux, int n_io) {
  RowsLayout l;
  l.w = 0;
  l.a = l.w + ((w_bytes + 1023) & ~1023);
  l.aux = l.a + s_a * kASlotBytes;
  l.io = l.aux + (has_aux ? 2 * kTileBytes : 0);
  l.misc = l.io + n_io * kTileBytes;
  l.total = l.misc + 1024;
  return l;
}

struct RowsMisc {
  float scale[64];
  float bias[64];
  uint64_t w_full;
  uint64_t a_full[kMaxASlots];
  uint64_t step_done[kStepRing];   // tcgen05.commit after every step (one source row)
  uint64_t acc_free[kAccRingMax];  // epilogue -> MMA: accumulator slot drained
  uint64_t par_done;               // MMA -> epilogue: partition 1x1 accumulators of a row are ready
  uint64_t aux_full[2];
  uint64_t id_full[kMaxIoSlots];
  uint64_t io_empty[kMaxIoSlots];
  uint32_t tmem_base;
  uint32_t go_step;                // scout -> MMA: steps whose barriers have all completed
  uint32_t go_par;                 // epilogue -> MMA: epilogue-warp reads of the partition region (8 or 4 per row)
  uint32_t slot_free;              // split roles: output rows whose TMA stores have finished reading their staging slot
  uint64_t dy_full[kMaxIoSlots];   // split roles: region readers -> main epilogue: the row's 1x1 blend is parked
  uint64_t peer_w;                 // pair mode, leader: the other CTA's weights have landed
};
static_assert(sizeof(RowsMisc) <= 1024, "misc region overflow");

// A CTA owns the tiles [t_begin, t_end) in (image, strip, row) order; a segment is a maximal run of
// consecutive rows of one strip.  Steps j = j_first..j_last are the in-image source rows y_b + j.
struct Segment {
  int n, strip, y_b, len, j_first, j_last;
};

struct SegIter {
  int t, t_end, H, strips, n, strip, y_b, dcol;
  // rank: this CTA's position in its pair (pair mode: tiles count column PAIRS, the CTA walks column 2*pair + rank)
  __device__ SegIter(const ConvParams& p, int b, int e, int rank = 0) : t(b), t_end(e), H(p.H), strips(p.strips) {
    int col = b / p.H;
    y_b = b - col * p.H;
    dcol = p.pair ? 2 : 1;
    if (p.pair) col = 2 * col + rank;
    n = col / p.strips;
    strip = col - n * p.strips;
  }
  __device__ __forceinline__ bool valid() const { return t < t_end; }
  __device__ __forceinline__ Segment get() const {
    Segment s;
    s.n = n;
    s.strip = strip;
    s.y_b = y_b;
    s.len = min(H - y_b, t_end - t);
    s.j_first = (y_b > 0) ? -1 : 0;
    s.j_last = (y_b + s.len < H) ? s.len : s.len - 1;
    return s;
  }
  __device__ __forceinline__ void next(const Segment& s) {
    t += s.len;
    y_b = 0;
    strip += dcol;
    while (strip >= strips) {
      strip -= strips;
      ++n;
    }
  }
};

struct Ring {
  uint32_t slot, phase, size;
  __device__ explicit Ring(uint32_t n) : slot(0), phase(0), size(n) {}
  __device__ __forceinline__ void advance() {
    if (++slot == size) {
      slot = 0;
      phase ^= 1;
    }
  }
};

__device__ __forceinline__ float act_fn(float v, int act) {
  if (act == kActLrelu) return v > 0.f ? v : 0.1f * v;
  if (act == kActRelu) return fmaxf(v, 0.f);
  return v;
}

}  // namespace

template <bool kPar, bool kScale, bool kPair>
__global__ void __launch_bounds__(kPar ? kRowsThreadsPar : kRowsThreads, 1)
conv3x3_rows_kernel(const __grid_constant__ ConvParams p) {
  constexpr int kAccRing = kPar ? 5 : 8;
  const int rank = kPair ? (int)cluster_ctarank() : 0;        // position in the CTA pair; 0 = leader
  const int unit = kPair ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;   // tile ranges are per CTA / per pair
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t sbase = (raw + 1023u) & ~1023u;
  uint8_t* sgen = smem_raw + (sbase - raw);
  const int tap_n = p.tap_n;                            // 64, or 16 for the 64->3 tail
  const int dx_block_bytes = 3 * tap_n * 128;           // [3 dy sub-blocks][tap_n rows][128 B]
  // bytes of weights resident in THIS CTA.  Pair mode: half of the rows of every block, twice (N-split layout for
  // whole N = 3*tap_n windows, per-sub-block-split layout for the N = tap_n MMAs of wrapped / clipped windows)
  const int w_bytes = kPair ? 3 * dx_block_bytes + (p.aux_k16 > 0 ? kWChunkBytes / 2 : 0) + (kPar ? 3 * 64 * 128 / 2 : 0)
                            : 3 * dx_block_bytes + (p.aux_k16 > 0 ? kWChunkBytes : 0) + (kPar ? 3 * 64 * 128 : 0);
  const RowsLayout L = rows_layout(w_bytes, p.s_a, p.aux_k16 > 0, p.n_io);
  RowsMisc* misc = reinterpret_cast<RowsMisc*>(sgen + L.misc);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // Tile range.  cpi > 0: `cpi` CTAs per image, so that a CTA never crosses an image and can use that image's own
  // weights / bias (clips with different CRF / QP conditions in ONE launch: the reference's groups=batch grouped conv,
  // sr_backbone_utils.py:196-204).
  int t_begin, t_end, img = 0;
  if (p.cpi > 0) {
    img = unit / p.cpi;
    const int tiles_img = (kPair ? p.strips >> 1 : p.strips) * p.H;     // pair mode: strips is even here
    t_begin = img * tiles_img + (unit - img * p.cpi) * p.tiles_per_cta;
    t_end = min((img + 1) * tiles_img, t_begin + p.tiles_per_cta);
  } else {
    t_begin = unit * p.tiles_per_cta;
    t_end = min(p.tiles_total, t_begin + p.tiles_per_cta);
  }
  // Operands that change per frame step come from the launch table in table mode (constant kernel parameters
  // otherwise).  The table and the step word were written by stream operations that completed before the first
  // kernel of this step started, so they may be read ahead of griddepcontrol.wait.
  const DynEntry* dyn = p.dyn.entry();
  const long long* img_off = dyn ? reinterpret_cast<const long long*>(dyn->p[5]) : p.img_off;
  const long long w_off = img_off ? img_off[2 * img] : 0, b_off = img_off ? img_off[2 * img + 1] : 0;
  const uint8_t* const wpack = (dyn ? reinterpret_cast<const uint8_t*>(dyn->p[0]) : static_cast<const uint8_t*>(p.wpack)) + w_off;
  const float* const bias_g = p.has_bias ? (dyn ? reinterpret_cast<const float*>(dyn->p[1]) : p.bias) + b_off : nullptr;
  const float* const par_g = dyn ? reinterpret_cast<const float*>(dyn->p[2]) : p.par;
  const float* const lq_g = dyn ? reinterpret_cast<const float*>(dyn->p[3]) : p.lq;
  float* const outf_g = dyn ? reinterpret_cast<float*>(dyn->p[4]) : p.outf;
  const int src_f = dyn ? dyn->i[0] : 0, aux_f = dyn ? dyn->i[1] : 0, idt_f = dyn ? dyn->i[2] : 0,
            out_f = dyn ? dyn->i[3] : 0;
  const int s_a = p.s_a;
  const int n_io = p.n_io;
  const bool last_mode = (p.mode == kModeLast);
  // flip_y: the image is walked bottom-up (weights are packed with ky mirrored), so that a launch
  // reads first what the previous launch wrote last -- those rows are still in L2.
  const int y_flip_base = p.flip_y ? p.H - 1 : 0;
  const int y_sign = p.flip_y ? -1 : 1;
#define PNP_Y(yy) (y_flip_base + y_sign * (yy))

  if (threadIdx.x < 64) {
    misc->scale[threadIdx.x] = p.scale ? p.scale[threadIdx.x] : 1.0f;
    const int nb = last_mode ? 3 : 64;
    misc->bias[threadIdx.x] = (bias_g && threadIdx.x < nb) ? bias_g[threadIdx.x] : 0.0f;
  }
  if (warp == 0) {
    if (lane == 0) {
      mbar_init(smem_u32(&misc->w_full), 1);
      for (int i = 0; i < kMaxASlots; ++i) mbar_init(smem_u32(&misc->a_full[i]), 1);
      for (int i = 0; i < kStepRing; ++i) mbar_init(smem_u32(&misc->step_done[i]), 1);
      // pair mode: the leader's acc_free barriers collect the reader warps of both CTAs
      const int acc_readers = kEpilogueWarps * (kPair ? 2 : 1);
      for (int i = 0; i < kAccRingMax; ++i) mbar_init(smem_u32(&misc->acc_free[i]), acc_readers);
      mbar_init(smem_u32(&misc->peer_w), 1);
      for (int i = 0; i < kMaxIoSlots; ++i) mbar_init(smem_u32(&misc->dy_full[i]), 4);
      misc->slot_free = 0;
      mbar_init(smem_u32(&misc->par_done), 1);
      for (int i = 0; i < 2; ++i) mbar_init(smem_u32(&misc->aux_full[i]), 1);
      for (int i = 0; i < kMaxIoSlots; ++i) {
        mbar_init(smem_u32(&misc->id_full[i]), 1);
        mbar_init(smem_u32(&misc->io_empty[i]), 1);
      }
      misc->go_step = 0;
      misc->go_par = 0;
      mbar_fence_init();
      tma_prefetch_desc(&p.tm_src);
      if (!last_mode) tma_prefetch_desc(&p.tm_out);
    }
    __syncwarp();
    if (kPair) tmem_alloc2(smem_u32(&misc->tmem_base), kTmemCols);
    else tmem_alloc(smem_u32(&misc->tmem_base), kTmemCols);
  }
  tc_fence_before();
  // pair mode: the peer's barriers must be initialised before the first remote arrival / TMA completion reaches them
  if (kPair) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = misc->tmem_base;
  // Programmatic dependent launch: launch latency, block scheduling and the prologue above overlap
  // the tail of the previous kernel in the stream; nothing below touches global memory before the
  // previous kernel has completed (packed weights may have been written by the kernel just before).
  griddep_launch_dependents();
  const uint32_t w_smem_early = sbase + L.w;
  auto load_weights = [&]() {                 // one elected lane of warp 0
    const uint32_t wbar = smem_u32(&misc->w_full);
    mbar_arrive_expect_tx(wbar, w_bytes);
    if (kPair) {
      // This CTA's halves, straight out of the ordinary pack [dx][dy sub-block][tap_n rows][128 B] (row counts are
      // multiples of 8, so the pre-applied 128B swizzle stays valid at the new 1024-aligned offsets):
      //   [0, 3*h192): per dx the rows [rank*3*tap_n/2, +3*tap_n/2) of the stacked block   (whole-window MMAs)
      //   then per (dx, sub-block) the rows [rank*tap_n/2, +tap_n/2) of the sub-block      (per-sub-block MMAs)
      //   then this CTA's half of the LR-im2col block (aux, N = 64) or of the stacked 1x1 block (kPar, N = 192)
      const int h192 = dx_block_bytes >> 1, h64 = (tap_n * 128) >> 1;
      for (int dx = 0; dx < 3; ++dx)
        bulk_load_1d(w_smem_early + dx * h192, wpack + dx * dx_block_bytes + rank * h192, h192, wbar);
      for (int b = 0; b < 9; ++b)
        bulk_load_1d(w_smem_early + 3 * h192 + b * h64, wpack + b * (tap_n * 128) + rank * h64, h64, wbar);
      const int extra = w_bytes - 3 * dx_block_bytes;
      if (extra > 0)
        bulk_load_1d(w_smem_early + 3 * dx_block_bytes, wpack + 3 * dx_block_bytes + rank * extra, extra, wbar);
    } else {
      for (int off = 0; off < w_bytes; off += kWChunkBytes) {
        const int n = min(kWChunkBytes, w_bytes - off);
        bulk_load_1d(w_smem_early + off, wpack + off, n, wbar);
      }
    }
  };
  // stable weights (packed long before this launch) are fetched while the previous kernel drains
  if (p.w_stable && warp == 0) {
    if (elect_one()) load_weights();
    __syncwarp();
  }
  griddep_wait();
  if (PNP_TRACING && threadIdx.x == 0) {            // per-CTA body start (cycles, ns): stored, not kept live
    p.trace[2048 + blockIdx.x] = -clock64();
    p.trace[2208 + blockIdx.x] = (long long)globaltimer_ns();
  }
  // Threads that merely wait for work poll patiently (one lane per warp, hardware suspend hint): hot
  // try_wait loops of 256 epilogue lanes compete with the MMA operand fetch for the shared-memory pipe
  // (measured: N=192 MMAs ~25 % slower).  debug bit 32 selects patient polling, bit 64 shortens the hint.
  const bool par_defer = kPar && p.par_split && PNP_DBG(1024);    // diagnostic, see the MMA issuer
  const bool hot_waits = !PNP_DBG(32);
  const uint32_t hint_ns = PNP_DBG(64) ? 40u : 200u;
  auto pwait = [&](uint32_t bar, uint32_t parity, int tag) {      // one elected lane
    if (hot_waits) mbar_wait(bar, parity, tag); else mbar_wait_patient(bar, parity, tag, hint_ns);
  };
  auto ewait = [&](uint32_t bar, uint32_t parity, int tag) {      // whole (converged) warp
    if (hot_waits) mbar_wait(bar, parity, tag); else mbar_wait_warp(bar, parity, tag, hint_ns);
  };
  // debug bit 2048: every output row of the epilogue starts ~2 us late, so the epilogue trails the MMA issuer by a full
  // accumulator ring -- the schedule the step-barrier ring (kStepRing) must survive; results stay exact
  auto slow_epilogue = [&]() {
    if (PNP_DBG(2048)) __nanosleep(2000);
  };
  const uint32_t w_smem = sbase + L.w;
  const uint32_t a_smem = sbase + L.a;
  const uint32_t aux_smem = sbase + L.aux;
  const uint32_t io_smem = sbase + L.io;

  if (warp == 0) {
    // ============================================================ TMA producer (one elected lane)
    if (elect_one()) {
      if (!p.w_stable) load_weights();
      const uint64_t pol_src = p.l2_src == 2 ? l2_policy_evict_last() : l2_policy_evict_first();
      Ring ar(s_a);
      uint32_t sc = 0, ord = 0;            // step counter, output-row ordinal
      uint32_t aux_step[2] = {0, 0};       // step in which each aux slot was last consumed
      for (SegIter it(p, t_begin, t_end, rank); it.valid();) {
        const Segment s = it.get();
        const int x0 = s.strip * kTilePx;
        for (int j = s.j_first; j <= s.j_last; ++j, ++sc, ar.advance()) {
          if (sc >= (uint32_t)s_a) {       // slot last used by step sc - s_a
            // with deferred 1x1 MMAs the row of step ps is still read during step ps + 1
            const uint32_t ps = sc - s_a + (par_defer ? 1u : 0u);
            pwait(smem_u32(&misc->step_done[ps & (kStepRing - 1)]), (ps >> kStepShift) & 1, 1);
          }
          const uint32_t fb = smem_u32(&misc->a_full[ar.slot]);
          if (kPair) {
            // both CTAs' rows complete on the LEADER's barrier, which expects the bytes of the two loads (a
            // completion that overtakes the leader's expect_tx only drives the pending count negative for a while)
            if (rank == 0) mbar_arrive_expect_tx(fb, 2 * kRowBytes);
            tma_load_4d_pair(a_smem + ar.slot * kASlotBytes, &p.tm_src, mapa_shared(fb, 0), 0, x0 - 1, PNP_Y(s.y_b + j),
                             s.n + src_f);
          } else if (PNP_DBG(1) && sc >= (uint32_t)s_a) {
            mbar_arrive(fb);
          } else {
            mbar_arrive_expect_tx(fb, kRowBytes);
            if (p.l2_src)
              tma_load_4d_hint(a_smem + ar.slot * kASlotBytes, &p.tm_src, fb, 0, x0 - 1, PNP_Y(s.y_b + j), s.n + src_f, pol_src);
            else
              tma_load_4d(a_smem + ar.slot * kASlotBytes, &p.tm_src, fb, 0, x0 - 1, PNP_Y(s.y_b + j), s.n + src_f);
          }
          if (j >= 0 && j < s.len) {       // per-output-row operands of row y_b + j
            if (p.aux_k16 > 0) {
              const uint32_t as = ord & 1;
              if (ord >= 2) {
                const uint32_t ps = aux_step[as];
                pwait(smem_u32(&misc->step_done[ps & (kStepRing - 1)]), (ps >> kStepShift) & 1, 2);
              }
              aux_step[as] = sc;           // consumed in this very step (centre row)
              const uint32_t ab = smem_u32(&misc->aux_full[as]);
              if (kPair) {
                if (rank == 0) mbar_arrive_expect_tx(ab, 2 * kTileBytes);
                tma_load_4d_pair(aux_smem + as * kTileBytes, &p.tm_aux, mapa_shared(ab, 0), 0, x0, PNP_Y(s.y_b + j),
                                 s.n + aux_f);
              } else {
                mbar_arrive_expect_tx(ab, p.aux_pitch64 ? kTileBytes / 2 : kTileBytes);
                tma_load_4d(aux_smem + as * kTileBytes, &p.tm_aux, ab, 0, x0, PNP_Y(s.y_b + j), s.n + aux_f);
              }
            }
            ++ord;
          }
        }
        it.next(s);
      }
    }
  } else if (warp == 1) {
    // ============================================================ MMA issuer (one elected lane; pair mode: leader only)
    if (kPair && rank != 0) {
      if (elect_one()) {      // the leader's MMAs read this CTA's weight halves as well: report them landed
        mbar_wait(smem_u32(&misc->w_full), 0, 4);
        mbar_arrive_cluster(mapa_shared(smem_u32(&misc->peer_w), 0));
      }
    } else if (elect_one()) {
      const uint32_t idesc0 = umma_idesc_bf16(kPair ? 256 : 128, 0);    // N field added per MMA
      const uint32_t idesc_step = ((uint32_t)tap_n >> 3) << 17;         // one dy sub-block of N
      const uint32_t w_lo = umma_desc_lo(w_smem);
      const uint32_t dxb = (uint32_t)dx_block_bytes >> 4;      // descriptor units per dx block
      const uint32_t sbb = (uint32_t)(tap_n * 128) >> 4;       // ... per dy sub-block
      const uint32_t aux_w_lo = w_lo + 3 * dxb;                 // LR im2col block (aux) ...
      const uint32_t aux_a_hi = p.aux_pitch64 ? kDescHiSw64 : kDescHiSw128;   // 64-byte or 128-byte aux pixels
      const uint32_t par_w_lo = w_lo + 3 * dxb;                 // ... or the stacked 1x1 block (kPar)
      // pair mode: this CTA's halves -- N-split dx blocks at w_lo, per-sub-block-split blocks behind them
      const uint32_t u192 = dxb >> 1, u64 = sbb >> 1, w64_lo = w_lo + 3 * (dxb >> 1);
      mbar_wait(smem_u32(&misc->w_full), 0, 4);
      if (kPair) mbar_wait(smem_u32(&misc->peer_w), 0, 14);
      // One step = one in-image source row.  `StepCtx` carries everything the issue code needs, so
      // the barriers of step s+1 can be checked in the MIDDLE of step s: an already-complete
      // mbarrier wait costs ~200 cycles and the tensor pipe only rides out ~300 cycles of silence
      // from this thread (tools/umma_bench.cu, "steps" rows), so waits between steps would stall it.
      struct StepCtx {
        bool valid;
        int j, len, j_first;
        uint32_t ord0, sc, a_slot, a_phase;
      };
      SegIter seg_it(p, t_begin, t_end, rank);
      Segment seg = seg_it.valid() ? seg_it.get() : Segment{0, 0, 0, 0, 0, -1};
      Ring ar(s_a);
      StepCtx cur{seg_it.valid(), seg.j_first, seg.len, seg.j_first, 0u, 0u, ar.slot, ar.phase};
      auto advance = [&](StepCtx& c) {        // next step in program order (crosses segments)
        ar.advance();
        c.sc += 1;
        c.a_slot = ar.slot;
        c.a_phase = ar.phase;
        if (c.j < seg.j_last) {
          c.j += 1;
          return;
        }
        const uint32_t next_ord0 = c.ord0 + (uint32_t)seg.len;
        seg_it.next(seg);
        c.valid = seg_it.valid();
        if (c.valid) {
          seg = seg_it.get();
          c.j = seg.j_first;
          c.len = seg.len;
          c.j_first = seg.j_first;
          c.ord0 = next_ord0;
        }
      };
      auto ranges = [](const StepCtx& c, int& lo, int& cnt, int& old_cnt) {
        lo = max(c.j - 1, 0);
        const int hi = min(c.j + 1, c.len - 1);
        cnt = hi - lo + 1;
        const int new_from = (c.j == c.j_first) ? lo : c.j + 1;   // rows first touched in this step
        old_cnt = min(max(new_from - lo, 0), cnt);
      };
      const uint32_t go_step = smem_u32(&misc->go_step), go_par = smem_u32(&misc->go_par);
      bool pend = false;
      uint32_t pend_bar = 0;
      auto commit = [&](uint32_t bar) {
        if (kPair) umma2_commit(bar); else umma_commit(bar);
      };

      // MMAs of one (dx,k) over `cnt` consecutive accumulator slots starting at slot_lo.  kWrap: the
      // range may run over the end of the ring and is issued as two MMAs.  The two cases are separate
      // straight-line bodies selected by ONE branch per step: a predicated-off tcgen05.mma is not free
      // (measured: steps with 12 squashed second halves took ~1790 cycles, steps whose ranges really
      // wrap -- 24 executed MMAs -- only ~1570).
      auto mma_range = [&](auto wrap_tag, uint32_t slot_lo, int cnt, uint32_t a_lo, uint32_t b_lo, uint32_t acc) {
        constexpr bool kWrap = decltype(wrap_tag)::value;
        if constexpr (!kWrap) {
          umma_bf16_lo(tmem_base + slot_lo * tap_n, a_lo, kDescHiSw128, b_lo, kDescHiSw128, idesc0 + cnt * idesc_step, acc);
        } else {
          // the two halves of a wrapped window share the A tile: the second MMA takes it from the collector
          // (tools/umma_collect_bench.cu) instead of fetching its 4 KB from shared memory again
          const int n1 = min(cnt, kAccRing - (int)slot_lo);
          if (cnt > n1) {
            umma1_bf16_lo<1>(tmem_base + slot_lo * tap_n, a_lo, b_lo, idesc0 + n1 * idesc_step, acc);
            umma1_bf16_lo<3>(tmem_base, a_lo, b_lo + n1 * sbb, idesc0 + (cnt - n1) * idesc_step, acc);
          } else {
            umma_bf16_lo(tmem_base + slot_lo * tap_n, a_lo, kDescHiSw128, b_lo, kDescHiSw128, idesc0 + n1 * idesc_step, acc);
          }
        }
      };

      // the four 1x1 MMAs of output row `od` (source row descriptor a_row_) + their own commit
      bool ppend = false;
      uint32_t pp_arow = 0, pp_od = 0;
      auto issue_par = [&](uint32_t a_row_, uint32_t od) {
        // every reader warp (of both CTAs in pair mode) has pulled row od-1's region into registers
        const uint32_t readers = (p.par_split ? 4u : (uint32_t)kEpilogueWarps) * (kPair ? 2u : 1u);
        if (kPair) {
          uint32_t spins = 0;
          while (ld_volatile_shared(go_par) < readers * od) {
            if (++spins > PNP_SPIN_LIMIT) {
              printf("pnp: flag wait timed out (tag 10, block %d, target %u)\n", (int)blockIdx.x, readers * od);
              __trap();
            }
          }
        } else {
          spin_until_ge(go_par, readers * od, 10);
        }
        tc_fence_after();
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          if (kPair)
            umma2_bf16_lo<0>(tmem_base + kParCol, a_row_ + 8 + 2 * k, par_w_lo + 2 * k, idesc0 + 3 * idesc_step, k > 0);
          else
            umma_bf16_lo(tmem_base + kParCol, a_row_ + 8 + 2 * k, kDescHiSw128, par_w_lo + 2 * k, kDescHiSw128,
                         idesc0 + 3 * idesc_step, k > 0);
        }
        commit(smem_u32(&misc->par_done));
      };

      // last value read from go_step: the scout usually runs several steps ahead (A ring depth, free
      // accumulator slots), so most steps need no shared-memory poll and no fence at all
      uint32_t go_seen = 0;
      const bool dbg_nopoll = PNP_DBG(8), dbg_nofence = PNP_DBG(16);
      if (cur.valid) go_seen = spin_until_ge_v(go_step, 1, 5);
      tc_fence_after();
      while (cur.valid) {
        const bool tr = PNP_TRACING && blockIdx.x == 0 && cur.sc < 64 && !PNP_DBG(128);
        if (tr) p.trace[cur.sc * 8 + 0] = clock64();
        int lo, cnt, old_cnt;
        ranges(cur, lo, cnt, old_cnt);
        const int new_cnt = cnt - old_cnt;
        const bool centre = (cur.j >= 0 && cur.j < cur.len);
        const uint32_t slot_lo = (cur.ord0 + lo) % kAccRing;
        const uint32_t a_row = umma_desc_lo(a_smem + cur.a_slot * kASlotBytes);
        const uint32_t sb_lo = (uint32_t)(lo - (cur.j - 1));                 // first dy sub-block in range
        const uint32_t b_row = w_lo + sb_lo * sbb;
        const uint32_t cur_sc = cur.sc;
        const uint32_t cur_od = cur.ord0 + (uint32_t)max(cur.j, 0);
        StepCtx nxt = cur;
        advance(nxt);
        // `emit(dx, k)` issues the MMAs of one (dx, k) of this step; everything else a step does between them -- the
        // previous row's deferred 1x1 convs, the look-ahead at the next step's barriers, the previous step's deferred
        // commit -- is common to the single-CTA and the pair form
        auto step_body = [&](auto emit) {
#pragma unroll
          for (int dx = 0; dx < 3; ++dx) {
            if (kPar && dx == 1 && ppend) {       // previous row's 1x1 convs, behind this step's dx = 0 group
              issue_par(pp_arow, pp_od);
              ppend = false;
            }
            if (tr && dx == 1) p.trace[cur_sc * 8 + 6] = clock64();
            if (dx == 2) {
              // barriers of the NEXT step, checked while ~8 MMAs of this step are still queued
              if (tr) p.trace[cur_sc * 8 + 7] = clock64();
              if (nxt.valid && go_seen < nxt.sc + 1 && !dbg_nopoll) {
                go_seen = spin_until_ge_v(go_step, nxt.sc + 1, 5);
                if (!dbg_nofence) tc_fence_after();
              }
              if (tr) p.trace[cur_sc * 8 + 2] = clock64();   // (slot 2 is otherwise the epilogue's)
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              emit(dx, k);
              if (dx == 0 && k == 0 && pend) {
                // the previous step's commit rides behind this step's first MMA
                commit(pend_bar);
                pend = false;
              }
              if (tr) p.trace[1024 + cur_sc * 16 + dx * 4 + k] = clock64();
            }
          }
        };
        if constexpr (kPair) {
          // Whole window (3 rows, not wrapping): ONE N = 3*tap_n MMA per (dx, k) out of the N-split blocks.  Otherwise,
          // and always for the first MMA of a step (its rows take different accumulate flags: rows touched before
          // accumulate, new rows are overwritten): one N = tap_n MMA per row out of the per-sub-block-split blocks,
          // chained through the A collector so that the A tile is fetched from shared memory once.
          uint32_t dcol[3];
#pragma unroll
          for (int i = 0; i < 3; ++i) {
            uint32_t sl = slot_lo + (uint32_t)i;
            if (sl >= (uint32_t)kAccRing) sl -= (uint32_t)kAccRing;
            dcol[i] = tmem_base + sl * tap_n;
          }
          const uint32_t idesc_sb = idesc0 + idesc_step, idesc_win = idesc0 + 3 * idesc_step;
          auto rows = [&](auto cnt_tag, int dx, int k, uint32_t a_lo, bool first) {
            constexpr int kCnt = decltype(cnt_tag)::value;
            const uint32_t b0 = w64_lo + ((uint32_t)dx * 3 + sb_lo) * u64 + 2 * k;
            const uint32_t acc0 = first ? (old_cnt > 0) : 1u, acc1 = first ? (old_cnt > 1) : 1u,
                           acc2 = first ? (old_cnt > 2) : 1u;
            if constexpr (kCnt == 1) {
              umma2_bf16_lo<0>(dcol[0], a_lo, b0, idesc_sb, acc0);
            } else if constexpr (kCnt == 2) {
              umma2_bf16_lo<1>(dcol[0], a_lo, b0, idesc_sb, acc0);
              umma2_bf16_lo<3>(dcol[1], a_lo, b0 + u64, idesc_sb, acc1);
            } else {
              umma2_bf16_lo<1>(dcol[0], a_lo, b0, idesc_sb, acc0);
              umma2_bf16_lo<2>(dcol[1], a_lo, b0 + u64, idesc_sb, acc1);
              umma2_bf16_lo<3>(dcol[2], a_lo, b0 + 2 * u64, idesc_sb, acc2);
            }
          };
          if (cnt == 3 && slot_lo + 3u <= (uint32_t)kAccRing) {
            step_body([&](int dx, int k) {
              const uint32_t a_lo = a_row + dx * 8 + 2 * k;
              if (dx == 0 && k == 0) rows(std::integral_constant<int, 3>{}, dx, k, a_lo, true);
              else umma2_bf16_lo<0>(dcol[0], a_lo, w_lo + (uint32_t)dx * u192 + 2 * k, idesc_win, 1);
            });
          } else if (cnt == 3) {
            step_body([&](int dx, int k) {
              rows(std::integral_constant<int, 3>{}, dx, k, a_row + dx * 8 + 2 * k, dx == 0 && k == 0);
            });
          } else if (cnt == 2) {
            step_body([&](int dx, int k) {
              rows(std::integral_constant<int, 2>{}, dx, k, a_row + dx * 8 + 2 * k, dx == 0 && k == 0);
            });
          } else {
            step_body([&](int dx, int k) {
              rows(std::integral_constant<int, 1>{}, dx, k, a_row + dx * 8 + 2 * k, dx == 0 && k == 0);
            });
          }
        } else {
          auto emit1 = [&](auto wrap_tag, int dx, int k) {
            const uint32_t a_lo = a_row + dx * 8 + 2 * k;
            const uint32_t b_lo = b_row + dx * dxb + 2 * k;
            if (dx == 0 && k == 0) {
              // first MMA of the step: rows touched before accumulate, new rows are overwritten
              if (old_cnt > 0) mma_range(wrap_tag, slot_lo, old_cnt, a_lo, b_lo, 1);
              if (new_cnt > 0)
                mma_range(wrap_tag, (slot_lo + old_cnt) % kAccRing, new_cnt, a_lo, b_lo + old_cnt * sbb, 0);
            } else {
              mma_range(wrap_tag, slot_lo, cnt, a_lo, b_lo, 1);
            }
          };
          if (slot_lo + (uint32_t)cnt > (uint32_t)kAccRing)
            step_body([&](int dx, int k) { emit1(std::true_type{}, dx, k); });
          else
            step_body([&](int dx, int k) { emit1(std::false_type{}, dx, k); });
        }
        if (p.aux_k16 > 0 && centre) {
          const uint32_t a_lo = umma_desc_lo(aux_smem + (cur_od & 1) * kTileBytes);
          for (int k = 0; k < p.aux_k16; ++k) {
            if (kPair)
              umma2_bf16_lo<0>(tmem_base + (cur_od % kAccRing) * tap_n, a_lo + 2 * k, aux_w_lo + 2 * k,
                               idesc0 + idesc_step, 1);
            else
              umma_bf16_lo(tmem_base + (cur_od % kAccRing) * tap_n, a_lo + 2 * k, aux_a_hi,
                           aux_w_lo + 2 * k, kDescHiSw128, idesc0 + idesc_step, 1);
          }
        }
        if (kPar && centre) {
          // Partition 1x1 convs of this row: centre pixel column (dx index 1), N = 192, own TMEM region.
          // Issued at the end of their own step.  Deferring them behind the dx = 0 group of the NEXT step (debug
          // bit 1024: the wait for the region then comes a third of a step later) measured no difference once the
          // region had its own reader warps (73.9 us either way): the step is bound by shared-memory wavefronts.
          if (par_defer) {
            ppend = true;
            pp_arow = a_row;
            pp_od = cur_od;
          } else {
            issue_par(a_row, cur_od);
          }
        }
        pend = true;
        pend_bar = smem_u32(&misc->step_done[cur_sc & (kStepRing - 1)]);
        if (tr) p.trace[cur_sc * 8 + 1] = clock64();
        cur = nxt;
      }
      if (kPar && ppend) issue_par(pp_arow, pp_od);      // the last row's 1x1 convs
      if (pend) commit(pend_bar);
    }
  } else if (warp == 10) {
    // ============================================================ barrier scout (one elected lane)
    // Walks the same step sequence as the MMA thread, one or more steps ahead, performs every
    // mbarrier wait the MMAs depend on (an already-complete try_wait costs 220-290 cycles in this
    // kernel) and publishes plain progress counters the MMA thread can poll in ~30 cycles.
    // Pair mode: the leader's scout alone -- its barriers collect both CTAs' loads and accumulator releases.
    if ((!kPair || rank == 0) && elect_one()) {
      const uint32_t go_step = smem_u32(&misc->go_step);
      Ring ar(s_a);
      uint32_t sc = 0, ord0 = 0;
      for (SegIter it(p, t_begin, t_end, rank); it.valid();) {
        const Segment s = it.get();
        for (int j = s.j_first; j <= s.j_last; ++j, ++sc, ar.advance()) {
          const bool trs = PNP_TRACING && blockIdx.x == 0 && sc < 64;
          if (trs) p.trace[2560 + sc * 4 + 0] = clock64();
          mbar_wait(smem_u32(&misc->a_full[ar.slot]), ar.phase, 5);
          if (trs) p.trace[2560 + sc * 4 + 1] = clock64();
          const int lo = max(j - 1, 0), hi = min(j + 1, s.len - 1);
          const int new_from = (j == s.j_first) ? lo : j + 1;
          for (int o = max(new_from, lo); o <= hi; ++o) {          // rows first touched in this step
            const uint32_t od = ord0 + o;
            mbar_wait(smem_u32(&misc->acc_free[od % kAccRing]), ((od / kAccRing) & 1) ^ 1, 6);
          }
          const bool centre = (j >= 0 && j < s.len);
          if (p.aux_k16 > 0 && centre) {
            const uint32_t od = ord0 + j;
            mbar_wait(smem_u32(&misc->aux_full[od & 1]), (od >> 1) & 1, 7);
          }
          st_release_shared(go_step, sc + 1);
          if (trs) p.trace[2560 + sc * 4 + 2] = clock64();
        }
        ord0 += s.len;
        it.next(s);
      }
    }
  } else if (warp >= 11 && !(kPar && p.par_split)) {
    // (block launch A with the single-role epilogue: the region-reader warps have nothing to do)
  } else {
    // ============================================================ epilogue (8 warps, 256 threads; + 4 region readers)
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;          // warps 2..9 only
    const int row = q * 32 + lane;
    const bool store_warp = (warp == 2);
    const uint32_t sw = (uint32_t)(row & 7);
    const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
    // non-partition variants keep the per-channel constants of this warp's 32 channels in registers;
    // the partition variant needs those registers for the 1x1 blend and re-reads them as float4
    // non-partition variants keep the per-channel constants of this warp's 32 channels in registers;
    // the partition variant is short of registers (1x1 blend) and re-reads them as float4
    float bias_r[kPar ? 1 : 32], scale_r[(kScale && !kPar) ? 32 : 1];
    if (!kPar) {
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        bias_r[j] = misc->bias[half * 32 + j];
        if (kScale) scale_r[j] = misc->scale[half * 32 + j];
      }
    }

    // flat cursor over this CTA's output rows (copyable: the partition path looks one row ahead)
    struct TileCur {
      SegIter it;
      Segment s;
      int o;
      uint32_t ord, sc0;
      bool valid;
    };
    TileCur cur{SegIter(p, t_begin, t_end, rank), Segment{0, 0, 0, 0, 0, -1}, 0, 0u, 0u, false};
    cur.valid = cur.it.valid();
    if (cur.valid) cur.s = cur.it.get();
    // "this accumulator slot / the 1x1 region has been read": in pair mode both CTAs report to the leader
    const uint32_t acc_free0 = kPair ? mapa_shared(smem_u32(&misc->acc_free[0]), 0) : smem_u32(&misc->acc_free[0]);
    const uint32_t go_par_a = kPair ? mapa_shared(smem_u32(&misc->go_par), 0) : smem_u32(&misc->go_par);
    auto acc_release = [&](uint32_t slot) {
      __syncwarp();
      if (lane == 0) {
        if (kPair) mbar_arrive_cluster(acc_free0 + slot * 8);
        else mbar_arrive(acc_free0 + slot * 8);
      }
    };
    auto par_release = [&]() {
      __syncwarp();
      if (lane == 0) {
        if (kPair) red_add_cluster(go_par_a);
        else asm volatile("red.relaxed.cta.shared::cta.add.u32 [%0], 1;" ::"r"(go_par_a) : "memory");
      }
    };
    // pair mode, odd number of (image, strip) columns: the last pair's second CTA walks a column that does not exist
    // (n == N).  Its loads may hit whatever follows in the pool, its results are never stored.
    auto phantom = [&](const Segment& sg) { return kPair && sg.n >= p.N; };
    auto tile_next = [](TileCur& c) {
      ++c.ord;
      if (++c.o < c.s.len) return;
      c.sc0 += (uint32_t)(c.s.j_last - c.s.j_first + 1);
      c.it.next(c.s);
      c.valid = c.it.valid();
      c.o = 0;
      if (c.valid) c.s = c.it.get();
    };

    // sum_k par_k * conv1x1_k(x) of a row: read the 3 x 32 columns of this warp's channel half from the
    // partition accumulators, blend with the pixel's partition values and park the result (bf16) in the
    // row's output staging slot -- in exactly the bytes this thread overwrites with the final value one
    // row later, so no register state is carried from row to row and no other thread is involved.
    auto blend_store = [&](uint8_t* slot_row, float q0, float q1, float q2) {
      // (the values were prefetched rows ago; they are first touched here, behind the barrier wait)
      if (p.par_sparse) par_sparse_select(q0, q1, q2);   // 1/255 for the surviving class, 0 for the others
#pragma unroll
      for (int gg = 0; gg < 2; ++gg) {
        float a1[16], a2[16], a3[16];
        const uint32_t col = kParCol + half * 32 + gg * 16;
        tmem_ld16(lane_base + col, a1);
        tmem_ld16(lane_base + col + 64, a2);
        tmem_ld16(lane_base + col + 128, a3);
        tmem_ld_wait();
        uint32_t w[8];
#pragma unroll
        for (int j = 0; j < 8; ++j)
          w[j] = pack_bf16x2(fmaf(q2, a3[2 * j], fmaf(q1, a2[2 * j], q0 * a1[2 * j])),
                             fmaf(q2, a3[2 * j + 1], fmaf(q1, a2[2 * j + 1], q0 * a1[2 * j + 1])));
        const int g = half * 2 + gg;
        *reinterpret_cast<uint4*>(slot_row + (((2 * g) ^ sw) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
        *reinterpret_cast<uint4*>(slot_row + (((2 * g + 1) ^ sw) << 4)) = make_uint4(w[4], w[5], w[6], w[7]);
      }
    };
    auto par_load = [&](const TileCur& c, float& q0, float& q1, float& q2) {
      const int x = c.s.strip * kTilePx + row;
      q0 = q1 = q2 = 0.f;
      if (x < p.W && !phantom(c.s)) {
        const float* pp = par_g + (long long)c.s.n * p.par_sn + (long long)PNP_Y(c.s.y_b + c.o) * p.par_sy + x;
        q0 = __ldg(pp);
        q1 = __ldg(pp + p.par_sc);
        q2 = __ldg(pp + 2 * p.par_sc);
      }
    };
    // ---------------------------------------------------------------------------------------------------
    // Split roles (kPar, p.par_split): warps 6..9 do nothing but drain the single 1x1 accumulator region --
    // wait for par_done, pull the 192 columns of their lane quarter into registers, hand the region back, blend
    // and park the result in the row's staging slot -- while warps 2..5 finish rows (all 64 channels of their 32
    // pixels).  The region's hand-back loop (commit -> reader -> release -> next 1x1 MMAs) then no longer
    // contains the main epilogue's loop top, store bookkeeping and row arithmetic.
    // ---------------------------------------------------------------------------------------------------
    if (kPar && p.par_split) {
      const uint32_t slot_free = smem_u32(&misc->slot_free);
      if (warp >= 11) {
        float pn0 = 0.f, pn1 = 0.f, pn2 = 0.f;
        if (cur.valid) par_load(cur, pn0, pn1, pn2);
        Ring sl(n_io);
        while (cur.valid) {
          TileCur nxt = cur;
          tile_next(nxt);
          float pf0 = 0.f, pf1 = 0.f, pf2 = 0.f;
          if (nxt.valid) par_load(nxt, pf0, pf1, pf2);      // one row ahead: consumed a whole step later
          const bool trr = PNP_TRACING && blockIdx.x == 0 && cur.ord < 64 && warp == 11 && lane == 0;
          if (trr) p.trace[3072 + cur.ord * 4 + 0] = clock64();
          mbar_wait(smem_u32(&misc->par_done), cur.ord & 1, 11);   // (one poller per warp measured no better)
          if (trr) p.trace[3072 + cur.ord * 4 + 1] = clock64();
          tc_fence_after();
          if (p.par_sparse) par_sparse_select(pn0, pn1, pn2);
          uint32_t wv[32];
          // four batches of 16 channels x 3 classes (48 values in flight: the 480-thread block leaves 128 registers)
#pragma unroll
          for (int b4 = 0; b4 < 4; ++b4) {
            float a1[16], a2[16], a3[16];
            const uint32_t col = kParCol + b4 * 16;
            tmem_ld16(lane_base + col, a1);
            tmem_ld16(lane_base + col + 64, a2);
            tmem_ld16(lane_base + col + 128, a3);
            tmem_ld_wait();
            if (b4 == 3) {                                   // everything is in registers: hand the region back first
              tc_fence_before();
              par_release();
              if (trr) p.trace[3072 + cur.ord * 4 + 2] = clock64();
            }
#pragma unroll
            for (int j = 0; j < 8; ++j)
              wv[b4 * 8 + j] = pack_bf16x2(fmaf(pn2, a3[2 * j], fmaf(pn1, a2[2 * j], pn0 * a1[2 * j])),
                                           fmaf(pn2, a3[2 * j + 1], fmaf(pn1, a2[2 * j + 1], pn0 * a1[2 * j + 1])));
          }
          // the row's staging slot was last used by row ord - n_io: its TMA store must have finished reading
          if (cur.ord >= (uint32_t)n_io) spin_until_ge(slot_free, cur.ord - (uint32_t)n_io + 1, 12);
          uint8_t* rowp = sgen + L.io + sl.slot * kTileBytes + row * 128;
#pragma unroll
          for (int c8 = 0; c8 < 8; ++c8)
            *reinterpret_cast<uint4*>(rowp + ((c8 ^ sw) << 4)) =
                make_uint4(wv[4 * c8], wv[4 * c8 + 1], wv[4 * c8 + 2], wv[4 * c8 + 3]);
          warp_arrive(smem_u32(&misc->dy_full[sl.slot]));    // release: the parked values are visible to warps 2..5
          if (trr) p.trace[3072 + cur.ord * 4 + 3] = clock64();
          sl.advance();
          pn0 = pf0;
          pn1 = pf1;
          pn2 = pf2;
          cur = nxt;
        }
      } else {
        Ring ior(n_io);
        while (cur.valid) {
          const Segment& s = cur.s;
          const uint32_t ord = cur.ord;
          const int y = PNP_Y(s.y_b + cur.o);
          const uint32_t sc_last = cur.sc0 + (uint32_t)(min(cur.o + 1, s.j_last) - s.j_first);
          const uint32_t slot = ord % kAccRing;
          const uint32_t taddr = lane_base + slot * tap_n;
          if (store_warp) {
            if (elect_one()) {
              tma_store_wait_read<1>();                      // stores of rows <= ord-2 no longer read shared memory
              if (ord >= 1) st_release_shared(slot_free, ord - 1);
            }
            __syncwarp();
          }
          const bool trm = PNP_TRACING && blockIdx.x == 0 && ord < 64 && warp == 2 && lane == 0;
          if (trm) p.trace[2816 + ord * 4 + 0] = clock64();
          slow_epilogue();
          mbar_wait(smem_u32(&misc->step_done[sc_last & (kStepRing - 1)]), (sc_last >> kStepShift) & 1, 9);
          if (trm) p.trace[2816 + ord * 4 + 1] = clock64();
          tc_fence_after();
          float v[32];                                       // this warp's 32 channels of its 32 pixels
          tmem_ld16(taddr + half * 32, v);
          tmem_ld16(taddr + half * 32 + 16, v + 16);
          tmem_ld_wait();
          tc_fence_before();
          acc_release(slot);                                 // accumulator is in registers: slot reusable
          if (trm) p.trace[2816 + ord * 4 + 2] = clock64();
          mbar_wait(smem_u32(&misc->dy_full[ior.slot]), ior.phase, 13);
          if (trm) p.trace[2816 + ord * 4 + 3] = clock64();
          uint8_t* rowp = sgen + L.io + ior.slot * kTileBytes + row * 128;
#pragma unroll
          for (int gg = 0; gg < 2; ++gg) {
            const int g = half * 2 + gg;
            float* vv = v + gg * 16;
            const float4* sc4 = reinterpret_cast<const float4*>(&misc->scale[g * 16]);
            const float4* bi4 = reinterpret_cast<const float4*>(&misc->bias[g * 16]);
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
              const float4 sc = kScale ? sc4[j4] : make_float4(1.f, 1.f, 1.f, 1.f);
              const float4 bi = bi4[j4];
              vv[4 * j4 + 0] = fmaf(vv[4 * j4 + 0], sc.x, bi.x);
              vv[4 * j4 + 1] = fmaf(vv[4 * j4 + 1], sc.y, bi.y);
              vv[4 * j4 + 2] = fmaf(vv[4 * j4 + 2], sc.z, bi.z);
              vv[4 * j4 + 3] = fmaf(vv[4 * j4 + 3], sc.w, bi.w);
            }
            uint4* c0 = reinterpret_cast<uint4*>(rowp + (((2 * g) ^ sw) << 4));
            uint4* c1 = reinterpret_cast<uint4*>(rowp + (((2 * g + 1) ^ sw) << 4));
            const uint4 i0 = *c0, i1 = *c1;                  // the row's parked 1x1 blend
            const uint32_t iw[8] = {i0.x, i0.y, i0.z, i0.w, i1.x, i1.y, i1.z, i1.w};
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              vv[2 * j] += bf16_lo(iw[j]);
              vv[2 * j + 1] += bf16_hi(iw[j]);
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) vv[j] = act_fn(vv[j], p.act);
            *c0 = make_uint4(pack_bf16x2(vv[0], vv[1]), pack_bf16x2(vv[2], vv[3]), pack_bf16x2(vv[4], vv[5]),
                             pack_bf16x2(vv[6], vv[7]));
            *c1 = make_uint4(pack_bf16x2(vv[8], vv[9]), pack_bf16x2(vv[10], vv[11]), pack_bf16x2(vv[12], vv[13]),
                             pack_bf16x2(vv[14], vv[15]));
          }
          fence_proxy_async_smem();
          named_bar_sync(2, 256);
          if (store_warp) {
            if (elect_one()) {
              if (!phantom(s)) {
                if (p.l2_out)
                  tma_store_4d_hint(&p.tm_out, io_smem + ior.slot * kTileBytes, 0, s.strip * kTilePx, y, s.n + out_f,
                                    p.l2_out == 2 ? l2_policy_evict_last() : l2_policy_evict_first());
                else
                  tma_store_4d(&p.tm_out, io_smem + ior.slot * kTileBytes, 0, s.strip * kTilePx, y, s.n + out_f);
              }
              tma_store_commit();
            }
            __syncwarp();
          }
          ior.advance();
          tile_next(cur);
        }
        if (store_warp) {
          if (elect_one()) tma_store_wait_all<0>();
          __syncwarp();
        }
      }
    } else {
    // partition values are fetched TWO rows ahead: the epilogue is the hand-back path of the single 1x1
    // accumulator region, so a global-load latency per row (measured: 1300-2400 cycles of "math") would
    // bound the whole pipeline.  pn* = values of the row after `cur`, loaded one iteration earlier.
    float pn0 = 0.f, pn1 = 0.f, pn2 = 0.f;
    if (kPar && cur.valid) {                 // first row of this CTA: staging slot 0 is free
      float q0, q1, q2;
      par_load(cur, q0, q1, q2);
      {
        TileCur n1 = cur;
        tile_next(n1);
        if (n1.valid) par_load(n1, pn0, pn1, pn2);
      }
      ewait(smem_u32(&misc->par_done), cur.ord & 1, 11);
      tc_fence_after();
      blend_store(sgen + L.io + row * 128, q0, q1, q2);
      tc_fence_before();
      par_release();
    }

    // Identity tiles are fetched by the epilogue's own store lane: it is the one who knows when a
    // staging slot has been drained (wait_group.read), so the TMA producer never blocks on them and
    // keeps its source rows s_a-1 steps ahead.  `idc` runs n_io-2 output rows ahead of `cur`.
    TileCur idc = cur;
    Ring idr(n_io);
    auto load_id = [&](const TileCur& c, uint32_t slot) {
      const uint32_t ib = smem_u32(&misc->id_full[slot]);
      mbar_arrive_expect_tx(ib, kTileBytes);
      if (p.l2_idt)
        tma_load_4d_hint(io_smem + slot * kTileBytes, &p.tm_id, ib, 0, c.s.strip * kTilePx, PNP_Y(c.s.y_b + c.o), c.s.n + idt_f,
                         p.l2_idt == 2 ? l2_policy_evict_last() : l2_policy_evict_first());
      else
        tma_load_4d(io_smem + slot * kTileBytes, &p.tm_id, ib, 0, c.s.strip * kTilePx, PNP_Y(c.s.y_b + c.o), c.s.n + idt_f);
    };
    if (p.has_id && store_warp) {
      if (elect_one()) {
        for (int i = 0; i < n_io && idc.valid; ++i) {     // all slots start out free
          load_id(idc, idr.slot);
          idr.advance();
          tile_next(idc);
        }
      }
      __syncwarp();
    }

    // kModeLast: `+ lq` (or its x4 bilinear upsampling) of the pixel this thread finishes in row `c`
    auto lq_fetch = [&](const TileCur& c, float* r) {
      r[0] = r[1] = r[2] = 0.f;
      if (!c.valid || half != 0) return;
      const int x = c.s.strip * kTilePx + row;
      const int y = PNP_Y(c.s.y_b + c.o);
      if (x >= p.W) return;
      if (p.lq_up4) {
        // base = nn.Upsample(scale_factor=4, mode='bilinear', align_corners=False)(lr), iconvsr_ipb_par.py:41,
        // 140-141, fused: ATen's source index scale*(dst+0.5)-0.5 clamped at 0, i1 = i0 + (i0 < size-1),
        // lambda1 = src - i0, row blend of the two column blends
        const int hl = p.H >> 2, wl = p.W >> 2;
        const float sy = fmaxf(0.25f * ((float)y + 0.5f) - 0.5f, 0.f), sx = fmaxf(0.25f * ((float)x + 0.5f) - 0.5f, 0.f);
        const int y0 = (int)sy, x0 = (int)sx;
        const int y1 = y0 + (y0 < hl - 1 ? 1 : 0), x1 = x0 + (x0 < wl - 1 ? 1 : 0);
        const float ly1 = sy - (float)y0, lx1 = sx - (float)x0;
        const float ly0 = 1.f - ly1, lx0 = 1.f - lx1;
        const float* b0 = lq_g + (long long)c.s.n * p.lq_sn + (long long)y0 * p.lq_sy;
        const float* b1 = lq_g + (long long)c.s.n * p.lq_sn + (long long)y1 * p.lq_sy;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
          const float* c0 = b0 + ch * p.lq_sc;
          const float* c1 = b1 + ch * p.lq_sc;
          r[ch] = ly0 * (lx0 * __ldg(c0 + x0) + lx1 * __ldg(c0 + x1)) + ly1 * (lx0 * __ldg(c1 + x0) + lx1 * __ldg(c1 + x1));
        }
      } else {
        const float* lp = lq_g + (long long)c.s.n * p.lq_sn + (long long)y * p.lq_sy + x;
        r[0] = __ldg(lp);
        r[1] = __ldg(lp + p.lq_sc);
        r[2] = __ldg(lp + 2 * p.lq_sc);
      }
    };
    float lq_a[3] = {0.f, 0.f, 0.f}, lq_b[3] = {0.f, 0.f, 0.f};
    if (last_mode) {
      lq_fetch(cur, lq_a);
      TileCur n1 = cur;
      if (n1.valid) tile_next(n1);
      lq_fetch(n1, lq_b);
    }

    Ring ior(n_io);
    while (cur.valid) {
      slow_epilogue();
      const Segment& s = cur.s;
      const int o = cur.o;
      const uint32_t ord = cur.ord;
      const int x = s.strip * kTilePx + row;
      const bool valid = x < p.W;
      const int y = PNP_Y(s.y_b + o);
      const uint32_t sc_last = cur.sc0 + (uint32_t)(min(o + 1, s.j_last) - s.j_first);
      const uint32_t slot = ord % kAccRing;
      const uint32_t taddr = lane_base + slot * tap_n;
      TileCur nxt = cur;
      tile_next(nxt);
      if (last_mode) {
        // lq values are fetched TWO rows ahead (lq_a: this row, lq_b: the next one): a row of this N=48 conv is only
        // ~500 MMA cycles, so a global-load latency inside the row's own iteration was the bound of the whole kernel
        // (46.5 us at 720p for 141 MB of traffic)
        const float r0 = lq_a[0], r1 = lq_a[1], r2 = lq_a[2];
        {
          TileCur n2 = nxt;
          if (n2.valid) tile_next(n2);
          lq_a[0] = lq_b[0];
          lq_a[1] = lq_b[1];
          lq_a[2] = lq_b[2];
          lq_fetch(n2, lq_b);
        }
        ewait(smem_u32(&misc->step_done[sc_last & (kStepRing - 1)]), (sc_last >> kStepShift) & 1, 9);
        tc_fence_after();
        float v[16];
        if (half == 0) {
          tmem_ld16(taddr, v);
          tmem_ld_wait();
        }
        tc_fence_before();
        acc_release(slot);
        if (valid && half == 0) {
          const long long o_off = (long long)s.n * p.of_sn + (long long)y * p.of_sy + x;
          const float o0 = v[0] + misc->bias[0] + r0, o1 = v[1] + misc->bias[1] + r1, o2 = v[2] + misc->bias[2] + r2;
          // the same fp32 sums, stored as tensor2img's uint8 values (kModeLast never has a partition operand: the kPar
          // instances leave the branch out)
          if (!kPar && p.out_u8) {
            uint8_t* op = reinterpret_cast<uint8_t*>(outf_g) + o_off;
            op[0] = (uint8_t)quant_u8(o0);
            op[p.of_sc] = (uint8_t)quant_u8(o1);
            op[2 * p.of_sc] = (uint8_t)quant_u8(o2);
          } else {
            float* op = outf_g + o_off;
            op[0] = o0;
            op[p.of_sc] = o1;
            op[2 * p.of_sc] = o2;
          }
        }
        cur = nxt;
        continue;
      }
      const bool tr = PNP_TRACING && blockIdx.x == 0 && ord < 64 && threadIdx.x == 64 && !PNP_DBG(128);
      // Partition path: the 1x1 accumulators of the NEXT row finish with the same step that completes
      // this row's 3x3 result (they are issued last in that step), so both are fetched from TMEM in
      // one batch behind one barrier wait; the blend of the next row is parked in its staging slot.
      float pf0 = 0.f, pf1 = 0.f, pf2 = 0.f;   // partition values of the row after next
      if (kPar && nxt.valid) {
        TileCur n2 = nxt;
        tile_next(n2);
        if (n2.valid) par_load(n2, pf0, pf1, pf2);
      }
      const uint32_t s_io = ior.slot;
      if (store_warp) {
        if (elect_one()) {
          tma_store_wait_read<1>();      // stores of output rows <= ord-2 no longer read smem
          if (p.has_id && ord >= 2 && idc.valid) {
            load_id(idc, idr.slot);      // slot of row ord-2 == slot of row ord-2+n_io
            idr.advance();
            tile_next(idc);
          }
        }
        __syncwarp();
      }
      if (p.has_id) {
        ewait(smem_u32(&misc->id_full[s_io]), ior.phase, 8);
      } else {
        named_bar_sync(1, 256);
      }
      if (kPar && nxt.valid) {
        // par_done of the next row is committed right behind its four 1x1 MMAs, which are the LAST MMAs of
        // the step that also completes this row's 3x3 result (a commit covers everything issued before
        // it), whereas that step's own step_done commit is deferred into the following step
        ewait(smem_u32(&misc->par_done), (ord + 1) & 1, 11);
      } else {
        ewait(smem_u32(&misc->step_done[sc_last & (kStepRing - 1)]), (sc_last >> kStepShift) & 1, 9);
      }
      tc_fence_after();
      if (tr) p.trace[ord * 8 + 3] = clock64();
      uint8_t* rowp = sgen + L.io + s_io * kTileBytes + row * 128;
      float v[32];
      if (PNP_DBG(4)) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = 0.f;
      } else {
        tmem_ld16(taddr + half * 32, v);
        tmem_ld16(taddr + half * 32 + 16, v + 16);
        if (kPar && nxt.valid) {
          // the NEXT row's 1x1 results (complete with the same step): blend into the next staging slot,
          // which the store of row ord-2 has drained (wait_group.read<1> + named barrier 1 above, n_io >= 3)
          const uint32_t s_nx = (s_io + 1 == (uint32_t)n_io) ? 0u : s_io + 1;
          blend_store(sgen + L.io + s_nx * kTileBytes + row * 128, pn0, pn1, pn2);
        } else {
          tmem_ld_wait();
        }
      }
      tc_fence_before();
      acc_release(slot);                              // accumulator is in registers: slot reusable
      if (kPar && nxt.valid) par_release();           // ... and so is the 1x1 region
#pragma unroll
      for (int gg = 0; gg < 2; ++gg) {
        const int g = half * 2 + gg;
        float* vv = v + gg * 16;
        if (kPar) {
          const float4* sc4 = reinterpret_cast<const float4*>(&misc->scale[g * 16]);
          const float4* bi4 = reinterpret_cast<const float4*>(&misc->bias[g * 16]);
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4) {
            const float4 sc = kScale ? sc4[j4] : make_float4(1.f, 1.f, 1.f, 1.f);
            const float4 bi = bi4[j4];
            vv[4 * j4 + 0] = fmaf(vv[4 * j4 + 0], sc.x, bi.x);
            vv[4 * j4 + 1] = fmaf(vv[4 * j4 + 1], sc.y, bi.y);
            vv[4 * j4 + 2] = fmaf(vv[4 * j4 + 2], sc.z, bi.z);
            vv[4 * j4 + 3] = fmaf(vv[4 * j4 + 3], sc.w, bi.w);
          }
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j)
            vv[j] = kScale ? fmaf(vv[j], scale_r[gg * 16 + j], bias_r[gg * 16 + j]) : vv[j] + bias_r[gg * 16 + j];
        }
        uint4* c0 = reinterpret_cast<uint4*>(rowp + (((2 * g) ^ sw) << 4));
        uint4* c1 = reinterpret_cast<uint4*>(rowp + (((2 * g + 1) ^ sw) << 4));
        if (p.has_id || kPar) {              // identity tile (TMA) or this row's parked 1x1 blend
          const uint4 i0 = *c0, i1 = *c1;
          const uint32_t iw[8] = {i0.x, i0.y, i0.z, i0.w, i1.x, i1.y, i1.z, i1.w};
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            vv[2 * j] += bf16_lo(iw[j]);
            vv[2 * j + 1] += bf16_hi(iw[j]);
          }
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) vv[j] = act_fn(vv[j], p.act);
        uint4 o0, o1;
        o0.x = pack_bf16x2(vv[0], vv[1]);
        o0.y = pack_bf16x2(vv[2], vv[3]);
        o0.z = pack_bf16x2(vv[4], vv[5]);
        o0.w = pack_bf16x2(vv[6], vv[7]);
        o1.x = pack_bf16x2(vv[8], vv[9]);
        o1.y = pack_bf16x2(vv[10], vv[11]);
        o1.z = pack_bf16x2(vv[12], vv[13]);
        o1.w = pack_bf16x2(vv[14], vv[15]);
        if (!PNP_DBG(2)) {
          *c0 = o0;
          *c1 = o1;
        }
      }
      if (tr) p.trace[ord * 8 + 4] = clock64();
      fence_proxy_async_smem();
      named_bar_sync(2, 256);
      if (tr) p.trace[ord * 8 + 5] = clock64();
      if (store_warp) {
        if (elect_one()) {
          if (!PNP_DBG(2)) {
            if (!phantom(s)) {
              if (p.l2_out)
                tma_store_4d_hint(&p.tm_out, io_smem + s_io * kTileBytes, 0, s.strip * kTilePx, y, s.n + out_f,
                                  p.l2_out == 2 ? l2_policy_evict_last() : l2_policy_evict_first());
              else
                tma_store_4d(&p.tm_out, io_smem + s_io * kTileBytes, 0, s.strip * kTilePx, y, s.n + out_f);
            }
            tma_store_commit();
          }
        }
        __syncwarp();
      }
      ior.advance();
      if (kPar) {
        pn0 = pf0;
        pn1 = pf1;
        pn2 = pf2;
      }
      cur = nxt;
    }
    if (store_warp) {
      if (elect_one()) tma_store_wait_all<0>();
      __syncwarp();
    }
    }   // !(kPar && p.par_split)
  }

  tc_fence_before();
  // pair mode: neither CTA may leave (or free its TMEM) while the other one's MMAs / arrivals can still reach it
  if (kPair) cluster_sync_all(); else __syncthreads();
  if (PNP_TRACING && threadIdx.x == 0) {            // per-CTA body cycles, start and end time (ns)
    p.trace[2048 + blockIdx.x] += clock64();
    p.trace[2368 + blockIdx.x] = (long long)globaltimer_ns();
  }
  if (warp == 0) {
    tc_fence_after();
    if (kPair) tmem_dealloc2(tmem_base, kTmemCols);
    else tmem_dealloc(tmem_base, kTmemCols);
  }
}

#undef PNP_Y

size_t conv_rows_smem_bytes(const ConvParams& p) {
  const int full = 3 * 3 * p.tap_n * 128;
  const int w_bytes = p.pair ? full + (p.aux_k16 > 0 ? kWChunkBytes / 2 : 0) + (p.has_par ? 3 * 64 * 128 / 2 : 0)
                             : full + (p.aux_k16 > 0 ? kWChunkBytes : 0) + (p.has_par ? 3 * 64 * 128 : 0);
  return rows_layout(w_bytes, p.s_a, p.aux_k16 > 0, p.n_io).total + 1024;
}

namespace {
constexpr int kMaxSmem = 232448;

template <bool kPar, bool kScale, bool kPair>
cudaError_t launch_rows_variant(const ConvParams& p, int grid, size_t smem, cudaStream_t stream) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kPar ? kRowsThreadsPar : kRowsThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (kPair) {
    attr[1].id = cudaLaunchAttributeClusterDimension;
    attr[1].val.clusterDim.x = 2;
    attr[1].val.clusterDim.y = 1;
    attr[1].val.clusterDim.z = 1;
    cfg.numAttrs = 2;
  }
  return cudaLaunchKernelEx(&cfg, conv3x3_rows_kernel<kPar, kScale, kPair>, p);
}
template <bool kPar, bool kScale, bool kPair>
cudaError_t prepare_variant(int* max_pairs) {
  cudaError_t e = cudaFuncSetAttribute(conv3x3_rows_kernel<kPar, kScale, kPair>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       kMaxSmem);
  if (e != cudaSuccess || !kPair) return e;
  // how many CTA pairs fit on the device at once (GPCs with an odd number of usable SMs leave one SM unpaired)
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * 148);
  cfg.blockDim = dim3(kPar ? kRowsThreadsPar : kRowsThreads);
  cfg.dynamicSmemBytes = kMaxSmem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int n = 0;
  e = cudaOccupancyMaxActiveClusters(&n, conv3x3_rows_kernel<kPar, kScale, kPair>, &cfg);
  if (e == cudaSuccess && n < *max_pairs) *max_pairs = n;
  return e;
}
}  // namespace

// once per device, before the first launch (and before any stream capture): the API layer calls it under call_once
cudaError_t conv_rows_prepare(int* max_pairs) {
  cudaError_t e;
  int pairs = 1 << 30;
  if ((e = prepare_variant<true, true, false>(&pairs)) != cudaSuccess) return e;
  if ((e = prepare_variant<true, false, false>(&pairs)) != cudaSuccess) return e;
  if ((e = prepare_variant<false, true, false>(&pairs)) != cudaSuccess) return e;
  if ((e = prepare_variant<false, false, false>(&pairs)) != cudaSuccess) return e;
  if ((e = prepare_variant<true, true, true>(&pairs)) != cudaSuccess) return e;
  if ((e = prepare_variant<true, false, true>(&pairs)) != cudaSuccess) return e;
  if ((e = prepare_variant<false, true, true>(&pairs)) != cudaSuccess) return e;
  if ((e = prepare_variant<false, false, true>(&pairs)) != cudaSuccess) return e;
  if (max_pairs) *max_pairs = pairs == (1 << 30) ? 0 : pairs;
  return cudaSuccess;
}

cudaError_t launch_conv_rows(const ConvParams& p, int grid, cudaStream_t stream) {
  const size_t smem = conv_rows_smem_bytes(p);
  const bool par = p.has_par != 0, scale = (p.scale != nullptr);
  if (p.pair) {
    if (par) return scale ? launch_rows_variant<true, true, true>(p, grid, smem, stream)
                          : launch_rows_variant<true, false, true>(p, grid, smem, stream);
    return scale ? launch_rows_variant<false, true, true>(p, grid, smem, stream)
                 : launch_rows_variant<false, false, true>(p, grid, smem, stream);
  }
  if (par) return scale ? launch_rows_variant<true, true, false>(p, grid, smem, stream)
                        : launch_rows_variant<true, false, false>(p, grid, smem, stream);
  return scale ? launch_rows_variant<false, true, false>(p, grid, smem, stream)
               : launch_rows_variant<false, false, false>(p, grid, smem, stream);
}

}  // namespace pnp
