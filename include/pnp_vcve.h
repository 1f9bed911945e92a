/*
 * pnp_vcve.h -- C ABI of libpnpvcve.so, the sm_100a kernels behind the BAE+CAA generator.
 *
 * The reference (ZeldaM1/PnP-VCVE) is pure Python/PyTorch and has no FFI of its own; every entry
 * point below replaces a group of library calls the reference makes on its hot path, cited as
 * reference file:line.  The Python class that mirrors the reference's registry interface
 * (pnpvcve_b200/backbone.py, same name / kwargs / state_dict as
 * mmedit/models/backbones/sr_backbones/iconvsr_ipb_par.py:16-44) binds these with ctypes; see
 * INTEGRATION.md for the stub a maintainer adds on the reference side.
 *
 * Conventions: plain pointers and sizes only (no torch types); all pointers are DEVICE pointers
 * unless stated; `stream` is a cudaStream_t passed as void*; nothing is allocated or retained by
 * the library (buffers, workspaces and packed weights are owned by the caller); every function
 * returns 0 on success or a negative pnp_status and never throws.  Kernels launch asynchronously
 * on `stream`.  sm_100a only: on any other device the calls return PNP_ERR_ARCH.
 */
#ifndef PNP_VCVE_H_
#define PNP_VCVE_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum pnp_status {
  PNP_OK = 0,
  PNP_ERR_ARG = -1,     /* null pointer / bad shape / misaligned pointer */
  PNP_ERR_ARCH = -2,    /* current device is not compute capability 10.x */
  PNP_ERR_CUDA = -3,    /* a CUDA runtime/driver call failed (see pnp_last_error) */
  PNP_ERR_RESOURCE = -4 /* shared-memory budget cannot be met */
} pnp_status;

/* Library / device info. */
int pnp_abi_version(void);
const char* pnp_last_error(void);          /* message of the last failing call in this thread */
int pnp_device_check(void);                /* PNP_OK iff the current device is sm_100 */
int pnp_set_pair_mode(int mode);           /* conv kernel form for later pnp_conv3x3 calls of this process: 0 single CTA,
                                              1 CTA pairs (tcgen05 cta_group::2) where the shape pairs up without waste,
                                              2 also with a phantom column, -1 follow the PNP_PAIR environment variable
                                              (default 0).  Same results either way.  Returns the previous setting. */
int pnp_device_pairs(void);                /* CTA pairs (clusters of two) the conv kernel's cta_group::2 form can keep
                                              resident on the current device; < 0: error code */

/*
 * Launch tables and CUDA graphs -- the launch-free frame loop.
 *
 * The reference's generator is a Python loop over frames that launches ~300 library kernels per frame
 * (mmedit/models/backbones/sr_backbones/iconvsr_ipb_par.py:71-147).  Here a frame step is a fixed sequence of
 * ~20-25 kernels whose operands differ from frame to frame only in a few pointers / image indices.  Those live in a
 * device-resident TABLE of 64-byte entries written once per clip; a kernel launched in table mode reads entry
 *     table[*step * stride + node]
 * so its kernel parameters are constant for the clip and the whole step can be captured ONCE in a CUDA graph and
 * replayed for every frame: per step the host sets the step word and launches one graph (pnp_graph_launch).
 * Entry layout by operation (unused fields are ignored):
 *   pnp_conv3x3  : p[0] wpack, p[1] bias, p[2] par, p[3] lq, p[4] outf, p[5] img_off (int64 pairs, see below) or 0;
 *                  i[0..3] first image of src / aux / idt / out inside the buffers the descriptor points to
 *   pnp_mv_warp  : p[1] flow_x, p[2] flow_y; i[0] / i[3] image of src / dst inside the call's src_pool
 *   pnp_lr_im2col: p[0] lr, p[1] dst
 */
typedef struct pnp_dyn_entry {
  uint64_t p[6];
  int32_t i[4];
} pnp_dyn_entry;

typedef struct pnp_dyn_ref {
  const pnp_dyn_entry* table; /* device memory; NULL = static launch (operands are the call's own arguments) */
  const int32_t* step;        /* device word holding the current step */
  int32_t node;               /* index of this launch inside its step */
  int32_t stride;             /* entries per step */
} pnp_dyn_ref;

/* Stream capture of the calls made between begin and end into an executable graph (thin wrappers over
 * cudaStreamBeginCapture / cudaStreamEndCapture / cudaGraphInstantiate; programmatic-dependent-launch edges between the
 * conv kernels are kept).  The graph handle is the only object this library ever owns; destroy it with
 * pnp_graph_destroy.  pnp_graph_launch first stores `step_value` into *step_word (stream ordered; NULL to skip) and
 * then launches the graph; pnp_set_step does only the store (for launching the same sequence without a graph). */
int pnp_graph_begin(void* stream);
int pnp_graph_end(void* stream, void** graph_exec);
int pnp_graph_launch(void* graph_exec, int32_t* step_word, int32_t step_value, void* stream);
int pnp_graph_destroy(void* graph_exec);
int pnp_set_step(int32_t* step_word, int32_t step_value, void* stream);
/* Stream-ordered copy of `bytes` (multiple of 16) from PAGE-LOCKED host memory into device memory by a kernel that
 * reads the host buffer over the bus -- for the launch table: a cudaMemcpyAsync would queue on the H2D copy engine
 * behind a clip that is being streamed in and hold back the first frame step for its whole upload. */
int pnp_fetch_pinned(void* dst, const void* src_pinned, int64_t bytes, void* stream);

/*
 * K1 -- MV-guided bilinear warp of a 64-channel feature map.
 * Replaces flow_warp (mmedit/models/common/flow_warp.py:6-50) as called by VOSAlignment.forward
 * (mmedit/models/backbones/sr_backbones/iconvsr_mv.py:17-18): grid_sample(bilinear, zeros,
 * align_corners=True) of x + mv, including the reference's fp32 normalise/un-normalise sequence.
 *   src, dst : bf16 NHWC (N, H, W, 64), 16-byte aligned, distinct buffers (N same-shape clips)
 *   flow_x/y : fp32 planes, element (n,y,x) at [n*flow_image_stride + y*flow_row_stride + x]
 *              (the (2,H,W) slices mvs[b0:b1, i, 2:4] or [.., 0:2] of the reference's `mvs`)
 *   dbg_x0/y0: optional int32 (H*W) outputs of the integer north-west tap (floor), N == 1 only
 */
int pnp_mv_warp(const void* src, const float* flow_x, const float* flow_y, int64_t flow_row_stride,
                int64_t flow_image_stride, void* dst, int N, int H, int W, int32_t* dbg_x0,
                int32_t* dbg_y0, void* stream);
/* table mode: the flow planes and the src / dst IMAGE INDICES inside the (src_pool_images, H, W, 64) buffer at src_pool
 * come from the launch table (no debug outputs): tap windows and output tiles move by TMA through tensor maps of that
 * buffer, built when the launch is recorded. */
int pnp_mv_warp_dyn(const pnp_dyn_ref* dyn, const void* src_pool, int src_pool_images, int64_t flow_row_stride,
                    int64_t flow_image_stride, int N, int H, int W, void* stream);

/*
 * LR frames -> im2col'd bf16 operand (N, H, W, dst_channels), channel k = tap*3 + c for k < 27, zero for
 * 27..31.  dst_channels = 32: 64-byte pixels, every byte written (the operand the conv reads through a
 * SWIZZLE_64B tile, pnp_conv_desc.aux_channels = 32); dst_channels = 64: 128-byte pixels whose channels 32..63
 * are not written (allocate the buffer zeroed once).  Carries the 3-channel slice of the reference's input conv
 * (basicvsr_net.py:484 on the cat at iconvsr_ipb_par.py:90,125).  lr is an fp32 (N,3,H,W) view with element
 * strides sn, sc, sy (x: 1).
 */
int pnp_lr_im2col(const float* lr, int64_t sn, int64_t sc, int64_t sy, void* dst, int N, int H, int W,
                  int dst_channels, void* stream);
/* table mode: lr / dst come from the launch table */
int pnp_lr_im2col_dyn(const pnp_dyn_ref* dyn, int64_t sn, int64_t sc, int64_t sy, int N, int H, int W, int dst_channels,
                      void* stream);

/*
 * K4 -- weight packing (run once per checkpoint / once per distinct (CRF, QP) condition, results stay resident).
 * Packed operands are 128-byte rows [out channel][64 in channels] bf16, pre-swizzled for the tensor-core
 * shared-memory layout (16-byte column group g of row r at g ^ (r & 7)).
 *   pnp_pack_conv3x3_rowstack: w is fp32 (E, out_ch, in_total, 3, 3); the result is sum_e coef[e]*w[e] restricted to
 *     input channels [in_begin, in_begin+in_count) (+ the slice at in_begin2 if >= 0), laid out per kx as one block of
 *     3*tap_n rows, sub-block sb = 0,1,2 holding ky = 2 - sb (flip_ky: ky = sb), so that one source row can be multiplied
 *     against the weights of the three output rows it feeds in a single N = 3*tap_n MMA.  tap_n is 64, or 16 for the
 *     64->3 tail; 9*tap_n*128 bytes.  coef is a DEVICE pointer to E floats or NULL (E must then be 1); it replaces the
 *     per-block, per-frame torch.mm expert mixing of Dynamic_conv2d_se.forward (sr_backbone_utils.py:198-199).
 *     row_scale is a DEVICE pointer to out_ch floats multiplied into the rows (the SE gain of
 *     sr_backbone_utils.py:207-208 folded into the kernel: (conv(x,W)+b)*g == conv(x, g*W) + g*b), or NULL.
 *   pnp_pack_rows: fp32 matrix (rows<=64, cols<=64; element strides) into packed rows row_offset.. of dst (the three
 *     1x1 partition convs, sr_backbone_utils.py:285-287, as 192 rows behind a row-stacked pack).
 *   pnp_pack_aux: first 3 input channels of w (out_ch, in_total, 3, 3) as one [64][tap*3+c] block.
 *   pnp_pack_mix_blocks: the block-launch-A packs of ALL n_blocks BAE blocks for one condition in one launch:
 *     w2 fp32 (n_blocks, E, 64, 64, 3, 3), w1x1 fp32 (n_blocks, 3, 64, 64); block b is written at
 *     dst + b*dst_block_stride as [row-stacked row_scale*sum_e coef[e]*w2[b][e] (73728 B)][192 rows of w1x1[b] (24576 B)].
 */
int pnp_pack_conv3x3_rowstack(const float* w, int n_experts, const float* coef, const float* row_scale,
                              int out_ch, int in_total, int in_begin, int in_begin2, int in_count, void* dst,
                              int tap_n, int flip_ky, void* stream);
int pnp_pack_rows(const float* w, int rows, int cols, int64_t row_stride, int64_t col_stride, void* dst,
                  int row_offset, void* stream);
int pnp_pack_aux(const float* w, int out_ch, int in_total, void* dst, void* stream);
int pnp_pack_mix_blocks(const float* w2, const float* w1x1, int n_blocks, int n_experts, const float* coef,
                        const float* row_scale, void* dst, int64_t dst_block_stride, void* stream);

/*
 * CAA heads for `frames` frames: experts (frames, n_experts) = Base_Predictor(base_qp)
 * (domain_aware.py:172-183), gamma (frames, 64) = SEModule(qp) (domain_aware.py:201-222).
 * Weights are the reference's parameters, fp32, contiguous.
 */
int pnp_caa_heads(const float* base_qp, const float* qp, int frames, const float* base0_w,
                  const float* base0_b, const float* base2_w, const float* base2_b, const float* se0_w,
                  const float* se2_w, int n_experts, int se_hidden, float* experts, float* gamma,
                  void* stream);
/* out[f][blk][c] = gamma[f][c] * sum_e experts[f][e] * conv2_bias[blk][e][c]
 * (sr_backbone_utils.py:200-208); conv2_bias is (n_blocks, n_experts, 64) contiguous. */
int pnp_mix_bias(const float* conv2_bias, int n_blocks, int n_experts, const float* experts,
                 const float* gamma, int frames, float* out, void* stream);

/*
 * Side-information rasteriser ("next" row of the scope table): per-block motion-vector records ->
 * dense motion fields and partition maps, bit-exact replacement of the per-record Python loop of
 * LoadImageFromFileList_ipb.__call__ (mmedit/datasets/pipelines/loading_ipb.py:328-369) followed by
 * RescaleToZeroOne on the partition maps (normalization.py:93-99) and FramesToTensor (formating.py:101-138).
 *   records       : fp32 (R,10): direction, w, h, src_x, src_y, dst_x, dst_y, motion_x, motion_y, scale
 *   frame_offsets : int32 (T+1): records of frame f are [frame_offsets[f], frame_offsets[f+1])
 *   is_b          : int32 (T): 1 for B slices
 *   p_target      : int32 (T): frame that receives the reversed direction>0 records of a non-B frame
 *                   (the previous non-B frame, loading_ipb.py:351-355,369), -1 if there is none
 *   owner_fwd/owner_bwd/part_mask : uint32 (T,H,W) workspaces, ZEROED by the caller
 *   mvs (T,4,H,W), partitions (T,3,H,W) : fp32 outputs, fully overwritten
 *   status        : device int32, OR-ed with 1 (block area not in {256,128,64}: KeyError in the reference)
 *                   and 2 (reversed record without a target frame)
 */
int pnp_mv_rasterize(const float* records, const int32_t* frame_offsets, const int32_t* is_b,
                     const int32_t* p_target, int T, int R, int H, int W, uint32_t* owner_fwd,
                     uint32_t* owner_bwd, uint32_t* part_mask, float* mvs, float* partitions,
                     int32_t* status, void* stream);
/* The planes of a frame window [a, b) of a clip, bit-identical to frames [a, b) of pnp_mv_rasterize on the whole clip
 * (what the reference computes when it slices the dense tensors of a whole clip, restoration_video_inference.py:121-128).
 * Only one later frame writes into the window: the TAIL frame e, the first non-B frame >= b, whose reversed records land
 * in the previous non-B frame.  The table holds the window's frames, then at most one tail frame, in clip order:
 *   records       : the records of frames [a, b), then (tail = 1) the direction>0 records of frame e
 *   frame_offsets : int32 (T+tail+1), window-relative; is_b, p_target : int32 (T+tail), window-relative frame indices
 *   p_target      : as above, plus -2 for a target before the window (the write is skipped, no status bit)
 *   tail          : 0 or 1; a tail record makes only its reversed write (no forward write, no partition mark, no
 *                   status bit 1: its frame lies outside the window, which owns none of its errors)
 *   T, owner_fwd/owner_bwd/part_mask, mvs, partitions, status: as above, T = b - a window frames.
 * An addition: the ABI version and every other entry point are unchanged. */
int pnp_mv_rasterize_window(const float* records, const int32_t* frame_offsets, const int32_t* is_b,
                            const int32_t* p_target, int T, int tail, int R, int H, int W, uint32_t* owner_fwd,
                            uint32_t* owner_bwd, uint32_t* part_mask, float* mvs, float* partitions,
                            int32_t* status, void* stream);

/*
 * Per-frame quality metrics of the reference's test loop, computed where the frames are ("next" row of the scope
 * table): BasicVSR.evaluate (mmedit/models/restorers/basicvsr.py:119-153) copies every frame to the host, quantises
 * it with tensor2img (mmedit/core/misc.py:9-74: clamp [0,1], x255, round half to even, uint8) and calls psnr / ssim
 * (mmedit/core/evaluation/metrics.py:170-215, 262-355; convert_to=None).
 *   a, b        : fp32 (F,3,H,W) views, unit x stride; *_sf/_sc/_sy = frame / channel / row strides in elements
 *   sse[F]      : EXACT integer sum over the cropped frame and the 3 channels of (a8 - b8)^2;
 *                 psnr = 20 log10(255 / sqrt(sse / (3 (H-2c) (W-2c)))), +inf when sse == 0
 *   ssim_sum[3F]: float64 sum of the SSIM map (11x11 Gaussian window, sigma 1.5, valid positions of the cropped frame)
 *                 of channel k at [3 f + k]; ssim = mean_k(sum_k / ((H-2c-10) (W-2c-10))).  Reference quirk, kept: with
 *                 crop_border != 0 only the first channel of the BGR image -- input channel 2 -- is evaluated
 *                 (metrics.py:347-352 index with a trailing None), and only [3 f] is written.
 * Both outputs are zeroed by the call.  H - 2 crop_border and W - 2 crop_border must be >= 11.
 */
int pnp_frame_quality(const float* a, int64_t a_sf, int64_t a_sc, int64_t a_sy, const float* b, int64_t b_sf,
                      int64_t b_sc, int64_t b_sy, int F, int H, int W, int crop_border, unsigned long long* sse,
                      double* ssim_sum, void* stream);
/* The same metrics with each operand fp32 or uint8: *_is_u8 = 1 makes that operand a uint8 (F,3,H,W) view (strides in
 * bytes) whose values are taken as they are; fp32 operands are quantised as above, so every operand mix sees the same
 * uint8 values: sse is identical, and so is every per-block float64 partial of ssim_sum (the partials meet in float64
 * atomics, whose order -- and with it the last bits of the total -- varies between launches for any operand types).
 * pnp_frame_quality is the fp32 / fp32 case. */
int pnp_frame_quality_u8(const void* a, int a_is_u8, int64_t a_sf, int64_t a_sc, int64_t a_sy, const void* b,
                         int b_is_u8, int64_t b_sf, int64_t b_sc, int64_t b_sy, int F, int H, int W, int crop_border,
                         unsigned long long* sse, double* ssim_sum, void* stream);

/*
 * 8-bit frames -> fp32 lq.  The reference's loader decodes PNGs to uint8 and RescaleToZeroOne computes
 * img.astype(np.float32) / 255. (mmedit/datasets/pipelines/normalization.py:93-99); dst = the correctly rounded fp32
 * quotient v / 255 of every sample (not v * (1/255f), which differs for 126 of the 256 values).
 *   src : uint8 (F,3,H,W) view, unit x stride; s_sf/s_sc/s_sy = frame / channel / row strides in bytes
 *   dst : fp32 (F,3,H,W) view, unit x stride; d_sf/d_sc/d_sy in elements
 * F <= 65535, H <= 21845.
 */
int pnp_unit_from_u8(const uint8_t* src, int64_t s_sf, int64_t s_sc, int64_t s_sy, float* dst, int64_t d_sf,
                     int64_t d_sc, int64_t d_sy, int F, int H, int W, void* stream);

/*
 * K2/K3/K5 -- fused 3x3 convolution on tcgen05 tensor cores (implicit GEMM, TMA fed, TMEM
 * accumulators).  One call replaces one F.conv2d of the reference plus the elementwise work
 * around it:
 *   acc  = conv3x3(src, W) [+ conv1x1(aux, Waux)]
 *   v    = acc * scale + bias [+ sum_k par_k * conv1x1_k(src)] [+ idt]      (fp32)
 *   out  = act(v)                       -> bf16 NHWC               (mode PNP_CONV_BF16)
 *   outf = v[0:3] + lq (or up4(lq))     -> fp32 NCHW view          (mode PNP_CONV_LAST; uint8 with out_u8)
 * Reference call sites: ResidualBlockNoBNDynamic_drt.forward (sr_backbone_utils.py:304-333),
 * input_conv (basicvsr_net.py:484,515), conv_hr/conv_last (iconvsr_ipb_par.py:144-146).
 */
enum { PNP_CONV_BF16 = 0, PNP_CONV_LAST = 1 };
enum { PNP_ACT_NONE = 0, PNP_ACT_LRELU = 1, PNP_ACT_RELU = 2 };

typedef struct pnp_conv_desc {
  const void* src;     /* bf16 (N,H,W,64) */
  const void* aux;     /* bf16 (N,H,W,64) -- or (N,H,W,32), see aux_channels -- im2col'd LR, or NULL */
  const void* idt;     /* bf16 (N,H,W,64) added before the activation, or NULL */
  void* out;           /* bf16 (N,H,W,64); PNP_CONV_BF16 only */
  const void* wpack;   /* pnp_pack_conv3x3_rowstack output (9*tap_n*128 bytes), followed by the 8192-byte
                          pnp_pack_aux block when aux is given, or by the three 1x1 partition convs as 192 packed rows
                          (pnp_pack_rows, offsets 0/64/128 from there) when par is given; par excludes aux and idt */
  const float* scale;  /* [64] or NULL */
  const float* bias;   /* [64] ([3] for PNP_CONV_LAST) or NULL */
  const float* par;    /* fp32 (N,3,H,W) view of the partition map or NULL: block launch A */
  int64_t par_sn, par_sc, par_sy;
  const float* lq;     /* PNP_CONV_LAST: fp32 (N,3,H,W) view */
  int64_t lq_sn, lq_sc, lq_sy;
  float* outf;         /* PNP_CONV_LAST: fp32 (N,3,H,W) view (uint8 with out_u8) */
  int64_t of_sn, of_sc, of_sy;
  int32_t N, H, W;
  int32_t tap_n;       /* 64, or 16 for PNP_CONV_LAST */
  int32_t aux_k16;     /* K/16 of aux (2 for the 27-entry LR im2col), 0 without aux */
  int32_t act;
  int32_t mode;
  int32_t flip_y;      /* process rows bottom-up.  The result is identical when wpack was packed with flip_ky = 1;
                          alternating directions between dependent launches makes each launch read first what its
                          predecessor wrote last (L2 hits). */
  int64_t out_spx, out_sy, out_sn; /* element strides of `out` between pixels / rows / images; all 0 = contiguous
                          (64, 64*W, 64*H*W).  A strided view makes the TMA store a scatter: launch g of a
                          PixelShufflePack (upsample.py:46-49, scale 2) writes its 64 channels to
                          up[:, i::2, j::2, :] -- the pixel shuffle is the store epilogue.  Multiples of 8. */
  int32_t lq_up4;      /* PNP_CONV_LAST: 1 = `lq` is the (N,3,H/4,W/4) low-resolution frame and the epilogue adds its
                          x4 bilinear upsampling (nn.Upsample(scale_factor=4, mode='bilinear', align_corners=False),
                          iconvsr_ipb_par.py:41,140-141) instead of lq itself */
  int32_t par_sparse;  /* 1: the reference's eval-mode sparse_val=True path (sr_backbone_utils.py:294-302): the 1x1 conv of
                          the LAST partition class whose map is non-zero at the pixel, divided by 255 -- the
                          map's value is not used.  0: dense sum_k par_k * conv1x1_k(src). */
  int32_t wpack_stable; /* 1: wpack was NOT written by the operation immediately preceding this launch in the stream
                          (weights are packed once per checkpoint / clip, long before the frame loop), so the
                          kernel may fetch it while the previous kernel is still draining (programmatic dependent
                          launch).  0: fetch it only after the previous kernel has completed. */
  int32_t per_image;   /* 1: every image of the launch has its OWN weights and bias (clips with different CRF / QP
                          conditions in one launch -- the reference's per-sample grouped conv, groups = batch,
                          sr_backbone_utils.py:196-204): image n uses wpack + img_off[2n] bytes and bias + img_off[2n+1]
                          floats.  CTAs are then partitioned by image; N must not exceed the SM count. */
  const int64_t* img_off; /* per_image (static launches): device array of N (weight byte offset, bias float offset) pairs */
  /* table mode (dyn.table != NULL): wpack / bias / par / lq / outf / img_off and the first-image indices of src / aux /
     idt / out come from the launch table; src / aux / idt / out above are then the BASES of buffers holding
     src_images / aux_images / idt_images / out_images images (0 = N) -- typically one pool that contains every frame's
     features and the work buffers -- and bias / par / lq / outf / aux / idt only say (non-NULL) that the operand exists. */
  pnp_dyn_ref dyn;
  int32_t src_images, aux_images, idt_images, out_images;
  int32_t aux_channels; /* channels per pixel of `aux`: 64 (or 0) = a (N,H,W,64) tensor; 32 = a (N,H,W,32) tensor of 64-byte
                          pixels as pnp_lr_im2col writes it with dst_channels = 32 (aux_k16 <= 2) */
  int32_t out_u8;      /* PNP_CONV_LAST: 1 = `outf` is a uint8 (N,3,H,W) view (of_* strides in bytes) and receives tensor2img's
                          value of every output sample (mmedit/core/misc.py:9-74): the same fp32 v + bias + lq as the fp32
                          store, clamped to [0,1], x255 (fp32), rounded half to even -- the uint8 frame the reference scores or
                          writes, and what pnp_frame_quality computes from the fp32 frame.  0 = fp32 store (the only value
                          accepted for PNP_CONV_BF16). */
} pnp_conv_desc;

int pnp_conv3x3(const pnp_conv_desc* desc, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PNP_VCVE_H_ */
