"""Host-side scheduler of the BAE+CAA forward: key-frame schedule, resident packed weights, the feature pool, the
per-call launch table and the CUDA graphs of the frame steps.

Restructures ``IconVSR_restore_wo_refill_mv_ipb_fast_domain_dynamic_with_par.forward``
(mmedit/models/backbones/sr_backbones/iconvsr_ipb_par.py:44-149) without changing its results:

* the key-frame indices come from ONE device->host copy of ``slices`` instead of ``int(torch.where(...))`` per frame
  and clip (:81, :116);
* expert mixing (sr_backbone_utils.py:198-202) is done once per distinct (CRF, QP) condition and kept resident;
* ``torch.cat`` of [lr, key_warp, neighbour(, backward feature)] (:90, :125) is never materialised: each source is its
  own K slice of ``input_conv.0.weight`` and is accumulated by a chain of conv launches; when the neighbour IS the
  warped key frame (:85-88) the two K slices are summed into one;
* SE gain, bias, partition-modulated 1x1 convs, ReLU/LeakyReLU, residual adds and the final ``out += lq`` run in the
  conv epilogues;
* the reference's Python frame loop (:71-147, ~300 library launches per frame) becomes ONE CUDA-graph launch per frame
  step: every frame's features and all work buffers live in one pool (one TMA tensor map), the operands that change
  from frame to frame sit in a device-resident launch table written once per call, and the six step variants
  (backward / forward x first / merged-neighbour / separate-neighbour) are captured once per clip shape;
* clips of one call that share the key-frame schedule run as ONE sequence with N images per launch even when their
  CRF / QP conditions differ: per-image weight and bias offsets in the launch (the reference's per-sample grouped conv,
  ``groups = batch``, sr_backbone_utils.py:196-204).
"""
import ctypes
import os

import numpy as np
import torch
import torch.nn.functional as F

from . import _lib, ops
from .ops import PNP_ACT_LRELU, PNP_ACT_NONE, PNP_ACT_RELU

SLICE_I, SLICE_P = 73, 80
ROW_BYTES = 9 * 64 * 128           # one row-stacked 64->64 pack
WORK = ("kw", "pa", "pb", "xa", "xb", "t", "hr", "zero")


def key_schedule(key_row):
    """Key-frame indices for one clip (iconvsr_ipb_par.py:60-62, :81, :116).

    key_row: list[bool] with first/last already forced.  Returns (bwd_key, fwd_key):
    bwd_key[i] = min{j > i : key[j]} for i < T-1, fwd_key[i] = max{j < i : key[j]} for i > 0, else -1.
    """
    t = len(key_row)
    bwd, fwd = [-1] * t, [-1] * t
    nxt = -1
    for i in range(t - 1, -1, -1):
        bwd[i] = nxt
        if key_row[i]:
            nxt = i
    prv = -1
    for i in range(t):
        fwd[i] = prv
        if key_row[i]:
            prv = i
    return bwd, fwd


def keyframe_rows(slices_host):
    """slices_host: (n,T) float tensor on the host -> list of per-clip bool lists."""
    key = (slices_host == SLICE_I) | (slices_host == SLICE_P)
    key[:, 0] = True
    key[:, -1] = True
    return key.tolist()


def group_clips(key_rows, max_batch, batch=True):
    """Runs of consecutive clips with the same key-frame schedule -> [b0, b1) ranges (at most max_batch clips each).
    Such clips take the same launch sequence at every step; their CRF / QP conditions may differ (per-image weights)."""
    groups = []
    for b, row in enumerate(key_rows):
        if batch and groups and row == key_rows[groups[-1][0]] and groups[-1][1] - groups[-1][0] < max_batch:
            groups[-1][1] = b + 1
        else:
            groups.append([b, b + 1])
    return [tuple(g) for g in groups]


def step_variants(bwd_key, fwd_key):
    """Variant name of each of the 2T frame steps: steps 0..T-1 are the backward-time pass (frame T-1-s), steps
    T..2T-1 the forward-time pass (frame s-T)."""
    t = len(bwd_key)
    names = []
    for s in range(t):
        i = t - 1 - s
        names.append("b_last" if i == t - 1 else ("b_merged" if bwd_key[i] == i + 1 else "b_sep"))
    for i in range(t):
        names.append("f_first" if i == 0 else ("f_merged" if fwd_key[i] == i - 1 else "f_sep"))
    return names


class _Program:
    """Everything that is fixed for one (clip count, T, H, W) shape: the feature pool, the launch table, the prebuilt
    descriptors of every step variant and their captured graphs."""

    def __init__(self, n, t, h, w, dev, maxn, nb, vsr, table_steps, lr_once=False):
        self.key = (n, t, h, w, dev, maxn, nb, vsr, lr_once)
        self.n, self.t, self.h, self.w, self.dev, self.maxn, self.nb, self.vsr = n, t, h, w, dev, maxn, nb, vsr
        self.img_bytes = h * w * 128
        # The LR im2col operand lives in its own (images, H, W, 32) tensor of 64-byte pixels (SWIZZLE_64B aux tiles).
        # lr_once: one image per frame and clip (frame-major like feats) -- the backward-time pass writes it, the
        # forward-time pass reads it again instead of recomputing it; otherwise one image per clip of a run.
        self.lr_once = lr_once
        self.lr = torch.zeros((t * n if lr_once else maxn, h, w, 32), dtype=torch.bfloat16, device=dev)
        self.lr_img_bytes = h * w * 64
        first_work = t * n
        self.pool_images = first_work + len(WORK) * maxn
        self.pool = torch.empty((self.pool_images, h, w, 64), dtype=torch.bfloat16, device=dev)
        self.feats = self.pool[: t * n].view(t, n, h, w, 64)      # frame-major: a run of clips at one frame is contiguous
        self.work = {}
        for k, name in enumerate(WORK):
            f0 = first_work + k * maxn
            self.work[name] = (f0, self.pool[f0:f0 + maxn])
        self.work["zero"][1].zero_()
        if vsr:      # x4 tail: 2Hx2W and 4Hx4W feature maps of one frame step
            self.u1 = ops.new_feature(maxn, 2 * h, 2 * w, dev)
            self.u2 = ops.new_feature(maxn, 4 * h, 4 * w, dev)
            self.hr4 = ops.new_feature(maxn, 4 * h, 4 * w, dev)
        self.stride = 8 + 2 * nb + (8 if vsr else 0)              # launch-table entries per step
        self.table_steps = 0
        self.table = self.img_off = self.host_table = self.host_off = None
        self.nodes = {}          # (variant, nn, per_image, sparse, out_u8) -> [(kind, label, args)]
        self.graphs = {}         # same key -> graph handle
        self.ensure_table(table_steps)
        self.step_word = torch.zeros(1, dtype=torch.int32, device=dev)
        self.cap_stream = torch.cuda.Stream(device=dev)   # stream capture is not allowed on the legacy default stream
        self.uploaded = None     # event behind the last table upload (the pinned staging buffers are reused)

    def ensure_table(self, steps):
        if steps <= self.table_steps:
            return
        steps = max(steps, 2 * self.t)
        self.release_graphs()    # the table address is baked into the captured kernel parameters
        self.nodes = {}
        self.table_steps = steps
        self.table = torch.zeros((steps, self.stride, _lib.DYN_ENTRY_WORDS), dtype=torch.int64, device=self.dev)
        self.img_off = torch.zeros((steps, self.maxn, 2), dtype=torch.int64, device=self.dev)
        self.host_table = torch.zeros((steps, self.stride, _lib.DYN_ENTRY_WORDS), dtype=torch.int64).pin_memory()
        self.host_off = torch.zeros((steps, self.maxn, 2), dtype=torch.int64).pin_memory()

    def release_graphs(self):
        graphs, self.graphs = getattr(self, "graphs", {}), {}
        if graphs:
            lib = _lib.load()
            for g in graphs.values():
                lib.pnp_graph_destroy(g)

    def __del__(self):
        try:
            self.release_graphs()
        except Exception:  # noqa: BLE001 - interpreter shutdown
            pass


class BaeEngine:
    """Owns the packed weights, the feature pool and the step graphs of one generator instance on one device."""

    def __init__(self, module):
        self.m = module
        self.static_key = None
        self.static = None
        self.mix_slots = {}       # (CRF, QP) -> slot of mix_pool
        self.mix_pool = None      # uint8 (slots, 2*nb, PACK_A_BYTES): expert-mixed block-launch-A packs
        self.prog = None
        self.launch_count = 0
        self.last_mode = "graph"  # how the last forward launched its frame steps: "graph" | "eager"
        self._done = None         # (device, event recorded behind the last forward)
        #: set to {label: []} (labels: "block_a", "block_b", "input", "hr", "last", "up", "warp", "im2col", "phases") to
        #: have the next forward bracket those launches with CUDA events on the launching stream (bench.py); such a
        #: forward launches its kernels one by one instead of replaying graphs.  prof_every = N brackets only every
        #: N-th launch of a label (event records between kernels defeat programmatic dependent launch).
        self.prof = None
        self.prof_every = 1
        #: replay one captured CUDA graph per frame step (default) or launch the same table-mode kernels one by one
        self.use_graphs = os.environ.get("PNP_GRAPHS", "1") != "0"
        #: batch runs of clips with the same key-frame schedule into N-image launches (up to max_batch clips)
        self.batch_clips = os.environ.get("PNP_BATCH_CLIPS", "1") != "0"
        #: LR im2col once per frame (kept in the pool between the two passes): None = when the memory is small against
        #: the device, True / False = forced (PNP_LR_ONCE=1 / 0)
        self.lr_once = {"0": False, "1": True}.get(os.environ.get("PNP_LR_ONCE", ""), None)
        self.max_batch = 16

    # ------------------------------------------------------------------ weights
    def _param_key(self):
        # data_ptr: updates through ``p.data`` (``p.data = ...``, EMA weight swaps) re-seat the storage without
        # bumping ``_version``; in-place writes through ``.data`` (``p.data.copy_``) change neither -- call
        # ``invalidate()`` (the module does it from ``load_state_dict`` / ``_apply``) after such updates
        return tuple((id(p), p._version, p.device, p.data_ptr()) for p in self.m.parameters())

    def invalidate(self):
        """Drop the packed / expert-mixed weights (re-packed by the next forward)."""
        self.static = self.static_key = None
        self.mix_slots = {}

    # Copies and pickles of the owning module get a FRESH engine: packed weights, the pool, graphs, ctypes
    # descriptors and events are per-process, per-device resources and are rebuilt on first use.
    def __getstate__(self):
        return {"m": self.m}

    def __setstate__(self, state):
        self.__init__(state["m"])

    def _pack_static(self, dev):
        """Weights that do not depend on the clip: packed once per checkpoint."""
        key = self._param_key()
        if self.static is not None and self.static_key == key:
            return self.static
        m = self.m
        nb = m.num_blocks
        st = {}

        def f32(p):
            return p.detach().to(dev, torch.float32).contiguous()

        conv1_w = torch.zeros((2 * nb, ROW_BYTES), dtype=torch.uint8, device=dev)
        conv1_b, c2w, c2b, w1x1 = [], [], [], []
        for br, (name, branch) in enumerate((("bwd", m.backward_resblocks), ("fwd", m.forward_resblocks))):
            w_in = f32(branch.input_conv[0].weight)
            st[name + "_in_bias"] = f32(branch.input_conv[0].bias)
            # K slices of the 131/195-channel input conv: [0:3] lr, [3:67] key_warp, [67:131] neighbour,
            # [131:195] backward feature (iconvsr_ipb_par.py:90,125)
            def pack(in_begin, in_begin2=-1, with_aux=False, w_in=w_in):
                buf = ops.new_wpack_rowstack(dev, with_aux=with_aux)
                ops.pack_conv3x3_rowstack(w_in, buf, in_begin=in_begin, in_begin2=in_begin2, in_count=64)
                if with_aux:
                    ops.pack_aux(w_in, buf[ROW_BYTES:])
                return buf
            if name == "bwd":
                st["bwd_key_aux"] = pack(3, with_aux=True)          # first pass, separate neighbour
                st["bwd_merged_aux"] = pack(3, 67, with_aux=True)   # neighbour == key_warp
                st["bwd_nb"] = pack(67)
            else:
                st["fwd_bf_aux"] = pack(131, with_aux=True)         # first pass: backward feature + lr
                st["fwd_key"] = pack(3)
                st["fwd_merged"] = pack(3, 67)
                st["fwd_nb"] = pack(67)
            for k, blk in enumerate(branch.main):
                # block launch B walks the image bottom-up (flip_y): launch A wrote its bottom rows
                # last, so B finds them in L2; B in turn writes the top rows last, where A starts
                ops.pack_conv3x3_rowstack(f32(blk.conv1.weight), conv1_w[br * nb + k], flip_ky=True)
                conv1_b.append(f32(blk.conv1.bias))
                c2w.append(f32(blk.conv2.weight))
                c2b.append(f32(blk.conv2.bias))
                w1x1.append(torch.stack([f32(c.weight).view(64, 64) for c in
                                         (blk.conv16x16, blk.conv16x8, blk.conv8x8)], 0))
        st["conv1_w"] = conv1_w
        st["conv1_b"] = torch.stack(conv1_b, 0).contiguous()          # (2nb, 64)
        st["conv2_w_all"] = torch.stack(c2w, 0).contiguous()          # (2nb, E, 64, 64, 3, 3)
        st["w1x1_all"] = torch.stack(w1x1, 0).contiguous()            # (2nb, 3, 64, 64)
        st["conv2_bias_all"] = torch.stack(c2b, 0).contiguous()       # (2nb, E, 64)
        hr = ops.new_wpack_rowstack(dev)
        ops.pack_conv3x3_rowstack(f32(m.conv_hr.weight), hr)
        st["hr_w"], st["hr_b"] = hr, f32(m.conv_hr.bias)
        last = ops.new_wpack_rowstack(dev, tap_n=16)
        ops.pack_conv3x3_rowstack(f32(m.conv_last.weight), last, tap_n=16)
        st["last_w"], st["last_b"] = last, f32(m.conv_last.bias)
        if m.vsr:
            # PixelShufflePack (common/upsample.py:46-49): conv 64 -> 256 then pixel_shuffle(2), i.e. output
            # channel c*4 + 2*i + j lands at (c, 2y+i, 2x+j).  Sliced by g = 2*i + j this is four 64 -> 64
            # convs whose 64 channels are one NHWC pixel of the upsampled map: the shuffle becomes the
            # (strided) store of launch g and LeakyReLU stays in its epilogue.
            for name, mod in (("up1", m.upsample1), ("up2", m.upsample2)):
                w_up, b_up = f32(mod.upsample_conv.weight), f32(mod.upsample_conv.bias)
                packs, biases = [], []
                for g in range(4):
                    buf = ops.new_wpack_rowstack(dev)
                    ops.pack_conv3x3_rowstack(w_up[g::4].contiguous(), buf)
                    packs.append(buf)
                    biases.append(b_up[g::4].contiguous())
                st[name + "_w"], st[name + "_b"] = packs, biases
        st["caa"] = dict(b0w=f32(m.BasePredictor.BaseNet[0].weight), b0b=f32(m.BasePredictor.BaseNet[0].bias),
                         b2w=f32(m.BasePredictor.BaseNet[2].weight), b2b=f32(m.BasePredictor.BaseNet[2].bias),
                         s0w=f32(m.BiasePredictor.fc[0].weight), s2w=f32(m.BiasePredictor.fc[2].weight))
        st["nb"] = nb
        self.static, self.static_key = st, key
        self.mix_slots = {}
        return st

    def _mix_slots_for(self, st, conds, experts, gamma, dev):
        """Slot of the expert-mixed packs of every (CRF, QP) condition in ``conds`` ({cond: flat frame index}).

        Dynamic_conv2d_se.forward (sr_backbone_utils.py:198-208) re-mixes per block and frame and multiplies the
        output by gamma; the mixture only depends on the frame's CRF and gamma on its QP, so the packed kernels
        gamma_o * sum_e a_e W_e of ALL 2*nb blocks are produced by one launch per distinct condition and kept in a
        pool -- 3 conditions per clip in the IPB configs, at most ~15 in the CRF config."""
        nb2 = 2 * st["nb"]
        pool = self.mix_pool
        if pool is not None and (pool.device != dev or pool.shape[1] != nb2):
            pool = self.mix_pool = None
            self.mix_slots = {}
        need = [c for c in conds if c not in self.mix_slots]
        cap = 0 if pool is None else pool.shape[0]
        if len(self.mix_slots) + len(need) > cap:
            # recycle every slot (whatever is still enqueued reads its packs in stream order); grow when one call alone
            # needs more conditions than the pool holds
            if len(conds) > cap:
                self.mix_pool = None
                self.mix_pool = torch.empty((max(48, 2 * len(conds)), nb2, ops.PACK_A_BYTES), dtype=torch.uint8, device=dev)
            self.mix_slots = {}
            need = list(conds)
        for c in need:
            slot = len(self.mix_slots)
            f = conds[c]
            ops.pack_mix_blocks(st["conv2_w_all"], st["w1x1_all"], experts[f], gamma[f], self.mix_pool[slot])
            self.mix_slots[c] = slot
        return self.mix_slots

    # ------------------------------------------------------------------ program (pool, table, descriptors, graphs)
    def _program(self, n, t, h, w, dev, maxn, steps):
        # LR im2col once per frame instead of once per pass: costs a second t*n-image region of the pool, taken when
        # it is small against the device (PNP_LR_ONCE=0/1 forces it off / on)
        extra = t * n * h * w * 64
        lr_once = self.lr_once if self.lr_once is not None else \
            extra <= torch.cuda.get_device_properties(dev).total_memory // 8
        key = (n, t, h, w, dev, maxn, self.m.num_blocks, bool(self.m.vsr), lr_once)
        if self.prog is None or self.prog.key != key:
            self.prog = None                         # release the old pool before allocating the new one
            self.prog = _Program(n, t, h, w, dev, maxn, self.m.num_blocks, bool(self.m.vsr), steps, lr_once)
        self.prog.ensure_table(steps)
        return self.prog

    def _build_nodes(self, pg, variant, nn, per_image, sparse, shapes, out_u8=False):
        """Launch sequence of one step variant for a run of ``nn`` clips: [(kind, label, ctypes args)], every operand
        that changes per step left to the launch table (node index = position in the list).  out_u8: conv_last stores
        uint8 frames (the descriptor, and with it a captured graph, differs)."""
        lib = _lib.load()
        nodes = []
        h, w, nb = pg.h, pg.w, pg.nb
        pool_ptr = pg.pool.data_ptr()

        def dyn(node):
            r = _lib.DynRef()
            r.table, r.step, r.node, r.stride = pg.table.data_ptr(), pg.step_word.data_ptr(), node, pg.stride
            return r

        def conv(label, aux=False, idt=False, bias=False, par=False, act=PNP_ACT_NONE, flip=False, last=False,
                 image=False, src=None, out=None, hh=h, ww=w, lq_up4=False):
            d = ops.ConvDesc()
            d.src = src.data_ptr() if src is not None else pool_ptr
            d.src_images = 0 if src is not None else pg.pool_images
            d.aux, d.aux_images = (pg.lr.data_ptr(), pg.lr.shape[0]) if aux else (None, 0)
            d.aux_channels = 32 if aux else 0
            d.idt, d.idt_images = (pool_ptr, pg.pool_images) if idt else (None, 0)
            d.out_spx = d.out_sy = d.out_sn = 0
            if last:
                d.out, d.out_images = None, 0
            elif out is not None:
                d.out, d.out_images = out.data_ptr(), 0
                if not out.is_contiguous():
                    d.out_sn, d.out_sy, d.out_spx = out.stride(0), out.stride(1), out.stride(2)
            else:
                d.out, d.out_images = pool_ptr, pg.pool_images
            d.wpack, d.scale = None, None
            d.bias = 1 if bias else None                       # table mode: non-NULL only says "there is a bias"
            if par:
                d.par = 1
                d.par_sn, d.par_sc, d.par_sy = shapes["par"]
            if last:
                d.lq, d.outf = 1, 1
                d.lq_sn, d.lq_sc, d.lq_sy = shapes["lq"]       # with lq_up4: strides of the LR frame itself
                d.of_sn, d.of_sc, d.of_sy = shapes["outf"]
                d.out_u8 = 1 if out_u8 else 0
            d.N, d.H, d.W = nn, hh, ww
            d.tap_n = 16 if last else 64
            d.aux_k16 = 2 if aux else 0
            d.act, d.mode = act, (ops.PNP_CONV_LAST if last else ops.PNP_CONV_BF16)
            d.flip_y = 1 if flip else 0
            d.lq_up4 = 1 if lq_up4 else 0
            d.par_sparse = 1 if (par and sparse) else 0
            d.wpack_stable = 1
            d.per_image = 1 if image else 0
            d.img_off = None
            d.dyn = dyn(len(nodes))
            nodes.append(("conv", label, (lib.pnp_conv3x3, ctypes.byref(d), d)))

        def im2col():
            r = dyn(len(nodes))
            sn, sc, sy = shapes["lq"]
            nodes.append(("im2col", "im2col", (lib.pnp_lr_im2col_dyn, ctypes.byref(r), r, sn, sc, sy, nn, h, w, 32)))

        def warp():
            r = dyn(len(nodes))
            fsy, fsn = shapes["flow"]
            nodes.append(("warp", "warp", (lib.pnp_mv_warp_dyn, ctypes.byref(r), r, ctypes.c_void_p(pool_ptr), pg.pool_images,
                                           fsy, fsn, nn, h, w)))

        bwd = variant.startswith("b_")
        if bwd or not pg.lr_once:
            im2col()
        if variant not in ("b_last", "f_first"):
            warp()
        if variant in ("b_last", "b_merged", "f_first"):
            conv("input", aux=True, bias=True, act=PNP_ACT_LRELU)
        elif variant in ("b_sep", "f_merged"):
            conv("input", aux=True, bias=True)
            conv("input", idt=True, act=PNP_ACT_LRELU)
        else:   # f_sep
            conv("input", aux=True, bias=True)
            conv("input", idt=True)
            conv("input", idt=True, act=PNP_ACT_LRELU)
        for _ in range(nb):     # ResidualBlockNoBNDynamic_drt, sr_backbone_utils.py:304-333: launch A then launch B
            conv("block_a", bias=True, par=True, act=PNP_ACT_RELU, image=per_image)
            conv("block_b", idt=True, bias=True, flip=True)
        if not bwd:
            if pg.vsr:
                # x4 tail (:135-142): lrelu(upsample1) -> lrelu(upsample2) -> lrelu(conv_hr) -> conv_last + bilinear x4 of
                # the LR frame.  Pixel shuffle = strided store of launch g, the bilinear base is computed inside
                # conv_last's epilogue from the LR frame.
                u1, u2, hr4 = pg.u1[:nn], pg.u2[:nn], pg.hr4[:nn]
                for g in range(4):
                    conv("up", bias=True, act=PNP_ACT_LRELU, out=u1[:, g >> 1::2, g & 1::2, :])
                for g in range(4):
                    conv("up", bias=True, act=PNP_ACT_LRELU, src=u1, out=u2[:, g >> 1::2, g & 1::2, :], hh=2 * h, ww=2 * w)
                conv("hr", bias=True, act=PNP_ACT_LRELU, src=u2, out=hr4, hh=4 * h, ww=4 * w)
                conv("last", bias=True, last=True, src=hr4, hh=4 * h, ww=4 * w, lq_up4=True)
            else:
                # out = conv_last(lrelu(conv_hr(x))) + lq   (:144-146)
                conv("hr", bias=True, act=PNP_ACT_LRELU)
                conv("last", bias=True, last=True)
        assert len(nodes) <= pg.stride
        return nodes

    def _fill_table(self, pg, st, g_idx, b0, nn, variants, bwd_key, fwd_key, slot_of, ptrs, per_image):
        """Launch-table rows [g_idx*2T, (g_idx+1)*2T) for one run of clips, vectorised over the steps of each variant."""
        t, n, nb, h, w = pg.t, pg.n, pg.nb, pg.h, pg.w
        tab = pg.host_table.numpy()[g_idx * 2 * t:(g_idx + 1) * 2 * t]
        off = pg.host_off.numpy()[g_idx * 2 * t:(g_idx + 1) * 2 * t]
        tab[:] = 0
        off[:] = 0
        steps = np.arange(2 * t)
        frame = np.where(steps < t, t - 1 - steps, steps - t)
        var = np.array(variants)
        img = pg.img_bytes
        pool_ptr = pg.pool.data_ptr()
        work = {k: v[0] for k, v in pg.work.items()}
        feats = lambda i: i * n + b0                                             # noqa: E731 - pool image of frame i
        bk, fk = np.array(bwd_key), np.array(fwd_key)
        up = 4 if pg.vsr else 1
        plane = h * w * 4
        lr_ptr = ptrs["lrs"] + (b0 * t + frame) * 3 * plane
        par_ptr = ptrs["par"] + (b0 * t + frame) * 3 * plane
        outf_ptr = ptrs["out"] + (b0 * t + frame) * 3 * h * w * up * up * ptrs["out_elem"]    # fp32 or uint8 frames
        mv_base = ptrs["mvs"] + (b0 * t + frame) * 4 * plane
        flow_x = np.where(steps < t, mv_base + 2 * plane, mv_base)               # bwd pass: channels 2,3; fwd: 0,1
        bias_row = 2 * nb * 64
        # expert-mixed packs / biases: per-image offsets (per_image) or folded into the base pointers
        slots = slot_of[b0:b0 + nn][:, frame]                                    # (nn, 2T)
        slot_stride = self.mix_pool.stride(0)
        if per_image:
            off[:, :nn, 0] = (slots * slot_stride).T
            off[:, :nn, 1] = (((b0 + np.arange(nn))[:, None] * t + frame[None, :]) * bias_row).T
            w_base = np.full(2 * t, self.mix_pool.data_ptr(), dtype=np.int64)
            b_base = np.full(2 * t, ptrs["bias_tab"], dtype=np.int64)
            off_ptr = pg.img_off.data_ptr() + (g_idx * 2 * t + steps) * pg.maxn * 16
        else:
            w_base = self.mix_pool.data_ptr() + slots[0] * slot_stride
            b_base = ptrs["bias_tab"] + (b0 * t + frame) * bias_row * 4
            off_ptr = np.zeros(2 * t, dtype=np.int64)

        def put(sel, node, p=(), i=(0, 0, 0, 0)):
            for k, v in enumerate(p):
                tab[sel, node, k] = v[sel] if isinstance(v, np.ndarray) else v
            iv = [np.asarray(x[sel] if isinstance(x, np.ndarray) else x, dtype=np.int64) & 0xFFFFFFFF for x in i]
            tab[sel, node, 6] = iv[0] | (iv[1] << 32)
            tab[sel, node, 7] = iv[2] | (iv[3] << 32)

        W = {k: v.data_ptr() for k, v in st.items() if isinstance(v, torch.Tensor)}
        # image of the frame's LR im2col operand in pg.lr: its own per-frame image (lr_once) or the run's first image
        lr64 = (frame * n + b0) if pg.lr_once else np.zeros(2 * t, dtype=np.int64)
        for v in set(variants):
            sel = var == v
            bwd = v.startswith("b_")
            br = 0 if bwd else 1
            node = 0
            if bwd or not pg.lr_once:
                put(sel, node, p=(lr_ptr, pg.lr.data_ptr() + lr64 * pg.lr_img_bytes))   # im2col
                node += 1
            cur = feats(frame)
            if v not in ("b_last", "f_first"):
                kidx = np.where(steps < t, bk[frame], fk[frame])
                put(sel, node, p=(0, flow_x, flow_x + plane, 0), i=(feats(kidx), 0, 0, work["kw"]))
                node += 1
            in_bias = W["bwd_in_bias"] if bwd else W["fwd_in_bias"]
            if v == "b_last":       # zeros for key_warp / neighbour (:69-70)
                put(sel, node, p=(W["bwd_merged_aux"], in_bias), i=(work["zero"], lr64, 0, work["xa"]))
                node += 1
            elif v == "b_merged":   # align_key: the neighbour is the warped key (:85-88)
                put(sel, node, p=(W["bwd_merged_aux"], in_bias), i=(work["kw"], lr64, 0, work["xa"]))
                node += 1
            elif v == "b_sep":
                put(sel, node, p=(W["bwd_key_aux"], in_bias), i=(work["kw"], lr64, 0, work["pa"]))
                put(sel, node + 1, p=(W["bwd_nb"],), i=(feats(frame + 1), 0, work["pa"], work["xa"]))
                node += 2
            elif v == "f_first":
                put(sel, node, p=(W["fwd_bf_aux"], in_bias), i=(cur, lr64, 0, work["xa"]))
                node += 1
            elif v == "f_merged":
                put(sel, node, p=(W["fwd_bf_aux"], in_bias), i=(cur, lr64, 0, work["pa"]))
                put(sel, node + 1, p=(W["fwd_merged"],), i=(work["kw"], 0, work["pa"], work["xa"]))
                node += 2
            else:                   # f_sep
                put(sel, node, p=(W["fwd_bf_aux"], in_bias), i=(cur, lr64, 0, work["pa"]))
                put(sel, node + 1, p=(W["fwd_key"],), i=(work["kw"], 0, work["pa"], work["pb"]))
                put(sel, node + 2, p=(W["fwd_nb"],), i=(feats(frame - 1), 0, work["pb"], work["xa"]))
                node += 3
            x, other = work["xa"], work["xb"]
            for k in range(nb):
                blk = br * nb + k
                put(sel, node, p=(w_base + blk * ops.PACK_A_BYTES, b_base + blk * 256, par_ptr, 0, 0, off_ptr),
                    i=(x, 0, 0, work["t"]))
                o = cur if k == nb - 1 else other
                put(sel, node + 1, p=(W["conv1_w"] + blk * ROW_BYTES, W["conv1_b"] + blk * 256),
                    i=(work["t"], 0, x, o))
                node += 2
                x, other = o, x
            if not bwd:
                if pg.vsr:
                    for name, src_f in (("up1", cur), ("up2", 0)):
                        for g in range(4):
                            put(sel, node, p=(st[name + "_w"][g].data_ptr(), st[name + "_b"][g].data_ptr()),
                                i=(src_f, 0, 0, 0))
                            node += 1
                    put(sel, node, p=(W["hr_w"], W["hr_b"]), i=(0, 0, 0, 0))
                    put(sel, node + 1, p=(W["last_w"], W["last_b"], 0, lr_ptr, outf_ptr), i=(0, 0, 0, 0))
                else:
                    put(sel, node, p=(W["hr_w"], W["hr_b"]), i=(cur, 0, 0, work["hr"]))
                    put(sel, node + 1, p=(W["last_w"], W["last_b"], 0, lr_ptr, outf_ptr), i=(work["hr"], 0, 0, 0))

    # ------------------------------------------------------------------ forward
    @torch.no_grad()
    def forward(self, lrs, *args, **kwargs):
        """Runs ``_forward`` with ``lrs.device`` as the current CUDA device (every launch of libpnpvcve goes to the
        current device / its current stream; the reference accepts a module on a non-current device) and orders the
        call behind the previous one: the pool is reused, so a call from another stream waits for the event
        the previous call recorded."""
        dev = lrs.device
        if dev.type != "cuda":
            raise RuntimeError("pnpvcve_b200 runs on sm_100 CUDA devices only; there is no CPU fallback")
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev)
            if self._done is not None and self._done[0] == dev:
                stream.wait_event(self._done[1])
            res = self._forward(lrs, *args, **kwargs)
            ev = self._done[1] if (self._done is not None and self._done[0] == dev) else torch.cuda.Event()
            ev.record(stream)
            self._done = (dev, ev)
        return res

    def _forward(self, lrs, QPs, slices, mvs, base_QPs, par_map, return_features=False, cond_host=None,
                 frame_ready=None, frame_done=None, out=None):
        """cond_host: optional host copies (slices, base_QPs, QPs), each (n,T) -- skips the one device->host copy.
        frame_ready(i): called (host side) before frame i's lq / mvs / par_map are first read, in the backward-time
        pass (i = T-1 .. 0); frame_done(i, out): called after frame i's output has been enqueued.  Both let a caller
        stream a clip in and out in chunks (driver.ClipStreamer): they typically enqueue an event wait / record.
        out: optional preallocated fp32 (n,T,3,Hout,Wout) result buffer (the caller guarantees nobody still reads it),
        or a uint8 one: conv_last then stores tensor2img's uint8 value of every output sample.
        lrs may be uint8 8-bit frames: value v stands for float32(v) / 255 (the reference loader's RescaleToZeroOne);
        the clip is dequantised into an fp32 device tensor first."""
        m = self.m
        dev = lrs.device
        lib = _lib.load()
        _lib.require_device()
        n, t, c, h_in, w_in = lrs.shape
        assert h_in >= 64 and w_in >= 64, (
            f"The height and width of inputs should be at least 64, but got {h_in} and {w_in}.")
        pad_h, pad_w = (4 - h_in % 4) % 4, (4 - w_in % 4) % 4
        lq_u8 = lrs.dtype == torch.uint8
        if frame_ready is not None and (pad_h or pad_w or lq_u8 or not (lrs.is_contiguous() and mvs.is_contiguous()
                                                                       and par_map.is_contiguous())):
            for i in range(t):                            # whole-tensor copies below: everything must have arrived
                frame_ready(i)
            frame_ready = None
        if lq_u8:                                         # 8-bit frames: v / 255 in fp32, before the reflect padding
            src = lrs if lrs.stride(-1) == 1 else lrs.contiguous()
            try:
                src.view(n * t, c, h_in, w_in)
            except RuntimeError:
                src = src.contiguous()
            lrs = ops.unit_from_u8(src, torch.empty(lrs.shape, dtype=torch.float32, device=dev))
        if pad_h or pad_w:                                # spatial_padding, iconvsr.py:371-394
            lrs = F.pad(lrs.reshape(-1, c, h_in, w_in), [0, pad_w, 0, pad_h], mode="reflect")
            lrs = lrs.view(n, t, c, h_in + pad_h, w_in + pad_w)
        h, w = lrs.shape[3:]
        if tuple(mvs.shape) != (n, t, 4, h, w) or tuple(par_map.shape) != (n, t, 3, h, w):
            # the reference fails inside flow_warp.py:27-29 / the partition multiply for these shapes
            raise ValueError(f"The spatial sizes of input ({(h, w)}) and flow ({tuple(mvs.shape[3:])})"
                             f" / partition map ({tuple(par_map.shape[3:])}) are not the same.")
        lrs = lrs.contiguous().float()
        mvs = mvs.contiguous().float()
        par_map = par_map.contiguous().float()
        # NOTE: the mirror-extended case (iconvsr.py:396-410) only changes how the SAME motion
        # vectors are indexed (iconvsr_ipb.py:33-46): flows_backward[-i] of the mirrored layout is
        # mvs[:, i, :2], i.e. exactly flows_forward[i-1].  No branch (and no host sync) is needed.

        st = self._pack_static(dev)
        # one D2H copy for everything the host needs (the reference syncs 2(T-1)n+1 times)
        if cond_host is not None:
            cond = torch.stack([torch.as_tensor(c, dtype=torch.float32).reshape(n, t).cpu() for c in cond_host], 0)
        else:
            cond = torch.stack([slices.reshape(n, t).float(), base_QPs.reshape(n, t).float(),
                                QPs.reshape(n, t).float()], 0).cpu()
        key_rows = keyframe_rows(cond[0])
        crf_host, qp_host = cond[1].numpy(), cond[2].numpy()

        experts, gamma = ops.caa_heads(base_QPs.reshape(-1).float().contiguous(),
                                       QPs.reshape(-1).float().contiguous(), st["caa"], m.num_experts)
        bias_tab = ops.mix_bias(st["conv2_bias_all"], experts, gamma)       # (n*t, 2*nb, 64)
        # expert-mixed packs of every distinct (CRF, QP) condition of the call, packed up front
        conds, cond_keys = {}, []
        for b in range(n):
            row = [(float(crf_host[b, i]), float(qp_host[b, i])) for i in range(t)]
            cond_keys.append(row)
            for i, k in enumerate(row):
                conds.setdefault(k, b * t + i)
        slot_map = self._mix_slots_for(st, conds, experts, gamma, dev)
        slot_of = np.array([[slot_map[k] for k in row] for row in cond_keys], dtype=np.int64)

        groups = group_clips(key_rows, self.max_batch, self.batch_clips)
        maxn = max(b1 - b0 for b0, b1 in groups)
        pg = self._program(n, t, h, w, dev, maxn, 2 * t * len(groups))
        up = 4 if m.vsr else 1
        if out is None:
            out = torch.empty((n, t, 3, up * h, up * w), dtype=torch.float32, device=dev)
        elif tuple(out.shape) != (n, t, 3, up * h, up * w) or out.dtype not in (torch.float32, torch.uint8) or \
                out.device != dev or not out.is_contiguous():
            raise ValueError(f"out must be a contiguous fp32 or uint8 {(n, t, 3, up * h, up * w)} tensor on {dev}")
        out_u8 = out.dtype == torch.uint8
        feats = pg.feats
        bwd_feats = torch.empty_like(feats) if return_features else None
        # the reference takes the sparse path only in eval mode (sr_backbone_utils.py:307: `self.sparse_val and
        # not self.training`); a module left in train() under no_grad computes the dense blend
        sparse = bool(m.sparse_val) and not m.training

        # ---------------- launch table of the whole call: one H2D copy
        if pg.uploaded is not None:
            pg.uploaded.synchronize()                     # the pinned staging buffers are reused between calls
        ptrs = dict(lrs=lrs.data_ptr(), par=par_map.data_ptr(), mvs=mvs.data_ptr(), out=out.data_ptr(),
                    out_elem=out.element_size(), bias_tab=bias_tab.data_ptr())
        plans = []
        for g_idx, (b0, b1) in enumerate(groups):
            bwd_key, fwd_key = key_schedule(key_rows[b0])
            variants = step_variants(bwd_key, fwd_key)
            per_image = bool((slot_of[b0:b1] != slot_of[b0:b0 + 1]).any())
            self._fill_table(pg, st, g_idx, b0, b1 - b0, variants, bwd_key, fwd_key, slot_of, ptrs, per_image)
            plans.append((b0, b1, variants, per_image))
        rows = 2 * t * len(groups)
        # (not a cudaMemcpyAsync: the H2D copy engine may be busy with the next clip's upload for tens of ms)
        ops.fetch_pinned(pg.table[:rows], pg.host_table[:rows])
        ops.fetch_pinned(pg.img_off[:rows], pg.host_off[:rows])
        pg.uploaded = torch.cuda.Event()
        pg.uploaded.record()

        plane = h * w
        shapes = dict(lq=(t * 3 * plane, plane, w), par=(t * 3 * plane, plane, w), flow=(w, t * 4 * plane),
                      outf=(t * 3 * plane * up * up, plane * up * up, w * up))
        prof = self.prof
        graphs = self.use_graphs and prof is None
        self.last_mode = "graph" if graphs else "eager"
        seen = {}
        stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        step_ptr = ctypes.c_void_p(pg.step_word.data_ptr())
        launches = 0

        def phase(name):
            """prof["phases"]: one event per phase boundary of a frame step"""
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            prof["phases"].append((name, ev))

        def run_nodes(nodes, stream):
            for kind, label, a in nodes:
                timed = prof is not None and label in prof
                if timed:                                  # bracket every prof_every-th launch of this label
                    k = seen.get(label, 0)
                    seen[label] = k + 1
                    timed = (k % self.prof_every) == 0
                if timed:
                    e0 = torch.cuda.Event(enable_timing=True)
                    e1 = torch.cuda.Event(enable_timing=True)
                    e0.record()
                if kind == "conv":
                    rc = a[0](a[1], stream)
                elif kind == "warp":
                    rc = a[0](a[1], a[3], a[4], a[5], a[6], a[7], a[8], a[9], stream)
                else:
                    rc = a[0](a[1], a[3], a[4], a[5], a[6], a[7], a[8], a[9], stream)
                if timed:
                    e1.record()
                    prof[label].append((e0, e1))
                if rc != 0:
                    _lib.check(rc, "pnp_" + kind)

        def run_step(step, variant, nn, per_image):
            nonlocal launches
            key = (variant, nn, per_image, sparse, out_u8)      # a captured graph bakes in the descriptors
            nodes = pg.nodes.get(key)
            if nodes is None:
                nodes = pg.nodes[key] = self._build_nodes(pg, variant, nn, per_image, sparse, shapes, out_u8)
            launches += len(nodes)
            if not graphs:
                _lib.check(lib.pnp_set_step(step_ptr, step, stream), "pnp_set_step")
                if prof is not None and "phases" in prof:
                    # events at the phase boundaries of the step: [im2col, warp, input convs] [blocks] [head]
                    n_in = sum(1 for k in nodes if k[1] in ("im2col", "warp", "input"))
                    n_blk = sum(1 for k in nodes if k[1] in ("block_a", "block_b"))
                    tag = "bwd" if variant.startswith("b_") else "fwd"
                    phase(tag + "_start")
                    run_nodes(nodes[:n_in], stream)
                    phase(tag + "_input_done")
                    run_nodes(nodes[n_in:n_in + n_blk], stream)
                    phase(tag + "_stack_done")
                    run_nodes(nodes[n_in + n_blk:], stream)
                    if tag == "fwd":
                        phase("fwd_head_done")
                else:
                    run_nodes(nodes, stream)
                return
            g = pg.graphs.get(key)
            if g is None:
                # capture (nothing executes) on the program's side stream, then replay in the caller's stream
                cap = ctypes.c_void_p(pg.cap_stream.cuda_stream)
                _lib.check(lib.pnp_graph_begin(cap), "pnp_graph_begin")
                handle = ctypes.c_void_p()
                try:
                    run_nodes(nodes, cap)
                finally:
                    rc = lib.pnp_graph_end(cap, ctypes.byref(handle))
                _lib.check(rc, "pnp_graph_end")
                g = pg.graphs[key] = handle
            rc = lib.pnp_graph_launch(g, step_ptr, step, stream)
            if rc != 0:
                _lib.check(rc, "pnp_graph_launch")

        for g_idx, (b0, b1, variants, per_image) in enumerate(plans):
            nn = b1 - b0
            base = g_idx * 2 * t
            # ---------------- backward-time propagation (iconvsr_ipb_par.py:67-100)
            for s in range(t):
                if frame_ready is not None:
                    frame_ready(t - 1 - s)
                run_step(base + s, variants[s], nn, per_image)
            if return_features:
                bwd_feats[:, b0:b1].copy_(feats[:, b0:b1])
            # ---------------- forward-time propagation + reconstruction (:102-147)
            for i in range(t):
                run_step(base + t + i, variants[t + i], nn, per_image)
                if frame_done is not None and b1 == n:
                    frame_done(i, out)
        self.launch_count = launches
        if return_features:
            return out, bwd_feats.transpose(0, 1), feats.clone().transpose(0, 1)     # (n, T, H, W, 64)
        return out
