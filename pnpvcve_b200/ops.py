"""Tensor-level wrappers over the C ABI (raw pointers + current CUDA stream).

PyTorch is used for device memory and streams only; all arithmetic happens in libpnpvcve.so.
Layouts: feature maps are bf16 NHWC ``(N, H, W, 64)``; frames / motion vectors / partition maps
stay in the reference's fp32 NCHW layout and are consumed through strided views.
"""
import ctypes

import torch

from . import _lib
from ._lib import (PNP_ACT_LRELU, PNP_ACT_NONE, PNP_ACT_RELU, PNP_CONV_BF16,  # noqa: F401
                   PNP_CONV_LAST, ConvDesc, DynRef)

CHUNK_BYTES = 8192


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _on_device_of(fn):
    """Public wrappers launch on the device of their first tensor argument (libpnpvcve launches on the CURRENT
    device / its current stream); the context switch is skipped when that device is already current."""
    import functools

    @functools.wraps(fn)
    def wrapped(t, *args, **kwargs):
        if not t.is_cuda:
            raise ValueError(f"{fn.__name__}: CUDA tensors only (there is no CPU path)")
        if t.device.index == torch.cuda.current_device():
            return fn(t, *args, **kwargs)
        with torch.cuda.device(t.device):
            return fn(t, *args, **kwargs)
    return wrapped


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _feat_check(t, name, strided=False):
    ok = t.dtype == torch.bfloat16 and t.dim() == 4 and t.shape[-1] == 64
    if ok and not t.is_contiguous():
        ok = strided and t.stride(3) == 1 and all(st % 8 == 0 and st > 0 for st in t.stride()[:3])
    if not ok:
        raise ValueError(f"{name} must be a contiguous bf16 (N,H,W,64) tensor, got "
                         f"{tuple(t.shape)} {t.dtype}")
    if not t.is_cuda:
        raise ValueError(f"{name} must live on a CUDA device")


def _plane_view_check(t, name):
    """fp32 (N,3|2,H,W)-like view whose innermost stride is 1."""
    if t.dtype != torch.float32 or t.stride(-1) != 1 or not t.is_cuda:
        raise ValueError(f"{name} must be an fp32 CUDA view with unit innermost stride")


def _frames_view(t, name, dtype):
    """(F,3,H,W) view of a (F,3,H,W) or (n,T,3,H,W) frame tensor of ``dtype`` with unit innermost stride."""
    if t.dtype != dtype or not t.is_cuda or t.dim() not in (4, 5) or t.shape[-3] != 3 or t.stride(-1) != 1:
        raise ValueError(f"{name} must be a {dtype} CUDA (F,3,H,W) or (n,T,3,H,W) view with unit innermost stride, got "
                         f"{tuple(t.shape)} {t.dtype}")
    if t.dim() == 5:
        try:
            t = t.view(-1, *t.shape[2:])
        except RuntimeError:
            raise ValueError(f"{name}: the (n,T) dimensions of a 5-D view must merge into one frame stride") from None
    return t


@_on_device_of
def unit_from_u8(src_u8, dst_f32):
    """8-bit frames -> fp32 frames in [0,1]: dst = float32(v) / 255, correctly rounded (the reference loader's
    ``img.astype(np.float32) / 255.``).  src_u8 uint8 and dst_f32 fp32 views of the same (F,3,H,W) or (n,T,3,H,W) shape,
    unit innermost stride."""
    if src_u8.shape != dst_f32.shape:
        raise ValueError(f"unit_from_u8: shapes {tuple(src_u8.shape)} / {tuple(dst_f32.shape)} differ")
    s = _frames_view(src_u8, "src_u8", torch.uint8)
    d = _frames_view(dst_f32, "dst_f32", torch.float32)
    if s.numel() == 0:
        return dst_f32
    f, _, h, w = s.shape
    lib = _lib.load()
    _lib.check(lib.pnp_unit_from_u8(_ptr(s), s.stride(0), s.stride(1), s.stride(2), _ptr(d), d.stride(0), d.stride(1),
                                    d.stride(2), f, h, w, _stream()), "pnp_unit_from_u8")
    return dst_f32


def fetch_pinned(dst, src):
    """dst (device) <- src (pinned host tensor of the same byte size), stream ordered, WITHOUT the copy engine (the
    launch table must not queue behind a clip that is being uploaded)."""
    nbytes = src.numel() * src.element_size()
    if not src.is_pinned() or not dst.is_cuda or not dst.is_contiguous() or not src.is_contiguous() or \
            dst.numel() * dst.element_size() != nbytes:
        raise ValueError("fetch_pinned: dst must be a contiguous CUDA tensor and src a pinned host tensor of the same size")
    with torch.cuda.device(dst.device):
        _lib.check(_lib.load().pnp_fetch_pinned(_ptr(dst), _ptr(src), nbytes, _stream()), "pnp_fetch_pinned")


def new_feature(n, h, w, device, zero=False):
    f = torch.zeros if zero else torch.empty
    return f((n, h, w, 64), dtype=torch.bfloat16, device=device)


@_on_device_of
def mv_warp(src, flow, dst, debug=False):
    """K1.  src/dst (N,H,W,64) bf16; flow (2,H,W) or (N,2,H,W) fp32 view (x then y).  Returns (x0,y0) if debug."""
    _feat_check(src, "src")
    _feat_check(dst, "dst")
    _plane_view_check(flow, "flow")
    n, h, w, _ = src.shape
    if flow.dim() == 3:
        flow = flow.unsqueeze(0)
    if tuple(flow.shape) != (n, 2, h, w) or dst.shape != src.shape:
        raise ValueError(f"The spatial sizes of input ({(h, w)}) and flow ({tuple(flow.shape[-2:])}) "
                         "are not the same.")
    dx = dy = None
    if debug:
        if n != 1:
            raise ValueError("mv_warp: debug tap outputs need N == 1")
        dx = torch.empty((h, w), dtype=torch.int32, device=src.device)
        dy = torch.empty((h, w), dtype=torch.int32, device=src.device)
    lib = _lib.load()
    _lib.check(lib.pnp_mv_warp(_ptr(src), _ptr(flow[0, 0]), _ptr(flow[0, 1]), flow.stride(2), flow.stride(0),
                               _ptr(dst), n, h, w, _ptr(dx), _ptr(dy), _stream()), "pnp_mv_warp")
    return (dx, dy) if debug else None


def _aux_check(t, name):
    """LR im2col operand: contiguous bf16 (N,H,W,64) with 32 channels used, or the compact (N,H,W,32) form."""
    if not (t.dtype == torch.bfloat16 and t.dim() == 4 and t.shape[-1] in (32, 64) and t.is_contiguous() and t.is_cuda):
        raise ValueError(f"{name} must be a contiguous bf16 (N,H,W,64) or (N,H,W,32) CUDA tensor, got "
                         f"{tuple(t.shape)} {t.dtype}")


@_on_device_of
def lr_im2col(lr, dst):
    """lr (N,3,H,W) fp32 view -> dst (N,H,W,64) bf16 (channels 0..31 written) or the compact (N,H,W,32) form."""
    _plane_view_check(lr, "lr")
    _aux_check(dst, "dst")
    n, c, h, w = lr.shape
    if c != 3 or tuple(dst.shape[:3]) != (n, h, w):
        raise ValueError("lr_im2col: shape mismatch")
    lib = _lib.load()
    _lib.check(lib.pnp_lr_im2col(_ptr(lr), lr.stride(0), lr.stride(1), lr.stride(2), _ptr(dst), n, h, w,
                                 int(dst.shape[3]), _stream()), "pnp_lr_im2col")


def rowstack_bytes(tap_n=64, with_aux=False, with_par=False):
    """Size of a row-stacked weight pack (see pnp_pack_conv3x3_rowstack)."""
    return 9 * tap_n * 128 + (CHUNK_BYTES if with_aux else 0) + (3 * CHUNK_BYTES if with_par else 0)


def new_wpack_rowstack(device, tap_n=64, with_aux=False, with_par=False):
    n = (rowstack_bytes(tap_n, with_aux, with_par) + 1023) // 1024 * 1024
    return torch.zeros(n, dtype=torch.uint8, device=device)


@_on_device_of
def pack_conv3x3_rowstack(w, dst, coef=None, in_begin=0, in_begin2=-1, in_count=None, tap_n=64,
                          row_scale=None, flip_ky=False):
    """w fp32 (O,I,3,3) or (E,O,I,3,3) -> row-stacked blocks [kx][ky=2,1,0][tap_n rows] in dst."""
    if w.dtype != torch.float32 or not w.is_contiguous():
        raise ValueError("pack_conv3x3_rowstack: w must be contiguous fp32")
    if w.dim() == 4:
        e, (o, i) = 1, w.shape[:2]
    else:
        e, o, i = w.shape[:3]
    in_count = i - in_begin if in_count is None else in_count
    lib = _lib.load()
    _lib.check(lib.pnp_pack_conv3x3_rowstack(_ptr(w), e, _ptr(coef), _ptr(row_scale), o, i, in_begin, in_begin2,
                                             in_count,
                                             _ptr(dst), tap_n, int(flip_ky), _stream()), "pnp_pack_conv3x3_rowstack")


@_on_device_of
def pack_rows(w2d, dst, row_offset):
    """fp32 (rows<=64, cols<=64) view -> packed rows row_offset.. of dst."""
    if w2d.dtype != torch.float32 or w2d.dim() != 2:
        raise ValueError("pack_rows: need an fp32 matrix")
    lib = _lib.load()
    _lib.check(lib.pnp_pack_rows(_ptr(w2d), w2d.shape[0], w2d.shape[1], w2d.stride(0), w2d.stride(1),
                                 _ptr(dst), row_offset, _stream()), "pnp_pack_rows")


@_on_device_of
def pack_aux(w, dst):
    if w.dtype != torch.float32 or not w.is_contiguous() or w.dim() != 4:
        raise ValueError("pack_aux: w must be contiguous fp32 (O,I,3,3)")
    lib = _lib.load()
    _lib.check(lib.pnp_pack_aux(_ptr(w), w.shape[0], w.shape[1], _ptr(dst), _stream()), "pnp_pack_aux")


PACK_A_BYTES = 12 * CHUNK_BYTES      # block-launch-A pack: row-stacked conv2 mix (72 KB) + three stacked 1x1 (24 KB)


@_on_device_of
def pack_mix_blocks(w2, w1x1, coef, row_scale, dst):
    """All block-launch-A packs of one (CRF, QP) condition: w2 fp32 (B,E,64,64,3,3), w1x1 fp32 (B,3,64,64), coef (E,),
    row_scale (64,) -> dst uint8 (B, PACK_A_BYTES)."""
    b, e = w2.shape[:2]
    if w2.dtype != torch.float32 or w1x1.dtype != torch.float32 or not w2.is_contiguous() or not w1x1.is_contiguous() \
            or tuple(w2.shape[2:]) != (64, 64, 3, 3) or tuple(w1x1.shape) != (b, 3, 64, 64):
        raise ValueError("pack_mix_blocks: need contiguous fp32 (B,E,64,64,3,3) and (B,3,64,64)")
    if dst.dtype != torch.uint8 or dst.dim() != 2 or dst.shape[0] != b or dst.shape[1] < PACK_A_BYTES or dst.stride(1) != 1:
        raise ValueError("pack_mix_blocks: dst must be uint8 (B, >= PACK_A_BYTES)")
    lib = _lib.load()
    _lib.check(lib.pnp_pack_mix_blocks(_ptr(w2), _ptr(w1x1), b, e, _ptr(coef), _ptr(row_scale), _ptr(dst),
                                       dst.stride(0), _stream()), "pnp_pack_mix_blocks")


@_on_device_of
def caa_heads(base_qp, qp, params, n_experts):
    """base_qp/qp: fp32 (F,) -> experts (F,E), gamma (F,64).  params: dict of the six CAA tensors."""
    f = base_qp.numel()
    dev = base_qp.device
    experts = torch.empty((f, n_experts), dtype=torch.float32, device=dev)
    gamma = torch.empty((f, 64), dtype=torch.float32, device=dev)
    lib = _lib.load()
    _lib.check(lib.pnp_caa_heads(_ptr(base_qp), _ptr(qp), f, _ptr(params["b0w"]), _ptr(params["b0b"]),
                                 _ptr(params["b2w"]), _ptr(params["b2b"]), _ptr(params["s0w"]),
                                 _ptr(params["s2w"]), n_experts, params["s0w"].numel(), _ptr(experts),
                                 _ptr(gamma), _stream()), "pnp_caa_heads")
    return experts, gamma


@_on_device_of
def mix_bias(conv2_bias, experts, gamma):
    """conv2_bias (B,E,64), experts (F,E), gamma (F,64) -> (F,B,64)."""
    b, e, _ = conv2_bias.shape
    f = experts.shape[0]
    out = torch.empty((f, b, 64), dtype=torch.float32, device=experts.device)
    lib = _lib.load()
    _lib.check(lib.pnp_mix_bias(_ptr(conv2_bias), b, e, _ptr(experts), _ptr(gamma), f, _ptr(out),
                                _stream()), "pnp_mix_bias")
    return out


def fill_conv_desc(d, src, wpack, out=None, aux=None, idt=None, scale=None, bias=None, par=None,
                   act=PNP_ACT_NONE, lq=None, outf=None, flip_y=False, wpack_stable=False,
                   lq_up4=False, par_sparse=False, img_off=None):
    """Fill a ConvDesc in place (static launch: every operand is in the descriptor).  `out` may be a strided
    (N,H,W,64) view with unit channel stride (e.g. up[:, i::2, j::2, :]: pixel shuffle as the store epilogue).
    img_off: int64 (N,2) device tensor of per-image (weight byte offset, bias float offset) -> per-image launch."""
    n, h, w, _ = src.shape
    last = outf is not None
    d.src, d.aux, d.idt = src.data_ptr(), (aux.data_ptr() if aux is not None else None), \
        (idt.data_ptr() if idt is not None else None)
    d.out = out.data_ptr() if out is not None else None
    if out is not None and not out.is_contiguous():
        d.out_sn, d.out_sy, d.out_spx = out.stride(0), out.stride(1), out.stride(2)
    else:
        d.out_sn = d.out_sy = d.out_spx = 0
    d.lq_up4 = 1 if lq_up4 else 0
    d.par_sparse = 1 if (par_sparse and par is not None) else 0
    d.wpack = wpack.data_ptr()
    d.scale = scale.data_ptr() if scale is not None else None
    d.bias = bias.data_ptr() if bias is not None else None
    if par is not None:
        d.par, d.par_sn, d.par_sc, d.par_sy = par.data_ptr(), par.stride(0), par.stride(1), par.stride(2)
    else:
        d.par, d.par_sn, d.par_sc, d.par_sy = None, 0, 0, 0
    d.out_u8 = 0
    if last:
        d.lq, d.lq_sn, d.lq_sc, d.lq_sy = lq.data_ptr(), lq.stride(0), lq.stride(1), lq.stride(2)
        d.outf, d.of_sn, d.of_sc, d.of_sy = outf.data_ptr(), outf.stride(0), outf.stride(1), outf.stride(2)
        d.out_u8 = 1 if outf.dtype == torch.uint8 else 0
    else:
        d.lq, d.lq_sn, d.lq_sc, d.lq_sy = None, 0, 0, 0
        d.outf, d.of_sn, d.of_sc, d.of_sy = None, 0, 0, 0
    d.N, d.H, d.W = n, h, w
    d.tap_n = 16 if last else 64
    d.aux_k16 = 2 if aux is not None else 0
    d.aux_channels = int(aux.shape[3]) if aux is not None else 0
    d.act = act
    d.mode = PNP_CONV_LAST if last else PNP_CONV_BF16
    d.flip_y = 1 if flip_y else 0
    d.wpack_stable = 1 if wpack_stable else 0
    d.per_image = 1 if img_off is not None else 0
    d.img_off = img_off.data_ptr() if img_off is not None else None
    d.dyn.table, d.dyn.step, d.dyn.node, d.dyn.stride = None, None, 0, 0
    d.src_images = d.aux_images = d.idt_images = d.out_images = 0
    return d


@_on_device_of
def conv3x3(src, wpack, out=None, aux=None, idt=None, scale=None, bias=None, par=None,
            act=PNP_ACT_NONE, lq=None, outf=None, flip_y=False, wpack_stable=False, lq_up4=False,
            par_sparse=False, img_off=None):
    """Fused tcgen05 3x3 conv (see include/pnp_vcve.h: pnp_conv3x3).  `out` may be a strided view with unit
    channel stride (pixel shuffle as the store epilogue); lq_up4: lq is the (N,3,H/4,W/4) frame whose x4
    bilinear upsampling is added; img_off: per-image weight / bias offsets (one launch, N differently
    conditioned images).  A uint8 `outf` receives tensor2img's uint8 values of the fp32 result (out_u8)."""
    _feat_check(src, "src")
    for t, nm in ((out, "out"), (idt, "idt")):
        if t is not None:
            _feat_check(t, nm, strided=(nm == "out"))
            if t.shape != src.shape:
                raise ValueError(f"conv3x3: {nm} shape {tuple(t.shape)} != src {tuple(src.shape)}")
    if aux is not None:
        _aux_check(aux, "aux")
        if aux.shape[:3] != src.shape[:3]:
            raise ValueError(f"conv3x3: aux shape {tuple(aux.shape)} does not match src {tuple(src.shape)}")
    for t, nm in ((par, "par"), (lq, "lq"), (outf, "outf")):
        if t is not None:
            if nm == "outf" and t.dtype == torch.uint8:
                if t.stride(-1) != 1 or not t.is_cuda:
                    raise ValueError("outf must be a CUDA view with unit innermost stride")
            else:
                _plane_view_check(t, nm)
            hw = tuple(src.shape[1:3])
            if nm == "lq" and lq_up4:
                hw = (src.shape[1] // 4, src.shape[2] // 4)
            if t.dim() != 4 or t.shape[1] != 3 or t.shape[0] != src.shape[0] or tuple(t.shape[2:]) != hw:
                raise ValueError(f"conv3x3: {nm} must be (N,3,H,W) matching src" + (" / 4" if hw[0] != src.shape[1] else ""))
    if img_off is not None and (img_off.dtype != torch.int64 or tuple(img_off.shape) != (src.shape[0], 2) or
                                not img_off.is_contiguous() or not img_off.is_cuda):
        raise ValueError("conv3x3: img_off must be a contiguous int64 (N,2) CUDA tensor")
    d = fill_conv_desc(ConvDesc(), src, wpack, out, aux, idt, scale, bias, par, act, lq, outf, flip_y,
                       wpack_stable, lq_up4, par_sparse, img_off)
    need = rowstack_bytes(d.tap_n, aux is not None, par is not None)
    if img_off is None and wpack.numel() < need:
        raise ValueError("conv3x3: packed weight buffer too small for this configuration")
    lib = _lib.load()
    _lib.check(lib.pnp_conv3x3(ctypes.byref(d), _stream()), "pnp_conv3x3")
    return out if outf is None else outf
