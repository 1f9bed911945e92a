"""Quality metrics of the reference's test loop without leaving the GPU.

``BasicVSR.evaluate`` (mmedit/models/restorers/basicvsr.py:119-153) moves every output / GT frame to the host,
quantises it to uint8 (``tensor2img``, mmedit/core/misc.py:9-74) and calls ``psnr`` / ``ssim``
(mmedit/core/evaluation/metrics.py:170-215, 262-355) in numpy / OpenCV -- 2 T device->host copies and syncs per
clip.  Here ``pnp_frame_quality`` accumulates the exact integer squared error and the float64 SSIM-map sums per
frame on the device; the few remaining scalar operations are torch ops on the same stream, so a whole clip's
metrics are one small tensor that can go straight into the fixed-shape gather of ``driver.gather_metrics``.
convert_to=None only (what the shipped configs use).  Either operand may also be an 8-bit frame (uint8, the value
tensor2img would produce), read as is: a uint8 GT scores exactly like the fp32 GT ``gt / 255`` it was decoded to.
"""
import math

import torch

from . import _lib
from .ops import _ptr, _stream

_DTYPES = (torch.float32, torch.uint8)


def frame_quality(out, gt, crop_border=0):
    """out, gt: (n,T,3,H,W) (or (F,3,H,W)) fp32 or uint8 CUDA tensors with unit innermost stride (fp32 frames are
    quantised like tensor2img, uint8 frames are taken as they are).

    Returns dict(psnr, ssim: float64, sse: int64), each shaped like the leading dims, on the device, no host sync.
    """
    if out.shape != gt.shape or out.shape[-3] != 3 or out.dim() not in (4, 5):
        raise ValueError(f"frame_quality: shapes {tuple(out.shape)} / {tuple(gt.shape)} must match (...,3,H,W)")
    if out.dtype not in _DTYPES or gt.dtype not in _DTYPES or not out.is_cuda or not gt.is_cuda:
        raise ValueError("frame_quality: fp32 or uint8 CUDA tensors expected (there is no CPU path)")
    lead = out.shape[:-3]
    h, w = out.shape[-2:]
    a = out.reshape(-1, 3, h, w)
    b = gt.reshape(-1, 3, h, w)
    if a.stride(-1) != 1:
        a = a.contiguous()
    if b.stride(-1) != 1:
        b = b.contiguous()
    f = a.shape[0]
    c = int(crop_border)
    sse = torch.empty(f, dtype=torch.int64, device=out.device)
    ssum = torch.empty((f, 3), dtype=torch.float64, device=out.device)
    lib = _lib.load()
    with torch.cuda.device(out.device):
        rc = lib.pnp_frame_quality_u8(_ptr(a), int(a.dtype == torch.uint8), a.stride(0), a.stride(1), a.stride(2),
                                      _ptr(b), int(b.dtype == torch.uint8), b.stride(0), b.stride(1), b.stride(2), f, h,
                                      w, c, _ptr(sse), _ptr(ssum), _stream())
    _lib.check(rc, "pnp_frame_quality")
    npix = 3 * (h - 2 * c) * (w - 2 * c)
    mse = sse.to(torch.float64) / npix
    psnr = torch.where(sse == 0, torch.full_like(mse, math.inf), 20.0 * torch.log10(255.0 / torch.sqrt(mse)))
    nwin = (h - 2 * c - 10) * (w - 2 * c - 10)
    ssim = (ssum / nwin).mean(dim=1) if c == 0 else ssum[:, 0] / nwin      # crop quirk: first BGR channel only
    return dict(psnr=psnr.view(lead), ssim=ssim.view(lead), sse=sse.view(lead))


def evaluate(out, gt, crop_border=0, metrics=("PSNR", "SSIM")):
    """``BasicVSR.evaluate`` for a sequence (n,T,3,H,W): per-frame metrics averaged over the frames
    (basicvsr.py:137-145).  Returns {name: 0-d float64 device tensor}; call ``.item()`` when you need the number."""
    q = frame_quality(out, gt, crop_border)
    res = {}
    for m in metrics:
        if m not in ("PSNR", "SSIM"):
            raise KeyError(m)
        res[m] = q[m.lower()].mean()
    return res
