"""PNG files of 8-bit frames, encoded on the device (``pnp_png_encode``).

The reference's test loop saves every output frame with ``mmcv.imwrite(tensor2img(frame))`` (tools/test.py
--save-path, ``forward_test(save_image=True)``).  ``encode`` turns the uint8 frames that ``conv_last`` stores
(``out_dtype=torch.uint8``) into complete PNG files where they are, so the host does no compression and only writes
bytes.  The output buffer holds ``frame_bound`` bytes per frame (the raw scanlines plus block and chunk headers), so
downloading it whole moves slightly more than the uint8 frame itself.  A file holds exactly its uint8 frame as 8-bit
RGB (red = channel 0, what OpenCV makes of the BGR array), padded frames at their padded size; its pixels equal
OpenCV's, its compressed bytes do not.
"""
import ctypes
import os

import torch

from . import _lib
from .ops import _frames_view, _on_device_of, _ptr, _stream


def frame_bound(h, w):
    """Exact size of the largest PNG file of an h x w frame (every segment a stored block), chunk framing included."""
    n = _lib.load().pnp_png_frame_bound(int(h), int(w))
    if n < 0:
        _lib.check(int(n), "pnp_png_frame_bound")
    return int(n)


@_on_device_of
def encode(frames_u8, out=None, sizes=None):
    """uint8 (F,3,H,W) or (n,T,3,H,W) device view, unit x stride -> (out, sizes): PNG f is ``out[f, :sizes[f]]``.

    ``out`` is a (F, >= frame_bound(H, W)) uint8 device tensor with unit inner stride and ``sizes`` an (F,) int64 device
    tensor (both allocated when not given).  Runs on the current stream; nothing is synchronised."""
    f = _frames_view(frames_u8, "frames_u8", torch.uint8)
    n, _, h, w = f.shape
    bound = frame_bound(h, w)
    if out is None:
        out = torch.empty((n, bound), dtype=torch.uint8, device=f.device)
    if sizes is None:
        sizes = torch.empty(n, dtype=torch.int64, device=f.device)
    if out.dtype != torch.uint8 or out.dim() != 2 or out.shape[0] != n or out.shape[1] < bound or \
            out.stride(1) != 1 or out.device != f.device:
        raise ValueError(f"out must be a ({n}, >= {bound}) uint8 tensor on {f.device} with unit inner stride, got "
                         f"{tuple(out.shape)} {out.dtype}")
    if sizes.dtype != torch.int64 or tuple(sizes.shape) != (n,) or sizes.stride(0) != 1 or sizes.device != f.device:
        raise ValueError(f"sizes must be a contiguous ({n},) int64 tensor on {f.device}")
    if n == 0:
        return out, sizes
    lib = _lib.load()
    nbytes = lib.pnp_png_workspace_bytes(n, h, w)
    if nbytes < 0:
        _lib.check(int(nbytes), "pnp_png_workspace_bytes")
    work = torch.empty(int(nbytes), dtype=torch.uint8, device=f.device)    # (stream ordered: reused after this call)
    _lib.check(lib.pnp_png_encode(_ptr(f), f.stride(0), f.stride(1), f.stride(2), n, h, w, _ptr(out),
                                  out.stride(0), _ptr(sizes), _ptr(work), ctypes.c_int64(int(nbytes)), _stream()),
               "pnp_png_encode")
    return out, sizes


def write(buf_host, sizes_host, paths):
    """Write PNG k (``buf_host[k, :sizes_host[k]]``, host tensors) to ``paths[k]``; a path of None is skipped.  Parent
    directories are created, as ``mmcv.imwrite(auto_mkdir=True)`` does.  Raises OSError."""
    sizes = sizes_host.tolist()
    for k, path in enumerate(paths):
        if path is None:
            continue
        path = os.fspath(path)
        parent = os.path.dirname(path)
        if parent:
            os.makedirs(parent, exist_ok=True)
        with open(path, "wb") as fh:
            fh.write(memoryview(buf_host[k, :sizes[k]].numpy()))


def save_frames(frames_u8, path_of):
    """Encode device frames (n,T,3,H,W) uint8 and write frame (j, i) to ``path_of(j, i)`` (None skips it), before
    returning.  For frames that stay on the device; host-resident clips are saved by ``driver.ClipStreamer``."""
    for j in range(frames_u8.shape[0]):
        paths = [path_of(j, i) for i in range(frames_u8.shape[1])]
        if all(p is None for p in paths):
            continue
        buf, sizes = encode(frames_u8[j])
        sizes_h = sizes.cpu()
        write(buf[:, :int(sizes_h.max())].cpu(), sizes_h, paths)
