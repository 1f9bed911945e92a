"""Compact codec side information -> dense generator inputs, on the GPU.

The reference ships 7 dense fp32 planes per pixel and frame to the GPU (``mvs`` 4 + ``partitions`` 3:
25.8 MB per 720p frame) after rasterising the per-block motion-vector records in a Python loop
(mmedit/datasets/pipelines/loading_ipb.py:328-369, up to 14 400 iterations per 720p frame).  Here the
records themselves (40 bytes per block) are uploaded and ``pnp_mv_rasterize`` produces exactly the
tensors the generator expects -- same integer truncation, numpy slice wrapping, record-order overwrite,
P-frame reversal into the previous non-B frame and partition one-hot/255 encoding.

Record layout (loading_ipb.py:339): direction, w, h, src_x, src_y, dst_x, dst_y, motion_x, motion_y, scale.
"""
import ctypes

import numpy as np
import torch

from . import _lib

SLICE_ORD = {"I": 73, "P": 80, "B": 66}


def p_targets(slice_types):
    """Frame that receives the reversed (direction>0) records of each non-B frame.

    loading_ipb.py:353-355,369: ``mvs[-p_offset]`` with ``p_offset = p_offset + 1 if B else 1`` updated
    after every frame, i.e. the previous non-B frame; -1 when ``p_offset`` is still unbound (first frame)
    or would point before the clip.
    """
    tgt, p_off = [], None
    for f, st in enumerate(slice_types):
        t = -1
        if st != "B" and p_off is not None and f - p_off >= 0:
            t = f - p_off
        tgt.append(t)
        p_off = (p_off + 1) if (st == "B" and p_off is not None) else 1
    return tgt


def _launch(rec, offs, is_b, tgt, t, h, w, work, mvs, par, status, tail=None):
    """pnp_mv_rasterize on the current stream of the tensors' device; ``work`` (3,T,H,W) int32 must be zeroed.
    ``tail`` (0 or 1) makes it pnp_mv_rasterize_window on a ``window_side`` table of T frames + ``tail`` tail frames."""
    lib = _lib.load()
    vp = ctypes.c_void_p
    stream = vp(torch.cuda.current_stream(mvs.device).cuda_stream)
    head = (vp(rec.data_ptr() if rec.numel() else 0), vp(offs.data_ptr()), vp(is_b.data_ptr()), vp(tgt.data_ptr()), t)
    rest = (rec.shape[0], h, w, vp(work[0].data_ptr()), vp(work[1].data_ptr()), vp(work[2].data_ptr()),
            vp(mvs.data_ptr()), vp(par.data_ptr()), vp(status.data_ptr()), stream)
    if tail is None:
        _lib.check(lib.pnp_mv_rasterize(*head, *rest), "pnp_mv_rasterize")
    else:
        _lib.check(lib.pnp_mv_rasterize_window(*head, int(tail), *rest), "pnp_mv_rasterize_window")


def raise_for_status(st):
    """The reference's loader errors for a device status word of pnp_mv_rasterize."""
    if st & 1:
        raise KeyError("block area w*h not in {256, 128, 64} (partition_ch lookup, loading_ipb.py:361)")
    if st & 2:
        raise ValueError("reversed P-frame record without a previous non-B frame (p_offset unbound)")


def rasterize_clip(records, frame_offsets, slice_types, h, w, device=None, check=True):
    """records (R,10) fp32, frame_offsets (T+1,) int, slice_types: sequence of 'I'|'P'|'B'.

    Returns (mvs (T,4,H,W), partitions (T,3,H,W)) fp32 on ``device`` -- the per-clip tensors of the
    reference pipeline after ``FramesToTensor`` (add a leading batch dim for the generator).
    ``check`` synchronises once and raises like the reference (KeyError for a block area outside
    {256,128,64}; ValueError for a reversed record without a target frame).
    """
    dev = torch.device(device if device is not None else "cuda")
    t = len(slice_types)
    rec = torch.as_tensor(np.asarray(records, dtype=np.float32).reshape(-1, 10)).to(dev).contiguous()
    offs = torch.as_tensor(np.asarray(frame_offsets, dtype=np.int32)).to(dev)
    if offs.numel() != t + 1:
        raise ValueError("frame_offsets must have T+1 entries")
    is_b = torch.tensor([1 if s == "B" else 0 for s in slice_types], dtype=torch.int32, device=dev)
    tgt = torch.tensor(p_targets(slice_types), dtype=torch.int32, device=dev)
    work = torch.zeros((3, t, h, w), dtype=torch.int32, device=dev)        # owner fwd / bwd, partition bits
    mvs = torch.empty((t, 4, h, w), dtype=torch.float32, device=dev)
    par = torch.empty((t, 3, h, w), dtype=torch.float32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _launch(rec, offs, is_b, tgt, t, h, w, work, mvs, par, status)
    if check:
        raise_for_status(int(status.item()))
    return mvs, par


def pack_side(records, frame_offsets, slice_types):
    """Host form of one clip's side information for ``driver.ClipStreamer`` / ``driver.enhance_clips`` (the ``side``
    entry of a host clip that carries no dense ``mvs`` / ``partitions``): pinned records (R,10) fp32 and ONE pinned
    int32 vector [frame_offsets (T+1) | is_b (T) | p_target (T)] -- two contiguous uploads per clip."""
    t = len(slice_types)
    rec = torch.as_tensor(np.ascontiguousarray(np.asarray(records, dtype=np.float32).reshape(-1, 10)))
    offs = np.asarray(frame_offsets, dtype=np.int32).reshape(-1)
    if offs.size != t + 1:
        raise ValueError("frame_offsets must have T+1 entries")
    meta = np.concatenate([offs, np.asarray([1 if s == "B" else 0 for s in slice_types], dtype=np.int32),
                           np.asarray(p_targets(slice_types), dtype=np.int32)])
    return _pinned_side(rec, torch.as_tensor(meta), t=t)


def _pinned_side(rec, meta, **kw):
    pin = torch.cuda.is_available()
    return dict(records=rec.pin_memory() if pin else rec, meta=meta.pin_memory() if pin else meta, **kw)


def window_side(side, a, b):
    """The packed side information of frames [a, b) of a clip, from the clip's ``pack_side`` entry: rasterised by
    ``pnp_mv_rasterize_window``, it gives exactly frames [a, b) of the whole clip's planes.

    Records: those of frames [a, b), then -- as a tail frame -- the direction>0 rows of frame e, the first non-B frame
    >= b, when their target (the previous non-B frame) lies inside the window: no other later frame writes into it.
    ``meta`` is [frame_offsets (n+1) | is_b (n) | p_target (n)] of the n = (b - a) + tail table frames, window-relative;
    a target before the window becomes -2 (the write lands outside it), -1 (frame 0 of the clip has no target) stays.
    Returns the ``pack_side`` form plus ``tail`` (0 or 1)."""
    t = side["t"]
    if not 0 <= a < b <= t:
        raise ValueError(f"window [{a}, {b}) is not inside a clip of {t} frames")
    meta = side["meta"].tolist()
    offs, is_b, tgt = meta[:t + 1], meta[t + 1:2 * t + 1], meta[2 * t + 1:]
    rec = side["records"]
    parts = [rec[offs[a]:offs[b]]]
    rel = [v - a if v >= a else (-2 if v >= 0 else v) for v in tgt[a:b]]
    w_offs = [o - offs[a] for o in offs[a:b + 1]]
    w_is_b = list(is_b[a:b])
    e = next((f for f in range(b, t) if not is_b[f]), None)
    tail = int(e is not None and tgt[e] >= a)
    if tail:
        rows = rec[offs[e]:offs[e + 1]]
        rows = rows[rows[:, 0] > 0]
        parts.append(rows)
        w_offs.append(w_offs[-1] + rows.shape[0])
        w_is_b.append(0)
        rel.append(tgt[e] - a)
    return _pinned_side(torch.cat(parts, 0).contiguous(), torch.tensor(w_offs + w_is_b + rel, dtype=torch.int32),
                        t=b - a, tail=tail)


def mv_record_path(frame_path, dataset="reds"):
    """Where the reference's loader finds the motion-vector records of an LQ frame (loading_ipb.py:316-323):
    ``.../png/.../00000012.png -> .../mv/.../00000012.npy``; vimeo septuplets ``.../png/.../im3.png -> .../mv/.../00000002.npy``;
    KITTI pairs (loading_ipb_kitti.py, same raster loop) ``<root>/png/.../000012_11.png -> <root>/mv/000012/00000001.npy``."""
    import os
    if dataset == "vimeo":
        d, idx = frame_path.split("/im")
        return os.path.join(d.replace("png", "mv"), "{:08d}.npy".format(int(idx.split(".png")[0]) - 1))
    if dataset == "kitti":
        # loading_ipb_kitti.py:102-103,127-129: frames are named <sequence>_<index>.png, index 10 is the first frame
        name = os.path.basename(frame_path)
        seq, idx = name.split("_")[0], name.split("_")[1].split(".")[0]
        return "{}/mv/{}/{:08d}.npy".format(frame_path.split("/png/")[0], seq, int(idx) - 10)
    return frame_path.replace(".png", ".npy").replace("png", "mv")


def side_from_files(frame_paths, slice_types, dataset="reds"):
    """The compact feed of one clip straight from the files the reference's loader reads: per LQ frame path the ``.npy``
    record table next to it (``np.load(...).astype(np.float32)``, loading_ipb.py:325; an I frame's table may be empty or
    missing rows) -> ``pack_side``.  Replaces the raster loop of ``LoadImageFromFileList_ipb`` (:328-369) plus
    ``RescaleToZeroOne`` / ``FramesToTensor`` on ``mvs`` / ``partitions``: the planes are built on the GPU instead."""
    if len(frame_paths) != len(slice_types):
        raise ValueError("one slice type per frame path")
    tables = [np.load(mv_record_path(str(p), dataset)).astype(np.float32).reshape(-1, 10) for p in frame_paths]
    flat = np.concatenate(tables, 0) if tables else np.zeros((0, 10), np.float32)
    offs = np.cumsum([0] + [len(tb) for tb in tables])
    return pack_side(flat, offs, list(slice_types))


def upload_side(side, device):
    """Enqueue the two H2D copies of one clip's packed side information (``pack_side``) on the current stream;
    returns the device tensors (records, meta) and the bytes that cross the bus."""
    rec = side["records"].to(device, non_blocking=True)
    meta = side["meta"].to(device, non_blocking=True)
    return rec, meta, rec.numel() * 4 + meta.numel() * 4


def rasterize_uploaded(rec, meta, t, mvs, par, work, status, tail=None):
    """Rasterise uploaded side information (``upload_side``) into ``mvs`` (T,4,H,W) / ``par`` (T,3,H,W) on the CURRENT
    stream without any host synchronisation; ``work`` (3,T,H,W) int32 is zeroed here, ``status`` accumulates the error
    bits (check it with ``raise_for_status`` after a synchronisation).  ``tail``: the entry is a frame window
    (``window_side``) of T frames with that many (0 or 1) tail frames; None: a whole clip (``pack_side``)."""
    h, w = mvs.shape[-2], mvs.shape[-1]
    n = t + (tail or 0)
    if tuple(mvs.shape) != (t, 4, h, w) or tuple(par.shape) != (t, 3, h, w) or meta.numel() != 3 * n + 1:
        raise ValueError(f"side information of {t} frames does not match outputs {tuple(mvs.shape)} / {tuple(par.shape)}")
    work.zero_()
    _launch(rec, meta[:n + 1], meta[n + 1:2 * n + 1], meta[2 * n + 1:], t, h, w, work, mvs, par, status, tail)


def synthetic_records(h, w, pattern, seed=0, messy=False):
    """Seeded per-frame record lists with the structure of an H.264 partition tree.

    Every frame but I frames is tiled with 16x16 macroblocks split at random into 16x16 / 16x8 / 8x16 /
    8x8 blocks (areas 256 / 128 / 64); motion in quarter pels with scale 4.  B frames carry forward and
    (for a random subset) backward records, P frames forward records plus direction>0 records that the
    loader reverses into the previous non-B frame.  ``messy`` adds what the loader tolerates: blocks
    hanging over the frame edges (numpy slice wrapping), duplicates (overwrite order), direction 0 rows.
    """
    rng = np.random.RandomState(seed)
    frames = []
    for f, st in enumerate(pattern):
        rows = []
        if st != "I":
            for y0 in range(0, h, 16):
                for x0 in range(0, w, 16):
                    split = rng.randint(0, 4)
                    blocks = {0: [(0, 0, 16, 16)], 1: [(0, 0, 16, 8), (0, 8, 16, 8)],
                              2: [(0, 0, 8, 16), (8, 0, 8, 16)],
                              3: [(0, 0, 8, 8), (8, 0, 8, 8), (0, 8, 8, 8), (8, 8, 8, 8)]}[split]
                    for (bx, by, bw, bh) in blocks:
                        cx, cy = x0 + bx + bw // 2, y0 + by + bh // 2
                        mx, my = rng.randint(-64, 65), rng.randint(-64, 65)
                        sx, sy = cx + mx // 4, cy + my // 4
                        rows.append([-1, bw, bh, sx, sy, cx, cy, mx, my, 4])
                        if st == "B" and rng.rand() < 0.6:
                            rows.append([1, bw, bh, cx - mx // 4, cy - my // 4, cx, cy, -mx, -my, 4])
                        if st == "P" and f > 0 and rng.rand() < 0.5:
                            rows.append([1, bw, bh, sx, sy, cx, cy, mx, my, 4])
            if messy and rows:
                for _ in range(12):
                    r = list(rows[rng.randint(0, len(rows))])
                    kind = rng.randint(0, 4)
                    if kind == 0:          # hangs over the top/left edge: negative slice start wraps
                        r[5], r[6] = rng.randint(-6, 4), rng.randint(-6, 4)
                    elif kind == 1:        # hangs over the bottom/right edge: clamped
                        r[5], r[6] = w - rng.randint(0, 6), h - rng.randint(0, 6)
                    elif kind == 2:        # duplicate with another vector: later record wins
                        r[7], r[8] = rng.randint(-64, 65), rng.randint(-64, 65)
                    else:                  # direction 0: partition only
                        r[0] = 0
                    if r[0] > 0 and st == "P":
                        r[3], r[4] = rng.randint(-8, w + 8), rng.randint(-8, h + 8)
                    rows.append(r)
        frames.append(np.asarray(rows, dtype=np.float32).reshape(-1, 10))
    return frames
