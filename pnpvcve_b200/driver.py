"""Clip-sharded / frame-window-sharded multi-GPU driver: one process per GPU, no data-path collective.

The reference shards its test set by rank-strided sampling (mmedit/datasets/samplers/
distributed_sampler.py:51-72) and gathers pickled results with two all_gathers
(mmedit/apis/test.py:190-234).  Clips are independent, so here clip ``c`` goes to rank
``c mod world`` and the only communication is ONE fixed-shape all_gather of per-frame metrics.
"""
import threading
import weakref
from concurrent.futures import ThreadPoolExecutor

import torch
import torch.distributed as dist

from . import pngio

N_METRICS = 2  # per frame: max-abs error vs. a reference frame (or 0), mean squared error


def shard_clips(num_clips, rank, world):
    """Rank-strided clip indices (clip c -> rank c % world)."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError(f"bad rank/world: {rank}/{world}")
    return list(range(rank, num_clips, world))


def clips_per_rank(num_clips, world):
    return (num_clips + world - 1) // world


def _unit(x):
    """Frames in [0,1] units: 8-bit frames as float32(v) / 255 (the loader's RescaleToZeroOne), others as they are."""
    return x.float() / 255.0 if x.dtype == torch.uint8 else x


def frame_metrics(out, ref=None):
    """out (n,T,3,H,W) -> (n,T,N_METRICS) fp32 on the same device (no host sync).  uint8 frames (out or ref) are
    compared in [0,1] units, so max-abs and mse mean the same for fp32 and 8-bit frames."""
    out = _unit(out)
    d = out.float() if ref is None else (out - _unit(ref)).float()
    return torch.stack([d.abs().amax(dim=(2, 3, 4)), (d * d).mean(dim=(2, 3, 4))], dim=-1)


def gather_metrics(local, num_clips, rank, world, group=None):
    """local: (len(shard_clips), T, N_METRICS) -> (num_clips, T, N_METRICS) in clip order on every rank.

    One all_gather of a fixed-shape tensor (ranks with fewer clips pad with NaN rows).
    """
    per = clips_per_rank(num_clips, world)
    t = local.shape[1] if local.dim() == 3 else 0
    nm = local.shape[2] if local.dim() == 3 else N_METRICS      # any per-frame metric vector (e.g. + PSNR, SSIM)
    padded = torch.full((per, t, nm), float("nan"), dtype=torch.float32, device=local.device)
    padded[: local.shape[0]] = local
    if world == 1:
        parts = [padded]
    else:
        parts = [torch.empty_like(padded) for _ in range(world)]
        dist.all_gather(parts, padded, group=group)
    full = torch.empty((num_clips, t, nm), dtype=torch.float32, device=local.device)
    for r in range(world):
        idx = shard_clips(num_clips, r, world)
        if idx:
            full[idx] = parts[r][: len(idx)]
    return full


@torch.no_grad()
def enhance_clips(net, clips, rank=0, world=1, refs=None, gts=None, crop_border=0, device=None, out_hosts=None,
                  chunk=10, out_dtype=torch.float32, save_png=None):
    """Run this rank's share of ``clips``: a list of clip dicts as produced by pnpvcve_b200.synthetic, each holding
    n >= 1 equally shaped clips (n, T, ...); entries of other ranks may be None.

    Device-resident entries are enhanced in place; HOST-resident entries (CPU tensors, pinned or not) stream through
    ``ClipStreamer`` on ``device``: chunked uploads and downloads overlap the kernels, the upload of the next entry
    overlaps the kernels of the current one, and the frames land in ``out_hosts[c]`` (pinned buffers, allocated here
    when not given).  Returns (outputs of the local entries -- device tensors, or the pinned host buffers --, gathered
    metrics (num_entries * n, T, M) for all clips on every rank).  With ``gts`` (ground truth, (n,T,3,H,W) per entry) the
    per-frame metric vector is [max-abs, mse, PSNR, SSIM]: PSNR / SSIM as BasicVSR.evaluate computes them
    (mmedit/models/restorers/basicvsr.py:119-153), but on the device (pnpvcve_b200.metrics) -- the reference's test loop
    copies every frame to the host and pickles per-clip results through two all_gathers (mmedit/apis/test.py:190-234);
    here nothing but the frames themselves leaves the GPU before the single fixed-shape gather.

    8-bit frames: ``lq`` may be uint8 (value v stands for float32(v) / 255, what the reference's loader makes of a PNG),
    and ``out_dtype=torch.uint8`` returns tensor2img's uint8 frames (mmedit/core/misc.py:9-74) of the fp32 result,
    stored by the last conv itself -- same (n,T,3,H,W) layout, a quarter of the bytes over the bus and in pinned
    memory.  ``out_hosts`` must then be uint8; ``gts`` / ``refs`` may be uint8 too.

    ``save_png``: a callable (clip, frame) -> path that saves every frame as a PNG file, as the reference's
    ``forward_test(save_image=True)`` does with ``mmcv.imwrite(tensor2img(...))``; clip is the row of the returned
    metrics (``entry * n + j``).  mmedit's naming is one such callable:
    ``lambda c, i: f"{save_path}/{folders[c]}/{i:08d}.png"``.  Needs ``out_dtype=torch.uint8``.  The files are encoded
    on the device (``pngio``, pixel-identical to OpenCV's).  The frames of host entries are not downloaded -- their PNG
    buffers are, written by host threads while later frames are computed -- and their ``outs`` are None;
    device-resident entries return their frames as before.  The call returns after every file has been written and
    raises the first OSError of a write.
    """
    from .synthetic import generator_args
    from . import metrics as _metrics
    if out_dtype not in (torch.float32, torch.uint8):
        raise ValueError(f"out_dtype must be torch.float32 or torch.uint8, got {out_dtype}")
    if save_png is not None and out_dtype != torch.uint8:
        raise ValueError("save_png needs out_dtype=torch.uint8 (PNG files hold tensor2img's uint8 frames)")
    if save_png is not None and out_hosts is not None:
        raise ValueError("save_png does not download the frames of host entries; leave out_hosts at None")
    if out_hosts is not None:
        bad = [c for c, o in enumerate(out_hosts) if o is not None and o.dtype != out_dtype]
        if bad:
            raise ValueError(f"out_hosts[{bad[0]}] is {out_hosts[bad[0]].dtype}, out_dtype is {out_dtype}")
    mine = shard_clips(len(clips), rank, world)
    first = next(c for c in clips if c is not None)["lq"]
    shape_of = first.shape
    n, t = shape_of[:2]
    host = not first.is_cuda                 # (a rank without work of its own still takes part in the gather, on its GPU)
    dev = torch.device(device) if device is not None else \
        (torch.device("cuda", torch.cuda.current_device()) if host else first.device)
    outs, mets = [], []

    def measure(c, out):
        m = frame_metrics(out, None if refs is None else refs[c].to(out.device))
        if gts is not None:
            q = _metrics.frame_quality(out, gts[c].to(out.device), crop_border)
            m = torch.cat([m, q["psnr"].float()[..., None], q["ssim"].float()[..., None]], dim=-1)
        mets.append(m)

    if host and mine:
        up = 4 if getattr(net, "vsr", False) else 1
        # (`side`: compact side information packed by sideinfo.pack_side, already pinned -- see ClipStreamer.upload)
        pinned = {c: {k: (v if k == "side" or v.is_pinned() else v.pin_memory()) for k, v in clips[c].items()}
                  for c in mine}
        streamer = streamer_for(net, dev, chunk)
        ticket = streamer.upload(pinned[mine[0]])
        for i, c in enumerate(mine):
            oshape = (n, t, 3, shape_of[-2] * up, shape_of[-1] * up)
            if save_png is not None:        # the frames stay on the device (a meta tensor carries shape and dtype)
                dst = torch.empty(oshape, dtype=out_dtype, device="meta")
                png = lambda j, k, c=c: save_png(c * n + j, k)        # noqa: E731
            else:
                dst = out_hosts[c] if out_hosts is not None else torch.empty(oshape, dtype=out_dtype).pin_memory()
                png = None
            out = streamer.run(ticket, dst) if png is None else streamer.run(ticket, dst, png=png)
            ticket = streamer.upload(pinned[mine[i + 1]]) if i + 1 < len(mine) else None   # overlaps clip c's kernels
            measure(c, out)                 # on the device copy, before its buffer is recycled two entries later
            outs.append(None if save_png is not None else dst)
        streamer.finish(check=True)
    else:
        for c in mine:
            if out_dtype == torch.uint8:
                lq = clips[c]["lq"]
                up = 4 if getattr(net, "vsr", False) else 1
                buf = torch.empty(tuple(lq.shape[:3]) + ((lq.shape[3] + 3) // 4 * 4 * up, (lq.shape[4] + 3) // 4 * 4 * up),
                                  dtype=torch.uint8, device=lq.device)
                out = net.forward_streamed(*generator_args(clips[c]), out=buf)
            else:
                out = net(*generator_args(clips[c]))
            outs.append(out)
            measure(c, out)
            if save_png is not None:
                pngio.save_frames(out, lambda j, k, c=c: save_png(c * n + j, k))
    nm = N_METRICS + (2 if gts is not None else 0)
    local = torch.cat(mets, 0) if mets else torch.empty((0, t, nm), device=dev)
    per_entry = gather_metrics(local.view(len(mine), n * t, nm) if mets else local.view(0, n * t, nm),
                               len(clips), rank, world)
    return outs, per_entry.view(len(clips) * n, t, nm)


# ------------------------------------------------------------------------------------------------
# frame-window sharding: ONE long clip (or a few) spread over the GPUs
# ------------------------------------------------------------------------------------------------
def frame_windows(t, window):
    """Consecutive windows [a, b) of at most ``window`` frames, as the reference's recurrent inference with
    ``max_seq_len`` cuts a sequence (mmedit/apis/restoration_video_inference.py:121-128: ``data[:, i:i + max_seq_len]``
    for i in range(0, T, max_seq_len), results concatenated).  Every window is enhanced as a clip of its own, so its
    first and last frame become forced key frames (iconvsr_ipb_par.py:61-62) and no state crosses a window border."""
    if window < 1:
        raise ValueError(f"window must be >= 1, got {window}")
    return [(a, min(a + window, t)) for a in range(0, t, window)]


def balanced_window(t, world, min_window=2):
    """Window length that cuts a T-frame clip into ``world`` windows of (almost) equal length."""
    return max(min_window, (t + world - 1) // world)


def shard_windows(num_clips, t, window, rank, world):
    """This rank's (clip, a, b) work items: the windows of all clips in (clip, window) order, item k -> rank k % world."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError(f"bad rank/world: {rank}/{world}")
    items = [(c, a, b) for c in range(num_clips) for a, b in frame_windows(t, window)]
    return items[rank::world]


def clip_window(clip, a, b, overlap=0):
    """Views of frames [a - overlap, b + overlap) (clamped to the clip) of every tensor of a clip dict, and the position
    [lo, hi) of the core frames [a, b) inside that window.  ``overlap`` > 0 runs extra context frames whose outputs are
    discarded: the forced key frames then sit ``overlap`` frames away from the frames that are kept, which bounds the
    seam error against the uncut clip at the price of (2 overlap / window) extra work.  overlap = 0 is the reference's
    ``max_seq_len`` semantics exactly.  Compact side information (``side``) is cut by ``sideinfo.window_side``: the
    window's records plus the ones a later frame writes into it, new pinned host tensors."""
    t = clip["lq"].shape[1]
    a0, b0 = max(0, a - overlap), min(t, b + overlap)
    win = {k: v[:, a0:b0] for k, v in clip.items() if k != "side"}
    if "side" in clip:
        from . import sideinfo
        win["side"] = [sideinfo.window_side(sd, a0, b0) for sd in clip["side"]]
    return win, a - a0, b - a0


def _pinned(v):
    """``v`` itself when it is already contiguous pinned memory (a window of a pinned clip is), else a pinned copy;
    without a CUDA device (the CPU tests of the sharding logic) a contiguous one."""
    if not torch.cuda.is_available():
        return v.contiguous()
    return v if v.is_contiguous() and v.is_pinned() else v.contiguous().pin_memory()


@torch.no_grad()
def enhance_windows(net, clips, window, rank=0, world=1, overlap=0, refs=None, gather_output=False, group=None,
                    device=None, chunk=10, gts=None, crop_border=0, out_dtype=torch.float32, save_png=None):
    """Frame-window sharding (north_star: "sharding independent clips or frame windows per GPU"): the windows of
    ``clips`` (equally shaped (1,T,...) clip dicts) are dealt to the ranks round robin and enhanced independently.
    HOST-resident clips stream their windows through the cached ``ClipStreamer`` of (net, device, chunk) on ``device``
    (only a rank's own windows ever reach its GPU), device-resident clips are sliced in place.

    A host clip may carry ``side`` (one ``sideinfo.pack_side`` entry of the whole clip) instead of the dense ``mvs`` /
    ``partitions``: each rank uploads only the records of its own windows (``sideinfo.window_side``, overlap included)
    and rasterises them on the device, bit-identical to the same frames of the whole clip's planes.  Device-resident
    clips and stand-in callables take dense planes only.

    8-bit frames: ``lq`` may be uint8, and ``out_dtype=torch.uint8`` returns tensor2img's uint8 frames, stored by the
    last conv (as in ``enhance_clips``).  ``gts`` (per clip (1,T,3,H,W), fp32 or uint8) adds PSNR / SSIM
    (``metrics.frame_quality`` with ``crop_border``) to every frame's metric vector: [max-abs, mse, PSNR, SSIM].

    ``save_png``: a callable (clip, frame) -> path, frame counted in the whole clip, that saves the core frames of every
    window (never its overlap frames) as PNG files encoded on the device, as in ``enhance_clips`` -- so each frame of a
    clip is written exactly once, by the rank that owns it.  Needs ``out_dtype=torch.uint8`` and excludes
    ``gather_output``; the frames of host clips are then not downloaded.

    Returns (outs, metrics): outs = {(clip, a, b): (1, b-a, 3, H, W) frames} of this rank's windows (device tensors)
    -- or, with ``gather_output``, the complete (num_clips, T, 3, H, W) result on every rank (one fixed-shape all_gather
    of frames over NVLink, in ``out_dtype``) --, metrics = (num_clips, T, M) of ALL frames on every rank (one
    fixed-shape all_gather).  No collective touches the data path of a window."""
    from .synthetic import generator_args
    from . import metrics as _metrics
    if out_dtype not in (torch.float32, torch.uint8):
        raise ValueError(f"out_dtype must be torch.float32 or torch.uint8, got {out_dtype}")
    if save_png is not None and out_dtype != torch.uint8:
        raise ValueError("save_png needs out_dtype=torch.uint8 (PNG files hold tensor2img's uint8 frames)")
    if save_png is not None and gather_output:
        raise ValueError("save_png writes each rank's own windows; it cannot be combined with gather_output")
    num_clips = len(clips)
    t = clips[0]["lq"].shape[1]
    # host-resident clips are streamed when `net` is the generator (anything else -- a stand-in callable in the CPU tests
    # of the sharding logic -- is simply called on the tensors where they are)
    host = not clips[0]["lq"].is_cuda and hasattr(net, "forward_streamed")
    if not host and any("side" in c for c in clips):
        raise ValueError("frame windows of device-resident clips are cut from dense mvs / partitions planes; rasterise "
                         "compact side information first (pnpvcve_b200.sideinfo.rasterize_clip) or pass host clips")
    dev = torch.device(device) if device is not None else \
        (torch.device("cuda", torch.cuda.current_device()) if host else clips[0]["lq"].device)
    mine = shard_windows(num_clips, t, window, rank, world)
    up = 4 if getattr(net, "vsr", False) else 1
    outs = {}
    nm = N_METRICS + (2 if gts is not None else 0)
    local = torch.full((num_clips, t, nm), float("nan"), dtype=torch.float32, device=dev)
    streamer, ticket, wins, dsts = None, None, [], {}
    if host and mine:
        streamer = streamer_for(net, dev, chunk)
        for c, a, b in mine:          # pinned windows of this rank (views when the clip itself is pinned)
            win, lo, hi = clip_window(clips[c], a, b, overlap)
            wins.append(({k: v if k == "side" else _pinned(v) for k, v in win.items()}, lo, hi))
        ticket = streamer.upload(wins[0][0])
    for i, (c, a, b) in enumerate(mine):
        if host:
            hwin, lo, hi = wins[i]
            shape = (1, hwin["lq"].shape[1], 3, hwin["lq"].shape[-2] * up, hwin["lq"].shape[-1] * up)
            png = None
            if save_png is not None:  # core frames only, numbered in the whole clip; no frame download
                dsts.setdefault(shape, torch.empty(shape, dtype=out_dtype, device="meta"))
                png = lambda j, k, c=c, lo=lo, hi=hi, a0=a - lo: save_png(c, a0 + k) if lo <= k < hi else None  # noqa
            elif shape not in dsts:   # one download target per window shape, written in stream order
                dsts[shape] = _pinned(torch.empty(shape, dtype=out_dtype))
            full = streamer.run(ticket, dsts[shape]) if png is None else streamer.run(ticket, dsts[shape], png=png)
            ticket = streamer.upload(wins[i + 1][0]) if i + 1 < len(mine) else None
            out = full[:, lo:hi].clone()            # (the streamer recycles its device buffer two windows later)
        else:
            win, lo, hi = clip_window(clips[c], a, b, overlap)
            args = generator_args({k: v.contiguous() for k, v in win.items()})
            if out_dtype == torch.uint8:
                lq = win["lq"]
                buf = torch.empty(tuple(lq.shape[:3]) + ((lq.shape[3] + 3) // 4 * 4 * up, (lq.shape[4] + 3) // 4 * 4 * up),
                                  dtype=torch.uint8, device=lq.device)
                out = net.forward_streamed(*args, out=buf)[:, lo:hi]
            else:
                out = net(*args)[:, lo:hi]
            if save_png is not None:
                pngio.save_frames(out, lambda j, k, c=c, a=a: save_png(c, a + k))
        outs[(c, a, b)] = out
        m = frame_metrics(out, None if refs is None else refs[c][:, a:b].to(dev))[0]
        if gts is not None:
            q = _metrics.frame_quality(out, gts[c][:, a:b].to(dev), crop_border)
            m = torch.cat([m, q["psnr"][0].float()[:, None], q["ssim"][0].float()[:, None]], dim=-1)
        local[c, a:b] = m
    if streamer is not None:
        streamer.finish(check=True)
    metrics = merge_sharded(local, world, group)
    if not gather_output:
        return outs, metrics
    # frames: every rank contributes ONLY its own windows, packed into a fixed (items, window, 3, H, W) block
    h, w = clips[0]["lq"].shape[-2] * up, clips[0]["lq"].shape[-1] * up
    items_all = [shard_windows(num_clips, t, window, r, world) for r in range(world)]
    max_items = max(len(it) for it in items_all)
    wlen = min(window, t)
    block = torch.zeros((max_items, wlen, 3, h, w), dtype=out_dtype, device=dev)
    for i, (c, a, b) in enumerate(mine):
        block[i, :b - a] = outs[(c, a, b)][0]
    if world == 1:
        parts = block[None]
    else:
        parts = torch.empty((world,) + tuple(block.shape), dtype=out_dtype, device=dev)
        dist.all_gather(list(parts.unbind(0)), block, group=group)
    frames = torch.empty((num_clips, t, 3, h, w), dtype=out_dtype, device=dev)
    for r in range(world):
        for i, (c, a, b) in enumerate(items_all[r]):
            frames[c, a:b] = parts[r, i, :b - a]
    return frames, metrics


def merge_sharded(local, world, group=None):
    """Every rank holds a tensor of the SAME shape with its own entries filled and NaN elsewhere; returns the union on
    every rank (one all_gather of that fixed shape).  Entries nobody owns stay NaN."""
    if world == 1:
        return local
    parts = [torch.empty_like(local) for _ in range(world)]
    dist.all_gather(parts, local.contiguous(), group=group)
    full = parts[0]
    for p in parts[1:]:
        full = torch.where(torch.isnan(full), p, full)
    return full


# ------------------------------------------------------------------------------------------------
# host-resident clips: chunked upload / download overlapped with the kernels
# ------------------------------------------------------------------------------------------------
#: net -> {(device, chunk): ClipStreamer}.  enhance_clips keeps its streamer (copy streams, double-buffered device copies
#: of the inputs, result buffers, rasteriser workspace: ~11 GB for 720p x 100 clips) alive between calls: a new one per
#: call hands GB-sized blocks back and forth through the caching allocator, which showed up as one-off stalls of
#: 50-300 ms in the first call after a change of feed (profiles/r02_notes.md section 13).  release_streamers() drops them.
_STREAMERS = weakref.WeakKeyDictionary()


def streamer_for(net, device, chunk=10):
    """The cached ClipStreamer of (net, device, chunk); created on first use, released with the net."""
    key = (str(torch.device(device)), int(chunk))
    try:
        per_net = _STREAMERS.setdefault(net, {})
    except TypeError:                      # a stand-in callable that cannot be weakly referenced
        return ClipStreamer(net, device, chunk=chunk)
    st = per_net.get(key)
    if st is None:
        st = per_net[key] = ClipStreamer(net, device, chunk=chunk)
    return st


def release_streamers(net=None):
    """Drop the cached streamers (of one generator, or all) and with them their device buffers."""
    if net is None:
        _STREAMERS.clear()
    else:
        _STREAMERS.pop(net, None)


class ClipStreamer:
    """Enhances clips that live in PINNED HOST memory and returns the frames to pinned host memory.

    The reference's test loop uploads a whole clip, runs the generator, then copies every frame back
    (mmedit/apis/test.py:38-60, restorers/basicvsr.py:176-182).  Here the clip is uploaded in chunks of frames in
    the order the backward-time pass consumes them (last frame first) on a copy stream, the generator waits per
    chunk (``forward_streamed``), and finished frames go back to the host chunk by chunk on a second copy stream
    while later frames are still being computed; the upload of clip k+1 overlaps the kernels of clip k (two sets of
    device buffers).  Every clip still pays its full H2D and D2H -- they are just never exposed, except the first
    chunk in and the last chunk out.  A call takes a batch of n >= 1 clips (n, T, ...): every copy is issued per clip
    so that it is one contiguous DMA transfer (a strided (n, chunk) slice of a pinned tensor would be staged through a
    pageable bounce buffer by the framework and stall the host).

    PNG files (``run(..., png=...)``): at the end of each chunk its frames are encoded on the kernels' stream
    (``pngio.encode``; on a side stream the encoder would share the SMs with the persistent conv kernels and slow them),
    the files go down on the download stream into pinned buffers (the whole frame bound per frame), and a small pool of
    host threads writes them once that copy has completed.  The kernels' stream never waits on the host; at most
    ``PNG_IN_FLIGHT`` chunks wait for their writes, and ``finish`` joins the writers.
    """

    PNG_WRITERS = 4
    #: chunks whose pinned PNG buffers may wait for their writes; beyond that the host (never the kernels' stream) waits
    #: for the oldest write, so that a slow disk cannot make locked host memory grow with the length of a call
    PNG_IN_FLIGHT = 8

    BIG = ("lq", "mvs", "partitions")
    SMALL = ("QPs", "slices", "base_QPs")

    def __init__(self, net, device, chunk=10):
        # (weak: streamers are cached per generator in a WeakKeyDictionary, a strong reference would keep it alive)
        try:
            self._net = weakref.ref(net)
        except TypeError:
            self._net = lambda: net
        self.dev, self.chunk = torch.device(device), int(chunk)
        self.up = torch.cuda.Stream(device=self.dev)
        self.down = torch.cuda.Stream(device=self.dev)
        self.slots = [None, None]          # double-buffered device copies of the inputs
        self.outs = [None, None]           # ... and result buffers: (tensor, event "its last download has finished")
        self.turn = 0
        self.h2d_bytes = self.d2h_bytes = 0
        self.raster_work = self.raster_status = None     # compact side information: rasteriser workspace / error bits
        self.pngs = [None, None]           # per slot: (device PNG buffer, sizes, event "its last download has finished")
        self._png_host = {}                # (frames, bound) -> free pinned (buffer, sizes) pairs
        self._png_lock = threading.Lock()
        self._writers = None               # ThreadPoolExecutor, created on first use
        self._png_jobs = []
        self._png_error = None
        #: diagnostics (tools/e2e_probe.py): skip the big H2D / D2H copies to see what each direction costs
        self.copy_in = self.copy_out = True

    @property
    def net(self):
        return self._net()

    def _chunks(self, t):
        """Frame ranges [a, b) in ascending order.  The clip's LAST frames are the first the kernels read (backward-time
        pass) and the last they deliver, so the chunks there are short (2, 4, 8 frames, then ``chunk``): the first
        kernel waits for 2 frames instead of ``chunk``, and only 2 frames' download is left when the last one is done."""
        out, b, size = [], t, min(2, self.chunk)
        while b > 0:
            a = max(0, b - size)
            out.append((a, b))
            b = a
            size = min(self.chunk, size * 2)
        return out[::-1]

    @staticmethod
    def _chunk_of(chunks, t):
        """frame index -> its chunk"""
        owner = [None] * t
        for c in chunks:
            for i in range(c[0], c[1]):
                owner[i] = c
        return owner

    def upload(self, host_clip):
        """Enqueue the upload of one clip; returns a ticket for ``run``.

        8-bit frames: a uint8 ``lq`` is streamed as uint8 into a uint8 device copy; ``run`` dequantises each chunk into the
        fp32 ``lq`` the kernels read as soon as it has arrived, on the kernels' stream.

        COMPACT side information: a host clip that carries ``side`` (a list of n ``sideinfo.pack_side`` dicts: the
        codec's per-block motion-vector records, 40 bytes per block) instead of the dense ``mvs`` / ``partitions``
        planes uploads those records and rasterises them on the device (``pnp_mv_rasterize``, the bit-exact
        replacement of the loader's per-record loop, loading_ipb.py:328-369) -- 0.5 instead of 25.8 MB per 720p frame
        over the bus; only ``lq`` is then streamed in chunks.  A frame window's entry (``sideinfo.window_side``) is
        rasterised by ``pnp_mv_rasterize_window``."""
        t = host_clip["lq"].shape[1]
        slot = self.turn
        self.turn ^= 1
        side = host_clip.get("side")
        tensors = {k: v for k, v in host_clip.items() if k != "side"}
        n, _, _, h, w = host_clip["lq"].shape
        lq_u8 = host_clip["lq"].dtype == torch.uint8
        if side is not None:
            if len(side) != n or any(sd["t"] != t for sd in side):
                raise ValueError(f"side information must hold one packed entry of {t} frames per clip ({n})")
            shapes = dict({k: (tuple(v.shape), v.dtype) for k, v in tensors.items()},
                          mvs=((n, t, 4, h, w), torch.float32), partitions=((n, t, 3, h, w), torch.float32))
        else:
            shapes = {k: (tuple(v.shape), v.dtype) for k, v in tensors.items()}
        if lq_u8:                          # the uint8 chunks land in lq_u8, the kernels read the fp32 lq
            shapes["lq_u8"] = shapes["lq"]
            shapes["lq"] = (shapes["lq"][0], torch.float32)
        key = tuple((k, sh, dt) for k, (sh, dt) in sorted(shapes.items()))
        fresh = self.slots[slot] is None or self.slots[slot][0] != key
        if fresh:
            self.slots[slot] = (key, {k: torch.empty(sh, dtype=dt, device=self.dev) for k, (sh, dt) in shapes.items()},
                                None)
        dclip = self.slots[slot][1]
        busy = self.slots[slot][2]         # kernels of the clip that last used these buffers
        events = {}
        side_bytes, side_dev, side_ev = 0, [], None
        main = torch.cuda.current_stream(self.dev)
        with torch.cuda.stream(self.up):
            if fresh:
                # new buffers come from the caller's stream's pool: a block freed there may still be written by work
                # enqueued on that stream (the previous clip's temporaries), so the copies into it wait for that work
                self.up.wait_stream(main)
            if busy is not None:
                self.up.wait_event(busy)
            for k in self.SMALL:
                dclip[k].copy_(host_clip[k], non_blocking=True)
            if side is not None:
                # only the records cross the bus here; they are rasterised by `run` on the kernels' own stream (on this
                # copy stream the rasteriser would share the SMs with the previous clip's persistent conv kernels for
                # tens of ms and slow them: measured 268 instead of 299 frames/s)
                from . import sideinfo
                for c in range(n):
                    rec, meta, nbytes = sideinfo.upload_side(side[c], self.dev)
                    side_dev.append((rec, meta, side[c].get("tail")))
                    side_bytes += nbytes
                side_ev = torch.cuda.Event()
                side_ev.record(self.up)
            big = [k for k in self.BIG if k in tensors]
            for a, b in reversed(self._chunks(t)):
                for k in big if self.copy_in else ():
                    dk = "lq_u8" if (k == "lq" and lq_u8) else k
                    for c in range(n):
                        dclip[dk][c, a:b].copy_(host_clip[k][c, a:b], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self.up)
                events[(a, b)] = ev
        self.h2d_bytes = sum(v.numel() * v.element_size() for v in tensors.values()) + side_bytes
        return dict(slot=slot, dclip=dclip, events=events, t=t, side_dev=side_dev, side_ev=side_ev, lq_u8=lq_u8,
                    cond=(host_clip["slices"], host_clip["base_QPs"], host_clip["QPs"]))

    @torch.no_grad()
    def run(self, ticket, out_host, png=None):
        """Enqueue the kernels of an uploaded clip and the chunked download of its frames into ``out_host`` (fp32, or
        uint8: the last conv then stores tensor2img's uint8 frames).  An ``out_host`` on the meta device only gives the
        shape and dtype: the frames are then not downloaded.  ``png``: a callable (clip of the batch, frame) -> path or
        None; the uint8 frames with a path are saved as PNG files (see the class docstring)."""
        main = torch.cuda.current_stream(self.dev)
        t, dclip, events = ticket["t"], ticket["dclip"], ticket["events"]
        chunks = self._chunks(t)
        owner = self._chunk_of(chunks, t)
        waited = set()

        def arrive(ch):
            """the kernels' stream waits for chunk ``ch``; 8-bit frames are then dequantised there (on the copy stream
            the kernel would share the SMs with the previous clip's persistent conv kernels)"""
            waited.add(ch)
            main.wait_event(events[ch])
            if ticket["lq_u8"]:
                from . import ops
                a, b = ch
                with torch.cuda.device(self.dev):
                    for c in range(dclip["lq"].shape[0]):
                        ops.unit_from_u8(dclip["lq_u8"][c, a:b], dclip["lq"][c, a:b])

        def frame_ready(i):
            c = owner[i]
            if c not in waited:
                arrive(c)

        download = self.copy_out and out_host.device.type != "meta"
        png_bytes = [0]

        def frame_done(i, out):
            a, b = owner[i]
            if i == b - 1:
                if png is not None:
                    png_bytes[0] += self._png_chunk(out, a, b, png, main, slot)
                ev = torch.cuda.Event()
                ev.record(main)
                with torch.cuda.stream(self.down):
                    self.down.wait_event(ev)
                    for c in range(out.shape[0]) if download else ():
                        out_host[c, a:b].copy_(out[c, a:b], non_blocking=True)

        arrive(chunks[-1])                           # small tensors + the first chunk the kernels need
        if ticket["side_dev"]:
            # compact side information: records -> dense mvs / partitions of the whole clip, ahead of its first kernel
            # (~47 us per 720p frame).  The planes' previous readers ran on this stream, so plain stream order suffices.
            from . import sideinfo
            main.wait_event(ticket["side_ev"])
            h, w = dclip["lq"].shape[-2:]
            if self.raster_work is None or tuple(self.raster_work.shape[1:]) != (t, h, w):
                self.raster_work = torch.empty((3, t, h, w), dtype=torch.int32, device=self.dev)
            if self.raster_status is None:
                self.raster_status = torch.zeros(1, dtype=torch.int32, device=self.dev)
            with torch.cuda.device(self.dev):
                for c, (rec, meta, tail) in enumerate(ticket["side_dev"]):
                    rec.record_stream(main)          # allocated on the copy stream, read here
                    meta.record_stream(main)
                    sideinfo.rasterize_uploaded(rec, meta, t, dclip["mvs"][c], dclip["partitions"][c],
                                                self.raster_work, self.raster_status, tail)
            ticket["side_dev"] = []
        from .synthetic import generator_args
        # result buffers are owned here and recycled under events: a fresh torch.empty per clip that another stream
        # still reads (record_stream) keeps the caching allocator from reusing the block and ends in cudaMalloc stalls
        slot = ticket["slot"]
        if png is not None:
            if out_host.dtype != torch.uint8:
                raise ValueError("PNG files are written from uint8 frames")
            bound = pngio.frame_bound(out_host.shape[-2], out_host.shape[-1])
            pshape = tuple(out_host.shape[:2]) + (bound,)
            if self.pngs[slot] is not None and self.pngs[slot][2] is not None:
                main.wait_event(self.pngs[slot][2])  # (also before a buffer of another shape replaces it)
            if self.pngs[slot] is None or tuple(self.pngs[slot][0].shape) != pshape:
                self.pngs[slot] = (torch.empty(pshape, dtype=torch.uint8, device=self.dev),
                                   torch.empty(pshape[:2], dtype=torch.int64, device=self.dev), None)
        if self.outs[slot] is not None:
            main.wait_event(self.outs[slot][1])      # (also before a buffer of another shape replaces it)
        if self.outs[slot] is not None and tuple(self.outs[slot][0].shape) == tuple(out_host.shape) and \
                self.outs[slot][0].dtype == out_host.dtype:
            obuf = self.outs[slot][0]
        else:
            obuf = torch.empty(out_host.shape, dtype=out_host.dtype, device=self.dev)
        out = self.net.forward_streamed(*generator_args(dclip), cond_host=ticket["cond"], frame_ready=frame_ready,
                                        frame_done=frame_done, out=obuf)
        free_ev = torch.cuda.Event()
        free_ev.record(self.down)                    # behind the last chunk's download
        self.outs[slot] = (obuf, free_ev)
        if png is not None:
            self.pngs[slot] = self.pngs[slot][:2] + (free_ev,)
        done = torch.cuda.Event()
        done.record(main)
        self.slots[ticket["slot"]] = (self.slots[ticket["slot"]][0], dclip, done)
        self.d2h_bytes = (out.numel() * out.element_size() if download else 0) + png_bytes[0]
        return out

    def _png_chunk(self, out, a, b, png, main, slot):
        """Encode frames [a, b) of every clip of ``out`` that have a path (on the kernels' stream), enqueue their download
        into pinned buffers and hand the writes to the writer threads.  Returns the bytes copied."""
        n = out.shape[0]
        paths = [[png(c, i) for i in range(a, b)] for c in range(n)]
        have = [k for k in range(b - a) if any(p[k] is not None for p in paths)]
        if not have:
            return 0
        lo, hi = a + have[0], a + have[-1] + 1
        pbuf, psizes = self.pngs[slot][:2]
        with torch.cuda.stream(main), torch.cuda.device(self.dev):
            for c in range(n):
                pngio.encode(out[c, lo:hi], out=pbuf[c, lo:hi], sizes=psizes[c, lo:hi])
        ev = torch.cuda.Event()
        ev.record(main)
        key = (n * (hi - lo), pbuf.shape[-1])
        while len(self._png_jobs) >= self.PNG_IN_FLIGHT:
            self._png_jobs.pop(0).result()
        with self._png_lock:
            free = self._png_host.setdefault(key, [])
            hbuf, hsizes = free.pop() if free else (torch.empty(key, dtype=torch.uint8, pin_memory=True),
                                                     torch.empty(key[0], dtype=torch.int64, pin_memory=True))
        with torch.cuda.stream(self.down):
            self.down.wait_event(ev)
            for c in range(n):
                k = slice(c * (hi - lo), (c + 1) * (hi - lo))
                hbuf[k].copy_(pbuf[c, lo:hi], non_blocking=True)
                hsizes[k].copy_(psizes[c, lo:hi], non_blocking=True)
            copied = torch.cuda.Event()
            copied.record(self.down)
        if self._writers is None:
            self._writers = ThreadPoolExecutor(max_workers=self.PNG_WRITERS, thread_name_prefix="png-writer")
        flat = [p[i - a] for p in paths for i in range(lo, hi)]
        self._png_jobs.append(self._writers.submit(self._png_write, copied, hbuf, hsizes, flat, key))
        return hbuf.numel() + hsizes.numel() * hsizes.element_size()

    def _png_write(self, copied, hbuf, hsizes, paths, key):
        """writer thread: wait for the download, write the files, return the pinned buffers to the pool"""
        try:
            copied.synchronize()
            if self._png_error is None:
                pngio.write(hbuf, hsizes, paths)
        except OSError as e:
            with self._png_lock:
                if self._png_error is None:
                    self._png_error = e
        finally:
            with self._png_lock:
                self._png_host[key].append((hbuf, hsizes))

    def finish(self, check=False):
        """Order the caller's stream behind the last download.  ``check``: synchronise and raise what the reference's
        loader raises for malformed side information (KeyError / ValueError, see sideinfo.raise_for_status)."""
        torch.cuda.current_stream(self.dev).wait_stream(self.down)
        jobs, self._png_jobs = self._png_jobs, []
        for j in jobs:
            j.result()
        if check and self._png_error is not None:
            err, self._png_error = self._png_error, None
            raise err
        if check and self.raster_status is not None:
            from . import sideinfo
            st = int(self.raster_status.item())
            if st:
                self.raster_status.zero_()     # the streamer may serve further calls
            sideinfo.raise_for_status(st)


def stream_clips(net, host_clips, out_hosts, device, chunk=10):
    """Enhance a sequence of pinned host clips into pinned host outputs (see ClipStreamer); returns the streamer."""
    s = ClipStreamer(net, device, chunk)
    ticket = s.upload(host_clips[0])
    for k in range(len(host_clips)):
        s.run(ticket, out_hosts[k])
        ticket = s.upload(host_clips[k + 1]) if k + 1 < len(host_clips) else None    # overlaps clip k's kernels
    s.finish()
    return s
