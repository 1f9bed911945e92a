"""PNG files of the enhanced frames: the device encoder alone, its cost inside enhance_clips, and the host zlib it replaces.

   python tools/png_out_probe.py [--frames T] [--steps K] [--json PATH]

1. ``pngio.encode`` alone: us per frame from CUDA events over >= 200 frames (chunks of 10, as ClipStreamer encodes them;
   the frames span more than the L2), for generator output at 1280x720, 320x180 and the x4 ``vsr`` output of 320x180
   (1280x720), and the compression ratio (raw RGB bytes / file bytes) of generator output, uniform noise and zeros.
2. ``driver.enhance_clips`` on C2 (1280x720, T frames, compact side information, uint8 lq, pinned host entries):
   arm "u8" returns uint8 frames in pinned memory, arm "png" writes every frame with ``save_png`` into a directory on
   tmpfs (/dev/shm when it exists).  Arms alternate, three timed repetitions each, in one process; median frames/s.
3. The host encoder it replaces: ``zlib.compress`` levels 1 and 3 of the Up-filtered scanlines of the same 720p generator
   frames, one thread, ms per frame.
"""
import argparse
import json
import os
import shutil
import sys
import tempfile
import time
import zlib

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from u8_io_probe import gpu_info, host_entry  # noqa: E402


def generator_frames(dev, h, w, t, vsr):
    """(t, 3, H, W) uint8 frames of the generator (random weights, synthetic clip), tensor2img-exact"""
    import pnpvcve_b200 as P
    from pnpvcve_b200 import synthetic, weights
    net = P.build_backbone(dict(bench.GEN_CFG, vsr=vsr))
    net.load_state_dict(weights.random_state_dict(0, vsr=vsr), strict=True)
    net = net.to(dev).eval()
    clip = synthetic.make_clip(h, w, t, seed=5)
    up = 4 if vsr else 1
    with torch.no_grad():
        out = torch.empty((1, t, 3, h * up, w * up), dtype=torch.uint8, device=dev)
        net.forward_streamed(*[v.to(dev) for v in synthetic.generator_args(clip)], out=out)
    return out[0]


def time_encoder(frames, total, chunk=10):
    """us per frame of pngio.encode over `total` frames, `chunk` frames per call"""
    from pnpvcve_b200 import pngio
    reps = -(-total // frames.shape[0])
    pool = frames.repeat(reps, 1, 1, 1)[:total].contiguous()
    h, w = pool.shape[-2:]
    buf = torch.empty((chunk, pngio.frame_bound(h, w)), dtype=torch.uint8, device=pool.device)
    sizes = torch.empty(chunk, dtype=torch.int64, device=pool.device)
    for k in range(0, chunk * 3, chunk):                      # warm-up
        pngio.encode(pool[k:k + chunk], out=buf, sizes=sizes)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(0, total, chunk):
        pngio.encode(pool[k:k + chunk], out=buf[:min(chunk, total - k)], sizes=sizes[:min(chunk, total - k)])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / total


def ratio(frames):
    from pnpvcve_b200 import pngio
    _, sizes = pngio.encode(frames)
    return frames[0].numel() * frames.shape[0] / float(sizes.sum().item())


def up_filtered(frame):
    """(3, H, W) uint8 -> the PNG scanlines with filter 2 (Up) on every row, as bytes"""
    px = frame.permute(1, 2, 0).reshape(frame.shape[1], -1).cpu().numpy().astype(np.int16)
    above = np.vstack([np.zeros((1, px.shape[1]), np.int16), px[:-1]])
    rows = ((px - above) & 255).astype(np.uint8)
    return np.hstack([np.full((rows.shape[0], 1), 2, np.uint8), rows]).tobytes()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--frames", type=int, default=100, help="frames of the C2 clip")
    ap.add_argument("--steps", type=int, default=2, help="C2 entries per timed repetition")
    ap.add_argument("--encode-frames", type=int, default=200)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("png_out_probe.py measures on a B200; there is no CPU path")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    import __graft_entry__
    __graft_entry__.build()
    import pnpvcve_b200 as P
    from pnpvcve_b200 import driver, weights

    info = gpu_info()
    print(f"devices (name, power limit): {info}", flush=True)
    res = dict(devices=info, encoder={}, ratio={}, enhance_clips={}, host_zlib={})

    # ---- 1. encoder alone
    gen = {"1280x720": generator_frames(dev, 720, 1280, 10, False),
           "320x180": generator_frames(dev, 180, 320, 10, False),
           "vsr_1280x720": generator_frames(dev, 180, 320, 10, True)}
    for name, frames in gen.items():
        us = time_encoder(frames, args.encode_frames)
        res["encoder"][name] = dict(us_per_frame=us, frames=args.encode_frames)
        print(f"encoder {name}: {us:8.1f} us/frame over {args.encode_frames} frames (generator output)", flush=True)
    g = torch.Generator(device=dev).manual_seed(1)
    for name, frames in (("generator_1280x720", gen["1280x720"]), ("generator_vsr_1280x720", gen["vsr_1280x720"]),
                         ("noise_1280x720", torch.randint(0, 256, (10, 3, 720, 1280), generator=g, dtype=torch.uint8,
                                                          device=dev)),
                         ("zeros_1280x720", torch.zeros((10, 3, 720, 1280), dtype=torch.uint8, device=dev))):
        res["ratio"][name] = ratio(frames)
        print(f"compression ratio {name}: {res['ratio'][name]:.3f}", flush=True)
    noise_us = time_encoder(torch.randint(0, 256, (10, 3, 720, 1280), generator=g, dtype=torch.uint8, device=dev),
                            args.encode_frames)
    res["encoder"]["noise_1280x720"] = dict(us_per_frame=noise_us, frames=args.encode_frames)
    print(f"encoder noise_1280x720: {noise_us:8.1f} us/frame", flush=True)

    # ---- 3. host zlib on the same 720p frames
    filtered = [up_filtered(f) for f in gen["1280x720"]]
    for level in (1, 3):
        t0 = time.perf_counter()
        n_out = sum(len(zlib.compress(b, level)) for b in filtered)
        ms = (time.perf_counter() - t0) * 1e3 / len(filtered)
        res["host_zlib"][f"level{level}"] = dict(ms_per_frame=ms, ratio=sum(map(len, filtered)) / n_out)
        print(f"host zlib level {level}: {ms:.1f} ms/frame, ratio {res['host_zlib'][f'level{level}']['ratio']:.3f} "
              f"(one thread, Up filter)", flush=True)

    # ---- 2. enhance_clips: uint8 frames out vs PNG files out
    t = args.frames
    net = P.build_backbone(dict(bench.GEN_CFG))
    net.load_state_dict(weights.random_state_dict(0), strict=True)
    net = net.to(dev).eval()
    entry, _, _ = host_entry(720, 1280, t, 1, 3000)
    out_host = torch.empty((1, t, 3, 720, 1280), dtype=torch.uint8).pin_memory()
    shm = "/dev/shm" if os.path.isdir("/dev/shm") else None
    root = tempfile.mkdtemp(prefix="png_out_probe_", dir=shm)
    res["enhance_clips"]["save_dir_on"] = shm or tempfile.gettempdir()
    rates = {"u8": [], "png": []}

    def run(arm, steps):
        entries = [entry] * steps
        if arm == "u8":
            driver.enhance_clips(net, entries, device=dev, chunk=10, out_dtype=torch.uint8,
                                 out_hosts=[out_host] * steps)
        else:
            driver.enhance_clips(net, entries, device=dev, chunk=10, out_dtype=torch.uint8,
                                 save_png=lambda c, i: f"{root}/{c:03d}/{i:08d}.png")
    try:
        with torch.no_grad():
            for arm in ("u8", "png"):
                run(arm, 1)
            for _ in range(3):
                for arm in ("u8", "png"):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    run(arm, args.steps)                 # returns after the files are written
                    torch.cuda.synchronize()
                    rates[arm].append(args.steps * t / (time.perf_counter() - t0))
                    shutil.rmtree(root, ignore_errors=True)
    finally:
        shutil.rmtree(root, ignore_errors=True)
    for arm, r in rates.items():
        res["enhance_clips"][arm] = dict(frames_per_s=sorted(r)[1], repetitions=r)
        print(f"enhance_clips C2 1280x720 T={t} compact feed, uint8 lq, {arm}: {sorted(r)[1]:.1f} frames/s "
              f"({' '.join(f'{x:.1f}' for x in r)})", flush=True)
    step_us = 1e6 / res["enhance_clips"]["u8"]["frames_per_s"]
    res["enhance_clips"]["encoder_share_of_frame_step"] = res["encoder"]["1280x720"]["us_per_frame"] / step_us
    print(f"encoder share of a 720p frame step: {100 * res['enhance_clips']['encoder_share_of_frame_step']:.1f} %",
          flush=True)
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
