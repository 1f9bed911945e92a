"""fp32 against 8-bit frames through the host-clip API: driver.enhance_clips on pinned host entries fed with compact
side information, arm "f32" = fp32 lq in / fp32 frames out, arm "u8" = uint8 lq in / tensor2img uint8 frames out (the
same clips: the fp32 lq is the uint8 one / 255).  Arms alternate, three timed repetitions each, in one process.

   python tools/u8_io_probe.py [--steps K] [--frames T] [--json PATH]
   torchrun --nproc-per-node 8 tools/u8_io_probe.py ...     (clip-sharded like bench.py's e2e leg)

Per arm: frames/s (median and all three repetitions), H2D and D2H bytes per frame, pinned host bytes per entry."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402

#: name -> (H, W, clips per entry, vsr)
CASES = {"C2_720p": (720, 1280, 1, False), "C4_180x320_x16": (180, 320, 16, False), "vsr_180x320": (180, 320, 1, True)}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError):
        q = []
    return q


def host_entry(h, w, t, n, seed):
    """n clips of (h, w, t) with uint8 lq and compact side information, pinned"""
    from pnpvcve_b200 import sideinfo, synthetic
    clips = [synthetic.make_clip(h, w, t, seed=seed + c, crf=(15, 25, 35)[c % 3], ipb=True) for c in range(n)]
    entry = synthetic.cat_clips(clips)
    types = [chr(int(v)) for v in entry["slices"][0].flatten()]
    tmpl = sideinfo.synthetic_records(h, w, "IBBP", seed=77)       # record lists of an I, two B and a P frame
    per_type = {"I": [tmpl[0]], "B": [tmpl[1], tmpl[2]], "P": [tmpl[3]]}
    recs = [per_type[st][f % len(per_type[st])] for f, st in enumerate(types)]
    flat = np.concatenate(recs, 0)
    offs = np.cumsum([0] + [len(r) for r in recs])
    u8 = (entry["lq"].clamp(0, 1) * 255.0).round().to(torch.uint8)
    small = {k: entry[k].pin_memory() for k in ("QPs", "slices", "base_QPs")}
    side = [sideinfo.pack_side(flat, offs, types) for _ in range(n)]
    side_bytes = sum(sd["records"].numel() * 4 + sd["meta"].numel() * 4 for sd in side)
    return dict(small, lq=u8.pin_memory(), side=side), dict(small, lq=(u8.float() / 255.0).pin_memory(), side=side), \
        side_bytes


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=3, help="entries per rank and timed repetition")
    ap.add_argument("--frames", type=int, default=100)
    ap.add_argument("--cases", default=",".join(CASES))
    ap.add_argument("--json", default=None, help="write the results here (rank 0)")
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("u8_io_probe.py measures on a B200; there is no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    import __graft_entry__
    __graft_entry__.build()
    import pnpvcve_b200 as P
    from pnpvcve_b200 import driver, weights

    def log(msg):
        if rank == 0:
            print(msg, flush=True)

    info = gpu_info()
    log(f"devices (name, power limit): {info}; world {world}")
    res = dict(devices=info, world=world, steps=args.steps, frames=args.frames, cases={})
    t = args.frames
    for name in args.cases.split(","):
        h, w, n, vsr = CASES[name]
        net = P.build_backbone(dict(bench.GEN_CFG, vsr=vsr))
        net.load_state_dict(weights.random_state_dict(0, vsr=vsr), strict=True)
        net = net.to(dev).eval()
        e_u8, e_f32, side_bytes = host_entry(h, w, t, n, 3000 + 100 * rank)
        up = 4 if vsr else 1
        arms = {}
        for arm, entry, dt in (("f32", e_f32, torch.float32), ("u8", e_u8, torch.uint8)):
            out = torch.empty((n, t, 3, up * h, up * w), dtype=dt).pin_memory()
            arms[arm] = dict(entry=entry, out=out, rates=[],
                             pinned_bytes_per_entry=entry["lq"].numel() * entry["lq"].element_size() +
                             out.numel() * out.element_size() + side_bytes)

        def run(arm, steps):
            a = arms[arm]
            entries = [a["entry"] if c % world == rank else None for c in range(world * steps)]
            driver.enhance_clips(net, entries, rank, world, device=dev, out_hosts=[a["out"]] * len(entries),
                                 chunk=min(10, t), out_dtype=a["out"].dtype)
            st = driver.streamer_for(net, dev, min(10, t))
            a["h2d_bytes_per_frame"] = st.h2d_bytes / (n * t)
            a["d2h_bytes_per_frame"] = st.d2h_bytes / (n * t)

        with torch.no_grad():
            for arm in ("f32", "u8"):          # warm-up: two entries each (the streamer allocates its buffers)
                run(arm, 2)
            for _ in range(3):
                for arm in ("f32", "u8"):
                    if world > 1:
                        dist.barrier()
                    torch.cuda.synchronize()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    run(arm, args.steps)
                    e1.record()
                    torch.cuda.synchronize()
                    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
                    if world > 1:
                        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
                    arms[arm]["rates"].append(world * args.steps * n * t / (float(ms.item()) / 1e3))
        out = {}
        for arm, a in arms.items():
            out[arm] = dict(frames_per_s=sorted(a["rates"])[1], repetitions=a["rates"],
                            h2d_bytes_per_frame=a["h2d_bytes_per_frame"], d2h_bytes_per_frame=a["d2h_bytes_per_frame"],
                            pinned_bytes_per_entry=a["pinned_bytes_per_entry"])
            log(f"{name} {w}x{h} n={n} T={t} vsr={vsr} {arm}: {out[arm]['frames_per_s']:8.1f} frames/s "
                f"({' '.join(f'{r:.1f}' for r in a['rates'])}), H2D {a['h2d_bytes_per_frame'] / 1e6:.3f} MB/frame, "
                f"D2H {a['d2h_bytes_per_frame'] / 1e6:.3f} MB/frame, pinned {a['pinned_bytes_per_entry'] / 1e6:.1f} MB/entry")
        res["cases"][name] = dict(h=h, w=w, clips_per_entry=n, vsr=vsr, **out)
        driver.release_streamers(net)
        del net, arms, e_u8, e_f32
        torch.cuda.empty_cache()
    if rank == 0 and args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
