"""Frame-window sharding of ONE long host-resident clip (driver.enhance_windows), fed two ways: arm "dense" = fp32 lq and
dense fp32 mvs / partitions planes in, fp32 frames out (the feed the window path had before it took records); arm
"records" = uint8 lq and the codec's per-block records (sideinfo.pack_side) in, tensor2img uint8 frames out.  Same clip
(the dense planes are the device rasterisation of the same records, the fp32 lq is the uint8 one / 255), arms alternate,
three timed repetitions each, in one process; the gathered frames of the two arms are compared (uint8 == tensor2img of
fp32).

   python tools/window_feed_probe.py [--steps K] [--json PATH]
   torchrun --nproc-per-node 8 tools/window_feed_probe.py ...

Workload: one 1280x720 clip of T = 40 x world frames, one window of 40 frames per rank, gather_output=True (every rank
ends with all frames).  Per arm: frames/s (max-over-ranks device time), H2D and D2H bytes per frame, host memory pinned
per rank (the clip as the caller holds it, and what the call itself pins)."""
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

H, W, PER_RANK = 720, 1280, 40


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError):
        q = []
    return q


def host_clips(t, dev):
    """(dense fp32 clip, compact uint8 clip) of the same pinned host clip"""
    from pnpvcve_b200 import sideinfo, synthetic
    clip = synthetic.make_clip(H, W, t, seed=4000, crf=25, ipb=True)
    types = [chr(int(v)) for v in clip["slices"].flatten()]
    tmpl = sideinfo.synthetic_records(H, W, "IBBP", seed=77)       # record lists of an I, two B and a P frame
    per_type = {"I": [tmpl[0]], "B": [tmpl[1], tmpl[2]], "P": [tmpl[3]]}
    recs = [per_type[st][f % len(per_type[st])] for f, st in enumerate(types)]
    flat = np.concatenate(recs, 0)
    offs = np.cumsum([0] + [len(r) for r in recs])
    mvs, par = sideinfo.rasterize_clip(flat, offs, types, H, W, device=dev)
    u8 = (clip["lq"].clamp(0, 1) * 255.0).round().to(torch.uint8)
    small = {k: clip[k].pin_memory() for k in ("QPs", "slices", "base_QPs")}
    dense = dict(small, lq=(u8.float() / 255.0).pin_memory(), mvs=mvs.cpu()[None].pin_memory(),
                 partitions=par.cpu()[None].pin_memory())
    compact = dict(small, lq=u8.pin_memory(), side=[sideinfo.pack_side(flat, offs, types)])
    return dense, compact


def nbytes(clip):
    n = sum(v.numel() * v.element_size() for k, v in clip.items() if k != "side")
    return n + sum(sd["records"].numel() * 4 + sd["meta"].numel() * 4 for sd in clip.get("side", []))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=5, help="enhance_windows calls per timed repetition")
    ap.add_argument("--json", default=None, help="write the results here (rank 0)")
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("window_feed_probe.py measures on a B200; there is no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    import __graft_entry__
    __graft_entry__.build()
    import pnpvcve_b200 as P
    from pnpvcve_b200 import driver, sideinfo, weights

    def log(msg):
        if rank == 0:
            print(msg, flush=True)

    info = gpu_info()
    log(f"devices (name, power limit): {info}; world {world}")
    t = PER_RANK * world
    chunk = 10
    net = P.build_backbone(dict(bench.GEN_CFG))
    net.load_state_dict(weights.random_state_dict(0), strict=True)
    net = net.to(dev).eval()
    dense, compact = host_clips(t, dev)
    (c, a, b), = driver.shard_windows(1, t, PER_RANK, rank, world)
    records_pinned = nbytes(dict(side=[sideinfo.window_side(compact["side"][0], a, b)]))
    arms = {}
    for arm, clip, dt in (("dense", dense, torch.float32), ("records", compact, torch.uint8)):
        result_pinned = PER_RANK * 3 * H * W * torch.empty((), dtype=dt).element_size()
        arms[arm] = dict(clip=clip, dtype=dt, rates=[], clip_pinned_bytes=nbytes(clip),
                         call_pinned_bytes=result_pinned + (records_pinned if arm == "records" else 0))

    def run(arm):
        x = arms[arm]
        frames, _ = driver.enhance_windows(net, [x["clip"]], PER_RANK, rank, world, gather_output=True, device=dev,
                                           chunk=chunk, out_dtype=x["dtype"])
        st = driver.streamer_for(net, dev, chunk)
        x["h2d_bytes_per_frame"] = st.h2d_bytes / PER_RANK
        x["d2h_bytes_per_frame"] = st.d2h_bytes / PER_RANK
        return frames

    with torch.no_grad():
        outs = {arm: run(arm) for arm in arms}          # warm-up (every shape), and the outputs of the two arms
        run("dense"), run("records")
        torch.cuda.synchronize()
        same = bool(torch.equal(outs["records"], (outs["dense"].clamp(0, 1) * 255.0).round().to(torch.uint8)))
        del outs
        for _ in range(3):
            for arm in arms:
                if world > 1:
                    dist.barrier()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.steps):
                    run(arm)
                e1.record()
                torch.cuda.synchronize()
                ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
                if world > 1:
                    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
                arms[arm]["rates"].append(args.steps * t / (float(ms.item()) / 1e3))
    res = dict(devices=info, world=world, frames=t, window=PER_RANK, steps=args.steps, chunk=chunk,
               workload=f"one {W}x{H}x{t} host clip, one {PER_RANK}-frame window per rank, gather_output=True",
               records_equal_tensor2img_of_dense=same, arms={})
    log(f"records arm == tensor2img(dense arm), all {t} frames: {same}")
    for arm, x in arms.items():
        res["arms"][arm] = dict(frames_per_s=sorted(x["rates"])[1], repetitions=x["rates"],
                                h2d_bytes_per_frame=x["h2d_bytes_per_frame"], d2h_bytes_per_frame=x["d2h_bytes_per_frame"],
                                clip_pinned_bytes_per_rank=x["clip_pinned_bytes"],
                                call_pinned_bytes_per_rank=x["call_pinned_bytes"])
        log(f"{arm:8s}: {res['arms'][arm]['frames_per_s']:8.1f} frames/s ({' '.join(f'{r:.1f}' for r in x['rates'])}), "
            f"H2D {x['h2d_bytes_per_frame'] / 1e6:.3f} MB/frame, D2H {x['d2h_bytes_per_frame'] / 1e6:.3f} MB/frame, "
            f"pinned per rank: clip {x['clip_pinned_bytes'] / 1e6:.1f} MB, by the call {x['call_pinned_bytes'] / 1e6:.1f} MB")
    if rank == 0 and args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)
    driver.release_streamers(net)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
