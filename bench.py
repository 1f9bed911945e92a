#!/usr/bin/env python
"""Benchmark of the BAE+CAA enhancement hot path (BASELINE.json: 720p enhanced frames/s + roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config C2|C3|C4|C5] [--frames T] [--clips n]
                    [--impl ours|reference] [--dump-outputs DIR]

A *step* is one batch of synthetic clips of the selected BASELINE.json config per GPU through the registry-built
generator: C2 (default at N=1) one REDS4-shape clip 1280x720x100, per-frame random QPs, CRF cycling 15/25/35 over the
steps; C3 (default at N>1, the config BASELINE.json quotes for 1/2/4/8 GPUs) the same with slice-type (IPB) conditioning;
C4 sixteen 320x180x100 LR clips with MIXED CRFs in one call; C5 sixteen KITTI-shape 1244x376 frame pairs.  The N=1 line
also carries `other_configs`: short resident runs of the configs that are not the selected one (frames/s, Mpx/s, and
max-abs error of a sample against the CPU oracle port).  N>1 is launched by torchrun (one process per GPU); clips are
independent, so ranks share nothing on the data path (weak scaling) and only gather per-frame metrics.
Rank 0 prints ONE JSON line:

  value        frames/s with the clip already resident in HBM (CUDA events around the steps, NO events inside
               them, max over ranks)
  e2e          same from pinned HOST buffers through the public host-clip API (driver.enhance_clips on host entries,
               ClipStreamer underneath): H2D of every input and D2H of the enhanced frames inside the timed region,
               overlapped with the kernels
  e2e_sideinfo the same public call fed with COMPACT side information: per-block motion-vector records (40 bytes per
               block) over the bus instead of the dense mvs / partitions planes, rasterised on the device
               (pnp_mv_rasterize); informational, `e2e` stays the reference's dense interface
  roofline     dominant kernel (block launch A: 3x3 conv + three partition 1x1 convs): algorithmic FLOPs per
               launch / mean launch duration, CUDA events bracketing every 8th such launch in a separate pass of
               the same steps (an upper bound: the bracketed launch loses its programmatic-dependent-launch
               overlap), against the measured sustained bf16 peak of MEASURED_PEAKS.json; block_pair = in-situ
               time of a launch A + launch B pair from phase-boundary events around the undisturbed stacks
  roofline_warp  K1 (HBM bound), algorithmic bytes 264 B/px
  cpu_baseline the oracle port of the reference on this box's host cores, bounded sample
  parity       max-abs error of the CUDA path against that oracle sample (same inputs, tolerance 2e-3)
  frame_windows  ONE clip of the config cut into one window per GPU (driver.enhance_windows: the reference's max_seq_len
               windows, each a clip of its own; frames and metrics gathered on every rank): strong scaling of a single
               clip stream, beside the weak-scaling `value`

--impl reference times the reference's own algorithm (oracle port, PyTorch CPU, all host threads) on
the same metric.  The oracle is only ever the thing measured beside us, never part of the product.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W = 720, 1280                            # the selected config's frame size (set by select_config)
CRFS = (15, 25, 35)
#: BASELINE.json configs 2-5 (config 1 is the CPU-runnable case of the parity tests)
CONFIGS = {
    "C2": dict(h=720, w=1280, t=100, ipb=False, clips=1, mv_qpel=64, pattern="IBBP", tag="720p",
               desc="C2 HR_davis_LR_128x128 BAE+CAA forward, synthetic REDS4-shape clips 1280x720, per-frame random QPs"),
    "C3": dict(h=720, w=1280, t=100, ipb=True, clips=1, mv_qpel=64, pattern="IBBP", tag="720p",
               desc="C3 HR_davis_LR_128x128_IPB (slice-type I/P/B conditioning) BAE+CAA forward, synthetic 720p clips 1280x720"),
    "C4": dict(h=180, w=320, t=100, ipb=True, clips=16, mv_qpel=32, pattern="IBBP", tag="lr_320x180",
               desc="C4 HR_davis_LR_128x128_IPB_LR_test BAE+CAA forward, synthetic LR clips 320x180, many clips per call with mixed CRFs"),
    "C5": dict(h=376, w=1244, t=2, ipb=True, clips=16, mv_qpel=64, pattern="IP", tag="kitti_1244x376",
               desc="C5 HR_davis_LR_128x128_IPB BAE+CAA forward, synthetic KITTI-shape frame pairs 1242x375 pre-padded to 1244x376"),
}
CFG = dict(CONFIGS["C2"], name="C2")


def select_config(args):
    """Fix the workload: --config (default C2 at N=1, C3 at N>1), --frames / --clips override its T / clips per step."""
    global H, W, CFG, METRIC
    name = args.config or ("C2" if args.gpus <= 1 else "C3")
    CFG = dict(CONFIGS[name], name=name)
    if args.frames:
        CFG["t"] = args.frames
    if args.clips:
        CFG["clips"] = args.clips
    args.frames, args.clips = CFG["t"], CFG["clips"]
    H, W = CFG["h"], CFG["w"]
    METRIC = "enhanced_frames_per_sec_" + CFG["tag"]
    return CFG
FLOP_PER_PX_FRAME = 3205248                 # SURVEY.md section 8(d): dense convs, 2 FLOP per MAC
FLOP_BLOCK_A_PER_PX = 2 * (64 * 64 * 9 + 3 * 64 * 64)
WARP_BYTES_PER_PX = 2 * 64 * 2 + 8          # bf16 features in + out, fp32 2-channel flow
METRIC = "enhanced_frames_per_sec_720p"
GEN_CFG = dict(
    type="IconVSR_restore_wo_refill_mv_ipb_fast_domain_dynamic_with_par", mid_channels=64, num_blocks=8,
    padding=3, with_cat=True, use_base_qp=True, num_experts=6, expert_softmax=True, init_weight=True,
    with_bias=True, with_se=True, with_par=True, one_layer=True, blocktype="drt", channel_first=True,
    sparse_val=False, align_key=True, vsr=False)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], bf16_tflops=p["bf16_tflops"],
                    bf16_tflops_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=10)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        busy = [x for x in sm if x > 0.5 * max(sm)] if sm else []
        return dict(sm_mhz=statistics.median(busy) if busy else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


# ---------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the oracle port on the host cores
# ---------------------------------------------------------------------------------------------
def cpu_oracle_step(sd, clip, keep=None):
    from oracle import bae_oracle
    from pnpvcve_b200 import synthetic
    t0 = time.perf_counter()
    out = bae_oracle.generator_forward(sd, *synthetic.generator_args(clip))
    dt = time.perf_counter() - t0
    if keep is not None:
        keep.append(out)
    return dt


def cpu_px_rate():
    """Pixels x frames per second of the oracle port on this host (probe on 128x128, scaled for large frames)."""
    from pnpvcve_b200 import synthetic, weights
    sd = weights.random_state_dict(0)
    probe = synthetic.make_clip(128, 128, 2, seed=1)
    cpu_oracle_step(sd, probe)                                   # page in / thread pool warm-up
    dt = cpu_oracle_step(sd, probe)
    return 2 * 128 * 128 / dt * 0.45                             # large frames run ~2x slower per pixel


def cpu_sample(budget_s, n_steps, cfg=None):
    """The bounded sample of the workload one CPU step runs: (h, w, frames).  The config's own frame size with 2 frames
    (I,B / I,P) or 1 frame (I) whenever n_steps of it fit the budget -- otherwise a centred crop, and the caller says so."""
    cfg = cfg or CFG
    rate = cpu_px_rate()
    for (h, w) in ((cfg["h"], cfg["w"]), (cfg["h"] // 2, cfg["w"] // 2), (cfg["h"] // 4, cfg["w"] // 4)):
        h, w = max(64, h // 4 * 4), max(64, w // 4 * 4)
        for frames in (2, 1):
            if n_steps * (frames * h * w / rate) <= budget_s:
                return h, w, frames
    return 64, 64, 1


def make_cpu_clip(cfg, h, w, frames, crf=25):
    from pnpvcve_b200 import synthetic
    return synthetic.make_clip(h, w, frames, seed=2000, crf=crf, mv_qpel=cfg["mv_qpel"], ipb=cfg["ipb"],
                               pattern=cfg["pattern"])


def sample_text(cfg, h, w, frames):
    full = (h, w) == (cfg["h"], cfg["w"])
    return (f"{frames} frame{'s' if frames > 1 else ''} of a {w}x{h} synthetic clip"
            + ("" if full else f" (crop of the {cfg['w']}x{cfg['h']} workload; value scaled by pixel count)"))


def run_reference_arm(args):
    """--impl reference: rank 0 only; other ranks exit without work."""
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    from pnpvcve_b200 import weights
    cfg = select_config(args)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    h, w, frames = cpu_sample(200.0, args.steps + args.warmup)
    sd = weights.random_state_dict(0)
    clip = make_cpu_clip(cfg, h, w, frames)
    for _ in range(args.warmup):
        cpu_oracle_step(sd, clip)
    times = [cpu_oracle_step(sd, clip) for _ in range(args.steps)]
    total = sum(times)
    value = args.steps * frames * (h * w) / float(H * W) / total      # frames of the config's size per second
    sample = f"oracle port (PyTorch fp32, {cores} threads), per step " + sample_text(cfg, h, w, frames)
    config = workload_config(args, 1)
    # what this arm REALLY ran per step (a bounded sample of the workload above, tier rule 4)
    config.update(sample=sample_text(cfg, h, w, frames), sample_height=h, sample_width=w, sample_frames=frames)
    line = dict(metric=METRIC, value=value, unit="frames/s", n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=1e3 * total / args.steps, higher_is_better=True,
                scaling="weak", vs_baseline=None, dtype="f32", data="synthetic", impl="reference",
                config=config,
                cpu_baseline=dict(value=value, unit="frames/s", cores=cores, kind="port", sample=sample),
                e2e=dict(value=value, unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0)
    _emit(line)
    return 0


def workload_config(args, world):
    return dict(workload=f"{CFG['desc']}, {args.clips} clip(s) x {args.frames} frames per GPU per step, "
                         f"CRF 15/25/35 {'mixed inside the batch' if args.clips > 1 else 'cycling over the steps'}, "
                         "random-init weights",
                config=CFG["name"], frames_per_clip=args.frames, clips_per_gpu_per_step=args.clips, height=H, width=W,
                conditioning="slice type (IPB)" if CFG["ipb"] else "per-frame QP",
                parallelism=f"clip-sharded x{world} (no data-path collective)",
                l2=f"inputs ({40 * H * W * args.clips * args.frames / 1e6:.0f} MB per step) and every feature map "
                   "pass exceed L2 between reuses; no flush needed" if 40 * H * W * args.clips * args.frames > 200e6
                   else "three resident batches are rotated so that consecutive steps read different inputs")


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
def make_device_batch(cfg, frames, n, seed, crf0, dev):
    """n clips of the config's shape; CRFs cycle inside the batch starting at index crf0 (mixed-CRF batches)."""
    from pnpvcve_b200 import synthetic
    return synthetic.cat_clips([
        synthetic.make_clip(cfg["h"], cfg["w"], frames, seed=seed + 3 * k, crf=CRFS[(crf0 + k) % len(CRFS)],
                            mv_qpel=cfg["mv_qpel"], ipb=cfg["ipb"], pattern=cfg["pattern"], device=dev)
        for k in range(n)])


def mean_event_ms(pairs):
    return sum(a.elapsed_time(b) for a, b in pairs) / max(len(pairs), 1)


def ncu_traffic(substr):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch (bytes) of the first kernel whose name contains
    `substr`, read from the newest committed capture profiles/r*_kernels_ncu_summary.csv (720p launches)."""
    import csv
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_kernels_ncu_summary.csv")))
    for path in reversed(files):
        with open(path, newline="") as f:
            rows = list(csv.reader(f))
        if len(rows) < 3:
            continue
        hdr, units = rows[0], rows[1]
        try:
            ir, iw = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
        except ValueError:
            continue
        scale = {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}
        for r in rows[2:]:
            if substr in r[0] and len(r) > max(ir, iw):
                return (float(r[ir]) * scale.get(units[ir], 1.0) + float(r[iw]) * scale.get(units[iw], 1.0),
                        os.path.relpath(path, ROOT))
    return None, None


#: the ONE JSON line goes to the process's original stdout; everything else that native libraries print there
#: (NCCL announces its version on stdout on some boxes) is sent to stderr
_JSON_OUT = None


def _claim_stdout():
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def _emit(line):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


#: --dump-outputs keeps at most this many values of the enhanced frames (16 MB of float32)
DUMP_MAX_VALUES = 1 << 22


def dump_outputs(path, out):
    """--dump-outputs: what the last timed step returned to its caller, as .npy files under `path`.

    frames.npy         the enhanced frames (n, T, 3, H, W) float32, when they hold at most DUMP_MAX_VALUES values
    frames_sample.npy  otherwise: the values at DUMP_MAX_VALUES flat positions drawn with a fixed seed, in ascending
                       position order (the same positions for the same arguments)
    frame_metrics.npy  (n, T, 2) float32 per-frame max-abs and mean square of the whole frames (driver.frame_metrics)
    """
    import numpy as np
    from pnpvcve_b200 import driver
    os.makedirs(path, exist_ok=True)
    flat = out.reshape(-1)
    if flat.numel() <= DUMP_MAX_VALUES:
        np.save(os.path.join(path, "frames.npy"), out.float().cpu().numpy())
    else:
        g = torch.Generator().manual_seed(0)
        pos = torch.randint(flat.numel(), (DUMP_MAX_VALUES,), generator=g).sort().values
        np.save(os.path.join(path, "frames_sample.npy"), flat[pos.to(flat.device)].float().cpu().numpy())
    np.save(os.path.join(path, "frame_metrics.npy"), driver.frame_metrics(out).cpu().numpy())


def timed_resident(net, batches, steps, warmup, dev):
    """frames/s of `steps` resident steps (CUDA events, no events inside the steps)."""
    from pnpvcve_b200 import synthetic
    with torch.no_grad():
        for i in range(warmup):
            net(*synthetic.generator_args(batches[i % len(batches)]))
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            net(*synthetic.generator_args(batches[(warmup + i) % len(batches)]))
        e1.record()
        torch.cuda.synchronize()
    n, t = batches[0]["lq"].shape[:2]
    return steps * n * t / (e0.elapsed_time(e1) * 1e-3), net.gpu_launches


def other_configs_block(net, dev, main_name, cpu_budget_s=45.0):
    """Short resident runs of the BASELINE configs that are not the selected one + a CPU-oracle sample of each
    (CPU frames/s beside ours and the max-abs error of the CUDA path on that very sample)."""
    from pnpvcve_b200 import synthetic, weights
    res = {}
    sd = weights.random_state_dict(0)
    plan = dict(C2=dict(t=20, steps=2, warm=1), C3=dict(t=20, steps=2, warm=1), C4=dict(t=100, steps=2, warm=1),
                C5=dict(t=2, steps=20, warm=3))
    names = [n for n in ("C3", "C4", "C5", "C2") if n != main_name][:3]
    for name in names:
        cfg = dict(CONFIGS[name], name=name)
        pl = plan[name]
        net._engine.prog = None
        torch.cuda.empty_cache()
        batches = [make_device_batch(cfg, pl["t"], cfg["clips"], 5000 + 100 * j, j, dev) for j in range(2)]
        fps, launches = timed_resident(net, batches, pl["steps"], pl["warm"], dev)
        del batches
        h, w, frames = cpu_sample(cpu_budget_s / len(names), 1, cfg)
        clip = make_cpu_clip(cfg, h, w, frames, crf=35)
        kept = []
        dt = cpu_oracle_step(sd, clip, keep=kept)
        with torch.no_grad():
            got = net(*[a.to(dev) for a in synthetic.generator_args(clip)]).float().cpu()
        res[name] = dict(workload=f"{cfg['desc']}, {cfg['clips']} clip(s) x {pl['t']} frames per step, mixed CRFs",
                         frames_per_s=fps, mpx_per_s=fps * cfg["h"] * cfg["w"] / 1e6, steps=pl["steps"],
                         gpu_launches_per_step=launches,
                         tflops=FLOP_PER_PX_FRAME * cfg["h"] * cfg["w"] * fps / 1e12,
                         max_abs_err=float((got - kept[0]).abs().max()), tolerance=2e-3,
                         cpu_frames_per_s=frames * (h * w) / float(cfg["h"] * cfg["w"]) / dt,
                         sample=sample_text(cfg, h, w, frames) + ", CUDA path vs CPU oracle port, CRF 35")
    net._engine.prog = None
    torch.cuda.empty_cache()
    return res


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3,
                    help="timed steps of the headline value and of the e2e, e2e_sideinfo (three repetitions) and "
                         "frame_windows blocks; other_configs and the kernel profiling pass use fixed counts")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default=None, choices=sorted(CONFIGS),
                    help="BASELINE.json config (default: C2 at --gpus 1, C3 at --gpus > 1)")
    ap.add_argument("--frames", type=int, default=0, help="frames per clip (default: the config's)")
    ap.add_argument("--clips", type=int, default=0, help="clips per GPU per step (default: the config's)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--no-sideinfo", action="store_true", help="skip the compact side-information end-to-end block")
    ap.add_argument("--no-windows", action="store_true", help="skip the frame-window (single clip, strong scaling) block")
    ap.add_argument("--prof-every", type=int, default=8,
                    help="bracket every N-th launch of the profiled kernels with CUDA events")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frames the last timed step computed (rank 0) as .npy files into DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the CUDA path's frames; it does not apply to --impl reference")
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch.distributed as dist
    import __graft_entry__
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback for the product path")
    cfg = select_config(args)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    __graft_entry__.build()
    import pnpvcve_b200 as P
    from pnpvcve_b200 import driver, synthetic, weights

    net = P.build_backbone(GEN_CFG)
    net.load_state_dict(weights.random_state_dict(0), strict=True)
    net = net.to(dev).eval()
    T = args.frames
    nc = args.clips
    px = H * W * nc                              # pixels per launch (nc images)
    # three resident batches of `nc` clips, reused across steps (generation is not part of the job); with one clip
    # per step the CRF cycles 15/25/35 over the steps, with several the CRFs are mixed inside every batch
    clips = [make_device_batch(cfg, T, nc, 2000 + 10 * rank + 100 * j, j, dev) for j in range(len(CRFS))]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident(i):
        clip = clips[i % len(clips)]
        out = net(*synthetic.generator_args(clip))
        local = driver.frame_metrics(out)
        driver.gather_metrics(local.mean(0, keepdim=True), world, rank, world)   # the job's only collective
        return out

    # ---------------- device-resident throughput (value)
    with torch.no_grad():
        for i in range(args.warmup):
            step_resident(i)
        barrier()
        sampler = ClockSampler(local_rank) if rank == 0 else None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches = 0
        e0.record()
        for i in range(args.steps):
            out = step_resident(args.warmup + i)
            launches += net.gpu_launches
            if i + 1 < args.steps:
                del out                            # only the last step's frames outlive their step
        e1.record()
        barrier()
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, out)
        del out
        # Per-kernel durations come from a SEPARATE pass of the same steps, right behind the timed one (same
        # clocks, same thermal state): an event record between two launches defeats programmatic dependent
        # launch for both neighbours, and bracketing every 8th launch was measured to slow the whole step by
        # ~10 % (round-1 measurement: 151 -> 167 us per block).  `value` is therefore timed without any events
        # inside the step; the bracketed durations below include the launch overhead PDL normally hides.
        net._engine.prof = {"block": [], "block_a": [], "warp": [], "block_b": []}
        net._engine.prof_every = args.prof_every
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        prof_steps = min(args.steps, 2)
        p0.record()
        for i in range(prof_steps):
            step_resident(args.warmup + i)
        p1.record()
        barrier()
        prof = net._engine.prof
        prof_step_ms = p0.elapsed_time(p1) / prof_steps
        # ... and one more step with events only at the phase boundaries of a frame (7 per frame instead of ~12 per
        # block): the 8-block stacks are timed undisturbed, which gives the in-situ duration of a launch A + launch B pair
        net._engine.prof = {"phases": []}
        step_resident(args.warmup)
        barrier()
        clocks = sampler.stop() if sampler else None
        phases = net._engine.prof["phases"]
        net._engine.prof = None
        stack_us = [a.elapsed_time(b) * 1e3 for (n0, a), (n1, b) in zip(phases[:-1], phases[1:])
                    if n0.endswith("input_done") and n1.endswith("stack_done")]
        pair_us = sum(stack_us) / len(stack_us) / GEN_CFG["num_blocks"] if stack_us else 0.0
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    total_ms = float(ms.item())
    frames_total = world * args.steps * T * nc
    value = frames_total / (total_ms / 1e3)

    peaks = measured_peaks()
    a_ms = mean_event_ms(prof["block_a"])
    b_ms = mean_event_ms(prof["block_b"])
    w_ms = mean_event_ms(prof["warp"])
    a_tflops = FLOP_BLOCK_A_PER_PX * px / (a_ms * 1e-3) / 1e12 if a_ms else 0.0
    w_gbs = WARP_BYTES_PER_PX * px / (w_ms * 1e-3) / 1e9 if w_ms else 0.0
    steps_ms = total_ms / args.steps
    # share of the (profiled) step spent in this kernel: bracketed launches x sampling stride / profiled step time
    share_a = a_ms * len(prof["block_a"]) * args.prof_every / prof_steps / prof_step_ms if a_ms else 0.0
    # dram__bytes_read.sum + dram__bytes_write.sum per launch at 720p from the newest committed ncu capture (algorithmic
    # bytes of launch A: 118 (x) + 11 (partition planes) + 118 (t) = 247 MB; of the warp: 243 MB); null off 720p
    at_720p = (H, W, nc) == (720, 1280, 1)
    a_traffic, a_src = ncu_traffic("conv3x3_rows_kernel<1") if at_720p else (None, None)
    w_traffic, w_src = ncu_traffic("mv_warp_kernel") if at_720p else (None, None)
    per_gpu_tflops = FLOP_PER_PX_FRAME * H * W * (value / world) / 1e12
    pair_flop = (FLOP_BLOCK_A_PER_PX + 2 * 64 * 64 * 9) * px
    roofline = dict(bound="tensor", kernel="conv3x3_rows_kernel<1,0> (block launch A: row-stacked 3x3 + three partition 1x1 convs, N=192 MMAs, split-role epilogue)",
                    achieved=a_tflops, peak=peaks["bf16_tflops_sustained"], unit="TFLOP/s",
                    frac=a_tflops / peaks["bf16_tflops_sustained"],
                    traffic=a_traffic, traffic_unit="bytes/launch", traffic_source=a_src,
                    algorithmic_flop_per_launch=FLOP_BLOCK_A_PER_PX * px,
                    peak_source=f"{peaks['source']} sustained cuBLAS bf16 (kernel timed inside a long step)",
                    ms_per_launch=a_ms, launches_timed=len(prof["block_a"]), timed_every=args.prof_every,
                    share_of_step=share_a,
                    # launch A + launch B of one BAE block, from phase-boundary events around the undisturbed 8-block stacks
                    block_pair=dict(us=pair_us, tflops=pair_flop / (pair_us * 1e-6) / 1e12 if pair_us else 0.0,
                                    frac=pair_flop / (pair_us * 1e-6) / 1e12 / peaks["bf16_tflops_sustained"] if pair_us else 0.0,
                                    note="bracketing single launches defeats programmatic dependent launch, so ms_per_launch "
                                         "is an upper bound; this is the in-situ time of the A+B pair"),
                    # per GPU: the all-rank value divided by the world size
                    whole_path_tflops=per_gpu_tflops,
                    whole_path_frac=per_gpu_tflops / peaks["bf16_tflops_sustained"])
    roofline_warp = dict(bound="hbm", kernel="mv_warp_kernel", achieved=w_gbs, peak=peaks["hbm_gbs"],
                         unit="GB/s", frac=w_gbs / peaks["hbm_gbs"],
                         traffic=w_traffic, traffic_unit="bytes/launch", traffic_source=w_src,
                         algorithmic_bytes_per_launch=WARP_BYTES_PER_PX * px, ms_per_launch=w_ms,
                         launches_timed=len(prof["warp"]), peak_source=peaks["source"])

    # ---------------- end to end from pinned host buffers (e2e)
    host = [{k: v.cpu().pin_memory() for k, v in c.items()} for c in clips[:1]]
    out_host = torch.empty((nc, T, 3, H, W), dtype=torch.float32).pin_memory()
    h2d = sum(v.numel() * v.element_size() for v in host[0].values())
    d2h = out_host.numel() * out_host.element_size()
    def run_e2e(n_steps, entry=None):
        entry = host[0] if entry is None else entry
        """The public host-clip API, driver.enhance_clips on HOST-resident entries: this rank's share of world x n_steps
        entries streams through driver.ClipStreamer -- frames are uploaded in chunks in the order the backward-time pass
        reads them, finished frames are downloaded chunk by chunk, the next entry's upload overlaps the kernels; every
        step still copies all of its inputs from pinned host memory and all of its frames back inside the timed region,
        and the per-frame metrics of all ranks meet in the job's one fixed-shape gather."""
        entries = [entry if c % world == rank else None for c in range(world * n_steps)]
        driver.enhance_clips(net, entries, rank, world, device=dev, out_hosts=[out_host] * len(entries),
                             chunk=max(1, min(10, T)))

    del clips
    torch.cuda.empty_cache()
    with torch.no_grad():
        # two warm-up steps: the streamer double-buffers its device copies, so the second step still allocates
        # (GB-sized cudaMallocs inside the timed region made this number swing between 230 and 300 frames/s)
        e2e_warm = min(args.warmup, 2) if args.frames >= 50 else args.warmup
        run_e2e(max(e2e_warm, 2))
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e2e_steps = args.steps
        f0.record()
        run_e2e(e2e_steps)
        f1.record()
        barrier()
    ms2 = torch.tensor([f0.elapsed_time(f1)], device=dev)
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    e2e_value = world * e2e_steps * T * nc / (float(ms2.item()) / 1e3)

    # ---------------- the same call fed with COMPACT side information (SURVEY 8(f-1)): the codec's per-block records
    # (40 bytes per block) go over the bus instead of the dense mvs / partitions planes and are rasterised on the
    # device inside the streamer (pnp_mv_rasterize, bit-exact replacement of loading_ipb.py:328-369)
    e2e_side = None
    if not args.no_sideinfo:
        import numpy as np
        from pnpvcve_b200 import sideinfo
        types = [chr(int(v)) for v in host[0]["slices"][0].flatten()]
        tmpl = sideinfo.synthetic_records(H, W, "IBBP", seed=77)          # record lists of an I, two B and a P frame
        per_type = {"I": [tmpl[0]], "B": [tmpl[1], tmpl[2]], "P": [tmpl[3]]}
        recs = [per_type[st][f % len(per_type[st])] for f, st in enumerate(types)]
        flat = np.concatenate(recs, 0)
        offs = np.cumsum([0] + [len(r) for r in recs])
        compact = {k: v for k, v in host[0].items() if k not in ("mvs", "partitions")}
        compact["side"] = [sideinfo.pack_side(flat, offs, types) for _ in range(nc)]
        side_h2d = sum(v.numel() * v.element_size() for k, v in compact.items() if k != "side") + \
            sum(sd["records"].numel() * 4 + sd["meta"].numel() * 4 for sd in compact["side"])
        # informational block: three timed repetitions of K steps, the median is reported next to all three (single
        # repetitions of this leg have shown one-off host-side stalls of 50-150 ms on some boxes)
        rates = []
        with torch.no_grad():
            run_e2e(2, compact)
            barrier()
            for _ in range(3):
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s0.record()
                run_e2e(e2e_steps, compact)
                s1.record()
                barrier()
                ms4 = torch.tensor([s0.elapsed_time(s1)], device=dev)
                if world > 1:
                    dist.all_reduce(ms4, op=dist.ReduceOp.MAX)
                rates.append(world * e2e_steps * T * nc / (float(ms4.item()) / 1e3))
        e2e_side = dict(value=sorted(rates)[1], unit="frames/s", repetitions=rates,
                        h2d_bytes_per_step=side_h2d, d2h_bytes_per_step=d2h, steps=e2e_steps,
                        records_per_frame=int(len(flat) / max(1, T)),
                        api="pnpvcve_b200.driver.enhance_clips on pinned host entries carrying `side` (per-block motion-"
                            "vector records of a synthetic H.264-style partition tree) instead of dense mvs / partitions")
    del host, out_host
    driver.release_streamers(net)          # (the legs below want the memory back)
    torch.cuda.empty_cache()

    # ---------------- frame-window sharding: ONE clip of the config cut into `world` windows, one per rank (strong
    # scaling of a single clip stream; north_star: "sharding independent clips or frame windows per GPU")
    windows = None
    if nc == 1 and T >= 2 * world and not args.no_windows:
        wclip = make_device_batch(cfg, T, 1, 7000, 0, dev)              # the same clip on every rank
        wlen = driver.balanced_window(T, world)
        with torch.no_grad():
            for _ in range(2):
                driver.enhance_windows(net, [wclip], wlen, rank, world, gather_output=True)
            barrier()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            wsteps = args.steps
            g0.record()
            for _ in range(wsteps):
                driver.enhance_windows(net, [wclip], wlen, rank, world, gather_output=True)
            g1.record()
            barrier()
        ms3 = torch.tensor([g0.elapsed_time(g1)], device=dev)
        if world > 1:
            dist.all_reduce(ms3, op=dist.ReduceOp.MAX)
        windows = dict(value=wsteps * T / (float(ms3.item()) / 1e3), unit="frames/s", scaling="strong",
                       workload=f"ONE {W}x{H}x{T} clip cut into {len(driver.frame_windows(T, wlen))} windows of <= {wlen} "
                                "frames, one per GPU, each enhanced as a clip of its own (window ends are forced key "
                                "frames); every rank ends with all frames and metrics (two fixed-shape NCCL all_gathers)",
                       steps=wsteps, window_frames=wlen, api="pnpvcve_b200.driver.enhance_windows")
        del wclip
        net._engine.prog = None
        torch.cuda.empty_cache()

    # ---------------- CPU baseline (rank 0, N=1 only): oracle port on a bounded sample
    cpu_baseline = None
    parity = None
    others = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        h, w, frames = cpu_sample(30.0, 1)
        sd = weights.random_state_dict(0)
        clip = make_cpu_clip(cfg, h, w, frames)
        kept = []
        dt = cpu_oracle_step(sd, clip, keep=kept)
        # the oracle's frames of that sample double as the checker of the CUDA path on the same inputs (max-abs on
        # [0,1] frames, tolerance 2e-3 of north_star) -- the sample has the config's frame size whenever the budget allows
        with torch.no_grad():
            got = net(*[a.to(dev) for a in synthetic.generator_args(clip)]).float().cpu()
        parity = dict(max_abs_err=float((got - kept[0]).abs().max()), tolerance=2e-3,
                      sample=sample_text(cfg, h, w, frames) + ", CUDA path vs CPU oracle port; the headline lengths "
                             "(T=100) are covered by tests/test_gpu_headline.py, table in profiles/r02_error_vs_frame.json")
        cpu_baseline = dict(value=frames * (h * w) / float(H * W) / dt, unit="frames/s", cores=cores, kind="port",
                            sample=f"oracle port (PyTorch fp32, {cores} threads), " + sample_text(cfg, h, w, frames)
                                   + ", one timed run after a 128x128 warm-up")
        if not args.no_other_configs:
            others = other_configs_block(net, dev, cfg["name"])

    if rank == 0:
        line = dict(metric=METRIC, value=value, unit="frames/s", n_gpus=world, steps=args.steps,
                    warmup=args.warmup, ms_per_step=steps_ms, higher_is_better=True, scaling="weak",
                    vs_baseline=None, dtype="bf16", data="synthetic", config=workload_config(args, world),
                    clocks=clocks, e2e=dict(value=e2e_value, unit="frames/s", h2d_bytes_per_step=h2d,
                                            d2h_bytes_per_step=d2h, steps=e2e_steps,
                                            api="pnpvcve_b200.driver.enhance_clips on pinned host entries (ClipStreamer: "
                                                "chunked H2D/D2H overlapped with the kernels)"),
                    e2e_sideinfo=e2e_side, frame_windows=windows,
                    gpu_launches=launches * world, launch_mode=net._engine.last_mode, roofline=roofline,
                    roofline_warp=roofline_warp,
                    kernels_ms=dict(block=mean_event_ms(prof["block"]), block_a=a_ms, block_b=b_ms, warp=w_ms),
                    mpx_per_s=value * H * W / 1e6, cpu_baseline=cpu_baseline, parity=parity, other_configs=others)
        _emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
