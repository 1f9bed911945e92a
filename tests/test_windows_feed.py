"""Frame windows fed with the codec's per-block records: sideinfo.window_side (CPU), pnp_mv_rasterize_window against the
whole clip's planes (GPU), and driver.enhance_windows with compact side information, uint8 frames and PSNR / SSIM."""
import os
import weakref

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import mv_raster_oracle as R
from pnpvcve_b200 import driver, sideinfo, synthetic

from test_sideinfo import CASES as GOLDEN_CASES, load_case

#: (name, pattern, H, W, messy)
PATTERNS = [("ibbp", "IBBPBBPBBP", 32, 48, False), ("allB", "BBBBBB", 32, 32, False),
            ("p_only", "PPPPPPP", 32, 32, False), ("starts_B", "BBPBBPBP", 32, 48, False),
            ("messy", "IBBPBPPBBP", 48, 64, True)]
LENGTHS, OVERLAPS = range(1, 6), range(0, 3)


def pattern_case(name):
    """(per-frame record lists, slice types, H, W) of one named case: a synthetic pattern or a committed raster golden"""
    for n, pattern, h, w, messy in PATTERNS:
        if n == name:
            return sideinfo.synthetic_records(h, w, pattern, seed=len(pattern) * 7 + h, messy=messy), list(pattern), h, w
    _, recs, pattern, h, w = load_case(name)
    return recs, pattern, h, w


def pack(recs, types):
    flat = np.concatenate(recs, 0) if recs else np.zeros((0, 10), np.float32)
    return sideinfo.pack_side(flat, np.cumsum([0] + [len(r) for r in recs]), types)


def all_windows(t):
    """every [a0, b0) enhance_windows cuts from a t-frame clip with windows of 1-5 frames and overlaps 0-2"""
    out = set()
    for length in LENGTHS:
        for ov in OVERLAPS:
            for a, b in driver.frame_windows(t, length):
                out.add((max(0, a - ov), min(t, b + ov)))
    return sorted(out)


def unpack(ws):
    n = ws["t"] + ws["tail"]
    meta = ws["meta"].tolist()
    return n, meta[:n + 1], meta[n + 1:2 * n + 1], meta[2 * n + 1:]


def emulate_window(ws, h, w):
    """The reference loader's loop (oracle/mv_raster_oracle.py) run over a window table with the rules of
    pnp_mv_rasterize_window: a tail record makes only its reversed write, a -2 target is skipped.  Returns
    (mvs, partitions, status bits)."""
    n, offs, is_b, tgt = unpack(ws)
    t = ws["t"]
    rec = ws["records"].numpy()
    mv = np.zeros((t, h, w, 4), np.float32)
    part = np.zeros((t, h, w, 3), np.float32)
    status = 0
    for f in range(n):
        for r in rec[offs[f]:offs[f + 1]]:
            direction, bw, bh, xs, ys, x, y, mx, my, sc = r
            x, y, bw, bh, xs, ys = int(x), int(y), int(bw), int(bh), int(xs), int(ys)
            mx, my = mx / sc, my / sc
            dst = (slice(y - bh // 2, y + bh // 2), slice(x - bw // 2, x + bw // 2))
            if f == t:
                assert direction > 0
            if direction < 0 and f < t:
                mv[f][dst + (0,)], mv[f][dst + (1,)] = mx, my
            elif direction > 0 and f < t and is_b[f]:
                mv[f][dst + (2,)], mv[f][dst + (3,)] = mx, my
            elif direction > 0:
                if tgt[f] == -1:
                    status |= 2
                elif tgt[f] >= 0:
                    src = (slice(ys - bh // 2, ys + bh // 2), slice(xs - bw // 2, xs + bw // 2))
                    mv[tgt[f]][src + (2,)], mv[tgt[f]][src + (3,)] = -mx, -my
            if f < t:
                if bw * bh in R.PARTITION_CHANNEL:
                    part[f][dst + (R.PARTITION_CHANNEL[bw * bh],)] = 1
                else:
                    status |= 1
    return mv.transpose(0, 3, 1, 2), (part / 255).astype(np.float32).transpose(0, 3, 1, 2), status


# ------------------------------------------------------------------ CPU: window_side
@pytest.mark.parametrize("name", [p[0] for p in PATTERNS] + GOLDEN_CASES)
def test_window_side_selects_the_records_that_reach_the_window(name):
    recs, types, h, w = pattern_case(name)
    t = len(types)
    side = pack(recs, types)
    emv, epar = R.rasterize_clip(recs, types, h, w)
    targets = sideinfo.p_targets(types)
    for a, b in all_windows(t):
        ws = sideinfo.window_side(side, a, b)
        n, offs, is_b, tgt = unpack(ws)
        assert ws["t"] == b - a and ws["tail"] in (0, 1)
        # records: the window's rows, then only the reversed rows of e = the first non-B frame >= b, in clip order
        e = next((f for f in range(b, t) if types[f] != "B"), None)
        want = [recs[f] for f in range(a, b)]
        if ws["tail"]:
            assert e is not None and a <= targets[e] < b
            want.append(recs[e][recs[e][:, 0] > 0])
        else:
            assert e is None or targets[e] < a
        assert torch.equal(ws["records"], torch.from_numpy(np.concatenate(want, 0).reshape(-1, 10)))
        # window-relative offsets, B flags and targets
        assert offs == np.cumsum([0] + [len(r) for r in want]).tolist()
        assert is_b == [int(types[f] == "B") for f in range(a, b)] + [0] * ws["tail"]
        for i, f in enumerate(list(range(a, b)) + ([e] if ws["tail"] else [])):
            g = targets[f]
            assert tgt[i] == (g - a if g >= a else -2 if g >= 0 else -1)
            if types[f] != "B" and tgt[i] == -1:
                assert f == 0                            # -1 survives only for frame 0 of the clip
        # the window table computes frames [a, b) of the whole clip
        mv, par, status = emulate_window(ws, h, w)
        assert status == 0
        assert np.array_equal(mv, emv[a:b]) and np.array_equal(par, epar[a:b]), (a, b)


def test_window_side_rejects_windows_outside_the_clip():
    side = pack(*pattern_case("ibbp")[:2])
    for a, b in ((0, 0), (-1, 2), (3, 11), (5, 4)):
        with pytest.raises(ValueError):
            sideinfo.window_side(side, a, b)


def error_case():
    """P B B P B P: frame 0 carries a reversed record (ValueError: p_offset unbound), frame 3 a block of area 16
    among its reversed rows (KeyError)"""
    types = list("PBBPBP")
    recs = sideinfo.synthetic_records(32, 32, types, seed=3)
    recs[0] = np.concatenate([recs[0], np.array([[1, 8, 8, 8, 8, 8, 8, 1, 1, 4]], np.float32)], 0)
    recs[3] = np.concatenate([recs[3], np.array([[1, 4, 4, 9, 9, 9, 9, 2, 2, 4]], np.float32)], 0)
    return recs, types


def expected_status(a, b):
    return (1 if a <= 3 < b else 0) | (2 if a == 0 else 0)


def test_window_errors_stay_with_the_frame_that_causes_them():
    recs, types = error_case()
    side = pack(recs, types)
    for a, b in all_windows(len(types)):
        ws = sideinfo.window_side(side, a, b)
        if b <= 3 and a <= 0:
            assert ws["tail"] == 1                       # frame 3 rides along as a tail; its KeyError is not reported
        assert emulate_window(ws, 32, 32)[2] == expected_status(a, b), (a, b)


# ------------------------------------------------------------------ CPU: enhance_windows with a stand-in streamer
def _stand_in(lq):
    """depends on the window's first and last frame, as the generator does through the forced key frames"""
    return lq * 2.0 + lq[:, :1] - lq[:, -1:]


class _Net:
    """stand-in generator: enhance_windows streams host clips through `forward_streamed` nets"""
    vsr = False

    def forward_streamed(self, *args, **kw):
        raise AssertionError("called through the streamer")


class _Streamer:
    """ClipStreamer's interface on the CPU: records what is uploaded and into which host buffers it downloads"""
    made = 0

    def __init__(self, net, device, chunk=10):
        type(self).made += 1
        self._net = weakref.ref(net)
        self.uploads, self.targets = [], []

    def upload(self, host_clip):
        self.uploads.append(host_clip)
        return host_clip

    def run(self, ticket, out_host):
        lq = ticket["lq"].float() / 255.0 if ticket["lq"].dtype == torch.uint8 else ticket["lq"]
        y = _stand_in(lq)
        out_host.copy_((y.clamp(0, 1) * 255.0).round().to(torch.uint8) if out_host.dtype == torch.uint8 else y)
        self.targets.append(out_host)
        return out_host.clone()

    def finish(self, check=False):
        pass


def _host_clip(t, seed):
    clip = synthetic.make_clip(32, 32, t, seed=seed, ipb=True)
    types = [chr(int(v)) for v in clip["slices"].flatten()]
    side = pack(sideinfo.synthetic_records(32, 32, types, seed=seed), types)
    clip["lq"] = (clip["lq"] * 255.0).round().to(torch.uint8)
    return dict({k: v for k, v in clip.items() if k not in ("mvs", "partitions")}, side=[side])


def test_enhance_windows_reuses_the_cached_streamer_and_result_buffers(monkeypatch):
    monkeypatch.setattr(driver, "ClipStreamer", _Streamer)
    _Streamer.made = 0
    net = _Net()
    clip = _host_clip(17, 5)
    try:
        for call in range(2):
            outs, met = driver.enhance_windows(net, [clip], 4, overlap=1, device="cpu", out_dtype=torch.uint8)
            assert _Streamer.made == 1
            st = driver.streamer_for(net, "cpu", 10)
            # one download target per window shape (windows of 5, 6, 6, 6 and 2 frames with the overlap)
            targets = st.targets[5 * call:]
            assert [x.shape[1] for x in targets] == [5, 6, 6, 6, 2]
            assert len({id(x) for x in targets}) == 3 and all(x is targets[1] for x in targets[1:4])
        assert all(o.dtype == torch.uint8 for o in outs.values()) and met.shape == (1, 17, driver.N_METRICS)
    finally:
        driver.release_streamers(net)


def test_enhance_windows_checks_the_output_dtype():
    with pytest.raises(ValueError):
        driver.enhance_windows(_stand_in, [synthetic.make_clip(32, 32, 4, seed=1)], 2, out_dtype=torch.float16)


def _gloo_worker(rank, world, port, t, window, overlap, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    driver.ClipStreamer = _Streamer
    net = _Net()
    full, met = driver.enhance_windows(net, [_host_clip(t, 9)], window, rank, world, overlap=overlap,
                                       gather_output=True, device="cpu", out_dtype=torch.uint8)
    st = driver.streamer_for(net, "cpu", 10)
    # (numpy: pickled by value -- a torch tensor would travel as a shared-memory handle that dies with this process)
    q.put((rank, full.numpy(), met.numpy(), [u["side"][0]["records"].numpy() for u in st.uploads]))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("t,window,overlap", [(11, 4, 0), (9, 3, 2)])
def test_windows_world2_upload_own_records_and_gather_uint8(t, window, overlap):
    """Two ranks over gloo: each uploads only the records of its own windows (overlap included), and every rank ends
    with all frames as uint8."""
    import socket
    world = 2
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_gloo_worker, args=(r, world, port, t, window, overlap, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = [q.get(timeout=300) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    clip = _host_clip(t, 9)
    exp = torch.empty((1, t, 3, 32, 32), dtype=torch.uint8)
    for a, b in driver.frame_windows(t, window):
        a0, b0 = max(0, a - overlap), min(t, b + overlap)
        y = _stand_in(clip["lq"][:, a0:b0].float() / 255.0)[:, a - a0:b - a0]
        exp[:, a:b] = (y.clamp(0, 1) * 255.0).round().to(torch.uint8)
    whole = clip["side"][0]["records"].shape[0]
    for rank, full, met, uploaded in got:
        assert full.dtype == np.uint8 and np.array_equal(full, exp.numpy())
        assert met.shape == (1, t, driver.N_METRICS) and not np.isnan(met).any()
        mine = driver.shard_windows(1, t, window, rank, world)
        assert len(uploaded) == len(mine)
        for (c, a, b), rec in zip(mine, uploaded):
            ws = sideinfo.window_side(clip["side"][0], max(0, a - overlap), min(t, b + overlap))
            assert np.array_equal(rec, ws["records"].numpy()) and len(rec) < whole


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pnpvcve_b200 import _lib
    _lib.require_device()
    return torch.device("cuda:0")


def rasterize_window(ws, h, w, dev):
    """window_side entry -> (mvs, partitions, status bits) through pnp_mv_rasterize_window"""
    rec, meta, _ = sideinfo.upload_side(ws, dev)
    t = ws["t"]
    mvs = torch.full((t, 4, h, w), float("nan"), device=dev)
    par = torch.full((t, 3, h, w), float("nan"), device=dev)
    work = torch.empty((3, t, h, w), dtype=torch.int32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        sideinfo.rasterize_uploaded(rec, meta, t, mvs, par, work, status, ws["tail"])
    return mvs.cpu(), par.cpu(), int(status.item())


@pytest.mark.gpu
@pytest.mark.parametrize("name", [p[0] for p in PATTERNS] + GOLDEN_CASES)
def test_window_planes_equal_the_whole_clip_slice(dev, name):
    recs, types, h, w = pattern_case(name)
    side = pack(recs, types)
    emv, epar = R.rasterize_clip(recs, types, h, w)
    flat = side["records"].numpy()
    kmv, kpar = sideinfo.rasterize_clip(flat, side["meta"][:len(types) + 1].numpy(), types, h, w, device=dev)
    kmv, kpar = kmv.cpu(), kpar.cpu()
    assert torch.equal(kmv, torch.from_numpy(emv)) and torch.equal(kpar, torch.from_numpy(epar))
    for a, b in all_windows(len(types)):
        mv, par, status = rasterize_window(sideinfo.window_side(side, a, b), h, w, dev)
        assert status == 0, (a, b)
        assert torch.equal(mv, kmv[a:b]) and torch.equal(par, kpar[a:b]), (a, b)


@pytest.mark.gpu
def test_window_errors_are_raised_by_the_owning_window_only(dev):
    recs, types = error_case()
    side = pack(recs, types)
    for a, b in all_windows(len(types)):
        st = rasterize_window(sideinfo.window_side(side, a, b), 32, 32, dev)[2]
        assert st == expected_status(a, b), (a, b)
        if st & 1:
            with pytest.raises(KeyError):
                sideinfo.raise_for_status(st)
        elif st & 2:
            with pytest.raises(ValueError):
                sideinfo.raise_for_status(st)


@pytest.mark.gpu
@pytest.mark.parametrize("overlap", [0, 2])
def test_enhance_windows_records_uint8_in_and_out(dev, overlap):
    """Host clip with `side`, uint8 lq, uint8 frames out: every window equals tensor2img of the dense fp32 run on
    oracle-rasterised planes; gather_output gives the same frames; PSNR / SSIM equal frame_quality on them."""
    from pnpvcve_b200 import metrics
    from test_frames_u8 import _net, quant
    net = _net(dev)
    h, w, t, window = 64, 96, 10, 4
    clip = synthetic.make_clip(h, w, t, seed=81, ipb=True)
    types = [chr(int(v)) for v in clip["slices"].flatten()]
    recs = sideinfo.synthetic_records(h, w, types, seed=82, messy=True)
    emv, epar = R.rasterize_clip(recs, types, h, w)
    u8 = (clip["lq"] * 255.0).round().to(torch.uint8)
    dense = dict(clip, lq=u8.float() / 255.0, mvs=torch.from_numpy(emv)[None], partitions=torch.from_numpy(epar)[None])
    compact = dict({k: v for k, v in clip.items() if k not in ("mvs", "partitions")}, lq=u8, side=[pack(recs, types)])
    gts = [torch.randint(0, 256, (1, t, 3, h, w), generator=torch.Generator().manual_seed(83), dtype=torch.uint8)]
    outs_f, _ = driver.enhance_windows(net, [dense], window, overlap=overlap, device=dev, chunk=3)
    outs_u, met_u = driver.enhance_windows(net, [compact], window, overlap=overlap, device=dev, chunk=3,
                                           out_dtype=torch.uint8)
    frames, met_g = driver.enhance_windows(net, [compact], window, overlap=overlap, device=dev, chunk=3,
                                           out_dtype=torch.uint8, gather_output=True, gts=[g.to(dev) for g in gts])
    torch.cuda.synchronize()
    assert outs_u.keys() == outs_f.keys()
    for k in outs_u:
        assert outs_u[k].dtype == torch.uint8 and torch.equal(outs_u[k], quant(outs_f[k])), k
    assert frames.dtype == torch.uint8 and tuple(frames.shape) == (1, t, 3, h, w)
    for (c, a, b), o in outs_u.items():
        assert torch.equal(frames[c, a:b], o[0])
    assert torch.equal(met_g[..., :2], met_u) and met_g.shape == (1, t, driver.N_METRICS + 2)
    q = metrics.frame_quality(frames, gts[0].to(dev))
    assert torch.equal(met_g[..., 2], q["psnr"].float())                 # the SSE, bit for bit
    assert (met_g[..., 3].double() - q["ssim"]).abs().max().item() <= 1e-7   # fp32 of an SSIM equal to ~1e-16
    ev = metrics.evaluate(frames, gts[0].to(dev))
    assert abs(ev["SSIM"].item() - q["ssim"].mean().item()) <= 1e-15
    assert torch.equal(ev["PSNR"], q["psnr"].mean())
