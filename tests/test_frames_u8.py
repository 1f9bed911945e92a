"""8-bit frames end to end: uint8 lq in (value v stands for float32(v) / 255, the reference loader's RescaleToZeroOne),
tensor2img-exact uint8 frames out (the uint8 store of conv_last), and the metrics on uint8 operands."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import metrics_oracle as M
from pnpvcve_b200 import _lib, driver, ops, synthetic

from helpers import metric_cases


def dequant_table():
    """float32(v) / 255 for v = 0..255, correctly rounded (the float64 quotient rounded once to float32)."""
    return (np.arange(256, dtype=np.float64) / 255.0).astype(np.float32)


def quant(x):
    """tensor2img's uint8 value of fp32 samples: clamp to [0,1], x255 in fp32, round half to even."""
    return (x.clamp(0.0, 1.0) * 255.0).round().to(torch.uint8)


def to_u8(x):
    """8-bit frames of fp32 frames in [0,1] (any uint8 values would do)."""
    return quant(x)


def dequant(u8):
    """numpy's dequantisation of 8-bit frames, as the reference's loader computes it."""
    return torch.from_numpy(u8.cpu().numpy().astype(np.float32) / 255.)


# ------------------------------------------------------------------ CPU
def test_dequantisation_rule_over_all_values():
    v = np.arange(256, dtype=np.uint8)
    loader = v.astype(np.float32) / 255.                              # normalization.py:93-99
    assert loader.dtype == np.float32
    assert np.array_equal(loader.view(np.uint32), dequant_table().view(np.uint32))
    # what the driver's metrics use for uint8 frames is the same number
    assert torch.equal(torch.arange(256, dtype=torch.uint8).float() / 255.0, torch.from_numpy(dequant_table()))
    # multiplying by fl(1/255) is not the same rule
    assert int((v.astype(np.float32) * np.float32(1 / 255) != loader).sum()) == 126
    # tensor2img(v / 255) == v: a uint8 GT and the fp32 GT it was decoded to score identically
    chw = np.broadcast_to(loader, (3, 1, 256)).copy()
    assert np.array_equal(M.tensor2img_u8(chw)[0, :, 0], v)           # (HWC, BGR: channel 0 is input channel 2)


def test_new_entry_points_reject_null_pointers_without_gpu():
    lib = _lib.load()
    assert lib.pnp_unit_from_u8(None, 0, 0, 0, None, 0, 0, 0, 1, 4, 4, None) == -1
    assert b"null" in lib.pnp_last_error()
    assert lib.pnp_frame_quality_u8(None, 1, 0, 0, 0, None, 0, 0, 0, 0, 1, 16, 16, 0, None, None, None) == -1
    assert b"null" in lib.pnp_last_error()
    # out_u8 is a PNP_CONV_LAST option only
    d = _lib.ConvDesc()
    d.src, d.wpack, d.out = 1 << 12, 2 << 12, 3 << 12
    d.N, d.H, d.W, d.tap_n, d.mode, d.out_u8 = 1, 64, 64, 64, ops.PNP_CONV_BF16, 1
    assert lib.pnp_conv3x3(ctypes.byref(d), None) == -1
    assert b"out_u8" in lib.pnp_last_error()


def test_enhance_clips_checks_the_output_dtype():
    clip = synthetic.make_clip(64, 64, 2, seed=1)
    with pytest.raises(ValueError):
        driver.enhance_clips(None, [clip], out_dtype=torch.float16)
    with pytest.raises(ValueError):
        driver.enhance_clips(None, [clip], out_dtype=torch.uint8, out_hosts=[torch.empty((1, 2, 3, 64, 64))])
    with pytest.raises(ValueError):
        driver.enhance_clips(None, [clip], out_hosts=[torch.empty((1, 2, 3, 64, 64), dtype=torch.uint8)])


def test_frame_metrics_take_uint8_frames_in_unit_scale():
    g = torch.Generator().manual_seed(3)
    u = torch.randint(0, 256, (1, 2, 3, 8, 8), generator=g, dtype=torch.uint8)
    r = torch.randint(0, 256, (1, 2, 3, 8, 8), generator=g, dtype=torch.uint8)
    assert torch.equal(driver.frame_metrics(u), driver.frame_metrics(u.float() / 255.0))
    assert torch.equal(driver.frame_metrics(u, r), driver.frame_metrics(u.float() / 255.0, r.float() / 255.0))


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    _lib.require_device()
    return torch.device("cuda:0")


@pytest.mark.gpu
def test_unit_from_u8_all_values_and_strided_views(dev):
    table = torch.from_numpy(dequant_table()).to(dev)
    v = torch.arange(256, dtype=torch.uint8, device=dev).view(1, 1, 1, 256).expand(2, 3, 4, 256).contiguous()
    out = torch.full(v.shape, float("nan"), device=dev)
    ops.unit_from_u8(v, out)
    assert torch.equal(out, table[v.long()])
    # 720p strided views on both sides: a crop of a larger uint8 clip into a channel-strided fp32 buffer
    g = torch.Generator(device=dev).manual_seed(7)
    big = torch.randint(0, 256, (3, 3, 724, 1290), generator=g, dtype=torch.uint8, device=dev)
    src = big[:, :, 2:722, 5:1285]
    dst_buf = torch.full((3, 4, 720, 1296), -1.0, device=dev)
    dst = dst_buf[:, 1:, :, 8:1288]
    ops.unit_from_u8(src, dst)
    assert torch.equal(dst, table[src.long()])
    assert (dst_buf[:, 0] == -1).all() and (dst_buf[..., :8] == -1).all() and (dst_buf[..., 1288:] == -1).all()
    # (n,T,3,H,W) form, as the engine calls it
    five = big[:2].reshape(1, 2, 3, 724, 1290)
    o5 = torch.empty(five.shape, device=dev)
    ops.unit_from_u8(five, o5)
    assert torch.equal(o5, table[five.long()])
    with pytest.raises(ValueError):
        ops.unit_from_u8(src.float(), dst)


def _last_table_launch(x, wp, bias, lq, outf, lq_up4):
    """the same conv_last launch in table mode: wpack / bias / lq / outf come from a one-step launch table"""
    dev = x.device
    n, h, w, _ = x.shape
    table = torch.zeros((1, 1, _lib.DYN_ENTRY_WORDS), dtype=torch.int64)
    table[0, 0, :5] = torch.tensor([wp.data_ptr(), bias.data_ptr(), 0, lq.data_ptr(), outf.data_ptr()])
    table = table.to(dev)
    step = torch.zeros(1, dtype=torch.int32, device=dev)
    d = ops.ConvDesc()
    d.src, d.src_images = x.data_ptr(), n
    d.bias, d.lq, d.outf = 1, 1, 1
    d.lq_sn, d.lq_sc, d.lq_sy = lq.stride(0), lq.stride(1), lq.stride(2)
    d.of_sn, d.of_sc, d.of_sy = outf.stride(0), outf.stride(1), outf.stride(2)
    d.N, d.H, d.W, d.tap_n, d.mode, d.wpack_stable = n, h, w, 16, ops.PNP_CONV_LAST, 1
    d.lq_up4 = 1 if lq_up4 else 0
    d.out_u8 = 1 if outf.dtype == torch.uint8 else 0
    d.dyn.table, d.dyn.step, d.dyn.node, d.dyn.stride = table.data_ptr(), step.data_ptr(), 0, 1
    _lib.check(_lib.load().pnp_conv3x3(ctypes.byref(d), ops._stream()), "pnp_conv3x3 (table)")
    torch.cuda.current_stream().synchronize()          # (the table lives only as long as this call)


@pytest.mark.gpu
@pytest.mark.parametrize("n,h,w", [(1, 64, 64), (2, 72, 200), (1, 376, 1244), (1, 720, 1280)])
def test_conv_last_uint8_store_equals_quantised_fp32_store(dev, n, h, w):
    """out_u8 on conv_last: plain and lq_up4 forms, single-CTA and CTA-pair mode, static and table launches -- the uint8
    frame is quant_u8 of the fp32 frame the same launch stores, bit for bit."""
    lib = _lib.load()
    g = torch.Generator(device=dev).manual_seed(n * 7 + h + w)
    x = torch.randn((n, 64, h, w), generator=g, device=dev).permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)
    wl = torch.randn((3, 64, 3, 3), generator=g, device=dev) * 0.04
    bias = torch.randn(3, generator=g, device=dev) * 0.1
    wp = ops.new_wpack_rowstack(dev, tap_n=16)
    ops.pack_conv3x3_rowstack(wl, wp, tap_n=16)
    for lq_up4 in (False, True):
        lq = torch.rand((n, 3, h // 4, w // 4) if lq_up4 else (n, 3, h, w), generator=g, device=dev) * 1.2 - 0.1
        ref = torch.empty((n, 3, h, w), device=dev)
        ops.conv3x3(x, wp, bias=bias, lq=lq, outf=ref, lq_up4=lq_up4)
        want = quant(ref)
        assert (ref < 0).any() and (ref > 1).any()           # both clamps are exercised
        prev = lib.pnp_set_pair_mode(0)
        try:
            for mode in (0, 1):
                lib.pnp_set_pair_mode(mode)
                got = torch.full((n, 3, h, w), 7, dtype=torch.uint8, device=dev)
                ops.conv3x3(x, wp, bias=bias, lq=lq, outf=got, lq_up4=lq_up4)
                assert torch.equal(got, want), f"static, pair mode {mode}, lq_up4={lq_up4}"
                got.fill_(7)
                _last_table_launch(x, wp, bias, lq, got, lq_up4)
                assert torch.equal(got, want), f"table, pair mode {mode}, lq_up4={lq_up4}"
                f32 = torch.empty_like(ref)
                _last_table_launch(x, wp, bias, lq, f32, lq_up4)
                assert torch.equal(f32, ref)
        finally:
            lib.pnp_set_pair_mode(prev)
    # a strided uint8 destination (a crop of a wider buffer): the strides are in bytes
    buf = torch.zeros((n, 3, h, w + 16), dtype=torch.uint8, device=dev)
    ops.conv3x3(x, wp, bias=bias, lq=lq, outf=buf[..., 8:8 + w], lq_up4=True)
    assert torch.equal(buf[..., 8:8 + w], want) and not buf[..., :8].any() and not buf[..., 8 + w:].any()


# ------------------------------------------------------------------ generator
def _net(dev, **kw):
    import pnpvcve_b200 as P
    from pnpvcve_b200 import weights
    from test_gpu_parity import GENERATOR_CFG
    net = P.build_backbone(dict(GENERATOR_CFG, num_blocks=2, **kw))
    net.load_state_dict(weights.random_state_dict(11, num_blocks=2, vsr=bool(kw.get("vsr"))), strict=True)
    return net.to(dev).eval()


def _case(name):
    """(generator kwargs, clip dict on the host with uint8 lq) of one case"""
    if name == "c1":
        clip = synthetic.make_config_clip("C1")
        kw = {}
    elif name == "ipb_n2_crf":
        clip = synthetic.cat_clips([synthetic.make_clip(96, 128, 6, seed=21 + c, crf=(15, 35)[c], ipb=True)
                                    for c in range(2)])
        kw = {}
    elif name == "pad_66x130":
        clip = synthetic.make_clip(66, 130, 5, seed=31)
        for k, ch in (("mvs", 4), ("partitions", 3)):            # the pad contract: planes at the padded size, zeros
            padded = torch.zeros((1, 5, ch, 68, 132))
            padded[..., :66, :130] = clip[k]
            clip[k] = padded
        kw = {}
    elif name == "vsr":
        clip = synthetic.make_clip(64, 80, 5, seed=41)
        kw = dict(vsr=True)
    elif name == "sparse":
        clip = synthetic.overlap_partitions(synthetic.make_clip(64, 96, 6, seed=51, ipb=True), 52)
        kw = dict(sparse_val=True)
    else:                                                         # 720p, short
        clip = synthetic.make_config_clip("C2", t=3)
        kw = {}
    clip["lq"] = to_u8(clip["lq"])
    return kw, clip


CASES = ["c1", "ipb_n2_crf", "pad_66x130", "vsr", "sparse", "720p"]


def _args(clip, dev, lq=None):
    a = [v.to(dev) for v in synthetic.generator_args(clip)]
    if lq is not None:
        a[0] = lq.to(dev)
    return a


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_generator_uint8_lq_equals_dequantised_fp32_lq(dev, name):
    kw, clip = _case(name)
    net = _net(dev, **kw)
    with torch.no_grad():
        a = net(*_args(clip, dev))
        b = net(*_args(clip, dev, dequant(clip["lq"])))
        # a non-contiguous uint8 view (every other frame of a longer clip) takes the same path
        t = clip["lq"].shape[1]
        twice = torch.stack([clip["lq"], torch.zeros_like(clip["lq"])], 2).flatten(1, 2).to(dev)
        c = net(*_args(clip, dev, twice[:, 0:2 * t:2]))
    assert a.dtype == torch.float32 and torch.equal(a, b) and torch.equal(a, c)


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_generator_uint8_output_equals_quantised_fp32_output(dev, name):
    """forward_streamed(out=uint8) == quant_u8(fp32 output), with graphs and in table mode without graphs; fp32 and
    uint8 calls alternate on one generator, so the graph / node cache must keep the two outputs apart."""
    kw, clip = _case(name)
    net = _net(dev, **kw)
    eng = net._engine
    args = _args(clip, dev)
    with torch.no_grad():
        for graphs in (True, False):
            eng.use_graphs = graphs
            for rep in range(2):
                ref = net(*args)
                u8 = torch.full(ref.shape, 3, dtype=torch.uint8, device=dev)
                got = net.forward_streamed(*args, out=u8)
                assert got is u8 and eng.last_mode == ("graph" if graphs else "eager")
                assert torch.equal(u8, quant(ref)), f"graphs={graphs}, round {rep}"
                f32 = torch.empty_like(ref)
                net.forward_streamed(*args, out=f32)
                assert torch.equal(f32, ref)
    keys = list(eng.prog.nodes)
    assert any(k[-1] for k in keys) and any(not k[-1] for k in keys)


@pytest.mark.gpu
@pytest.mark.parametrize("feed", ["dense", "side"])
def test_enhance_clips_uint8_frames_in_and_out(dev, feed):
    from oracle import mv_raster_oracle as R
    from test_sideinfo import _side_entries
    net = _net(dev)
    h, w, t, n = 64, 96, 7, 2
    dense, compact = _side_entries(h, w, t, n, 60, R.rasterize_clip)
    entries = dense if feed == "dense" else compact
    g = torch.Generator().manual_seed(9)
    for d, c in zip(dense, compact):
        d["lq"] = c["lq"] = to_u8(d["lq"])
    gts_u8 = [torch.randint(0, 256, (n, t, 3, h, w), generator=g, dtype=torch.uint8) for _ in entries]
    gts_f32 = [x.float() / 255.0 for x in gts_u8]
    # device-resident entries (dense planes) with uint8 frames in and out
    dev_entries = [{k: v.to(dev) for k, v in e.items()} for e in dense]
    outs_dev, _ = driver.enhance_clips(net, dev_entries, out_dtype=torch.uint8)
    outs_u8, met_u8 = driver.enhance_clips(net, entries, device=dev, chunk=3, out_dtype=torch.uint8,
                                           gts=[x.to(dev) for x in gts_u8])
    st = driver.streamer_for(net, dev, 3)
    h2d_u8, d2h_u8 = st.h2d_bytes, st.d2h_bytes
    _, met_u8_f = driver.enhance_clips(net, entries, device=dev, chunk=3, out_dtype=torch.uint8,
                                       gts=[x.to(dev) for x in gts_f32])
    fp_entries = [dict(e, lq=dequant(e["lq"]).pin_memory()) for e in entries]
    outs_f32, met_f32 = driver.enhance_clips(net, fp_entries, device=dev, chunk=3, gts=[x.to(dev) for x in gts_u8])
    h2d_f32, d2h_f32 = st.h2d_bytes, st.d2h_bytes
    torch.cuda.synchronize()
    for a, b, f in zip(outs_u8, outs_dev, outs_f32):
        assert a.dtype == torch.uint8 and a.is_pinned() and torch.equal(a, b.cpu())
        assert torch.equal(a, quant(f))
    # 1-byte frames: the last entry's lq and output bytes
    assert d2h_u8 == n * t * 3 * h * w and d2h_f32 == 4 * d2h_u8
    assert h2d_f32 - h2d_u8 == 3 * n * t * 3 * h * w
    # PSNR / SSIM: uint8 GT == fp32 GT = gt / 255, and uint8 output == fp32 output -- exactly, up to the order of the
    # float64 atomics that add up the SSIM map (one fp32 ulp of the gathered value at most)
    assert torch.equal(met_u8[..., :3], met_u8_f[..., :3]) and torch.equal(met_u8[..., 2], met_f32[..., 2])
    for other in (met_u8_f, met_f32):
        assert (met_u8[..., 3] - other[..., 3]).abs().max().item() <= 1e-7
    assert torch.isfinite(met_u8).all()


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(metric_cases()))
def test_frame_quality_uint8_operands_equal_fp32_path(dev, name):
    from pnpvcve_b200 import metrics
    out, gt, crop = metric_cases()[name]
    out, gt = out[None].to(dev), gt[None].to(dev)
    ref = metrics.frame_quality(out, gt, crop)
    for a, b in ((quant(out), quant(gt)), (quant(out), gt), (out, quant(gt))):
        q = metrics.frame_quality(a, b, crop)
        for k in ("sse", "psnr"):                            # exact integer work
            assert torch.equal(q[k], ref[k]), (k, a.dtype, b.dtype)
        # the per-block float64 partial sums of the SSIM map are equal; they meet in float64 atomics whose order varies
        # from launch to launch for any operand types, so the totals agree to the last few bits
        assert (q["ssim"] - ref["ssim"]).abs().max().item() <= 1e-13, (a.dtype, b.dtype)
    ev = metrics.evaluate(quant(out), gt, crop)
    assert abs(ev["SSIM"].item() - ref["ssim"].mean().item()) <= 1e-13
    with pytest.raises(ValueError):
        metrics.frame_quality(out.half(), gt, crop)


@pytest.mark.gpu
def test_enhance_windows_takes_a_uint8_host_clip(dev):
    net = _net(dev)
    clip = synthetic.make_clip(64, 96, 9, seed=71)
    clip["lq"] = to_u8(clip["lq"])
    fp = dict(clip, lq=dequant(clip["lq"]))
    outs_u8, met_u8 = driver.enhance_windows(net, [clip], 4, overlap=1, device=dev, chunk=3)
    outs_f32, met_f32 = driver.enhance_windows(net, [fp], 4, overlap=1, device=dev, chunk=3)
    torch.cuda.synchronize()
    assert outs_u8.keys() == outs_f32.keys()
    for k in outs_u8:
        assert outs_u8[k].dtype == torch.float32 and torch.equal(outs_u8[k], outs_f32[k])
    assert torch.equal(met_u8, met_f32)
    # device-resident uint8 clip: the engine dequantises it
    outs_d, _ = driver.enhance_windows(net, [{k: v.to(dev) for k, v in clip.items()}], 4, overlap=1)
    for k in outs_u8:
        assert torch.equal(outs_d[k], outs_f32[k])
