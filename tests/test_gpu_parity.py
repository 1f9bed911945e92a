"""End-to-end parity of the registry-built generator on a B200 against the reference's golden
vectors and the CPU oracle.  north_star tolerance: max-abs 2e-3 on [0,1] frames, PSNR delta
<= 0.02 dB, key schedule / tap indices bit exact (taps: tests/test_gpu_kernels.py)."""
import pytest
import torch

from oracle import bae_oracle as O
import pnpvcve_b200 as P
from pnpvcve_b200 import synthetic, weights

from helpers import build_case, check_against_golden, golden_cases

pytestmark = pytest.mark.gpu

TOL = 2e-3
GENERATOR_CFG = dict(
    type="IconVSR_restore_wo_refill_mv_ipb_fast_domain_dynamic_with_par",
    mid_channels=64, num_blocks=8, padding=3, with_cat=True, use_base_qp=True, num_experts=6,
    expert_softmax=True, init_weight=True, with_bias=True, with_se=True, with_par=True,
    one_layer=True, blocktype="drt", channel_first=True, sparse_val=False, align_key=True, vsr=False)


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def build(sd, dev, **over):
    cfg = dict(GENERATOR_CFG)
    cfg.update(over)
    net = P.build_backbone(cfg)
    net.load_state_dict(sd, strict=True)
    return net.to(dev).eval()


def run(net, clip, dev):
    args = [a.to(dev) for a in synthetic.generator_args(clip)]
    with torch.no_grad():
        out = net(*args)
    torch.cuda.synchronize()
    return out


CASES = [c for c in golden_cases() if c != "warp_720p"]


@pytest.mark.parametrize("name", CASES)
def test_generator_matches_reference_golden(dev, name):
    sd, clip, gold = build_case(name)
    case = golden_cases()[name]
    net = build(sd, dev, vsr=bool(case.get("vsr")), sparse_val=bool(case.get("sparse_val")))
    out = run(net, clip, dev)
    assert out.dtype == torch.float32 and out.is_cuda
    err = check_against_golden(out, gold, tol=TOL, lq=clip["lq"], vsr=bool(case.get("vsr")))
    assert net.gpu_launches > 0
    print(f"{name}: max-abs vs reference golden {err:.2e}")


@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("name", CASES)
def test_generator_in_pair_form_matches_reference_golden(dev, name, mode):
    """The whole generator with every eligible conv launch in the CTA-pair (cta_group::2) form (mode 2: phantom
    columns included), for every golden case with its vsr / sparse_val flags: same reference goldens, and bit-identical
    to the default form.  Catches a pair-form defect on an optional path: the strided PixelShufflePack stores of the vsr
    tail, the sparse partition blend, all-B / mirrored / one-frame schedules."""
    from pnpvcve_b200 import _lib
    lib = _lib.load()
    sd, clip, gold = build_case(name)
    case = golden_cases()[name]
    flags = dict(vsr=bool(case.get("vsr")), sparse_val=bool(case.get("sparse_val")))
    ref = run(build(sd, dev, **flags), clip, dev)
    prev = lib.pnp_set_pair_mode(mode)
    try:
        out = run(build(sd, dev, **flags), clip, dev)
    finally:
        lib.pnp_set_pair_mode(prev)
    check_against_golden(out, gold, tol=TOL, lq=clip["lq"], vsr=flags["vsr"])
    assert torch.equal(out, ref)


def psnr_delta(out, ref, seed=0):
    """PSNR (tensor2img uint8, metrics.py psnr) of both outputs against a synthetic ground truth."""
    g = torch.Generator().manual_seed(seed)
    worst = 0.0
    for b in range(out.shape[0]):
        for i in range(out.shape[1]):
            gt = (ref[b, i] + 0.02 * torch.randn(ref[b, i].shape, generator=g)).clamp(0, 1)
            gt8 = O.tensor2img_u8(gt)
            worst = max(worst, abs(O.psnr_u8(O.tensor2img_u8(out[b, i]), gt8)
                                   - O.psnr_u8(O.tensor2img_u8(ref[b, i]), gt8)))
    return worst


def test_generator_matches_oracle_features_and_psnr(dev):
    """C1 shape, both propagation feature stacks + output + PSNR delta against the CPU oracle."""
    sd = weights.random_state_dict(7)
    clip = synthetic.make_config_clip("C1", clip_idx=3, crf=35)
    ref, bwd_ref, fwd_ref = O.generator_forward(sd, *synthetic.generator_args(clip), return_features=True)
    net = build(sd, dev)
    args = [a.to(dev) for a in synthetic.generator_args(clip)]
    out, bwd, fwd = net.forward_with_features(*args)
    out = out.cpu()
    assert (out - ref).abs().max().item() <= TOL
    t = ref.shape[1]
    for i in range(t):
        for got, exp in ((bwd[0, i], bwd_ref[0][i][0]), (fwd[0, i], fwd_ref[0][i][0])):
            got = got.float().permute(2, 0, 1).cpu()
            scale = exp.abs().max().item()
            assert (got - exp).abs().max().item() <= 0.03 * scale + 1e-2
    assert psnr_delta(out, ref) <= 0.02


def test_generator_kitti_shape_edges_and_ipb(dev):
    """C5: 376x1244 (non multiple of the 128-pixel tile), I/P pair, IPB conditioning."""
    sd = weights.random_state_dict(9)
    clip = synthetic.make_config_clip("C5", clip_idx=1, crf=25)
    ref = O.generator_forward(sd, *synthetic.generator_args(clip))
    out = run(build(sd, dev), clip, dev).cpu()
    assert out.shape == ref.shape
    assert (out - ref).abs().max().item() <= TOL
    assert psnr_delta(out, ref) <= 0.02


def test_generator_720p_short_clip(dev):
    """C2/C3 shape, T=3 (I B B -> keys 0 and forced 2), CPU-oracle spot check."""
    sd = weights.random_state_dict(11)
    clip = synthetic.make_config_clip("C3", clip_idx=0, t=3, crf=15)
    ref = O.generator_forward(sd, *synthetic.generator_args(clip))
    out = run(build(sd, dev), clip, dev).cpu()
    assert (out - ref).abs().max().item() <= TOL
    assert psnr_delta(out, ref) <= 0.02


def test_generator_batch_equals_single_clips(dev):
    """n=2 with different slice patterns / CRFs == the two clips run alone (bit identical)."""
    sd = weights.random_state_dict(13)
    a = synthetic.make_clip(64, 96, 5, seed=1, crf=15, pattern="IBBP", ipb=True)
    b = synthetic.make_clip(64, 96, 5, seed=2, crf=35, pattern="allB", ipb=True)
    net = build(sd, dev)
    both = run(net, synthetic.cat_clips([a, b]), dev)
    assert torch.equal(both[0:1], run(net, a, dev))
    assert torch.equal(both[1:2], run(net, b, dev))


def test_generator_batches_identically_conditioned_clips(dev):
    """Clips with the same slice pattern / CRF / QPs share launches (N images per kernel); results must
    equal the clips run alone, and the mixed batch [same, same, different] must split into two runs."""
    sd = weights.random_state_dict(17)
    a = synthetic.make_clip(64, 96, 5, seed=11, crf=25, pattern="IBBP", ipb=True)
    b = synthetic.make_clip(64, 96, 5, seed=12, crf=25, pattern="IBBP", ipb=True)
    c = synthetic.make_clip(64, 96, 5, seed=13, crf=35, pattern="IP", ipb=True)
    net = build(sd, dev)
    single = [run(net, x, dev) for x in (a, b, c)]
    launches_single = net.gpu_launches
    both = run(net, synthetic.cat_clips([a, b, c]), dev)
    assert net.gpu_launches < 3 * launches_single                      # a and b shared their launches
    for k in range(3):
        assert torch.equal(both[k:k + 1], single[k])
    net._engine.batch_clips = False
    unb = run(net, synthetic.cat_clips([a, b, c]), dev)
    assert torch.equal(unb, both)


def test_generator_reflect_padding_and_size_errors(dev):
    sd = weights.random_state_dict(1, num_blocks=2)
    net = build(sd, dev, num_blocks=2)
    clip = synthetic.make_clip(64, 64, 2, seed=1)
    small = {k: (v[..., :60, :60].contiguous() if v.dim() == 5 and v.shape[-1] == 64 else v)
             for k, v in clip.items()}
    with pytest.raises(AssertionError):
        run(net, small, dev)
    clip = synthetic.make_clip(66, 70, 2, seed=1)       # reference raises for non-x4 sizes too
    with pytest.raises(ValueError):
        run(net, clip, dev)
    # C5 contract: lq NOT pre-padded (reflect-padded inside), mvs / partitions zero-padded by caller
    clip = synthetic.make_clip(68, 72, 2, seed=4, pattern="IP")
    lq = clip["lq"][..., :66, :70].contiguous()
    ref = O.generator_forward(sd, lq, *synthetic.generator_args(clip)[1:], num_blocks=2)
    clip2 = dict(clip, lq=lq)
    out = run(net, clip2, dev).cpu()
    assert out.shape[-2:] == (68, 72)
    assert (out - ref).abs().max().item() <= TOL


def test_unsupported_kwargs_raise():
    with pytest.raises(NotImplementedError):
        P.build_backbone(dict(GENERATOR_CFG, with_se=False))
    with pytest.raises(NotImplementedError):
        P.build_backbone(dict(GENERATOR_CFG, blocktype="sft"))


def test_clip_streamer_equals_plain_forward(dev):
    """Host-resident clips through driver.ClipStreamer (chunked H2D in backward-time order, chunked D2H, recycled
    device buffers) give bit-identical frames to the plain call -- the streaming hooks only reorder copies."""
    from pnpvcve_b200 import driver
    sd = weights.random_state_dict(9, num_blocks=2)
    net = build(sd, dev, num_blocks=2)
    clips = [synthetic.make_clip(64, 96, 13, seed=600 + i, crf=(15, 35)[i % 2]) for i in range(3)]
    refs = [run(net, c, dev).cpu() for c in clips]
    hosts = [{k: v.pin_memory() for k, v in c.items()} for c in clips]
    outs = [torch.empty_like(r).pin_memory() for r in refs]
    st = driver.stream_clips(net, hosts, outs, dev, chunk=5)
    torch.cuda.synchronize()
    for o, r in zip(outs, refs):
        assert torch.equal(o, r)
    assert st.h2d_bytes == sum(v.numel() * v.element_size() for v in hosts[0].values())
    assert st.d2h_bytes == refs[0].numel() * 4


def test_clip_streamer_orders_fresh_buffers_behind_pending_work(dev):
    """ClipStreamer takes new device buffers from the caller's stream's pool whenever a clip shape changes (frame
    windows of different lengths), but fills its input buffers on the upload stream and empties its result buffers on
    the download stream.  A block freed by work still queued on one stream must not be written through another before
    that work is done: the upload into fresh input buffers waits for the caller's stream, and a result buffer of another
    shape replaces the old one only behind the old one's download.  Without that order the next clip's inputs can land
    in a block that a queued kernel still writes (seen as frame-window metrics that differ between identical calls).
    A long sleep on one stream makes the order observable."""
    from pnpvcve_b200 import driver
    sd = weights.random_state_dict(9, num_blocks=2)
    net = build(sd, dev, num_blocks=2)
    clips = [synthetic.make_clip(64, 96, t, seed=620 + t) for t in (4, 4, 2)]
    refs = [run(net, c, dev).cpu() for c in clips]
    hosts = [{k: v.pin_memory() for k, v in c.items()} for c in clips]
    outs = [torch.empty_like(r).pin_memory() for r in refs]
    sleep = 10 ** 9                                  # cycles: ~0.5 s, far longer than these clips' launches
    st = driver.ClipStreamer(net, dev, chunk=4)
    main = torch.cuda.current_stream(dev)
    torch.cuda.synchronize()
    torch.cuda._sleep(sleep)
    busy = torch.cuda.Event()
    busy.record(main)
    ticket = st.upload(hosts[0])                     # fresh input buffers
    for ev in ticket["events"].values():
        ev.synchronize()
    assert busy.query(), "the upload into fresh buffers overtook work queued on the caller's stream"
    with torch.cuda.stream(st.down):                 # clip 0's downloads queue up behind a sleep
        torch.cuda._sleep(sleep)
        slow = torch.cuda.Event()
        slow.record(st.down)
    st.run(ticket, outs[0])                          # slot 0
    ticket = st.upload(hosts[1])
    st.run(ticket, outs[1])                          # slot 1
    ticket = st.upload(hosts[2])
    st.run(ticket, outs[2])                          # slot 0 again, T=2: a new result buffer replaces clip 0's
    done = torch.cuda.Event()
    done.record(main)
    done.synchronize()
    assert slow.query(), "a result buffer was replaced before its download had finished"
    st.finish()
    torch.cuda.synchronize()
    for o, r in zip(outs, refs):
        assert torch.equal(o, r)


def test_frame_windows_match_oracle_on_the_same_windows(dev):
    """Frame-window sharding (driver.enhance_windows): every window is a clip of its own -- compared with the oracle run
    on the SAME windows (the reference's max_seq_len semantics); with overlap the kept frames move away from the forced
    key frames and the seam error against the UNCUT clip does not grow."""
    from pnpvcve_b200 import driver
    sd = weights.random_state_dict(21, num_blocks=2)
    net = build(sd, dev, num_blocks=2)
    clip = synthetic.make_clip(64, 96, 11, seed=640, crf=25)
    dclip = {k: v.to(dev) for k, v in clip.items()}
    full, met = driver.enhance_windows(net, [dclip], 4, gather_output=True)
    assert full.shape == (1, 11, 3, 64, 96) and not torch.isnan(full).any() and met.shape == (1, 11, driver.N_METRICS)
    for a, b in driver.frame_windows(11, 4):
        win, _, _ = driver.clip_window(clip, a, b)
        ref = O.generator_forward(sd, *synthetic.generator_args({k: v.contiguous() for k, v in win.items()}), num_blocks=2)
        err = (full[:, a:b].cpu() - ref).abs().max().item()
        assert err <= TOL, f"window [{a},{b}): {err}"
    uncut = O.generator_forward(sd, *synthetic.generator_args(clip), num_blocks=2)
    seam0 = (full.cpu() - uncut).abs().max().item()
    lapped, _ = driver.enhance_windows(net, [dclip], 4, overlap=2, gather_output=True)
    seam2 = (lapped.cpu() - uncut).abs().max().item()
    print(f"seam error vs the uncut clip: {seam0:.3e} without overlap, {seam2:.3e} with 2 frames of overlap")
    assert seam2 <= seam0 + 1e-6
    # host-resident clip: the windows stream through ClipStreamer, same frames
    hosted, met_h = driver.enhance_windows(net, [clip], 4, overlap=2, gather_output=True, device=dev, chunk=3)
    assert torch.equal(hosted, lapped) and met_h.shape == met.shape


def test_enhance_clips_streams_host_clips(dev):
    """driver.enhance_clips on HOST-resident entries (n = 2 clips each) goes through ClipStreamer: same frames as the
    device-resident call, frames delivered to pinned host buffers, metrics gathered for every clip."""
    from pnpvcve_b200 import driver
    sd = weights.random_state_dict(22, num_blocks=2)
    net = build(sd, dev, num_blocks=2)
    entries = [synthetic.cat_clips([synthetic.make_clip(64, 96, 7, seed=700 + 2 * i + j, crf=(15, 35)[j]) for j in range(2)])
               for i in range(3)]
    on_dev = [{k: v.to(dev) for k, v in e.items()} for e in entries]
    outs_d, met_d = driver.enhance_clips(net, on_dev)
    outs_h, met_h = driver.enhance_clips(net, entries, device=dev, chunk=3)
    torch.cuda.synchronize()
    assert met_d.shape == (6, 7, driver.N_METRICS)
    for od, oh in zip(outs_d, outs_h):
        assert oh.is_pinned() and torch.equal(od.cpu(), oh)
    assert torch.equal(met_d, met_h)


def test_profiled_launch_path_equals_fast_path(dev):
    """bench.py's profile pass brackets block launches with events and therefore takes the per-launch descriptor path;
    the default path patches pre-filled descriptors.  Same kernels, same arguments: bit-identical frames."""
    sd = weights.random_state_dict(11, num_blocks=3)
    net = build(sd, dev, num_blocks=3)
    clip = synthetic.make_clip(72, 136, 5, seed=700, crf=25, ipb=True)
    fast = run(net, clip, dev).clone()
    net._engine.prof = {"block_a": [], "block_b": [], "warp": [], "phases": []}
    net._engine.prof_every = 2
    try:
        slow = run(net, clip, dev)
        assert len(net._engine.prof["block_a"]) > 0 and len(net._engine.prof["phases"]) > 0
    finally:
        net._engine.prof = None
    assert torch.equal(fast, slow)


def test_lr_operand_kept_per_frame_equals_recomputed(dev):
    """The LR im2col operand of a frame is written once by the backward-time pass and read again by the forward-time
    pass (engine.lr_once, the default when the pool has room) -- bit-identical to recomputing it in both passes, with
    one launch fewer per forward step, for single clips, batched runs of clips and several runs in one call."""
    sd = weights.random_state_dict(19, num_blocks=2)
    net = build(sd, dev, num_blocks=2)
    a = synthetic.make_clip(72, 136, 6, seed=21, crf=15, pattern="IBBP", ipb=True)
    b = synthetic.make_clip(72, 136, 6, seed=22, crf=35, pattern="IBBP", ipb=True)
    c = synthetic.make_clip(72, 136, 6, seed=23, crf=25, pattern="allB", ipb=True)
    for clip in (a, synthetic.cat_clips([a, b, c])):
        net._engine.lr_once = False
        twice = run(net, clip, dev).clone()
        launches_twice = net.gpu_launches
        net._engine.lr_once = True
        once = run(net, clip, dev)
        assert net._engine.prog.lr_once
        assert net.gpu_launches < launches_twice
        assert torch.equal(once, twice)
