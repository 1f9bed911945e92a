"""The optional generator paths at full size: the x4 tail (`vsr=True`), `sparse_val=True`, the CTA-pair form of the conv
kernel on the whole generator, and the process-wide switches PNP_PAR_SPLIT, PNP_WARP_TMA and PNP_L2_HINTS.

Their kernel code differs from the default path's, so each is held to a plain reference (the fp32 GPU oracle with TF32
off, or float64 conv2d / pixel_shuffle / interpolate) or to bit-identity with the default path.  The library reads the
switches once per process, so every setting runs in a child pytest process of its own.
"""
import contextlib
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

from oracle import bae_oracle as O
from pnpvcve_b200 import _lib, ops, synthetic, weights

from helpers import build_case, golden_cases
from test_gpu_kernels import assert_bf16_close, bf, nchw, nhwc
from test_gpu_parity import TOL, build, run

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    _lib.require_device()
    return torch.device("cuda:0")


@pytest.fixture(autouse=True)
def fp32_oracle():
    """The GPU oracle and the fp64 references must not run in TF32."""
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


@contextlib.contextmanager
def pair_mode(mode):
    """pnp_set_pair_mode(mode) for the duration of a with-block."""
    lib = _lib.load()
    prev = lib.pnp_set_pair_mode(mode)
    try:
        yield
    finally:
        lib.pnp_set_pair_mode(prev)


def per_frame_errors(out, ref, seed=0):
    """(n,T) max-abs and PSNR delta (tensor2img uint8 + psnr of the reference's test loop, against a synthetic ground
    truth near the reference output), computed on the device."""
    n, t = out.shape[:2]
    g = torch.Generator(device=out.device).manual_seed(seed)
    err = (out - ref).abs().amax(dim=(2, 3, 4))
    gt = (ref + 0.02 * torch.randn(ref.shape, generator=g, device=ref.device)).clamp(0, 1)
    q = lambda x: (x.clamp(0, 1) * 255.0).round()       # noqa: E731

    def psnr(a):
        mse = ((q(a) - q(gt)).double() ** 2).mean(dim=(2, 3, 4))
        return 20.0 * torch.log10(255.0 / mse.sqrt())
    return err.cpu(), (psnr(out) - psnr(ref)).abs().cpu()


# ------------------------------------------------------------------ x4 tail kernels at real shapes
@pytest.mark.parametrize("n,h,w", [(1, 180, 320), (1, 360, 640), (2, 96, 312), (1, 64, 64)])
def test_pixel_shuffle_store_at_real_shapes_in_both_conv_forms(dev, n, h, w):
    """PixelShufflePack as four 64->64 launches whose strided stores interleave one 2H x 2W map, at the LR shapes of the
    vsr tail (C4's 180x320 and its 360x640 second stage, C5's 96x312) in pair modes 0, 1 and 2.  180x320, 360x640 and
    64x64 have an odd (image, strip) column count, so mode 2 pairs them with a phantom column.  Catches a pair-form
    strided store that misses the phantom column's neighbour pixels or writes the phantom's results, a strided store
    that drops the last strip's clipped columns, and a form that computes other values than the single-CTA one."""
    assert _lib.load().pnp_device_pairs() >= 8
    g = torch.Generator(device=dev).manual_seed(n * 100000 + h * 1000 + w)
    x = bf(torch.randn((n, 64, h, w), generator=g, device=dev))
    w_up = bf(torch.randn((256, 64, 3, 3), generator=g, device=dev) * 0.05)
    b_up = torch.randn(256, generator=g, device=dev) * 0.1
    ref = F.leaky_relu(F.pixel_shuffle(F.conv2d(x.double(), w_up.double(), b_up.double(), padding=1), 2), 0.1)
    xs = nhwc(x)
    packs = []
    for k in range(4):
        wp = ops.new_wpack_rowstack(dev)
        ops.pack_conv3x3_rowstack(w_up[k::4].contiguous(), wp)
        packs.append(wp)
    outs = []
    for mode in (0, 1, 2):
        up = torch.full((n, 2 * h, 2 * w, 64), float("nan"), dtype=torch.bfloat16, device=dev)
        with pair_mode(mode):
            for k in range(4):
                ops.conv3x3(xs, packs[k], out=up[:, k >> 1::2, k & 1::2, :], bias=b_up[k::4].contiguous(),
                            act=ops.PNP_ACT_LRELU)
            torch.cuda.synchronize()
        assert torch.isfinite(up.float()).all(), f"mode {mode}: {int((~torch.isfinite(up.float())).sum())} values not written"
        got = nchw(up).double()
        assert_bf16_close(got, ref, f"pixel shuffle store, mode {mode}")
        outs.append(up)
    print(f"pixel shuffle {n}x{h}x{w}: max-abs vs fp64 {(nchw(outs[0]).double() - ref).abs().max().item():.2e}")
    for mode in (1, 2):
        assert torch.equal(outs[mode], outs[0]), f"mode {mode}: {int((outs[mode] != outs[0]).sum())} values differ"


@pytest.mark.parametrize("n,hl,wl", [(1, 180, 320), (2, 96, 312)])
def test_conv_last_bilinear_base_at_real_shapes(dev, n, hl, wl):
    """conv_last with the x4 bilinear base of the LR frame computed in its epilogue (lq_up4), at 720x1280 from C4's
    180x320 and 384x1248 from C5's 96x312.  The LR values span [-0.1, 1.1] (the generator's LR input is not clamped),
    so the base is not flat at the borders.  Catches a wrong clamp of the source index at the right and bottom borders
    (i1 = i0 + (i0 < size - 1)), a half-pixel offset error and a pixel left unwritten."""
    g = torch.Generator(device=dev).manual_seed(n * 1000 + hl + wl)
    hh, ww = 4 * hl, 4 * wl
    y = bf(torch.randn((n, 64, hh, ww), generator=g, device=dev))
    wl_ = bf(torch.randn((3, 64, 3, 3), generator=g, device=dev) * 0.05)
    bl = torch.randn(3, generator=g, device=dev) * 0.1
    lr = torch.rand((n, 3, hl, wl), generator=g, device=dev) * 1.2 - 0.1
    wpl = ops.new_wpack_rowstack(dev, tap_n=16)
    ops.pack_conv3x3_rowstack(wl_, wpl, tap_n=16)
    outf = torch.full((n, 3, hh, ww), float("nan"), device=dev)
    ops.conv3x3(nhwc(y), wpl, bias=bl, lq=lr, outf=outf, lq_up4=True)
    base = F.interpolate(lr.double(), scale_factor=4, mode="bilinear", align_corners=False)
    ref = F.conv2d(y.double(), wl_.double(), bl.double(), padding=1) + base
    assert torch.isfinite(outf).all(), "pixels not written"
    err = (outf.double() - ref).abs()
    print(f"conv_last + x4 base {n}x{hh}x{ww}: max-abs vs fp64 {err.max().item():.2e}")
    assert err.max().item() < 1e-4


# ------------------------------------------------------------------ optional generator variants at full size
SPARSE_1X1_GAIN = 500.0


def sparse_state_dict(seed):
    """Random weights whose three partition 1x1 convs are scaled by SPARSE_1X1_GAIN.  At the reference init scale the
    sparse and the dense blend move the output by ~2e-5, far inside TOL, so an oracle check could not tell them apart;
    with the gain they differ by several TOL while the features stay in their usual range."""
    sd = weights.random_state_dict(seed)
    for k in sd:
        if k.endswith(("conv16x16.weight", "conv16x8.weight", "conv8x8.weight")):
            sd[k] = sd[k] * SPARSE_1X1_GAIN
    return sd


def zero_pad_planes(clip, h, w):
    """The C5 contract: lq as it comes, motion vectors and partition maps zero-padded to the x4 size by the caller."""
    for k in ("mvs", "partitions"):
        v = clip[k]
        padded = torch.zeros((*v.shape[:3], h, w))
        padded[..., :v.shape[3], :v.shape[4]] = v
        clip[k] = padded
    return clip


def variant_case(name):
    """(state_dict, clip, generator flags) of a full-size optional-path case."""
    if name == "vsr_c4_n2_180x320_t6":
        clips = [synthetic.make_config_clip("C4", clip_idx=k, t=6, crf=crf) for k, crf in enumerate((15, 35))]
        return weights.random_state_dict(41, vsr=True), synthetic.cat_clips(clips), dict(vsr=True)
    if name == "vsr_c5_94x310_t2_unpadded":
        clip = synthetic.make_clip(94, 310, 2, seed=5042, crf=25, mv_qpel=64, ipb=True, pattern="IP")
        return weights.random_state_dict(42, vsr=True), zero_pad_planes(clip, 96, 312), dict(vsr=True)
    if name == "sparse_c3_720p_t3":
        clip = synthetic.overlap_partitions(synthetic.make_config_clip("C3", clip_idx=7, t=3, crf=25), 3043)
        return sparse_state_dict(43), clip, dict(sparse_val=True)
    if name == "sparse_c5_376x1244_t2":
        clip = synthetic.overlap_partitions(synthetic.make_config_clip("C5", clip_idx=2, crf=35), 5044)
        return sparse_state_dict(44), clip, dict(sparse_val=True)
    raise KeyError(name)


VARIANTS = ["vsr_c4_n2_180x320_t6", "vsr_c5_94x310_t2_unpadded", "sparse_c3_720p_t3", "sparse_c5_376x1244_t2"]


@pytest.mark.parametrize("name", VARIANTS)
def test_optional_variant_matches_gpu_oracle_in_every_launch_form(dev, name):
    """vsr at C4's shape (two 180x320 clips with different CRFs -> 720x1280) and under the C5 contract (94x310 LR,
    reflect-padded inside -> 384x1248), sparse_val at 720p and at 376x1244: per-frame max-abs <= TOL and PSNR delta
    <= 0.02 dB against the fp32 GPU oracle; pair modes 1 and 2 and table mode without graphs are bit-identical to the
    default run; for vsr the uint8 store of conv_last is tensor2img of the fp32 frames.  Catches a vsr tail that is
    wrong only at sizes whose upsampled maps span several strips (odd column counts, the phantom column of pair mode 2),
    a wrong bilinear base under the C5 padding, a sparse blend that keeps the dense sum or the wrong class, and a
    per-image (mixed-CRF) launch that differs between the launch forms."""
    sd, clip, flags = variant_case(name)
    args = [a.to(dev) for a in synthetic.generator_args(clip)]
    with torch.no_grad():
        ref = O.generator_forward(sd, *args, **flags)
    net = build(sd, dev, **flags)
    with torch.no_grad():
        out = net(*args)
    torch.cuda.synchronize()
    assert out.shape == ref.shape
    err, dps = per_frame_errors(out, ref)
    print(f"{name}: max-abs {float(err.max()):.2e} psnr-delta {float(dps.max()):.4f} dB vs the fp32 GPU oracle")
    assert err.max().item() <= TOL
    assert dps.max().item() <= 0.02
    if flags.get("sparse_val"):
        with torch.no_grad():
            dense = O.generator_forward(sd, *args)
        gap = (out - dense).abs().max().item()
        print(f"{name}: max-abs {gap:.2e} vs the dense-blend oracle")
        assert gap > TOL, "the check cannot tell the sparse blend from the dense one on this case"
    del ref
    for mode in (1, 2):
        with pair_mode(mode):
            paired = run(build(sd, dev, **flags), clip, dev)
        assert torch.equal(paired, out), f"pair mode {mode}: {int((paired != out).sum())} values differ"
        del paired
    net._engine.use_graphs = False
    eager = run(net, clip, dev)
    assert net._engine.last_mode == "eager"
    assert torch.equal(eager, out), f"table mode without graphs: {int((eager != out).sum())} values differ"
    if flags.get("vsr"):
        net._engine.use_graphs = True
        u8 = torch.full(out.shape, 3, dtype=torch.uint8, device=dev)
        with torch.no_grad():
            net.forward_streamed(*args, out=u8)
        torch.cuda.synchronize()
        assert torch.equal(u8, O.tensor2img_u8(out))


# ------------------------------------------------------------------ process-wide switches, one child process each
KNOBS = ("PNP_PAR_SPLIT", "PNP_WARP_TMA", "PNP_L2_HINTS", "PNP_PAIR", "PNP_RINGS")
SAVE_ENV = "PNP_TEST_SWITCH_SAVE"          # set by the parent: where the child saves its golden-case outputs
SWITCH_GOLDENS = ["c1_128x128_t7", "n2_64x96_t6_ipb", "sparse_64x64_t3", "edge_68x132_t3"]
_K = "tests/test_gpu_kernels.py::"
_GOLDEN_IDS = [f"tests/test_gpu_parity.py::test_generator_matches_reference_golden[{n}]" for n in SWITCH_GOLDENS]
_PAR_TESTS = [_K + "test_conv_variants_match_fp32_conv2d", _K + "test_conv_par_sparse_selects_last_nonzero_class",
              _K + "test_conv_per_image_weights_equal_separate_launches"]
_WARP_TESTS = [_K + "test_mv_warp_taps_bit_exact_and_values", _K + "test_mv_warp_matches_reference_golden",
               _K + "test_mv_warp_zero_and_integer_flow", _K + "test_mv_warp_per_pixel_flow_takes_the_gather_path"]
_C3 = ["tests/test_gpu_headline.py::test_c3_720p_t12_ipb_crf15"]
#: setting -> (environment, tests the child runs besides the goldens)
SWITCHES = {
    "PNP_PAR_SPLIT=0": (dict(PNP_PAR_SPLIT="0"), _PAR_TESTS),
    "PNP_WARP_TMA=0": (dict(PNP_WARP_TMA="0"), _WARP_TESTS),
    "PNP_L2_HINTS=1": (dict(PNP_L2_HINTS="1"), _C3),
    "PNP_L2_HINTS=2": (dict(PNP_L2_HINTS="2"), _C3),
    "PNP_L2_HINTS=3": (dict(PNP_L2_HINTS="3"), _C3),
}


def golden_case_output(name, dev):
    sd, clip, _ = build_case(name)
    case = golden_cases()[name]
    return run(build(sd, dev, vsr=bool(case.get("vsr")), sparse_val=bool(case.get("sparse_val"))), clip, dev).cpu()


@pytest.mark.skipif(SAVE_ENV not in os.environ, reason="runs in the child process of test_process_wide_switch")
def test_switch_child_saves_golden_outputs(dev):
    """Child side of test_process_wide_switch: the switch golden cases' outputs under this process's switches."""
    torch.save({name: golden_case_output(name, dev) for name in SWITCH_GOLDENS}, os.environ[SAVE_ENV])


@pytest.fixture(scope="module")
def default_golden_outputs(dev):
    return {name: golden_case_output(name, dev) for name in SWITCH_GOLDENS}


@pytest.mark.parametrize("setting", list(SWITCHES))
def test_process_wide_switch(dev, tmp_path, setting, default_golden_outputs):
    """Each switch in a child pytest process: its kernel tests, the generator goldens (and for the L2 hints the 720p
    C3 oracle test) must pass there, and the goldens' outputs must be bit-identical to this process's default run.

    * PNP_PAR_SPLIT=0, the single-role epilogue of block launch A: both epilogues blend the 1x1 results with the same
      fmaf chain, round the blend to bf16 once when they park it in the staging slot, and add it after the same
      scale / bias fmaf, so the switch is held to bit-identity.  Catches a single-role epilogue that drops or misplaces
      the parked blend of a CTA's first or last row, or applies the sparse class selection differently.
    * PNP_WARP_TMA=0, every tap by global gathers (block-constant fields too): same taps and blend as the staged
      path.  Catches a gather path that is wrong at image borders or for block-constant vectors.
    * PNP_L2_HINTS=1/2/3, cache-policy operands on the TMA loads and stores of launches A and B: a hint must not
      change a value.  Catches a hinted load or store with other coordinates than the plain one."""
    if any(k in os.environ for k in KNOBS):
        pytest.skip("this process runs with a switch set: its outputs are not the default path's")
    env_set, tests = SWITCHES[setting]
    saved = tmp_path / "golden_outputs.pt"
    env = {k: v for k, v in os.environ.items() if k not in KNOBS}
    env.update(env_set)
    env[SAVE_ENV] = str(saved)
    cmd = [sys.executable, "-m", "pytest", *tests, *_GOLDEN_IDS,
           "tests/test_optional_paths.py::test_switch_child_saves_golden_outputs", "-x", "-q", "-p", "no:cacheprovider"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
    tail = (res.stdout + res.stderr)[-2000:]
    assert res.returncode == 0, tail
    summary = res.stdout.strip().splitlines()[-1]
    assert " passed" in summary and "skipped" not in summary, tail
    print(f"{setting}: child {summary}")
    child = torch.load(saved)
    for name in SWITCH_GOLDENS:
        a, b = child[name], default_golden_outputs[name]
        assert torch.equal(a, b), f"{setting}, {name}: {int((a != b).sum())} values differ from the default path, " \
                                  f"max {(a - b).abs().max().item():.2e}"
