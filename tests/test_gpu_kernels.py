"""Kernel-level parity on a real B200, every call going through the C ABI (libpnpvcve.so)."""
import os

import pytest
import torch
import torch.nn.functional as F

from oracle import bae_oracle as O
from pnpvcve_b200 import _lib, ops, weights

from helpers import warp_case

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    _lib.require_device()            # raises if libpnpvcve.so is missing or the device is not sm_100
    return torch.device("cuda:0")


def bf(x):
    return x.to(torch.bfloat16).float()


def nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)


def nchw(x):
    return x.float().permute(0, 3, 1, 2).contiguous()


def assert_bf16_close(got, ref, what, extra=None):
    """within one bf16 rounding step of the fp32 reference result (+ an optional per-element allowance)"""
    tol = ref.abs() * 2.0 ** -7 + 2e-3
    if extra is not None:
        tol = tol + extra
    bad = (got - ref).abs() > tol
    assert not bad.any(), f"{what}: {int(bad.sum())} of {bad.numel()} off, max {float((got - ref).abs().max())}"


# ------------------------------------------------------------------ K1 warp
@pytest.mark.parametrize("h,w,qpel", [(720, 1280, 64), (376, 1244, 64), (180, 320, 32), (64, 64, 200)])
def test_mv_warp_taps_bit_exact_and_values(dev, h, w, qpel):
    g = torch.Generator().manual_seed(h * 7 + w)
    x = bf(torch.randn((64, h, w), generator=g))
    fb = torch.randint(-qpel, qpel + 1, (2, (h + 7) // 8, (w + 7) // 8), generator=g).float() / 4.0
    flow = fb.repeat_interleave(8, 1).repeat_interleave(8, 2)[:, :h, :w].contiguous()
    src = nhwc(x[None]).to(dev)
    dst = ops.new_feature(1, h, w, dev)
    x0, y0 = ops.mv_warp(src, flow.to(dev), dst, debug=True)
    torch.cuda.synchronize()
    ex0, ey0 = O.warp_taps(flow, h, w)                 # CPU oracle: integer taps must be identical
    assert torch.equal(x0.cpu(), ex0), "x tap indices differ from the oracle"
    assert torch.equal(y0.cpu(), ey0), "y tap indices differ from the oracle"
    ref = O.warp_bilinear(x, flow)                     # fp32 CPU oracle on the same bf16-valued input
    assert_bf16_close(nchw(dst)[0].cpu(), ref, "warp values")


def test_mv_warp_matches_reference_golden(dev):
    x, flow, gold = warp_case()                        # reference flow_warp output (fp32 input)
    xb = torch.zeros((1, 64, 720, 1280))
    xb[:, :2] = bf(x)
    dst = ops.new_feature(1, 720, 1280, dev)
    ops.mv_warp(nhwc(xb).to(dev), flow[0].to(dev), dst)
    got = nchw(dst)[0, :2, ::8, ::8].cpu()
    lat = torch.from_numpy(gold["lattice"])[0]
    # input rounded to bf16 (2^-9 relative) and output rounded to bf16: tolerance 2^-6 relative
    assert ((got - lat).abs() <= lat.abs() * 2.0 ** -6 + 4e-2).all()
    assert (got - lat).abs().mean().item() < 6e-3


def test_mv_warp_zero_and_integer_flow(dev):
    g = torch.Generator().manual_seed(3)
    x = bf(torch.randn((1, 64, 72, 136), generator=g))
    src = nhwc(x).to(dev)
    dst = ops.new_feature(1, 72, 136, dev)
    ops.mv_warp(src, torch.zeros((2, 72, 136), device=dev), dst)
    assert_bf16_close(nchw(dst).cpu(), x, "zero flow")
    flow = torch.zeros((2, 72, 136))
    flow[0] += 5.0
    flow[1] -= 3.0
    ops.mv_warp(src, flow.to(dev), dst)
    exp = torch.zeros_like(x)
    exp[:, :, 3:, : 136 - 5] = x[:, :, : 72 - 3, 5:]
    assert_bf16_close(nchw(dst).cpu(), exp, "integer shift")


def test_mv_warp_per_pixel_flow_takes_the_gather_path(dev):
    """A flow field that is NOT block constant (every pixel its own vector, up to +-40 px): the 8 x 8 blocks' taps do not
    fit the staged 10 x 10 windows, so they are read by global gathers -- same taps, same values as the oracle; mixed
    with block-constant regions in one launch, and with n = 2 images."""
    g = torch.Generator().manual_seed(5)
    h, w = 72, 136
    x = bf(torch.randn((2, 64, h, w), generator=g))
    flow = (torch.rand((2, 2, h, w), generator=g) - 0.5) * 80.0
    flow[:, :, :32, :64] = 2.25                                   # a block-constant corner: staged windows
    src = nhwc(x).to(dev)
    dst = ops.new_feature(2, h, w, dev)
    ops.mv_warp(src, flow.to(dev), dst)
    torch.cuda.synchronize()
    for i in range(2):
        ref = O.warp_bilinear(x[i], flow[i])
        assert_bf16_close(nchw(dst[i:i + 1])[0].cpu(), ref, f"image {i}")
        x0, y0 = ops.mv_warp(src[i:i + 1].contiguous(), flow[i].to(dev), ops.new_feature(1, h, w, dev), debug=True)
        ex0, ey0 = O.warp_taps(flow[i], h, w)
        assert torch.equal(x0.cpu(), ex0) and torch.equal(y0.cpu(), ey0)


def test_mv_warp_rejects_bad_arguments(dev):
    a = ops.new_feature(1, 64, 64, dev)
    with pytest.raises(ValueError):
        ops.mv_warp(a, torch.zeros((2, 60, 64), device=dev), ops.new_feature(1, 64, 64, dev))
    with pytest.raises(_lib.PnpError):
        ops.mv_warp(a, torch.zeros((2, 64, 64), device=dev), a)      # aliasing
    with pytest.raises(_lib.PnpError):                               # smaller than one staged tap window
        ops.mv_warp(ops.new_feature(1, 8, 64, dev), torch.zeros((2, 8, 64), device=dev), ops.new_feature(1, 8, 64, dev))


# ------------------------------------------------------------------ conv
# (image, strip) column counts 1, 2, 4, 3, 10, 15: an even count or >= 15 columns takes the CTA-pair (cta_group::2) form
# of the kernel -- 15 with a phantom column in the last pair --, the others the single-CTA form
SHAPES = [(1, 64, 64), (1, 68, 132), (2, 72, 200), (1, 180, 320), (1, 376, 1244), (5, 40, 320)]


def _pack(wt, dev, **kw):
    """Pack a 3x3 conv in the row-stacked weight layout."""
    tap_n = 16 if wt.shape[-4] <= 16 else 64
    wp = ops.new_wpack_rowstack(dev, tap_n=tap_n, with_aux=True)
    ops.pack_conv3x3_rowstack(wt, wp, tap_n=tap_n, **kw)
    return wp


def _pack_par(wt, w1, dev, **kw):
    """Block-launch-A pack: row-stacked 3x3 followed by the three 1x1 partition convs as 192 rows."""
    wpp = ops.new_wpack_rowstack(dev, with_par=True)
    ops.pack_conv3x3_rowstack(wt, wpp, **kw)
    for j in range(3):
        ops.pack_rows(w1[j], wpp[9 * ops.CHUNK_BYTES:], 64 * j)
    return wpp


@pytest.mark.parametrize("n,h,w", SHAPES)
def test_conv_variants_match_fp32_conv2d(dev, n, h, w):
    g = torch.Generator(device=dev).manual_seed(n * 100000 + h * 1000 + w)
    x = bf(torch.randn((n, 64, h, w), generator=g, device=dev))
    wt = bf(torch.randn((64, 64, 3, 3), generator=g, device=dev) * 0.05)
    bias = torch.randn(64, generator=g, device=dev) * 0.1
    scale = torch.rand(64, generator=g, device=dev) + 0.5
    xs = nhwc(x)
    ref0 = F.conv2d(x, wt, padding=1)
    wp = _pack(wt, dev)
    out = ops.new_feature(n, h, w, dev)

    ops.conv3x3(xs, wp, out=out)
    assert_bf16_close(nchw(out), ref0, "plain")
    ops.conv3x3(xs, wp, out=out, bias=bias, act=ops.PNP_ACT_LRELU)
    assert_bf16_close(nchw(out), F.leaky_relu(ref0 + bias.view(1, -1, 1, 1), 0.1), "bias+lrelu")
    idt = bf(torch.randn((n, 64, h, w), generator=g, device=dev))
    ops.conv3x3(xs, wp, out=out, bias=bias, scale=scale, idt=nhwc(idt), act=ops.PNP_ACT_RELU)
    assert_bf16_close(nchw(out), F.relu(ref0 * scale.view(1, -1, 1, 1) + bias.view(1, -1, 1, 1) + idt),
                      "scale+bias+id+relu")

    # LR frame through the im2col'd aux operand == the first 3 input channels of a 131-ch conv
    lr = torch.rand((n, 3, h, w), generator=g, device=dev)
    w_in = bf(torch.randn((64, 131, 3, 3), generator=g, device=dev) * 0.05)
    wpa = _pack(w_in, dev, in_begin=3, in_count=64)
    ops.pack_aux(w_in, wpa[9 * ops.CHUNK_BYTES:])
    lr64 = ops.new_feature(n, h, w, dev, zero=True)
    ops.lr_im2col(lr, lr64)
    ops.conv3x3(xs, wpa, out=out, aux=lr64, bias=bias, act=ops.PNP_ACT_LRELU)
    ref = F.leaky_relu(F.conv2d(torch.cat([bf(lr), x], 1), w_in[:, :67], bias, padding=1), 0.1)
    assert_bf16_close(nchw(out), ref, "aux")

    # merged K slices (neighbour == key_warp): weights of two input slices summed
    wpm = _pack(w_in, dev, in_begin=3, in_begin2=67, in_count=64)
    ops.conv3x3(xs, wpm, out=out)
    assert_bf16_close(nchw(out), F.conv2d(x, bf(w_in[:, 3:67] + w_in[:, 67:131]), padding=1), "merged")

    # 3x3 + three partition-modulated 1x1 convs, general (non one-hot) float partition map
    par = torch.rand((n, 3, h, w), generator=g, device=dev) * \
        (torch.rand((n, 3, h, w), generator=g, device=dev) > 0.5)
    w1 = [bf(torch.randn((64, 64), generator=g, device=dev) * 0.1) for _ in range(3)]
    wpp = _pack_par(wt, w1, dev)
    ops.conv3x3(xs, wpp, out=out, scale=scale, bias=bias, par=par, act=ops.PNP_ACT_RELU)
    ref = ref0 * scale.view(1, -1, 1, 1) + bias.view(1, -1, 1, 1)
    dyres = torch.zeros_like(ref0)
    for j in range(3):
        dyres = dyres + F.conv2d(x, w1[j].view(64, 64, 1, 1)) * par[:, j:j + 1]
    ref = ref + dyres
    # the row-stacked kernel parks the 1x1 blend in bf16 before adding it: one more rounding of that addend
    # (this test's partition values are O(1); the real maps are {0, 1/255}, where it is ~1e-5)
    extra = dyres.abs() * 2.0 ** -8
    assert_bf16_close(nchw(out), F.relu(ref), "par", extra)
    ops.conv3x3(xs, wpp, out=out, bias=bias, par=par, act=ops.PNP_ACT_NONE)
    assert_bf16_close(nchw(out), ref - ref0 * scale.view(1, -1, 1, 1) + ref0, "par without scale", extra)

    # reconstruction tail: 64 -> 3, + lq, fp32 NCHW output
    wl = bf(torch.randn((3, 64, 3, 3), generator=g, device=dev) * 0.05)
    bl = torch.randn(3, generator=g, device=dev) * 0.1
    wpl = _pack(wl, dev)
    outf = torch.empty((n, 3, h, w), device=dev)
    ops.conv3x3(xs, wpl, bias=bl, lq=lr, outf=outf)
    assert (outf - (F.conv2d(x, wl, bl, padding=1) + lr)).abs().max().item() < 1e-4


def test_conv_expert_mixing_matches_reference_formula(dev):
    """pack_conv3x3_rowstack with coef == torch.mm(softmax_attention, weight) of Dynamic_conv2d_se."""
    g = torch.Generator(device=dev).manual_seed(11)
    w = torch.randn((6, 64, 64, 3, 3), generator=g, device=dev) * 0.05
    coef = torch.softmax(torch.randn(6, generator=g, device=dev), 0)
    x = bf(torch.randn((1, 64, 64, 96), generator=g, device=dev))
    wp = ops.new_wpack_rowstack(dev)
    ops.pack_conv3x3_rowstack(w, wp, coef=coef)
    out = ops.new_feature(1, 64, 96, dev)
    ops.conv3x3(nhwc(x), wp, out=out)
    mixed = torch.mm(coef.view(1, 6), w.view(6, -1)).view(64, 64, 3, 3)
    assert_bf16_close(nchw(out), F.conv2d(x, bf(mixed), padding=1), "expert mix")


def test_conv_full_720p_linearity_and_identity(dev):
    """Size-independent properties at the full REDS4 shape: identity kernel and linearity."""
    g = torch.Generator(device=dev).manual_seed(5)
    h, w = 720, 1280
    x = nhwc(bf(torch.randn((1, 64, h, w), generator=g, device=dev)))
    y = nhwc(bf(torch.randn((1, 64, h, w), generator=g, device=dev)))
    eye = torch.zeros((64, 64, 3, 3), device=dev)
    eye[:, :, 1, 1] = torch.eye(64, device=dev)
    wp = _pack(eye, dev)
    out = ops.new_feature(1, h, w, dev)
    ops.conv3x3(x, wp, out=out)
    assert torch.equal(out, x)
    # conv(x) + y through the id operand with the identity kernel == x + y (bf16 rounded once)
    ops.conv3x3(x, wp, out=out, idt=y)
    assert torch.equal(out, (x.float() + y.float()).to(torch.bfloat16))
    # shift kernel: tap (0,2) moves the image one pixel left with zero fill at the right edge
    sh = torch.zeros((64, 64, 3, 3), device=dev)
    sh[:, :, 0, 2] = torch.eye(64, device=dev)
    wp = _pack(sh, dev)
    ops.conv3x3(x, wp, out=out)
    exp = torch.zeros_like(x)
    exp[:, 1:, : w - 1] = x[:, : h - 1, 1:]
    assert torch.equal(out, exp)


def test_conv_rejects_bad_descriptors(dev):
    x = ops.new_feature(1, 64, 64, dev)
    wp = ops.new_wpack_rowstack(dev, with_par=True)
    with pytest.raises(_lib.PnpError):
        ops.conv3x3(x, wp, out=x)                       # out aliases src
    with pytest.raises(ValueError):
        ops.conv3x3(x, wp, out=ops.new_feature(1, 64, 68, dev))
    with pytest.raises(ValueError):
        ops.conv3x3(x.float(), wp, out=ops.new_feature(1, 64, 64, dev))


# ------------------------------------------------------------------ CAA heads
def test_caa_heads_match_oracle(dev):
    sd = weights.random_state_dict(3)
    crf = torch.tensor([15, 25, 35, 25, 51, 0], dtype=torch.float32) / 255.0
    qp = torch.tensor([73, 66, 80, 20, 30, 40], dtype=torch.float32) / 255.0
    params = dict(b0w=sd["BasePredictor.BaseNet.0.weight"], b0b=sd["BasePredictor.BaseNet.0.bias"],
                  b2w=sd["BasePredictor.BaseNet.2.weight"], b2b=sd["BasePredictor.BaseNet.2.bias"],
                  s0w=sd["BiasePredictor.fc.0.weight"], s2w=sd["BiasePredictor.fc.2.weight"])
    params = {k: v.to(dev).contiguous() for k, v in params.items()}
    experts, gamma = ops.caa_heads(crf.to(dev), qp.to(dev), params, 6)
    e_ref = O.base_predictor(sd, crf.view(1, -1, 1, 1, 1))[0]
    g_ref = O.se_module(sd, qp.view(1, -1, 1, 1, 1))[0]
    assert (experts.cpu() - e_ref).abs().max().item() < 1e-6
    assert (gamma.cpu() - g_ref).abs().max().item() < 1e-6
    b2 = torch.randn((4, 6, 64), device=dev)
    tab = ops.mix_bias(b2, experts, gamma)
    ref = torch.einsum("fe,bec->fbc", experts, b2) * gamma[:, None, :]
    assert (tab - ref).abs().max().item() < 1e-5


def test_pack_row_scale_equals_output_gain(dev):
    """SE gain folded at pack time: conv(x, g*W) == g * conv(x, W)  (sr_backbone_utils.py:207-208)."""
    g = torch.Generator(device=dev).manual_seed(21)
    w = bf(torch.randn((64, 64, 3, 3), generator=g, device=dev) * 0.05)
    gain = torch.rand(64, generator=g, device=dev) * 2.0
    x = bf(torch.randn((1, 64, 64, 128), generator=g, device=dev))
    out = ops.new_feature(1, 64, 128, dev)
    wp = ops.new_wpack_rowstack(dev)
    ops.pack_conv3x3_rowstack(w, wp, row_scale=gain)
    ops.conv3x3(nhwc(x), wp, out=out)
    assert_bf16_close(nchw(out), F.conv2d(x, bf(w * gain.view(-1, 1, 1, 1)), padding=1), "row_scale")


@pytest.mark.parametrize("n,h,w", [(1, 68, 132), (2, 72, 200), (1, 376, 1244)])
def test_conv_rowstack_bottom_up_equals_top_down(dev, n, h, w):
    """flip_y + weights packed with mirrored ky: same convolution, rows accumulated in the other order
    (fp32 sums differ in the last bit, so compare against conv2d, not bit for bit)."""
    g = torch.Generator(device=dev).manual_seed(h + w)
    x = nhwc(bf(torch.randn((n, 64, h, w), generator=g, device=dev)))
    idt = nhwc(bf(torch.randn((n, 64, h, w), generator=g, device=dev)))
    wt = bf(torch.randn((64, 64, 3, 3), generator=g, device=dev) * 0.05)
    bias = torch.randn(64, generator=g, device=dev) * 0.1
    down, up = ops.new_wpack_rowstack(dev), ops.new_wpack_rowstack(dev)
    ops.pack_conv3x3_rowstack(wt, down)
    ops.pack_conv3x3_rowstack(wt, up, flip_ky=True)
    a, b = ops.new_feature(n, h, w, dev), ops.new_feature(n, h, w, dev)
    ops.conv3x3(x, down, out=a, idt=idt, bias=bias, act=ops.PNP_ACT_LRELU)
    ops.conv3x3(x, up, out=b, idt=idt, bias=bias, act=ops.PNP_ACT_LRELU, flip_y=True)
    ref = F.leaky_relu(F.conv2d(nchw(x), wt, bias, padding=1) + nchw(idt), 0.1)
    assert_bf16_close(nchw(a), ref, "top-down")
    assert_bf16_close(nchw(b), ref, "bottom-up")
    assert (a.float() - b.float()).abs().max().item() <= 0.07
    # 64 -> 3 tail with fp32 output
    wl = bf(torch.randn((3, 64, 3, 3), generator=g, device=dev) * 0.05)
    lq = torch.rand((n, 3, h, w), generator=g, device=dev)
    d16, u16 = ops.new_wpack_rowstack(dev, tap_n=16), ops.new_wpack_rowstack(dev, tap_n=16)
    ops.pack_conv3x3_rowstack(wl, d16, tap_n=16)
    ops.pack_conv3x3_rowstack(wl, u16, tap_n=16, flip_ky=True)
    o1, o2 = torch.empty((n, 3, h, w), device=dev), torch.empty((n, 3, h, w), device=dev)
    ops.conv3x3(x, d16, lq=lq, outf=o1)
    ops.conv3x3(x, u16, lq=lq, outf=o2, flip_y=True)
    ref = F.conv2d(nchw(x), wl, padding=1) + lq
    assert (o1 - ref).abs().max().item() < 1e-4 and (o2 - ref).abs().max().item() < 1e-4


# ------------------------------------------------------------------ sparse_val partition path
def test_conv_par_sparse_selects_last_nonzero_class(dev):
    """sparse_val eval path (sr_backbone_utils.py:294-302): W_k x / 255 of the LAST class whose map is non-zero,
    whatever the map's value; pixels with all-zero maps get nothing.  1x1 weights are large here so that the
    term is O(1) and a wrong class / a dense blend would be far outside the tolerance."""
    n, h, w = 2, 40, 136
    g = torch.Generator(device=dev).manual_seed(11)
    x = bf(torch.randn((n, 64, h, w), generator=g, device=dev))
    wt = bf(torch.randn((64, 64, 3, 3), generator=g, device=dev) * 0.05)
    w1 = [bf(torch.randn((64, 64), generator=g, device=dev) * 20.0) for _ in range(3)]
    bias = torch.randn(64, generator=g, device=dev) * 0.1
    par = (torch.rand((n, 3, h, w), generator=g, device=dev) > 0.6).float() * \
        torch.randint(1, 4, (n, 3, h, w), generator=g, device=dev).float() / 255.0
    wpp = _pack_par(wt, w1, dev)
    out = ops.new_feature(n, h, w, dev)
    ops.conv3x3(nhwc(x), wpp, out=out, bias=bias, par=par, act=ops.PNP_ACT_NONE, par_sparse=True)
    dy = torch.zeros_like(x)
    for j in range(3):                                   # later classes overwrite earlier ones
        m = (par[:, j:j + 1] != 0)
        dy = torch.where(m, F.conv2d(x, w1[j].view(64, 64, 1, 1)), dy)
    dy = dy / 255
    ref = F.conv2d(x, wt, bias, padding=1) + dy
    assert dy.abs().mean().item() > 0.1                  # the term under test is not negligible
    extra = dy.abs() * 2.0 ** -8
    assert_bf16_close(nchw(out), ref, "par_sparse", extra)
    # and it is NOT what the dense blend gives on these maps
    ops.conv3x3(nhwc(x), wpp, out=out, bias=bias, par=par, act=ops.PNP_ACT_NONE)
    assert (nchw(out) - ref).abs().max().item() > 0.05


# ------------------------------------------------------------------ x4 tail epilogues (vsr=True)
@pytest.mark.parametrize("n,h,w", [(1, 64, 64), (2, 36, 132)])
def test_pixel_shuffle_store_and_bilinear_base_epilogues(dev, n, h, w):
    """PixelShufflePack (common/upsample.py:46-49) as four 64->64 launches with strided stores, and conv_last
    with the x4 bilinear base of the LR frame added in its epilogue (iconvsr_ipb_par.py:139-141)."""
    g = torch.Generator(device=dev).manual_seed(n * 1000 + h + w)
    x = bf(torch.randn((n, 64, h, w), generator=g, device=dev))
    w_up = bf(torch.randn((256, 64, 3, 3), generator=g, device=dev) * 0.05)
    b_up = torch.randn(256, generator=g, device=dev) * 0.1
    up = torch.full((n, 2 * h, 2 * w, 64), float("nan"), dtype=torch.bfloat16, device=dev)
    for k in range(4):
        wp = ops.new_wpack_rowstack(dev)
        ops.pack_conv3x3_rowstack(w_up[k::4].contiguous(), wp)
        ops.conv3x3(nhwc(x), wp, out=up[:, k >> 1::2, k & 1::2, :], bias=b_up[k::4].contiguous(),
                    act=ops.PNP_ACT_LRELU)
    ref = F.leaky_relu(F.pixel_shuffle(F.conv2d(x, w_up, b_up, padding=1), 2), 0.1)
    assert torch.isfinite(up.float()).all(), "pixels not covered by the four strided stores"
    assert_bf16_close(nchw(up), ref, "pixel shuffle store")

    hh, ww = 4 * h, 4 * w
    y = bf(torch.randn((n, 64, hh, ww), generator=g, device=dev))
    wl = bf(torch.randn((3, 64, 3, 3), generator=g, device=dev) * 0.05)
    bl = torch.randn(3, generator=g, device=dev) * 0.1
    lr = torch.rand((n, 3, h, w), generator=g, device=dev)
    wpl = ops.new_wpack_rowstack(dev, tap_n=16)
    ops.pack_conv3x3_rowstack(wl, wpl, tap_n=16)
    outf = torch.empty((n, 3, hh, ww), device=dev)
    ops.conv3x3(nhwc(y), wpl, bias=bl, lq=lr, outf=outf, lq_up4=True)
    base = F.interpolate(lr, scale_factor=4, mode="bilinear", align_corners=False)
    assert (outf - (F.conv2d(y, wl, bl, padding=1) + base)).abs().max().item() < 1e-4


# ------------------------------------------------------------------ per-image weights, batched packer, table mode
def test_pack_mix_blocks_equals_per_block_packers(dev):
    """One launch packs the block-launch-A weights of ALL blocks for one (CRF, QP) condition: byte-identical to
    pack_conv3x3_rowstack(coef, row_scale) + pack_rows per block."""
    g = torch.Generator(device=dev).manual_seed(31)
    nbk, e = 5, 6
    w2 = torch.randn((nbk, e, 64, 64, 3, 3), generator=g, device=dev) * 0.05
    w1 = torch.randn((nbk, 3, 64, 64), generator=g, device=dev) * 0.1
    coef = torch.softmax(torch.randn(e, generator=g, device=dev), 0)
    gain = torch.rand(64, generator=g, device=dev) * 2.0
    dst = torch.zeros((nbk, ops.PACK_A_BYTES), dtype=torch.uint8, device=dev)
    ops.pack_mix_blocks(w2, w1, coef, gain, dst)
    for b in range(nbk):
        ref = _pack_par(w2[b].contiguous(), [w1[b, j] for j in range(3)], dev, coef=coef, row_scale=gain)
        assert torch.equal(dst[b], ref[:ops.PACK_A_BYTES]), f"block {b}"


@pytest.mark.parametrize("n,h,w", [(2, 72, 200), (5, 64, 136), (16, 180, 320)])
def test_conv_per_image_weights_equal_separate_launches(dev, n, h, w):
    """per_image: every image of ONE launch uses its own weights and bias (the reference's groups=batch grouped conv,
    sr_backbone_utils.py:196-204) -- bit-identical to one launch per image."""
    g = torch.Generator(device=dev).manual_seed(n * 7 + h)
    x = nhwc(bf(torch.randn((n, 64, h, w), generator=g, device=dev)))
    par = torch.rand((n, 3, h, w), generator=g, device=dev) * (torch.rand((n, 3, h, w), generator=g, device=dev) > 0.5)
    n_cond = 3
    packs = torch.zeros((n_cond, ops.PACK_A_BYTES), dtype=torch.uint8, device=dev)
    biases = torch.randn((n_cond, 64), generator=g, device=dev) * 0.1
    for c in range(n_cond):
        wt = bf(torch.randn((64, 64, 3, 3), generator=g, device=dev) * 0.05)
        w1 = [bf(torch.randn((64, 64), generator=g, device=dev) * 0.1) for _ in range(3)]
        packs[c] = _pack_par(wt, w1, dev)[:ops.PACK_A_BYTES]
    cond = [(3 * i + 1) % n_cond for i in range(n)]
    off = torch.tensor([[c * ops.PACK_A_BYTES, c * 64] for c in cond], dtype=torch.int64, device=dev)
    out = ops.new_feature(n, h, w, dev)
    ops.conv3x3(x, packs, out=out, bias=biases, par=par, act=ops.PNP_ACT_RELU, img_off=off)
    for i in range(n):
        one = ops.new_feature(1, h, w, dev)
        ops.conv3x3(x[i:i + 1], packs[cond[i]], out=one, bias=biases[cond[i]], par=par[i:i + 1], act=ops.PNP_ACT_RELU)
        assert torch.equal(out[i:i + 1], one), f"image {i}"


@pytest.mark.parametrize("n,h,w,mode", [(1, 68, 132, 1), (2, 72, 200, 1), (1, 376, 1244, 1), (1, 180, 320, 2),
                                        (1, 64, 64, 2), (5, 40, 320, 1), (1, 720, 1280, 1)])
def test_conv_pair_form_is_bit_identical_to_single_cta_form(dev, n, h, w, mode):
    """The CTA-pair form of the conv kernel (cluster of two, tcgen05 cta_group::2, N-split weights, A-collector chains
    for wrapped / clipped accumulator windows; pnp_set_pair_mode) against the single-CTA form: every operand variant,
    even and odd column counts (mode 2: phantom column), per-image weights -- torch.equal."""
    lib = _lib.load()
    assert lib.pnp_device_pairs() >= 8
    g = torch.Generator(device=dev).manual_seed(n * 31 + h + w)
    x = nhwc(bf(torch.randn((n, 64, h, w), generator=g, device=dev)))
    idt = nhwc(bf(torch.randn((n, 64, h, w), generator=g, device=dev)))
    wt = bf(torch.randn((64, 64, 3, 3), generator=g, device=dev) * 0.05)
    bias = torch.randn(64, generator=g, device=dev) * 0.1
    scale = torch.rand(64, generator=g, device=dev) + 0.5
    wp = _pack(wt, dev)
    lr = torch.rand((n, 3, h, w), generator=g, device=dev)
    w_in = bf(torch.randn((64, 131, 3, 3), generator=g, device=dev) * 0.05)
    wpa = _pack(w_in, dev, in_begin=3, in_count=64)
    ops.pack_aux(w_in, wpa[9 * ops.CHUNK_BYTES:])
    lr64 = ops.new_feature(n, h, w, dev, zero=True)
    ops.lr_im2col(lr, lr64)
    par = torch.rand((n, 3, h, w), generator=g, device=dev) * (torch.rand((n, 3, h, w), generator=g, device=dev) > 0.5)
    w1 = [bf(torch.randn((64, 64), generator=g, device=dev) * 0.1) for _ in range(3)]
    wpp = _pack_par(wt, w1, dev)
    wpf = _pack(wt, dev, flip_ky=True)
    packs = torch.stack([_pack_par(bf(torch.randn((64, 64, 3, 3), generator=g, device=dev) * 0.05), w1, dev)[:ops.PACK_A_BYTES]
                         for _ in range(2)], 0)
    off = torch.tensor([[(i % 2) * ops.PACK_A_BYTES, (i % 2) * 64] for i in range(n)], dtype=torch.int64, device=dev)
    biases = torch.randn((2, 64), generator=g, device=dev) * 0.1
    variants = {
        "plain": lambda o: ops.conv3x3(x, wp, out=o),
        "bias+lrelu": lambda o: ops.conv3x3(x, wp, out=o, bias=bias, act=ops.PNP_ACT_LRELU),
        "scale+idt+relu": lambda o: ops.conv3x3(x, wp, out=o, bias=bias, scale=scale, idt=idt, act=ops.PNP_ACT_RELU),
        "idt bottom-up": lambda o: ops.conv3x3(x, wpf, out=o, bias=bias, idt=idt, flip_y=True),
        "aux": lambda o: ops.conv3x3(x, wpa, out=o, aux=lr64, bias=bias, act=ops.PNP_ACT_LRELU),
        "par": lambda o: ops.conv3x3(x, wpp, out=o, bias=bias, par=par, act=ops.PNP_ACT_RELU),
        "par sparse": lambda o: ops.conv3x3(x, wpp, out=o, bias=bias, par=par, act=ops.PNP_ACT_RELU, par_sparse=True),
        "par per image": lambda o: ops.conv3x3(x, packs, out=o, bias=biases, par=par, act=ops.PNP_ACT_RELU, img_off=off),
    }
    prev = lib.pnp_set_pair_mode(0)
    try:
        for name, fn in variants.items():
            lib.pnp_set_pair_mode(0)
            single = ops.new_feature(n, h, w, dev)
            fn(single)
            lib.pnp_set_pair_mode(mode)
            paired = ops.new_feature(n, h, w, dev)
            paired.fill_(7.0)
            fn(paired)
            torch.cuda.synchronize()
            assert torch.equal(single, paired), f"{name}: {int((single != paired).sum())} values differ"
    finally:
        lib.pnp_set_pair_mode(prev)


def test_fetch_pinned_copies_without_the_copy_engine(dev):
    """pnp_fetch_pinned: stream-ordered device copy of a PINNED host buffer by a kernel (the launch table's way up);
    pageable memory and odd sizes are refused."""
    src = torch.arange(3 * 24 * 8, dtype=torch.int64).view(3, 24, 8).pin_memory()
    dst = torch.zeros((3, 24, 8), dtype=torch.int64, device=dev)
    ops.fetch_pinned(dst, src)
    torch.cuda.synchronize()
    assert torch.equal(dst.cpu(), src)
    with pytest.raises(ValueError):
        ops.fetch_pinned(dst, torch.zeros((3, 24, 8), dtype=torch.int64))            # not pinned
    lib = _lib.load()
    assert lib.pnp_fetch_pinned(dst.data_ptr(), src.data_ptr(), 24, None) == -1      # not a multiple of 16 bytes
    pageable = torch.zeros(64, dtype=torch.int64)
    assert lib.pnp_fetch_pinned(dst.data_ptr(), pageable.data_ptr(), 64, None) != 0


def test_conv_720p_survives_a_slow_epilogue(dev, tmp_path, monkeypatch):
    """Regression for the step-barrier ABA (pnp_conv_rows.cu, kStepRing): with 8 step barriers the CTA whose tile range
    ends a few rows into a new column (720p: CTA 102) dead-locked whenever its epilogue fell a full accumulator ring
    behind the MMA thread -- once in ~10^6 launches natively, every time the epilogue warps are slowed but the tensor
    pipe is not.  A diagnostics build of the library (PNP_DIAG, debug bit 2048) delays every epilogue row by ~2 us;
    the 720p conv variants (both kernel forms) must run through with it and stay bit-identical.  That delay does reach
    the full-ring schedule (tools/epilogue_lag.py, profiles/r03_epilogue_lag.log; CTA 0 of a 720p launch, B200 at
    1000 W): when the epilogue takes a row, the issuer has begun 5 steps beyond the one completing it (plain conv; 2 with
    the partition 1x1 convs), i.e. all 8 (5) accumulators are held, against 1 step without the delay."""
    import subprocess
    import sys
    from pnpvcve_b200 import build
    lib = str(tmp_path / "libpnpvcve_diag.so")
    monkeypatch.setenv("PNP_DIAG", "1")
    build.build(force=True, lib=lib)
    env = dict(os.environ, PNP_LIB_PATH=lib, PNP_DEBUG_SKIP="2048")
    cmd = [sys.executable, "-m", "pytest", os.path.abspath(__file__), "-m", "gpu", "-x", "-q", "-p", "no:cacheprovider",
           "-k", "pair_form and 720"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env,
                         cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    tail = (res.stdout + res.stderr)[-1500:]
    assert res.returncode == 0, tail
    assert "1 passed" in res.stdout, tail


def test_table_mode_launches_equal_static_launches(dev):
    """Launch-table mode (operands from a device-resident table selected by a step word) of the warp, the LR im2col and
    the conv, eagerly and replayed from a captured graph: bit-identical to the static launches."""
    import ctypes
    lib = _lib.load()
    g = torch.Generator(device=dev).manual_seed(77)
    n, h, w, frames = 2, 72, 136, 3
    pool = bf(torch.randn((frames * n + 3 * n, h, w, 64), generator=g, device=dev)).to(torch.bfloat16)
    flow = (torch.randint(-32, 33, (frames, n, 2, h, w), generator=g, device=dev).float() / 4.0)
    lr = torch.rand((frames, n, 3, h, w), generator=g, device=dev)
    idt_f, kw_f, out_f = frames * n, frames * n + n, frames * n + 2 * n
    wt = bf(torch.randn((64, 64, 3, 3), generator=g, device=dev) * 0.05)
    wp = _pack(wt, dev)
    bias = torch.randn(64, generator=g, device=dev) * 0.1
    img = h * w * 128
    # expected: static launches per "step" s: warp(frame s -> kw), conv(kw + idt -> out)
    exp = []
    for s in range(frames):
        kw = ops.new_feature(n, h, w, dev)
        ops.mv_warp(pool[s * n:(s + 1) * n], flow[s], kw)
        o = ops.new_feature(n, h, w, dev)
        ops.conv3x3(kw, wp, out=o, idt=pool[idt_f:idt_f + n], bias=bias, act=ops.PNP_ACT_LRELU)
        aux = ops.new_feature(n, h, w, dev, zero=True)
        ops.lr_im2col(lr[s], aux)
        exp.append((o.clone(), aux.clone()))
    stride = 4
    table = torch.zeros((frames, stride, 8), dtype=torch.int64)
    for s in range(frames):
        table[s, 0, :4] = torch.tensor([0, flow[s, 0, 0].data_ptr(), flow[s, 0, 1].data_ptr(), 0])
        table[s, 0, 6] = s * n                   # warp: src image | - << 32
        table[s, 0, 7] = kw_f << 32              #       - | dst image << 32
        table[s, 1, :2] = torch.tensor([wp.data_ptr(), bias.data_ptr()])
        table[s, 1, 6] = kw_f                    # src image | aux image << 32
        table[s, 1, 7] = idt_f | (out_f << 32)   # idt image | out image << 32
    table = table.to(dev)
    step = torch.zeros(1, dtype=torch.int32, device=dev)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def ref(node):
        r = _lib.DynRef()
        r.table, r.step, r.node, r.stride = table.data_ptr(), step.data_ptr(), node, stride
        return r

    r0 = ref(0)
    d = ops.ConvDesc()
    d.src = d.idt = d.out = pool.data_ptr()
    d.src_images = d.idt_images = d.out_images = pool.shape[0]
    d.bias = 1
    d.N, d.H, d.W, d.tap_n, d.act, d.mode, d.wpack_stable = n, h, w, 64, ops.PNP_ACT_LRELU, ops.PNP_CONV_BF16, 1
    d.dyn = ref(1)

    def sequence(st):
        _lib.check(lib.pnp_mv_warp_dyn(ctypes.byref(r0), ctypes.c_void_p(pool.data_ptr()), pool.shape[0], flow.stride(3),
                                       flow.stride(1), n, h, w, st), "warp_dyn")
        _lib.check(lib.pnp_conv3x3(ctypes.byref(d), st), "conv dyn")

    for s in range(frames):                                              # eager table mode
        _lib.check(lib.pnp_set_step(ctypes.c_void_p(step.data_ptr()), s, stream), "set_step")
        sequence(stream)
        assert torch.equal(pool[out_f:out_f + n], exp[s][0]), f"eager step {s}"
    side = torch.cuda.Stream(device=dev)
    cap = ctypes.c_void_p(side.cuda_stream)
    _lib.check(lib.pnp_graph_begin(cap), "graph_begin")
    sequence(cap)
    handle = ctypes.c_void_p()
    _lib.check(lib.pnp_graph_end(cap, ctypes.byref(handle)), "graph_end")
    for s in reversed(range(frames)):                                    # graph replay, any step order
        pool[out_f:out_f + n].zero_()
        _lib.check(lib.pnp_graph_launch(handle, ctypes.c_void_p(step.data_ptr()), s, stream), "graph_launch")
        assert torch.equal(pool[out_f:out_f + n], exp[s][0]), f"graph step {s}"
    _lib.check(lib.pnp_graph_destroy(handle), "graph_destroy")
    # LR im2col in table mode
    t2 = torch.zeros((frames, 1, 8), dtype=torch.int64)
    aux = ops.new_feature(n, h, w, dev, zero=True)
    for s in range(frames):
        t2[s, 0, 0], t2[s, 0, 1] = lr[s].data_ptr(), aux.data_ptr()
    t2 = t2.to(dev)
    r2 = _lib.DynRef()
    r2.table, r2.step, r2.node, r2.stride = t2.data_ptr(), step.data_ptr(), 0, 1
    for s in range(frames):
        _lib.check(lib.pnp_set_step(ctypes.c_void_p(step.data_ptr()), s, stream), "set_step")
        _lib.check(lib.pnp_lr_im2col_dyn(ctypes.byref(r2), lr.stride(1), lr.stride(2), lr.stride(3), n, h, w, 64, stream),
                   "im2col_dyn")
        assert torch.equal(aux, exp[s][1]), f"im2col step {s}"


@pytest.mark.parametrize("n,h,w", [(1, 64, 64), (2, 72, 200), (1, 180, 320), (1, 376, 1244), (1, 720, 1280)])
def test_compact_lr_operand_is_bit_identical(dev, n, h, w):
    """The LR im2col operand as a (N,H,W,32) tensor of 64-byte pixels (what the engine uses: contiguous stores, half the
    bytes, read by the conv through a SWIZZLE_64B tile and a 64B-swizzle A descriptor) against the (N,H,W,64) form whose
    upper 32 channels are dead: same operand values, bit-identical conv results -- also next to an identity operand."""
    g = torch.Generator(device=dev).manual_seed(h * 7 + w)
    lr = torch.rand((n, 3, h, w), generator=g, device=dev)
    x = nhwc(bf(torch.randn((n, 64, h, w), generator=g, device=dev)))
    w_in = bf(torch.randn((64, 131, 3, 3), generator=g, device=dev) * 0.05)
    bias = torch.randn(64, generator=g, device=dev) * 0.1
    wpa = _pack(w_in, dev, in_begin=3, in_count=64)
    ops.pack_aux(w_in, wpa[9 * ops.CHUNK_BYTES:])
    lr64 = ops.new_feature(n, h, w, dev, zero=True)
    lr32 = torch.full((n, h, w, 32), float("nan"), dtype=torch.bfloat16, device=dev)
    ops.lr_im2col(lr, lr64)
    ops.lr_im2col(lr, lr32)
    assert torch.equal(lr32, lr64[..., :32])
    a = ops.new_feature(n, h, w, dev)
    b = ops.new_feature(n, h, w, dev)
    ops.conv3x3(x, wpa, out=a, aux=lr64, bias=bias, act=ops.PNP_ACT_LRELU)
    ops.conv3x3(x, wpa, out=b, aux=lr32, bias=bias, act=ops.PNP_ACT_LRELU)
    assert torch.equal(a, b)
    lib = _lib.load()
    prev = lib.pnp_set_pair_mode(1)          # (the compact operand always takes the single-CTA form)
    try:
        ops.conv3x3(x, wpa, out=b, aux=lr32, bias=bias, act=ops.PNP_ACT_LRELU)
    finally:
        lib.pnp_set_pair_mode(prev)
    assert torch.equal(a, b)
