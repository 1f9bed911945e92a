"""The oracle (oracle/bae_oracle.py) against the reference's golden vectors -- CPU only."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import bae_oracle as O
from oracle import refshim
from pnpvcve_b200 import synthetic, weights

from helpers import build_case, check_against_golden, golden_cases, warp_case

CASES = [c for c in golden_cases() if c != "warp_720p"]


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_reference_golden(name):
    sd, clip, gold = build_case(name)
    case = golden_cases()[name]
    out = O.generator_forward(sd, *synthetic.generator_args(clip), vsr=bool(case.get("vsr")),
                              sparse_val=bool(case.get("sparse_val")))
    err = check_against_golden(out, gold, tol=2e-6, lq=clip["lq"], vsr=bool(case.get("vsr")))
    assert err < 2e-6


def test_oracle_warp_matches_reference_golden():
    x, flow, gold = warp_case()
    y = O.warp_bilinear(x[0], flow[0])
    lat = torch.from_numpy(gold["lattice"])[0]
    assert (y[:, ::8, ::8] - lat).abs().max().item() <= 2e-6
    assert abs(y.double().sum().item() - float(gold["out_sum"])) <= 1e-3


def test_oracle_warp_equals_aten_grid_sample_taps():
    """Tap indices: the restated coordinates floor to the taps ATen's grid_sample uses.

    A plane holding its own linear index is warped with nearest-free bilinear sampling at
    exactly-integer coordinates; any disagreement in floor() would show as a different value.
    """
    h, w = 96, 160
    g = torch.Generator().manual_seed(5)
    flow = torch.randint(-40, 41, (2, h, w), generator=g).float() / 4.0
    x = torch.randn((3, h, w), generator=g)
    gy, gx = torch.meshgrid(torch.arange(h, dtype=torch.float32),
                            torch.arange(w, dtype=torch.float32), indexing="ij")
    nx = 2.0 * (gx + flow[0]) / max(w - 1, 1) - 1.0
    ny = 2.0 * (gy + flow[1]) / max(h - 1, 1) - 1.0
    ref = F.grid_sample(x[None], torch.stack((nx, ny), 2)[None], mode="bilinear",
                        padding_mode="zeros", align_corners=True)[0]
    out = O.warp_bilinear(x, flow)
    assert (out - ref).abs().max().item() <= 1e-6


def test_warp_zero_flow_is_identity_and_integer_flow_is_shift():
    g = torch.Generator().manual_seed(1)
    x = torch.randn((4, 64, 80), generator=g)
    zero = torch.zeros(2, 64, 80)
    assert torch.allclose(O.warp_bilinear(x, zero), x, atol=2e-4)  # fp32 coordinate round trip
    ix, iy = O.warp_taps(zero, 64, 80)
    # NOTE: the fp32 normalise/un-normalise round trip may land a hair below the integer, so the
    # floor can be one less with the weight entirely on the +1 tap; values, not taps, are identity.
    flow = torch.zeros(2, 64, 80)
    flow[0] += 3.0
    flow[1] -= 2.0
    y = O.warp_bilinear(x, flow)
    exp = torch.zeros_like(x)
    exp[:, 2:, : 80 - 3] = x[:, : 64 - 2, 3:]
    assert torch.allclose(y, exp, atol=2e-4)


def test_key_schedule_rules():
    # I B B P B B P B  -> keys at 0,3,6 and forced last (7)
    sl = torch.tensor([73, 66, 66, 80, 66, 66, 80, 66], dtype=torch.float32).view(1, 8, 1, 1, 1)
    key = O.keyframe_mask(sl)[0].tolist()
    assert key == [True, False, False, True, False, False, True, True]
    bwd, fwd = O.key_schedule(key)
    assert bwd == [3, 3, 3, 6, 6, 6, 7, -1]
    assert fwd == [-1, 0, 0, 0, 3, 3, 3, 6]
    allb = O.keyframe_mask(torch.full((1, 4, 1, 1, 1), 66.0))[0].tolist()
    assert allb == [True, False, False, True]
    assert O.key_schedule(allb) == ([3, 3, 3, -1], [-1, 0, 0, 0])


def test_oracle_size_errors_like_reference():
    sd = weights.random_state_dict(0, num_blocks=1)
    clip = synthetic.make_clip(64, 64, 2, seed=1)
    small = {k: (v[..., :60, :60] if v.dim() == 5 and v.shape[-1] == 64 else v)
             for k, v in clip.items()}
    with pytest.raises(AssertionError):
        O.generator_forward(sd, *synthetic.generator_args(small), num_blocks=1)
    clip = synthetic.make_clip(66, 70, 2, seed=1)          # not multiples of 4
    with pytest.raises(ValueError):
        O.generator_forward(sd, *synthetic.generator_args(clip), num_blocks=1)


def test_caa_heads_ranges():
    sd = weights.random_state_dict(0)
    crf = torch.tensor([15, 25, 35], dtype=torch.float32).view(1, 3, 1, 1, 1) / 255.0
    w = O.base_predictor(sd, crf)
    assert w.shape == (1, 3, 6)
    assert torch.allclose(w.sum(-1), torch.ones(1, 3), atol=1e-6)
    g = O.se_module(sd, crf)
    assert g.shape == (1, 3, 64) and g.min() >= 0 and g.max() <= 2.0


@pytest.mark.skipif(not refshim.available(),
                    reason="runs the upstream PnP-VCVE generator from its source tree (PNP_REFERENCE_ROOT), which is not "
                           "part of this repository; its stored outputs of the golden cases are checked by "
                           "test_oracle_matches_reference_golden")
def test_oracle_matches_live_reference():
    net = refshim.build_reference(seed=0)
    sd = net.state_dict()
    assert set(sd) == set(weights.state_dict_shapes())
    assert all(tuple(sd[k].shape) == s for k, s in weights.state_dict_shapes().items())
    clips = [synthetic.make_clip(64, 96, 5, seed=77, crf=15, pattern="IBBP"),
             synthetic.make_clip(64, 96, 5, seed=78, crf=35, pattern="allB", ipb=True)]
    clip = synthetic.cat_clips(clips)
    with torch.no_grad():
        ref = net(*synthetic.generator_args(clip))
    out = O.generator_forward(sd, *synthetic.generator_args(clip))
    assert (ref - out).abs().max().item() <= 1e-6
