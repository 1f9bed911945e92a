"""Drop-in at the RESTORER level: the reference's own ``BasicVSR`` (mmedit/models/restorers/basicvsr.py:155-233,
basic_restorer.py:49,65-98 -- loaded unmodified through oracle/refshim.py) builds the B200 generator from the
shipped config dict through its own registry / builder, loads a ``generator.``-prefixed checkpoint, and routes
``model(test_mode=True, **data)`` positionally into it.  Needs the reference tree (build container only); without a
GPU the call must end in the product's loud no-fallback error, on a GPU it must equal the direct call."""
import os

import pytest
import torch

from oracle import refshim
import pnpvcve_b200 as P
from pnpvcve_b200 import synthetic, weights

pytestmark = pytest.mark.skipif(
    not refshim.available(),
    reason="executes the upstream PnP-VCVE restorer code from its source tree (PNP_REFERENCE_ROOT), which is not part of "
           "this repository")

GENERATOR_CFG = dict(
    type="IconVSR_restore_wo_refill_mv_ipb_fast_domain_dynamic_with_par",
    mid_channels=64, num_blocks=8, padding=3, with_cat=True, use_base_qp=True, num_experts=6,
    expert_softmax=True, init_weight=True, with_bias=True, with_se=True, with_par=True,
    one_layer=True, blocktype="drt", channel_first=True, sparse_val=False, align_key=True, vsr=False)


class _Cfg(dict):
    """test_cfg is an mmcv ConfigDict in the reference: attribute + .get access."""
    __getattr__ = dict.__getitem__


def _build(test_cfg=None, pretrained=None):
    r = refshim.load_restorer()
    # the reference's registry resolves `type` to OUR class: force-registration under the same name, as INTEGRATION.md
    # tells a maintainer to do (mmcv: MODELS.register_module(force=True))
    r["BACKBONES"].register_module(name=GENERATOR_CFG["type"], force=True, module=P.BAEGenerator)
    model_cfg = dict(type="BasicVSR", generator=dict(GENERATOR_CFG),
                     pixel_loss=dict(type="CharbonnierLoss", loss_weight=1.0, reduction="mean"), pretrained=pretrained)
    return r["build_model"](model_cfg, train_cfg=None, test_cfg=test_cfg)


def _data(clip, gt=None):
    d = dict(lq=clip["lq"], QPs=clip["QPs"], slices=clip["slices"], mvs=clip["mvs"], base_QPs=clip["base_QPs"],
             partitions=clip["partitions"])
    if gt is not None:
        d["gt"] = gt
    return d


def test_reference_restorer_builds_loads_and_reaches_the_generator(tmp_path, monkeypatch):
    model = _build()
    assert isinstance(model.generator, P.BAEGenerator)
    # checkpoint layout of tools/test.py: keys prefixed with `generator.` (+ the restorer's own step_counter buffer)
    sd = weights.random_state_dict(3)
    ckpt = {"generator." + k: v for k, v in sd.items()}
    ckpt["step_counter"] = torch.zeros(1)
    missing, unexpected = model.load_state_dict(ckpt, strict=True)
    assert not missing and not unexpected
    for k, v in sd.items():
        assert torch.equal(model.generator.state_dict()[k], v)
    # BasicRestorer.init_weights(pretrained) -> generator.init_weights(str): iconvsr.py:510-523
    path = os.path.join(tmp_path, "ckpt.pth")
    torch.save({"state_dict": ckpt}, path)
    model2 = _build(pretrained=path)
    assert torch.equal(model2.generator.state_dict()["conv_last.weight"], sd["conv_last.weight"])
    with pytest.raises(TypeError):
        model.generator.init_weights(pretrained=3)
    if torch.cuda.is_available():
        pytest.skip("CPU-box half of the test")
    # no GPU here: forward_test must arrive in the generator and fail LOUDLY (no CPU fallback)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    clip = synthetic.make_clip(64, 64, 3, seed=1)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        model(test_mode=True, **_data(clip))


@pytest.mark.gpu
def test_reference_restorer_forward_test_on_gpu():
    """GPU half (runs where both a B200 and the reference tree exist): forward_test == direct generator call, and the
    restorer's evaluate() (reference psnr on tensor2img frames) agrees with pnpvcve_b200.metrics."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    dev = torch.device("cuda:0")
    model = _build(test_cfg=_Cfg(metrics=["PSNR"], crop_border=0))
    sd = weights.random_state_dict(3)
    model.generator.load_state_dict(sd)
    model = model.to(dev).eval()
    clip = {k: v.to(dev) for k, v in synthetic.make_clip(64, 96, 4, seed=2).items()}
    gt = (clip["lq"] * 0.9 + 0.05).contiguous()
    res = model(test_mode=True, **_data(clip, gt))
    with torch.no_grad():
        direct = model.generator(*synthetic.generator_args(clip))
    from pnpvcve_b200 import metrics
    ours = metrics.evaluate(direct, gt, 0, metrics=("PSNR",))["PSNR"].item()
    assert abs(res["eval_result"]["PSNR"] - ours) <= 1e-4
