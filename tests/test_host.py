"""Host-side logic and the C-ABI surface -- runs without a GPU."""
import ctypes
import os
import re
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import pnpvcve_b200 as P
from oracle import bae_oracle as O
from oracle import refshim
from pnpvcve_b200 import _lib, driver, engine, synthetic, weights

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GEN = "IconVSR_restore_wo_refill_mv_ipb_fast_domain_dynamic_with_par"
CFG = dict(type=GEN, mid_channels=64, num_blocks=8, padding=3, with_cat=True, use_base_qp=True,
           num_experts=6, expert_softmax=True, init_weight=True, with_bias=True, with_se=True,
           with_par=True, one_layer=True, blocktype="drt", channel_first=True, sparse_val=False,
           align_key=True, vsr=False)


# ------------------------------------------------------------------ C ABI
def header_symbols():
    text = open(os.path.join(ROOT, "include", "pnp_vcve.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(pnp_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    import __graft_entry__
    __graft_entry__.build()
    lib = ctypes.CDLL(_lib.LIB_PATH)
    syms = header_symbols()
    assert len(syms) >= 12
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/pnp_vcve.h but not exported"
    assert sorted(_lib.EXPORTS) == syms
    assert _lib.load().pnp_abi_version() == 10


def test_abi_argument_errors_without_gpu():
    lib = _lib.load()
    assert lib.pnp_conv3x3(None, None) == -1                      # PNP_ERR_ARG
    assert b"null" in lib.pnp_last_error()
    assert lib.pnp_mv_warp(None, None, None, 0, 0, None, 1, 4, 4, None, None, None) == -1
    assert lib.pnp_graph_launch(None, None, 0, None) == -1
    assert lib.pnp_set_step(None, 0, None) == -1
    assert lib.pnp_mv_warp_dyn(None, None, 0, 0, 0, 1, 4, 4, None) == -1
    assert lib.pnp_graph_destroy(None) == 0
    if not torch.cuda.is_available():
        assert lib.pnp_device_check() != 0                         # no device: loud failure, no fallback
        with pytest.raises(_lib.PnpError):
            _lib.require_device()


def test_conv_desc_matches_header_layout():
    """ctypes mirror of struct pnp_conv_desc / pnp_dyn_ref (the library static_asserts the same offsets)."""
    d = _lib.ConvDesc()
    assert ctypes.sizeof(d) == 280 and ctypes.sizeof(_lib.DynRef) == 24
    assert _lib.ConvDesc.N.offset == 152 and _lib.ConvDesc.mode.offset == 176 and _lib.ConvDesc.flip_y.offset == 180
    assert _lib.ConvDesc.out_spx.offset == 184 and _lib.ConvDesc.out_sn.offset == 200
    assert _lib.ConvDesc.lq_up4.offset == 208 and _lib.ConvDesc.per_image.offset == 220
    assert _lib.ConvDesc.img_off.offset == 224 and _lib.ConvDesc.dyn.offset == 232
    assert _lib.ConvDesc.src_images.offset == 256 and _lib.ConvDesc.out_images.offset == 268
    assert _lib.DYN_ENTRY_WORDS * 8 == 64


# ------------------------------------------------------------------ registry / boundary
def test_registry_builds_generator_and_state_dict_layout():
    assert GEN in P.BACKBONES
    net = P.build_backbone(CFG)
    sd = net.state_dict()
    shapes = weights.state_dict_shapes()
    assert set(sd) == set(shapes)
    assert all(tuple(sd[k].shape) == shapes[k] for k in shapes)
    assert sum(p.numel() for p in net.parameters()) == 4559885
    assert not list(net.buffers())
    net.load_state_dict(weights.random_state_dict(0), strict=True)
    with pytest.raises(KeyError):
        P.build_backbone(dict(CFG, type="NoSuchBackbone"))
    # vsr=True (x4 tail) is supported: two PixelShufflePack holders with the reference's key names
    vsr_net = P.build_backbone(dict(CFG, vsr=True))
    vsr_shapes = weights.state_dict_shapes(vsr=True)
    assert {k: tuple(v.shape) for k, v in vsr_net.state_dict().items()} == vsr_shapes
    assert set(vsr_shapes) - set(shapes) == {f"upsample{i}.upsample_conv.{p}" for i in (1, 2) for p in ("weight", "bias")}
    for bad in (dict(blocktype="sft"), dict(with_se=False), dict(deform="fvc"),
                dict(one_layer=False), dict(mid_channels=32)):
        with pytest.raises(NotImplementedError):
            P.build_backbone(dict(CFG, **bad))


def test_init_weights_contract(tmp_path):
    net = P.build_backbone(CFG)
    net.init_weights(None)
    with pytest.raises(TypeError):
        net.init_weights(123)
    sd = weights.random_state_dict(5)
    path = str(tmp_path / "ckpt.pth")
    torch.save({"state_dict": {"generator." + k: v for k, v in sd.items()}}, path)
    net.init_weights(path, strict=True)
    assert torch.equal(net.state_dict()["conv_last.weight"], sd["conv_last.weight"])


def test_forward_refuses_cpu_and_training():
    net = P.build_backbone(CFG)
    clip = synthetic.make_clip(64, 64, 2, seed=0)
    with pytest.raises(RuntimeError):
        net(*synthetic.generator_args(clip))                       # training mode + grad
    net.eval()
    with torch.no_grad(), pytest.raises(RuntimeError):
        net(*synthetic.generator_args(clip))                       # CPU tensors: no fallback


def test_config_loader_base_inheritance(tmp_path):
    (tmp_path / "base.py").write_text(
        "model = dict(type='BasicVSR', generator=dict(type='%s', num_blocks=8, vsr=False))\n"
        "data = dict(test=dict(type='A', lq_folder='x'))\n" % GEN)
    (tmp_path / "child.py").write_text(
        "_base_ = './base.py'\nmodel = dict(generator=dict(num_blocks=4))\n"
        "data = dict(test=dict(_delete_=True, type='B'))\n")
    cfg = P.Config.fromfile(str(tmp_path / "child.py"))
    assert cfg.model.generator.type == GEN and cfg.model.generator.num_blocks == 4
    assert cfg.model.generator.vsr is False and cfg.model.type == "BasicVSR"
    assert dict(cfg.data.test) == {"type": "B"}


@pytest.mark.skipif(not refshim.available(),
                    reason="reads the upstream PnP-VCVE config files from its source tree (PNP_REFERENCE_ROOT), which is "
                           "not part of this repository")
@pytest.mark.parametrize("cfgname", ["HR_davis_LR_128x128.py", "HR_davis_LR_128x128_IPB.py",
                                     "HR_davis_LR_128x128_IPB_LR_test.py"])
def test_reference_configs_build_unchanged(cfgname):
    cfg = P.Config.fromfile(os.path.join(refshim.REFERENCE_ROOT, "configs", cfgname))
    net = P.build_backbone(cfg.model.generator)
    assert type(net).__name__ == GEN and net.num_blocks == 8 and net.num_experts == 6


# ------------------------------------------------------------------ schedule
def test_key_schedule_equals_oracle_on_random_patterns():
    g = torch.Generator().manual_seed(0)
    for t in (1, 2, 3, 7, 16, 100):
        for _ in range(5):
            s = torch.tensor([[73, 80, 66][i] for i in torch.randint(0, 3, (t,), generator=g)])
            sl = s.float().view(1, t, 1, 1, 1)
            rows = engine.keyframe_rows(sl.view(1, t).clone())
            assert rows == O.keyframe_mask(sl).tolist()
            if t > 1:
                assert engine.key_schedule(rows[0]) == O.key_schedule(rows[0])


def test_step_variants_and_clip_grouping():
    """Host logic of the launch-free frame loop: which of the six step graphs each frame step replays, and which
    clips of a call share one launch sequence (same key-frame schedule; CRF / QP may differ)."""
    key = [True, False, False, True, False, True]                   # I B B P B (last forced)
    bwd, fwd = engine.key_schedule(key)
    v = engine.step_variants(bwd, fwd)
    assert v[:6] == ["b_last", "b_merged", "b_sep", "b_merged", "b_sep", "b_sep"]      # frames 5,4,3,2,1,0
    assert v[6:] == ["f_first", "f_merged", "f_sep", "f_sep", "f_merged", "f_sep"]     # frames 0..5
    assert engine.step_variants(*engine.key_schedule([True])) == ["b_last", "f_first"]
    a, b, c = [True, False, True], [True, False, True], [True, True, True]
    assert engine.group_clips([a, b, c, c, a], 16) == [(0, 2), (2, 4), (4, 5)]
    assert engine.group_clips([a] * 5, 2) == [(0, 2), (2, 4), (4, 5)]
    assert engine.group_clips([a, b], 16, batch=False) == [(0, 1), (1, 2)]


def test_synthetic_clip_semantics():
    c = synthetic.make_config_clip("C1")
    assert c["lq"].shape == (1, 7, 3, 128, 128) and c["mvs"].shape == (1, 7, 4, 128, 128)
    assert c["slices"].flatten().tolist() == [73, 66, 66, 80, 66, 66, 80]
    assert c["mvs"][0, 0].abs().max() == 0 and c["partitions"][0, 0].abs().max() == 0   # I frame
    p = c["partitions"][0, 1]
    assert torch.unique(p).tolist() == [0.0, torch.tensor(1.0 / 255.0).item()]
    assert torch.allclose(p.sum(0), torch.full((128, 128), 1.0 / 255.0))
    assert torch.equal(c["mvs"][0, 1] * 4, (c["mvs"][0, 1] * 4).round())                # quarter pel
    assert torch.equal(c["mvs"][0, 1, :, :8, :8], c["mvs"][0, 1, :, :1, :1].expand(4, 8, 8))
    c3 = synthetic.make_config_clip("C3", t=4)
    assert torch.equal(c3["QPs"], c3["slices"] / 255.0)
    again = synthetic.make_config_clip("C1")
    assert all(torch.equal(c[k], again[k]) for k in c)


# ------------------------------------------------------------------ multi-process (gloo, world 2)
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, num_clips, t, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    mine = driver.shard_clips(num_clips, rank, world)
    local = torch.stack([torch.full((t, driver.N_METRICS), float(c)) for c in mine], 0) if mine \
        else torch.empty((0, t, driver.N_METRICS))
    full = driver.gather_metrics(local, num_clips, rank, world)
    q.put((rank, full))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("num_clips", [5, 4, 1])
def test_clip_sharding_and_metric_gather_world2(num_clips):
    world, t = 2, 3
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, num_clips, t, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = [q.get(timeout=300) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    exp = torch.arange(num_clips, dtype=torch.float32).view(-1, 1, 1).expand(num_clips, t, driver.N_METRICS)
    for _, full in got:
        assert torch.equal(full, exp)
    assert sorted(driver.shard_clips(5, 0, 2) + driver.shard_clips(5, 1, 2)) == list(range(5))


def _fake_net(lq, *rest):
    """stands in for the generator on the CPU: the result depends on the window's first and last frame, as the real
    one does through the forced key frames"""
    return lq * 2.0 + lq[:, :1] - lq[:, -1:]


def _window_worker(rank, world, port, num_clips, t, window, overlap, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    clips = [synthetic.make_clip(16, 16, t, seed=70 + c) for c in range(num_clips)]
    full, met = driver.enhance_windows(_fake_net, clips, window, rank, world, overlap=overlap, gather_output=True)
    # (numpy: pickled by value -- a torch tensor would travel as a shared-memory handle that dies with this process)
    q.put((rank, full.numpy(), met.numpy(), len(driver.shard_windows(num_clips, t, window, rank, world))))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("num_clips,t,window,overlap", [(1, 11, 4, 0), (2, 10, 5, 0), (1, 9, 3, 1), (1, 5, 8, 0)])
def test_frame_window_sharding_world2(num_clips, t, window, overlap):
    """Frame windows of one (or two) clips dealt to two ranks: every rank ends up with the frames and the metrics of
    ALL windows, each window computed exactly as a clip of its own (the reference's max_seq_len semantics,
    restoration_video_inference.py:121-128), overlap frames computed and dropped."""
    world = 2
    assert driver.frame_windows(11, 4) == [(0, 4), (4, 8), (8, 11)]
    assert driver.balanced_window(100, 8) == 13 and len(driver.frame_windows(100, 13)) == 8
    items = [driver.shard_windows(num_clips, t, window, r, world) for r in range(world)]
    assert sorted(items[0] + items[1]) == [(c, a, b) for c in range(num_clips) for a, b in driver.frame_windows(t, window)]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_window_worker, args=(r, world, port, num_clips, t, window, overlap, q))
             for r in range(world)]
    for p in procs:
        p.start()
    got = [q.get(timeout=300) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    clips = [synthetic.make_clip(16, 16, t, seed=70 + c) for c in range(num_clips)]
    exp = torch.empty((num_clips, t, 3, 16, 16))
    for c in range(num_clips):
        for a, b in driver.frame_windows(t, window):
            a0, b0 = max(0, a - overlap), min(t, b + overlap)
            exp[c, a:b] = _fake_net(clips[c]["lq"][:, a0:b0])[0, a - a0:b - a0]
    for rank, full, met, n_items in got:
        full, met = torch.from_numpy(full), torch.from_numpy(met)
        assert n_items == len(items[rank])
        assert torch.equal(full, exp)
        assert met.shape == (num_clips, t, driver.N_METRICS) and not torch.isnan(met).any()
        assert torch.equal(met[..., 0], exp.abs().amax(dim=(2, 3, 4)))


def test_clip_streamer_chunk_layout():
    """Chunks cover the clip in order; the clip's last frames -- read first by the backward-time pass, delivered last by
    the forward-time pass -- come in short chunks (2, 4, 8, then `chunk` frames)."""
    st = driver.ClipStreamer.__new__(driver.ClipStreamer)
    for t, chunk in ((100, 10), (7, 3), (13, 5), (1, 10), (2, 1), (40, 10)):
        st.chunk = chunk
        ch = st._chunks(t)
        assert ch[0][0] == 0 and ch[-1][1] == t and all(a[1] == b[0] for a, b in zip(ch, ch[1:]))
        assert all(0 < b - a <= max(chunk, 1) for a, b in ch)
        owner = st._chunk_of(ch, t)
        assert all(owner[i][0] <= i < owner[i][1] for i in range(t))
    st.chunk = 10
    assert st._chunks(100)[-3:] == [(86, 94), (94, 98), (98, 100)]


def test_frame_windows_reject_compact_side_information():
    """Windows are cut from dense planes: a clip that carries per-block records instead raises before any work."""
    from pnpvcve_b200 import driver
    clip = synthetic.make_clip(64, 64, 4, seed=1)
    compact = dict({k: v for k, v in clip.items() if k not in ("mvs", "partitions")}, side=[None])
    with pytest.raises(ValueError, match="dense"):
        driver.enhance_windows(_fake_net, [compact], 2)


def test_streamer_cache_is_per_generator_and_dies_with_it(monkeypatch):
    """driver.streamer_for: one ClipStreamer per (generator, device, chunk), kept between enhance_clips calls, released
    with the generator (the streamer itself only holds a weak reference to it) or by release_streamers()."""
    import gc
    import weakref
    from pnpvcve_b200 import driver

    class Net(torch.nn.Module):
        pass

    class Fake(driver.ClipStreamer):
        def __init__(self, net, device, chunk=10):      # no CUDA streams on the CPU box
            self._net = weakref.ref(net)
            self.dev, self.chunk = torch.device(device), int(chunk)

    monkeypatch.setattr(driver, "ClipStreamer", Fake)
    a, b = Net(), Net()
    sa = driver.streamer_for(a, "cpu", 10)
    assert driver.streamer_for(a, "cpu", 10) is sa and sa.net is a
    assert driver.streamer_for(a, "cpu", 5) is not sa and driver.streamer_for(b, "cpu", 10) is not sa
    driver.release_streamers(b)
    assert b not in driver._STREAMERS and a in driver._STREAMERS
    ref = weakref.ref(a)
    del a, sa
    gc.collect()
    assert ref() is None and len(driver._STREAMERS) == 0
