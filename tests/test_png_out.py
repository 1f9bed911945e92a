"""PNG files of 8-bit frames encoded on the device (pnp_png_*, pngio) and the drivers' ``save_png``.

The oracle is a plain numpy PNG reader: it checks the signature, IHDR, every chunk CRC and IEND, inflates the IDAT data
with zlib (which checks the Adler-32) and undoes all five scanline filters."""
import ctypes
import os
import struct
import zlib

import numpy as np
import pytest
import torch

from pnpvcve_b200 import _lib, driver, pngio, synthetic


# ------------------------------------------------------------------ reader (the oracle) and a reference writer
def _paeth(a, b, c):
    p = a + b - c
    pa, pb, pc = abs(p - a), abs(p - b), abs(p - c)
    return np.where((pa <= pb) & (pa <= pc), a, np.where(pb <= pc, b, c))


def read_png(data):
    """bytes of an 8-bit RGB PNG -> (H, W, 3) uint8; raises ValueError on anything malformed."""
    data = bytes(data)
    if data[:8] != b"\x89PNG\r\n\x1a\n":
        raise ValueError("bad signature")
    pos, chunks = 8, []
    while pos < len(data):
        if pos + 12 > len(data):
            raise ValueError("truncated chunk header")
        n, kind = struct.unpack(">I4s", data[pos:pos + 8])
        if pos + 12 + n > len(data):
            raise ValueError(f"truncated {kind} chunk")
        body = data[pos + 8:pos + 8 + n]
        (crc,) = struct.unpack(">I", data[pos + 8 + n:pos + 12 + n])
        if zlib.crc32(kind + body) != crc:
            raise ValueError(f"bad CRC of a {kind} chunk")
        chunks.append((kind, body))
        pos += 12 + n
    if not chunks or chunks[0][0] != b"IHDR" or chunks[-1] != (b"IEND", b""):
        raise ValueError("IHDR must come first and an empty IEND last")
    w, h, depth, ctype, comp, filt, interlace = struct.unpack(">IIBBBBB", chunks[0][1])
    if (depth, ctype, comp, filt, interlace) != (8, 2, 0, 0, 0):
        raise ValueError("not 8-bit truecolour without interlace")
    kinds = [k for k, _ in chunks[1:-1]]
    if not kinds or set(kinds) != {b"IDAT"}:
        raise ValueError("expected IDAT chunks only between IHDR and IEND")
    try:
        raw = zlib.decompress(b"".join(b for _, b in chunks[1:-1]))
    except zlib.error as e:
        raise ValueError(f"IDAT data: {e}") from None
    stride = 3 * w + 1
    if len(raw) != h * stride:
        raise ValueError("wrong amount of image data")
    rows = np.frombuffer(raw, np.uint8).reshape(h, stride)
    img = np.zeros((h, 3 * w), np.int32)
    prev = np.zeros(3 * w, np.int32)
    for y in range(h):
        ft, x = int(rows[y, 0]), rows[y, 1:].astype(np.int32)
        if ft in (0, 2):
            cur = (x + (prev if ft == 2 else 0)) & 255
        elif ft in (1, 3, 4):                         # these read the reconstructed left neighbour: pixel by pixel
            cur = np.zeros(3 * w, np.int32)
            for i in range(0, 3 * w, 3):
                a = cur[i - 3:i] if i else np.zeros(3, np.int32)
                b = prev[i:i + 3]
                c = prev[i - 3:i] if i else np.zeros(3, np.int32)
                pred = a if ft == 1 else ((a + b) >> 1 if ft == 3 else _paeth(a, b, c))
                cur[i:i + 3] = (x[i:i + 3] + pred) & 255
        else:
            raise ValueError(f"bad filter type {ft}")
        img[y] = cur
        prev = cur
    return img.astype(np.uint8).reshape(h, w, 3)


def write_png(img, filters):
    """reference writer: (H, W, 3) uint8 with filter type filters[y % len(filters)] on row y, zlib.compress"""
    h, w, _ = img.shape
    px = img.reshape(h, 3 * w).astype(np.int32)
    out = []
    for y in range(h):
        ft = filters[y % len(filters)]
        x = px[y]
        b = px[y - 1] if y else np.zeros_like(x)
        a = np.concatenate([np.zeros(3, np.int32), x[:-3]])
        c = np.concatenate([np.zeros(3, np.int32), b[:-3]])
        pred = [0, a, b, (a + b) >> 1, _paeth(a, b, c)][ft]
        out.append(bytes([ft]) + ((x - pred) & 255).astype(np.uint8).tobytes())

    def chunk(kind, body):
        return struct.pack(">I", len(body)) + kind + body + struct.pack(">I", zlib.crc32(kind + body))
    return (b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 8, 2, 0, 0, 0)) +
            chunk(b"IDAT", zlib.compress(b"".join(out), 6)) + chunk(b"IEND", b""))


def row_filters(data):
    """the filter type of every scanline of a PNG file"""
    chunks, pos = [], 8
    while pos < len(data):
        n, kind = struct.unpack(">I4s", data[pos:pos + 8])
        if kind == b"IDAT":
            chunks.append(data[pos + 8:pos + 8 + n])
        pos += 12 + n
    w = struct.unpack(">I", data[16:20])[0]
    return np.frombuffer(zlib.decompress(b"".join(chunks)), np.uint8).reshape(-1, 3 * w + 1)[:, 0]


def libpng_filters(img):
    """per row of an (H, W, 3) image the filter with the smallest sum of |signed byte| (libpng's heuristic, the first
    minimum wins)"""
    h, w, _ = img.shape
    x = img.reshape(h, 3 * w).astype(np.int32)
    b = np.vstack([np.zeros((1, 3 * w), np.int32), x[:-1]])
    a = np.hstack([np.zeros((h, 3), np.int32), x[:, :-3]])
    c = np.hstack([np.zeros((h, 3), np.int32), b[:, :-3]])
    sums = []
    for pred in (0, a, b, (a + b) >> 1, _paeth(a, b, c)):
        v = (x - pred) & 255
        sums.append(np.where(v < 128, v, 256 - v).sum(axis=1))
    return np.argmin(np.stack(sums), axis=0)


def worst_case_bytes(h, w):
    """the size of a file whose every segment is one stored block: signature, IHDR, per segment an IDAT chunk (12
    bytes of framing, 5 bytes of block header, the filtered rows), zlib header and Adler-32, IEND"""
    line = 3 * w + 1
    rows = min(h, max(1, 32768 // line))
    segments = -(-h // rows)
    return 8 + 25 + segments * (12 + 5) + h * line + 2 + 4 + 12


# ------------------------------------------------------------------ CPU
def test_reader_undoes_every_filter_and_rejects_damage():
    g = np.random.default_rng(5)
    img = np.clip(np.cumsum(g.integers(-9, 10, (23, 17, 3)), axis=1) + 128, 0, 255).astype(np.uint8)
    for filters in ([0], [1], [2], [3], [4], [0, 1, 2, 3, 4], [4, 3, 2, 1, 0, 0]):
        assert np.array_equal(read_png(write_png(img, filters)), img), filters
    data = write_png(img, [0, 1, 2, 3, 4])
    idat = data.index(b"IDAT")
    flipped = bytearray(data)
    flipped[idat + 4 + struct.unpack(">I", data[idat - 4:idat])[0] + 1] ^= 0x10     # a byte of the IDAT CRC
    with pytest.raises(ValueError, match="CRC"):
        read_png(flipped)
    with pytest.raises(ValueError):
        read_png(data[:idat + 40])                                                       # truncated IDAT
    n = struct.unpack(">I", data[idat - 4:idat])[0]
    short = bytearray(data[:idat - 4])                                                   # IDAT whose stream stops early
    body = data[idat + 4:idat + 4 + n - 7]
    short += struct.pack(">I", len(body)) + b"IDAT" + body + struct.pack(">I", zlib.crc32(b"IDAT" + body))
    short += data[idat + 8 + n:]
    with pytest.raises(ValueError, match="IDAT"):
        read_png(bytes(short))


def test_png_entry_points_reject_bad_arguments_without_gpu():
    lib = _lib.load()
    p = ctypes.c_void_p(1 << 12)
    bound = lib.pnp_png_frame_bound(64, 64)
    ws = lib.pnp_png_workspace_bytes(2, 64, 64)
    assert ws > 0
    assert lib.pnp_png_encode(None, 0, 0, 0, 1, 64, 64, p, bound, p, p, ws, None) == -1
    assert b"null" in lib.pnp_last_error()
    assert lib.pnp_png_encode(p, 0, 0, 0, 1, 64, 64, p, bound, None, p, ws, None) == -1
    assert b"null" in lib.pnp_last_error()
    for f, h, w in ((0, 64, 64), (1, 0, 64), (1, 64, 0), (1, 4, 21845), (65536, 4, 4)):
        assert lib.pnp_png_encode(p, 0, 0, 0, f, h, w, p, bound, p, p, 1 << 40, None) == -1
        assert b"bad size" in lib.pnp_last_error()
    assert lib.pnp_png_encode(p, 0, 0, 0, 2, 64, 64, p, bound - 1, p, p, ws, None) == -1
    assert b"stride" in lib.pnp_last_error()
    assert lib.pnp_png_encode(p, 0, 0, 0, 2, 64, 64, p, bound, p, p, ws - 1, None) == -1
    assert b"workspace" in lib.pnp_last_error()
    assert lib.pnp_png_frame_bound(0, 5) == -1 and lib.pnp_png_frame_bound(5, 21845) == -1
    assert lib.pnp_png_workspace_bytes(1, 5, 0) == -1
    assert b"bad size" in lib.pnp_last_error()


@pytest.mark.parametrize("h,w", [(1, 1), (5, 1), (40000, 1), (64, 64), (68, 132), (180, 320), (720, 1280),
                                 (2880, 5120), (3, 21844)])
def test_frame_bound_is_the_all_stored_size(h, w):
    assert pngio.frame_bound(h, w) == worst_case_bytes(h, w)


def test_save_png_needs_uint8_frames_and_no_gather():
    clip = synthetic.make_clip(64, 64, 2, seed=1)
    save = lambda c, i: f"/nonexistent/{c}/{i:08d}.png"       # noqa: E731
    with pytest.raises(ValueError, match="uint8"):
        driver.enhance_clips(None, [clip], save_png=save)
    with pytest.raises(ValueError, match="out_hosts"):
        driver.enhance_clips(None, [clip], out_dtype=torch.uint8, save_png=save,
                             out_hosts=[torch.empty((1, 2, 3, 64, 64), dtype=torch.uint8)])
    with pytest.raises(ValueError, match="uint8"):
        driver.enhance_windows(lambda *a: None, [clip], 1, save_png=save)
    with pytest.raises(ValueError, match="gather_output"):
        driver.enhance_windows(lambda *a: None, [clip], 1, out_dtype=torch.uint8, gather_output=True, save_png=save)


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    _lib.require_device()
    return torch.device("cuda:0")


def _decode_all(buf, sizes):
    buf, sizes = buf.cpu(), sizes.cpu().tolist()
    return [bytes(buf[k, :sizes[k]].numpy()) for k in range(len(sizes))]


def _check(frames, files):
    """every file decodes (reader and zlib) to its (3, H, W) frame"""
    frames = frames.cpu().numpy()
    assert len(files) == len(frames)
    for k, data in enumerate(files):
        assert np.array_equal(read_png(data), frames[k].transpose(1, 2, 0)), k


def _contents(kind, f, h, w, dev, seed=0):
    g = torch.Generator(device=dev).manual_seed(seed)
    if kind == "zeros":
        return torch.zeros((f, 3, h, w), dtype=torch.uint8, device=dev)
    if kind == "ones":
        return torch.full((f, 3, h, w), 255, dtype=torch.uint8, device=dev)
    if kind == "noise":
        return torch.randint(0, 256, (f, 3, h, w), generator=g, dtype=torch.uint8, device=dev)
    # gradients: long matches, every filter has something to do
    y = torch.arange(h, device=dev).view(1, 1, h, 1)
    x = torch.arange(w, device=dev).view(1, 1, 1, w)
    c = torch.arange(3, device=dev).view(1, 3, 1, 1)
    k = torch.arange(f, device=dev).view(f, 1, 1, 1)
    return ((x * (c + 1) + y * 2 + k * 37 + (x * y) // 97) % 256).to(torch.uint8)


@pytest.mark.gpu
@pytest.mark.parametrize("h,w", [(64, 64), (68, 132), (180, 320), (376, 1244), (720, 1280)])
@pytest.mark.parametrize("kind", ["zeros", "ones", "gradient", "noise"])
def test_encode_decodes_to_the_frames(dev, h, w, kind):
    f = 3 if h * w > 200000 else 5
    frames = _contents(kind, f, h, w, dev, seed=h + w)
    buf, sizes = pngio.encode(frames)
    files = _decode_all(buf, sizes)
    _check(frames, files)
    bound = pngio.frame_bound(h, w)
    assert buf.shape == (f, bound) and all(len(d) <= bound for d in files)
    for k, data in enumerate(files):         # the filter of every row is libpng's choice
        want = libpng_filters(frames[k].cpu().numpy().transpose(1, 2, 0))
        assert np.array_equal(row_filters(data), want), k
    if kind == "gradient":
        assert len(set(row_filters(files[0]).tolist())) >= 2
    if kind == "noise":                      # nothing to gain: every segment is a stored block
        assert all(len(d) == bound for d in files)
    elif kind in ("zeros", "ones"):
        assert all(len(d) < bound // 20 for d in files)


@pytest.mark.gpu
def test_encode_batches_strided_views_and_is_deterministic(dev):
    h, w = 68, 132
    g = torch.Generator(device=dev).manual_seed(3)
    big = torch.randint(0, 256, (2, 13, 3, h + 4, w + 8), generator=g, dtype=torch.uint8, device=dev)
    big[:, ::2] //= 16                                            # some frames compress, some do not
    for f in range(1, 13):
        view = big[1, :f, :, 2:2 + h, 3:3 + w]                    # a strided (F,3,H,W) view of an (n,T,3,H,W) tensor
        _check(view, _decode_all(*pngio.encode(view)))
    every_other = big[0, 0:12:2, :, 1:1 + h, 5:5 + w]
    _check(every_other, _decode_all(*pngio.encode(every_other)))
    batch = _decode_all(*pngio.encode(big[1, :12, :, 2:2 + h, 3:3 + w]))
    side = torch.cuda.Stream(device=dev)
    for k in (0, 5, 11):
        alone = _decode_all(*pngio.encode(big[1, k:k + 1, :, 2:2 + h, 3:3 + w].contiguous()))
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            other = pngio.encode(big[1, k:k + 1, :, 2:2 + h, 3:3 + w])
        torch.cuda.current_stream().wait_stream(side)
        assert alone[0] == batch[k] == _decode_all(*other)[0], k
    # into a caller's buffer, one frame per row of a wider tensor
    out = torch.zeros((12, pngio.frame_bound(h, w) + 64), dtype=torch.uint8, device=dev)
    sizes = torch.zeros(12, dtype=torch.int64, device=dev)
    pngio.encode(big[1, :12, :, 2:2 + h, 3:3 + w], out=out, sizes=sizes)
    assert _decode_all(out, sizes) == batch


def _net(dev, **kw):
    from test_frames_u8 import _net as net
    return net(dev, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("name,h,w,kw", [("720p", 720, 1280, {}), ("vsr", 180, 320, {"vsr": True})])
def test_encode_generator_output(dev, name, h, w, kw):
    net = _net(dev, **kw)
    clip = synthetic.make_clip(h, w, 3, seed=61)
    with torch.no_grad():
        args = [v.to(dev) for v in synthetic.generator_args(clip)]
        ref = net(*args)
        u8 = torch.empty(ref.shape, dtype=torch.uint8, device=dev)
        net.forward_streamed(*args, out=u8)
    frames = u8[0]
    assert frames.shape[-2:] == (720, 1280)
    buf, sizes = pngio.encode(frames)
    _check(frames, _decode_all(buf, sizes))
    assert int(sizes.max()) <= pngio.frame_bound(720, 1280)


def _files(root):
    found = {}
    for d, _, names in os.walk(root):
        for nm in names:
            found[os.path.relpath(os.path.join(d, nm), root)] = os.path.join(d, nm)
    return found


@pytest.mark.gpu
@pytest.mark.parametrize("feed", ["dense", "side"])
def test_enhance_clips_saves_every_frame_once(dev, feed, tmp_path):
    from oracle import mv_raster_oracle as R
    from test_frames_u8 import to_u8
    from test_sideinfo import _side_entries
    net = _net(dev)
    h, w, t, n = 64, 96, 7, 2
    dense, compact = _side_entries(h, w, t, n, 80, R.rasterize_clip)
    for d, c in zip(dense, compact):
        d["lq"] = c["lq"] = to_u8(d["lq"])
    entries = dense if feed == "dense" else compact
    gts = [torch.randint(0, 256, (n, t, 3, h, w), dtype=torch.uint8).to(dev) for _ in entries]
    want, met = driver.enhance_clips(net, entries, device=dev, chunk=3, out_dtype=torch.uint8, gts=gts)
    calls = []

    def save(c, i):
        calls.append((c, i))
        return str(tmp_path / "host" / f"clip{c:03d}" / f"{i:08d}.png")
    outs, met_png = driver.enhance_clips(net, entries, device=dev, chunk=3, out_dtype=torch.uint8, gts=gts,
                                         save_png=save)
    assert outs == [None] * len(entries)
    assert sorted(calls) == [(c, i) for c in range(len(entries) * n) for i in range(t)]
    assert torch.equal(met_png[..., :3], met[..., :3])
    assert (met_png[..., 3] - met[..., 3]).abs().max().item() <= 1e-7      # (float64 atomics, see test_frames_u8)
    files = _files(tmp_path / "host")
    assert len(files) == len(entries) * n * t
    for e, frames in enumerate(want):
        for j in range(n):
            for i in range(t):
                with open(files[os.path.join(f"clip{e * n + j:03d}", f"{i:08d}.png")], "rb") as fh:
                    assert np.array_equal(read_png(fh.read()), frames[j, i].numpy().transpose(1, 2, 0))
    # device-resident entries: frames returned as before, files written as well
    dev_entries = [{k: v.to(dev) for k, v in e.items()} for e in dense]
    outs_d, _ = driver.enhance_clips(net, dev_entries, out_dtype=torch.uint8,
                                     save_png=lambda c, i: str(tmp_path / "dev" / f"{c}_{i}.png"))
    assert len(_files(tmp_path / "dev")) == len(entries) * n * t
    for e, frames in enumerate(outs_d):
        assert torch.equal(frames.cpu(), want[e])
        with open(tmp_path / "dev" / f"{e * n + 1}_{t - 1}.png", "rb") as fh:
            assert np.array_equal(read_png(fh.read()), want[e][1, t - 1].numpy().transpose(1, 2, 0))


@pytest.mark.gpu
def test_enhance_windows_saves_core_frames_once(dev, tmp_path):
    from test_frames_u8 import to_u8
    net = _net(dev)
    clips = [synthetic.make_clip(64, 96, 9, seed=91 + c) for c in range(2)]
    for clip in clips:
        clip["lq"] = to_u8(clip["lq"])
    frames, met = driver.enhance_windows(net, clips, 4, overlap=1, device=dev, chunk=3, out_dtype=torch.uint8,
                                         gather_output=True)
    calls = []

    def save(c, i):
        calls.append((c, i))
        return str(tmp_path / f"{c}" / f"{i:08d}.png")
    outs, met_png = driver.enhance_windows(net, clips, 4, overlap=1, device=dev, chunk=3, out_dtype=torch.uint8,
                                           save_png=save)
    assert sorted(calls) == [(c, i) for c in range(2) for i in range(9)]
    assert torch.equal(met_png, met)
    assert len(_files(tmp_path)) == 18
    for c in range(2):
        for i in range(9):
            with open(tmp_path / f"{c}" / f"{i:08d}.png", "rb") as fh:
                assert np.array_equal(read_png(fh.read()), frames[c, i].cpu().numpy().transpose(1, 2, 0))
    for (c, a, b), o in outs.items():
        assert torch.equal(o[0], frames[c, a:b])


@pytest.mark.gpu
def test_write_errors_surface_and_the_streamer_recovers(dev, tmp_path):
    from test_frames_u8 import to_u8
    net = _net(dev)
    clip = synthetic.make_clip(64, 96, 5, seed=97)
    clip["lq"] = to_u8(clip["lq"])
    locked = tmp_path / "locked"
    locked.mkdir()
    locked.chmod(0o500)
    bad = locked / "sub"
    if os.access(locked, os.W_OK):             # (a superuser writes anywhere: a regular file as the parent fails too)
        (tmp_path / "file").write_bytes(b"")
        bad = tmp_path / "file"
    try:
        with pytest.raises(OSError):
            driver.enhance_clips(net, [clip], device=dev, chunk=2, out_dtype=torch.uint8,
                                 save_png=lambda c, i: str(bad / f"{i}.png"))
        _, met = driver.enhance_clips(net, [clip], device=dev, chunk=2, out_dtype=torch.uint8,
                                      save_png=lambda c, i: str(tmp_path / "ok" / f"{i}.png"))
        want, met_ref = driver.enhance_clips(net, [clip], device=dev, chunk=2, out_dtype=torch.uint8)
        assert torch.equal(met, met_ref)
        for i in range(5):
            with open(tmp_path / "ok" / f"{i}.png", "rb") as fh:
                assert np.array_equal(read_png(fh.read()), want[0][0, i].numpy().transpose(1, 2, 0))
    finally:
        locked.chmod(0o700)
