"""s2d_png_decode on the device: every frame equals cv2.imdecode(IMREAD_COLOR) byte for byte (every legal colour type /
bit depth, every filter type, every deflate variant, widths 1-2000, files written by cv2 and PIL), malformed streams get
a status and leave their neighbours and every byte outside their own ranges alone, and load_label_maps / the drop-in
load_masks reproduce the host route."""
import ctypes as C
import io
import os
import warnings
import zlib

import cv2
import numpy as np
import pytest
import torch
from PIL import Image

from s2d_b200 import _lib, png
from tests import png_reference as pr

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0") if torch.cuda.is_available() else None


def _cv2_rgb(data: bytes):
    bgr = cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)
    return cv2.cvtColor(bgr, cv2.COLOR_BGR2RGB)


def _check_all(blobs):
    dec = png.decode_pngs(blobs, DEV)
    assert dec.accepted.all(), dec.status
    for i, b in enumerate(blobs):
        assert np.array_equal(dec.frames[i].cpu().numpy(), _cv2_rgb(b)), i


def _samples(rng, H, W, ct, bd, flat=True):
    hi = 1 << min(bd, 8) if ct == 3 else 1 << bd
    s = rng.integers(0, hi, (H, W, pr.CHANNELS[ct]), dtype=np.uint32)
    if flat:                                                       # label-map-like: flat runs
        s[:, W // 3:] = s[:, W // 3:W // 3 + 1]
    return s


def _pal(rng, bd):
    return rng.integers(0, 256, (1 << min(bd, 8), 3), dtype=np.uint8)


@pytest.mark.parametrize("ct,bd", pr.LEGAL)
def test_every_pair_every_filter_every_width(ct, bd):
    rng = np.random.default_rng(ct * 37 + bd)
    blobs = []
    for W in (1, 2, 3, 7, 31, 32, 33, 100, 333, 2000):
        for filters in ([0], [1], [2], [3], [4], [0, 1, 2, 3, 4]):
            pal = _pal(rng, bd) if ct == 3 else None
            blobs.append(pr.write_png(_samples(rng, 6, W, ct, bd, flat=W > 3), ct, bd, palette=pal, filters=filters))
    _check_all(blobs)


@pytest.mark.parametrize("variant", ["l0", "l1", "l6", "l9", "fixed", "huffman", "rle", "filtered"])
def test_every_deflate_variant(variant):
    rng = np.random.default_rng(len(variant))
    level = {"l0": 0, "l1": 1, "l9": 9}.get(variant, 6)
    strategy = {"fixed": zlib.Z_FIXED, "huffman": zlib.Z_HUFFMAN_ONLY, "rle": zlib.Z_RLE,
                "filtered": zlib.Z_FILTERED}.get(variant, zlib.Z_DEFAULT_STRATEGY)
    blobs = []
    for ct, bd, W, H in ((2, 8, 1280, 30), (3, 8, 640, 40), (6, 16, 500, 12), (0, 1, 2000, 9), (2, 8, 4000, 20)):
        pal = _pal(rng, bd) if ct == 3 else None
        s = _samples(rng, H, W, ct, bd)
        blobs.append(pr.write_png(s, ct, bd, palette=pal, filters=[1, 0, 2, 4, 3], level=level, strategy=strategy))
    # stored blocks of 65535 bytes and distances up to 32768 (a 12 KB row repeated three rows further down)
    s = rng.integers(0, 256, (12, 4000, 3), dtype=np.uint32)
    s[3::3] = s[0]
    blobs.append(pr.write_png(s, 2, 8, filters=[0], level=level, strategy=strategy))
    _check_all(blobs)


def test_cv2_and_pil_files_and_allowed_chunks():
    rng = np.random.default_rng(3)
    lab = np.zeros((72, 128), np.uint8)
    for k in range(1, 12):
        y, x = rng.integers(0, 60), rng.integers(0, 100)
        lab[y:y + rng.integers(5, 30), x:x + rng.integers(5, 60)] = k
    pal = rng.integers(0, 256, (256, 3), dtype=np.uint8)
    pal[0] = 0
    blobs = []
    for params in ([], [cv2.IMWRITE_PNG_COMPRESSION, 0], [cv2.IMWRITE_PNG_COMPRESSION, 9]):
        blobs.append(cv2.imencode(".png", pal[lab][..., ::-1], params)[1].tobytes())
    blobs.append(cv2.imencode(".png", lab * 20)[1].tobytes())                       # gray
    blobs.append(cv2.imencode(".png", (pal[lab].astype(np.uint16) * 257)[..., ::-1])[1].tobytes())   # 16-bit
    blobs.append(cv2.imencode(".png", np.dstack([pal[lab][..., ::-1], lab * 9]))[1].tobytes())       # RGBA
    im = Image.fromarray(lab, "P")
    im.putpalette(pal.tobytes())
    for kw in ({}, {"transparency": 0}, {"transparency": bytes(range(12))}, {"optimize": True}):
        b = io.BytesIO()
        im.save(b, "PNG", **kw)
        blobs.append(b.getvalue())
    b = io.BytesIO()
    Image.fromarray(pal[lab]).save(b, "PNG")
    blobs.append(b.getvalue())
    s = _samples(rng, 20, 50, 2, 8)
    extra = {b"gAMA": b"\0\0\xb1\x8f", b"cHRM": bytes(32), b"sRGB": b"\0", b"pHYs": bytes(9),
             b"tEXt": b"Software\0test", b"zTXt": b"Comment\0\0" + zlib.compress(b"hello"),
             b"iTXt": b"Title\0\0\0\0\0hi", b"tIME": b"\x07\xea\x0a\x15\x0c\0\0", b"bKGD": b"\0\x10\0\x20\0\x30"}
    for t, body in extra.items():
        blobs.append(pr.write_png(s, 2, 8, extra=[(t, body)], filters=[1]))
    blobs.append(pr.write_png(s[..., :1] * 0 + 3, 0, 8, trns=b"\0\3"))                  # gray with tRNS
    blobs.append(pr.write_png(s, 2, 8, trns=b"\0\1\0\2\0\3"))                           # RGB with tRNS
    for b in blobs:
        assert png.parse_png(b) is not None
    _check_all(blobs)


# ---- malformed streams, guard bytes -----------------------------------------------------------------------------

class _BitW:
    def __init__(self):
        self.v, self.n = 0, 0

    def put(self, x, k):
        self.v |= x << self.n
        self.n += k

    def put_code(self, code, k):                                    # Huffman codes go MSB first
        self.put(int(format(code, f"0{k}b")[::-1], 2), k)

    def bytes(self):
        return self.v.to_bytes((self.n + 7) // 8, "little")


def _fixed_stream_with_far_distance():
    """fixed block: literal 0, then a match of 3 at distance 7 (only one byte written so far)"""
    w = _BitW()
    w.put(1, 1); w.put(1, 2)
    w.put_code(0x30, 8)                   # literal 0
    w.put_code(1, 7)                      # 257: length 3
    w.put_code(5, 5); w.put(0, 1)         # distance code 5: 7 + 0
    w.put_code(0, 7)                      # end of block
    return b"\x78\x9c" + w.bytes() + b"\0\0\0\0"


def _launch(items, gap=64):
    """items: (ParsedPng, zdata) -> (status, rgb frames) decoded from one call whose RGB ranges and scanline ranges are
    separated by `gap` guard bytes; asserts that no guard byte changed."""
    ps = [p for p, _ in items]
    zs = [z for _, z in items]
    N = len(ps)
    raw_off, rgb_off, a, b = [], [], gap, gap
    for p in ps:
        raw_off.append(a); a += p.raw_bytes + gap
        rgb_off.append(b); b += p.height * p.width * 3 + gap
    descs = torch.from_numpy(png.pack_descs(ps, raw_off, rgb_off).view(np.uint8).copy()).to(DEV)
    z_off = np.concatenate([[0], np.cumsum([len(z) for z in zs])]).astype(np.int64)
    zdata = torch.from_numpy(np.frombuffer(b"".join(zs) + b"\0", np.uint8).copy()).to(DEV)
    nw = C.c_int64()
    _lib.call("s2d_png_decode_work_ints", N, a, C.byref(nw))
    work = torch.full((nw.value,), 0x5A5A5A5A, dtype=torch.int32, device=DEV)
    rgb = torch.full((b,), 0xA5, dtype=torch.uint8, device=DEV)
    st = torch.full((N,), -7, dtype=torch.int32, device=DEV)
    _lib.call("s2d_png_decode", zdata.data_ptr(), torch.from_numpy(z_off).to(DEV).data_ptr(), descs.data_ptr(), N,
              work.data_ptr(), rgb.data_ptr(), st.data_ptr(), torch.cuda.current_stream(DEV).cuda_stream)
    torch.cuda.synchronize()
    rgb_h = rgb.cpu().numpy()
    scratch = work.cpu().numpy().view(np.uint8)[(N + 3) // 4 * 16:]
    mask_rgb, mask_raw = np.ones(b, bool), np.ones(a, bool)
    for p, o in zip(ps, rgb_off):
        mask_rgb[o:o + p.height * p.width * 3] = False
    for p, o in zip(ps, raw_off):
        mask_raw[o:o + p.raw_bytes] = False
    assert (rgb_h[mask_rgb] == 0xA5).all(), "RGB guard bytes written"
    assert (scratch[:a][mask_raw] == 0x5A).all(), "scanline guard bytes written"
    frames = [rgb_h[o:o + p.height * p.width * 3].reshape(p.height, p.width, 3) for p, o in zip(ps, rgb_off)]
    return st.cpu().numpy(), frames


def test_malformed_streams_are_flagged_and_neighbours_decode():
    rng = np.random.default_rng(8)
    s = _samples(rng, 16, 45, 2, 8)
    good_png = pr.write_png(s, 2, 8, filters=[1, 2, 4])
    good = png.parse_png(good_png)
    raw = pr.filter_rows(pr.pack_rows(s, 2, 8), 3, [1])
    items, want = [], []

    def add(z, bits, p=good):
        items.append((p, z)); want.append(bits)
        items.append((good, good.zdata)); want.append(0)

    z = good.zdata
    for k in range(5):                                              # flipped bits
        zb = bytearray(z)
        i = int(rng.integers(2, len(z) - 4))
        zb[i] ^= 1 << int(rng.integers(0, 8))
        add(bytes(zb), None)
    add(z[:len(z) // 2], None)                                      # truncated
    add(z[:-1], None)
    add(z + b"\0", None)                                            # data after the adler32
    add(_fixed_stream_with_far_distance(), 1)                       # distance before the stream's start
    add(b"\x78\x9c\x07\0\0\0\0\0", 1)                               # block type 3
    bad_f = bytearray(raw); bad_f[(45 * 3 + 1) * 5] = 5             # filter byte 5 in row 5
    add(pr.compress(bytes(bad_f)), 4)
    add(z[:-4] + bytes(4), 8)                                       # wrong adler32
    add(pr.compress(raw + b"\0" * 10), 2)                           # stream longer than the frame
    add(pr.compress(raw[:-(45 * 3 + 1)]), 2)                        # a row short
    stored = pr.compress(raw, 0)
    add(stored[:3] + bytes([stored[3] ^ 1]) + stored[4:], 1)        # stored LEN / NLEN disagree
    pal_png = pr.write_png(rng.integers(0, 4, (6, 9, 1), dtype=np.uint32), 3, 2, palette=_pal(rng, 2)[:3])
    pp = png.parse_png(pal_png)
    add(pp.zdata, 32, pp)                                           # index 3 of a 3-entry palette
    st, frames = _launch(items)
    ref = _cv2_rgb(good_png)
    for (p, _), w, s_, f in zip(items, want, st, frames):
        if w == 0:
            assert s_ == 0 and np.array_equal(f, ref)
        elif w is None:
            assert s_ != 0
        else:
            assert s_ & w, (s_, w)


def test_wrong_descriptor_size_is_flagged():
    rng = np.random.default_rng(2)
    s = _samples(rng, 10, 20, 0, 8)
    p = png.parse_png(pr.write_png(s, 0, 8))
    tall = png.ParsedPng(p.width, p.height + 1, 8, 0, b"", p.zdata)
    short = png.ParsedPng(p.width, p.height - 1, 8, 0, b"", p.zdata)
    wide = png.ParsedPng(20000, 1, 8, 2, b"", p.zdata)
    bad_pair = png.ParsedPng(p.width, p.height, 16, 3, b"\0" * 3, p.zdata)
    st, frames = _launch([(tall, p.zdata), (p, p.zdata), (short, p.zdata), (wide, p.zdata), (bad_pair, p.zdata)])
    assert st[0] & 2 and st[1] == 0 and st[2] & 2 and st[3] == 16 and st[4] == 16
    assert np.array_equal(frames[1], np.repeat(s.astype(np.uint8), 3, axis=2))


def test_graph_capture():
    rng = np.random.default_rng(4)
    blobs = [pr.write_png(_samples(rng, 8, 40, 2, 8), 2, 8, filters=[1]) for _ in range(3)]
    dec = png.decode_pngs(blobs, DEV)
    ps = [png.parse_png(b) for b in blobs]
    N = len(ps)
    raw_off = np.cumsum([0] + [p.raw_bytes for p in ps])
    rgb_off = np.cumsum([0] + [p.height * p.width * 3 for p in ps])
    descs = torch.from_numpy(png.pack_descs(ps, raw_off[:-1], rgb_off[:-1]).view(np.uint8).copy()).to(DEV)
    z_off = torch.from_numpy(np.cumsum([0] + [len(p.zdata) for p in ps]).astype(np.int64)).to(DEV)
    zd = torch.from_numpy(np.frombuffer(b"".join(p.zdata for p in ps), np.uint8).copy()).to(DEV)
    nw = C.c_int64()
    _lib.call("s2d_png_decode_work_ints", N, int(raw_off[-1]), C.byref(nw))
    work = torch.empty(nw.value, dtype=torch.int32, device=DEV)
    rgb = torch.zeros(int(rgb_off[-1]), dtype=torch.uint8, device=DEV)
    st = torch.full((N,), -1, dtype=torch.int32, device=DEV)
    s = torch.cuda.Stream(DEV)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            _lib.call("s2d_png_decode", zd.data_ptr(), z_off.data_ptr(), descs.data_ptr(), N, work.data_ptr(),
                      rgb.data_ptr(), st.data_ptr(), s.cuda_stream)
    g.replay()
    torch.cuda.synchronize()
    assert (st.cpu().numpy() == 0).all()
    assert torch.equal(rgb, torch.cat([f.reshape(-1) for f in dec.frames]))


# ---- end to end --------------------------------------------------------------------------------------------------

def _palette(seed):
    pal = np.random.default_rng(seed).choice(1 << 24, 255, replace=False)
    rgb = np.stack([(pal >> 16) & 255, (pal >> 8) & 255, pal & 255], axis=1).astype(np.uint8)
    return np.concatenate([np.zeros((1, 3), np.uint8), rgb])


def _write_scene(tmp, labels, pal, kind):
    paths = []
    for t, lab in enumerate(labels):
        p = os.path.join(tmp, f"{t:05d}.png")
        if kind == "rgb":
            cv2.imwrite(p, pal[lab][..., ::-1])
        else:
            im = Image.fromarray(lab, "P")
            im.putpalette(pal.tobytes())
            im.save(p)
        paths.append(p)
    return paths


@pytest.mark.parametrize("shape", ["c1", "c2"])
@pytest.mark.parametrize("kind", ["rgb", "palette"])
def test_load_label_maps_synth_scenes(tmp_path, shape, kind):
    from s2d_b200.keymask_ident.crw_utils import rgb_to_label_ids
    from s2d_b200.synth import make_scene_device
    T, H, W, M = {"c1": (24, 480, 854, 10), "c2": (36, 720, 1280, 20)}[shape]
    labels = make_scene_device(2024, T, H, W, M, 64, DEV)["labels"].cpu().numpy()
    pal = _palette(1)
    paths = _write_scene(str(tmp_path), labels, pal, kind)
    got = png.load_label_maps(paths, DEV)
    want = np.stack([rgb_to_label_ids(pal[lab]) for lab in labels])
    assert got.shape == (T, H, W) and got.dtype == torch.uint8
    assert np.array_equal(got.cpu().numpy(), want)
    dec = png.decode_pngs([open(p, "rb").read() for p in paths], DEV)
    assert dec.accepted.all()


def _adam7_png(rgb):
    H, W = rgb.shape[:2]
    raw = b""
    for x0, y0, dx, dy in ((0, 0, 8, 8), (4, 0, 8, 8), (0, 4, 4, 8), (2, 0, 4, 4), (0, 2, 2, 4), (1, 0, 2, 2), (0, 1, 1, 2)):
        sub = rgb[y0::dy, x0::dx]
        if sub.size:
            raw += pr.filter_rows(sub.reshape(sub.shape[0], -1), 3, [0])
    import struct
    return (b"\x89PNG\r\n\x1a\n" + pr.chunk(b"IHDR", struct.pack(">IIBBBBB", W, H, 8, 2, 0, 0, 1)) +
            pr.chunk(b"IDAT", zlib.compress(raw)) + pr.chunk(b"IEND", b""))


def _host_only(monkeypatch, fn, *a):
    with monkeypatch.context() as m:
        m.setattr(torch.cuda, "is_available", lambda: False)
        return fn(*a)


def test_load_masks_mixed_folder_equals_host_route(tmp_path, monkeypatch):
    from s2d_b200.keymask_ident import crw_utils
    rng = np.random.default_rng(6)
    pal = _palette(2)
    lab = rng.integers(0, 6, (5, 48, 64)).astype(np.uint8)
    lab = np.repeat(np.repeat(lab[:, ::4, ::4], 4, axis=1), 4, axis=2)
    d = str(tmp_path)
    _write_scene(d, lab[:3], pal, "rgb")
    with open(os.path.join(d, "00003.png"), "wb") as f:
        f.write(_adam7_png(pal[lab[3]]))
    with open(os.path.join(d, "00004.png"), "wb") as f:
        f.write(b"not a png at all")
    im = Image.fromarray(lab[4], "P"); im.putpalette(pal.tobytes()); im.save(os.path.join(d, "00005.png"))
    with warnings.catch_warnings(record=True) as w_dev:
        warnings.simplefilter("always")
        got = crw_utils.load_masks(d)
    with warnings.catch_warnings(record=True) as w_host:
        warnings.simplefilter("always")
        want = _host_only(monkeypatch, crw_utils.load_masks, d)
    assert got.dtype == want.dtype == torch.int64 and got.shape == want.shape == (5, 48, 64, 1)
    assert torch.equal(got, want)
    assert [str(x.message) for x in w_dev] == [str(x.message) for x in w_host] and len(w_host) == 1
    # mixed shapes keep the host colour -> id route, and raise what it raises
    cv2.imwrite(os.path.join(d, "00006.png"), pal[lab[0, :40]][..., ::-1])
    with pytest.raises(ValueError) as e_dev:
        crw_utils.load_masks(d)
    with pytest.raises(ValueError) as e_host:
        _host_only(monkeypatch, crw_utils.load_masks, d)
    assert str(e_dev.value) == str(e_host.value)
    # no readable frame / empty folder
    e = tmp_path / "bad"
    e.mkdir()
    (e / "a.png").write_bytes(b"\x89PNG garbage")
    with pytest.raises(RuntimeError, match="No valid mask images"):
        crw_utils.load_masks(str(e))
    with pytest.raises(ValueError, match="No .png masks"):
        crw_utils.load_masks(str(tmp_path / "none"))
