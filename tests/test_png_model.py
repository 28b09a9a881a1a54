"""Host models of the PNG decoder (no GPU): the inflate kernel's Huffman tables, the unfilter kernel's decomposition of
the row filters, the RGB conversion rules against cv2 itself, and s2d_b200.png.parse_png."""
import io
import struct
import zlib

import cv2
import numpy as np
import pytest
from PIL import Image

from s2d_b200.png import parse_png
from tests import png_reference as pr


def _corpus_bytes(rng, n):
    """label-map-like bytes: long flat runs, a few noisy stretches, repeats far back"""
    parts = []
    while sum(map(len, parts)) < n:
        k = int(rng.integers(0, 4))
        m = int(rng.integers(1, 3000))
        if k == 0:
            parts.append(bytes([int(rng.integers(0, 256))]) * m)
        elif k == 1:
            parts.append(rng.integers(0, 256, m, dtype=np.uint8).tobytes())
        elif k == 2 and parts:
            parts.append(parts[int(rng.integers(0, len(parts)))][:m])
        else:
            parts.append(bytes(rng.integers(0, 8, m, dtype=np.uint8)))
    return b"".join(parts)[:n]


@pytest.mark.parametrize("level", list(range(10)))
def test_inflate_model_levels(level):
    raw = _corpus_bytes(np.random.default_rng(level), 60000)
    assert pr.inflate_model(pr.compress(raw, level)) == raw


@pytest.mark.parametrize("strategy", [zlib.Z_FIXED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FILTERED])
def test_inflate_model_strategies(strategy):
    raw = _corpus_bytes(np.random.default_rng(strategy + 20), 60000)
    assert pr.inflate_model(pr.compress(raw, 6, strategy)) == raw


def test_inflate_model_stored_blocks_of_65535_bytes():
    raw = np.random.default_rng(3).integers(0, 256, 3 * 65535 + 17, dtype=np.uint8).tobytes()
    z = pr.compress(raw, 0)
    assert z[2] & 6 == 0 and struct.unpack_from("<H", z, 3)[0] == 65535
    assert pr.inflate_model(z) == raw


def test_inflate_model_distances_up_to_32768():
    rng = np.random.default_rng(4)
    block = rng.integers(0, 256, 32768, dtype=np.uint8).tobytes()
    raw = block + block[:5000] + rng.integers(0, 256, 100, dtype=np.uint8).tobytes() + block[-300:]
    z = pr.compress(raw, 9)
    assert pr.inflate_model(z) == raw


def test_table_model_long_codes_use_sub_tables():
    """a skewed alphabet: codes of 10-15 bits, reached through the sub-tables; all tables within zlib's ENOUGH"""
    rng = np.random.default_rng(5)
    p = 0.5 ** np.arange(1, 40)
    syms = rng.choice(np.arange(39), size=200000, p=p / p.sum())
    raw = (syms * 6 + 1).astype(np.uint8).tobytes()
    z = pr.compress(raw, 9, zlib.Z_HUFFMAN_ONLY)
    assert pr.inflate_model(z) == raw
    lens = [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 15]
    tab, used = pr.build_table(lens + [0] * 270, 9, 852)
    assert used > 512 and used <= 852
    assert pr.build_table([1, 1, 1], 9, 852) is None                 # oversubscribed
    assert pr.build_table([2, 2, 2], 9, 852) is None                 # incomplete
    assert pr.build_table([1, 0, 0], 6, 592) is not None             # one code of length 1: allowed


@pytest.mark.parametrize("bpp", [1, 2, 3, 4, 6, 8])
def test_unfilter_model_matches_per_byte_loop(bpp):
    rng = np.random.default_rng(bpp)
    for rb in (bpp, 31, 32, 33, 97, 130):
        rb = max(rb - rb % bpp, bpp)
        H = 10
        rows = rng.integers(0, 256, (H, rb), dtype=np.uint8)
        rows[3] = rows[2]
        raw = pr.filter_rows(rows, bpp, [0, 1, 2, 3, 4, 1, 1, 3, 4, 2])
        want = pr.unfilter_reference(raw, H, rb, bpp)
        assert np.array_equal(want, rows)
        assert np.array_equal(pr.unfilter_model(raw, H, rb, bpp), want)


def _samples(rng, H, W, ct, bd, pal_n=None):
    hi = (1 << bd) - 1 if ct != 3 else (pal_n or (1 << bd)) - 1
    return rng.integers(0, hi + 1, (H, W, pr.CHANNELS[ct]), dtype=np.uint32)


@pytest.mark.parametrize("ct,bd", pr.LEGAL)
def test_conversion_rules_match_cv2(ct, bd):
    """The reference conversion the kernel implements equals cv2.imdecode(IMREAD_COLOR) for every legal pair."""
    rng = np.random.default_rng(ct * 100 + bd)
    H, W = 7, 37
    pal = rng.integers(0, 256, (1 << min(bd, 8), 3), dtype=np.uint8) if ct == 3 else None
    s = _samples(rng, H, W, ct, bd)
    png = pr.write_png(s, ct, bd, palette=pal, filters=[0, 1, 2, 3, 4])
    got = cv2.cvtColor(cv2.imdecode(np.frombuffer(png, np.uint8), cv2.IMREAD_COLOR), cv2.COLOR_BGR2RGB)
    assert np.array_equal(pr.to_rgb_reference(pr.pack_rows(s, ct, bd), W, ct, bd, pal), got)
    p = parse_png(png)
    assert p is not None and (p.width, p.height, p.bit_depth, p.color_type) == (W, H, bd, ct)
    assert zlib.decompress(p.zdata) == pr.filter_rows(pr.pack_rows(s, ct, bd), max(1, pr.CHANNELS[ct] * bd // 8),
                                                      [0, 1, 2, 3, 4])


def _rgb_png():
    rng = np.random.default_rng(9)
    return pr.write_png(_samples(rng, 20, 33, 2, 8), 2, 8, filters=[1])


def test_parse_png_idat_in_one_byte_chunks():
    rng = np.random.default_rng(10)
    s = _samples(rng, 20, 33, 2, 8)
    a, b = parse_png(pr.write_png(s, 2, 8)), parse_png(pr.write_png(s, 2, 8, idat_split=1))
    assert a is not None and b is not None and a.zdata == b.zdata


def test_parse_png_rejects():
    png = _rgb_png()
    assert parse_png(png) is not None
    bad = bytearray(png)
    bad[40] ^= 1                                                      # inside IDAT: its CRC no longer matches
    assert parse_png(bytes(bad)) is None
    for cut in (7, 20, 33, 50, len(png) - 1, len(png) - 12):
        assert parse_png(png[:cut]) is None
    assert parse_png(png + b"\x00") is None
    assert parse_png(b"GIF89a" + png[6:]) is None
    ihdr = struct.pack(">IIBBBBB", 33, 20, 8, 2, 0, 0, 1)             # Adam7
    assert parse_png(png[:8] + pr.chunk(b"IHDR", ihdr) + png[33:]) is None
    for t in (b"acTL", b"eXIf", b"sPLT", b"abCd", b"iCCP"):
        assert parse_png(png[:33] + pr.chunk(t, b"\0" * 8) + png[33:]) is None
    for t in (b"gAMA", b"tEXt", b"pHYs"):
        assert parse_png(png[:33] + pr.chunk(t, b"\0" * 9) + png[33:]) is not None
    ihdr16 = struct.pack(">IIBBBBB", 33, 20, 16, 3, 0, 0, 0)          # 16-bit palette: not a legal pair
    assert parse_png(png[:8] + pr.chunk(b"IHDR", ihdr16) + png[33:]) is None
    zbad = pr.write_png(_samples(np.random.default_rng(1), 4, 4, 0, 8), 0, 8, zdata=b"\x78\x9d" + b"\0" * 8)
    assert parse_png(zbad) is None                                   # preset dictionary flag


def test_parse_png_of_pil_and_cv2_files():
    rng = np.random.default_rng(11)
    lab = rng.integers(0, 5, (30, 40)).astype(np.uint8)
    pal = rng.integers(0, 256, (256, 3), dtype=np.uint8)
    im = Image.fromarray(lab, "P")
    im.putpalette(pal.tobytes())
    for kw in ({}, {"transparency": 0}):
        b = io.BytesIO()
        im.save(b, "PNG", **kw)
        p = parse_png(b.getvalue())
        assert p is not None and p.color_type == 3
    ok, enc = cv2.imencode(".png", pal[lab])
    p = parse_png(enc.tobytes())
    assert ok and p is not None and p.color_type == 2 and zlib.decompress(p.zdata)[0] == 1   # cv2 writes Sub rows
