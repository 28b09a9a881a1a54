"""Test helpers for the PNG decoder: a minimal PNG writer (struct, zlib, crc32) that forces a filter type per row and
a deflate variant, host models of the kernels' Huffman tables and row filters, and per-byte reference loops."""
from __future__ import annotations

import struct
import zlib

import numpy as np

CHANNELS = {0: 1, 2: 3, 3: 1, 4: 2, 6: 4}
LEGAL = [(0, 1), (0, 2), (0, 4), (0, 8), (0, 16), (2, 8), (2, 16), (3, 1), (3, 2), (3, 4), (3, 8), (4, 8), (4, 16),
         (6, 8), (6, 16)]


def chunk(ctype: bytes, body: bytes) -> bytes:
    return struct.pack(">I", len(body)) + ctype + body + struct.pack(">I", zlib.crc32(ctype + body))


def pack_rows(samples: np.ndarray, ct: int, bd: int) -> np.ndarray:
    """[H, W, C] integer samples -> [H, rowbytes] uint8 scanlines (unfiltered)."""
    H, W = samples.shape[:2]
    s = samples.reshape(H, W * CHANNELS[ct]).astype(np.uint32)
    if bd == 16:
        return np.stack([s >> 8, s & 0xFF], axis=-1).reshape(H, -1).astype(np.uint8)
    if bd == 8:
        return s.astype(np.uint8)
    per = 8 // bd
    rb = (W * CHANNELS[ct] * bd + 7) // 8
    pad = np.zeros((H, rb * per), np.uint32)
    pad[:, :s.shape[1]] = s
    g = pad.reshape(H, rb, per)
    out = np.zeros((H, rb), np.uint32)
    for k in range(per):
        out |= g[:, :, k] << (8 - bd * (k + 1))
    return out.astype(np.uint8)


def paeth(a, b, c):
    p = a + b - c
    pa, pb, pc = abs(p - a), abs(p - b), abs(p - c)
    return a if pa <= pb and pa <= pc else b if pb <= pc else c


def filter_rows(rows: np.ndarray, bpp: int, types) -> bytes:
    """Filtered scanlines: row y gets filter types[y % len(types)]."""
    H, rb = rows.shape
    out = bytearray()
    prev = np.zeros(rb, np.int32)
    for y in range(H):
        f = types[y % len(types)]
        cur = rows[y].astype(np.int32)
        left = np.concatenate([np.zeros(bpp, np.int32), cur[:-bpp]]) if rb > bpp else np.zeros(rb, np.int32)
        left = left[:rb]
        ul = np.concatenate([np.zeros(bpp, np.int32), prev[:-bpp]])[:rb]
        if f == 0:
            r = cur
        elif f == 1:
            r = cur - left
        elif f == 2:
            r = cur - prev
        elif f == 3:
            r = cur - (left + prev) // 2
        else:
            r = cur - np.array([paeth(int(a), int(b), int(c)) for a, b, c in zip(left, prev, ul)], np.int32)
        out.append(f)
        out += (r & 0xFF).astype(np.uint8).tobytes()
        prev = cur
    return bytes(out)


def compress(raw: bytes, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, wbits=15) -> bytes:
    c = zlib.compressobj(level, zlib.DEFLATED, wbits, 9, strategy)
    return c.compress(raw) + c.flush()


def write_png(samples: np.ndarray, ct: int, bd: int, palette: np.ndarray | None = None, filters=(0,), level=6,
              strategy=zlib.Z_DEFAULT_STRATEGY, extra=(), idat_split=None, zdata: bytes | None = None,
              trns: bytes | None = None) -> bytes:
    """PNG of [H, W, C] samples with forced per-row filters and deflate settings; `extra` chunks (type, body) go
    before IDAT; idat_split cuts the stream into IDAT chunks of that many bytes; zdata replaces the stream."""
    H, W = samples.shape[:2]
    rows = pack_rows(samples, ct, bd)
    bpp = max(1, CHANNELS[ct] * bd // 8)
    raw = filter_rows(rows, bpp, filters)
    z = zdata if zdata is not None else compress(raw, level, strategy)
    out = b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", W, H, bd, ct, 0, 0, 0))
    for t, b in extra:
        out += chunk(t, b)
    if palette is not None:
        out += chunk(b"PLTE", np.asarray(palette, np.uint8).tobytes())
    if trns is not None:
        out += chunk(b"tRNS", trns)
    step = idat_split or max(1, len(z))
    for i in range(0, max(1, len(z)), step):
        out += chunk(b"IDAT", z[i:i + step])
    return out + chunk(b"IEND", b"")


# ---- host model of the inflate kernel's tables -------------------------------------------------------------------

PTR = 1 << 24


def rev_bits(x: int, n: int) -> int:
    return int(format(x, f"0{n}b")[::-1], 2) if n else 0


def build_table(lens, root: int, cap: int):
    """The kernel's build_table: counts per length, canonical codes in (length, symbol) order, short codes replicated
    over their primary slots, each primary slot with longer codes pointing to a sub-table of 2^(its longest code -
    root) entries, placed by an exclusive scan over the slots. None for an oversubscribed or incomplete code."""
    n = len(lens)
    cnt = [0] * 16
    for l in lens:
        if l:
            cnt[l] += 1
    left, code, nxt, maxl = 1, 0, [0] * 16, 0
    for l in range(1, 16):
        left = (left << 1) - cnt[l]
        if left < 0:
            return None
        code = (code + cnt[l - 1]) << 1
        nxt[l] = code
        if cnt[l]:
            maxl = l
    if left > 0 and maxl > 1:
        return None
    tab = [0] * cap
    sub = [0] * (1 << root)
    codes = [0] * n
    for s, l in enumerate(lens):                  # rank within a length = symbol order (the kernel's match_any rank)
        if not l:
            continue
        codes[s] = nxt[l]
        nxt[l] += 1
        if l <= root:
            r = rev_bits(codes[s], l)
            for k in range(1 << (root - l)):
                tab[r | (k << l)] = s | (l << 16)
        else:
            p = rev_bits(codes[s] >> (l - root), root)
            sub[p] = max(sub[p], l - root)
    off = 1 << root
    for p in range(1 << root):
        if sub[p]:
            tab[p] = off | (sub[p] << 16) | PTR
            off += 1 << sub[p]
    if off > cap:
        return None
    for s, l in enumerate(lens):
        if l > root:
            e = tab[rev_bits(codes[s] >> (l - root), root)]
            b, o, ls = (e >> 16) & 0xFF, e & 0xFFFF, l - root
            r = rev_bits(codes[s] & ((1 << ls) - 1), ls)
            for k in range(1 << (b - ls)):
                tab[o + (r | (k << ls))] = s | (l << 16)
    return tab, off


LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEN_EXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
             6145, 8193, 12289, 16385, 24577]
DIST_EXTRA = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]
CLEN_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]


class _Bits:
    def __init__(self, data: bytes, pos: int):
        self.d = bytes(data[pos:]) + bytes(8)
        self.n = 8 * (len(data) - pos)
        self.at = 0

    def peek(self, k):
        q = self.at >> 3
        return (int.from_bytes(self.d[q:q + 4], "little") >> (self.at & 7)) & ((1 << k) - 1)

    def take(self, k):
        x = self.peek(k)
        self.at += k
        if self.at > self.n:
            raise ValueError("truncated")
        return x


def _sym(bits, tab, root):
    e = tab[bits.peek(root)]
    if e & PTR:
        b = (e >> 16) & 0xFF
        e = tab[(e & 0xFFFF) + ((bits.peek(root + b) >> root) & ((1 << b) - 1))]
    l = (e >> 16) & 0xFF
    if not l:
        raise ValueError("bad code")
    bits.take(l)
    return e & 0xFFFF


def inflate_model(z: bytes) -> bytes:
    """zlib stream -> bytes with the kernel's tables (primary 9 / 6 / 7 bits plus sub-tables)."""
    bits = _Bits(z, 2)
    out = bytearray()
    last = False
    while not last:
        last = bits.take(1)
        t = bits.take(2)
        if t == 0:
            bits.take((-bits.at) % 8)
            ln, nln = bits.take(16), bits.take(16)
            assert ln ^ 0xFFFF == nln
            p = 2 + bits.at // 8
            out += z[p:p + ln]
            bits.at += 8 * ln
            continue
        if t == 1:
            lens = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
            dl = [5] * 32
        else:
            nlen, ndist, ncl = bits.take(5) + 257, bits.take(5) + 1, bits.take(4) + 4
            cl = [0] * 19
            for i in range(ncl):
                cl[CLEN_ORDER[i]] = bits.take(3)
            ctab, _ = build_table(cl, 7, 128)
            ll = []
            while len(ll) < nlen + ndist:
                s = _sym(bits, ctab, 7)
                if s < 16:
                    ll.append(s)
                elif s == 16:
                    ll += [ll[-1]] * (3 + bits.take(2))
                elif s == 17:
                    ll += [0] * (3 + bits.take(3))
                else:
                    ll += [0] * (11 + bits.take(7))
            lens, dl = ll[:nlen], ll[nlen:]
        lt, lused = build_table(lens, 9, 852)
        dt, dused = build_table(dl, 6, 592)
        assert lused <= 852 and dused <= 592
        while True:
            s = _sym(bits, lt, 9)
            if s < 256:
                out.append(s)
                continue
            if s == 256:
                break
            ln = LEN_BASE[s - 257] + bits.take(LEN_EXTRA[s - 257])
            d = _sym(bits, dt, 6)
            dist = DIST_BASE[d] + bits.take(DIST_EXTRA[d])
            assert dist <= len(out)
            for _ in range(ln):
                out.append(out[-dist])
    return bytes(out)


# ---- row filters: the kernel's decomposition and a per-byte reference --------------------------------------------

def unfilter_reference(raw: bytes, H: int, rb: int, bpp: int) -> np.ndarray:
    out = np.zeros((H, rb), np.uint8)
    prev = [0] * rb
    for y in range(H):
        f = raw[y * (rb + 1)]
        r = raw[y * (rb + 1) + 1:(y + 1) * (rb + 1)]
        cur = [0] * rb
        for x in range(rb):
            a = cur[x - bpp] if x >= bpp else 0
            b = prev[x]
            c = prev[x - bpp] if x >= bpp else 0
            pred = [0, a, b, (a + b) // 2, paeth(a, b, c)][f]
            cur[x] = (r[x] + pred) & 0xFF
        out[y] = cur
        prev = cur
    return out


def unfilter_model(raw: bytes, H: int, rb: int, bpp: int) -> np.ndarray:
    """png_unfilter_kernel's order of work: 32-byte steps, Sub as a stride-bpp Hillis-Steele scan over the 32 lanes
    plus the carry from lane 32 - bpp + lane % bpp of the previous step; Avg / Paeth one chain per byte of a pixel."""
    row = np.zeros(rb, np.uint32)
    out = np.zeros((H, rb), np.uint8)
    lanes = np.arange(32)
    for y in range(H):
        f = raw[y * (rb + 1)]
        r = np.frombuffer(raw, np.uint8, rb, y * (rb + 1) + 1).astype(np.uint32)
        if f <= 2:
            prev_out = np.zeros(32, np.uint32)
            for x0 in range(0, rb, 32):
                x = x0 + lanes
                v = np.where(x < rb, r[np.minimum(x, rb - 1)], 0).astype(np.uint32)
                o = v.copy()
                if f == 1:
                    k = bpp
                    while k < 32:
                        u = np.concatenate([np.zeros(k, np.uint32), o[:-k]])
                        o = o + u
                        k <<= 1
                    c = prev_out[32 - bpp + lanes % bpp]
                    o = o + (c if x0 else 0)
                elif f == 2:
                    o = o + np.where(x < rb, row[np.minimum(x, rb - 1)], 0)
                o &= 0xFF
                prev_out = o
                ok = x < rb
                row[x[ok]] = o[ok]
        else:
            for lane in range(bpp):
                a = c = 0
                for x in range(lane, rb, bpp):
                    b = int(row[x])
                    pred = (a + b) >> 1 if f == 3 else paeth(a, b, c)
                    o = (int(r[x]) + pred) & 0xFF
                    row[x] = o
                    a, c = o, b
        out[y] = row
    return out


def to_rgb_reference(rows: np.ndarray, W: int, ct: int, bd: int, palette: np.ndarray | None) -> np.ndarray:
    """Unfiltered scanlines -> [H, W, 3] RGB as cv2.imread(IMREAD_COLOR) returns them (after BGR -> RGB)."""
    H = rows.shape[0]
    ch = CHANNELS[ct]
    if bd < 8:
        bits = np.unpackbits(rows, axis=1)[:, :W * bd].reshape(H, W, bd)
        s = (bits * (1 << np.arange(bd - 1, -1, -1))).sum(-1).astype(np.uint32)
        if ct == 3:
            return np.asarray(palette, np.uint8).reshape(-1, 3)[s]
        return np.repeat((s * {1: 255, 2: 85, 4: 17}[bd]).astype(np.uint8)[..., None], 3, axis=2)
    hi = rows.reshape(H, W * ch, bd // 8)[..., 0].reshape(H, W, ch)
    if ct == 3:
        return np.asarray(palette, np.uint8).reshape(-1, 3)[hi[..., 0]]
    if ct in (0, 4):
        return np.repeat(hi[..., :1], 3, axis=2)
    return np.ascontiguousarray(hi[..., :3])
