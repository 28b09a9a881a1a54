"""Host models of the COCO RLE decode kernels (s2d_b200/csrc/rle_decode.cu), no GPU:
- the parallel parse of rp_write_kernel - value ends from the continuation bit, each value assembled from the groups since
  the previous end, the two interleaved chains (odd indices from 1, even from 2) as prefix sums in uint32, the status
  rules - against the serial coco_rle.from_string;
- the tiled decode of rd_tile_kernel - run starts by a prefix sum, per tile column a search for the run covering the
  tile's first row, the one-run fast path, rows placed at their address mod 16 - against oracle.coco_rle.decode."""
import numpy as np
import pytest

from oracle import coco_rle as oc
from s2d_b200.keymask_ident.annotations import coco_rle

TC, TR = 128, 64


def parse_model(s: bytes):
    """(counts, status) the way rp_write_kernel computes them, vectorised over the characters."""
    c = (np.frombuffer(s, np.uint8).astype(np.int64) - 48) & 0x3F
    ends = (c & 0x20) == 0
    bad = bool(len(c)) and not ends[-1]
    idx = np.nonzero(ends)[0]
    starts = np.concatenate(([0], idx[:-1] + 1)) if len(idx) else idx
    xs = []
    for a, b in zip(starts, idx):                     # value = groups a..b, sign-extended from the last group's 0x10
        g = c[a:b + 1] & 0x1F
        k = len(g)
        lo = 0
        for j in range(min(k, 12)):
            lo |= int(g[j]) << (5 * j)
        neg = bool(g[-1] & 0x10)
        high = g[12:]
        big = bool((high != 0x1F).any()) if neg else bool((high != 0).any())
        x = lo - (1 << min(5 * k, 60)) if neg else lo
        bad |= big or not (-(1 << 31) < x < (1 << 31))
        xs.append(x)
    u = np.asarray(xs, np.int64).astype(np.uint32)
    j = np.arange(len(u))
    odd = np.cumsum(np.where(j % 2 == 1, u, 0), dtype=np.uint32)
    even = np.cumsum(np.where((j % 2 == 0) & (j >= 2), u, 0), dtype=np.uint32)
    cnt = np.where(j == 0, u, np.where(j % 2 == 1, odd, even)).astype(np.uint32)
    bad |= bool((cnt >= 2 ** 31).any())
    return cnt.astype(np.int64).tolist(), int(bad)


def host_reference(s: bytes):
    """from_string's counts, and whether it fails or leaves [0, 2^31)"""
    try:
        cnts = coco_rle.from_string(s.decode("latin-1"))
    except IndexError:
        return None, 1
    return cnts, int(any(not (0 <= x < 2 ** 31) for x in cnts))


def random_counts(rng, n, big=False):
    hi = 2 ** 31 - 1 if big else 3000
    return rng.integers(0 if big else 1, hi, size=n).tolist()


@pytest.mark.parametrize("seed", range(6))
def test_parse_model_equals_from_string(seed):
    rng = np.random.default_rng(seed)
    for n in list(range(6)) + [100, 257, 640]:
        for big in (False, True):
            cnts = random_counts(rng, n, big)
            if n > 3 and not big:
                cnts[rng.integers(3, n)] = 0                      # negative delta and a zero run
            s = coco_rle.to_string(cnts).encode()
            got, st = parse_model(s)
            assert st == 0 and got == cnts == coco_rle.from_string(s.decode())


def test_parse_model_extremes_and_malformed():
    cases = [[2 ** 31 - 1, 2 ** 31 - 1, 0, 2 ** 31 - 1, 0, 1], [0, 2 ** 31 - 1, 2 ** 31 - 1, 0, 2 ** 31 - 1]]
    for cnts in cases:
        got, st = parse_model(coco_rle.to_string(cnts).encode())
        assert st == 0 and got == cnts
    rng = np.random.default_rng(5)
    ok = coco_rle.to_string(random_counts(rng, 40)).encode()
    bad_inputs = [
        ok + b"P",                                             # last character continues ('P' - 48 = 0x20)
        b"\x2f",                                               # byte 47: c = -1, continuation bit set
        coco_rle.to_string([5, -3]).encode(),                  # a negative count
        coco_rle.to_string([5, 2 ** 31]).encode(),             # a count of 2^31
        coco_rle.to_string([1, 5, 3, 2 ** 31 + 4]).encode(),   # delta 2^31 - 1 in range, cnts[3] = 5 + delta is not
        b"P" * 14 + b"1",                                      # 15 groups, 2^70
        b"o" * 14 + b"?",                                      # 15 groups of -1 then 0x0F: not the sign pattern
    ]
    for s in bad_inputs:
        got, st = parse_model(s)
        want, wst = host_reference(s)
        assert st == wst == 1, s
        if want is not None and len(want) == len(got):
            assert [x % 2 ** 32 for x in want] == got
    # long values that stay small: redundant groups above the sign (-1 in 15 groups is still a bad count)
    for s, wst in ((b"o" * 14 + b"O", 1), (b"P" * 13 + b"0", 0), (b"1" + b"P" * 20 + b"0", 0)):
        got, st = parse_model(s)
        want, _ = host_reference(s)
        assert st == wst and got == [x % 2 ** 32 for x in want]
    # bytes outside '0'..'o' follow byte - 48
    s = bytes([48 + 5, 200, 10, 48 + 7])
    got, st = parse_model(s)
    want, wst = host_reference(s)
    assert st == wst and (st or got == want)


def decode_model(cnts, h, w, out_off=0):
    """rd_tile_kernel's tiles on a flat buffer (the mask at byte out_off of a 16-aligned buffer); returns [h, w]."""
    st = np.concatenate(([0], np.cumsum(np.asarray(cnts, np.int64))))
    nc, total = len(cnts), int(st[-1])
    buf = np.full(out_off + h * w + 32, 0xEE, np.uint8)
    for y0 in range(0, h, TR):
        for x0 in range(0, w, TC):
            rows, cols = min(TR, h - y0), min(TC, w - x0)
            col_r, col_v, uni = [], [], []
            for x in range(x0, x0 + cols):
                p0 = x * h + y0
                if p0 >= total:
                    r, v, u = nc, 0, True
                else:
                    r = int(np.searchsorted(st[:nc], p0, side="right")) - 1
                    v, u = r & 1, st[r + 1] >= p0 + rows
                col_r.append(r)
                col_v.append(v)
                uni.append(u)
            fast = all(uni) and len(set(col_v)) == 1
            tile = np.full((rows, cols), 0xAA, np.uint8)
            for ci in range(cols):
                p0 = (x0 + ci) * h + y0
                if fast:
                    tile[:, ci] = col_v[0]
                    continue
                r, y = col_r[ci], 0
                while y < rows:
                    end = min(int(st[r + 1]) - p0, rows) if r < nc else rows
                    b = r & 1 if r < nc else 0
                    tile[y:max(y, end), ci] = b
                    y = max(y, end)
                    r += 1
            for yy in range(rows):
                a = out_off + (y0 + yy) * w + x0
                buf[a:a + cols] = tile[yy]
    assert (buf[:out_off] == 0xEE).all() and (buf[out_off + h * w:] == 0xEE).all()
    return buf[out_off:out_off + h * w].reshape(h, w)


def blob(rng, h, w):
    yy, xx = np.mgrid[:h, :w]
    m = np.zeros((h, w), bool)
    for _ in range(3):
        cy, cx, r = rng.integers(0, h), rng.integers(0, w), rng.integers(1, max(2, min(h, w) // 2))
        m |= (yy - cy) ** 2 + (xx - cx) ** 2 < r * r
    return m


@pytest.mark.parametrize("shape", [(1, 1), (1, 300), (300, 1), (7, 13), (65, 129), (130, 257), (64, 128), (200, 77)])
def test_decode_model_equals_oracle(shape):
    h, w = shape
    rng = np.random.default_rng(h * 1000 + w)
    masks = [np.zeros((h, w), bool), np.ones((h, w), bool), blob(rng, h, w),
             (np.add.outer(np.arange(h), np.arange(w)) % 2).astype(bool)]
    p = np.zeros((h, w), bool)
    p[0, 0] = True
    masks.append(p)
    for m in masks:
        cnts = oc.counts(m)
        for off in (0, 3, 21):
            assert np.array_equal(decode_model(cnts, h, w, off), oc.decode(cnts, h, w))


def test_decode_model_wrong_sums():
    h, w = 70, 150
    m = blob(np.random.default_rng(3), h, w)
    cnts = oc.counts(m)
    short = cnts[:-1]
    want = oc.decode(short, h, w)
    assert np.array_equal(decode_model(short, h, w, 5), want)
    long = cnts[:-1] + [cnts[-1] + 500, 40, 9]
    assert np.array_equal(decode_model(long, h, w, 5), m.astype(np.uint8))
