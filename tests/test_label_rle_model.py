"""Host model of stage E's device encoding (s2d_b200/csrc/label_rle.cu), checked against the restatement of maskApi.c
(oracle/coco_rle.py) and the host string helpers. Runs without a GPU.

Label RLE: in column-major order a transition a -> b between pixel labels is an edge of mask a and of mask b only; the
kernels find the transitions per strip of columns, number each label's edges per strip, and place a strip's edges
after those of the strips to its left. String packing: every count is packed from itself and the count two places
back, so lengths and digits are independent per count."""
import numpy as np
import pytest

from oracle import coco_rle as cr
from s2d_b200.keymask_ident.annotations import coco_rle

NONE = 256


def _edges_by_strips(lab: np.ndarray, labels, S: int):
    """The kernels' bookkeeping: pass 1 counts the edges of each label per strip of S columns, a prefix over strips
    gives each strip's first slot, pass 2 writes the edges of a strip in its walk order (column by column, top to
    bottom) at prefix + rank. Returns {label: edge positions (column-major pixel index)}."""
    H, W = lab.shape
    strips = [(x0, min(W, x0 + S)) for x0 in range(0, W, S)]
    walk = []                                           # per strip: [(pos, a, b)] in the strip's walk order
    for x0, x1 in strips:
        carry = int(lab[H - 1, x0 - 1]) if x0 > 0 else NONE
        ev = []
        for x in range(x0, x1):
            col = lab[:, x].astype(np.int64)
            prev = np.concatenate(([carry], col[:-1]))
            for y in np.nonzero(col != prev)[0]:
                ev.append((x * H + int(y), int(prev[y]), int(col[y])))
            carry = int(col[-1])
        walk.append(ev)
    counts = np.zeros((len(strips), 257), np.int64)
    for s, ev in enumerate(walk):
        for _, a, b in ev:
            counts[s, a] += 1
            counts[s, b] += 1
    first = np.cumsum(counts, axis=0) - counts         # exclusive prefix over strips
    out = {l: np.full(int(counts[:, l].sum()), -1, np.int64) for l in labels}
    for s, ev in enumerate(walk):
        rank = first[s].copy()
        for pos, a, b in ev:
            for l in (a, b):
                if l in out:
                    out[l][rank[l]] = pos
                    rank[l] += 1
    return out


def _runs_and_box(edges: np.ndarray, H: int, W: int):
    """lr_diff_kernel: runs are the differences of 0, the edges and H * W; set runs [e_2k, e_2k+1) give the box, a set
    run that crosses a column boundary spans all rows."""
    e = np.concatenate((edges, [H * W]))
    runs = np.diff(np.concatenate(([0], e))).tolist()
    xs = ys = 1 << 30
    xe = ye = -1
    for k in range(0, len(edges), 2):
        lo, hi = int(e[k]), int(e[k + 1]) - 1
        xs, xe = min(xs, lo // H), max(xe, hi // H)
        if lo // H != hi // H:
            ys, ye = 0, H - 1
        else:
            ys, ye = min(ys, lo % H), max(ye, hi % H)
    return runs, [float(xs), float(ys), float(xe - xs + 1), float(ye - ys + 1)]


def _maps(H, W, seed):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    blobs = np.zeros((H, W), np.uint8)
    for l in range(1, 9):
        cy, cx = rng.uniform(0, H), rng.uniform(0, W)
        ry, rx = rng.uniform(1, max(2, H / 3)), rng.uniform(1, max(2, W / 3))
        blobs[((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 <= 1] = l
    corners = np.zeros((H, W), np.uint8)
    corners[0, 0] = 3
    corners[-1, -1] = 9
    top = np.where((xx + yy) % 5 < 2, 255, 0).astype(np.uint8)
    return {"blobs": blobs, "random": rng.integers(0, 256, size=(H, W)).astype(np.uint8),
            "full": np.full((H, W), 7, np.uint8), "background": np.zeros((H, W), np.uint8), "corners": corners,
            "label255": top, "stripes": (yy // 3 % 4).astype(np.uint8)}


@pytest.mark.parametrize("H,W", [(1, 1), (1, 9), (7, 1), (31, 33), (40, 70), (97, 131)])
@pytest.mark.parametrize("S", [32, 16, 1])
def test_transition_rule_equals_rle_encode(H, W, S):
    for name, lab in _maps(H, W, H * 1000 + W).items():
        present = [int(l) for l in np.unique(lab)]
        edges = _edges_by_strips(lab, present, S)
        for l in present:
            m = lab == l
            assert (edges[l] >= 0).all() and np.all(np.diff(edges[l]) > 0), (name, l)
            runs, box = _runs_and_box(edges[l], H, W)
            assert runs == cr.counts(m), (name, l)
            assert box == cr.bbox(m), (name, l)
            assert sum(runs[1::2]) == int(m.sum())


def _pack_model(cnts):
    """rs_kernel: per count, the value x = c[i] - c[i-2] (i > 2) in int32 arithmetic, its 5-bit digit count, a scan of
    the lengths, then the digits; continuation bit on every digit but the last."""
    c = np.asarray(cnts, np.int64)
    xs = [int(np.int32(c[i] - (c[i - 2] if i > 2 else 0))) for i in range(len(c))]

    def length(x):
        n = 0
        while True:
            d = x & 0x1F
            x >>= 5
            n += 1
            if not ((x != -1) if (d & 0x10) else (x != 0)):
                return n

    lens = [length(x) for x in xs]
    offs = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    out = bytearray(int(offs[-1]))
    for i, x in enumerate(xs):
        for k in range(lens[i]):
            d = x & 0x1F
            x >>= 5
            out[offs[i] + k] = (d | (0x20 if k + 1 < lens[i] else 0)) + 48
    return out.decode("ascii"), max(lens, default=0)


def test_string_packer_rule_equals_to_string():
    rng = np.random.default_rng(5)
    big = 2 ** 31 - 1
    cases = [[0], [5], [0, 1], [3, 4, 5], [0, 10, 3, 2, 100, 1], [1, big], [0, big, 1, big - 1, 0, 1],
             [big, 0, big, 0, 1, big], [7, 2 ** 20, 3, 1, 2 ** 25, 2 ** 30 + 3, 0, big]]
    cases += [rng.integers(0, 2000, size=int(rng.integers(1, 60))).tolist() for _ in range(200)]
    cases += [rng.integers(0, 2 ** 31, size=int(rng.integers(1, 30))).tolist() for _ in range(100)]
    cases += [cr.counts(m) for m in _maps(37, 53, 3).values()]
    widest = 0
    for c in cases:
        s, w = _pack_model(c)
        widest = max(widest, w)
        assert s == coco_rle.to_string(c), c
        assert coco_rle.from_string(s) == [int(x) for x in c]
    assert widest == 7                      # 31-bit values with a sign: seven 5-bit digits, no more
