"""Host model of the annotation json (s2d_b200/csrc/annotation_json.cu), checked against Python's json.dumps on the
annotations of synthetic batches, and the file envelope of write_video_annotations for bytes. Runs without a GPU.

The kernels print one2x from k = round_half_even(100 * gs / gn) computed in integers from the double's mantissa and
exponent, write '\\' as "\\\\", and give every annotation the length of its text plus 2 (its ", " or the video's brackets)
before a scan places it."""
import json
import math
import os
import struct

import numpy as np
import pytest

from tests.annotation_reference import reference, synthetic_batch
from tests.test_annotation_layout_model import model_layout


def one2x_text(gs: int, gn: int) -> str:
    """AjOut::one2x: repr(round(gs / gn, 2)), 0.0 when gn == 0"""
    x = gs / gn if gn else 0.0
    sign = "-" if math.copysign(1.0, x) < 0 else ""
    bits = struct.unpack("<Q", struct.pack("<d", abs(x)))[0]
    ex, m = bits >> 52, bits & ((1 << 52) - 1)
    if ex == 0:
        e = -1074
    else:
        m |= 1 << 52
        e = ex - 1075
    n100 = 100 * m
    if e >= 0:
        k = n100 << e
    elif -e > 62:
        k = 0
    else:
        s = -e
        q, r, half = n100 >> s, n100 & ((1 << s) - 1), 1 << (s - 1)
        k = q + (r > half or (r == half and q & 1))
    f = k % 100
    return f"{sign}{k // 100}." + (str(f // 10) if f % 10 == 0 else f"{f:02d}")


def test_one2x_exhaustive_small():
    for gn in range(1, 1001):
        for gs in range(0, 4 * gn + 1):
            assert one2x_text(gs, gn) == repr(round(gs / gn, 2)), (gs, gn)
    assert one2x_text(0, 0) == "0.0" == repr(0.0)
    assert one2x_text(7, 0) == "0.0"


def test_one2x_random_and_ties():
    rng = np.random.default_rng(0)
    gs = rng.integers(0, 2 ** 31, size=10 ** 6).tolist()
    gn = rng.integers(1, 2 ** 31, size=10 ** 6).tolist()
    small = rng.integers(1, 2 ** 16, size=10 ** 5).tolist()
    for a, b in zip(gs, gn):
        assert one2x_text(a, b) == repr(round(a / b, 2)), (a, b)
    for a, b in zip(gs[:10 ** 5], small):          # ratios far above 1
        assert one2x_text(a, b) == repr(round(a / b, 2)), (a, b)
    ties = [(1, 8), (3, 8), (5, 8), (7, 8), (1, 200)]
    for m in range(1, 2000):
        for k in range(0, 200, 7):
            if 200 * m < 2 ** 31 and m * (2 * k + 1) < 2 ** 31:
                ties.append((m * (2 * k + 1), 200 * m))
    for a, b in ties:
        assert one2x_text(a, b) == repr(round(a / b, 2)), (a, b)
    assert [one2x_text(a, b) for a, b in ties[:5]] == ["0.12", "0.38", "0.62", "0.88", "0.01"]


def model_text(H, W, T, aid, gs, gn, mems, strings, pairs):
    """aj_text_kernel's text of one annotation, piece by piece as the kernel emits it. mems: (frame, x0, y0, x1, y1,
    area) in frame order; strings: the members' RLE strings; pairs: (start, end) of the cluster's runs."""
    out = [f'{{"video_id": 1, "iscrowd": 0, "height": {H}, "width": {W}, "length": {T}']
    for sec, head in enumerate((', "segmentations": [', '], "bboxes": [', '], "areas": [')):
        out.append(head)
        prev = -1
        for (f, x0, y0, x1, y1, area), s in zip(mems, strings):
            out.append("null, " * (f - prev - 1))
            if sec == 0:
                out.append(f'{{"size": [{H}, {W}], "counts": "' + s.replace("\\", "\\\\") + '"}')
            elif sec == 1:
                out.append(f"[{x0}.0, {y0}.0, {x1 - x0 + 1}.0, {y1 - y0 + 1}.0]")
            else:
                out.append(str(area))
            if f < T - 1:
                out.append(", ")
            prev = f
        if T - 1 - prev > 0:
            out.append("null, " * (T - 1 - prev - 1) + "null")
    out.append(f'], "category_id": 1, "id": {aid}, "one2x": {one2x_text(gs, gn)}, "visibility_ranges": [')
    out.append(", ".join(f"[{s}, {e}]" for s, e in pairs))
    out.append("]}")
    return "".join(out)


def model_length(H, W, T, aid, gs, gn, mems, strings, pairs):
    """aj_text_kernel<false>: the byte count alone, strings counted as length + backslashes"""
    digits = lambda x: len(str(x))
    n = len('{"video_id": 1, "iscrowd": 0, "height": , "width": , "length": ') + digits(H) + digits(W) + digits(T)
    n += len(', "segmentations": [') + len('], "bboxes": [') + len('], "areas": [')
    frames = [m[0] for m in mems]
    n += 3 * (4 * (T - len(mems)) + 2 * (T - 1))                       # nulls and separators of the three lists
    for (f, x0, y0, x1, y1, area), s in zip(mems, strings):
        n += len('{"size": [, ], "counts": ""}') + digits(H) + digits(W) + len(s) + s.count("\\")
        n += len("[.0, .0, .0, .0]") + digits(x0) + digits(y0) + digits(x1 - x0 + 1) + digits(y1 - y0 + 1)
        n += digits(area)
    n += len('], "category_id": 1, "id": , "one2x": , "visibility_ranges": []}') + digits(aid) + len(one2x_text(gs, gn))
    n += sum(len("[, ]") + digits(s) + digits(e) for s, e in pairs) + 2 * max(0, len(pairs) - 1)
    assert frames == sorted(set(frames))
    return n


def model_videos(t):
    """per video the model's annotation texts and lengths from the layout tables of a synthetic batch"""
    tabs = model_layout(t)
    vann, ann = tabs["vann"].reshape(-1, 2), tabs["ann"].reshape(-1, 7)
    mem, moff = tabs["members"].reshape(-1, 6), tabs["member_off"].tolist() + [len(tabs["chars"])]
    chars = tabs["chars"].tobytes().decode("ascii")
    clusters, pairs = tabs["clusters"].reshape(-1, 2), tabs["pairs"].reshape(-1, 2)
    out = []
    for vi, d in enumerate(t.descs):
        if t.vidinfo[vi, 3] != 1:
            out.append(None)
            continue
        n, a0 = (int(x) for x in vann[vi])
        anns = []
        for a in range(a0, a0 + n):
            _, _, gn, gs, ci, m0, nm = (int(x) for x in ann[a])
            ms = [tuple(int(x) for x in mem[m]) for m in range(m0, m0 + nm)]
            ss = [chars[moff[m]:moff[m + 1]] for m in range(m0, m0 + nm)]
            p0, npairs = (int(x) for x in clusters[ci])
            pr = [tuple(int(x) for x in p) for p in pairs[p0:p0 + npairs]]
            args = (d.H, d.W, d.T, a - a0 + 1, gs, gn, ms, ss, pr)
            anns.append((model_text(*args), model_length(*args)))
        out.append(anns)
    return out


@pytest.mark.parametrize("seed", range(8))
def test_model_length_equals_json_dumps(seed):
    t = synthetic_batch(seed, nvideos=6)
    want = reference(t)
    got = model_videos(t)
    for w, g in zip(want, got):
        assert (w is None) == (g is None)
        if w is None:
            continue
        for a, (text, n) in zip(w, g):
            assert text == json.dumps(a)
            assert n == len(json.dumps(a))
        # the video's text: "[" + annotations joined by ", " + "]" = the lengths + 2 each, or "[]"
        assert (sum(n + 2 for _, n in g) if g else 2) == len(json.dumps(w))


def test_synthetic_batches_cover_escapes_and_large_one2x():
    bs = big = False
    for seed in range(8):
        for w in reference(synthetic_batch(seed, nvideos=6)):
            if w is None:
                continue
            s = json.dumps(w)
            bs |= "\\\\" in s
            big |= any(a["one2x"] > 1 for a in w)
    assert bs and big


def test_write_video_annotations_bytes_envelope(tmp_path):
    from PIL import Image

    from s2d_b200.keymask_ident.annotations import _dump_video_json, _video_entry, write_video_annotations
    vdir = tmp_path / "vidéo_1"
    vdir.mkdir()
    for i in range(3):
        Image.fromarray(np.zeros((7, 11, 3), np.uint8)).save(vdir / f"{i:05d}.jpg")
    anns = [a for a in reference(synthetic_batch(1, nvideos=6)) if a][0]
    for lst in (anns, []):
        out_list, out_bytes = tmp_path / "list", tmp_path / "bytes"
        _dump_video_json(_video_entry(str(vdir)), lst, str(out_list), str(vdir))
        write_video_annotations(str(vdir), json.dumps(lst).encode(), str(out_bytes))
        name = os.path.basename(str(vdir)) + ".json"
        a, b = (out_list / name).read_bytes(), (out_bytes / name).read_bytes()
        assert a == b and json.loads(b)["annotations"] == json.loads(json.dumps(lst))
    write_video_annotations(str(vdir), None, str(tmp_path / "none"))
    assert not (tmp_path / "none").exists()
