"""COCO RLE decode on the device (s2d_rle_from_strings, s2d_rle_decode, coco_rle.decode_batch,
decode_video_annotations) against the host parser coco_rle.from_string and oracle.coco_rle.decode, and stage E's json
decoded back to the label maps it came from."""
import ctypes as C
import json

import numpy as np
import pytest
import torch

from oracle import coco_rle as oc
from s2d_b200.keymask_ident.annotations import coco_rle, decode_video_annotations
from tests.conftest import GOLDEN_CASES, load_golden

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _parse_cabi(blobs, capacity=None, guard=-77):
    """s2d_rle_from_strings on byte strings; returns (counts buffer incl. 64 guard ints, offsets, status, needed, cap)"""
    from s2d_b200 import _lib
    offs = np.zeros(len(blobs) + 1, np.int64)
    offs[1:] = np.cumsum([len(b) for b in blobs])
    chars = _dev(np.frombuffer(b"".join(blobs) + b"\0", np.uint8).copy())
    cap = int(offs[-1]) if capacity is None else capacity
    n = C.c_int64()
    _lib.call("s2d_rle_from_strings_work_ints", len(blobs), int(offs[-1]), C.byref(n))
    work = torch.empty(n.value, dtype=torch.int32, device=DEV)
    counts = torch.full((cap + 64,), guard, dtype=torch.int32, device=DEV)
    coff = torch.full((len(blobs) + 1,), -1, dtype=torch.int64, device=DEV)
    status = torch.full((len(blobs),), -1, dtype=torch.int32, device=DEV)
    need = torch.full((1,), -1, dtype=torch.int64, device=DEV)
    d_off = _dev(offs)
    _lib.call("s2d_rle_from_strings", chars.data_ptr(), d_off.data_ptr(), len(blobs), work.data_ptr(), cap,
              counts.data_ptr(), coff.data_ptr(), status.data_ptr(), need.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return counts.cpu().numpy(), coff.cpu().numpy(), status.cpu().numpy(), int(need.item()), cap


def _edge_strings(rng):
    lists = [[], [0], [5], [0, 7], [3, 4, 5], [2 ** 31 - 1], [0, 2 ** 31 - 1, 2 ** 31 - 1, 1],
             [2 ** 30 + 12345, 2 ** 31 - 2, 17, 2 ** 31 - 1]]               # 7-character values
    lists += [rng.integers(0, 3000, size=rng.integers(0, 400)).tolist() for _ in range(300)]
    lists += [rng.integers(0, 2 ** 31 - 1, size=rng.integers(1, 60)).tolist() for _ in range(40)]
    return lists


def test_parse_equals_from_string():
    rng = np.random.default_rng(0)
    lists = _edge_strings(rng)
    long = rng.integers(0, 2 ** 31 - 1, size=190_000).tolist()                # > 10^6 characters
    lists.insert(150, long)
    blobs = [coco_rle.to_string(x).encode() for x in lists]
    assert max(len(b) for b in blobs) > 10 ** 6
    counts, coff, status, need, cap = _parse_cabi(blobs)
    assert need == coff[-1] == sum(len(x) for x in lists) and (status == 0).all()
    for i, x in enumerate(lists):
        assert counts[coff[i]:coff[i + 1]].tolist() == x == coco_rle.from_string(blobs[i].decode()), i
    assert (counts[cap:] == -77).all()
    # the public call returns the same on the device
    c2, o2, s2 = coco_rle.counts_from_strings_device(blobs[:20] + [b.decode() for b in blobs[20:40]])
    o2 = o2.cpu().numpy()
    assert (s2.cpu().numpy() == 0).all() and np.array_equal(o2, coff[:41] - coff[0])
    assert np.array_equal(c2.cpu().numpy()[:o2[-1]], counts[:coff[40]])


@pytest.mark.parametrize("n", [1, 31, 1023, 1024, 1025, 2048, 2049, 5000])
def test_parse_offsets_across_scan_blocks(n):
    """count_offsets of n strings, n on both sides of the 1024-element steps of the single-CTA offsets scan"""
    rng = np.random.default_rng(n)
    lists = [rng.integers(0, 3000, size=rng.integers(0, 40)).tolist() for _ in range(n)]
    blobs = [coco_rle.to_string(x).encode() for x in lists]
    counts, coff, status, need, _ = _parse_cabi(blobs)
    want = np.zeros(n + 1, np.int64)
    want[1:] = np.cumsum([len(x) for x in lists])
    assert np.array_equal(coff, want) and need == coff[-1] and (status == 0).all()


def test_parse_flags_malformed_without_disturbing_neighbours():
    rng = np.random.default_rng(1)
    good = [rng.integers(0, 3000, size=rng.integers(1, 200)).tolist() for _ in range(64)]
    blobs = [coco_rle.to_string(x).encode() for x in good]
    bad = {3: blobs[3] + b"P", 10: b"\x2f", 17: coco_rle.to_string([5, -3]).encode(),
           22: coco_rle.to_string([5, 2 ** 31]).encode(), 30: coco_rle.to_string([1, 5, 3, 2 ** 31 + 4]).encode(),
           41: b"P" * 14 + b"1", 50: b"o" * 14 + b"?"}
    for i, b in bad.items():
        blobs[i] = b
    counts, coff, status, need, _ = _parse_cabi(blobs)
    assert sorted(np.nonzero(status)[0].tolist()) == sorted(bad) and set(status.tolist()) == {0, 1}
    for i, x in enumerate(good):
        if i not in bad:
            assert counts[coff[i]:coff[i + 1]].tolist() == x
    # a string of values outside '0'..'o' that is well formed: byte - 48 as from_string computes for ASCII
    s = bytes([48 + 5, 40, 10, 126 - 32, 48 + 7])
    counts, coff, status, _, _ = _parse_cabi([s])
    want = coco_rle.from_string(s.decode())
    assert status[0] == int(any(not 0 <= x < 2 ** 31 for x in want))
    if status[0] == 0:
        assert counts[:coff[1]].tolist() == want


def test_parse_short_capacity_reports_need():
    rng = np.random.default_rng(2)
    lists = _edge_strings(rng)[:120]
    blobs = [coco_rle.to_string(x).encode() for x in lists]
    full, coff_full, _, need_full, _ = _parse_cabi(blobs)
    for cap in (0, 1, need_full // 2, need_full - 1):
        counts, coff, status, need, _ = _parse_cabi(blobs, capacity=cap, guard=-99)
        assert need == need_full and np.array_equal(coff, coff_full) and (status == 0).all()
        assert np.array_equal(counts[:cap], full[:cap]) and (counts[cap:] == -99).all()


def _checker(h, w):
    return (np.add.outer(np.arange(h), np.arange(w)) % 2).astype(bool)


def _blob(rng, h, w):
    yy, xx = np.ogrid[:h, :w]
    m = np.zeros((h, w), bool)
    for _ in range(4):
        cy, cx, r = rng.integers(0, h), rng.integers(0, w), rng.integers(1, max(2, min(h, w) // 3))
        m |= (yy - cy) ** 2 + (xx - cx) ** 2 < r * r
    return m


def _masks(h, w, rng):
    p = np.zeros((h, w), bool)
    p[0, 0] = True
    return [np.zeros((h, w), bool), np.ones((h, w), bool), p, _checker(h, w), _blob(rng, h, w), _blob(rng, h, w)]


@pytest.mark.parametrize("shape", [(1, 1), (1, 333), (333, 1), (7, 13), (37, 91), (129, 257), (480, 854), (720, 1280),
                                   (1080, 1920), (1920, 1080)])
def test_decode_equals_oracle(shape):
    h, w = shape
    rng = np.random.default_rng(h + 7 * w)
    masks = _masks(h, w, rng)
    rles = [{"size": [h, w], "counts": coco_rle.to_string(oc.counts(m)) if k != 3 or h * w < 10 ** 5 else oc.counts(m)}
            for k, m in enumerate(masks)]
    got = coco_rle.decode_batch(rles).cpu().numpy()
    assert got.shape == (len(masks), h, w)
    for k, m in enumerate(masks):
        cnts = oc.counts(m)
        want = oc.decode(cnts, h, w) if len(cnts) < 10 ** 5 else m.astype(np.uint8)
        assert np.array_equal(want, m) and np.array_equal(got[k], want), k
    single = coco_rle.decode_batch(rles[4])
    assert single.shape == (h, w) and np.array_equal(single.cpu().numpy(), masks[4])


def _decode_cabi(cnt_lists, sizes, out_offsets, nbytes, sentinel=0xC3):
    from s2d_b200 import _lib
    offs = np.zeros(len(cnt_lists) + 1, np.int64)
    offs[1:] = np.cumsum([len(x) for x in cnt_lists])
    counts = _dev(np.concatenate([np.asarray(x, np.int64) for x in cnt_lists] + [np.zeros(1, np.int64)]).astype(np.int32))
    n = C.c_int64()
    _lib.call("s2d_rle_decode_work_ints", len(cnt_lists), int(offs[-1]), C.byref(n))
    work = torch.empty(n.value, dtype=torch.int32, device=DEV)
    out = torch.full((nbytes,), sentinel, dtype=torch.uint8, device=DEV)
    status = torch.zeros(len(cnt_lists), dtype=torch.int32, device=DEV)
    sz = np.asarray(sizes, np.int32)
    hs, ws, oo, d_off = _dev(sz[:, 0]), _dev(sz[:, 1]), _dev(np.asarray(out_offsets, np.int64)), _dev(offs)
    _lib.call("s2d_rle_decode", counts.data_ptr(), d_off.data_ptr(), len(cnt_lists), hs.data_ptr(), ws.data_ptr(),
              oo.data_ptr(), work.data_ptr(), out.data_ptr(), status.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return out.cpu().numpy(), status.cpu().numpy()


def test_decode_mixed_sizes_gaps_and_wrong_sums():
    rng = np.random.default_rng(3)
    sizes = [(37, 91), (1, 1), (720, 1280), (5, 300), (129, 257), (64, 128), (33, 17), (200, 77)]
    masks = [_blob(rng, h, w) for h, w in sizes]
    lists = [oc.counts(m) for m in masks]
    # 5: runs that stop short of H * W; 6: runs past H * W; 7: one huge run
    lists[5] = lists[5][:-1] if len(lists[5]) > 1 else [10]
    lists[6] = lists[6] + [500, 40]
    lists[7] = [3, 2 ** 31 - 1]
    offsets, pos = [], 29                                              # unaligned start, gaps of odd sizes
    for h, w in sizes:
        offsets.append(pos)
        pos += h * w + 13
    out, status = _decode_cabi(lists, sizes, offsets, pos + 64)
    assert status.tolist() == [0, 0, 0, 0, 0, 2, 2, 2]
    covered = np.zeros(len(out), bool)
    for k, ((h, w), o) in enumerate(zip(sizes, offsets)):
        if k == 7:
            flat = np.zeros(h * w, np.uint8)
            flat[3:] = 1
            want = flat.reshape((h, w), order="F")
        else:
            want = oc.decode(lists[k], h, w)
        assert np.array_equal(out[o:o + h * w].reshape(h, w), want), k
        covered[o:o + h * w] = True
    assert (out[~covered] == 0xC3).all()


def test_decode_batch_errors_and_status():
    m = np.zeros((10, 12), bool)
    m[2:5, 3:7] = True
    ok = {"size": [10, 12], "counts": coco_rle.to_string(oc.counts(m))}
    with pytest.raises(ValueError, match="different sizes"):
        coco_rle.decode_batch([ok, {"size": [12, 10], "counts": ok["counts"]}])
    with pytest.raises(ValueError, match="segmentation 2: malformed"):
        coco_rle.decode_batch([ok, ok, {"size": [10, 12], "counts": ok["counts"] + "P"}])
    with pytest.raises(ValueError, match="segmentation 1: runs do not sum"):
        coco_rle.decode_batch([ok, {"size": [10, 12], "counts": [5, 5]}])
    with pytest.raises(ValueError, match="outside"):
        coco_rle.decode_batch([{"size": [10, 12], "counts": [5, -5]}])
    masks, status = coco_rle.decode_batch([ok, {"size": [10, 12], "counts": ok["counts"].encode() + b"P"},
                                           {"size": [10, 12], "counts": oc.counts(m)}, {"size": [10, 12], "counts": [7]}],
                                          check=False)
    assert status.cpu().tolist() == [0, 1, 0, 2]
    assert np.array_equal(masks[0].cpu().numpy(), m) and np.array_equal(masks[2].cpu().numpy(), m)


def test_encode_then_decode_round_trip():
    rng = np.random.default_rng(4)
    masks = np.stack([_blob(rng, 96, 160) for _ in range(40)] + [np.zeros((96, 160), bool), _checker(96, 160)])
    enc = coco_rle.encode_batch(masks)
    got = coco_rle.decode_batch([r for r, _, _ in enc]).cpu().numpy()
    assert np.array_equal(got, masks.astype(np.uint8))


def _check_video(anns, labels):
    """every non-null frame of every annotation is labels[f] == v, v the label under its first set pixel; area and box as
    the json has them; null frames zero"""
    masks = decode_video_annotations(anns)
    if isinstance(anns, (bytes, bytearray)):
        anns = json.loads(anns)
    A, T = len(anns), labels.shape[0]
    assert masks.shape == (A, T) + tuple(labels.shape[1:])
    lab = labels.to(DEV) if torch.is_tensor(labels) else _dev(labels)
    for a, ann in enumerate(anns):
        for t, seg in enumerate(ann["segmentations"]):
            m = masks[a, t]
            if seg is None:
                assert not m.any()
                continue
            first = int(torch.argmax(m.reshape(-1)))
            assert m.reshape(-1)[first] == 1
            v = lab[t].reshape(-1)[first]
            assert torch.equal(m.bool(), lab[t] == v), (a, t)
            assert int(m.sum()) == ann["areas"][t]
            ys, xs = torch.nonzero(m.any(dim=1)).reshape(-1), torch.nonzero(m.any(dim=0)).reshape(-1)
            assert ann["bboxes"][t] == [float(xs[0]), float(ys[0]), float(xs[-1] - xs[0] + 1), float(ys[-1] - ys[0] + 1)]
    return masks


def _golden_batch(names):
    from s2d_b200.pipeline import Batch, Params, VideoInput
    vids = []
    for n in names:
        _, labels, tracks, vis = load_golden(n)
        vids.append(VideoInput(*(torch.from_numpy(x).to(DEV) for x in (labels, tracks, vis)), name=n))
    g = load_golden(names[0])[0]
    b = Batch(vids, stages="LVBDE")
    b.run(Params(g["visibility_threshold"], g["matching_threshold"]))
    return b


@pytest.mark.parametrize("case", GOLDEN_CASES)
def test_stage_e_json_decodes_to_label_maps_golden(case):
    b = _golden_batch([case])
    text = b.annotation_json()[0]
    if text is None:
        pytest.skip(f"{case}: status is not 1, no annotations")
    labels = load_golden(case)[1]
    _check_video(text, labels)
    assert torch.equal(decode_video_annotations(b.annotations()[0]), decode_video_annotations(text))


def test_stage_e_json_decodes_mixed_status():
    thr = lambda n: (load_golden(n)[0]["visibility_threshold"], load_golden(n)[0]["matching_threshold"])
    by_thr = {}
    for n in GOLDEN_CASES:
        by_thr.setdefault(thr(n), []).append(n)
    names = max(by_thr.values(), key=lambda ns: len({load_golden(n)[0]["status"] == 1 for n in ns}) * 100 + len(ns))
    b = _golden_batch(names)
    texts = b.annotation_json()
    assert any(t is None for t in texts) and any(texts)
    for n, t in zip(names, texts):
        if t is not None:
            _check_video(t, load_golden(n)[1])


@pytest.mark.parametrize("order", ["raster", "random"])
def test_stage_e_json_decodes_c2_shape(order):
    from s2d_b200.pipeline import Batch, Params, VideoInput
    from s2d_b200.synth import make_scene_device
    sc = make_scene_device(2024, 36, 720, 1280, 20, 4096, torch.device(DEV), point_order=order)
    b = Batch([VideoInput(sc["labels"], sc["tracks"], sc["vis"])], stages="LVBDE")
    b.run(Params())
    text = b.annotation_json()[0]
    assert text and text != b"[]"
    masks = _check_video(text, sc["labels"])
    assert masks.sum() > 0


def test_graph_capture_replays_same_bytes():
    from s2d_b200 import _lib
    rng = np.random.default_rng(5)
    h, w = 180, 333
    masks = [_blob(rng, h, w) for _ in range(24)]
    blobs = [coco_rle.to_string(oc.counts(m)).encode() for m in masks]
    n = len(blobs)
    offs = np.zeros(n + 1, np.int64)
    offs[1:] = np.cumsum([len(b) for b in blobs])
    chars, d_off = _dev(np.frombuffer(b"".join(blobs), np.uint8).copy()), _dev(offs)
    nw = C.c_int64()
    _lib.call("s2d_rle_from_strings_work_ints", n, int(offs[-1]), C.byref(nw))
    pwork = torch.empty(nw.value, dtype=torch.int32, device=DEV)
    _lib.call("s2d_rle_decode_work_ints", n, int(offs[-1]), C.byref(nw))
    dwork = torch.empty(nw.value, dtype=torch.int32, device=DEV)
    counts = torch.empty(int(offs[-1]), dtype=torch.int32, device=DEV)
    coff = torch.empty(n + 1, dtype=torch.int64, device=DEV)
    status = torch.empty(n, dtype=torch.int32, device=DEV)
    need = torch.empty(1, dtype=torch.int64, device=DEV)
    hs, ws = torch.full((n,), h, dtype=torch.int32, device=DEV), torch.full((n,), w, dtype=torch.int32, device=DEV)
    oo = torch.arange(n, dtype=torch.int64, device=DEV) * h * w
    out = torch.zeros((n, h, w), dtype=torch.uint8, device=DEV)

    def run():
        st = torch.cuda.current_stream().cuda_stream
        _lib.call("s2d_rle_from_strings", chars.data_ptr(), d_off.data_ptr(), n, pwork.data_ptr(), counts.numel(),
                  counts.data_ptr(), coff.data_ptr(), status.data_ptr(), need.data_ptr(), st)
        _lib.call("s2d_rle_decode", counts.data_ptr(), coff.data_ptr(), n, hs.data_ptr(), ws.data_ptr(), oo.data_ptr(),
                  dwork.data_ptr(), out.data_ptr(), status.data_ptr(), st)

    run()
    torch.cuda.synchronize()
    direct = out.clone()
    assert np.array_equal(direct.cpu().numpy(), np.stack(masks)) and not status.any()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        run()
    out.fill_(7)
    counts.fill_(-1)
    status.fill_(-1)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, direct) and not status.any()
