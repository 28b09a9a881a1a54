"""Stage E on the device (s2d_label_rle, s2d_rle_strings, Batch.annotations, discover_keymasks(annotations=True))
against the restatement of maskApi.c, the reference's stage-D folder tree (goldens) and the file-based drop-in."""
import json
import os
import re

import numpy as np
import pytest
import torch

from oracle import coco_rle as cr
from tests.conftest import GOLDEN_CASES, load_golden

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _maps(H, W, seed):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    blobs = np.zeros((H, W), np.uint8)
    for l in range(1, 13):
        cy, cx = rng.uniform(0, H), rng.uniform(0, W)
        ry, rx = rng.uniform(1, max(2, H / 3)), rng.uniform(1, max(2, W / 3))
        blobs[((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 <= 1] = l
    corners = np.zeros((H, W), np.uint8)
    corners[0, 0] = 3
    corners[-1, -1] = 9
    nearly_full = np.full((H, W), 7, np.uint8)
    nearly_full[H // 2, W // 2] = 0
    l255 = np.where(blobs > 0, 255, 0).astype(np.uint8)
    l255[blobs == 1] = 254
    return [blobs, rng.integers(0, 256, size=(H, W)).astype(np.uint8), np.full((H, W), 7, np.uint8), nearly_full,
            np.zeros((H, W), np.uint8), l255, corners]


def _label_batch(label_list, capacity=None):
    """A stage-E batch over label maps only: K0 enumerates the rows, every video is given final status 1."""
    from s2d_b200 import _lib
    from s2d_b200.pipeline import Batch, VideoInput
    vids = []
    for lab in label_list:
        T, H, W = lab.shape
        nm = 0
        for t in range(T):
            nm += max(0, len(np.unique(lab[t])) - 1)
        vids.append(VideoInput(labels=torch.from_numpy(np.ascontiguousarray(lab)).to(DEV), dims={"Nm": max(1, nm), "P": 2}))
    b = Batch(vids, stages="LDE")
    if capacity is not None:
        b._alloc_rle(*capacity)
    b.run(stages="L")
    for i in range(len(vids)):
        b.vidinfo[i * _lib.S2D_VIDINFO_WORDS + 3] = 1
    b.run(stages="E")
    return b


def _check_rows(b, label_list, tab):
    from s2d_b200.keymask_ident.annotations import coco_rle
    gid_of = b.gid_of.cpu().numpy().reshape(-1, 256)
    area = b.area.cpu().numpy().reshape(-1, 256)
    offs, counts, bbox, soff, chars = tab["offsets"], tab["counts"], tab["bbox"], tab["str_off"], tab["chars"]
    nrows = 0
    for vi, lab in enumerate(label_list):
        d = b.host_descs[vi]
        T, H, W = lab.shape
        for t in range(T):
            present = np.unique(lab[t])
            for l in range(256):
                g = int(gid_of[d.frame0 + t, l])
                assert (g >= 0) == (l in present[1:]), (t, l, g)
                if g < 0:
                    continue
                r = d.row0 + g
                m = lab[t] == l
                c = counts[offs[r]:offs[r + 1]].tolist()
                assert c == cr.counts(m), (vi, t, l)
                assert np.array_equal(cr.decode(c, H, W), m.astype(np.uint8))
                x0, y0, x1, y1 = (int(v) for v in bbox[r])
                assert [float(x0), float(y0), float(x1 - x0 + 1), float(y1 - y0 + 1)] == cr.bbox(m)
                assert int(area[d.frame0 + t, l]) == cr.area(m)
                assert chars[soff[r]:soff[r + 1]] == coco_rle.to_string(c)
                nrows += 1
    return nrows


@pytest.mark.parametrize("H,W", [(1, 1), (31, 33), (97, 131), (480, 854), (720, 1280), (1080, 1920)])
def test_label_rle_vs_restatement(H, W):
    lab = np.stack(_maps(H, W, H * 7 + W))
    b = _label_batch([lab])
    tab = b.rle_tables(counts=True)
    assert _check_rows(b, [lab], tab) > 0 or H * W == 1


def test_overflow_reports_need_and_batch_retries():
    """A capacity below the need: the device reports the need, nothing at or past the capacity changes; the batch's
    retry (rle_tables) grows the buffers and gives the right tables. Per-pixel random labels: ~2 edges per pixel."""
    rng = np.random.default_rng(11)
    labs = [rng.integers(0, 256, size=(3, 64, 96)).astype(np.uint8), np.stack(_maps(45, 77, 3))]
    b = _label_batch(labs, capacity=(1000, 500))
    cnt_pad, chr_pad = torch.full((1000 + 4096,), -7, dtype=torch.int32, device=DEV), torch.full((500 + 4096,), 0x5A, dtype=torch.uint8, device=DEV)
    b.rle_counts, b.rle_chars = cnt_pad, chr_pad          # capacities stay 1000 / 500: the tails must stay untouched
    b.run(stages="E")
    torch.cuda.synchronize()
    need = b.rle_need.cpu().tolist()
    assert need[0] > 2 * 3 * 64 * 96 and need[1] > 0
    assert (cnt_pad[1000:] == -7).all() and (chr_pad[500:] == 0x5A).all()
    assert b.rle_off.cpu().numpy()[-1] == need[0]
    tab = b.rle_tables(counts=True)
    assert b.rle_cap >= need[0]
    rows = sum(len(np.unique(lab[t])) - 1 for lab in labs for t in range(lab.shape[0]))
    assert _check_rows(b, labs, tab) == rows


@pytest.mark.parametrize("n", [1, 31, 1023, 1024, 1025, 2048, 2049, 5000])
def test_rle_strings_offsets_across_scan_blocks(n):
    """s2d_rle_strings of n run-length lists, n on both sides of the 1024-element steps of the single-CTA offsets scan"""
    from s2d_b200 import _lib
    from s2d_b200.keymask_ident.annotations import coco_rle
    rng = np.random.default_rng(n)
    lists = [rng.integers(0, 5000, size=rng.integers(1, 40)).tolist() for _ in range(n)]
    strings = [coco_rle.to_string(x) for x in lists]
    offs = np.zeros(n + 1, np.int64)
    offs[1:] = np.cumsum([len(x) for x in lists])
    want = np.zeros(n + 1, np.int64)
    want[1:] = np.cumsum([len(s) for s in strings])
    counts = torch.from_numpy(np.concatenate(lists).astype(np.int32)).to(DEV)
    d_off = torch.from_numpy(offs).to(DEV)
    work = torch.empty(n, dtype=torch.int32, device=DEV)
    chars = torch.empty(int(want[-1]), dtype=torch.uint8, device=DEV)
    soff = torch.full((n + 1,), -1, dtype=torch.int64, device=DEV)
    need = torch.full((1,), -1, dtype=torch.int64, device=DEV)
    _lib.call("s2d_rle_strings", counts.data_ptr(), d_off.data_ptr(), n, int(offs[-1]), work.data_ptr(), int(want[-1]),
              chars.data_ptr(), soff.data_ptr(), need.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert np.array_equal(soff.cpu().numpy(), want) and int(need.item()) == want[-1]
    assert chars.cpu().numpy().tobytes().decode("ascii") == "".join(strings)


def _groups_from_files(files):
    """(cluster, group) -> {frame: largest mask id} from the reference's group_files (tie rule of the batched path)."""
    out = {}
    for f in files:
        c, g, name = f.split("/")
        fr, m = (int(x) for x in re.match(r"frame(\d+)_mask(\d+)\.png", name).groups())
        d = out.setdefault((c, g), {})
        d[fr] = max(d.get(fr, -1), m)
    return out


def _run_golden(names):
    from s2d_b200.pipeline import Params, VideoInput, discover_keymasks
    vids, gs = [], []
    for n in names:
        g, labels, tracks, vis = load_golden(n)
        vids.append(VideoInput(torch.from_numpy(labels).to(DEV), torch.from_numpy(tracks).to(DEV), torch.from_numpy(vis).to(DEV), name=n))
        gs.append((g, labels))
    p = Params(gs[0][0]["visibility_threshold"], gs[0][0]["matching_threshold"])
    return discover_keymasks(vids, p, want_comps=False, annotations=True), gs


@pytest.mark.parametrize("case", GOLDEN_CASES)
def test_membership_equals_reference_group_files(case):
    (res,), ((g, labels),) = _run_golden([case])
    if g["status"] != 1:
        assert res["annotations"] is None
        return
    want = _groups_from_files(g["group_files"])
    order = sorted(want)                                   # cluster_*, then group_*: lexicographic, like the reference
    anns = res["annotations"]
    assert [a["id"] for a in anns] == list(range(1, len(anns) + 1)) and len(anns) == len(order)
    T, H, W = labels.shape
    for a, key in zip(anns, order):
        got = {}
        for f, seg in enumerate(a["segmentations"]):
            if seg is None:
                assert a["areas"][f] is None and a["bboxes"][f] is None
                continue
            m = cr.decode(cr_from(seg["counts"]), H, W).astype(bool)
            vals = np.unique(labels[f][m])
            assert len(vals) == 1 and np.array_equal(m, labels[f] == vals[0])
            got[f] = int(vals[0])
            assert a["areas"][f] == int(m.sum()) and a["bboxes"][f] == cr.bbox(m)
        assert got == want[key], (case, key)
        assert a["visibility_ranges"] == next(c["ranges"] for c in g["clusters"] if f"cluster_{c['cluster_id']}" == key[0])


def cr_from(s):
    from s2d_b200.keymask_ident.annotations import coco_rle
    return coco_rle.from_string(s)


@pytest.mark.parametrize("case", [c for c in GOLDEN_CASES if load_golden(c)[0]["status"] == 1])
def test_equals_dropin_json(case, tmp_path, monkeypatch):
    """discover_keymasks(annotations=True) + write_video_annotations writes json-for-json what the drop-in's stage E
    writes after its stages A-D on the same video, with group folders listed in ascending mask-id order (the batched
    path's tie rule)."""
    from s2d_b200.keymask_ident import (_engine, annotations as ann, cotracker_matching, cotracker_occlusions, crw_utils,
                                       identify_visibility_windows, keymask_utils)
    from tests.test_dropin_gpu import _Model, _Replay, _write_video
    g, labels, tracks, vis = load_golden(case)
    root = str(tmp_path)
    vdir, mdir = _write_video(root, labels)
    rp = _Replay(labels, tracks, vis)
    _engine.set_tracker_factory(lambda checkpoint=None: _Model(rp))
    _engine._label_cache.clear()
    real_listdir = os.listdir

    def by_mask(p):
        def key(f):
            m = re.search(r"mask(\d+)", f)
            return (int(m.group(1)) if m else -1, f)
        return sorted(real_listdir(p), key=key)

    class _Os:
        def __getattr__(self, k):
            return by_mask if k == "listdir" else getattr(os, k)
    try:
        vm, vc, save = os.path.join(root, "vm"), os.path.join(root, "vc"), os.path.join(root, "seg")
        a = cotracker_occlusions.extract_object_visibility_data(vdir, mdir, os.path.join(root, "videos"), vm, False)
        w = identify_visibility_windows.get_visibility_windows_for_video(a, "ytvis2021", "train", "vid0", vc,
                                                                         g["visibility_threshold"], False)
        imgs, imgs_orig, lbls, meta = crw_utils.load_frames_and_masks(vdir, mdir, w, "ytvis2021")
        cm = keymask_utils.save_segmentation_masks(imgs, imgs_orig, lbls, meta, save, False)
        assert cotracker_matching.temporal_correspondence_match(vdir, mdir, cm, vm, vc, g["matching_threshold"], False) == 1
        monkeypatch.setattr(ann, "os", _Os())
        ann.write_annotation_for_video(vdir, cm, os.path.join(root, "dropin"), w)
        monkeypatch.undo()
    finally:
        _engine.set_tracker_factory(None)
    (res,), _ = _run_golden([case])
    ann.write_video_annotations(vdir, res["annotations"], os.path.join(root, "batched"))
    with open(os.path.join(root, "dropin", "vid0.json")) as f:
        want = json.load(f)
    with open(os.path.join(root, "batched", "vid0.json")) as f:
        got = json.load(f)
    assert got == want


def test_c2_shape_keymasks_decode_to_label_masks():
    from s2d_b200.pipeline import Params, VideoInput, discover_keymasks
    from s2d_b200.synth import make_scene_device
    vids, labs = [], []
    for order in ("raster", "random"):
        sc = make_scene_device(2024, 36, 720, 1280, 20, 4096, torch.device(DEV), point_order=order)
        vids.append(VideoInput(sc["labels"], sc["tracks"], sc["vis"]))
        labs.append(sc["labels"].cpu().numpy())
    res = discover_keymasks(vids, Params(), want_comps=False, annotations=True)
    nseg = 0
    for r, lab in zip(res, labs):
        assert r["status"] == 1 and r["annotations"]
        T, H, W = lab.shape
        for a in r["annotations"]:
            assert (a["height"], a["width"], a["length"]) == (H, W, T)
            for f, seg in enumerate(a["segmentations"]):
                if seg is None:
                    continue
                m = cr.decode(cr_from(seg["counts"]), H, W).astype(bool)
                v = lab[f][m]
                assert v.size and (v == v[0]).all() and np.array_equal(m, lab[f] == v[0])
                assert a["areas"][f] == int(m.sum()) and a["bboxes"][f] == cr.bbox(m)
                nseg += 1
    assert nseg > 100


def test_graph_replay_and_batch_invariance():
    from s2d_b200.pipeline import Batch, Params, VideoInput
    ok = [c for c in GOLDEN_CASES if load_golden(c)[0]["status"] == 1]
    thr = lambda n: (load_golden(n)[0]["visibility_threshold"], load_golden(n)[0]["matching_threshold"])
    names = [c for c in ok if thr(c) == thr(ok[0])][:3]
    gl = {n: load_golden(n) for n in names}
    mk = lambda n: VideoInput(*(torch.from_numpy(x).to(DEV) for x in gl[n][1:]), name=n)
    p = Params(gl[names[0]][0]["visibility_threshold"], gl[names[0]][0]["matching_threshold"])
    assert len(names) >= 2
    alone = []
    for n in names:
        b = Batch([mk(n)], stages="LVBDE")
        b.run(p)
        alone.append(b.annotations()[0])
    b = Batch([mk(n) for n in names], stages="LVBDE")
    b.run(p)
    direct = b.annotations()
    assert direct == alone
    b.capture(p)
    torch.cuda.synchronize()
    for x in (b.rle_counts, b.rle_chars, b.rle_bbox):
        x.fill_(0x11)
    b.replay()
    assert b.annotations() == direct
    # stage E is enqueued only when asked for: the default step launches what it launched before
    d = Batch([mk(n) for n in names])
    assert d.stages == "LVBD" and d.rle_counts is None
    n_default = d.run(p)
    assert b.run(p, stages="LVBD") == n_default and b.run(p) == n_default + 8
