"""Annotation json on the device (s2d_annotation_json, Batch.annotation_json, HostPipeline(annotations="json")) against
json.dumps of the annotation lists of the Python route (Batch.annotations, tests/annotation_reference.py)."""
import ctypes as C
import dataclasses
import json

import numpy as np
import pytest
import torch

from tests.annotation_reference import reference, synthetic_batch
from tests.conftest import GOLDEN_CASES, load_golden
from tests.test_annotation_layout_gpu import _golden_video, _grow, _host_videos, _scenes

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _dumps(anns):
    return [None if a is None else json.dumps(a).encode() for a in anns]


@pytest.mark.parametrize("case", GOLDEN_CASES)
def test_batch_json_equals_dumps_golden(case):
    from s2d_b200.pipeline import Batch, Params
    g = load_golden(case)[0]
    b = Batch([_golden_video(case)], stages="LVBDE")
    b.run(Params(g["visibility_threshold"], g["matching_threshold"]))
    got = b.annotation_json()
    assert got == _dumps(b.annotations())
    assert (got[0] is None) == (g["status"] != 1)


def test_batch_json_equals_dumps_mixed_status():
    from s2d_b200.pipeline import Batch, Params
    thr = lambda n: (load_golden(n)[0]["visibility_threshold"], load_golden(n)[0]["matching_threshold"])
    by_thr = {}
    for n in GOLDEN_CASES:
        by_thr.setdefault(thr(n), []).append(n)
    names = max(by_thr.values(), key=lambda ns: len({load_golden(n)[0]["status"] == 1 for n in ns}) * 100 + len(ns))
    b = Batch([_golden_video(n) for n in names], stages="LVBDE")
    b.run(Params(*thr(names[0])))
    got = b.annotation_json()
    assert got == _dumps(b.annotations())
    assert any(a is None for a in got) and any(a for a in got)


@pytest.mark.parametrize("order", ["raster", "random"])
def test_batch_json_equals_dumps_c2_shape(order):
    from s2d_b200.pipeline import Batch, Params, VideoInput
    from s2d_b200.synth import make_scene_device
    sc = make_scene_device(2024, 36, 720, 1280, 20, 4096, torch.device(DEV), point_order=order)
    b = Batch([VideoInput(sc["labels"], sc["tracks"], sc["vis"])], stages="LVBDE")
    b.run(Params())
    got = b.annotation_json()
    assert got[0] and got[0] != b"[]" and got == _dumps(b.annotations())


def _crafted_ties(t):
    """status-1 videos whose group sums hit one2x ties (1/8, 3/8, 5/8, 7/8, 1/200, m(2k+1) / 200m), and a status-1 video
    that gets no annotation (no row has a cluster)"""
    rng = np.random.default_rng(17)
    ties = [(1, 8), (3, 8), (5, 8), (7, 8), (1, 200), (3, 600), (5, 1000), (201, 200), (1001, 2000), (0, 7), (9, 0)]
    pick = rng.integers(0, len(ties), size=len(t.grp_n))
    t.grp_one2x = np.asarray([a for a, _ in ties], np.int32)[pick]
    t.grp_n = np.asarray([b for _, b in ties], np.int32)[pick]
    t.vidinfo[:, 3] = 1
    d = t.descs[0]
    t.rowinfo[d.row0:d.row0 + d.Nm, 0] = -1
    return t


def _run_cabi(t, capacity=None, sentinel=0x5A, layout_cap=None, beyond=None):
    """layout then json through the C ABI on synthetic tables; returns (needed, video_off, out buffer, capacity).
    layout_cap: the layout's string capacity (default: all strings fit); beyond: byte written into the layout's string
    buffer from layout_cap on, before the json call"""
    from s2d_b200 import _lib
    nv, R, F = len(t.descs), t.total_rows, t.total_frames
    descs = (_lib.VideoDesc * nv)()
    for i, d in enumerate(t.descs):
        x = descs[i]
        x.T, x.H, x.W, x.Nm, x.TW, x.row0, x.frame0, x.xbits_off = d.T, d.H, d.W, d.Nm, d.TW, d.row0, d.frame0, d.xbits_off
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    ddesc = dev(np.frombuffer(bytes(descs), np.uint8).copy())
    vidinfo = dev(t.vidinfo.reshape(-1))
    ins = [vidinfo, dev(t.rowinfo.reshape(-1)), dev(t.winbits), dev(t.rsbits), dev(t.rebits),
           dev(t.glabel), dev(t.qframe), dev(t.qlabel), dev(t.grp_n), dev(t.grp_one2x), dev(t.area.reshape(-1)),
           dev(t.gid_of.reshape(-1)), dev(t.bbox.reshape(-1)), dev(t.str_off),
           dev(np.frombuffer(t.chars.encode() + b"\0", np.uint8).copy())]
    n = C.c_int64()
    _lib.call("s2d_annotation_layout_work_ints", R, nv, C.byref(n))
    z = lambda k, dt=torch.int32: torch.full((k,), -7, dtype=dt, device=DEV)
    nchars = len(t.chars)
    o = dict(work=z(n.value), vann=z(2 * nv), ann=z(7 * R), members=z(6 * R), member_off=z(R, torch.int64),
             clusters=z(32 * nv), pairs=z(16 * (F + nv)), chars=torch.zeros(nchars + 64, dtype=torch.uint8, device=DEV),
             sizes=z(5, torch.int64))
    st = torch.cuda.current_stream().cuda_stream
    lcap = nchars if layout_cap is None else layout_cap
    _lib.call("s2d_annotation_layout", ddesc.data_ptr(), nv, R, *(x.data_ptr() for x in ins), nchars,
              o["work"].data_ptr(), o["vann"].data_ptr(), o["ann"].data_ptr(), o["members"].data_ptr(),
              o["member_off"].data_ptr(), o["clusters"].data_ptr(), o["pairs"].data_ptr(), lcap, o["chars"].data_ptr(),
              o["sizes"].data_ptr(), st)
    if beyond is not None:
        o["chars"][lcap:] = beyond
    _lib.call("s2d_annotation_json_work_ints", R, nv, C.byref(n))
    work = z(n.value)
    cap = 4 * nchars + 4096 * R if capacity is None else capacity
    out = torch.full((cap + 256,), sentinel, dtype=torch.uint8, device=DEV)
    voff, need = z(nv + 1, torch.int64), z(1, torch.int64)
    _lib.call("s2d_annotation_json", ddesc.data_ptr(), nv, R, vidinfo.data_ptr(), o["vann"].data_ptr(),
              o["ann"].data_ptr(), o["members"].data_ptr(), o["member_off"].data_ptr(), o["chars"].data_ptr(), lcap,
              o["clusters"].data_ptr(), o["pairs"].data_ptr(), o["sizes"].data_ptr(), work.data_ptr(), cap,
              out.data_ptr(), voff.data_ptr(), need.data_ptr(), st)
    torch.cuda.synchronize()
    return int(need.item()), voff.cpu().tolist(), out.cpu().numpy(), cap


@pytest.mark.parametrize("seed", range(5))
def test_json_kernel_on_synthetic_tables(seed):
    """escapes, one2x with gs > gn, failed videos; seed 3 adds a video of > 4096 rows, seed 4 crafted one2x ties and a
    status-1 video without annotation"""
    t = synthetic_batch(seed, nvideos=6)
    if seed == 3:
        t = _grow(t)
    if seed == 4:
        t = _crafted_ties(t)
    want = reference(t)
    need, off, out, cap = _run_cabi(t)
    assert need == off[-1] <= cap and (out[cap:] == 0x5A).all()
    got = [out[off[v]:off[v + 1]].tobytes() if off[v + 1] > off[v] else None for v in range(len(t.descs))]
    assert got == _dumps(want)
    if seed == 4:
        assert got[0] == b"[]"
        ones = {a["one2x"] for w in want for a in w}
        assert len(ones & {0.12, 0.38, 0.62, 0.88, 0.01}) >= 3 and ones & {1.0, 0.5}


def test_json_kernel_short_capacity_reports_need():
    t = synthetic_batch(2, nvideos=6)
    need_full, off_full, out_full, _ = _run_cabi(t)
    for cap in (0, 7, need_full // 3, need_full - 1):
        need, off, out, _ = _run_cabi(t, capacity=cap, sentinel=0xA5)
        assert need == need_full and off == off_full
        assert (out[cap:] == 0xA5).all()                           # nothing at or past the capacity
    assert need_full > 0


def test_json_kernel_reads_no_string_byte_past_the_layout_capacity():
    """Stage E short of string capacity: the layout reports more string bytes than its buffer holds (the caller re-runs
    stage E). The json call must read nothing from the layout's buffer at or past that capacity: bytes placed there, '~'
    (outside the RLE alphabet) or '\\' (which would lengthen the text), change neither the text nor its length."""
    t = synthetic_batch(2, nvideos=6)
    lcap = 64
    runs = [_run_cabi(t, layout_cap=lcap, beyond=b) for b in (ord("~"), ord("\\"), 0)]
    (need, off, out, cap), *others = runs
    assert need < _run_cabi(t)[0]                                  # the strings were cut at the capacity
    for n2, off2, out2, _ in others:
        assert n2 == need and off2 == off and (out2[:need] == out[:need]).all()
    assert b"~" not in out[:need].tobytes()


def _scene_batch():
    from s2d_b200.pipeline import Batch, VideoInput
    b = Batch([VideoInput(*(torch.from_numpy(x).to(DEV) for x in (sc.labels, sc.tracks, sc.vis))) for sc in _scenes()],
              stages="LVBDE")
    b.run()
    return b


def test_batch_json_short_capacity_reruns():
    b = _scene_batch()
    want = _dumps(b.annotations())
    assert any(want)
    b.aj_out, b.aj_cap = torch.full((16,), 0xA5, dtype=torch.uint8, device=DEV), 16
    assert b.annotation_json() == want
    assert b.aj_cap == sum(len(a) for a in want if a is not None)


def test_json_graph_capture_replays_same_bytes():
    b = _scene_batch()
    direct = b.annotation_json()                                       # settles every capacity first
    assert any(direct)
    n = b.aj_video_off[-1].item()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        b.layout()
        b.serialize()
    b.aj_out.fill_(0)
    b.aj_video_off.fill_(-1)
    g.replay()
    torch.cuda.synchronize()
    off = b.aj_video_off.cpu().tolist()
    text = b.aj_out[:n].cpu().numpy().tobytes()
    assert [text[off[v]:off[v + 1]] if off[v + 1] > off[v] else None for v in range(b.nv)] == direct


def _pipe_json(outs):
    return [a for o in outs for a in o["annotation_json"]]


@pytest.mark.parametrize("bits", [False, True])
def test_host_pipeline_json_equals_dumps(bits):
    from s2d_b200.hostpipe import HostPipeline
    hv = _host_videos(_scenes(), bits)
    lists = HostPipeline(hv[:2], DEV, chunk=2, annotations=True)
    want = _dumps([a for o in lists.run(hv) for a in o["annotations"]])
    assert any(want)
    pipe = HostPipeline(hv[:2], DEV, chunk=2, annotations="json")
    for _ in range(2):                                   # second run reuses the staging sets and host buffers
        outs = pipe.run(hv)
        assert _pipe_json(outs) == want
        assert all("annotations" not in o for o in outs)
    # launches: annotations=True plus the json call per chunk; copies: the used json bytes, offsets, sizes, tables
    assert pipe.reruns == 0 and lists.reruns == 0
    assert pipe.launches == lists.launches + 3 * 2
    tables = sum(o[k].numel() * o[k].element_size() for o in outs for k in HostPipeline.RESULT_TABLES)
    used = sum(len(a) for a in want if a is not None)
    assert pipe.d2h_bytes == tables + used + 2 * (8 * (2 + 1) + 8 * 3)


def test_host_pipeline_json_grows_and_reruns_short_capacity():
    """noisy label maps and tiny forced stage-E and json capacities: every first chunk on a staging set re-runs, and the
    json of all four chunks is right"""
    from s2d_b200.hostpipe import HostPipeline
    from s2d_b200.pipeline import Batch, VideoInput
    base = _scenes()[:2]
    scenes = []
    for c in range(4):
        for j, sc in enumerate(base):
            rng = np.random.default_rng(10 * c + j)
            lab = sc.labels.copy()
            for t in range(lab.shape[0]):
                present = np.unique(lab[t])[1:]
                bg = (lab[t] == 0) & (rng.random(lab[t].shape) < 0.5)
                lab[t][bg] = rng.choice(present, size=int(bg.sum()))
            scenes.append(dataclasses.replace(sc, labels=lab))
    want = []
    for sc in scenes:
        b = Batch([VideoInput(*(torch.from_numpy(x).to(DEV) for x in (sc.labels, sc.tracks, sc.vis)))], stages="LVBDE")
        b.run()
        want += _dumps(b.annotations())
    assert sum(a is not None for a in want) >= 4
    hv = _host_videos(scenes, False)
    pipe = HostPipeline(hv[:2], DEV, chunk=2, annotations="json")
    for _, b in pipe.sets:
        b._alloc_rle(64, 64)
        b.aj_out, b.aj_cap = torch.empty(64, dtype=torch.uint8, device=DEV), 64
    outs = pipe.run(hv)
    assert pipe.reruns >= 4
    assert _pipe_json(outs) == want


def test_discover_keymasks_json_and_file(tmp_path):
    from PIL import Image

    from s2d_b200.keymask_ident.annotations import write_video_annotations
    from s2d_b200.pipeline import VideoInput, discover_keymasks
    vs = [VideoInput(*(torch.from_numpy(x).to(DEV) for x in (sc.labels, sc.tracks, sc.vis))) for sc in _scenes()]
    lists = [r["annotations"] for r in discover_keymasks(vs, want_comps=False, annotations=True)]
    res = discover_keymasks(vs, want_comps=False, annotations="json")
    assert all("annotations" not in r for r in res)
    assert [r["annotation_json"] for r in res] == _dumps(lists)
    i = next(i for i, a in enumerate(lists) if a)
    lst, text = lists[i], res[i]["annotation_json"]
    vdir = tmp_path / "video_7"
    vdir.mkdir()
    for i in range(10):
        Image.fromarray(np.zeros((64, 96, 3), np.uint8)).save(vdir / f"{i:05d}.jpg")
    write_video_annotations(str(vdir), lst, str(tmp_path / "from_list"))
    write_video_annotations(str(vdir), text, str(tmp_path / "from_bytes"))
    a = (tmp_path / "from_list" / "video_7.json").read_bytes()
    assert a == (tmp_path / "from_bytes" / "video_7.json").read_bytes() and json.loads(a)["annotations"] == lst
