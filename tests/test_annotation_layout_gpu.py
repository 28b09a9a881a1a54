"""Annotation layout on the device (s2d_annotation_layout, Batch.annotations, HostPipeline(annotations=True)) against
the frozen Python assembly it replaced (tests/annotation_reference.py) and the device-resident batch."""
import ctypes as C
import dataclasses

import numpy as np
import pytest
import torch

from tests.annotation_reference import frozen_annotations, reference, synthetic_batch
from tests.conftest import GOLDEN_CASES, load_golden

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _frozen(b):
    """the assembly before the device layout, on decode() + rle_tables() of the same step"""
    area = b.area.cpu().numpy().reshape(-1, 256)
    gid_of = b.gid_of.cpu().numpy().reshape(-1, 256)
    return frozen_annotations(b.decode(want_comps=False), b.rle_tables(), area, gid_of, b.host_descs)


def _golden_video(n):
    from s2d_b200.pipeline import VideoInput
    g, labels, tracks, vis = load_golden(n)
    return VideoInput(*(torch.from_numpy(x).to(DEV) for x in (labels, tracks, vis)), name=n)


@pytest.mark.parametrize("case", GOLDEN_CASES)
def test_batch_equals_frozen_assembly_golden(case):
    from s2d_b200.pipeline import Batch, Params
    g = load_golden(case)[0]
    b = Batch([_golden_video(case)], stages="LVBDE")
    b.run(Params(g["visibility_threshold"], g["matching_threshold"]))
    got = b.annotations()
    assert got == _frozen(b)
    assert (got[0] is None) == (g["status"] != 1)


def test_batch_equals_frozen_assembly_mixed_status():
    from s2d_b200.pipeline import Batch, Params
    thr = lambda n: (load_golden(n)[0]["visibility_threshold"], load_golden(n)[0]["matching_threshold"])
    by_thr = {}
    for n in GOLDEN_CASES:
        by_thr.setdefault(thr(n), []).append(n)
    names = max(by_thr.values(), key=lambda ns: len({load_golden(n)[0]["status"] == 1 for n in ns}) * 100 + len(ns))
    assert {load_golden(n)[0]["status"] == 1 for n in names} == {True, False}, "no threshold group mixes statuses"
    b = Batch([_golden_video(n) for n in names], stages="LVBDE")
    b.run(Params(*thr(names[0])))
    got = b.annotations()
    assert got == _frozen(b)
    assert any(a is None for a in got) and any(a for a in got)


@pytest.mark.parametrize("order", ["raster", "random"])
def test_batch_equals_frozen_assembly_c2_shape(order):
    from s2d_b200.pipeline import Batch, Params, VideoInput
    from s2d_b200.synth import make_scene_device
    sc = make_scene_device(2024, 36, 720, 1280, 20, 4096, torch.device(DEV), point_order=order)
    b = Batch([VideoInput(sc["labels"], sc["tracks"], sc["vis"])], stages="LVBDE")
    b.run(Params())
    got = b.annotations()
    assert got[0] and got == _frozen(b)


@pytest.mark.parametrize("seed", range(4))
def test_layout_kernel_on_synthetic_tables(seed):
    """ties, more than 10 groups, clusters without candidates, status other than 1, videos of more rows than the
    shared-memory sort holds"""
    from s2d_b200 import _lib
    from s2d_b200.pipeline import LAYOUT_TABLES, annotations_from_layout
    t = synthetic_batch(seed, nvideos=6)
    if seed == 3:                                            # a video of > 4096 rows sorts in global memory
        t = _grow(t)
    nv, R, F = len(t.descs), t.total_rows, t.total_frames
    descs = (_lib.VideoDesc * nv)()
    for i, d in enumerate(t.descs):
        x = descs[i]
        x.T, x.H, x.W, x.Nm, x.TW, x.row0, x.frame0, x.xbits_off = d.T, d.H, d.W, d.Nm, d.TW, d.row0, d.frame0, d.xbits_off
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    ddesc = dev(np.frombuffer(bytes(descs), np.uint8).copy())
    ins = [dev(t.vidinfo.reshape(-1)), dev(t.rowinfo.reshape(-1)), dev(t.winbits), dev(t.rsbits), dev(t.rebits),
           dev(t.glabel), dev(t.qframe), dev(t.qlabel), dev(t.grp_n), dev(t.grp_one2x), dev(t.area.reshape(-1)),
           dev(t.gid_of.reshape(-1)), dev(t.bbox.reshape(-1)), dev(t.str_off),
           dev(np.frombuffer(t.chars.encode() + b"\0", np.uint8).copy())]
    n = C.c_int64()
    _lib.call("s2d_annotation_layout_work_ints", R, nv, C.byref(n))
    z = lambda k, dt=torch.int32: torch.full((k,), -7, dtype=dt, device=DEV)
    nchars = len(t.chars)
    outs = dict(work=z(n.value), vann=z(2 * nv), ann=z(7 * R), members=z(6 * R), member_off=z(R, torch.int64),
                clusters=z(32 * nv), pairs=z(16 * (F + nv)), chars=torch.full((nchars + 64,), 0x5A, dtype=torch.uint8, device=DEV),
                sizes=z(5, torch.int64))
    o = outs
    _lib.call("s2d_annotation_layout", ddesc.data_ptr(), nv, R, *(x.data_ptr() for x in ins[:-1]), ins[-1].data_ptr(),
              nchars, o["work"].data_ptr(), o["vann"].data_ptr(), o["ann"].data_ptr(), o["members"].data_ptr(),
              o["member_off"].data_ptr(), o["clusters"].data_ptr(), o["pairs"].data_ptr(), nchars, o["chars"].data_ptr(),
              o["sizes"].data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    sizes = o["sizes"].cpu().tolist()
    assert sizes[2] <= nchars and (o["chars"][nchars:] == 0x5A).all()
    tabs = {"vann": o["vann"].cpu().numpy(),
            **{k: o[k][:w * sizes[i]].cpu().numpy() for k, (w, i) in LAYOUT_TABLES.items()}}
    assert annotations_from_layout(t.descs, t.vidinfo[:, 3], tabs) == reference(t)


def _grow(t):
    """append a status-1 video of 6000 rows (one cluster, 40 groups) to a synthetic batch"""
    from types import SimpleNamespace
    rng = np.random.default_rng(99)
    T, per = 750, 8
    Nm, TW = T * per, (T + 31) // 32
    d = SimpleNamespace(T=T, H=9, W=9, Nm=Nm, TW=TW, row0=t.total_rows, frame0=t.total_frames,
                        xbits_off=len(t.rsbits))
    gid = np.full((T, 256), -1, np.int32)
    qf, ql = np.repeat(np.arange(T), per).astype(np.int32), np.tile(np.arange(1, per + 1), T).astype(np.int32)
    gid[qf, ql] = np.arange(Nm)
    rs, re, wb = (np.zeros((Nm, TW), np.int32) for _ in range(3))
    rs[0, 0], re[0, 0] = 1, 2                                # cluster 0: one run [0, 1]
    wb[:, 0] = 1
    ri = np.zeros((Nm, 4), np.int32)
    ri[:, 1] = np.where(rng.random(Nm) < 0.3, 0, -1)
    gl = rng.integers(-1, 40, size=Nm).astype(np.int32)
    vid = np.zeros((1, 8), np.int32)
    vid[0, 0], vid[0, 3] = 1, 1
    lens = rng.integers(0, 20, size=Nm)
    so = t.str_off[-1] + np.cumsum(lens)
    extra = "".join(chr(48 + int(x)) for x in rng.integers(0, 64, size=int(lens.sum())))
    bb = np.tile(np.array([[1, 2, 3, 4]], np.int32), (Nm, 1))
    cat = np.concatenate
    return SimpleNamespace(
        descs=t.descs + [d], vidinfo=cat([t.vidinfo, vid]), rowinfo=cat([t.rowinfo, ri]), glabel=cat([t.glabel, gl]),
        qframe=cat([t.qframe, qf]), qlabel=cat([t.qlabel, ql]), rsbits=cat([t.rsbits, rs.reshape(-1)]),
        rebits=cat([t.rebits, re.reshape(-1)]), winbits=cat([t.winbits, wb.reshape(-1)]),
        grp_n=cat([t.grp_n[:16 * t.total_rows], rng.integers(0, 6, size=16 * Nm).astype(np.int32)]),
        grp_one2x=cat([t.grp_one2x[:16 * t.total_rows], rng.integers(0, 6, size=16 * Nm).astype(np.int32)]),
        gid_of=cat([t.gid_of, gid]), area=cat([t.area, rng.integers(1, 99, size=(T, 256)).astype(np.int32)]),
        bbox=cat([t.bbox, bb]), str_off=cat([t.str_off, so]), chars=t.chars + extra,
        total_rows=t.total_rows + Nm, total_frames=t.total_frames + T)


def _scenes():
    from s2d_b200.synth import make_scene
    shapes = [(12, 64, 96, 4, 64), (10, 48, 80, 3, 32), (12, 64, 96, 4, 64), (10, 48, 80, 3, 32)]   # slots 0 / 1 of two chunks
    scenes = [make_scene(300 + (i % 2), T, H, W, M, P) for i, (T, H, W, M, P) in enumerate(shapes)]
    scenes[2].tracks[:] = scenes[0].tracks[::-1].copy()
    scenes[3].tracks[:] = scenes[1].tracks + 0.25
    return scenes


def _resident(sc_list):
    from s2d_b200.pipeline import Batch, VideoInput
    out = []
    for sc in sc_list:
        b = Batch([VideoInput(*(torch.from_numpy(x).to(DEV) for x in (sc.labels, sc.tracks, sc.vis)))], stages="LVBDE")
        b.run()
        out.append(b.annotations()[0])
    return out


def _host_videos(sc_list, bits):
    from s2d_b200.hostpipe import HostVideo
    from s2d_b200.pipeline import pack_vis_bits
    hv = []
    for sc in sc_list:
        v = torch.from_numpy(sc.vis)
        hv.append(HostVideo(torch.from_numpy(sc.labels).pin_memory(), torch.from_numpy(sc.tracks).pin_memory(),
                            (pack_vis_bits(v) if bits else v).pin_memory(), vis_bits=bits))
    return hv


@pytest.mark.parametrize("bits", [False, True])
def test_host_pipeline_annotations_match_device_batch(bits):
    from s2d_b200.hostpipe import HostPipeline
    scenes = _scenes()
    want = _resident(scenes)
    assert any(a for a in want)
    hv = _host_videos(scenes, bits)
    pipe = HostPipeline(hv[:2], DEV, chunk=2, annotations=True)
    for _ in range(2):                                   # second run reuses the staging sets and host buffers
        outs = pipe.run(hv)
    assert [a for o in outs for a in o["annotations"]] == want


def test_host_pipeline_grows_and_reruns_short_capacity():
    """Noise in the background of the label maps (about two edges per noisy pixel) and a tiny forced capacity: the
    first chunk on each staging set overflows and is re-run (about twice: once for the counts, once for the exact
    string size) before chunk 2 or 3 reuses that set, and the annotations of all four chunks are right. Later chunks
    re-run only if they need more than the grown buffers hold."""
    from s2d_b200.hostpipe import HostPipeline
    base = _scenes()[:2]
    scenes = []
    for c in range(4):                                   # 4 chunks: each staging set is reused once
        for j, sc in enumerate(base):
            rng = np.random.default_rng(10 * c + j)
            lab = sc.labels.copy()
            for t in range(lab.shape[0]):
                present = np.unique(lab[t])[1:]
                bg = (lab[t] == 0) & (rng.random(lab[t].shape) < 0.5)
                lab[t][bg] = rng.choice(present, size=int(bg.sum()))
            scenes.append(dataclasses.replace(sc, labels=lab))
    want = _resident(scenes)
    assert sum(a is not None for a in want) >= 4
    hv = _host_videos(scenes, False)
    pipe = HostPipeline(hv[:2], DEV, chunk=2, annotations=True)
    for _, b in pipe.sets:
        b._alloc_rle(64, 64)
    outs = pipe.run(hv)
    assert pipe.reruns >= 4
    assert [a for o in outs for a in o["annotations"]] == want


def test_host_pipeline_default_is_unchanged():
    from s2d_b200.hostpipe import HostPipeline
    from s2d_b200.pipeline import Batch
    scenes = _scenes()
    hv = _host_videos(scenes, True)
    plain = HostPipeline(hv[:2], DEV, chunk=2)
    withE = HostPipeline(hv[:2], DEV, chunk=2, annotations=True)
    assert all(b.stages == "LVBD" and b.rle_counts is None and b.al_work is None for _, b in plain.sets)
    a = plain.run(hv)
    launches, d2h = plain.launches, plain.d2h_bytes
    a = [{k: o[k].clone() for k in HostPipeline.RESULT_TABLES} for o in a]
    b = withE.run(hv)
    for x, y in zip(a, b):
        assert set(x) == set(HostPipeline.RESULT_TABLES) and "annotations" in y
        for k in HostPipeline.RESULT_TABLES:
            assert torch.equal(x[k], y[k]), k
    per_chunk = Batch(plain.sets[0][0]).run()
    assert launches == 2 * per_chunk
    assert d2h == sum(o[k].numel() * o[k].element_size() for o in a for k in HostPipeline.RESULT_TABLES)
    assert withE.launches == 2 * (per_chunk + 8 + 3) + 11 * withE.reruns
