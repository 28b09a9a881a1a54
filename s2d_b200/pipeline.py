"""Batched, device-resident keymask discovery: the arithmetic of the reference's per-video loop
(keymask_ident/main_keymask_ident.py:91-128, stages A-D) as one sequence of CUDA launches over a
whole batch of videos, with no host round trip between the stages.

torch is used for device memory and streams only; every number is produced by the kernels in
s2d_b200/csrc through the C ABI (include/s2d_b200.h). `decode()` turns the raw device results
into the same python structures the reference builds (stage-B json schema, matches_data,
groupings, one2x, coverage) - it only unpacks bit masks and index tables.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field
from typing import List, Optional, Union

import numpy as np
import torch

from . import _lib
from ._lib import (S2D_CLINFO_WORDS, S2D_MAX_CLUSTERS, S2D_MAX_LABELS, S2D_PV_TMAP_BYTES, S2D_VIDINFO_WORDS, VideoDesc)


@dataclass
class VideoInput:
    """Device tensors of one video (see s2d_b200.synth for the layout)."""
    labels: Optional[torch.Tensor] = None   # u8  [T,H,W]
    tracks: Optional[torch.Tensor] = None   # f32 [Nm,T,P,2]
    vis: Optional[torch.Tensor] = None      # u8/bool [Nm,T,P]; or int32 [Nm,T,ceil(P/32)] bit-packed (pack_vis_bits) with vis_bits=True
    vis_bits: bool = False                  # `vis` holds the flags bit-packed by the producer (1/8 of the bytes on the wire)
    npts: Optional[torch.Tensor] = None     # i32 [Nm]
    tstart: Optional[torch.Tensor] = None   # i32 [Nm]: tracks hold frames [tstart[q], tstart[q] + tracks.shape[1]) only
    max_label: Optional[int] = None         # upper bound of the label ids (default 255)
    name: str = ""
    # stage-wise callers (the file-based drop-in modules) may omit tensors a stage does not read
    # and give the missing dimensions here: keys T, H, W, P, Nm
    dims: Optional[dict] = None


@dataclass
class Params:
    """Constants the reference hard-codes (SURVEY.md section 5, config row) with its defaults."""
    visibility_threshold: float = 0.3       # --visibility-threshold
    matching_threshold: float = 0.5         # --matching-threshold
    dbscan1_eps: float = 0.2                # identify_visibility_windows.py:114
    dbscan1_min_samples: int = 5
    winner_fraction: float = 0.3            # identify_visibility_windows.py:166
    one2x_iou: float = 0.25                 # cotracker_matching.py:1085
    one2x_frames: int = 5                   # cotracker_matching.py:1111


def _i32(n, device, fill=None):
    t = torch.empty(int(n), dtype=torch.int32, device=device)
    if fill is not None:
        t.fill_(fill)
    return t


class Batch:
    """Descriptor table + workspace for a list of videos. Allocation happens here, once; `run`
    only enqueues kernels, so a Batch can be re-run (benchmarks) without touching the allocator."""

    def __init__(self, videos: List[VideoInput], device=None, stages: str = "LVBD", persistent_votes: bool = True,
                 label_tmaps: bool = True, gram_min_rows: int = 2048):
        """`persistent_votes=False` runs K2 as one CTA per tile (the library's fallback for odd P / unaligned
        tracks), `label_tmaps=False` makes the persistent kernel fetch its label tables row by row instead of as TMA
        boxes; both exist for tests and profiling comparisons, the defaults are the product path."""
        assert len(videos) > 0
        self.videos = videos
        first = next(t for t in (videos[0].labels, videos[0].tracks, videos[0].vis) if t is not None) \
            if any(t is not None for t in (videos[0].labels, videos[0].tracks, videos[0].vis)) else None
        self.device = device or (first.device if first is not None else torch.device("cuda:0"))
        dev = self.device
        nv = len(videos)
        descs = (VideoDesc * nv)()
        row0 = frame0 = vt = hits = xw = mw = 0
        self.max_T = self.max_Nm = self.max_TW = self.max_NW = self.max_P = 0
        self.max_npix = self.max_rows_x_T = self.max_rows_x_TW = 0
        self.vec4 = 1
        self._keep = []
        for i, v in enumerate(videos):
            dm = dict(v.dims or {})
            if v.labels is not None:
                assert v.labels.dtype == torch.uint8 and v.labels.is_contiguous() and v.labels.dim() == 3
                dm["T"], dm["H"], dm["W"] = v.labels.shape
            if v.tracks is not None:
                assert v.tracks.dtype == torch.float32 and v.tracks.is_contiguous() and v.tracks.dim() == 4
                assert v.tracks.shape[3] == 2
                if v.tstart is None:
                    assert dm.setdefault("T", v.tracks.shape[1]) == v.tracks.shape[1]
                dm["Nm"], dm["P"] = v.tracks.shape[0], v.tracks.shape[2]
            if v.vis is not None:
                assert v.vis.is_contiguous() and v.vis.dim() == 3
                if v.vis_bits:
                    assert v.vis.dtype == torch.int32 and "P" in dm, "bit-packed flags need P (from tracks or dims)"
                    assert v.vis.shape[2] == (dm["P"] + 31) // 32 and dm.setdefault("Nm", v.vis.shape[0]) == v.vis.shape[0]
                    assert dm.setdefault("T", v.vis.shape[1]) == v.vis.shape[1]
                else:
                    assert v.vis.dtype in (torch.uint8, torch.bool)
                    if v.tracks is not None and v.tstart is None:
                        assert tuple(v.vis.shape) == (dm["Nm"], dm["T"], dm["P"]), "inconsistent video tensors"
                    else:
                        assert dm.setdefault("T", v.vis.shape[1]) == v.vis.shape[1]
                        assert dm.setdefault("Nm", v.vis.shape[0]) == v.vis.shape[0]
                        assert dm.setdefault("P", v.vis.shape[2]) == v.vis.shape[2]
            T, H, W = dm["T"], dm.get("H", 1), dm.get("W", 1)
            Nm, P = dm["Nm"], dm.get("P", 1)
            assert Nm >= 1 and T >= 1
            assert H <= 65535 and W <= 65535 and P <= 32768 and T <= 1024
            L = min(S2D_MAX_LABELS, (v.max_label if v.max_label is not None else 255) + 1)
            d = descs[i]
            d.T, d.H, d.W, d.P, d.Nm, d.L = T, H, W, P, Nm, L
            d.TW, d.NW = (T + 31) // 32, (Nm + 31) // 32
            d.row0, d.frame0 = row0, frame0
            d.labels = v.labels.data_ptr() if v.labels is not None else None
            d.tracks = v.tracks.data_ptr() if v.tracks is not None else None
            d.vis = v.vis.data_ptr() if v.vis is not None else None
            d.npts = v.npts.data_ptr() if v.npts is not None else None
            d.tstart = v.tstart.data_ptr() if v.tstart is not None else None
            d.Ttr = v.tracks.shape[1] if v.tracks is not None else T
            d.flags = _lib.S2D_DESC_VIS_BITS if (v.vis is not None and v.vis_bits) else 0
            d.vt_off, d.hits_off, d.xbits_off, d.mbits_off = vt, hits, xw, mw
            if P % 2 or (v.tracks is not None and v.tracks.data_ptr() % 16):
                self.vec4 = 0
            row0 += Nm; frame0 += T; vt += Nm * T; hits += Nm * T * L
            xw += Nm * d.TW; mw += Nm * d.NW
            self.max_T = max(self.max_T, T); self.max_Nm = max(self.max_Nm, Nm)
            self.max_TW = max(self.max_TW, d.TW); self.max_NW = max(self.max_NW, d.NW)
            self.max_P = max(self.max_P, P); self.max_npix = max(self.max_npix, H * W)
            self.max_rows_x_T = max(self.max_rows_x_T, Nm * T)
            self.max_rows_x_TW = max(self.max_rows_x_TW, Nm * d.TW)
        self.nv = nv
        self.stages = stages
        self.host_descs = descs
        self.total_rows, self.total_frames, self.total_vt = row0, frame0, vt
        self.total_hits, self.total_xw, self.total_mw = hits, xw, mw
        raw = np.frombuffer(bytes(descs), dtype=np.uint8)
        self.descs = torch.from_numpy(raw.copy()).to(dev)

        # workspace / outputs: only what the requested stages touch
        st = set(stages)
        z = lambda n, fill=None: _i32(n, dev, fill)
        n = C.c_int64()
        self.vidinfo = z(nv * S2D_VIDINFO_WORDS, 0)
        self.qframe = z(row0, 0)
        self.qlabel = z(row0, 0)
        self.rowinfo = z(row0 * 4, -1)
        self.clusterinfo = z(nv * S2D_MAX_CLUSTERS * S2D_CLINFO_WORDS, 0)
        self.labels1 = z(row0, -1)
        self.area = self.gid_of = self.frameinfo = None
        if st & set("LD"):
            self.area = z(frame0 * S2D_MAX_LABELS)
            self.gid_of = z(frame0 * S2D_MAX_LABELS)
            self.frameinfo = z(frame0 * 4)
        self.cnt = self.V = None
        if st & set("VB"):
            self.cnt = z(vt)
            self.V = torch.empty(vt, dtype=torch.float32, device=dev)
        self.xbits = self.dbwork = self.ccount = self.clrow = None
        self.majbits = self.rsbits = self.rebits = self.winbits = None
        if "B" in st:
            self.xbits = z(xw)
            _lib.call("s2d_dbscan_work_ints", row0, nv, C.byref(n))
            self.dbwork = z(n.value + 2)
            self.ccount = z(vt)
            self.clrow = z(row0 * 4)
            self.majbits, self.rsbits, self.rebits, self.winbits = z(xw), z(xw), z(xw), z(xw)
        self.pvwork = self.pvtmaps = self.hits = self.uniq = self.mbits = self.one2x = self.nmatch = None
        self.grpwork = self.glabel = self.grp_n = self.grp_one2x = None
        if "D" in st:
            _lib.call("s2d_point_votes_work_ints", row0, C.byref(n))
            self.pvwork = z(n.value + 4)
            # TMA descriptors of the label maps (host-encoded once per batch)
            if label_tmaps and all(v.labels is not None for v in videos):
                hbuf = np.zeros(nv * S2D_PV_TMAP_BYTES, np.uint8)
                _lib.call("s2d_point_votes_tmaps", descs, nv, hbuf.ctypes.data)
                self.pvtmaps = torch.from_numpy(hbuf).to(dev)
                assert self.pvtmaps.data_ptr() % 64 == 0
            self.hits = z(hits)
            self.uniq = z(vt)
            self.mbits = z(mw)
            self.one2x = z(row0)
            self.nmatch = z(row0)
            _lib.call("s2d_group_work_ints", row0, nv, C.byref(n))
            self.grpwork = z(n.value + 2)
            self.glabel = z(row0)
            self.grp_n = z(16 * row0)
            self.grp_one2x = z(16 * row0)
            # DBSCAN #2 of videos with many rows: the pairwise distances come from one int8 Gram contraction of the
            # video's match rows on the tensor cores (O(Nm^2) reads in the DBSCAN passes instead of O(Nm^3 / 32) bit ops)
            self.gram = self.gram_off = self.gram_planes = None
            big = [i for i in range(nv) if descs[i].Nm >= gram_min_rows]
            if big:
                offs, tot, pmax = [-1] * nv, 0, 0
                for i in big:
                    offs[i] = tot
                    tot += descs[i].Nm * descs[i].Nm
                    tot += (-tot) % 4                         # 16-byte aligned matrices
                    pmax = max(pmax, descs[i].Nm * descs[i].NW * 32)
                self.gram = z(tot)
                self.gram_off = torch.tensor(offs, dtype=torch.int64, device=dev)
                self.gram_planes = torch.empty(pmax, dtype=torch.uint8, device=dev)
                self._gram_videos = [(i, offs[i]) for i in big]
        # stage E: COCO RLE of every keymask row from the label maps (counts, offsets, boxes) and its strings
        self.rle_work = self.rle_counts = self.rle_off = self.rle_bbox = self.rle_need = None
        self.str_work = self.str_off = self.rle_chars = self.al_work = self.al_chars = None
        self.aj_work = self.aj_out = None
        self.aj_cap = 0
        self.rle_cap = self.str_cap = 0
        if "E" in st:
            assert "L" in st and "D" in st, 'stage "E" reads K0\'s gid_of ("L") and the final status of K4 ("D")'
            self.max_H = max(descs[i].H for i in range(nv))
            self.max_W = max(descs[i].W for i in range(nv))
            _lib.call("s2d_label_rle_work_ints", frame0, row0, self.max_H, self.max_W, C.byref(n))
            self.rle_work = z(n.value)
            self.rle_off = torch.empty(row0 + 1, dtype=torch.int64, device=dev)
            self.rle_bbox = z(4 * row0)
            self.rle_need = torch.zeros(2, dtype=torch.int64, device=dev)    # counts, string bytes the run needed
            self.str_work = z(row0)
            self.str_off = torch.empty(row0 + 1, dtype=torch.int64, device=dev)
            # annotation layout (s2d_annotation_layout): annotations and members number at most one per row, the
            # packed strings at most stage E's, clusters S2D_MAX_CLUSTERS and runs ceil(T / 2) per cluster per video
            _lib.call("s2d_annotation_layout_work_ints", row0, nv, C.byref(n))
            self.al_work = z(n.value)
            self.al_vann = z(2 * nv)
            self.al_ann = z(7 * row0)
            self.al_members = z(6 * row0)
            self.al_member_off = torch.empty(row0, dtype=torch.int64, device=dev)
            self.al_clusters = z(2 * S2D_MAX_CLUSTERS * nv)
            self.al_pairs = z(2 * (S2D_MAX_CLUSTERS // 2) * (frame0 + nv))
            self.al_sizes = torch.zeros(5, dtype=torch.int64, device=dev)     # annotations, members, string bytes, clusters, pairs
            # first guess: blob-like maps have about two edges per (object, column); too small re-runs (annotations())
            cap = sum(descs[i].T * 8 * descs[i].W for i in range(nv)) + 2 * row0
            self._alloc_rle(cap, 3 * cap)
            # annotation json (s2d_annotation_json): the text buffer is allocated by the first serialize(), sized as the
            # layout's string capacity plus 128 bytes of fixed text per row (segmentation header, box, area, separators,
            # nulls); a short guess re-runs the json call alone
            _lib.call("s2d_annotation_json_work_ints", row0, nv, C.byref(n))
            self.aj_work = z(n.value)
            self.aj_video_off = torch.zeros(nv + 1, dtype=torch.int64, device=dev)
            self.aj_need = torch.zeros(1, dtype=torch.int64, device=dev)
            self.aj_out, self.aj_cap = None, self.str_cap + 128 * row0
        self._graph = None
        self.kernel_launches_per_run = 0
        # persistent TMA-fed votes kernel (the library falls back by itself when P is odd)
        self.use_tma = bool(persistent_votes)

    # ------------------------------------------------------------------ enqueue
    def run(self, params: Params = Params(), stream=None, stages: Optional[str] = None, timers=None):
        """Enqueue the whole path on `stream` (default: torch's current stream). Returns the
        number of kernel launches enqueued. `timers`: optional dict name -> list; a pair of CUDA
        events is recorded around every C-ABI call on torch's current stream (bench.py)."""
        with torch.cuda.device(self.device):       # events and launches on the batch's device, whatever is current
            return self._run(params, stream, stages, timers)

    def _run(self, params, stream, stages, timers):
        st = stream if stream is not None else torch.cuda.current_stream(self.device).cuda_stream
        p = lambda t: t.data_ptr() if t is not None else None
        d, nv = p(self.descs), self.nv
        launches = 0
        stages = self.stages if stages is None else stages
        assert set(stages) <= set(self.stages), f"batch was built for stages {self.stages!r}"

        def call(tag, nk, name, *args):
            nonlocal launches
            if timers is not None:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                _lib.call(name, *args)
                e1.record()
                timers.setdefault(tag, []).append((e0, e1))
            else:
                _lib.call(name, *args)
            launches += nk

        if "L" in stages:
            call("label_stats", 2, "s2d_label_stats", d, nv, self.max_T, self.max_npix, self.total_frames,
                 p(self.area), p(self.gid_of), p(self.frameinfo), p(self.qframe), p(self.qlabel), p(self.vidinfo), st)
        if "V" in stages:
            call("vis_reduce", 1, "s2d_vis_reduce", d, nv, self.max_rows_x_T, p(self.cnt), p(self.V), st)
        if "B" in stages:
            call("binarize", 1, "s2d_binarize", d, nv, self.max_rows_x_TW, p(self.V),
                 float(np.float32(params.visibility_threshold)), p(self.xbits), st)
            call("dbscan1", 6, "s2d_dbscan_visibility", d, nv, self.max_Nm, self.max_TW, self.total_rows,
                 p(self.xbits), params.dbscan1_eps, params.dbscan1_min_samples, p(self.dbwork), p(self.labels1),
                 p(self.vidinfo), st)
            call("windows", 4, "s2d_windows", d, nv, self.max_rows_x_TW, self.max_TW, self.total_rows,
                 self.total_vt, p(self.xbits), p(self.labels1), p(self.qframe),
                 float(np.float32(params.winner_fraction)), p(self.ccount), p(self.clrow), p(self.majbits),
                 p(self.rsbits), p(self.rebits), p(self.winbits), p(self.rowinfo), p(self.vidinfo),
                 p(self.clusterinfo), st)
        if "D" in stages:
            call("point_votes", 3 if self.use_tma else 1, "s2d_point_votes_sized", d, nv, self.max_T, self.max_Nm, self.max_P,
                 self.vec4, self.total_rows, p(self.rowinfo), p(self.vidinfo),
                 p(self.pvwork) if self.use_tma else None, p(self.pvtmaps), self.max_npix, p(self.hits), p(self.uniq), st)
            call("select", 1, "s2d_select", d, nv, self.max_Nm, self.total_mw, p(self.hits), p(self.uniq),
                 p(self.gid_of), p(self.rowinfo), params.matching_threshold, params.one2x_iou,
                 params.one2x_frames, p(self.mbits), p(self.one2x), p(self.nmatch), p(self.vidinfo), st)
            self._enqueue_group(call, st, True)
        if "E" in stages:
            call("label_rle", 5, "s2d_label_rle", d, nv, self.max_T, self.max_H, self.max_W, self.max_Nm,
                 self.total_frames, self.total_rows, p(self.gid_of), p(self.vidinfo), p(self.rle_work), self.rle_cap,
                 p(self.rle_counts), p(self.rle_off), p(self.rle_bbox), p(self.rle_need), st)
            call("rle_strings", 3, "s2d_rle_strings", p(self.rle_counts), p(self.rle_off), self.total_rows, self.rle_cap,
                 p(self.str_work), self.str_cap, p(self.rle_chars), p(self.str_off), p(self.rle_need) + 8, st)
        self.kernel_launches_per_run = launches
        return launches

    def _enqueue_group(self, call, st, gram: bool):
        """DBSCAN #2 and the grouping of stage D on the match tables in place (mbits, rowinfo, one2x, vidinfo). Videos with a
        Gram buffer first contract their match rows with themselves; `gram=False` takes every video's distances from the
        bit rows instead."""
        p = lambda t: t.data_ptr() if t is not None else None
        use = gram and self.gram is not None
        if use:
            for i, off in self._gram_videos:               # match rows -> u8 planes -> G = X X^T (tcgen05 kind::i8)
                hd = self.host_descs[i]
                mb = self.mbits.data_ptr() + 4 * hd.mbits_off
                call("group", 1, "s2d_unpack_bits", mb, hd.Nm, hd.NW, hd.NW * 32, p(self.gram_planes), st)
                call("group", 2, "s2d_overlap_i8", p(self.gram_planes), hd.Nm, p(self.gram_planes), hd.Nm, hd.NW * 32,
                     self.gram.data_ptr() + 4 * off, st)
        call("group", 8, "s2d_group_gram", p(self.descs), self.nv, self.max_Nm, self.max_NW, self.total_rows, p(self.mbits),
             p(self.rowinfo), p(self.one2x), p(self.grpwork), p(self.glabel), p(self.grp_n), p(self.grp_one2x),
             p(self.vidinfo), p(self.clusterinfo), p(self.gram) if use else None, p(self.gram_off) if use else None, st)

    def group(self, stream=None, gram: bool = True):
        """Enqueue stage D's grouping alone (what run() does after s2d_select) on the match tables as they stand: callers
        that fill mbits / rowinfo / one2x / vidinfo themselves, and re-runs of one step's grouping with `gram=False`."""
        assert "D" in self.stages, 'the grouping needs a batch built with stage "D"'
        st = stream if stream is not None else torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            self._enqueue_group(lambda tag, nk, name, *args: _lib.call(name, *args), st, gram)

    def _alloc_rle(self, counts_cap: int, chars_cap: int):
        self.rle_cap, self.str_cap = int(counts_cap), int(chars_cap)
        self.rle_counts = torch.empty(max(1, self.rle_cap), dtype=torch.int32, device=self.device)
        self.rle_chars = torch.empty(max(1, self.str_cap), dtype=torch.uint8, device=self.device)
        self.al_chars = torch.empty(max(1, self.str_cap), dtype=torch.uint8, device=self.device)

    def capture(self, params: Params = Params(), stages: Optional[str] = None):
        """Record the whole path of this batch once as a CUDA graph; replay() then costs one launch
        instead of ~20 (small batches - a single short video - are launch-bound). The C-ABI calls only
        enqueue kernels and memsets on the current stream, so they capture as they are; the first,
        un-captured run() configures the kernels' attributes."""
        with torch.cuda.device(self.device):
            self.run(params, stages=stages)
            torch.cuda.synchronize(self.device)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self.run(params, stages=stages)
        self._graph = g
        self._graph_args = (params, stages)
        return g

    def replay(self):
        self._graph.replay()

    def votes_all(self, stream=None):
        """K2 over every (query, frame) of every video, ignoring candidates/status (tests, bench)."""
        st = stream if stream is not None else torch.cuda.current_stream(self.device).cuda_stream
        _lib.call("s2d_point_votes_sized", self.descs.data_ptr(), self.nv, self.max_T, self.max_Nm, self.max_P, self.vec4,
                  self.total_rows, None, None, self.pvwork.data_ptr() if self.use_tma else None,
                  self.pvtmaps.data_ptr() if self.pvtmaps is not None else None, self.max_npix,
                  self.hits.data_ptr(), self.uniq.data_ptr(), st)

    # ------------------------------------------------------------------ results
    def fetch_summary(self):
        """The small device->host read of a step's result: status, cluster table, per-row
        (cluster, candidate, window), group labels, one2x flags."""
        out = dict(vidinfo=self.vidinfo.cpu().numpy().reshape(self.nv, S2D_VIDINFO_WORDS),
                   clusterinfo=self.clusterinfo.cpu().numpy().reshape(self.nv, S2D_MAX_CLUSTERS, S2D_CLINFO_WORDS),
                   rowinfo=self.rowinfo.cpu().numpy().reshape(-1, 4),
                   glabel=self.glabel.cpu().numpy(), one2x=self.one2x.cpu().numpy())
        return out

    def upload_visibility(self, V: np.ndarray, qframe: np.ndarray, vi: int = 0):
        """Stage-wise entry (file-based drop-in): place an existing visibility matrix [Nm,T] and
        the rows' frame ids for video `vi` before run(stages="B")."""
        d = self.host_descs[vi]
        assert V.shape == (d.Nm, d.T)
        self.V[d.vt_off:d.vt_off + d.Nm * d.T] = torch.from_numpy(np.ascontiguousarray(V, np.float32).reshape(-1)).to(self.device)
        self.qframe[d.row0:d.row0 + d.Nm] = torch.from_numpy(np.ascontiguousarray(qframe, np.int32)).to(self.device)

    def upload_stage_b(self, rowinfo: np.ndarray, nclusters: int, status: int, vi: int = 0):
        """Stage-wise entry: rows' (cluster, candidate run, v0, v1) and the stage-B status as the
        host derived them from the stage-B json / stage-C folder, before run(stages="LD")."""
        d = self.host_descs[vi]
        assert rowinfo.shape == (d.Nm, 4)
        self.rowinfo[4 * d.row0:4 * (d.row0 + d.Nm)] = torch.from_numpy(np.ascontiguousarray(rowinfo, np.int32).reshape(-1)).to(self.device)
        v = torch.tensor([nclusters, status, -1, -1, int((rowinfo[:, 1] >= 0).sum())], dtype=torch.int32, device=self.device)
        self.vidinfo[vi * S2D_VIDINFO_WORDS:vi * S2D_VIDINFO_WORDS + 5] = v
        self.labels1[d.row0:d.row0 + d.Nm] = torch.from_numpy(np.ascontiguousarray(rowinfo[:, 0], np.int32)).to(self.device)

    def decode(self, want_comps: bool = True, check_rows: bool = True):
        """Full results in the reference's python structures, one dict per video (same schema as
        oracle.keymask_oracle.discover)."""
        h = {k: getattr(self, k).cpu().numpy() for k in
             ("qframe", "qlabel", "vidinfo", "V", "labels1", "clrow", "rsbits", "rebits", "winbits", "rowinfo",
              "clusterinfo", "one2x", "nmatch", "mbits", "glabel", "grp_n", "grp_one2x", "area", "gid_of")
             if getattr(self, k) is not None}
        have_b = self.xbits is not None
        if want_comps and self.hits is not None:
            h["hits"] = self.hits.cpu().numpy()
            h["uniq"] = self.uniq.cpu().numpy()
        vidinfo = h["vidinfo"].reshape(self.nv, S2D_VIDINFO_WORDS)
        clinfo = h["clusterinfo"].reshape(self.nv, S2D_MAX_CLUSTERS, S2D_CLINFO_WORDS)
        rowinfo = h["rowinfo"].reshape(-1, 4)
        clrow = h["clrow"].reshape(-1, 4) if have_b else None
        area = h["area"].reshape(-1, S2D_MAX_LABELS) if "area" in h else None
        gid_of = h["gid_of"].reshape(-1, S2D_MAX_LABELS) if "gid_of" in h else None
        want_comps = want_comps and "hits" in h
        results = []
        for vi in range(self.nv):
            d = self.host_descs[vi]
            T, Nm, TW, NW, L = d.T, d.Nm, d.TW, d.NW, d.L
            r0, f0 = d.row0, d.frame0
            if check_rows and int(vidinfo[vi, 5]) != Nm:
                raise _lib.S2DError(f"video {vi}: tracks hold {Nm} queries but the label maps enumerate "
                                    f"{int(vidinfo[vi, 5])} objects")
            qf = h["qframe"][r0:r0 + Nm].astype(np.int64)
            ql = h["qlabel"][r0:r0 + Nm].astype(np.int64)
            res = {"query_frame": qf, "query_label": ql}
            if "V" in h:
                res["V"] = h["V"][d.vt_off:d.vt_off + Nm * T].reshape(Nm, T)
            lab1 = h["labels1"][r0:r0 + Nm].astype(np.int64)
            res["labels1"] = lab1
            ri = rowinfo[r0:r0 + Nm]
            bits = lambda name: h[name][d.xbits_off:d.xbits_off + Nm * TW].reshape(Nm, TW).view(np.uint32)
            if have_b:
                rs, re, wb = bits("rsbits"), bits("rebits"), bits("winbits")
            k = int(vidinfo[vi, 0])
            clusters = []
            for c in range(k if have_b else 0):
                starts = _setbits(rs[c], T)
                ends = _setbits(re[c], T)
                rows = np.nonzero(lab1 == c)[0]
                all_cands, all_vis = [], []
                for r, (s, e) in enumerate(zip(starts, ends)):
                    cands = []
                    for g in rows:
                        if (wb[g, r >> 5] >> (r & 31)) & 1:
                            all_vis.append({"frame_id": int(qf[g]), "mask_id": int(ql[g])})
                            if ri[g, 1] == r:
                                cands.append({"start_frame": s, "end_frame": e, "frame_id": int(qf[g]),
                                              "mask_id": int(ql[g])})
                    all_cands.append({"range": [s, e], "candidates": cands})
                clusters.append({"cluster_id": c, "cluster_size": int(clrow[r0 + c, 0]),
                                 "ranges": [[s, e] for s, e in zip(starts, ends)],
                                 "all_candidates": all_cands, "all_visible_masks": all_vis})
            res["clusters"] = clusters
            status = int(vidinfo[vi, 3]) if self.mbits is not None else -1
            res["status"] = status
            res["stage_b_status"] = int(vidinfo[vi, 1])
            res["queries"] = []
            res["groupings"] = None
            if status == 1:
                mb = h["mbits"][d.mbits_off:d.mbits_off + Nm * NW].reshape(Nm, NW).view(np.uint32)
                if want_comps:
                    hits = h["hits"][d.hits_off:d.hits_off + Nm * T * L].reshape(Nm, T, L)
                    uniq = h["uniq"][d.vt_off:d.vt_off + Nm * T].reshape(Nm, T)
                    # windowed track storage: frames without stored tracks were not voted on (their hits / uniq are
                    # whatever the buffers held); they count as intersection 0 / union 0, like in s2d_select
                    tsv = self.videos[vi].tstart
                    ts_h = tsv.cpu().numpy().astype(np.int64) if tsv is not None else None
                queries = []
                for c in range(k):
                    rows = np.nonzero((ri[:, 0] == c) & (ri[:, 1] >= 0))[0]
                    # processing order: files sorted lexicographically by name, then stable by frame
                    names = sorted((f"cluster{c}_frame{int(qf[g])}_mask{int(ql[g])}.png", int(g)) for g in rows)
                    order = sorted(names, key=lambda ng: int(qf[ng[1]]))
                    for _, g in order:
                        v0, v1 = int(ri[g, 2]), int(ri[g, 3])
                        a = int(area[f0 + int(qf[g]), int(ql[g])])
                        q = {"cluster_id": c, "frame_id": int(qf[g]), "mask_id": int(ql[g]), "overall_mask_id": g,
                             "one2x": int(h["one2x"][r0 + g]), "matches": _setbits(mb[g], Nm),
                             "v_range": (v0, v1), "grid_size": max(min(a // 800, 50), 25),
                             "backward_tracking": int(qf[g]) > v0}
                        if want_comps:
                            comps = []
                            for t in range(v0, v1 + 1):
                                gids = gid_of[f0 + t]
                                stored = ts_h is None or ts_h[g] <= t < ts_h[g] + d.Ttr
                                for o in np.nonzero(gids >= 0)[0]:
                                    I, U = (int(hits[g, t, o]), int(uniq[g, t])) if stored else (0, 0)
                                    comps.append((t, int(o), int(gids[o]), I, U, 0.0 if U == 0 else I / U))
                            q["comps"] = comps
                        queries.append(q)
                res["queries"] = queries
                groupings, cov = [], []
                tot_m = tot_n = 0
                one2x_video = {}
                for c in range(k):
                    ci = clinfo[vi, c]
                    rows = np.nonzero(ri[:, 0] == c)[0]
                    gl = h["glabel"][r0:r0 + Nm]
                    groups = {}
                    for g in rows:
                        if gl[g] >= 0:
                            groups.setdefault(int(gl[g]), []).append((int(qf[g]), int(ql[g])))
                    groupings.append({"cluster_id": c, "visibility_to_temporal_factor": int(ci[11]),
                                      "overall_mask_ids_per_label": groups})
                    cov.append(int(ci[12]) / int(ci[14]) if ci[14] else 0)     # matched / candidates of the cluster
                    tot_m += int(ci[12]); tot_n += int(ci[14])
                    od = {"avg_one2x_cluster": int(ci[13]) / int(ci[14]) if ci[14] else float("nan")}
                    base = 16 * r0 + c * Nm
                    for lab in groups:
                        n_, s_ = int(h["grp_n"][base + lab]), int(h["grp_one2x"][base + lab])
                        avg = s_ / n_ if n_ else 0
                        od[f"group_{lab}"] = {"avg_one2x": avg, "one2x_counts": n_, "noisy": bool(avg > 0.5)}
                    one2x_video[f"cluster_{c}"] = od
                res["groupings"] = groupings
                res["cluster_coverages"] = cov
                res["video_coverage"] = tot_m / tot_n if tot_n else 0
                res["one2x"] = one2x_video
            results.append(res)
        return results


    def rle_tables(self, counts: bool = False):
        """Host copy of stage E's device tables after run() / replay(): per row (global id) `offsets` of its runs,
        `bbox` (xmin, ymin, xmax, ymax), `str_off` of its string in `chars`; `counts` (the runs) on request. When a
        buffer was too small for this batch (the device reports what it needed; noise-like label maps have about two
        edges per pixel) it is grown and stage E re-run - its inputs are still in place - and a captured graph is
        recorded again on the new buffers."""
        assert "E" in self.stages, 'stage-E tables need a batch built with stage "E"'
        with torch.cuda.device(self.device):
            need = self._settle_rle()
            out = {"offsets": self.rle_off.cpu().numpy(), "bbox": self.rle_bbox.cpu().numpy().reshape(-1, 4),
                   "str_off": self.str_off.cpu().numpy(),
                   "chars": self.rle_chars[:max(1, need[1])].cpu().numpy().tobytes()[:need[1]].decode("ascii")}
            if counts:
                out["counts"] = self.rle_counts[:max(1, need[0])].cpu().numpy()[:need[0]]
        return out

    def _settle_rle(self):
        """Wait for the step, and grow the stage-E buffers and re-run stage E (re-recording a captured graph) while
        the device reports that a capacity was short. Returns the final `need` (counts, string bytes)."""
        torch.cuda.synchronize(self.device)
        need = self.rle_need.cpu().tolist()
        if self.rle_fits(need):
            return need
        while not self.rle_fits(need):
            self.grow_rle(need)
            self.run(stages="E")
            torch.cuda.synchronize(self.device)
            need = self.rle_need.cpu().tolist()
        if self._graph is not None:
            self.capture(*self._graph_args)
            torch.cuda.synchronize(self.device)
        return need

    def rle_fits(self, need) -> bool:
        """Whether stage E's tables are complete, given a host copy of `rle_need`."""
        return need[0] <= self.rle_cap and need[1] <= self.str_cap

    def grow_rle(self, need):
        """Grow the stage-E buffers (and the layout's string buffer) to a host copy of `rle_need`; stage E has to be
        run again. Once the counts fit, the string size the device reports is exact, so at most two rounds are needed."""
        self._alloc_rle(max(need[0], self.rle_cap), max(need[1], self.str_cap))

    def layout(self, stream=None) -> int:
        """Enqueue the annotation layout (s2d_annotation_layout) of this step's stage-E tables on `stream` (default:
        torch's current stream): per video the annotations, their members and strings and the clusters' visibility
        runs, packed in the reference's order into the `al_*` tables, their used lengths into `al_sizes`. Returns the
        number of kernel launches."""
        assert "E" in self.stages, 'the annotation layout needs a batch built with stage "E"'
        st = stream if stream is not None else torch.cuda.current_stream(self.device).cuda_stream
        p = lambda t: t.data_ptr()
        with torch.cuda.device(self.device):
            _lib.call("s2d_annotation_layout", p(self.descs), self.nv, self.total_rows, p(self.vidinfo), p(self.rowinfo),
                      p(self.winbits), p(self.rsbits), p(self.rebits), p(self.glabel), p(self.qframe), p(self.qlabel),
                      p(self.grp_n), p(self.grp_one2x), p(self.area), p(self.gid_of), p(self.rle_bbox), p(self.str_off),
                      p(self.rle_chars), self.str_cap, p(self.al_work), p(self.al_vann), p(self.al_ann), p(self.al_members),
                      p(self.al_member_off), p(self.al_clusters), p(self.al_pairs), self.str_cap, p(self.al_chars),
                      p(self.al_sizes), st)
        return 3

    def layout_views(self, sizes):
        """Device views of the used part of every layout table, given a host copy of `al_sizes`."""
        return {"vann": self.al_vann, **{k: getattr(self, "al_" + k)[:w * int(sizes[i])] for k, (w, i) in LAYOUT_TABLES.items()}}

    def annotations(self, results=None):
        """Stage E: per video the `annotations` list of the YTVIS json the reference writes for it
        (keymask_ident/annotations.py:8-140), or None when the video's final status is not 1 (the reference writes
        none). Needs a batch built with "E" in its stages, after run() or replay(). `results` is accepted for
        compatibility and unused: the annotations no longer come from decode().

        The device lays them out (layout(), after the stage-E capacities are settled) in the reference's order:
        cluster directories with candidates in lexicographic order of `cluster_{c}`, groups in lexicographic order
        of `group_{l}`, ids from 1 across the video. A group with two members on one frame keeps the member with the
        largest label id (the reference keeps whichever PNG its directory listing returns last). The host copies the
        used part of the tables back and slices them into json objects."""
        with torch.cuda.device(self.device):
            self._settle_rle()
            self.layout()
            sizes = self.al_sizes.cpu().tolist()
            tabs = {k: t.cpu().numpy() for k, t in self.layout_views(sizes).items()}
            status = self.vidinfo.cpu().numpy()[3::S2D_VIDINFO_WORDS]
        return annotations_from_layout(self.host_descs, status, tabs)

    def serialize(self, stream=None) -> int:
        """Enqueue the annotation json (s2d_annotation_json) of the layout tables on `stream` (default: torch's current
        stream): per video the text of its `annotations` list at aj_out[aj_video_off[v]:aj_video_off[v + 1]], the bytes
        the batch needs in `aj_need`. Follows layout(). The first call allocates the text buffer, so call it once
        before capturing it in a graph. Returns the number of kernel launches."""
        assert "E" in self.stages, 'the annotation json needs a batch built with stage "E"'
        if self.aj_out is None:
            self.grow_json(self.aj_cap)
        st = stream if stream is not None else torch.cuda.current_stream(self.device).cuda_stream
        p = lambda t: t.data_ptr()
        with torch.cuda.device(self.device):
            _lib.call("s2d_annotation_json", p(self.descs), self.nv, self.total_rows, p(self.vidinfo), p(self.al_vann),
                      p(self.al_ann), p(self.al_members), p(self.al_member_off), p(self.al_chars), self.str_cap,
                      p(self.al_clusters), p(self.al_pairs), p(self.al_sizes), p(self.aj_work), self.aj_cap, p(self.aj_out),
                      p(self.aj_video_off), p(self.aj_need), st)
        return 3

    def grow_json(self, need: int):
        """(Re)allocate the json text buffer for at least `need` bytes; serialize() has to be run again."""
        self.aj_cap = max(int(need), self.aj_cap if self.aj_out is not None else 0)
        self.aj_out = torch.empty(max(1, self.aj_cap), dtype=torch.uint8, device=self.device)

    def annotation_json(self):
        """Per video the json text of its `annotations` list as bytes, byte-identical to
        `json.dumps(self.annotations()[v]).encode()`, or None when the video's final status is not 1. Needs a batch
        built with "E" in its stages, after run() or replay(). The stage-E capacities are settled as in annotations(),
        then the layout and the json are enqueued on the device; only the used bytes and the offsets are copied back.
        When the text buffer was short it is grown and the json call alone re-run (the layout tables are intact).
        keymask_ident.annotations.write_video_annotations writes the bytes into the video's file."""
        with torch.cuda.device(self.device):
            self._settle_rle()
            self.layout()
            self.serialize()
            need = int(self.aj_need.item())
            if need > self.aj_cap:
                self.grow_json(need)
                self.serialize()
            off = self.aj_video_off.cpu().tolist()
            text = self.aj_out[:need].cpu().numpy().tobytes()
        return [text[off[v]:off[v + 1]] if off[v + 1] > off[v] else None for v in range(self.nv)]


# layout table -> (int32 / int64 / byte elements per entry, index of its entry count in al_sizes)
LAYOUT_TABLES = {"ann": (7, 0), "members": (6, 1), "member_off": (1, 1), "chars": (1, 2), "clusters": (2, 3), "pairs": (2, 4)}


def annotations_from_layout(descs, status, tabs):
    """The `annotations` lists of a batch from host copies of its layout tables (Batch.layout_views): per video the
    reference's json objects, None when `status` (vidinfo[3] per video) is not 1. Only slices: every choice was made
    on the device."""
    vann = tabs["vann"].reshape(-1, 2).tolist()
    ann = tabs["ann"].reshape(-1, 7).tolist()
    mem = tabs["members"].reshape(-1, 6).tolist()
    moff = tabs["member_off"].tolist() + [len(tabs["chars"])]
    chars = tabs["chars"].tobytes().decode("ascii")
    clusters = tabs["clusters"].reshape(-1, 2).tolist()
    pairs = tabs["pairs"].reshape(-1, 2).tolist()
    out = []
    for vi, d in enumerate(descs):
        if int(status[vi]) != 1:
            out.append(None)
            continue
        T, H, W = d.T, d.H, d.W
        n, a0 = vann[vi]
        anns = []
        for k in range(n):
            _, _, gn, gs, ci, m0, nm = ann[a0 + k]
            segs, boxes, areas = [None] * T, [None] * T, [None] * T
            for m in range(m0, m0 + nm):
                f, x0, y0, x1, y1, a = mem[m]
                segs[f] = {"size": [H, W], "counts": chars[moff[m]:moff[m + 1]]}
                boxes[f] = [float(x0), float(y0), float(x1 - x0 + 1), float(y1 - y0 + 1)]
                areas[f] = a
            p0, npairs = clusters[ci]
            anns.append({"video_id": 1, "iscrowd": 0, "height": H, "width": W, "length": T,
                         "segmentations": segs, "bboxes": boxes, "areas": areas, "category_id": 1,
                         "id": k + 1, "one2x": round(gs / gn, 2) if gn else 0.0,
                         "visibility_ranges": [list(x) for x in pairs[p0:p0 + npairs]]})
        out.append(anns)
    return out


def pack_vis_bits(vis: torch.Tensor) -> torch.Tensor:
    """[Nm,T,P] visibility flags (bool / u8) -> int32 [Nm,T,ceil(P/32)] words, bit p % 32 of word p // 32 = flag p: the
    producer-side wire format of S2D_DESC_VIS_BITS (torch plumbing; one pass over the flags where they are born)."""
    Nm, T, P = vis.shape
    pw = (P + 31) // 32
    b = (vis != 0)
    if pw * 32 != P:
        b = torch.nn.functional.pad(b, (0, pw * 32 - P))
    w = b.reshape(Nm, T, pw, 32).to(torch.int64) << torch.arange(32, device=vis.device, dtype=torch.int64)
    w = w.sum(dim=3)
    return torch.where(w >= 2 ** 31, w - 2 ** 32, w).to(torch.int32).contiguous()


def _setbits(words: np.ndarray, limit: int):
    out = []
    for w, m in enumerate(words.tolist()):
        m &= 0xFFFFFFFF
        while m:
            b = (m & -m).bit_length() - 1
            m &= m - 1
            i = w * 32 + b
            if i < limit:
                out.append(i)
    return out


def discover_keymasks(videos: List[VideoInput], params: Params = Params(), want_comps: bool = True,
                      annotations: Union[bool, str] = False):
    """Public in-memory entry point: run stages A-D for a batch of videos on their device and
    return one result dict per video. annotations=True runs stage E as well: each dict gains "annotations", the
    YTVIS annotation list the reference writes for the video (None when its status is not 1; see
    Batch.annotations and keymask_ident.annotations.write_video_annotations). annotations="json" gains
    "annotation_json" instead: the json text of that list as bytes, serialised on the device (Batch.annotation_json)."""
    if annotations not in (False, True, "json"):
        raise ValueError(f"annotations must be False, True or 'json', not {annotations!r}")
    b = Batch(videos, stages="LVBDE" if annotations else "LVBD")
    b.run(params)
    torch.cuda.synchronize(b.device)
    res = b.decode(want_comps=want_comps)
    if annotations == "json":
        for r, a in zip(res, b.annotation_json()):
            r["annotation_json"] = a
    elif annotations:
        for r, a in zip(res, b.annotations(res)):
            r["annotations"] = a
    return res
