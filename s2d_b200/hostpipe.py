"""End-to-end entry for HOST buffers: keymask discovery of a list of videos whose label maps, tracks and visibility
flags live in (page-locked) host memory - what a caller has when the upstream producers ran elsewhere. Chunks of
videos are staged into two device sets on two copy streams, so the host -> device DMA of chunk c + 1 overlaps the
kernels of chunk c; per chunk only the small result tables travel back (status, clusters, windows, group labels,
one2x flags: ~70 KB per video).

This is the path bench.py's `e2e` record times. It is bound by the DMA (61 GB per C2 batch at ~55 GB/s per GPU
against 14 ms of kernels), which is why the wire format matters: visibility flags travel bit-packed
(S2D_DESC_VIS_BITS, 1/8 of the bytes), tracks stay float32 as the tracker produced them."""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Sequence, Union

import torch

from ._lib import S2D_VIDINFO_WORDS
from .pipeline import LAYOUT_TABLES, Batch, Params, VideoInput, annotations_from_layout


@dataclass
class HostVideo:
    """host tensors of one video (ideally inside a hostmem.PinnedPool)"""
    labels: torch.Tensor                 # u8 [T,H,W]
    tracks: torch.Tensor                 # f32 [Nm,T,P,2]
    vis: torch.Tensor                    # u8 [Nm,T,P] or int32 [Nm,T,ceil(P/32)] when vis_bits
    vis_bits: bool = False
    max_label: Optional[int] = None

    @property
    def nbytes(self) -> int:
        return sum(t.numel() * t.element_size() for t in (self.labels, self.tracks, self.vis))

    def signature(self):
        return (tuple(self.labels.shape), tuple(self.tracks.shape), tuple(self.vis.shape), self.vis_bits, self.max_label)


class HostPipeline:
    """Two staging sets + batches for chunks of `chunk` videos. `like` gives the shapes of the slots: `chunk` entries
    (both sets alike) or 2 * `chunk` entries (even chunks land in the first half's shapes, odd chunks in the second
    half's). The allocation happens here, once; run() only enqueues copies and kernels.

    `annotations=True` adds stage E and its annotation layout (Batch.layout) to every chunk, and run() gives each
    video's YTVIS annotation list as well. Before a staging set is reused, the host reads the stage-E needs and layout
    sizes of the chunk it holds (the next chunk's copies are in flight meanwhile): a short capacity is grown and stage
    E and the layout re-run on that set, whose label maps are still staged; then only the used part of the layout
    tables is copied back.

    `annotations="json"` adds the annotation json (Batch.serialize) after the layout instead: the json text of every
    video's annotation list is made on the device, and only its used bytes and the video offsets are copied back, with
    no Python annotation objects built. The host reads the stage-E needs and the json size before a set is reused;
    a short stage-E capacity re-runs stage E, the layout and the json, a short json buffer the json call alone."""

    RESULT_TABLES = ("vidinfo", "clusterinfo", "rowinfo", "glabel", "one2x")

    def __init__(self, like: Sequence[HostVideo], device, params: Params = Params(), chunk: Optional[int] = None,
                 annotations: Union[bool, str] = False):
        if annotations not in (False, True, "json"):
            raise ValueError(f"annotations must be False, True or 'json', not {annotations!r}")
        self.device = torch.device(device)
        self.params = params
        self.chunk = int(chunk) if chunk else len(like)
        self.annotations = annotations if annotations == "json" else bool(annotations)
        self.json = annotations == "json"
        assert len(like) in (self.chunk, 2 * self.chunk)
        halves = [list(like[:self.chunk]), list(like[-self.chunk:])]
        self.sigs = [[v.signature() for v in h] for h in halves]
        self.sets = []
        with torch.cuda.device(self.device):
            for h in halves:
                dv = [VideoInput(torch.empty(v.labels.shape, dtype=torch.uint8, device=self.device),
                                 torch.empty(v.tracks.shape, dtype=torch.float32, device=self.device),
                                 torch.empty(v.vis.shape, dtype=v.vis.dtype, device=self.device),
                                 vis_bits=v.vis_bits, max_label=v.max_label) for v in h]
                b = Batch(dv, device=self.device, stages="LVBDE" if self.annotations else "LVBD")
                self.sets.append((dv, b))
            self.copy_streams = [torch.cuda.Stream(self.device), torch.cuda.Stream(self.device)]
            self.compute_stream = torch.cuda.Stream(self.device)
        self.host_results: List[dict] = []          # one set of pinned result tables per chunk, grown on first use
        self.host_sizes: List[torch.Tensor] = []    # annotations: per chunk stage E's need (2) and the layout sizes (5)
        #                                             or, with "json", the json bytes (1)
        self.host_layout: List[dict] = []           # annotations: per chunk pinned layout tables (with "json": the json
        #                                             text and video offsets), grown on demand
        self.h2d_bytes = 0
        self.d2h_bytes = 0
        self.launches = 0
        self.reruns = 0

    def run(self, videos: Sequence[HostVideo]) -> List[dict]:
        """All videos, chunk by chunk. Returns one dict of pinned host result tables per chunk (owned by the pipeline,
        overwritten by the next run); with annotations=True each dict also holds "annotations": per video of the chunk,
        in list order, its annotation list (keymask_ident.annotations.write_video_annotations) or None when its status
        is not 1; with annotations="json" it holds "annotation_json" instead: per video the json text of that list as
        bytes, or None. Synchronises the device once at the end, and with annotations twice per chunk as well."""
        assert len(videos) % self.chunk == 0, "the list must be a whole number of chunks"
        nchunks = len(videos) // self.chunk
        while len(self.host_results) < nchunks:      # first call only: pinned result tables for every chunk
            b0 = self.sets[len(self.host_results) % 2][1]
            self.host_results.append({k: torch.empty(getattr(b0, k).shape, dtype=getattr(b0, k).dtype, pin_memory=True)
                                      for k in self.RESULT_TABLES})
            if self.annotations:
                self.host_sizes.append(torch.empty(3 if self.json else 7, dtype=torch.int64, pin_memory=True))
                self.host_layout.append({})
        done = [None, None]
        self.h2d_bytes = self.d2h_bytes = self.launches = self.reruns = 0
        with torch.cuda.device(self.device):
            for c in range(nchunks):
                s = c % 2
                dv, b = self.sets[s]
                copied = None
                if done[s] is not None:
                    if self.annotations:
                        copied = self._collect(c - 2, done[s])    # chunk c - 2 is complete before its set is reused
                    self.copy_streams[s].wait_event(done[s])          # staging set s is free again
                with torch.cuda.stream(self.copy_streams[s]):
                    for j in range(self.chunk):
                        hv = videos[c * self.chunk + j]
                        assert hv.signature() == self.sigs[s][j], "video does not fit the staging slot it lands in"
                        dv[j].labels.copy_(hv.labels, non_blocking=True)
                        dv[j].tracks.copy_(hv.tracks, non_blocking=True)
                        dv[j].vis.copy_(hv.vis, non_blocking=True)
                        self.h2d_bytes += hv.nbytes
                    ready = torch.cuda.Event()
                    ready.record()
                self.compute_stream.wait_event(ready)
                with torch.cuda.stream(self.compute_stream):
                    self.launches += b.run(self.params)
                    if self.annotations:
                        self.launches += b.layout()
                        if self.json:
                            self.launches += b.serialize()
                        self._copy_sizes(c, b)
                    for k in self.RESULT_TABLES:
                        hbuf = self.host_results[c][k]
                        hbuf.copy_(getattr(b, k), non_blocking=True)
                        self.d2h_bytes += hbuf.numel() * hbuf.element_size()
                    done[s] = torch.cuda.Event()
                    done[s].record()
                if copied is not None:
                    # chunk c's copies and step are enqueued: the DMA stays busy while chunk c - 2's json objects are built
                    copied.synchronize()
                    self._assemble(c - 2)
            if self.annotations:
                for c in range(max(0, nchunks - 2), nchunks):
                    self._collect(c, done[c % 2]).synchronize()
                    self._assemble(c)
            self.compute_stream.synchronize()
        return self.host_results[:nchunks]

    def _assemble(self, c):
        """chunk c's annotation lists from its pinned layout tables (copied back already)"""
        b = self.sets[c % 2][1]
        if self.json:
            hl = self.host_layout[c]
            off = hl["video_off"].tolist()
            text = hl["text"][:off[-1]].numpy().tobytes()
            self.host_results[c]["annotation_json"] = [text[off[v]:off[v + 1]] if off[v + 1] > off[v] else None
                                                       for v in range(b.nv)]
            return
        hs = self.host_sizes[c].tolist()
        n = {k: w * int(hs[2 + i]) for k, (w, i) in LAYOUT_TABLES.items()}
        n["vann"] = 2 * b.nv
        tabs = {k: t[:n[k]].numpy() for k, t in self.host_layout[c].items()}
        status = self.host_results[c]["vidinfo"].numpy()[3::S2D_VIDINFO_WORDS]
        self.host_results[c]["annotations"] = annotations_from_layout(b.host_descs, status, tabs)

    def _copy_sizes(self, c, b):
        hs = self.host_sizes[c]
        hs[:2].copy_(b.rle_need, non_blocking=True)
        hs[2:].copy_(b.aj_need if self.json else b.al_sizes, non_blocking=True)
        self.d2h_bytes += hs.numel() * hs.element_size()

    def _collect(self, c, done):
        """Chunk c's annotations: wait for its step, grow and re-run stage E and the layout on its set while a capacity
        was short, then copy the used part of the layout tables to pinned host buffers. Enqueued on the set's copy
        stream, so the set's next host -> device copies follow it. Returns an event recorded after the copies."""
        b = self.sets[c % 2][1]
        st = self.copy_streams[c % 2]
        done.synchronize()
        hs = self.host_sizes[c]
        if self.json:
            return self._collect_json(c, b, st)
        with torch.cuda.stream(st):
            while not b.rle_fits(hs[:2].tolist()):
                b.grow_rle(hs[:2].tolist())
                self.launches += b.run(self.params, stages="E") + b.layout()
                self.reruns += 1
                self._copy_sizes(c, b)
                st.synchronize()
            hl = self.host_layout[c]
            for k, t in b.layout_views(hs[2:].tolist()).items():
                if k not in hl or hl[k].numel() < t.numel():
                    hl[k] = torch.empty(t.numel() + t.numel() // 4 + 64, dtype=t.dtype, pin_memory=True)
                hl[k][:t.numel()].copy_(t, non_blocking=True)
                self.d2h_bytes += t.numel() * t.element_size()
            copied = torch.cuda.Event()
            copied.record()
        return copied

    def _collect_json(self, c, b, st):
        """_collect for annotations="json": re-run what a short capacity left incomplete (stage E, the layout and the json
        when a stage-E buffer was short, the json call alone when its text buffer was), then copy the used json bytes
        and the video offsets to pinned host buffers."""
        hs = self.host_sizes[c]
        with torch.cuda.stream(st):
            while True:
                need = hs.tolist()
                if not b.rle_fits(need[:2]):
                    b.grow_rle(need[:2])
                    self.launches += b.run(self.params, stages="E") + b.layout() + b.serialize()
                elif need[2] > b.aj_cap:
                    b.grow_json(need[2])
                    self.launches += b.serialize()
                else:
                    break
                self.reruns += 1
                self._copy_sizes(c, b)
                st.synchronize()
            hl = self.host_layout[c]
            n = int(hs[2])
            if "text" not in hl or hl["text"].numel() < n:
                hl["text"] = torch.empty(n + n // 4 + 64, dtype=torch.uint8, pin_memory=True)
                hl["video_off"] = torch.empty(b.nv + 1, dtype=torch.int64, pin_memory=True)
            hl["text"][:n].copy_(b.aj_out[:n], non_blocking=True)
            hl["video_off"].copy_(b.aj_video_off, non_blocking=True)
            self.d2h_bytes += n + hl["video_off"].numel() * 8
            copied = torch.cuda.Event()
            copied.record()
        return copied
