"""BASELINE.json's multi-video configurations as runnable workloads: lists of seeded synthetic videos of mixed shapes
(C4: MOSE + VIPSeg mixture), long windowed videos (C3: SA-V-shaped) and the stress sweep (C5), run through the device
pipeline in chunks sized for HBM, with a digest of every video's result tables so that runs on 1, 2, 4 or 8 GPUs can
be compared bit for bit. Generation (the upstream producers' stand-in) is never inside a timed region; the timed
regions are device-timed with CUDA events."""
from __future__ import annotations

import hashlib
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import partition
from ._lib import S2D_CLINFO_WORDS, S2D_MAX_CLUSTERS, S2D_VIDINFO_WORDS
from .pipeline import Batch, Params, VideoInput


@dataclass(frozen=True)
class VideoSpec:
    name: str
    seed: int
    T: int
    H: int
    W: int
    M: int
    P: int
    window: int = 0            # > 0: stage D tracks are stored (and voted) for `window` frames per query only
    vis_bits: bool = False     # visibility flags handed over bit-packed

    @property
    def nq(self) -> int:       # upper bound of the (frame, mask) queries
        return self.M * self.T

    def device_bytes(self) -> int:
        ttr = self.window if self.window > 0 else self.T
        tracks = 8 * self.nq * ttr * self.P
        vis = self.nq * self.T * (((self.P + 31) // 32) * 4 if self.vis_bits else self.P)
        work = 4 * self.nq * self.T * (self.M + 2) + 16 * self.nq * self.T
        gen = (8 if self.window == 0 else 2) * 256 * ttr * self.P * 4      # generator temporaries
        return tracks + vis + self.T * self.H * self.W + work + gen

    def cost(self) -> float:
        ttr = self.window if self.window > 0 else self.T
        return partition.video_cost(ttr, self.H, self.W, self.nq, self.P) + float(self.nq) * self.T * self.P / (8 if self.vis_bits else 1)


def c4_specs(n: int = 512, seed: int = 4, P: int = 1024) -> List[VideoSpec]:
    """BASELINE.json configs[3]: a MOSE + VIPSeg mixture. Even indices are MOSE-like (480p / 720p / 1080p, 20-60 frames),
    odd ones VIPSeg-like (720p, 50-120 frames); 5-30 masks per frame; P tracks per query. Costs span two orders of
    magnitude, which is what the LPT partition is for."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        if i % 2 == 0:
            H, W = [(480, 854), (720, 1280), (1080, 1920)][int(rng.integers(0, 3))]
            T = int(rng.integers(20, 61))
        else:
            H, W, T = 720, 1280, int(rng.integers(50, 121))
        M = int(rng.integers(5, 31))
        out.append(VideoSpec(f"c4_{i:03d}", 40000 + i, T, H, W, M, P))
    return out


def c3_specs(n: int = 16, T: int = 300, H: int = 1080, W: int = 1920, M: int = 30, P: int = 8192, window: int = 64) -> List[VideoSpec]:
    """BASELINE.json configs[2]: SA-V-shaped long videos; per query only a window of <= 64 frames is tracked and voted."""
    return [VideoSpec(f"c3_{i:02d}", 30000 + i, T, H, W, M, P, window=window, vis_bits=True) for i in range(n)]


def c5_points():
    """BASELINE.json configs[4]: masks/frame 10-100 x tracks 1k-16k x window 8-64 frames (480 x 854 videos whose
    length is the window)."""
    return [(M, P, Tw) for M in (10, 20, 50, 100) for P in (1024, 4096, 16384) for Tw in (8, 16, 32, 64)]


def c5_specs(M: int, P: int, Tw: int, target_bytes: float = 3e9, max_videos: int = 16) -> List[VideoSpec]:
    one = VideoSpec("x", 0, Tw, 480, 854, M, P)
    n = int(max(1, min(max_videos, target_bytes // max(1, 9 * one.nq * Tw * P))))
    return [VideoSpec(f"c5_m{M}_p{P}_t{Tw}_{i}", 50000 + 1000 * M + 10 * Tw + P % 7 + i, Tw, 480, 854, M, P) for i in range(n)]


def window_starts(qframe: torch.Tensor, rowinfo4: torch.Tensor, T: int, window: int) -> torch.Tensor:
    """first stored frame per query: the window is centred on the query's own frame, kept inside the cluster's
    visibility window [v0, v1] where that is possible, and inside the video. Device ops, no host round trip."""
    v0 = rowinfo4[:, 2].clamp(min=0)
    v1 = rowinfo4[:, 3].clamp(min=0)
    ts = qframe - window // 2
    ts = torch.minimum(torch.maximum(ts, v0), torch.maximum(v1 + 1 - window, v0))
    return ts.clamp(min=0, max=max(T - window, 0)).to(torch.int32)


def video_digest(summ: dict, vi: int, row0: int, nm: int) -> str:
    """sha256 over the result tables of one video: status / cluster table / per-row (cluster, candidate run, window) /
    group labels / one2x flags - everything decode() builds its output from."""
    h = hashlib.sha256()
    h.update(np.ascontiguousarray(summ["vidinfo"][vi]).tobytes())
    h.update(np.ascontiguousarray(summ["clusterinfo"][vi]).tobytes())
    h.update(np.ascontiguousarray(summ["rowinfo"][row0:row0 + nm]).tobytes())
    h.update(np.ascontiguousarray(summ["glabel"][row0:row0 + nm]).tobytes())
    h.update(np.ascontiguousarray(summ["one2x"][row0:row0 + nm]).tobytes())
    return h.hexdigest()


def list_digest(results: Sequence[dict]) -> str:
    h = hashlib.sha256()
    for r in results:
        h.update(r["name"].encode())
        h.update(r["digest"].encode())
    return h.hexdigest()


class DeviceRunner:
    """Runs a list of VideoSpec through the device pipeline in chunks that fit `budget_bytes` of HBM."""

    def __init__(self, device, params: Params = Params(), budget_bytes: float = 110e9, point_order: str = "raster"):
        self.device = torch.device(device)
        self.params = params
        self.budget = float(budget_bytes)
        self.point_order = point_order

    def chunks(self, specs: Sequence[VideoSpec]) -> List[List[int]]:
        out, cur, used = [], [], 0.0
        for i, s in enumerate(specs):
            b = s.device_bytes()
            if cur and used + b > self.budget:
                out.append(cur)
                cur, used = [], 0.0
            cur.append(i)
            used += b
        if cur:
            out.append(cur)
        return out

    def run_list(self, specs: Sequence[VideoSpec], reps: int = 1, keep_batch: bool = False, warm: int = 0):
        """Every chunk of the list runs `warm` untimed repetitions, then `reps` timed ones. Returns (per-video results of
        the last repetition in list order, stats). stats: device_ms (event-timed kernels + result read-back, summed over
        chunks and timed repetitions), stage_ms, k2 bytes / tiles, frames and launches of all timed repetitions."""
        from .synth import make_scene_device
        dev = self.device
        results: List[Optional[dict]] = [None] * len(specs)
        stats = {"device_ms": 0.0, "frames": 0, "k2_bytes": 0, "k2_tiles": 0, "k2_ms": 0.0, "vis_bytes": 0, "vis_ms": 0.0,
                 "launches": 0, "chunks": 0, "stage_ms": {}}
        last = None
        reps = max(1, reps)
        with torch.cuda.device(dev):
            for idx in self.chunks(specs):
                scenes, vids = [], []
                for i in idx:
                    s = specs[i]
                    sc = make_scene_device(s.seed, s.T, s.H, s.W, s.M, s.P, dev, point_order=self.point_order,
                                           window=s.window, vis_bits=s.vis_bits)
                    scenes.append(sc)
                    vids.append(VideoInput(sc["labels"], sc["tracks"], sc["vis"], tstart=sc.get("tstart"), vis_bits=s.vis_bits,
                                           max_label=s.M, name=s.name))
                batch = Batch(vids, device=dev)
                windowed = any(specs[i].window > 0 for i in idx)
                host = {k: torch.empty(getattr(batch, k).shape, dtype=getattr(batch, k).dtype, pin_memory=True)
                        for k in ("vidinfo", "clusterinfo", "rowinfo", "glabel", "one2x")}
                ms, st = 0.0, {}
                for rep in range(warm + reps):
                    timers = {}
                    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
                    torch.cuda.synchronize(dev)
                    if windowed:
                        ev[0].record()
                        n1 = batch.run(self.params, stages="LVB", timers=timers)
                        ev[1].record()
                        # the windowed tracker run of stage D: untimed (upstream producer), driven by stage B's windows
                        ri = batch.rowinfo.view(-1, 4)
                        for j, i in enumerate(idx):
                            s, d = specs[i], batch.host_descs[j]
                            if s.window > 0:
                                ts = window_starts(batch.qframe[d.row0:d.row0 + d.Nm], ri[d.row0:d.row0 + d.Nm], s.T, s.window)
                                scenes[j]["tstart"].copy_(ts)
                                if rep == 0:
                                    scenes[j]["fill_window"](ts)
                        ev[2].record()
                        n2 = batch.run(self.params, stages="D", timers=timers)
                    else:
                        ev[0].record(); ev[1].record(); ev[2].record()
                        n1, n2 = batch.run(self.params, timers=timers), 0
                    for k, hbuf in host.items():
                        hbuf.copy_(getattr(batch, k), non_blocking=True)
                    ev[3].record()
                    ev[3].synchronize()
                    if rep >= warm:
                        ms += ev[0].elapsed_time(ev[1]) + ev[2].elapsed_time(ev[3])
                        for k, v in timers.items():
                            st[k] = st.get(k, 0.0) + sum(a.elapsed_time(b) for a, b in v)
                stats["device_ms"] += ms
                stats["launches"] += (n1 + n2) * reps
                stats["chunks"] += 1
                for k, v in st.items():
                    stats["stage_ms"][k] = stats["stage_ms"].get(k, 0.0) + v
                summ = dict(vidinfo=host["vidinfo"].numpy().reshape(batch.nv, S2D_VIDINFO_WORDS),
                            clusterinfo=host["clusterinfo"].numpy().reshape(batch.nv, S2D_MAX_CLUSTERS, S2D_CLINFO_WORDS),
                            rowinfo=host["rowinfo"].numpy().reshape(-1, 4), glabel=host["glabel"].numpy(), one2x=host["one2x"].numpy())
                ri = summ["rowinfo"]
                for j, i in enumerate(idx):
                    s, d = specs[i], batch.host_descs[j]
                    rows = ri[d.row0:d.row0 + d.Nm]
                    ok = summ["vidinfo"][j, 1] > 0
                    cand = rows[:, 1] >= 0
                    if s.window > 0:
                        ts = scenes[j]["tstart"].cpu().numpy()
                        lo = np.maximum(rows[:, 2], ts)
                        hi = np.minimum(rows[:, 3], ts + s.window - 1)
                    else:
                        lo, hi = rows[:, 2], rows[:, 3]
                    tiles = int((np.maximum(hi - lo + 1, 0) * cand).sum()) if ok else 0
                    stats["k2_tiles"] += tiles * reps
                    stats["k2_bytes"] += (8 * s.P * tiles + s.T * s.H * s.W + 4 * (d.L + 1) * tiles) * reps
                    stats["vis_bytes"] += (d.Nm * d.T * ((((s.P + 31) // 32) * 4) if s.vis_bits else s.P) + 8 * d.Nm * d.T) * reps
                    stats["frames"] += s.T * reps
                    gl = summ["glabel"][d.row0:d.row0 + d.Nm]
                    results[i] = {"name": s.name, "frames": s.T, "queries": int(d.Nm), "candidates": int(cand.sum()),
                                  "status": int(summ["vidinfo"][j, 3]), "clusters": int(summ["vidinfo"][j, 0]),
                                  "keymasks": int((gl >= 0).sum()), "tiles": tiles,
                                  "digest": video_digest(summ, j, d.row0, d.Nm)}
                stats["k2_ms"] += st.get("point_votes", 0.0)
                stats["vis_ms"] += st.get("vis_reduce", 0.0)
                if keep_batch:
                    last = (batch, scenes, vids)
                else:
                    del batch, scenes, vids, host
                    torch.cuda.empty_cache()
        return results, stats, last
