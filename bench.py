#!/usr/bin/env python
"""Keymask-discovery throughput (frames/s) on B200 - BASELINE.json's metric.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c1|target] [--impl reference]

A step = one pass of the whole hot path (stages A-D: label stats, visibility reduce, DBSCAN #1,
windows, point votes, selection, grouping) over one batch of synthetic videos per GPU. The
default workload is BASELINE.json configs[1]: 64 videos x 36 frames 720p, 20 masks/frame,
4096 tracks per query (one such batch per GPU: videos are independent, so N GPUs run N batches
- weak scaling, no collective on the data path). One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (videos per GPU, T, H, W, masks/frame, tracks/query, description)
    "c2": (64, 36, 720, 1280, 20, 4096, "YouTubeVIS-2021-shaped batch: 64 videos x 36 frames 720p, 20 masks/frame, 4k tracks"),
    "c1": (1, 24, 480, 854, 10, 1000, "single synthetic 24-frame 480x854 video, 10 masks/frame, 1k tracks"),
    "target": (64, 36, 480, 854, 20, 4096, "480p videos, 20 masks/frame, 4k tracks (north_star target shape)"),
    "tiny": (4, 12, 120, 160, 6, 256, "tiny self-test shape"),
}
LIST_WORKLOADS = {
    "c3": "SA-V-shaped long videos: 16 videos x 300 frames 1080p, 30 masks/frame, 8k tracks, windowed overlap (<= 64 frames per query)",
    "c4": "MOSE+VIPSeg mixture: 512 videos (480p-1080p, 20-120 frames, 5-30 masks/frame, 1k tracks) partitioned by video across the GPUs",
    "c5": "stress sweep: masks/frame 10-100 x tracks 1k-16k x window 8-64 frames (480x854), every point vs the CPU baseline",
}
METRIC = "keymask_discovery_frames_per_sec"
UNIT = "frames/s"


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            j = json.load(f)
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu_index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def host_threads():
    """host cores this process may use (cgroup / affinity aware)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def make_config(args, nq):
    """`config` of the JSON line: identical keys and values in both arms (ours / --impl reference)."""
    nvid, T, H, W, M, P, desc = WORKLOADS[args.workload]
    return {"workload": f"{args.workload}: {desc}", "videos_per_gpu": nvid, "frames_per_video": T,
            "resolution": [H, W], "masks_per_frame": M, "tracks_per_query": P, "queries_per_video": int(nq),
            "point_order": args.point_order, "partition": "by video, one batch of videos per GPU (weak scaling)",
            "cache": "inputs per step (tracks+flags+labels) >> 126 MB L2, no flush needed"}


def build_videos(workload, device, seed0, point_order="raster"):
    import torch
    from s2d_b200.pipeline import VideoInput
    from s2d_b200.synth import make_scene_device
    nvid, T, H, W, M, P, _ = WORKLOADS[workload]
    vids = []
    for i in range(nvid):
        sc = make_scene_device(seed0 + i, T, H, W, M, P, device, point_order=point_order)
        vids.append(VideoInput(sc["labels"], sc["tracks"], sc["vis"], max_label=M, name=f"v{i}"))
    torch.cuda.synchronize(device)
    return vids


def cpu_sample(vid, nq, threads=None):
    """Dense torch-CPU port of the reference (oracle/dense_port.py) on `nq` queries of one video over
    the whole video as window; returns (frames/s extrapolated to the video, seconds, pairs)."""
    import numpy as np
    import torch
    from oracle import dense_port
    if threads:
        torch.set_num_threads(threads)
    labels = vid.labels.cpu().numpy()
    T = labels.shape[0]
    Nm = vid.tracks.shape[0]
    qs = list(np.linspace(0, Nm - 1, nq).astype(int))
    tracks = {int(q): vid.tracks[int(q)].cpu().numpy() for q in qs}
    vis = {int(q): vid.vis[int(q)].cpu().numpy() for q in qs}
    lab = torch.from_numpy(labels.astype(np.int64))[..., None]
    t0 = time.perf_counter()
    npairs = 0
    for q in qs:
        _ = dense_port.visibility_rows(torch.from_numpy(vis[int(q)][None].astype(bool)))
        m, c, o = dense_port.match_query_dense(lab, torch.from_numpy(tracks[int(q)]), 0, T - 1,
                                               labels.shape[1], labels.shape[2], 0.5)
        npairs += len(c)
    dt = time.perf_counter() - t0
    per_video = dt / len(qs) * Nm
    return T / per_video, dt, npairs, len(qs)


def reference_arm(args):
    """--impl reference: the reference's CPU algorithm (dense torch-CPU port, all host threads) on a
    bounded sample of the same workload. Rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1 to its workers: the CPU arm must use every host core whatever N is
    ncores = host_threads()
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = str(ncores)
    import torch
    torch.set_num_threads(ncores)
    nvid, T, H, W, M, P, desc = WORKLOADS[args.workload]
    dev = torch.device("cuda:0") if torch.cuda.is_available() else torch.device("cpu")
    from s2d_b200.pipeline import VideoInput
    from s2d_b200.synth import make_scene_device
    sc = make_scene_device(2024, T, H, W, M, P, dev, point_order=args.point_order)
    vid = VideoInput(sc["labels"], sc["tracks"], sc["vis"], max_label=M)
    nq = args.ref_queries
    for _ in range(args.warmup):
        cpu_sample(vid, 1)
    vals, secs = [], []
    for _ in range(args.steps):
        fps, dt, npairs, n = cpu_sample(vid, nq)
        vals.append(fps); secs.append(dt)
    v = sum(vals) / len(vals)
    cores = torch.get_num_threads()
    sample = (f"{nq} of {vid.tracks.shape[0]} queries of one {args.workload} video per step, full-video window "
              f"({T} frames x ~{M} masks per query), dense torch-CPU port of cotracker_matching.extract_mask_matches; "
              f"frames/s extrapolated linearly in queries")
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000 * sum(secs) / len(secs), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int64/u8 (torch CPU)", "data": "synthetic",
            "config": make_config(args, vid.tracks.shape[0]),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default 10); c3 / c4 / c5: timed passes over the list (default 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c2", choices=list(WORKLOADS) + list(LIST_WORKLOADS))
    ap.add_argument("--list-videos", type=int, default=0, help="c3 / c4: number of videos in the list (default 16 / 512)")
    ap.add_argument("--list-scale", type=float, default=1.0, help="c3 / c4 / c5: scale frame size by this factor (smoke runs)")
    ap.add_argument("--hbm-budget-gb", type=float, default=110.0, help="c3 / c4 / c5: HBM per chunk of videos")
    ap.add_argument("--digest-file", default="", help="c3 / c4: JSON file with the digest of a reference run (any GPU count) to compare with")
    ap.add_argument("--write-digest", default="", help="c3 / c4: JSON file that receives this run's digest (merged by workload key)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ref-queries", type=int, default=8, help="queries per step of the reference arm")
    ap.add_argument("--cpu-queries", type=int, default=48, help="queries in the cpu_baseline sample")
    ap.add_argument("--videos", type=int, default=0, help="override videos per GPU (profiling runs)")
    ap.add_argument("--point-order", default="raster", choices=["raster", "random"],
                    help="order of a query's points: raster (CoTracker-like grid order) or random (worst case)")
    ap.add_argument("--graph", action="store_true",
                    help="replay the step as one CUDA graph (launch-bound small workloads such as c1); per-stage "
                         "times then come from one extra un-timed pass")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-vis", default="bits", choices=["bits", "bytes"], help="wire format of the visibility flags in the e2e leg")
    ap.add_argument("--e2e-pool", default="huge", choices=["huge", "torch"],
                    help="host staging pool of the e2e leg: huge-page mapping + cudaHostRegister, or torch pin_memory")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-k1", action="store_true")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the results of the last timed step to DIR/<name>.npy (batch workloads: rank 0's batch)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 1 if args.workload in LIST_WORKLOADS and args.impl == "ours" else 10
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.workload in LIST_WORKLOADS:
        return list_workload(args)
    if args.videos > 0:
        w = WORKLOADS[args.workload]
        WORKLOADS[args.workload] = (args.videos,) + w[1:]
    if args.impl == "reference":
        return reference_arm(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from s2d_b200.pipeline import Batch, Params

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    from s2d_b200 import hostmem
    all_cores = os.sched_getaffinity(0)
    # cores (and with them the first-touch placement of the pinned pools) next to this rank's GPU
    binding = hostmem.bind_to_gpu(local_rank, local_rank, int(os.environ.get("LOCAL_WORLD_SIZE", world)))
    if world > 1:
        # NCCL prints its version banner on STDOUT (NCCL_DEBUG=VERSION/WARN in this image): send its log to
        # stderr so that stdout holds the one JSON line the driver parses
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"          # no version banner on stdout
        dist.init_process_group("nccl", device_id=dev)

    nvid, T, H, W, M, P, desc = WORKLOADS[args.workload]
    vids = build_videos(args.workload, dev, 2024 + 1000 * rank, args.point_order)
    batch = Batch(vids)
    params = Params()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    if args.graph:
        batch.capture(params)
    for _ in range(args.warmup):
        batch.replay() if args.graph else batch.run(params)
    barrier()
    clocks = ClockSampler(local_rank)
    clocks.start()
    timers = {}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    launches = 0
    for _ in range(args.steps):
        if args.graph:
            batch.replay()
            launches += batch.kernel_launches_per_run
        else:
            launches += batch.run(params, timers=timers)
    e1.record()
    barrier()
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, batch)
    if args.graph:                       # per-stage times of the same work, outside the timed region
        for _ in range(3):
            batch.run(params, timers=timers)
        torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    tms = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms_max = float(tms.item())
    frames = nvid * T * world
    value = frames * args.steps / (ms_max / 1000.0)

    stage_ms = {k: sum(a.elapsed_time(b) for a, b in v) / len(v) for k, v in timers.items()}

    # ---- roofline of the dominant kernel (K2 point votes), algorithmic bytes / measured time
    summ = batch.fetch_summary()
    ri = summ["rowinfo"]
    ok = np.repeat(summ["vidinfo"][:, 1] > 0, [d.Nm for d in batch.host_descs])
    cand = (ri[:, 1] >= 0) & ok
    tiles = int(((ri[:, 3] - ri[:, 2] + 1) * cand).sum())
    alg_bytes = 8 * P * tiles + nvid * T * H * W + 4 * (M + 1 + 1) * tiles
    peak, peak_src = _peaks()
    k2_ms = stage_ms["point_votes"]
    achieved = alg_bytes / (k2_ms / 1000.0) / 1e9
    vr_bytes = sum(d.Nm * d.T * d.P + 8 * d.Nm * d.T for d in batch.host_descs)
    pv_name = ("point_votes_warp_kernel (persistent, one warp per tile: tracks by cp.async.bulk, bitmap of the bounding box in "
               "shared memory, labels of first points straight from the label map)" if batch.use_tma and batch.vec4 and P <= 1024 and H * W <= 524288
               else "point_votes_tab_kernel (persistent; tile's tracks by cp.async.bulk, bbox of the label map by TMA "
               "boxes into the same smem buffer, one shared atomic per point)" if batch.use_tma and batch.vec4 and P <= 16384
               else "point_votes_kernel (one CTA per tile)")
    # DRAM traffic of the same launch from the committed `ncu --set full` capture (profiles/), if it
    # was taken on this workload: dram__bytes_read.sum + dram__bytes_write.sum
    traffic = None
    tpath = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "k2_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        from s2d_b200 import _lib
        # only a capture of THIS library revision on THIS workload counts; anything else reads as "not measured"
        if (tj.get("workload") == args.workload and int(tj.get("videos", -1)) == nvid and tj.get("point_order") == args.point_order
                and int(tj.get("lib_version", -1)) == int(_lib.load().s2d_version())):
            traffic = float(tj["dram_bytes_per_launch"])
    roofline = {"kernel": pv_name, "bound": "hbm", "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes, "ms_per_launch": k2_ms, "tiles_per_launch": tiles,
                "share_of_step": k2_ms / (ms / args.steps),
                "vis_reduce": {"achieved": vr_bytes / (stage_ms["vis_reduce"] / 1000.0) / 1e9,
                               "frac": vr_bytes / (stage_ms["vis_reduce"] / 1000.0) / 1e9 / peak,
                               "algorithmic_bytes_per_launch": vr_bytes, "ms_per_launch": stage_ms["vis_reduce"]}}

    # ---- parity spot check against the oracle (outside the timed region)
    parity = "skipped"
    if rank == 0:
        from oracle import keymask_oracle as ko
        v0 = vids[0]
        lab_h = v0.labels.cpu().numpy()
        d0 = batch.host_descs[0]
        hits = batch.hits[d0.hits_off:d0.hits_off + d0.Nm * d0.T * d0.L].cpu().numpy().reshape(d0.Nm, d0.T, d0.L)
        uniq = batch.uniq[d0.vt_off:d0.vt_off + d0.Nm * d0.T].cpu().numpy().reshape(d0.Nm, d0.T)
        qs = [q for q in np.linspace(0, d0.Nm - 1, 6).astype(int) if ri[q, 1] >= 0]
        good = True
        for q in qs:
            a, b = int(ri[q, 2]), int(ri[q, 3])
            h, u = ko.point_votes(v0.tracks[int(q)].cpu().numpy(), lab_h, a, b, nbins=d0.L)
            good &= bool(np.array_equal(u, uniq[q, a:b + 1]) and np.array_equal(h, hits[q, a:b + 1]))
        Vd = batch.V[d0.vt_off:d0.vt_off + d0.Nm * d0.T].cpu().numpy().reshape(d0.Nm, d0.T)
        good &= bool(np.array_equal(Vd[qs], ko.visibility_mean(v0.vis[qs].cpu().numpy())))
        parity = "ok" if good else "MISMATCH"

    # ---- e2e: host buffers, H2D of every video's inputs + D2H of the summary inside the timed region
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, vids, dev, world, params, barrier, binding)

    # ---- K1 on the tensor cores: one-hot Gram matrix of each video's label maps (outside the timed step)
    k1 = None
    if rank == 0 and not args.no_k1:
        k1 = run_k1(vids, batch, M + 1)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        os.sched_setaffinity(0, all_cores)            # the CPU baseline uses every host core, not just the GPU's node
        fps, dt, npairs, n = cpu_sample(vids[0], args.cpu_queries, threads=host_threads())
        cpu = {"value": fps, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
               "sample": (f"{n} of {vids[0].tracks.shape[0]} queries of video 0, full-video window, {npairs} (query,mask) "
                          f"pairs in {dt:.1f} s with the dense torch-CPU port of the reference (oracle/dense_port.py); "
                          f"frames/s extrapolated linearly in queries")}
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "u8/int32 (f32 tracks, f64 scores)",
                "data": "synthetic",
                "config": make_config(args, batch.host_descs[0].Nm), "cuda_graph": bool(args.graph),
                "input_bytes_per_step_per_gpu": int(sum(v.tracks.numel() * 4 + v.vis.numel() + v.labels.numel() for v in vids)),
                "clocks": clk, "e2e": e2e, "gpu_launches": launches, "roofline": roofline,
                "stage_ms": stage_ms, "parity_check": parity, "overlap_gemm": k1, "cpu_baseline": cpu}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


DUMP_BUDGET = 60_000_000          # bytes of all --dump-outputs files together


def write_arrays(out_dir, src, budget=DUMP_BUDGET, seed=0):
    """One out_dir/<name>.npy per entry of `src` (name -> (rows, bytes per row, get(row indices or None) -> array)). The
    arrays share `budget` bytes, smallest first; one that does not fit its share is replaced by rows drawn with a fixed
    seed, whose row numbers go to <name>_rows.npy."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    left = budget
    for i, name in enumerate(sorted(src, key=lambda k: src[k][0] * src[k][1])):
        nrows, row_bytes, get = src[name]
        share = left // (len(src) - i)
        idx = None
        if nrows * row_bytes > share:
            idx = np.sort(np.random.default_rng(seed).choice(nrows, share // (row_bytes + 8), replace=False))
            np.save(os.path.join(out_dir, f"{name}_rows.npy"), idx.astype(np.float64))
            left -= 8 * len(idx)
        a = get(idx)
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
        left -= a.nbytes


def _whole(arrays):
    """write_arrays entries of arrays held in host memory"""
    return {k: (len(a), a[:1].nbytes, lambda idx, a=a: a if idx is None else a[idx]) for k, a in arrays.items()}


def dump_outputs(out_dir, batch, budget=DUMP_BUDGET, seed=0):
    """--dump-outputs of a batch workload: what a caller of the timed path reads back after a step, integers as float64
    (exact), the visibility means V as float32: Batch.fetch_summary's result tables, the query identities and first-stage
    cluster labels per row, V [row, frame], the match bit words, and `votes`, one row per voted (query, frame) tile:
    [row, frame, points inside the frame, points per label 0 .. L-1]. Only entries the step writes are included, so two
    runs with the same arguments give identical files."""
    import numpy as np
    import torch
    descs = batch.host_descs
    T, L = descs[0].T, descs[0].L
    assert all(d.T == T and d.L == L for d in descs), "the batch workloads have one video shape"
    summ = batch.fetch_summary()
    ri = summ["rowinfo"]
    ok = np.repeat(summ["vidinfo"][:, 1] > 0, [d.Nm for d in descs])
    cand = np.nonzero((ri[:, 1] >= 0) & ok)[0]
    n = (ri[cand, 3] - ri[cand, 2] + 1).astype(np.int64)
    rows = np.repeat(cand, n)
    frames = ri[rows, 2] + np.arange(len(rows)) - np.repeat(np.cumsum(n) - n, n)
    f64 = lambda a: np.asarray(a, np.float64)

    def votes(idx):
        r, f = (rows, frames) if idx is None else (rows[idx], frames[idx])
        rt, ft = torch.from_numpy(r).to(batch.device), torch.from_numpy(f.astype(np.int64)).to(batch.device)
        hits = batch.hits.view(-1, T, L)[rt, ft].cpu().numpy()
        uniq = batch.uniq.view(-1, T)[rt, ft].cpu().numpy()
        return np.concatenate([f64(r)[:, None], f64(f)[:, None], f64(uniq)[:, None], f64(hits)], axis=1)

    host = {k: f64(v) for k, v in summ.items()}
    host.update(query_frame=f64(batch.qframe.cpu()), query_label=f64(batch.qlabel.cpu()), labels1=f64(batch.labels1.cpu()),
                V=batch.V.view(-1, T).cpu().numpy(), match_bits=f64(batch.mbits.cpu().numpy().view(np.uint32)))
    src = _whole(host)
    src["votes"] = (len(rows), (3 + L) * 8, votes)
    write_arrays(out_dir, src, budget, seed)


def dump_list_results(out_dir, results):
    """--dump-outputs of a list workload: the per-video results of the last timed pass, in list order, that the digest is
    computed from: `videos` [frames, queries, candidates, status, clusters, keymasks, K2 tiles] and `digests`, the 32
    bytes of each video's sha256 over its result tables (s2d_b200.workloads.video_digest), all as float64."""
    import numpy as np
    keys = ("frames", "queries", "candidates", "status", "clusters", "keymasks", "tiles")
    videos = np.asarray([[r[k] for k in keys] for r in results], np.float64).reshape(-1, len(keys))
    digests = np.asarray([list(bytes.fromhex(r["digest"])) for r in results], np.float64).reshape(-1, 32)
    write_arrays(out_dir, _whole({"videos": videos, "digests": digests}))


def list_specs(args):
    """the video list of a list workload (identical on every rank)"""
    from dataclasses import replace
    from s2d_b200 import workloads as wl
    if args.workload == "c3":
        specs = wl.c3_specs(args.list_videos or 16)
    elif args.workload == "c4":
        specs = wl.c4_specs(args.list_videos or 512)
    else:
        raise ValueError(args.workload)
    if args.list_scale != 1.0:
        f = args.list_scale
        specs = [replace(s, H=max(32, int(s.H * f) // 2 * 2), W=max(32, int(s.W * f) // 2 * 2)) for s in specs]
    return specs


def cpu_sample_spec(spec, nq, threads, device):
    """dense torch-CPU port on `nq` queries of one generated video of `spec` (windowed specs: over the stored window)."""
    import numpy as np
    import torch
    from oracle import dense_port
    from s2d_b200.synth import make_scene_device
    from s2d_b200.workloads import window_starts
    torch.set_num_threads(threads)
    sc = make_scene_device(spec.seed, spec.T, spec.H, spec.W, spec.M, spec.P, device, window=spec.window, vis_bits=spec.vis_bits)
    Nm = sc["tracks"].shape[0]
    qs = [int(q) for q in np.linspace(0, Nm - 1, nq).astype(int)]
    lab = sc["labels"].cpu().long()[..., None]
    T = spec.T
    if spec.window > 0:
        ri = torch.zeros((Nm, 4), dtype=torch.int32, device=sc["query_frame"].device)
        ri[:, 3] = T - 1
        ts = window_starts(sc["query_frame"], ri, T, spec.window)
        sc["fill_window"](ts)
    t0 = time.perf_counter()
    npairs = 0
    for q in qs:
        if spec.window > 0:
            a = int(ts[q])
            full = torch.full((T, spec.P, 2), float("nan"))
            full[a:a + spec.window] = sc["tracks"][q].cpu()
            v0, v1 = a, a + spec.window - 1
        else:
            full, v0, v1 = sc["tracks"][q].cpu(), 0, T - 1
        m, c, o = dense_port.match_query_dense(lab, full, v0, v1, spec.H, spec.W, 0.5)
        npairs += len(c)
    dt = time.perf_counter() - t0
    return T / (dt / len(qs) * Nm), dt, npairs, len(qs), Nm


def list_workload(args):
    """--workload c3 | c4 | c5: a LIST of videos (mixed shapes / long windowed videos / the sweep's points) instead of one
    homogeneous batch per GPU. The list is the same on every rank; s2d_b200.partition assigns videos to ranks (LPT over
    the byte cost), every rank runs its share through the device pipeline in HBM-sized chunks (device-timed), rank 0
    gathers the per-video results (timed) and hashes them: the digest must not depend on the number of GPUs.
    Strong scaling: the total work is fixed. --steps K times K passes over the list: every chunk of videos runs K times
    on the device, the partition and the gather are done K times."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from s2d_b200 import hostmem, partition
    from s2d_b200 import workloads as wl
    from s2d_b200.pipeline import Params

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        if rank != 0:
            return
        ncores = host_threads()
        for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS"):
            os.environ[k] = str(ncores)
        dev = torch.device("cuda:0") if torch.cuda.is_available() else torch.device("cpu")
        if args.workload == "c5":
            specs = [wl.c5_specs(M, P, Tw)[0] for (M, P, Tw) in wl.c5_points()[:: max(1, 48 // max(1, args.ref_queries))]]
        else:
            specs = list_specs(args)
            specs = [specs[i] for i in np.linspace(0, len(specs) - 1, min(len(specs), 3)).astype(int)]
        vals, secs = [], []
        for _ in range(max(1, args.steps)):
            fr, tt, meas = 0.0, 0.0, 0.0
            for sp in specs:
                fps, dt, npairs, n, Nm = cpu_sample_spec(sp, 1, ncores, dev)
                fr += sp.T; tt += sp.T / fps; meas += dt
            vals.append(fr / tt); secs.append(meas)
        v = sum(vals) / len(vals)
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1000 * sum(secs) / len(secs), "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "int64/u8 (torch CPU)", "data": "synthetic",
                "config": {"workload": f"{args.workload}: {LIST_WORKLOADS[args.workload]}", "point_order": args.point_order},
                "cpu_baseline": {"value": v, "unit": UNIT, "cores": ncores, "kind": "port",
                                 "sample": f"1 query of each of {len(specs)} videos spread over the list, dense torch-CPU port, "
                                           f"frames/s extrapolated linearly in queries and averaged by frames"},
                "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), flush=True)
        return

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    all_cores = os.sched_getaffinity(0)
    binding = hostmem.bind_to_gpu(local_rank, local_rank, int(os.environ.get("LOCAL_WORLD_SIZE", world)))
    host_pg = None
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"          # no version banner on stdout
        dist.init_process_group("nccl", device_id=dev)
        # the gather of the per-video results is a HOST exchange (python objects, KBs): its own gloo group, connected
        # before the timed region (one small gather), so that the timed gather is the exchange and not the rendezvous
        host_pg = dist.new_group(backend="gloo")
        warm = [None] * world if rank == 0 else None
        dist.gather_object(("warm", rank), warm, dst=0, group=host_pg)
    runner = wl.DeviceRunner(dev, Params(), budget_bytes=args.hbm_budget_gb * 1e9, point_order=args.point_order)
    peak, peak_src = _peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    clocks = ClockSampler(local_rank)
    if args.workload == "c5":
        return c5_sweep(args, runner, rank, world, dev, barrier, max_over_ranks, clocks, peak, peak_src, all_cores, host_pg)

    specs = list_specs(args)
    costs = [s.cost() for s in specs]
    # warm-up: W small videos through every kernel of the path (attribute opt-ins, allocator, clocks)
    warm = [wl.VideoSpec(f"warm{i}", 7 + i, 24, 240, 426, 8, specs[0].P, window=min(specs[0].window, 16), vis_bits=specs[0].vis_bits)
            for i in range(max(3, args.warmup))]
    runner.run_list(warm)
    barrier()
    clocks.start()
    local_stats = {}

    def worker(idx):
        res, st, _ = runner.run_list([specs[i] for i in idx], reps=args.steps)
        local_stats.update(st)
        return res

    # the gather is timed on its own, after a barrier, so that it measures the exchange and not the ranks' drift
    parts = partition.lpt_partition(costs, world)
    t_part0 = time.perf_counter()
    for _ in range(args.steps):
        mine = partition.lpt_partition(costs, world)[rank]
    t_part = time.perf_counter() - t_part0
    local = worker(mine)
    barrier()
    t_gather = 0.0
    for _ in range(args.steps):
        if world > 1:
            dist.barrier(group=host_pg)               # host-side rendezvous right before the timed exchange
        tg0 = time.perf_counter()
        if world > 1:
            gathered = [None] * world if rank == 0 else None
            dist.gather_object(list(zip(mine, local)), gathered, dst=0, group=host_pg)
            merged = sorted((p for part in gathered for p in part), key=lambda x: x[0]) if rank == 0 else None
        else:
            merged = sorted(zip(mine, local), key=lambda x: x[0])
        t_gather += time.perf_counter() - tg0
    clk = clocks.stop()
    dev_ms = max_over_ranks(local_stats["device_ms"])
    sum_ms = torch.tensor([local_stats["device_ms"], local_stats["k2_ms"], float(local_stats["k2_bytes"]), float(local_stats["k2_tiles"]),
                           float(local_stats["launches"]), local_stats["vis_ms"], float(local_stats["vis_bytes"])], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(sum_ms)
    tot = sum_ms.tolist()
    if rank == 0:
        results = [r for _, r in merged]
        assert [i for i, _ in merged] == list(range(len(specs)))
        digest = wl.list_digest(results)
        if args.dump_outputs:
            dump_list_results(args.dump_outputs, results)
        frames = sum(r["frames"] for r in results)
        total_s = dev_ms / 1000.0 + t_gather + t_part
        ref_digest, equal = None, None
        dpath = args.digest_file or os.path.join(ROOT, "profiles", f"{args.workload}_digest.json")
        if os.path.exists(dpath):
            dj = json.load(open(dpath))
            key = f"{args.workload}/{len(specs)}/{args.list_scale}/{args.point_order}"
            if key in dj:
                ref_digest, equal = dj[key]["digest"], dj[key]["digest"] == digest
        if args.write_digest:
            dj = json.load(open(args.write_digest)) if os.path.exists(args.write_digest) else {}
            dj[f"{args.workload}/{len(specs)}/{args.list_scale}/{args.point_order}"] = {
                "digest": digest, "n_gpus": world, "videos": len(specs), "frames": frames,
                "videos_ok": sum(1 for r in results if r["status"] == 1), "keymasks": sum(r["keymasks"] for r in results)}
            with open(args.write_digest, "w") as f:
                json.dump(dj, f, indent=1, sort_keys=True)
        loads = [sum(costs[i] for i in p) for p in parts]
        k2_gbs = tot[2] / (tot[1] / 1000.0) / 1e9 if tot[1] > 0 else 0.0
        line = {"metric": METRIC, "value": frames * args.steps / total_s, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": len(warm), "ms_per_step": 1000 * total_s / args.steps, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None,
                "dtype": "u8/int32 (f32 tracks, f64 scores)", "data": "synthetic",
                "config": {"workload": f"{args.workload}: {LIST_WORKLOADS[args.workload]}", "videos": len(specs),
                           "frames": frames, "queries": sum(r["queries"] for r in results), "list_scale": args.list_scale,
                           "point_order": args.point_order, "hbm_budget_gb": args.hbm_budget_gb,
                           "partition": f"LPT by video over {world} GPU(s), host gather of per-video results (gather_object over gloo)",
                           "cache": "every chunk's inputs >> 126 MB L2, no flush needed"},
                "timed_region": {"device_ms_max_over_ranks": dev_ms, "gather_ms": 1000 * t_gather, "partition_ms": 1000 * t_part,
                                 "note": "device_ms = CUDA-event time of every chunk's kernels + result read-back, summed over chunks and "
                                         "steps per rank, max over ranks; generation of the synthetic inputs (upstream producers) is outside; "
                                         "gather and partition summed over steps, each gather timed after a barrier"},
                "balance": {"max_over_mean_cost": max(loads) / (sum(loads) / len(loads)), "device_ms_sum_over_ranks": tot[0]},
                "clocks": clk, "gpu_launches": int(tot[4]),
                "roofline": {"kernel": "point_votes_tab_kernel (all chunks of all ranks)", "bound": "hbm", "achieved": k2_gbs, "peak": peak,
                             "unit": "GB/s", "frac": k2_gbs / peak, "traffic": None, "peak_source": peak_src,
                             "algorithmic_bytes": tot[2], "ms_sum_over_ranks": tot[1], "tiles": int(tot[3]),
                             "vis_reduce": {"achieved": tot[6] / (tot[5] / 1000.0) / 1e9 if tot[5] > 0 else None, "algorithmic_bytes": tot[6], "ms": tot[5]}},
                "results": {"digest": digest, "reference_digest": ref_digest, "results_equal": equal,
                            "videos_ok": sum(1 for r in results if r["status"] == 1), "keymasks": sum(r["keymasks"] for r in results),
                            "candidates": sum(r["candidates"] for r in results)},
                "stage_ms_rank0": {k: round(v, 3) for k, v in local_stats["stage_ms"].items()},
                "e2e": None, "cpu_binding": binding}
        if world == 1 and not args.no_cpu:
            os.sched_setaffinity(0, all_cores)
            sp = specs[len(specs) // 2]
            fps, dt, npairs, n, Nm = cpu_sample_spec(sp, 1, host_threads(), dev)
            line["cpu_baseline"] = {"value": fps, "unit": UNIT, "cores": host_threads(), "kind": "port",
                                    "sample": f"1 of {Nm} queries of video {sp.name} ({sp.T} x {sp.H}x{sp.W}, window {sp.window or sp.T}), "
                                              f"{npairs} pairs in {dt:.1f} s, extrapolated linearly in queries"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def c5_sweep(args, runner, rank, world, dev, barrier, max_over_ranks, clocks, peak, peak_src, all_cores, host_pg=None):
    """the 48 points of the sweep are dealt to the ranks round-robin by cost; per point: frames/s of the device path, the
    K2 roofline fraction, and the CPU port on one query of the same video (all host cores / ranks per rank). Every point's
    videos run once untimed (it warms the shape), then --steps timed times."""
    import torch
    import torch.distributed as dist
    from s2d_b200 import partition
    from s2d_b200 import workloads as wl
    pts = wl.c5_points()
    plists = [wl.c5_specs(M, P, Tw) for (M, P, Tw) in pts]
    if args.list_scale != 1.0:
        from dataclasses import replace
        f = args.list_scale
        plists = [[replace(s, H=max(32, int(s.H * f) // 2 * 2), W=max(32, int(s.W * f) // 2 * 2)) for s in pl] for pl in plists]
    costs = [sum(s.cost() for s in pl) for pl in plists]
    mine = partition.lpt_partition(costs, world)[rank]
    runner.run_list([wl.VideoSpec(f"warm{i}", 7 + i, 16, 240, 426, 8, 1024) for i in range(3)])
    barrier()
    clocks.start()
    out = []
    dev_ms = 0.0
    threads = max(1, len(all_cores) // world)
    for pi in mine:
        M, P, Tw = pts[pi]
        res, st, _ = runner.run_list(plists[pi], reps=args.steps, warm=1)
        dev_ms += st["device_ms"]
        k2 = st["k2_bytes"] / (st["k2_ms"] / 1000.0) / 1e9 if st["k2_ms"] > 0 else 0.0
        rec = {"masks_per_frame": M, "tracks": P, "window": Tw, "videos": len(plists[pi]), "frames": st["frames"],
               "frames_per_s": st["frames"] / (st["device_ms"] / 1000.0), "device_ms": st["device_ms"],
               "k2_gbs": k2, "k2_frac": k2 / peak, "k2_ms": st["k2_ms"], "videos_ok": sum(1 for r in res if r["status"] == 1),
               "digest": wl.list_digest(res)}
        if not args.no_cpu:
            fps, dt, npairs, n, Nm = cpu_sample_spec(plists[pi][0], 1, threads, dev)
            rec["cpu_frames_per_s"] = fps
            rec["cpu_sample"] = f"1 of {Nm} queries, {npairs} pairs in {dt:.2f} s on {threads} threads"
        out.append((pi, rec, res))
    barrier()
    clk = clocks.stop()
    if world > 1:
        gathered = [None] * world if rank == 0 else None
        dist.gather_object(out, gathered, dst=0, group=host_pg)
        merged = sorted((p for part in gathered for p in part), key=lambda x: x[0]) if rank == 0 else None
    else:
        merged = sorted(out, key=lambda x: x[0])
    t_max = max_over_ranks(dev_ms)
    if rank == 0:
        recs = [r for _, r, _ in merged]
        if args.dump_outputs:
            dump_list_results(args.dump_outputs, [v for _, _, res in merged for v in res])
        frames = sum(r["frames"] for r in recs)
        fr = [r["k2_frac"] for r in recs]
        line = {"metric": METRIC, "value": frames / (t_max / 1000.0), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": 3,
                "ms_per_step": t_max / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "u8/int32 (f32 tracks, f64 scores)", "data": "synthetic",
                "config": {"workload": f"c5: {LIST_WORKLOADS['c5']}", "points": len(recs), "list_scale": args.list_scale,
                           "partition": f"LPT by sweep point over {world} GPU(s)", "cache": "inputs per point >> 126 MB L2"},
                "clocks": clk, "roofline": {"kernel": "point_votes_tab_kernel", "bound": "hbm", "unit": "GB/s", "peak": peak, "peak_source": peak_src,
                                           "frac_min": min(fr), "frac_median": sorted(fr)[len(fr) // 2], "frac_max": max(fr),
                                           "achieved": sorted(r["k2_gbs"] for r in recs)[len(recs) // 2], "frac": sorted(fr)[len(fr) // 2], "traffic": None},
                "cpu_baseline": None if args.no_cpu else {
                    "value": frames / sum(r["frames"] / r["cpu_frames_per_s"] for r in recs), "unit": UNIT, "cores": threads, "kind": "port",
                    "sample": "1 query of the first video of every sweep point, dense torch-CPU port, extrapolated linearly in queries; frames-weighted"},
                "sweep": recs, "e2e": None}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_k1(vids, batch, L):
    """Cross-frame mask-overlap matrix of a video (all (frame,label) masks against each other) as an int8
    contraction on the tensor cores, operands synthesised on-chip from the label maps. Reports achieved
    TOP/s against an int8 GEMM peak measured here with cuBLASLt (torch._int_mm 8192^3)."""
    import ctypes as C
    import numpy as np
    import torch
    from s2d_b200 import _lib
    dev = vids[0].labels.device
    st = torch.cuda.current_stream(dev).cuda_stream

    def timeit(fn, iters, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize(dev)
        return a.elapsed_time(b) / iters

    n = 8192
    x = torch.randint(-3, 3, (n, n), dtype=torch.int8, device=dev)
    y = torch.randint(-3, 3, (n, n), dtype=torch.int8, device=dev)
    peak = 2.0 * n ** 3 / (timeit(lambda: torch._int_mm(x, y), 10) * 1e-3) / 1e12
    del x, y
    T, H, W = vids[0].labels.shape
    if (H * W) % 16:
        return {"skipped": "pixel count is not a multiple of 16"}
    R = T * L
    nv = min(8, len(vids))
    nw = C.c_int64()
    _lib.call("s2d_overlap_gram_work_ints", T, L, H * W, C.byref(nw))
    work = torch.empty(nw.value, dtype=torch.int32, device=dev)
    G = torch.empty(R * R, dtype=torch.int32, device=dev)

    def run():
        for v in vids[:nv]:
            _lib.call("s2d_overlap_gram_labels", v.labels.data_ptr(), T, L, H * W, work.data_ptr(), G.data_ptr(), st)
    ms = timeit(run, 5) / nv
    # exact check of the WHOLE matrix of the last video run against two independent paths: (i) the bit-packed
    # AND + popc kernel of this library on explicit one-hot planes (s2d_overlap_bits, itself checked against the oracle
    # in tests/), (ii) cuBLASLt's int8 GEMM on the same planes; and its diagonal against K0's mask areas
    d = batch.host_descs[nv - 1]
    area = batch.area[d.frame0 * 256:(d.frame0 + T) * 256].reshape(T, 256)[:, :L].reshape(-1)
    Gm = G.reshape(R, R)
    lab = vids[nv - 1].labels.reshape(T, 1, H * W)
    X = (lab == torch.arange(L, dtype=torch.uint8, device=dev)[None, :, None]).reshape(R, H * W).to(torch.uint8)
    nwords = (H * W + 31) // 32
    Xb = torch.empty((R, nwords), dtype=torch.int32, device=dev)
    _lib.call("s2d_pack_bits", X.data_ptr(), R, H * W, Xb.data_ptr(), st)
    Gb = torch.empty((R, R), dtype=torch.int32, device=dev)
    aA = torch.empty(R, dtype=torch.int32, device=dev)
    aB = torch.empty(R, dtype=torch.int32, device=dev)
    _lib.call("s2d_overlap_bits", Xb.data_ptr(), R, Xb.data_ptr(), R, nwords, Gb.data_ptr(), aA.data_ptr(), aB.data_ptr(), st)
    checks = {"vs_overlap_bits_full_matrix": bool(torch.equal(Gm, Gb)),
              "diagonal_vs_label_areas": bool(torch.equal(Gm.diagonal(), area)),
              "symmetric": bool(torch.equal(Gm, Gm.t()))}
    try:
        Rp8 = (R + 7) // 8 * 8
        Xp = torch.zeros((Rp8, H * W), dtype=torch.int8, device=dev)
        Xp[:R] = X.view(torch.int8)
        Gc = torch._int_mm(Xp, Xp.t().contiguous())[:R, :R]
        checks["vs_cublaslt_int8_full_matrix"] = bool(torch.equal(Gm, Gc))
        del Xp, Gc
    except Exception as e:                       # the library check is optional; the repo's own path above is not
        checks["vs_cublaslt_int8_full_matrix"] = f"not run: {type(e).__name__}"
    del X, Xb, Gb
    ops = 2.0 * R * R * H * W                      # algorithmic: every pair of rows once
    tops = ops / (ms * 1e-3) / 1e12
    ex = C.c_double()
    _lib.call("s2d_overlap_gram_executed_ops", T, L, H * W, C.byref(ex))   # what the tensor cores really execute
    tops_exec = ex.value / (ms * 1e-3) / 1e12
    tiling = C.c_int(-1)
    _lib.call("s2d_overlap_gram_tiling", T, L, C.byref(tiling))
    kname = {2: "gram_labels2_kernel: one-hot operands synthesised in smem by two producer groups on alternate k-blocks, two "
                "tcgen05.mma kind::i8 M128xN256 groups per k-block into 512 int32 TMEM columns; only the 256x256 blocks on or "
                "above the diagonal of the symmetric overlap matrix are executed",
             1: "gram_labels_kernel<256>: one-hot operands synthesised in smem, tcgen05.mma kind::i8 M128xN256, int32 in TMEM; "
                "only the 128x256 tiles touching the upper triangle are executed (too few labels per frame for the label "
                "ring of the 256x256 kernel)",
             0: "gram_labels_kernel<128>: one-hot operands synthesised in smem, tcgen05.mma kind::i8 M128xN128, int32 in TMEM; "
                "only the 128x128 tiles touching the upper triangle are executed (small matrix, or too few labels per frame "
                "for the label ring of the wider tilings)"}[tiling.value]
    return {"kernel": kname, "tiling": tiling.value,
            "rows": R, "pixels": H * W, "ms_per_video": ms, "achieved": tops_exec, "unit": "TOP/s",
            "peak": peak, "peak_source": "measured here: torch._int_mm 8192^3 (cuBLASLt int8)", "frac": tops_exec / peak,
            "frac_of_nominal_4500": tops_exec / 4500.0,
            "note": "achieved / frac count the EXECUTED tensor-core ops (upper-triangle tiles only, partial tiles in full)",
            "algorithmic": {"ops_per_video": ops, "achieved": tops, "frac": tops / peak},
            "hbm_bytes_per_video": int(T * H * W),
            "check": "ok" if all(v is True or isinstance(v, str) for v in checks.values()) and checks["vs_overlap_bits_full_matrix"] else "MISMATCH",
            "checks": checks}


def run_e2e(args, vids, dev, world, params, barrier, binding):
    """Same metric through the public host-buffer API (s2d_b200.hostpipe.HostPipeline): every step copies every video's
    inputs from page-locked host memory (a pool of distinct videos, cycled), runs the path, reads the result tables
    back. Chunks of videos are double-buffered on two copy streams so the DMA overlaps the kernels. Visibility flags
    travel bit-packed (the producer-side wire format, S2D_DESC_VIS_BITS) unless --e2e-vis bytes."""
    import torch
    import torch.distributed as dist
    from s2d_b200 import hostmem
    from s2d_b200.hostpipe import HostPipeline, HostVideo
    from s2d_b200.pipeline import pack_vis_bits
    nvid, T, H, W, M, P, _ = WORKLOADS[args.workload]
    chunk = min(4, nvid)
    npool = min(nvid, 2 * chunk)
    bits = args.e2e_vis == "bits"
    src = []
    for i in range(npool):
        v = vids[i]
        src += [v.labels, v.tracks, pack_vis_bits(v.vis) if bits else v.vis]
    if args.e2e_pool == "huge":
        pool, host = hostmem.pooled_copies(src, huge=True)
        pool_desc = {"kind": "anonymous mapping + cudaHostRegister", "transparent_huge_pages": bool(pool.huge), "bytes": pool.nbytes}
    else:
        pool, host = None, [t.cpu().pin_memory() for t in src]
        pool_desc = {"kind": "cudaHostAlloc (torch pin_memory)"}
    del src
    hv = [HostVideo(host[3 * i], host[3 * i + 1], host[3 * i + 2], vis_bits=bits, max_label=M) for i in range(npool)]
    pipe = HostPipeline(hv[:2 * chunk] if npool >= 2 * chunk else hv[:chunk], dev, params, chunk=chunk)
    steps = args.steps
    order = [hv[i % npool] for i in range(nvid)]

    pipe.run(order)                                   # warm-up (allocates the pinned result tables)
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        pipe.run(order)
    barrier()
    dt = time.perf_counter() - t0
    tt = torch.tensor([dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dt = float(tt.item())
    # what the platform gives a bare copy loop at this GPU count: the same pool, cudaMemcpyAsync only, all ranks at once
    barrier()
    probe_bytes, tp0 = 0, time.perf_counter()
    dst = pipe.sets[0][0]
    with torch.cuda.device(dev):
        while time.perf_counter() - tp0 < 1.0:
            for j in range(chunk):
                dst[j].tracks.copy_(hv[j].tracks, non_blocking=True)
                probe_bytes += hv[j].tracks.numel() * 4
            torch.cuda.synchronize(dev)
    tp = time.perf_counter() - tp0
    barrier()
    probe = torch.tensor([probe_bytes / tp / 1e9], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(probe, op=dist.ReduceOp.MIN)
    nchunks = nvid // chunk
    return {"value": nvid * T * world * steps / dt, "unit": UNIT, "h2d_bytes_per_step": int(pipe.h2d_bytes),
            "d2h_bytes_per_step": int(pipe.d2h_bytes), "steps": steps, "ms_per_step": 1000 * dt / steps,
            "h2d_gbs_per_gpu": pipe.h2d_bytes * steps / dt / 1e9,
            "h2d_probe_gbs_per_gpu": float(probe.item()),
            "h2d_probe": "bare cudaMemcpyAsync loop over the same pinned pool, all ranks concurrently, min over ranks: the platform's "
                         "host -> device ceiling at this GPU count",
            "gpu_launches_per_step": pipe.launches,
            "wire_format": {"tracks": "f32 (x, y) as produced", "labels": "u8",
                            "visibility": "bit-packed u32 (S2D_DESC_VIS_BITS)" if bits else "u8 flags"},
            "host_pool": pool_desc, "cpu_binding": binding,
            "note": f"{nchunks} chunks of {chunk} videos per step from a page-locked pool of {npool} distinct videos, "
                    f"copies double-buffered against compute; bound by the host -> device DMA"}


if __name__ == "__main__":
    main()
