"""Stage E on the device at C2 scale: bench.py's C2 batch (64 videos x 36 frames 720p, 20 masks/frame, 4096 tracks,
same generator and seed) run with stages "LVBDE".

Reports from CUDA events after warm-up: the time of the label-RLE call (s2d_label_rle, 5 kernels) and the string call
(s2d_rle_strings, 3 kernels), label-map bytes over the label-RLE time as a fraction of the copy peak bench.py uses,
the step time with and without "E" (alternated in one run), the keymask / count / string-byte totals, the host time of
Batch.annotations(), and - for comparison - the previous route on 4 of the videos: keymask planes materialised,
s2d_rle_encode, host string packing. A separate torch.profiler pass gives each kernel's time. The sha256 of the
annotations of a direct run and of a CUDA-graph replay are both recorded (they must be equal).

The annotation layout (s2d_annotation_layout, 3 kernels) is timed with CUDA events around Batch.layout(), and
annotations() with a host clock (it ends in a device synchronise). HostPipeline's frames/s over the 64 videos (a pool
of 8 distinct pinned videos cycled, chunks of 4, bit-packed flags: bench.py's e2e set-up) is measured with and without
annotations, alternated in this one run.

    python tools/stage_e_bench.py --out profiles/r04_annotation_layout_c2.json
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, plim, clk = (x.strip() for x in out.split(","))
        return {"name": name, "power_limit": plim, "sm_max_clock": clk}
    except Exception as e:  # noqa: BLE001
        return {"name": None, "error": str(e)}


def sha(anns):
    return hashlib.sha256(json.dumps(anns, sort_keys=True).encode()).hexdigest()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_annotation_layout_c2.json"))
    args = ap.parse_args()

    import numpy as np
    import torch

    import bench
    from s2d_b200 import _lib
    from s2d_b200.keymask_ident.annotations import coco_rle
    from s2d_b200.pipeline import Batch, Params

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    info = card()
    vids = bench.build_videos("c2", dev, 2024)
    nv, T, H, W, M, P, _ = bench.WORKLOADS["c2"]
    label_bytes = sum(v.labels.numel() for v in vids)
    peak, peak_src = bench._peaks()
    p = Params()
    bE, b0 = Batch(vids, stages="LVBDE"), Batch(vids)
    for _ in range(args.warmup):
        bE.run(p)
        b0.run(p)
    tab = bE.rle_tables()                       # grows the buffers once if the first guess was short
    need = bE.rle_need.cpu().tolist()
    for _ in range(2):
        bE.run(p)
    torch.cuda.synchronize()

    # alternated steps with and without stage E; per-call events inside the E steps
    ev = lambda: torch.cuda.Event(enable_timing=True)
    step_e, step_0, timers = [], [], {}
    for _ in range(args.steps):
        for b, acc, tm in ((bE, step_e, timers), (b0, step_0, None)):
            e0, e1 = ev(), ev()
            e0.record()
            b.run(p, timers=tm)
            e1.record()
            acc.append((e0, e1))
    torch.cuda.synchronize()
    ms = lambda pairs: [a.elapsed_time(b) for a, b in pairs]
    t_e, t_0 = ms(step_e), ms(step_0)
    t_lr, t_rs = ms(timers["label_rle"]), ms(timers["rle_strings"])
    med = lambda x: float(np.median(x))

    # annotation layout on the device, then annotations() end to end (layout, copies, json objects)
    bE.annotations()
    lay = []
    for _ in range(args.steps):
        e0, e1 = ev(), ev()
        e0.record()
        bE.layout()
        e1.record()
        lay.append((e0, e1))
    torch.cuda.synchronize()
    t_lay = ms(lay)
    hosts = []
    for _ in range(3):
        h0 = time.perf_counter()
        anns = bE.annotations()
        hosts.append(time.perf_counter() - h0)
    t_host = min(hosts)
    res = bE.decode(want_comps=False)
    nkeymask = sum(sum(len(a["segmentations"]) - a["segmentations"].count(None) for a in x) for x in anns if x)
    sha_direct = sha(anns)
    bE.capture(p)
    torch.cuda.synchronize()
    bE.rle_chars.fill_(0)
    bE.rle_counts.fill_(0)
    bE.replay()
    sha_graph = sha(bE.annotations(res))

    # per-kernel times: a short profiled run of its own
    kern = {}
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            bE.run(p, stages="E")
        torch.cuda.synchronize()
    for e in prof.key_averages():
        if e.key.startswith(("void s2d::lr_", "void s2d::rs_", "s2d::lr_", "s2d::rs_")) or "lr_strip" in e.key or "rs_kernel" in e.key \
                or "offsets_kernel" in e.key or "lr_diff" in e.key or "lr_frame" in e.key:
            kern[e.key] = {"calls": e.count, "avg_us": (getattr(e, "device_time", None) or e.cuda_time)}

    # previous route on 4 videos: materialised keymask planes -> s2d_rle_encode -> host packer
    st = torch.cuda.current_stream().cuda_stream
    gid_of = bE.gid_of.cpu().numpy().reshape(-1, 256)
    planes, nmask = [], 0
    for vi in range(4):
        d = bE.host_descs[vi]
        for t in range(d.T):
            labs = np.nonzero(gid_of[d.frame0 + t] >= 0)[0]
            planes.append((vids[vi].labels[t][None] == torch.as_tensor(labs, device=dev, dtype=torch.uint8)[:, None, None]))
            nmask += len(labs)
    masks = torch.cat(planes).to(torch.uint8).contiguous()
    n = masks.shape[0]
    max_runs = min(H * W + 1, 8 * W + 64)
    nw = C.c_int64()
    _lib.call("s2d_rle_work_ints", n, H, W, max_runs, C.byref(nw))
    work = torch.empty(nw.value, dtype=torch.int32, device=dev)
    counts = torch.empty((n, max_runs), dtype=torch.int32, device=dev)
    nruns, area, bbox = (torch.empty(k, dtype=torch.int32, device=dev) for k in (n, n, 4 * n))
    enc = []
    for _ in range(3):
        e0, e1 = ev(), ev()
        e0.record()
        _lib.call("s2d_rle_encode", masks.data_ptr(), n, H, W, max_runs, work.data_ptr(), counts.data_ptr(),
                  nruns.data_ptr(), area.data_ptr(), bbox.data_ptr(), st)
        e1.record()
        enc.append((e0, e1))
    torch.cuda.synchronize()
    nr, cn = nruns.cpu().numpy(), counts.cpu().numpy()
    assert int(nr.max()) <= max_runs
    h0 = time.perf_counter()
    for i in range(n):
        coco_rle.to_string(cn[i, :nr[i]].tolist())
    t_pack = time.perf_counter() - h0
    lr = med(t_lr)
    out = {
        "tool": "tools/stage_e_bench.py", "card": info, "version": _lib.load().s2d_version(),
        "workload": "c2: 64 videos x 36 frames 720x1280, 20 masks/frame, 4096 tracks, seed 2024 (bench.py generator)",
        "steps": args.steps, "warmup": args.warmup,
        "label_rle_ms": {"median": lr, "all": t_lr},
        "rle_strings_ms": {"median": med(t_rs), "all": t_rs},
        "stage_e_ms": lr + med(t_rs),
        "label_map_bytes": label_bytes,
        "label_rle_gbs": label_bytes / (lr * 1e-3) / 1e9,
        "label_rle_fraction_of_copy_peak": label_bytes / (lr * 1e-3) / 1e9 / peak,
        "copy_peak_gbs": peak, "copy_peak_source": peak_src,
        "label_rle_reads_of_label_maps": 2,
        "step_ms_with_E": {"median": med(t_e), "all": t_e},
        "step_ms_without_E": {"median": med(t_0), "all": t_0},
        "keymask_rows": int(bE.total_rows), "annotated_keymasks": nkeymask, "counts": int(need[0]), "string_bytes": int(need[1]),
        "counts_capacity_first_guess_fit": bool(tab is not None and need[0] <= bE.rle_cap),
        "annotations_host_s": t_host, "annotations_host_s_all": hosts,
        "annotation_layout_ms": {"median": med(t_lay), "all": t_lay},
        "annotation_layout_sizes": dict(zip(("annotations", "members", "string_bytes", "clusters", "range_pairs"),
                                            bE.al_sizes.cpu().tolist())),
        "hostpipe_frames_per_s": hostpipe_fps(vids, nv, T, dev, p, args.steps),
        "kernels_profiler_us": kern,
        "previous_route_4_videos": {"masks": n, "mask_plane_bytes": int(masks.numel()),
                                    "s2d_rle_encode_ms": med(ms(enc)), "host_pack_s": t_pack},
        "annotations_sha256_direct": sha_direct, "annotations_sha256_graph_replay": sha_graph,
    }
    assert sha_direct == sha_graph, "graph replay gave different annotations"
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("card", "label_rle_ms", "rle_strings_ms", "label_rle_fraction_of_copy_peak",
                                          "step_ms_with_E", "step_ms_without_E", "annotations_host_s",
                                          "annotation_layout_ms", "hostpipe_frames_per_s", "annotations_sha256_direct")},
                     default=str)[:3000])


def hostpipe_fps(vids, nv, T, dev, params, rounds, modes=(("without", False), ("with_annotations", True))):
    """HostPipeline over the whole list for each (name, annotations=) of `modes`, alternated (bench.py's e2e pool and
    chunks); by default without and with annotations"""
    import torch

    from s2d_b200.hostpipe import HostPipeline, HostVideo
    from s2d_b200.pipeline import pack_vis_bits
    chunk, npool = 4, 8
    hv = [HostVideo(v.labels.cpu().pin_memory(), v.tracks.cpu().pin_memory(), pack_vis_bits(v.vis).cpu().pin_memory(),
                    vis_bits=True, max_label=v.max_label) for v in vids[:npool]]
    order = [hv[i % npool] for i in range(nv)]
    pipes = {k: HostPipeline(hv, dev, params, chunk=chunk, annotations=a) for k, a in modes}
    for p in pipes.values():
        p.run(order)                                   # warm-up: pinned host tables, buffer growth
    t = {k: [] for k in pipes}
    for _ in range(max(1, rounds // 3)):
        for k, p in pipes.items():
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            p.run(order)
            t[k].append(nv * T / (time.perf_counter() - t0))
    out = {k: {"median": float(sorted(v)[len(v) // 2]), "all": v} for k, v in t.items()}
    if "with_annotations" in pipes:
        out["reruns_with_annotations"] = pipes["with_annotations"].reruns
    out["reruns"] = {k: p.reruns for k, p in pipes.items()}
    out["d2h_bytes"] = {k: p.d2h_bytes for k, p in pipes.items()}
    return out


if __name__ == "__main__":
    main()
