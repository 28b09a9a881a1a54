"""The annotation json of stage E (s2d_annotation_json) at C2 scale: bench.py's C2 batch (64 videos x 36 frames 720p, 20
masks/frame, 4096 tracks, same generator and seed) run with stages "LVBDE", measured in one run.

- the json call (3 kernels) with CUDA events around Batch.serialize(), median after warm-up, with the bytes it reads
  (the layout tables and strings, twice: a length pass and a write pass) and writes (the text);
- Batch.annotation_json() end to end against Batch.annotations() plus json.dumps per video (host clock, both end in a
  device synchronise), alternated;
- writing the 64 per-video files with write_video_annotations from the bytes against from the lists (json.dump),
  alternated, into a temporary directory (each video folder holds 36 one-pixel images);
- HostPipeline frames/s with annotations off, True and "json", alternated (a pool of 8 distinct pinned videos cycled,
  chunks of 4, bit-packed flags: bench.py's e2e set-up);
- the sha256 of the concatenated json bytes and of json.dumps of annotations() in the same run (they must be equal).

    python tools/annotation_json_bench.py --out profiles/r05_annotation_json_c2.json
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import shutil
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_annotation_json_c2.json"))
    args = ap.parse_args()

    import numpy as np
    import torch
    from PIL import Image

    import bench
    from s2d_b200 import _lib
    from s2d_b200.keymask_ident.annotations import write_video_annotations
    from s2d_b200.pipeline import Batch, Params
    from stage_e_bench import card, hostpipe_fps

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    info = card()
    vids = bench.build_videos("c2", dev, 2024)
    nv, T, H, W, M, P, _ = bench.WORKLOADS["c2"]
    p = Params()
    b = Batch(vids, stages="LVBDE")
    for _ in range(args.warmup):
        b.run(p)
    anns = b.annotations()                              # settles the stage-E capacities
    texts = b.annotation_json()                         # settles the json capacity
    torch.cuda.synchronize()

    ev = lambda: torch.cuda.Event(enable_timing=True)
    ms = lambda pairs: [a.elapsed_time(c) for a, c in pairs]
    med = lambda x: float(np.median(x))
    for _ in range(args.warmup):
        b.serialize()
    kern = []
    for _ in range(args.steps):
        e0, e1 = ev(), ev()
        e0.record()
        b.serialize()
        e1.record()
        kern.append((e0, e1))
    torch.cuda.synchronize()
    t_kern = ms(kern)
    sizes = b.al_sizes.cpu().tolist()
    need = int(b.aj_need.item())
    A, Mm, S, K, R = (int(x) for x in sizes)
    table_bytes = 28 * A + 3 * 24 * Mm + 8 * Mm + 8 * K + 8 * R   # ann rows, member rows (3 lists), offsets, clusters, pairs
    bytes_read = 2 * (S + table_bytes)

    # end to end: annotation_json() against annotations() + json.dumps, alternated
    e2e_json, e2e_lists = [], []
    for _ in range(5):
        h0 = time.perf_counter()
        texts = b.annotation_json()
        e2e_json.append(time.perf_counter() - h0)
        h0 = time.perf_counter()
        anns = b.annotations()
        dumped = [None if a is None else json.dumps(a).encode() for a in anns]
        e2e_lists.append(time.perf_counter() - h0)
    sha_json = hashlib.sha256(b"".join(x for x in texts if x is not None)).hexdigest()
    sha_lists = hashlib.sha256(b"".join(x for x in dumped if x is not None)).hexdigest()
    identical = texts == dumped

    # the 64 files, from bytes and from lists
    tmp = tempfile.mkdtemp(prefix="s2d_json_bench_")
    try:
        px = os.path.join(tmp, "px.jpg")
        Image.fromarray(np.zeros((1, 1, 3), np.uint8)).save(px)
        dirs = []
        for v in range(nv):
            d = os.path.join(tmp, "videos", f"video_{v:03d}")
            os.makedirs(d)
            for f in range(T):
                shutil.copyfile(px, os.path.join(d, f"{f:05d}.jpg"))
            dirs.append(d)
        w_bytes, w_lists = [], []
        for r in range(3):
            for src, acc, tag in ((texts, w_bytes, "bytes"), (anns, w_lists, "lists")):
                out = os.path.join(tmp, f"out_{tag}_{r}")
                h0 = time.perf_counter()
                for d, a in zip(dirs, src):
                    write_video_annotations(d, a, out)
                acc.append(time.perf_counter() - h0)
        files_identical = all(
            open(os.path.join(tmp, "out_bytes_0", n), "rb").read() == open(os.path.join(tmp, "out_lists_0", n), "rb").read()
            for n in os.listdir(os.path.join(tmp, "out_lists_0")))
        nfiles = len(os.listdir(os.path.join(tmp, "out_lists_0")))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)

    out = {
        "tool": "tools/annotation_json_bench.py", "card": info, "version": _lib.load().s2d_version(),
        "workload": "c2: 64 videos x 36 frames 720x1280, 20 masks/frame, 4096 tracks, seed 2024 (bench.py generator)",
        "steps": args.steps, "warmup": args.warmup,
        "annotation_json_ms": {"median": med(t_kern), "all": t_kern,
                               "note": "CUDA events around Batch.serialize(): aj_text_kernel<length>, aj_scan_kernel, "
                                       "aj_text_kernel<write>; inputs are L2-resident after the layout"},
        "layout_sizes": dict(zip(("annotations", "members", "string_bytes", "clusters", "range_pairs"), sizes)),
        "json_bytes_written": need, "bytes_read_two_passes": bytes_read,
        "json_write_gbs": need / (med(t_kern) * 1e-3) / 1e9,
        "annotation_json_e2e_s": {"min": min(e2e_json), "all": e2e_json},
        "annotations_plus_dumps_e2e_s": {"min": min(e2e_lists), "all": e2e_lists},
        "files_written": nfiles,
        "write_files_from_bytes_s": {"min": min(w_bytes), "all": w_bytes},
        "write_files_from_lists_s": {"min": min(w_lists), "all": w_lists},
        "files_byte_identical": files_identical,
        "hostpipe_frames_per_s": hostpipe_fps(vids, nv, T, dev, p, args.steps,
                                              (("without", False), ("annotations", True), ("json", "json"))),
        "sha256_json_bytes": sha_json, "sha256_dumps_of_annotations": sha_lists, "json_equals_dumps": identical,
    }
    assert identical and sha_json == sha_lists and files_identical, "json bytes differ from json.dumps of the lists"
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("card", "annotation_json_ms", "json_bytes_written", "annotation_json_e2e_s",
                                          "annotations_plus_dumps_e2e_s", "write_files_from_bytes_s",
                                          "write_files_from_lists_s", "hostpipe_frames_per_s", "sha256_json_bytes")},
                     default=str)[:3000])


if __name__ == "__main__":
    main()
