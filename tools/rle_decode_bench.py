"""COCO RLE decode on the device (s2d_rle_from_strings, s2d_rle_decode) at C2 scale: bench.py's C2 batch (64 videos x 36
frames 720p, 20 masks/frame, 4096 tracks, same generator and seed) run with stages "LVBDE", its annotation json decoded.

- parse: every segmentation string of the 64 videos' json in one s2d_rle_from_strings call, CUDA events, median after
  warm-up, against the host parser coco_rle.from_string over the same strings (one pass, host clock);
- decode: the members of the first video with annotations (every non-null segmentation) in one s2d_rle_decode call, CUDA events, median after
  warm-up; bytes written (H * W per mask; the output is larger than the 126 MB L2) over time, and its fraction of the
  6548.2 GB/s copy peak DESIGN.md uses;
- decode_video_annotations(json bytes) of that video end to end (json.loads, uploads, parse, decode; host clock around a
  device synchronise), and a check that the decoded masks' areas equal the json's.

    python tools/rle_decode_bench.py --out profiles/r06_rle_decode_c2.json
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

COPY_PEAK_GBS = 6548.2


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_rle_decode_c2.json"))
    args = ap.parse_args()

    import numpy as np
    import torch

    import bench
    from s2d_b200 import _lib
    from s2d_b200.keymask_ident.annotations import coco_rle, decode_video_annotations
    from s2d_b200.pipeline import Batch, Params
    from stage_e_bench import card

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    info = card()
    vids = bench.build_videos("c2", dev, 2024)
    b = Batch(vids, stages="LVBDE")
    b.run(Params())
    texts = b.annotation_json()
    anns = [json.loads(t) if t is not None else [] for t in texts]
    strings = [s["counts"] for a in anns for ann in a for s in ann["segmentations"] if s is not None]
    blobs = [s.encode("ascii") for s in strings]
    nstr, nchars = len(blobs), sum(len(x) for x in blobs)

    ev = lambda: torch.cuda.Event(enable_timing=True)
    med = lambda x: float(np.median(x))
    st = torch.cuda.current_stream(dev).cuda_stream

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        pairs = []
        for _ in range(args.steps):
            e0, e1 = ev(), ev()
            e0.record()
            fn()
            e1.record()
            pairs.append((e0, e1))
        torch.cuda.synchronize()
        return [a.elapsed_time(c) for a, c in pairs]

    # parse: all strings of the batch
    offs = np.zeros(nstr + 1, np.int64)
    offs[1:] = np.cumsum([len(x) for x in blobs])
    chars = torch.frombuffer(bytearray(b"".join(blobs)), dtype=torch.uint8).to(dev)
    d_off = torch.from_numpy(offs).to(dev)
    n = C.c_int64()
    _lib.call("s2d_rle_from_strings_work_ints", nstr, nchars, C.byref(n))
    pwork = torch.empty(n.value, dtype=torch.int32, device=dev)
    counts = torch.empty(nchars, dtype=torch.int32, device=dev)
    coff = torch.empty(nstr + 1, dtype=torch.int64, device=dev)
    status = torch.empty(nstr, dtype=torch.int32, device=dev)
    need = torch.empty(1, dtype=torch.int64, device=dev)
    parse = lambda: _lib.call("s2d_rle_from_strings", chars.data_ptr(), d_off.data_ptr(), nstr, pwork.data_ptr(), nchars,
                              counts.data_ptr(), coff.data_ptr(), status.data_ptr(), need.data_ptr(), st)
    t_parse = timed(parse)
    ncounts = int(need.item())
    assert not status.any()
    h0 = time.perf_counter()
    host = [coco_rle.from_string(s) for s in strings]
    t_host = time.perf_counter() - h0
    co = coff.cpu().numpy()
    parse_equal = bool(np.array_equal(counts[:ncounts].cpu().numpy(), np.concatenate([np.asarray(x, np.int64) for x in host])) and
                       np.array_equal(np.diff(co), [len(x) for x in host]))

    # decode: the members of video v0, the first with annotations (status 1)
    v0 = next(v for v, t in enumerate(texts) if t is not None and anns[v])
    _, _, H, W, _, _, _ = bench.WORKLOADS["c2"]
    segs = [s for ann in anns[v0] for s in ann["segmentations"] if s is not None]
    m = len(segs)
    vb = [s["counts"].encode("ascii") for s in segs]
    vcounts, vcoff, vstatus = coco_rle.counts_from_strings_device(vb)
    vn = int(vcoff[-1].item())
    _lib.call("s2d_rle_decode_work_ints", m, vn, C.byref(n))
    dwork = torch.empty(n.value, dtype=torch.int32, device=dev)
    hs = torch.full((m,), H, dtype=torch.int32, device=dev)
    ws = torch.full((m,), W, dtype=torch.int32, device=dev)
    oo = torch.arange(m, dtype=torch.int64, device=dev) * H * W
    out = torch.empty((m, H, W), dtype=torch.uint8, device=dev)
    decode = lambda: _lib.call("s2d_rle_decode", vcounts.data_ptr(), vcoff.data_ptr(), m, hs.data_ptr(), ws.data_ptr(),
                               oo.data_ptr(), dwork.data_ptr(), out.data_ptr(), vstatus.data_ptr(), st)
    t_dec = timed(decode)
    assert not vstatus.any()
    areas = [a for ann in anns[v0] for a, s in zip(ann["areas"], ann["segmentations"]) if s is not None]
    areas_equal = out.reshape(m, -1).sum(1, dtype=torch.int64).cpu().tolist() == areas
    written = m * H * W
    gbs = written / (med(t_dec) * 1e-3) / 1e9

    # decode_video_annotations of that video from its json bytes
    for _ in range(args.warmup):
        decode_video_annotations(texts[v0])
    torch.cuda.synchronize()
    e2e = []
    for _ in range(max(5, args.steps // 2)):
        h0 = time.perf_counter()
        vm = decode_video_annotations(texts[v0])
        torch.cuda.synchronize()
        e2e.append(time.perf_counter() - h0)
    slots = [a * vm.shape[1] + t for a, ann in enumerate(anns[v0]) for t, s in enumerate(ann["segmentations"])
             if s is not None]
    video_equal = bool(torch.equal(vm.reshape(-1, H, W)[slots], out))

    res = {
        "tool": "tools/rle_decode_bench.py", "card": info, "version": _lib.load().s2d_version(),
        "workload": "c2: 64 videos x 36 frames 720x1280, 20 masks/frame, 4096 tracks, seed 2024 (bench.py generator), "
                    "stages LVBDE, Batch.annotation_json()",
        "steps": args.steps, "warmup": args.warmup,
        "parse": {"strings": nstr, "chars": nchars, "counts": ncounts, "device_ms": {"median": med(t_parse), "all": t_parse},
                  "host_from_string_s": t_host, "equal_to_from_string": parse_equal,
                  "note": "CUDA events around s2d_rle_from_strings (rp_count_kernel, offsets_kernel, rp_write_kernel); "
                          "host: coco_rle.from_string over the same strings, one pass"},
        "decode_one_video": {"video": v0, "masks": m, "H": H, "W": W, "counts": vn, "ms": {"median": med(t_dec), "all": t_dec},
                          "bytes_written": written, "write_gbs": gbs, "copy_peak_gbs": COPY_PEAK_GBS,
                          "fraction_of_copy_peak": gbs / COPY_PEAK_GBS, "areas_equal_json": areas_equal,
                          "note": "CUDA events around s2d_rle_decode (rd_scan_kernel, rd_tile_kernel); output "
                                  f"{written / 1e6:.0f} MB, larger than L2"},
        "decode_video_annotations_s": {"median": med(e2e), "min": min(e2e), "all": e2e,
                                       "equals_direct_decode": video_equal},
    }
    assert parse_equal and areas_equal and video_equal, "device decode differs from the host parser or the json"
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("card", "parse", "decode_one_video", "decode_video_annotations_s")}, default=str)[:3000])


if __name__ == "__main__":
    main()
