"""PNG label-map decode of the C2 batch on the device (s2d_png_decode, then s2d_color_to_labels) against cv2.imdecode on
every host core. Inputs: the 64 x 36 = 2304 720p label maps of bench.py's C2 batch (make_scene_device, seed 2024 + video)
encoded two ways: (a) RGB PNGs written by cv2 with its default settings, (b) PIL palette PNGs (DAVIS / YTVIS style).
Device times are CUDA events, median of --reps launches after a warm-up; the working set (6.4 GB of scanlines and as
much RGB for (a)) is far larger than L2.

    python tools/png_decode_bench.py --out profiles/r08_png_decode_c2.json
"""
import argparse
import ctypes as C
import io
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import cv2
import numpy as np
import torch
from PIL import Image

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from s2d_b200 import _lib, png  # noqa: E402
from s2d_b200.keymask_ident import _engine  # noqa: E402
from s2d_b200.synth import make_scene_device  # noqa: E402


def _palette():
    pal = np.random.default_rng(1).choice(1 << 24, 255, replace=False)
    rgb = np.stack([(pal >> 16) & 255, (pal >> 8) & 255, pal & 255], axis=1).astype(np.uint8)
    return np.concatenate([np.zeros((1, 3), np.uint8), rgb])


def _enc_rgb(args):
    lab, pal = args
    return cv2.imencode(".png", pal[lab][..., ::-1])[1].tobytes()


def _enc_pal(args):
    lab, pal = args
    im = Image.fromarray(lab, "P")
    im.putpalette(pal.tobytes())
    b = io.BytesIO()
    im.save(b, "PNG")
    return b.getvalue()


def _events(fn, reps):
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), float(np.min(ts))


def measure(blobs, labels_want, dev, reps, pool):
    r = {"files": len(blobs), "png_bytes": int(sum(map(len, blobs)))}
    t = time.perf_counter()
    parsed = [png.parse_png(b) for b in blobs]
    r["host_parse_ms"] = (time.perf_counter() - t) * 1e3
    assert all(p is not None for p in parsed)
    r["raw_bytes"] = int(sum(p.raw_bytes for p in parsed))
    torch.cuda.synchronize()
    t = time.perf_counter()
    sp = png.stage_pngs(parsed, dev)
    torch.cuda.synchronize()
    r["stage_upload_ms"] = (time.perf_counter() - t) * 1e3
    rgb, st = png.launch_decode(sp)
    nw = C.c_int64()
    _lib.call("s2d_png_decode_work_ints", len(parsed), int(sp.raw_off[-1]), C.byref(nw))
    work = torch.empty(nw.value, dtype=torch.int32, device=dev)
    assert (st.cpu().numpy() == 0).all()
    H, W = parsed[0].height, parsed[0].width
    frames = rgb.view(len(parsed), H, W, 3)
    labels, _ = _engine.color_frames_to_labels(frames)
    assert torch.equal(labels, labels_want), "device labels differ from the scene's"
    r["decode_ms_median"], r["decode_ms_min"] = _events(lambda: png.launch_decode(sp, work, rgb, st), reps)
    r["decode_colour_to_ids_ms_median"], r["decode_colour_to_ids_ms_min"] = _events(
        lambda: (png.launch_decode(sp, work, rgb, st), _engine.color_frames_to_labels(frames)), reps)
    r["rgb_bytes"] = int(rgb.numel())
    # load_label_maps' device path end to end from bytes in host memory: parse, stage + upload, decode, colour -> ids
    ts = []
    for _ in range(3):
        torch.cuda.synchronize()
        t = time.perf_counter()
        dec = png.decode_pngs(blobs, dev)
        lab = png.rgb_frames_to_labels(dec.frames)
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t) * 1e3)
    assert torch.equal(lab, labels_want)
    r["end_to_end_from_bytes_ms_median"] = float(np.median(ts))
    # cv2.imdecode of the same bytes on every host core
    dec1 = lambda b: cv2.imdecode(np.frombuffer(b, np.uint8), cv2.IMREAD_COLOR)   # noqa: E731
    list(pool.map(dec1, blobs[:64]))
    t = time.perf_counter()
    list(pool.map(dec1, blobs))
    r["cv2_imdecode_all_cores_ms"] = (time.perf_counter() - t) * 1e3
    t = time.perf_counter()
    for b in blobs[:64]:
        dec1(b)
    r["cv2_imdecode_one_core_ms_per_file"] = (time.perf_counter() - t) * 1e3 / 64
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--videos", type=int, default=64)
    ap.add_argument("--frames", type=int, default=36)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    pal = _palette()
    labs = []
    for i in range(args.videos):
        sc = make_scene_device(2024 + i, args.frames, 720, 1280, 20, 4096, dev)
        labs.append(sc["labels"].cpu().numpy())
        del sc
    labs = np.concatenate(labs)
    ncpu = os.cpu_count()
    res = {"workload": f"c2: {args.videos} videos x {args.frames} frames 720x1280 label maps, seed 2024 (bench.py generator)",
           "gpu": torch.cuda.get_device_name(dev), "nvidia_smi": smi[0] if smi else "", "host_cpus": ncpu, "reps": args.reps}
    with ThreadPoolExecutor(ncpu) as pool:
        labels_want = torch.cat([_engine.color_frames_to_labels(torch.from_numpy(pal[labs[i:i + args.frames]]).to(dev))[0]
                                 for i in range(0, len(labs), args.frames)])
        for kind, enc in (("cv2_rgb", _enc_rgb), ("pil_palette", _enc_pal)):
            blobs = list(pool.map(enc, [(l, pal) for l in labs]))
            res[kind] = measure(blobs, labels_want, dev, args.reps, pool)
            print(kind, json.dumps(res[kind]), flush=True)
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
