"""Drop-in for keymask_ident/annotations.py (stage E): single-video YTVIS json from the
`cluster_*/group_*/frame{f}_mask{m}.png` tree. The reference calls pycocotools per keymask
(mask_util.encode / area / toBbox, annotations.py:94-106); here all keymasks of a video are encoded
in one batch on the GPU (s2d_rle_encode: column-major run lengths, area, bounding box; s2d_rle_strings: the
base-48 string packing of maskApi.c rleToString). Batched callers that got their annotations from
s2d_b200.pipeline (stage E on the device) write the same json with write_video_annotations.
pycocotools is not installable in the build container, so parity at the RLE boundary is pinned by
the published algorithm and by decode round trips only (tests/test_dropin_gpu.py)."""
from __future__ import annotations

import ctypes as C
import json
import os
import re

import numpy as np
import torch
from PIL import Image

try:
    from . import _engine
except ImportError:
    import _engine


class coco_rle:
    """COCO compressed-RLE strings (maskApi.c rleToString / rleFrString) and the GPU batch encoder. to_string /
    from_string are the host helpers; encode_batch packs on the device (s2d_rle_strings), byte for byte the same."""

    @staticmethod
    def to_string(cnts):
        out = []
        for i, x in enumerate(cnts):
            x = int(x)
            if i > 2:
                x -= int(cnts[i - 2])
            more = True
            while more:
                c = x & 0x1F
                x >>= 5
                more = (x != -1) if (c & 0x10) else (x != 0)
                if more:
                    c |= 0x20
                out.append(chr(c + 48))
        return "".join(out)

    @staticmethod
    def from_string(s):
        cnts, p = [], 0
        while p < len(s):
            x, k, more = 0, 0, True
            while more:
                c = ord(s[p]) - 48
                x |= (c & 0x1F) << (5 * k)
                more = bool(c & 0x20)
                p += 1
                k += 1
                if not more and (c & 0x10):
                    x |= -1 << (5 * k)
            if len(cnts) > 2:
                x += cnts[-2]
            cnts.append(x)
        return cnts

    @staticmethod
    def encode_batch(masks):
        """masks [N,H,W] (bool / uint8, numpy or torch) -> list of (rle dict, area int, bbox [x,y,w,h] floats),
        what mask_util.encode / area / toBbox return per mask."""
        from s2d_b200 import _lib
        dev = _engine.device()
        m = torch.as_tensor(np.asarray(masks)) if not torch.is_tensor(masks) else masks
        m = (m != 0).to(dev, torch.uint8).contiguous()
        n, h, w = m.shape
        if n == 0:
            return []
        st = torch.cuda.current_stream(dev).cuda_stream
        max_runs = min(h * w + 1, 8 * w + 64)
        while True:
            need = C.c_int64()
            _lib.call("s2d_rle_work_ints", n, h, w, max_runs, C.byref(need))
            work = torch.empty(need.value, dtype=torch.int32, device=dev)
            counts = torch.empty((n, max_runs), dtype=torch.int32, device=dev)
            nruns = torch.empty(n, dtype=torch.int32, device=dev)
            area = torch.empty(n, dtype=torch.int32, device=dev)
            bbox = torch.empty((n, 4), dtype=torch.int32, device=dev)
            _lib.call("s2d_rle_encode", m.data_ptr(), n, h, w, max_runs, work.data_ptr(), counts.data_ptr(),
                      nruns.data_ptr(), area.data_ptr(), bbox.data_ptr(), st)
            nr = nruns.cpu().numpy()
            if int(nr.max()) <= max_runs:
                break
            max_runs = int(nr.max())                   # a mask with more runs than the first guess: once more
        # the masks' runs back to back, then the strings of all of them in one device pass
        flat = counts[torch.arange(max_runs, device=dev)[None, :] < nruns[:, None].to(torch.int64)].contiguous()
        offs = np.zeros(n + 1, np.int64)
        offs[1:] = np.cumsum(nr.astype(np.int64))
        strings = coco_rle.strings_device(flat, offs, dev)
        ar, bb = area.cpu().numpy(), bbox.cpu().numpy()
        out = []
        for i in range(n):
            rle = {"size": [int(h), int(w)], "counts": strings[i]}
            if ar[i] == 0:
                box = [0.0, 0.0, 0.0, 0.0]
            else:
                box = [float(bb[i, 0]), float(bb[i, 1]), float(bb[i, 2] - bb[i, 0] + 1), float(bb[i, 3] - bb[i, 1] + 1)]
            out.append((rle, int(ar[i]), box))
        return out


    @staticmethod
    def strings_device(counts, offsets, dev):
        """rleToString of N run-length lists on the device: counts (device int32, the lists back to back), offsets
        (host int64 [N + 1]) -> list of N strings."""
        from s2d_b200 import _lib
        n = len(offsets) - 1
        ncounts = int(offsets[-1])
        st = torch.cuda.current_stream(dev).cuda_stream
        d_off = torch.from_numpy(np.ascontiguousarray(offsets, np.int64)).to(dev)
        work = torch.empty(n, dtype=torch.int32, device=dev)
        soff = torch.empty(n + 1, dtype=torch.int64, device=dev)
        need = torch.zeros(1, dtype=torch.int64, device=dev)
        cap = 2 * ncounts + 16                      # most runs of a keymask take one or two characters
        while True:
            chars = torch.empty(cap, dtype=torch.uint8, device=dev)
            _lib.call("s2d_rle_strings", counts.data_ptr(), d_off.data_ptr(), n, ncounts, work.data_ptr(), cap,
                      chars.data_ptr(), soff.data_ptr(), need.data_ptr(), st)
            total = int(need.item())
            if total <= cap:
                break
            cap = total
        text = chars[:max(1, total)].cpu().numpy().tobytes()[:total].decode("ascii")
        so = soff.cpu().numpy()
        return [text[so[i]:so[i + 1]] for i in range(n)]


def rle_area_bbox_batch(rles):
    """[(area int, bbox [x, y, w, h] floats)] of COCO RLE dicts ({"size": [h, w], "counts": str | bytes | list})
    without decoding the masks: mask_util.area / toBbox for a whole list in one GPU launch (s2d_rle_area_bbox)."""
    from s2d_b200 import _lib
    if not rles:
        return []
    dev = _engine.device()
    lists = []
    for r in rles:
        c = r["counts"]
        if isinstance(c, bytes):
            c = c.decode("ascii")
        lists.append(coco_rle.from_string(c) if isinstance(c, str) else [int(x) for x in c])
    offs = np.zeros(len(lists) + 1, np.int64)
    offs[1:] = np.cumsum([len(x) for x in lists])
    flat = np.concatenate([np.asarray(x, np.int64) for x in lists] + [np.zeros(1, np.int64)]).astype(np.int32)
    counts = torch.from_numpy(flat).to(dev)
    offsets = torch.from_numpy(offs).to(dev)
    hs = torch.tensor([int(r["size"][0]) for r in rles], dtype=torch.int32, device=dev)
    area = torch.empty(len(rles), dtype=torch.int32, device=dev)
    bbox = torch.empty((len(rles), 4), dtype=torch.int32, device=dev)
    _lib.call("s2d_rle_area_bbox", counts.data_ptr(), offsets.data_ptr(), len(rles), hs.data_ptr(), area.data_ptr(),
              bbox.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
    a, b = area.cpu().numpy(), bbox.cpu().numpy()
    return [(int(a[i]), [float(v) for v in b[i]]) for i in range(len(rles))]


def _video_entry(video_path):
    """The `videos` entry the reference builds from the video's image folder (annotations.py:13-40), None without
    images."""
    video_name = os.path.basename(video_path)
    video_files = sorted(f for f in os.listdir(video_path) if f.endswith((".jpg", ".png", ".jpeg")))
    if not video_files:
        print(f"No image files found in {video_path}")
        return None
    with Image.open(os.path.join(video_path, video_files[0])) as img:
        width, height = img.size
    return {"license": 1, "coco_url": "", "height": height, "width": width, "length": len(video_files),
            "date_captured": "2019-04-11 00:55:41.903902",
            "file_names": [os.path.join(video_name, f) for f in video_files], "flickr_url": "", "id": 1}


_CATEGORIES = [{"supercategory": "object", "id": 1, "name": "fg"}]


def _dump_video_json(video, annotations, annotation_output_path, video_path):
    """`{videos, annotations, categories}` of one video to <annotation_output_path>/<video name>.json
    (annotations.py:131-140). `annotations` is the list, or its json text as bytes (Batch.annotation_json): then the
    other parts are json.dumps'ed around it, which gives the file json.dump writes for the list."""
    os.makedirs(annotation_output_path, exist_ok=True)
    path = os.path.join(annotation_output_path, f"{os.path.basename(video_path)}.json")
    if isinstance(annotations, (bytes, bytearray)):
        with open(path, "wb") as f:
            f.write(b'{"videos": ' + json.dumps([video]).encode() + b', "annotations": ' + bytes(annotations) +
                    b', "categories": ' + json.dumps(_CATEGORIES).encode() + b"}")
        return
    with open(path, "w") as f:
        json.dump({"videos": [video], "annotations": annotations, "categories": _CATEGORIES}, f)


def write_video_annotations(video_path, annotations, annotation_output_path):
    """The json write_annotation_for_video produces, for annotations computed elsewhere - the device stage E of the
    batched path (s2d_b200.pipeline: Batch.annotations, discover_keymasks(..., annotations=True)). `annotations` may
    also be the json text of the list as bytes (Batch.annotation_json, discover_keymasks(..., annotations="json")):
    the file is the same. Nothing is written for a video without annotations (None: the reference writes no json for
    a failed video) or without images."""
    if annotations is None:
        return
    video = _video_entry(video_path)
    if video is not None:
        _dump_video_json(video, annotations, annotation_output_path, video_path)


def write_annotation_for_video(video_path, cluster_masks_path, annotation_output_path, visibility_data):
    """Same contract as the reference (annotations.py:8-140)."""
    video = _video_entry(video_path)
    if video is None:
        return
    height, width = video["height"], video["width"]
    cluster_dirs = sorted(d for d in os.listdir(cluster_masks_path)
                          if os.path.isdir(os.path.join(cluster_masks_path, d)) and d.startswith("cluster_")
                          and any(f.endswith(".png") for f in os.listdir(os.path.join(cluster_masks_path, d))))
    with open(os.path.join(cluster_masks_path, "video_one2x_data.json")) as f:
        one2x_data = json.load(f)
    annotations, ann_id, n = [], 1, video["length"]
    pending = []
    for cname in cluster_dirs:
        cdir = os.path.join(cluster_masks_path, cname)
        groups = sorted(d for d in os.listdir(cdir) if os.path.isdir(os.path.join(cdir, d)) and d.startswith("group_"))
        try:
            cid = int(cname.replace("cluster_", ""))
            ranges = next((c for c in visibility_data["clusters"] if c["cluster_id"] == cid), None)["ranges"]
        except KeyError:
            ranges = [(-1, -1)]
        if cname not in one2x_data:
            print(f"Could not find one2x data for {cname}.")
            continue
        for gname in groups:
            gdir = os.path.join(cdir, gname)
            segs, boxes, areas = [None] * n, [None] * n, [None] * n
            for mf in (f for f in os.listdir(gdir) if f.endswith(".png")):
                m = re.search(r"frame(\d+)", mf)
                if not m or int(m.group(1)) >= n:
                    continue
                binary = np.array(Image.open(os.path.join(gdir, mf)).convert("L")) > 0
                pending.append((segs, areas, boxes, int(m.group(1)), binary))     # encoded in one GPU batch below
            annotations.append({"video_id": 1, "iscrowd": 0, "height": height, "width": width, "length": n,
                                "segmentations": segs, "bboxes": boxes, "areas": areas, "category_id": 1,
                                "id": ann_id, "one2x": round(float(one2x_data[cname][gname]["avg_one2x"]), 2),
                                "visibility_ranges": ranges})
            ann_id += 1
    # later files of a group overwrite earlier ones on the same frame, like the reference's loop
    by_shape = {}
    for item in pending:
        by_shape.setdefault(item[4].shape, []).append(item)
    for items in by_shape.values():
        enc = coco_rle.encode_batch(np.stack([it[4] for it in items]))
        for (segs, areas, boxes, fidx, _), (rle, area, box) in zip(items, enc):
            segs[fidx], areas[fidx], boxes[fidx] = rle, area, box
    _dump_video_json(video, annotations, annotation_output_path, video_path)
