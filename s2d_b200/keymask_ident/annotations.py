"""Drop-in for keymask_ident/annotations.py (stage E): single-video YTVIS json from the
`cluster_*/group_*/frame{f}_mask{m}.png` tree. The reference calls pycocotools per keymask
(mask_util.encode / area / toBbox, annotations.py:94-106); here all keymasks of a video are encoded
in one batch on the GPU (s2d_rle_encode: column-major run lengths, area, bounding box; s2d_rle_strings: the
base-48 string packing of maskApi.c rleToString). Batched callers that got their annotations from
s2d_b200.pipeline (stage E on the device) write the same json with write_video_annotations.
coco_rle.decode_batch and decode_video_annotations turn the strings back into masks on the device (mask_util.decode:
s2d_rle_from_strings, s2d_rle_decode).
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

    @staticmethod
    def counts_from_strings_device(strings):
        """rleFrString of N strings (str or bytes, ASCII) on the device, in one launch sequence (s2d_rle_from_strings) ->
        (counts int32, offsets int64 [N + 1], status int32 [N]), device tensors: list n is counts[offsets[n]:offsets[n +
        1]], status[n] = 1 marks a malformed string (its last character continues, or a count falls outside [0, 2^31)).
        No host synchronisation."""
        dev = _engine.device()
        blobs = [s.encode("ascii") if isinstance(s, str) else bytes(s) for s in strings]
        counts = torch.empty(max(1, sum(len(b) for b in blobs)), dtype=torch.int32, device=dev)
        status = torch.empty(len(blobs), dtype=torch.int32, device=dev)
        if not blobs:
            return counts[:0], torch.zeros(1, dtype=torch.int64, device=dev), status
        return counts, coco_rle._parse_device(blobs, dev, counts, status), status

    @staticmethod
    def _parse_device(blobs, dev, counts, status):
        """s2d_rle_from_strings of the byte strings `blobs` into counts (capacity: one count per character at most, so
        it is never short) and status [len(blobs)]; returns the device offsets [len(blobs) + 1]."""
        from s2d_b200 import _lib
        n = len(blobs)
        offs = np.zeros(n + 1, np.int64)
        offs[1:] = np.cumsum([len(b) for b in blobs])
        nchars = int(offs[-1])
        assert counts.numel() >= nchars and status.numel() >= n
        chars = torch.frombuffer(bytearray(b"".join(blobs) or b"\0"), dtype=torch.uint8).to(dev)
        d_off = torch.from_numpy(offs).to(dev)
        need = C.c_int64()
        _lib.call("s2d_rle_from_strings_work_ints", n, nchars, C.byref(need))
        work = torch.empty(need.value, dtype=torch.int32, device=dev)
        count_off = torch.empty(n + 1, dtype=torch.int64, device=dev)
        needed = torch.empty(1, dtype=torch.int64, device=dev)
        _lib.call("s2d_rle_from_strings", chars.data_ptr(), d_off.data_ptr(), n, work.data_ptr(), counts.numel(),
                  counts.data_ptr(), count_off.data_ptr(), status.data_ptr(), needed.data_ptr(),
                  torch.cuda.current_stream(dev).cuda_stream)
        return count_off

    @staticmethod
    def _decode_into(rles, out, out_offsets):
        """rleDecode of the RLE dicts `rles` into the uint8 device buffer `out`, mask i at byte out_offsets[i] (host
        int64): one parse launch sequence for all compressed strings, one decode launch sequence for all masks. Returns
        the device status int32 [len(rles)] (1: malformed string, 2: runs do not sum to H * W). Uncompressed counts
        (lists) and non-ASCII strings (host from_string) are range-checked here and uploaded as they are."""
        from s2d_b200 import _lib
        dev = out.device
        n = len(rles)
        blobs, s_idx, lists, l_idx = [], [], [], []
        for i, r in enumerate(rles):
            c = r["counts"]
            if isinstance(c, str):
                try:
                    c = c.encode("ascii")
                except UnicodeEncodeError:
                    try:
                        c = coco_rle.from_string(c)
                    except IndexError:
                        raise ValueError(f"segmentation {i}: malformed RLE string") from None
            if isinstance(c, (bytes, bytearray)):
                blobs.append(c)
                s_idx.append(i)
                continue
            c = np.asarray(c, dtype=np.int64).reshape(-1)
            if c.size and (c.min() < 0 or c.max() >= 2 ** 31):
                raise ValueError(f"segmentation {i}: RLE counts outside [0, 2^31)")
            lists.append(c.astype(np.int32))
            l_idx.append(i)
        # lists first, then the parsed strings: one contiguous counts buffer and one offsets array for the decode
        l_off = np.zeros(len(lists) + 1, np.int64)
        l_off[1:] = np.cumsum([len(x) for x in lists])
        nl = int(l_off[-1])
        nchars = sum(len(b) for b in blobs)
        counts = torch.empty(nl + max(1, nchars), dtype=torch.int32, device=dev)
        if nl:
            counts[:nl] = torch.from_numpy(np.concatenate(lists)).to(dev)
        status = torch.zeros(n, dtype=torch.int32, device=dev)
        count_off = torch.from_numpy(l_off).to(dev)
        if blobs:
            s_off = coco_rle._parse_device(blobs, dev, counts[nl:], status[len(lists):])
            count_off = torch.cat([count_off[:-1], s_off + nl])
        order = l_idx + s_idx
        size = np.asarray([[int(rles[i]["size"][0]), int(rles[i]["size"][1])] for i in order], np.int32).reshape(-1, 2)
        hs = torch.from_numpy(np.ascontiguousarray(size[:, 0])).to(dev)
        ws = torch.from_numpy(np.ascontiguousarray(size[:, 1])).to(dev)
        oo = torch.from_numpy(np.asarray(out_offsets, np.int64)[order]).to(dev)
        need = C.c_int64()
        _lib.call("s2d_rle_decode_work_ints", n, nl + nchars, C.byref(need))
        work = torch.empty(need.value, dtype=torch.int32, device=dev)
        _lib.call("s2d_rle_decode", counts.data_ptr(), count_off.data_ptr(), n, hs.data_ptr(), ws.data_ptr(), oo.data_ptr(),
                  work.data_ptr(), out.data_ptr(), status.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
        back = torch.empty_like(status)
        back[torch.tensor(order, dtype=torch.int64, device=dev)] = status
        return back

    @staticmethod
    def decode_batch(rles, check=True):
        """mask_util.decode on the device: one RLE dict ({"size": [h, w], "counts": str | bytes | list}) -> uint8 [H, W];
        a list of them, all of one size (ValueError otherwise) -> uint8 [N, H, W]. Unlike pycocotools, which returns
        [H, W, N], the mask index comes first. Values are 0 / 1. With check=True a malformed string or runs that do not
        sum to H * W raise ValueError naming the first such index; with check=False the call returns (masks, status) -
        status int32 ([N] or a scalar; 1: malformed string, 2: wrong sum) - without synchronising the host."""
        single = isinstance(rles, dict)
        lst = [rles] if single else list(rles)
        sizes = {(int(r["size"][0]), int(r["size"][1])) for r in lst}
        if len(sizes) > 1:
            raise ValueError(f"decode_batch: masks of different sizes {sorted(sizes)} in one call")
        h, w = sizes.pop() if sizes else (0, 0)
        dev = _engine.device()
        buf = torch.empty(max(1, len(lst) * h * w), dtype=torch.uint8, device=dev)
        out = buf[:len(lst) * h * w].view(len(lst), h, w)
        status = (coco_rle._decode_into(lst, buf, np.arange(len(lst), dtype=np.int64) * h * w) if lst
                  else torch.zeros(0, dtype=torch.int32, device=dev))
        if single:
            out, status = out[0], status[0]
        if not check:
            return out, status
        _raise_on_status(status.reshape(-1), "segmentation")
        return out


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


def _raise_on_status(status, what):
    bad = torch.nonzero(status).reshape(-1).cpu()
    if bad.numel():
        i = int(bad[0])
        s = int(status[i])
        why = "malformed RLE string" if s & 1 else "runs do not sum to H * W"
        raise ValueError(f"{what} {i}: {why} (status {s}; {bad.numel()} bad in all)")


def decode_video_annotations(annotations, check=True):
    """The masks of one video's YTVIS `annotations` - the list Batch.annotations() returns, its json text as bytes
    (Batch.annotation_json()) or the "annotations" of a loaded file - as uint8 [A, T, H, W] on the device: annotation a,
    frame t is mask_util.decode of segmentations[t], zero where the segmentation is null. All segmentations go through
    one parse and one decode launch sequence. check=True raises ValueError on a malformed segmentation (named by
    annotation and frame); check=False returns (masks, status int32 [A, T]) without synchronising the host."""
    if isinstance(annotations, (bytes, bytearray, str)):
        annotations = json.loads(annotations)
    dev = _engine.device()
    A = len(annotations)
    T = len(annotations[0]["segmentations"]) if A else 0
    rles, slots, hw = [], [], set()
    for a, ann in enumerate(annotations):
        segs = ann["segmentations"]
        if len(segs) != T:
            raise ValueError(f"annotation {a}: {len(segs)} frames, annotation 0 has {T}")
        for t, s in enumerate(segs):
            if s is not None:
                rles.append(s)
                slots.append(a * T + t)
                hw.add((int(s["size"][0]), int(s["size"][1])))
    if len(hw) > 1:
        raise ValueError(f"decode_video_annotations: segmentations of different sizes {sorted(hw)}")
    H, W = hw.pop() if hw else ((int(annotations[0]["height"]), int(annotations[0]["width"])) if A else (0, 0))
    buf = torch.zeros(max(1, A * T * H * W), dtype=torch.uint8, device=dev)
    out = buf[:A * T * H * W].view(A, T, H, W)
    status = torch.zeros(A * T, dtype=torch.int32, device=dev)
    if rles:
        status[torch.tensor(slots, dtype=torch.int64, device=dev)] = coco_rle._decode_into(
            rles, buf, np.asarray(slots, np.int64) * H * W)
    status = status.view(A, T)
    if not check:
        return out, status
    bad = torch.nonzero(status).cpu()
    if bad.shape[0]:
        a, t = (int(x) for x in bad[0])
        s = int(status[a, t])
        why = "malformed RLE string" if s & 1 else "runs do not sum to H * W"
        raise ValueError(f"annotation {a} frame {t}: {why} (status {s}; {bad.shape[0]} bad in all)")
    return out


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
