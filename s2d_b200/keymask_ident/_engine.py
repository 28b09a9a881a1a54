"""Glue shared by the drop-in modules: device selection, per-process caches, tracker access,
dataset/split naming, and the stage-wise GPU calls (through s2d_b200.pipeline / the C ABI)."""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

_ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if _ROOT not in sys.path:
    sys.path.insert(0, _ROOT)

from s2d_b200.pipeline import Batch, Params, VideoInput  # noqa: E402

# substrings looked for in the video path, in the reference's order
# (cotracker_occlusions.py:265-293, cotracker_matching.py:943-971)
_DATASETS = [("DAVIS", "DAVIS"), ("ytvis2021", "ytvis2021"), ("ytvis2019", "ytvis2019"), ("ovis", "ovis"),
             ("VIPSeg", "VIPSeg"), ("MOSE", "MOSE"), ("sa-v", "SA-V")]
_SPLITS = ["train", "valid", "test", "val", "imgs"]


def dataset_and_split(video_path: str):
    for needle, name in _DATASETS:
        if needle in video_path:
            break
    else:
        raise ValueError("Unknown dataset")
    for sp in _SPLITS:
        if sp in video_path:
            return name, sp
    return name, "all"


def device():
    if not torch.cuda.is_available():
        raise RuntimeError("s2d_b200 needs a CUDA device: the keymask kernels have no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def checkpoint_dir():
    """same lookup as the reference (cotracker_occlusions.py:309-315)"""
    for p in ("/mnt/data/checkpoints", "/mnt/hdd/leon/checkpoints/"):
        if os.path.exists(p):
            return p
    raise FileNotFoundError("Checkpoint directory not found. Please ensure the path is correct. Add it for the new cluster")


_tracker_factory = None


def set_tracker_factory(factory):
    """Install a callable `factory(checkpoint=...) -> model` used instead of
    cotracker.predictor.CoTrackerPredictor (precomputed tracks, tests)."""
    global _tracker_factory
    _tracker_factory = factory


def make_tracker():
    """CoTracker is an upstream producer of this path (BASELINE.json north_star): use the real
    predictor when the `cotracker` package is importable, else an installed factory."""
    if _tracker_factory is not None:
        return _tracker_factory(checkpoint=None)
    from cotracker.predictor import CoTrackerPredictor   # third-party, as in the reference
    model = CoTrackerPredictor(checkpoint=os.path.join(checkpoint_dir(), "scaled_offline.pth"))
    if torch.cuda.is_available():
        model = model.cuda()
    return model


# ---- label maps: loaded once per mask folder (the reference re-reads them three times) -------
_label_cache = {}


def cached_labels(mask_folder, loader):
    key = os.path.abspath(mask_folder)
    ent = _label_cache.get(key)
    if ent is None:
        masks = loader(mask_folder)
        if masks is None:
            return None
        ent = masks
        _label_cache.clear()          # one video at a time, like the driver
        _label_cache[key] = ent
    return ent


def labels_u8_device(masks_thw1: torch.Tensor):
    lab = masks_thw1[..., 0]
    if int(lab.max()) > 255:
        raise ValueError("s2d_b200 supports at most 255 masks per frame")
    return lab.to(torch.uint8).contiguous().to(device())


def enumerate_objects(labels_dev: torch.Tensor):
    """K0 on the GPU: (qframe, qlabel, area[T,256]) of sort(unique(label[t]))[1:] per frame."""
    T, H, W = labels_dev.shape
    # Nm is not known yet: an upper bound of 255 objects per frame sizes the row arrays
    b = Batch([VideoInput(labels=labels_dev, dims={"Nm": 255 * T, "P": 2})], stages="L")
    b.run()
    torch.cuda.synchronize(b.device)
    nm = int(b.vidinfo[5].item())
    return (b.qframe[:nm].cpu().numpy().astype(np.int64), b.qlabel[:nm].cpu().numpy().astype(np.int64),
            b.area.cpu().numpy().reshape(T, 256))


def visibility_mean(vis_rows, T: int):
    """K3a on the GPU. vis_rows: list of [T,P_q] bool arrays/tensors (ragged P)."""
    nm = len(vis_rows)
    pmax = max(int(v.shape[1]) for v in vis_rows)
    pmax += pmax % 2
    dev = device()
    vis = torch.zeros((nm, T, pmax), dtype=torch.uint8, device=dev)
    npts = torch.empty(nm, dtype=torch.int32)
    for q, v in enumerate(vis_rows):
        v = torch.as_tensor(v)
        vis[q, :, : v.shape[1]] = v.to(dev).to(torch.uint8)
        npts[q] = v.shape[1]
    b = Batch([VideoInput(vis=vis, npts=npts.to(dev))], stages="V")
    b.run()
    torch.cuda.synchronize(dev)
    return b.V.cpu().numpy().reshape(nm, T)


def visibility_windows(V: np.ndarray, qframe, qlabel, visibility_threshold: float):
    """K3b/c on the GPU: returns the `clusters` list of the stage-B json."""
    nm, T = V.shape
    b = Batch([VideoInput(dims={"Nm": nm, "T": T, "P": 2})], device=device(), stages="B")
    b.upload_visibility(V, np.asarray(qframe))
    b.qlabel[:nm] = torch.from_numpy(np.asarray(qlabel, np.int32)).to(b.device)
    b.run(Params(visibility_threshold=visibility_threshold))
    torch.cuda.synchronize(b.device)
    return b.decode(want_comps=False, check_rows=False)[0]["clusters"]


def color_frames_to_labels(rgb_frames: np.ndarray):
    """f1 on the GPU: [F,H,W,3] uint8 RGB frames (numpy, or a tensor already on the device) -> ([F,H,W] uint8 label
    ids on the device, colours per frame). Same ids as crw_utils.rgb_to_label_ids (rank of the RGB tuple among the
    non-black colours)."""
    import ctypes as C
    from s2d_b200 import _lib
    F, H, W, _ = rgb_frames.shape
    if torch.is_tensor(rgb_frames):
        rgb = rgb_frames.contiguous()
        dev = rgb.device
    else:
        dev = device()
        rgb = torch.from_numpy(np.ascontiguousarray(rgb_frames)).to(dev)
    n = C.c_int64()
    _lib.call("s2d_color_to_labels_work_ints", F, C.byref(n))
    work = torch.empty(n.value, dtype=torch.int32, device=dev)
    labels = torch.empty((F, H, W), dtype=torch.uint8, device=dev)
    ncol = torch.empty(F, dtype=torch.int32, device=dev)
    _lib.call("s2d_color_to_labels", rgb.data_ptr(), F, H * W, work.data_ptr(), labels.data_ptr(), ncol.data_ptr(),
              torch.cuda.current_stream(dev).cuda_stream)
    ncol_h = ncol.cpu().numpy()
    if int(ncol_h.max()) > 255:
        raise ValueError("s2d_b200 supports at most 255 masks per frame")
    return labels, ncol_h


def appearance_events(vis: torch.Tensor, smoothing_window: int = 1, thresh: float = 0.95, min_run_length: int = 4):
    """K3d through the C ABI: {row: list(zip(starts, ends))} exactly as the reference builds it."""
    from s2d_b200 import _lib
    dev = device()
    v = vis.to(dev, torch.float32).contiguous()
    n, T = v.shape
    p1, p2 = (int(smoothing_window) - 1) // 2, (int(min_run_length) - 1) // 2
    if p1 >= T or p2 >= T or p2 >= T + 2 * p2 - int(min_run_length) + 1:
        raise RuntimeError("Padding size should be less than the corresponding input dimension")   # what torch raises
    cap = T // 2 + 2                                # a row cannot hold more transitions of one kind
    ns = torch.empty(n, dtype=torch.int32, device=dev)
    ne = torch.empty(n, dtype=torch.int32, device=dev)
    st = torch.empty((n, cap), dtype=torch.int32, device=dev)
    en = torch.empty((n, cap), dtype=torch.int32, device=dev)
    _lib.call("s2d_appearance_events", v.data_ptr(), n, T, int(smoothing_window), float(np.float32(thresh)),
              int(min_run_length), cap, ns.data_ptr(), ne.data_ptr(), st.data_ptr(), en.data_ptr(), None,
              torch.cuda.current_stream(dev).cuda_stream)
    ns, ne, st, en = ns.cpu().numpy(), ne.cpu().numpy(), st.cpu().numpy(), en.cpu().numpy()
    return {i: list(zip(st[i, :ns[i]].tolist(), en[i, :ne[i]].tolist())) for i in range(n)}


def boolean_visibility(vis: torch.Tensor, threshold: float = 0.3) -> torch.Tensor:
    from s2d_b200 import _lib
    dev = device()
    v = vis.to(dev, torch.float32).contiguous()
    out = torch.empty(v.shape, dtype=torch.uint8, device=dev)
    if v.numel():
        _lib.call("s2d_boolean_visibility", v.data_ptr(), v.numel(), float(np.float32(threshold)), out.data_ptr(),
                  torch.cuda.current_stream(dev).cuda_stream)
    return out.to(torch.bool).to(vis.device)
