"""Drop-in for keymask_ident/crw_utils.py: CLI flags, robust image loading, colour-PNG -> label
ids, frame/mask loading. Host-side I/O only (SURVEY.md section 8 rows a1, a9); the dead dataset
classes of the CRW code base are not part of the keymask path and are not reproduced."""
from __future__ import annotations

import argparse
import glob
import os
import random
import time
import warnings
from pathlib import Path

import cv2
import numpy as np
import torch
import torch.nn.functional as F
from PIL import Image


def keymask_args():
    """Same flags and defaults as the reference (crw_utils.py:28-82)."""
    ap = argparse.ArgumentParser(description="Keymask Identification")
    ap.add_argument("--workers", default=4, type=int, metavar="N")
    ap.add_argument("--manualSeed", type=int, default=777)
    ap.add_argument("--gpu-id", default="0", type=str)
    ap.add_argument("--batchSize", default=1, type=int)
    ap.add_argument("--video-base-path", default="/mnt/data/datasets/DAVIS/JPEGImages/480p", type=str)
    ap.add_argument("--mask-base-path", default="/mnt/data/outputs/DAVIS/cuts3d/pseudo_annotations", type=str)
    ap.add_argument("--save-path", default="/mnt/data/outputs/cotracker/segmentation_masks/DAVIS/all/", type=str)
    ap.add_argument("--video-output-dir", default="/mnt/data/outputs/cotracker/videos", type=str)
    ap.add_argument("--visibility-maps-output-base", default="/mnt/data/outputs/cotracker/visibility_maps", type=str)
    ap.add_argument("--visibility-clusters-output-base", default="/mnt/data/outputs/cotracker/visibility_clusters", type=str)
    ap.add_argument("--annotation-output-path", default="/mnt/data/outputs/cotracker/annotations/DAVIS/all/", type=str)
    ap.add_argument("--visibility-threshold", default=0.3, type=float)
    ap.add_argument("--matching-threshold", default=0.5, type=float)
    ap.add_argument("--job-id", default=0, type=int)
    ap.add_argument("--videos-per-job", default=-1, type=int)
    ap.add_argument("--debug", default=False, action="store_true")
    args = ap.parse_args()
    os.environ["CUDA_VISIBLE_DEVICES"] = args.gpu_id
    args.device = "cuda" if torch.cuda.is_available() else "cpu"
    random.seed(args.manualSeed)
    torch.manual_seed(args.manualSeed)
    if args.device == "cuda":
        torch.cuda.manual_seed_all(args.manualSeed)
    return args


def safe_exists(p):
    try:
        return Path(p).exists()
    except OSError as e:
        print(f"Warning: I/O error checking {p}: {e}")
        return False


def load_image_robust(path, max_retries=3, backoff=0.1):
    """BGR image like cv2.imread, None when the file is missing or unreadable after retries
    (OpenCV first, PIL as a fallback) - crw_utils.py:310-346."""
    path = Path(path)
    if not safe_exists(path):
        warnings.warn(f"File does not exist or the loading gracefully failed for: {path!s}")
        return None
    err = None
    for attempt in range(1, max_retries + 1):
        try:
            with open(path, "rb") as f:
                if len(f.read(16)) == 0:
                    raise IOError("File appears empty or unreadable")
            img = cv2.imread(str(path), cv2.IMREAD_COLOR)
            if img is not None:
                return img
            with Image.open(path) as pil:
                pil.verify()
            return cv2.cvtColor(np.array(Image.open(path)), cv2.COLOR_RGB2BGR)
        except Exception as e:  # noqa: BLE001
            err = e
            time.sleep(backoff * attempt)
    warnings.warn(f"Failed to load image {path!s} after {max_retries} attempts. Last error: {err}")
    return None


def load_image(img_path):
    img = load_image_robust(img_path)
    if img is None:
        return None
    rgb = (img.astype(np.float32) / 255.0)[:, :, ::-1].copy()
    return torch.from_numpy(np.transpose(rgb, (2, 0, 1))).float()


def color_normalize(x, mean, std):
    if x.size(0) == 1:
        x = x.repeat(3, 1, 1)
    for ch, m, s in zip(x, mean, std):
        ch.sub_(m).div_(s)
    return x


def rgb_to_label_ids(rgb: np.ndarray) -> np.ndarray:
    """label id = rank of the pixel's RGB tuple among the frame's non-black colours in
    lexicographic order, 0 for black (crw_utils.py:688-711 / cotracker_matching.py:54-71).
    Vectorised: the lexicographic order of (R,G,B) equals the numeric order of R<<16|G<<8|B."""
    key = (rgb[..., 0].astype(np.uint32) << 16) | (rgb[..., 1].astype(np.uint32) << 8) | rgb[..., 2].astype(np.uint32)
    colours, inv = np.unique(key, return_inverse=True)
    rank = np.arange(len(colours), dtype=np.int64)
    if colours[0] != 0:          # no black pixel: ranks start at 1
        rank += 1
    return rank[inv].reshape(key.shape)


def convert_lblimg_to_maskid(lblimg: np.ndarray):
    return rgb_to_label_ids(lblimg)[..., None]


def load_masks(mask_folder: str):
    """(T, H, W, 1) int64 label maps from a folder of colour PNGs."""
    paths = sorted(glob.glob(os.path.join(mask_folder, "*.png")))
    if not paths:
        raise ValueError(f"No .png masks found in {mask_folder!r}")
    if torch.cuda.is_available():
        # PNG decode and colour -> id on the GPU (s2d_png_decode, s2d_color_to_labels); files the device decoder does
        # not take go through load_image_robust, as below
        from s2d_b200 import png
        frames = png.load_rgb_frames(paths)
        if not frames:
            raise RuntimeError("No valid mask images could be read.")
        if len({tuple(f.shape) for f in frames}) == 1:
            return png.rgb_frames_to_labels(frames).cpu().to(torch.int64)[..., None]
        frames = [f.cpu().numpy() for f in frames]
        return torch.from_numpy(np.stack([rgb_to_label_ids(f)[..., None] for f in frames], axis=0))
    frames = []
    for p in paths:
        bgr = load_image_robust(p)
        if bgr is None:
            continue
        frames.append(cv2.cvtColor(bgr, cv2.COLOR_BGR2RGB))
    if not frames:
        raise RuntimeError("No valid mask images could be read.")
    return torch.from_numpy(np.stack([rgb_to_label_ids(f)[..., None] for f in frames], axis=0))


def make_paths(folder_path, label_path, dataset_name="DAVIS"):
    imgs = [i for i in os.listdir(folder_path) if i.endswith((".jpg", ".png", ".jpeg"))]
    lbls = [l for l in os.listdir(label_path) if "npy" not in l]
    under = lambda x: int(x.split("_")[1].split(".")[0])
    plain = lambda x: int(x.split(".")[0])
    if dataset_name == "SA-V":
        imgs.sort(key=under); lbls.sort(key=under)
    elif dataset_name == "ovis":
        imgs.sort(key=under)          # the reference sorts only the images for ovis (crw_utils.py:782-783)
    else:
        imgs.sort(key=plain); lbls.sort(key=plain)
    n = len(imgs)
    return ["%s/%s" % (folder_path, imgs[i]) for i in range(n)], ["%s/%s" % (label_path, lbls[i]) for i in range(n)]


def load_frames_and_masks(video_path, label_path, visibility_data, dataset_name="DAVIS"):
    """imgs (normalised), imgs_orig, lbls (T,1,H,W) int64 nearest-resized to the frame size,
    meta - or four Nones when a file cannot be read (crw_utils.py:796-857)."""
    frame_num = len(os.listdir(video_path))
    mean, std = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
    img_paths, lbl_paths = make_paths(video_path, label_path, dataset_name)
    imgs, imgs_orig = [], []
    for i in range(frame_num):
        img = load_image(img_paths[i])
        if img is None or load_image_robust(lbl_paths[i]) is None:
            return None, None, None, None
        imgs_orig.append(img.clone())
        imgs.append(color_normalize(img, mean, std))
    meta = dict(video_path=video_path, img_paths=img_paths, lbl_paths=lbl_paths, visibility=visibility_data)
    imgs = torch.stack(imgs)
    imgs_orig = torch.stack(imgs_orig)
    try:
        from . import _engine
    except ImportError:      # imported as a top-level module, like the reference's layout
        import _engine
    lbls = _engine.cached_labels(label_path, load_masks).permute(0, 3, 1, 2)
    if lbls.shape[-2:] != imgs.shape[-2:]:
        lbls = F.interpolate(lbls.float(), size=(imgs.size(2), imgs.size(3)), mode="nearest").long()
    return imgs, imgs_orig, lbls, meta
