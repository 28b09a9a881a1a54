"""PNG label maps on the device: mask folders decoded straight into label ids.

The host walks each file's chunks (`parse_png`, per chunk, never per byte); one `s2d_png_decode` call inflates every
accepted file's zlib stream, undoes the row filters and writes the RGB pixels `cv2.imread(path, cv2.IMREAD_COLOR)`
returns (in RGB order); `s2d_color_to_labels` then turns the frames into label ids.

Files the device path does not take are decoded on the host through `crw_utils.load_image_robust`, exactly as before:
interlaced (Adam7) files, animated PNGs, files with a chunk outside `ALLOWED_CHUNKS`, a bad CRC, a truncated file, and
any file the kernel flags (malformed deflate data, wrong size, bad filter byte, adler32 mismatch, palette index past the
palette). Files that cannot be read at all follow load_image_robust's rules (warning, frame skipped)."""
from __future__ import annotations

import ctypes as C
import struct
import zlib
from dataclasses import dataclass
from typing import NamedTuple

import numpy as np
import torch

from . import _lib

PNG_SIGNATURE = b"\x89PNG\r\n\x1a\n"
# chunks cv2's IMREAD_COLOR decode ignores (or, tRNS, drops with the alpha channel); each is covered by a GPU test
ALLOWED_CHUNKS = frozenset({b"IHDR", b"PLTE", b"IDAT", b"IEND", b"tRNS", b"gAMA", b"cHRM", b"sRGB", b"pHYs", b"tEXt",
                            b"zTXt", b"iTXt", b"tIME", b"bKGD"})
LEGAL_DEPTHS = {0: (1, 2, 4, 8, 16), 2: (8, 16), 3: (1, 2, 4, 8), 4: (8, 16), 6: (8, 16)}
CHANNELS = {0: 1, 2: 3, 3: 1, 4: 2, 6: 4}
MAX_ROWBYTES = 16384            # S2D_PNG_MAX_ROWBYTES
MAX_RAW_BYTES = 1 << 30         # S2D_PNG_MAX_RAW_BYTES

DESC_DTYPE = np.dtype([("width", "<i4"), ("height", "<i4"), ("bit_depth", "<i4"), ("color_type", "<i4"),
                       ("raw_offset", "<i8"), ("rgb_offset", "<i8"), ("palette_size", "<i4"), ("reserved", "<i4"),
                       ("palette", "u1", (768,))])
assert DESC_DTYPE.itemsize == 808   # sizeof(s2d_png_desc)


@dataclass
class ParsedPng:
    width: int
    height: int
    bit_depth: int
    color_type: int
    palette: bytes          # PLTE (RGB triples), empty unless colour type 3
    zdata: bytes            # the IDAT payloads joined: one zlib stream

    @property
    def rowbytes(self) -> int:
        return (self.width * CHANNELS[self.color_type] * self.bit_depth + 7) // 8

    @property
    def raw_bytes(self) -> int:
        return self.height * (1 + self.rowbytes)


def parse_png(data) -> ParsedPng | None:
    """IHDR, PLTE and the joined IDAT payloads of a PNG file, or None for a file the device decoder does not take:
    not a PNG, interlaced, an APNG or any chunk outside ALLOWED_CHUNKS, a bad chunk CRC, chunks out of order, a
    truncated file, a size past the kernel's limits, or a zlib header other than deflate with a window <= 32 KB and no
    preset dictionary."""
    mv = memoryview(data)
    n = len(mv)
    if n < 8 or bytes(mv[:8]) != PNG_SIGNATURE:
        return None
    pos, ihdr, plte, idat, idat_done = 8, None, b"", [], False
    while True:
        if pos + 12 > n:
            return None                                             # truncated: no IEND
        length, = struct.unpack_from(">I", mv, pos)
        ctype = bytes(mv[pos + 4:pos + 8])
        end = pos + 12 + length
        if length >= 1 << 31 or end > n:
            return None
        if zlib.crc32(mv[pos + 4:pos + 8 + length]) != struct.unpack_from(">I", mv, pos + 8 + length)[0]:
            return None
        if ctype not in ALLOWED_CHUNKS or (ihdr is None) != (ctype == b"IHDR"):
            return None
        body = mv[pos + 8:pos + 8 + length]
        if ctype == b"IHDR":
            if length != 13:
                return None
            ihdr = struct.unpack(">IIBBBBB", body)
        elif ctype == b"PLTE":
            if plte or idat or length == 0 or length % 3 or length > 768:
                return None
            plte = bytes(body)
        elif ctype == b"IDAT":
            if idat_done:
                return None                                         # IDAT chunks must be consecutive
            idat.append(body)
        elif idat:
            idat_done = True
        pos = end
        if ctype == b"IEND":
            break
    if pos != n or not idat:
        return None
    w, h, bd, ct, method, filt, interlace = ihdr
    if method or filt or interlace or bd not in LEGAL_DEPTHS.get(ct, ()) or not (1 <= w <= MAX_ROWBYTES) or h < 1:
        return None
    if (ct == 3) != bool(plte) or (ct == 3 and len(plte) // 3 > 1 << bd):
        return None
    p = ParsedPng(w, h, bd, ct, plte, b"".join(idat))
    if p.rowbytes > MAX_ROWBYTES or p.raw_bytes > MAX_RAW_BYTES or len(p.zdata) < 6:
        return None
    cmf, flg = p.zdata[0], p.zdata[1]
    if cmf & 15 != 8 or cmf >> 4 > 7 or flg & 0x20 or (cmf * 256 + flg) % 31:
        return None
    return p


def pack_descs(parsed, raw_offsets, rgb_offsets) -> np.ndarray:
    """s2d_png_desc [N] of parsed files whose scanlines / RGB frames go to the given byte offsets."""
    d = np.zeros(len(parsed), DESC_DTYPE)
    for i, p in enumerate(parsed):
        d[i]["width"], d[i]["height"], d[i]["bit_depth"], d[i]["color_type"] = p.width, p.height, p.bit_depth, p.color_type
        d[i]["raw_offset"], d[i]["rgb_offset"] = raw_offsets[i], rgb_offsets[i]
        if p.palette:
            d[i]["palette_size"] = len(p.palette) // 3
            d[i]["palette"][:len(p.palette)] = np.frombuffer(p.palette, np.uint8)
    return d


class DecodedPngs(NamedTuple):
    frames: list            # [H, W, 3] uint8 RGB on the device per file, None where not accepted
    accepted: np.ndarray    # bool [n]: parsed and decoded without a flag
    status: np.ndarray      # int32 [n]: the kernel's S2D_PNG_BAD_* bits, -1 where parse_png returned None


class StagedPngs(NamedTuple):
    """Parsed files uploaded for one s2d_png_decode call (descs | z_offsets | zdata in one device buffer)."""
    parsed: list
    dbuf: torch.Tensor
    o_z: int                # byte offset of z_offsets in dbuf
    o_data: int             # byte offset of zdata in dbuf
    raw_off: np.ndarray     # int64 [N + 1] scanline offsets (the last = the scratch bytes)
    rgb_off: np.ndarray     # int64 [N + 1] RGB offsets (the last = the output bytes)


def stage_pngs(parsed, device) -> StagedPngs:
    """Lay out parsed files back to back and upload them with one async copy from one pinned buffer."""
    N = len(parsed)
    z_off = np.concatenate([[0], np.cumsum([len(p.zdata) for p in parsed])]).astype(np.int64)
    raw_off = np.concatenate([[0], np.cumsum([p.raw_bytes for p in parsed])]).astype(np.int64)
    rgb_off = np.concatenate([[0], np.cumsum([p.height * p.width * 3 for p in parsed])]).astype(np.int64)
    descs = pack_descs(parsed, raw_off[:-1], rgb_off[:-1])
    o_z = N * DESC_DTYPE.itemsize
    o_data = o_z + 8 * (N + 1)
    staged = torch.empty(o_data + int(z_off[-1]), dtype=torch.uint8, pin_memory=True)
    buf = staged.numpy()
    buf[:o_z] = descs.view(np.uint8)
    buf[o_z:o_data] = z_off.view(np.uint8)
    for p, a in zip(parsed, z_off[:-1]):
        buf[o_data + a:o_data + a + len(p.zdata)] = np.frombuffer(p.zdata, np.uint8)
    return StagedPngs(parsed, staged.to(device, non_blocking=True), o_z, o_data, raw_off, rgb_off)


def launch_decode(sp: StagedPngs, work=None, rgb=None, status=None):
    """Enqueue s2d_png_decode of staged files on the current stream; returns (rgb bytes, status int32 [N]) on the
    device. work / rgb / status may be passed in to reuse buffers."""
    device = sp.dbuf.device
    N = len(sp.parsed)
    if work is None:
        nw = C.c_int64()
        _lib.call("s2d_png_decode_work_ints", N, int(sp.raw_off[-1]), C.byref(nw))
        work = torch.empty(nw.value, dtype=torch.int32, device=device)
    rgb = torch.empty(int(sp.rgb_off[-1]), dtype=torch.uint8, device=device) if rgb is None else rgb
    status = torch.empty(N, dtype=torch.int32, device=device) if status is None else status
    base = sp.dbuf.data_ptr()
    _lib.call("s2d_png_decode", base + sp.o_data, base + sp.o_z, base, N, work.data_ptr(), rgb.data_ptr(),
              status.data_ptr(), torch.cuda.current_stream(device).cuda_stream)
    return rgb, status


def decode_pngs(blobs, device=None) -> DecodedPngs:
    """Decode a list of PNG files (bytes) on the device with one upload and one s2d_png_decode call. The accepted
    files' frames are views of one buffer, back to back in list order."""
    device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    n = len(blobs)
    parsed = [parse_png(b) for b in blobs]
    idx = [i for i, p in enumerate(parsed) if p is not None]
    frames, status = [None] * n, np.full(n, -1, np.int32)
    if not idx:
        return DecodedPngs(frames, np.zeros(n, bool), status)
    sp = stage_pngs([parsed[i] for i in idx], device)
    rgb, st = launch_decode(sp)
    st_h = st.cpu().numpy()
    for k, i in enumerate(idx):
        status[i] = st_h[k]
        if st_h[k] == 0:
            p = sp.parsed[k]
            frames[i] = rgb[sp.rgb_off[k]:sp.rgb_off[k + 1]].view(p.height, p.width, 3)
    return DecodedPngs(frames, status == 0, status)


def _read(path):
    try:
        with open(path, "rb") as f:
            return f.read()
    except OSError:
        return None


def load_rgb_frames(paths, device=None) -> list:
    """RGB frames ([H, W, 3] uint8 on the device) of the mask files that can be read, in path order, as
    cv2.cvtColor(load_image_robust(p), COLOR_BGR2RGB) gives them: PNGs the device decoder takes are decoded there,
    every other file goes through load_image_robust (with its warnings; None skips the frame)."""
    from .keymask_ident import crw_utils
    device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    blobs = [_read(p) for p in paths]
    dec = decode_pngs([b if b is not None else b"" for b in blobs], device)
    out = []
    for p, f in zip(paths, dec.frames):
        if f is None:
            import cv2
            bgr = crw_utils.load_image_robust(p)
            if bgr is None:
                continue
            f = torch.from_numpy(np.ascontiguousarray(cv2.cvtColor(bgr, cv2.COLOR_BGR2RGB))).to(device)
        out.append(f)
    return out


def _stack(frames) -> torch.Tensor:
    """[T, H, W, 3] of same-shape frames: a view when they already lie back to back in one buffer."""
    f0 = frames[0]
    step = f0.numel()
    if all(f.is_contiguous() and f.untyped_storage().data_ptr() == f0.untyped_storage().data_ptr()
           and f.data_ptr() == f0.data_ptr() + k * step for k, f in enumerate(frames)):
        return f0.new_empty(0).set_(f0.untyped_storage(), f0.storage_offset(), (len(frames),) + tuple(f0.shape))
    return torch.stack(frames)


def rgb_frames_to_labels(frames) -> torch.Tensor:
    """uint8 [T, H, W] label ids of same-shape RGB frames on the device (s2d_color_to_labels, one call)."""
    from .keymask_ident import _engine
    labels, _ = _engine.color_frames_to_labels(_stack(frames))
    return labels


def load_label_maps(paths, device=None):
    """Label maps of a folder's mask files (label = 1 + rank of the pixel's colour among the frame's non-black colours,
    0 for black), decoded and converted on the device. Returns uint8 [T, H, W] on the device when the frames share one
    shape, else a list of [H, W] maps (one s2d_color_to_labels call per distinct shape). Unreadable files are skipped
    as load_masks skips them; RuntimeError when none can be read."""
    frames = load_rgb_frames(paths, device)
    if not frames:
        raise RuntimeError("No valid mask images could be read.")
    shapes = sorted({tuple(f.shape) for f in frames})
    if len(shapes) == 1:
        return rgb_frames_to_labels(frames)
    out = [None] * len(frames)
    for s in shapes:
        ks = [k for k, f in enumerate(frames) if tuple(f.shape) == s]
        lab = rgb_frames_to_labels([frames[k] for k in ks])
        for j, k in enumerate(ks):
            out[k] = lab[j]
    return out
