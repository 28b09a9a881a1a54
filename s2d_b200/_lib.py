"""ctypes binding of libs2d_b200.so (C ABI in include/s2d_b200.h).

There is no CPU fallback: if the CUDA library has not been built, or an entry point fails,
this raises - the product path never silently degrades (the numpy oracle under oracle/ is test
infrastructure and is never imported from here)."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("S2D_B200_LIB") or os.path.join(_HERE, "libs2d_b200.so")   # override: debug builds (make check)

S2D_MAX_LABELS = 256
S2D_MAX_CLUSTERS = 16
S2D_VIDINFO_WORDS = 8
S2D_CLINFO_WORDS = 16
S2D_PV_TMAP_BYTES = 32 * 128 + 128
S2D_DESC_VIS_BITS = 1


class VideoDesc(C.Structure):
    """mirror of s2d_video_desc"""
    _fields_ = [
        ("T", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("P", C.c_int32),
        ("Nm", C.c_int32), ("L", C.c_int32), ("TW", C.c_int32), ("NW", C.c_int32),
        ("row0", C.c_int64), ("frame0", C.c_int64),
        ("labels", C.c_void_p), ("tracks", C.c_void_p), ("vis", C.c_void_p), ("npts", C.c_void_p),
        ("tstart", C.c_void_p), ("Ttr", C.c_int32), ("flags", C.c_int32),
        ("vt_off", C.c_int64), ("hits_off", C.c_int64), ("xbits_off", C.c_int64), ("mbits_off", C.c_int64),
    ]


_P, _I, _L, _D, _F = C.c_void_p, C.c_int, C.c_int64, C.c_double, C.c_float

# name -> argtypes (restype is int unless listed in _RESTYPES); must list every symbol the
# header declares (tests/test_cabi.py checks this against include/s2d_b200.h)
SIGNATURES = {
    "s2d_last_error": [],
    "s2d_version": [],
    "s2d_desc_size": [],
    "s2d_device_sm_count": [_I],
    "s2d_host_register": [_P, _L],
    "s2d_host_unregister": [_P],
    "s2d_device_pci_bus_id": [_I, C.c_char_p, _I],
    "s2d_label_stats": [_P, _I, _I, _L, _L, _P, _P, _P, _P, _P, _P, _P],
    "s2d_vis_reduce": [_P, _I, _L, _P, _P, _P],
    "s2d_binarize": [_P, _I, _L, _P, _F, _P, _P],
    "s2d_dbscan_work_ints": [_L, _I, C.POINTER(C.c_int64)],
    "s2d_dbscan_visibility": [_P, _I, _I, _I, _L, _P, _D, _I, _P, _P, _P, _P],
    "s2d_windows": [_P, _I, _L, _I, _L, _L, _P, _P, _P, _F, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "s2d_point_votes_variant": [_I],
    "s2d_point_votes_work_ints": [_L, C.POINTER(C.c_int64)],
    "s2d_point_votes_tmaps": [_P, _I, _P],
    "s2d_point_votes": [_P, _I, _I, _I, _I, _I, _L, _P, _P, _P, _P, _P, _P, _P],
    "s2d_point_votes_sized": [_P, _I, _I, _I, _I, _I, _L, _P, _P, _P, _P, _L, _P, _P, _P],
    "s2d_appearance_events": [_P, _I, _I, _I, _F, _I, _I, _P, _P, _P, _P, _P, _P],
    "s2d_boolean_visibility": [_P, _L, _F, _P, _P],
    "s2d_rle_work_ints": [_I, _I, _I, _I, C.POINTER(C.c_int64)],
    "s2d_rle_encode": [_P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P],
    "s2d_rle_area_bbox": [_P, _P, _I, _P, _P, _P, _P],
    "s2d_label_rle_work_ints": [_L, _L, _I, _I, C.POINTER(C.c_int64)],
    "s2d_label_rle": [_P, _I, _I, _I, _I, _I, _L, _L, _P, _P, _P, _L, _P, _P, _P, _P, _P],
    "s2d_rle_strings": [_P, _P, _I, _L, _P, _L, _P, _P, _P, _P],
    "s2d_rle_from_strings_work_ints": [_I, _L, C.POINTER(C.c_int64)],
    "s2d_rle_from_strings": [_P, _P, _I, _P, _L, _P, _P, _P, _P, _P],
    "s2d_rle_decode_work_ints": [_I, _L, C.POINTER(C.c_int64)],
    "s2d_rle_decode": [_P, _P, _I, _P, _P, _P, _P, _P, _P, _P],
    "s2d_png_decode_work_ints": [_I, _L, C.POINTER(C.c_int64)],
    "s2d_png_decode": [_P, _P, _P, _I, _P, _P, _P, _P],
    "s2d_annotation_layout_work_ints": [_L, _I, C.POINTER(C.c_int64)],
    "s2d_annotation_layout": [_P, _I, _L] + [_P] * 15 + [_L, _P, _P, _P, _P, _P, _P, _P, _L, _P, _P, _P],
    "s2d_annotation_json_work_ints": [_L, _I, C.POINTER(C.c_int64)],
    "s2d_annotation_json": [_P, _I, _L] + [_P] * 6 + [_L] + [_P] * 4 + [_L, _P, _P, _P, _P],
    "s2d_select": [_P, _I, _I, _L, _P, _P, _P, _P, _D, _D, _I, _P, _P, _P, _P, _P],
    "s2d_group_work_ints": [_L, _I, C.POINTER(C.c_int64)],
    "s2d_group": [_P, _I, _I, _I, _L, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "s2d_group_gram": [_P, _I, _I, _I, _L, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "s2d_unpack_bits": [_P, _I, _I, _L, _P, _P],
    "s2d_hamming_dbscan": [_P, _I, _I, _I, _D, _I, _P, _P, _P],
    "s2d_pack_bits": [_P, _I, _L, _P, _P],
    "s2d_overlap_bits": [_P, _I, _P, _I, _L, _P, _P, _P, _P],
    "s2d_overlap_i8": [_P, _I, _P, _I, _L, _P, _P],
    "s2d_overlap_gram_work_ints": [_I, _I, _L, C.POINTER(C.c_int64)],
    "s2d_overlap_gram_tiling": [_I, _I, C.POINTER(C.c_int)],
    "s2d_overlap_gram_band_work_ints": [_I, _I, _L, _I, C.POINTER(C.c_int64)],
    "s2d_overlap_gram_labels_banded": [_P, _I, _I, _L, _I, _P, _P, _P],
    "s2d_overlap_gram_executed_ops": [_I, _I, _L, C.POINTER(C.c_double)],
    "s2d_overlap_gram_labels": [_P, _I, _I, _L, _P, _P, _P],
    "s2d_color_to_labels_work_ints": [_I, C.POINTER(C.c_int64)],
    "s2d_color_to_labels": [_P, _I, _L, _P, _P, _P, _P],
    "s2d_rasterise_tracks": [_P, _I, _I, _I, _I, _P, _P],
}
_RESTYPES = {"s2d_last_error": C.c_char_p}

_lib = None


class S2DError(RuntimeError):
    pass


def load():
    """Load the shared library (once). Raises if it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise S2DError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C s2d_b200/csrc`). s2d_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = _RESTYPES.get(name, C.c_int)
    if lib.s2d_desc_size() != C.sizeof(VideoDesc):
        raise S2DError(f"s2d_video_desc size mismatch: C {lib.s2d_desc_size()} vs ctypes {C.sizeof(VideoDesc)}")
    _lib = lib
    return lib


def call(name, *args):
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise S2DError(f"{name} failed ({rc}): {lib.s2d_last_error().decode()}")
    return rc
