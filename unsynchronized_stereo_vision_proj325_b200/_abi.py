"""ctypes mirror of include/usv_b200.h (PODs and constants only)."""
import ctypes as C

import numpy as np

USV_ABI_VERSION = 5
USV_OK, USV_ERR_INVALID_ARG, USV_ERR_CUDA, USV_ERR_NO_DEVICE, USV_ERR_UNSUPPORTED, USV_ERR_NOMEM = 0, -1, -2, -3, -4, -5
COST_SAD, COST_SSD, COST_NCC, COST_ZNCC, COST_CENSUS = 0, 1, 2, 3, 4
COST_NAMES = {"sad": COST_SAD, "ssd": COST_SSD, "ncc": COST_NCC, "zncc": COST_ZNCC, "census": COST_CENSUS}
DIST_NONE, DIST_PINHOLE, DIST_POWERLAW = 0, 1, 2
LEFT_CAM, RIGHT_CAM = 1, 0
NO_MATCH = 0xFFFFFFFF
NO_DISPARITY = 0xFFFF
NO_SUBPIXEL = -2**31  # disparity_x16 of a window without a refined disparity (INT32_MIN)

OUT_MATCHES, OUT_RIGHT_INDEX, OUT_RAW_COST, OUT_SCORE = 0x01, 0x02, 0x04, 0x08
OUT_DISTANCE, OUT_DISTANCE_F32, OUT_DISPARITY_U16, OUT_RAW_COST_U16 = 0x10, 0x20, 0x40, 0x80
OUT_RESOLVED_DISPARITY_U16 = 0x100

# numpy view of the reference's 16-byte `class Match` (P/Match.hpp:4-12)
MATCH_DTYPE = np.dtype([("LeftIndex", "<u4"), ("RightIndex", "<u4"), ("MatchValue", "<f8")], align=True)
assert MATCH_DTYPE.itemsize == 16


class Match(C.Structure):
    _fields_ = [("LeftIndex", C.c_uint32), ("RightIndex", C.c_uint32), ("MatchValue", C.c_double)]


class SearchParams(C.Structure):
    _fields_ = [
        ("tmpl_w", C.c_int32), ("tmpl_h", C.c_int32),
        ("search_min", C.c_int32), ("search_max", C.c_int32),
        ("stride_x", C.c_int32), ("stride_y", C.c_int32),
        ("cost_kind", C.c_int32), ("camera_side", C.c_int32),
        ("distance_kind", C.c_int32), ("reserved", C.c_int32),
        ("accept_threshold", C.c_double),
    ]


class FrameDesc(C.Structure):
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32), ("channels", C.c_int32),
        ("row_stride", C.c_int32), ("frame_stride", C.c_int64),
    ]


PRE_OPENCV3, PRE_OPENCV4 = 3, 4


class PreprocessParams(C.Structure):
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32), ("src_stride", C.c_int32), ("dst_stride", C.c_int32),
        ("src_frame_stride", C.c_int64), ("dst_frame_stride", C.c_int64), ("flavour", C.c_int32), ("lighting", C.c_int32),
    ]


class Outputs(C.Structure):
    _fields_ = [
        ("matches", C.c_void_p), ("right_index", C.c_void_p), ("raw_cost", C.c_void_p),
        ("score", C.c_void_p), ("distance", C.c_void_p), ("distance_f32", C.c_void_p),
        ("disparity_u16", C.c_void_p), ("raw_cost_u16", C.c_void_p), ("resolved_disparity_u16", C.c_void_p),
    ]


OUTPUT_FIELDS = (
    # name, mask bit, numpy dtype
    ("matches", OUT_MATCHES, MATCH_DTYPE),
    ("right_index", OUT_RIGHT_INDEX, np.dtype("<u4")),
    ("raw_cost", OUT_RAW_COST, np.dtype("<u4")),
    ("score", OUT_SCORE, np.dtype("<f8")),
    ("distance", OUT_DISTANCE, np.dtype("<f8")),
    ("distance_f32", OUT_DISTANCE_F32, np.dtype("<f4")),
    ("disparity_u16", OUT_DISPARITY_U16, np.dtype("<u2")),
    ("raw_cost_u16", OUT_RAW_COST_U16, np.dtype("<u2")),
    ("resolved_disparity_u16", OUT_RESOLVED_DISPARITY_U16, np.dtype("<u2")),
)


def make_params(tmpl_w=16, tmpl_h=16, search_min=0, search_max=1 << 20, stride_x=1, stride_y=1,
                cost="sad", camera_side=LEFT_CAM, distance_kind=DIST_PINHOLE, accept_threshold=0.75):
    """Search spec; defaults follow the reference (accept < 0.75, P/Main.cpp:417)."""
    kind = COST_NAMES[cost] if isinstance(cost, str) else int(cost)
    return SearchParams(tmpl_w, tmpl_h, search_min, search_max, stride_x, stride_y, kind,
                        int(camera_side), int(distance_kind), 0, float(accept_threshold))


def frame_desc_for(arr):
    """FrameDesc of a [n, H, W] or [n, H, W, C] uint8 batch (C-contiguous rows)."""
    assert arr.dtype == np.uint8 and arr.ndim in (3, 4)
    n, h, w = arr.shape[:3]
    c = arr.shape[3] if arr.ndim == 4 else 1
    return FrameDesc(w, h, c, arr.strides[1], arr.strides[0])
