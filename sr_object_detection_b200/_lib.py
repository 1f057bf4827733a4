"""ctypes loader for libyolo2_b200.so (the C-ABI declared in include/*.h).

There is no fallback: if the shared library is missing it is built in-tree with nvcc,
and if that fails the import error propagates.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

from . import build as _build

_LIB = None


class Y2Error(RuntimeError):
    pass


class ConvDesc(C.Structure):
    """Mirror of `y2_conv_desc` (include/yolo2_b200_kernels.h)."""
    _fields_ = [
        ("in_", C.c_void_p), ("in_cs", C.c_int), ("cin", C.c_int),
        ("batch", C.c_int), ("h", C.c_int), ("w", C.c_int), ("ksize", C.c_int),
        ("wt", C.c_void_p), ("cout", C.c_int), ("npad", C.c_int),
        ("block_n", C.c_int), ("block_k", C.c_int),
        ("alpha", C.c_void_p), ("beta", C.c_void_p), ("act", C.c_int),
        ("out", C.c_void_p), ("out_cs", C.c_int), ("out_mode", C.c_int), ("in_order", C.c_int),
    ]


class Det(C.Structure):
    """Mirror of `y2_det`."""
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("w", C.c_float), ("h", C.c_float),
                ("prob", C.c_float), ("obj_id", C.c_int), ("box_index", C.c_int)]


class FrameWindow(C.Structure):
    """Mirror of `y2_frame_window`: where one frame of a packed frame list sits and the window it fills."""
    _fields_ = [("offset", C.c_ulonglong), ("src_w", C.c_int), ("src_h", C.c_int), ("dx", C.c_int), ("dy", C.c_int),
                ("new_w", C.c_int), ("new_h", C.c_int), ("w_scale", C.c_float), ("h_scale", C.c_float)]


def frame_list_layout(sizes, w: int, h: int, letterbox: bool):
    """y2_frame_list_layout for frames of sizes [(frame_w, frame_h), ...] on a w x h network: (records, table offset,
    packed size in bytes)."""
    lib = load()
    n = len(sizes)
    fw = (C.c_int * max(n, 1))(*[s[0] for s in sizes])
    fh = (C.c_int * max(n, 1))(*[s[1] for s in sizes])
    win = (FrameWindow * max(n, 1))()
    toff = C.c_size_t()
    total = lib.y2_frame_list_layout(n, fw, fh, w, h, int(letterbox), win, C.byref(toff))
    return list(win)[:n], toff.value, total


class StreamSrc(C.Structure):
    """Mirror of `y2_stream_src`: where the 3 ring slots of an image's stream come from, and the ring row it commits."""
    _fields_ = [("src", C.c_int * 3), ("commit", C.c_int)]


def stream_plan(stream_ids, max_streams: int, frame_index, frames_seen):
    """y2_stream_plan for one list of stream ids: (records, advanced frame_index, advanced frames_seen).  The counter
    lists are not modified; a bad id raises Y2Error."""
    lib = load()
    n = len(stream_ids)
    ids = (C.c_int * max(n, 1))(*stream_ids)
    fi = (C.c_int * max_streams)(*frame_index)
    seen = (C.c_int * max_streams)(*frames_seen)
    plan = (StreamSrc * max(n, 1))()
    check(lib.y2_stream_plan(n, ids, max_streams, fi, seen, plan), "y2_stream_plan")
    return list(plan)[:n], list(fi), list(seen)


class TrackImg(C.Structure):
    """Mirror of `y2_track_img`: one image of a tracked batch and its stream's history position before it."""
    _fields_ = [("image", C.c_int), ("stream", C.c_int), ("w", C.c_int), ("h", C.c_int), ("head", C.c_int),
                ("len", C.c_int), ("restart", C.c_int)]


def track_plan(stream_ids, sizes, max_streams: int, story: int, head, length, restart):
    """y2_track_plan for one list of stream ids with frame sizes [(w, h), ...]: (records, offsets, advanced head,
    advanced len, advanced restart).  The counter lists are not modified; a bad argument raises Y2Error."""
    lib = load()
    n = len(stream_ids)
    ids = (C.c_int * max(n, 1))(*stream_ids)
    fw = (C.c_int * max(n, 1))(*[s[0] for s in sizes])
    fh = (C.c_int * max(n, 1))(*[s[1] for s in sizes])
    hd, ln, rs = ((C.c_int * max_streams)(*v) for v in (head, length, restart))
    recs = (TrackImg * max(n, 1))()
    offsets = (C.c_int * (n + 1))()
    k = lib.y2_track_plan(n, ids, fw, fh, max_streams, story, hd, ln, rs, recs, offsets)
    check(0 if k >= 1 else k, "y2_track_plan")
    return list(recs)[:n], list(offsets)[:k + 1], list(hd), list(ln), list(rs)


def lib_path() -> Path:
    return _build.LIB


def load() -> C.CDLL:
    global _LIB
    if _LIB is not None:
        return _LIB
    path = _build.LIB
    if not path.exists():
        _build.build()
    if not path.exists():
        raise Y2Error(f"{path} is missing and could not be built; the CUDA extension is mandatory")
    lib = C.CDLL(str(path), mode=C.RTLD_GLOBAL)
    _declare(lib)
    _LIB = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().y2_last_error().decode(errors="replace")
        raise Y2Error(f"{what or 'y2 call'} failed (rc={rc}): {msg}")


def _declare(lib: C.CDLL) -> None:
    vp, i, f = C.c_void_p, C.c_int, C.c_float
    sigs = {
        "y2_last_error": (C.c_char_p, []),
        "y2_version": (C.c_char_p, []),
        "y2_device_count": (i, [C.POINTER(i)]),
        "y2_set_device": (i, [i]),
        "y2_malloc": (i, [C.POINTER(vp), C.c_size_t]),
        "y2_free": (i, [vp]),
        "y2_memset": (i, [vp, i, C.c_size_t, vp]),
        "y2_host_alloc": (i, [C.POINTER(vp), C.c_size_t]),
        "y2_host_free": (i, [vp]),
        "y2_memcpy_h2d": (i, [vp, vp, C.c_size_t, vp]),
        "y2_memcpy_d2h": (i, [vp, vp, C.c_size_t, vp]),
        "y2_stream_create": (i, [C.POINTER(vp)]),
        "y2_stream_destroy": (i, [vp]),
        "y2_stream_sync": (i, [vp]),
        "y2_device_sync": (i, []),
        "y2_graph_begin": (i, [vp]),
        "y2_graph_end": (i, [vp, C.POINTER(vp)]),
        "y2_graph_launch": (i, [vp, vp]),
        "y2_graph_destroy": (i, [vp]),
        "y2_event_create": (i, [C.POINTER(vp)]),
        "y2_event_record": (i, [vp, vp]),
        "y2_event_elapsed_ms": (i, [vp, vp, C.POINTER(f)]),
        "y2_event_sync": (i, [vp]),
        "y2_stream_wait_event": (i, [vp, vp]),
        "y2_event_destroy": (i, [vp]),
        "y2_conv_plan_create": (i, [C.POINTER(ConvDesc), C.POINTER(vp)]),
        "y2_conv_plan_launch": (i, [vp, vp]),
        "y2_conv_plan_destroy": (None, [vp]),
        "y2_conv_plan_tiles": (i, [vp]),
        "y2_conv_plan_variant": (i, [vp]),
        "y2_conv_plan_order": (i, [vp]),
        "y2_stem_prepare": (i, []),
        "y2_stem_conv_pool": (i, [vp, i, i, i, i, vp, i, vp, vp, i, vp, i, vp]),
        "y2_stem_conv_pool_u8": (i, [vp, i, i, i, vp, i, vp, vp, i, vp, i, vp]),
        "y2_pack_nchw_f32": (i, [vp, vp, i, i, i, i, i, i, vp]),
        "y2_pack_patches_f32": (i, [vp, vp, i, i, i, i, i, i, vp]),
        "y2_gather_patches_f32": (i, [vp, vp, i, i, i, i, i, i, i, i, i, i, vp]),
        "y2_gather_patches_bf16": (i, [vp, i, i, i, i, vp, i, i, i, i, i, i, vp]),
        "y2_gather_rows_f32": (i, [vp, vp, i, i, i, i, i, i, i, i, i, i, vp]),
        "y2_resize_u8_to_f32": (i, [vp, vp, i, i, i, i, i, vp]),
        "y2_frame_list_layout": (C.c_size_t, [i, C.POINTER(i), C.POINTER(i), i, i, i, C.POINTER(FrameWindow),
                                              C.POINTER(C.c_size_t)]),
        "y2_frames_u8_to_f32": (i, [vp, vp, i, vp, i, i, i, vp]),
        "y2_stream_plan": (i, [i, C.POINTER(i), i, C.POINTER(i), C.POINTER(i), C.POINTER(StreamSrc)]),
        "y2_stream_mean": (i, [vp, vp, vp, i, i, vp, vp]),
        "y2_stream_commit": (i, [vp, vp, vp, i, i, vp]),
        "y2_track_plan": (i, [i, C.POINTER(i), C.POINTER(i), C.POINTER(i), i, i, C.POINTER(i), C.POINTER(i),
                              C.POINTER(i), C.POINTER(TrackImg), C.POINTER(i)]),
        "y2_stream_track": (i, [vp, i, vp, vp, vp, i, i, i, i, vp, vp, vp, vp, i, vp]),
        "y2_unpack_to_nchw_f32": (i, [vp, vp, i, i, i, i, i, vp]),
        "y2_flat_to_nchw_f32": (i, [vp, vp, i, i, i, i, vp]),
        "y2_nchw_to_flat_f32": (i, [vp, vp, i, i, i, vp]),
        "y2_maxpool": (i, [vp, i, vp, i, i, i, i, i, i, i, i, i, i, vp]),
        "y2_reorg": (i, [vp, i, vp, i, i, i, i, i, i, vp]),
        "y2_reorg_table": (i, [vp, i, i, i, i, i, vp]),
        "y2_reorg_gather": (i, [vp, i, vp, i, vp, i, i, i, i, i, vp]),
        "y2_copy_channels": (i, [vp, i, vp, i, i, i, i, i, vp]),
        "y2_region_forward": (i, [vp, vp, i, i, i, i, i, i, vp, vp, vp]),
        "y2_region_boxes": (i, [vp, vp, vp, vp, i, i, i, i, i, f, f, f, i, i, i, vp, vp, i, vp]),
        "y2_nms_sort": (i, [vp, vp, i, i, i, f, vp]),
        "y2_collect": (i, [vp, vp, i, i, i, f, vp, vp, i, vp]),
        "y2_avgpool_flat": (i, [vp, vp, i, i, i, i, vp]),
        "y2_softmax_rows": (i, [vp, vp, i, i, f, vp]),
        "y2_shortcut": (i, [vp, i, vp, i, i, i, i, vp, i, i, i, i, i, i, i, vp, i, vp, vp]),
    }
    for name, (res, args) in sigs.items():
        fn = getattr(lib, name, None)
        if fn is None:
            continue  # symbol presence is asserted by tests/test_abi.py against include/*.h
        fn.restype = res
        fn.argtypes = args
