"""CPU tests of the frame-descriptor entries (RGB, BGR or NV12 frames with a row pitch, in host or device memory): the
NV12 rule against OpenCV's output, the layout that stages a descriptor list, the Python descriptor builder, the ctypes
mirror, and the refusal of every entry on a network without a device plan."""
import ctypes as C
import hashlib
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from sr_object_detection_b200 import _lib, darknet as dn, synth
from tests.golden.make_nv12_golden import SMALL, nv12_pattern

ROOT = Path(__file__).resolve().parents[1]
GOLDEN = ROOT / "tests" / "golden" / "nv12_rgb.npz"


def nv12_to_rgb(nv12: np.ndarray) -> np.ndarray:
    """uint8 [h*3/2][w] NV12 -> uint8 [h][w][3] RGB: BT.601 limited range in OpenCV's 20-bit fixed point"""
    h, w = nv12.shape[0] * 2 // 3, nv12.shape[1]
    uv = nv12[h:].reshape(h // 2, w // 2, 2).astype(np.int64)
    u = uv[..., 0].repeat(2, 0).repeat(2, 1) - 128
    v = uv[..., 1].repeat(2, 0).repeat(2, 1) - 128
    y = np.maximum(nv12[:h].astype(np.int64) - 16, 0) * 1220542
    half = 1 << 19
    r = (y + half + 1673527 * v) >> 20
    g = (y + half - 852492 * v - 409993 * u) >> 20
    b = (y + half + 2116026 * u) >> 20
    return np.stack([r, g, b], -1).clip(0, 255).astype(np.uint8)


def to_rgb(frame: np.ndarray, fmt: int) -> np.ndarray:
    """the tight RGB bytes the frame-list entries would be fed for a frame of format fmt"""
    if fmt == dn.FRAME_NV12:
        return nv12_to_rgb(frame)
    return np.ascontiguousarray(frame[..., ::-1] if fmt == dn.FRAME_BGR24 else frame)


# ---- the NV12 rule ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("w,h", SMALL)
def test_nv12_rule_equals_opencv(w, h):
    d = np.load(GOLDEN)
    nv12 = d[f"nv12_{w}x{h}"]
    y, uv = nv12[:h], nv12[h:]
    assert y.min() <= 16 or w * h < 16  # the small frames reach both ends of every plane
    if w * h >= 64 * 48:
        assert y.min() <= 16 and y.max() >= 235 and uv.min() == 0 and uv.max() == 255
    assert np.array_equal(nv12_to_rgb(nv12), d[f"rgb_{w}x{h}"]), str(d["opencv_version"])


def test_nv12_rule_equals_opencv_on_every_uv_pair_at_1080p():
    frame = nv12_pattern(1920, 1080)
    pairs = frame[1080:].reshape(-1, 2)
    assert len(np.unique(pairs[:, 0].astype(np.int32) * 256 + pairs[:, 1])) == 65536
    got = hashlib.sha256(nv12_to_rgb(frame).tobytes()).hexdigest()
    assert got == str(np.load(GOLDEN)["pattern_1920x1080_sha256"])


# ---- layout -------------------------------------------------------------------------------------------------------
def _desc(w, h, fmt, on_device=0, data=0x1000, pitch=0, uv=0, uv_pitch=0):
    d = dn.FrameDesc()
    d.data, d.uv, d.w, d.h, d.pitch, d.uv_pitch, d.format, d.on_device = data, uv or None, w, h, pitch, uv_pitch, \
        fmt, on_device
    return d


MIXED = [(_desc(1920, 1080, dn.FRAME_NV12), 1920 * 1080 * 3 // 2), (_desc(5, 3, dn.FRAME_RGB24), 45),
         (_desc(64, 48, dn.FRAME_NV12, on_device=1, data=0x7f0000001001, pitch=80), 0),
         (_desc(7, 9, dn.FRAME_BGR24), 189), (_desc(2, 2, dn.FRAME_NV12), 6),
         (_desc(33, 17, dn.FRAME_BGR24, on_device=1, data=0x7f0000100003, pitch=101), 0),
         (_desc(16, 10, dn.FRAME_NV12, on_device=1, data=0x7f0000200000, pitch=16, uv=0x7f0000300005, uv_pitch=24), 0),
         (_desc(500, 375, dn.FRAME_RGB24), 500 * 375 * 3)]


@pytest.mark.parametrize("letterbox", [False, True])
def test_layout_packs_host_frames_and_leaves_device_frames_in_place(letterbox):
    descs = [d for d, _ in MIXED]
    recs, toff, total = _lib.frame_desc_layout(descs, 416, 416, letterbox)
    wins, _, _ = _lib.frame_list_layout([(d.w, d.h) for d in descs], 416, 416, letterbox)
    end = 0
    for r, win, (d, staged) in zip(recs, wins, MIXED):
        # the geometry of the frame-list record, the offset aside
        for f in ("src_w", "src_h", "dx", "dy", "new_w", "new_h", "w_scale", "h_scale"):
            assert getattr(r.win, f) == getattr(win, f), f
        assert r.format == d.format
        row = d.w * (1 if d.format == dn.FRAME_NV12 else 3)
        if d.on_device:  # its own addresses, the defaults applied
            assert r.win.offset == d.data and r.pitch == (d.pitch or row)
            if d.format == dn.FRAME_NV12:
                assert r.uv == (d.uv or d.data + d.h * r.pitch) and r.uv_pitch == (d.uv_pitch or r.pitch)
            continue
        assert r.win.offset % 16 == 0 and end <= r.win.offset < end + 16  # aligned, in list order, packed
        assert r.pitch == row
        if d.format == dn.FRAME_NV12:  # the Y plane, then the UV plane, tight
            assert r.uv == r.win.offset + row * d.h and r.uv_pitch == row
        end = r.win.offset + staged
    assert toff % 16 == 0 and end <= toff < end + 16
    assert total == toff + len(descs) * C.sizeof(_lib.FrameSrc)
    assert C.sizeof(_lib.FrameSrc) == 64 and _lib.FrameSrc.uv.offset == C.sizeof(_lib.FrameWindow)


def test_layout_of_an_all_device_list_is_the_table_alone():
    descs = [d for d, staged in MIXED if not staged]
    recs, toff, total = _lib.frame_desc_layout(descs, 608, 608, False)
    assert toff == 0 and total == len(descs) * C.sizeof(_lib.FrameSrc)


@pytest.mark.parametrize("bad", [dict(w=0), dict(h=-2), dict(format=3), dict(format=-1), dict(w=7, format=2),
                                 dict(h=5, format=2), dict(pitch=23), dict(pitch=-24), dict(format=2, pitch=7),
                                 dict(format=2, uv_pitch=7), dict(format=2, uv_pitch=-8),
                                 dict(w=715827883)])
def test_layout_refuses_a_bad_descriptor(bad):
    args = dict(w=8, h=6, fmt=dn.FRAME_RGB24)
    args.update({("fmt" if k == "format" else k): v for k, v in bad.items()})
    d = _desc(args.pop("w"), args.pop("h"), args.pop("fmt"), **args)
    assert _lib.frame_desc_layout([_desc(4, 4, dn.FRAME_RGB24), d], 416, 416, False)[2] == 0
    assert _lib.frame_desc_layout([_desc(4, 4, dn.FRAME_RGB24)], 416, 416, False)[2] > 0
    assert _lib.frame_desc_layout([], 416, 416, False)[2] == 0


def test_ctypes_mirror_matches_the_library():
    lib = dn.lib()
    assert lib.y2_abi_sizeof(7) == C.sizeof(dn.FrameDesc) == 40


# ---- the Python descriptor builder ---------------------------------------------------------------------------------
def test_frame_desc_reads_the_pitch_from_the_row_stride():
    wide = np.zeros((10, 20, 3), np.uint8)
    d = dn.frame_desc(wide[:, 3:11], dn.FRAME_BGR24)
    assert (d.w, d.h, d.pitch, d.format, d.on_device) == (8, 10, 60, dn.FRAME_BGR24, 0)
    assert d.data == wide.ctypes.data + 9
    nv12 = np.zeros((18, 32), np.uint8)[:, :8]
    d = dn.frame_desc(nv12, dn.FRAME_NV12)
    assert (d.w, d.h, d.pitch, d.uv) == (8, 12, 32, None)
    y, uv = np.zeros((12, 8), np.uint8), np.zeros((6, 16, 2), np.uint8)[:, :4]
    d = dn.frame_desc((y, uv), dn.FRAME_NV12)
    assert (d.w, d.h, d.pitch, d.uv, d.uv_pitch) == (8, 12, 8, uv.ctypes.data, 32)

    class Dev:  # what a torch or cupy tensor on the GPU exposes
        __cuda_array_interface__ = {"shape": (4, 6, 3), "typestr": "|u1", "data": (0x7f0000000010, False),
                                    "strides": (32, 3, 1), "version": 3}
    d = dn.frame_desc(Dev(), dn.FRAME_RGB24)
    assert (d.data, d.w, d.h, d.pitch, d.on_device) == (0x7f0000000010, 6, 4, 32, 1)


@pytest.mark.parametrize("case", ["planar", "float", "channels4", "odd_nv12", "nv12_rows", "reversed", "uv_shape",
                                  "not_an_array", "format", "overlapping_rows"])
def test_frame_desc_refuses_what_is_not_interleaved_pixel_rows(case):
    a = np.zeros((6, 8, 3), np.uint8)
    obj, fmt = {
        "planar": (np.zeros((3, 6, 8), np.uint8).transpose(1, 2, 0), dn.FRAME_RGB24),
        "float": (a.astype(np.float32), dn.FRAME_RGB24),
        "channels4": (np.zeros((6, 8, 4), np.uint8), dn.FRAME_RGB24),
        "odd_nv12": (np.zeros((9, 5), np.uint8), dn.FRAME_NV12),
        "nv12_rows": (np.zeros((10, 8), np.uint8), dn.FRAME_NV12),
        "reversed": (a[::-1], dn.FRAME_RGB24),
        "uv_shape": ((np.zeros((6, 8), np.uint8), np.zeros((3, 6), np.uint8)), dn.FRAME_NV12),
        "not_an_array": ([[1, 2, 3]], dn.FRAME_RGB24),
        "format": (a, 7),
        "overlapping_rows": (np.lib.stride_tricks.as_strided(a, (6, 8, 3), (12, 3, 1)), dn.FRAME_RGB24),
    }[case]
    with pytest.raises((ValueError, TypeError)):
        dn.frame_desc(obj, fmt)


# ---- refusal without a device plan ---------------------------------------------------------------------------------
DESCS = "[dn.frame_desc(np.zeros((12, 16, 3), np.uint8), dn.FRAME_BGR24), " \
        "dn.frame_desc(np.zeros((6, 8), np.uint8), dn.FRAME_NV12)][:net.batch]"
CALLS = {
    "detect_batch": f"dn.network_detect_frame_descs(net, {DESCS}, .5, .4)",
    "detect_submit": f"dn.network_detect_submit_frame_descs(net, {DESCS}, .5, .4)",
    "classify_batch": f"dn.network_classify_frame_descs(net, {DESCS}, top=3)",
    "classify_submit": f"dn.network_classify_submit_frame_descs(net, {DESCS}, top=3)",
    "streams_batch": f"dn.network_detect_streams_descs(net, [0], {DESCS}, .5, .4)",
    "streams_submit": f"dn.network_detect_submit_streams_descs(net, [0], {DESCS}, .5, .4)",
    "tracked_batch": f"dn.network_detect_streams_tracked_descs(net, [0], {DESCS}, .5, .4)",
    "tracked_submit": f"dn.network_detect_submit_streams_tracked_descs(net, [0], {DESCS}, .5, .4)",
    "staging": f"dn.network_pipeline_staging_frame_descs(net, 0, {DESCS})",
}


@pytest.mark.parametrize("call", sorted(CALLS))
def test_frame_descs_without_a_device_plan_exit_through_error(tmp_path, call):
    cfg = tmp_path / "net.cfg"
    cfg.write_text(synth.exact_classifier_cfg(batch=1))
    code = ("import sys, numpy as np; sys.path.insert(0, %r)\n"
            "from sr_object_detection_b200 import darknet as dn\n"
            "dn.set_gpu_index(-1)\n"
            "net = dn.parse_network_cfg(%r)\n"
            "%s\n"
            "print('COMPUTED')\n" % (str(ROOT), str(cfg), CALLS[call]))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert r.returncode != 0 and "COMPUTED" not in r.stdout
    assert "no device plan" in r.stderr, r.stderr[-2000:]
