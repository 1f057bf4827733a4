"""CPU tests of the frame-list entries (frames of their own sizes in one batch): the layout helper that packs the
frames and their window records, and the refusal of every frame-list entry on a network without a device plan."""
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from sr_object_detection_b200 import _lib, synth
from tests.test_classify_host import SOURCES, TARGETS, _geometry

ROOT = Path(__file__).resolve().parents[1]
LIST = SOURCES + [(1, 1), (1, 300), (300, 1), (416, 416), (3, 2)]


def _same_f32(a, b):
    return np.array([a], np.float32).view(np.uint32)[0] == np.array([b], np.float32).view(np.uint32)[0] or \
        (np.isnan(a) and np.isnan(b))


@pytest.mark.parametrize("w,h", TARGETS)
@pytest.mark.parametrize("letterbox", [False, True])
def test_layout_packs_the_frames_and_the_table(w, h, letterbox):
    win, toff, total = _lib.frame_list_layout(LIST, w, h, letterbox)
    assert len(win) == len(LIST)
    end = 0
    for f, (sw, sh) in zip(win, LIST):
        assert f.offset % 16 == 0 and f.offset >= end, (f.offset, end)  # aligned, in list order, no overlap
        assert f.offset - end < 16  # and packed: only the alignment gap between frames
        end = f.offset + sw * sh * 3
        assert (f.src_w, f.src_h) == (sw, sh)
    assert toff % 16 == 0 and end <= toff < end + 16
    assert total == toff + len(LIST) * _lib.C.sizeof(_lib.FrameWindow)


@pytest.mark.parametrize("w,h", TARGETS)
@pytest.mark.parametrize("letterbox", [False, True])
def test_layout_windows_and_scales(w, h, letterbox):
    win, _, _ = _lib.frame_list_layout(LIST, w, h, letterbox)
    with np.errstate(divide="ignore", invalid="ignore"):
        for f, (sw, sh) in zip(win, LIST):
            if letterbox:
                nw, nh, dx, dy = _geometry(sw, sh, w, h)
            else:
                nw, nh, dx, dy = w, h, 0, 0
            assert (f.new_w, f.new_h, f.dx, f.dy) == (nw, nh, dx, dy), (sw, sh, w, h)
            # resize_image's scales (image.c:1954-1955) in float32: (float)(im.w - 1) / (w - 1)
            assert _same_f32(f.w_scale, np.float32(sw - 1) / np.float32(nw - 1)), (sw, nw, f.w_scale)
            assert _same_f32(f.h_scale, np.float32(sh - 1) / np.float32(nh - 1)), (sh, nh, f.h_scale)


def test_layout_of_one_frame_and_of_bad_lists():
    win, toff, total = _lib.frame_list_layout([(5, 3)], 8, 8, False)
    assert win[0].offset == 0 and toff == 48 and total == 48 + _lib.C.sizeof(_lib.FrameWindow)
    assert _lib.frame_list_layout([], 8, 8, False)[2] == 0
    assert _lib.frame_list_layout([(5, 3), (0, 4)], 8, 8, False)[2] == 0
    assert _lib.frame_list_layout([(5, -1)], 8, 8, True)[2] == 0
    assert _lib.frame_list_layout([(5, 3)], 0, 8, True)[2] == 0


FRAMES = "[np.zeros((12, 16, 3), np.uint8), np.zeros((5, 7, 3), np.uint8)][:net.batch]"
CALLS = {
    "detect_batch": f"dn.network_detect_frame_list(net, {FRAMES}, .5, .4)",
    "detect_submit": f"dn.network_detect_submit_frame_list(net, {FRAMES}, .5, .4)",
    "classify_batch": f"dn.network_classify_batch(net, frame_list={FRAMES}, top=3)",
    "classify_submit": f"dn.network_classify_submit(net, frame_list={FRAMES}, top=3)",
    "staging": "dn.network_pipeline_staging_frame_list(net, 0, [(16, 12)])",
}


@pytest.mark.parametrize("call", sorted(CALLS))
def test_frame_list_without_a_device_plan_exits_through_error(tmp_path, call):
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
