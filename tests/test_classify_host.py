"""CPU tests of the batched classification extension (network_classify_*): the struct mirror, the letterbox
geometry shared by letterbox_image and the device letterbox, and the refusal of the classify entries on a network
without a device plan."""
import ctypes as C
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from sr_object_detection_b200 import darknet as dn, synth

ROOT = Path(__file__).resolve().parents[1]
SOURCES = [(640, 480), (300, 200), (448, 448), (1920, 1080), (37, 53), (1, 9), (25, 16), (1, 100), (9, 1),
           (2, 64), (1, 1), (500, 375)]
TARGETS = [(448, 448), (256, 256), (64, 32), (32, 32), (16, 12), (1, 1)]


def test_class_hit_mirror_matches_the_library():
    lib = dn.lib()
    assert lib.y2_abi_sizeof(5) == C.sizeof(dn.ClassHit) == 8


def _geometry(sw, sh, w, h):
    lib = dn.lib()
    lib.y2_letterbox_geometry.restype = None
    lib.y2_letterbox_geometry.argtypes = [C.c_int] * 4 + [C.POINTER(C.c_int)] * 4
    out = [C.c_int() for _ in range(4)]
    lib.y2_letterbox_geometry(sw, sh, w, h, *[C.byref(v) for v in out])
    return tuple(v.value for v in out)


def _rule(sw, sh, w, h):
    """image.c:1624-1644 restated: float comparison of the two scales, integer divisions"""
    if np.float32(w) / np.float32(sw) < np.float32(h) / np.float32(sh):
        nw, nh = w, (sh * w) // sw
    else:
        nw, nh = (sw * h) // sh, h
    return nw, nh, (w - nw) // 2, (h - nh) // 2


@pytest.mark.parametrize("w,h", TARGETS)
def test_letterbox_geometry_is_what_letterbox_image_draws(w, h):
    """The window the helper reports is exactly the part of letterbox_image's canvas that is not the .5 grey (a
    source of zeros resizes to zeros), over wider, taller, equal and 1-pixel sources."""
    lib = dn.lib()
    for sw, sh in SOURCES:
        nw, nh, dx, dy = _geometry(sw, sh, w, h)
        assert (nw, nh, dx, dy) == _rule(sw, sh, w, h), (sw, sh, w, h)
        if nh == 1 and nw > 0:
            continue  # resize_image has no defined result for a 1-pixel-high target
        im = np.zeros((3, sh, sw), np.float32)
        out = lib.letterbox_image(dn.Image(sh, sw, 3, im.ctypes.data_as(C.POINTER(C.c_float))), w, h)
        got = np.ctypeslib.as_array(out.data, shape=(3, h, w)).copy()
        lib.free_image(out)
        inside = np.zeros((h, w), bool)
        inside[dy:dy + nh, dx:dx + nw] = True
        assert np.all(got[:, ~inside] == np.float32(.5)), (sw, sh, w, h)
        assert np.all(got[:, inside] == 0), (sw, sh, w, h)


CALLS = {
    "batch_frames": "dn.network_classify_batch(net, frames=np.zeros((1, 12, 16, 3), np.uint8), top=3)",
    "batch": "dn.network_classify_batch(net, images=np.zeros((1, 3, 12, 16), np.float32), top=3)",
    "device": "dn.network_classify_batch(net, top=3)",
    "submit_frames": "dn.network_classify_submit(net, frames=np.zeros((1, 12, 16, 3), np.uint8), top=3)",
    "submit_resident": "dn.network_classify_submit(net, top=3)",
}


@pytest.mark.parametrize("call", sorted(CALLS))
def test_classify_without_a_device_plan_exits_through_error(tmp_path, call):
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
