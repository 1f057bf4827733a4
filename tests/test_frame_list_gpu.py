"""Frame lists (frames of their own sizes in one batch; y2_frames_u8_to_f32, network_*_frame_list) against the host
chains they replace, per frame: byte/255. then resize_image (detection) or letterbox_image (classification), then the
uniform entries.  Every comparison is bit for bit."""
import ctypes as C
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from sr_object_detection_b200 import _lib, darknet as dn, synth
from tests.test_classify_gpu import NETS, _host_letterbox, _host_topk, _planar, _same

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
_fp = C.POINTER(C.c_float)


def _host_resize(u8, w, h):
    lib = dn.lib()
    im = _planar(u8)
    out = lib.resize_image(dn.Image(im.shape[1], im.shape[2], 3, im.ctypes.data_as(_fp)), w, h)
    got = np.ctypeslib.as_array(out.data, shape=(3, h, w)).copy()
    lib.free_image(out)
    return got


def _frames(sizes, seed):
    rng = np.random.default_rng(seed)
    return [rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8) for w, h in sizes]


def _sized(frames, w, h, letterbox, batch):
    """the host chain's network input for a list, the canvas behind it .5f"""
    x = np.full((batch, 3, h, w), np.float32(.5), np.float32)
    for i, f in enumerate(frames):
        x[i] = _host_letterbox(f, w, h) if letterbox else _host_resize(f, w, h)
    return x


# ---- kernel -----------------------------------------------------------------------------------------------------
MIXED = [(1920, 1080), (640, 480), (37, 53), (1, 1), (1, 9), (9, 1), (2, 64), (500, 375), (375, 500), (64, 1)]


@pytest.mark.parametrize("letterbox,side", [(False, 416), (True, 448), (False, 64), (True, 32)])
def test_kernel_on_a_mixed_list_equals_the_host_chain(letterbox, side):
    sizes = MIXED + [(side, side)]
    if letterbox:  # a letterbox window 1 pixel high has no defined result
        sizes = [(w, h) for w, h in sizes if _window_h(w, h, side) != 1]
    frames = _frames(sizes, seed=side + letterbox)
    win, toff, total = _lib.frame_list_layout(sizes, side, side, letterbox)
    packed = np.zeros(total, np.uint8)
    for f, r in zip(frames, win):
        packed[r.offset:r.offset + f.nbytes] = f.reshape(-1)
    packed[toff:] = np.frombuffer((_lib.FrameWindow * len(win))(*win), np.uint8)
    batch = len(sizes) + 3
    d_packed = torch.from_numpy(packed).cuda()
    d_dst = torch.full((batch, 3, side, side), -7.0, dtype=torch.float32, device="cuda")  # sentinel
    lib = _lib.load()
    _lib.check(lib.y2_frames_u8_to_f32(d_packed.data_ptr(), d_packed.data_ptr() + toff, len(sizes), d_dst.data_ptr(),
                                       batch, side, side, None), "frames_u8_to_f32")
    torch.cuda.synchronize()
    got = d_dst.cpu().numpy()
    want = _sized(frames, side, side, letterbox, batch)
    for i, (w, h) in enumerate(sizes):
        assert np.array_equal(got[i].view(np.uint32), want[i].view(np.uint32)), (w, h, side, letterbox)
    assert np.all(got[len(sizes):] == np.float32(.5))


def _window_h(w, h, side):
    g = [C.c_int() for _ in range(4)]
    lib = _lib.load()
    lib.y2_letterbox_geometry.restype = None
    lib.y2_letterbox_geometry.argtypes = [C.c_int] * 4 + [C.POINTER(C.c_int)] * 4
    lib.y2_letterbox_geometry(w, h, side, side, *[C.byref(v) for v in g])
    return g[1].value


# ---- detection ----------------------------------------------------------------------------------------------------
def _detector(tmp_path, name, batch):
    text = synth.CFGS[name](batch=batch, w=416, h=416)
    (tmp_path / f"{name}.cfg").write_text(text)
    synth.write_weights(tmp_path / f"{name}.weights", text, seed=1234)
    dn.set_gpu_index(0)
    net = dn.parse_network_cfg(tmp_path / f"{name}.cfg")
    dn.load_weights(net, tmp_path / f"{name}.weights")
    return net


THRESH, NMS, MAX_DET = 0.02, 0.4, 256
VOC_LIKE = [(500, 375), (375, 500), (416, 416), (500, 333), (1920, 1080), (353, 500)]


def _host_detect(net, frames):
    want, _ = dn.network_detect_batch(net, _sized(frames, net.w, net.h, False, net.batch), THRESH, NMS, MAX_DET)
    return want[:len(frames)]


def _same_dets(got, want, what):
    assert len(got) == len(want), what
    for b, (g, w) in enumerate(zip(got, want)):
        assert g.tobytes() == w.tobytes(), f"{what}: image {b}"


@pytest.mark.parametrize("name", ["tiny-yolo-voc", "yolo-voc"])
def test_detect_frame_list_equals_host_resize_then_detect(tmp_path, name):
    net = _detector(tmp_path, name, 4)
    try:
        for sizes, seed in ((VOC_LIKE[:4], 1), (VOC_LIKE[4:], 2), (VOC_LIKE[1:2], 3)):  # n == batch and n < batch
            frames = _frames(sizes, seed)
            want = _host_detect(net, frames)
            assert any(len(w) for w in want), "test needs at least one detection"
            got, counts = dn.network_detect_frame_list(net, frames, THRESH, NMS, MAX_DET)
            assert len(counts) == len(frames)
            _same_dets(got, want, f"{name} {sizes}")
        # a frame at the network size equals the uint8 first-layer path
        frames = _frames([(416, 416)] * 4, seed=4)
        u8 = np.ascontiguousarray(np.stack(frames))
        dets = (dn.Detection * (4 * MAX_DET))()
        counts = (C.c_int * 4)()
        dn.lib().network_detect_batch_u8(net, dn._as_u8(u8), THRESH, NMS, dets, counts, MAX_DET)
        want = [np.ctypeslib.as_array(dets)[b * MAX_DET:b * MAX_DET + min(counts[b], MAX_DET)].copy() for b in range(4)]
        _same_dets(dn.network_detect_frame_list(net, frames[:2], THRESH, NMS, MAX_DET)[0], want[:2], "net size")
    finally:
        dn.free_network(net)


# ---- classification -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["darknet19_448", "resnet50", "exact-tree"])
def test_classify_frame_list_equals_the_host_chain(tmp_path, name, monkeypatch):
    monkeypatch.chdir(tmp_path)  # the exact tree classifier reads t.tree relative to the cwd
    net = NETS[name](tmp_path)
    top = 5
    try:
        for sizes, seed in (([(500, 375), (net.w, net.h)], 1), ([(37, 1920)], 2), ([(1920, 1080), (3, 2)], 3)):
            frames = _frames(sizes, seed)
            out = dn.network_predict(net, _sized(frames, net.w, net.h, True, net.batch))
            want = _host_topk(out[:len(frames)], top, hierarchy=net.hierarchy if net.hierarchy else None)
            _same(dn.network_classify_batch(net, frame_list=frames, top=top), want)
    finally:
        dn.free_network(net)


# ---- pipeline -----------------------------------------------------------------------------------------------------
def _stage(net, frames):
    """frames written straight into the next slot's pinned staging buffer"""
    views = dn.network_pipeline_staging_frame_list(net, dn.lib().network_pipeline_next_slot(net),
                                                   [(f.shape[1], f.shape[0]) for f in frames])
    for v, f in zip(views, frames):
        v[...] = f
    return views


def _resident(net, x):
    dev = dn.lib().network_pipeline_input_device(net, dn.lib().network_pipeline_next_slot(net))
    _lib.check(_lib.load().y2_memcpy_h2d(dev, x.ctypes.data, x.nbytes, None), "h2d")
    _lib.check(_lib.load().y2_stream_sync(None))


def test_detect_pipeline_interleaves_frame_lists_with_every_kind(tmp_path):
    net = _detector(tmp_path, "tiny-yolo-voc", 3)
    lib, B = dn.lib(), net.batch
    try:
        small, large = _frames([(500, 375)], 5), _frames([(1920, 1080), (640, 480), (375, 500)], 6)
        x = synth.images(B, 3, net.h, net.w, seed=7)
        u8 = np.ascontiguousarray(np.stack(_frames([(416, 416)] * B, 8)))
        frames = np.ascontiguousarray(np.stack(_frames([(333, 517)] * B, 9)))
        res = synth.images(B, 3, net.h, net.w, seed=10)
        seq = [("list", small), ("f32", x), ("staged", large), ("u8", u8), ("list", large), ("frames", frames),
               ("staged", small), ("resident", res), ("list", small)]

        def host(kind, a):
            if kind in ("list", "staged", "frames"):
                return _host_detect(net, list(a))
            if kind == "u8":
                a = np.ascontiguousarray(np.stack([_planar(f) for f in a]))
            return dn.network_detect_batch(net, a, THRESH, NMS, MAX_DET)[0]

        want = [host(k, a) for k, a in seq]  # the synchronous calls before anything is in flight

        def submit(kind, a):
            if kind in ("list", "staged"):
                return dn.network_detect_submit_frame_list(net, _stage(net, a) if kind == "staged" else a, THRESH,
                                                           NMS, MAX_DET)
            if kind == "f32":
                return lib.network_detect_submit(net, dn._as_fp(a), THRESH, NMS, MAX_DET)
            if kind == "u8":
                return lib.network_detect_submit_u8(net, dn._as_u8(a), THRESH, NMS, MAX_DET)
            if kind == "frames":
                return lib.network_detect_submit_frames(net, dn._as_u8(a), a.shape[2], a.shape[1], THRESH, NMS,
                                                        MAX_DET)
            _resident(net, a)
            return lib.network_detect_submit_resident(net, THRESH, NMS, MAX_DET)

        def check(i):
            kind, a = seq[i]
            n = len(a) if kind in ("list", "staged") else B
            got, counts = dn.network_detect_wait_n(net, n, MAX_DET)
            assert len(counts) == n
            _same_dets(got, want[i], f"{i} {kind}")

        submit(*seq[0])
        for i in range(1, len(seq)):
            submit(*seq[i])  # two batches in flight
            check(i - 1)
        check(len(seq) - 1)
    finally:
        dn.free_network(net)


def test_classify_pipeline_interleaves_frame_lists_with_every_kind(tmp_path):
    net = NETS["darknet19_448"](tmp_path)
    lib, B, top = dn.lib(), net.batch, 5
    try:
        small, large = _frames([(500, 375)], 5), _frames([(1920, 1080), (353, 500)], 6)
        x = synth.images(B, 3, net.h, net.w, seed=7)
        u8 = np.ascontiguousarray(np.stack(_frames([(net.w, net.h)] * B, 8)))
        frames = np.ascontiguousarray(np.stack(_frames([(640, 480)] * B, 9)))
        res = synth.images(B, 3, net.h, net.w, seed=10)
        seq = [("list", small), ("f32", x), ("staged", large), ("u8", u8), ("frames", frames), ("staged", small),
               ("resident", res), ("list", large)]

        def host(kind, a):
            if kind in ("list", "staged"):
                out = dn.network_predict(net, _sized(a, net.w, net.h, True, B))
                return _host_topk(out[:len(a)], top)
            if kind == "u8":
                a = np.ascontiguousarray(np.stack([_planar(f) for f in a]))
            elif kind == "frames":
                a = _sized(list(a), net.w, net.h, True, B)
            return dn.network_classify_batch(net, images=a, top=top)

        want = [host(k, a) for k, a in seq]

        def submit(kind, a):
            if kind in ("list", "staged"):
                return dn.network_classify_submit(net, frame_list=_stage(net, a) if kind == "staged" else a, top=top)
            if kind == "f32":
                return dn.network_classify_submit(net, images=a, top=top)
            if kind == "u8":
                return dn.network_classify_submit(net, u8=a, top=top)
            if kind == "frames":
                return dn.network_classify_submit(net, frames=a, top=top)
            _resident(net, a)
            return dn.network_classify_submit(net, top=top)

        def n_of(kind, a):
            return len(a) if kind in ("list", "staged") else B

        submit(*seq[0])
        for i in range(1, len(seq)):
            submit(*seq[i])
            _same(dn.network_classify_wait(net, top=top, n=n_of(*seq[i - 1])), want[i - 1])
        _same(dn.network_classify_wait(net, top=top, n=n_of(*seq[-1])), want[-1])
    finally:
        dn.free_network(net)


# ---- refusals -------------------------------------------------------------------------------------------------------
REFUSE = """
import sys, ctypes as C, numpy as np
sys.path.insert(0, {root!r})
from sr_object_detection_b200 import darknet as dn
dn.set_gpu_index(0)
net = dn.parse_network_cfg({cfg!r})
dn.load_weights(net, {weights!r})
f = np.zeros((12, 16, 3), np.uint8)
lib = dn.lib()
{call}
print("RETURNED")
"""


@pytest.mark.parametrize("case", ["n0", "n_over_batch", "null_frame", "zero_size", "negative_size", "one_channel",
                                  "wait_on_detect", "wait_on_classify", "staging_n0"])
def test_frame_list_refusals_exit_through_error(tmp_path, case):
    if case in ("wait_on_detect", "wait_on_classify"):
        cfg_text = synth.exact_detector_cfg(batch=2) if case == "wait_on_detect" else \
            synth.exact_classifier_cfg(batch=2)
    elif case == "one_channel":
        cfg_text = synth.exact_classifier_cfg(batch=2).replace("channels=3", "channels=1")
        assert "channels=1" in cfg_text
    else:
        cfg_text = synth.exact_classifier_cfg(batch=2)
    (tmp_path / "n.cfg").write_text(cfg_text)
    synth.write_weights(tmp_path / "n.weights", cfg_text, seed=3)
    ptrs = "(C.POINTER(C.c_ubyte) * 2)(dn._as_u8(f), {})"
    sizes = "(C.c_int * 2)(16, 16), (C.c_int * 2)({}, 12)"
    call, msg = {
        "n0": ("lib.network_classify_submit_frame_list(net, 0, %s, %s, 3)" % (ptrs.format("dn._as_u8(f)"),
                                                                             sizes.format(16)), "1 .. batch frames"),
        "n_over_batch": ("dn.network_classify_batch(net, frame_list=[f, f, f], top=3)", "1 .. batch frames"),
        "null_frame": ("lib.network_classify_submit_frame_list(net, 2, %s, %s, 3)" % (ptrs.format("None"),
                                                                                     sizes.format(16)),
                       "NULL frame pointer"),
        "zero_size": ("lib.network_classify_submit_frame_list(net, 2, %s, %s, 3)" % (ptrs.format("dn._as_u8(f)"),
                                                                                    sizes.format(0)),
                      "frame size of 0 or less"),
        "negative_size": ("lib.network_classify_batch_frame_list(net, 2, %s, %s, 3, (dn.ClassHit * 6)())"
                          % (ptrs.format("dn._as_u8(f)"), sizes.format(-4)), "frame size of 0 or less"),
        "one_channel": ("dn.network_classify_batch(net, frame_list=[f], top=3)", "3 input channels"),
        "wait_on_detect": ("dn.network_detect_submit_frame_list(net, [f], .5, .4)\n"
                           "dn.network_classify_wait(net, top=3, n=1)", "is a detection batch"),
        "wait_on_classify": ("dn.network_classify_submit(net, frame_list=[f], top=3)\n"
                             "dn.network_detect_wait_n(net, 1)", "is a classify batch"),
        "staging_n0": ("dn.network_pipeline_staging_frame_list(net, 0, [])", "1 .. batch frames"),
    }[case]
    code = REFUSE.format(root=str(ROOT), cfg=str(tmp_path / "n.cfg"), weights=str(tmp_path / "n.weights"), call=call)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert r.returncode != 0 and "RETURNED" not in r.stdout, r.stdout
    assert msg in r.stderr, r.stderr[-2000:]
