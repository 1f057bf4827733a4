"""Video streams (network_streams_open, network_detect_*_streams): each frame detected on the 3-frame mean of its
stream, against the Detector's own flow (yolo_v2_class.cpp:206-216) restated on the host: the plain frame-list
path's region outputs, a numpy ring per stream, mean_arrays in float32, then the host get_region_boxes, do_nms_sort
and the max_index pick.  Every comparison is bit for bit."""
import ctypes as C
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from sr_object_detection_b200 import _lib, darknet as dn, synth
from tests.test_frame_list_gpu import _frames, _stage

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
_fp = C.POINTER(C.c_float)
F0, F3 = np.float32(0), np.float32(3)


def _mean3(a, b, c):
    """mean_arrays (utils.c:420-433) of three float32 rows: ((0 + a) + b) + c) / 3"""
    return (((F0 + a) + b) + c) / F3


def _same_bits(got, want, what):
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan), what
    assert np.array_equal(got[~nan].view(np.uint32), want[~nan].view(np.uint32)), what


# ---- kernels ------------------------------------------------------------------------------------------------------
def _special_rows(rng, rows, outputs):
    x = rng.standard_normal((rows, outputs)).astype(np.float32)
    specials = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1e-40, -1e-45, 3e38, -3e38, 1.17549435e-38],
                        np.float32)
    pick = rng.random((rows, outputs)) < .3
    x[pick] = rng.choice(specials, int(pick.sum()))
    k = min(len(specials), outputs)
    for r in range(rows):  # the first columns: every special, rotated row by row (narrow rows see them all too)
        x[r, :k] = np.roll(specials, r)[:k]
    return x


@pytest.mark.parametrize("outputs", [1, 7, 1024, 1029, 4100, 21125])
def test_mean_and_commit_kernels_equal_numpy(outputs):
    rng = np.random.default_rng(outputs)
    max_streams = 4
    # stream 2 five times in one list, stream 0 with a full ring, stream 1 fresh, stream 3 with one frame before
    ids = [2, 0, 2, 2, 1, 2, 3, 2, 0]
    fi, seen = [1, 0, 0, 1], [3, 0, 0, 1]
    plan, _, _ = _lib.stream_plan(ids, max_streams, fi, seen)
    n = len(ids)
    out = _special_rows(rng, n + 2, outputs)
    ring = _special_rows(rng, 3 * max_streams, outputs)
    table = np.frombuffer((_lib.StreamSrc * n)(*plan), np.int32).reshape(n, 4)
    d_out, d_ring = torch.from_numpy(out).cuda(), torch.from_numpy(ring).cuda()
    d_table = torch.from_numpy(table.copy()).cuda()
    d_mean = torch.full((n, outputs), -7.0, dtype=torch.float32, device="cuda")
    lib = _lib.load()
    _lib.check(lib.y2_stream_mean(d_out.data_ptr(), d_ring.data_ptr(), d_table.data_ptr(), n, outputs,
                                  d_mean.data_ptr(), None), "stream_mean")
    _lib.check(lib.y2_stream_commit(d_out.data_ptr(), d_ring.data_ptr(), d_table.data_ptr(), n, outputs, None),
               "stream_commit")
    torch.cuda.synchronize()

    def row(code):
        if code >= 0:
            return out[code]
        return np.zeros(outputs, np.float32) if code == -1 else ring[-2 - code]

    want_mean = np.stack([_mean3(*[row(c) for c in r.src]) for r in plan])
    _same_bits(d_mean.cpu().numpy(), want_mean, f"mean, outputs {outputs}")
    want_ring = ring.copy()
    for i, r in enumerate(plan):
        if r.commit >= 0:
            want_ring[r.commit] = out[i]
    assert [r.commit >= 0 for r in plan] == [False, True, False, True, True, True, True, True, True]  # stream 2: last 3
    _same_bits(d_ring.cpu().numpy(), want_ring, f"ring, outputs {outputs}")


# ---- the host reference ---------------------------------------------------------------------------------------------
class HostStreams:
    """The Detector's state per stream (zero ring of 3 region outputs, frame_index) and its decode of the mean."""

    def __init__(self, net):
        self.net = net
        self.outputs = dn.region_layer(net).outputs
        self.rings = {}

    def frame(self, s, region_out, thresh, nms):
        ring, idx = self.rings.get(s, ([np.zeros(self.outputs, np.float32) for _ in range(3)], 0))
        ring[idx] = region_out.copy()
        self.rings[s] = (ring, (idx + 1) % 3)
        return _host_decode(self.net, np.ascontiguousarray(_mean3(*ring)), thresh, nms)


def _host_decode(net, pred, thresh, nms):
    """get_region_boxes on pred (a Layer copy whose output points at it), do_nms_sort when nms, max_index pick"""
    l = dn.Layer.from_buffer_copy(dn.region_layer(net))
    l.output = pred.ctypes.data_as(_fp)
    total, classes = l.w * l.h * l.n, l.classes
    probs = np.zeros((total, classes), np.float32)
    boxes = np.zeros((total, 4), np.float32)
    rows = (_fp * total)(*[C.cast(probs.ctypes.data + j * classes * 4, _fp) for j in range(total)])
    dn.lib().get_region_boxes(l, 1, 1, thresh, rows, boxes.ctypes.data_as(C.POINTER(dn.Box)), 0, None)
    if nms:
        dn.do_nms_sort(boxes, probs, nms)
    obj = np.argmax(probs, axis=1)  # max_index: the first of equal maxima
    prob = probs[np.arange(total), obj]
    keep = np.nonzero(prob > thresh)[0]
    out = np.zeros(len(keep), np.dtype([("x", "<f4"), ("y", "<f4"), ("w", "<f4"), ("h", "<f4"), ("prob", "<f4"),
                                        ("obj_id", "<i4"), ("box_index", "<i4")]))
    for f, k in zip("xywh", range(4)):
        out[f] = boxes[keep, k]
    out["prob"], out["obj_id"], out["box_index"] = prob[keep], obj[keep], keep
    return out


def _same_dets(got, want, what):
    assert len(got) == len(want), what
    for b, (g, w) in enumerate(zip(got, want)):
        assert g.tobytes() == w.tobytes(), f"{what}: image {b}"


def _region_outputs(net, frames, thresh, nms, max_det):
    """the plain frame-list path on the same frames: its detections and its region outputs"""
    dets = dn.network_detect_frame_list(net, frames, thresh, nms, max_det)
    return dets, dn.get_network_output_layer(net, net.n - 1)[:len(frames)]


def _check_sequence(net, host, batches, thresh, nms, max_det, tag):
    """batches: (ids, frames) or a callable applied between batches; every streams batch against the host reference"""
    found = 0
    for k, item in enumerate(batches):
        if callable(item):
            item()
            continue
        ids, frames = item
        _, region = _region_outputs(net, frames, thresh, nms, max_det)
        want = [host.frame(s, region[i], thresh, nms) for i, s in enumerate(ids)]
        got, counts = dn.network_detect_streams(net, ids, frames, thresh, nms, max_det)
        assert counts == [len(w) for w in want], f"{tag} batch {k}"
        _same_dets(got, want, f"{tag} batch {k}")
        found += sum(counts)
    assert found > 0, "test needs detections"


def _detector(tmp_path, name, batch, side=416, head_gain=1.0):
    text = synth.CFGS[name](batch=batch, w=side, h=side)
    (tmp_path / f"{name}.cfg").write_text(text)
    synth.write_weights(tmp_path / f"{name}.weights", text, seed=1234, head_gain=head_gain)
    dn.set_gpu_index(0)
    net = dn.parse_network_cfg(tmp_path / f"{name}.cfg")
    dn.load_weights(net, tmp_path / f"{name}.weights")
    return net


THRESH, NMS = 0.02, 0.4
SIZES = [(500, 375), (375, 500), (416, 416), (640, 480), (353, 500), (1280, 720)]  # stream s: frames of SIZES[s]
LISTS = [[0, 1, 2, 0, 3, 0, 4, 5], [1, 1, 2, 5, 5, 5, 0, 3], [4, 2, 0, 0, 1, 3], [5, 4, 3, 2, 1, 0, 0, 0]]


def _stream_frames(ids, seed):
    return _frames([SIZES[s] for s in ids], seed)


# ---- networks -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["tiny-yolo-voc", "yolo-voc"])
def test_streams_equal_the_detector_flow(tmp_path, name):
    net = _detector(tmp_path, name, 8)
    try:
        dn.network_streams_open(net, 6)
        batches = [(ids, _stream_frames(ids, 10 + k)) for k, ids in enumerate(LISTS)]
        _check_sequence(net, HostStreams(net), batches, THRESH, NMS, 1024, name)
    finally:
        dn.free_network(net)


def test_streams_on_yolo_608_with_1080p_frames(tmp_path):
    net = _detector(tmp_path, "yolo", 4, side=608, head_gain=24.0)  # 80 classes: detections at the Detector's .24
    try:
        dn.network_streams_open(net, 2)
        batches = [(ids, _frames([(1920, 1080)] * len(ids), 20 + k))
                   for k, ids in enumerate([[0, 1, 0], [1, 1, 0, 1], [0, 0]])]
        _check_sequence(net, HostStreams(net), batches, 0.24, NMS, 2048, "yolo 608")
    finally:
        dn.free_network(net)


# ---- the reference's own class --------------------------------------------------------------------------------------
def _bbox_line(i, dets, w, h):
    """the scenario's dump of Detector::detect's bbox_t list (yolo_v2_class.cpp:224-236, detector_scenario.cpp)"""
    line = f"mean {i} {len(dets)}"
    for d in dets:
        bx, by, bw, bh = (float(np.float32(d[f])) for f in "xywh")
        x = int(max(0.0, (bx - bw / 2.0) * w))
        y = int(max(0.0, (by - bh / 2.0) * h))
        line += " %d %d %d %d %.9g %d 0" % (x, y, int(np.float32(bw) * np.float32(w)),
                                            int(np.float32(bh) * np.float32(h)), float(d["prob"]), int(d["obj_id"]))
    return line


def test_streams_reproduce_the_reference_detector_mean_lines(tmp_path):
    g = json.loads((ROOT / "tests" / "golden" / "detector_ref.json").read_text())
    want = [l for l in g["lines"] if l.startswith("mean ")]
    assert len(want) == g["n"] == 6
    w, h, B = g["w"], g["h"], 4
    cfg = g["cfg"].replace("batch=1", f"batch={B}")
    assert f"batch={B}" in cfg
    (tmp_path / "net.cfg").write_text(cfg)
    synth.write_exact_weights(tmp_path / "net.weights", g["cfg"])
    frames = synth.exact_frames(g["n"], h, w)
    others = synth.exact_frames(8, h, w, seed=31)
    dn.set_gpu_index(0)
    net = dn.parse_network_cfg(tmp_path / "net.cfg")
    dn.load_weights(net, tmp_path / "net.weights")
    lib = _lib.load()

    def run(lists):
        """lists of (stream, frame) through the resident entry; the lines of stream 0's frames in order"""
        lines = []
        for items in lists:
            x = np.zeros((B, 3, h, w), np.float32)
            for i, (_, f) in enumerate(items):
                x[i] = f
            dev = dn.lib().network_pipeline_input_device(net, dn.lib().network_pipeline_next_slot(net))
            _lib.check(lib.y2_memcpy_h2d(dev, x.ctypes.data, x.nbytes, None), "h2d")
            _lib.check(lib.y2_stream_sync(None))
            dn.network_detect_submit_streams_resident(net, [s for s, _ in items], g["thresh"], g["nms"], 1024)
            got, _ = dn.network_detect_wait_n(net, len(items), 1024)
            lines += [d for (s, _), d in zip(items, got) if s == 0]
        return [_bbox_line(i, d, w, h) for i, d in enumerate(lines)]

    try:
        dn.network_streams_open(net, 1)
        assert run([[(0, frames[i])] for i in range(3)] + [[(0, frames[3]), (0, frames[4]), (0, frames[5])]]) == want
        dn.network_streams_open(net, 3)
        spread = [[(1, others[0]), (0, frames[0]), (2, others[1]), (0, frames[1])],
                  [(0, frames[2]), (1, others[2]), (0, frames[3]), (0, frames[4])],
                  [(2, others[3]), (2, others[4]), (1, others[5]), (0, frames[5])]]
        assert run(spread) == want
    finally:
        dn.free_network(net)


# ---- pipeline -----------------------------------------------------------------------------------------------------
def test_streams_interleave_with_plain_frame_lists_in_the_pipeline(tmp_path):
    net = _detector(tmp_path, "tiny-yolo-voc", 4)
    max_det = 1024
    try:
        plain = [_frames([(500, 375), (1920, 1080)], 40), _frames([(375, 500)] * 4, 41), _frames([(640, 480)], 42)]
        streams = [([0, 1, 0], _stream_frames([0, 1, 0], 43)), ([2, 0, 0, 1], _stream_frames([2, 0, 0, 1], 44)),
                   ([1], _stream_frames([1], 45)), ([0, 2, 2], _stream_frames([0, 2, 2], 46))]
        want_plain = [dn.network_detect_frame_list(net, f, THRESH, NMS, max_det)[0] for f in plain]
        dn.network_streams_open(net, 3)
        want_streams = [dn.network_detect_streams(net, ids, f, THRESH, NMS, max_det)[0] for ids, f in streams]
        assert any(len(d) for w in want_streams for d in w)
        dn.network_streams_open(net, 3)  # every stream over again
        seq = [("s", 0, False), ("p", 0, True), ("s", 1, True), ("p", 1, False), ("s", 2, False), ("p", 2, True),
               ("s", 3, False)]

        def submit(kind, k, staged):
            if kind == "p":
                f = _stage(net, plain[k]) if staged else plain[k]
                return dn.network_detect_submit_frame_list(net, f, THRESH, NMS, max_det)
            ids, f = streams[k]
            return dn.network_detect_submit_streams(net, ids, _stage(net, f) if staged else f, THRESH, NMS, max_det)

        def check(kind, k, _staged):
            n = len(plain[k]) if kind == "p" else len(streams[k][0])
            got, _ = dn.network_detect_wait_n(net, n, max_det)
            _same_dets(got, (want_plain if kind == "p" else want_streams)[k], f"{kind}{k}")

        submit(*seq[0])
        for i in range(1, len(seq)):
            submit(*seq[i])  # two batches in flight
            check(*seq[i - 1])
        check(*seq[-1])
    finally:
        dn.free_network(net)


def test_reset_between_submissions_affects_only_the_later_batch(tmp_path):
    net = _detector(tmp_path, "tiny-yolo-voc", 4)
    max_det = 1024
    try:
        first, second = _stream_frames([0, 0, 0], 50), _stream_frames([0, 1], 51)
        dn.network_streams_open(net, 2)
        want_first = dn.network_detect_streams(net, [0, 0, 0], first, THRESH, NMS, max_det)[0]
        dn.network_streams_open(net, 2)
        want_second = dn.network_detect_streams(net, [0, 1], second, THRESH, NMS, max_det)[0]  # fresh streams
        assert any(len(d) for d in want_first + want_second)
        dn.network_streams_open(net, 2)
        dn.network_detect_submit_streams(net, [1], _stream_frames([1], 52), THRESH, NMS, max_det)
        dn.network_detect_wait_n(net, 1, max_det)  # stream 1 is not fresh when it is reset
        dn.network_detect_submit_streams(net, [0, 0, 0], first, THRESH, NMS, max_det)
        dn.network_stream_reset(net, 0)
        dn.network_stream_reset(net, 1)
        dn.network_detect_submit_streams(net, [0, 1], second, THRESH, NMS, max_det)
        _same_dets(dn.network_detect_wait_n(net, 3, max_det)[0], want_first, "before the reset")
        _same_dets(dn.network_detect_wait_n(net, 2, max_det)[0], want_second, "after the reset")
    finally:
        dn.free_network(net)


def test_set_batch_network_keeps_the_rings(tmp_path):
    net = _detector(tmp_path, "tiny-yolo-voc", 4)
    try:
        dn.network_streams_open(net, 3)
        lists = [[0, 1, 0], [2, 0, 1, 1], [0, 2, 0, 1, 1, 2, 0], [1, 0]]
        batches = [(lists[0], _stream_frames(lists[0], 60)), (lists[1], _stream_frames(lists[1], 61)),
                   lambda: dn.set_batch_network(net, 8),  # beyond the planned capacity: a re-plan
                   (lists[2], _stream_frames(lists[2], 62)),
                   lambda: dn.set_batch_network(net, 2),
                   (lists[3], _stream_frames(lists[3], 63))]
        _check_sequence(net, HostStreams(net), batches, THRESH, NMS, 1024, "set_batch")
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


@pytest.mark.parametrize("case", ["not_opened", "id_over", "id_negative", "null_ids", "tree_head", "resized",
                                  "list_over_batch", "null_frame", "resident_n0", "reset_id", "open_zero"])
def test_streams_refusals_exit_through_error(tmp_path, case):
    extra = ""
    if case == "tree_head":
        synth.write_tree(tmp_path / "t.tree", n=4, fanout=2, roots=2)
        extra = f"tree={tmp_path / 't.tree'}\n"
    cfg_text = synth.exact_detector_cfg(batch=2, extra=extra)
    (tmp_path / "n.cfg").write_text(cfg_text)
    synth.write_exact_weights(tmp_path / "n.weights", cfg_text)
    opened = "dn.network_streams_open(net, 2)\n"
    call, msg = {
        "not_opened": ("dn.network_detect_streams(net, [0], [f], .5, .4)", "streams not opened"),
        "id_over": (opened + "dn.network_detect_submit_streams(net, [0, 2], [f, f], .5, .4)", "stream id outside"),
        "id_negative": (opened + "dn.network_detect_submit_streams_resident(net, [-1], .5, .4)", "stream id outside"),
        "null_ids": (opened + "lib.network_detect_submit_streams_resident(net, 1, None, .5, .4, 16)",
                     "NULL stream id array"),
        "tree_head": ("dn.network_streams_open(net, 2)", "flat-softmax region head"),
        "resized": (opened + "dn.resize_network(net, 64, 48)\n"
                    "dn.network_detect_submit_streams_resident(net, [0], .5, .4)", "region output size differs"),
        "list_over_batch": (opened + "dn.network_detect_streams(net, [0, 1, 0], [f, f, f], .5, .4)",
                            "1 .. batch frames"),
        "null_frame": (opened + "lib.network_detect_submit_streams(net, 1, (C.c_int * 1)(0), "
                       "(C.POINTER(C.c_ubyte) * 1)(None), (C.c_int * 1)(16), (C.c_int * 1)(12), .5, .4, 16)",
                       "NULL frame pointer"),
        "resident_n0": (opened + "lib.network_detect_submit_streams_resident(net, 0, (C.c_int * 1)(0), .5, .4, 16)",
                        "1 .. batch images"),
        "reset_id": (opened + "dn.network_stream_reset(net, 2)", "stream id outside"),
        "open_zero": ("dn.network_streams_open(net, 0)", "max_streams must be 1 or more"),
    }[case]
    code = REFUSE.format(root=str(ROOT), cfg=str(tmp_path / "n.cfg"), weights=str(tmp_path / "n.weights"), call=call)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert r.returncode != 0 and "RETURNED" not in r.stdout, r.stdout
    assert msg in r.stderr, r.stderr[-2000:]
