"""Tracked video streams (network_streams_track, network_detect_*_streams_tracked, y2_stream_track) against the
Detector's own flow, per stream: detect(img, thresh, use_mean) and then tracking(result, frames_story)
(yolo_v2_class.cpp:173-304).  The kernel is checked on crafted detection lists against the restatement of
Detector::tracking that tests/test_detector_cpp.py pins to the C++ class; the entries against the C++ Detector itself and
the reference Detector's golden `track` lines.  Every comparison is bit for bit."""
import ctypes as C
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from sr_object_detection_b200 import _lib, darknet as dn, synth
from tests.test_detector_cpp import _track_reference
from tests.test_frame_list_gpu import _frames, _stage

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
LIBDIR = ROOT / "sr_object_detection_b200"


# ---- the kernel through y2_stream_track -----------------------------------------------------------------------------
def _to_bbox(bx, by, bw, bh, w, h):
    """yolo_v2_class.cpp:228-236 on float32 box values: corner in double clamped at 0, extent in float"""
    bx, by, bw, bh = (float(np.float32(v)) for v in (bx, by, bw, bh))
    x = int(max(0.0, (bx - bw / 2.0) * w))
    y = int(max(0.0, (by - bh / 2.0) * h))
    return x, y, int(np.float32(bw) * np.float32(w)), int(np.float32(bh) * np.float32(h))


class KernelRun:
    """The device state of S streams and the host counters; batches of (stream, dets, w, h) through the kernel, and
    per stream the sequence of frames since its last start-over for the reference."""

    def __init__(self, S, story, total, classes):
        self.S, self.story, self.total, self.classes = S, story, total, classes
        self.hist = torch.zeros(S * story * total * 7, dtype=torch.int32, device="cuda")
        self.hist_cnt = torch.zeros(S * story, dtype=torch.int32, device="cuda")
        self.next_id = torch.full((S * classes,), 12345, dtype=torch.int32, device="cuda")
        self.head, self.len, self.restart = [0] * S, [0] * S, [1] * S
        self.segments = {s: [[]] for s in range(S)}  # stream -> list of segments of (frame in pixels, prob, got)

    def reset(self, s):
        self.head[s], self.len[s], self.restart[s] = 0, 0, 1
        self.segments[s].append([])

    def batch(self, items):
        """items: (stream, [(bx, by, bw, bh, prob, obj)], w, h) per image"""
        n, total = len(items), self.total
        det = np.zeros((n, total), np.dtype([("x", "<f4"), ("y", "<f4"), ("w", "<f4"), ("h", "<f4"),
                                             ("prob", "<f4"), ("obj_id", "<i4"), ("box_index", "<i4")]))
        det["box_index"] = -9
        count = np.array([len(d) for _, d, _, _ in items], np.int32)
        for i, (_, dets, _, _) in enumerate(items):
            for m, (bx, by, bw, bh, p, obj) in enumerate(dets):
                det[i, m] = (bx, by, bw, bh, p, obj, m)
        recs, offsets, self.head, self.len, self.restart = _lib.track_plan(
            [s for s, _, _, _ in items], [(w, h) for _, _, w, h in items], self.S, self.story, self.head, self.len,
            self.restart)
        d_det = torch.from_numpy(det.view(np.uint8).reshape(-1).copy()).cuda()
        d_cnt = torch.from_numpy(count).cuda()
        d_recs = torch.from_numpy(np.frombuffer((_lib.TrackImg * n)(*recs), np.uint8).copy()).cuda()
        d_off = torch.tensor(offsets, dtype=torch.int32, device="cuda")
        d_out = torch.full((n * total * 7,), -1, dtype=torch.int32, device="cuda")
        _lib.check(_lib.load().y2_stream_track(d_det.data_ptr(), total, d_cnt.data_ptr(), d_recs.data_ptr(),
                                               d_off.data_ptr(), len(offsets) - 1, total, self.classes, self.story,
                                               self.hist.data_ptr(), self.hist_cnt.data_ptr(), self.next_id.data_ptr(),
                                               d_out.data_ptr(), total, None), "y2_stream_track")
        out = d_out.cpu().numpy().reshape(n, total, 7)
        for i, (s, dets, w, h) in enumerate(items):
            px = [_to_bbox(bx, by, bw, bh, w, h) + (obj,) for bx, by, bw, bh, _, obj in dets]
            probs = [np.float32(p) for *_, p, _ in dets]
            self.segments[s][-1].append((px, probs, out[i, :len(dets)].copy()))

    def check(self, tag):
        boxes = 0
        for s, segs in self.segments.items():
            for k, seg in enumerate(segs):
                want = _track_reference([px for px, _, _ in seg], self.story)
                for f, ((_, probs, got), w) in enumerate(zip(seg, want)):
                    got_rows = [(int(r[0]), int(r[1]), int(r[2]), int(r[3]), int(r[5]), int(r[6])) for r in
                                got.view(np.uint32)]
                    assert got_rows == [tuple(b) for b in w], f"{tag}: stream {s} segment {k} frame {f}"
                    assert got[:, 4].tobytes() == np.array(probs, np.float32).view(np.int32).tobytes()
                    boxes += len(w)
        return boxes


def _px(x, y, w, h, obj, prob=0.5):
    """a box given in pixels of a 1 x 1 frame: the conversion is exact (centre x + w/2 in float32)"""
    return (x + w / 2, y + h / 2, w, h, prob, obj)


# frames of one stream, in pixels: (x, y, w, h, obj)
CRAFTED = {
    "dist_99": [[(0, 0, 10, 10, 0)], [(99, 0, 10, 10, 0)]],
    "dist_100": [[(0, 0, 10, 10, 0)], [(100, 0, 10, 10, 0)]],
    "equal_distances": [[(100, 100, 10, 10, 0)], [(60, 100, 10, 10, 0), (140, 100, 10, 10, 0)]],
    "best_updated_not_chosen": [[(0, 0, 10, 10, 0), (30, 0, 10, 10, 0)],
                                [(10, 0, 10, 10, 0), (20, 0, 10, 10, 0), (80, 0, 10, 10, 0)]],
    "id_taken": [[(0, 0, 10, 10, 0)], [(2, 0, 10, 10, 0)], [(4, 0, 10, 10, 0), (6, 0, 10, 10, 0)]],
    "width_average_moves_a_match": [[(0, 0, 200, 10, 0), (150, 0, 10, 10, 0)], [(10, 0, 10, 10, 0)],
                                    [(60, 0, 120, 10, 0), (110, 0, 10, 10, 0)]],
    "empty_frames": [[], [(5, 5, 10, 10, 1)], [], [], [(8, 5, 10, 10, 1)], []],
    "only_empty_history": [[], [], [(5, 5, 10, 10, 0), (50, 5, 10, 10, 0)], [(6, 5, 10, 10, 0)]],
    "full_story": [[(i * 30, 0, 10, 10, 0)] for i in range(9)] + [[(0, 0, 10, 10, 0), (250, 0, 10, 10, 0)]],
    "classes": [[(0, 0, 10, 10, 0), (0, 0, 10, 10, 1), (0, 0, 10, 10, 2)],
                [(1, 1, 10, 10, 2), (1, 1, 10, 10, 0), (300, 300, 4, 4, 1), (2, 2, 10, 10, 1)]],
    "reference_script": [[(10, 10, 40, 40, 0), (200, 200, 50, 50, 0), (300, 20, 30, 60, 1)],
                         [(14, 12, 44, 40, 0), (205, 190, 50, 54, 0), (500, 400, 30, 30, 1)], [],
                         [(20, 15, 40, 40, 0), (290, 30, 30, 60, 1), (295, 28, 30, 60, 1)], [(400, 400, 10, 10, 2)],
                         [(22, 18, 40, 40, 0), (402, 398, 12, 12, 2), (60, 60, 40, 40, 0)]],
}


@pytest.mark.parametrize("case", sorted(CRAFTED))
@pytest.mark.parametrize("story", [1, 3, 6])
def test_kernel_on_crafted_sequences(case, story):
    run = KernelRun(1, story, 16, 3)
    for frame in CRAFTED[case]:
        run.batch([(0, [_px(*b) for b in frame], 1, 1)])
    run.check(case)
    if case in ("dist_99", "dist_100") and story >= 1:
        ids = [int(r[6]) for r in run.segments[0][0][1][2].view(np.uint32)]
        assert ids == ([1] if case == "dist_99" else [2])


def _random_frames(rng, n_frames, max_boxes, classes):
    """drifting boxes in relative units: most of a frame's boxes stay within 100 pixels of the last frame's"""
    frames, prev = [], []
    for _ in range(n_frames):
        k = int(rng.integers(0, max_boxes + 1))
        cur = []
        for m in range(k):
            if prev and rng.random() < .7:
                bx, by, bw, bh, _, obj = prev[int(rng.integers(0, len(prev)))]
                bx, by = bx + rng.normal(0, .02), by + rng.normal(0, .02)
                bw, bh = bw * rng.uniform(.8, 1.25), bh * rng.uniform(.8, 1.25)
            else:
                bx, by, bw, bh = rng.uniform(-.05, 1.05), rng.uniform(-.05, 1.05), rng.uniform(.01, .6), \
                    rng.uniform(.01, .6)
                obj = int(rng.integers(0, classes))
            cur.append((bx, by, bw, bh, float(rng.random()), obj))
        frames.append(cur)
        prev = cur or prev
    return frames


@pytest.mark.parametrize("seed", range(6))
def test_kernel_on_many_streams_with_repeats_and_resets(seed):
    rng = np.random.default_rng(seed)
    S, story, classes = 5, int(rng.integers(1, 9)), 4
    total = [845, 125, 13][seed % 3]
    sizes = [(640, 480), (1920, 1080), (416, 416), (353, 500), (37, 53)]
    queues = {s: _random_frames(rng, 200, min(total, 200 if s == 0 else 30), classes) for s in range(S)}
    run = KernelRun(S, story, total, classes)
    for b in range(12):
        ids = [int(v) for v in rng.integers(0, S, int(rng.integers(1, 17)))]
        run.batch([(s, queues[s].pop(), *sizes[s]) for s in ids])
        if rng.random() < .3:
            run.reset(int(rng.integers(0, S)))
    assert run.check(f"seed {seed}") > 100


def test_kernel_on_frames_of_every_box():
    rng = np.random.default_rng(99)
    total = 845
    run = KernelRun(2, 2, total, 20)
    frames = _random_frames(rng, 4, total, 20)
    for f in frames:
        f += [f[0]] * (total - len(f)) if f else []
    run.batch([(0, frames[0], 640, 480), (1, frames[1], 500, 375), (0, frames[2], 640, 480)])
    run.batch([(0, frames[3], 640, 480)])
    assert run.check("every box") > total


# ---- the entries against the C++ Detector ---------------------------------------------------------------------------
def _build_driver(tmp_path):
    from sr_object_detection_b200 import build as b
    b.build()
    exe = tmp_path / "detector_track"
    cmd = ["g++", "-O1", "-std=c++17", "-I", str(ROOT / "include"), str(ROOT / "tests" / "cpp" / "detector_track.cpp"),
           "-L", str(LIBDIR), "-lyolo2_b200", f"-Wl,-rpath,{LIBDIR}", "-o", str(exe)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return exe


def _detector_runs(tmp_path, cfg, weights, thresh, nms, story, segments):
    """segments: lists of (uint8 frame, use_mean), each run by a fresh C++ Detector; the tracked bbox_t lists as
    (n, 7) uint32 arrays (prob as its bits), in segment order"""
    exe = _build_driver(tmp_path)
    blob, spec, off = [], [], 0
    for seg in segments:
        spec.append("new")
        for f, use_mean in seg:
            spec.append(f"frame {off} {f.shape[1]} {f.shape[0]} {int(use_mean)}")
            blob.append(f.reshape(-1))
            off += f.size
    (tmp_path / "frames.u8").write_bytes(np.concatenate(blob).tobytes())
    (tmp_path / "spec.txt").write_text("\n".join(spec) + "\n")
    r = subprocess.run([str(exe), str(cfg), str(weights), str(thresh), str(nms), str(story),
                        str(tmp_path / "frames.u8"), str(tmp_path / "spec.txt"), "0"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l.split() for l in r.stdout.splitlines() if l.startswith("track ")]
    out = []
    for t in lines:
        n = int(t[2])
        rows = np.zeros((n, 7), np.uint32)
        for m in range(n):
            v = t[3 + 7 * m:10 + 7 * m]
            rows[m] = [int(v[0]), int(v[1]), int(v[2]), int(v[3]), np.float32(float(v[4])).view(np.uint32),
                       int(v[5]), int(v[6])]
        out.append(rows)
    it = iter(out)
    return [[next(it) for _ in seg] for seg in segments]


def _rows(arr):
    return np.ascontiguousarray(arr).view(np.uint32).reshape(-1, 7)


def _detector(tmp_path, name, batch):
    text = synth.CFGS[name](batch=batch, w=416, h=416)
    cfg, weights = tmp_path / f"{name}.cfg", tmp_path / f"{name}.weights"
    cfg.write_text(text)
    synth.write_weights(weights, text, seed=1234)
    dn.set_gpu_index(0)
    net = dn.parse_network_cfg(cfg)
    dn.load_weights(net, weights)
    return net, cfg, weights  # the Detector sets batch 1 itself


THRESH, NMS, STORY = 0.02, 0.4, 4
SIZES = [(500, 375), (640, 480), (416, 416), (1280, 720)]  # tracked stream s: frames of SIZES[s]


@pytest.mark.parametrize("name", ["tiny-yolo-voc", "yolo-voc"])
def test_tracked_streams_equal_the_cpp_detector(tmp_path, name):
    net, cfg, weights = _detector(tmp_path, name, 6)
    max_det = 64  # below the detections of some frames: tracking still sees them all
    wide = 1024  # untracked batches ask for more detections than the 845 boxes of a frame: longer list rows
    rng = np.random.default_rng(7)
    segments = {s: [[]] for s in range(4)}  # the Detector's view: frames (and use_mean) since the last start-over
    got = {s: [[]] for s in range(4)}
    counts_seen = []

    def frames_of(ids, seed):
        fr = _frames([SIZES[s] for s in ids], seed)
        for i, f in enumerate(fr):  # consecutive frames of a stream alike, so that tracks continue
            if segments[ids[i]][-1]:
                base = segments[ids[i]][-1][-1][0]
                f[:] = np.clip(base.astype(np.int16) + rng.integers(-12, 13, f.shape), 0, 255).astype(np.uint8)
        return fr

    def record(ids, fr, use_mean, result):
        boxes, counts = result
        counts_seen.extend(counts)
        for i, s in enumerate(ids):
            segments[s][-1].append((fr[i], use_mean))
            got[s][-1].append((_rows(boxes[i]), counts[i]))

    def reset(s):
        dn.network_stream_reset(net, s)
        segments[s].append([])
        got[s].append([])

    try:
        dn.network_streams_open(net, 6)
        dn.network_streams_track(net, STORY)
        warm = _frames([(640, 480)] * 3, 99)
        for _ in range(2):  # both pipeline slots hold wide detection lists before the first tracked batch
            dn.network_detect_frame_list(net, warm, THRESH, NMS, wide)
        plan = [([0, 1, 0, 2, 0], True, "batch"), ([3, 3, 1, 2], False, "submit"), ([0, 1, 2, 3, 3, 3], True, "staged"),
                "reset1", ([1, 1, 0, 2], False, "batch"), "set_batch", ([2, 0, 3, 1, 0, 0, 0, 2], True, "submit"),
                ([0, 2], False, "batch"), "reset0", ([0, 0, 1], True, "staged")]
        k = 0
        for step in plan:
            if step == "reset1":
                reset(1)
                continue
            if step == "reset0":
                reset(0)
                continue
            if step == "set_batch":
                dn.set_batch_network(net, 8)  # beyond the planned capacity: a re-plan keeps the tracks
                continue
            ids, use_mean, how = step
            fr = frames_of(ids, 100 + k)
            k += 1
            if how == "batch":
                record(ids, fr, use_mean, dn.network_detect_streams_tracked(net, ids, fr, THRESH, NMS, use_mean,
                                                                           max_det))
                continue
            # interleaved with an untracked streams batch (stream 5) and a plain frame list
            other = _frames([(640, 480)] * 2, 200 + k)
            dn.network_detect_submit_streams(net, [5, 5], other, THRESH, NMS, wide)
            dn.network_detect_submit_streams_tracked(net, ids, _stage(net, fr) if how == "staged" else fr, THRESH,
                                                     NMS, use_mean, max_det)
            dn.network_detect_wait_n(net, 2, wide)
            dn.network_detect_submit_frame_list(net, other, THRESH, NMS, wide)
            record(ids, fr, use_mean, dn.network_detect_wait_tracked(net, len(ids), max_det))
            dn.network_detect_wait_n(net, 2, wide)
        want = _detector_runs(tmp_path, cfg, weights, THRESH, NMS, STORY,
                              [seg for s in range(4) for seg in segments[s]])
        it = iter(want)
        continued = 0  # boxes that carry on a track of the stream's previous frame
        for s in range(4):
            for k, seg in enumerate(got[s]):
                w_seg = next(it)
                assert len(w_seg) == len(seg)
                for f, ((g, count), w) in enumerate(zip(seg, w_seg)):
                    assert count == len(w), f"{name}: stream {s} segment {k} frame {f}"
                    assert np.array_equal(g, w[:max_det]), f"{name}: stream {s} segment {k} frame {f}"
                    if f:
                        prev = {(int(r[5]), int(r[6])) for r in w_seg[f - 1]}
                        continued += sum((int(r[5]), int(r[6])) in prev for r in w)
        assert max(counts_seen) > max_det, "test needs frames with more detections than max_det"
        assert continued > 0
    finally:
        dn.free_network(net)


def test_resident_entry_equals_the_cpp_detector(tmp_path):
    net, cfg, weights = _detector(tmp_path, "tiny-yolo-voc", 4)
    lib = _lib.load()
    try:
        dn.network_streams_open(net, 2)
        dn.network_streams_track(net, 3)
        base = _frames([(416, 416)] * 2, 300)
        rng = np.random.default_rng(3)
        seq = [[np.clip(b.astype(np.int16) + rng.integers(-10, 11, b.shape), 0, 255).astype(np.uint8) for b in base]
               for _ in range(5)]
        lists = [[0, 1], [1, 0, 0], [0], [1, 1, 0]]
        use = [True, False, True, False]
        pos = [0, 0]
        segs = {0: [], 1: []}
        got = {0: [], 1: []}
        sizes = {0: (416, 416), 1: (832, 624)}  # stream 1's boxes scaled as for a frame twice the size
        for ids, use_mean in zip(lists, use):
            x = np.zeros((4, 3, 416, 416), np.float32)
            for i, s in enumerate(ids):
                f = seq[pos[s]][s]
                pos[s] += 1
                x[i] = (f.transpose(2, 0, 1).astype(np.float64) / 255.).astype(np.float32)
                segs[s].append((f, use_mean))
            dev = dn.lib().network_pipeline_input_device(net, dn.lib().network_pipeline_next_slot(net))
            _lib.check(lib.y2_memcpy_h2d(dev, x.ctypes.data, x.nbytes, None), "h2d")
            _lib.check(lib.y2_stream_sync(None))
            dn.network_detect_submit_streams_tracked_resident(net, ids, [sizes[s] for s in ids], THRESH, NMS,
                                                              use_mean, 1024)
            boxes, _ = dn.network_detect_wait_tracked(net, len(ids), 1024)
            for i, s in enumerate(ids):
                got[s].append(_rows(boxes[i]))
        # stream 0 as the Detector sees it; stream 1's boxes are scaled to the frame size given for it
        want = _detector_runs(tmp_path, cfg, weights, THRESH, NMS, 3, [segs[0]])[0]
        assert len(want) == len(got[0])
        for f, (g, w) in enumerate(zip(got[0], want)):
            assert np.array_equal(g, w), f"frame {f}"
        assert sum(len(w) for w in want) > 0
        assert max(int(g[:, 0].max() + g[:, 2].max()) for g in got[1] if len(g)) > 416  # scaled to the frame size
    finally:
        dn.free_network(net)


# ---- the reference's own class --------------------------------------------------------------------------------------
def test_tracked_streams_reproduce_the_reference_detector_track_lines(tmp_path):
    g = json.loads((ROOT / "tests" / "golden" / "detector_ref.json").read_text())
    want = [l for l in g["lines"] if l.startswith("track ")]
    assert len(want) == g["n"] == 6
    w, h, B = g["w"], g["h"], 4
    cfg = g["cfg"].replace("batch=1", f"batch={B}")
    (tmp_path / "net.cfg").write_text(cfg)
    synth.write_exact_weights(tmp_path / "net.weights", g["cfg"])
    frames = synth.exact_frames(g["n"], h, w)
    others = synth.exact_frames(8, h, w, seed=31)
    dn.set_gpu_index(0)
    net = dn.parse_network_cfg(tmp_path / "net.cfg")
    dn.load_weights(net, tmp_path / "net.weights")
    lib = _lib.load()

    def run(lists):
        lines = []
        for items in lists:
            x = np.zeros((B, 3, h, w), np.float32)
            for i, (_, f) in enumerate(items):
                x[i] = f
            dev = dn.lib().network_pipeline_input_device(net, dn.lib().network_pipeline_next_slot(net))
            _lib.check(lib.y2_memcpy_h2d(dev, x.ctypes.data, x.nbytes, None), "h2d")
            _lib.check(lib.y2_stream_sync(None))
            ids = [s for s, _ in items]
            dn.network_detect_submit_streams_tracked_resident(net, ids, [(w, h)] * len(ids), g["thresh"], g["nms"],
                                                              False, 1024)
            got, _ = dn.network_detect_wait_tracked(net, len(items), 1024)
            lines += [d for (s, _), d in zip(items, got) if s == 0]
        return ["track %d %d" % (i, len(d)) + "".join(" %d %d %d %d %.9g %d %d" % (b["x"], b["y"], b["w"], b["h"],
                                                                                   float(b["prob"]), b["obj_id"],
                                                                                   b["track_id"]) for b in d)
                for i, d in enumerate(lines)]

    try:
        dn.network_streams_open(net, 1)
        dn.network_streams_track(net, g["story"])
        assert run([[(0, frames[i])] for i in range(3)] + [[(0, frames[3]), (0, frames[4]), (0, frames[5])]]) == want
        dn.network_streams_open(net, 3)
        dn.network_streams_track(net, g["story"])
        spread = [[(1, others[0]), (0, frames[0]), (2, others[1]), (0, frames[1])],
                  [(0, frames[2]), (1, others[2]), (0, frames[3]), (0, frames[4])],
                  [(2, others[3]), (2, others[4]), (1, others[5]), (0, frames[5])]]
        assert run(spread) == want
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
I1 = (C.c_int * 1)
{call}
print("RETURNED")
"""


@pytest.mark.parametrize("case", ["not_opened", "not_tracked", "story_zero", "story_over", "use_mean_2",
                                  "resident_null_w", "resident_size_0", "id_over", "list_over_batch", "reopen_drops",
                                  "wait_wrong_kind", "wait_tracked_wrong_kind", "track_not_opened", "too_many_boxes"])
def test_tracked_refusals_exit_through_error(tmp_path, case):
    # 96 x 80 cells of 3 anchors: 23040 boxes a frame, more than Y2_TRACK_MAX_TOTAL
    cfg_text = synth.exact_detector_cfg(batch=2, **({"w": 96, "h": 80} if case == "too_many_boxes" else {}))
    (tmp_path / "n.cfg").write_text(cfg_text)
    synth.write_exact_weights(tmp_path / "n.weights", cfg_text)
    opened = "dn.network_streams_open(net, 2)\n"
    tracked = opened + "dn.network_streams_track(net, 6)\n"
    call, msg = {
        "not_opened": ("dn.network_detect_streams_tracked(net, [0], [f], .5, .4)", "streams not opened"),
        "not_tracked": (opened + "dn.network_detect_streams_tracked(net, [0], [f], .5, .4)", "tracking not enabled"),
        "story_zero": (opened + "dn.network_streams_track(net, 0)", "frames_story must be in"),
        "story_over": (opened + "dn.network_streams_track(net, 33)", "frames_story must be in"),
        "use_mean_2": (tracked + "dn.network_detect_submit_streams_tracked(net, [0], [f], .5, .4, 2)",
                       "use_mean must be 0 or 1"),
        "resident_null_w": (tracked + "lib.network_detect_submit_streams_tracked_resident(net, 1, I1(0), None, I1(9), "
                            ".5, .4, 1, 16)", "NULL frame width or height array"),
        "resident_size_0": (tracked + "dn.network_detect_submit_streams_tracked_resident(net, [0], [(16, 0)], .5, .4)",
                            "a frame size of 0 or less"),
        "id_over": (tracked + "dn.network_detect_submit_streams_tracked(net, [0, 2], [f, f], .5, .4)",
                    "stream id outside"),
        "list_over_batch": (tracked + "dn.network_detect_streams_tracked(net, [0, 1, 0], [f, f, f], .5, .4)",
                            "1 .. batch frames"),
        "reopen_drops": (tracked + opened + "dn.network_detect_streams_tracked(net, [0], [f], .5, .4)",
                         "tracking not enabled"),
        "wait_wrong_kind": (tracked + "dn.network_detect_submit_streams_tracked(net, [0], [f], .5, .4)\n"
                            "dn.network_detect_wait_n(net, 1)", "is a tracked batch, call network_detect_wait_tracked"),
        "wait_tracked_wrong_kind": (opened + "dn.network_detect_submit_streams(net, [0], [f], .5, .4)\n"
                                    "dn.network_detect_wait_tracked(net, 1)", "an untracked detection batch"),
        "track_not_opened": ("dn.network_streams_track(net, 6)", "streams not opened"),
        "too_many_boxes": (opened + "dn.network_streams_track(net, 6)", "more region boxes per image than"),
    }[case]
    code = REFUSE.format(root=str(ROOT), cfg=str(tmp_path / "n.cfg"), weights=str(tmp_path / "n.weights"), call=call)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert r.returncode != 0 and "RETURNED" not in r.stdout, r.stdout
    assert msg in r.stderr, r.stderr[-2000:]
