"""CPU tests of tracked video streams: the y2_bbox mirror, the tracking plan y2_track_plan against a restatement of the
Detector's history (yolo_v2_class.cpp:251-304: push_front, pop_back beyond frames_story, ids from 1 per fresh
Detector), and the refusal of every tracked entry on a network without a device plan."""
import ctypes as C
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from sr_object_detection_b200 import _lib, darknet as dn, synth

ROOT = Path(__file__).resolve().parents[1]


def test_bbox_mirror_has_the_layout_of_bbox_t():
    lib = dn.lib()
    assert lib.y2_abi_sizeof(6) == C.sizeof(dn.BBox) == 28
    assert [f for f, _ in dn.BBox._fields_] == ["x", "y", "w", "h", "prob", "obj_id", "track_id"]


class DetectorHistories:
    """One Detector per stream: its deque of remembered frames (newest first, at most story) and whether its ids
    are fresh.  A frame is named by (batch, image)."""

    def __init__(self, max_streams, story):
        self.story = story
        self.deque = [[] for _ in range(max_streams)]
        self.fresh = [True] * max_streams

    def reset(self, s):
        self.deque[s] = []
        self.fresh[s] = True

    def frame(self, s, name):
        """the frames its tracking() matches against, and whether its ids start over; then remember it"""
        before, fresh = list(self.deque[s]), self.fresh[s]
        self.deque[s].insert(0, name)
        del self.deque[s][self.story:]
        self.fresh[s] = False
        return before, fresh


def _run(max_streams, story, batches, seed):
    """batches: (ids, sizes, streams reset before it).  Checks the CSR order, the sizes and flags, and that the history
    slots each record names hold exactly the frames the Detector remembers, newest first."""
    ref = DetectorHistories(max_streams, story)
    head, length, restart = [0] * max_streams, [0] * max_streams, [1] * max_streams
    slots = [[None] * story for _ in range(max_streams)]  # the frame each device history slot holds
    for b, (ids, sizes, resets) in enumerate(batches):
        for s in resets:
            ref.reset(s)
            head[s], length[s], restart[s] = 0, 0, 1  # network_stream_reset: host counters only
        recs, offsets, head, length, restart = _lib.track_plan(ids, sizes, max_streams, story, head, length, restart)
        distinct = list(dict.fromkeys(ids))
        assert len(offsets) == len(distinct) + 1 and offsets[0] == 0 and offsets[-1] == len(ids)
        for k, s in enumerate(distinct):
            run = recs[offsets[k]:offsets[k + 1]]
            assert [r.image for r in run] == [i for i, v in enumerate(ids) if v == s], (seed, b)
            assert all(r.stream == s for r in run)
        for r in recs:
            i, s = r.image, r.stream
            assert (r.w, r.h) == sizes[i]
            before, fresh = ref.frame(s, (b, i))
            assert bool(r.restart) == fresh, (seed, b, i)
            assert 0 <= r.head < story and r.len == len(before), (seed, b, i)
            assert [slots[s][(r.head - k) % story] for k in range(1, r.len + 1)] == before, (seed, b, i)
            slots[s][r.head] = (b, i)


@pytest.mark.parametrize("seed", range(40))
def test_plan_equals_the_detector_histories(seed):
    rng = np.random.default_rng(seed)
    max_streams = int(rng.integers(1, 9))
    story = int(rng.integers(1, 33))
    batches = []
    for _ in range(int(rng.integers(1, 9))):
        n = int(rng.integers(1, 17))
        ids = [int(v) for v in rng.integers(0, max_streams, n)]
        sizes = [(int(rng.integers(1, 2000)), int(rng.integers(1, 2000))) for _ in range(n)]
        resets = [int(v) for v in rng.choice(max_streams, int(rng.integers(0, 3)))] if rng.random() < .4 else []
        batches.append((ids, sizes, resets))
    _run(max_streams, story, batches, seed)


def test_plan_of_one_stream_repeated_past_its_story():
    recs, offsets, head, length, restart = _lib.track_plan([1] * 5, [(8, 6)] * 5, 3, 2, [0] * 3, [0] * 3, [1] * 3)
    assert offsets == [0, 5]
    assert [(r.head, r.len, r.restart) for r in recs] == [(0, 0, 1), (1, 1, 0), (0, 2, 0), (1, 2, 0), (0, 2, 0)]
    assert head == [0, 1, 0] and length == [0, 2, 0] and restart == [1, 0, 1]


def test_plan_refuses_bad_arguments_and_changes_nothing():
    lib = _lib.load()
    for ids, w, story in (([0, 3], 4, 2), ([-1], 4, 2), ([0, 1], 0, 2), ([0], 4, 0), ([0], 4, 33)):
        n = len(ids)
        head, length, restart = (C.c_int * 3)(1, 0, 0), (C.c_int * 3)(1, 0, 0), (C.c_int * 3)(0, 1, 1)
        recs, offsets = (_lib.TrackImg * 3)(), (C.c_int * 4)()
        fw, fh = (C.c_int * n)(*[w] * n), (C.c_int * n)(*[5] * n)
        assert lib.y2_track_plan(n, (C.c_int * n)(*ids), fw, fh, 3, story, head, length, restart, recs, offsets) < 0
        assert list(head) == [1, 0, 0] and list(length) == [1, 0, 0] and list(restart) == [0, 1, 1]


FRAMES = "[np.zeros((12, 16, 3), np.uint8)]"
CALLS = {
    "track": "dn.network_streams_track(net, 6)",
    "batch": f"dn.network_detect_streams_tracked(net, [0], {FRAMES}, .5, .4)",
    "submit": f"dn.network_detect_submit_streams_tracked(net, [0], {FRAMES}, .5, .4)",
    "submit_resident": "dn.network_detect_submit_streams_tracked_resident(net, [0], [(16, 12)], .5, .4)",
    "wait": "dn.network_detect_wait_tracked(net, 1)",
}


@pytest.mark.parametrize("call", sorted(CALLS))
def test_tracked_entries_without_a_device_plan_exit_through_error(tmp_path, call):
    cfg = tmp_path / "net.cfg"
    cfg.write_text(synth.exact_detector_cfg(batch=1))
    code = ("import sys, numpy as np; sys.path.insert(0, %r)\n"
            "from sr_object_detection_b200 import darknet as dn\n"
            "dn.set_gpu_index(-1)\n"
            "net = dn.parse_network_cfg(%r)\n"
            "%s\n"
            "print('COMPUTED')\n" % (str(ROOT), str(cfg), CALLS[call]))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert r.returncode != 0 and "COMPUTED" not in r.stdout
    assert ("no device plan" if call != "wait" else "nothing in flight") in r.stderr, r.stderr[-2000:]
