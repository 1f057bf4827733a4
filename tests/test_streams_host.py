"""CPU tests of the video-streams entries (each frame detected on the 3-frame mean of its stream): the ring plan
y2_stream_plan against a restatement of the Detector's own ring (yolo_v2_class.cpp:206-216), and the refusal of every
streams entry on a network without a device plan."""
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from sr_object_detection_b200 import _lib, synth

ROOT = Path(__file__).resolve().parents[1]


class DetectorRings:
    """yolo_v2_class.cpp:206-216 per stream: ring[frame_index] = this frame, mean over the 3 slots, advance.  A slot
    holds the id of the frame that wrote it (None: not written since the start / reset)."""

    def __init__(self, max_streams):
        self.ring = [[None] * 3 for _ in range(max_streams)]
        self.index = [0] * max_streams
        self.seen = [0] * max_streams

    def reset(self, s):
        self.ring[s] = [None] * 3
        self.index[s] = 0
        self.seen[s] = 0

    def frame(self, s, frame_id):
        """the slot the frame writes and the 3 slots its mean reads"""
        slot = self.index[s]
        self.ring[s][slot] = frame_id
        self.index[s] = (slot + 1) % 3
        self.seen[s] = min(self.seen[s] + 1, 3)
        return slot, list(self.ring[s])


def _run(max_streams, batches, seed):
    """batches: list of (id list, streams reset before it).  Checks every record of every batch exactly, and that
    the ring the records describe holds what the Detector's ring holds."""
    ref = DetectorRings(max_streams)
    fi, seen = [0] * max_streams, [0] * max_streams
    device_ring = [None] * (3 * max_streams)  # frame id each ring row holds after the commits so far
    for b, (ids, resets) in enumerate(batches):
        for s in resets:
            ref.reset(s)
            fi[s], seen[s] = 0, 0  # network_stream_reset: host counters only, the ring is not touched
        plan, fi, seen = _lib.stream_plan(ids, max_streams, fi, seen)
        assert len(plan) == len(ids)
        frames = [ref.frame(s, (b, i)) for i, s in enumerate(ids)]  # (slot written, the 3 slots the mean reads)
        for i, s in enumerate(ids):
            slot = frames[i][0]
            later = any(ids[k] == s and frames[k][0] == slot for k in range(i + 1, len(ids)))
            assert plan[i].commit == (-1 if later else 3 * s + slot), (seed, b, i, ids)
            for j in range(3):
                code = plan[i].src[j]
                held = frames[i][1][j]
                if held is None:
                    want = -1
                elif held[0] == b:
                    want = held[1]
                else:
                    want = -2 - (3 * s + j)
                assert code == want, (seed, b, i, j, ids, code, want)
                # what the record names is what the Detector's slot holds
                if code >= 0:
                    assert code <= i and (b, code) == held
                elif code <= -2:
                    assert device_ring[-2 - code] == held
        for i, r in enumerate(plan):
            if r.commit >= 0:
                device_ring[r.commit] = (b, i)
        assert fi == ref.index and seen == ref.seen, (seed, b)


@pytest.mark.parametrize("seed", range(40))
def test_plan_equals_the_detector_ring(seed):
    rng = np.random.default_rng(seed)
    max_streams = int(rng.integers(1, 9))
    batches = []
    for _ in range(int(rng.integers(1, 7))):
        n = int(rng.integers(1, 17))
        active = int(rng.integers(1, max_streams + 1))  # streams >= active never appear in this list
        ids = [int(v) for v in rng.integers(0, active, n)]
        resets = [int(v) for v in rng.choice(max_streams, int(rng.integers(0, 3)))] if rng.random() < .4 else []
        batches.append((ids, resets))
    _run(max_streams, batches, seed)


def test_plan_of_one_stream_repeated_and_of_fresh_streams():
    # one stream five times in one list: slots 0,1,2,0,1; only the last writer of a slot commits
    plan, fi, seen = _lib.stream_plan([2] * 5, 4, [0] * 4, [0] * 4)
    assert [list(r.src) for r in plan] == [[0, -1, -1], [0, 1, -1], [0, 1, 2], [3, 1, 2], [3, 4, 2]]
    assert [r.commit for r in plan] == [-1, -1, 8, 6, 7]
    assert fi == [0, 0, 2, 0] and seen == [0, 0, 3, 0]
    # the next list reads the committed rows
    plan, fi, seen = _lib.stream_plan([2], 4, fi, seen)
    assert list(plan[0].src) == [-2 - 6, -2 - 7, 0] and plan[0].commit == 8
    # a stream reset by its counters reads zeros again, another one keeps its ring
    plan, _, _ = _lib.stream_plan([2, 1], 4, [0, 0, 0, 0], [0, 0, 0, 0])
    assert list(plan[0].src) == [0, -1, -1] and list(plan[1].src) == [1, -1, -1]


def test_plan_refuses_a_bad_id_and_changes_nothing():
    lib = _lib.load()
    C = _lib.C
    for bad in ([0, 3], [-1], [1, 2, 7]):
        fi = (C.c_int * 3)(1, 2, 0)
        seen = (C.c_int * 3)(3, 3, 0)
        plan = (_lib.StreamSrc * 3)()
        ids = (C.c_int * len(bad))(*bad)
        assert lib.y2_stream_plan(len(bad), ids, 3, fi, seen, plan) != 0
        assert list(fi) == [1, 2, 0] and list(seen) == [3, 3, 0]
    assert lib.y2_stream_plan(0, (C.c_int * 1)(0), 3, (C.c_int * 3)(), (C.c_int * 3)(), (_lib.StreamSrc * 1)()) != 0


FRAMES = "[np.zeros((12, 16, 3), np.uint8)]"
CALLS = {
    "open": "dn.network_streams_open(net, 4)",
    "reset": "dn.network_stream_reset(net, 0)",
    "batch": f"dn.network_detect_streams(net, [0], {FRAMES}, .5, .4)",
    "submit": f"dn.network_detect_submit_streams(net, [0], {FRAMES}, .5, .4)",
    "submit_resident": "dn.network_detect_submit_streams_resident(net, [0], .5, .4)",
}


@pytest.mark.parametrize("call", sorted(CALLS))
def test_streams_without_a_device_plan_exit_through_error(tmp_path, call):
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
    assert "no device plan" in r.stderr, r.stderr[-2000:]
