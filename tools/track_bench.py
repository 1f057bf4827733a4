#!/usr/bin/env python
"""Developer tool (GPU box): cost of tracking video streams (network_detect_submit_streams_tracked) for yolo-voc 416 at
batch 64 with 64 streams (frame i of a batch belongs to stream i), in one process:
  - the streams step with and without tracking, both decoded on the 3-frame means: ms per batch with two batches in
    flight (submit / wait, host clock, pageable 416x416 frames), the two alternated round by round on the same frames;
  - the tracking kernel alone (y2_stream_track) on a full history (frames_story 6, every frame of every stream
    holding D boxes, D = 10, 100 and 845, the same boxes each frame so that every old box matches): its device time
    from CUDA events around a row of launches queued behind a device-side sleep, so that the host's launch rate is not
    what is timed.
Prints one JSON line with the device name and power limit.

    python tools/track_bench.py --steps 30 --out profiles/track_bench_yolo-voc.json
"""
import argparse
import json
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from sr_object_detection_b200 import _lib, darknet as dn, synth  # noqa: E402

THRESH, NMS, MAX_DET, STORY = 0.02, 0.4, 256, 6
DETS = (10, 100, 845)


def device_info():
    r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, _, power = r.stdout.strip().partition(", ")
    return name or None, power or None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--steps", type=int, default=30, help="batches per timed round")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the two paths")
    ap.add_argument("--launches", type=int, default=50, help="kernel launches per event-timed row")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if min(args.batch, args.steps, args.rounds, args.launches) < 1:
        ap.error("--batch, --steps, --rounds and --launches must be >= 1")

    B = args.batch
    lib, klib = dn.lib(), _lib.load()
    tmp = Path(tempfile.mkdtemp(prefix="y2track_"))
    text = synth.yolo_voc_cfg(batch=B, w=416, h=416)
    (tmp / "n.cfg").write_text(text)
    synth.write_weights(tmp / "n.weights", text, seed=1234)
    dn.set_gpu_index(0)
    lib.cuda_set_device(0)
    net = dn.parse_network_cfg(tmp / "n.cfg")
    dn.load_weights(net, tmp / "n.weights")
    l = dn.region_layer(net)
    total, classes = l.w * l.h * l.n, l.classes

    rng = np.random.default_rng(7)
    frames = [rng.integers(0, 256, size=(416, 416, 3), dtype=np.uint8) for _ in range(B)]
    ids = list(range(B))
    dn.network_streams_open(net, B)
    dn.network_streams_track(net, STORY)

    def pipelined_ms(submit, wait, steps):
        """ms per batch with two batches in flight; ends in the wait for the last one"""
        submit()
        t0 = time.perf_counter()
        for _ in range(steps):
            submit()
            wait()
        wait()
        return (time.perf_counter() - t0) * 1e3 / (steps + 1)

    def untracked():
        dn.network_detect_submit_streams(net, ids, frames, THRESH, NMS, MAX_DET)

    def tracked():
        dn.network_detect_submit_streams_tracked(net, ids, frames, THRESH, NMS, True, MAX_DET)

    def wait_untracked():
        dn.network_detect_wait_n(net, B, MAX_DET)

    def wait_tracked():
        dn.network_detect_wait_tracked(net, B, MAX_DET)

    pipelined_ms(untracked, wait_untracked, args.warmup)
    pipelined_ms(tracked, wait_tracked, args.warmup)
    t_plain, t_track = [], []
    for _ in range(args.rounds):
        t_plain.append(pipelined_ms(untracked, wait_untracked, args.steps))
        t_track.append(pipelined_ms(tracked, wait_tracked, args.steps))
    tracked()
    _, counts = dn.network_detect_wait_tracked(net, B, MAX_DET)
    mu, mt = statistics.median(t_plain), statistics.median(t_track)
    step = {"frame": "416x416", "streams": B, "frames_story": STORY,
            "untracked_ms_per_batch": round(mu, 4), "tracked_ms_per_batch": round(mt, 4),
            "tracking_overhead_ms_per_batch": round(mt - mu, 4),
            "untracked_rounds_ms": [round(t, 4) for t in t_plain], "tracked_rounds_ms": [round(t, 4) for t in t_track],
            "detections_per_frame_mean": round(float(np.mean(counts)), 1)}
    print(json.dumps(step), file=sys.stderr, flush=True)
    dn.free_network(net)

    kernels = []
    for D in DETS:  # the kernel alone, one frame per stream, every stream's history full
        det = np.zeros((B, total, 7), np.float32)
        box = rng.uniform(.05, .95, (B, D, 4)).astype(np.float32)
        box[..., 2:] *= .3
        det[:, :D, :4] = box
        det[:, :D, 4] = .5
        det = det.view(np.int32)
        det[:, :D, 5] = rng.integers(0, classes, (B, D))
        det[:, :, 6] = np.arange(total)
        d_det = torch.from_numpy(det.reshape(-1).copy()).cuda()
        d_cnt = torch.full((B,), D, dtype=torch.int32, device="cuda")
        hist = torch.zeros(B * STORY * total * 7, dtype=torch.int32, device="cuda")
        hist_cnt = torch.zeros(B * STORY, dtype=torch.int32, device="cuda")
        next_id = torch.zeros(B * classes, dtype=torch.int32, device="cuda")
        out = torch.zeros(B * total * 7, dtype=torch.int32, device="cuda")
        head, length, restart = [0] * B, [0] * B, [1] * B
        sizes = [(416, 416)] * B

        def launch(recs, offsets):
            _lib.check(klib.y2_stream_track(d_det.data_ptr(), total, d_cnt.data_ptr(), recs.data_ptr(),
                                            offsets.data_ptr(), B, total, classes, STORY, hist.data_ptr(),
                                            hist_cnt.data_ptr(), next_id.data_ptr(), out.data_ptr(), total, None),
                            "y2_stream_track")

        def plan():
            nonlocal head, length, restart
            recs, offsets, head, length, restart = _lib.track_plan(ids, sizes, B, STORY, head, length, restart)
            return (torch.from_numpy(np.frombuffer((_lib.TrackImg * B)(*recs), np.uint8).copy()).cuda(),
                    torch.tensor(offsets, dtype=torch.int32, device="cuda"))

        for _ in range(STORY):  # fill every history
            launch(*plan())
        steady = plan()  # a full history from here on; each launch rewrites the same slot with the same boxes
        launch(*steady)
        torch.cuda.synchronize()
        times = []
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda._sleep(50_000_000)
            e0.record()
            for _ in range(args.launches):
                launch(*steady)
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) / args.launches)
        kernels.append({"detections_per_frame": D, "frames_story": STORY, "streams": B,
                        "history_boxes_per_frame": STORY * D, "kernel_us": round(statistics.median(times) * 1e3, 2),
                        "rows_us": [round(t * 1e3, 2) for t in times]})
        print(json.dumps(kernels[-1]), file=sys.stderr, flush=True)
    name, power = device_info()
    res = {"tool": "track_bench", "cfg": "yolo-voc", "side": 416, "batch": B, "total": total, "steps": args.steps,
           "rounds": args.rounds, "launches": args.launches, "device": name, "power_limit": power, "step": step,
           "kernels": kernels}
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
