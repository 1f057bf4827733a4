#!/usr/bin/env python
"""Developer tool (GPU box): cost of the video-streams path (network_detect_submit_streams: every frame decoded on the
3-frame mean of its stream) against the plain frame-list path on the same frames, for yolo-voc 416.

For 1, 8 and 64 streams (frame i of a batch belongs to stream i % streams) and for frames at the network size and of
500x375, in one process:
  - end-to-end images/s with two batches in flight (submit / wait, host clock, pageable frames), the streams path and
    network_detect_submit_frame_list alternated round by round on the same frames;
  - the mean and commit kernels alone (y2_stream_mean, y2_stream_commit) on a steady state plan (every ring slot
    written): their device durations from torch.profiler (CUDA activities) over many launches, after the end-to-end
    rounds, so the profiler slows none of them.  A launch from Python through ctypes takes longer than these kernels
    run, so timing a row of launches with events would measure the host.  With their bytes, n * outputs * 4 *
    (3 read + 1 written) for the mean and 2 * 4 * outputs per committed row, the rate those bytes give.  The working
    set (a few to 16 MB) fits the L2, so the rates are for L2-resident operands, as in the pipeline, where the
    forward pass has just written the region output.
Prints one JSON line with the device name and power limit.

    python tools/streams_bench.py --batch 64 --steps 30 --out profiles/streams_bench_yolo-voc.json
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
from torch.profiler import ProfilerActivity, profile  # noqa: E402

from sr_object_detection_b200 import _lib, darknet as dn, synth  # noqa: E402

THRESH, NMS, MAX_DET = 0.02, 0.4, 256
STREAMS = (1, 8, 64)
SIZES = ((416, 416), (500, 375))


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
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the two paths per case")
    ap.add_argument("--launches", type=int, default=200, help="kernel launches per profiled timing")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if min(args.batch, args.steps, args.rounds, args.launches) < 1:
        ap.error("--batch, --steps, --rounds and --launches must be >= 1")

    B = args.batch
    lib, klib = dn.lib(), _lib.load()
    tmp = Path(tempfile.mkdtemp(prefix="y2streams_"))
    text = synth.yolo_voc_cfg(batch=B, w=416, h=416)
    (tmp / "n.cfg").write_text(text)
    synth.write_weights(tmp / "n.weights", text, seed=1234)
    dn.set_gpu_index(0)
    lib.cuda_set_device(0)
    net = dn.parse_network_cfg(tmp / "n.cfg")
    dn.load_weights(net, tmp / "n.weights")
    outputs = dn.region_layer(net).outputs

    def pipelined_ms(submit, steps):
        """ms per batch with two batches in flight; ends in the wait for the last one"""
        submit()
        t0 = time.perf_counter()
        for _ in range(steps):
            submit()
            dn.network_detect_wait_n(net, B, MAX_DET)
        dn.network_detect_wait_n(net, B, MAX_DET)
        return (time.perf_counter() - t0) * 1e3 / (steps + 1)

    def kernel_ms(fn, kernel):
        """mean device duration of `kernel` over args.launches calls of fn"""
        for _ in range(10):
            fn()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.launches):
                fn()
            torch.cuda.synchronize()
        hits = [e for e in prof.key_averages() if kernel in e.key]
        if len(hits) != 1 or hits[0].count != args.launches:
            raise RuntimeError(f"profiler saw {[(e.key, e.count) for e in hits]} for {kernel}")
        return hits[0].device_time_total / hits[0].count / 1e3

    rng = np.random.default_rng(7)
    cases, kernel_runs = [], []
    for w, h in SIZES:
        frames = [rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8) for _ in range(B)]
        for n_streams in STREAMS:
            ids = [i % n_streams for i in range(B)]
            dn.network_streams_open(net, n_streams)

            def plain():
                dn.network_detect_submit_frame_list(net, frames, THRESH, NMS, MAX_DET)

            def streams():
                dn.network_detect_submit_streams(net, ids, frames, THRESH, NMS, MAX_DET)

            pipelined_ms(plain, args.warmup)
            pipelined_ms(streams, args.warmup)
            t_plain, t_streams = [], []
            for _ in range(args.rounds):
                t_plain.append(pipelined_ms(plain, args.steps))
                t_streams.append(pipelined_ms(streams, args.steps))
            mp, ms_ = statistics.median(t_plain), statistics.median(t_streams)
            cases.append({
                "frame": f"{w}x{h}", "streams": n_streams,
                "plain_ms_per_batch": round(mp, 4), "streams_ms_per_batch": round(ms_, 4),
                "plain_images_per_s": round(B * 1e3 / mp, 1), "streams_images_per_s": round(B * 1e3 / ms_, 1),
                "streams_over_plain_time": round(ms_ / mp, 4),
                "plain_rounds_ms": [round(t, 4) for t in t_plain], "streams_rounds_ms": [round(t, 4) for t in t_streams],
            })
            print(json.dumps(cases[-1]), file=sys.stderr, flush=True)
    dn.free_network(net)

    for n_streams in STREAMS:  # the kernels alone, steady state: every slot of every stream written before the batch
        ids = [i % n_streams for i in range(B)]
        plan, _, _ = _lib.stream_plan(ids, n_streams, [0] * n_streams, [3] * n_streams)
        table = np.frombuffer((_lib.StreamSrc * B)(*plan), np.int32).copy()
        committed = sum(r.commit >= 0 for r in plan)
        bufs = [dn._DevBuf(B * outputs * 4), dn._DevBuf(3 * n_streams * outputs * 4),
                dn._DevBuf(table.nbytes, table), dn._DevBuf(B * outputs * 4)]
        out, ring, tab, mean = (b.ptr for b in bufs)
        _lib.check(klib.y2_memset(out, 0, B * outputs * 4, None))
        _lib.check(klib.y2_memset(ring, 0, 3 * n_streams * outputs * 4, None))
        t_mean = kernel_ms(lambda: _lib.check(klib.y2_stream_mean(out, ring, tab, B, outputs, mean, None)),
                           "stream_mean_kernel")
        t_commit = kernel_ms(lambda: _lib.check(klib.y2_stream_commit(out, ring, tab, B, outputs, None)),
                             "stream_commit_kernel")
        for b in bufs:
            b.free()
        mean_bytes, commit_bytes = B * outputs * 4 * 4, committed * 2 * 4 * outputs
        step = min(c["plain_ms_per_batch"] for c in cases if c["streams"] == n_streams)
        kernel_runs.append({
            "streams": n_streams, "mean_kernel_us": round(t_mean * 1e3, 3), "mean_bytes": mean_bytes,
            "mean_GBps": round(mean_bytes / (t_mean * 1e-3) / 1e9, 1),
            "commit_kernel_us": round(t_commit * 1e3, 3), "committed_rows": committed, "commit_bytes": commit_bytes,
            "commit_GBps": round(commit_bytes / (t_commit * 1e-3) / 1e9, 1),
            "kernels_share_of_plain_batch": round((t_mean + t_commit) / step, 5),
        })
        print(json.dumps(kernel_runs[-1]), file=sys.stderr, flush=True)
    name, power = device_info()
    res = {"tool": "streams_bench", "cfg": "yolo-voc", "side": 416, "batch": B, "outputs": outputs,
           "steps": args.steps, "rounds": args.rounds, "launches": args.launches, "device": name,
           "power_limit": power, "cases": cases, "kernels": kernel_runs}
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
