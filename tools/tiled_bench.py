#!/usr/bin/env python
"""Developer tool (GPU box): throughput of tiled detection (network_detect_submit_tiled_descs) on 1920x1080 NV12 frames
for yolo-voc 416 at batch 64 (synthetic weights, the head scaled as smoke() scales it), host and device frames, for
three tilings:
  1x1      one tile per frame, no whole frame (the plain descriptor path):  64 frames a batch
  2x2o64f  2x2 grid, overlap 64, plus the whole frame: 5 tiles a frame,     12 frames a batch (60 images)
  3x2o64f  3x2 grid, overlap 64, plus the whole frame: 7 tiles a frame,      9 frames a batch (63 images)

Prints one JSON line with the device name and power limit and, per tiling:
  - frames/s and network images/s end to end with two batches in flight (submit / wait, host clock; host frames are
    passed as numpy arrays, so their staging copy is included);
  - the forward-only time of a batch (submit_resident / wait);
  - the merge tail (y2_tile_map + y2_tile_nms + y2_tile_collect) by CUDA events on the batch's own region output, at
    thresh .24 and at a low thresh, with the candidate counts of the busiest (frame, class) pair and the tail's share
    of the end-to-end batch time.
Each end-to-end rate is the median of `--repeats` runs, the kinds alternated.

    python tools/tiled_bench.py --steps 20 --out profiles/tiled_bench.json
"""
import argparse
import ctypes as C
import json
import sys
import tempfile
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent))
import numpy as np  # noqa: E402

from frame_list_bench import device_info  # noqa: E402
from sr_object_detection_b200 import _lib, darknet as dn, synth  # noqa: E402

FW, FH, SIDE, B = 1920, 1080, 416, 64
NMS, MAX_DET = 0.45, 256
THRESH, LOW_THRESH = 0.24, 0.005
HEAD_GAIN = 30.0  # synthetic head weights scaled as smoke() does, so that some boxes clear .24 (plain random: none)
TILINGS = {"1x1": (1, 1, 0, 0), "2x2o64f": (2, 2, 64, 1), "3x2o64f": (3, 2, 64, 1)}
KINDS = ["host_nv12", "device_nv12"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if args.steps < 1 or args.repeats < 1:
        ap.error("--steps and --repeats must be >= 1")
    klib = _lib.load()
    lib = dn.lib()
    dn.set_gpu_index(0)
    lib.cuda_set_device(0)
    sig = {"y2_region_boxes_counted": (C.c_int, [C.c_void_p] * 4 + [C.c_int] * 5 + [C.c_float] * 3 + [C.c_int] * 3 +
                                       [C.c_void_p] * 2 + [C.c_int, C.c_void_p, C.c_void_p])}
    for k, (res, argt) in sig.items():
        getattr(klib, k).restype, getattr(klib, k).argtypes = res, argt
    name, power = device_info()

    tmp = Path(tempfile.mkdtemp(prefix="y2tl_"))
    text = synth.yolo_voc_cfg(batch=B, w=SIDE, h=SIDE)
    (tmp / "n.cfg").write_text(text)
    synth.write_weights(tmp / "n.weights", text, seed=1234, head_gain=HEAD_GAIN)
    net = dn.parse_network_cfg(tmp / "n.cfg")
    dn.load_weights(net, tmp / "n.weights")
    stream = C.c_void_p(lib.network_stream(net))
    l = dn.region_layer(net)
    total, classes = l.w * l.h * l.n, l.classes

    rng = np.random.default_rng(2024)
    host = [rng.integers(0, 256, size=(FH * 3 // 2, FW), dtype=np.uint8) for _ in range(B)]
    per = host[0].nbytes
    dev = C.c_void_p()
    _lib.check(klib.y2_malloc(C.byref(dev), per * B))
    for i, f in enumerate(host):
        _lib.check(klib.y2_memcpy_h2d(dev.value + i * per, f.ctypes.data, per, None))
    _lib.check(klib.y2_stream_sync(None))
    host_descs = [dn.frame_desc(f, dn.FRAME_NV12) for f in host]
    dev_descs = []
    for i in range(B):
        d = dn.FrameDesc()
        d.data, d.w, d.h, d.format, d.on_device = dev.value + i * per, FW, FH, dn.FRAME_NV12, 1
        dev_descs.append(d)

    dets = (dn.Detection * (B * MAX_DET))()
    counts = (C.c_int * B)()

    def wait():
        lib.network_detect_wait(net, dets, counts, MAX_DET)

    def host_ms(submit, steps):
        """two batches in flight; ends in the wait for the last batch, i.e. after the device finished"""
        def run(k):
            submit()
            for _ in range(1, k):
                submit()
                wait()
            wait()
        run(args.warmup)
        t0 = time.perf_counter()
        run(steps)
        return (time.perf_counter() - t0) * 1e3 / steps

    ev = [C.c_void_p() for _ in range(4)]
    for e in ev:
        _lib.check(klib.y2_event_create(C.byref(e)))

    def elapsed(a, b):
        ms = C.c_float()
        _lib.check(klib.y2_event_elapsed_ms(a, b, C.byref(ms)))
        return ms.value

    x = synth.images(B, 3, SIDE, SIDE, seed=1)
    for s in (0, 1):
        _lib.check(klib.y2_memcpy_h2d(lib.network_pipeline_input_device(net, s), x.ctypes.data, x.nbytes, None))
    _lib.check(klib.y2_stream_sync(None))

    res = {"tool": "tiled_bench", "network": f"yolo-voc 416 (synthetic weights, head_gain {HEAD_GAIN})", "batch": B,
           "frame": f"{FW}x{FH}", "format": "NV12", "nms": NMS, "steps": args.steps, "repeats": args.repeats,
           "device": name, "power_limit": power}
    plans = {}
    for tname, tiling in TILINGS.items():
        per_frame = tiling[3] + tiling[0] * tiling[1]
        n = B // per_frame
        arrs = {"host_nv12": dn._descs_arg(host_descs[:n]), "device_nv12": dn._descs_arg(dev_descs[:n])}
        t = dn.Tiling(*tiling)
        plans[tname] = (n, per_frame, arrs, t)

    def submit_fn(tname, kind):
        n, _, arrs, t = plans[tname]
        cnt, arr = arrs[kind]
        return lambda: lib.network_detect_submit_tiled_descs(net, cnt, arr, C.byref(t), None, THRESH, NMS, MAX_DET)

    ms = {tn: {k: [] for k in KINDS} for tn in TILINGS}
    resident = []
    for _ in range(args.repeats):
        for tn in TILINGS:
            for k in KINDS:
                ms[tn][k].append(host_ms(submit_fn(tn, k), args.steps))
        resident.append(host_ms(lambda: lib.network_detect_submit_resident(net, THRESH, NMS, MAX_DET), args.steps))
    resident_ms = float(np.median(resident))
    res["forward_only_ms_per_batch"] = round(resident_ms, 4)
    res["forward_only_runs_ms"] = [round(v, 4) for v in resident]

    # the merge tail on each tiling's own region output (device frames), timed alone
    boxes_b, probs_b, pred_b, cnt_b, det_b, dcnt_b, tab_b, ws_b = (C.c_void_p() for _ in range(8))
    outputs = l.outputs
    _lib.check(klib.y2_malloc(C.byref(boxes_b), B * total * 16))
    _lib.check(klib.y2_malloc(C.byref(probs_b), B * total * classes * 4))
    _lib.check(klib.y2_malloc(C.byref(pred_b), B * outputs * 4))
    _lib.check(klib.y2_malloc(C.byref(cnt_b), B * classes * 4))
    _lib.check(klib.y2_memset(cnt_b, 0, B * classes * 4, None))
    _lib.check(klib.y2_malloc(C.byref(det_b), B * MAX_DET * C.sizeof(dn.Detection)))
    _lib.check(klib.y2_malloc(C.byref(dcnt_b), B * 4))
    biases = np.ctypeslib.as_array(l.biases, shape=(2 * l.n,)).astype(np.float32)
    bias_b = C.c_void_p()
    _lib.check(klib.y2_malloc(C.byref(bias_b), biases.nbytes))
    _lib.check(klib.y2_memcpy_h2d(bias_b, biases.ctypes.data, biases.nbytes, None))
    ws_bytes = 0
    for tname, tiling in TILINGS.items():
        n, per_frame, arrs, t = plans[tname]
        cnt, arr = arrs["device_nv12"]
        lib.network_detect_batch_tiled_descs(net, cnt, arr, C.byref(t), None, THRESH, NMS, dets, counts, MAX_DET)
        out = dn.get_network_output_layer(net, net.n - 1)
        _lib.check(klib.y2_memcpy_h2d(pred_b, out.ctypes.data, out.nbytes, None))
        rc, lay, _, tiles, spans = _lib.tile_plan(dev_descs[:n], t, SIDE, SIDE, B)
        tab = bytes((_lib.Tile * len(tiles))(*tiles)) + bytes((_lib.TileSpan * len(spans))(*spans))
        tb = np.frombuffer(tab, np.uint8).copy()
        _lib.check(klib.y2_malloc(C.byref(tab_b), tb.nbytes))
        _lib.check(klib.y2_memcpy_h2d(tab_b, tb.ctypes.data, tb.nbytes, None))
        tiles_d, spans_d = tab_b.value, tab_b.value + len(tiles) * C.sizeof(_lib.Tile)
        T = lay.n_tiles
        need = klib.y2_tile_nms_ws_bytes(n, classes, per_frame * total)
        if need > ws_bytes:
            if ws_b.value:
                klib.y2_free(ws_b)
            _lib.check(klib.y2_malloc(C.byref(ws_b), need))
            ws_bytes = need
        _lib.check(klib.y2_stream_sync(None))
        tail = {}
        for label, thresh in (("thresh_0.24", THRESH), (f"thresh_{LOW_THRESH}", LOW_THRESH)):
            def decode():
                _lib.check(klib.y2_region_boxes_counted(pred_b, bias_b, boxes_b, probs_b, T, l.w, l.h, l.n, classes,
                                                        1.0, 1.0, thresh, 0, l.classfix, 0, None, None, 0, cnt_b,
                                                        stream))

            def merge():
                _lib.check(klib.y2_tile_map(boxes_b, tiles_d, T, total, stream))
                _lib.check(klib.y2_tile_nms(boxes_b, probs_b, cnt_b, spans_d, n, total, classes, per_frame, NMS, ws_b,
                                            ws_bytes, stream))
                _lib.check(klib.y2_tile_collect(boxes_b, probs_b, spans_d, n, total, classes, thresh, det_b, dcnt_b,
                                                MAX_DET, cnt_b, stream))
            decode()
            counts_h = np.zeros((T, classes), np.int32)
            _lib.check(klib.y2_memcpy_d2h(counts_h.ctypes.data, cnt_b, counts_h.nbytes, stream))
            _lib.check(klib.y2_stream_sync(stream))
            per_pair = counts_h.reshape(n, per_frame, classes).sum(axis=1)
            merge()
            for _ in range(args.warmup):
                decode()
                merge()
            tail_ms = dec_ms = 0.0
            for _ in range(args.steps):
                _lib.check(klib.y2_event_record(ev[0], stream))
                decode()
                _lib.check(klib.y2_event_record(ev[1], stream))
                merge()
                _lib.check(klib.y2_event_record(ev[2], stream))
                _lib.check(klib.y2_event_sync(ev[2]))
                dec_ms += elapsed(ev[0], ev[1])
                tail_ms += elapsed(ev[1], ev[2])
            tail_ms /= args.steps
            dec_ms /= args.steps
            batch_ms = float(np.median(ms[tname]["device_nv12"]))
            tail[label] = {"merge_ms": round(tail_ms, 4), "decode_ms": round(dec_ms, 4),
                           "merge_share_of_batch": round(tail_ms / batch_ms, 4),
                           "merge_share_of_forward": round(tail_ms / resident_ms, 4),
                           "candidates_busiest_pair": int(per_pair.max()),
                           "candidates_mean_pair": round(float(per_pair.mean()), 1),
                           "pairs_with_2_or_more": int((per_pair >= 2).sum())}
        klib.y2_free(tab_b)
        med = {k: float(np.median(v)) for k, v in ms[tname].items()}
        res[tname] = {
            "tiling": dict(zip(("cols", "rows", "overlap", "full"), tiling)), "frames_per_batch": n,
            "images_per_batch": n * per_frame, "union_boxes_per_frame": per_frame * total,
            "frames_per_s": {k: round(n * 1e3 / v, 1) for k, v in med.items()},
            "images_per_s": {k: round(n * per_frame * 1e3 / v, 1) for k, v in med.items()},
            "ms_per_batch": {k: round(v, 4) for k, v in med.items()},
            "runs_ms_per_batch": {k: [round(x, 4) for x in v] for k, v in ms[tname].items()},
            "merge_tail": tail,
        }
    for p in (boxes_b, probs_b, pred_b, cnt_b, det_b, dcnt_b, bias_b, ws_b, dev):
        if p.value:
            klib.y2_free(p)
    for e in ev:
        klib.y2_event_destroy(e)
    dn.free_network(net)
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
