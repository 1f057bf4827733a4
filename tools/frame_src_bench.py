#!/usr/bin/env python
"""Developer tool (GPU box): throughput of the frame-descriptor entries (network_*_submit_frame_descs: RGB, BGR or NV12
frames in host or device memory, converted and resized or letterboxed on the device) on 1920x1080 frames, for
yolo-voc 416 (detection) and darknet19_448 (classification), against today's host-RGB frame list.

Prints one JSON line with the device name and power limit and, per network, for `batch` 1920x1080 frames:
  - end-to-end images/s with two batches in flight (submit / wait, host clock), the host frames already in the slots'
    pinned staging buffers: host RGB (network_*_submit_frame_list), host NV12, device RGB and device NV12 (descriptor
    entries; device frames read in place, only the record table is uploaded);
  - the forward-only rate (submit_resident / wait on the same network);
  - the host -> device ceiling of plain pinned cudaMemcpyAsync (CUDA events) and what it allows in RGB and NV12
    frames/s;
  - the conversion kernel alone per format (y2_frames_src_to_f32 on device frames, CUDA events) with touched bytes (the
    source rows the bilinear taps read, whole rows, plus the table and the fp32 output) and TB/s.
Each end-to-end rate is the median of `--repeats` runs, the kinds alternated.

    python tools/frame_src_bench.py --batch 64 --steps 30 --out profiles/frame_src_bench.json
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

from frame_list_bench import device_info, rows_read  # noqa: E402
from sr_object_detection_b200 import _lib, darknet as dn, synth  # noqa: E402

CFGS = {"yolo-voc": (synth.yolo_voc_cfg, 416, False), "darknet19_448": (synth.darknet19_448_cfg, 448, True)}
FW, FH = 1920, 1080
THRESH, NMS, MAX_DET, TOP = 0.02, 0.4, 256, 5
KINDS = ["host_rgb", "host_nv12", "device_rgb", "device_nv12"]


def run_cfg(cfg, args, klib):
    make_cfg, side, letterbox = CFGS[cfg]
    B = args.batch
    lib = dn.lib()
    tmp = Path(tempfile.mkdtemp(prefix="y2fs_"))
    text = make_cfg(batch=B, w=side, h=side)
    (tmp / "n.cfg").write_text(text)
    synth.write_weights(tmp / "n.weights", text, seed=1234)
    net = dn.parse_network_cfg(tmp / "n.cfg")
    dn.load_weights(net, tmp / "n.weights")
    stream = C.c_void_p(lib.network_stream(net))
    ev = [C.c_void_p(), C.c_void_p()]
    for e in ev:
        _lib.check(klib.y2_event_create(C.byref(e)))

    def event_ms(fn, steps):
        for _ in range(args.warmup):
            fn()
        _lib.check(klib.y2_event_record(ev[0], stream))
        for _ in range(steps):
            fn()
        _lib.check(klib.y2_event_record(ev[1], stream))
        _lib.check(klib.y2_event_sync(ev[1]))
        ms = C.c_float()
        _lib.check(klib.y2_event_elapsed_ms(ev[0], ev[1], C.byref(ms)))
        return ms.value / steps

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

    if letterbox:
        hits = (dn.ClassHit * (B * TOP))()

        def wait():
            lib.network_classify_wait(net, hits, TOP)

        def submit_list(a):
            lib.network_classify_submit_frame_list(net, *a, TOP)

        def submit_descs(n, arr):
            lib.network_classify_submit_frame_descs(net, n, arr, None, TOP)

        def submit_resident():
            lib.network_classify_submit_resident(net, TOP)
    else:
        dets = (dn.Detection * (B * MAX_DET))()
        counts = (C.c_int * B)()

        def wait():
            lib.network_detect_wait(net, dets, counts, MAX_DET)

        def submit_list(a):
            lib.network_detect_submit_frame_list(net, *a, THRESH, NMS, MAX_DET)

        def submit_descs(n, arr):
            lib.network_detect_submit_frame_descs(net, n, arr, None, THRESH, NMS, MAX_DET)

        def submit_resident():
            lib.network_detect_submit_resident(net, THRESH, NMS, MAX_DET)

    rng = np.random.default_rng(2024)
    rgb = [rng.integers(0, 256, size=(FH, FW, 3), dtype=np.uint8) for _ in range(B)]
    nv12 = [rng.integers(0, 256, size=(FH * 3 // 2, FW), dtype=np.uint8) for _ in range(B)]

    # host frames written in place in both slots' pinned buffers, built once per slot
    list_views, nv12_descs = [], []
    for s in (0, 1):
        vs = dn.network_pipeline_staging_frame_list(net, s, [(FW, FH)] * B)
        for v, f in zip(vs, rgb):
            v[...] = f
        list_views.append(dn._frame_list_args(vs))
    # the NV12 layout is smaller: the RGB list's buffer holds it and nothing moves.  Its frames overwrite the start of
    # the RGB ones; no rate here depends on the pixel values.
    for s in (0, 1):
        vs = dn.network_pipeline_staging_frame_descs(net, s, [dn.frame_desc(f, dn.FRAME_NV12) for f in nv12])
        for v, f in zip(vs, nv12):
            v[...] = f
        nv12_descs.append(dn._descs_arg([dn.frame_desc(v, dn.FRAME_NV12) for v in vs]))

    # device frames: one allocation per format, frames back to back
    dev = {}
    for fmt, frames in ((dn.FRAME_RGB24, rgb), (dn.FRAME_NV12, nv12)):
        per = frames[0].nbytes
        p = C.c_void_p()
        _lib.check(klib.y2_malloc(C.byref(p), per * B))
        for i, f in enumerate(frames):
            _lib.check(klib.y2_memcpy_h2d(p.value + i * per, f.ctypes.data, per, None))
        descs = []
        for i in range(B):
            d = dn.FrameDesc()
            d.data, d.w, d.h, d.format, d.on_device = p.value + i * per, FW, FH, fmt, 1
            descs.append(d)
        dev[fmt] = (p, dn._descs_arg(descs), descs)
    _lib.check(klib.y2_stream_sync(None))

    submit = {
        "host_rgb": lambda: submit_list(list_views[lib.network_pipeline_next_slot(net)]),
        "host_nv12": lambda: submit_descs(*nv12_descs[lib.network_pipeline_next_slot(net)]),
        "device_rgb": lambda: submit_descs(*dev[dn.FRAME_RGB24][1]),
        "device_nv12": lambda: submit_descs(*dev[dn.FRAME_NV12][1]),
    }
    x = synth.images(B, 3, side, side, seed=1)
    for s in (0, 1):
        _lib.check(klib.y2_memcpy_h2d(lib.network_pipeline_input_device(net, s), x.ctypes.data, x.nbytes, None))
    _lib.check(klib.y2_stream_sync(None))
    ms = {k: [] for k in KINDS + ["resident"]}
    for _ in range(args.repeats):
        for k in KINDS:
            ms[k].append(host_ms(submit[k], args.steps))
        ms["resident"].append(host_ms(submit_resident, args.steps))
    med = {k: float(np.median(v)) for k, v in ms.items()}

    # host -> device ceiling: one batch of RGB frames, pinned
    total = rgb[0].nbytes * B
    hbuf, dbuf = C.c_void_p(), C.c_void_p()
    _lib.check(klib.y2_host_alloc(C.byref(hbuf), total))
    _lib.check(klib.y2_malloc(C.byref(dbuf), total))
    h2d_ms = event_ms(lambda: _lib.check(klib.y2_memcpy_h2d(dbuf, hbuf, total, stream)), args.steps)
    h2d_gbps = total / (h2d_ms * 1e6)
    klib.y2_host_free(hbuf)
    klib.y2_free(dbuf)

    # the conversion kernel alone, device frames of each format
    kernel = {}
    out = C.c_void_p()
    out_bytes = B * 3 * side * side * 4
    _lib.check(klib.y2_malloc(C.byref(out), out_bytes))
    for name, fmt in (("rgb", dn.FRAME_RGB24), ("bgr", dn.FRAME_BGR24), ("nv12", dn.FRAME_NV12)):
        descs = dev[dn.FRAME_NV12 if fmt == dn.FRAME_NV12 else dn.FRAME_RGB24][2]
        for d in descs:
            d.format = fmt
        recs, _, _ = _lib.frame_desc_layout(descs, side, side, letterbox)
        tab = np.frombuffer((_lib.FrameSrc * B)(*recs), np.uint8).copy()
        dtab = C.c_void_p()
        _lib.check(klib.y2_malloc(C.byref(dtab), tab.nbytes))
        _lib.check(klib.y2_memcpy_h2d(dtab, tab.ctypes.data, tab.nbytes, None))
        _lib.check(klib.y2_stream_sync(None))
        k_ms = event_ms(lambda: _lib.check(klib.y2_frames_src_to_f32(dtab, B, out, B, side, side, stream)), args.steps)
        klib.y2_free(dtab)
        f = recs[0].win
        rows = rows_read(f)
        if fmt == dn.FRAME_NV12:
            ys = set()
            for r in range(f.new_h):
                iy = min(int(np.float32(r) * np.float32(f.h_scale)), f.src_h - 1)
                ys.add(iy >> 1)
                if not (r == f.new_h - 1 or f.src_h == 1):
                    ys.add(min(iy + 1, f.src_h - 1) >> 1)
            src_bytes = (rows + len(ys)) * FW
        else:
            src_bytes = rows * FW * 3
        touched = B * src_bytes + tab.nbytes + out_bytes
        kernel[name] = {"ms": round(k_ms, 4), "touched_bytes": touched,
                        "touched_TB_per_s": round(touched / (k_ms * 1e9), 3)}
    klib.y2_free(out)
    for p, _, _ in dev.values():
        klib.y2_free(p)
    for e in ev:
        klib.y2_event_destroy(e)
    dn.free_network(net)

    ips = {k: B * 1e3 / med[k] for k in med}
    return {
        "side": side, "batch": B, "letterbox": letterbox,
        "images_per_s": {k: round(v, 1) for k, v in ips.items()},
        "ms_per_step": {k: round(v, 4) for k, v in med.items()},
        "runs_ms_per_step": {k: [round(x, 4) for x in v] for k, v in ms.items()},
        "host_nv12_over_host_rgb": round(ips["host_nv12"] / ips["host_rgb"], 4),
        "device_nv12_over_resident": round(ips["device_nv12"] / ips["resident"], 4),
        "device_rgb_over_resident": round(ips["device_rgb"] / ips["resident"], 4),
        "h2d_ceiling": {"GB_per_s": round(h2d_gbps, 2), "rgb_frames_per_s": round(h2d_gbps * 1e9 / (FW * FH * 3), 1),
                        "nv12_frames_per_s": round(h2d_gbps * 1e9 / (FW * FH * 3 // 2), 1)},
        "kernel": kernel,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cfg", choices=sorted(CFGS), action="append", help="default: both")
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if args.steps < 1 or args.batch < 1 or args.repeats < 1:
        ap.error("--steps, --batch and --repeats must be >= 1")
    klib = _lib.load()
    dn.lib()
    dn.set_gpu_index(0)
    dn.lib().cuda_set_device(0)
    name, power = device_info()
    res = {"tool": "frame_src_bench", "frame": f"{FW}x{FH}", "steps": args.steps, "repeats": args.repeats,
           "device": name, "power_limit": power}
    for cfg in args.cfg or sorted(CFGS, reverse=True):
        res[cfg] = run_cfg(cfg, args, klib)
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
