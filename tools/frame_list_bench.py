#!/usr/bin/env python
"""Developer tool (GPU box): throughput of frame lists (network_*_frame_list: frames of their own sizes in one batch,
resized or letterboxed on the device) for yolo-voc 416 (detection) or darknet19_448 (classification).

Prints one JSON line with the device name and power limit and, for a seeded list of `batch` frames drawn from a size
mix (voc: 500x375, 375x500, 500x333, 353x500, 640x480; camera: 1920x1080, 1280x720, 640x480):
  - end-to-end images/s with two batches in flight (submit_frame_list / wait, host clock), with the frames already in
    the slots' pinned staging buffers and from pageable arrays (one host copy per frame);
  - the device-resident rate (submit_resident / wait on the same network) and the host -> device ceiling of plain
    pinned cudaMemcpyAsync of the packed list (CUDA events), and the bound min(resident, ceiling / mean frame bytes);
  - the conversion kernel alone (y2_frames_u8_to_f32, CUDA events) with nominal bytes (every frame byte, the table and
    the fp32 output) and touched bytes (the source rows the bilinear taps read, whole rows, plus the output);
  - a list of 1920x1080 frames against network_detect_submit_frames / network_classify_submit_frames at that size,
    both staged, alternated;
  - the uniform conversion entries (y2_letterbox_u8_to_f32 / y2_resize_u8_to_f32) on 448x448 -> 448 letterbox,
    500x375 -> 448 letterbox and 1920x1080 -> 416 resize, and, with --baseline-lib, the same entries of another build
    of the library (e.g. the commit before the frame-list kernel) alternated with them in this process;
  - the host chain the entries replace: host resize_image (letterbox_image) per frame + network_detect_batch
    (network_classify_batch).

    python tools/frame_list_bench.py --cfg yolo-voc --mix voc --batch 64 --steps 30 --out profiles/x.json
"""
import argparse
import ctypes as C
import json
import subprocess
import sys
import tempfile
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np  # noqa: E402

from sr_object_detection_b200 import _lib, darknet as dn, synth  # noqa: E402

CFGS = {"yolo-voc": (synth.yolo_voc_cfg, 416, False), "darknet19_448": (synth.darknet19_448_cfg, 448, True)}
MIXES = {"voc": [(500, 375), (375, 500), (500, 333), (353, 500), (640, 480)],
         "camera": [(1920, 1080), (1280, 720), (640, 480)]}
UNIFORM = [((448, 448), 448, True), ((500, 375), 448, True), ((1920, 1080), 416, False)]
THRESH, NMS, MAX_DET, TOP = 0.02, 0.4, 256, 5


def device_info():
    r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, _, power = r.stdout.strip().partition(", ")
    return name or None, power or None


def rows_read(f):
    """source rows the kernel's vertical taps read for one frame's window (resize_image's y pass in float32)"""
    if f.new_w <= 0 or f.new_h <= 0:
        return 0
    rows = set()
    for r in range(f.new_h):
        iy = min(int(np.float32(r) * np.float32(f.h_scale)), f.src_h - 1)
        rows.add(iy)
        if not (r == f.new_h - 1 or f.src_h == 1):
            rows.add(min(iy + 1, f.src_h - 1))
    return len(rows)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cfg", choices=sorted(CFGS), default="yolo-voc")
    ap.add_argument("--mix", choices=sorted(MIXES), default="voc")
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--host-steps", type=int, default=2, help="batches through the host chain")
    ap.add_argument("--baseline-lib", help="another build of libyolo2_b200.so whose uniform conversion entries are "
                                           "timed alternately with this build's")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if args.steps < 1 or args.batch < 1 or args.host_steps < 1:
        ap.error("--steps, --batch and --host-steps must be >= 1")

    make_cfg, side, letterbox = CFGS[args.cfg]
    B = args.batch
    lib = dn.lib()
    klib = _lib.load()
    base = C.CDLL(args.baseline_lib, mode=C.RTLD_LOCAL) if args.baseline_lib else None
    for L in (klib, base) if base else (klib,):
        for name in ("y2_resize_u8_to_f32", "y2_letterbox_u8_to_f32"):
            getattr(L, name).restype = C.c_int
            getattr(L, name).argtypes = [C.c_void_p, C.c_void_p] + [C.c_int] * 5 + [C.c_void_p]
    tmp = Path(tempfile.mkdtemp(prefix="y2fl_"))
    text = make_cfg(batch=B, w=side, h=side)
    (tmp / "n.cfg").write_text(text)
    synth.write_weights(tmp / "n.weights", text, seed=1234)
    dn.set_gpu_index(0)
    lib.cuda_set_device(0)
    net = dn.parse_network_cfg(tmp / "n.cfg")
    dn.load_weights(net, tmp / "n.weights")
    stream = C.c_void_p(lib.network_stream(net))
    ev = [C.c_void_p(), C.c_void_p()]
    for e in ev:
        _lib.check(klib.y2_event_create(C.byref(e)))

    def event_ms(fn, steps, on=stream):
        for _ in range(args.warmup):
            fn()
        _lib.check(klib.y2_event_record(ev[0], on))
        for _ in range(steps):
            fn()
        _lib.check(klib.y2_event_record(ev[1], on))
        _lib.check(klib.y2_event_sync(ev[1]))
        ms = C.c_float()
        _lib.check(klib.y2_event_elapsed_ms(ev[0], ev[1], C.byref(ms)))
        return ms.value / steps

    def host_ms(fn, steps):
        """fn(steps) ends in a wait for its last batch, i.e. after the device finished"""
        fn(args.warmup)
        t0 = time.perf_counter()
        fn(steps)
        return (time.perf_counter() - t0) * 1e3 / steps

    if letterbox:
        hits = (dn.ClassHit * (B * TOP))()

        def submit_list(a):
            lib.network_classify_submit_frame_list(net, *a, TOP)

        def wait():
            lib.network_classify_wait(net, hits, TOP)

        def submit_resident():
            lib.network_classify_submit_resident(net, TOP)

        def submit_frames(p, fw, fh):
            lib.network_classify_submit_frames(net, p, fw, fh, TOP)
    else:
        dets = (dn.Detection * (B * MAX_DET))()
        counts = (C.c_int * B)()

        def submit_list(a):
            lib.network_detect_submit_frame_list(net, *a, THRESH, NMS, MAX_DET)

        def wait():
            lib.network_detect_wait(net, dets, counts, MAX_DET)

        def submit_resident():
            lib.network_detect_submit_resident(net, THRESH, NMS, MAX_DET)

        def submit_frames(p, fw, fh):
            lib.network_detect_submit_frames(net, p, fw, fh, THRESH, NMS, MAX_DET)

    def two_in_flight(submit):
        def run(steps):
            submit()
            for _ in range(1, steps):
                submit()
                wait()
            wait()
        return run

    # device-resident rate
    x = synth.images(B, 3, side, side, seed=1)
    for s in (0, 1):
        _lib.check(klib.y2_memcpy_h2d(lib.network_pipeline_input_device(net, s), x.ctypes.data, x.nbytes, None))
    _lib.check(klib.y2_stream_sync(None))
    resident_ms = host_ms(two_in_flight(submit_resident), args.steps)

    # the mixed list, staged in both slots and as pageable arrays
    rng = np.random.default_rng(2024)
    mix = MIXES[args.mix]
    sizes = [mix[i] for i in rng.integers(0, len(mix), B)]
    frames = [rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8) for w, h in sizes]
    frame_bytes = sum(f.nbytes for f in frames)

    def staged_views(frs):
        views = []
        for s in (0, 1):
            vs = dn.network_pipeline_staging_frame_list(net, s, [(f.shape[1], f.shape[0]) for f in frs])
            for v, f in zip(vs, frs):
                v[...] = f
            views.append(dn._frame_list_args(vs))  # (n, pointers, widths, heights), built once
        return views

    views = staged_views(frames)
    staged_ms = host_ms(two_in_flight(lambda: submit_list(views[lib.network_pipeline_next_slot(net)])), args.steps)
    pageable = dn._frame_list_args(frames)
    pageable_ms = host_ms(two_in_flight(lambda: submit_list(pageable)), args.steps)

    # host -> device ceiling and the conversion kernel alone, on the packed list
    win, toff, total = _lib.frame_list_layout(sizes, side, side, letterbox)
    packed = np.zeros(total, np.uint8)
    for f, r in zip(frames, win):
        packed[r.offset:r.offset + f.nbytes] = f.reshape(-1)
    packed[toff:] = np.frombuffer((_lib.FrameWindow * B)(*win), np.uint8)
    host, dsrc, ddst = C.c_void_p(), C.c_void_p(), C.c_void_p()
    out_bytes = B * 3 * side * side * 4
    _lib.check(klib.y2_host_alloc(C.byref(host), total))
    _lib.check(klib.y2_malloc(C.byref(dsrc), total))
    _lib.check(klib.y2_malloc(C.byref(ddst), out_bytes))
    C.memmove(host, packed.ctypes.data, total)
    h2d_ms = event_ms(lambda: _lib.check(klib.y2_memcpy_h2d(dsrc, host, total, stream)), args.steps)
    kernel_ms = event_ms(lambda: _lib.check(klib.y2_frames_u8_to_f32(dsrc, dsrc.value + toff, B, ddst, B, side, side,
                                                                       stream)), args.steps)
    touched = sum(rows_read(f) * f.src_w * 3 for f in win) + B * C.sizeof(_lib.FrameWindow) + out_bytes
    nominal = total + out_bytes
    klib.y2_host_free(host)
    klib.y2_free(dsrc)
    klib.y2_free(ddst)

    # all 1920x1080: the frame list against the uniform frames entry, both staged, alternated
    fw, fh = 1920, 1080
    hd = [np.random.default_rng(7 + i).integers(0, 256, size=(fh, fw, 3), dtype=np.uint8) for i in range(B)]
    hd_views = staged_views(hd)
    uni_stage = [lib.network_pipeline_staging_frames(net, s, fw, fh) for s in (0, 1)]
    hd_packed = np.ascontiguousarray(np.stack(hd))
    for p in uni_stage:
        C.memmove(p, hd_packed.ctypes.data, hd_packed.nbytes)
    hd_list, hd_uniform = [], []
    for _ in range(3):
        hd_list.append(host_ms(two_in_flight(lambda: submit_list(hd_views[lib.network_pipeline_next_slot(net)])),
                               args.steps))
        hd_uniform.append(host_ms(two_in_flight(
            lambda: submit_frames(uni_stage[lib.network_pipeline_next_slot(net)], fw, fh)), args.steps))
    del hd_views  # the staging buffers move below

    # uniform batches: this build's entries (the frame-list kernel with one record) and the baseline's, alternated
    uniform = {}
    for (sw, sh), t, lb in UNIFORM:
        nb = B * sh * sw * 3
        src, dst = C.c_void_p(), C.c_void_p()
        _lib.check(klib.y2_malloc(C.byref(src), nb))
        _lib.check(klib.y2_malloc(C.byref(dst), B * 3 * t * t * 4))
        u = np.random.default_rng(sw + sh).integers(0, 256, size=nb, dtype=np.uint8)
        _lib.check(klib.y2_memcpy_h2d(src, u.ctypes.data, nb, None))
        name = "y2_letterbox_u8_to_f32" if lb else "y2_resize_u8_to_f32"
        libs = {"new": klib} | ({"old": base} if base else {})
        ms = {k: [] for k in libs}
        for _ in range(5):
            for k, L in libs.items():
                fn = getattr(L, name)
                ms[k].append(event_ms(lambda fn=fn: _lib.check(fn(src, dst, B, sw, sh, t, t, None)), args.steps,
                                      on=None))
        entry = {f"{k}_ms": round(float(np.median(v)), 4) for k, v in ms.items()}
        entry["nominal_bytes"] = nb + B * 3 * t * t * 4
        if base:
            entry["new_over_old"] = round(float(np.median(ms["new"]) / np.median(ms["old"])), 4)
        uniform[f"{sw}x{sh}->{t} {'letterbox' if lb else 'resize'}"] = entry
        klib.y2_free(src)
        klib.y2_free(dst)

    # the host chain being replaced
    hl = dn.lib()

    def host_chain(steps):
        for _ in range(steps):
            xs = np.empty((B, 3, side, side), np.float32)
            for i, f in enumerate(frames):
                im = np.ascontiguousarray((f.transpose(2, 0, 1).astype(np.float64) / 255.0).astype(np.float32))
                img = dn.Image(f.shape[0], f.shape[1], 3, im.ctypes.data_as(C.POINTER(C.c_float)))
                out = (hl.letterbox_image if letterbox else hl.resize_image)(img, side, side)
                xs[i] = np.ctypeslib.as_array(out.data, shape=(3, side, side))
                hl.free_image(out)
            if letterbox:
                dn.network_classify_batch(net, images=xs, top=TOP)
            else:
                dn.network_detect_batch(net, xs, THRESH, NMS, MAX_DET)

    host_chain(1)
    t0 = time.perf_counter()
    host_chain(args.host_steps)
    host_chain_ms = (time.perf_counter() - t0) * 1e3 / args.host_steps

    for e in ev:
        klib.y2_event_destroy(e)
    dn.free_network(net)

    resident_ips = B * 1e3 / resident_ms
    h2d_gbps = total / (h2d_ms * 1e6)
    ceiling_ips = h2d_gbps * 1e9 / (frame_bytes / B)
    staged_ips = B * 1e3 / staged_ms
    name, power = device_info()
    res = {
        "tool": "frame_list_bench", "cfg": args.cfg, "side": side, "batch": B, "mix": args.mix, "steps": args.steps,
        "device": name, "power_limit": power,
        "sizes": {f"{w}x{h}": sizes.count((w, h)) for w, h in sorted(set(sizes))},
        "mean_frame_bytes": round(frame_bytes / B, 1),
        "e2e_staged": {"images_per_s": round(staged_ips, 1), "ms_per_step": round(staged_ms, 4)},
        "e2e_pageable": {"images_per_s": round(B * 1e3 / pageable_ms, 1), "ms_per_step": round(pageable_ms, 4)},
        "resident": {"images_per_s": round(resident_ips, 1), "ms_per_step": round(resident_ms, 4)},
        "h2d_ceiling": {"bytes": total, "GB_per_s": round(h2d_gbps, 2), "images_per_s": round(ceiling_ips, 1)},
        "staged_over_bound": round(staged_ips / min(resident_ips, ceiling_ips), 4),
        "kernel": {"ms": round(kernel_ms, 4), "nominal_bytes": nominal,
                   "nominal_GB_per_s": round(nominal / (kernel_ms * 1e6), 1), "touched_bytes": touched,
                   "touched_GB_per_s": round(touched / (kernel_ms * 1e6), 1)},
        "hd_1920x1080": {"frame_list_ms": round(float(np.median(hd_list)), 4),
                         "uniform_frames_ms": round(float(np.median(hd_uniform)), 4),
                         "list_over_uniform": round(float(np.median(hd_list) / np.median(hd_uniform)), 4)},
        "uniform_kernels": uniform,
        "host_chain": {"images_per_s": round(B * 1e3 / host_chain_ms, 1), "ms_per_step": round(host_chain_ms, 2)},
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
