#!/usr/bin/env python
"""Developer tool (GPU box): throughput of the batched classify path (network_classify_*) of one classifier cfg.

Prints one JSON line: the device name and power limit, forward-only ms/step (CUDA events), the top-k kernel alone
on the network's output (CUDA events), device-resident classify ms/step (submit_resident / wait, two batches in
flight, host clock), end-to-end images/s through submit_frames / wait with two batches in flight for frames at the
network size and at 500x375 and 1920x1080, the host -> device ceiling of plain pinned cudaMemcpyAsync in the same run,
and the letterbox kernel's time with two byte counts: nominal (every frame byte plus the canvas) and touched (the
source rows the window's bilinear taps read, whole rows, plus the canvas).  Weights and frames come from fixed seeds
(synth).

    python tools/classify_bench.py --cfg darknet19_448 --batch 64 --steps 30 --out profiles/x.json
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

CFGS = {"darknet19_448": (synth.darknet19_448_cfg, 448), "resnet50": (synth.resnet50_cfg, 256)}
TOP = 5


def device_info():
    r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, _, power = r.stdout.strip().partition(", ")
    return name or None, power or None


def rows_read(fw, fh, w, h):
    """source rows the letterbox kernel's vertical taps read for one frame (resize_image's y pass, image.c:1979-1990,
    in float32 as the kernel computes it)"""
    lib = _lib.load()
    g = [C.c_int() for _ in range(4)]
    lib.y2_letterbox_geometry(fw, fh, w, h, *[C.byref(v) for v in g])
    nw, nh = g[0].value, g[1].value
    if nw <= 0 or nh <= 0:
        return 0
    h_scale = np.float32(fh - 1) / np.float32(nh - 1) if nh > 1 else np.float32(0)
    rows = set()
    for r in range(nh):
        iy = min(int(np.float32(r) * h_scale), fh - 1)
        rows.add(iy)
        if not (r == nh - 1 or fh == 1):
            rows.add(min(iy + 1, fh - 1))
    return len(rows)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cfg", choices=sorted(CFGS), default="darknet19_448")
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--frames", default="net,500x375,1920x1080",
                    help="comma-separated frame sizes WxH for the end-to-end figures; 'net' = the network size")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if args.steps < 1 or args.batch < 1:
        ap.error("--steps and --batch must be >= 1")

    make_cfg, side = CFGS[args.cfg]
    B = args.batch
    lib = dn.lib()
    klib = _lib.load()
    klib.y2_letterbox_u8_to_f32.restype = C.c_int
    klib.y2_letterbox_u8_to_f32.argtypes = [C.c_void_p, C.c_void_p] + [C.c_int] * 5 + [C.c_void_p]
    klib.y2_letterbox_geometry.restype = None
    klib.y2_letterbox_geometry.argtypes = [C.c_int] * 4 + [C.POINTER(C.c_int)] * 4
    klib.y2_classify_topk.restype = C.c_int
    klib.y2_classify_topk.argtypes = [C.c_void_p] + [C.c_int] * 4 + [C.c_void_p, C.c_void_p, C.c_void_p]
    klib.y2_stem_u8_supported.restype = C.c_int
    klib.y2_stem_u8_supported.argtypes = [C.c_int, C.c_int]
    tmp = Path(tempfile.mkdtemp(prefix="y2cls_"))
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

    x = synth.images(B, 3, side, side, seed=1)
    staging = lib.network_input_staging(net)
    C.memmove(staging, x.ctypes.data, x.nbytes)
    lib.network_upload_input(net, staging)
    fwd_ms = event_ms(lambda: lib.network_forward_device(net), args.steps)

    hits = (dn.ClassHit * (B * TOP))()
    for s in (0, 1):
        _lib.check(klib.y2_memcpy_h2d(lib.network_pipeline_input_device(net, s), staging, x.nbytes, stream))
    _lib.check(klib.y2_stream_sync(stream))

    def resident(steps):
        lib.network_classify_submit_resident(net, TOP)
        for _ in range(1, steps):
            lib.network_classify_submit_resident(net, TOP)
            lib.network_classify_wait(net, hits, TOP)
        lib.network_classify_wait(net, hits, TOP)

    resident_ms = host_ms(resident, args.steps)

    # the top-k kernel alone, on the output layer of the last forward pass (fp32 [B][outputs] for these cfgs)
    oi = max(i for i in range(net.n) if net.layers[i].type != dn.COST)
    ol = net.layers[oi]
    hits_dev = C.c_void_p()
    _lib.check(klib.y2_malloc(C.byref(hits_dev), B * TOP * C.sizeof(dn.ClassHit)))
    out_dev = C.cast(ol.output_gpu, C.c_void_p)
    topk_ms = event_ms(lambda: _lib.check(klib.y2_classify_topk(out_dev, ol.outputs, B, ol.outputs, TOP, None,
                                                                hits_dev, stream)), args.steps)
    klib.y2_free(hits_dev)
    # the predicate network_classify_submit_frames applies to frames at the network size
    u8_path = lib.network_conv_kernel(net, 0) == 4 and klib.y2_stem_u8_supported(side, side) == 1

    e2e = {}
    biggest = (0, 0)
    for spec in args.frames.split(","):
        fw, fh = (side, side) if spec == "net" else map(int, spec.split("x"))
        if fw * fh > biggest[0] * biggest[1]:
            biggest = (fw, fh)
        frames = np.random.default_rng(fw * 7 + fh).integers(0, 256, size=(B, fh, fw, 3), dtype=np.uint8)
        stage = [lib.network_pipeline_staging_frames(net, s, fw, fh) for s in (0, 1)]
        for p in stage:
            C.memmove(p, frames.ctypes.data, frames.nbytes)

        def run(steps, fw=fw, fh=fh, stage=stage):
            lib.network_classify_submit_frames(net, stage[lib.network_pipeline_next_slot(net)], fw, fh, TOP)
            for _ in range(1, steps):
                lib.network_classify_submit_frames(net, stage[lib.network_pipeline_next_slot(net)], fw, fh, TOP)
                lib.network_classify_wait(net, hits, TOP)
            lib.network_classify_wait(net, hits, TOP)

        ms = host_ms(run, args.steps)
        e2e[f"{fw}x{fh}"] = {"images_per_s": round(B * 1e3 / ms, 1), "ms_per_step": round(ms, 4),
                             "h2d_bytes_per_step": int(frames.nbytes),
                             "path": "uint8 first layer" if (fw, fh) == (side, side) and u8_path
                             else "letterbox kernel"}

    # host -> device ceiling and the letterbox kernel alone, on the largest frames
    fw, fh = biggest
    nbytes = B * fh * fw * 3
    host, dsrc, ddst = C.c_void_p(), C.c_void_p(), C.c_void_p()
    _lib.check(klib.y2_host_alloc(C.byref(host), nbytes))
    _lib.check(klib.y2_malloc(C.byref(dsrc), nbytes))
    out_bytes = B * 3 * side * side * 4
    _lib.check(klib.y2_malloc(C.byref(ddst), out_bytes))
    frames = np.random.default_rng(5).integers(0, 256, size=nbytes, dtype=np.uint8)
    C.memmove(host, frames.ctypes.data, nbytes)
    h2d_ms = event_ms(lambda: _lib.check(klib.y2_memcpy_h2d(dsrc, host, nbytes, stream)), args.steps)
    lb_ms = event_ms(lambda: _lib.check(klib.y2_letterbox_u8_to_f32(dsrc, ddst, B, fw, fh, side, side, stream)),
                     args.steps)
    klib.y2_host_free(host)
    klib.y2_free(dsrc)
    klib.y2_free(ddst)
    for e in ev:
        klib.y2_event_destroy(e)
    dn.free_network(net)
    rows = rows_read(fw, fh, side, side)
    touched = B * rows * fw * 3 + out_bytes

    name, power = device_info()
    res = {
        "tool": "classify_bench", "cfg": args.cfg, "batch": B, "side": side, "top": TOP, "steps": args.steps,
        "device": name, "power_limit": power,
        "forward_ms_per_step": round(fwd_ms, 4),
        "forward_images_per_s": round(B * 1e3 / fwd_ms, 1),
        "resident_classify_ms_per_step": round(resident_ms, 4),
        "topk_kernel_ms": round(topk_ms, 4),
        "resident_minus_forward_ms": round(resident_ms - fwd_ms, 4),
        "e2e_frames": e2e,
        "h2d_ceiling": {"frame": f"{fw}x{fh}", "bytes": nbytes, "GB_per_s": round(nbytes / (h2d_ms * 1e6), 2),
                        "images_per_s": round(B * 1e3 / h2d_ms, 1)},
        "letterbox_kernel": {"frame": f"{fw}x{fh}", "ms": round(lb_ms, 4),
                             "nominal_bytes": nbytes + out_bytes,
                             "nominal_GB_per_s": round((nbytes + out_bytes) / (lb_ms * 1e6), 1),
                             "source_rows_read": rows, "touched_bytes": touched,
                             "touched_GB_per_s": round(touched / (lb_ms * 1e6), 1)},
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
