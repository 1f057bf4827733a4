#!/usr/bin/env python
"""Headline benchmark: YOLOv2-416 (yolo-voc.cfg) images/sec, batch 64 per GPU, on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path

A step = one pass of the hot path over one batch of synthetic images: forward (23 tcgen05
convolutions, 5 maxpools, reorg, in-place routes, region layer) + get_region_boxes + do_nms_sort +
final pick.  `value` is measured with the batch resident in HBM, `e2e` through the public C API
with host buffers (pinned H2D of the images and D2H of the detection lists inside the timed
region).  One JSON line on stdout (rank 0).

    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR

also writes the detections of the last timed step of `value` as DIR/*.npy (see dump_outputs), so that two
builds can be compared output for output: weights and images come from fixed seeds.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

WORKLOAD = "yolo-voc.cfg 416x416 batch 64 per GPU, forward + region decode + NMS"
CFG_NAME = "yolo-voc"
BATCH = 64
SIDE = 416
THRESH = 0.24   # detector.c:602 default -thresh
NMS = 0.4       # detector.c:456 / yolo_v2_class.hpp:45
MAX_DET = 256
SEED_W, SEED_X = 1234, 42
# The detection head of the random-init weights is scaled by this factor (synth.write_weights): with the plain
# init no box of a random network reaches the 0.24 threshold and decode / NMS / pick would run on an empty
# candidate set; at 13 about 8 % of the 845 boxes of an image clear it (SURVEY.md section 8d asks for ~5 %) and
# NMS keeps ~8 of them.  The reference arm reads the same weights file.
HEAD_GAIN = 13.0
GATHER_CAP = 32  # detections per image carried by the fixed-size host gather of the multi-rank e2e loop
DUMP_MAX_BYTES = 64 << 20  # --dump-outputs: larger detection tables are replaced by a fixed, seeded sample of rows


def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "tflops_burst": d["bf16_tflops"],
                "hbm_gbs": d["hbm_gbs"], "source": "measured (MEASURED_PEAKS.json)"}
    return {"tflops_sustained": 1400.0, "tflops_burst": 1590.0, "hbm_gbs": 6650.0,
            "source": "fallback (B200_PROFILING.md)"}


def _ncu_evidence():
    """DRAM traffic and tensor-pipe utilisation of the dominant kernel from the committed ncu capture
    (profiles/dominant_kernel_ncu.json names the raw summary it was taken from)."""
    p = ROOT / "profiles" / "dominant_kernel_ncu.json"
    try:
        return json.loads(p.read_text())
    except Exception:
        return None


def _cpu_model() -> str:
    try:
        for line in Path("/proc/cpuinfo").read_text().splitlines():
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def _host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            self.path = tempfile.NamedTemporaryFile(prefix="clocks_", suffix=".csv", delete=False).name
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        for line in Path(self.path).read_text().splitlines():
            f = [t.strip() for t in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0])); smax.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        # "under load": samples in the upper half of the power range
        thr = (max(power) + min(power)) / 2
        load = [s for s, p in zip(sm, power) if p >= thr] or sm
        return {"sm_mhz": statistics.median(load), "sm_max_mhz": max(smax), "power_w_max": max(power),
                "samples": len(sm), "reasons": sorted(reasons)}


def _write_inputs(tmp: Path, batch: int):
    from sr_object_detection_b200 import synth
    cfg_text = synth.CFGS[CFG_NAME](batch=batch, w=SIDE, h=SIDE)
    cfg = tmp / f"{CFG_NAME}_b{batch}.cfg"
    cfg.write_text(cfg_text)
    weights = tmp / f"{CFG_NAME}.weights"
    if not weights.exists():
        synth.write_weights(weights, cfg_text, seed=SEED_W, head_gain=HEAD_GAIN)
    return cfg, weights


def _ref_binary():
    ref = ROOT / "oracle" / "_ref" / "darknet_ref"
    if ref.exists():
        return ref, "reference"
    ref = ROOT / "oracle" / "_build" / "y2_oracle"
    return (ref, "port") if ref.exists() else (None, "unavailable")


def _time_reference(ref, cfg, weights, inp, warmup, iters, threads):
    """One timed run of the CPU path.  torchrun exports OMP_NUM_THREADS=1 to its workers: the thread count is
    always set explicitly here."""
    env = dict(os.environ)
    env["OMP_NUM_THREADS"] = str(threads)
    env.pop("OMP_PROC_BIND", None)
    r = subprocess.run([str(ref), "time", str(cfg), str(weights), str(inp), str(THRESH), str(NMS), str(warmup),
                        str(iters)], capture_output=True, text=True, env=env)
    if r.returncode != 0:
        raise RuntimeError(r.stderr[-200:])
    return json.loads(r.stdout.strip().splitlines()[-1])


def cpu_baseline(tmp: Path, iters: int = 20, warmup: int = 1) -> dict:
    """The reference's own CPU path (oracle/_ref, compiled from the reference sources) on the
    host cores, bounded sample of the same workload: batch-1 forward + decode + NMS, with all host
    threads and with one (BASELINE.md section 4)."""
    from sr_object_detection_b200 import synth
    ref, kind = _ref_binary()
    if ref is None:
        return {"value": None, "unit": "images/s", "cores": 0, "kind": "unavailable",
                "sample": "oracle binaries not built (run __graft_entry__.build())"}
    cfg, weights = _write_inputs(tmp, 1)
    inp = tmp / "cpu_input.f32"
    synth.images(1, 3, SIDE, SIDE, seed=SEED_X).tofile(inp)
    threads = _host_threads()
    try:
        d = _time_reference(ref, cfg, weights, inp, warmup, iters, threads)
        d1 = _time_reference(ref, cfg, weights, inp, 0, 1, 1)
    except RuntimeError as e:
        return {"value": None, "unit": "images/s", "cores": 0, "kind": kind, "sample": "failed: " + str(e)}
    return {"value": round(d["images_per_s"], 4), "unit": "images/s", "cores": threads, "kind": kind,
            "one_thread_value": round(d1["images_per_s"], 4), "cpu_model": _cpu_model(),
            "sample": f"{iters} x batch-1 {CFG_NAME} {SIDE}x{SIDE} forward+decode+NMS after {warmup} warm-up, "
                      f"OMP_NUM_THREADS={threads} ({d['seconds']:.1f} s); one image with OMP_NUM_THREADS=1 "
                      f"({d1['seconds']:.1f} s)"}


def dump_outputs(out: Path, dets, counts) -> None:
    """What network_detect_wait handed to the caller after the last timed step, for rank 0's batch:
    counts.npy      [batch]          detections the library reported per image;
    detections.npy  [n][8]           image, box_index, obj_id, prob, x, y, w, h of every returned detection,
                                     image by image in the library's order (at most MAX_DET per image).
    float64 holds the int32 and float32 fields of y2_det exactly.  Should the two files exceed DUMP_MAX_BYTES (only
    at very large --batch), detections.npy keeps a seeded sample of its rows, in their original order."""
    import numpy as np
    counts = np.asarray(counts, np.float64)
    rows = [np.zeros((0, 8))]
    for b, n in enumerate(counts):
        d = dets[b * MAX_DET:b * MAX_DET + min(int(n), MAX_DET)]
        rows.append(np.stack([np.full(len(d), b), d["box_index"], d["obj_id"], d["prob"], d["x"], d["y"], d["w"],
                              d["h"]], axis=1).astype(np.float64))
    det = np.concatenate(rows)
    keep = (DUMP_MAX_BYTES - counts.nbytes - 1024) // (det.itemsize * 8)  # 1 KB for the two .npy headers
    if len(det) > keep:
        det = det[np.sort(np.random.default_rng(0).choice(len(det), keep, replace=False))]
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / "counts.npy", counts)
    np.save(out / "detections.npy", det)


def run_reference(args) -> int:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    with tempfile.TemporaryDirectory(prefix="y2bench_") as t:
        tmp = Path(t)
        from sr_object_detection_b200 import synth
        ref, kind = _ref_binary()
        if ref is None:
            _emit({"impl": "reference", "unavailable": "oracle binaries not built"})
            return 0
        cfg, weights = _write_inputs(tmp, 1)
        inp = tmp / "cpu_input.f32"
        synth.images(1, 3, SIDE, SIDE, seed=SEED_X).tofile(inp)
        threads = _host_threads()
        try:
            d = _time_reference(ref, cfg, weights, inp, args.warmup, args.steps, threads)
        except RuntimeError as e:
            _emit({"impl": "reference", "unavailable": "oracle run failed: " + str(e)[-160:]})
            return 0
        ips = d["images_per_s"]
        line = {
            "impl": "reference", "metric": "images/sec", "value": round(ips, 4), "unit": "images/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(1000.0 * d["seconds"] / args.steps, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sample": "one image per step (batch 1), host CPU",
                       "omp_threads": threads, "cpu_model": _cpu_model(), "head_gain": HEAD_GAIN},
            "cpu_baseline": {"value": round(ips, 4), "unit": "images/s", "cores": threads, "kind": kind,
                             "cpu_model": _cpu_model(),
                             "sample": f"{args.steps} steps x 1 image, forward+decode+NMS, OMP_NUM_THREADS={threads}"},
            "e2e": {"value": round(ips, 4), "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        _emit(line)
    return 0


_JSON_OUT = None


def _claim_stdout():
    """stdout must carry exactly ONE JSON line.  Libraries write banners to file descriptor 1 on their
    own (NCCL prints "NCCL version ..." from C), so keep a private duplicate of the real stdout for the
    JSON line and point fd 1 at stderr for everything else in this process."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
    return _JSON_OUT


def _emit(line: dict) -> None:
    out = _claim_stdout()
    out.write(json.dumps(line) + "\n")
    out.flush()


def main() -> int:
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    # Defaults: 300 timed steps (~0.55 s) after 30 warm-up steps.  The 1 kW power limiter needs ~70 ms of this
    # load to settle (the first 40 steps after idle run ~10 % faster, 1.70 vs 1.88 ms), so a 20-step timed
    # region would sit entirely inside that burst window and nvidia-smi (100 ms period) could not even sample
    # it; 300 steps measure the sustained rate with the clocks sampled inside the timed region itself.
    # The reference arm (one CPU image per step, ~0.5 s each) defaults to 20 steps.
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-out", default=None, help="write the per-layer timing table (json) here")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the detections of the last timed step as DIR/<name>.npy (rank 0's batch)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 20 if args.impl == "reference" else 300
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup is None:
        args.warmup = 3 if args.impl == "reference" else 30
    if args.impl == "reference":
        return run_reference(args)
    if args.warmup < 3:
        args.warmup = 3

    import numpy as np
    import torch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    host_group = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # stdout carries exactly one JSON line: NCCL's own banner / logs go to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        # the detection lists live on the host when network_detect_wait returns: they are gathered there
        host_group = dist.new_group(backend="gloo")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local_rank)

    from sr_object_detection_b200 import _lib, synth
    from sr_object_detection_b200 import darknet as dn
    from sr_object_detection_b200 import dp

    lib = dn.lib()
    B = args.batch
    tmpdir = tempfile.TemporaryDirectory(prefix=f"y2bench_r{rank}_")
    tmp = Path(tmpdir.name)
    cfg, weights = _write_inputs(tmp, B)
    dn.set_gpu_index(local_rank)
    lib.cuda_set_device(local_rank)
    # this rank's host thread (submits, staging copies, detection gather) stays on the CPUs next to its GPU
    lib.y2_bind_thread_to_device.restype = C.c_int
    cpus_bound = int(lib.y2_bind_thread_to_device(local_rank))
    net = dn.parse_network_cfg(cfg)
    dn.load_weights(net, weights)
    lo, hi = dp.shard_range(rank, world, B * world)  # this rank's slice of the global batch (weak scaling)
    assert hi - lo == B
    images = synth.images(B, 3, SIDE, SIDE, seed=SEED_X + lo)
    stream = C.c_void_p(lib.network_stream(net))

    # stage the batch once in the pinned buffer; `value` keeps it resident in HBM
    staging = lib.network_input_staging(net)
    C.memmove(staging, images.ctypes.data, images.nbytes)
    lib.network_upload_input(net, staging)
    dets = (dn.Detection * (B * MAX_DET))()
    counts = (C.c_int * B)()
    dets_np = np.ctypeslib.as_array(dets)
    counts_np = np.ctypeslib.as_array(counts)

    def step_device():  # synchronous form: the host waits for every step's detections before launching the next
        lib.network_forward_device(net)
        lib.network_detect_device(net, THRESH, NMS, dets, counts, MAX_DET)

    # `value`: the same work with the batch resident in HBM and two steps in flight, so that the device does not idle
    # while the host picks up a step's detection lists (459 KB D2H + a stream sync per step in the synchronous form).
    # Both slots of the pipeline get the batch once, before the timed region.
    for s in (0, 1):
        _lib.check(lib.y2_memcpy_h2d(lib.network_pipeline_input_device(net, s), staging, images.nbytes, stream))
    _lib.check(lib.y2_stream_sync(stream))

    def run_device(steps):
        lib.network_detect_submit_resident(net, THRESH, NMS, MAX_DET)
        for _ in range(1, steps):
            lib.network_detect_submit_resident(net, THRESH, NMS, MAX_DET)
            lib.network_detect_wait(net, dets, counts, MAX_DET)
        lib.network_detect_wait(net, dets, counts, MAX_DET)

    gathered = {"images": 0, "detections": 0}

    def gather():
        """multi-rank runs: the per-image detection lists of every rank end up on rank 0, in image order (the only
        thing that crosses ranks); a fixed-size host gather over gloo, inside the e2e timed region"""
        if world == 1:
            return
        res = dp.gather_detection_arrays(dets_np, counts_np, MAX_DET, GATHER_CAP, group=host_group)
        if res is not None:
            gathered["images"] += len(res[1])
            gathered["detections"] += int(res[1].sum())

    def step_e2e_sync():
        lib.network_detect_batch(net, staging, THRESH, NMS, dets, counts, MAX_DET)
        gather()

    # pipelined public API: every step uploads its own batch from pinned host memory (slots
    # alternate), runs forward + decode + NMS and reads the detection lists back; two batches are in
    # flight so the H2D copy of step i+1 overlaps the forward pass of step i
    pipe_stage = [lib.network_pipeline_staging(net, s) for s in (0, 1)]
    for ps in pipe_stage:
        C.memmove(ps, images.ctypes.data, images.nbytes)

    def submit():
        lib.network_detect_submit(net, pipe_stage[lib.network_pipeline_next_slot(net)], THRESH, NMS, MAX_DET)

    def run_e2e_pipelined(steps):
        submit()
        for _ in range(1, steps):
            submit()
            lib.network_detect_wait(net, dets, counts, MAX_DET)
            gather()
        lib.network_detect_wait(net, dets, counts, MAX_DET)
        gather()

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    ev = [C.c_void_p() for _ in range(2)]
    for e in ev:
        _lib.check(lib.y2_event_create(C.byref(e)))

    def timed(fn, steps, on_stream=stream):
        barrier()
        _lib.check(lib.y2_event_record(ev[0], on_stream))
        for _ in range(steps):
            fn()
        _lib.check(lib.y2_event_record(ev[1], on_stream))
        torch.cuda.synchronize()
        ms = C.c_float()
        _lib.check(lib.y2_event_elapsed_ms(ev[0], ev[1], C.byref(ms)))
        barrier()
        if world > 1:
            t = torch.tensor([ms.value], device="cuda")
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            return float(t.item())
        return ms.value

    run_device(args.warmup)
    torch.cuda.synchronize()
    launches_fwd = lib.network_launch_count(net)
    det_per_image = float(np.mean([min(c, MAX_DET) for c in counts]))
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_dev = timed(lambda: run_device(args.steps), 1)
    # the steps below reuse dets / counts (the uint8 pipeline on other images): keep this step's result now
    last_dets, last_counts = dets_np.copy(), counts_np.copy()
    sampling = "nvidia-smi -lms 100 over the timed region"
    if ms_dev < 400.0:
        # a short timed region (--steps given by the caller): nvidia-smi samples every 100 ms, so keep the same
        # step running (untimed) for ~1.5 s more so that the clock record really is taken under this load
        t_probe = time.time()
        while time.time() - t_probe < 1.5:
            run_device(10)
        torch.cuda.synchronize()
        sampling += " + 1.5 s of the same step repeated (the timed region itself was shorter than 0.4 s)"
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["sampling"] = sampling
    for _ in range(3):
        step_device()
    ms_dev_sync = timed(step_device, args.steps)

    # the same pipeline fed with raw uint8 RGB images (what an image decoder hands over): a quarter of the upload
    u8_images = np.random.default_rng(SEED_X + lo).integers(0, 256, size=(B, SIDE, SIDE, 3), dtype=np.uint8)
    pipe_stage_u8 = [lib.network_pipeline_staging_u8(net, s) for s in (0, 1)]
    for ps in pipe_stage_u8:
        C.memmove(ps, u8_images.ctypes.data, u8_images.nbytes)

    def submit_u8():
        lib.network_detect_submit_u8(net, pipe_stage_u8[lib.network_pipeline_next_slot(net)], THRESH, NMS, MAX_DET)

    def run_e2e_u8(steps):
        submit_u8()
        for _ in range(1, steps):
            submit_u8()
            lib.network_detect_wait(net, dets, counts, MAX_DET)
            gather()
        lib.network_detect_wait(net, dets, counts, MAX_DET)
        gather()

    for _ in range(3):
        step_e2e_sync()
    ms_e2e_sync = timed(step_e2e_sync, args.steps)
    run_e2e_pipelined(3)
    gathered["images"] = gathered["detections"] = 0
    ms_e2e = timed(lambda: run_e2e_pipelined(args.steps), 1)
    gathered_e2e = dict(gathered)
    run_e2e_u8(3)
    ms_e2e_u8 = timed(lambda: run_e2e_u8(args.steps), 1)

    # host -> device ceiling of this box with the same ranks copying at the same time: plain pinned
    # cudaMemcpyAsync of the fp32 batch, nothing else running (what the fp32 e2e entry is bound by)
    h2d_reps = max(5, min(args.steps, 20))

    def h2d_copy():
        _lib.check(lib.y2_memcpy_h2d(lib.network_input_device(net), pipe_stage[0], images.nbytes, stream))

    for _ in range(2):
        h2d_copy()
    ms_h2d = timed(h2d_copy, h2d_reps)
    h2d_gbs_per_gpu = images.nbytes * h2d_reps / (ms_h2d * 1e6)
    lib.network_upload_input(net, staging)  # restore the resident batch for the layer profile below

    # per-layer device times (eager pass with CUDA events on the network stream), for the
    # roofline of the dominant kernel: the tcgen05 convolution
    n_layers = net.n
    layer_ms = np.zeros(n_layers, np.float32)
    prof_steps = max(3, min(args.steps, 10))
    buf = (C.c_float * n_layers)()
    for _ in range(prof_steps):
        if ms_dev >= 400.0:
            # sustained regime: the H2D measurement above left the GPU idle long enough for the power limiter to
            # relax; put ~0.1 s of the same load in front of every profiled pass so that the per-layer times (and
            # the dominant kernel's roofline) are taken at the clocks the timed region ran at
            for _ in range(60):
                step_device()
        lib.network_profile_layers(net, buf, n_layers)
        layer_ms += np.ctypeslib.as_array(buf)
    layer_ms /= prof_steps
    conv_ms = 0.0
    conv_launches = 0
    table = []
    flops_img = lib.network_conv_flops(net)
    KERNELS = {0: "conv_tcgen05_kernel (per-tap)", 1: "conv_slab_kernel", 2: "conv_pair_kernel (cta_group::2)",
               3: "conv_pool_kernel (conv + maxpool)", 4: "stem_conv_pool_kernel"}
    per_kernel = {}  # variant -> [ms, flops, launches]
    for i in range(n_layers):
        l = net.layers[i]
        fl = 2.0 * l.n * l.size * l.size * l.c * l.out_h * l.out_w * B if l.type == dn.CONVOLUTIONAL else 0.0
        kern = lib.network_conv_kernel(net, i)
        if l.type == dn.CONVOLUTIONAL:
            conv_ms += float(layer_ms[i])
            conv_launches += 1
            acc = per_kernel.setdefault(kern, [0.0, 0.0, 0])
            acc[0] += float(layer_ms[i])
            acc[1] += fl
            acc[2] += 1
        table.append({"layer": i, "type": int(l.type), "ms": round(float(layer_ms[i]), 4),
                      "kernel": KERNELS.get(kern),
                      "tflops": round(float(fl / (float(layer_ms[i]) * 1e9)), 1) if fl and layer_ms[i] > 0 else None})

    total_images = B * world * args.steps
    value = total_images / (ms_dev / 1000.0)
    e2e_value = total_images / (ms_e2e / 1000.0)
    peaks = _peaks()
    # the peak that matches the regime of THIS run: a timed region shorter than ~0.4 s sits in the window before
    # the power limiter settles (compare with the burst cuBLAS figure), a longer one runs at the sustained clocks
    sustained = ms_dev >= 400.0
    peak = peaks["tflops_sustained"] if sustained else peaks["tflops_burst"]
    step_flops = flops_img * B
    achieved_tf = step_flops / (conv_ms * 1e9) if conv_ms > 0 else 0.0
    detect_launches = 3  # region_boxes (+ candidate count), nms_mark, collect (+ argmax for wide class rows)
    # dominant kernel = the convolution kernel with the largest share of the step (the CTA-pair kernel on
    # yolo-voc): algorithmic FLOPs of the layers it runs / the CUDA-event time of those launches
    dom = max(per_kernel, key=lambda k: per_kernel[k][0]) if per_kernel else None
    dom_ms, dom_fl, dom_n = per_kernel.get(dom, [0.0, 0.0, 0])
    dom_tf = dom_fl / (dom_ms * 1e9) if dom_ms > 0 else 0.0
    ncu = _ncu_evidence() or {}
    ncu_ok = dom == 2 and str(ncu.get("kernel", "")).startswith("conv_pair")
    roofline = {
        "bound": "tensor", "kernel": f"{KERNELS.get(dom)} ({dom_n} launches per step)",
        "achieved": round(dom_tf, 1), "peak": peak, "unit": "TFLOP/s",
        "frac": round(dom_tf / peak, 4),
        "peak_regime": "sustained" if sustained else "burst",
        "frac_vs_burst_peak": round(dom_tf / peaks["tflops_burst"], 4),
        "frac_vs_sustained_peak": round(dom_tf / peaks["tflops_sustained"], 4),
        "peak_burst": peaks["tflops_burst"], "peak_sustained": peaks["tflops_sustained"],
        "peak_source": peaks["source"],
        # dram__bytes_read.sum + dram__bytes_write.sum of one launch and the tensor-pipe utilisation, from the
        # committed ncu capture of the dominant kernel (BASELINE.json's second metric)
        "traffic": (ncu.get("dram_bytes_read", 0) + ncu.get("dram_bytes_write", 0)) if ncu_ok else None,
        "tensor_pipe_pct": ncu.get("tensor_pipe_pct_elapsed") if ncu_ok else None,
        "tensor_pipe_pct_of_active_cycles": ncu.get("tensor_pipe_pct_active") if ncu_ok else None,
        "traffic_of": (f"{ncu.get('launch')}; ncu --set full, {ncu.get('source')}; algorithmic operand bytes of that "
                       f"launch: {ncu.get('algorithmic_operand_bytes')}") if ncu_ok else None,
        "ms_per_step": round(dom_ms, 4), "share_of_step": round(dom_ms / max(float(layer_ms.sum()), 1e-9), 3),
        "all_convolutions": {"launches": conv_launches, "ms_per_step": round(conv_ms, 4),
                             "achieved": round(achieved_tf, 1), "frac": round(achieved_tf / peak, 4)},
        "per_kernel": {KERNELS.get(k): {"launches": v[2], "ms": round(v[0], 4),
                                        "tflops": round(v[1] / (v[0] * 1e9), 1) if v[0] > 0 else None}
                       for k, v in sorted(per_kernel.items())},
        "step_ms_eager": round(float(layer_ms.sum()), 4)}
    d2h_bytes = int(B * MAX_DET * C.sizeof(dn.Detection) + B * 4)
    gather_note = ("; the detection lists of all ranks are gathered on rank 0 every step (host-side gloo gather, "
                   f"{GATHER_CAP} detections per image per message)") if world > 1 else ""
    line = {
        "metric": "images/sec", "value": round(value, 1), "unit": "images/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_dev / args.steps, 4),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": WORKLOAD, "cfg": "yolo-voc (YOLOv2-VOC)", "batch_per_gpu": B,
                   "global_batch": B * world, "input": f"{SIDE}x{SIDE}x3 fp32", "parallelism": f"dp{world}",
                   "thresh": THRESH, "nms": NMS,
                   "l2": "inputs larger than L2 (133 MB fp32 batch, 2.5 GB activations per step)",
                   "weights": f"random-init synthetic .weights (seed 1234), detection head scaled x{HEAD_GAIN:g} so "
                              "that decode / NMS / pick have candidates to work on",
                   "detections_per_image": round(det_per_image, 2),
                   "schedule": "CUDA graph replay; batch resident in HBM, two steps in flight (network_detect_submit_resident / "
                               "network_detect_wait): every step's detection lists are read back to the host",
                   "sync_value": round(total_images / (ms_dev_sync / 1000.0), 1),
                   "sync_schedule": "network_forward_device + network_detect_device: the host waits for each step's "
                                    "detections before it launches the next",
                   "host_thread_cpus": cpus_bound or "unbound (PCI topology not visible)",
                   "algorithmic_gflop_per_image": round(flops_img / 1e9, 3),
                   "regime": ("sustained: timed region of %.2f s under the 1 kW power cap" % (ms_dev / 1000.0))
                   if sustained else
                   ("burst window: timed region of %.0f ms; the power limiter settles after ~70 ms of this load, "
                    "the sustained rate is ~10%% lower (default --steps 300 measures it)" % ms_dev)},
        "model_tflops": round(value / world * flops_img / 1e12, 1),
        "model_frac_of_peak": round(value / world * flops_img / 1e12 / peak, 4),
        "roofline": roofline,
        "e2e": {"value": round(e2e_value, 1), "unit": "images/s", "ms_per_step": round(ms_e2e / args.steps, 4),
                "h2d_bytes_per_step": int(images.nbytes),
                "d2h_bytes_per_step": d2h_bytes,
                "api": "network_detect_submit(net, pinned_host_images, thresh, nms, max_det) / network_detect_wait(net, "
                       "dets, counts, max_det), two batches in flight" + gather_note,
                "h2d_ceiling_gbs_per_gpu": round(h2d_gbs_per_gpu, 2),
                "h2d_ceiling_gbs_total": round(h2d_gbs_per_gpu * world, 2),
                "h2d_ceiling_how": f"{h2d_reps} back-to-back pinned cudaMemcpyAsync of the {images.nbytes >> 20} MB fp32 "
                                   f"batch on all {world} rank(s) at once, max over ranks",
                "frac_of_h2d_ceiling": round(e2e_value / world * (images.nbytes / B) / (h2d_gbs_per_gpu * 1e9), 4),
                "sync_value": round(total_images / (ms_e2e_sync / 1000.0), 1),
                "sync_api": "network_detect_batch(net, host_images, thresh, nms, dets, counts, max_det)"},
        "e2e_u8": {"value": round(total_images / (ms_e2e_u8 / 1000.0), 1), "unit": "images/s",
                   "ms_per_step": round(ms_e2e_u8 / args.steps, 4), "h2d_bytes_per_step": int(u8_images.nbytes),
                   "d2h_bytes_per_step": d2h_bytes,
                   "api": "network_detect_submit_u8(net, pinned_uint8_rgb_images, ...) / network_detect_wait: raw decoded "
                          "images, byte/255 on the device (bit-identical detections to the float call)" + gather_note},
        "gpu_launches": int((launches_fwd + detect_launches) * args.steps),
        "clocks": clocks,
    }
    if world > 1:
        line["e2e"]["gathered_on_rank0"] = gathered_e2e
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(tmp)
        if args.dump_outputs:  # before the bench line: a dump that cannot be written fails the run with no line out
            dump_outputs(Path(args.dump_outputs), last_dets, last_counts)
        _emit(line)
        if args.profile_out:
            Path(args.profile_out).write_text(json.dumps({"batch": B, "layers": table, "line": line}, indent=1))
    dn.free_network(net)
    if world > 1:
        torch.distributed.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
