#!/usr/bin/env python
"""Developer tool (GPU box): device-memory leak check - parse / predict / detect / resize / free in a loop,
parse / classify / change the batch / free for a classifier, frame lists whose packed size grows and shrinks, frame
descriptor lists (host and device, RGB, BGR and NV12) whose staged size grows and shrinks, video streams (open,
submit with repeats, reset, reopen larger, change the batch, free) and tracked video streams (enable tracking, submit
with repeats, reset, reopen and enable again, change the batch, free)."""
import sys
import tempfile
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from sr_object_detection_b200 import darknet as dn, synth  # noqa: E402

tmp = Path(tempfile.mkdtemp())
dn.set_gpu_index(0)
torch.cuda.init()


def cycle(name, side, batch):
    text = synth.CFGS[name](batch=batch, w=side, h=side)
    (tmp / "n.cfg").write_text(text)
    w = tmp / f"{name}.weights"
    if not w.exists():
        synth.write_weights(w, text, seed=1234)
    net = dn.parse_network_cfg(tmp / "n.cfg")
    dn.load_weights(net, w)
    x = synth.images(batch, 3, side, side, seed=1)
    dn.network_predict(net, x)
    dn.network_detect_batch(net, x, 0.02, 0.4, 64)
    lib = dn.lib()
    import ctypes as C
    dets = (dn.Detection * (batch * 64))()
    counts = (C.c_int * batch)()
    for _ in range(2):  # two batches in flight, then drain
        slot = lib.network_pipeline_next_slot(net)
        lib.network_detect_submit(net, lib.network_pipeline_staging(net, slot), 0.02, 0.4, 64)
    lib.network_detect_wait(net, dets, counts, 64)
    lib.network_detect_wait(net, dets, counts, 64)
    dn.set_batch_network(net, max(1, batch // 2))
    dn.network_predict(net, np.ascontiguousarray(x[:max(1, batch // 2)]))
    dn.resize_network(net, side - 32, side - 32)
    dn.free_network(net)


def classify_cycle(name, side, batch):
    text = synth.CFGS[name](batch=batch, w=side, h=side)
    (tmp / "c.cfg").write_text(text)
    w = tmp / f"{name}.weights"
    if not w.exists():
        synth.write_weights(w, text, seed=1234)
    net = dn.parse_network_cfg(tmp / "c.cfg")
    dn.load_weights(net, w)
    frames = np.random.default_rng(1).integers(0, 256, size=(batch, 375, 500, 3), dtype=np.uint8)
    dn.network_classify_batch(net, frames=frames, top=5)
    lib = dn.lib()
    for _ in range(2):  # two batches in flight, then drain
        slot = lib.network_pipeline_next_slot(net)
        lib.network_classify_submit_frames(net, lib.network_pipeline_staging_frames(net, slot, 500, 375), 500, 375, 5)
    dn.network_classify_wait(net, top=5)
    dn.network_classify_wait(net, top=5)
    dn.set_batch_network(net, max(1, batch // 2))
    dn.network_classify_batch(net, frames=np.ascontiguousarray(frames[:max(1, batch // 2)]), top=5)
    dn.free_network(net)


def frame_list_cycle(name, side, batch):
    text = synth.CFGS[name](batch=batch, w=side, h=side)
    (tmp / "f.cfg").write_text(text)
    w = tmp / f"{name}.weights"
    if not w.exists():
        synth.write_weights(w, text, seed=1234)
    net = dn.parse_network_cfg(tmp / "f.cfg")
    dn.load_weights(net, w)
    rng = np.random.default_rng(2)
    # packed sizes small, large, small, larger: the slots' staging buffers grow between batches
    for n, (fw, fh) in ((1, (500, 375)), (batch, (1280, 720)), (2, (640, 480)), (batch, (1920, 1080))):
        frames = [rng.integers(0, 256, size=(fh - i, fw + i, 3), dtype=np.uint8) for i in range(n)]
        dn.network_detect_submit_frame_list(net, frames, 0.02, 0.4, 64)
        views = dn.network_pipeline_staging_frame_list(net, dn.lib().network_pipeline_next_slot(net),
                                                       [(f.shape[1], f.shape[0]) for f in frames])
        for v, f in zip(views, frames):
            v[...] = f
        dn.network_detect_submit_frame_list(net, views, 0.02, 0.4, 64)
        dn.network_detect_wait_n(net, n, 64)
        dn.network_detect_wait_n(net, n, 64)
    dn.free_network(net)


def descs_cycle(name, side, batch):
    text = synth.CFGS[name](batch=batch, w=side, h=side)
    (tmp / "d.cfg").write_text(text)
    w = tmp / f"{name}.weights"
    if not w.exists():
        synth.write_weights(w, text, seed=1234)
    net = dn.parse_network_cfg(tmp / "d.cfg")
    dn.load_weights(net, w)
    rng = np.random.default_rng(5)
    fmts = (dn.FRAME_RGB24, dn.FRAME_NV12, dn.FRAME_BGR24)
    # staged sizes small, large, all on the device (the table alone), larger: host and device frames mixed
    for n, (fw, fh), host in ((1, (500, 376), True), (batch, (1280, 720), True), (batch, (1920, 1080), False),
                              (batch, (1920, 1080), True)):
        frames, descs = [], []
        for i in range(n):
            fmt = fmts[i % 3]
            shape = (fh * 3 // 2, fw) if fmt == dn.FRAME_NV12 else (fh, fw, 3)
            a = rng.integers(0, 256, size=shape, dtype=np.uint8)
            if not (host and i % 2 == 0):
                a = torch.from_numpy(a).cuda()
            frames.append(a)
            descs.append(dn.frame_desc(a, fmt))
        torch.cuda.synchronize()
        dn.network_detect_submit_frame_descs(net, descs, 0.02, 0.4, 64)
        dn.network_detect_submit_frame_descs(net, descs[::-1], 0.02, 0.4, 64)
        dn.network_detect_wait_n(net, n, 64)
        dn.network_detect_wait_n(net, n, 64)
        del frames, descs
    dn.free_network(net)


def tiled_cycle(name, side, batch):
    text = synth.CFGS[name](batch=batch, w=side, h=side)
    (tmp / "tl.cfg").write_text(text)
    w = tmp / f"{name}.weights"
    if not w.exists():
        synth.write_weights(w, text, seed=1234)
    net = dn.parse_network_cfg(tmp / "tl.cfg")
    dn.load_weights(net, w)
    rng = np.random.default_rng(6)
    frames, descs = [], []
    for i, fmt in enumerate((dn.FRAME_NV12, dn.FRAME_RGB24, dn.FRAME_BGR24)):
        a = rng.integers(0, 256, size=(1620, 1920) if fmt == dn.FRAME_NV12 else (1080, 1920, 3), dtype=np.uint8)
        if i == 1:
            a = torch.from_numpy(a).cuda()
        frames.append(a)
        descs.append(dn.frame_desc(a, fmt))
    torch.cuda.synchronize()
    # the spill scratch of the merge grows with the tiles of a frame and the candidates (a low thresh)
    dn.network_detect_submit_tiled_descs(net, descs, (2, 2, 64, 1), 0.02, 0.45, 64)
    dn.network_detect_submit_tiled_descs(net, descs[:2], (3, 2, 64, 1), 0.0001, 0.45, 64)
    dn.network_detect_wait_n(net, 3, 64)
    dn.network_detect_wait_n(net, 2, 64)
    dn.network_detect_tiled_descs(net, descs[1:2], (4, 3, 32, 1), 0.0001, 0.45, 64)
    dn.set_batch_network(net, batch * 2)  # a re-plan drops the scratch with the region's buffers
    dn.network_detect_tiled_descs(net, descs, (3, 3, 16, 0), 0.02, 0.45, 64)
    dn.free_network(net)
    del frames, descs


def streams_cycle(name, side, batch):
    text = synth.CFGS[name](batch=batch, w=side, h=side)
    (tmp / "s.cfg").write_text(text)
    w = tmp / f"{name}.weights"
    if not w.exists():
        synth.write_weights(w, text, seed=1234)
    net = dn.parse_network_cfg(tmp / "s.cfg")
    dn.load_weights(net, w)
    rng = np.random.default_rng(3)
    frames = [rng.integers(0, 256, size=(375, 500, 3), dtype=np.uint8) for _ in range(batch)]
    dn.network_streams_open(net, 4)
    ids = [i % 3 for i in range(batch)]  # every stream several times in one list
    dn.network_detect_submit_streams(net, ids, frames, 0.02, 0.4, 64)
    dn.network_detect_submit_streams(net, ids[::-1], frames, 0.02, 0.4, 64)
    dn.network_stream_reset(net, 1)
    dn.network_detect_wait_n(net, batch, 64)
    dn.network_detect_wait_n(net, batch, 64)
    dn.network_streams_open(net, 64)  # reopen larger
    dn.network_detect_streams(net, list(range(batch)), frames, 0.02, 0.4, 64)
    dn.set_batch_network(net, batch * 2)  # a re-plan that keeps the streams, and a larger mean buffer
    dn.network_detect_streams(net, [5] * batch, frames, 0.02, 0.4, 64)
    dn.free_network(net)


def tracked_cycle(name, side, batch):
    text = synth.CFGS[name](batch=batch, w=side, h=side)
    (tmp / "t.cfg").write_text(text)
    w = tmp / f"{name}.weights"
    if not w.exists():
        synth.write_weights(w, text, seed=1)
    net = dn.parse_network_cfg(tmp / "t.cfg")
    dn.load_weights(net, w)
    rng = np.random.default_rng(4)
    frames = [rng.integers(0, 256, size=(375, 500, 3), dtype=np.uint8) for _ in range(batch)]
    dn.network_streams_open(net, 4)
    dn.network_streams_track(net, 6)
    ids = [i % 3 for i in range(batch)]
    dn.network_detect_submit_streams_tracked(net, ids, frames, 0.02, 0.4, True, 64)
    dn.network_detect_submit_streams_tracked(net, ids[::-1], frames, 0.02, 0.4, False, 64)
    dn.network_stream_reset(net, 1)
    dn.network_detect_wait_tracked(net, batch, 64)
    dn.network_detect_wait_tracked(net, batch, 64)
    dn.network_streams_open(net, 64)  # reopen larger: tracking is dropped, enable it again with a longer story
    dn.network_streams_track(net, 32)
    dn.network_detect_streams_tracked(net, list(range(batch)), frames, 0.02, 0.4, True, 64)
    dn.set_batch_network(net, batch * 2)  # a re-plan that keeps the tracks
    dn.network_detect_streams_tracked(net, [5] * batch, frames, 0.02, 0.4, False, 64)
    dn.free_network(net)


for fn, name, side, batch in ((cycle, "tiny-yolo-voc", 416, 8), (cycle, "yolo-voc", 416, 64),
                              (classify_cycle, "darknet19_448", 448, 16), (frame_list_cycle, "tiny-yolo-voc", 416, 16),
                              (descs_cycle, "tiny-yolo-voc", 416, 16), (tiled_cycle, "tiny-yolo-voc", 416, 16),
                              (streams_cycle, "tiny-yolo-voc", 416, 16), (tracked_cycle, "tiny-yolo-voc", 416, 16)):
    fn(name, side, batch)  # warm: allocator pools, per-device scratch
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info()
    for _ in range(15):
        fn(name, side, batch)
    torch.cuda.synchronize()
    free1, _ = torch.cuda.mem_get_info()
    print(f"{name} b{batch}: free before {free0 >> 20} MiB, after 15 cycles {free1 >> 20} MiB, delta {(free0 - free1) >> 20} MiB")
