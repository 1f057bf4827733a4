"""Frame descriptors (RGB, BGR or NV12 frames with a row pitch, in host or device memory; y2_frames_src_to_f32,
network_*_frame_descs, network_*_streams_*descs) against the tight host-RGB frame-list path fed with the same frames
converted to RGB bytes.  Every comparison is bit for bit."""
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from sr_object_detection_b200 import _lib, darknet as dn, synth
from tests.test_classify_gpu import NETS, _same
from tests.test_frame_list_gpu import _detector, _same_dets, _window_h
from tests.test_frame_src_host import to_rgb

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
RGB, BGR, NV12 = dn.FRAME_RGB24, dn.FRAME_BGR24, dn.FRAME_NV12
THRESH, NMS, MAX_DET = 0.02, 0.4, 256


def _frame(w, h, fmt, rng):
    shape = (h * 3 // 2, w) if fmt == NV12 else (h, w, 3)
    return rng.integers(0, 256, size=shape, dtype=np.uint8)


def _device(frame, pitch_extra, offset, keep):
    """frame's bytes in a torch allocation of their own, rows pitch_extra bytes wider than the frame's and the first
    row `offset` bytes into the allocation (an unaligned base for an odd offset)"""
    rows, row = frame.shape[0], frame.size // frame.shape[0]
    pitch = row + pitch_extra
    buf = torch.zeros(offset + rows * pitch, dtype=torch.uint8, device="cuda")
    strides = (pitch, frame.shape[2], 1) if frame.ndim == 3 else (pitch, 1)
    t = buf.as_strided(frame.shape, strides, offset)
    t.copy_(torch.from_numpy(frame))
    keep.append(buf)
    return t


def _desc(frame, fmt, where, keep):
    """a descriptor of frame: host (tight), host_pitched, device (tight) or device_pitched (unaligned bases; NV12 as a
    (y, uv) pair of separate allocations with different pitches)"""
    if where == "host":
        return dn.frame_desc(frame, fmt)
    if where == "host_pitched":
        wide = np.zeros((frame.shape[0], frame.shape[1] + 5) + frame.shape[2:], np.uint8)
        wide[:, 2:2 + frame.shape[1]] = frame
        keep.append(wide)
        return dn.frame_desc(wide[:, 2:2 + frame.shape[1]], fmt)
    if where == "device":
        return dn.frame_desc(_device(frame, 0, 0, keep), fmt)
    if fmt != NV12:
        return dn.frame_desc(_device(frame, 29, 3, keep), fmt)
    h = frame.shape[0] * 2 // 3
    y = _device(np.ascontiguousarray(frame[:h]), 29, 3, keep)
    uv = _device(np.ascontiguousarray(frame[h:]).reshape(h // 2, -1, 2), 45, 1, keep)
    return dn.frame_desc((y, uv), fmt)


WHERE = ["host", "device_pitched", "host_pitched", "device"]


def _list(specs, seed, keep):
    """(descriptors, tight RGB frames) for specs [(w, h, fmt, where), ...]"""
    rng = np.random.default_rng(seed)
    descs, rgb = [], []
    for w, h, fmt, where in specs:
        f = _frame(w, h, fmt, rng)
        descs.append(_desc(f, fmt, where, keep))
        rgb.append(to_rgb(f, fmt))
    torch.cuda.synchronize()  # the device frames are written before the network's stream reads them
    return descs, rgb


def _mixed(sizes, shift):
    """every format on every placement, in turn"""
    return [(w, h, (RGB, BGR, NV12)[(i + shift) % 3], WHERE[(i + i // 3 + shift) % 4])
            for i, (w, h) in enumerate(sizes)]


# ---- kernel -----------------------------------------------------------------------------------------------------
def _frames_u8(rgb, side, letterbox, batch):
    """y2_frames_u8_to_f32 on tight RGB frames"""
    win, toff, total = _lib.frame_list_layout([(f.shape[1], f.shape[0]) for f in rgb], side, side, letterbox)
    packed = np.zeros(total, np.uint8)
    for f, r in zip(rgb, win):
        packed[r.offset:r.offset + f.nbytes] = f.reshape(-1)
    packed[toff:] = np.frombuffer((_lib.FrameWindow * len(win))(*win), np.uint8)
    d_packed = torch.from_numpy(packed).cuda()
    dst = torch.full((batch, 3, side, side), -7.0, dtype=torch.float32, device="cuda")
    _lib.check(_lib.load().y2_frames_u8_to_f32(d_packed.data_ptr(), d_packed.data_ptr() + toff, len(rgb),
                                               dst.data_ptr(), batch, side, side, None), "frames_u8_to_f32")
    torch.cuda.synchronize()
    return dst.cpu().numpy()


def _frames_src(descs, side, letterbox, batch, keep):
    """y2_frames_src_to_f32 on a descriptor list: host frames staged tight in a device buffer as the pipeline does"""
    recs, toff, total = _lib.frame_desc_layout(descs, side, side, letterbox)
    assert total
    staged = np.zeros(max(toff, 1), np.uint8)
    for d, r in zip(descs, recs):
        if d.on_device:
            continue
        src = np.ascontiguousarray(d._keep).reshape(-1)  # host frames here are single arrays
        staged[r.win.offset:r.win.offset + src.size] = src
    d_staged = torch.from_numpy(staged).cuda()
    keep.append(d_staged)
    for d, r in zip(descs, recs):
        if not d.on_device:
            r.win.offset += d_staged.data_ptr()
            if d.format == NV12:
                r.uv += d_staged.data_ptr()
    table = torch.from_numpy(np.frombuffer((_lib.FrameSrc * len(recs))(*recs), np.uint8).copy()).cuda()
    dst = torch.full((batch, 3, side, side), -7.0, dtype=torch.float32, device="cuda")
    _lib.check(_lib.load().y2_frames_src_to_f32(table.data_ptr(), len(descs), dst.data_ptr(), batch, side, side, None),
               "frames_src_to_f32")
    torch.cuda.synchronize()
    return dst.cpu().numpy()


KERNEL_SIZES = [(1920, 1080), (2, 2), (640, 480), (38, 54), (2, 64), (500, 376), (64, 2), (416, 416), (1280, 720),
                (10, 6), (376, 500), (8, 8)]


@pytest.mark.parametrize("letterbox,side", [(False, 416), (False, 608), (True, 448), (True, 32)])
def test_kernel_equals_the_frame_list_kernel_on_the_converted_frames(letterbox, side):
    keep = []
    # host frames staged tight; the device frames of every format pitched at unaligned bases and tight
    specs = [(w, h, (RGB, BGR, NV12)[i % 3], ("host", "device_pitched", "device")[(i // 3) % 3])
             for i, (w, h) in enumerate(KERNEL_SIZES) if not letterbox or _window_h(w, h, side) != 1]
    descs, rgb = _list(specs, side + letterbox, keep)
    batch = len(specs) + 2  # a partial list: the .5 canvas behind it
    got = _frames_src(descs, side, letterbox, batch, keep)
    want = _frames_u8(rgb, side, letterbox, batch)
    for i, spec in enumerate(specs):
        assert np.array_equal(got[i].view(np.uint32), want[i].view(np.uint32)), (spec, side, letterbox)
    assert np.all(got[len(specs):] == np.float32(.5))


# ---- detection ----------------------------------------------------------------------------------------------------
SIZES = [(500, 376), (1920, 1080), (416, 416), (640, 480), (2, 2), (354, 500), (1280, 720)]


@pytest.mark.parametrize("name", ["tiny-yolo-voc", "yolo-voc"])
def test_detect_frame_descs_equal_the_frame_list_on_the_converted_frames(tmp_path, name):
    net = _detector(tmp_path, name, 4)
    keep = []
    try:
        for sizes, seed in ((SIZES[:4], 1), (SIZES[4:], 2), (SIZES[1:2], 3)):  # n == batch and n < batch
            for shift in range(3):  # each frame in each format
                specs = [(w, h, (RGB, BGR, NV12)[(i + shift) % 3], WHERE[(i + seed + shift) % 4])
                         for i, (w, h) in enumerate(sizes)]
                descs, rgb = _list(specs, seed * 10 + shift, keep)
                want = dn.network_detect_frame_list(net, rgb, THRESH, NMS, MAX_DET)
                assert any(len(w) for w in want[0]), "test needs at least one detection"
                got = dn.network_detect_frame_descs(net, descs, THRESH, NMS, MAX_DET)
                assert got[1] == want[1], specs
                _same_dets(got[0], want[0], f"{name} {specs}")
    finally:
        dn.free_network(net)


# ---- classification -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["darknet19_448", "exact-tree"])
def test_classify_frame_descs_equal_the_frame_list_on_the_converted_frames(tmp_path, name, monkeypatch):
    monkeypatch.chdir(tmp_path)  # the exact tree classifier reads t.tree relative to the cwd
    net = NETS[name](tmp_path)
    keep = []
    try:
        for sizes, seed in (([(500, 376), (net.w, net.h)], 1), ([(38, 1920)], 2), ([(1920, 1080), (4, 2)], 3)):
            for shift in range(3):
                specs = [(w, h, (RGB, BGR, NV12)[(i + shift) % 3], WHERE[(i + seed + shift) % 4])
                         for i, (w, h) in enumerate(sizes)]
                descs, rgb = _list(specs, seed * 10 + shift, keep)
                _same(dn.network_classify_frame_descs(net, descs, top=5),
                      dn.network_classify_batch(net, frame_list=rgb, top=5))
    finally:
        dn.free_network(net)


# ---- streams --------------------------------------------------------------------------------------------------------
STREAM_SIZES = [(640, 480), (500, 376), (1280, 720)]  # stream s: frames of STREAM_SIZES[s]
STREAM_BATCHES = [([0, 1, 2, 0], None), ([1, 1, 2], None), ([2, 0, 1, 1], 1), ([0, 2], None), ([1, 0, 2, 2], 0)]


def _stream_lists(keep):
    """per batch: (ids, stream reset before it, descriptors with device NV12 among them, tight RGB frames)"""
    out = []
    for b, (ids, reset) in enumerate(STREAM_BATCHES):
        specs = [(*STREAM_SIZES[s], (NV12, RGB, BGR)[(i + b) % 3], ("device_pitched", "host", "device", "host_pitched")
                  [(i + 2 * b) % 4]) for i, s in enumerate(ids)]
        descs, rgb = _list(specs, 100 + b, keep)
        out.append((ids, reset, descs, rgb))
    assert any(d.format == NV12 and d.on_device for _, _, descs, _ in out for d in descs)
    return out


def test_streams_descs_equal_the_host_rgb_streams_entries(tmp_path):
    net = _detector(tmp_path, "tiny-yolo-voc", 4)
    keep = []
    try:
        batches = _stream_lists(keep)
        runs = []
        for use_descs in (False, True):
            dn.network_streams_open(net, 3)
            got = []
            for ids, reset, descs, rgb in batches:
                if reset is not None:
                    dn.network_stream_reset(net, reset)
                if use_descs:
                    got.append(dn.network_detect_streams_descs(net, ids, descs, THRESH, NMS, MAX_DET))
                else:
                    got.append(dn.network_detect_streams(net, ids, rgb, THRESH, NMS, MAX_DET))
            runs.append(got)
        for b, (want, got) in enumerate(zip(*runs)):
            assert got[1] == want[1], b
            _same_dets(got[0], want[0], f"batch {b}")
        # the same through the submit/wait pipeline, two batches in flight
        dn.network_streams_open(net, 3)
        for b, (ids, reset, descs, rgb) in enumerate(batches):
            if reset is not None:
                dn.network_stream_reset(net, reset)
            dn.network_detect_submit_streams_descs(net, ids, descs, THRESH, NMS, MAX_DET)
            if b:
                _same_dets(dn.network_detect_wait_n(net, len(batches[b - 1][0]), MAX_DET)[0], runs[0][b - 1][0],
                           f"pipelined batch {b - 1}")
        _same_dets(dn.network_detect_wait_n(net, len(batches[-1][0]), MAX_DET)[0], runs[0][-1][0], "last batch")
    finally:
        dn.free_network(net)


def test_tracked_streams_descs_equal_the_host_rgb_tracked_entries(tmp_path):
    net = _detector(tmp_path, "tiny-yolo-voc", 4)
    keep = []
    max_det = 64
    try:
        batches = _stream_lists(keep)
        runs = []
        for use_descs in (False, True):
            dn.network_streams_open(net, 3)
            dn.network_streams_track(net, 4)
            got = []
            for b, (ids, reset, descs, rgb) in enumerate(batches):
                use_mean = b % 2 == 0
                if reset is not None:
                    dn.network_stream_reset(net, reset)
                if use_descs:
                    got.append(dn.network_detect_streams_tracked_descs(net, ids, descs, THRESH, NMS, use_mean,
                                                                       max_det))
                else:
                    got.append(dn.network_detect_streams_tracked(net, ids, rgb, THRESH, NMS, use_mean, max_det))
            runs.append(got)
        assert any(len(r) for g in runs[0] for r in g[0]), "test needs tracked boxes"
        for b, (want, got) in enumerate(zip(*runs)):
            assert got[1] == want[1], b
            _same_dets(got[0], want[0], f"tracked batch {b}")
        dn.network_streams_open(net, 3)
        dn.network_streams_track(net, 4)
        for b, (ids, reset, descs, rgb) in enumerate(batches):
            if reset is not None:
                dn.network_stream_reset(net, reset)
            dn.network_detect_submit_streams_tracked_descs(net, ids, descs, THRESH, NMS, b % 2 == 0, max_det)
            if b:
                _same_dets(dn.network_detect_wait_tracked(net, len(batches[b - 1][0]), max_det)[0], runs[0][b - 1][0],
                           f"pipelined tracked batch {b - 1}")
        _same_dets(dn.network_detect_wait_tracked(net, len(batches[-1][0]), max_det)[0], runs[0][-1][0], "last")
    finally:
        dn.free_network(net)


# ---- pipeline -----------------------------------------------------------------------------------------------------
def _staged_descs(net, specs, seed, keep):
    """host frames written straight into the next slot's pinned buffer, device frames in torch allocations"""
    descs, rgb = _list(specs, seed, keep)
    views = dn.network_pipeline_staging_frame_descs(net, dn.lib().network_pipeline_next_slot(net), descs)
    out = []
    for d, v in zip(descs, views):
        if v is None:
            assert d.on_device
            out.append(d)
            continue
        v[...] = np.asarray(d._keep)
        out.append(dn.frame_desc(v, d.format))
    for d, v in zip(out, views):
        assert v is None or d.data == v.ctypes.data
    return out


def test_detect_pipeline_interleaves_frame_descs_with_frame_lists_and_u8(tmp_path):
    net = _detector(tmp_path, "tiny-yolo-voc", 3)
    lib, B = dn.lib(), net.batch
    keep = []
    try:
        d1, r1 = _list(_mixed([(1920, 1080), (640, 480), (376, 500)], 0), 5, keep)
        d2, r2 = _list(_mixed([(500, 376), (2, 2)], 1), 6, keep)
        rng = np.random.default_rng(7)
        lst = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for w, h in [(333, 517), (640, 480)]]
        u8 = rng.integers(0, 256, (B, 416, 416, 3), dtype=np.uint8)
        staged_specs = [(640, 480, NV12, "host"), (1280, 720, BGR, "device_pitched"), (500, 376, RGB, "host")]
        seq = [("descs", (d1, r1)), ("list", lst), ("u8", u8), ("staged", None), ("descs", (d2, r2)), ("list", lst),
               ("staged", None), ("descs", (d1, r1))]
        staged_rgb = _list(staged_specs, 8, keep)[1]
        want = []
        for kind, a in seq:  # the synchronous calls before anything is in flight
            if kind == "descs":
                want.append(dn.network_detect_frame_list(net, a[1], THRESH, NMS, MAX_DET)[0])
            elif kind == "staged":
                want.append(dn.network_detect_frame_list(net, staged_rgb, THRESH, NMS, MAX_DET)[0])
            elif kind == "list":
                want.append(dn.network_detect_frame_list(net, a, THRESH, NMS, MAX_DET)[0])
            else:
                want.append(dn.network_detect_batch(net, np.ascontiguousarray(
                    u8.transpose(0, 3, 1, 2).astype(np.float32) / np.float32(255.)), THRESH, NMS, MAX_DET)[0])

        def submit(kind, a):
            if kind == "descs":
                return dn.network_detect_submit_frame_descs(net, a[0], THRESH, NMS, MAX_DET)
            if kind == "staged":
                return dn.network_detect_submit_frame_descs(net, _staged_descs(net, staged_specs, 8, keep), THRESH, NMS,
                                                            MAX_DET)
            if kind == "list":
                return dn.network_detect_submit_frame_list(net, a, THRESH, NMS, MAX_DET)
            return lib.network_detect_submit_u8(net, dn._as_u8(a), THRESH, NMS, MAX_DET)

        def n_of(kind, a):
            return {"descs": lambda: len(a[0]), "staged": lambda: 3, "list": lambda: len(a), "u8": lambda: B}[kind]()

        submit(*seq[0])
        for i in range(1, len(seq)):
            submit(*seq[i])  # two batches in flight
            _same_dets(dn.network_detect_wait_n(net, n_of(*seq[i - 1]), MAX_DET)[0], want[i - 1], f"{i - 1}")
        _same_dets(dn.network_detect_wait_n(net, n_of(*seq[-1]), MAX_DET)[0], want[-1], "last")
    finally:
        dn.free_network(net)


def test_classify_pipeline_interleaves_frame_descs_with_frame_lists_and_u8(tmp_path):
    net = NETS["darknet19_448"](tmp_path)
    B, top = net.batch, 5
    keep = []
    try:
        d1, r1 = _list(_mixed([(1920, 1080), (376, 500)], 2), 5, keep)
        d2, r2 = _list(_mixed([(640, 480)], 0), 6, keep)
        rng = np.random.default_rng(9)
        u8 = rng.integers(0, 256, (B, net.h, net.w, 3), dtype=np.uint8)
        seq = [("descs", (d1, r1)), ("list", r2), ("u8", u8), ("descs", (d2, r2)), ("descs", (d1, r1))]
        want = [dn.network_classify_batch(net, frame_list=a[1] if k == "descs" else a, top=top) if k != "u8" else
                dn.network_classify_batch(net, images=np.ascontiguousarray(
                    u8.transpose(0, 3, 1, 2).astype(np.float32) / np.float32(255.)), top=top) for k, a in seq]

        def submit(kind, a):
            if kind == "descs":
                return dn.network_classify_submit_frame_descs(net, a[0], top=top)
            if kind == "list":
                return dn.network_classify_submit(net, frame_list=a, top=top)
            return dn.network_classify_submit(net, u8=a, top=top)

        def n_of(kind, a):
            return len(a[0]) if kind == "descs" else len(a) if kind == "list" else B

        submit(*seq[0])
        for i in range(1, len(seq)):
            submit(*seq[i])
            _same(dn.network_classify_wait(net, top=top, n=n_of(*seq[i - 1])), want[i - 1])
        _same(dn.network_classify_wait(net, top=top, n=n_of(*seq[-1])), want[-1])
    finally:
        dn.free_network(net)


# ---- the ready event ------------------------------------------------------------------------------------------------
def test_ready_event_orders_device_frames_written_on_another_stream(tmp_path):
    net = _detector(tmp_path, "tiny-yolo-voc", 3)
    keep = []
    try:
        specs = [(1920, 1080, NV12, "device_pitched"), (640, 480, BGR, "device"), (500, 376, RGB, "host")]
        src, rgb = _list(specs, 11, keep)
        want = dn.network_detect_frame_list(net, rgb, THRESH, NMS, MAX_DET)
        assert any(len(w) for w in want[0])
        # empty device frames of the same layout, filled on a side stream behind a sleep
        blank, _ = _list(specs, 11, keep)
        targets = []
        for d in blank:
            if d.on_device:
                for t in (d._keep if isinstance(d._keep, tuple) else (d._keep,)):
                    targets.append(t)
                    t.zero_()
        sources = [t for d in src if d.on_device for t in (d._keep if isinstance(d._keep, tuple) else (d._keep,))]
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        ready = torch.cuda.Event()
        with torch.cuda.stream(side):
            torch.cuda._sleep(200_000_000)
            for t, s in zip(targets, sources):
                t.copy_(s)
            ready.record(side)
        dn.network_detect_submit_frame_descs(net, [blank[0], blank[1], src[2]], THRESH, NMS, MAX_DET,
                                             ready=ready.cuda_event)
        got = dn.network_detect_wait_n(net, 3, MAX_DET)
        assert got[1] == want[1]
        _same_dets(got[0], want[0], "ready")
    finally:
        torch.cuda.synchronize()
        dn.free_network(net)


# ---- refusals -------------------------------------------------------------------------------------------------------
REFUSE = """
import sys, ctypes as C, numpy as np
sys.path.insert(0, {root!r})
from sr_object_detection_b200 import darknet as dn
dn.set_gpu_index(0)
net = dn.parse_network_cfg({cfg!r})
dn.load_weights(net, {weights!r})
lib = dn.lib()
host = np.zeros((64, 64, 3), np.uint8)
dev = dn._DevBuf(4096)


def desc(w=16, h=12, fmt=0, on_device=0, data=None, pitch=0, uv=None, uv_pitch=0):
    d = dn.FrameDesc()
    d.data = data if data is not None else (dev.ptr.value if on_device else host.ctypes.data)
    d.uv, d.w, d.h, d.pitch, d.uv_pitch, d.format, d.on_device = uv, w, h, pitch, uv_pitch, fmt, on_device
    return d


def submit(*descs, n=None):
    arr = (dn.FrameDesc * max(len(descs), 1))(*descs)
    lib.network_classify_submit_frame_descs(net, len(descs) if n is None else n, arr, None, 3)


{call}
print("RETURNED")
"""
REFUSALS = {
    "n0": ("submit(desc(), n=0)", "1 .. batch frames"),
    "n_over_batch": ("submit(desc(), desc(), desc())", "1 .. batch frames"),
    "null_descs": ("lib.network_classify_submit_frame_descs(net, 1, None, None, 3)", "NULL descriptor array"),
    "null_frame": ("submit(desc(), desc(data=0))", "NULL frame pointer"),
    "zero_size": ("submit(desc(w=0))", "frame size of 0 or less"),
    "format": ("submit(desc(fmt=3))", "unknown format"),
    "odd_nv12": ("submit(desc(fmt=2, w=15))", "even width and height"),
    "pitch": ("submit(desc(pitch=47))", "pitch smaller than the row"),
    "row_over_int_max": ("submit(desc(w=715827883, h=2))", "a row of more than INT_MAX bytes"),
    "uv_pitch": ("submit(desc(fmt=2, uv_pitch=15))", "uv_pitch smaller than the row"),
    "device_frame_in_host_memory": ("submit(desc(on_device=1, data=host.ctypes.data))", "not device or managed memory"),
    "device_frame_past_its_allocation": ("submit(desc(w=1920, h=1080, on_device=1))", "not device or managed memory"),
    "device_uv_in_host_memory": ("submit(desc(fmt=2, on_device=1, w=16, h=8, uv=host.ctypes.data))",
                                 "not device or managed memory"),
    "host_frame_in_device_memory": ("submit(desc(data=dev.ptr.value))", "in device memory"),
    "staging_format": ("dn.network_pipeline_staging_frame_descs(net, 0, [desc(fmt=9)])", "unknown format"),
}


@pytest.mark.parametrize("case", sorted(REFUSALS))
def test_frame_desc_refusals_exit_through_error(tmp_path, case):
    cfg_text = synth.exact_classifier_cfg(batch=2)
    (tmp_path / "n.cfg").write_text(cfg_text)
    synth.write_weights(tmp_path / "n.weights", cfg_text, seed=3)
    call, msg = REFUSALS[case]
    code = REFUSE.format(root=str(ROOT), cfg=str(tmp_path / "n.cfg"), weights=str(tmp_path / "n.weights"), call=call)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert r.returncode != 0 and "RETURNED" not in r.stdout, r.stdout
    assert msg in r.stderr, r.stderr[-2000:]
