"""Tiled detection (network_*_tiled_descs) against the host chain: each tile run as an ordinary frame descriptor of
the crop (the existing entry, pinned to the host chain by test_frame_src_gpu), get_region_boxes per tile, then the
numpy restatement of the mapping, the union's do_nms_sort and the pick (tests/test_tiled_host.py).  Every comparison is
bit for bit."""
import ctypes as C
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from sr_object_detection_b200 import darknet as dn, synth
from tests.test_frame_list_gpu import _detector, _same_dets
from tests.test_frame_src_gpu import _list, _mixed
from tests.test_tiled_host import merge, tile_geometry

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
RGB, BGR, NV12 = dn.FRAME_RGB24, dn.FRAME_BGR24, dn.FRAME_NV12
NMS, MAX_DET = 0.45, 4096
SMEM_CANDIDATES = 2048  # candidates of one class a block of y2_tile_nms stages in shared memory


def _crop(d, x0, y0, tw, th):
    """a descriptor of the tile (x0, y0, tw, th) of frame d, read in place with the frame's pitch"""
    bpp = 1 if d.format == NV12 else 3
    pitch = d.pitch or d.w * bpp
    c = dn.FrameDesc()
    c.data = d.data + y0 * pitch + x0 * bpp
    c.w, c.h, c.pitch, c.format, c.on_device = tw, th, pitch, d.format, d.on_device
    if d.format == NV12:
        uv, uv_pitch = (d.uv or d.data + d.h * pitch), (d.uv_pitch or pitch)
        c.uv, c.uv_pitch = uv + (y0 // 2) * uv_pitch + x0, uv_pitch
    c._keep = d._keep
    return c


def _tile_outputs(net, descs, tiling):
    """per frame: its tiles' geometry, and a function thresh -> the tiles' (boxes, probs) relative to each tile, from
    the crops run through network_detect_frame_descs and get_region_boxes"""
    geoms = [tile_geometry(d.w, d.h, d.format, *tiling) for d in descs]
    crops = [_crop(d, *g) for d, gs in zip(descs, geoms) for g in gs]
    outputs = []  # region outputs per chunk of net.batch crops
    l = dn.region_layer(net)
    for i in range(0, len(crops), net.batch):
        chunk = crops[i:i + net.batch]
        dn.network_detect_frame_descs(net, chunk, 0.5, NMS, 1)
        outputs.append((len(chunk), dn.get_network_output_layer(net, net.n - 1).copy()))

    def at(thresh):
        boxes, probs = [], []
        for n, out in outputs:
            C.memmove(l.output, out.ctypes.data, out.nbytes)  # the host l.output get_region_boxes reads
            for b in range(n):
                bx, pr = dn.get_region_boxes(net, b, thresh)
                boxes.append(bx)
                probs.append(pr)
        per_frame, k = [], 0
        for gs in geoms:
            per_frame.append((boxes[k:k + len(gs)], probs[k:k + len(gs)]))
            k += len(gs)
        return per_frame

    return geoms, at


def _low_thresh(per_frame, target=2600):
    """a thresh at which the class with the most candidates of one frame's union has `target` of them"""
    t = 0.0
    for _, probs in per_frame:
        u = np.concatenate(probs)
        t = max(t, float(np.sort(u, axis=0)[::-1][min(target, len(u) - 1)].max()))
    return t


def _host_chain(descs, geoms, per_frame, thresh, nms, library_nms):
    """the frames' y2_det rows by the numpy chain; with library_nms each union's do_nms_sort is also checked against
    the library's dn.do_nms_sort"""
    out = []
    for d, gs, (boxes, probs) in zip(descs, geoms, per_frame):
        dets, ub, pre, post = merge(boxes, probs, gs, d.w, d.h, thresh, nms)
        if library_nms:
            lp = pre.copy()
            dn.do_nms_sort(np.ascontiguousarray(ub), lp, nms)
            assert lp.tobytes() == post.tobytes(), "numpy do_nms_sort != the library's on the union"
        out.append(dets)
    return out


def _check(got, want, max_det, what):
    dets, counts = got
    assert counts == [len(w) for w in want], what
    _same_dets(dets, [w[:max_det] for w in want], what)


# ---- 1 x 1 without the whole frame is the plain descriptor entry --------------------------------------------------
SIZES = [(500, 376), (1920, 1080), (416, 416), (640, 480), (2, 2), (354, 500), (1280, 720), (334, 518)]


@pytest.mark.parametrize("name", ["tiny-yolo-voc", "yolo-voc"])
def test_one_by_one_equals_the_frame_descs_entry(tmp_path, name):
    net = _detector(tmp_path, name, 4)
    keep = []
    try:
        for sizes, seed in ((SIZES[:4], 1), (SIZES[4:], 2), (SIZES[1:2], 3)):
            for shift in range(3):
                descs, _ = _list(_mixed(sizes, shift + seed), seed * 10 + shift, keep)
                want = dn.network_detect_frame_descs(net, descs, 0.02, NMS, 256)
                assert any(len(w) for w in want[0])
                for tiling in ((1, 1, 0, 0), (1, 1, 64, 0)):
                    got = dn.network_detect_tiled_descs(net, descs, tiling, 0.02, NMS, 256)
                    assert got[1] == want[1], (sizes, tiling)
                    _same_dets(got[0], want[0], f"{name} {sizes} {tiling}")
    finally:
        dn.free_network(net)


# ---- against the host chain -----------------------------------------------------------------------------------------
TILED_SPECS = [(1920, 1080, NV12, "device_pitched"), (333, 517, BGR, "host_pitched")]


@pytest.mark.parametrize("tiling", [(2, 2, 64, 1), (3, 2, 0, 0)], ids=["2x2o64full", "3x2o0"])
@pytest.mark.parametrize("name", ["tiny-yolo-voc", "yolo-voc"])
def test_tiled_equals_the_host_chain(tmp_path, name, tiling):
    net = _detector(tmp_path, name, 12)
    keep = []
    try:
        descs, _ = _list(TILED_SPECS, 21, keep)
        geoms, at = _tile_outputs(net, descs, tiling)
        low = _low_thresh(at(0.0))
        for thresh in (0.24, 0.02, low):
            per_frame = at(thresh)
            most = max(int((np.concatenate(p) != 0).sum(axis=0).max()) for _, p in per_frame)
            if thresh == low:
                assert most > SMEM_CANDIDATES, most  # the spill path runs
            want = _host_chain(descs, geoms, per_frame, thresh, NMS, library_nms=True)
            got = dn.network_detect_tiled_descs(net, descs, tiling, thresh, NMS, MAX_DET)
            _check(got, want, MAX_DET, f"{name} {tiling} thresh {thresh}")
            if thresh == 0.02:
                assert any(len(w) for w in want)
                # nms <= 0: the union unsuppressed
                want0 = _host_chain(descs, geoms, per_frame, thresh, 0.0, library_nms=False)
                _check(dn.network_detect_tiled_descs(net, descs, tiling, thresh, 0.0, MAX_DET), want0, MAX_DET,
                       "no nms")
    finally:
        dn.free_network(net)


def test_yolo_608_three_by_two_with_the_whole_frame(tmp_path):
    """12 635 boxes in the union, beyond what the library's do_nms_sort stages"""
    net = _detector_608(tmp_path)
    keep = []
    try:
        tiling = (3, 2, 64, 1)
        descs, _ = _list([(1920, 1080, NV12, "device")], 31, keep)
        geoms, at = _tile_outputs(net, descs, tiling)
        l = dn.region_layer(net)
        assert len(geoms[0]) * l.w * l.h * l.n == 12635
        for thresh in (0.24, _low_thresh(at(0.0), 2300)):
            want = _host_chain(descs, geoms, at(thresh), thresh, NMS, library_nms=False)
            got = dn.network_detect_tiled_descs(net, descs, tiling, thresh, NMS, MAX_DET)
            _check(got, want, MAX_DET, f"yolo 608 thresh {thresh}")
        assert any(len(w) for w in want)
    finally:
        dn.free_network(net)


def _detector_608(tmp_path):
    text = synth.CFGS["yolo"](batch=7, w=608, h=608)
    (tmp_path / "yolo.cfg").write_text(text)
    synth.write_weights(tmp_path / "yolo.weights", text, seed=1234)
    dn.set_gpu_index(0)
    net = dn.parse_network_cfg(tmp_path / "yolo.cfg")
    dn.load_weights(net, tmp_path / "yolo.weights")
    return net


# ---- max_det, the pipeline ------------------------------------------------------------------------------------------
def test_max_det_cuts_the_lists_and_counts_hold_the_full_number(tmp_path):
    net = _detector(tmp_path, "tiny-yolo-voc", 12)
    keep = []
    try:
        descs, _ = _list(TILED_SPECS, 41, keep)
        full = dn.network_detect_tiled_descs(net, descs, (2, 2, 64, 1), 0.02, NMS, MAX_DET)
        assert max(full[1]) > 3 and max(full[1]) < MAX_DET
        for max_det in (1, 3):
            got = dn.network_detect_tiled_descs(net, descs, (2, 2, 64, 1), 0.02, NMS, max_det)
            assert got[1] == full[1]
            _same_dets(got[0], [f[:max_det] for f in full[0]], f"max_det {max_det}")
    finally:
        dn.free_network(net)


def test_pipeline_interleaves_tiled_batches_with_frame_lists_streams_and_u8(tmp_path):
    net = _detector(tmp_path, "tiny-yolo-voc", 12)
    lib, B = dn.lib(), net.batch
    keep = []
    try:
        t1, _ = _list(TILED_SPECS, 51, keep)
        t2, _ = _list([(1280, 720, RGB, "host"), (640, 480, NV12, "host"), (500, 376, BGR, "device")], 52, keep)
        rng = np.random.default_rng(53)
        lst = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for w, h in [(333, 517), (640, 480)]]
        u8 = rng.integers(0, 256, (B, 416, 416, 3), dtype=np.uint8)
        seq = [("tiled", (t1, (2, 2, 64, 1))), ("list", lst), ("streams", ([0, 1], lst)),
               ("tiled", (t2, (2, 1, 32, 1))), ("u8", u8), ("tiled", (t1, (3, 2, 0, 0))), ("streams", ([1, 0], lst)), ("tiled", (t2, (1, 1, 0, 0)))]

        def run(kind, a, submit):
            if kind == "tiled":
                f = dn.network_detect_submit_tiled_descs if submit else dn.network_detect_tiled_descs
                return f(net, a[0], a[1], 0.02, NMS, 256)
            if kind == "list":
                f = dn.network_detect_submit_frame_list if submit else dn.network_detect_frame_list
                return f(net, a, 0.02, NMS, 256)
            if kind == "streams":
                f = dn.network_detect_submit_streams if submit else dn.network_detect_streams
                return f(net, a[0], a[1], 0.02, NMS, 256)
            if submit:
                return lib.network_detect_submit_u8(net, dn._as_u8(a), 0.02, NMS, 256)
            return dn.network_detect_batch(net, np.ascontiguousarray(
                a.transpose(0, 3, 1, 2).astype(np.float32) / np.float32(255.)), 0.02, NMS, 256)

        def n_of(kind, a):
            return {"tiled": lambda: len(a[0]), "list": lambda: len(a), "streams": lambda: len(a[0]),
                    "u8": lambda: B}[kind]()

        dn.network_streams_open(net, 2)
        want = [run(k, a, False)[0] for k, a in seq]
        assert any(len(w) for w in want[0])
        dn.network_streams_open(net, 2)
        run(*seq[0], True)
        for i in range(1, len(seq)):
            run(*seq[i], True)  # two batches in flight
            _same_dets(dn.network_detect_wait_n(net, n_of(*seq[i - 1]), 256)[0], want[i - 1], f"{i - 1}")
        _same_dets(dn.network_detect_wait_n(net, n_of(*seq[-1]), 256)[0], want[-1], "last")
    finally:
        dn.free_network(net)


# ---- refusals -------------------------------------------------------------------------------------------------------
REFUSE = """
import sys, ctypes as C, numpy as np
sys.path.insert(0, {root!r})
from sr_object_detection_b200 import darknet as dn
dn.set_gpu_index(0)
net = dn.parse_network_cfg({cfg!r})
{load}
lib = dn.lib()
host = np.zeros((64, 64, 3), np.uint8)


def desc(w=16, h=12):
    d = dn.FrameDesc()
    d.data, d.w, d.h, d.format = host.ctypes.data, w, h, dn.FRAME_RGB24
    return d


def submit(tiling, *descs, n=None):
    arr = (dn.FrameDesc * max(len(descs), 1))(*descs)
    t = C.byref(dn.Tiling(*tiling)) if tiling is not None else None
    lib.network_detect_submit_tiled_descs(net, len(descs) if n is None else n, arr, t, None, .24, .45, 16)


{call}
print("RETURNED")
"""
REFUSALS = {
    "n0": ("submit((1, 1, 0, 0), desc(), n=0)", "1 .. batch frames"),
    "n_over_batch": ("submit((1, 1, 0, 0), *[desc()] * 5)", "1 .. batch frames"),
    "desc_rule": ("submit((1, 1, 0, 0), desc(w=0))", "frame size of 0 or less"),
    "null_tiling": ("submit(None, desc())", "NULL tiling"),
    "cols0": ("submit((0, 1, 0, 0), desc())", "cols and rows must be in 1 .. Y2_TILE_MAX"),
    "cols17": ("submit((17, 1, 0, 0), desc())", "cols and rows must be in 1 .. Y2_TILE_MAX"),
    "rows17": ("submit((1, 17, 0, 0), desc())", "cols and rows must be in 1 .. Y2_TILE_MAX"),
    "overlap": ("submit((2, 2, -1, 0), desc())", "overlap must be 0 or more"),
    "full": ("submit((2, 2, 0, 2), desc())", "full must be 0 or 1"),
    "too_many_tiles": ("submit((2, 2, 8, 0), desc(), desc())", "more tiles than the network's batch"),
    "batch_entry_too_many_tiles": ("lib.network_detect_batch_tiled_descs(net, 1, (dn.FrameDesc * 1)(desc()), "
                                   "C.byref(dn.Tiling(5, 1, 0, 0)), None, .24, .45, None, None, 16)",
                                   "more tiles than the network's batch"),
    "softmax_tree": ("submit((1, 1, 0, 0), desc())", "softmax-tree heads are not supported"),
}


@pytest.mark.parametrize("case", sorted(REFUSALS))
def test_tiled_refusals_exit_through_error(tmp_path, case):
    if case == "softmax_tree":
        d = np.load(ROOT / "tests" / "golden" / "mini_yolo_tree.npz")
        (tmp_path / "t.tree").write_text(str(d["aux_t_tree"]))
        (tmp_path / "n.cfg").write_text(str(d["cfg"]).replace("batch=1", "batch=4", 1))
        (tmp_path / "n.weights").write_bytes(d["weights"].tobytes())
        load = f"dn.load_weights(net, {str(tmp_path / 'n.weights')!r})"
    else:
        cfg_text = synth.exact_detector_cfg(batch=4)
        (tmp_path / "n.cfg").write_text(cfg_text)
        synth.write_exact_weights(tmp_path / "n.weights", cfg_text)
        load = f"dn.load_weights(net, {str(tmp_path / 'n.weights')!r})"
    call, msg = REFUSALS[case]
    code = REFUSE.format(root=str(ROOT), cfg=str(tmp_path / "n.cfg"), load=load, call=call)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode != 0 and "RETURNED" not in r.stdout, r.stdout
    assert msg in r.stderr, r.stderr[-2000:]
