"""Tiled detection, host side: the tile plan (y2_tile_plan) against the rule it implements, and a numpy restatement of
do_nms_sort, the tile-to-frame mapping and the final pick.  The restatement is checked against the reference's own
do_nms_sort results (tests/golden/region_*.npz) and is the reference the GPU tests use for unions larger than the
library's do_nms_sort stages."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

from sr_object_detection_b200 import _lib, darknet as dn

GOLDEN = Path(__file__).resolve().parent / "golden"
RGB, BGR, NV12 = dn.FRAME_RGB24, dn.FRAME_BGR24, dn.FRAME_NV12


# ---- the host chain: numpy restatement ------------------------------------------------------------------------------
def tile_geometry(W, H, fmt, cols, rows, overlap, full):
    """the tiles (x0, y0, tw, th) of one W x H frame, in order"""
    nv12 = fmt == NV12

    def extent(ext, k):
        t = min(ext, -(-(ext + (k - 1) * overlap) // k))
        return t + (t & 1) if nv12 else t

    def origin(i, k, ext, t):
        o = 0 if k == 1 else (i * (ext - t)) // (k - 1)
        return o & ~1 if nv12 else o

    tw, th = extent(W, cols), extent(H, rows)
    out = [(0, 0, W, H)] if full else []
    for j in range(rows):
        for i in range(cols):
            out.append((origin(i, cols, W, tw), origin(j, rows, H, th), tw, th))
    return out


def map_boxes(boxes, x0, y0, tw, th, W, H):
    """boxes [n][4] (x, y, w, h) relative to a tile -> relative to its frame, in float32 without contraction"""
    b = np.array(boxes, np.float32, copy=True)
    f = np.float32
    if not (x0 == 0 and tw == W):
        b[:, 0] = (f(x0) + b[:, 0] * f(tw)) / f(W)
        b[:, 2] = (b[:, 2] * f(tw)) / f(W)
    if not (y0 == 0 and th == H):
        b[:, 1] = (f(y0) + b[:, 1] * f(th)) / f(H)
        b[:, 3] = (b[:, 3] * f(th)) / f(H)
    return b


def _iou(a, b):
    """box_iou (box.c:67-97) of box a against the rows of b, in float32"""
    two = np.float32(2)

    def overlap(x1, w1, x2, w2):
        left = np.maximum(x1 - w1 / two, x2 - w2 / two)
        right = np.minimum(x1 + w1 / two, x2 + w2 / two)
        return right - left

    w = overlap(a[0], a[2], b[:, 0], b[:, 2])
    h = overlap(a[1], a[3], b[:, 1], b[:, 3])
    inter = np.where((w < 0) | (h < 0), np.float32(0), w * h).astype(np.float32)
    union = (a[2] * a[3] + b[:, 2] * b[:, 3]) - inter
    return inter / union


def do_nms_sort(boxes, probs, thresh):
    """box.c:249-277: per class in order, a stable sort of all boxes by that class's probability (descending) from the
    order the previous class left, then every box still non-zero zeroes the later boxes with IoU > thresh.  Returns the
    new probabilities; the arguments are not modified."""
    boxes = np.asarray(boxes, np.float32)
    probs = np.array(probs, np.float32, copy=True)
    thresh = np.float32(thresh)
    order = np.arange(probs.shape[0])
    for k in range(probs.shape[1]):
        order = order[np.argsort(-probs[order, k].astype(np.float64), kind="stable")]
        cand = order[probs[order, k] != 0]  # zero entries neither suppress nor change when suppressed
        for i in range(len(cand) - 1):
            if probs[cand[i], k] == 0:
                continue
            later = cand[i + 1:]
            hit = later[_iou(boxes[cand[i]], boxes[later]) > thresh]
            probs[hit, k] = 0
    return probs


def pick(boxes, probs, thresh):
    """the final pick of Detector::detect (max_index, first maximum; kept when > thresh) as y2_det rows"""
    arg = np.argmax(probs, axis=1)
    best = probs[np.arange(len(probs)), arg]
    keep = np.nonzero(best > np.float32(thresh))[0]
    out = np.zeros(len(keep), dtype=np.dtype(dn.Detection))
    for f in ("x", "y", "w", "h"):
        out[f] = boxes[keep, "xywh".index(f)]
    out["prob"], out["obj_id"], out["box_index"] = best[keep], arg[keep], keep
    return out


def merge(tile_boxes, tile_probs, geoms, W, H, thresh, nms):
    """the tiles of one frame (boxes and probabilities relative to each tile) -> the frame's y2_det rows and the
    union before / after NMS"""
    boxes = np.concatenate([map_boxes(b, *g, W, H) for b, g in zip(tile_boxes, geoms)])
    pre = np.concatenate(tile_probs)
    post = do_nms_sort(boxes, pre, nms) if nms > 0 else pre
    return pick(boxes, post, thresh), boxes, pre, post


@pytest.mark.parametrize("name", sorted(p.stem for p in GOLDEN.glob("region_*.npz")))
def test_numpy_do_nms_sort_reproduces_the_reference(name):
    d = np.load(GOLDEN / f"{name}.npz")
    batch = d["region_in"].shape[0]
    boxes = d["boxes"].reshape(batch, -1, 4)
    pre = d["probs_pre"].reshape(batch, boxes.shape[1], -1)
    post = d["probs_post"].reshape(pre.shape)
    assert (pre != post).any(), "the fixture must suppress something"
    for b in range(batch):
        got = do_nms_sort(boxes[b], pre[b], float(d["nms"]))
        assert got.tobytes() == post[b].tobytes(), f"{name} image {b}"


def test_map_boxes_identity_and_rounding():
    rng = np.random.default_rng(1)
    b = rng.random((50, 4), dtype=np.float32)
    assert map_boxes(b, 0, 0, 640, 480, 640, 480).tobytes() == b.tobytes()
    m = map_boxes(b, 0, 37, 640, 200, 640, 480)
    assert m[:, [0, 2]].tobytes() == b[:, [0, 2]].tobytes()
    x = float(np.float32(np.float32(np.float32(37) + b[3, 1] * np.float32(200)) / np.float32(480)))
    assert m[3, 1] == np.float32(x)


# ---- the plan -----------------------------------------------------------------------------------------------------
PLAN_CASES = [  # (W, H, format, cols, rows, overlap, full)
    (1920, 1080, RGB, 3, 2, 64, 1),
    (1920, 1080, NV12, 3, 2, 64, 1),
    (1920, 1080, BGR, 2, 2, 64, 0),
    (100, 50, RGB, 2, 3, 400, 0),        # tiles wider than the frame
    (641, 480, BGR, 1, 3, 16, 1),        # one column
    (333, 517, RGB, 5, 7, 31, 0),        # odd sizes
    (1282, 722, NV12, 3, 3, 63, 0),      # odd overlap, odd tile before rounding
    (1278, 718, NV12, 4, 5, 0, 1),
    (2, 2, NV12, 16, 16, 5, 1),
    (1, 1, RGB, 16, 16, 0, 0),
    (4000, 30, RGB, 16, 1, 1000, 0),     # large overlap
    (1000, 700, RGB, 7, 4, 0, 0),
]
PLAN_IDS = [f"{c[0]}x{c[1]}f{c[2]}_{c[3]}x{c[4]}o{c[5]}F{c[6]}" for c in PLAN_CASES]


def _fake_desc(W, H, fmt, on_device, data=0x10000000, pitch=0, uv=0, uv_pitch=0):
    d = dn.FrameDesc()
    d.data, d.uv, d.w, d.h, d.pitch, d.uv_pitch, d.format, d.on_device = data, uv or None, W, H, pitch, uv_pitch, fmt, \
        on_device
    return d


def _bpp(fmt):
    return 1 if fmt == NV12 else 3


@pytest.mark.parametrize("case", PLAN_CASES, ids=PLAN_IDS)
def test_plan_matches_the_rule_and_the_crop_descriptors(case):
    W, H, fmt, cols, rows, overlap, full = case
    pitch = W * _bpp(fmt) + 40
    uv, uv_pitch = (0x30000000, W + 8) if fmt == NV12 else (0, 0)
    dev = _fake_desc(W, H, fmt, 1, pitch=pitch, uv=uv, uv_pitch=uv_pitch)
    host = _fake_desc(W, H, fmt, 0)
    tiling = dn.Tiling(cols, rows, overlap, full)
    geoms = tile_geometry(W, H, fmt, cols, rows, overlap, full)
    n_t = len(geoms)
    rc, lay, recs, tiles, spans = _lib.tile_plan([host, dev, host], tiling, 416, 320, 3 * n_t)
    assert rc == 0
    assert lay.n_tiles == 3 * n_t and lay.max_tiles == n_t
    assert [(s.first, s.count) for s in spans] == [(0, n_t), (n_t, n_t), (2 * n_t, n_t)]
    assert [(t.frame, t.x0, t.y0, t.w, t.h, t.frame_w, t.frame_h) for t in tiles] == \
        [(f, *g, W, H) for f in range(3) for g in geoms]
    frame_recs, _, _ = _lib.frame_desc_layout([host, dev, host], 416, 320, False)
    for t, (x0, y0, tw, th) in enumerate(geoms):
        # a device frame's tile: exactly the record of a descriptor of the crop, read with the frame's pitch
        crop = _fake_desc(tw, th, fmt, 1, data=dev.data + y0 * pitch + x0 * _bpp(fmt), pitch=pitch,
                          uv=(uv + (y0 // 2) * uv_pitch + x0) if fmt == NV12 else 0, uv_pitch=uv_pitch)
        want = _lib.frame_desc_layout([crop], 416, 320, False)[0][0]
        assert bytes(recs[n_t + t]) == bytes(want), (t, x0, y0)
        # a host frame's tile: the same window at the frame's one staged copy (tight rows)
        for f in (0, 2):
            fr, r = frame_recs[f], recs[f * n_t + t]
            row = W * _bpp(fmt)
            assert r.pitch == row and bytes(r.win)[8:] == bytes(want.win)[8:]
            assert r.win.offset == fr.win.offset + y0 * row + x0 * _bpp(fmt)
            if fmt == NV12:
                assert r.uv == fr.uv + (y0 // 2) * row + x0 and r.uv_pitch == row


@pytest.mark.parametrize("case", PLAN_CASES, ids=PLAN_IDS)
def test_tiles_cover_the_frame_and_overlap(case):
    W, H, fmt, cols, rows, overlap, full = case
    rc, lay, recs, tiles, spans = _lib.tile_plan([_fake_desc(W, H, fmt, 0)], dn.Tiling(cols, rows, overlap, full),
                                                 416, 416, 1000)
    assert rc == 0
    if full:
        assert (tiles[0].x0, tiles[0].y0, tiles[0].w, tiles[0].h) == (0, 0, W, H)
    grid = tiles[full:]
    assert len(grid) == cols * rows
    cover = np.zeros((H, W), np.int32)
    for t in grid:
        assert 0 <= t.x0 and t.x0 + t.w <= W and 0 <= t.y0 and t.y0 + t.h <= H
        cover[t.y0:t.y0 + t.h, t.x0:t.x0 + t.w] += 1
        if fmt == NV12:
            assert t.x0 % 2 == 0 and t.y0 % 2 == 0 and t.w % 2 == 0 and t.h % 2 == 0
    assert (cover > 0).all()
    need = max(overlap - (fmt == NV12), 0)
    for j in range(rows):  # row-major, left to right then top to bottom
        for i in range(cols):
            t = grid[j * cols + i]
            if i:
                left = grid[j * cols + i - 1]
                assert left.y0 == t.y0 and left.x0 <= t.x0
                assert left.x0 + left.w - t.x0 >= min(need, W)
            if j:
                up = grid[(j - 1) * cols + i]
                assert up.x0 == t.x0 and up.y0 <= t.y0
                assert up.y0 + up.h - t.y0 >= min(need, H)
    assert grid[0].x0 == 0 and grid[0].y0 == 0
    assert grid[-1].x0 + grid[-1].w == W and grid[-1].y0 + grid[-1].h == H


def test_each_host_frame_is_staged_once_and_device_frames_take_no_bytes():
    host = [_fake_desc(1920, 1080, NV12, 0), _fake_desc(333, 517, RGB, 0)]
    dev = [_fake_desc(1920, 1080, BGR, 1), _fake_desc(640, 480, NV12, 1, uv=0x30000000)]
    tiling = dn.Tiling(3, 2, 64, 1)
    frames = (1920 * 1080 * 3 // 2 + 15) // 16 * 16 + (333 * 517 * 3 + 15) // 16 * 16
    for descs in (host, host + dev, dev + host, dev):
        rc, lay, recs, tiles, spans = _lib.tile_plan(descs, tiling, 416, 416, 64)
        assert rc == 0
        assert lay.recs_offset == _lib.frame_desc_layout(descs, 416, 416, False)[1]
        assert lay.recs_offset == (frames if any(not d.on_device for d in descs) else 0)
        assert lay.tiles_offset == lay.recs_offset + lay.n_tiles * C.sizeof(_lib.FrameSrc)
        assert lay.spans_offset >= lay.tiles_offset + lay.n_tiles * C.sizeof(_lib.Tile)
        assert lay.bytes == lay.spans_offset + len(descs) * C.sizeof(_lib.TileSpan)
        for t, r in zip(tiles, recs):
            if descs[t.frame].on_device:
                assert r.win.offset >= 0x10000000
            else:
                assert r.win.offset < frames


@pytest.mark.parametrize("tiling,max_tiles,descs,code", [
    (None, 64, None, 2),
    ((0, 1, 0, 0), 64, None, 3),
    ((17, 1, 0, 0), 64, None, 3),
    ((1, 0, 0, 0), 64, None, 3),
    ((1, 17, 0, 0), 64, None, 3),
    ((2, 2, -1, 0), 64, None, 4),
    ((2, 2, 0, 2), 64, None, 5),
    ((2, 2, 0, -1), 64, None, 5),
    ((2, 2, 64, 1), 9, None, 6),   # 2 frames x 5 tiles
    ((2, 2, 64, 1), 10, None, 0),
    ((2, 2, 0, 0), 64, "odd_nv12", 1),
    ((2, 2, 0, 0), 64, "empty", 1),
])
def test_plan_refusals_return_their_code(tiling, max_tiles, descs, code):
    good = [_fake_desc(640, 480, RGB, 0), _fake_desc(1920, 1080, NV12, 0)]
    lst = {None: good, "odd_nv12": [_fake_desc(641, 480, NV12, 0)], "empty": []}[descs]
    t = dn.Tiling(*tiling) if tiling is not None else None
    assert _lib.tile_plan(lst, t, 416, 416, max_tiles)[0] == code
    assert _lib.load().y2_abi_sizeof(8) == C.sizeof(dn.Tiling)
