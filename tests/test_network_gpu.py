"""End-to-end GPU parity: the drop-in C API (parse_network_cfg / load_weights / network_predict /
get_region_boxes / do_nms_sort) on the B200 against the reference's CPU implementation on the
same seeded synthetic weights and images: the reference itself (oracle/_ref/darknet_ref) where its
sources were compiled, else the in-tree oracle port (oracle/y2_oracle.c).  tests/test_oracle_golden.py
pins the port bit for bit to stored reference outputs of the layer types it restates; cfgs with
layer types it does not restate (REF_ONLY) are checked against the compiled reference only.

Tolerances (north star): layer activations max|a-b| / max|b| <= 1e-2 (bf16 operands, fp32
accumulate); box indices and the post-NMS keep set bit-exact on identical region inputs.
"""
import numpy as np
import pytest

from sr_object_detection_b200 import darknet as dn
from sr_object_detection_b200 import synth
from tests import ref_util as R

pytestmark = pytest.mark.gpu

ACT_TOL = 1e-2
# connected / dropout layers, elu / tanh, reverse reorg: not restated by the oracle port
REF_ONLY = {"mini-alexnet", "mini-reorg-reverse"}


def _setup(tmp_path, name, batch, w=416, h=416, **kw):
    cfg_text = synth.CFGS[name](batch=batch, w=w, h=h, **kw)
    cfg = tmp_path / f"{name}.cfg"
    cfg.write_text(cfg_text)
    weights = tmp_path / f"{name}.weights"
    synth.write_weights(weights, cfg_text, seed=1234)
    x = synth.images(batch, 3, h, w, seed=42)
    inp = tmp_path / "input.f32"
    x.tofile(inp)
    return cfg, weights, x, inp


@pytest.mark.parametrize("name,batch,side", [("tiny-yolo-voc", 2, 416), ("yolo-voc", 2, 416), ("yolo", 1, 608),
                                             ("darknet19_448", 1, 448), ("yolo-voc", 3, 320),
                                             ("resnet50", 2, 256), ("resnet50", 1, 224),
                                             ("yolo9000", 1, 544),
                                             # non-square and odd extents: 15x11 and 13x9 cells, 2/1 pool on an odd row count
                                             ("tiny-yolo-voc", 2, (480, 352)), ("yolo-voc", 1, (416, 288)),
                                             # nested routes (a route that concatenates another route's output)
                                             ("mini-dense", 3, 64),
                                             # concat inputs with padding channels (48 / 24 / 40 filters): packed by copies
                                             ("mini-dense-odd", 3, 64),
                                             # classifier cfgs: connected / dropout layers, relu / elu / tanh
                                             ("mini-alexnet", 3, 32),
                                             # depth-to-space: a reorg layer with reverse=1
                                             ("mini-reorg-reverse", 2, 32)])
def test_layer_activations_match_reference(tmp_path, name, batch, side):
    """BASELINE.json configs 1-5 (at a batch the CPU reference finishes in seconds): every layer of
    the B200 forward pass against the reference's CPU forward on the same weights and images."""
    if name in REF_ONLY and not R.have_ref():
        pytest.skip(f"{name} needs the compiled reference (oracle/_ref/darknet_ref): the oracle port does not restate "
                    "its layer types")
    kw = {}
    if name == "yolo9000":  # config 4: 9418-way WordTree softmax (cfg/9k.tree of the reference is corrupt)
        synth.write_tree(tmp_path / "9k.tree")
        kw["tree"] = str(tmp_path / "9k.tree")
    w, h = side if isinstance(side, tuple) else (side, side)
    cfg, weights, x, inp = _setup(tmp_path, name, batch, w=w, h=h, **kw)
    ref_dir = tmp_path / "ref"
    R.forward(R.checker_bin(), cfg, weights, inp, ref_dir, thresh=0.24, nms=0.4)

    dn.set_gpu_index(0)
    net = dn.parse_network_cfg(cfg)
    dn.load_weights(net, weights)
    out = dn.network_predict(net, x)
    worst = (0.0, -1)
    for i in range(net.n):
        l = net.layers[i]
        if l.type == dn.COST:
            continue
        ref = R.load(ref_dir, "layer_%03d.f32" % i, (batch, l.outputs))
        got = dn.get_network_output_layer(net, i)
        err = float(np.abs(got - ref).max() / max(np.abs(ref).max(), 1e-30))
        worst = max(worst, (err, i))
        assert err <= ACT_TOL, f"{name} layer {i} (type {l.type}): max err / max|ref| = {err:.3e}"
    ref_out = R.load(ref_dir, "output.f32", out.shape)
    err = float(np.abs(out - ref_out).max() / np.abs(ref_out).max())
    assert err <= ACT_TOL, f"network output err {err:.3e}"
    print(f"{name}: worst layer error {worst[0]:.3e} at layer {worst[1]}, output err {err:.3e}")
    dn.free_network(net)


@pytest.mark.parametrize("name,classes,n,side,thresh,nms", [
    ("yolo-voc", 20, 5, 13, 0.24, 0.4),
    ("yolo-voc", 20, 5, 13, 0.005, 0.45),
    ("yolo", 80, 5, 19, 0.24, 0.4),
])
def test_decode_and_nms_bit_exact_on_identical_region_inputs(tmp_path, name, classes, n, side, thresh, nms):
    """Region forward + get_region_boxes + do_nms_sort: device kernels vs the reference's C code
    on the SAME region-layer input tensor."""
    import ctypes as C
    import torch
    from sr_object_detection_b200 import _lib
    batch = 3
    wh = side * 32
    cfg_text = synth.CFGS[name](batch=batch, w=wh, h=wh)
    cfg = tmp_path / "net.cfg"
    cfg.write_text(cfg_text)
    x = synth.region_inputs(batch, n, classes, side, side, seed=11)
    rin = tmp_path / "region_in.f32"
    x.tofile(rin)
    ref_dir = tmp_path / "ref"
    R.region(R.checker_bin(), cfg, rin, ref_dir, thresh=thresh, nms=nms)
    total = side * side * n
    size = classes + 5
    ref_out = R.load(ref_dir, "region_out.f32", (batch, total, size))
    ref_boxes = R.load(ref_dir, "boxes.f32", (batch, total, 4))
    ref_pre = R.load(ref_dir, "probs_pre.f32", (batch, total, classes))
    ref_post = R.load(ref_dir, "probs_post.f32", (batch, total, classes))

    lib = _lib.load()
    dev = torch.device("cuda:0")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    xin = torch.from_numpy(x).to(dev)
    flat = torch.empty(batch, side * side, n * size, device=dev)
    _lib.check(lib.y2_nchw_to_flat_f32(xin.data_ptr(), flat.data_ptr(), batch, n * size, side * side, st))
    out = torch.empty_like(flat)
    _lib.check(lib.y2_region_forward(flat.data_ptr(), out.data_ptr(), batch, side * side, n, classes, 1, 0,
                                     None, None, st))
    anchors = [float(v) for v in (synth.VOC_ANCHORS if classes == 20 else synth.COCO_ANCHORS).split(",")]
    biases = torch.tensor(anchors, device=dev)
    boxes = torch.empty(batch, total, 4, device=dev)
    probs = torch.empty(batch, total, classes, device=dev)
    _lib.check(lib.y2_region_boxes(out.data_ptr(), biases.data_ptr(), boxes.data_ptr(), probs.data_ptr(), batch,
                                   side, side, n, classes, 1.0, 1.0, thresh, 0, 0, 0, None, None, 0, st))
    pre = probs.clone()
    _lib.check(lib.y2_nms_sort(boxes.data_ptr(), probs.data_ptr(), batch, total, classes, nms, st))
    torch.cuda.synchronize()
    got_out = out.view(batch, total, size).cpu().numpy()
    got_boxes = boxes.cpu().numpy()
    got_pre = pre.cpu().numpy()
    got_post = probs.cpu().numpy()
    # values: identical expressions, double exp on both sides -> expect bit equality
    assert np.array_equal(got_out, ref_out), f"region output differs in {(got_out != ref_out).sum()} values"
    assert np.array_equal(got_boxes, ref_boxes), f"boxes differ in {(got_boxes != ref_boxes).sum()} values"
    assert np.array_equal(got_pre, ref_pre)
    # the keep set, and the kept values
    assert np.array_equal(got_post != 0, ref_post != 0), \
        f"keep set differs in {((got_post != 0) != (ref_post != 0)).sum()} entries"
    assert np.array_equal(got_post, ref_post)
    assert (ref_pre != 0).sum() > (ref_post != 0).sum() > 0  # the case actually suppresses something


def test_pipelined_submit_wait_equals_synchronous_detect(tmp_path):
    """network_detect_submit / network_detect_wait (two batches in flight, H2D of batch i+1 overlapping
    the forward of batch i) must hand out exactly the detections of the synchronous
    network_detect_batch, batch by batch and in submission order."""
    import ctypes as C
    batch, max_det = 4, 256
    cfg, weights, _, _ = _setup(tmp_path, "tiny-yolo-voc", batch)
    dn.set_gpu_index(0)
    net = dn.parse_network_cfg(cfg)
    dn.load_weights(net, weights)
    lib = dn.lib()
    batches = [synth.images(batch, 3, 416, 416, seed=100 + i) for i in range(5)]
    thresh, nms = 0.02, 0.4  # random-init weights: class scores sit near objectness / classes

    def as_list(dets, counts):
        out = []
        for b in range(batch):
            n = min(counts[b], max_det)
            out.append([(d.box_index, d.obj_id, d.prob, d.x, d.y, d.w, d.h)
                        for d in dets[b * max_det:b * max_det + n]])
        return out

    want = []
    for x in batches:
        per_img, _ = dn.network_detect_batch(net, x, thresh, nms, max_det)
        want.append([[(int(d["box_index"]), int(d["obj_id"]), float(d["prob"]), float(d["x"]), float(d["y"]),
                       float(d["w"]), float(d["h"])) for d in img] for img in per_img])
    assert any(len(img) for res in want for img in res), "test needs at least one detection"

    dets = (dn.Detection * (batch * max_det))()
    counts = (C.c_int * batch)()
    got = []
    stage = [lib.network_pipeline_staging(net, s) for s in (0, 1)]

    def submit(i):
        slot = lib.network_pipeline_next_slot(net)
        C.memmove(stage[slot], batches[i].ctypes.data, batches[i].nbytes)
        assert lib.network_detect_submit(net, stage[slot], thresh, nms, max_det) == slot

    submit(0)
    for i in range(1, len(batches)):
        submit(i)
        lib.network_detect_wait(net, dets, counts, max_det)
        got.append(as_list(dets, counts))
    lib.network_detect_wait(net, dets, counts, max_det)
    got.append(as_list(dets, counts))
    assert got == want

    # the same with the batches already resident in the slots' DEVICE inputs (network_detect_submit_resident): two
    # different batches uploaded once, then alternated without any host -> device copy
    from sr_object_detection_b200 import _lib
    stream = C.c_void_p(lib.network_stream(net))
    for slot in (0, 1):
        C.memmove(stage[slot], batches[slot].ctypes.data, batches[slot].nbytes)
        _lib.check(lib.y2_memcpy_h2d(lib.network_pipeline_input_device(net, slot), stage[slot], batches[slot].nbytes, stream))
    _lib.check(lib.y2_stream_sync(stream))
    got = []
    assert lib.network_detect_submit_resident(net, thresh, nms, max_det) == lib.network_pipeline_next_slot(net) ^ 1
    for i in range(1, 6):
        lib.network_detect_submit_resident(net, thresh, nms, max_det)
        lib.network_detect_wait(net, dets, counts, max_det)
        got.append(as_list(dets, counts))
    lib.network_detect_wait(net, dets, counts, max_det)
    got.append(as_list(dets, counts))
    first = lib.network_pipeline_next_slot(net)  # six submissions: the next slot is the one the first one used
    assert got == [want[(first + i) & 1] for i in range(6)]
    dn.free_network(net)


@pytest.mark.parametrize("side", [416, 320, 608])
def test_u8_input_detections_equal_float_input(tmp_path, side):
    """network_detect_batch_u8 / network_detect_submit_u8 on raw uint8 RGB images must give exactly the
    detections of the float calls on the image the reference's loaders derive from it (byte / 255.)."""
    import ctypes as C
    batch, max_det = 3, 256
    cfg, weights, _, _ = _setup(tmp_path, "tiny-yolo-voc", batch, w=side, h=side)
    dn.set_gpu_index(0)
    net = dn.parse_network_cfg(cfg)
    dn.load_weights(net, weights)
    lib = dn.lib()
    rng = np.random.default_rng(3)
    u8 = rng.integers(0, 256, size=(batch, side, side, 3), dtype=np.uint8)
    planar = (u8.transpose(0, 3, 1, 2).astype(np.float32).astype(np.float64) / 255.0).astype(np.float32)
    thresh, nms = 0.02, 0.4
    want, _ = dn.network_detect_batch(net, np.ascontiguousarray(planar), thresh, nms, max_det)
    assert any(len(w) for w in want), "test needs at least one detection"
    dets = (dn.Detection * (batch * max_det))()
    counts = (C.c_int * batch)()
    lib.network_detect_batch_u8(net, u8.ctypes.data_as(C.POINTER(C.c_ubyte)), thresh, nms, dets, counts, max_det)
    arr = np.ctypeslib.as_array(dets)
    for b in range(batch):
        got = arr[b * max_det:b * max_det + min(counts[b], max_det)]
        assert got.tobytes() == want[b].tobytes(), f"image {b}: uint8 and float paths disagree"
    # and through the pipeline, twice per slot
    stage = [lib.network_pipeline_staging_u8(net, s) for s in (0, 1)]
    for _ in range(4):
        slot = lib.network_pipeline_next_slot(net)
        C.memmove(stage[slot], u8.ctypes.data, u8.nbytes)
        lib.network_detect_submit_u8(net, stage[slot], thresh, nms, max_det)
        lib.network_detect_wait(net, dets, counts, max_det)
        arr = np.ctypeslib.as_array(dets)
        for b in range(batch):
            assert arr[b * max_det:b * max_det + min(counts[b], max_det)].tobytes() == want[b].tobytes()
    dn.free_network(net)


def test_frames_of_any_size_equal_host_resize_then_float_detect(tmp_path):
    """network_detect_batch_frames (raw uint8 frames of any size; byte/255. + resize_image on the device)
    must give exactly the detections of the reference's host chain: load_image -> resize_image ->
    network_predict -> get_region_boxes -> do_nms_sort (yolo_v2_class.cpp:173-239)."""
    import ctypes as C
    batch, max_det = 2, 256
    cfg, weights, _, _ = _setup(tmp_path, "tiny-yolo-voc", batch)
    dn.set_gpu_index(0)
    net = dn.parse_network_cfg(cfg)
    dn.load_weights(net, weights)
    lib = dn.lib()
    thresh, nms = 0.02, 0.4
    dets = (dn.Detection * (batch * max_det))()
    counts = (C.c_int * batch)()
    for fw, fh in [(640, 480), (416, 416), (333, 517)]:
        rng = np.random.default_rng(fw)
        u8 = rng.integers(0, 256, size=(batch, fh, fw, 3), dtype=np.uint8)
        planar = (u8.transpose(0, 3, 1, 2).astype(np.float32).astype(np.float64) / 255.0).astype(np.float32)
        sized = np.empty((batch, 3, 416, 416), dtype=np.float32)
        for b in range(batch):
            src = np.ascontiguousarray(planar[b])
            out = lib.resize_image(dn.Image(fh, fw, 3, src.ctypes.data_as(C.POINTER(C.c_float))), 416, 416)
            sized[b] = np.ctypeslib.as_array(out.data, shape=(3, 416, 416))
            lib.free_image(out)
        want, _ = dn.network_detect_batch(net, sized, thresh, nms, max_det)
        assert any(len(w) for w in want), "test needs at least one detection"
        lib.network_detect_batch_frames(net, u8.ctypes.data_as(C.POINTER(C.c_ubyte)), fw, fh, thresh, nms, dets,
                                        counts, max_det)
        arr = np.ctypeslib.as_array(dets)
        for b in range(batch):
            got = arr[b * max_det:b * max_det + min(counts[b], max_det)]
            assert got.tobytes() == want[b].tobytes(), f"{fw}x{fh} image {b}: device and host resize paths disagree"
    # pipelined, frames written straight into the pinned staging buffer
    fw, fh = 640, 480
    u8 = np.random.default_rng(fw).integers(0, 256, size=(batch, fh, fw, 3), dtype=np.uint8)
    lib.network_detect_batch_frames(net, u8.ctypes.data_as(C.POINTER(C.c_ubyte)), fw, fh, thresh, nms, dets, counts,
                                    max_det)
    ref = [np.ctypeslib.as_array(dets)[b * max_det:b * max_det + min(counts[b], max_det)].tobytes() for b in range(batch)]
    for _ in range(4):
        slot = lib.network_pipeline_next_slot(net)
        stage = lib.network_pipeline_staging_frames(net, slot, fw, fh)
        C.memmove(stage, u8.ctypes.data, u8.nbytes)
        lib.network_detect_submit_frames(net, stage, fw, fh, thresh, nms, max_det)
        lib.network_detect_wait(net, dets, counts, max_det)
        arr = np.ctypeslib.as_array(dets)
        for b in range(batch):
            assert arr[b * max_det:b * max_det + min(counts[b], max_det)].tobytes() == ref[b]
    dn.free_network(net)


def test_set_batch_and_resize_replan_the_device_side(tmp_path):
    """set_batch_network (network.c:308-320) down and UP (the device plan is rebuilt when the batch grows) and
    resize_network (network.c:322-388): every image's output must be what a network parsed directly at that
    batch / resolution produces - exactly, the kernels' accumulation order per output does not depend on either."""
    cfg4, weights, x6, _ = _setup(tmp_path, "tiny-yolo-voc", 6)
    cfg_text = synth.CFGS["tiny-yolo-voc"](batch=4, w=416, h=416)
    (tmp_path / "b4.cfg").write_text(cfg_text)
    dn.set_gpu_index(0)
    net = dn.parse_network_cfg(tmp_path / "b4.cfg")
    dn.load_weights(net, weights)
    full = dn.network_predict(net, np.ascontiguousarray(x6[:4]))
    dn.set_batch_network(net, 2)
    assert net.batch == 2
    assert np.array_equal(dn.network_predict(net, np.ascontiguousarray(x6[:2])), full[:2])
    dn.set_batch_network(net, 6)  # beyond the cfg batch: buffers and plans are rebuilt
    assert net.batch == 6
    out6 = dn.network_predict(net, x6)
    assert np.array_equal(out6[:4], full)
    dets, _ = dn.network_detect_batch(net, x6, 0.02, 0.4, 256)
    assert len(dets) == 6 and any(len(d) for d in dets)
    # resize 416 -> 320 and compare with a network parsed at 320
    assert dn.resize_network(net, 320, 320) == 0
    assert (net.w, net.h) == (320, 320)
    x320 = synth.images(6, 3, 320, 320, seed=77)
    got = dn.network_predict(net, x320)
    (tmp_path / "s320.cfg").write_text(synth.CFGS["tiny-yolo-voc"](batch=6, w=320, h=320))
    ref_net = dn.parse_network_cfg(tmp_path / "s320.cfg")
    dn.load_weights(ref_net, weights)
    want = dn.network_predict(ref_net, x320)
    assert got.shape == want.shape == (6, 10 * 10 * 125)
    assert np.array_equal(got, want)
    # two networks alive in one process: interleaved calls do not disturb each other
    again = dn.network_predict(net, x320)
    assert np.array_equal(again, got)
    dn.free_network(ref_net)
    dn.free_network(net)


@pytest.mark.timeout(300)
@pytest.mark.parametrize("name,side,batch", [("tiny-yolo-voc", 416, 64), ("tiny-yolo-voc", 608, 33), ("yolo-voc", 544, 48),
                                             ("yolo", 608, 16), ("darknet19_448", 448, 32), ("resnet50", 224, 32)])
def test_networks_at_serving_batches(tmp_path, name, side, batch):
    """Whole networks at batch sizes where every CTA walks many tiles (the parity tests above use batches the
    CPU reference finishes in seconds): must complete - an epilogue race in the conv+pool kernel once hung
    tiny-yolo-voc at batch 64 - and EVERY image's output must equal what the batch-1 network computes for that
    image up to bf16 roundings (kernel variant, work distribution and tile order change with the batch; against the
    reference itself these batch sizes are checked in test_baseline_batches_gpu.py)."""
    text1 = synth.CFGS[name](batch=1, w=side, h=side)
    textb = synth.CFGS[name](batch=batch, w=side, h=side)
    (tmp_path / "b1.cfg").write_text(text1)
    (tmp_path / "bn.cfg").write_text(textb)
    synth.write_weights(tmp_path / "n.weights", text1, seed=1234)
    x = synth.images(batch, 3, side, side, seed=42)
    dn.set_gpu_index(0)
    net1 = dn.parse_network_cfg(tmp_path / "b1.cfg")
    dn.load_weights(net1, tmp_path / "n.weights")
    rows = np.stack([dn.network_predict(net1, np.ascontiguousarray(x[b:b + 1]))[0] for b in range(batch)])
    dn.free_network(net1)
    net = dn.parse_network_cfg(tmp_path / "bn.cfg")
    dn.load_weights(net, tmp_path / "n.weights")
    out = dn.network_predict(net, x)
    assert np.isfinite(out).all()
    err = np.abs(out - rows).max(axis=1) / np.abs(rows).max(axis=1)
    assert err.max() <= 5e-3, \
        f"image {int(err.argmax())} at batch {batch} differs from its batch-1 run by {err.max():.2e} of the row maximum"
    again = dn.network_predict(net, x)
    assert np.array_equal(again, out), "two runs of the same batch must be bit-identical"
    if net.layers[net.n - 1].type == dn.REGION:
        dets, counts = dn.network_detect_batch(net, x, 0.02, 0.4, 256)
        assert len(dets) == batch
    dn.free_network(net)


def _device_count():
    import ctypes as C
    from sr_object_detection_b200 import _lib
    n = C.c_int(0)
    _lib.check(_lib.load().y2_device_count(C.byref(n)))
    return n.value


@pytest.mark.parametrize("replicas", [2, 3])
def test_multi_gpu_entry_one_thread_per_replica_equals_single_network(tmp_path, replicas):
    """network_detect_batch_multi / _u8_multi / submit_multi + wait_multi: one host thread per replica, image order
    preserved, detections identical to ONE network run over the whole batch.  Replicas go to distinct GPUs when the
    box has them; on a one-GPU box they share cuda:0, which is the stricter test of the per-network scratch (two
    networks in flight on one device from two host threads)."""
    import ctypes as C
    per, max_det = 3, 845
    total = per * replicas
    cfg, weights, _, _ = _setup(tmp_path, "tiny-yolo-voc", total)
    synth.write_weights(weights, cfg.read_text(), seed=1234, head_gain=30.0)
    x = synth.images(total, 3, 416, 416, seed=42)
    thresh, nms = 0.24, 0.4
    dn.set_gpu_index(0)
    lib = dn.lib()
    net = dn.parse_network_cfg(cfg)
    dn.load_weights(net, weights)
    want, want_counts = dn.network_detect_batch(net, x, thresh, nms, max_det)
    dn.free_network(net)
    assert sum(want_counts) > 20, "the case must produce detections"
    ndev = _device_count()
    gpus = (C.c_int * replicas)(*[i % ndev for i in range(replicas)])
    nets = lib.parse_network_cfg_multi(str(cfg).encode(), str(weights).encode(), gpus, replicas, per)
    assert lib.network_multi_batch(nets, replicas) == total
    dets = (dn.Detection * (total * max_det))()
    counts = (C.c_int * total)()

    def check(tag):
        arr = np.ctypeslib.as_array(dets)
        assert list(counts) == want_counts, tag
        for b in range(total):
            assert arr[b * max_det:b * max_det + counts[b]].tobytes() == want[b].tobytes(), f"{tag}: image {b}"

    with dn._quiet_stderr():
        pass
    lib.network_detect_batch_multi(nets, replicas, x.ctypes.data_as(C.POINTER(C.c_float)), thresh, nms, dets, counts, max_det)
    check("batch_multi")
    # pipelined: two global batches in flight, results in submission order
    x2 = np.ascontiguousarray(x[::-1])
    lib.network_detect_submit_multi(nets, replicas, x.ctypes.data_as(C.POINTER(C.c_float)), thresh, nms, max_det)
    lib.network_detect_submit_multi(nets, replicas, x2.ctypes.data_as(C.POINTER(C.c_float)), thresh, nms, max_det)
    lib.network_detect_wait_multi(nets, replicas, dets, counts, max_det)
    check("submit/wait first")
    lib.network_detect_wait_multi(nets, replicas, dets, counts, max_det)
    arr = np.ctypeslib.as_array(dets)
    for b in range(total):
        assert counts[b] == want_counts[total - 1 - b]
        assert arr[b * max_det:b * max_det + counts[b]].tobytes() == want[total - 1 - b].tobytes()
    # raw uint8 frames
    u8 = np.random.default_rng(5).integers(0, 256, size=(total, 416, 416, 3), dtype=np.uint8)
    planar = (u8.transpose(0, 3, 1, 2).astype(np.float32).astype(np.float64) / 255.0).astype(np.float32)
    lib.network_detect_batch_multi(nets, replicas, np.ascontiguousarray(planar).ctypes.data_as(C.POINTER(C.c_float)),
                                   thresh, nms, dets, counts, max_det)
    ref_bytes = [np.ctypeslib.as_array(dets)[b * max_det:b * max_det + counts[b]].tobytes() for b in range(total)]
    ref_counts = list(counts)
    lib.network_detect_batch_u8_multi(nets, replicas, u8.ctypes.data_as(C.POINTER(C.c_ubyte)), thresh, nms, dets, counts,
                                      max_det)
    assert list(counts) == ref_counts
    arr = np.ctypeslib.as_array(dets)
    for b in range(total):
        assert arr[b * max_det:b * max_det + counts[b]].tobytes() == ref_bytes[b]
    lib.free_network_multi(nets, replicas)
