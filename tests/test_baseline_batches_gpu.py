"""Parity at the batch sizes BASELINE.json states, EVERY image, against the reference's CPU forward (call sequence
of detector.c:454-512; ref_util.checker_bin: the compiled reference oracle/_ref/darknet_ref where present, else the
oracle port oracle/y2_oracle.c, which tests/test_oracle_golden.py pins bit for bit to stored reference outputs of every
layer type these cfgs use), plus the end-to-end detection agreement:

  * every dumped layer and the network output, all images of the batch:
      max|a-b| / max|b|  over the batch       <= 1e-2   (bf16 operands, fp32 accumulate: the north star's bf16 bound),
      the same per IMAGE (each image against its own maximum) <= 1.5e-2,
      relative L2 error  ||a-b|| / ||b||      <= 6e-3,
    and the element-wise figure is printed: the share of elements with |b| >= 5 % of the image maximum whose own
    relative error exceeds 1e-2.  These are the figures bf16 OPERANDS alone produce: tools/bf16_error_model.py (a
    PyTorch fp32 model of the same networks in which only the convolution inputs and weights are rounded to bf16)
    gives per-image maxima of 5e-3 ... 9e-3 and relative L2 of 3e-3 ... 4.5e-3 on two images, the extreme value
    over 64 images sits a little higher (profiles/r2_bf16_error_model.txt);
  * GPU network_detect_batch == the reference's region forward + get_region_boxes + do_nms_sort + final pick
    applied to the GPU's OWN head output: bit-exact, all images (the decode/NMS contract on identical inputs,
    closed end to end through the network's detection entry);
  * against the reference's full pipeline (its own forward): every confident reference candidate is found by the
    GPU with the same class and a box within BOX_TOL, and the GPU reports no candidate the reference scores
    clearly below the threshold (pre-NMS sets with a relative margin MARGIN around the threshold; the post-NMS
    overlap is printed - with random-init weights the class scores of neighbouring boxes are nearly equal, so
    the winner of a suppression is decided by roundings).

The detection head of the synthetic weights is scaled (synth.write_weights head_gain) so that a few per cent of
the boxes clear the 0.24 threshold, as SURVEY.md section 8d prescribes.
"""
import os

import numpy as np
import pytest

from sr_object_detection_b200 import darknet as dn
from sr_object_detection_b200 import synth
from tests import ref_util as R

pytestmark = pytest.mark.gpu

ACT_TOL = 1e-2   # max|a-b| / max|b| per layer, maxima over the whole batch
IMG_TOL = 1.5e-2  # the same with every image normalised by its own maximum (extreme value over up to 64 images)
L2_TOL = 6e-3    # ||a-b||_2 / ||b||_2, per layer over the batch (operand-rounding floor: 3e-3 ... 4.5e-3)
MARGIN = 0.10    # relative band around the detection threshold inside which the two sides may disagree
BOX_TOL = 2e-2   # |box coordinate difference| in units of the image (x, y, w, h are relative)


def _errors(got, ref):
    """got, ref: [B][n].  (batch max-normalised error, worst per-image max-normalised error, relative L2, share of
    significant elements with a relative error above 1e-2)"""
    d = np.abs(got - ref)
    mx = np.maximum(np.abs(ref).max(axis=1), 1e-30)
    per_img = d.max(axis=1) / mx
    whole = float(d.max() / mx.max())
    l2 = float(np.sqrt((d.astype(np.float64) ** 2).sum() / max((ref.astype(np.float64) ** 2).sum(), 1e-60)))
    sig = np.abs(ref) >= 0.05 * mx[:, None]
    rel_bad = float((d[sig] > 1e-2 * np.abs(ref[sig])).mean()) if sig.any() else 0.0
    return whole, float(per_img.max()), l2, rel_bad


def _dets_by_image(rows, batch):
    out = [dict() for _ in range(batch)]
    for r in rows.reshape(-1, 8):
        out[int(r[0])][int(r[1])] = (int(r[2]), np.float32(r[3]), r[4:8].astype(np.float32))
    return out


def _pick(probs, boxes, thresh):
    """final pick over a [total][classes] probability matrix (used for the PRE-NMS candidate sets only)"""
    obj = probs.argmax(axis=1)
    p = probs[np.arange(len(obj)), obj]
    return {int(i): (int(obj[i]), np.float32(p[i]), boxes[i]) for i in np.nonzero(p > thresh)[0]}


CASES = [
    # name, side, batch, head_gain, thresh          BASELINE.json config
    ("yolo-voc", 416, 64, 13.0, 0.24),            # C2: yolo-voc 416 at batch 64
    ("yolo", 608, 32, 24.0, 0.24),                # C3: yolo.cfg 608, 256 over 8 GPUs = 32 per GPU
    ("yolo9000", 544, 8, 13.0, 0.24),              # C4 at the largest batch the CPU side finishes in seconds
    ("darknet19_448", 448, 32, 1.0, None),        # C5
    ("resnet50", 256, 64, 1.0, None),             # C5
]


@pytest.mark.timeout(1500)
@pytest.mark.parametrize("name,side,batch,head_gain,thresh", CASES)
def test_every_image_of_a_baseline_batch_matches_the_reference(tmp_path, name, side, batch, head_gain, thresh):
    checker = R.checker_bin()
    nms = 0.4
    kw = {}
    if name == "yolo9000":
        synth.write_tree(tmp_path / "9k.tree")
        kw["tree"] = str(tmp_path / "9k.tree")
    cfg_text = synth.CFGS[name](batch=batch, w=side, h=side, **kw)
    cfg = tmp_path / "net.cfg"
    cfg.write_text(cfg_text)
    weights = tmp_path / "net.weights"
    synth.write_weights(weights, cfg_text, seed=1234, head_gain=head_gain)
    x = synth.images(batch, 3, side, side, seed=42)
    inp = tmp_path / "input.f32"
    x.tofile(inp)
    ref_dir = tmp_path / "ref"
    # layers above 400 MB per batch (the first two or three full-resolution tensors) are not dumped: they are
    # covered image by image at small batch in test_network_gpu.py and by the kernel tests at batch 64
    ref_dir.mkdir()
    R.run_raw([checker, "forward", cfg, weights, inp, ref_dir, thresh or 0.24, nms, 1],
              env={"Y2_DUMP_MAX_MB": "400", "OMP_NUM_THREADS": str(os.cpu_count())})

    dn.set_gpu_index(0)
    net = dn.parse_network_cfg(cfg)
    dn.load_weights(net, weights)
    out = dn.network_predict(net, x)
    ref_out = R.load(ref_dir, "output.f32", out.shape)
    assert np.isfinite(out).all()
    worst = (0.0, -1)
    worst_img = (0.0, -1)
    worst_l2 = (0.0, -1)
    worst_rel = (0.0, -1)
    checked = 0
    for i in range(net.n):
        l = net.layers[i]
        f = ref_dir / ("layer_%03d.f32" % i)
        if l.type == dn.COST or not f.exists():
            continue
        ref = R.load(ref_dir, f.name, (batch, l.outputs))
        got = dn.get_network_output_layer(net, i)
        e_max, e_img, e_l2, e_rel = _errors(got, ref)
        worst, worst_l2, worst_rel = max(worst, (e_max, i)), max(worst_l2, (e_l2, i)), max(worst_rel, (e_rel, i))
        worst_img = max(worst_img, (e_img, i))
        assert e_max <= ACT_TOL, f"{name} b{batch} layer {i}: max err / max|ref| = {e_max:.3e}"
        assert e_img <= IMG_TOL, f"{name} b{batch} layer {i}: worst image max err / its max|ref| = {e_img:.3e}"
        assert e_l2 <= L2_TOL, f"{name} b{batch} layer {i}: relative L2 error {e_l2:.3e}"
        checked += 1
        os.unlink(f)
    assert checked >= net.n // 2
    e_max, e_img, e_l2, e_rel = _errors(out, ref_out)
    assert e_max <= ACT_TOL and e_img <= IMG_TOL and e_l2 <= L2_TOL, \
        f"{name} b{batch} output: max {e_max:.3e}, per image {e_img:.3e}, L2 {e_l2:.3e}"
    print(f"\n{name} {side} b{batch}: {checked} layers x {batch} images; worst max-normalised error {worst[0]:.2e} "
          f"(layer {worst[1]}), per image {worst_img[0]:.2e} (layer {worst_img[1]}), worst relative L2 {worst_l2[0]:.2e} (layer {worst_l2[1]}), worst share "
          f"of significant elements with own relative error > 1e-2: {worst_rel[0]:.2e} (layer {worst_rel[1]}); "
          f"output: max {e_max:.2e}, L2 {e_l2:.2e}")
    if thresh is None:
        # classifier: the top-1 class must agree wherever the reference's top-2 gap exceeds the activation tolerance
        top_ref, top_got = ref_out.argmax(1), out.argmax(1)
        srt = np.sort(ref_out, axis=1)
        clear = (srt[:, -1] - srt[:, -2]) > 2 * ACT_TOL * np.abs(ref_out).max(axis=1)
        assert (top_ref[clear] == top_got[clear]).all()
        dn.free_network(net)
        return

    # ---- end-to-end detections --------------------------------------------------------------------------------
    lr = net.layers[net.n - 1]
    total, classes = lr.w * lr.h * lr.n, lr.classes
    lr_w, lr_h = lr.w, lr.h
    max_det = total
    dets, counts = dn.network_detect_batch(net, x, thresh, nms, max_det)
    dets0, _ = dn.network_detect_batch(net, x, thresh, 0.0, max_det)   # pre-NMS candidates
    head = dn.get_network_output_layer(net, net.n - 2)                 # the GPU's own head output, conv layout
    dn.free_network(net)

    # (a) the reference's decode + NMS + pick on the GPU's head output: bit-exact
    rin = tmp_path / "gpu_head.f32"
    head.tofile(rin)
    own_dir = tmp_path / "ref_on_gpu_head"
    anchors, classes_, num = synth.REGION_PARAMS[name]
    rcfg = tmp_path / "region_only.cfg"  # the region layer alone: no need to allocate the whole detector again
    rcfg.write_text(synth.region_only_cfg(batch, lr_w, lr_h, anchors, classes_, num,
                                          f"tree={kw['tree']}\n" if "tree" in kw else ""))
    R.region(checker, rcfg, rin, own_dir, thresh=thresh, nms=nms, cwd=tmp_path)
    want = _dets_by_image(R.load(own_dir, "dets.f32"), batch)
    n_exact = 0
    for b in range(batch):
        got = {int(d["box_index"]): (int(d["obj_id"]), np.float32(d["prob"]),
                                     np.array([d["x"], d["y"], d["w"], d["h"]], np.float32)) for d in dets[b]}
        assert sorted(got) == sorted(want[b]), f"image {b}: kept boxes differ from the reference's on the same head output"
        assert [int(d["box_index"]) for d in dets[b]] == sorted(got), "detections must come in box-index order"
        for k, (obj, p, bx) in got.items():
            wobj, wp, wbx = want[b][k]
            assert obj == wobj and p.tobytes() == wp.tobytes() and bx.tobytes() == wbx.tobytes(), \
                f"image {b} box {k}: ({obj}, {p}, {bx}) vs reference ({wobj}, {wp}, {wbx})"
        n_exact += len(got)

    # (b) against the reference's own forward: candidate sets with a margin around the threshold
    ref_boxes = R.load(ref_dir, "boxes.f32", (batch, total, 4))
    ref_pre = R.load(ref_dir, "probs_pre.f32", (batch, total, classes))
    ref_post = _dets_by_image(R.load(ref_dir, "dets.f32"), batch)
    ref_region = ref_out.reshape(batch, total, classes + 5)
    tree = name == "yolo9000"  # two coupled thresholds (hierarchy value > .5, objectness > thresh): printed only
    n_ref = n_found = n_gpu = 0
    worst_box = worst_prob = 0.0
    inter = union = 0
    for b in range(batch):
        ref_c = _pick(ref_pre[b], ref_boxes[b], thresh)
        got_c = {int(d["box_index"]): (int(d["obj_id"]), np.float32(d["prob"]),
                                       np.array([d["x"], d["y"], d["w"], d["h"]], np.float32)) for d in dets0[b]}
        n_gpu += len(got_c)
        got_keys = set(int(d["box_index"]) for d in dets[b])
        inter += len(got_keys & set(ref_post[b]))
        union += len(got_keys | set(ref_post[b]))
        if tree:
            n_ref += len(ref_c)
            n_found += len(set(ref_c) & set(got_c))
            continue
        for k, (obj, p, bx) in ref_c.items():
            if p <= thresh * (1 + MARGIN):
                continue
            n_ref += 1
            assert k in got_c, f"image {b}: reference candidate box {k} (prob {p:.4f}) missing on the GPU"
            gobj, gp, gbx = got_c[k]
            row = np.sort(ref_pre[b, k])
            if row[-1] - row[-2] > MARGIN * row[-1]:
                assert gobj == obj, f"image {b} box {k}: class {gobj} vs reference {obj}"
            worst_box = max(worst_box, float(np.abs(gbx - bx).max()))
            worst_prob = max(worst_prob, abs(float(gp) - float(p)) / float(p))
            n_found += 1
        # a GPU candidate the reference scores clearly below the threshold would be a false detection
        for k in got_c:
            raw = float(ref_region[b, k, 4] * ref_region[b, k, 5:].max())
            assert raw > thresh * (1 - MARGIN), f"image {b} box {k}: GPU candidate, reference probability {raw:.4f}"
    assert n_ref > 0, "the case must produce confident detections"
    assert worst_box <= BOX_TOL, f"box coordinates differ by {worst_box:.3e}"
    assert worst_prob <= MARGIN, f"detection probabilities differ by {worst_prob:.3e} (relative)"
    print(f"{name} b{batch} detections: {n_exact} kept boxes bit-exact against the reference decode+NMS of the same head "
          f"output; {n_found}/{n_ref} confident reference candidates found ({n_gpu} GPU candidates), worst box "
          f"difference {worst_box:.2e}, worst relative probability difference {worst_prob:.2e}; post-NMS keep sets "
          f"vs the reference's own forward: {inter}/{union} common")
