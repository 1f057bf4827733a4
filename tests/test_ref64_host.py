"""CPU tests of tests/ref64.py, the float64 layer reference the GPU layer checks (test_ref64_gpu.py) rest on:

1. pinned to the unmodified reference: chained in float64 over the stored inputs and weights of the golden fixtures,
   every layer agrees with the reference's fp32 forward within a stated fp32-versus-fp64 bound;
2. its 13 activations agree with the host activate_array (the reference's expressions in double) within 1 fp32 ulp;
3. its interval checker has teeth: it rejects each of a list of plausible kernel mistakes on a realistic layer, and
   it accepts a result rounded to bf16 toward zero instead of to nearest (the bound is not tighter than the
   arithmetic).
"""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

from tests import ref64 as R

GOLDEN = Path(__file__).resolve().parent / "golden"
# |ref64 - reference| <= 2^-18 * max|reference| per layer: the reference's fp32 forward rounds every product sum and
# activation once, and the roundings carry through the chain (measured worst: 6.6e-7 of the layer maximum)
PIN_TOL = 2.0 ** -18


@pytest.mark.parametrize("name", ["mini_yolo", "mini_resnet", "mini_yolo_tree"])
def test_ref64_chain_matches_reference_golden(name):
    """convolution (3x3, 1x1, 7x7/2), maxpool (2/2 and 2/1), forward reorg, one- and two-input routes, shortcuts with
    channel mismatch and stride 2, avgpool, softmax; the softmax-tree detector up to the region input"""
    d = np.load(GOLDEN / f"{name}.npz")
    batch, layers = R.parse_cfg(str(d["cfg"]))
    weights = R.read_weights(d["weights"].tobytes(), layers)
    upto = next((i for i, l in enumerate(layers) if l.type in ("region", "cost")), len(layers))
    outs = R.chain(layers, d["input"].astype(np.float64), weights, upto)
    assert len(outs) >= 13
    kinds = set()
    for i, o in enumerate(outs):
        want = d["layer_%03d" % i].reshape(batch, -1).astype(np.float64)
        assert o.shape == want.shape, (i, o.shape, want.shape)
        err = float(np.abs(o - want).max() / np.abs(want).max())
        assert err <= PIN_TOL, f"{name} layer {i} ({layers[i].type}): max|ref64 - ref| / max|ref| = {err:.3e}"
        kinds.add(layers[i].type)
    assert {"convolutional", "maxpool"} <= kinds


def _activation_grid():
    pts = [0.0]
    for b in R.BREAKPOINTS:
        pts += [b, np.nextafter(np.float32(b), np.float32(-np.inf)), np.nextafter(np.float32(b), np.float32(np.inf))]
    pts += list(np.arange(-10, 10.5, 0.5))                    # stair: integers and half-integers
    pts += [s * v for s in (1, -1) for v in (2.0 ** -20, 1e-3, 0.1, 0.4999, 0.5001, 354.0, 400.0)]
    pts += list(np.linspace(-30, 30, 4097))
    return np.unique(np.float32(pts))


def test_activations_match_host_activate_array():
    """All 13 activations against activate_array (activations.c:64-101, double math, one rounding to float) within
    1 fp32 ulp.  tanh is left out beyond |x| > 354: the reference's exp(2x) overflows there and it returns NaN."""
    from sr_object_detection_b200 import darknet as dn
    lib = dn.lib()
    x = _activation_grid()
    for a in range(13):
        xs = x[np.abs(x) <= 354] if a == R.TANH else x
        host = xs.copy()
        lib.activate_array(host.ctypes.data_as(C.POINTER(C.c_float)), host.size, a)
        want = R.act64(xs, a)
        ulps = np.abs(host.astype(np.float64) - want) / R.ulp_f32(np.abs(want))
        k = int(np.argmax(ulps))
        assert ulps[k] <= 1.0, f"{R.ACT_NAMES[a]}({xs[k]!r}): host {host[k]!r}, float64 {want[k]!r}"


# ---- teeth ---------------------------------------------------------------------------------------------------------
C_ACC = R.C_ACC


def _conv_case(act, cin=512, cout=64, h=13, w=11, batch=2, seed=3):
    """a 3x3 batchnorm convolution over a realistic input (the previous layer's leaky output), weights at the
    reference's init scale (synth.write_weights)"""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((batch, cin, h, w))
    x = np.where(x > 0, x, 0.1 * x)
    s = np.sqrt(2.0 / (9 * cin))
    wd = {"weights": rng.uniform(-s, s, (cout, cin, 3, 3)), "biases": rng.uniform(-0.1, 0.1, cout),
          "scales": rng.uniform(0.5, 1.5, cout), "mean": rng.uniform(-0.1, 0.1, cout), "var": rng.uniform(0.5, 1.5, cout)}
    l = R.L("convolutional", {}, c=cin, h=h, w=w, out_c=cout, out_h=h, out_w=w, act=act, n=cout, size=3, stride=1,
            pad=1, bn=True)
    return l, x, wd, R.layer_ref(l, [x], wd)


def _padded(v, cs):
    b, c, h, w = v.shape
    buf = np.zeros((b, h + 1, w + 1, cs))
    buf[:, :h, :w, :c] = v.transpose(0, 2, 3, 1)
    return buf


def _rejects(label, rep):
    print(f"teeth: {label}: rejected, {rep}")
    assert not rep.ok, f"{label}: the checker accepted it ({rep})"


def test_checker_rejects_kernel_mistakes_and_accepts_round_toward_zero():
    l, x, wd, g = _conv_case(R.LEAKY)
    e = g.e_pre(C_ACC)
    good = R.bf16_rn(g.out)
    assert R.check(good, g.pre, e, R.LEAKY).ok
    rz = R.check(R.bf16_rz(g.out), g.pre, e, R.LEAKY)
    print(f"teeth: bf16 rounded toward zero: accepted, {rz}")
    assert rz.ok, rz

    # one 64-channel K block (one tap, channels 128..191) missing from the sum
    wd2 = dict(wd, weights=wd["weights"].copy())
    wd2["weights"][:, 128:192, 1, 1] = 0
    _rejects("one 64-channel K block dropped (3x3, cin 512)",
             R.check(R.bf16_rn(R.layer_ref(l, [x], wd2).out), g.pre, e, R.LEAKY))
    _rejects("leaky slope 0.125", R.check(R.bf16_rn(np.where(g.pre > 0, g.pre, .125 * g.pre)), g.pre, e, R.LEAKY))
    _rejects("RELIE in place of LEAKY", R.check(R.bf16_rn(R.act64(g.pre, R.RELIE)), g.pre, e, R.LEAKY))
    _rejects("LEAKY in place of RELIE", R.check(R.bf16_rn(R.act64(g.pre, R.LEAKY)), g.pre, e, R.RELIE))
    _rejects("LOGGY in place of TANH", R.check(R.bf16_rn(R.act64(g.pre, R.LOGGY)), g.pre, e, R.TANH))
    _rejects("TANH in place of LOGGY", R.check(R.bf16_rn(R.act64(g.pre, R.TANH)), g.pre, e, R.LOGGY))
    # ((acc - mean) / sd + bias) * scale instead of (acc - mean) / sd * scale + bias
    bias, scale = wd["biases"].reshape(1, -1, 1, 1), wd["scales"].reshape(1, -1, 1, 1)
    _rejects("bias added before the batchnorm scale",
             R.check(R.bf16_rn(R.act64(g.pre - bias + bias * scale, R.LEAKY)), g.pre, e, R.LEAKY))
    last_row = good.copy()
    last_row[1, :, -1, :] = 0
    _rejects("one image's last output row left at zero", R.check(last_row, g.pre, e, R.LEAKY))
    # padded NHWC with 8 storage channels behind the 64 real ones
    lc, gc = _conv_case(R.LOGISTIC, cin=64, cout=56)[0], _conv_case(R.LOGISTIC, cin=64, cout=56)[3]
    buf = _padded(R.bf16_rn(gc.out), 64)
    assert R.check_padded(buf, lc.out_c, lc.out_h, lc.out_w, gc.pre, gc.e_pre(C_ACC), R.LOGISTIC).ok
    for label, sl in [("halo column holding f(0) = 0.5", np.s_[:, :, -1, :]),
                      ("padding channel holding f(0) = 0.5", np.s_[..., 60])]:
        bad = buf.copy()
        bad[sl] = 0.5
        _rejects(label, R.check_padded(bad, lc.out_c, lc.out_h, lc.out_w, gc.pre, gc.e_pre(C_ACC), R.LOGISTIC))


def test_checker_rejects_connected_weights_in_channel_major_order():
    """connected layer over a 24-channel 3x5 tensor: the device packs its input position-major ((y*w + x)*c + ch)
    and must permute the weights to match; weights left in the reference's channel-major order are rejected"""
    rng = np.random.default_rng(8)
    c, h, w, n, batch = 24, 3, 5, 40, 3
    x = R.bf16_rn(rng.uniform(0, 1, (batch, c, h, w)))
    s = np.sqrt(2.0 / (c * h * w))
    wd = {"weights": R.bf16_rn(rng.uniform(-s, s, (n, c * h * w))), "biases": rng.uniform(-0.1, 0.1, n)}
    l = R.L("connected", {}, c=c, h=h, w=w, out_c=n, out_h=1, out_w=1, act=R.RELU, n=n)
    g = R.layer_ref(l, [x], wd)
    e = g.e_pre(C_ACC)
    assert R.check(np.float32(g.out), g.pre, e, R.RELU, out="f32").ok
    x_pos_major = x.transpose(0, 2, 3, 1).reshape(batch, -1)
    wrong = R.act64(x_pos_major @ wd["weights"].T + wd["biases"], R.RELU)
    _rejects("connected weights in channel-major order", R.check(np.float32(wrong), g.pre, e, R.RELU, out="f32"))


def test_reorg_directions_are_inverse_index_maps():
    """forward = 0 (space-to-depth of yolo-voc's reorg) and forward = 1 (reverse = 1, depth-to-space) of reorg_cpu:
    restated loops, each the inverse of the other on the shapes the network uses"""
    rng = np.random.default_rng(1)
    for c, h, w, s in [(64, 26, 26, 2), (72, 9, 15, 3), (8, 8, 8, 2)]:
        x = rng.standard_normal((2, c, h, w))
        y = R.reorg(x, s, 1)
        assert y.shape == (2, c // (s * s), h * s, w * s)
        # depth-to-space: output (c2, h2, w2) is input channel ((h2 % s) * s + w2 % s) * (c / s^2) + c2 at (h2/s, w2/s)
        oc = c // (s * s)
        c2, h2, w2 = 1, h * s - 1, 2
        assert y[1, c2, h2, w2] == x[1, ((h2 % s) * s + w2 % s) * oc + c2, h2 // s, w2 // s]
        assert np.array_equal(R.reorg(y.reshape(x.shape), s, 0).reshape(x.shape), x)
