"""Plain float64 reference of the layer forward pass, and the per-element interval checker built on it.

Every function restates one piece of the reference's CPU forward (file:line of the reference cited) in float64 with
numpy, without the reference's float roundings: it is the exact value those layers approximate.  The GPU kernels
are compared with it per element under error bounds derived from their arithmetic (check, Gemm.e_pre below), not
relative to the largest element of a tensor, so that an error on small elements (a leaky tail, a padding channel, a
dropped K block in a deep layer) shows.

The network description is parsed here from the cfg text (parse_cfg), and the weights are read from the `.weights`
file (read_weights), independently of the library's parser and loader: a loader or weight-packing bug cannot hide
behind a reference that reads the same wrong numbers.
"""
from __future__ import annotations

import struct
from dataclasses import dataclass, field

import numpy as np

# ACTIVATION of activations.h:6-8, in enum order
ACT_NAMES = ["logistic", "relu", "relie", "linear", "ramp", "tanh", "plse", "leaky", "elu", "loggy", "stair",
             "hardtan", "lhtan"]
LOGISTIC, RELU, RELIE, LINEAR, RAMP, TANH, PLSE, LEAKY, ELU, LOGGY, STAIR, HARDTAN, LHTAN = range(13)
# activations whose value changes slope or form at these points (activations.h:22-60)
BREAKPOINTS = [-88.0, -20.0, -4.0, -1.0, 0.0, 1.0, 4.0, 20.0, 88.0]
BN_EPS = .000001  # normalize_cpu, blas.c:115-126

# unit roundoff / spacing constants of the device number formats
BF16_U = 2.0 ** -8     # bf16 keeps 8 significant bits: round-to-nearest moves a value by at most 2^-8 of it
F32_U = 2.0 ** -24
# accumulation error of the tensor-core GEMMs per unit of |alpha| * sum |x||w| (Gemm.e_pre): 2^-16; the largest
# observed on a B200 was 1.3e-7 = 2^-22.9 (test_ref64_gpu.py)
C_ACC = 2.0 ** -16


# ---- activations (activations.h:22-60) --------------------------------------------------------------------------
def act64(x, a: int) -> np.ndarray:
    """activate(x, a) in float64.  The formulas are the reference's; tanh, elu and loggy are evaluated in forms that
    do not cancel near 0 (tanh, expm1), which are the same functions."""
    x = np.asarray(x, np.float64)
    with np.errstate(over="ignore"):
        if a == LOGISTIC:
            return 1.0 / (1.0 + np.exp(-x))                               # activations.h:35
        if a == RELU:
            return np.where(x > 0, x, 0.0)                                # activations.h:37
        if a == RELIE:
            return np.where(x > 0, x, .01 * x)                            # activations.h:39
        if a == LINEAR:
            return x.copy()                                               # activations.h:34
        if a == RAMP:
            return np.where(x > 0, x, 0.0) + .1 * x                       # activations.h:40
        if a == TANH:
            return np.tanh(x)                                             # activations.h:43: (e^2x-1)/(e^2x+1)
        if a == PLSE:                                                     # activations.h:44-49
            return np.where(x < -4, .01 * (x + 4), np.where(x > 4, .01 * (x - 4) + 1, .125 * x + .5))
        if a == LEAKY:
            return np.where(x > 0, x, .1 * x)                             # activations.h:41
        if a == ELU:
            return np.where(x >= 0, x, np.expm1(np.minimum(x, 0.0)))      # activations.h:38: exp(x)-1
        if a == LOGGY:
            return np.tanh(x / 2)                                         # activations.h:36: 2/(1+e^-x)-1
        if a == STAIR:                                                    # activations.h:22-27
            n = np.floor(x)
            odd = np.fmod(n, 2) != 0                                      # C's n % 2: -3 % 2 == -1
            # (x - n) is float - int in the reference: rounded to float, which is all of the value near -0
            frac = (x - n).astype(np.float32).astype(np.float64)
            return np.where(odd, frac + np.floor(x / 2.), np.floor(x / 2.))
        if a == HARDTAN:
            return np.clip(x, -1.0, 1.0)                                  # activations.h:28-32
        if a == LHTAN:                                                    # activations.h:50-54
            return np.where(x < 0, .001 * x, np.where(x > 1, .001 * (x - 1) + 1, x))
    raise ValueError(f"activation {a}")


def bf16_rn(x) -> np.ndarray:
    """float -> bf16 with round-to-nearest-even, as float64 (the values the tensor cores read)"""
    f = np.ascontiguousarray(x, np.float32)
    u = f.view(np.uint32).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16
    r = np.where(np.isnan(f), u | 0x400000, r)
    return r.astype(np.uint32).view(np.float32).astype(np.float64).reshape(np.shape(x))


def bf16_rz(x) -> np.ndarray:
    """float -> bf16 truncated toward zero"""
    f = np.ascontiguousarray(x, np.float32)
    return (f.view(np.uint32) & np.uint32(0xFFFF0000)).view(np.float32).astype(np.float64).reshape(np.shape(x))


def ulp_bf16(m) -> np.ndarray:
    """spacing of bf16 values at magnitude m (8 significant bits, fp32 exponent range)"""
    m = np.asarray(m, np.float64)
    _, e = np.frexp(np.maximum(m, 2.0 ** -126))
    return np.ldexp(1.0, e - 8)


def ulp_f32(m) -> np.ndarray:
    m = np.asarray(m, np.float64)
    _, e = np.frexp(np.maximum(m, 2.0 ** -126))
    return np.ldexp(1.0, e - 24)


# ---- the interval checker -----------------------------------------------------------------------------------------
@dataclass
class Report:
    ok: bool
    worst: float           # max over elements of |got - centre| / half-width (<= 1 passes); inf for a failed exact part
    where: tuple = ()      # index of the worst element
    got: float = 0.0
    lo: float = 0.0
    hi: float = 0.0
    note: str = ""

    def __str__(self):
        s = f"worst ratio to the bound {self.worst:.3g}"
        if self.where:
            s += f" at {self.where}: got {self.got:.9g}, allowed [{self.lo:.9g}, {self.hi:.9g}]"
        return s + (f" ({self.note})" if self.note else "")


def check(got, pre, e_pre, act: int, out: str = "bf16", fp32_ulps: int = 4) -> Report:
    """Every activation here is monotone non-decreasing, so the exact output lies in [act(pre - e), act(pre + e)]
    when the device's pre-activation is within e_pre of `pre`; the activation's slope is applied through the
    interval (logistic and elu tails, leaky's 0.1 side are bounded by their own slope).  The interval is then widened
    by the output rounding: one bf16 ulp at max(|lo|, |hi|) for bf16 outputs (round-to-nearest needs half of it; a
    kernel that truncates toward zero must pass too: the bound is about the arithmetic, not the rounding mode), or
    `fp32_ulps` fp32 ulps for fp32 outputs (the output rounding plus the device's exp)."""
    got = np.asarray(got, np.float64)
    pre = np.asarray(pre, np.float64)
    e_pre = np.broadcast_to(np.asarray(e_pre, np.float64), pre.shape)
    lo, hi = act64(pre - e_pre, act), act64(pre + e_pre, act)
    m = np.maximum(np.abs(lo), np.abs(hi))
    widen = ulp_bf16(m) if out == "bf16" else fp32_ulps * ulp_f32(m)
    lo, hi = lo - widen, hi + widen
    return _interval_report(got, lo, hi)


def _interval_report(got, lo, hi) -> Report:
    centre, half = (lo + hi) / 2, (hi - lo) / 2
    dev = np.abs(got - centre)
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.where(half > 0, dev / np.where(half > 0, half, 1), np.where(dev == 0, 0.0, np.inf))
    ratio = np.where(np.isnan(got), np.inf, ratio)
    if ratio.size == 0:
        return Report(True, 0.0)
    k = np.unravel_index(int(np.argmax(ratio)), ratio.shape)
    worst = float(ratio[k])
    return Report(worst <= 1.0, worst, tuple(int(v) for v in k), float(got[k]), float(lo[k]), float(hi[k]))


def check_pooled(got, pre, e_pre, act: int, size: int, stride: int, pad: int, out: str = "bf16") -> Report:
    """A convolution checked through the maxpool behind it: max is monotone, so the pooled output lies in
    [pool(lo), pool(hi)] of the convolution's per-element interval (widened by the output rounding)."""
    pre = np.asarray(pre, np.float64)
    e_pre = np.broadcast_to(np.asarray(e_pre, np.float64), pre.shape)
    lo = maxpool(act64(pre - e_pre, act), size, stride, pad)
    hi = maxpool(act64(pre + e_pre, act), size, stride, pad)
    m = np.maximum(np.abs(lo), np.abs(hi))
    widen = ulp_bf16(m) if out == "bf16" else 4 * ulp_f32(m)
    return _interval_report(np.asarray(got, np.float64), lo - widen, hi + widen)


def check_padded(buf, c: int, h: int, w: int, pre, e_pre, act: int) -> Report:
    """A bf16 padded-NHWC buffer [B][h+1][w+1][cs] (as float): the real values under `check`, and the pad row, the pad
    column and the storage channels c..cs exactly zero, whatever act(0) is."""
    buf = np.asarray(buf, np.float64)
    pads = [np.abs(buf[:, h]).max(), np.abs(buf[:, :, w]).max()]
    if buf.shape[3] > c:
        pads.append(np.abs(buf[..., c:]).max())
    pad_max = float(max(pads))
    if pad_max != 0:
        return Report(False, float("inf"), note=f"pads / padding channels hold values up to {pad_max:g}")
    return check(buf[:, :h, :w, :c].transpose(0, 3, 1, 2), pre, e_pre, act)


def exact(got, want) -> Report:
    """bit-for-bit comparison of float32 values (byte / index layers)"""
    g = np.ascontiguousarray(got, np.float32)
    wv = np.ascontiguousarray(want, np.float32)
    diff = g.view(np.uint32) != wv.view(np.uint32)
    n = int(diff.sum())
    if n == 0:
        return Report(True, 0.0)
    k = np.unravel_index(int(np.argmax(diff)), diff.shape)
    return Report(False, float("inf"), tuple(int(v) for v in k), float(g[k]), float(wv[k]), float(wv[k]),
                  note=f"{n} of {diff.size} values differ")


# ---- cfg and weights ------------------------------------------------------------------------------------------------
@dataclass
class L:
    """one layer of a parsed cfg, with the extents parse_network_cfg computes (parser.c:585-700)"""
    type: str
    opt: dict
    c: int = 0
    h: int = 0
    w: int = 0
    out_c: int = 0
    out_h: int = 0
    out_w: int = 0
    act: int = LINEAR
    n: int = 0                 # filters / outputs
    size: int = 1
    stride: int = 1
    pad: int = 0
    bn: bool = False
    inputs: list = field(default_factory=list)   # producer layer indices (-1: the network input)
    groups: int = 1
    temperature: float = 1.0
    reverse: bool = False

    @property
    def outputs(self):
        return self.out_c * self.out_h * self.out_w


def _sections(text: str):
    out = []
    for raw in text.splitlines():
        line = "".join(raw.split())
        if not line or line[0] in "#;":
            continue
        if line.startswith("["):
            out.append((line[1:-1], {}))
        else:
            k, _, v = line.partition("=")
            out[-1][1][k] = v
    return out


def parse_cfg(text: str):
    """(batch, [L]) for a cfg text: the layer graph and extents of parse_network_cfg"""
    secs = _sections(text)
    assert secs[0][0] in ("net", "network")
    net = secs[0][1]
    batch = int(net.get("batch", 1))
    c, h, w = int(net.get("channels", 0)), int(net.get("height", 0)), int(net.get("width", 0))
    layers: list[L] = []
    for idx, (kind, opt) in enumerate(secs[1:]):
        l = L(kind, opt, c=c, h=h, w=w, inputs=[idx - 1])
        if kind == "convolutional":                                   # parser.c:140-175
            l.n, l.size, l.stride = int(opt.get("filters", 1)), int(opt.get("size", 1)), int(opt.get("stride", 1))
            l.pad = l.size // 2 if int(opt.get("pad", 0)) else int(opt.get("padding", 0))
            l.act = ACT_NAMES.index(opt.get("activation", "logistic"))
            l.bn = bool(int(opt.get("batch_normalize", 0)))
            l.out_c = l.n
            l.out_h = (h + 2 * l.pad - l.size) // l.stride + 1
            l.out_w = (w + 2 * l.pad - l.size) // l.stride + 1
        elif kind == "connected":                                     # parser.c:177-188
            l.n = int(opt.get("output", 1))
            l.act = ACT_NAMES.index(opt.get("activation", "logistic"))
            l.bn = bool(int(opt.get("batch_normalize", 0)))
            l.out_c, l.out_h, l.out_w = l.n, 1, 1
        elif kind == "maxpool":                                       # parser.c:296-308
            l.stride = int(opt.get("stride", 1))
            l.size = int(opt.get("size", l.stride))
            l.pad = int(opt.get("padding", (l.size - 1) // 2))
            l.out_c, l.out_h, l.out_w = c, (h + 2 * l.pad) // l.stride, (w + 2 * l.pad) // l.stride
        elif kind == "avgpool":
            l.out_c, l.out_h, l.out_w = c, 1, 1
        elif kind == "softmax":                                       # parser.c:190-204
            l.groups = int(opt.get("groups", 1))
            l.temperature = float(opt.get("temperature", 1))
            l.out_c, l.out_h, l.out_w = c * h * w, 1, 1
        elif kind == "route":                                         # parser.c:416-452
            l.inputs = [(idx + int(v)) if int(v) < 0 else int(v) for v in opt["layers"].split(",")]
            first = layers[l.inputs[0]]
            l.out_h, l.out_w = first.out_h, first.out_w
            l.out_c = sum(layers[k].out_c for k in l.inputs)
        elif kind == "reorg":                                         # reorg_layer.c:10-30
            l.stride = int(opt.get("stride", 1))
            l.reverse = bool(int(opt.get("reverse", 0)))
            s = l.stride
            if l.reverse:
                l.out_c, l.out_h, l.out_w = c // (s * s), h * s, w * s
            else:
                l.out_c, l.out_h, l.out_w = c * s * s, h // s, w // s
        elif kind == "shortcut":                                      # parser.c:374-387
            frm = int(opt["from"])
            l.inputs = [idx - 1, idx + frm if frm < 0 else frm]
            l.act = ACT_NAMES.index(opt.get("activation", "linear"))
            l.out_c, l.out_h, l.out_w = c, h, w
        elif kind in ("dropout", "cost", "region"):
            l.out_c, l.out_h, l.out_w = c, h, w
        else:
            raise ValueError(f"layer kind {kind}")
        layers.append(l)
        c, h, w = l.out_c, l.out_h, l.out_w
    return batch, layers


def read_weights(data: bytes, layers) -> dict:
    """The `.weights` bytes in the layout synth.write_weights writes and load_weights_upto reads
    (parser.c:1009-1082): int32 major, minor, revision, then `seen` (int64 when major*10 + minor >= 2); per
    convolutional layer biases[n], [scales[n], rolling_mean[n], rolling_variance[n]], weights[n][c][k][k]; per
    connected layer biases[n], weights[n][inputs], then the batchnorm vectors (load_connected_weights,
    parser.c:897-913).  Returns {layer index: {"biases", "weights", ["scales", "mean", "var"]}} in float64."""
    major, minor, _ = struct.unpack_from("<iii", data, 0)
    off = 12 + (8 if major * 10 + minor >= 2 else 4)

    def take(n):
        nonlocal off
        a = np.frombuffer(data, np.float32, n, off).astype(np.float64)
        off += 4 * n
        return a

    out = {}
    for i, l in enumerate(layers):
        if l.type == "convolutional":
            d = {"biases": take(l.n)}
            if l.bn:
                d["scales"], d["mean"], d["var"] = take(l.n), take(l.n), take(l.n)
            d["weights"] = take(l.n * l.c * l.size * l.size).reshape(l.n, l.c, l.size, l.size)
            out[i] = d
        elif l.type == "connected":
            inputs = l.c * l.h * l.w
            d = {"biases": take(l.n), "weights": take(l.n * inputs).reshape(l.n, inputs)}
            if l.bn:
                d["scales"], d["mean"], d["var"] = take(l.n), take(l.n), take(l.n)
            out[i] = d
    assert off == len(data), f"{len(data) - off} bytes of the weights file left over"
    return out


# ---- layers -----------------------------------------------------------------------------------------------------------
def _affine(wd):
    """(alpha, mean, bias) with which pre = alpha * (acc - mean) + bias: normalize_cpu + scale_bias + add_bias
    (convolutional_layer.c:401-423 -> blas.c:115-126, connected_layer.c:271-293); no batchnorm: 1, 0, bias"""
    if "scales" in wd:
        return wd["scales"] / (np.sqrt(wd["var"]) + BN_EPS), wd["mean"], wd["biases"]
    n = len(wd["biases"])
    return np.ones(n), np.zeros(n), wd["biases"]


def conv_sums(x, wt, stride: int, pad: int):
    """(sum x*w, sum |x|*|w|) of a convolution (im2col_cpu + gemm, convolutional_layer.c:401-410), [B][n][oh][ow]"""
    b, c, h, w = x.shape
    n, _, k, _ = wt.shape
    oh, ow = (h + 2 * pad - k) // stride + 1, (w + 2 * pad - k) // stride + 1
    xp = np.zeros((b, c, h + 2 * pad + stride, w + 2 * pad + stride))
    xp[:, :, pad:pad + h, pad:pad + w] = x
    acc = np.zeros((b, oh, ow, n))
    sab = np.zeros((b, oh, ow, n))
    for r in range(k):
        for s in range(k):
            tap = xp[:, :, r:r + stride * oh:stride, s:s + stride * ow:stride]
            acc += np.tensordot(tap, wt[:, :, r, s], axes=([1], [1]))
            sab += np.tensordot(np.abs(tap), np.abs(wt[:, :, r, s]), axes=([1], [1]))
    return acc.transpose(0, 3, 1, 2), sab.transpose(0, 3, 1, 2)


@dataclass
class Gemm:
    """A convolutional or connected layer evaluated in float64: pre-activation, the error scales of its bound, act"""
    pre: np.ndarray     # alpha*(acc - mean) + bias
    sabs: np.ndarray    # |alpha| * sum |x||w|
    affine: np.ndarray  # |alpha*mean| + |bias|: what the fp32 fold beta = bias - mean*alpha is computed from
    act: int

    @property
    def out(self):
        return act64(self.pre, self.act)

    def e_pre(self, c_acc: float, post_act: bool = False) -> np.ndarray:
        """e_pre = c_acc*|alpha|*sum|x||w| + 2^-22*(|alpha*mean| + |bias|) [+ 2^-8*|pre| when the activation runs
        behind a bf16 round trip of the pre-activation (post_act): bf16 round-to-nearest moves a value by at most
        2^-8 of it].  The second term covers alpha and beta held in fp32 and the fp32 affine of the epilogue."""
        e = c_acc * self.sabs + 2.0 ** -22 * self.affine
        if post_act:
            e = e + BF16_U * (np.abs(self.pre) + e)
        return e


def convolutional(l: L, x, wd, round_operands: bool = True) -> Gemm:
    """forward_convolutional_layer (convolutional_layer.c:395-430) on bf16-rounded operands when round_operands"""
    wt = wd["weights"]
    if round_operands:
        x, wt = bf16_rn(x), bf16_rn(wt)
    acc, sab = conv_sums(x, wt, l.stride, l.pad)
    alpha, mean, bias = (v.reshape(1, -1, 1, 1) for v in _affine(wd))
    return Gemm(alpha * (acc - mean) + bias, np.abs(alpha) * sab, np.abs(alpha * mean) + np.abs(bias) + 0 * acc, l.act)


def connected(l: L, x, wd, round_operands: bool = True) -> Gemm:
    """forward_connected_layer (connected_layer.c:122-155): out = W x over the flat NCHW input, then batchnorm,
    then bias, then the activation"""
    x = np.asarray(x, np.float64).reshape(len(x), -1)
    wt = wd["weights"]
    if round_operands:
        x, wt = bf16_rn(x), bf16_rn(wt)
    acc = x @ wt.T
    sab = np.abs(x) @ np.abs(wt).T
    alpha, mean, bias = (v.reshape(1, -1) for v in _affine(wd))
    return Gemm(alpha * (acc - mean) + bias, np.abs(alpha) * sab, np.abs(alpha * mean) + np.abs(bias) + 0 * acc, l.act)


def maxpool(x, size: int, stride: int, pad: int):
    """forward_maxpool_layer (maxpool_layer.c:79-114): window rows [i*stride - pad, i*stride - pad + size), cells
    outside the image skipped"""
    x = np.asarray(x, np.float64)
    b, c, h, w = x.shape
    oh, ow = (h + 2 * pad) // stride, (w + 2 * pad) // stride
    xp = np.full((b, c, h + 2 * pad + size + stride, w + 2 * pad + size + stride), -np.inf)
    xp[:, :, pad:pad + h, pad:pad + w] = x
    out = np.full((b, c, oh, ow), -np.inf)
    for r in range(size):
        for s in range(size):
            out = np.maximum(out, xp[:, :, r:r + stride * oh:stride, s:s + stride * ow:stride])
    return out


def reorg(x, stride: int, forward: int):
    """reorg_cpu(x, w, h, c, batch, stride, forward, out) of blas.c:8-29 for x [B][c][h][w] (the layer's INPUT
    extent, as reorg_layer.c:97-104 calls it): forward = 0 -> out[in_index] = x[out_index], forward = 1 ->
    out[out_index] = x[in_index]; the loop over (k, j, i) restated with index arrays"""
    x = np.asarray(x)
    b, c, h, w = x.shape
    out_c = c // (stride * stride)
    k, j, i = np.meshgrid(np.arange(c), np.arange(h), np.arange(w), indexing="ij")
    in_index = (i + w * (j + h * k)).ravel()
    c2 = k % out_c
    offset = k // out_c
    w2 = i * stride + offset % stride
    h2 = j * stride + offset // stride
    out_index = (w2 + w * stride * (h2 + h * stride * c2)).ravel()
    xf = x.reshape(b, -1)
    out = np.empty_like(xf)
    if forward:
        out[:, out_index] = xf[:, in_index]
        return out.reshape(b, out_c, h * stride, w * stride)
    out[:, in_index] = xf[:, out_index]
    return out.reshape(b, c * stride * stride, h // stride, w // stride)


def route(xs):
    """forward_route_layer (route_layer.c:73-86): the inputs' flat outputs one after the other per image"""
    return np.concatenate([np.asarray(x).reshape(len(x), -1) for x in xs], axis=1)


def shortcut(x, add, act: int):
    """forward_shortcut_layer (shortcut_layer.c:39-44): copy, shortcut_cpu (blas.c:57-81), activate"""
    x = np.array(x, np.float64)
    _, c2, h2, w2 = x.shape
    _, c1, h1, w1 = add.shape
    stride, sample = max(w1 // w2, 1), max(w2 // w1, 1)
    minw, minh, minc = min(w1, w2), min(h1, h2), min(c1, c2)
    x[:, :minc, 0:minh * sample:sample, 0:minw * sample:sample] += \
        add[:, :minc, 0:minh * stride:stride, 0:minw * stride:stride]
    return act64(x, act)


def avgpool(x):
    """forward_avgpool_layer (avgpool_layer.c:40-55): the mean over h*w per channel"""
    x = np.asarray(x, np.float64)
    return x.reshape(x.shape[0], x.shape[1], -1).mean(axis=2)


def softmax(x, groups: int = 1, temperature: float = 1.0):
    """forward_softmax_layer (softmax_layer.c:49-61) -> softmax (blas.c:205-221) per group of inputs/groups"""
    x = np.asarray(x, np.float64)
    b = x.shape[0]
    g = x.reshape(b * groups, -1) / temperature
    e = np.exp(g - g.max(axis=1, keepdims=True))
    return (e / e.sum(axis=1, keepdims=True)).reshape(b, -1)


def layer_ref(l: L, inputs, weights=None, round_operands: bool = True):
    """One layer on given inputs (NCHW arrays, or [B][n] vectors for flat producers).  Convolutional and connected
    layers return a Gemm (pre-activation and error scales), every other layer its output array."""
    t = l.type
    if t == "convolutional":
        return convolutional(l, np.asarray(inputs[0]).reshape(-1, l.c, l.h, l.w), weights, round_operands)
    if t == "connected":
        return connected(l, inputs[0], weights, round_operands)
    x = inputs[0]
    if t == "maxpool":
        return maxpool(np.asarray(x).reshape(-1, l.c, l.h, l.w), l.size, l.stride, l.pad)
    if t == "reorg":
        return reorg(np.asarray(x).reshape(-1, l.c, l.h, l.w), l.stride, int(l.reverse))
    if t == "route":
        return route(inputs)
    if t in ("dropout", "cost"):                                  # dropout_layer.c:40: identity at inference
        return np.array(x, copy=True)
    if t == "shortcut":
        return shortcut(np.asarray(x).reshape(-1, l.out_c, l.out_h, l.out_w), inputs[1], l.act)
    if t == "avgpool":
        return avgpool(np.asarray(x).reshape(-1, l.c, l.h, l.w))
    if t == "softmax":
        return softmax(np.asarray(x).reshape(len(x), -1), l.groups, l.temperature)
    raise ValueError(f"no reference for {t}")


def chain(layers, x, weights, upto: int | None = None, round_operands: bool = False):
    """the whole forward pass in float64 (no bf16 rounding by default: the reference's own fp32 forward is what it is
    compared with).  Returns the list of layer outputs as [B][outputs] arrays."""
    outs = []
    for i, l in enumerate(layers[:upto]):
        ins = []
        for k in l.inputs:
            if k < 0:
                ins.append(x)
            else:
                src = layers[k]
                ins.append(outs[k].reshape(-1, src.out_c, src.out_h, src.out_w))
        r = layer_ref(l, ins, weights.get(i), round_operands)
        if isinstance(r, Gemm):
            r = r.out
        outs.append(np.asarray(r).reshape(len(x), -1))
    return outs
