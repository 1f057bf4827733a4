"""GPU layers against the float64 reference of tests/ref64.py, per element.

Floating-point layers are checked under the interval bound of ref64.check: the device value must lie in
[act(pre - e_pre), act(pre + e_pre)], widened by the output rounding, with

    e_pre = C_ACC * |alpha| * sum|x||w|  +  2^-22 * (|alpha*mean| + |bias|)  [+ 2^-8 * |pre| behind a bf16 round trip]

on the bf16 operands the kernels read.  C_ACC = 2^-16 (ref64.C_ACC).  Each test prints its worst ratio to the bound
(<= 1 passes) and the fp32-output linear tests the observed |got - pre| / (|alpha| sum|x||w|).  Measured on one
NVIDIA B200 at a 1000 W power limit: the accumulation ratio was at most 1.3e-7 (2^-22.9) on the fp32 heads, the same
for the per-tap, slab and CTA-pair kernels; the worst ratios to the bound were 0.81 for every kernel and variant on
the bf16 convolution cases (per-tap, slab, pair, conv + maxpool, stem), 0.50 for the logistic epilogues, 0.014 for
the fp32 heads and connected layers, and 0.99 in the network tests (relu outputs at 0 where pre - e_pre < 0 < pre +
e_pre: the edge of the interval by construction).
Byte and index layers (reorg, the connected layer's input packing, maxpool, route, dropout) must match bit for bit.

Layer types no other test runs without the compiled reference (connected, dropout, reverse reorg, the activations
the epilogue lacks) are covered here from a clean checkout: the network tests build their cfgs, write synthetic
weights and read those weights back from the file for the reference, never from the library's layer structs.
"""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from sr_object_detection_b200 import _lib  # noqa: E402
from sr_object_detection_b200 import darknet as dn  # noqa: E402
from sr_object_detection_b200 import synth  # noqa: E402
from tests import ref64 as R  # noqa: E402
from tests.test_kernels_gpu import CONV_CASES  # noqa: E402

pytestmark = pytest.mark.gpu

Y2_ACT = {R.LINEAR: 0, R.LEAKY: 1, R.LOGISTIC: 2}   # epilogue codes of yolo2_b200_kernels.h
OUT_BF16, OUT_F32, OUT_POOLED = 0, 1, 2
VARIANT_NAMES = {0: "pertap", 1: "slab", 2: "pair", 3: "conv+pool", 4: "stem"}


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _fn(name, args):
    f = getattr(_lib.load(), name)
    f.restype, f.argtypes = C.c_int, args
    return f


vp, i32 = C.c_void_p, C.c_int


@pytest.fixture(params=["auto", "slab", "pertap", "pair", "roundrobin"])
def conv_variant(request, monkeypatch):
    """test_kernels_gpu.py's kernel choices: the default (CTA-pair kernel for wide layers), the halo-slab kernel, the
    per-tap fallback, the pair kernel wherever its shape constraints allow it, and the pair kernel on whole tiles
    round-robin (Y2_CONV_VARIANT / Y2_PAIR_BALANCE are read at plan creation)"""
    monkeypatch.delenv("Y2_PAIR_BALANCE", raising=False)
    if request.param in ("auto", "roundrobin"):
        monkeypatch.delenv("Y2_CONV_VARIANT", raising=False)
        if request.param == "roundrobin":
            monkeypatch.setenv("Y2_PAIR_BALANCE", "0")
    else:
        monkeypatch.setenv("Y2_CONV_VARIANT", request.param)
    return request.param


# ---- activations -----------------------------------------------------------------------------------------------------
def _bf16_grid(n):
    """n bf16-exact values: every breakpoint and its neighbours, integers and half-integers, small magnitudes
    around 0, and a dense sweep of [-30, 30]"""
    pts = [0.0]
    for b in R.BREAKPOINTS + list(np.arange(-10, 10.5, 0.5)):
        pts += [b, b - 2.0 ** -6, b + 2.0 ** -6]
    pts += [s * 2.0 ** -e for s in (1, -1) for e in range(1, 24)]
    pts += list(np.linspace(-30, 30, n))
    return np.unique(R.bf16_rn(np.float32(pts)))


def _bf16_ok(got, x64, a):
    """got == bf16_rn(act64(x)), or one bf16 ulp off where act64(x) lies within 2^-20 of a rounding boundary"""
    v = R.act64(x64, a)
    want = R.bf16_rn(v)
    same = got == want
    mid = (got + want) / 2
    near = (np.abs(got - want) <= R.ulp_bf16(np.maximum(np.abs(got), np.abs(want)))) & \
        (np.abs(v - mid) <= 2.0 ** -20 * np.abs(v))
    return same | near, want


@pytest.mark.parametrize("act", range(13), ids=R.ACT_NAMES)
def test_activate_bf16_matches_act64(act):
    """y2_activate_bf16 (the separate activation pass behind a LINEAR epilogue) on a bf16 padded-NHWC tensor with
    storage channels behind the real ones and odd h and w: real values = bf16_rn(act64(x)); pad row, pad column and
    channels c..cs keep their sentinel"""
    dev = torch.device("cuda:0")
    batch, h, w, c, cs = 2, 7, 9, 36, 40
    grid = _bf16_grid(2000)
    n = batch * h * w * c
    vals = np.resize(grid, n)
    np.random.default_rng(act).shuffle(vals)
    buf = np.full((batch, h + 1, w + 1, cs), 7.0, np.float32)
    buf[:, :h, :w, :c] = vals.reshape(batch, h, w, c)
    d = torch.from_numpy(buf).to(torch.bfloat16).to(dev)
    f = _fn("y2_activate_bf16", [vp, i32, i32, i32, i32, i32, i32, vp])
    _lib.check(f(d.data_ptr(), cs, c, batch, h, w, act, _stream()), "y2_activate_bf16")
    torch.cuda.synchronize()
    out = d.float().cpu().numpy().astype(np.float64)
    got = out[:, :h, :w, :c]
    ok, want = _bf16_ok(got, buf[:, :h, :w, :c].astype(np.float64), act)
    k = np.unravel_index(int(np.argmin(ok)), ok.shape)
    assert ok.all(), (f"{R.ACT_NAMES[act]}({buf[:, :h, :w, :c][k]!r}) = {got[k]!r}, bf16_rn(act64) = {want[k]!r}; "
                      f"{(~ok).sum()} of {ok.size} values")
    assert (out[:, h] == 7.0).all() and (out[:, :, w] == 7.0).all() and (out[..., c:] == 7.0).all()


VEC_ULPS = 4  # the device's fp32 expressions (tanhf, expm1f, expf, a constant product) round a few times


@pytest.mark.parametrize("act", range(13), ids=R.ACT_NAMES)
def test_vec_activate_matches_act64(act):
    """y2_vec_activate (activate_array_ongpu, and the post-activation of fp32 heads and connected layers) against
    act64 directly, within VEC_ULPS fp32 ulps: 4097 points over [-30, 30], every breakpoint and its float
    neighbours, and small magnitudes down to 2^-40 where tanh, elu and loggy are most easily computed with
    cancellation"""
    dev = torch.device("cuda:0")
    pts = list(np.linspace(-30, 30, 4097)) + [s * 2.0 ** -e for s in (1, -1) for e in range(1, 41)]
    for b in R.BREAKPOINTS + list(np.arange(-10, 10.5, 0.5)):
        fb = np.float32(b)
        pts += [fb, np.nextafter(fb, np.float32(-np.inf)), np.nextafter(fb, np.float32(np.inf))]
    x = np.unique(np.float32(pts))
    d = torch.from_numpy(x.copy()).to(dev)
    f = _fn("y2_vec_activate", [vp, C.c_longlong, i32, vp])
    _lib.check(f(d.data_ptr(), x.size, act, _stream()), "y2_vec_activate")
    torch.cuda.synchronize()
    got = d.cpu().numpy().astype(np.float64)
    want = R.act64(x.astype(np.float64), act)
    ulps = np.abs(got - want) / R.ulp_f32(np.abs(want))
    k = int(np.argmax(ulps))
    print(f"y2_vec_activate {R.ACT_NAMES[act]}: worst {ulps[k]:.2f} ulp at x = {x[k]!r}")
    assert ulps[k] <= VEC_ULPS, f"{R.ACT_NAMES[act]}({x[k]!r}) = {got[k]!r}, act64 = {want[k]!r} ({ulps[k]:.0f} ulp)"


# ---- single convolutions -------------------------------------------------------------------------------------------
def _operands(batch, cin, h, w, cout, ksize, seed, x_lo=-1.0):
    rng = np.random.default_rng(seed)
    x = R.bf16_rn(rng.uniform(x_lo, 1, (batch, cin, h, w)))
    s = (2.0 / (ksize * ksize * cin)) ** 0.5
    wt = R.bf16_rn(rng.uniform(-s, s, (cout, cin, ksize, ksize)))
    alpha = np.float32(rng.uniform(0.5, 1.5, cout))
    beta = np.float32(rng.uniform(-0.5, 0.5, cout))
    return x, wt, alpha, beta


_REF_CACHE = {}


def _ref(key, x, wt, alpha, beta, act):
    """float64 pre-activation and error scales of a stride-1 'same' convolution, cached per case (the kernel
    variants share it; the last few cases are kept)"""
    if key not in _REF_CACHE:
        acc, sab = R.conv_sums(x, wt, 1, wt.shape[2] // 2)
        a, b = alpha.astype(np.float64).reshape(1, -1, 1, 1), beta.astype(np.float64).reshape(1, -1, 1, 1)
        while len(_REF_CACHE) >= 6:
            _REF_CACHE.pop(next(iter(_REF_CACHE)))
        _REF_CACHE[key] = (a * acc + b, np.abs(a) * sab, np.abs(b))
    pre, sabs, aff = _REF_CACHE[key]
    return R.Gemm(pre, sabs, aff, act)


def _padded_in(x, cs=None, off=0, fill=0.0):
    b, c, h, w = x.shape
    cs = cs or c
    buf = np.full((b, h + 1, w + 1, cs), fill, np.float32)
    buf[:, h] = 0
    buf[:, :, w] = 0
    buf[:, :h, :w, off:off + c] = x.transpose(0, 2, 3, 1)
    return torch.from_numpy(buf).to(torch.bfloat16).cuda()


def _packed_weights(wt, npad):
    """[n][c][k][k] -> bf16 [npad][k*k*c], K index = (r*k + s)*c + c (y2_conv_desc)"""
    n, c, k, _ = wt.shape
    out = np.zeros((npad, k * k * c), np.float32)
    out[:n] = wt.transpose(0, 2, 3, 1).reshape(n, -1)
    return torch.from_numpy(out).to(torch.bfloat16).cuda()


def _launch(x_dev, in_cs, cin, batch, h, w, ksize, wt_dev, cout, npad, block_n, block_k, alpha, beta, act, out,
            out_cs, out_mode, out_off=0, in_off=0):
    lib = _lib.load()
    a = torch.zeros(npad, device="cuda")
    b = torch.zeros(npad, device="cuda")
    a[:len(alpha)] = torch.from_numpy(alpha).cuda()
    b[:len(beta)] = torch.from_numpy(beta).cuda()
    d = _lib.ConvDesc()
    d.in_ = x_dev.data_ptr() + in_off * 2; d.in_cs = in_cs; d.cin = cin
    d.batch = batch; d.h = h; d.w = w; d.ksize = ksize
    d.wt = wt_dev.data_ptr(); d.cout = cout; d.npad = npad; d.block_n = block_n; d.block_k = block_k
    d.alpha = a.data_ptr(); d.beta = b.data_ptr(); d.act = act
    d.out = out.data_ptr() + out_off * out.element_size(); d.out_cs = out_cs; d.out_mode = out_mode
    plan = C.c_void_p()
    _lib.check(lib.y2_conv_plan_create(C.byref(d), C.byref(plan)), "conv_plan_create")
    try:
        variant = lib.y2_conv_plan_variant(plan)
        _lib.check(lib.y2_conv_plan_launch(plan, _stream()), "conv_plan_launch")
        torch.cuda.synchronize()
    finally:
        lib.y2_conv_plan_destroy(plan)
    return VARIANT_NAMES.get(variant, str(variant))


def _report(tag, rep, g=None, got=None):
    s = f"{tag}: {rep}"
    if g is not None and got is not None and g.act == R.LINEAR:
        with np.errstate(divide="ignore", invalid="ignore"):
            r = np.where(g.sabs > 0, np.abs(got - g.pre) / g.sabs, 0)
        s += f"; accumulation |got - pre| / (|alpha| sum|x||w|) = {r.max():.2e}"
    print(s)
    assert rep.ok, s


@pytest.mark.parametrize("ksize", [1, 3])
def test_logistic_epilogue_bf16_padded(conv_variant, ksize):
    """Y2_ACT_LOGISTIC in the epilogue of every kernel, bf16 padded output: pads exactly zero (not f(0) = 0.5)"""
    batch, cin, h, w, cout = (16, 256, 13, 11, 256) if ksize == 1 else (8, 128, 13, 11, 256)
    x, wt, alpha, beta = _operands(batch, cin, h, w, cout, ksize, seed=40 + ksize)
    beta = np.float32(beta * 8)   # both tails of the logistic
    g = _ref(("lg", ksize), x, wt, alpha, beta, R.LOGISTIC)
    out = torch.full((batch, h + 1, w + 1, cout), 7.0, dtype=torch.bfloat16, device="cuda")
    v = _launch(_padded_in(x), cin, cin, batch, h, w, ksize, _packed_weights(wt, cout), cout, cout, 256, 64, alpha,
                beta, 2, out, cout, OUT_BF16)
    buf = out.float().cpu().numpy()
    _report(f"logistic {ksize}x{ksize} bf16 [{conv_variant} -> {v}]",
            R.check_padded(buf, cout, h, w, g.pre, g.e_pre(R.C_ACC), R.LOGISTIC))


@pytest.mark.parametrize("cout,cs,act", [(125, 125, R.LOGISTIC), (1101, 1104, R.LOGISTIC), (1101, 1104, R.LINEAR)])
def test_fp32_heads_logistic_and_linear(conv_variant, cout, cs, act):
    """fp32 flat heads [B][H*W][cs]: 125 filters, and the staged wide head of 1101 filters whose row padding
    (cs > cout) is nobody's to write; logistic epilogue and the linear reference measurement of the accumulation"""
    batch, cin, h, w = 3, 1024 if cout == 125 else 128, 13, 9
    x, wt, alpha, beta = _operands(batch, cin, h, w, cout, 1, seed=cout)
    g = _ref(("head", cout, act), x, wt, alpha, beta, act)
    npad = (cout + 255) // 256 * 256 if cout > 256 else 128
    out = torch.full((batch, h * w, cs), 7.0, dtype=torch.float32, device="cuda")
    v = _launch(_padded_in(x), cin, cin, batch, h, w, 1, _packed_weights(wt, npad), cout, npad,
                256 if cout > 256 else 128, 64, alpha, beta, Y2_ACT[act], out, cs, OUT_F32)
    o = out.cpu().numpy()
    got = o[:, :, :cout].reshape(batch, h, w, cout).transpose(0, 3, 1, 2).astype(np.float64)
    _report(f"{R.ACT_NAMES[act]} fp32 head {cout} [{conv_variant} -> {v}]",
            R.check(got, g.pre, g.e_pre(R.C_ACC), act, out="f32"), g, got)
    if cs > cout:
        assert (o[:, :, cout:] == 7.0).all()


def test_logistic_into_channel_slice_of_concat_buffer(conv_variant):
    """input read from a channel slice, output written at a channel offset of a wider buffer (in-place route):
    neighbouring channels and the row padding of the other slices untouched, own pads zero"""
    batch, cin, h, w, cout = 2, 64, 13, 15, 128
    x, wt, alpha, beta = _operands(batch, cin, h, w, cout, 3, seed=99)
    beta = np.float32(beta * 8)
    g = _ref("slice", x, wt, alpha, beta, R.LOGISTIC)
    xin = _padded_in(x, cs=192, off=64, fill=3.0)
    out = torch.full((batch, h + 1, w + 1, 320), 5.0, dtype=torch.bfloat16, device="cuda")
    v = _launch(xin, 192, cin, batch, h, w, 3, _packed_weights(wt, cout), cout, cout, 128, 64, alpha, beta, 2, out,
                320, OUT_BF16, out_off=64, in_off=64)
    buf = out.float().cpu().numpy()
    _report(f"logistic into a concat slice [{conv_variant} -> {v}]",
            R.check_padded(buf[..., 64:64 + cout], cout, h, w, g.pre, g.e_pre(R.C_ACC), R.LOGISTIC))
    assert (buf[..., :64] == 5.0).all() and (buf[..., 64 + cout:] == 5.0).all()


@pytest.mark.parametrize("case", CONV_CASES, ids=lambda c: "b%d_c%d_%dx%d_n%d_k%d_bn%d_bk%d_a%d" % c)
def test_conv_cases_per_element(case, monkeypatch):
    """test_kernels_gpu.CONV_CASES (every kernel, tile shape and store mode the convolution tests reach) under the
    per-element bound instead of 1e-2 of the tensor maximum, each under the five kernel choices of conv_variant
    (one float64 reference per case)"""
    batch, cin, h, w, cout, ksize, block_n, block_k, act = case
    a64 = R.LEAKY if act == 1 else R.LINEAR
    x, wt, alpha, beta = _operands(batch, cin, h, w, cout, ksize, seed=1234 + cin + cout)
    beta = np.float32(beta * 0.2)
    acc, sab = R.conv_sums(x, wt, 1, ksize // 2)
    a, b = alpha.astype(np.float64).reshape(1, -1, 1, 1), beta.astype(np.float64).reshape(1, -1, 1, 1)
    g = R.Gemm(a * acc + b, a * sab, np.abs(b), a64)
    e = g.e_pre(R.C_ACC)
    npad = (cout + block_n - 1) // block_n * block_n
    x_d, wt_d = _padded_in(x), _packed_weights(wt, npad)
    for variant in ("auto", "slab", "pertap", "pair", "roundrobin"):
        monkeypatch.delenv("Y2_PAIR_BALANCE", raising=False)
        monkeypatch.delenv("Y2_CONV_VARIANT", raising=False)
        if variant == "roundrobin":
            monkeypatch.setenv("Y2_PAIR_BALANCE", "0")
        elif variant != "auto":
            monkeypatch.setenv("Y2_CONV_VARIANT", variant)
        out = torch.full((batch, h + 1, w + 1, cout), 7.0, dtype=torch.bfloat16, device="cuda")
        v = _launch(x_d, cin, cin, batch, h, w, ksize, wt_d, cout, npad, block_n, block_k, alpha, beta, act, out, cout,
                    OUT_BF16)
        _report(f"conv {case} [{variant} -> {v}]", R.check_padded(out.float().cpu().numpy(), cout, h, w, g.pre, e, a64))


@pytest.mark.parametrize("batch,c,h,w,n", [(2, 3, 50, 38, 32), (3, 3, 64, 96, 16), (1, 1, 33, 35, 8), (4, 3, 416, 416, 32)])
def test_stem_conv_pool_per_element(batch, c, h, w, n):
    """the fused first layer (conv 3x3 + affine + leaky + 2x2/2 maxpool from fp32 NCHW) through its maxpool"""
    rng = np.random.default_rng(99 + h + n)
    x = rng.uniform(0, 1, (batch, c, h, w)).astype(np.float32)
    s = (2.0 / (9 * c)) ** 0.5
    wt = R.bf16_rn(rng.uniform(-s, s, (n, c, 3, 3)))
    alpha = np.zeros(32, np.float32)
    beta = np.zeros(32, np.float32)
    alpha[:n] = rng.uniform(0.5, 1.5, n)
    beta[:n] = rng.uniform(-0.2, 0.2, n)
    wt_p = np.zeros((32, 32), np.float32)
    wt_p[:n, :c * 9] = wt.reshape(n, c * 9)
    dev = torch.device("cuda:0")
    wt_d = torch.from_numpy(wt_p).to(torch.bfloat16).to(dev)
    a_d, b_d, x_d = (torch.from_numpy(v).to(dev) for v in (alpha, beta, x))
    oh, ow = h // 2, w // 2
    out = torch.zeros(batch, oh + 1, ow + 1, 32, dtype=torch.bfloat16, device=dev)   # pads: zero at plan time
    _lib.check(_lib.load().y2_stem_conv_pool(x_d.data_ptr(), batch, c, h, w, wt_d.data_ptr(), 32, a_d.data_ptr(),
                                             b_d.data_ptr(), 1, out.data_ptr(), 32, _stream()), "stem")
    torch.cuda.synchronize()
    acc, sab = R.conv_sums(R.bf16_rn(x), wt, 1, 1)
    a, b = alpha[:n].astype(np.float64).reshape(1, -1, 1, 1), beta[:n].astype(np.float64).reshape(1, -1, 1, 1)
    g = R.Gemm(a * acc + b, a * sab, np.abs(b) + 0 * acc, R.LEAKY)
    buf = out.float().cpu().numpy()
    _report(f"stem b{batch} c{c} {h}x{w} n{n}",
            R.check_pooled(buf[:, :oh, :ow, :n].transpose(0, 3, 1, 2), g.pre, g.e_pre(R.C_ACC), R.LEAKY, 2, 2, 0))
    assert (buf[:, oh] == 0).all() and (buf[:, :, ow] == 0).all() and (buf[..., n:] == 0).all()


# the conv+pool shapes of test_kernels_gpu.py: one and several patches per CTA, odd row pairs per patch, 32 / 64 channels
@pytest.mark.parametrize("batch,cin,h,w,cout", [(2, 32, 208, 208, 64), (2, 64, 104, 104, 128), (1, 32, 50, 38, 64),
                                                (3, 64, 26, 30, 64), (2, 32, 13, 13, 128), (64, 32, 104, 104, 64),
                                                (64, 64, 52, 52, 128), (16, 32, 304, 304, 64), (24, 64, 152, 152, 128)])
def test_conv_pool_fused_per_element(batch, cin, h, w, cout):
    """Y2_OUT_BF16_POOLED (3x3 conv + affine + leaky + 2x2/2 maxpool in one launch) through its maxpool; the
    neighbouring channels of the wider buffer and the pads stay zero"""
    x, wt, alpha, beta = _operands(batch, cin, h, w, cout, 3, seed=5 + cin + cout + h)
    beta = np.float32(beta * 0.2)
    g = _ref(("pool", batch, cin, h, w, cout), x, wt, alpha, beta, R.LEAKY)
    oh, ow = h // 2, w // 2
    out = torch.zeros(batch, oh + 1, ow + 1, cout + 64, dtype=torch.bfloat16, device="cuda")
    _launch(_padded_in(x), cin, cin, batch, h, w, 3, _packed_weights(wt, cout), cout, cout, cout, cin, alpha, beta, 1,
            out, cout + 64, OUT_POOLED)
    buf = out.float().cpu().numpy()
    _report(f"conv+pool b{batch} c{cin} {h}x{w} n{cout}",
            R.check_pooled(buf[:, :oh, :ow, :cout].transpose(0, 3, 1, 2), g.pre, g.e_pre(R.C_ACC), R.LEAKY, 2, 2, 0))
    assert (buf[:, oh] == 0).all() and (buf[:, :, ow] == 0).all() and (buf[..., cout:] == 0).all()


@pytest.mark.parametrize("general", [False, True])
def test_shortcut_logistic(general, monkeypatch):
    """y2_shortcut with Y2_ACT_LOGISTIC (the general kernel: the elementwise one maps 0 to 0 only): pads zero, not
    f(0) = 0.5; bf16 output within the bound of one fp32 add and the device's expf"""
    if general:
        monkeypatch.setenv("Y2_SHORTCUT_GENERAL", "1")
    rng = np.random.default_rng(12)
    batch, c, h, w = 3, 64, 9, 13
    x = R.bf16_rn(rng.standard_normal((batch, c, h, w)) * 4)
    add = R.bf16_rn(rng.standard_normal((batch, c, h, w)) * 4)
    out = torch.full((batch, h + 1, w + 1, c), 3.0, dtype=torch.bfloat16, device="cuda")
    xp, ap = _padded_in(x), _padded_in(add)
    _lib.check(_lib.load().y2_shortcut(xp.data_ptr(), c, ap.data_ptr(), c, c, h, w, out.data_ptr(), c, c, c, h, w,
                                       batch, 2, None, c, None, _stream()), "shortcut")
    torch.cuda.synchronize()
    pre = x + add
    _report(f"shortcut logistic general={general}",
            R.check_padded(out.float().cpu().numpy(), c, h, w, pre, R.F32_U * np.abs(pre), R.LOGISTIC))


# ---- byte layers ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c,s,h,w,in_cs,out_cs", [(64, 2, 6, 10, 96, 32), (72, 3, 5, 7, 80, 16), (128, 2, 13, 9, 128, 32)])
def test_reverse_reorg_bit_exact(c, s, h, w, in_cs, out_cs):
    """y2_reorg_table_reverse + y2_reorg_gather_reverse (reverse = 1, depth-to-space) against ref64's forward = 1
    loop: a channel slice of a wider input, padding channels of the output left zero, pads zero"""
    dev = torch.device("cuda:0")
    batch = 3
    oc, oh, ow = c // (s * s), h * s, w * s
    x = R.bf16_rn(np.random.default_rng(c + s).standard_normal((batch, c, h, w)))
    xin = _padded_in(x, cs=in_cs, fill=9.0)
    out = torch.full((batch, oh + 1, ow + 1, out_cs), 2.0, dtype=torch.bfloat16, device=dev)
    out[..., oc:] = 0
    table = torch.zeros(oh * ow * oc, dtype=torch.int32, device=dev)
    _lib.check(_fn("y2_reorg_table_reverse", [vp, i32, i32, i32, i32, i32, vp])(
        table.data_ptr(), in_cs, c, h, w, s, _stream()), "table")
    _lib.check(_fn("y2_reorg_gather_reverse", [vp, i32, vp, i32, vp, i32, i32, i32, i32, i32, vp])(
        xin.data_ptr(), in_cs, out.data_ptr(), out_cs, table.data_ptr(), batch, c, h, w, s, _stream()), "gather")
    torch.cuda.synchronize()
    buf = out.float().cpu().numpy()
    rep = R.exact(buf[:, :oh, :ow, :oc].transpose(0, 3, 1, 2), R.reorg(x, s, 1))
    assert rep.ok, str(rep)
    assert (buf[:, oh] == 0).all() and (buf[:, :, ow] == 0).all() and (buf[..., oc:] == 0).all()


@pytest.mark.parametrize("c,h,w,in_cs", [(24, 3, 5, 32), (40, 2, 7, 64), (13, 4, 3, 32)])
def test_fc_pack_bit_exact(c, h, w, in_cs):
    """y2_fc_pack_tensor: one position-major row ((y*w + x)*c + ch) per image from a padded tensor with storage
    channels; y2_fc_pack_vec: an fp32 vector with a row stride > n, rounded to bf16.  Zero up to kpad"""
    dev = torch.device("cuda:0")
    batch = 3
    n = c * h * w
    kpad = (n + 63) // 64 * 64 + 64
    x = R.bf16_rn(np.random.default_rng(c).standard_normal((batch, c, h, w)))
    xin = _padded_in(x, cs=in_cs, fill=4.0)
    dst = torch.zeros(batch, 2, 2, kpad, dtype=torch.bfloat16, device=dev)
    _lib.check(_fn("y2_fc_pack_tensor", [vp, i32, i32, i32, i32, vp, i32, i32, vp])(
        xin.data_ptr(), in_cs, c, h, w, dst.data_ptr(), kpad, batch, _stream()), "fc_pack_tensor")
    torch.cuda.synchronize()
    got = dst.float().cpu().numpy()
    assert R.exact(got[:, 0, 0, :n], x.transpose(0, 2, 3, 1).reshape(batch, n)).ok
    assert (got[:, 0, 0, n:] == 0).all() and (got[:, 0, 1:] == 0).all() and (got[:, 1] == 0).all()
    stride = n + 5
    v = np.random.default_rng(n).standard_normal((batch, stride)).astype(np.float32)
    dst.zero_()
    vd = torch.from_numpy(v).to(dev)
    _lib.check(_fn("y2_fc_pack_vec", [vp, i32, i32, vp, i32, i32, vp])(
        vd.data_ptr(), stride, n, dst.data_ptr(), kpad, batch, _stream()), "fc_pack_vec")
    torch.cuda.synchronize()
    got = dst.float().cpu().numpy()
    assert R.exact(got[:, 0, 0, :n], R.bf16_rn(v[:, :n])).ok
    assert (got[:, 0, 0, n:] == 0).all() and (got[:, 0, 1:] == 0).all() and (got[:, 1] == 0).all()


# ---- networks, layer-local -----------------------------------------------------------------------------------------
def _net(batch, w, h, c=3):
    return f"[net]\nbatch={batch}\nsubdivisions=1\nheight={h}\nwidth={w}\nchannels={c}\n\n"


def _conv(filters, size, stride=1, bn=1, act="leaky", pad=1):
    return (f"[convolutional]\n" + ("batch_normalize=1\n" if bn else "") +
            f"filters={filters}\nsize={size}\nstride={stride}\npad={pad}\nactivation={act}\n\n")


def every_activation_cfg(batch=3, w=40, h=24):
    """One convolution per activation, 1x1 and 3x3 alternating (the first a 1x1 over the 3-channel input: packed_in),
    filter counts with and without storage padding; a
    logistic convolution (epilogue); plse (f(0) = 0.5) feeding a 3x3 convolution, so that a non-zero halo would
    show; a relu head on an fp32 flat output feeding avgpool and softmax (post-activation on the F32 head)"""
    acts = ["relu", "relie", "ramp", "linear", "plse", "tanh", "leaky", "elu", "loggy", "stair", "hardtan", "lhtan",
            "logistic"]
    s = _net(batch, w, h)
    for k, a in enumerate(acts):
        s += _conv([24, 40, 32, 64][k % 4], 3 if k % 2 else 1, bn=k % 3 != 1, act=a)
    return s + _conv(10, 1, bn=0, act="relu") + "[avgpool]\n\n[softmax]\ngroups=1\n\n"


def gathered_cfg(batch=3, first=11):
    """convolutions off the native 1x1 / 3x3 'same' path: an 11x11/4 (use_patches 1) or 5x5 (use_patches 3) first
    layer, then a 3/2 maxpool on an odd extent, 5x5 pad 2, 3x3 pad 0, 1x1 stride 2 and 3x3 stride 2 layers
    (use_patches 2)"""
    s = _net(batch, 100, 76) + _conv(32, 11, stride=4) if first == 11 else _net(batch, 63, 47) + _conv(24, 5, act="relu")
    s += "[maxpool]\nsize=3\nstride=2\n\n"
    s += _conv(64, 5) + _conv(32, 3, pad=0, act="elu") + _conv(64, 1, stride=2) + _conv(32, 3, stride=2, act="tanh")
    return s + _conv(20, 1, bn=0, act="linear")


def packed_input_cfg(batch=3, w=30, h=22):
    """a 4-channel input under a 1x1 first layer (packed_in), then a 3x3 layer and a linear head"""
    return _net(batch, w, h, c=4) + _conv(32, 1) + _conv(64, 3, act="logistic") + _conv(16, 1, bn=0, act="linear")


def connected_cfg(batch=3, w=36, h=20):
    """a dropout between a convolution and a maxpool (tensor alias), a connected layer from a 24-channel tensor with
    h, w > 1, connected -> dropout -> connected with batchnorm and tanh (the fp32 vector path), softmax"""
    s = _net(batch, w, h) + _conv(16, 3) + "[dropout]\nprobability=.5\n\n[maxpool]\nsize=2\nstride=2\n\n"
    s += _conv(24, 3, act="relu") + "[maxpool]\nsize=2\nstride=2\n\n"
    s += "[connected]\noutput=50\nactivation=relu\n\n[dropout]\nprobability=.5\n\n"
    s += "[connected]\nbatch_normalize=1\noutput=30\nactivation=tanh\n\n"
    s += "[connected]\noutput=10\nactivation=linear\n\n[softmax]\ngroups=1\n\n"
    return s


def _write_weights(path, layers, seed, bias):
    """synth.write_weights' layout with a chosen bias spread (biases ~ U(-bias, bias)): pre-activations on both sides
    of every breakpoint"""
    with open(path, "wb") as f:
        f.write(np.int32([0, 1, 0, 0]).tobytes())
        for i, l in enumerate(layers):
            if l.type not in ("convolutional", "connected"):
                continue
            rng = np.random.default_rng(seed + i)
            k = l.size if l.type == "convolutional" else 1
            cin = l.c if l.type == "convolutional" else l.c * l.h * l.w
            s = np.sqrt(2.0 / (k * k * cin))
            b = np.float32(rng.uniform(-bias, bias, l.n))
            wt = np.float32(rng.uniform(-s, s, l.n * cin * k * k))
            bn = [np.float32(rng.uniform(lo, hi, l.n)) for lo, hi in ((.5, 1.5), (-.1, .1), (.5, 1.5))] if l.bn else []
            f.write(b.tobytes())
            if l.type == "convolutional":
                f.write(b"".join(v.tobytes() for v in bn) + wt.tobytes())
            else:
                f.write(wt.tobytes() + b"".join(v.tobytes() for v in bn))


EPILOGUE = (R.LEAKY, R.LINEAR, R.LOGISTIC)


def _gathered(l):
    return not (l.stride == 1 and l.size in (1, 3) and l.pad == l.size // 2)


def _expected_launches(layers, kernels):
    """launches of one forward pass as the paths under test take them: a conv is its plan, plus a gather or pack
    when it is the first layer or off the native path, plus the activation pass when the epilogue lacks its
    activation (stem-fused: one launch; the maxpool of a fused pair: none); a connected layer packs, runs its plan and
    activates when needed"""
    n = 0
    for i, l in enumerate(layers):
        if l.type == "convolutional":
            if kernels[i] == 4:
                n += 1
            else:
                n += 1 + int(i == 0 or _gathered(l)) + int(l.act not in EPILOGUE)
        elif l.type == "connected":
            n += 2 + int(l.act not in EPILOGUE)
        elif l.type == "maxpool":
            n += 0 if kernels[i - 1] in (3, 4) else 1
        elif l.type in ("reorg", "avgpool", "softmax", "region", "shortcut"):
            n += 1
        elif l.type == "route":
            assert len(l.inputs) == 1
    return n


def _check_network(tmp_path, name, cfg_text, bias=0.1, seed=1234):
    batch, layers = R.parse_cfg(cfg_text)
    cfg = tmp_path / f"{name}.cfg"
    cfg.write_text(cfg_text)
    wpath = tmp_path / f"{name}.weights"
    if bias == 0.1:
        synth.write_weights(wpath, cfg_text, seed=seed)
    else:
        _write_weights(wpath, layers, seed, bias)
    weights = R.read_weights(wpath.read_bytes(), layers)
    x = synth.images(batch, layers[0].c, layers[0].h, layers[0].w, seed=42)
    dn.set_gpu_index(0)
    net = dn.parse_network_cfg(cfg)
    dn.load_weights(net, wpath)
    lib = dn.lib()
    try:
        dn.network_predict(net, x)
        launches = lib.network_launch_count(net)
        kernels = [lib.network_conv_kernel(net, i) for i in range(net.n)]
        exports = {}
        for i, l in enumerate(layers):
            if l.type not in ("cost", "region"):
                exports[i] = dn.get_network_output_layer(net, i).astype(np.float64)
    finally:
        dn.free_network(net)
    assert launches == _expected_launches(layers, kernels), \
        f"{name}: {launches} launches, the paths under test take {_expected_launches(layers, kernels)} (kernels {kernels})"

    def inp(i, k):
        if k < 0:
            return x.astype(np.float64)
        s = layers[k]
        return exports[k].reshape(batch, s.out_c, s.out_h, s.out_w)

    flat_out = {i for i, l in enumerate(layers) if l.type == "convolutional" and
                (i + 1 == len(layers) or layers[i + 1].type in ("avgpool", "region"))}
    worst = []
    for i, l in enumerate(layers):
        if i not in exports:
            continue
        got = exports[i].reshape(batch, -1)
        ins = [inp(i, k) for k in l.inputs]
        tag = f"{name} layer {i} {l.type}"
        if l.type in ("convolutional", "connected"):
            g = R.layer_ref(l, ins, weights[i])
            f32 = l.type == "connected" or i in flat_out
            post = l.act not in EPILOGUE and not f32
            rep = R.check(got.reshape(g.pre.shape), g.pre, g.e_pre(R.C_ACC, post_act=post), l.act,
                          out="f32" if f32 else "bf16")
            tag += f" {R.ACT_NAMES[l.act]} [{VARIANT_NAMES.get(kernels[i], 'fc')}{' post_act' if l.act not in EPILOGUE else ''}" \
                   f"{' gathered' if l.type == 'convolutional' and (i == 0 or _gathered(l)) else ''}]"
            if l.type == "convolutional" and kernels[i] in (3, 4):   # the fused kernel's own output: the maxpool's
                m = layers[i + 1]
                prep = R.check_pooled(exports[i + 1].reshape(batch, m.out_c, m.out_h, m.out_w), g.pre,
                                      g.e_pre(R.C_ACC), l.act, m.size, m.stride, m.pad)
                print(f"{name} layer {i + 1} maxpool fused into {VARIANT_NAMES[kernels[i]]}: {prep}")
                assert prep.ok
                worst.append(prep.worst)
        elif l.type == "maxpool" and kernels[i - 1] in (3, 4):
            continue
        elif l.type == "avgpool":
            xin = ins[0]
            want = R.avgpool(xin)
            hw = l.h * l.w
            bound = (hw + 2) * R.F32_U * np.abs(xin).reshape(batch, l.c, -1).mean(axis=2)   # sequential fp32 sum
            rep = R._interval_report(got, want - bound, want + bound)
        elif l.type == "softmax":
            xin = ins[0].reshape(batch, -1)
            want = R.softmax(xin, l.groups, l.temperature)
            n = xin.shape[1] // l.groups
            spread = (xin.max(axis=1, keepdims=True) - xin.min(axis=1, keepdims=True)) / l.temperature
            bound = want * R.F32_U * (n + 4 + 2 * spread)   # exp of float differences, float sum, divide
            rep = R._interval_report(got, want - bound, want + bound)
        else:
            rep = R.exact(got, np.asarray(R.layer_ref(l, ins)).reshape(batch, -1))
        print(f"{tag}: {rep}")
        assert rep.ok, f"{tag}: {rep}"
        worst.append(rep.worst)
    return layers, kernels, max(worst)


def test_mini_alexnet_layer_local(tmp_path):
    """relu and elu convolutions (post-activation), connected layers from a tensor and from a vector, one with
    batchnorm and tanh, dropout aliases, softmax"""
    text = synth.mini_alexnet_cfg(batch=3, w=48, h=32)
    layers, kernels, worst = _check_network(tmp_path, "mini-alexnet", text)
    kinds = [l.type for l in layers]
    assert kinds.count("connected") == 3 and kinds.count("dropout") == 2
    assert {R.ACT_NAMES[l.act] for l in layers if l.type == "convolutional"} == {"relu", "elu"}


def test_mini_reorg_reverse_layer_local(tmp_path):
    layers, kernels, worst = _check_network(tmp_path, "mini-reorg-reverse",
                                            synth.mini_reorg_reverse_cfg(batch=3, w=48, h=32))
    assert any(l.type == "reorg" and l.reverse for l in layers)


def test_every_activation_layer_local(tmp_path):
    layers, kernels, worst = _check_network(tmp_path, "every-activation", every_activation_cfg(), bias=5.0)
    convs = [l for l in layers if l.type == "convolutional"]
    assert {l.act for l in convs} == set(range(13))
    plse = next(i for i, l in enumerate(layers) if l.act == R.PLSE and l.type == "convolutional")
    assert layers[plse + 1].size == 3


@pytest.mark.parametrize("first", [11, 5])
def test_gathered_convolutions_layer_local(tmp_path, first):
    layers, kernels, worst = _check_network(tmp_path, f"gathered-{first}", gathered_cfg(first=first), bias=1.0)
    assert sum(_gathered(l) for l in layers if l.type == "convolutional") == 5
    pool = next(l for l in layers if l.type == "maxpool")
    assert (pool.size, pool.stride) == (3, 2) and (pool.h % 2, pool.w % 2) != (0, 0)


def test_packed_input_layer_local(tmp_path):
    layers, kernels, worst = _check_network(tmp_path, "packed-input", packed_input_cfg(), bias=1.0)
    assert layers[0].c == 4 and layers[0].size == 1


def test_connected_variants_layer_local(tmp_path):
    layers, kernels, worst = _check_network(tmp_path, "connected", connected_cfg(), bias=0.5)
    kinds = [l.type for l in layers]
    assert kinds[1:3] == ["dropout", "maxpool"] and kernels[0] != 4
    fc = layers[kinds.index("connected")]
    assert fc.c == 24 and fc.h > 1 and fc.w > 1
