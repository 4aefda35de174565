"""NormalConv1d / NormalConv2d at the edges of the implicit-GEMM conv path (SampledConv2dImplicit: NHWC activations through
a TMA im2col tensor map, weights in (o, kh, kw, c) order) against torch's fp64 conv on the same eps: output, input
gradient and the gradients of weight and bias mean / scale.

  A  1-d layers (a height-1 2-d conv with stride (1, s), dilation (1, d), padding (0, p)), including a sequence that spans
     many 128-row tiles and a patch embedding with kernel = stride;
  B  strides with sh != sw (the im2col element strides and the (h, w) split of an output row);
  C  output and channel edges: odd / small / > 256 output channels, feature maps too large for the fused transposing pass,
     every P % 4, 1x1 outputs, no bias;
  D  both sides of every limit of the im2col descriptor: the kernel on the eligible side, the explicit lowering on the
     other, both exact;
  E  the in-kernel Philox draw against the weights `.materialize` reports for the same draw;
  F  the explicit NHWC lowering (bnn_im2col_nhwc / bnn_col2im_nhwc) and the weight layout on their own.
"""
import pytest
import torch
import torch.nn.functional as F

import bayesianneuralnetworks_b200 as bnn
from bayesianneuralnetworks_b200 import _C, runtime
from bayesianneuralnetworks_b200.nn import FlipOutNormalConv2d, NormalConv1d, NormalConv2d

pytestmark = pytest.mark.gpu

TOL = {"fp32": 2e-5, "tf32": 2e-3}
# fp32 mode accumulates a long reduction with an error that grows linearly in its length (see
# test_conv_layer_at_configuration_scale_matches_torch_conv2d): the weight gradient of the 2001-long sequence below (8004
# terms per element) is 3e-5 off on a B200, so weight and bias gradients of more than 4096 terms get 1e-4
LONG_REDUCTION, LONG_TOL = 4096, 1e-4
GRAD_NAMES = ("dx", "d mean_w", "d scale_w", "d mean_b", "d scale_b")


@pytest.fixture(autouse=True)
def _defaults():
    def reset():
        bnn.set_precision("fp32")
        bnn.set_conv_output_format("contiguous")
        bnn.graph_safe_rng(False)
        bnn.set_mc_batching("auto")
    reset()
    yield
    reset()


def rel_err(got, ref):
    """max-norm relative error |got - ref|_max / |ref|_max."""
    ref = ref.detach().double()
    return float((got.detach().double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def _params(layer):
    return [layer.weight.mean, layer.weight.scale] + ([layer.bias.mean, layer.bias.scale] if layer.bias is not None else [])


def forward(layer, x, S, B, shared, eps=None):
    """The layer in a batched Monte-Carlo pass of S samples (shared: x is the B-row network input, else S*B sample-major
    rows), eps injected when given; returns the leaf input and the output."""
    layer.zero_grad(set_to_none=True)
    x = x.detach().clone().requires_grad_(True)
    ctx = runtime.MCContext(S, B)
    ctx.expanded = not shared
    with bnn.injected_eps(eps or {}), runtime.mc_batch(ctx):
        y = layer(x)
    return x, y


def reference(layer, x, S, B, shared, dy, eps_w, eps_b):
    """fp64 torch, one conv per sample with W_s = mean + (1e-10 + softplus(scale)) eps_s; output and gradients."""
    conv = F.conv1d if isinstance(layer, NormalConv1d) else F.conv2d
    xd = x.detach().double().requires_grad_(True)
    p = [t.detach().double().requires_grad_(True) for t in _params(layer)]
    outs = []
    for s in range(S):
        w = p[0] + (1e-10 + F.softplus(p[1])) * eps_w[s].double()
        b = p[2] + (1e-10 + F.softplus(p[3])) * eps_b[s].double() if layer.bias is not None else None
        outs.append(conv(xd if shared else xd[s * B:(s + 1) * B], w, b, layer.stride, layer.padding, layer.dilation))
    ref = torch.cat(outs)
    ref.backward(dy.double())
    return ref, [xd.grad] + [t.grad for t in p]


def assert_matches(layer, x, y, ref, ref_grads, prec):
    assert y.shape == ref.shape
    err = rel_err(y, ref)
    assert err < TOL[prec], ("y", err)
    terms = y.shape[0] * y[0, 0].numel()                # S*B*OH*OW products per weight / bias gradient element
    long = prec == "fp32" and terms > LONG_REDUCTION
    for i, (name, got, want) in enumerate(zip(GRAD_NAMES, [x.grad] + [t.grad for t in _params(layer)], ref_grads)):
        err = rel_err(got, want)
        assert err < (LONG_TOL if long and i > 0 else TOL[prec]), (name, err)


def parity(layer, x_shape, S, B, shared, prec, seed, channels_last=False):
    """Injected-eps parity of one layer; returns the layer's output."""
    bnn.set_precision(prec)
    assert layer._implicit
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn((B if shared else S * B,) + tuple(x_shape), device="cuda", generator=g)
    if channels_last:
        bnn.set_conv_output_format("preserve")
        x = x.contiguous(memory_format=torch.channels_last)
    eps_w = torch.randn((S,) + tuple(layer.weight.mean.shape), device="cuda", generator=g)
    eps = {layer.weight: eps_w}
    eps_b = None
    if layer.bias is not None:
        eps_b = eps[layer.bias] = torch.randn(S, layer.out_channels, device="cuda", generator=g)
    x, y = forward(layer, x, S, B, shared, eps)
    dy = torch.randn(y.shape, device="cuda", generator=g)
    if channels_last:                   # 'preserve': the result follows the input's format, as torch's conv does
        assert y.is_contiguous(memory_format=torch.channels_last)
        dy = dy.contiguous(memory_format=torch.channels_last)
    else:
        assert y.is_contiguous()
    y.backward(dy)
    ref, ref_grads = reference(layer, x, S, B, shared, dy, eps_w, eps_b)
    assert_matches(layer, x, y, ref, ref_grads, prec)
    return y


# ------------------------------------------------------------------------------------------------ A. NormalConv1d
CONV1D = {
    # (B, S, Cin, Cout, L, k, stride, padding, dilation, bias)
    "s1": (3, 2, 32, 32, 37, 3, 1, 1, 1, True),             # stride-1 input-gradient gather with H = 1
    "s2_odd_len": (2, 3, 64, 48, 41, 5, 2, 2, 1, False),    # stride 2 on an odd length, no bias, Cout % 32 != 0
    "s3_d2": (2, 2, 96, 64, 50, 3, 3, 2, 2, True),          # stride 3 with dilation 2
    "long_seq": (2, 2, 32, 64, 2001, 3, 1, 1, 1, True),     # 16 row blocks per sequence, CTA-pair eligible, P % 4 == 1
    "patch_k4s4": (3, 2, 64, 10, 32, 4, 4, 0, 1, True),     # kernel = stride = 4, Cout = 10 (dY pitch not 16-byte aligned)
}


@pytest.mark.parametrize("prec", ["fp32", "tf32"])
@pytest.mark.parametrize("shared", [True, False])
@pytest.mark.parametrize("case", list(CONV1D))
def test_conv1d_matches_torch(case, shared, prec):
    B, S, Cin, Cout, L, k, s, p, d, bias = CONV1D[case]
    torch.manual_seed(101)
    layer = NormalConv1d(Cin, Cout, k, stride=s, padding=p, dilation=d, bias=bias).cuda()
    y = parity(layer, (Cin, L), S, B, shared, prec, seed=102)
    assert y.shape == (S * B, Cout, (L + 2 * p - d * (k - 1) - 1) // s + 1)


# ------------------------------------------------------------------------------------------------ B. sh != sw
ASYMMETRIC = {
    # (B, S, Cin, Cout, H, W, k, stride, padding, dilation)
    "s1x2": (2, 2, 32, 32, 7, 10, (3, 2), (1, 2), (1, 0), 1),
    "s2x1": (2, 2, 32, 64, 11, 6, (2, 3), (2, 1), (0, 1), 1),
    "s3x2": (2, 2, 64, 32, 13, 9, (3, 1), (3, 2), (1, 0), 1),
    "s2x3_d1x2": (2, 2, 32, 40, 8, 14, (1, 3), (2, 3), (0, 1), (1, 2)),
}


@pytest.mark.parametrize("prec", ["fp32", "tf32"])
@pytest.mark.parametrize("layout", ["nchw", "channels_last"])
@pytest.mark.parametrize("shared", [True, False])
@pytest.mark.parametrize("case", list(ASYMMETRIC))
def test_asymmetric_stride_matches_torch(case, shared, layout, prec):
    B, S, Cin, Cout, H, W, k, s, p, d = ASYMMETRIC[case]
    torch.manual_seed(201)
    layer = NormalConv2d(Cin, Cout, k, stride=s, padding=p, dilation=d).cuda()
    parity(layer, (Cin, H, W), S, B, shared, prec, seed=202, channels_last=layout == "channels_last")


# ------------------------------------------------------------------------------------------------ C. output / channel edges
EDGES = {
    # (B, S, Cin, Cout, H, W, k, padding, bias, what the fused NCHW -> NHWC + bias-gradient pass returns per backward)
    "cout3_p30": (2, 2, 32, 3, 6, 5, 3, 1, True, ["nhwc"]),          # P % 4 == 2, scalar transposing pass
    "cout10_p25": (2, 2, 32, 10, 5, 5, 3, 1, True, ["nhwc"]),        # P % 4 == 1
    "cout33_p15": (2, 2, 64, 33, 7, 5, 3, 0, True, ["nhwc"]),        # P % 4 == 3
    "cout288_p16": (2, 2, 32, 288, 4, 4, 3, 1, True, [None]),        # > 256 channels with a bias: the pass declines
    "map32x32_cout64": (1, 2, 32, 64, 32, 32, 3, 1, True, [None]),   # (Cout + 1) * P * 4 > 48 KiB: the pass declines
    "out1x1": (3, 2, 32, 32, 3, 3, 3, 0, True, []),                  # dY is NCHW- and NHWC-contiguous: no pass
    "no_bias": (2, 2, 64, 64, 6, 6, 3, 1, False, ["nhwc"]),
}


@pytest.mark.parametrize("prec", ["fp32", "tf32"])
@pytest.mark.parametrize("shared", [True, False])
@pytest.mark.parametrize("case", list(EDGES))
def test_output_and_channel_edges_match_torch(case, shared, prec, monkeypatch):
    B, S, Cin, Cout, H, W, k, p, bias, passes = EDGES[case]
    returned = []
    real = _C.nchw_to_nhwc_bias_grad

    def recording(*a, **kw):
        out = real(*a, **kw)
        returned.append(None if out is None else "nhwc")
        return out
    monkeypatch.setattr(_C, "nchw_to_nhwc_bias_grad", recording)
    torch.manual_seed(301)
    layer = NormalConv2d(Cin, Cout, k, padding=p, bias=bias).cuda()
    parity(layer, (Cin, H, W), S, B, shared, prec, seed=302)
    assert returned == passes


# ------------------------------------------------------------------------------------------------ D. descriptor limits
# im2col tensor maps of rank 4 take filter-window corners in [-128, 127], tap offsets (k - 1) * d < 256 and element
# strides <= 8 (conv_ok; the stride-1 input gradient has its own corners, tma_conv_dgrad).  Outside them the C entry points
# refuse and the layer lowers explicitly.  (kernel runs for: forward, input gradient, weight gradient)
LIMITS = {
    # (cls, Cout, spatial, k, stride, padding, dilation, (fwd, dgrad, wgrad) on the kernels)
    "stride_w8": (NormalConv2d, 32, (3, 20), 3, (1, 8), 1, 1, (True, False, True)),
    "stride_w9": (NormalConv2d, 32, (3, 20), 3, (1, 9), 1, 1, (False, False, False)),
    "stride8": (NormalConv2d, 32, (18, 18), 3, 8, 1, 1, (True, False, True)),
    "stride9": (NormalConv2d, 32, (20, 20), 3, 9, 1, 1, (False, False, False)),
    "pad127_k1": (NormalConv2d, 32, (2, 3), 1, 1, (0, 127), 1, (True, True, True)),
    "pad128_k1": (NormalConv2d, 32, (2, 3), 1, 1, (0, 128), 1, (False, False, False)),     # upper corner 128
    "pad128_k3": (NormalConv2d, 32, (2, 3), (1, 3), 1, (0, 128), 1, (True, True, True)),
    "pad129_k3": (NormalConv2d, 32, (2, 3), (1, 3), 1, (0, 129), 1, (False, False, False)),  # lower corner -129
    # padding 128 at k = 2 keeps every corner in range: only the filter extent (k - 1) * d differs
    "extent255": (NormalConv2d, 32, (2, 3), (1, 2), 1, (0, 128), (1, 255), (True, True, True)),
    "extent256": (NormalConv2d, 32, (2, 3), (1, 2), 1, (0, 128), (1, 256), (False, False, False)),
    "corner_m128": (NormalConv2d, 32, (2, 140), (1, 3), 1, 0, (1, 64), (True, True, True)),
    "corner_m130": (NormalConv2d, 32, (2, 140), (1, 3), 1, 0, (1, 65), (False, False, False)),
    "conv1d_s16": (NormalConv1d, 64, (64,), 16, 16, 0, 1, (False, False, False)),          # 1-d patch embedding
}


def _record_lowering(monkeypatch):
    """Names of the explicit-lowering calls (bnn_im2col_nhwc / bnn_col2im_nhwc) made from now on."""
    calls = []
    for name in ("im2col_nhwc", "col2im_nhwc"):
        real = getattr(_C, name)
        monkeypatch.setattr(_C, name, lambda *a, _real=real, _name=name: calls.append(_name) or _real(*a))
    return calls


@pytest.mark.parametrize("shared", [True, False])
@pytest.mark.parametrize("case", list(LIMITS))
def test_descriptor_limits_take_the_kernel_or_the_explicit_lowering(case, shared, monkeypatch):
    """TF32 mode on both sides of each im2col descriptor limit: every request matches fp64 torch, the eligible side runs
    on the kernels and the other lowers explicitly (forward: bnn_im2col_nhwc; input gradient: bnn_col2im_nhwc; weight
    gradient: bnn_im2col_nhwc) instead of raising BNN_ERR_UNSUPPORTED."""
    cls, Cout, spatial, k, s, p, d, (fwd, dgrad, wgrad) = LIMITS[case]
    Cin, B, S = 32, 2, 2
    bnn.set_precision("tf32")
    torch.manual_seed(401)
    layer = cls(Cin, Cout, k, stride=s, padding=p, dilation=d).cuda()
    assert layer._implicit
    g = torch.Generator(device="cuda").manual_seed(402)
    x = torch.randn((B if shared else S * B, Cin) + spatial, device="cuda", generator=g)
    eps_w = torch.randn((S,) + tuple(layer.weight.mean.shape), device="cuda", generator=g)
    eps_b = torch.randn(S, Cout, device="cuda", generator=g)
    calls = _record_lowering(monkeypatch)
    x, y = forward(layer, x, S, B, shared, {layer.weight: eps_w, layer.bias: eps_b})
    assert calls == ([] if fwd else ["im2col_nhwc"])
    calls.clear()
    dy = torch.randn(y.shape, device="cuda", generator=g)
    y.backward(dy)
    assert calls == ([] if dgrad else ["col2im_nhwc"]) + ([] if wgrad else ["im2col_nhwc"])
    ref, ref_grads = reference(layer, x, S, B, shared, dy, eps_w, eps_b)
    assert_matches(layer, x, y, ref, ref_grads, "tf32")


def test_flipout_conv_beyond_the_stride_limit_lowers_explicitly(monkeypatch):
    """FlipOutNormalConv2d with stride 9 in TF32 mode: both of its convolutions (mean, and stddev on the sign-flipped input)
    lower explicitly in both directions, and the layer matches conv(x, mean) + conv(x * S, stddev) * R in fp64."""
    bnn.set_precision("tf32")
    torch.manual_seed(411)
    layer = FlipOutNormalConv2d(32, 32, 3, stride=9).cuda()
    x = torch.randn(4, 32, 20, 20, device="cuda", requires_grad=True)
    calls = _record_lowering(monkeypatch)
    y = layer(x)
    assert calls == ["im2col_nhwc"] * 2
    calls.clear()
    dy = torch.randn(y.shape, device="cuda")
    y.backward(dy)
    assert sorted(calls) == ["col2im_nhwc"] * 2 + ["im2col_nhwc"] * 2
    R, Sg = layer.R.double(), layer.S.double()
    xd = x.detach().double().requires_grad_(True)
    mu = layer.weight.mean.detach().double().requires_grad_(True)
    rho = layer.weight.scale.detach().double().requires_grad_(True)
    ref = F.conv2d(xd, mu, None, 9) + F.conv2d(xd * Sg, 1e-10 + F.softplus(rho), None, 9) * R
    ref.backward(dy.double())
    assert y.shape == ref.shape
    for name, got, want in (("y", y, ref), ("dx", x.grad, xd.grad), ("d mean", layer.weight.mean.grad, mu.grad),
                            ("d scale", layer.weight.scale.grad, rho.grad)):
        err = rel_err(got, want)
        assert err < TOL["tf32"], (name, err)


# ------------------------------------------------------------------------------------------------ E. Philox draws
@pytest.mark.parametrize("graph_rng", [False, True])
@pytest.mark.parametrize("prec", ["fp32", "tf32"])
@pytest.mark.parametrize("kind", ["conv2d_s1", "conv1d_s2"])
def test_philox_draw_matches_the_materialised_weights(kind, prec, graph_rng):
    """Without injection the kernels draw eps in-kernel (forward, and again in the input- and weight-gradient kernels).
    The eps of the draw, recovered from `.materialize` of the same draw as (W_s - mean) / stddev in fp64, must reproduce
    the output and every gradient through torch: stride 1 (the transposed-filter input-gradient gather in TF32) and a
    strided 1-d layer, S = 4 on a shared input, on a second forward (draw begin != 0), and once with the device-side step
    counter after advance_rng_step()."""
    bnn.set_precision(prec)
    S, B = 4, 2
    torch.manual_seed(501)
    if kind == "conv2d_s1":
        layer, x_shape = NormalConv2d(32, 64, 3, padding=1).cuda(), (32, 6, 5)
    else:
        layer, x_shape = NormalConv1d(64, 32, 3, stride=2, padding=1).cuda(), (64, 23)
    assert layer._implicit
    g = torch.Generator(device="cuda").manual_seed(502)
    x0 = torch.randn((B,) + x_shape, device="cuda", generator=g)
    forward(layer, x0, S, B, True)                  # the first pass; the checked one draws from a later counter
    if graph_rng:
        bnn.graph_safe_rng(True)
        bnn.advance_rng_step()
    x, y = forward(layer, x0, S, B, True)
    assert layer.weight._last[0] != 0 and layer.weight._last[1] == S
    dy = torch.randn(y.shape, device="cuda", generator=g)
    y.backward(dy)
    eps = []
    with torch.no_grad():
        for w in (layer.weight, layer.bias):
            W_s = w.materialize(*w._last).double()
            eps.append((W_s - w.mean.double()) / (1e-10 + F.softplus(w.scale.double())))
    e = eps[0]
    assert abs(float(e.mean())) < 0.05 and 0.9 < float(e.std()) < 1.1       # a standard-normal draw ...
    assert not torch.equal(e[0], e[1])                                       # ... fresh for every sample
    ref, ref_grads = reference(layer, x, S, B, True, dy, eps[0], eps[1])
    assert_matches(layer, x, y, ref, ref_grads, prec)


# ------------------------------------------------------------------------------------------------ F. explicit lowering
LOWERING = {
    # (C, H, W, (kh, kw), (sh, sw), (ph, pw), (dh, dw)): the geometries of A-D, plus C = 4
    "c4": (4, 5, 7, (3, 3), (1, 1), (1, 1), (1, 1)),
    "a_s1": (32, 1, 37, (1, 3), (1, 1), (0, 1), (1, 1)),
    "a_s2_odd": (64, 1, 41, (1, 5), (1, 2), (0, 2), (1, 1)),
    "a_s3_d2": (96, 1, 50, (1, 3), (1, 3), (0, 2), (1, 2)),
    "a_long": (32, 1, 2001, (1, 3), (1, 1), (0, 1), (1, 1)),
    "a_k4s4": (64, 1, 32, (1, 4), (1, 4), (0, 0), (1, 1)),
    "b_s1x2": (32, 7, 10, (3, 2), (1, 2), (1, 0), (1, 1)),
    "b_s2x1": (32, 11, 6, (2, 3), (2, 1), (0, 1), (1, 1)),
    "b_s3x2": (64, 13, 9, (3, 1), (3, 2), (1, 0), (1, 1)),
    "b_s2x3_d1x2": (32, 8, 14, (1, 3), (2, 3), (0, 1), (1, 2)),
    "c_out1x1": (32, 3, 3, (3, 3), (1, 1), (0, 0), (1, 1)),
    "c_map32": (32, 32, 32, (3, 3), (1, 1), (1, 1), (1, 1)),
    "d_stride9": (32, 20, 20, (3, 3), (9, 9), (1, 1), (1, 1)),
    "d_pad128_k1": (32, 2, 3, (1, 1), (1, 1), (0, 128), (1, 1)),
    "d_pad129_k3": (32, 2, 3, (1, 3), (1, 1), (0, 129), (1, 1)),
    "d_extent256": (32, 2, 3, (1, 2), (1, 1), (0, 128), (1, 256)),
    "d_corner_m130": (32, 2, 140, (1, 3), (1, 1), (0, 0), (1, 65)),
    "d_conv1d_s16": (32, 1, 64, (1, 16), (1, 16), (0, 0), (1, 1)),
}


@pytest.mark.parametrize("case", list(LOWERING))
def test_nhwc_lowering_matches_unfold_and_fold(case):
    """bnn_im2col_nhwc is F.unfold with its columns reordered from (c, kh, kw) to (kh, kw, c), bit for bit;
    bnn_col2im_nhwc is F.fold of the same reordering (every input pixel written, also those no window reaches)."""
    C, H, W, k, s, p, d = LOWERING[case]
    n = 3
    OH = (H + 2 * p[0] - d[0] * (k[0] - 1) - 1) // s[0] + 1
    OW = (W + 2 * p[1] - d[1] * (k[1] - 1) - 1) // s[1] + 1
    L, taps = OH * OW, k[0] * k[1]
    geom = _C.conv_geom(n, H, W, C, OH, OW, 1, k[0], k[1], s, p, d)
    g = torch.Generator(device="cuda").manual_seed(601)
    x = torch.randn(n, C, H, W, device="cuda", generator=g).contiguous(memory_format=torch.channels_last)
    col = _C.im2col_nhwc(x, geom, n)
    want = F.unfold(x, k, d, p, s).view(n, C, taps, L).permute(0, 3, 2, 1).reshape(n * L, taps * C)
    assert col.shape == want.shape and torch.equal(col, want)
    dcol = torch.randn(n * L, taps * C, device="cuda", generator=g)
    dx = torch.full((n, C, H, W), float("nan"), device="cuda").contiguous(memory_format=torch.channels_last)
    _C.col2im_nhwc(dcol, dx, geom, n)
    want = F.fold(dcol.double().view(n, L, taps, C).permute(0, 3, 2, 1).reshape(n, C * taps, L), (H, W), k, d, p, s)
    assert bool(torch.isfinite(dx).all())
    assert rel_err(dx, want) < 1e-6


@pytest.mark.parametrize("shape", [(64, 32, 3, 3), (10, 64, 1, 4), (33, 96, 3, 2), (288, 32, 3, 3), (3, 4, 5, 5)])
def test_conv_weight_layout_round_trips_and_carries_the_stddev(shape):
    """bnn_conv2d_weight_layout writes mean, sigma and scale in (o, kh, kw, c) order, sigma bit-identical to bnn_stddev;
    bnn_conv2d_weight_unlayout brings all three back to OIHW unchanged."""
    g = torch.Generator(device="cuda").manual_seed(701)
    mu = torch.randn(shape, device="cuda", generator=g)
    rho = torch.randn(shape, device="cuda", generator=g) * 8 - 2      # scale in every softplus regime, some above 20
    rho.view(-1)[:3] = torch.tensor([25.0, -40.0, 20.0])
    sigma = _C.stddev(rho)
    wl = _C.conv_weight_layout(mu, rho)

    def ohwc(t):
        return t.permute(0, 2, 3, 1).reshape(-1)
    assert torch.equal(wl[0], ohwc(mu)) and torch.equal(wl[1], ohwc(sigma)) and torch.equal(wl[2], ohwc(rho))
    back = _C.conv_weight_unlayout(wl, shape)
    assert torch.equal(back[0], mu) and torch.equal(back[1], sigma) and torch.equal(back[2], rho)
