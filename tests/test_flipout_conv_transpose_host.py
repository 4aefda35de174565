"""FlipOutNormalConvTranspose1d / 2d / 3d without a GPU: constructor contract, validation shared with
NormalConvTranspose*, signs, output_size, the CPU composite against the formula and against fp64 autograd, and the C entry
points of the sign passes rejecting bad arguments."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from bayesianneuralnetworks_b200 import _C
import bayesianneuralnetworks_b200.nn as bnn_nn
from bayesianneuralnetworks_b200.nn import (BayesianConvNd, FlipOutNormalConvTranspose1d, FlipOutNormalConvTranspose2d,
                                            FlipOutNormalConvTranspose3d, FlipOutNormalConvTransposeNd,
                                            NormalConvTranspose1d, NormalConvTranspose2d, NormalConvTranspose3d,
                                            NormalConvTransposeNd)

_OPS = {1: F.conv_transpose1d, 2: F.conv_transpose2d, 3: F.conv_transpose3d}


def test_constructor_contract_and_attributes():
    layer = FlipOutNormalConvTranspose2d(16, 12, (3, 5), stride=(2, 1), padding=1, output_padding=(1, 0), groups=2,
                                         dilation=(1, 2))
    assert isinstance(layer, FlipOutNormalConvTransposeNd) and isinstance(layer, NormalConvTransposeNd)
    assert isinstance(layer, BayesianConvNd)
    assert layer.transposed is True and layer.bias is None
    assert layer._fused is False and layer._mc_composite is True
    assert tuple(layer.weight.mean.shape) == (16, 6, 3, 5) and tuple(layer.weight.scale.shape) == (16, 6, 3, 5)
    assert layer.stride == (2, 1) and layer.padding == (1, 1) and layer.output_padding == (1, 0)
    assert layer.dilation == (1, 2) and layer.groups == 2 and layer.kernel_size == (3, 5)
    assert layer.in_channels == 16 and layer.out_channels == 12
    one = FlipOutNormalConvTranspose1d(32, 64, 4, stride=2, padding=1)
    assert tuple(one.weight.mean.shape) == (32, 64, 4) and one.output_padding == (0,) and one.stride == (2,)
    three = FlipOutNormalConvTranspose3d(8, 4, (1, 4, 4), stride=(1, 2, 2), padding=(0, 1, 1))
    assert tuple(three.weight.mean.shape) == (8, 4, 1, 4, 4) and three.padding == (0, 1, 1)
    # the reference's init: scale ~ N(-2, 0.15), mean kaiming-uniform
    big = FlipOutNormalConvTranspose2d(64, 64, 3)
    assert abs(float(big.weight.scale.detach().mean()) + 2.0) < 0.02
    bound = 1 / (64 * 9) ** 0.5                  # kaiming_uniform(a = sqrt 5) of a [Cin, Cout, 3, 3] tensor
    assert float(big.weight.mean.detach().abs().max()) <= bound + 1e-7
    for name in ("FlipOutNormalConvTransposeNd", "FlipOutNormalConvTranspose1d", "FlipOutNormalConvTranspose2d",
                 "FlipOutNormalConvTranspose3d"):
        assert name in bnn_nn.__all__ and getattr(bnn_nn, name) is not None


def test_state_dict_keys():
    for layer in (FlipOutNormalConvTranspose1d(4, 6, 3), FlipOutNormalConvTranspose2d(4, 6, 3),
                  FlipOutNormalConvTranspose3d(4, 6, 3)):
        assert set(layer.state_dict()) == {"weight.mean", "weight.scale"}


@pytest.mark.parametrize("kw", [
    dict(stride=2, output_padding=2),
    dict(stride=1, output_padding=1),
    dict(stride=2, dilation=3, output_padding=3),
    dict(stride=(2, 1), output_padding=(0, 1)),
    dict(groups=4),
    dict(groups=3),
])
def test_validation_errors_match_normal_conv_transpose(kw):
    in_ch, out_ch = (6, 4) if kw.get("groups") == 4 else (6, 8) if kw.get("groups") == 3 else (4, 4)
    with pytest.raises(ValueError) as want:
        NormalConvTranspose2d(in_ch, out_ch, 3, **kw)
    with pytest.raises(ValueError) as got:
        FlipOutNormalConvTranspose2d(in_ch, out_ch, 3, **kw)
    assert str(got.value) == str(want.value)


def test_legal_output_padding_below_dilation_is_accepted():
    assert FlipOutNormalConvTranspose2d(4, 4, 3, stride=1, dilation=2, output_padding=1).output_padding == (1, 1)


def test_signs_shapes_and_draw_order():
    layer = FlipOutNormalConvTranspose2d(6, 4, 3, stride=2, groups=2)
    x = torch.randn(5, 6, 3, 3)
    torch.manual_seed(11)
    layer(x)
    R, S = layer.sampled
    assert tuple(R.shape) == (5, 4, 1, 1) and tuple(S.shape) == (5, 6, 1, 1)
    assert set(R.unique().tolist()) <= {-1.0, 1.0} and set(S.unique().tolist()) <= {-1.0, 1.0}
    torch.manual_seed(11)
    r = (torch.rand(5, 4, 1, 1) - .5).sign()                           # R first, then S
    s = (torch.rand(5, 6, 1, 1) - .5).sign()
    assert torch.equal(R, r) and torch.equal(S, s)
    layer.sample(3, (1, 1, 1))
    assert tuple(layer.R.shape) == (3, 4, 1, 1, 1) and tuple(layer.S.shape) == (3, 6, 1, 1, 1)
    one = FlipOutNormalConvTranspose1d(3, 5, 3)
    one(torch.randn(2, 3, 7))
    assert tuple(one.R.shape) == (2, 5, 1) and tuple(one.S.shape) == (2, 3, 1)


def test_sample_false_reuses_the_signs_and_checks_the_batch():
    layer = FlipOutNormalConvTranspose2d(3, 4, 3, stride=2)
    x = torch.randn(2, 3, 4, 4)
    y = layer(x)
    R, S = layer.sampled
    assert torch.equal(layer(x, sample=False), y)
    assert layer.R is R and layer.S is S
    with pytest.raises(RuntimeError, match=r"for this batch of 3 examples; the layer holds R \(2, 4, 1, 1\)"):
        layer(torch.randn(3, 3, 4, 4), sample=False)


def test_sample_false_before_any_forward_is_a_clear_error():
    layer = FlipOutNormalConvTranspose2d(3, 4, 3, stride=2)         # construction draws signs without spatial dims
    with pytest.raises(RuntimeError, match=r"must be R \(1, 4, 1, 1\) and S \(1, 3, 1, 1\)"):
        layer(torch.randn(1, 3, 4, 4), sample=False)
    del layer.R
    with pytest.raises(RuntimeError, match="the layer holds no signs"):
        layer(torch.randn(1, 3, 4, 4), sample=False)
    layer.sample(1, (1, 1))
    assert layer(torch.randn(1, 3, 4, 4), sample=False).shape == (1, 4, 9, 9)


def _geom2d(Cin, Cout, k, s, p, d, n_in):
    """The conv view of a transposed layer with a 1 x n_in input (the 1-d layers' form)."""
    n_out = (n_in - 1) * s - 2 * p + d * (k - 1) + 1
    return _C.conv_geom(1, 1, n_out, Cout, 1, n_in, Cin, 1, k, (1, s), (0, p), (1, d))


def test_one_predicate_decides_all_three_passes_without_a_gpu():
    """bnn_conv_transpose{2,3}d_supported: the forward's phase corners AND the gradients' conv-view corners.  With
    stride >= 2 the forward's corners are divided by the stride, so these layers pass the forward's own check but not
    the gradients' (conv-view corner -(k - 1) d < -128 or extent >= 256)."""
    assert _C.conv_transpose_supported(_geom2d(32, 32, 4, 2, 1, 1, 5))
    assert not _C.conv_transpose_supported(_geom2d(32, 32, 200, 2, 0, 1, 5))          # conv-view corner -199
    assert not _C.conv_transpose_supported(_geom2d(32, 32, 3, 2, 0, 65, 5))          # extent 130, corner -130
    assert not _C.conv_transpose_supported(_geom2d(32, 32, 3, 2, 130, 1, 200))       # padding beyond 128
    assert not _C.conv_transpose_supported(_geom2d(16, 32, 4, 2, 1, 1, 5))           # Cin % 32 != 0
    assert not _C.conv_transpose_supported(_geom2d(32, 3, 4, 2, 1, 1, 5))            # Cout % 32 != 0
    g3 = _C.conv3d_geom(1, 4, 4, 4, 32, 2, 2, 2, 32, (2, 2, 2), (2, 2, 2), (0, 0, 0), (1, 1, 1))
    assert _C.conv_transpose_supported(g3)
    g3 = _C.conv3d_geom(1, 34, 34, 34, 32, 2, 2, 2, 32, (3, 3, 3), (1, 1, 1), (1, 1, 1), (17, 17, 17))
    assert not _C.conv_transpose_supported(g3)                                       # extent 34 beyond rank-5 limits
    bad = _C.conv_geom(1, 1, 9, 32, 1, 5, 32, 1, 4, (1, 2), (0, 1), (1, 1))           # OW does not match the geometry
    with pytest.raises(_C.BnnError, match="do not match"):
        _C.conv_transpose_supported(bad)


@pytest.mark.parametrize("size", [(9, 9), (10, 10), (1, 2, 9, 10), (9, 10)])
def test_output_size_matches_torch(size):
    ref = torch.nn.ConvTranspose2d(3, 4, 3, stride=2, padding=1, bias=False)
    layer = FlipOutNormalConvTranspose2d(3, 4, 3, stride=2, padding=1)
    x = torch.randn(1, 3, 5, 5)
    y = layer(x, output_size=size)
    assert y.shape == ref(x, output_size=size).shape


@pytest.mark.parametrize("size", [(8, 8), (11, 11), (9,)])
def test_output_size_errors_match_torch(size):
    ref = torch.nn.ConvTranspose2d(3, 4, 3, stride=2, padding=1, bias=False)
    layer = FlipOutNormalConvTranspose2d(3, 4, 3, stride=2, padding=1)
    x = torch.randn(1, 3, 5, 5)
    with pytest.raises(ValueError) as want:
        ref(x, output_size=size)
    with pytest.raises(ValueError) as got:
        layer(x, output_size=size)
    assert str(got.value) == str(want.value)


_CASES = [
    (FlipOutNormalConvTranspose1d, dict(kernel_size=4, stride=2, padding=1), (3, 4, 7)),
    (FlipOutNormalConvTranspose2d, dict(kernel_size=3, stride=2, padding=1, output_padding=1), (3, 4, 5, 6)),
    (FlipOutNormalConvTranspose2d, dict(kernel_size=3, stride=1, dilation=2, output_padding=1, groups=2), (2, 4, 5, 5)),
    (FlipOutNormalConvTranspose3d, dict(kernel_size=(1, 4, 4), stride=(1, 2, 2), padding=(0, 1, 1)), (2, 4, 3, 4, 4)),
]


@pytest.mark.parametrize("cls,kw,shape", _CASES)
def test_cpu_forward_is_the_flipout_formula(cls, kw, shape):
    torch.manual_seed(0)
    layer = cls(shape[1], 6, **kw)
    x = torch.randn(*shape)
    y = layer(x)
    R, S = layer.sampled
    nd = x.dim() - 2
    args = (layer.stride, layer.padding, layer.output_padding, layer.groups, layer.dilation)
    mean, stddev = layer.weight.mean, layer.weight.stddev
    want = _OPS[nd](x, mean, None, *args) + _OPS[nd](x * S, stddev, None, *args) * R
    assert y.shape == want.shape and y.is_contiguous()
    torch.testing.assert_close(y, want, rtol=0, atol=0)


@pytest.mark.parametrize("cls,kw,shape", _CASES)
def test_cpu_backward_matches_fp64_autograd(cls, kw, shape):
    torch.manual_seed(1)
    layer = cls(shape[1], 6, **kw).double()
    x = torch.randn(*shape, dtype=torch.float64, requires_grad=True)
    y = layer(x)
    R, S = (t.double() for t in layer.sampled)
    g = torch.randn_like(y)
    (y * g).sum().backward()
    nd = x.dim() - 2
    args = (layer.stride, layer.padding, layer.output_padding, layer.groups, layer.dilation)
    x2 = x.detach().clone().requires_grad_()
    mean = layer.weight.mean.detach().clone().requires_grad_()
    scale = layer.weight.scale.detach().clone().requires_grad_()
    stddev = 1e-10 + F.softplus(scale)
    want = _OPS[nd](x2, mean, None, *args) + _OPS[nd](x2 * S, stddev, None, *args) * R
    (want * g).sum().backward()
    torch.testing.assert_close(x.grad, x2.grad, rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(layer.weight.mean.grad, mean.grad, rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(layer.weight.scale.grad, scale.grad, rtol=1e-12, atol=1e-12)


def test_sign_pass_symbols_are_exported():
    names = ("bnn_flipout_split", "bnn_flipout_combine", "bnn_conv_transpose2d_supported",
             "bnn_conv_transpose3d_supported")
    lib = _C.lib()
    for name in names:
        assert name in _C.EXPORTED_SYMBOLS and hasattr(lib, name)


def test_sign_passes_reject_bad_arguments_without_a_gpu():
    lib = _C.lib()
    bad = 1                                       # BNN_ERR_BAD_ARGUMENT, checked before any device query
    p = ctypes.c_void_p(16)                       # never dereferenced: the call returns before launching
    assert lib.bnn_flipout_split(None, 0, p, p, p, 1, 1, 1, None) == bad
    assert lib.bnn_flipout_split(p, 0, p, None, p, 1, 1, 1, None) == bad          # a_cl needed for an NCHW input
    assert lib.bnn_flipout_split(p, 1, None, None, p, 1, 1, 1, None) == bad
    assert lib.bnn_flipout_split(p, 0, p, p, p, -1, 1, 1, None) == bad
    assert lib.bnn_flipout_split(p, 0, p, p, p, 1, 0, 1, None) == bad
    assert lib.bnn_flipout_split(p, 0, p, p, p, 1, 1, -5, None) == bad
    assert lib.bnn_flipout_split(p, 0, p, p, p, 1 << 40, 1 << 20, 1 << 20, None) == bad   # n*C*P beyond 64 bits
    assert lib.bnn_flipout_combine(p, None, p, p, 0, 1, 1, 1, None) == bad
    assert lib.bnn_flipout_combine(p, p, p, None, 1, 1, 1, 1, None) == bad
    assert lib.bnn_flipout_combine(p, p, p, p, 0, 0, 1, 1, None) == bad
    assert lib.bnn_flipout_combine(p, p, p, p, 0, 1, -3, 1, None) == bad
    assert "bad shape" in lib.bnn_last_error_string().decode()
    with pytest.raises(RuntimeError, match="runs on CUDA"):
        _C.flipout_split(torch.zeros(2, 3, 4), torch.ones(2, 3))
    with pytest.raises(RuntimeError, match="runs on CUDA"):
        _C.flipout_combine(torch.zeros(2, 3, 4), torch.zeros(2, 3, 4), torch.ones(2, 3), channels_last=False)
