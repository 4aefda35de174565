"""NormalConvTranspose1d / 2d without a GPU: constructor contract, validation, state_dict, the CUDA-only error and the
host-side phase plan of the strided transposed-filter gather."""
import itertools

import pytest
import torch

from bayesianneuralnetworks_b200 import _C
from bayesianneuralnetworks_b200.nn import (BayesianConvNd, NormalConvNd, NormalConvTranspose1d, NormalConvTranspose2d,
                                            NormalConvTransposeNd)
import bayesianneuralnetworks_b200.nn as bnn_nn


def test_constructor_contract_and_attributes():
    layer = NormalConvTranspose2d(16, 12, (3, 5), stride=(2, 1), padding=1, output_padding=(1, 0), groups=2,
                                  dilation=(1, 2))
    assert isinstance(layer, NormalConvTransposeNd) and isinstance(layer, NormalConvNd) and isinstance(layer, BayesianConvNd)
    assert layer.transposed is True
    assert tuple(layer.weight.mean.shape) == (16, 6, 3, 5) and tuple(layer.weight.scale.shape) == (16, 6, 3, 5)
    assert tuple(layer.bias.mean.shape) == (12,)
    assert layer.stride == (2, 1) and layer.padding == (1, 1) and layer.output_padding == (1, 0)
    assert layer.dilation == (1, 2) and layer.groups == 2 and layer.kernel_size == (3, 5)
    assert layer.in_channels == 16 and layer.out_channels == 12
    assert not layer._implicit                                    # groups > 1: NCHW lowering, storage-order eps
    one = NormalConvTranspose1d(32, 64, 4, stride=2, padding=1, bias=False)
    assert tuple(one.weight.mean.shape) == (32, 64, 4) and one.bias is None and one.output_padding == (0,)
    assert one._implicit and one.weight._eps_layout == (32, 64, 4)      # conv view: in_channels = 64
    assert not NormalConvTranspose2d(64, 3, 4)._implicit             # a 3-channel output
    # the reference's init: scale ~ N(-2, 0.15), bias mean within 1 / sqrt(fan_in)
    big = NormalConvTranspose2d(64, 64, 3)
    assert abs(float(big.weight.scale.detach().mean()) + 2.0) < 0.02
    fan_in = 64 * 9                      # torch's fan-in of a [Cin, Cout, k, k] tensor: dim 1 x receptive field
    assert float(big.bias.mean.detach().abs().max()) <= 1 / fan_in ** 0.5 + 1e-7
    for name in ("NormalConvTransposeNd", "NormalConvTranspose1d", "NormalConvTranspose2d"):
        assert name in bnn_nn.__all__


@pytest.mark.parametrize("kw", [
    dict(stride=2, output_padding=2),
    dict(stride=1, output_padding=1),
    dict(stride=2, dilation=3, output_padding=3),
    dict(stride=(2, 1), output_padding=(0, 1)),
])
def test_output_padding_is_validated_at_construction(kw):
    with pytest.raises(ValueError, match="output_padding"):
        NormalConvTranspose2d(4, 4, 3, **kw)


def test_legal_output_padding_below_dilation_is_accepted():
    layer = NormalConvTranspose2d(4, 4, 3, stride=1, dilation=2, output_padding=1)
    assert layer.output_padding == (1, 1)


def test_channel_counts_must_divide_groups():
    with pytest.raises(ValueError):
        NormalConvTranspose2d(6, 4, 3, groups=4)


def test_state_dict_keys():
    assert set(NormalConvTranspose2d(4, 6, 3).state_dict()) == {"weight.mean", "weight.scale", "bias.mean", "bias.scale"}
    assert set(NormalConvTranspose1d(4, 6, 3, bias=False).state_dict()) == {"weight.mean", "weight.scale"}


def test_cpu_input_raises_the_cuda_error():
    layer = NormalConvTranspose2d(4, 6, 3, stride=2)
    with pytest.raises(RuntimeError, match="runs on CUDA"):
        layer(torch.zeros(2, 4, 5, 5))


def _out(n, k, s, p, op, d):
    return (n - 1) * s - 2 * p + d * (k - 1) + op + 1


def test_phase_plan_assigns_every_pixel_tap_pair_once():
    """bnn_debug_conv_transpose_phases (the plan the forward launches walk): over a sweep of kernel, stride, dilation,
    padding and output_padding, every (output row, tap, input row) triple of torch's conv_transpose definition
    (oh = ih * s - p + kh * d) is produced by exactly one phase, and nothing else is."""
    cases = 0
    for k, s, d in itertools.product(range(1, 6), range(1, 5), range(1, 3)):
        for p in range(0, (k - 1) * d // 2 + 1):
            for op in range(0, max(s, d)):
                if op >= s:
                    continue         # the layer folds output_padding >= stride into extra input rows first
                for n_in in (1, 3, 4):
                    n_out = _out(n_in, k, s, p, op, d)
                    if n_out <= 0:
                        continue
                    g = _C.conv_geom(1, n_out, n_out, 4, n_in, n_in, 32, k, k, (s, s), (p, p), (d, d))
                    phases = _C.conv_transpose_phases(g)
                    assert len(phases) == min(s, n_out) ** 2
                    want = {(oh, kh, ih) for ih in range(n_in) for kh in range(k)
                            for oh in [ih * s - p + kh * d] if 0 <= oh < n_out}
                    got = []
                    rows_seen = set()
                    for ph in phases:
                        if ph["rw"] != 0:
                            continue             # the plan is separable: one column of phases covers the rows
                        r, rows, taps = ph["rh"], ph["rows_h"], ph["taps_h"]
                        assert rows == len(range(r, n_out, s))
                        rows_seen.update(range(r, n_out, s))
                        for i in range(rows):
                            for j in range(taps):
                                kh = ph["last_h"] - j * ph["tap_step_h"]
                                ih = i + ph["first_h"] + j * ph["in_step_h"]
                                assert 0 <= kh < k
                                assert r + s * i == ih * s - p + kh * d
                                if 0 <= ih < n_in:
                                    got.append((r + s * i, kh, ih))
                    assert rows_seen == set(range(n_out))
                    assert len(got) == len(set(got)) and set(got) == want, (k, s, d, p, op, n_in)
                    cases += 1
    assert cases > 300
