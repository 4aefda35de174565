"""NormalConvTranspose3d and `forward(output_size=...)` of the transposed layers without a GPU: constructor contract,
validation, state_dict, the CUDA-only error, output_size resolution against torch, and the host-side phase plan of the
3-d transposed-filter gather."""
import itertools

import pytest
import torch

from bayesianneuralnetworks_b200 import _C
from bayesianneuralnetworks_b200.nn import (BayesianConvNd, NormalConvNd, NormalConvTranspose1d, NormalConvTranspose2d,
                                            NormalConvTranspose3d, NormalConvTransposeNd)
import bayesianneuralnetworks_b200.nn as bnn_nn


def test_constructor_contract_and_attributes():
    layer = NormalConvTranspose3d(16, 12, (3, 5, 2), stride=(2, 1, 3), padding=1, output_padding=(1, 0, 2), groups=2,
                                  dilation=(1, 2, 1))
    assert isinstance(layer, NormalConvTransposeNd) and isinstance(layer, NormalConvNd) and isinstance(layer, BayesianConvNd)
    assert layer.transposed is True
    assert tuple(layer.weight.mean.shape) == (16, 6, 3, 5, 2) and tuple(layer.weight.scale.shape) == (16, 6, 3, 5, 2)
    assert tuple(layer.bias.mean.shape) == (12,)
    assert layer.stride == (2, 1, 3) and layer.padding == (1, 1, 1) and layer.output_padding == (1, 0, 2)
    assert layer.dilation == (1, 2, 1) and layer.groups == 2 and layer.kernel_size == (3, 5, 2)
    assert layer.in_channels == 16 and layer.out_channels == 12
    assert not layer._implicit and layer.weight._eps_layout is None        # groups > 1: storage-order eps
    up = NormalConvTranspose3d(128, 64, 2, stride=2, bias=False)
    assert tuple(up.weight.mean.shape) == (128, 64, 2, 2, 2) and up.bias is None and up.output_padding == (0, 0, 0)
    assert up._implicit and up.weight._eps_layout == (128, 64, 8)        # conv view: (o = Cin, taps, c = Cout)
    assert not NormalConvTranspose3d(64, 1, 2, stride=2)._implicit       # a 1-channel output
    big = NormalConvTranspose3d(32, 32, 3)
    assert abs(float(big.weight.scale.detach().mean()) + 2.0) < 0.02
    fan_in = 32 * 27                     # torch's fan-in of a [Cin, Cout, k, k, k] tensor: dim 1 x receptive field
    assert float(big.bias.mean.detach().abs().max()) <= 1 / fan_in ** 0.5 + 1e-7
    assert "NormalConvTranspose3d" in bnn_nn.__all__


@pytest.mark.parametrize("kw", [
    dict(stride=2, output_padding=2),
    dict(stride=1, output_padding=1),
    dict(stride=2, dilation=3, output_padding=3),
    dict(stride=(2, 1, 1), output_padding=(0, 1, 0)),
])
def test_output_padding_is_validated_at_construction(kw):
    with pytest.raises(ValueError, match="output_padding"):
        NormalConvTranspose3d(4, 4, 3, **kw)


def test_legal_output_padding_below_dilation_is_accepted():
    assert NormalConvTranspose3d(4, 4, 3, stride=1, dilation=2, output_padding=1).output_padding == (1, 1, 1)


def test_channel_counts_must_divide_groups():
    with pytest.raises(ValueError):
        NormalConvTranspose3d(6, 4, 3, groups=4)


def test_state_dict_keys():
    assert set(NormalConvTranspose3d(4, 6, 3).state_dict()) == {"weight.mean", "weight.scale", "bias.mean", "bias.scale"}
    assert set(NormalConvTranspose3d(4, 6, 3, bias=False).state_dict()) == {"weight.mean", "weight.scale"}


@pytest.mark.parametrize("cin,cout,groups", [(32, 32, 1), (4, 6, 1), (4, 6, 2)])
def test_cpu_input_raises_the_cuda_error(cin, cout, groups):
    layer = NormalConvTranspose3d(cin, cout, 3, stride=2, groups=groups)
    with pytest.raises(RuntimeError, match="runs on CUDA"):
        layer(torch.zeros(2, cin, 3, 3, 3))


# ---- output_size: torch's _ConvTransposeNd._output_padding is the reference -------------------------------------------
_TORCH = {1: torch.nn.ConvTranspose1d, 2: torch.nn.ConvTranspose2d, 3: torch.nn.ConvTranspose3d}
_OURS = {1: NormalConvTranspose1d, 2: NormalConvTranspose2d, 3: NormalConvTranspose3d}


def _resolve(mod, x, output_size):
    n = len(mod.kernel_size)
    return mod._output_padding(x, output_size, list(mod.stride), list(mod.padding), list(mod.kernel_size), n,
                               list(mod.dilation))


@pytest.mark.parametrize("n", [1, 2, 3])
def test_output_size_resolves_like_torch(n):
    cases = 0
    for k, s, p, d in itertools.product((1, 2, 3, 4), (1, 2, 3), (0, 1), (1, 2)):
        if p > (k - 1) * d // 2:
            continue
        kw = dict(stride=s, padding=p, dilation=d)
        ref, ours = _TORCH[n](2, 2, k, **kw), _OURS[n](2, 2, k, **kw)
        spatial = (3, 4, 5)[:n]
        x = torch.zeros((1, 2) + spatial)
        lo = [(i - 1) * s - 2 * p + d * (k - 1) + 1 for i in spatial]
        for extra in range(-1, s + 1):
            size = [m + extra for m in lo]
            for form in (size, [1, 2] + size, torch.Size(size)):
                try:
                    want = tuple(_resolve(ref, x, form))
                except ValueError as e:
                    with pytest.raises(ValueError) as got:
                        ours._output_padding(x, form)
                    assert str(got.value) == str(e)
                    continue
                assert ours._output_padding(x, form) == want
                cases += 1
    assert cases > 50


def test_output_size_of_wrong_length_raises_like_torch():
    ref, ours = torch.nn.ConvTranspose3d(2, 2, 3, stride=2), NormalConvTranspose3d(2, 2, 3, stride=2)
    x = torch.zeros(1, 2, 3, 3, 3)
    with pytest.raises(ValueError) as want:
        _resolve(ref, x, [7, 7])
    with pytest.raises(ValueError) as got:
        ours._output_padding(x, [7, 7])
    assert str(got.value) == str(want.value)


def test_output_size_none_keeps_the_layer_output_padding():
    layer = NormalConvTranspose2d(2, 2, 3, stride=2, output_padding=1)
    assert layer._output_padding(torch.zeros(1, 2, 4, 4), None) == (1, 1)


def test_output_size_is_the_third_forward_argument():
    """Appended after `sample`, so existing positional calls keep their meaning."""
    import inspect
    for cls in (NormalConvTranspose1d, NormalConvTranspose2d, NormalConvTranspose3d):
        assert list(inspect.signature(cls.forward).parameters) == ["self", "x", "sample", "output_size"]


# ---- the phase plan of bnn_sampled_conv_transpose3d_fwd -----------------------------------------------------------------
def _out(n, k, s, p, op, d):
    return (n - 1) * s - 2 * p + d * (k - 1) + op + 1


def _plan_triples(g, dims):
    """{(output voxel, tap, input voxel)} produced by the phases; asserts every phase row is one of torch's triples."""
    got = []
    for ph in _C.conv_transpose3d_phases(g):
        per_dim = []
        for a, (n_in, k, s, p, d) in zip("dhw", dims):
            r, rows, taps = ph[f"r_{a}"], ph[f"rows_{a}"], ph[f"taps_{a}"]
            items = []
            for i in range(rows):
                for j in range(taps):
                    kk = ph[f"last_{a}"] - j * ph[f"tap_step_{a}"]
                    ii = i + ph[f"first_{a}"] + j * ph[f"in_step_{a}"]
                    assert 0 <= kk < k and r + s * i == ii * s - p + kk * d
                    if 0 <= ii < n_in:
                        items.append((r + s * i, kk, ii))
            per_dim.append(items)
        for (od, kd, id_), (oh, kh, ih), (ow, kw, iw) in itertools.product(*per_dim):
            got.append(((od, oh, ow), (kd, kh, kw), (id_, ih, iw)))
    return got


def _want_triples(dims, outs):
    per_dim = []
    for (n_in, k, s, p, d), n_out in zip(dims, outs):
        per_dim.append([(o, kk, i) for i in range(n_in) for kk in range(k) for o in [i * s - p + kk * d] if 0 <= o < n_out])
    return {((a[0], b[0], c[0]), (a[1], b[1], c[1]), (a[2], b[2], c[2])) for a, b, c in itertools.product(*per_dim)}


def test_phase_plan_assigns_every_voxel_tap_pair_once():
    """bnn_debug_conv_transpose3d_phases (the plan the forward launches walk): over k 1-4, s 1-3, d 1-2, every padding and
    output_padding below the stride, isotropic and anisotropic, every (output voxel, tap, input voxel) triple of torch's
    conv_transpose3d definition (o = i s - p + k d per dimension) is produced by exactly one phase, and nothing else is;
    the phases cover every output voxel."""
    cases = 0
    iso = []
    for k, s, d in itertools.product(range(1, 5), range(1, 4), range(1, 3)):
        for p in range(0, (k - 1) * d // 2 + 1):
            for op in range(0, s):
                iso.append(((k, s, p, op, d),) * 3)
    aniso = [((1, 1, 0, 0, 1), (4, 2, 1, 0, 1), (4, 2, 1, 1, 1)), ((3, 1, 1, 0, 1), (4, 2, 1, 0, 1), (4, 2, 1, 0, 1)),
             ((2, 2, 0, 1, 1), (3, 3, 1, 2, 2), (1, 1, 0, 0, 1)), ((4, 3, 2, 1, 2), (2, 1, 0, 0, 1), (3, 2, 0, 1, 2)),
             ((2, 3, 0, 2, 1), (1, 2, 0, 0, 1), (4, 1, 3, 0, 2))]
    for spec in iso + aniso:
        for n_in in ((1, 3, 2), (3, 2, 4), (2, 4, 1)):
            dims = [(n, k, s, p, d) for n, (k, s, p, op, d) in zip(n_in, spec)]
            outs = [_out(n, k, s, p, op, d) for n, (k, s, p, op, d) in zip(n_in, spec)]
            if min(outs) <= 0:
                continue
            (kd, sd, pd, _, dd), (kh, sh, ph, _, dh), (kw, sw, pw, _, dw) = spec
            g = _C.conv3d_geom(1, *outs, 32, *n_in, 32, (kd, kh, kw), (sd, sh, sw), (pd, ph, pw), (dd, dh, dw))
            phases = _C.conv_transpose3d_phases(g)
            assert len(phases) == min(sd, outs[0]) * min(sh, outs[1]) * min(sw, outs[2])
            covered = set()
            for ph in phases:
                covered.update(itertools.product(*[range(ph[f"r_{a}"], n, s) for a, n, s in
                                                   zip("dhw", outs, (sd, sh, sw))]))
            assert covered == set(itertools.product(*[range(n) for n in outs]))
            got = _plan_triples(g, dims)
            assert len(got) == len(set(got)) and set(got) == _want_triples(dims, outs), (spec, n_in)
            cases += 1
    assert cases > 300


def test_phase_plan_rejects_a_geometry_that_does_not_match():
    g = _C.conv3d_geom(1, 8, 8, 8, 32, 5, 4, 4, 32, (2, 2, 2), (2, 2, 2), (0, 0, 0), (1, 1, 1))   # input depth 4, not 5
    with pytest.raises(_C.BnnError):
        _C.conv_transpose3d_phases(g)
