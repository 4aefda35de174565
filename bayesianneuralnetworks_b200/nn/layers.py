"""Bayesian Linear / Conv layers (mirror of pytorch_bayesian/nn/dense.py:9-60 and conv.py:9-142).

Constructor signatures, attributes (`weight`, `bias`, `sampled`, `sample()`, priors, conv geometry)
and `forward(x, sample=True)` follow the reference; the arithmetic runs in libbnn_b200.so:
NormalLinear, NormalConv1d/2d and NormalConvTranspose1d/2d/3d call the fused sample-and-contract kernels (no sampled
weight in memory), NormalConv3d contracts materialised samples with torch's conv3d.
"""
import math

import torch
from torch.distributions.normal import Normal
from torch.nn import init

from .. import _C, runtime
from ..functional import (ConvTranspose3dRefused, CudnnConvTranspose, SampledConv2d, SampledConv2dImplicit,
                          SampledConvTranspose2d, SampledConvTranspose2dImplicit, SampledConvTranspose3dImplicit,
                          SampledLinear, conv_implicit_eligible, conv_output_nchw)
from ..utils.traversal import _pair, _single, _triple
from .container import BayesianModule
from .variational import WeightNormal


def _init_normal_posterior(layer):
    """dense.py:34-44 / conv.py:53-63: mean ~ kaiming_uniform(a=sqrt 5), scale ~ N(-2, 0.15);
    bias mean ~ U(+-1/sqrt(fan_in)), bias scale ~ N(-2, 0.15); then a fresh draw."""
    init.kaiming_uniform_(layer.weight.mean, a=math.sqrt(5))
    init.normal_(layer.weight.scale, -2.0, 0.15)
    if layer.bias is not None:
        fan_in, _ = init._calculate_fan_in_and_fan_out(layer.weight.mean)
        bound = 1 / math.sqrt(fan_in)
        init.uniform_(layer.bias.mean, -bound, bound)
        init.normal_(layer.bias.scale, -2.0, 0.15)
    layer.sample()


class _FusedBayesianLayer:
    """Mixin of the layers whose forward is one fused launch over all Monte-Carlo samples."""
    _fused = True         # subclasses evaluated by torch ops (Flipout) switch this off

    def _mc_shape(self, x):
        """(S, shared, sample offset, draws to reserve) for this call from the MC context."""
        ctx = runtime.current_mc()
        if ctx is None:
            return 1, True, 0, 1, None
        if not ctx.expanded:
            if x.shape[0] != ctx.rows:
                raise RuntimeError("batched Monte-Carlo forward: the first Bayesian layer must see the network "
                                   f"input rows ({ctx.rows}), got {x.shape[0]}")
            return ctx.samples, True, ctx.sample_offset, ctx.total_samples, ctx
        return ctx.samples, False, ctx.sample_offset, ctx.total_samples, ctx

    def _draws(self, sample, S, offset, total):
        """DrawSpecs of weight and bias for this forward; `sample=False` reuses the previous draw
        (dense.py:56-60)."""
        if sample:
            wb = self.weight.advance(S, offset, total)          # W first, then b (dense.py:47,51)
            bb = self.bias.advance(S, offset, total) if self.bias is not None else None
        else:
            wb, wc = self.weight._last
            if wc != S:
                raise RuntimeError(f"forward(sample=False) reuses the previous draw of {wc} MC samples, "
                                   f"but this call evaluates {S}")
            bb = self.bias._last[0] if self.bias is not None else None
        spec_w = self.weight.draw_spec(wb, S)
        spec_b = self.bias.draw_spec(bb, S) if self.bias is not None else None
        return spec_w, spec_b

    def sample(self):
        """dense.py:46-54 / conv.py:65-73."""
        self.weight.sample()
        if self.bias is not None:
            self.bias.sample()

    @property
    def sampled(self):
        """(W, b | None) of the most recent draw — a 2-tuple as in the reference."""
        return (self.weight.sampled, self.bias.sampled if self.bias is not None else None)


# ------------------------------------------------------------------------------------------------ dense
class BayesianLinear(BayesianModule):
    """dense.py:9-24."""

    def __init__(self, in_features, out_features, bias, weight, prior, bias_prior=None):
        super(BayesianLinear, self).__init__(in_features, out_features, prior, bias_prior)
        self.weight = weight(out_features, in_features)
        if bias:
            self.bias = weight(out_features)
        else:
            self.register_parameter('bias', None)
        self.reset_parameters()

    def reset_parameters(self):
        pass


class NormalLinear(_FusedBayesianLayer, BayesianLinear):
    """dense.py:27-60."""

    def __init__(self, in_features, out_features, bias=True, prior=Normal(0, .1)):
        super(NormalLinear, self).__init__(in_features, out_features, bias, WeightNormal, prior)

    def reset_parameters(self):
        _init_normal_posterior(self)

    def forward(self, x, sample=True):
        S, shared, offset, total, ctx = self._mc_shape(x)
        spec_w, spec_b = self._draws(sample, S, offset, total)
        lead = x.shape[:-1]
        x2 = x.reshape(-1, x.shape[-1])
        y = SampledLinear.apply(x2, self.weight.mean, self.weight.scale,
                                self.bias.mean if self.bias is not None else None,
                                self.bias.scale if self.bias is not None else None,
                                S, shared, spec_w, spec_b, runtime.precision())
        if ctx is not None:
            ctx.expanded = True
        if shared and S > 1:
            return y.view((S * lead[0],) + tuple(lead[1:]) + (y.shape[-1],))
        return y.view(tuple(lead) + (y.shape[-1],))


# ------------------------------------------------------------------------------------------------ conv
class BayesianConvNd(BayesianModule):
    """conv.py:9-40."""

    def __init__(self, in_channels, out_channels, kernel_size, stride, padding, dilation, transposed, groups,
                 bias, weight, prior, bias_prior=None):
        super(BayesianConvNd, self).__init__(in_channels, out_channels, prior, bias_prior)
        if in_channels % groups != 0:
            raise ValueError('in_channels must be divisible by groups')
        if out_channels % groups != 0:
            raise ValueError('out_channels must be divisible by groups')
        self.kernel_size = kernel_size
        self.stride = stride
        self.padding = padding
        self.dilation = dilation
        self.transposed = transposed
        self.groups = groups
        if transposed:
            self.weight = weight(in_channels, out_channels // groups, *kernel_size)
        else:
            self.weight = weight(out_channels, in_channels // groups, *kernel_size)
        if bias:
            self.bias = weight(out_channels)
        else:
            self.register_parameter('bias', None)
        self.reset_parameters()

    def reset_parameters(self):
        pass


class NormalConvNd(BayesianConvNd):
    """conv.py:43-73."""

    def __init__(self, in_channels, out_channels, kernel_size, stride, padding, dilation, transposed, groups,
                 bias, prior):
        kernel_size = _single(kernel_size)
        super(NormalConvNd, self).__init__(in_channels, out_channels, kernel_size, stride, padding, dilation,
                                           transposed, groups, bias, WeightNormal, prior)

    def reset_parameters(self):
        _init_normal_posterior(self)

    def sample(self):
        self.weight.sample()
        if self.bias is not None:
            self.bias.sample()

    @property
    def sampled(self):
        return (self.weight.sampled, self.bias.sampled if self.bias is not None else None)


def _mark_implicit(layer):
    """Layers with groups == 1 and in_channels % 32 == 0 run the implicit-GEMM path; their weight's eps stream is keyed in
    (o, kh, kw, c) order (variational.WeightNormal._eps_layout).  A transposed layer is judged by its conv view (the
    convolution from its output back to its input, whose in_channels are the layer's out_channels)."""
    w = layer.weight.mean
    layer._implicit = conv_implicit_eligible(layer.out_channels if layer.transposed else layer.in_channels, layer.groups)
    if layer._implicit:
        layer.weight._eps_layout = (w.shape[0], w.shape[1], w.numel() // (w.shape[0] * w.shape[1]))


def _sampled_conv2d(layer, x, w_shape, S, shared, spec_w, spec_b, stride, padding, dilation):
    bias = layer.bias
    mean, scale = layer.weight.mean.view(w_shape), layer.weight.scale.view(w_shape)
    if layer._implicit:
        return SampledConv2dImplicit.apply(x, mean, scale, bias.mean if bias is not None else None,
                                           bias.scale if bias is not None else None, S, shared, spec_w, spec_b,
                                           runtime.precision(), stride, padding, dilation)
    return SampledConv2d.apply(x, mean, scale, bias.mean if bias is not None else None,
                               bias.scale if bias is not None else None, S, shared, spec_w, spec_b, runtime.precision(),
                               stride, padding, dilation, layer.groups)


class NormalConv2d(_FusedBayesianLayer, NormalConvNd):
    """conv.py:99-119."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1,
                 bias=True, prior=Normal(0, .1)):
        super(NormalConv2d, self).__init__(in_channels, out_channels, _pair(kernel_size), _pair(stride),
                                           _pair(padding), _pair(dilation), False, groups, bias, prior)
        _mark_implicit(self)

    def forward(self, x, sample=True):
        S, shared, offset, total, ctx = self._mc_shape(x)
        spec_w, spec_b = self._draws(sample, S, offset, total)
        y = _sampled_conv2d(self, x, tuple(self.weight.mean.shape), S, shared, spec_w, spec_b, tuple(self.stride),
                            tuple(self.padding), tuple(self.dilation))
        if ctx is not None:
            ctx.expanded = True
        return y


class NormalConv1d(_FusedBayesianLayer, NormalConvNd):
    """conv.py:76-96 — evaluated as a 2-d convolution with a height of one."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1,
                 bias=True, prior=Normal(0, .1)):
        super(NormalConv1d, self).__init__(in_channels, out_channels, _single(kernel_size), _single(stride),
                                           _single(padding), _single(dilation), False, groups, bias, prior)
        _mark_implicit(self)

    def forward(self, x, sample=True):
        S, shared, offset, total, ctx = self._mc_shape(x)
        spec_w, spec_b = self._draws(sample, S, offset, total)
        w_shape = (self.weight.mean.shape[0], self.weight.mean.shape[1], 1, self.weight.mean.shape[2])
        y = _sampled_conv2d(self, x.unsqueeze(2), w_shape, S, shared, spec_w, spec_b, (1, tuple(self.stride)[0]),
                            (0, tuple(self.padding)[0]), (1, tuple(self.dilation)[0]))
        if ctx is not None:
            ctx.expanded = True
        return y.squeeze(2)


class NormalConvTransposeNd(NormalConvNd):
    """Bayesian transposed convolution: weight [in_channels, out_channels // groups, *kernel_size] as the reference's
    BayesianConvNd(transposed=True) stores it (conv.py:26-28), plus `output_padding`.  The reference never wrote its forward;
    this one computes F.conv_transposeNd(x, W_s, b_s, stride, padding, output_padding, groups, dilation) for all
    Monte-Carlo samples in one fused call."""

    def __init__(self, in_channels, out_channels, kernel_size, stride, padding, output_padding, groups, bias, dilation,
                 prior):
        super(NormalConvTransposeNd, self).__init__(in_channels, out_channels, kernel_size, stride, padding, dilation,
                                                    True, groups, bias, prior)
        for op, s, d in zip(output_padding, self.stride, self.dilation):
            if not 0 <= op < max(s, d):
                raise ValueError(f"output_padding {tuple(output_padding)} must be smaller than either stride "
                                 f"{tuple(self.stride)} or dilation {tuple(self.dilation)} in every dimension")
        self.output_padding = output_padding
        _mark_implicit(self)

    def _output_padding(self, x, output_size):
        """output_padding of this call: the layer's own, or the one that gives `output_size` (torch's
        _ConvTransposeNd._output_padding: the same accepted sizes, [min, min + stride - 1] per dimension, and errors)."""
        if output_size is None:
            return tuple(self.output_padding)
        n = len(self.kernel_size)
        non_spatial = 2 if x.dim() == n + 2 else 1
        if len(output_size) == non_spatial + n:
            output_size = output_size[non_spatial:]
        if len(output_size) != n:
            raise ValueError(f"ConvTranspose{n}D: for {x.dim()}D input, output_size must have {n} or {non_spatial + n} "
                             f"elements (got {len(output_size)})")
        min_sizes = [(x.size(d + non_spatial) - 1) * self.stride[d] - 2 * self.padding[d] +
                     self.dilation[d] * (self.kernel_size[d] - 1) + 1 for d in range(n)]
        max_sizes = [m + s - 1 for m, s in zip(min_sizes, self.stride)]
        for size, lo, hi in zip(output_size, min_sizes, max_sizes):
            if size < lo or size > hi:
                raise ValueError(f"requested an output size of {output_size}, but valid sizes range from {min_sizes} "
                                 f"to {max_sizes} (for an input of {x.size()[2:]})")
        return tuple(size - lo for size, lo in zip(output_size, min_sizes))

    def _conv_transpose2d(self, x, w_shape, S, shared, spec_w, spec_b, stride, padding, output_padding, dilation):
        # output_padding >= stride (possible when dilation > stride): the rows beyond the conv view are reached by
        # appending zero input rows, which leaves output_padding % stride
        extra = [op // s for op, s in zip(output_padding, stride)]
        if any(extra):
            x = torch.nn.functional.pad(x, (0, extra[1], 0, extra[0]))
            output_padding = tuple(op % s for op, s in zip(output_padding, stride))
        bias = self.bias
        mean, scale = self.weight.mean.view(w_shape), self.weight.scale.view(w_shape)
        args = (x, mean, scale, bias.mean if bias is not None else None, bias.scale if bias is not None else None, S,
                shared, spec_w, spec_b, runtime.precision(), stride, padding, output_padding, dilation)
        if self._implicit:
            return SampledConvTranspose2dImplicit.apply(*args)
        return SampledConvTranspose2d.apply(*args, self.groups)


class NormalConvTranspose2d(_FusedBayesianLayer, NormalConvTransposeNd):
    """torch.nn.ConvTranspose2d's constructor order with a Normal variational posterior on weight and bias."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, output_padding=0, groups=1,
                 bias=True, dilation=1, prior=Normal(0, .1)):
        super(NormalConvTranspose2d, self).__init__(in_channels, out_channels, _pair(kernel_size), _pair(stride),
                                                    _pair(padding), _pair(output_padding), groups, bias,
                                                    _pair(dilation), prior)

    def forward(self, x, sample=True, output_size=None):
        output_padding = self._output_padding(x, output_size)
        S, shared, offset, total, ctx = self._mc_shape(x)
        spec_w, spec_b = self._draws(sample, S, offset, total)
        y = self._conv_transpose2d(x, tuple(self.weight.mean.shape), S, shared, spec_w, spec_b, tuple(self.stride),
                                   tuple(self.padding), output_padding, tuple(self.dilation))
        if ctx is not None:
            ctx.expanded = True
        return y


class NormalConvTranspose1d(_FusedBayesianLayer, NormalConvTransposeNd):
    """torch.nn.ConvTranspose1d's constructor order — evaluated as a 2-d transposed convolution with a height of one."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, output_padding=0, groups=1,
                 bias=True, dilation=1, prior=Normal(0, .1)):
        super(NormalConvTranspose1d, self).__init__(in_channels, out_channels, _single(kernel_size), _single(stride),
                                                    _single(padding), _single(output_padding), groups, bias,
                                                    _single(dilation), prior)

    def forward(self, x, sample=True, output_size=None):
        output_padding = self._output_padding(x, output_size)
        S, shared, offset, total, ctx = self._mc_shape(x)
        spec_w, spec_b = self._draws(sample, S, offset, total)
        w = self.weight.mean.shape
        y = self._conv_transpose2d(x.unsqueeze(2), (w[0], w[1], 1, w[2]), S, shared, spec_w, spec_b,
                                   (1, tuple(self.stride)[0]), (0, tuple(self.padding)[0]),
                                   (0, output_padding[0]), (1, tuple(self.dilation)[0]))
        if ctx is not None:
            ctx.expanded = True
        return y.squeeze(2)


class NormalConvTranspose3d(_FusedBayesianLayer, NormalConvTransposeNd):
    """torch.nn.ConvTranspose3d's constructor order with a Normal variational posterior on weight and bias — the
    upsampling layer of Bayesian volumetric decoders (3-D U-Nets, V-Nets).  CUDA, TF32, groups == 1 with in_ and
    out_channels multiples of 32 and a geometry within the rank-5 im2col descriptor's limits: the 3-d implicit-GEMM kernels
    (SampledConvTranspose3dImplicit, all Monte-Carlo samples in one call per output phase).  Everything else — fp32 mode,
    other channel counts (e.g. a 1-channel output), groups > 1, geometry outside those limits — contracts the S
    materialised draws (the same draws: WeightNormal.materialize applies the layer's eps order) with one
    F.conv_transpose3d per sample, with cuDNN's TF32 off in fp32 mode."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, output_padding=0, groups=1,
                 bias=True, dilation=1, prior=Normal(0, .1)):
        super(NormalConvTranspose3d, self).__init__(in_channels, out_channels, _triple(kernel_size), _triple(stride),
                                                    _triple(padding), _triple(output_padding), groups, bias,
                                                    _triple(dilation), prior)

    def _materialized(self, x, S, shared, spec_w, spec_b, stride, padding, output_padding, dilation):
        """The reference's form: W_s (autograd-tracked) and one cuDNN transposed convolution per sample."""
        def begin(spec):
            return (spec.step << 32) | spec.sample_begin
        # contiguous: the draws of a layer with the (o, kd, kh, kw, c) eps order come back as a strided view
        w = self.weight.materialize(begin(spec_w), S).contiguous()
        b = self.bias.materialize(begin(spec_b), S) if self.bias is not None else None
        xs = x if shared else x.reshape((S, x.shape[0] // S) + tuple(x.shape[1:]))
        tf32 = runtime.precision() == _C.PREC_TF32
        y = torch.cat([CudnnConvTranspose.apply(x if shared else xs[s], w[s], b[s] if b is not None else None, stride,
                                                  padding, output_padding, self.groups, dilation, tf32)
                       for s in range(S)], 0)
        return y.contiguous() if conv_output_nchw(x) else y

    def _conv_transpose3d(self, x, S, shared, spec_w, spec_b, output_padding):
        stride, padding, dilation = tuple(self.stride), tuple(self.padding), tuple(self.dilation)
        if self._implicit and runtime.precision() == _C.PREC_TF32:
            # output_padding >= stride (dilation > stride): zero input rows appended, as in _conv_transpose2d
            extra = [op // s for op, s in zip(output_padding, stride)]
            xi, opi = x, output_padding
            if any(extra):
                xi = torch.nn.functional.pad(x, (0, extra[2], 0, extra[1], 0, extra[0]))
                opi = tuple(op % s for op, s in zip(output_padding, stride))
            bias = self.bias
            try:
                return SampledConvTranspose3dImplicit.apply(xi, self.weight.mean, self.weight.scale,
                                                            bias.mean if bias is not None else None,
                                                            bias.scale if bias is not None else None, S, shared, spec_w,
                                                            spec_b, stride, padding, opi, dilation)
            except ConvTranspose3dRefused:
                pass
        return self._materialized(x, S, shared, spec_w, spec_b, stride, padding, output_padding, dilation)

    def forward(self, x, sample=True, output_size=None):
        output_padding = self._output_padding(x, output_size)
        S, shared, offset, total, ctx = self._mc_shape(x)
        spec_w, spec_b = self._draws(sample, S, offset, total)
        y = self._conv_transpose3d(x, S, shared, spec_w, spec_b, output_padding)
        if ctx is not None:
            ctx.expanded = True
        return y


_UNFOLD_LIMIT_BYTES = 1 << 30      # NormalConv3d: largest lowered activation matrix the fused path builds


class NormalConv3d(_FusedBayesianLayer, NormalConvNd):
    """conv.py:122-142.  CUDA, groups == 1: the input is lowered by torch (pad + three `unfold`s: a differentiable
    strided view, one copy into a `[B·OD·OH·OW, C·kd·kh·kw]` matrix whose column order IS the weight's memory order) and
    contracted by the sample-and-contract kernels (`SampledLinear`: all S Monte-Carlo samples in one launch, the sampled
    weights never materialised, eps regenerated in the backward pass); autograd carries the input gradient back through
    the lowering.  Grouped layers, CPU tensors and lowered matrices above 1 GiB keep the reference's form: the sampled
    weights are materialised by the library (autograd-tracked) and contracted by torch's conv3d, one sample per call."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1,
                 bias=True, prior=Normal(0, .1)):
        super(NormalConv3d, self).__init__(in_channels, out_channels, _triple(kernel_size), _triple(stride),
                                           _triple(padding), _triple(dilation), False, groups, bias, prior)
        self._fused = groups == 1

    def _lowered_bytes(self, x):
        k, s, p, d = (tuple(self.kernel_size), tuple(self.stride), tuple(self.padding), tuple(self.dilation))
        out = [(x.shape[2 + i] + 2 * p[i] - d[i] * (k[i] - 1) - 1) // s[i] + 1 for i in range(3)]
        return 4 * x.shape[0] * max(out[0], 0) * max(out[1], 0) * max(out[2], 0) * x.shape[1] * k[0] * k[1] * k[2]

    def forward(self, x, sample=True):
        fused = (self._fused and x.is_cuda and x.dim() == 5 and x.dtype == torch.float32
                 and self._lowered_bytes(x) <= _UNFOLD_LIMIT_BYTES)
        if not fused:
            if runtime.current_mc() is not None:
                raise RuntimeError("NormalConv3d: this call does not qualify for the batched Monte-Carlo forward")
            if sample:
                self.sample()
            return torch.nn.functional.conv3d(x, *self.sampled, self.stride, self.padding, self.dilation, self.groups)
        S, shared, offset, total, ctx = self._mc_shape(x)
        spec_w, spec_b = self._draws(sample, S, offset, total)
        k, s, p, d = (tuple(self.kernel_size), tuple(self.stride), tuple(self.padding), tuple(self.dilation))
        cols = torch.nn.functional.pad(x, (p[2], p[2], p[1], p[1], p[0], p[0])) if any(p) else x
        for i in range(3):                 # [rows, C, OD, OH, OW, kd, kh, kw]: window axes are appended in order
            cols = cols.unfold(2 + i, (k[i] - 1) * d[i] + 1, s[i])
            if d[i] > 1:
                cols = cols[..., ::d[i]]
        rows, C, OD, OH, OW = cols.shape[:5]
        col = cols.permute(0, 2, 3, 4, 1, 5, 6, 7).reshape(rows * OD * OH * OW, C * k[0] * k[1] * k[2])
        O = self.weight.mean.shape[0]
        y = SampledLinear.apply(col, self.weight.mean.view(O, -1), self.weight.scale.view(O, -1),
                                self.bias.mean if self.bias is not None else None,
                                self.bias.scale if self.bias is not None else None,
                                S, shared, spec_w, spec_b, runtime.precision())
        if ctx is not None:
            ctx.expanded = True
        return y.view(-1, OD, OH, OW, O).permute(0, 4, 1, 2, 3).contiguous()
