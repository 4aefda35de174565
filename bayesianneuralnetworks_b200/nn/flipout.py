"""Flipout layers (Wen et al. 2018) — SURVEY §8(f) rank 1: `FlipoutNormalLinear` (pytorch_bayesian/nn/dense.py:63-83)
and `FlipOutNormalConvNd/1d/2d/3d` (conv.py:145-251).

The perturbation is sigma itself with random sign flips,
    y = op(x, mean) + op(x * S, stddev) * R,        R, S in {-1, +1}.
Reference quirks kept: no bias; the Linear signs are per feature and shared by the whole batch (dense.py:71-75), the conv
signs are per example (conv.py:154-161).

* FlipoutNormalLinear (CUDA): because R and S are shared by the batch,  (x * S) sigma^T * R = x (sigma o (R S^T))^T, so the
  layer IS a sampled contraction  y = x (mean + sigma o eps)^T  with the rank-one sign noise eps = R S^T: ONE launch of the
  sample-and-contract kernels (bnn_rng.row_sign / col_sign: the generator warps read the two sign vectors instead of
  drawing Philox normals), where the reference runs two GEMMs and two elementwise passes; the backward kernels form
  d mean and d scale with the same eps.  R / S are still drawn by torch and kept as attributes (`sampled`).
* The conv layers' signs differ per example, which makes the perturbed filter example specific: there is no common
  sampled weight, the layer really is TWO convolutions with unsampled weights, conv(x, mean) + conv(x * S, stddev) * R.
  FlipOutNormalConv1d / 2d (CUDA, groups == 1, in_channels % 32 == 0) run both through the library's implicit-GEMM
  contraction kernels (the sample-and-contract kernels with injected eps = 0, i.e. W = the given tensor; TMA im2col
  operand, tcgen05 MMAs; forward, input gradient and weight gradients), with the sign products and d stddev / d scale
  left to torch element-wise ops; everything else (3-d, grouped, odd channel counts, CPU tensors) evaluates the
  reference's composite with torch's convolutions.
* FlipOutNormalConvTranspose1d / 2d / 3d: the transposed form the reference prepared (`transposed=True`) but never built,
  on the transposed-convolution kernels, with the sign products and layout changes in two bandwidth kernels
  (bnn_flipout_split / bnn_flipout_combine, functional.FlipoutConvTransposeImplicit).
Their variational tensor is a WeightNormal, hence KLDivergence and PruneNormal treat them like every other Bayesian layer
(the fused KL / prune kernels).
"""
import torch
import torch.nn.functional as F
from torch.distributions.normal import Normal

from .. import _C, runtime
from ..functional import (CudnnConvTranspose, FlipoutContractionRefused, FlipoutConvTransposeImplicit,
                          conv_implicit_eligible, conv_output_nchw)
from ..utils.traversal import _pair, _single, _triple
from .layers import NormalConvNd, NormalConvTransposeNd, NormalLinear


def _signs(*shape, device):
    return (torch.rand(*shape, device=device) - .5).sign()


_FUSED_LINEAR = {"on": True}
_KERNEL_CONV = {"on": True}


def set_fused_flipout_linear(flag=True):
    """False: FlipoutNormalLinear evaluates the reference's two-contraction composite on CUDA too (A/B comparisons)."""
    _FUSED_LINEAR["on"] = bool(flag)


def set_flipout_conv_kernels(flag=True):
    """False: FlipOutNormalConv1d / 2d and FlipOutNormalConvTranspose1d / 2d / 3d evaluate the reference's composite with
    torch's convolutions on CUDA too."""
    _KERNEL_CONV["on"] = bool(flag)


class FlipoutNormalLinear(NormalLinear):
    _fused = False        # not a Philox-noise layer: the container treats it as a composite ...
    _mc_composite = True  # ... that takes part in the batched Monte-Carlo forward (S sign draws in one call)

    def __init__(self, in_features, out_features, prior=Normal(0, .1)):
        super(FlipoutNormalLinear, self).__init__(in_features, out_features, False, prior)

    def sample(self):
        self.R = _signs(self.weight.size(0), device=self.weight.device)
        self.S = _signs(self.weight.size(1), device=self.weight.device)
        self._signs = None

    @property
    def sampled(self):
        return (self.R, self.S)

    def _forward_fused(self, x, sample):
        """One sampled contraction with eps = R S^T per Monte-Carlo sample (module doc)."""
        from ..functional import DrawSpec, SampledLinear
        ctx = runtime.current_mc()
        S = 1 if ctx is None else ctx.samples
        shared = ctx is None or not ctx.expanded
        if ctx is not None and shared and x.shape[0] != ctx.rows:
            raise RuntimeError("batched Monte-Carlo forward: the first Bayesian layer must see the network "
                               f"input rows ({ctx.rows}), got {x.shape[0]}")
        dev = self.weight.device
        if sample:
            R = _signs(S, self.weight.size(0), device=dev)
            Sg = _signs(S, self.weight.size(1), device=dev)
            self._signs = (R, Sg)
            self.R, self.S = R[-1], Sg[-1]
        elif S == 1:              # dense.py:77-79: reuse the attributes (a previous draw, sample(), or set by the caller)
            self._signs = (self.R.reshape(1, -1).to(dev, torch.float32).contiguous(),
                           self.S.reshape(1, -1).to(dev, torch.float32).contiguous())
        elif getattr(self, "_signs", None) is None or self._signs[0].shape[0] != S:
            raise RuntimeError("forward(sample=False) needs a previous draw with the same number of MC samples")
        spec = DrawSpec(0, 0, 0, signs=self._signs)
        lead = x.shape[:-1]
        y = SampledLinear.apply(x.reshape(-1, x.shape[-1]), self.weight.mean, self.weight.scale, None, None, S, shared,
                                spec, None, runtime.precision())
        if ctx is not None:
            ctx.expanded = True
        if shared and S > 1:
            return y.view((S * lead[0],) + tuple(lead[1:]) + (y.shape[-1],))
        return y.view(tuple(lead) + (y.shape[-1],))

    def forward(self, x, sample=True):
        if x.is_cuda and _FUSED_LINEAR["on"] and x.dtype == torch.float32:
            return self._forward_fused(x, sample)
        S, x, ctx = runtime.mc_expand_rows(x)
        if ctx is not None and S > 1 and sample:
            # S Monte-Carlo passes at once: one sign pair per sample, shared by that sample's B rows (dense.py:71-75)
            R = _signs(S, 1, self.weight.size(0), device=self.weight.device)
            Sg = _signs(S, 1, self.weight.size(1), device=self.weight.device)
            self.R, self.S = R[-1, 0], Sg[-1, 0]
            x3 = x.reshape(S, -1, x.shape[-1])
            perturbation = ((x3 * Sg).matmul(self.weight.stddev.t()) * R).reshape(x.shape[:-1] + (self.weight.size(0),))
            return F.linear(x, self.weight.mean) + perturbation
        if sample:
            self.sample()
        perturbation = (x * self.S).matmul(self.weight.stddev.t()) * self.R
        return F.linear(x, self.weight.mean, perturbation)       # dense.py:81-83: the perturbation rides in as the bias


class FlipOutNormalConvNd(NormalConvNd):
    _op = None            # set by the dimensional subclasses
    _fused = False
    _mc_composite = True  # the signs are per example (conv.py:154-161): S*B rows simply draw S*B sign sets

    def __init__(self, in_channels, out_channels, kernel_size, stride, padding, dilation, transposed, groups, prior):
        super(FlipOutNormalConvNd, self).__init__(in_channels, out_channels, _single(kernel_size), stride, padding,
                                                  dilation, transposed, groups, False, prior)

    def sample(self, batch_size=1, additional_dims=()):
        self.R = _signs(batch_size, self.weight.size(0), *additional_dims, device=self.weight.device)
        self.S = _signs(batch_size, self.weight.size(1), *additional_dims, device=self.weight.device)

    @property
    def sampled(self):
        return (self.R, self.S)

    def _kernel_path(self, x, nd):
        return (_KERNEL_CONV["on"] and nd <= 2 and x.is_cuda and x.dtype == torch.float32 and x.dim() == nd + 2
                and not self.transposed and conv_implicit_eligible(self.in_channels, self.groups))

    def _contract(self, x4, w4, geometry):
        """conv2d(x4, w4) through the implicit-GEMM contraction kernels: the sample-and-contract path with ONE sample and
        injected eps = 0 (W = w4 exactly); autograd returns d x4 and d w4 from the library's input- / weight-gradient
        kernels."""
        from ..functional import DrawSpec, SampledConv2dImplicit
        zero = getattr(self, "_zero_eps", None)
        if zero is None or zero.device != w4.device or zero.numel() != w4.numel():
            zero = torch.zeros(1, w4.numel(), device=w4.device, dtype=torch.float32)
            self._zero_eps = zero
        spec = DrawSpec(0, 0, 0, eps=zero)
        return SampledConv2dImplicit.apply(x4, w4, self.weight.scale.detach().view(w4.shape), None, None, 1, True, spec,
                                           None, runtime.precision(), *geometry)

    def _flipout(self, x, nd, sample):
        _, x, _ = runtime.mc_expand_rows(x)
        if sample:
            self.sample(x.size(0), (1,) * nd)
        if self._kernel_path(x, nd):
            xs = x * self.S.expand_as(x)
            mean, stddev = self.weight.mean, self.weight.stddev
            if nd == 1:            # a 2-d convolution with a height of one
                shape4 = (mean.shape[0], mean.shape[1], 1, mean.shape[2])
                geometry = ((1, tuple(self.stride)[0]), (0, tuple(self.padding)[0]), (1, tuple(self.dilation)[0]))
                x, xs, mean, stddev = x.unsqueeze(2), xs.unsqueeze(2), mean.view(shape4), stddev.view(shape4)
            else:
                geometry = (tuple(self.stride), tuple(self.padding), tuple(self.dilation))
            out = self._contract(x, mean, geometry)
            pert = self._contract(xs, stddev, geometry)
            if nd == 1:
                out, pert = out.squeeze(2), pert.squeeze(2)
            return out + pert * self.R.expand_as(out)
        op = type(self)._op
        args = (self.stride, self.padding, self.dilation, self.groups)
        out = op(x, self.weight.mean, self.bias, *args)
        return out + op(x * self.S.expand_as(x), self.weight.stddev, self.bias, *args) * self.R.expand_as(out)


class FlipOutNormalConv1d(FlipOutNormalConvNd):
    _op = staticmethod(F.conv1d)

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1,
                 prior=Normal(0, .1)):
        super(FlipOutNormalConv1d, self).__init__(in_channels, out_channels, _single(kernel_size), _single(stride),
                                                  _single(padding), _single(dilation), False, groups, prior)

    def forward(self, x, sample=True):
        return self._flipout(x, 1, sample)


class FlipOutNormalConv2d(FlipOutNormalConvNd):
    _op = staticmethod(F.conv2d)

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1,
                 prior=Normal(0, .1)):
        super(FlipOutNormalConv2d, self).__init__(in_channels, out_channels, _pair(kernel_size), _pair(stride),
                                                  _pair(padding), _pair(dilation), False, groups, prior)

    def forward(self, x, sample=True):
        return self._flipout(x, 2, sample)


class FlipOutNormalConv3d(FlipOutNormalConvNd):
    _op = staticmethod(F.conv3d)

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1,
                 prior=Normal(0, .1)):
        super(FlipOutNormalConv3d, self).__init__(in_channels, out_channels, _triple(kernel_size), _triple(stride),
                                                  _triple(padding), _triple(dilation), False, groups, prior)

    def forward(self, x, sample=True):
        return self._flipout(x, 3, sample)


class FlipOutNormalConvTransposeNd(NormalConvTransposeNd):
    """Flipout transposed convolution: the reference's FlipOutNormalConvNd takes `transposed` like BayesianConvNd but
    never built the transposed forward; this one is

        y = conv_transposeNd(x, mean) + R o conv_transposeNd(x o S, stddev),

    with per-example signs (conv.py:154-161) R [B, out_channels, 1, ...] and S [B, in_channels, 1, ...], no bias, and the
    geometry, validation and `output_size` of NormalConvTransposeNd.  CUDA, TF32, groups == 1, in_ and out_channels
    multiples of 32 and a geometry the transposed-convolution kernels take: two contractions of those kernels per pass,
    with the sign products and layout changes in two bandwidth kernels (functional.FlipoutConvTransposeImplicit).
    Everything else — CPU tensors, fp32 mode (cuDNN's TF32 off in both passes), groups > 1, other channel counts,
    geometry the kernels refuse, set_flipout_conv_kernels(False) — evaluates the composite with torch's
    conv_transposeNd."""
    _fused = False
    _mc_composite = True  # per-example signs: S*B rows of the batched Monte-Carlo forward draw S*B sign sets

    def __init__(self, in_channels, out_channels, kernel_size, stride, padding, output_padding, groups, dilation, prior):
        super(FlipOutNormalConvTransposeNd, self).__init__(in_channels, out_channels, kernel_size, stride, padding,
                                                           output_padding, groups, False, dilation, prior)

    def sample(self, batch_size=1, additional_dims=()):
        """R over the out_channels, then S over the in_channels.  FlipOutNormalConvNd.sample reads the two counts from
        weight.size(0) and weight.size(1), which for a transposed weight [in_channels, out_channels // groups, *k] are
        the in_channels and out_channels // groups: the wrong channels, and too few of them for groups > 1."""
        self.R = _signs(batch_size, self.out_channels, *additional_dims, device=self.weight.device)
        self.S = _signs(batch_size, self.in_channels, *additional_dims, device=self.weight.device)

    @property
    def sampled(self):
        return (self.R, self.S)

    def _kernel_path(self, x):
        w = self.weight.mean
        return (_KERNEL_CONV["on"] and x.is_cuda and x.dtype == torch.float32 and w.is_cuda and w.dtype == torch.float32
                and runtime.precision() == _C.PREC_TF32 and self.groups == 1 and self.in_channels % 32 == 0
                and self.out_channels % 32 == 0)

    def _kernels(self, x, nd, output_padding):
        """The kernel path; FlipoutContractionRefused when the kernels do not take the geometry."""
        stride, padding, dilation = tuple(self.stride), tuple(self.padding), tuple(self.dilation)
        mean, scale = self.weight.mean, self.weight.scale
        if nd == 1:               # a 2-d transposed convolution with a height of one
            x = x.unsqueeze(2)
            shape4 = (mean.shape[0], mean.shape[1], 1, mean.shape[2])
            mean, scale = mean.view(shape4), scale.view(shape4)
            stride, padding, output_padding, dilation = ((1, stride[0]), (0, padding[0]), (0, output_padding[0]),
                                                         (1, dilation[0]))
        nchw_out = conv_output_nchw(x)
        # output_padding >= stride (dilation > stride): zero input rows appended, as in NormalConvTransposeNd
        extra = [op // s for op, s in zip(output_padding, stride)]
        if any(extra):
            pad = []
            for e in reversed(extra):
                pad += [0, e]
            x = F.pad(x, pad)
            output_padding = tuple(op % s for op, s in zip(output_padding, stride))
        if not (x.is_contiguous() or x.permute(0, *range(2, x.dim()), 1).is_contiguous()):
            x = x.contiguous()
        zero = getattr(self, "_zero_eps", None)
        if zero is None or zero.device != mean.device or zero.numel() != mean.numel():
            zero = torch.zeros(1, mean.numel(), device=mean.device, dtype=torch.float32)
            self._zero_eps = zero
        n = x.shape[0]
        R = self.R.reshape(n, -1).to(x.device, torch.float32).contiguous()
        S = self.S.reshape(n, -1).to(x.device, torch.float32).contiguous()
        y = FlipoutConvTransposeImplicit.apply(x, mean, scale, R, S, zero, stride, padding, output_padding, dilation,
                                               nchw_out)
        return y.squeeze(2) if nd == 1 else y

    def _composite(self, x, output_padding):
        """The reference's form with torch's conv_transposeNd; cuDNN's TF32 follows the precision mode."""
        tf32 = runtime.precision() == _C.PREC_TF32
        args = (tuple(self.stride), tuple(self.padding), tuple(output_padding), self.groups, tuple(self.dilation), tf32)
        R, S = self.R.to(x.device), self.S.to(x.device)
        out = CudnnConvTranspose.apply(x, self.weight.mean, None, *args)
        y = out + CudnnConvTranspose.apply(x * S.expand_as(x), self.weight.stddev, None, *args) * R.expand_as(out)
        return y.contiguous() if conv_output_nchw(x) else y

    def _flipout(self, x, nd, sample, output_size):
        output_padding = self._output_padding(x, output_size)
        _, x, _ = runtime.mc_expand_rows(x)
        if sample:
            self.sample(x.size(0), (1,) * nd)
        else:
            # the signs of an earlier forward (or sample(B, (1,) * nd)); the draw at construction has no spatial dims
            n, ones = x.size(0), (1,) * nd
            R, S = getattr(self, "R", None), getattr(self, "S", None)
            if (R is None or S is None or tuple(R.shape) != (n, self.out_channels) + ones
                    or tuple(S.shape) != (n, self.in_channels) + ones):
                have = "no signs" if R is None or S is None else f"R {tuple(R.shape)} and S {tuple(S.shape)}"
                raise RuntimeError(f"forward(sample=False) reuses the signs of an earlier forward, which must be "
                                   f"R {(n, self.out_channels) + ones} and S {(n, self.in_channels) + ones} for this "
                                   f"batch of {n} examples; the layer holds {have}")
        if self._kernel_path(x):
            try:
                return self._kernels(x, nd, output_padding)
            except FlipoutContractionRefused:
                pass
        return self._composite(x, output_padding)


class FlipOutNormalConvTranspose1d(FlipOutNormalConvTransposeNd):
    """torch.nn.ConvTranspose1d's constructor order without `bias` — evaluated as a 2-d transposed convolution with a
    height of one on the kernel path."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, output_padding=0, groups=1,
                 dilation=1, prior=Normal(0, .1)):
        super(FlipOutNormalConvTranspose1d, self).__init__(in_channels, out_channels, _single(kernel_size),
                                                           _single(stride), _single(padding), _single(output_padding),
                                                           groups, _single(dilation), prior)

    def forward(self, x, sample=True, output_size=None):
        return self._flipout(x, 1, sample, output_size)


class FlipOutNormalConvTranspose2d(FlipOutNormalConvTransposeNd):
    """torch.nn.ConvTranspose2d's constructor order without `bias`."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, output_padding=0, groups=1,
                 dilation=1, prior=Normal(0, .1)):
        super(FlipOutNormalConvTranspose2d, self).__init__(in_channels, out_channels, _pair(kernel_size), _pair(stride),
                                                           _pair(padding), _pair(output_padding), groups, _pair(dilation),
                                                           prior)

    def forward(self, x, sample=True, output_size=None):
        return self._flipout(x, 2, sample, output_size)


class FlipOutNormalConvTranspose3d(FlipOutNormalConvTransposeNd):
    """torch.nn.ConvTranspose3d's constructor order without `bias`."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, output_padding=0, groups=1,
                 dilation=1, prior=Normal(0, .1)):
        super(FlipOutNormalConvTranspose3d, self).__init__(in_channels, out_channels, _triple(kernel_size),
                                                           _triple(stride), _triple(padding), _triple(output_padding),
                                                           groups, _triple(dilation), prior)

    def forward(self, x, sample=True, output_size=None):
        return self._flipout(x, 3, sample, output_size)
