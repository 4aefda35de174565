"""FlipOutNormalConvTranspose1d / 2d / 3d on the B200: the sign passes (bnn_flipout_split / _combine) bit for bit against
torch, the layers against an fp64 composite with the same signs (forward, input gradient, d mean, d scale) on the kernel
path and on every fallback, input and output formats, the batched Monte-Carlo forward, and KL / pruning / ELBOAdam over
the new layer's weight."""
import copy

import pytest
import torch
import torch.nn.functional as F

import bayesianneuralnetworks_b200 as bnn
from bayesianneuralnetworks_b200 import _C, functional
from bayesianneuralnetworks_b200.nn import (BayesianNetworkModule, FlipOutNormalConvTranspose1d,
                                            FlipOutNormalConvTranspose2d, FlipOutNormalConvTranspose3d, KLDivergence,
                                            NormalConvTranspose2d, WeightNormal)
from bayesianneuralnetworks_b200.nn.flipout import set_flipout_conv_kernels
from bayesianneuralnetworks_b200.prune import PruneNormal

pytestmark = pytest.mark.gpu

_OPS = {1: F.conv_transpose1d, 2: F.conv_transpose2d, 3: F.conv_transpose3d}


@pytest.fixture(autouse=True)
def _defaults():
    bnn.set_precision("tf32")
    bnn.set_mc_batching("auto")
    bnn.set_conv_output_format("contiguous")
    set_flipout_conv_kernels(True)
    yield
    bnn.set_precision("fp32")
    bnn.set_mc_batching("auto")
    bnn.set_conv_output_format("contiguous")
    set_flipout_conv_kernels(True)


@pytest.fixture
def paths(monkeypatch):
    """Which path each call took: 'kernel' (FlipoutConvTransposeImplicit ran) or 'composite' (torch's conv_transposeNd,
    through CudnnConvTranspose)."""
    seen = []
    real_kernel = functional.FlipoutConvTransposeImplicit.apply
    real_cudnn = functional.CudnnConvTranspose.apply

    def kernel(*a):
        y = real_kernel(*a)
        seen.append("kernel")
        return y

    def cudnn(*a):
        seen.append("composite")
        return real_cudnn(*a)
    monkeypatch.setattr(functional.FlipoutConvTransposeImplicit, "apply", kernel)
    monkeypatch.setattr(functional.CudnnConvTranspose, "apply", cudnn)
    return seen


@pytest.fixture
def no_torch_conv(monkeypatch):
    """torch's transposed convolutions raise: the kernel path must not touch them, forward or backward."""
    def boom(*a, **k):
        raise AssertionError("torch's conv_transpose ran on the kernel path")
    for n in ("conv_transpose1d", "conv_transpose2d", "conv_transpose3d"):
        monkeypatch.setattr(F, n, boom)
        monkeypatch.setattr(torch, n, boom)


def rel_err(got, ref):
    ref = ref.detach().double()
    return float((got.detach().double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


# ---------------------------------------------------------------------------------------------------- sign passes
def _as(t, channels_last):
    if not channels_last:
        return t.contiguous()
    return t.movedim(1, -1).contiguous().movedim(-1, 1)


@pytest.mark.parametrize("C", [1, 3, 32, 33, 256])
@pytest.mark.parametrize("P", [1, 7, 16, 1024, 32 ** 3])
def test_split_and_combine_are_bit_identical_to_torch(C, P):
    torch.manual_seed(C * 131 + P)
    for n in (1, 3, 5):
        if n * C * P > 1 << 26:
            continue
        a = torch.randn(n, C, P, device="cuda")
        b = torch.randn(n, C, P, device="cuda")
        sign = (torch.rand(n, C, device="cuda") - .5).sign()
        s = sign[:, :, None]
        for cl_in in (False, True):
            src = _as(a, cl_in)
            a_cl, sa_cl = _C.flipout_split(src, sign)
            assert a_cl.movedim(1, -1).is_contiguous() and sa_cl.movedim(1, -1).is_contiguous()
            assert torch.equal(a_cl, a) and torch.equal(sa_cl, a * s)
            if cl_in:
                assert a_cl.data_ptr() == src.data_ptr()                 # nothing written for a channels-last input
        for cl_out in (False, True):
            y = _C.flipout_combine(_as(a, True), _as(b, True), sign, channels_last=cl_out)
            assert (y.movedim(1, -1) if cl_out else y).is_contiguous()
            assert torch.equal(y, a + b * s)


@pytest.mark.parametrize("shape", [(2, 64, 16, 16), (3, 32, 16, 24), (2, 16, 8, 16, 16)])
def test_sign_passes_on_images_above_the_48_kib_transposition_limit(shape):
    """Images whose (C + 1) x P block exceeds the 48 KiB of bnn_nchw_to_nhwc_bias_grad: the tiled pass has no such
    limit.  4-d and 5-d tensors in both formats."""
    n, C = shape[0], shape[1]
    assert (C + 1) * (torch.Size(shape[2:]).numel()) * 4 > 48 * 1024
    fmt = torch.channels_last if len(shape) == 4 else torch.channels_last_3d
    a = torch.randn(shape, device="cuda")
    b = torch.randn(shape, device="cuda").contiguous(memory_format=fmt)
    sign = (torch.rand(n, C, device="cuda") - .5).sign()
    s = sign.view((n, C) + (1,) * (len(shape) - 2))
    a_cl, sa_cl = _C.flipout_split(a, sign)
    assert a_cl.is_contiguous(memory_format=fmt) and sa_cl.is_contiguous(memory_format=fmt)
    assert torch.equal(a_cl, a) and torch.equal(sa_cl, a * s)
    for cl_out in (False, True):
        y = _C.flipout_combine(a_cl, b, sign, channels_last=cl_out)
        assert y.is_contiguous(memory_format=fmt if cl_out else torch.contiguous_format)
        assert torch.equal(y, a + b * s)


# ---------------------------------------------------------------------------------------------------- layers
def run(layer, x, gy, **kw):
    x = x.detach().clone().requires_grad_(True)
    y = layer(x, **kw)
    (y * gy).sum().backward()
    return y, [x.grad, layer.weight.mean.grad, layer.weight.scale.grad]


def composite64(layer, x, gy, output_padding=None):
    """fp64 torch: conv_transposeNd(x, mean) + R o conv_transposeNd(x o S, stddev) with the layer's last signs."""
    nd = x.dim() - 2
    R, S = (t.double() for t in layer.sampled)
    x = x.detach().double().clone().requires_grad_(True)
    mean = layer.weight.mean.detach().double().clone().requires_grad_(True)
    scale = layer.weight.scale.detach().double().clone().requires_grad_(True)
    op = layer.output_padding if output_padding is None else output_padding
    args = (layer.stride, layer.padding, op, layer.groups, layer.dilation)
    y = _OPS[nd](x, mean, None, *args) + _OPS[nd](x * S, 1e-10 + F.softplus(scale), None, *args) * R
    (y * gy.double()).sum().backward()
    return y, [x.grad, mean.grad, scale.grad]


def check(layer, x, tol, output_size=None):
    kw = {} if output_size is None else dict(output_size=output_size)
    with torch.no_grad():
        shape = layer(x, **kw).shape
    gy = torch.randn(shape, device="cuda")
    y, grads = run(layer, x, gy, **kw)
    op = None if output_size is None else layer._output_padding(x, output_size)
    y64, g64 = composite64(layer, x, gy, op)
    assert y.shape == y64.shape and y.is_contiguous()
    for name, a, b in zip(("y", "dx", "d mean", "d scale"), [y] + grads, [y64] + g64):
        assert rel_err(a, b) <= tol, (name, rel_err(a, b))


# (Cin, Cout, k, stride, padding, output_padding, dilation, H, W)
CASES_2D = [
    (32, 32, 4, 2, 1, 0, 1, 5, 6),              # the decoder layer: k4 s2 p1
    (64, 32, 3, 2, 1, 1, 1, 7, 5),              # k3 s2 p1 op1
    (32, 64, 2, 2, 0, 0, 1, 4, 4),              # k2 s2
    (32, 32, 3, 1, 1, 0, 1, 6, 6),              # k3 s1 p1
    (32, 32, 3, 1, 0, 1, 2, 5, 5),              # dilation 2, output_padding >= stride
    (32, 32, 3, (1, 2), 1, (0, 1), 1, 5, 6),    # stride (1, 2)
    (32, 32, 1, 2, 0, 1, 1, 4, 5),              # k < s: phases without taps
]


@pytest.mark.parametrize("case", CASES_2D, ids=[str(i) for i in range(len(CASES_2D))])
def test_flipout_conv_transpose2d_kernel_path(case, paths, no_torch_conv):
    Cin, Cout, k, s, p, op, d, H, W = case
    torch.manual_seed(hash(case) % 1000)
    layer = FlipOutNormalConvTranspose2d(Cin, Cout, k, stride=s, padding=p, output_padding=op, dilation=d).cuda()
    x = torch.randn(3, Cin, H, W, device="cuda")
    check(layer, x, 2e-3)
    assert paths and set(paths) == {"kernel"}


def test_flipout_conv_transpose2d_output_size(paths, no_torch_conv):
    layer = FlipOutNormalConvTranspose2d(32, 32, 3, stride=2, padding=1).cuda()
    x = torch.randn(2, 32, 5, 6, device="cuda")
    check(layer, x, 2e-3, output_size=(10, 12))
    assert set(paths) == {"kernel"}


def test_flipout_conv_transpose1d_kernel_path(paths, no_torch_conv):
    layer = FlipOutNormalConvTranspose1d(32, 64, 4, stride=2).cuda()
    check(layer, torch.randn(4, 32, 9, device="cuda"), 2e-3)
    assert set(paths) == {"kernel"}


# (Cin, Cout, k, stride, padding, D, H, W)
CASES_3D = [
    (32, 32, 2, 2, 0, 3, 4, 4),
    (32, 64, 4, 2, 1, 3, 3, 4),
    (64, 32, (1, 4, 4), (1, 2, 2), (0, 1, 1), 2, 4, 5),
]


@pytest.mark.parametrize("case", CASES_3D, ids=[str(i) for i in range(len(CASES_3D))])
def test_flipout_conv_transpose3d_kernel_path(case, paths, no_torch_conv):
    Cin, Cout, k, s, p, D, H, W = case
    torch.manual_seed(7)
    layer = FlipOutNormalConvTranspose3d(Cin, Cout, k, stride=s, padding=p).cuda()
    check(layer, torch.randn(2, Cin, D, H, W, device="cuda"), 2e-3)
    assert set(paths) == {"kernel"}


@pytest.mark.parametrize("make,shape,prec,tol", [
    (lambda: FlipOutNormalConvTranspose2d(32, 32, 4, stride=2, padding=1, groups=2), (2, 32, 5, 5), "tf32", 2e-3),
    (lambda: FlipOutNormalConvTranspose2d(32, 3, 4, stride=2, padding=1), (2, 32, 5, 5), "tf32", 2e-3),
    (lambda: FlipOutNormalConvTranspose2d(16, 32, 3, stride=2, padding=1, output_padding=1), (2, 16, 5, 5), "tf32",
     2e-3),
    (lambda: FlipOutNormalConvTranspose2d(32, 32, 4, stride=2, padding=1), (2, 32, 5, 5), "fp32", 1e-5),
    (lambda: FlipOutNormalConvTranspose1d(32, 32, 4, stride=2), (2, 32, 7), "fp32", 1e-5),
    (lambda: FlipOutNormalConvTranspose3d(32, 32, 2, stride=2), (2, 32, 3, 3, 3), "fp32", 1e-5),
    # a filter extent (k - 1) d = 34 beyond the rank-5 im2col descriptor: refused by the 3-d predicate
    (lambda: FlipOutNormalConvTranspose3d(32, 32, 3, stride=1, padding=1, dilation=17), (1, 32, 2, 2, 2), "tf32", 2e-3),
    # stride 2: the forward's phase corners are within the im2col limits, the conv view the gradients use is not
    (lambda: FlipOutNormalConvTranspose1d(32, 32, 200, stride=2), (2, 32, 5), "tf32", 2e-3),
    (lambda: FlipOutNormalConvTranspose2d(32, 32, 3, stride=2, dilation=65), (1, 32, 3, 3), "tf32", 2e-3),
], ids=["groups2", "cout3", "cin16", "fp32", "fp32_1d", "fp32_3d", "refused3d", "refused1d_k200", "refused2d_d65"])
def test_fallbacks_take_the_composite(make, shape, prec, tol, paths):
    bnn.set_precision(prec)
    torch.manual_seed(5)
    layer = make().cuda()
    check(layer, torch.randn(shape, device="cuda"), tol)
    assert paths and "kernel" not in paths and "composite" in paths


def test_switch_off_takes_the_composite(paths):
    set_flipout_conv_kernels(False)
    layer = FlipOutNormalConvTranspose2d(32, 32, 4, stride=2, padding=1).cuda()
    check(layer, torch.randn(2, 32, 5, 5, device="cuda"), 2e-3)
    assert set(paths) == {"composite"}


def test_channels_last_input_and_preserve_format(paths, no_torch_conv):
    torch.manual_seed(9)
    layer = FlipOutNormalConvTranspose2d(32, 64, 4, stride=2, padding=1).cuda()
    x = torch.randn(2, 32, 6, 5, device="cuda").contiguous(memory_format=torch.channels_last)
    check(layer, x, 2e-3)                                      # 'contiguous': NCHW output whatever the input
    bnn.set_conv_output_format("preserve")
    y = layer(x)
    assert y.is_contiguous(memory_format=torch.channels_last)
    xg = x.detach().clone().requires_grad_(True)
    layer(xg, sample=False).sum().backward()
    assert xg.grad.is_contiguous(memory_format=torch.channels_last)
    gy = torch.randn(y.shape, device="cuda")
    layer.zero_grad()
    y2, grads = run(layer, x, gy, sample=False)
    y64, g64 = composite64(layer, x, gy)
    assert y2.is_contiguous(memory_format=torch.channels_last)
    for a, b in zip([y2] + grads, [y64] + g64):
        assert rel_err(a, b) <= 2e-3
    y3 = layer(torch.randn(2, 32, 6, 5, device="cuda"))
    assert y3.is_contiguous()                                  # 'preserve' with an NCHW input
    assert set(paths) == {"kernel"}


def test_misaligned_input_takes_the_kernel_path(paths, no_torch_conv):
    torch.manual_seed(6)
    layer = FlipOutNormalConvTranspose2d(32, 32, 4, stride=2, padding=1).cuda()
    flat = torch.randn(2 * 32 * 5 * 5 + 1, device="cuda", requires_grad=True)
    x = flat[1:].view(2, 32, 5, 5)                             # contiguous, 4 bytes past a 16-byte boundary
    assert x.data_ptr() % 16 != 0
    y = layer(x)
    gy = torch.randn(y.shape, device="cuda")
    (y * gy).sum().backward()
    y64, g64 = composite64(layer, x, gy)
    for a, b in zip([y, flat.grad[1:].view(x.shape), layer.weight.mean.grad, layer.weight.scale.grad], [y64] + g64):
        assert rel_err(a, b) <= 2e-3
    assert set(paths) == {"kernel"}


def test_non_contiguous_incoming_gradient(paths, no_torch_conv):
    torch.manual_seed(4)
    layer = FlipOutNormalConvTranspose2d(32, 32, 3, stride=2, padding=1, output_padding=1).cuda()
    x = torch.randn(2, 32, 5, 5, device="cuda")
    y = layer(x)
    g_full = torch.randn(y.shape[0], y.shape[1], y.shape[3], y.shape[2], device="cuda")
    gy = g_full.transpose(2, 3)                                # neither NCHW- nor channels-last-contiguous
    assert not gy.is_contiguous() and not gy.is_contiguous(memory_format=torch.channels_last)
    xg = x.clone().requires_grad_(True)
    layer.zero_grad()
    layer(xg, sample=False).backward(gy)
    _, g64 = composite64(layer, x, gy)
    for a, b in zip([xg.grad, layer.weight.mean.grad, layer.weight.scale.grad], g64):
        assert rel_err(a, b) <= 2e-3
    assert set(paths) == {"kernel"}


# ---------------------------------------------------------------------------------------------------- whole models
class Decoder(BayesianNetworkModule):
    def __init__(self, samples=4):
        super().__init__(32, 32, samples)
        self.up = NormalConvTranspose2d(32, 32, 4, stride=2, padding=1)
        self.act = torch.nn.ELU()
        self.flip = FlipOutNormalConvTranspose2d(32, 32, 4, stride=2, padding=1)

    def _forward(self, x):
        return self.flip(self.act(self.up(x)))


def test_batched_monte_carlo_forward_agrees_with_the_loop(paths):
    torch.manual_seed(3)
    S, B = 4, 3
    net = Decoder(S).cuda()
    assert net._mc_plan()[0] is True
    x = torch.rand(B, 32, 4, 4, device="cuda")
    saved = {n: p.detach().clone() for n, p in net.named_parameters()}
    with torch.no_grad():                                      # noise-free limit: sigma ~ 1e-10
        for n, p in net.named_parameters():
            if n.endswith(".scale"):
                p.fill_(-100.0)
        bnn.set_mc_batching("always")
        batched = net(x)
        assert tuple(net.flip.R.shape) == (S * B, 32, 1, 1)    # S*B rows draw S*B sign sets
        bnn.set_mc_batching("never")
        loop = net(x)
    assert isinstance(batched, list) and len(batched) == S and batched[0].shape == (B, 32, 16, 16)
    for a, b in zip(batched, loop):
        assert torch.allclose(a, b, rtol=5e-3, atol=2e-3)
    with torch.no_grad():
        for n, p in net.named_parameters():
            p.copy_(saved[n])
    # with noise: the moments of many batched samples agree with the loop's
    n_mc = 400
    bnn.set_mc_batching("always")
    with torch.no_grad():
        big = torch.stack(net(x, samples=n_mc))
        bnn.set_mc_batching("never")
        ref = torch.stack([torch.stack(net(x, samples=50)) for _ in range(n_mc // 50)]).flatten(0, 1)
    assert float(big.std(0).mean()) > 1e-3
    se = ref.std(0) / n_mc ** 0.5
    assert float(((big.mean(0) - ref.mean(0)).abs() > 6 * se + 1e-4).float().mean()) < 1e-3
    assert torch.allclose(big.std(0).mean(), ref.std(0).mean(), rtol=0.05)
    # gradients reach every variational parameter through the batched pass
    bnn.set_mc_batching("always")
    net.zero_grad()
    torch.stack(net(x)).square().mean().backward()
    for n, p in net.named_parameters():
        assert p.grad is not None and float(p.grad.abs().sum()) > 0, n
    assert "kernel" in paths and "composite" not in paths


class Net(BayesianNetworkModule):
    def __init__(self):
        super().__init__(32, 32, 2)
        self.flip = FlipOutNormalConvTranspose2d(32, 32, 4, stride=2, padding=1)

    def _forward(self, x):
        return self.flip(x)


def test_kl_pruning_and_elbo_adam_cover_the_layer():
    torch.manual_seed(12)
    model = Net().cuda()
    kld = KLDivergence(number_of_batches=3)
    w = model.flip.weight
    q = torch.distributions.Normal(w.mean.double(), 1e-10 + F.softplus(w.scale.double()))
    want = torch.distributions.kl_divergence(q, torch.distributions.Normal(0.0, 0.1)).mean() / 3
    assert [m for m in model.modules() if isinstance(m, WeightNormal)] == [w]
    assert float(kld(model).detach()) == pytest.approx(float(want), rel=1e-5)
    before = w.mean.detach().clone()
    PruneNormal()(model, 0.5)
    changed = w.mean != before
    assert int(changed.sum()) == int(0.5 * before.numel()) == int((w.scale == -30).sum())
    assert bool((w.mean[changed] == 0).all())
    ref_model, new_model = copy.deepcopy(model), copy.deepcopy(model)
    x = torch.randn(2, 32, 5, 5, device="cuda")
    target = torch.randn(2, 32, 10, 10, device="cuda")
    ref_opt = torch.optim.Adam(ref_model.parameters(), lr=2e-3)
    new_opt = bnn.optim.ELBOAdam(new_model, number_of_batches=3, lr=2e-3)
    for step in range(3):
        torch.manual_seed(100 + step)                         # the same signs for both models
        ref_opt.zero_grad()
        (bnn.nn.mc_mean_loss(F.mse_loss, ref_model(x), target) + kld(ref_model)).backward()
        ref_opt.step()
        torch.manual_seed(100 + step)
        new_opt.zero_grad()
        bnn.nn.mc_mean_loss(F.mse_loss, new_model(x), target).backward()
        new_opt.step()
    for (n, a), (_, b) in zip(ref_model.named_parameters(), new_model.named_parameters()):
        assert torch.allclose(a, b, rtol=2e-4, atol=2e-6), (n, float((a - b).abs().max()))
