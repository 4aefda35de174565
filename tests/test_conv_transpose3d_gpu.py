"""NormalConvTranspose3d on the B200 against torch's conv_transpose3d in fp64 with the same (injected) eps: output, input
gradient and the gradients of weight / bias mean and scale, over strides (isotropic and anisotropic), kernels, dilations,
output paddings, channel counts and groups on both sides of the 3-d kernels' eligibility, both sides of the rank-5 corner
limit, shared and per-sample inputs, both output formats and several Monte-Carlo sample counts; the in-kernel Philox
draw against `.sampled`, `output_size`, and a small 3-d encoder/decoder through the batched Monte-Carlo forward, KL,
pruning, ELBOAdam and CUDA-graph replay."""
import copy

import pytest
import torch
import torch.nn.functional as F

import bayesianneuralnetworks_b200 as bnn
from bayesianneuralnetworks_b200 import _C, functional
from bayesianneuralnetworks_b200.nn import (BayesianNetworkModule, KLDivergence, NormalConv3d, NormalConvTranspose2d,
                                            NormalConvTranspose3d, WeightNormal)
from bayesianneuralnetworks_b200.prune import PruneNormal

pytestmark = pytest.mark.gpu

TOL = {"fp32": 2e-5, "tf32": 2e-3}


@pytest.fixture(autouse=True)
def _defaults():
    bnn.set_precision("fp32")
    bnn.set_mc_batching("auto")
    bnn.set_conv_output_format("contiguous")
    bnn.manual_seed(0x3D)
    yield
    bnn.set_precision("fp32")
    bnn.set_mc_batching("auto")
    bnn.set_conv_output_format("contiguous")


@pytest.fixture
def paths(monkeypatch):
    """Records which path each forward took: 'kernel' (the 3-d gather accepted the request), 'refused' (it did not) and
    'cudnn' (one materialised-sample call per sample)."""
    seen = []
    real = _C.try_sampled_conv_transpose3d_fwd

    def fwd(*a):
        ok = real(*a)
        seen.append("kernel" if ok else "refused")
        return ok
    monkeypatch.setattr(_C, "try_sampled_conv_transpose3d_fwd", fwd)
    real_apply = functional.CudnnConvTranspose3d.apply

    def cudnn(*a):
        seen.append("cudnn")
        return real_apply(*a)
    monkeypatch.setattr(functional.CudnnConvTranspose3d, "apply", cudnn)
    return seen


def rel_err(got, ref):
    ref = ref.detach().double()
    return float((got.detach().double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def run_layer(layer, x, S, shared, eps_w, eps_b, gy):
    """The layer's own dispatch for S samples with injected eps; returns y and the gradients of x, weight and bias."""
    x = x.detach().clone().requires_grad_(True)
    inj = {layer.weight: eps_w}
    if layer.bias is not None:
        inj[layer.bias] = eps_b
    with bnn.injected_eps(inj):
        spec_w = layer.weight.draw_spec(0, S)
        spec_b = layer.bias.draw_spec(0, S) if layer.bias is not None else None
        y = layer._conv_transpose3d(x, S, shared, spec_w, spec_b, tuple(layer.output_padding))
    (y * gy).sum().backward()
    grads = [x.grad, layer.weight.mean.grad, layer.weight.scale.grad]
    if layer.bias is not None:
        grads += [layer.bias.mean.grad, layer.bias.scale.grad]
    return y, grads


def reference(layer, x, S, shared, eps_w, eps_b, gy):
    """fp64 torch: W_s = mean + (1e-10 + softplus(scale)) eps_s, one conv_transpose3d per sample."""
    x = x.detach().double().clone().requires_grad_(True)
    params = [layer.weight.mean, layer.weight.scale] + ([layer.bias.mean, layer.bias.scale] if layer.bias is not None else [])
    p64 = [p.detach().double().clone().requires_grad_(True) for p in params]
    B = x.shape[0] if shared else x.shape[0] // S
    ys = []
    for s in range(S):
        W = p64[0] + (1e-10 + F.softplus(p64[1])) * eps_w[s].double()
        b = p64[2] + (1e-10 + F.softplus(p64[3])) * eps_b[s].double() if layer.bias is not None else None
        xs = x if shared else x[s * B:(s + 1) * B]
        ys.append(F.conv_transpose3d(xs, W, b, layer.stride, layer.padding, layer.output_padding, layer.groups,
                                     layer.dilation))
    y = torch.cat(ys)
    (y * gy.double()).sum().backward()
    return y, [x.grad] + [p.grad for p in p64]


def _check(layer, x, S, shared, prec, memory_format=torch.contiguous_format, seed=0):
    torch.manual_seed(seed)
    Cout = layer.out_channels
    eps_w = torch.randn((S,) + tuple(layer.weight.mean.shape), device="cuda")
    eps_b = torch.randn(S, Cout, device="cuda")
    B = x.shape[0] if shared else x.shape[0] // S
    out = [functional.conv_transpose_out(n, k, s, p, o, d) for n, k, s, p, o, d in
           zip(x.shape[2:], layer.kernel_size, layer.stride, layer.padding, layer.output_padding, layer.dilation)]
    gy = torch.randn(S * B, Cout, *out, device="cuda").contiguous(memory_format=memory_format)
    layer.zero_grad()
    y_ref, g_ref = reference(layer, x, S, shared, eps_w, eps_b, gy)
    layer.zero_grad()
    y, grads = run_layer(layer, x, S, shared, eps_w, eps_b, gy)
    assert y.shape == y_ref.shape
    assert rel_err(y, y_ref) < TOL[prec]
    for name, a, b in zip(("dx", "dmu_w", "drho_w", "dmu_b", "drho_b"), grads, g_ref):
        assert rel_err(a, b) < TOL[prec], (name, rel_err(a, b))
    return y


# (Cin, Cout, k, stride, padding, output_padding, dilation, groups, (D, H, W), S, shared, path in TF32)
CASES = [
    (64, 32, 2, 2, 0, 0, 1, 1, (4, 5, 3), 3, False, "kernel"),                    # the 3-D U-Net up-conv: k2 s2
    (32, 32, 4, 2, 1, 0, 1, 1, (3, 4, 4), 3, False, "kernel"),                    # k4 s2 p1
    (32, 64, 3, 2, 1, 1, 1, 1, (3, 4, 3), 3, True, "kernel"),                     # k3 s2 p1 op1, shared input
    (32, 32, (1, 4, 4), (1, 2, 2), (0, 1, 1), 0, 1, 1, (3, 4, 5), 3, False, "kernel"),   # anisotropic (V3's layer)
    (32, 32, (3, 4, 4), (1, 2, 2), (1, 1, 1), (0, 1, 0), 1, 1, (3, 3, 4), 3, True, "kernel"),
    (32, 32, 3, 2, 2, 1, 2, 1, (4, 4, 3), 3, False, "kernel"),                    # dilation 2 with stride 2
    (32, 32, 1, 2, 0, 1, 1, 1, (3, 3, 4), 3, False, "kernel"),                    # k < s: bias-only phases
    (32, 32, 3, 1, 1, 0, 1, 1, (4, 3, 5), 3, True, "kernel"),                     # stride 1
    (32, 32, 3, 1, 0, 1, 2, 1, (4, 4, 3), 3, False, "kernel"),                    # output_padding >= stride (< dilation)
    (32, 32, 2, 2, 0, 0, 1, 1, (2, 2, 2), 1, False, "kernel"),                    # tensors under 128 KiB, S = 1
    (64, 32, 2, 2, 0, 0, 1, 1, (3, 3, 3), 16, False, "kernel"),                   # S = 16
    (48, 32, 3, 2, 1, 1, 1, 1, (3, 3, 3), 3, False, "refused"),                   # Cin % 32 != 0
    (32, 1, 2, 2, 0, 0, 1, 1, (3, 3, 3), 3, True, "cudnn"),                       # a 1-channel output
    (32, 64, 3, 2, 1, 1, 1, 2, (3, 3, 3), 3, False, "cudnn"),                     # groups 2
]


@pytest.mark.parametrize("prec", ["fp32", "tf32"])
@pytest.mark.parametrize("case", CASES, ids=[str(i) for i in range(len(CASES))])
def test_conv_transpose3d_parity(case, prec, paths):
    Cin, Cout, k, s, p, op, d, g, size, S, shared, path = case
    bnn.set_precision(prec)
    torch.manual_seed(7)
    layer = NormalConvTranspose3d(Cin, Cout, k, stride=s, padding=p, output_padding=op, groups=g, dilation=d).cuda()
    B = 2
    x = torch.randn((B if shared else S * B), Cin, *size, device="cuda")
    y = _check(layer, x, S, shared, prec)
    assert y.is_contiguous()
    if prec == "tf32" and path == "kernel":
        assert paths == ["kernel"]
    elif prec == "tf32" and path == "refused":
        assert paths == ["refused"] + ["cudnn"] * S
    else:
        assert paths == ["cudnn"] * S


@pytest.mark.parametrize("pad,path", [(16, "kernel"), (17, "refused")])
def test_rank5_corner_limit(pad, path, paths):
    """Depth taps 8 apart (extent 16): padding 16 puts a corner at -16, the rank-5 descriptor's limit; 17 is past it and
    the layer contracts materialised samples instead.  Both agree with fp64 torch."""
    bnn.set_precision("tf32")
    layer = NormalConvTranspose3d(32, 32, (3, 1, 1), padding=(pad, 0, 0), dilation=(8, 1, 1)).cuda()
    x = torch.randn(3 * 2, 32, 20, 2, 3, device="cuda")
    _check(layer, x, 3, False, "tf32")
    assert paths[0] == path


@pytest.mark.parametrize("shared", [False, True])
def test_preserve_format_gives_channels_last_3d_and_matches(shared, paths):
    bnn.set_precision("tf32")
    bnn.set_conv_output_format("preserve")
    S, B = 3, 2
    layer = NormalConvTranspose3d(32, 64, 4, stride=2, padding=1).cuda()
    x = torch.randn((B if shared else S * B), 32, 3, 4, 3, device="cuda").contiguous(memory_format=torch.channels_last_3d)
    y = _check(layer, x, S, shared, "tf32", memory_format=torch.channels_last_3d)
    assert y.is_contiguous(memory_format=torch.channels_last_3d)
    assert paths == ["kernel"]


@pytest.mark.parametrize("prec", ["fp32", "tf32"])
def test_bias_only_phases(prec):
    """k < s: phases without a tap hold exactly the sampled bias."""
    bnn.set_precision(prec)
    layer = NormalConvTranspose3d(32, 32, 1, stride=(2, 3, 2), output_padding=(1, 2, 1)).cuda()
    x = torch.randn(2, 32, 3, 3, 3, device="cuda")
    y = layer(x)
    w, b = layer.sampled
    assert rel_err(y, F.conv_transpose3d(x.double(), w.double(), b.double(), (2, 3, 2), 0, (1, 2, 1))) < TOL[prec]
    assert torch.allclose(y[:, :, 1::2, 2::3, 1::2], b.view(1, -1, 1, 1, 1).expand(2, 32, 3, 3, 3), atol=1e-6)


@pytest.mark.parametrize("cfg", [(64, 32, 2, 2, 0, 0), (32, 32, 4, 2, 1, 0), (32, 32, 3, 2, 1, 1), (32, 1, 2, 2, 0, 0)])
@pytest.mark.parametrize("prec", ["fp32", "tf32"])
def test_philox_forward_equals_torch_on_sampled(cfg, prec):
    """The in-kernel Philox draw (and the materialised path's) is the one `.sampled` shows."""
    Cin, Cout, k, s, p, op = cfg
    bnn.set_precision(prec)
    layer = NormalConvTranspose3d(Cin, Cout, k, stride=s, padding=p, output_padding=op).cuda()
    x = torch.randn(3, Cin, 3, 4, 3, device="cuda")
    y = layer(x)
    w, b = layer.sampled
    assert rel_err(y, F.conv_transpose3d(x.double(), w.double(), b.double(), s, p, op)) < TOL[prec]
    assert rel_err(layer(x, sample=False), y) < 1e-6          # the same draw (cuDNN need not sum in the same order)


@pytest.mark.parametrize("prec", ["fp32", "tf32"])
def test_output_size(prec):
    """forward(x, output_size=skip.shape): the U-Net decoder call with an odd skip size."""
    bnn.set_precision(prec)
    layer = NormalConvTranspose3d(32, 32, 3, stride=2, padding=1).cuda()
    x = torch.randn(2, 32, 3, 4, 3, device="cuda")
    skip = torch.zeros(2, 32, 6, 7, 6, device="cuda")
    y = layer(x, output_size=skip.shape)
    assert y.shape == skip.shape
    w, b = layer.sampled
    assert rel_err(y, F.conv_transpose3d(x.double(), w.double(), b.double(), 2, 1, (1, 0, 1))) < TOL[prec]
    two = NormalConvTranspose2d(32, 32, 3, stride=2, padding=1).cuda()
    y2 = two(torch.randn(2, 32, 4, 3, device="cuda"), output_size=(8, 5))
    assert y2.shape == (2, 32, 8, 5)


# ---- a small volumetric encoder / decoder ------------------------------------------------------------------------------
class UNet3d(BayesianNetworkModule):
    def __init__(self, samples):
        super().__init__(1, 1, samples)
        self.down = NormalConv3d(1, 32, 3, stride=2, padding=1)
        self.mid = NormalConv3d(32, 64, 3, padding=1)
        self.up = NormalConvTranspose3d(64, 32, 2, stride=2)
        self.head = NormalConvTranspose3d(32, 1, 3, padding=1)

    def _forward(self, x):
        h = torch.nn.functional.elu(self.mid(torch.nn.functional.elu(self.down(x))))
        return self.head(torch.nn.functional.elu(self.up(h, output_size=x.shape)))


@pytest.mark.parametrize("prec", ["fp32", "tf32"])
def test_batched_model_equals_the_loop(prec):
    bnn.set_precision(prec)
    torch.manual_seed(11)
    proto = UNet3d(3).cuda()
    x = torch.randn(2, 1, 8, 8, 8, device="cuda")
    runs = []
    for mode in ("auto", "never"):
        bnn.set_mc_batching(mode)
        net = copy.deepcopy(proto)
        assert (mode == "never") or net._mc_plan()[0]
        preds = net(x)
        assert isinstance(preds, list) and len(preds) == 3 and preds[0].shape == (2, 1, 8, 8, 8)
        torch.stack([p.square().sum() for p in preds]).mean().backward()
        runs.append((net, preds))
    (a, pa), (b, pb) = runs
    tol = 1e-5 if prec == "fp32" else 2e-3
    for s in range(3):
        assert rel_err(pa[s], pb[s]) < tol
    for (n1, p1), (_, p2) in zip(a.named_parameters(), b.named_parameters()):
        assert rel_err(p1.grad, p2.grad) < 10 * tol, n1


def test_whole_model_kl_prune_and_elbo_adam():
    torch.manual_seed(12)
    model = UNet3d(2).cuda()
    kld = KLDivergence(number_of_batches=3)
    terms = []
    for w in model.modules():
        if isinstance(w, WeightNormal):
            q = torch.distributions.Normal(w.mean.double(), 1e-10 + F.softplus(w.scale.double()))
            terms.append(torch.distributions.kl_divergence(q, torch.distributions.Normal(0.0, 0.1)).mean())
    assert len(terms) == 8
    assert float(kld(model)) == pytest.approx(float(torch.stack(terms).mean() / 3), rel=1e-5)
    up = model.up
    before = up.weight.mean.detach().clone()
    PruneNormal()(model, 0.5)
    changed = up.weight.mean != before
    assert int(changed.sum()) == int(0.5 * before.numel()) == int((up.weight.scale == -30).sum())
    assert bool((up.weight.mean[changed] == 0).all())
    state = {k: v.clone() for k, v in model.state_dict().items()}
    PruneNormal()(model, 0.5)
    assert all(torch.equal(state[k], v) for k, v in model.state_dict().items())
    ref_model, new_model = copy.deepcopy(model), copy.deepcopy(model)
    x = torch.randn(2, 1, 8, 8, 8, device="cuda")
    target = torch.randn(2, 1, 8, 8, 8, device="cuda")
    ref_opt = torch.optim.Adam(ref_model.parameters(), lr=2e-3)
    new_opt = bnn.optim.ELBOAdam(new_model, number_of_batches=3, lr=2e-3)

    def rewind(m, step):
        ids = iter(range(40_000, 50_000))
        for w in m.modules():
            if isinstance(w, WeightNormal):
                w._tensor_id, w._draw = next(ids), 2 * step

    for step in range(3):
        rewind(ref_model, step), rewind(new_model, step)
        ref_opt.zero_grad()
        (bnn.nn.mc_mean_loss(F.mse_loss, ref_model(x), target) + kld(ref_model)).backward()
        ref_opt.step()
        new_opt.zero_grad()
        bnn.nn.mc_mean_loss(F.mse_loss, new_model(x), target).backward()
        new_opt.step()
    for (n, a), (_, b) in zip(ref_model.named_parameters(), new_model.named_parameters()):
        assert torch.allclose(a, b, rtol=2e-4, atol=2e-6), (n, float((a - b).abs().max()))


@pytest.mark.parametrize("prec", ["fp32", "tf32"])
def test_graph_replay_equals_eager(prec):
    from bayesianneuralnetworks_b200 import runtime
    bnn.set_precision(prec)
    bnn.graph_safe_rng(True)
    try:
        layer = NormalConvTranspose3d(32, 64, 4, stride=2, padding=1).cuda()
        sx = torch.randn(2, 32, 3, 4, 3, device="cuda")
        runtime.step_counter(sx.device).zero_()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                layer.zero_grad(set_to_none=True)
                layer(sx).square().sum().backward()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        layer.zero_grad(set_to_none=True)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            bnn.advance_rng_step()
            out = layer(sx)
            out.square().sum().backward()
        outs = []
        tol = 1e-5 if prec == "fp32" else 2e-3
        for _ in range(3):
            g.replay()
            torch.cuda.synchronize()
            got = out.detach().clone()
            gm, gs = layer.weight.mean.grad.clone(), layer.weight.scale.grad.clone()
            outs.append(got)
            eager = copy.deepcopy(layer)
            eager.zero_grad(set_to_none=True)
            eager.weight._draw, eager.bias._draw = layer.weight._draw - 1, layer.bias._draw - 1
            y = eager(sx)
            y.square().sum().backward()
            assert rel_err(got, y) < tol
            assert rel_err(gm, eager.weight.mean.grad) < tol and rel_err(gs, eager.weight.scale.grad) < tol
            w, b = layer.sampled
            assert rel_err(got, F.conv_transpose3d(sx.double(), w.double(), b.double(), 2, 1)) < TOL[prec]
        assert not torch.equal(outs[0], outs[1])
    finally:
        bnn.graph_safe_rng(False)
