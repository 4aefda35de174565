"""NormalConvTranspose1d / 2d on the B200 against torch's conv_transpose in fp64 with the same (injected) eps: output,
input gradient and the gradients of weight / bias mean and scale, over strides, kernels, dilations, output paddings,
channel counts on both sides of the implicit-GEMM eligibility, groups, shared and per-sample inputs, both output formats
and several Monte-Carlo sample counts; plus the batched Monte-Carlo forward, the whole-model operations and graph
replay."""
import copy

import pytest
import torch
import torch.nn.functional as F

import bayesianneuralnetworks_b200 as bnn
from bayesianneuralnetworks_b200 import _C, functional
from bayesianneuralnetworks_b200.nn import (BayesianNetworkModule, KLDivergence, NormalConvTranspose1d,
                                            NormalConvTranspose2d, NormalLinear, WeightNormal)
from bayesianneuralnetworks_b200.prune import PruneNormal

pytestmark = pytest.mark.gpu

TOL = {"fp32": 2e-5, "tf32": 2e-3}


@pytest.fixture(autouse=True)
def _defaults():
    bnn.set_precision("fp32")
    bnn.set_mc_batching("auto")
    bnn.set_conv_output_format("contiguous")
    bnn.manual_seed(0x7A5)
    yield
    bnn.set_precision("fp32")
    bnn.set_mc_batching("auto")
    bnn.set_conv_output_format("contiguous")


def rel_err(got, ref):
    ref = ref.detach().double()
    return float((got.detach().double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def _pair(v):
    return tuple(v) if isinstance(v, (tuple, list)) else (v, v)


def run_layer(layer, x, S, shared, eps_w, eps_b, gy):
    """The layer's own dispatch for S samples with injected eps; returns y and the gradients of x, weight and bias."""
    x = x.detach().clone().requires_grad_(True)
    inj = {layer.weight: eps_w}
    if layer.bias is not None:
        inj[layer.bias] = eps_b
    with bnn.injected_eps(inj):
        spec_w = layer.weight.draw_spec(0, S)
        spec_b = layer.bias.draw_spec(0, S) if layer.bias is not None else None
        w = layer.weight.mean.shape
        if isinstance(layer, NormalConvTranspose1d):
            y = layer._conv_transpose2d(x.unsqueeze(2), (w[0], w[1], 1, w[2]), S, shared, spec_w, spec_b,
                                        (1, layer.stride[0]), (0, layer.padding[0]), (0, layer.output_padding[0]),
                                        (1, layer.dilation[0])).squeeze(2)
        else:
            y = layer._conv_transpose2d(x, tuple(w), S, shared, spec_w, spec_b, tuple(layer.stride), tuple(layer.padding),
                                        tuple(layer.output_padding), tuple(layer.dilation))
    (y * gy).sum().backward()
    grads = [x.grad, layer.weight.mean.grad, layer.weight.scale.grad]
    if layer.bias is not None:
        grads += [layer.bias.mean.grad, layer.bias.scale.grad]
    return y, grads


def reference(layer, x, S, shared, eps_w, eps_b, gy):
    """fp64 torch: W_s = mean + (1e-10 + softplus(scale)) eps_s, one conv_transpose per sample."""
    conv = F.conv_transpose1d if isinstance(layer, NormalConvTranspose1d) else F.conv_transpose2d
    x = x.detach().double().clone().requires_grad_(True)
    params = [layer.weight.mean, layer.weight.scale] + ([layer.bias.mean, layer.bias.scale] if layer.bias is not None else [])
    p64 = [p.detach().double().clone().requires_grad_(True) for p in params]
    B = x.shape[0] if shared else x.shape[0] // S
    ys = []
    for s in range(S):
        W = p64[0] + (1e-10 + F.softplus(p64[1])) * eps_w[s].double()
        b = p64[2] + (1e-10 + F.softplus(p64[3])) * eps_b[s].double() if layer.bias is not None else None
        xs = x if shared else x[s * B:(s + 1) * B]
        ys.append(conv(xs, W, b, layer.stride, layer.padding, layer.output_padding, layer.groups, layer.dilation))
    y = torch.cat(ys)
    (y * gy.double()).sum().backward()
    return y, [x.grad] + [p.grad for p in p64]


# (Cin, Cout, k, stride, padding, output_padding, dilation, groups, H, W, S, shared)
CASES = [
    (32, 32, 4, 2, 1, 0, 1, 1, 5, 6, 3, False),          # the decoder layer: k4 s2 p1
    (64, 32, 3, 2, 1, 1, 1, 1, 7, 5, 3, True),           # k3 s2 p1 op1, shared input
    (32, 64, 3, 3, 0, 2, 1, 1, 4, 4, 1, False),          # stride 3, uneven phases
    (32, 32, 5, 2, 2, 1, 2, 1, 6, 5, 3, False),          # dilation 2 with stride 2
    (32, 32, 3, (2, 1), 1, (1, 0), 1, 1, 5, 6, 3, True),  # stride (2, 1)
    (128, 32, 2, 2, 0, 0, 1, 1, 4, 4, 16, False),        # k2 s2, S = 16
    (32, 32, 1, 2, 0, 1, 1, 1, 4, 5, 3, False),          # k < s: bias-only phases
    (32, 32, 3, 3, 1, 0, 1, 1, 3, 4, 3, True),           # k = s with padding
    (32, 32, 3, 1, 1, 0, 2, 1, 6, 6, 3, False),          # stride 1, dilation 2
    (32, 32, 3, 1, 0, 1, 2, 1, 5, 5, 3, False),          # output_padding >= stride (below dilation)
    (48, 32, 3, 2, 1, 1, 1, 1, 5, 5, 3, False),          # Cin % 32 != 0: explicit forward, implicit backward
    (17, 64, 4, 2, 1, 0, 1, 1, 5, 5, 3, True),
    (32, 3, 4, 2, 1, 0, 1, 1, 5, 5, 3, True),            # RGB output: NCHW lowering
    (32, 17, 3, 2, 1, 1, 1, 1, 4, 6, 3, False),
    (32, 48, 3, 3, 1, 2, 1, 2, 4, 4, 3, False),          # groups 2
    (64, 64, 3, 2, 1, 1, 2, 4, 5, 5, 3, True),           # groups 4, dilation 2
    (16, 3, 5, 1, 2, 0, 1, 1, 6, 6, 16, False),
]


@pytest.mark.parametrize("prec", ["fp32", "tf32"])
@pytest.mark.parametrize("case", CASES, ids=[str(i) for i in range(len(CASES))])
def test_conv_transpose2d_parity(case, prec):
    Cin, Cout, k, s, p, op, d, g, H, W, S, shared = case
    bnn.set_precision(prec)
    torch.manual_seed(hash(case) % 1000)
    layer = NormalConvTranspose2d(Cin, Cout, k, stride=s, padding=p, output_padding=op, groups=g, dilation=d).cuda()
    B = 2
    x = torch.randn((B if shared else S * B), Cin, H, W, device="cuda")
    eps_w = torch.randn((S,) + tuple(layer.weight.mean.shape), device="cuda")
    eps_b = torch.randn(S, Cout, device="cuda")
    out = [functional.conv_transpose_out(n, k, s_, p_, o_, d_) for n, s_, p_, o_, d_ in
           zip((H, W), _pair(s), _pair(p), _pair(op), _pair(d))]
    gy = torch.randn(S * B, Cout, *out, device="cuda")
    layer.zero_grad()
    y_ref, g_ref = reference(layer, x, S, shared, eps_w, eps_b, gy)
    y, grads = run_layer(layer, x, S, shared, eps_w, eps_b, gy)
    assert y.shape == y_ref.shape and y.is_contiguous()
    assert rel_err(y, y_ref) < TOL[prec]
    for name, a, b in zip(("dx", "dmu_w", "drho_w", "dmu_b", "drho_b"), grads, g_ref):
        assert rel_err(a, b) < TOL[prec], (name, rel_err(a, b))


@pytest.mark.parametrize("prec", ["fp32", "tf32"])
def test_conv_transpose1d_parity(prec):
    bnn.set_precision(prec)
    S, B = 3, 2
    layer = NormalConvTranspose1d(32, 32, 4, stride=2, padding=1, output_padding=1).cuda()
    x = torch.randn(S * B, 32, 9, device="cuda")
    eps_w = torch.randn((S,) + tuple(layer.weight.mean.shape), device="cuda")
    eps_b = torch.randn(S, 32, device="cuda")
    gy = torch.randn(S * B, 32, 19, device="cuda")
    y_ref, g_ref = reference(layer, x, S, False, eps_w, eps_b, gy)
    y, grads = run_layer(layer, x, S, False, eps_w, eps_b, gy)
    assert y.shape == y_ref.shape
    assert rel_err(y, y_ref) < TOL[prec]
    for a, b in zip(grads, g_ref):
        assert rel_err(a, b) < TOL[prec]


@pytest.mark.parametrize("shared", [False, True])
def test_preserve_format_gives_channels_last_and_matches(shared):
    bnn.set_precision("tf32")
    bnn.set_conv_output_format("preserve")
    S, B = 3, 2
    layer = NormalConvTranspose2d(32, 64, 4, stride=2, padding=1).cuda()
    x = torch.randn((B if shared else S * B), 32, 6, 5, device="cuda").contiguous(memory_format=torch.channels_last)
    eps_w = torch.randn((S,) + tuple(layer.weight.mean.shape), device="cuda")
    eps_b = torch.randn(S, 64, device="cuda")
    gy = torch.randn(S * B, 64, 12, 10, device="cuda").contiguous(memory_format=torch.channels_last)
    y, grads = run_layer(layer, x, S, shared, eps_w, eps_b, gy)
    assert y.is_contiguous(memory_format=torch.channels_last)
    layer.zero_grad()
    y_ref, g_ref = reference(layer, x, S, shared, eps_w, eps_b, gy)
    assert rel_err(y, y_ref) < TOL["tf32"]
    for a, b in zip(grads, g_ref):
        assert rel_err(a, b) < TOL["tf32"]


@pytest.mark.parametrize("case", [CASES[0], CASES[1], CASES[2], CASES[6], CASES[9]], ids=["k4s2", "op1", "s3", "k1s2", "d2"])
def test_implicit_and_explicit_paths_agree_in_tf32(case, monkeypatch):
    Cin, Cout, k, s, p, op, d, g, H, W, S, shared = case
    bnn.set_precision("tf32")
    layer = NormalConvTranspose2d(Cin, Cout, k, stride=s, padding=p, output_padding=op, dilation=d).cuda()
    assert layer._implicit
    x = torch.randn((2 if shared else 2 * S), Cin, H, W, device="cuda")
    eps_w = torch.randn((S,) + tuple(layer.weight.mean.shape), device="cuda")
    eps_b = torch.randn(S, Cout, device="cuda")
    y0, _ = run_layer(layer, x, S, shared, eps_w, eps_b, torch.zeros(1, device="cuda"))
    gy = torch.randn(y0.shape, device="cuda")
    layer.zero_grad()
    launches = _C.launch_count
    y_k, g_k = run_layer(layer, x, S, shared, eps_w, eps_b, gy)
    assert _C.launch_count > launches
    g_k = [t.clone() for t in g_k]
    for name in ("try_sampled_conv_transpose2d_fwd", "try_sampled_conv_transpose2d_dgrad",
                 "try_sampled_conv_transpose2d_wgrad"):
        monkeypatch.setattr(_C, name, lambda *a, **k: False)
    layer.zero_grad()
    y_e, g_e = run_layer(layer, x, S, shared, eps_w, eps_b, gy)
    assert rel_err(y_k, y_e) < 2e-3
    for a, b in zip(g_k, g_e):
        assert rel_err(a, b) < 2e-3


def test_kernel_path_is_taken_in_tf32(monkeypatch):
    """The TF32 forward of an eligible layer is the phase-decomposed gather, not the explicit lowering."""
    bnn.set_precision("tf32")
    layer = NormalConvTranspose2d(64, 64, 4, stride=2, padding=1).cuda()
    calls = []
    monkeypatch.setattr(_C, "col2im_nhwc", lambda *a, **k: calls.append("col2im"))
    real = _C.try_sampled_conv_transpose2d_fwd
    monkeypatch.setattr(_C, "try_sampled_conv_transpose2d_fwd", lambda *a: calls.append("gather") or real(*a))
    layer(torch.randn(4, 64, 8, 8, device="cuda"))
    assert calls == ["gather"]


@pytest.mark.parametrize("prec", ["fp32", "tf32"])
def test_bias_only_phases(prec):
    """k < s: phases without a tap hold exactly the sampled bias."""
    bnn.set_precision(prec)
    layer = NormalConvTranspose2d(32, 32, 1, stride=3, output_padding=2).cuda()
    x = torch.randn(2, 32, 4, 4, device="cuda")
    y = layer(x)
    w, b = layer.sampled
    ref = F.conv_transpose2d(x.double(), w.double(), b.double(), 3, 0, 2)
    assert rel_err(y, ref) < TOL[prec]
    assert torch.allclose(y[:, :, 1::3, 2::3], b.view(1, -1, 1, 1).expand(2, 32, 4, 4), atol=1e-6)


@pytest.mark.parametrize("cfg", [(32, 64, 4, 2, 1, 0), (64, 3, 3, 2, 1, 1), (32, 32, 3, 1, 1, 0)])
@pytest.mark.parametrize("prec", ["fp32", "tf32"])
def test_philox_forward_equals_torch_on_sampled(cfg, prec):
    Cin, Cout, k, s, p, op = cfg
    bnn.set_precision(prec)
    layer = NormalConvTranspose2d(Cin, Cout, k, stride=s, padding=p, output_padding=op).cuda()
    x = torch.randn(3, Cin, 7, 6, device="cuda")
    y = layer(x)
    w, b = layer.sampled
    assert rel_err(y, F.conv_transpose2d(x.double(), w.double(), b.double(), s, p, op)) < TOL[prec]
    assert torch.equal(layer(x, sample=False), y)


class Unflatten(torch.nn.Module):
    def __init__(self, shape):
        super().__init__()
        self.shape = shape

    def forward(self, x):
        return x.view((x.shape[0],) + self.shape)


bnn.nn.register_rowwise_module(Unflatten)


class Decoder(BayesianNetworkModule):
    def __init__(self, samples):
        super().__init__(1, 1, samples)
        self.layers = torch.nn.Sequential(
            NormalLinear(8, 32 * 4 * 4), Unflatten((32, 4, 4)),
            NormalConvTranspose2d(32, 32, 4, stride=2, padding=1), torch.nn.ELU(),
            NormalConvTranspose2d(32, 3, 4, stride=2, padding=1), torch.nn.Sigmoid())

    def _forward(self, x):
        return self.layers(x)


@pytest.mark.parametrize("prec", ["fp32", "tf32"])
def test_batched_decoder_equals_the_loop(prec):
    bnn.set_precision(prec)
    torch.manual_seed(11)
    proto = Decoder(4).cuda()
    x = torch.randn(5, 8, device="cuda")
    runs = []
    for mode in ("auto", "never"):
        bnn.set_mc_batching(mode)
        net = copy.deepcopy(proto)
        assert (mode == "never") or net._mc_plan()[0]
        preds = net(x)
        assert isinstance(preds, list) and len(preds) == 4 and preds[0].shape == (5, 3, 16, 16)
        torch.stack([(p - 0.5).square().sum() for p in preds]).mean().backward()
        runs.append((net, preds))
    (a, pa), (b, pb) = runs
    tol = 1e-5 if prec == "fp32" else 2e-3
    for s in range(4):
        assert rel_err(pa[s], pb[s]) < tol
    for (n1, p1), (_, p2) in zip(a.named_parameters(), b.named_parameters()):
        assert rel_err(p1.grad, p2.grad) < 10 * tol, n1


def test_whole_model_kl_prune_and_elbo_adam():
    torch.manual_seed(12)
    model = Decoder(2).cuda()
    # KL divergence: the closed form of every variational tensor, found through the traversal
    kld = KLDivergence(number_of_batches=3)
    terms = []
    for w in model.modules():
        if isinstance(w, WeightNormal):
            q = torch.distributions.Normal(w.mean.double(), 1e-10 + F.softplus(w.scale.double()))
            terms.append(torch.distributions.kl_divergence(q, torch.distributions.Normal(0.0, 0.1)).mean())
    assert len(terms) == 6
    assert float(kld(model)) == pytest.approx(float(torch.stack(terms).mean() / 3), rel=1e-5)
    # pruning reaches the transposed layers: count and idempotence
    conv = model.layers[2]
    before = conv.weight.mean.detach().clone()
    PruneNormal()(model, 0.5)
    changed = conv.weight.mean != before
    assert int(changed.sum()) == int(0.5 * before.numel()) == int((conv.weight.scale == -30).sum())
    assert bool((conv.weight.mean[changed] == 0).all())
    state = {k: v.clone() for k, v in model.state_dict().items()}
    PruneNormal()(model, 0.5)
    assert all(torch.equal(state[k], v) for k, v in model.state_dict().items())
    # ELBOAdam walks the same trajectory as torch's Adam on likelihood + KL
    ref_model, new_model = copy.deepcopy(model), copy.deepcopy(model)
    x = torch.randn(6, 8, device="cuda")
    target = torch.rand(6, 3, 16, 16, device="cuda")
    ref_opt = torch.optim.Adam(ref_model.parameters(), lr=2e-3)
    new_opt = bnn.optim.ELBOAdam(new_model, number_of_batches=3, lr=2e-3)

    def rewind(m, step):
        ids = iter(range(30_000, 40_000))
        for w in m.modules():
            if isinstance(w, WeightNormal):
                w._tensor_id, w._draw = next(ids), 2 * step

    for step in range(4):
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
        layer = NormalConvTranspose2d(32, 64, 4, stride=2, padding=1).cuda()
        sx = torch.randn(4, 32, 6, 6, device="cuda")
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
        for _ in range(3):
            g.replay()
            torch.cuda.synchronize()
            got = out.detach().clone()
            gm, gs = layer.weight.mean.grad.clone(), layer.weight.scale.grad.clone()
            outs.append(got)
            # eager step with the same device step counter value
            eager = copy.deepcopy(layer)
            eager.zero_grad(set_to_none=True)
            eager.weight._draw, eager.bias._draw = layer.weight._draw - 1, layer.bias._draw - 1
            y = eager(sx)
            y.square().sum().backward()
            tol = 1e-5 if prec == "fp32" else 2e-3
            assert rel_err(got, y) < tol
            assert rel_err(gm, eager.weight.mean.grad) < tol and rel_err(gs, eager.weight.scale.grad) < tol
            w, b = layer.sampled
            assert rel_err(got, F.conv_transpose2d(sx.double(), w.double(), b.double(), 2, 1)) < TOL[prec]
        assert not torch.equal(outs[0], outs[1])
    finally:
        bnn.graph_safe_rng(False)


def test_d1_configuration_scale_tf32():
    """D1 at full size (B = 512, S = 16, shared input, 8x8 -> 16x16, 128 -> 128 channels) against fp64 torch."""
    bnn.set_precision("tf32")
    torch.manual_seed(13)
    S, B = 16, 512
    layer = NormalConvTranspose2d(128, 128, 4, stride=2, padding=1).cuda()
    x = torch.randn(B, 128, 8, 8, device="cuda")
    eps_w = torch.randn((S,) + tuple(layer.weight.mean.shape), device="cuda")
    eps_b = torch.randn(S, 128, device="cuda")
    gy = torch.randn(S * B, 128, 16, 16, device="cuda")
    y, grads = run_layer(layer, x, S, True, eps_w, eps_b, gy)
    y = y.detach()
    layer.zero_grad()
    y_ref, g_ref = reference(layer, x, S, True, eps_w, eps_b, gy)
    assert rel_err(y, y_ref) < TOL["tf32"]
    for a, b in zip(grads, g_ref):
        assert rel_err(a, b) < TOL["tf32"]
