"""CPU tests of the host-side mirror of the reference interface: traversal semantics (reference
tests/test_utils.py), containers (tests/test_nn/test_container.py), constructor contracts, state_dict
layout, the Monte-Carlo batching plan, draw bookkeeping — and that the C-ABI library loads and exports
every symbol include/bnn_b200.h declares.  No kernel is launched."""
import ctypes
import os
import re

import pytest
import torch

import bayesianneuralnetworks_b200 as bnn
from bayesianneuralnetworks_b200 import _C, runtime
from bayesianneuralnetworks_b200.nn import (BayesianModule, BayesianNetworkModule, NormalConv1d, NormalConv2d,
                                            NormalConv3d, NormalLinear, WeightNormal)
from bayesianneuralnetworks_b200.utils import _item_or_list, _pair, _single, _triple, apply_wb, traverse

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class Net(BayesianNetworkModule):
    def __init__(self, seq, samples=1):
        super().__init__(1, 1, samples)
        self.layers = seq

    def _forward(self, x):
        return self.layers(x)


# ------------------------------------------------------------------------------------------------ C ABI
def test_header_symbols_are_exported_by_the_library():
    header = open(os.path.join(ROOT, "include", "bnn_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(bnn_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    assert os.path.exists(_C.LIB_PATH), "libbnn_b200.so missing: run `python -m bayesianneuralnetworks_b200._build`"
    lib = ctypes.CDLL(_C.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/bnn_b200.h but not exported"
    assert declared == set(_C.EXPORTED_SYMBOLS), "ctypes binding and header disagree"
    assert _C.lib().bnn_abi_version() == 1
    assert isinstance(_C.lib().bnn_last_error_string(), bytes)


def test_binding_struct_sizes_match_the_header():
    assert ctypes.sizeof(_C.bnn_rng) == 64
    assert ctypes.sizeof(_C.bnn_view) == 24
    assert ctypes.sizeof(_C.bnn_conv2d_geom) == 64
    assert ctypes.sizeof(_C.bnn_kl_tensor) == 56
    assert ctypes.sizeof(_C.bnn_prune_tensor) == 56
    assert ctypes.sizeof(_C.bnn_prune_into_tensor) == 80
    assert ctypes.sizeof(_C.bnn_adam_tensor) == 88


def test_hot_path_rejects_cpu_tensors():
    layer = NormalLinear(3, 2)
    with pytest.raises(RuntimeError, match="CUDA"):
        layer(torch.zeros(1, 3))
    with pytest.raises(RuntimeError, match="CUDA"):
        layer.weight.sampled
    with pytest.raises(RuntimeError, match="CUDA"):
        bnn.prune.PruneNormal()(Net(torch.nn.Sequential(layer)), 0.5)


# ------------------------------------------------------------------------------------------------ utils
def test_item_or_list_and_ntuples():
    """reference tests/test_utils.py:6-24."""
    assert _item_or_list([1]) == 1 and _item_or_list([1, 2]) == [1, 2] and _item_or_list([]) == []
    assert _single(3) == (3,) and _pair(3) == (3, 3) and _triple(3) == (3, 3, 3)
    assert _pair((1, 2)) == (1, 2) and _pair([1, 2, 3]) == [1, 2, 3]      # iterables pass through unchecked


def test_apply_wb_semantics():
    """reference tests/test_utils.py:27-50."""
    m = NormalLinear(3, 3)
    assert apply_wb(m, lambda p: p.shape) == [(3, 3), (3,)]
    assert apply_wb(m, lambda p: None) is None
    assert apply_wb(m, lambda p, type: type, pass_type=True) == ['w', 'b']
    assert apply_wb(m, lambda p, module: module, pass_module=True) == [m, m]
    assert apply_wb(NormalLinear(3, 3, False), lambda p, type: type, pass_type=True) == ['w']
    assert apply_wb(m, lambda p, a, b=0: a + b, 1, b=2) == [3, 3]


def test_traverse_semantics():
    """reference tests/test_utils.py:53-65 and utils.py:50-67."""
    a, b = NormalLinear(3, 3), NormalConv2d(3, 4, 3)
    assert traverse(torch.nn.Linear(3, 3), lambda m: [1]) is None
    assert traverse(a, lambda m: [m]) == [a]
    assert traverse(a, lambda m: m) is None                      # non-list results are dropped
    seq = torch.nn.Sequential(a, torch.nn.ReLU(), torch.nn.Sequential(b), torch.nn.ModuleList([a]))
    assert traverse(seq, lambda m: [m]) == [a, b, a]             # registration order, nested containers
    assert traverse(torch.nn.Sequential(torch.nn.ReLU()), lambda m: [m]) is None

    class Block(torch.nn.Module):                                # not a traversed container type
        def __init__(self):
            super().__init__()
            self.inner = NormalLinear(3, 3)
    assert traverse(torch.nn.Sequential(Block()), lambda m: [m]) is None
    net = Net(torch.nn.Sequential(a, b))
    assert net.traverse(lambda m: [type(m).__name__]) == ['NormalLinear', 'NormalConv2d']


# ------------------------------------------------------------------------------------------------ containers / ctors
def test_containers():
    """reference tests/test_nn/test_container.py:16-33."""
    p, bp = torch.distributions.Normal(0, 1), torch.distributions.Normal(0, 2)
    m = BayesianModule(3, 4, p)
    assert (m.in_channels, m.out_channels, m.weight_prior, m.bias_prior) == (3, 4, p, p)
    assert BayesianModule(3, 4, p, bp).bias_prior is bp
    n = BayesianNetworkModule(3, 4, samples=7)
    assert (n.in_channels, n.out_channels, n.samples) == (3, 4, 7)
    with pytest.raises(NotImplementedError):
        n(torch.zeros(1, 3))


def test_constructor_signatures_and_state_dict_layout():
    lin = NormalLinear(3, 4, True, torch.distributions.Normal(0, 1))
    assert lin.weight.shape == (4, 3) and lin.bias.shape == (4,)
    assert float(lin.weight_prior.scale) == 1.0 and lin.bias_prior is lin.weight_prior
    quirk = NormalLinear(3, 3, torch.distributions.Normal(0, 1))      # reference tests/conftest.py:91 passes the
    assert quirk.bias is not None and float(quirk.weight_prior.scale) == pytest.approx(0.1)   # prior as `bias`
    c1, c2, c3 = NormalConv1d(4, 6, 3, groups=2), NormalConv2d(4, 6, 3, 2, 1, 1, 2, False), NormalConv3d(2, 2, (1, 2, 3))
    assert c1.weight.shape == (6, 2, 3) and c1.kernel_size == (3,) and c1.stride == (1,)
    assert c2.weight.shape == (6, 2, 3, 3) and c2.bias is None and c2.stride == (2, 2) and c2.groups == 2
    assert c3.weight.shape == (2, 2, 1, 2, 3) and c3.padding == (0, 0, 0) and not c3.transposed
    with pytest.raises(ValueError):
        NormalConv2d(3, 4, 3, groups=2)
    net = Net(torch.nn.Sequential(torch.nn.Conv2d(1, 2, 3), c2, lin))
    assert sorted(net.state_dict().keys()) == sorted([
        'layers.0.weight', 'layers.0.bias', 'layers.1.weight.mean', 'layers.1.weight.scale',
        'layers.2.weight.mean', 'layers.2.weight.scale', 'layers.2.bias.mean', 'layers.2.bias.scale'])
    # reference initialisation (dense.py:34-44): scale ~ N(-2, 0.15), |mean| <= 1/sqrt(fan_in)
    big = NormalLinear(400, 300)
    assert abs(float(big.weight.scale.mean()) + 2.0) < 0.01 and abs(float(big.weight.scale.std()) - 0.15) < 0.01
    assert float(big.weight.mean.abs().max()) <= 1 / 20 + 1e-6 and float(big.bias.mean.abs().max()) <= 1 / 20 + 1e-6


def test_draw_bookkeeping_and_partition_arithmetic():
    w = WeightNormal(3, 3)
    d0 = w._draw
    assert d0 == 1                               # the constructor's sample() (core.py:15)
    w.sample()
    assert w._last == (d0, 1) and w._draw == d0 + 1
    begin = w.advance(4, offset=8, total=16)     # rank 2 of 4, 4 samples each
    assert begin == d0 + 1 + 8 and w._last == (begin, 4) and w._draw == d0 + 17
    spec = w.draw_spec((1 << 32) + 5, 2)
    assert spec.sample_begin == 5 and spec.step == 1 and spec.tensor_id == w._tensor_id
    assert WeightNormal(2)._tensor_id != w._tensor_id
    with pytest.raises(ValueError):
        bnn.set_sample_partition(2, 2)
    with pytest.raises(ValueError):
        bnn.set_precision("bf16")


def test_mc_batching_plan():
    ok = Net(torch.nn.Sequential(torch.nn.Conv2d(1, 2, 3), torch.nn.BatchNorm2d(2), torch.nn.ELU(),
                                 NormalConv2d(2, 2, 3), torch.nn.Flatten(), NormalLinear(8, 3),
                                 torch.nn.Softmax(dim=-1)), samples=4)
    plan = ok._mc_plan()
    assert plan.ok and len(plan.bns) == 1 and not plan.probes
    ok.eval()
    assert ok._mc_plan().ok and ok._mc_plan().bns == []
    ok.layers[1].train()                          # a per-submodule toggle invalidates the cached plan
    assert len(ok._mc_plan().bns) == 1
    no_stats = Net(torch.nn.Sequential(torch.nn.BatchNorm1d(3, track_running_stats=False), NormalLinear(3, 3))).eval()
    assert len(no_stats._mc_plan().bns) == 1      # batch statistics even in eval mode: guarded
    assert not Net(torch.nn.Sequential(torch.nn.Linear(3, 3)))._mc_plan()[0]             # nothing Bayesian
    assert not Net(torch.nn.Sequential(NormalLinear(3, 3), torch.nn.Softmax(dim=0)))._mc_plan()[0]
    assert not Net(torch.nn.Sequential(torch.nn.Dropout(0.5), NormalLinear(3, 3)))._mc_plan()[0]

    class Custom(torch.nn.Module):
        def forward(self, x):
            return x.view(x.size(0), -1)
    probed = Net(torch.nn.Sequential(Custom(), NormalLinear(3, 3)))._mc_plan()
    assert probed.ok and len(probed.probes) == 1          # unknown stateless leaf: eligible, probed at run time
    bnn.nn.register_rowwise_module(Custom)
    registered = Net(torch.nn.Sequential(Custom(), NormalLinear(3, 3)))._mc_plan()
    assert registered.ok and not registered.probes
    bnn.nn.container._ROWWISE.remove(Custom)

    class Stateful(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.w = torch.nn.Parameter(torch.ones(3))

        def forward(self, x):
            return x * self.w
    assert not Net(torch.nn.Sequential(Stateful(), NormalLinear(3, 3)))._mc_plan()[0]     # unknown code with state
    assert not Net(torch.nn.Sequential(NormalConv3d(2, 2, 1, groups=2)))._mc_plan()[0]    # grouped 3-d layers: no fused path
    assert Net(torch.nn.Sequential(NormalConv3d(1, 1, 1)))._mc_plan()[0]                  # groups == 1: lowering + sampled GEMM


# ------------------------------------------------------------------------------------------------ C ABI error behaviour
def test_c_abi_rejects_bad_arguments_without_a_gpu():
    """Argument validation happens before any device work: status codes and the thread-local message (no GPU needed)."""
    lib = _C.lib()
    null = ctypes.c_void_p(None)
    one = ctypes.c_void_p(16)               # never dereferenced on these paths

    def msg():
        return lib.bnn_last_error_string().decode()

    assert lib.bnn_stddev(null, null, 8, null) == 1 and "NULL" in msg()
    assert lib.bnn_stddev(null, null, -1, null) == 1
    assert lib.bnn_stddev(null, null, 0, null) == 0                       # empty input is fine
    assert lib.bnn_kl(None, -1, null, null, null, null, 0, null) == 1
    assert lib.bnn_kl(None, 0, null, null, null, null, 0, null) == 0
    table = (_C.bnn_kl_tensor * 1)()
    table[0].mu, table[0].rho, table[0].numel, table[0].prior_scale = 16, 16, 4, 1.0
    assert lib.bnn_kl(table, 1, one, null, null, null, 0, null) == 5 and "workspace" in msg()      # BNN_ERR_WORKSPACE
    need = lib.bnn_kl_workspace_size(1)
    assert lib.bnn_kl(table, 1, one, null, null, ctypes.c_void_p(8), need, null) == 2              # BNN_ERR_MISALIGNED
    table[0].prior_scale = 0.0
    assert lib.bnn_kl(table, 1, one, null, null, ctypes.c_void_p(256), need, null) == 1 and "scale" in msg()
    pt = (_C.bnn_prune_tensor * 1)()
    pt[0].mu, pt[0].rho, pt[0].numel, pt[0].k = 16, 16, 10, 11
    ws = lib.bnn_prune_workspace_size(pt, 1)
    assert ws > 0
    assert lib.bnn_prune(pt, 1, ctypes.c_void_p(256), ws, null) == 1 and "k" in msg()
    rng = _C.make_rng(1, 0, 0)
    view = _C.make_view(16, 8, 1)
    # unknown precision, negative size, bias with only one of (mu_b, sigma_b)
    assert lib.bnn_sampled_gemm_fwd(one, 8, 0, one, one, null, null, null, null, view, 0, 4, 4, 8, 1, 0,
                                    ctypes.byref(rng), None, 7, null) == 1 and "precision" in msg()
    assert lib.bnn_sampled_gemm_fwd(one, 8, 0, one, one, null, null, null, null, view, 0, -4, 4, 8, 1, 0,
                                    ctypes.byref(rng), None, 0, null) == 1
    assert lib.bnn_sampled_gemm_fwd(one, 8, 0, one, one, one, null, null, null, view, 0, 4, 4, 8, 1, 0,
                                    ctypes.byref(rng), None, 0, null) == 1 and "bias" in msg()
    assert lib.bnn_sampled_gemm_fwd(one, 8, 0, one, one, null, null, null, null, view, 0, 4, 4, 8, 70000, 0,
                                    ctypes.byref(rng), None, 0, null) == 6                          # BNN_ERR_UNSUPPORTED
    geom = _C.bnn_conv2d_geom(1, 4, 8, 8, 2, 4, 3, 3, 6, 6, 1, 1, 0, 0, 1, 1)                       # c0 + Cg > C
    assert lib.bnn_im2col(one, one, ctypes.byref(geom), null) == 1 and "geometry" in msg()
    # likelihood tail: rows must be whole sample blocks, pitches must hold a row, the workspace is checked last
    ce_ws = lib.bnn_mc_cross_entropy_workspace_size()
    assert ce_ws >= 16 + 2 * 8 * 148
    assert lib.bnn_mc_cross_entropy_fwd(one, 4, one, 10, 3, 4, -100, one, one, one, one, ce_ws, null) == 1 and "sample blocks" in msg()
    assert lib.bnn_mc_cross_entropy_fwd(one, 3, one, 9, 3, 4, -100, one, one, one, one, ce_ws, null) == 1 and "pitch" in msg()
    assert lib.bnn_mc_cross_entropy_fwd(null, 4, one, 9, 3, 4, -100, one, one, one, one, ce_ws, null) == 1 and "NULL" in msg()
    assert lib.bnn_mc_cross_entropy_fwd(one, 4, one, 0, 3, 4, -100, one, one, one, one, ce_ws, null) == 1 and "empty" in msg()
    assert lib.bnn_mc_cross_entropy_bwd(one, 4, one, 9, 3, 4, -100, one, one, one, null, 4, null) == 1 and "NULL" in msg()
    assert lib.bnn_mc_cross_entropy_bwd(one, 4, one, 9, 3, 4, -100, one, one, one, one, 2, null) == 1 and "pitch" in msg()


def test_prune_workspace_plan_and_selftest_argument_checks():
    """bnn_prune_workspace_size is a pure host function: it must cover the general path's key workspace (4 B per
    element), the deferred list of small tensors (every element: 20 B each) and grow with every tensor added; the
    interval self test validates its arguments before touching the device."""
    lib = _C.lib()
    null = ctypes.c_void_p(None)

    def size(numels):
        t = (_C.bnn_prune_tensor * len(numels))()
        for i, n in enumerate(numels):
            t[i].mu, t[i].rho, t[i].numel, t[i].k = 16, 16, n, n // 2
        return lib.bnn_prune_workspace_size(t, len(numels))

    assert lib.bnn_prune_workspace_size(None, 0) == 256
    prev = 0
    for numels in ([10], [10, 4099], [10, 4099, 65536], [10, 4099, 65536, 65537], [10, 4099, 65536, 65537, 1 << 24]):
        s = size(numels)
        assert s % 256 == 0 and s > prev
        general = sum(4 * n for n in numels)
        small = sum(20 * n for n in numels if n <= 65536)
        assert s >= max(general, small) + len(numels) * (256 + 2 * 2049 * 4)
        prev = s
    assert size([1 << 24]) < 4.2 * (1 << 24) + (1 << 20)          # no more than the key workspace plus small change
    assert size([40] * 30) > size([40] * 24)                       # more than one group of descriptors
    at = (_C.bnn_adam_tensor * 1)()
    at[0].mu, at[0].rho, at[0].numel, at[0].kl_coeff, at[0].prior_scale = 16, 16, 4, 1.0, 0.1
    assert lib.bnn_adam_kl_step(at, 1, 1e-3, 0.9, 0.999, 1e-8, null, 1, null) == 1 and "moment" in lib.bnn_last_error_string().decode()
    assert lib.bnn_adam_kl_step(at, 1, 1e-3, 1.0, 0.999, 1e-8, null, 1, null) == 1                 # beta1 = 1
    assert lib.bnn_adam_kl_step(at, 1, 1e-3, 0.9, 0.999, 1e-8, null, 0, null) == 1 and "step" in lib.bnn_last_error_string().decode()
    assert lib.bnn_adam_kl_step(None, 0, 1e-3, 0.9, 0.999, 1e-8, null, 1, null) == 0
    assert lib.bnn_selftest_prune_interval(null, null, -1, null, null, 0, null) == 1
    assert lib.bnn_selftest_prune_interval(null, null, 4, null, null, 2, null) == 1
    assert lib.bnn_selftest_prune_interval(null, null, 4, null, null, 1, null) == 1 and "NULL" in lib.bnn_last_error_string().decode()
    assert lib.bnn_selftest_prune_interval(null, null, 0, null, null, 1, null) == 0


def test_mc_mean_loss_host_logic():
    """nn.mc_mean_loss == the reference loop body torch.stack([criterion(p, y) for p in preds]).mean()
    (examples/MNIST/train.py:59-61): one call over the batched rows when the list is an MCSamples of row blocks and
    the criterion is a row mean, the loop otherwise."""
    import torch.nn.functional as F
    from bayesianneuralnetworks_b200.nn import MCSamples, mc_mean_loss
    torch.manual_seed(0)
    S, B, C = 5, 7, 4
    base = torch.randn(S * B, C, requires_grad=True)
    y = torch.randint(0, C, (B,))
    preds = MCSamples(base.view(S, B, C).unbind(0))
    preds.batched = base
    assert isinstance(preds, list) and len(preds) == S
    w = torch.tensor([0.5, 1.0, 2.0, 1.5])
    for crit in (F.cross_entropy, torch.nn.CrossEntropyLoss(), torch.nn.CrossEntropyLoss(weight=w, label_smoothing=0.1),
                 torch.nn.CrossEntropyLoss(reduction='sum'), lambda p, t: F.cross_entropy(p, t) * 2):
        ref = torch.stack([crit(p, y) for p in preds]).mean()
        got = mc_mean_loss(crit, preds, y)
        assert torch.allclose(got, ref, rtol=1e-6, atol=1e-7)
        g_ref, = torch.autograd.grad(ref, base, retain_graph=True)
        g_got, = torch.autograd.grad(got, base)
        assert torch.allclose(g_got, g_ref, rtol=1e-5, atol=1e-8)
    # regression criterion with a [B, C] target, a plain list (no batched tensor), and the bare tensor of S == 1
    t2 = torch.randn(B, C)
    assert torch.allclose(mc_mean_loss(F.mse_loss, preds, t2), torch.stack([F.mse_loss(p, t2) for p in preds]).mean())
    plain = [p.detach() for p in preds]
    assert torch.allclose(mc_mean_loss(F.cross_entropy, plain, y), torch.stack([F.cross_entropy(p, y) for p in plain]).mean())
    assert torch.equal(mc_mean_loss(F.cross_entropy, plain[0], y), F.cross_entropy(plain[0], y))


def test_fused_cross_entropy_eligibility_and_gradient_buffers():
    """Which criteria nn.mc_mean_loss may send to bnn_mc_cross_entropy (plain mean cross-entropy over class indices,
    the examples' criterion, train.py:40) and the single zeroed buffer a layer's backward accumulates into."""
    import torch.nn.functional as F
    from bayesianneuralnetworks_b200.functional import _zero_grads
    from bayesianneuralnetworks_b200.nn.elbo import _plain_cross_entropy
    assert _plain_cross_entropy(F.cross_entropy) == -100
    assert _plain_cross_entropy(torch.nn.CrossEntropyLoss()) == -100
    assert _plain_cross_entropy(torch.nn.CrossEntropyLoss(ignore_index=3)) == 3
    for other in (torch.nn.CrossEntropyLoss(weight=torch.ones(4)), torch.nn.CrossEntropyLoss(label_smoothing=0.1),
                  torch.nn.CrossEntropyLoss(reduction='sum'), torch.nn.NLLLoss(), F.nll_loss,
                  lambda p, t: F.cross_entropy(p, t)):
        assert _plain_cross_entropy(other) is None

    class Sub(torch.nn.CrossEntropyLoss):          # a subclass may override forward: not assumed to be plain
        pass
    assert _plain_cross_entropy(Sub()) is None
    grads, bias = _zero_grads((6, 4, 3, 3), 6, 'cpu')
    assert grads.shape == (2, 6, 4, 3, 3) and bias.shape == (2, 6) and not grads.any() and not bias.any()
    assert grads.is_contiguous() and bias.is_contiguous()
    assert bias.data_ptr() == grads.data_ptr() + 4 * grads.numel()         # one allocation, one fill
    assert _zero_grads(None, None, 'cpu') == (None, None)
    assert _zero_grads(None, 5, 'cpu')[0] is None and _zero_grads((2, 3), None, 'cpu')[1] is None
    with pytest.raises(RuntimeError, match="CUDA"):
        _C.mc_cross_entropy_fwd(torch.zeros(4, 3), torch.zeros(2, dtype=torch.int64))


def test_elbo_adam_plans_the_same_tensors_and_coefficients_as_kl_divergence():
    """bnn.optim.ELBOAdam folds the gradient of KLDivergence(n_batches)(model) into its step: it must see the tensors the
    reference's traverse sees (weights and biases as separate entries, loss.py:30-38), give each the coefficient
    1 / (numel * n_tensors * n_batches), and leave every other parameter to torch's Adam."""
    from torch.nn import Conv2d, ELU, Flatten, Sequential

    class Hidden(torch.nn.Module):                 # a Bayesian layer inside a plain module: invisible to traverse
        def __init__(self):
            super().__init__()
            self.inner = NormalLinear(10, 10)

        def forward(self, x):
            return self.inner(x)

    class Net(BayesianNetworkModule):
        def __init__(self):
            super().__init__(1, 10, 2)
            self.layers = Sequential(Conv2d(1, 4, 3), ELU(), NormalConv2d(4, 4, 3), Flatten(),
                                     NormalLinear(16, 10, bias=False), Hidden())

        def _forward(self, x):
            return self.layers(x)

    net = Net()
    opt = bnn.optim.ELBOAdam(net, number_of_batches=5, lr=1e-2)
    seen = [e["w"] for e in opt._var]
    assert seen == [net.layers[2].weight, net.layers[2].bias, net.layers[4].weight]
    for e in opt._var:
        assert e["coeff"] == pytest.approx(1.0 / (e["w"].mean.numel() * 3 * 5)) and (e["loc"], e["scale"]) == (0.0, pytest.approx(0.1))
    assert opt.param_groups[0]["variational"] and not opt.param_groups[1]["variational"]       # a torch Optimizer
    assert {id(p) for p in opt.param_groups[0]["params"]} == {id(p) for w in seen for p in (w.mean, w.scale)}
    others = {id(p) for p in opt.param_groups[1]["params"]}
    assert others == {id(p) for p in list(net.layers[0].parameters()) + list(net.layers[5].parameters())}
    net.layers[0].weight.grad = torch.ones_like(net.layers[0].weight)
    opt.zero_grad()
    assert net.layers[0].weight.grad is None


def test_pair_kernel_tile_plans_cover_every_row_block_exactly_once():
    """sampled_gemm_tma.cu: TilePlan.  For a sweep of (row blocks per sample, samples) the plan the launcher would use
    (bnn_debug_pair_tile_plan, host arithmetic) is decoded exactly as the kernel decodes blockIdx.x and must (1) give
    every sample a run of tiles that starts at row block 0, is contiguous and covers all of its row blocks, spilling at
    most two block pairs past the end (those rows are masked), and (2) beat the uniform grid's list schedule."""
    import ctypes
    lib = _C.lib()
    slots = 74
    n_plans = 0
    for m_blocks in list(range(5, 80)) + [128, 200]:
        for S in (3, 8, 16, 19, 30, 50, 60):
            out = (ctypes.c_int32 * 7)()
            assert lib.bnn_debug_pair_tile_plan(m_blocks, S, slots, out) == 0
            on, n_a, s1, a1, b1, a2, b2 = list(out)
            if not on:
                continue
            n_plans += 1
            n_b = s1 * b1 + (S - s1) * b2
            assert n_a == s1 * a1 + (S - s1) * a2
            tiles = {s: [] for s in range(S)}
            for t in range(n_a + n_b):                      # the kernel's decode of t = blockIdx.x >> 1
                if t < n_a:
                    first = s1 * a1
                    if t < first:
                        s, j = divmod(t, a1)
                    else:
                        q, j = divmod(t - first, a2)
                        s = s1 + q
                    tiles[s].append((j * 8, 8))
                else:
                    v, first = t - n_a, s1 * b1
                    if v < first:
                        s, j = divmod(v, b1)
                        a = a1
                    else:
                        q, j = divmod(v - first, b2)
                        s, a = s1 + q, a2
                    tiles[s].append((a * 8 + j * 6, 6))
            for s in range(S):
                run = sorted(tiles[s])
                pos = 0
                for start, size in run:
                    assert start == pos, (m_blocks, S, s, run)
                    pos += size
                assert m_blocks <= pos <= m_blocks + 5, (m_blocks, S, s, pos)      # <= 2 block pairs (+ odd block) to spare
            # list schedule: all 8-block tiles first, then the 6-block ones, against the uniform grid
            def makespan(costs):
                load = [0] * slots
                for c in costs:
                    load[load.index(min(load))] += c
                return max(load)
            uniform = S * ((((m_blocks + 1) // 2) + 3) // 4)
            assert makespan([4] * n_a + [3] * n_b) * 100 <= makespan([4] * uniform) * 92
    assert n_plans > 20
    out = (ctypes.c_int32 * 7)()
    lib.bnn_debug_pair_tile_plan(64, 16, 74, out)           # C3 conv forward: 74 + 72 tiles on 74 pair slots
    assert out[0] == 1 and out[1] + out[2] * out[4] + (16 - out[2]) * out[6] <= 148


def _wgrad_plan(M, N, K, S, sms=148):
    out = (ctypes.c_int32 * 5)()
    rc = _C.lib().bnn_debug_wgrad_plan(M, N, K, S, sms, out)
    return rc, list(out)


def _assert_wgrad_plan_covers(M, N, K, S, plan, sms=148, forced_pair=None):
    """Decodes a weight-gradient plan exactly as wgrad_tma_kernel does (per from gridDim.z, units [z per, (z + 1) per),
    unit u = chunk u % n_chunks of sample u / n_chunks, chunk c = stages [c chunk_blocks, + chunk_blocks) clipped to
    m_total): every (sample, 64-row stage) is reduced exactly once, and no CTA is launched without work."""
    import numpy as np
    pair, n_chunks, cb, per, groups = plan
    m_total = (M + 63) // 64
    units = S * n_chunks
    n_tiles = (N + 127) // 128
    tiles = n_tiles * ((K + 127) // 128)
    assert 1 <= groups <= 65535 and n_chunks >= 1 and cb >= 1
    assert per == (units + groups - 1) // groups                     # what the kernel derives from gridDim.z
    z = np.arange(groups)
    s_begin, s_end = z * per, np.minimum(z * per + per, units)
    assert (s_begin < s_end).all(), "a CTA group without work"
    assert s_begin[0] == 0 and s_end[-1] == units and (s_begin[1:] == s_end[:-1]).all()
    u = np.arange(units)
    s, mb0 = u // n_chunks, (u % n_chunks) * cb
    nb = np.minimum(cb, m_total - mb0)
    assert (nb >= 1).all(), "an empty chunk"
    diff = np.zeros((S, m_total + 1), dtype=np.int64)
    np.add.at(diff, (s, mb0), 1)
    np.add.at(diff, (s, mb0 + nb), -1)
    assert (np.cumsum(diff, axis=1)[:, :m_total] == 1).all(), "a stage reduced twice or never"
    rule = n_tiles >= 2 and tiles * groups >= 2 * sms
    if forced_pair is None:
        assert pair == int(rule)
    else:
        assert pair == forced_pair and (not pair or n_tiles >= 2)


def test_wgrad_plans_reduce_every_stage_exactly_once():
    """sampled_gemm_tma.cu: wgrad_plan, the plan wgrad_plan_and_launch runs (bnn_debug_wgrad_plan, host arithmetic).  Over
    a sweep of M (ragged, 1 to 5 stages, thousands of rows), N and K on both sides of 128 and 256, and S from 1 to 64 on
    148 SMs, and over forced plans: every (sample, stage) covered once, no empty CTA, groups <= 65535, CTA pairs only
    under their rule.  Forced values the shape cannot take are refused, and the figures DESIGN states are pinned."""
    try:
        n_plans = n_pair = n_multi = 0
        chunk_stats = set()
        for M in (1, 63, 64, 100, 150, 250, 300, 777, 1000, 2100, 2304, 4100, 8192):
            for N in (4, 100, 128, 132, 256, 260, 512):
                for K in (4, 128, 132, 256, 288, 1152):
                    for S in (1, 2, 5, 16, 64):
                        rc, plan = _wgrad_plan(M, N, K, S)
                        assert rc == 0
                        _assert_wgrad_plan_covers(M, N, K, S, plan)
                        m_total, n_chunks, cb = (M + 63) // 64, plan[1], plan[2]
                        assert n_chunks <= max(1, min((m_total + 3) // 4, 64))   # the cost model's chunk limit
                        chunk_stats.add((m_total, n_chunks, cb, m_total - (n_chunks - 1) * cb))
                        n_plans, n_pair, n_multi = n_plans + 1, n_pair + plan[0], n_multi + (plan[3] > 1)
        assert n_plans > 2000 and n_pair >= 10 and n_multi > 100
        assert (5, 2, 3, 2) in chunk_stats                        # m_total = 5 is cut 3 + 2: units may be < 4 stages
        # forced plans, including ones the cost model never picks (every sample's stages a chunk of their own, one CTA
        # group walking every unit, units that cross sample boundaries)
        forced = [((1000, 260, 100, 5), (1, 4, 3)), ((1000, 260, 100, 5), (0, 4, 3)), ((1000, 260, 100, 5), (1, 1, 5)),
                  ((1000, 260, 100, 5), (0, 16, 1)), ((2100, 136, 96, 7), (1, 4, 3)), ((2100, 136, 96, 7), (0, 33, 2)),
                  ((300, 128, 64, 3), (0, 2, 6)), ((4100, 512, 32, 64), (1, 65, 8)), ((700, 260, 96, 3), (1, 2, 3))]
        for (M, N, K, S), (pair, n_chunks, per) in forced:
            assert _C.lib().bnn_debug_force_wgrad_plan(pair, n_chunks, per) == 0
            rc, plan = _wgrad_plan(M, N, K, S)
            assert rc == 0, _C.lib().bnn_last_error_string()
            assert (plan[0], plan[1], plan[3]) == (pair, n_chunks, per), ((M, N, K, S), plan)
            _assert_wgrad_plan_covers(M, N, K, S, plan, forced_pair=pair)
        assert _C.lib().bnn_debug_force_wgrad_plan(-1, 3, -1) == 0       # one value forced, the others chosen
        rc, plan = _wgrad_plan(2304, 64, 576, 8)
        assert rc == 0 and plan[1] == 3
        _assert_wgrad_plan_covers(2304, 64, 576, 8, plan)
        # values the shape cannot take: refused with a message naming them, never another plan
        for (M, N, K, S), (pair, n_chunks, per), word in [
                ((1000, 128, 100, 5), (1, -1, -1), "pair"),              # one n-tile
                ((300, 256, 64, 3), (-1, 4, -1), "n_chunks"),            # 5 stages in chunks of 2: 3 chunks, not 4
                ((300, 256, 64, 3), (-1, 6, -1), "n_chunks"),            # more chunks than stages
                ((300, 256, 64, 3), (-1, 2, 7), "units_per_cta"),        # more than S x n_chunks = 6 units
                ((300, 256, 64, 12), (-1, 1, 5), "units_per_cta"),       # 3 groups of 5 units: the kernel would walk 4
                ((64, 256, 64, 70000), (-1, 1, 1), "units_per_cta")]:    # 70000 groups
            assert _C.lib().bnn_debug_force_wgrad_plan(pair, n_chunks, per) == 0
            rc, _ = _wgrad_plan(M, N, K, S)
            assert rc == 1 and word in _C.lib().bnn_last_error_string().decode(), ((M, N, K, S), rc)
        for bad in [(2, -1, -1), (-1, 0, -1), (-1, -1, 0), (-2, -1, -1)]:
            assert _C.lib().bnn_debug_force_wgrad_plan(*bad) == 1
    finally:
        _C.lib().bnn_debug_force_wgrad_plan(-1, -1, -1)
    # the override is gone: the figures DESIGN states
    tiles_ctas = lambda M, N, K, S: (_wgrad_plan(M, N, K, S)[1], ((N + 127) // 128) * ((K + 127) // 128))
    plan, tiles = tiles_ctas(2304, 64, 576, 8)                   # C2 conv weight gradient
    assert plan[0] == 0 and tiles * plan[4] == 120
    plan, tiles = tiles_ctas(8192, 128, 1152, 16)                # C3 conv weight gradient
    assert plan[0] == 0 and tiles * plan[4] == 144 and plan[3] == 1
    plan, _ = tiles_ctas(1024, 4096, 4096, 2)                    # C4
    assert plan[0] == 1
    plan, _ = tiles_ctas(1024, 512, 1024, 16)                    # one CTA walks several samples
    assert plan[0] == 0 and plan[3] > 1
