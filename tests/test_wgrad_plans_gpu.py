"""The TMA weight gradient (wgrad_tma_kernel, TF32 mode) on every plan it can run, against float64 torch on the same eps.

wgrad_plan_and_launch picks CTA pairs, the number of M-chunks per sample and the work units (sample, chunk) each CTA
walks from a cost model, so the suite's small shapes reach few of its plans.  bnn_debug_force_wgrad_plan forces them;
bnn_debug_wgrad_plan reports the plan a launch will run, and every forced case asserts it first.  The forced plans
include a pair whose last CTA owns no n rows (three n-tiles), units that cross sample boundaries, a short last group,
one CTA walking every sample, one chunk per 64-row stage, and odd and even units per CTA (both TMEM accumulators end
a CTA).

  a  matrix mode (bnn_sampled_gemm_wgrad): injected eps, shared and per-sample A, an unforced multi-unit plan, and the
     in-kernel Philox draw (sample_begin != 0) against the eps `.materialize` reports;
  b  rank-one sign-noise mode (Flipout): eps_s = R_s Sg_s^T;
  c  2-d conv mode: NormalConv2d with 260 output channels (stride 1, and stride 2 with dilation 2) through the layer;
  d  NormalConvTranspose2d with 260 input channels (its conv view's weight gradient has N = 260, shared_dy when the
     input is shared);
  e  3-d mode: NormalConvTranspose3d with 160 input channels, each forward / input-gradient contraction variant forced
     at the same time (kMode 3, sum_samples for a shared input).

dmu and drho start from a random base about as large as the gradient: the kernels accumulate into them (red.global.add),
so out - base must equal the reference; a tile written twice or never shows up as an error of the gradient's size.
Tolerance: the TF32 class, max |out - (base + ref)| / max |ref| < 2e-3.
"""
import pytest
import torch
import torch.nn.functional as F

import bayesianneuralnetworks_b200 as bnn
from bayesianneuralnetworks_b200 import _C, runtime
from bayesianneuralnetworks_b200.nn import NormalConv2d, NormalConvTranspose2d, NormalConvTranspose3d

pytestmark = pytest.mark.gpu

TOL = 2e-3


@pytest.fixture(autouse=True)
def _defaults():
    def reset():
        _C.force_wgrad_plan()
        _C.force_contract_variant(None)
        bnn.set_precision("fp32")
        bnn.set_mc_batching("auto")
        bnn.set_conv_output_format("contiguous")
    reset()
    yield
    reset()


def rel_err(got, ref):
    ref = ref.detach().double()
    return float((got.detach().double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def force(M, N, K, S, pair, n_chunks, per):
    """Forces the plan and checks that the launcher will run exactly it."""
    _C.force_wgrad_plan(pair, n_chunks, per)
    plan = _C.wgrad_plan(M, N, K, S)
    assert (plan["pair"], plan["n_chunks"], plan["units_per_cta"]) == (pair, n_chunks, per), plan
    return plan


def assert_reaches_the_tma_launcher(call):
    """An impossible forced plan makes the TMA launcher refuse: `call` reaches it (the register-staged kernels would not
    look at the plan)."""
    _C.force_wgrad_plan(units_per_cta=1 << 30)
    with pytest.raises(_C.BnnError, match="units_per_cta"):
        call()
    _C.force_wgrad_plan()


# ------------------------------------------------------------------------------------------------ a, b: matrix modes
def wgrad_ref(a, dy, rho, eps):
    """float64: sum_s G_s and sum_s G_s o eps_s * sigmoid(rho), G_s = dy_s^T a_s."""
    S = dy.shape[0]
    G = torch.bmm(dy.double().transpose(1, 2), a.double().expand(S, -1, -1))            # [S, N, K]
    return G.sum(0), (G * eps.double()).sum(0) * torch.sigmoid(rho.double())


def random_base(ref, gen):
    return (torch.randn(ref.shape, generator=gen, device="cuda") * (float(ref.abs().max()) / 4)).float()


def run_wgrad(a, dy, rho, eps, base, rng, sample_begin=0):
    S, M, N = dy.shape
    K = a.shape[2]
    dmu, drho = base[0].clone(), base[1].clone()
    _C.sampled_gemm_wgrad(_C.make_view(dy.data_ptr(), N, 1), M * N, a, K, 0 if a.shape[0] == 1 else M * K, rho, eps, dmu,
                          drho, M, N, K, S, sample_begin, rng, 0)
    torch.cuda.synchronize()
    return dmu, drho


def matrix_case(M, N, K, S, shared, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    a = torch.randn((1 if shared else S, M, K), generator=g, device="cuda")
    dy = torch.randn((S, M, N), generator=g, device="cuda")
    rho = torch.randn((N, K), generator=g, device="cuda") * 0.15 - 2.0
    eps = torch.randn((S, N, K), generator=g, device="cuda")
    return a, dy, rho, eps, g


def check(out, base, ref):
    for name, o, b, r in zip(("dmu", "drho"), out, base, ref):
        err = float((o.double() - (b.double() + r)).abs().max() / r.abs().max())
        assert err < TOL, (name, err)


# (M, N, K, S, shared A): three n-tiles (the pair grid's fourth CTA owns no rows), K = 100 (the last 32-column group
# holds 4 columns), M % 64 = 40; and 33 stages of which the last holds 52 rows, shared A
MATRIX_SHAPES = [(1000, 260, 100, 5, False), (2100, 136, 96, 7, True)]
# (n_chunks, units per CTA) for each shape: units crossing sample boundaries with a short last group (odd), an even
# count, one CTA group walking every sample, one chunk per stage
MATRIX_PLANS = {(1000, 260, 100, 5): [(4, 3), (2, 4), (1, 5), (16, 1)],
                (2100, 136, 96, 7): [(4, 3), (3, 6), (1, 7), (33, 1)]}


@pytest.mark.parametrize("pair", [1, 0])
@pytest.mark.parametrize("M,N,K,S,shared", MATRIX_SHAPES)
def test_matrix_mode_on_forced_plans(M, N, K, S, shared, pair):
    a, dy, rho, eps, g = matrix_case(M, N, K, S, shared, seed=M + pair)
    ref = wgrad_ref(a, dy, rho, eps)
    base = [random_base(r, g) for r in ref]
    rng = _C.make_rng(0, 0, 0)
    assert_reaches_the_tma_launcher(lambda: run_wgrad(a, dy, rho, eps, base, rng))
    for n_chunks, per in MATRIX_PLANS[(M, N, K, S)]:
        plan = force(M, N, K, S, pair, n_chunks, per)
        out = run_wgrad(a, dy, rho, eps, base, rng)
        try:
            check(out, base, ref)
        except AssertionError as e:
            raise AssertionError(f"plan {plan}: {e}") from None


def test_matrix_mode_unforced_multi_unit_plan():
    """A shape whose own plan has single CTAs walking several units (TMEM double buffer, sums carried across units)."""
    M, N, K, S = 1024, 512, 1024, 16
    plan = _C.wgrad_plan(M, N, K, S)
    assert plan["pair"] == 0 and plan["units_per_cta"] > 1, plan
    a, dy, rho, eps, g = matrix_case(M, N, K, S, False, seed=21)
    ref = wgrad_ref(a, dy, rho, eps)
    base = [random_base(r, g) for r in ref]
    check(run_wgrad(a, dy, rho, eps, base, _C.make_rng(0, 0, 0)), base, ref)


def test_matrix_mode_philox_on_a_forced_multi_unit_pair_plan():
    """In-kernel Philox with sample_begin = 5 and elem_offset = 8 on a pair plan whose CTAs walk units of several
    samples: the same as the call on the eps `.materialize` reports for that key (atomics may reorder the sums)."""
    M, N, K, S = 1000, 260, 100, 5
    a, dy, rho, _, g = matrix_case(M, N, K, S, False, seed=22)
    rng = _C.make_rng(0xC0FFEE, 3, 17, elem_offset=8)
    _, eps = _C.materialize(torch.zeros(N, K, device="cuda"), torch.ones(N, K, device="cuda"), S, 5, rng, want_eps=True)
    ref = wgrad_ref(a, dy, rho, eps)
    base = [random_base(r, g) for r in ref]
    force(M, N, K, S, 1, 4, 3)
    check(run_wgrad(a, dy, rho, eps, base, rng, sample_begin=5), base, ref)
    zero = [torch.zeros_like(b) for b in base]
    inj = run_wgrad(a, dy, rho, eps, zero, rng, sample_begin=5)
    phx = run_wgrad(a, dy, rho, None, zero, rng, sample_begin=5)
    for name, p, i in zip(("dmu", "drho"), phx, inj):
        assert rel_err(p, i) < 1e-6, name


@pytest.mark.parametrize("pair", [1, 0])
@pytest.mark.parametrize("shared", [True, False])
def test_sign_noise_mode_on_forced_plans(shared, pair):
    """Flipout's rank-one sign noise eps_s = R_s Sg_s^T, regenerated per sample by the epilogue of each unit."""
    M, N, K, S = 700, 260, 96, 3
    a, dy, rho, _, g = matrix_case(M, N, K, S, shared, seed=30 + pair)
    R = (torch.randint(0, 2, (S, N), generator=g, device="cuda") * 2 - 1).float()
    Sg = (torch.randint(0, 2, (S, K), generator=g, device="cuda") * 2 - 1).float()
    ref = wgrad_ref(a, dy, rho, R.unsqueeze(2) * Sg.unsqueeze(1))
    base = [random_base(r, g) for r in ref]
    rng = _C.make_rng(0, 0, 0, signs=(R, Sg))
    for n_chunks, per in [(2, 3), (1, 2)]:              # 11 stages: 6 + 5 with units across samples; whole samples
        plan = force(M, N, K, S, pair, n_chunks, per)
        try:
            check(run_wgrad(a, dy, rho, None, base, rng), base, ref)
        except AssertionError as e:
            raise AssertionError(f"plan {plan}: {e}") from None


# ------------------------------------------------------------------------------------------------ c, d, e: conv layers
@pytest.fixture
def wgrad_calls(monkeypatch):
    """Wraps the conv weight-gradient entry points: fills the layer's zeroed dmu / drho with a random base before the
    kernel and takes it off afterwards, so the layer's gradients are right only if the kernel accumulated into the base;
    records whether the kernel took the request."""
    calls = []
    scale = {}
    gen = torch.Generator(device="cuda").manual_seed(99)

    def wrap(name):
        real = getattr(_C, name)

        def wrapped(*a):
            dmu, drho = a[5], a[6]
            base = [torch.randn(t.shape, generator=gen, device="cuda") * scale.get(i, 1.0)
                    for i, t in enumerate((dmu, drho))]
            dmu.copy_(base[0])
            drho.copy_(base[1])
            ok = real(*a)
            ok = True if ok is None else ok
            if ok:
                dmu.sub_(base[0])
                drho.sub_(base[1])
            calls.append(ok)
            return ok
        monkeypatch.setattr(_C, name, wrapped)
    for name in ("try_sampled_conv2d_wgrad", "try_sampled_conv_transpose2d_wgrad", "sampled_conv_transpose3d_wgrad"):
        wrap(name)
    return calls, scale


def layer_pass(layer, x, S, B, shared, eps_w, eps_b, dy):
    """The layer in a batched Monte-Carlo pass of S samples with injected eps; y and the gradients of x and the
    parameters."""
    layer.zero_grad(set_to_none=True)
    x = x.detach().clone().requires_grad_(True)
    ctx = runtime.MCContext(S, B)
    ctx.expanded = not shared
    with bnn.injected_eps({layer.weight: eps_w, layer.bias: eps_b}), runtime.mc_batch(ctx):
        y = layer(x)
    y.backward(dy)
    return y, [x.grad, layer.weight.mean.grad, layer.weight.scale.grad, layer.bias.mean.grad, layer.bias.scale.grad]


def layer_reference(layer, x, S, B, shared, eps_w, eps_b, gen):
    """float64 torch, one convolution per sample with W_s = mean + (1e-10 + softplus(scale)) eps_s: the output, a random
    output gradient dy and the gradients it gives."""
    xd = x.detach().double().requires_grad_(True)
    p = [t.detach().double().requires_grad_(True) for t in (layer.weight.mean, layer.weight.scale, layer.bias.mean,
                                                              layer.bias.scale)]
    outs = []
    for s in range(S):
        w = p[0] + (1e-10 + F.softplus(p[1])) * eps_w[s].double()
        b = p[2] + (1e-10 + F.softplus(p[3])) * eps_b[s].double()
        xs = xd if shared else xd[s * B:(s + 1) * B]
        if isinstance(layer, NormalConv2d):
            outs.append(F.conv2d(xs, w, b, layer.stride, layer.padding, layer.dilation))
        else:
            conv = F.conv_transpose3d if isinstance(layer, NormalConvTranspose3d) else F.conv_transpose2d
            outs.append(conv(xs, w, b, layer.stride, layer.padding, layer.output_padding, 1, layer.dilation))
    ref = torch.cat(outs)
    dy = torch.randn(ref.shape, generator=gen, device="cuda")
    ref.backward(dy.double())
    return ref, dy, [xd.grad] + [t.grad for t in p]


def layer_parity(layer, in_shape, S, B, shared, plan, wgrad_calls, seed):
    """Forced weight-gradient plan (M, N, K, pair, n_chunks, per) on one layer pass in TF32 against fp64 torch."""
    calls, scale = wgrad_calls
    bnn.set_precision("tf32")
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn((B if shared else S * B,) + tuple(in_shape), generator=g, device="cuda")
    eps_w = torch.randn((S,) + tuple(layer.weight.mean.shape), generator=g, device="cuda")
    eps_b = torch.randn((S,) + tuple(layer.bias.mean.shape), generator=g, device="cuda")
    ref, dy, ref_grads = layer_reference(layer, x, S, B, shared, eps_w, eps_b, g)
    scale[0] = float(ref_grads[1].abs().max()) / 4
    scale[1] = float(ref_grads[2].abs().max()) / 4
    M, N, K, pair, n_chunks, per = plan
    force(M, N, K, S, pair, n_chunks, per)
    del calls[:]
    y, grads = layer_pass(layer, x, S, B, shared, eps_w, eps_b, dy)
    assert calls == [True], calls
    assert y.shape == ref.shape and rel_err(y, ref) < TOL
    for name, got, want in zip(("dx", "d mean_w", "d scale_w", "d mean_b", "d scale_b"), grads, ref_grads):
        err = rel_err(got, want)
        assert err < TOL, (name, err)


# NormalConv2d(32, 260, 3): N = 260 (three n-tiles), K = 9 x 32 = 288; 2 x 24 x 24 = 1152 rows (18 stages) per sample
CONV2D = [dict(stride=1, padding=1, dilation=1, hw=24), dict(stride=2, padding=2, dilation=2, hw=48)]


@pytest.mark.parametrize("pair,n_chunks,per", [(1, 3, 2), (0, 3, 2), (1, 2, 3), (0, 2, 3)])
@pytest.mark.parametrize("shared", [True, False])
@pytest.mark.parametrize("cfg", CONV2D, ids=["s1", "s2d2"])
def test_conv2d_mode_on_forced_plans(cfg, shared, pair, n_chunks, per, wgrad_calls):
    S, B = 3, 2
    layer = NormalConv2d(32, 260, 3, stride=cfg["stride"], padding=cfg["padding"], dilation=cfg["dilation"]).cuda()
    layer_parity(layer, (32, cfg["hw"], cfg["hw"]), S, B, shared, (B * 24 * 24, 260, 288, pair, n_chunks, per),
                 wgrad_calls, seed=40 + pair + 2 * n_chunks)


@pytest.mark.parametrize("pair,n_chunks,per", [(1, 3, 2), (0, 2, 3)])
@pytest.mark.parametrize("shared", [True, False])
def test_conv_transpose2d_mode_on_forced_plans(shared, pair, n_chunks, per, wgrad_calls):
    """The weight gradient of NormalConvTranspose2d(260, 32, 4, stride 2) is its conv view's: N = in_channels = 260,
    K = 16 x 32, M = 2 x 24 x 24 input pixels; a shared input is read as sample 0 of dY by every sample (shared_dy)."""
    S, B = 3, 2
    layer = NormalConvTranspose2d(260, 32, 4, stride=2, padding=1).cuda()
    layer_parity(layer, (260, 24, 24), S, B, shared, (B * 24 * 24, 260, 512, pair, n_chunks, per), wgrad_calls,
                 seed=50 + pair)


@pytest.fixture
def gathers(monkeypatch):
    seen = []
    real = _C.try_sampled_conv_transpose3d_fwd
    monkeypatch.setattr(_C, "try_sampled_conv_transpose3d_fwd", lambda *a: seen.append(real(*a)) or seen[-1])
    return seen


# NormalConvTranspose3d(160, 32, ...): N = 160 (two n-tiles), 2 x 8 x 8 x 9 = 1152 input voxels (18 stages) per sample,
# more than 512 output rows per phase and sample (the forced contraction pair needs more than 4 row blocks)
CONV3D = [dict(kernel_size=2, stride=2, padding=0, K=8 * 32), dict(kernel_size=3, stride=1, padding=1, K=27 * 32)]


@pytest.mark.parametrize("variant,pair", [("pair", 1), ("mb4", 0), ("mb2", 1), ("mb1", 0)])
@pytest.mark.parametrize("shared", [True, False])
@pytest.mark.parametrize("cfg", CONV3D, ids=["k2s2", "k3s1p1"])
def test_conv_transpose3d_mode_on_forced_plans_and_contraction_variants(cfg, shared, variant, pair, wgrad_calls,
                                                                       gathers):
    """3-d mode of the weight gradient on forced plans, and each forward / input-gradient contraction variant forced
    through kMode 3 at the same time: the forward phases, and the input gradient (the conv view's forward, summing the
    samples inside the kernel for a shared input)."""
    S, B = 3, 2
    _C.force_contract_variant(variant)
    layer = NormalConvTranspose3d(160, 32, cfg["kernel_size"], stride=cfg["stride"], padding=cfg["padding"]).cuda()
    layer_parity(layer, (160, 8, 8, 9), S, B, shared, (B * 8 * 8 * 9, 160, cfg["K"], pair, 3, 2), wgrad_calls,
                 seed=60 + pair)
    assert gathers and all(gathers), gathers
