"""GPU parity tests of the raw C-ABI kernels (libbnn_b200.so through the ctypes binding) against
the CPU oracle (oracle/variational_oracle.py) on the same seeded inputs.

Tolerances (BASELINE.json north_star): eps-injected outputs and gradients within 1e-5 relative in
the fp32-class mode (FP32X3) and 2e-3 in TF32; prune masks bit-exact; Philox integers bit-exact
(checked through the float transform at 2e-5 absolute, the accuracy of the fast log/sincos).
Relative error is measured against the largest magnitude of the reference tensor (the scale of
the contraction), which is how a GEMM's rounding error is bounded.
"""
import hashlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import variational_oracle as orc

pytestmark = pytest.mark.gpu

TOL = {0: 2e-3, 1: 1e-5}   # bnn_precision -> relative tolerance


@pytest.fixture(scope="module")
def C():
    from bayesianneuralnetworks_b200 import _C
    _C.lib()
    assert _C.device_supported(0), "tests need a compute capability 10.x device"
    return _C


def rel_err(got, ref):
    ref = ref.double()
    scale = ref.abs().max().clamp_min(1e-30)
    return float((got.double().cpu() - ref).abs().max() / scale)


def init_params(shape, gen, fan_in=None):
    """mu ~ U(+-1/sqrt(fan_in)), rho ~ N(-2, 0.15): the reference initialisation (dense.py:34-44)."""
    fan_in = fan_in or (int(np.prod(shape[1:])) if len(shape) > 1 else shape[0])
    bound = 1.0 / np.sqrt(fan_in)
    mu = (torch.rand(shape, generator=gen) * 2 - 1) * bound
    rho = torch.randn(shape, generator=gen) * 0.15 - 2.0
    return mu, rho


# ------------------------------------------------------------------------------------------------
def test_abi_version_and_umma_selftest(C):
    assert C.abi_version() == 1
    err = C.selftest_umma()
    assert err < 1e-4, f"tcgen05 tile self test: max |err| = {err}"
    err = C.selftest_umma(mn_major=True)
    assert err < 1e-4, f"tcgen05 MN-major tile self test: max |err| = {err}"


def test_stddev_matches_oracle(C):
    g = torch.Generator().manual_seed(0)
    rho = torch.cat([torch.randn(10007, generator=g) * 3 - 2,
                     torch.tensor([-100.0, -30.0, -2.0, 0.0, 19.9, 20.0, 20.1, 50.0])])
    got = C.stddev(rho.cuda()).cpu()
    ref = orc.stddev(rho)
    assert torch.allclose(got, ref, rtol=2e-7, atol=0)
    assert got[-8] == pytest.approx(1e-10, rel=1e-6)          # rho = -100 (SURVEY appendix A1)
    assert got[-7] == pytest.approx(1.00094e-10, rel=1e-5)    # rho = -30 (pruned)


def test_materialize_injected_eps(C):
    g = torch.Generator().manual_seed(1)
    mu, rho = init_params((37, 53), g)
    eps = torch.randn(3, 37, 53, generator=g)
    sigma = C.stddev(rho.cuda())
    got = C.materialize(mu.cuda(), sigma, 3, 0, C.make_rng(1, 0, 0), eps_in=eps.cuda()).cpu()
    ref = torch.stack([orc.sample(mu, rho, eps[s]) for s in range(3)])
    assert torch.allclose(got, ref, rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("numel,offset", [(4096, 0), (1001, 0), (260, 8)])
def test_philox_stream_matches_oracle(C, numel, offset):
    seed, step, tid = 0x5EED1234ABCD, 7 + (3 << 32), 11
    mu = torch.zeros(numel, device="cuda")
    sigma = torch.ones(numel, device="cuda")
    rng = C.make_rng(seed, step, tid, elem_offset=offset)
    out, eps = C.materialize(mu, sigma, 2, 5, rng, want_eps=True)
    assert torch.equal(out, eps)                      # mu = 0, sigma = 1
    for s in range(2):
        ref = orc.philox_eps(seed, step, tid, 5 + s, numel, elem_offset=offset)
        err = np.abs(eps[s].cpu().numpy().astype(np.float64) - ref).max()
        assert err < 2e-5, f"sample {s}: max |eps - oracle| = {err}"


def test_philox_moments(C):
    n = 1 << 22
    mu = torch.zeros(n, device="cuda")
    sigma = torch.ones(n, device="cuda")
    eps = C.materialize(mu, sigma, 1, 0, C.make_rng(42, 0, 3)).double().flatten()
    # standard errors: mean 1/sqrt(n) = 4.9e-4, var sqrt(2/n) = 6.9e-4, kurt sqrt(24/n) = 2.4e-3; 5 sigma bounds
    assert abs(float(eps.mean())) < 2.5e-3
    assert abs(float(eps.var()) - 1.0) < 3.5e-3
    assert abs(float((eps ** 3).mean())) < 6e-3
    assert abs(float((eps ** 4).mean()) - 3.0) < 2.5e-2
    # different samples / tensors are uncorrelated
    e2 = C.materialize(mu, sigma, 1, 1, C.make_rng(42, 0, 3)).double().flatten()
    e3 = C.materialize(mu, sigma, 1, 0, C.make_rng(42, 0, 4)).double().flatten()
    assert abs(float((eps * e2).mean())) < 2.5e-3
    assert abs(float((eps * e3).mean())) < 2.5e-3


# ------------------------------------------------------------------------------------------------ KL
def kl_case(gen, shapes, loc=0.0, scale=0.1):
    return [init_params(s, gen) + (loc, scale) for s in shapes]


@pytest.mark.parametrize("shapes", [[(400, 784), (400,), (10, 400), (10,)], [(1,)], [(4097,), (3, 5, 7)],
                                    [(64, 64, 3, 3)] * 30])
def test_kl_sums_and_grads(C, shapes):
    g = torch.Generator().manual_seed(2)
    tensors = kl_case(g, shapes, loc=0.05, scale=0.3)
    ref_sums = orc.kl_tensor_sums(tensors)
    dev = [(m.cuda(), r.cuda()) for m, r, _, _ in tensors]
    entries = [(m, r, None, None, loc, sc, 0.0) for (m, r), (_, _, loc, sc) in zip(dev, tensors)]
    sums = C.kl(entries).cpu().tolist()
    for got, ref in zip(sums, ref_sums):
        assert got == pytest.approx(ref, rel=1e-5)
    # gradients of the reference reduction: mean over elements, mean over tensors, / n_batches
    n_batches = 7
    leaves = [(m.clone().requires_grad_(True), r.clone().requires_grad_(True)) for m, r, _, _ in tensors]
    total = orc.kl_divergence([(m, r, loc, sc) for (m, r), (_, _, loc, sc) in zip(leaves, tensors)], n_batches)
    total.backward()
    gbuf = [(torch.empty_like(m), torch.empty_like(r)) for m, r in dev]
    coeffs = [1.0 / (m.numel() * len(tensors) * n_batches) for m, _ in dev]
    entries = [(m, r, gm, gr, loc, sc, c) for (m, r), (gm, gr), (_, _, loc, sc), c in zip(dev, gbuf, tensors, coeffs)]
    sums2 = C.kl(entries).cpu().tolist()
    for got, ref in zip(sums2, ref_sums):
        assert got == pytest.approx(ref, rel=1e-5)
    for (gm, gr), (lm, lr) in zip(gbuf, leaves):
        assert rel_err(gm, lm.grad) < 1e-5
        assert rel_err(gr, lr.grad) < 1e-5
    # value of the full reduction
    got_total = sum(s / m.numel() for s, (m, _) in zip(sums, dev)) / len(dev) / n_batches
    assert got_total == pytest.approx(float(total), rel=1e-5)


def test_kl_grad_scale_and_extremes(C):
    mu = torch.tensor([0.0, 0.3, -2.0, 0.0, 1e-3, 0.5, 0.1, -0.1, 0.2])
    rho = torch.tensor([-30.0, -100.0, 25.0, 19.5, 0.0, -1.3862, -1.3864, 3.0, -10.0])
    ref = orc.kl_tensor_sums([(mu, rho, 0.0, 1.0)])[0]
    lm, lr = mu.clone().requires_grad_(True), rho.clone().requires_grad_(True)
    orc.kl_normal_elementwise(lm, lr, 0.0, 1.0).sum().backward()
    gm, gr = torch.empty(9, device="cuda"), torch.empty(9, device="cuda")
    scale = torch.tensor([0.5], device="cuda")
    s = C.kl([(mu.cuda(), rho.cuda(), gm, gr, 0.0, 1.0, 2.0)], grad_scale=scale).cpu().item()
    assert s == pytest.approx(ref, rel=1e-5)
    assert torch.allclose(gm.cpu(), lm.grad, rtol=1e-5, atol=1e-12)      # 2.0 * 0.5 = 1
    assert torch.allclose(gr.cpu(), lr.grad, rtol=2e-5, atol=1e-9)


# ------------------------------------------------------------------------------------------------ prune
def torch_keys_same_device(mu, rho):
    """The reference's key on the same device: Normal(mean, stddev).log_prob(0) (prune.py:11)."""
    torch.distributions.Distribution.set_default_validate_args(False)
    return torch.distributions.Normal(mu, 1e-10 + F.softplus(rho)).log_prob(0)


@pytest.mark.parametrize("shape,p", [((64, 64, 3, 3), 0.75), ((10, 576), 0.9), ((10,), 0.5), ((4099,), 0.0),
                                     ((4099,), 1.0), ((1000, 333), 0.3)])
def test_prune_bit_exact(C, prune_mode, shape, p):
    g = torch.Generator().manual_seed(3)
    mu, rho = init_params(shape, g)
    k = orc.prune_count(p, mu.numel())
    dmu, drho = mu.cuda(), rho.cuda()
    ref_keys = torch_keys_same_device(dmu, drho)
    mask = torch.empty(shape, dtype=torch.uint8, device="cuda")
    keys = torch.empty(shape, device="cuda")
    C.prune([(dmu, drho, k, mask, keys)])
    assert torch.equal(keys, ref_keys), "prune key differs from torch on the same device"
    # torch.topk mask on the same device (k-th key unique for these seeds -> must be identical)
    flat = ref_keys.flatten()
    ref_mask = torch.zeros_like(flat)
    if k > 0:
        ref_mask = ref_mask.scatter(0, torch.topk(flat, k).indices, 1)
    ref_mask = ref_mask.bool().view(shape)
    assert int(mask.sum()) == k
    assert torch.equal(mask.bool(), ref_mask)
    # the CPU oracle agrees too (keys differ from the CPU's by at most an ulp; masks identical
    # because the k-th key is separated from its neighbour)
    cpu_mask = orc.prune_mask_lowest_index(mu, rho, k)
    assert torch.equal(mask.bool().cpu(), cpu_mask)
    # in-place update: mean <- 0, scale <- -30 on the selected, untouched elsewhere
    em, er = orc.prune_apply(mu.clone(), rho.clone(), cpu_mask)
    assert torch.equal(dmu.cpu(), em) and torch.equal(drho.cpu(), er)
    # the request above asked for keys_out (general path); the default (sampled) path gives the same
    dmu2, drho2 = mu.cuda(), rho.cuda()
    mask2 = torch.empty(shape, dtype=torch.uint8, device="cuda")
    C.prune([(dmu2, drho2, k, mask2, None)])
    assert torch.equal(mask2, mask) and torch.equal(dmu2, dmu) and torch.equal(drho2, drho)


@pytest.mark.parametrize("numel,p", [(333000, 0.3), (333000, 0.75), (1 << 20, 0.9), (1 << 20, 0.999), (70001, 0.5),
                                     (200000, 1e-5), (200000, 0.99999)])
def test_prune_sampled_path_equals_general_path(C, prune_mode, numel, p):
    """The sampled two-sweep path and the general radix-select path are both exact: identical masks, and
    identical to the stable descending sort of torch's keys on the device."""
    g = torch.Generator().manual_seed(12)
    mu, rho = init_params((numel,), g, fan_in=400)
    k = max(1, orc.prune_count(p, numel)) if p < 0.5 else min(numel - 1, orc.prune_count(p, numel))
    ref = orc.prune_mask_from_keys(torch_keys_same_device(mu.cuda(), rho.cuda()), k)
    outs = []
    for flags in (0, C.PRUNE_GENERAL):
        dmu, drho = mu.cuda(), rho.cuda()
        mask = torch.empty(numel, dtype=torch.uint8, device="cuda")
        C.prune([(dmu, drho, k, mask, None)], flags=flags)
        assert int(mask.sum()) == k
        assert torch.equal(mask.bool(), ref)
        outs.append((dmu, drho))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    assert bool((outs[0][0][ref] == 0).all()) and bool((outs[0][1][ref] == -30).all())
    assert torch.equal(outs[0][0][~ref].cpu(), mu[~ref.cpu()])


@pytest.mark.parametrize("variant", [0, 1])
def test_prune_certified_intervals_contain_the_exact_key(C, variant):
    """The rigor of the sampled prune path rests on one claim: the fast-math interval [lo, hi] of an element contains
    the exact fp32 key that torch's op order produces (prune.py:11 -> Normal.log_prob(0)).  Checked directly on 2^22
    random elements per regime: every softplus regime of rho (variant 0 is the branch taken for rho <= ln(1/4) only),
    |mu| over 12 decades, pruned entries, and values placed next to the regime switches."""
    g = torch.Generator().manual_seed(77)
    n = 1 << 22
    regimes = []
    if variant == 0:
        regimes.append(torch.rand(n, generator=g) * 98.6 - 100.0)            # -100 .. ln(1/4)
        regimes.append(torch.randn(n, generator=g) * 0.15 - 2.0)             # the reference initialisation
        regimes.append(torch.full((n,), -1.3862944))
    else:
        regimes.append(torch.rand(n, generator=g) * 140.0 - 100.0)           # -100 .. 40
        regimes.append(torch.rand(n, generator=g) * 4.0 - 2.5)               # around e = 1/4
        regimes.append(torch.rand(n, generator=g) * 12.0 + 12.0)             # around rho = 15 and torch's threshold 20
        regimes.append(torch.randn(n, generator=g) * 0.15 - 2.0)
    worst = 0.0
    for rho in regimes:
        mu = torch.randn(n, generator=g) * torch.pow(10.0, torch.rand(n, generator=g) * 12 - 9)
        mu[::7] = 0.0
        dmu, drho = mu.cuda(), rho.cuda()
        lo, hi = C.selftest_prune_interval(dmu, drho, variant)
        key = torch_keys_same_device(dmu, drho)                              # fp32, torch's op order, same device
        key2 = (key.double() + 0.9189385332046727) * 1.4426950408889634
        finite = torch.isfinite(key2)
        assert bool(finite.float().mean() > 0.9)
        lo, hi = lo.double(), hi.double()
        assert bool((lo[finite] <= key2[finite]).all()), "exact key below its certified interval"
        assert bool((key2[finite] <= hi[finite]).all()), "exact key above its certified interval"
        assert bool((lo[finite] <= hi[finite]).all())
        # the margins are not loose either: width within 2 * (1.5e-5 * q + 5e-5) * log2(e) of the key magnitude scale
        q2 = (key2[finite] - lo[finite]).clamp_min(0) + (hi[finite] - key2[finite]).clamp_min(0)
        worst = max(worst, float((q2 / (1e-4 + 3e-5 * key2[finite].abs() + 3e-5 * (torch.log2(1e-10 + F.softplus(drho[finite].double())).abs()))).max()))
    assert worst < 4.0, worst


@pytest.mark.parametrize("kind", ["wide_rho", "pruned_mix", "strided_structure", "outliers", "nonfinite_free_extremes",
                                  "nan_entries"])
def test_prune_sampled_path_hard_distributions(C, prune_mode, kind):
    """Inputs that stress the certified-interval arithmetic of the sampled path (every softplus regime, rho above
    torch's threshold of 20, keys of very different magnitude, already pruned entries) or defeat its strided sample
    (structure with the sample's period: the bracket misses and the tensor must fall back to the general path).
    Masks must equal the stable descending order of torch's own keys on the device for every k."""
    n = 1 << 20
    g = torch.Generator().manual_seed(21)
    mu, rho = init_params((n,), g, fan_in=400)
    if kind == "wide_rho":
        rho = torch.rand(n, generator=g) * 70 - 40                       # -40 .. 30
        mu = torch.randn(n, generator=g) * torch.pow(10.0, torch.rand(n, generator=g) * 4 - 3)
    elif kind == "pruned_mix":
        dead = torch.rand(n, generator=g) < 0.6
        mu[dead], rho[dead] = 0.0, -30.0
    elif kind == "strided_structure":
        mu[::32] *= 1e-3                                                  # 2^20 / 32768 samples: stride 32
    elif kind == "outliers":
        mu[::1000] = 1e6
        rho[::1000] = -80.0
        mu[5::777] = 0.0
    elif kind == "nonfinite_free_extremes":
        rho[::3] = 25.0
        rho[1::3] = -100.0
        mu[1::3] *= 1e-8
    elif kind == "nan_entries":                                          # NaN keys rank first, as in torch.topk / sort
        mu[torch.randperm(n, generator=g)[:37]] = float("nan")
    keys = torch_keys_same_device(mu.cuda(), rho.cuda())
    assert kind == "nan_entries" or bool(torch.isfinite(keys).all())
    for k in (1, 20, n // 100, n // 3, int(0.7 * n), n - n // 50, n - 1):
        dmu, drho = mu.cuda(), rho.cuda()
        mask = torch.empty(n, dtype=torch.uint8, device="cuda")
        C.prune([(dmu, drho, k, mask, None)])
        ref = orc.prune_mask_from_keys(keys, k)
        assert int(mask.sum()) == k, (kind, k)
        assert torch.equal(mask.bool(), ref), (kind, k)
        assert bool((dmu[ref] == 0).all()) and bool((drho[ref] == -30).all())
        keep = ~ref.cpu()
        assert torch.equal(dmu.cpu()[keep], mu[keep], ) or kind == "nan_entries"
        assert torch.equal(drho.cpu()[keep], rho[keep])
        if kind == "nan_entries":                                         # NaN != NaN: compare the bit patterns
            assert torch.equal(dmu.cpu()[keep].view(torch.int32), mu[keep].view(torch.int32))


@pytest.mark.parametrize("classes", [1, 2, 3])
def test_prune_large_tie_classes(C, prune_mode, classes):
    """Huge tie classes on a tensor large enough for the sampled path: the bracket collapses onto one key
    (candidate-heavy resolve, index bound) or overflows the candidate buffer (device-side fallback)."""
    n = 300000
    base_mu = torch.tensor([0.0, 0.5, 1.0][:classes]).repeat(n // classes)
    base_rho = torch.full((base_mu.numel(),), -2.0)
    keys = torch_keys_same_device(base_mu.cuda(), base_rho.cuda())
    for k in sorted({1, n // classes - 1, n // classes, min(n // classes + 1, base_mu.numel()), n // 2,
                     base_mu.numel() - 1}):
        mu, rho = base_mu.clone().cuda(), base_rho.clone().cuda()
        mask = torch.empty(base_mu.numel(), dtype=torch.uint8, device="cuda")
        C.prune([(mu, rho, k, mask, None)])
        assert int(mask.sum()) == k
        assert torch.equal(mask.bool(), orc.prune_mask_from_keys(keys, k))


def test_prune_ties_lowest_index_first(C, prune_mode):
    # 3 distinct (mu, rho) pairs repeated: massive ties at the threshold
    base_mu = torch.tensor([0.0, 0.5, 1.0]).repeat(5000)
    base_rho = torch.full((15000,), -2.0)
    ref_keys = torch_keys_same_device(base_mu.cuda(), base_rho.cuda())
    assert torch.unique(ref_keys).numel() == 3
    for k in (1, 4999, 5000, 5001, 7777, 14999):
        mu, rho = base_mu.clone().cuda(), base_rho.clone().cuda()
        mask = torch.empty(15000, dtype=torch.uint8, device="cuda")
        C.prune([(mu, rho, k, mask, None)])
        ref = orc.prune_mask_from_keys(ref_keys, k)
        assert int(mask.sum()) == k
        assert torch.equal(mask.bool(), ref)
        # lowest index first: the selected members of each tie class form a prefix of that class
        for cls in range(3):
            sel = mask.bool()[cls::3]
            n = int(sel.sum())
            assert bool(sel[:n].all()) and not bool(sel[n:].any())


def test_prune_many_tensors_and_idempotent_order(C, prune_mode):
    g = torch.Generator().manual_seed(4)
    shapes = [(64, 64, 3, 3), (64,), (10, 576), (10,)] * 8        # 32 tensors: two launches' worth
    dev = [tuple(t.cuda() for t in init_params(s, g)) for s in shapes]
    for p in (0.5, 0.75):                                         # second sweep re-selects the pruned first
        masks = [torch.empty(s, dtype=torch.uint8, device="cuda") for s in shapes]
        before = [(m.clone(), r.clone()) for m, r in dev]
        C.prune([(m, r, orc.prune_count(p, m.numel()), mk, None) for (m, r), mk in zip(dev, masks)])
        for (m, r), mk, (bm, br) in zip(dev, masks, before):
            k = orc.prune_count(p, bm.numel())
            ref = orc.prune_mask_from_keys(torch_keys_same_device(bm, br), k)   # reference keys, same device
            assert torch.equal(mk.bool(), ref)
            if p == 0.75:
                assert bool(ref[bm == 0].all())           # everything pruned at p=0.5 is selected again first
            orc.prune_apply(bm, br, ref)
            assert torch.equal(m, bm) and torch.equal(r, br)


def test_prune_several_groups_of_large_tensors(C, prune_mode):
    """More tensors than one descriptor table holds (24), each large enough for the sampled path: bnn_prune_into runs the
    bracket / resolve / finish steps of a group on its side lane while the next group is swept.  Every mask must equal
    the stable sort of torch's keys; a second call on the results (75 % -> 80 %) re-selects what is pruned first."""
    g = torch.Generator().manual_seed(21)
    sizes = [150000 + 4099 * i for i in range(50)]
    dev = [tuple(t.cuda() for t in init_params((n,), g, fan_in=400)) for n in sizes]
    for p in (0.75, 0.8):
        before = [(m.clone(), r.clone()) for m, r in dev]
        masks = [torch.empty(n, dtype=torch.uint8, device="cuda") for n in sizes]
        C.prune([(m, r, orc.prune_count(p, m.numel()), mk, None) for (m, r), mk in zip(dev, masks)])
        for (m, r), mk, (bm, br) in zip(dev, masks, before):
            k = orc.prune_count(p, bm.numel())
            ref = orc.prune_mask_from_keys(torch_keys_same_device(bm, br), k)
            assert int(mk.sum()) == k
            assert torch.equal(mk.bool(), ref)
            orc.prune_apply(bm, br, ref)
            assert torch.equal(m, bm) and torch.equal(r, br)


def test_prune_into_reports_the_kl_sums_of_the_same_sweep(C):
    """north_star: "the pruning mask reuses that same pass".  bnn_prune_into's optional by-product — the KL element sum of
    every INPUT tensor, formed from the sigma / log sigma of the key arithmetic — against bnn_kl on the same tensors, for
    every kind of tensor the sweep distinguishes (sampled path, small tensor, k = 0, k = numel, forced general path,
    ragged length, rho above the fast-math regime); the masks are the ones the plain call produces."""
    g = torch.Generator().manual_seed(31)
    shapes = [(700001,), (1 << 20,), (64, 64, 3, 3), (10,), (300007,), (300007,), (500000,)]
    ks = [0.75, 0.9, 0.5, 0.5, 0.0, 1.0, 0.6]
    params = [init_params(sh, g, fan_in=400) for sh in shapes]
    params[6][1].mul_(-1.0).add_(-1.0)                     # rho around +1: the general softplus regime
    dev = [(m.cuda(), r.cuda()) for m, r in params]
    entries = [(m, r, orc.prune_count(p, m.numel()), None) for (m, r), p in zip(dev, ks)]
    priors = [(0.0, 0.1), (0.05, 0.2), (0.0, 0.1), (0.0, 1.0), (0.0, 0.1), (-0.1, 0.3), (0.0, 0.5)]
    ref = C.kl([(m, r, None, None, loc, sc, 1.0) for (m, r), (loc, sc) in zip(dev, priors)])
    plain = C.prune_into(entries)
    outs, sums = C.prune_into(entries, kl_priors=priors)
    torch.cuda.synchronize()
    assert sums.dtype == torch.float64 and sums.shape == (len(shapes),)
    for i in range(len(shapes)):
        assert float(sums[i]) == pytest.approx(float(ref[i]), rel=1e-5), (i, float(sums[i]), float(ref[i]))
        assert torch.equal(outs[i][0], plain[i][0]) and torch.equal(outs[i][1], plain[i][1])
    # forced general path: the sweep leaves the tensor to the fallback but still sums its KL
    outs_g, sums_g = C.prune_into(entries[:2], flags=C.PRUNE_GENERAL, kl_priors=priors[:2])
    for i in range(2):
        assert float(sums_g[i]) == pytest.approx(float(ref[i]), rel=1e-5)
        assert torch.equal(outs_g[i][0], plain[i][0]) and torch.equal(outs_g[i][1], plain[i][1])


def test_prune_into_kl_sums_over_several_descriptor_groups(C):
    """KL by-product + side-stream pipelining together: 53 tensors (three descriptor groups) with different priors; sums
    against bnn_kl, outputs against the call without the by-product, twice in a row (the side lane's events are reused)."""
    g = torch.Generator().manual_seed(41)
    sizes = [70000 + 1111 * i for i in range(53)]
    dev = [tuple(t.cuda() for t in init_params((n,), g, fan_in=300)) for n in sizes]
    priors = [(0.01 * (i % 5), 0.1 + 0.05 * (i % 4)) for i in range(53)]
    entries = [(m, r, orc.prune_count(0.7, m.numel()), None) for m, r in dev]
    ref = C.kl([(m, r, None, None, loc, sc, 1.0) for (m, r), (loc, sc) in zip(dev, priors)])
    plain = C.prune_into(entries)
    for _ in range(2):
        outs, sums = C.prune_into(entries, kl_priors=priors)
        torch.cuda.synchronize()
        assert torch.allclose(sums, ref, rtol=1e-5, atol=0)
        for (a, b), (c, d) in zip(outs, plain):
            assert torch.equal(a, c) and torch.equal(b, d)


# ------------------------------------------------------------------------------------------------ contractions
def gemm_inputs(M, N, K, S, shared_a, gen, bias=True):
    mu_w, rho_w = init_params((N, K), gen)
    mu_b, rho_b = init_params((N,), gen, fan_in=K) if bias else (None, None)
    a = torch.randn((1 if shared_a else S, M, K), generator=gen)
    eps_w = torch.randn(S, N, K, generator=gen)
    eps_b = torch.randn(S, N, generator=gen) if bias else None
    return a, mu_w, rho_w, mu_b, rho_b, eps_w, eps_b


def run_fwd(C, a, mu_w, rho_w, mu_b, rho_b, eps_w, eps_b, S, prec, rng_w=None, rng_b=None, sample_begin=0):
    _, M, K = a.shape
    N = mu_w.shape[0]
    da = a.cuda().contiguous()
    sig_w = C.stddev(rho_w.cuda())
    sig_b = C.stddev(rho_b.cuda()) if rho_b is not None else None
    y = torch.full((S, M, N), float("nan"), device="cuda")
    C.sampled_gemm_fwd(da, K, 0 if a.shape[0] == 1 else M * K, mu_w.cuda(), sig_w,
                       mu_b.cuda() if mu_b is not None else None, sig_b,
                       eps_w.cuda() if eps_w is not None else None,
                       eps_b.cuda() if eps_b is not None else None,
                       C.make_view(y.data_ptr(), N, 1), M * N, M, N, K, S, sample_begin,
                       rng_w or C.make_rng(0, 0, 0), rng_b or C.make_rng(0, 0, 1), prec)
    torch.cuda.synchronize()
    return y


GEMM_SHAPES = [
    # M, N, K, S, shared activations
    (128, 128, 32, 1, True),
    (77, 10, 576, 3, False),        # ragged everything (C2 linear head shape, odd M)
    (300, 400, 784, 2, True),       # C1 first layer, shared input
    (256, 130, 100, 2, False),      # N just over one tile
    (640, 64, 96, 2, False),        # M blocks > 4
    (5, 3, 7, 2, False),            # tiny, unaligned K (scalar paths)
    (1024, 256, 128, 2, False),     # > 512 rows per sample: CTA-pair (cta_group::2) kernels in TF32 mode
    (700, 136, 96, 3, True),        # CTA pair with a ragged second CTA, shared activations (dgrad sums the samples)
]


@pytest.mark.parametrize("prec", [0, 1])
@pytest.mark.parametrize("M,N,K,S,shared", GEMM_SHAPES)
def test_sampled_gemm_fwd_injected(C, M, N, K, S, shared, prec):
    g = torch.Generator().manual_seed(5)
    a, mu_w, rho_w, mu_b, rho_b, eps_w, eps_b = gemm_inputs(M, N, K, S, shared, g)
    y = run_fwd(C, a, mu_w, rho_w, mu_b, rho_b, eps_w, eps_b, S, prec)
    for s in range(S):
        ref = orc.linear_forward(a[0 if shared else s].double(), mu_w.double(), rho_w.double(), eps_w[s].double(),
                                 mu_b.double(), rho_b.double(), eps_b[s].double())
        assert rel_err(y[s], ref) < TOL[prec], f"sample {s}"


def test_sampled_gemm_fwd_no_bias(C):
    g = torch.Generator().manual_seed(6)
    a, mu_w, rho_w, _, _, eps_w, _ = gemm_inputs(130, 40, 64, 2, False, g, bias=False)
    y = run_fwd(C, a, mu_w, rho_w, None, None, eps_w, None, 2, 1)
    for s in range(2):
        ref = orc.linear_forward(a[s].double(), mu_w.double(), rho_w.double(), eps_w[s].double())
        assert rel_err(y[s], ref) < TOL[1]


def test_sampled_gemm_fwd_philox_equals_materialized(C):
    """In-kernel Philox inside the GEMM producers == the eps the materialize kernel reports."""
    g = torch.Generator().manual_seed(7)
    M, N, K, S = 200, 136, 260, 3
    a, mu_w, rho_w, mu_b, rho_b, _, _ = gemm_inputs(M, N, K, S, False, g)
    rng_w, rng_b = C.make_rng(99, 5, 20), C.make_rng(99, 5, 21)
    _, eps_w = C.materialize(mu_w.cuda(), C.stddev(rho_w.cuda()), S, 4, rng_w, want_eps=True)
    _, eps_b = C.materialize(mu_b.cuda(), C.stddev(rho_b.cuda()), S, 4, rng_b, want_eps=True)
    y_inj = run_fwd(C, a, mu_w, rho_w, mu_b, rho_b, eps_w.cpu(), eps_b.cpu(), S, 1)
    y_phx = run_fwd(C, a, mu_w, rho_w, mu_b, rho_b, None, None, S, 1, rng_w, rng_b, sample_begin=4)
    assert torch.equal(y_inj, y_phx)
    # partition invariance: samples [1, 3) computed alone reproduce the same slices
    y_part = run_fwd(C, a[1:], mu_w, rho_w, mu_b, rho_b, None, None, 2, 1, rng_w, rng_b, sample_begin=5)
    assert torch.equal(y_part, y_phx[1:])


@pytest.mark.parametrize("prec", [0, 1])
@pytest.mark.parametrize("M,N,K,S,shared", GEMM_SHAPES)
def test_sampled_gemm_backward_injected(C, M, N, K, S, shared, prec):
    g = torch.Generator().manual_seed(8)
    a, mu_w, rho_w, mu_b, rho_b, eps_w, eps_b = gemm_inputs(M, N, K, S, shared, g)
    dy = torch.randn(S, M, N, generator=g)
    # oracle: autograd through the restated forward, float64
    la = a.double().requires_grad_(True)
    leaves = [t.double().requires_grad_(True) for t in (mu_w, rho_w, mu_b, rho_b)]
    ref = torch.autograd.grad(
        [orc.linear_forward(la[0 if shared else s], leaves[0], leaves[1], eps_w[s].double(), leaves[2], leaves[3],
                            eps_b[s].double()) for s in range(S)],
        [la] + leaves, [dy[s].double() for s in range(S)])
    d_a, d_muw, d_rhow, d_mub, d_rhob = ref

    ddy = dy.cuda()
    sig_w = C.stddev(rho_w.cuda())
    dy_view = C.make_view(ddy.data_ptr(), N, 1)
    rng = C.make_rng(0, 0, 0)
    # dgrad
    da = torch.full(tuple(a.shape), float("nan"), device="cuda")
    C.sampled_gemm_dgrad(dy_view, M * N, mu_w.cuda(), sig_w, eps_w.cuda(), da, K, 0 if shared else M * K,
                         M, N, K, S, 0, rng, prec)
    assert rel_err(da, d_a) < TOL[prec]
    # wgrad
    dmu = torch.zeros(N, K, device="cuda")
    drho = torch.zeros(N, K, device="cuda")
    dev_a = a.cuda()
    C.sampled_gemm_wgrad(dy_view, M * N, dev_a, K, 0 if shared else M * K, rho_w.cuda(), eps_w.cuda(), dmu, drho,
                         M, N, K, S, 0, rng, prec)
    assert rel_err(dmu, d_muw) < TOL[prec]
    assert rel_err(drho, d_rhow) < TOL[prec]
    # bias
    dmub = torch.zeros(N, device="cuda")
    drhob = torch.zeros(N, device="cuda")
    C.bias_grad(dy_view, M * N, rho_b.cuda(), eps_b.cuda(), dmub, drhob, M, N, S, 0, rng)
    assert rel_err(dmub, d_mub) < 1e-5
    assert rel_err(drhob, d_rhob) < 1e-5


@pytest.mark.parametrize("variant", ["pair", "mb4", "mb2", "mb1"])
@pytest.mark.parametrize("M,N,K,S,shared", [(700, 136, 96, 3, True), (1024, 256, 128, 2, False), (1100, 64, 288, 2, True)])
def test_every_tma_contraction_variant_on_small_shapes(C, request, variant, M, N, K, S, shared):
    """The launcher picks rows-per-CTA / CTA pairs from a cost model, so small shapes normally run one variant only;
    bnn_debug_force_contract_variant forces each of them (TF32 mode) through forward and input gradient, shared
    activations (the input gradient sums the samples inside the kernel) and per-sample ones."""
    C.force_contract_variant(variant)
    request.addfinalizer(lambda: C.force_contract_variant(None))
    g = torch.Generator().manual_seed(12)
    a, mu_w, rho_w, mu_b, rho_b, eps_w, eps_b = gemm_inputs(M, N, K, S, shared, g)
    y = run_fwd(C, a, mu_w, rho_w, mu_b, rho_b, eps_w, eps_b, S, 0)
    dy = torch.randn(S, M, N, generator=g)
    d_a = torch.zeros(a.shape, dtype=torch.float64)
    for s in range(S):
        w = mu_w.double() + orc.stddev(rho_w.double()) * eps_w[s].double()
        ref = orc.linear_forward(a[0 if shared else s].double(), mu_w.double(), rho_w.double(), eps_w[s].double(),
                                 mu_b.double(), rho_b.double(), eps_b[s].double())
        assert rel_err(y[s], ref) < TOL[0], f"forward, sample {s}"
        d_a[0 if shared else s] += dy[s].double() @ w
    ddy = dy.cuda()
    da = torch.full(tuple(a.shape), float("nan"), device="cuda")
    C.sampled_gemm_dgrad(C.make_view(ddy.data_ptr(), N, 1), M * N, mu_w.cuda(), C.stddev(rho_w.cuda()), eps_w.cuda(), da,
                         K, 0 if shared else M * K, M, N, K, S, 0, C.make_rng(0, 0, 0), 0)
    assert rel_err(da, d_a) < TOL[0]


@pytest.mark.parametrize("M,N,K,S", [(2100, 128, 96, 30), (1300, 100, 64, 50), (3000, 128, 32, 19), (8192, 128, 64, 16),
                                     (1050, 64, 64, 60)])
def test_pair_kernel_tile_plan_covers_every_row_once(C, request, M, N, K, S):
    """Narrow layers (one column tile) whose uniform 1024-row pair tiles need a fraction of a wave more than the machine
    has slots are cut into 8- and 6-row-block tiles, two kinds of samples (sampled_gemm_tma.cu: TilePlan).  Forward and
    per-sample input gradient on shapes whose plans differ (different cuts per sample, ragged last block, a sample count
    that is not a multiple of anything): every output row must be written exactly once — NaN-filled outputs, torch fp64
    reference with the injected eps."""
    C.force_contract_variant("pair")
    request.addfinalizer(lambda: C.force_contract_variant(None))
    g = torch.Generator().manual_seed(33)
    a, mu_w, rho_w, mu_b, rho_b, eps_w, eps_b = gemm_inputs(M, N, K, S, False, g)
    y = run_fwd(C, a, mu_w, rho_w, mu_b, rho_b, eps_w, eps_b, S, 0)
    assert bool(torch.isfinite(y).all())
    sig = orc.stddev(rho_w.double())
    w = mu_w.double().unsqueeze(0) + sig.unsqueeze(0) * eps_w.double()                     # [S, N, K]
    b = mu_b.double().unsqueeze(0) + orc.stddev(rho_b.double()).unsqueeze(0) * eps_b.double()
    ref = torch.bmm(a.double(), w.transpose(1, 2)) + b.unsqueeze(1)
    assert rel_err(y, ref) < TOL[0]
    dy = torch.randn(S, M, N, generator=g)
    ddy = dy.cuda()
    da = torch.full(tuple(a.shape), float("nan"), device="cuda")
    C.sampled_gemm_dgrad(C.make_view(ddy.data_ptr(), N, 1), M * N, mu_w.cuda(), C.stddev(rho_w.cuda()), eps_w.cuda(), da,
                         K, M * K, M, N, K, S, 0, C.make_rng(0, 0, 0), 0)
    assert bool(torch.isfinite(da).all())
    assert rel_err(da, torch.bmm(dy.double(), w)) < TOL[0]


@pytest.mark.parametrize("variant", ["pair", "mb4", "mb2", "mb1"])
@pytest.mark.parametrize("shared", [True, False])
def test_every_tma_contraction_variant_in_the_conv_and_sign_noise_modes(C, request, variant, shared):
    """The single-CTA and CTA-pair kernels share one body in all three modes; force each variant through (a) the
    implicit-GEMM conv mode: stride-1 NormalConv2d forward and input gradient on injected eps against torch fp64, and (b)
    the rank-one sign-noise mode: the fused FlipoutNormalLinear forward and input gradient against the two-contraction
    formula.  765 and 700 rows per sample: more than 4 row blocks, which the forced pair variant needs.  NaN-filled
    outputs: every row must be written."""
    C.force_contract_variant(variant)
    request.addfinalizer(lambda: C.force_contract_variant(None))
    g = torch.Generator().manual_seed(14)
    # (a) conv, 3x3, padding 1: weights in (o, kh, kw, c) order, NHWC activations
    S, B, Cin, H, W, Cout = 2, 3, 32, 15, 17, 64
    M = B * H * W
    x = torch.randn(1 if shared else S, B, Cin, H, W, generator=g)
    mu_w, rho_w = init_params((Cout, Cin, 3, 3), g)
    mu_b, rho_b = init_params((Cout,), g, fan_in=Cin * 9)
    eps_w = torch.randn(S, Cout, Cin, 3, 3, generator=g)
    eps_b = torch.randn(S, Cout, generator=g)
    w = mu_w.double() + orc.stddev(rho_w.double()) * eps_w.double()                  # [S, Cout, Cin, 3, 3]
    b = mu_b.double() + orc.stddev(rho_b.double()) * eps_b.double()
    geom = C.conv_geom(B, H, W, Cin, H, W, Cout, 3, 3, (1, 1), (1, 1), (1, 1))
    mu_o, sig_o = mu_w.permute(0, 2, 3, 1).contiguous().cuda(), C.stddev(rho_w.permute(0, 2, 3, 1).contiguous().cuda())
    eps_o = eps_w.permute(0, 1, 3, 4, 2).contiguous().cuda()
    y = torch.full((S, M, Cout), float("nan"), device="cuda")
    C.sampled_conv2d_fwd(x.permute(0, 1, 3, 4, 2).contiguous().cuda(), 0 if shared else M * Cin, mu_o, sig_o, mu_b.cuda(),
                         C.stddev(rho_b.cuda()), eps_o, eps_b.cuda(), C.make_view(y.data_ptr(), Cout, 1), M * Cout, geom, S, 0,
                         C.make_rng(0, 0, 0), C.make_rng(0, 0, 1))
    dy = torch.randn(S, B, Cout, H, W, generator=g)
    dx = torch.full((1 if shared else S, B, H, W, Cin), float("nan"), device="cuda")
    C.sampled_conv2d_dgrad(dy.permute(0, 1, 3, 4, 2).contiguous().cuda(), mu_o, sig_o, eps_o, dx, 0 if shared else M * Cin,
                           geom, S, 0, C.make_rng(0, 0, 0))
    torch.cuda.synchronize()
    dx_ref = torch.zeros(dx.shape, dtype=torch.float64)
    for s in range(S):
        ref = F.conv2d(x[0 if shared else s].double(), w[s], b[s], padding=1)
        assert rel_err(y[s], ref.permute(0, 2, 3, 1).reshape(M, Cout)) < TOL[0], f"conv forward, sample {s}"
        dx_ref[0 if shared else s] += F.conv_transpose2d(dy[s].double(), w[s], padding=1).permute(0, 2, 3, 1)
    assert rel_err(dx, dx_ref) < TOL[0]
    # (b) rank-one sign noise eps_s = R_s Sg_s^T, no bias
    M, N, K, S = 700, 136, 96, 3
    a, mu_w, rho_w, _, _, _, _ = gemm_inputs(M, N, K, S, shared, g, bias=False)
    R = (torch.randint(0, 2, (S, N), generator=g) * 2 - 1).float()
    Sg = (torch.randint(0, 2, (S, K), generator=g) * 2 - 1).float()
    rng = C.make_rng(0, 0, 0, signs=(R.cuda(), Sg.cuda()))
    y = run_fwd(C, a, mu_w, rho_w, None, None, None, None, S, 0, rng_w=rng)
    dy = torch.randn(S, M, N, generator=g)
    da = torch.full(tuple(a.shape), float("nan"), device="cuda")
    sig = orc.stddev(rho_w.double())
    ddy = dy.cuda()
    C.sampled_gemm_dgrad(C.make_view(ddy.data_ptr(), N, 1), M * N, mu_w.cuda(), C.stddev(rho_w.cuda()), None, da, K,
                         0 if shared else M * K, M, N, K, S, 0, rng, 0)
    torch.cuda.synchronize()
    da_ref = torch.zeros(a.shape, dtype=torch.float64)
    for s in range(S):
        x_s, r, c = a[0 if shared else s].double(), R[s].double(), Sg[s].double()
        ref = x_s @ mu_w.double().t() + ((x_s * c) @ sig.t()) * r
        assert rel_err(y[s], ref) < TOL[0], f"sign-noise forward, sample {s}"
        da_ref[0 if shared else s] += dy[s].double() @ mu_w.double() + ((dy[s].double() * r) @ sig) * c
    assert rel_err(da, da_ref) < TOL[0]


def test_wgrad_philox_equals_injected(C):
    g = torch.Generator().manual_seed(9)
    M, N, K, S = 96, 72, 136, 5
    a, mu_w, rho_w, _, _, _, _ = gemm_inputs(M, N, K, S, False, g)
    dy = torch.randn(S, M, N, generator=g).cuda()
    rng = C.make_rng(1234, 2, 9)
    _, eps_w = C.materialize(mu_w.cuda(), C.stddev(rho_w.cuda()), S, 10, rng, want_eps=True)
    outs = []
    for eps in (eps_w, None):
        dmu = torch.zeros(N, K, device="cuda")
        drho = torch.zeros(N, K, device="cuda")
        C.sampled_gemm_wgrad(C.make_view(dy.data_ptr(), N, 1), M * N, a.cuda(), K, M * K, rho_w.cuda(), eps, dmu,
                             drho, M, N, K, S, 10, rng, 1)
        outs.append((dmu, drho))
    # the sample split over CTAs is the same in both runs; atomics may reorder fp32 sums slightly
    assert rel_err(outs[1][0], outs[0][0].cpu()) < 1e-6
    assert rel_err(outs[1][1], outs[0][1].cpu()) < 1e-6


# ------------------------------------------------------------------------------------------------ likelihood tail
@pytest.mark.parametrize("S,B,classes,pitch", [(8, 256, 10, 10), (3, 32, 4096, 4096), (5, 7, 13, 13), (2, 9, 12, 16),
                                               (1, 1, 1, 1), (4, 300, 100, 100)])
def test_mc_cross_entropy_matches_torch(C, S, B, classes, pitch):
    """bnn_mc_cross_entropy_fwd / _bwd == F.cross_entropy over the S*B rows with the labels replicated S times
    (the reference loop of train.py:59-61 is the mean of the S block means = the mean over all rows), fp32, 1e-6."""
    g = torch.Generator().manual_seed(13)
    store = torch.rand(S * B, pitch, generator=g).cuda()               # probabilities-like scores, as the models emit
    x = store[:, :classes]
    y = torch.randint(0, classes, (B,), generator=g).cuda()
    if B > 4:
        y[1] = -100                                                     # ignored rows (torch's default ignore_index)
    xr = x.detach().clone().contiguous().requires_grad_(True)
    ref = F.cross_entropy(xr, y.repeat(S))
    (ref * 3.0).backward()
    loss, lse, count = C.mc_cross_entropy_fwd(x, y)
    assert abs(float(loss) - float(ref)) <= 1e-6 * abs(float(ref)) + 1e-7
    assert float(count) == S * int((y != -100).sum())
    assert torch.allclose(lse, torch.logsumexp(x, dim=1), rtol=1e-6, atol=1e-6)
    dx = C.mc_cross_entropy_bwd(x, y, lse, count, torch.tensor(3.0, device="cuda"))
    assert torch.allclose(dx, xr.grad, rtol=1e-5, atol=1e-9)
    # widely spread logits (the online max / sum rescaling), same tolerances relative to the loss
    z = (torch.randn(S * B, classes, generator=g) * 30).cuda()
    zr = z.clone().requires_grad_(True)
    ref2 = F.cross_entropy(zr, y.repeat(S))
    ref2.backward()
    loss2, lse2, count2 = C.mc_cross_entropy_fwd(z, y)
    if bool((y != -100).any()):
        assert abs(float(loss2) - float(ref2)) <= 2e-6 * abs(float(ref2)) + 1e-6
        dz = C.mc_cross_entropy_bwd(z, y, lse2, count2, torch.tensor(1.0, device="cuda"))
        assert torch.allclose(dz, zr.grad, rtol=1e-4, atol=1e-8)


def test_mc_cross_entropy_edge_cases(C):
    x = torch.rand(6, 5, device="cuda")
    ignored = torch.full((3,), -100, dtype=torch.int64, device="cuda")
    loss, _, count = C.mc_cross_entropy_fwd(x, ignored)
    assert float(count) == 0 and bool(torch.isnan(loss))                # torch returns NaN as well
    bad = torch.tensor([0, 7, 1], device="cuda")                        # class 7 of 5: NaN instead of a device assert
    assert bool(torch.isnan(C.mc_cross_entropy_fwd(x, bad)[0]))
    with pytest.raises(ValueError):
        C.mc_cross_entropy_fwd(x, torch.zeros(4, dtype=torch.int64, device="cuda"))      # 6 rows, 4 labels
    with pytest.raises(TypeError):
        C.mc_cross_entropy_fwd(x, torch.zeros(3, dtype=torch.int32, device="cuda"))
    # back-to-back calls reuse the self-resetting workspace
    y = torch.tensor([1, 4, 0], device="cuda")
    a = [float(C.mc_cross_entropy_fwd(x, y)[0]) for _ in range(3)]
    assert a[0] == a[1] == a[2] and abs(a[0] - float(F.cross_entropy(x, y.repeat(2)))) < 1e-6


# ------------------------------------------------------------------------------------------------ conv lowering
CONV_CASES = [
    # B, C, H, W, Cout, k, stride, pad, dil, groups
    (2, 3, 10, 10, 4, 3, 1, 1, 1, 1),       # the reference's own conv test config (tests/conftest.py:270-277)
    (3, 64, 6, 6, 64, 3, 2, 1, 1, 1),       # C2 Bayesian conv
    (2, 8, 9, 7, 6, 3, 2, 0, 2, 2),         # stride, dilation, groups, non-square
    (1, 1, 10, 10, 1, 1, 1, 1, 1, 1),       # 1x1 kernel with padding (conftest.py:270)
    (4, 128, 4, 4, 128, 3, 1, 1, 1, 1),     # C3 Bayesian conv (staged lowering, several channel slices per image)
    (1, 16, 40, 40, 16, 3, 1, 1, 1, 1),     # col2im slab of one channel > 48 KiB: two-channel slices, scalar rows
    (1, 2, 224, 224, 2, 3, 2, 1, 1, 1),     # one channel exceeds the staging limit: generic kernels
]


@pytest.mark.parametrize("case", CONV_CASES)
def test_im2col_col2im_match_unfold_fold(C, case):
    B, Cin, H, W, Cout, k, s, p, d, groups = case
    g = torch.Generator().manual_seed(10)
    x = torch.randn(B, Cin, H, W, generator=g)
    OH = (H + 2 * p - d * (k - 1) - 1) // s + 1
    OW = (W + 2 * p - d * (k - 1) - 1) // s + 1
    Cg = Cin // groups
    dx = torch.full((B, Cin, H, W), float("nan"), device="cuda")
    for grp in range(groups):
        geom = C.bnn_conv2d_geom(B, Cin, H, W, grp * Cg, Cg, k, k, OH, OW, s, s, p, p, d, d)
        col = torch.empty(B * OH * OW, Cg * k * k, device="cuda")
        C.im2col(x.cuda(), col, geom)
        ref = F.unfold(x[:, grp * Cg:(grp + 1) * Cg], k, d, p, s)            # [B, Cg*k*k, OH*OW]
        ref = ref.transpose(1, 2).reshape(B * OH * OW, Cg * k * k)
        assert torch.equal(col.cpu(), ref)
        dcol = torch.randn(B * OH * OW, Cg * k * k, generator=g)
        C.col2im(dcol.cuda(), dx, geom, False)
        ref_dx = F.fold(dcol.reshape(B, OH * OW, -1).transpose(1, 2), (H, W), k, d, p, s)
        assert torch.allclose(dx[:, grp * Cg:(grp + 1) * Cg].cpu(), ref_dx, rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("prec", [0, 1])
@pytest.mark.parametrize("case", CONV_CASES)
def test_conv2d_forward_through_gemm_view(C, case, prec):
    """NormalConv2d forward = im2col + sampled GEMM writing through the NCHW view (conv.py:112-119)."""
    B, Cin, H, W, Cout, k, s, p, d, groups = case
    S = 2
    g = torch.Generator().manual_seed(11)
    x = torch.randn(S, B, Cin, H, W, generator=g)
    mu_w, rho_w = init_params((Cout, Cin // groups, k, k), g)
    mu_b, rho_b = init_params((Cout,), g, fan_in=Cin // groups * k * k)
    eps_w = torch.randn((S,) + tuple(mu_w.shape), generator=g)
    eps_b = torch.randn(S, Cout, generator=g)
    OH = (H + 2 * p - d * (k - 1) - 1) // s + 1
    OW = (W + 2 * p - d * (k - 1) - 1) // s + 1
    Cg, Ng, Kg = Cin // groups, Cout // groups, (Cin // groups) * k * k
    M = B * OH * OW
    y = torch.full((S, B, Cout, OH, OW), float("nan"), device="cuda")
    dx_ = x.cuda().reshape(S * B, Cin, H, W)
    sig_w, sig_b = C.stddev(rho_w.cuda()), C.stddev(rho_b.cuda())
    dmu_w, dmu_b = mu_w.cuda(), mu_b.cuda()
    deps_w, deps_b = eps_w.cuda(), eps_b.cuda()
    for grp in range(groups):
        geom = C.bnn_conv2d_geom(S * B, Cin, H, W, grp * Cg, Cg, k, k, OH, OW, s, s, p, p, d, d)
        col = torch.empty(S * M, Kg, device="cuda")
        C.im2col(dx_, col, geom)
        w_off = grp * Ng * Kg
        # eps for this group's slice of the weight: [S][Cout*Kg] with offset; pass a compact copy
        ew = deps_w.reshape(S, Cout * Kg)[:, w_off:w_off + Ng * Kg].contiguous()
        eb = deps_b[:, grp * Ng:(grp + 1) * Ng].contiguous()
        view = C.make_view(y.data_ptr() + 4 * grp * Ng * OH * OW, Cout * OH * OW, OH * OW)
        C.sampled_gemm_fwd(col, Kg, M * Kg, dmu_w.reshape(-1)[w_off:w_off + Ng * Kg], sig_w.reshape(-1)[w_off:w_off + Ng * Kg],
                           dmu_b[grp * Ng:(grp + 1) * Ng], sig_b[grp * Ng:(grp + 1) * Ng], ew, eb, view,
                           B * Cout * OH * OW, M, Ng, Kg, S, 0, C.make_rng(0, 0, 0), C.make_rng(0, 0, 1), prec)
    for smp in range(S):
        ref = orc.conv2d_forward(x[smp].double(), mu_w.double(), rho_w.double(), eps_w[smp].double(), mu_b.double(),
                                 rho_b.double(), eps_b[smp].double(), s, p, d, groups)
        assert rel_err(y[smp], ref) < TOL[prec]


def test_golden_checkpoint_prune_fingerprints(C, prune_mode):
    """SURVEY §8c: masks of PruneNormal on the reference's shipped MNIST checkpoint (bit-exact)."""
    import os
    path = os.path.join(os.path.dirname(__file__), "golden", "mnist_ckpt_bayes_layers.npz")
    if not os.path.exists(path):
        pytest.skip("golden checkpoint fixture not generated")
    z = np.load(path)
    gold = {0.75: ["310e7ec976ca", "9fa0d864f805", "3960c6460375", "13bb28a97059"],
            0.9: ["ac9219b949a6", "8647fb21bdf7", "0b495bc324e0", "94d272989317"]}
    names = ["conv_w", "conv_b", "lin_w", "lin_b"]
    for p, hashes in gold.items():
        for name, h in zip(names, hashes):
            mu = torch.from_numpy(z[name + "_mean"]).cuda()
            rho = torch.from_numpy(z[name + "_scale"]).cuda()
            mask = torch.empty(mu.shape, dtype=torch.uint8, device="cuda")
            C.prune([(mu, rho, orc.prune_count(torch.tensor(p), mu.numel()), mask, None)])
            got = hashlib.sha1(mask.bool().cpu().numpy().tobytes()).hexdigest()[:12]
            assert got == h, f"{name} p={p}"
