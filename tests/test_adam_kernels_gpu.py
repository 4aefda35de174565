"""bnn_adam_kl_step, bnn_adam_kl_step_peers, bnn_peer_average and bnn_pack_gradients on their own, against a float64
restatement of torch.optim.Adam on the same float32 inputs.

Reference: g = g_lik + kl_coeff * dKL (dKL by float64 autograd of the oracle's kl_normal_elementwise),
m = b1 m + (1 - b1) g, v = b2 v + (1 - b2) g^2, p -= lr / (1 - b1^t) * m / (sqrt(v) / sqrt(1 - b2^t) + eps).
The moments start random with v > 0, so the step is a smooth function of the gradient at every step number.
Errors are measured against the size of the terms that make up a result, not against the result (a sum can cancel):
m and v within 4 float32 rounding units of the sum of their terms' magnitudes plus what the float32 gradient's own
error bound gives (2 units of the likelihood gradient, 16 of the KL gradient's terms: expf / log1pf and a division);
the update within 1e-5 of the reference update plus 1e-6 lr plus one ulp of the parameter, plus what the bound on m
allows through m / denominator.  Hyper-parameters are rounded to float32 for the reference, as the kernel takes them.
Everything the kernels should do identically is checked bit for bit: step_dev against step_host, the scalar path
(misaligned arrays, numel tails) against the float4 path, table order, one launch against several, the peer average in
the optimizer kernel against bnn_peer_average.  Every array sits between NaN guard words that must survive.

bnn_peer_barrier is not here: on one device it needs two spinning launches resident at once, which nothing guarantees;
tests/test_multi_gpu.py covers it on two GPUs.
"""
import numpy as np
import pytest
import torch

from oracle import variational_oracle as orc

pytestmark = pytest.mark.gpu

U = 2.0 ** -24                # float32 unit roundoff
GUARD = 4                     # NaN words in front of (16 bytes: the array itself stays 16-byte aligned) and after each array
ARRAYS = ("mu", "rho", "g_mu", "g_rho", "m_mu", "v_mu", "m_rho", "v_rho")
DEV = "cuda"
SPECIAL_RHO = (-100.0, -80.0, -30.0, -10.0, 0.0, 19.9, 20.0, 20.1, 30.0)


def f32(x):
    return float(np.float32(x))


@pytest.fixture(scope="module")
def C():
    from bayesianneuralnetworks_b200 import _C
    _C.lib()
    assert _C.device_supported(0), "tests need a compute capability 10.x device"
    return _C


# ------------------------------------------------------------------------------------------------ table entries
class Entry:
    """One table entry: each array in its own NaN-filled buffer at `GUARD + offsets[name]` words."""

    def __init__(self, n, seed, variational=True, g_mu=True, g_rho=True, offsets=None, loc=0.0, scale=0.1, coeff=0.0):
        gen = torch.Generator().manual_seed(seed)
        offsets = offsets or {}
        self.n, self.variational = n, variational
        self.loc, self.scale = f32(loc), f32(scale)
        self.coeff = f32(coeff) if variational else 0.0
        present = {"mu", "g_mu", "m_mu", "v_mu"} if variational is False else set(ARRAYS)
        if not g_mu:
            present.discard("g_mu")
        if not g_rho or not variational:
            present.discard("g_rho")
        s = 1e-2                                                # size of the gradients and of m
        values = {
            "mu": (torch.rand(n, generator=gen, dtype=torch.float64) * 2 - 1) * 10,
            "rho": torch.randn(n, generator=gen, dtype=torch.float64) * 3 - 3,
            "g_mu": torch.randn(n, generator=gen, dtype=torch.float64) * s,
            "g_rho": torch.randn(n, generator=gen, dtype=torch.float64) * s,
        }
        for k in ("mu", "rho"):
            m = torch.randn(n, generator=gen, dtype=torch.float64) * s
            values["m_" + k] = m
            values["v_" + k] = (m * m + s * s * (0.5 + 1.5 * torch.rand(n, generator=gen, dtype=torch.float64)))
        values["rho"][: min(n, 3 * len(SPECIAL_RHO))] = torch.tensor(SPECIAL_RHO, dtype=torch.float64).repeat(3)[:n]
        self.bufs, self.views, self.offsets = {}, {}, {}
        for k in ARRAYS:
            if k not in present:
                self.bufs[k] = self.views[k] = None
                continue
            off = GUARD + offsets.get(k, 0)
            buf = torch.full((off + n + GUARD,), float("nan"), dtype=torch.float32, device=DEV)
            buf[off: off + n] = values[k].to(torch.float32).to(DEV)
            self.bufs[k], self.views[k], self.offsets[k] = buf, buf[off: off + n], off
        self.init = {k: None if v is None else v.clone() for k, v in self.views.items()}
        self.guards = {k: self._guard_bits(k) for k in present}

    def _guard_bits(self, k):
        b, off = self.bufs[k], self.offsets[k]
        return torch.cat([b[:off], b[off + self.n:]]).view(torch.int32).clone()

    def row(self):
        v = self.views
        return (v["mu"], v["rho"], v["g_mu"], v["g_rho"], v["m_mu"], v["v_mu"], v["m_rho"], v["v_rho"],
                self.loc, self.scale, self.coeff)

    def reset(self):
        for k, t in self.views.items():
            if t is not None:
                t.copy_(self.init[k])

    def outputs(self):
        return {k: self.views[k].clone() for k in ("mu", "rho", "m_mu", "v_mu", "m_rho", "v_rho") if self.views[k] is not None}

    def check_guards(self):
        for k, bits in self.guards.items():
            assert torch.equal(self._guard_bits(k), bits), f"{k}: a guard word was written"


def launch(C, entries, hyper, step, on_device):
    lr, b1, b2, eps = hyper
    if on_device:
        C.adam_kl_step([e.row() for e in entries], lr, b1, b2, eps,
                       step_dev=torch.tensor(float(step), dtype=torch.float32, device=DEV))
    else:
        C.adam_kl_step([e.row() for e in entries], lr, b1, b2, eps, step=step)


# ------------------------------------------------------------------------------------------------ the float64 reference
def kl_grads(mu, rho, loc, scale, coeff):
    """coeff * dKL/dmu, coeff * dKL/drho by float64 autograd, and the magnitudes of the terms of each."""
    mu = mu.detach().double().requires_grad_(True)
    rho = rho.detach().double().requires_grad_(True)
    with torch.enable_grad():
        (orc.kl_normal_elementwise(mu, rho, loc, scale).sum() * coeff).backward()
    with torch.no_grad():
        sigma = orc.stddev(rho)
        mag_mu = abs(coeff) * (mu - loc).abs() / scale ** 2
        mag_rho = abs(coeff) * (sigma / scale ** 2 + 1 / sigma) * torch.sigmoid(rho)
    return mu.grad, rho.grad, mag_mu, mag_rho


def adam_reference(p, g, g_mag, g_err, m, v, hyper, step):
    """float64 Adam on float32 inputs; returns (p, m, v, bound on |m error|, bound on |v error|, tolerance of the update).
    g_mag: sum of the magnitudes of the gradient's terms; g_err: bound on the error of the float32 gradient."""
    lr, b1, b2, eps = (f32(x) for x in hyper)
    p, m, v = p.double(), m.double(), v.double()
    bc1, bc2 = 1 - b1 ** step, 1 - b2 ** step
    m_new = b1 * m + (1 - b1) * g
    v_new = b2 * v + (1 - b2) * g * g
    denom = v_new.sqrt() / np.sqrt(bc2) + eps
    upd = -lr / bc1 * m_new / denom
    m_tol = 4 * U * (m.abs() + (1 - b1) * g_mag) + (1 - b1) * g_err
    v_tol = 4 * U * (b2 * v + (1 - b2) * g_mag * g_mag) + 2 * (1 - b2) * g_mag * g_err
    pf = p.float()
    ulp = (torch.nextafter(pf.abs(), torch.tensor(float("inf"), device=pf.device)) - pf.abs()).double()
    upd_tol = 1e-5 * upd.abs() + 1e-6 * lr + ulp + lr / bc1 * m_tol / denom
    return p + upd, m_new, v_new, m_tol, v_tol, upd_tol


def check_entry(e, hyper, step):
    """The entry's current arrays against one reference step from its initial arrays."""
    ini = {k: None if t is None else t.double() for k, t in e.init.items()}
    zero = torch.zeros(e.n, dtype=torch.float64, device=DEV)
    g_mu = ini["g_mu"] if ini["g_mu"] is not None else zero
    g_rho = ini["g_rho"] if ini["g_rho"] is not None else zero
    mag_mu, mag_rho = g_mu.abs(), g_rho.abs()
    err_mu, err_rho = 2 * U * mag_mu, 2 * U * mag_rho
    if e.variational and e.coeff != 0.0:
        # the float32 KL gradient goes through expf / log1pf (2 ulp each), a division and a few roundings
        k_mu, k_rho, km_mu, km_rho = kl_grads(ini["mu"], ini["rho"], e.loc, e.scale, e.coeff)
        g_mu, g_rho, mag_mu, mag_rho = g_mu + k_mu, g_rho + k_rho, mag_mu + km_mu, mag_rho + km_rho
        err_mu, err_rho = err_mu + 16 * U * km_mu, err_rho + 16 * U * km_rho
    pairs = [("mu", g_mu, mag_mu, err_mu)] + ([("rho", g_rho, mag_rho, err_rho)] if e.variational else [])
    for name, g, mag, g_err in pairs:
        p_ref, m_ref, v_ref, m_tol, v_tol, upd_tol = adam_reference(ini[name], g, mag, g_err, ini["m_" + name],
                                                                    ini["v_" + name], hyper, step)
        got_p, got_m, got_v = (e.views[k].double() for k in (name, "m_" + name, "v_" + name))
        for what, got, ref, tol in (("m", got_m, m_ref, m_tol), ("v", got_v, v_ref, v_tol),
                                    ("update", got_p - ini[name], p_ref - ini[name], upd_tol)):
            err = (got - ref).abs()
            bad = ~(err <= tol)
            if bool(bad.any()):
                i = int(bad.nonzero()[0])
                raise AssertionError(f"{name} {what}: {int(bad.sum())} of {e.n} elements out of bound; first at {i}: "
                                     f"got {float(got[i])!r}, want {float(ref[i])!r}, error {float(err[i]):.3g} > "
                                     f"{float(tol[i]):.3g} (rho {float(ini['rho'][i]) if e.variational else None})")
        if hyper[0] == 0.0:
            assert torch.equal(e.views[name], e.init[name]), f"{name} moved with lr = 0"
    e.check_guards()


# ------------------------------------------------------------------------------------------------ A: the update
NUMELS = (1, 3, 4, 5, 1023, 1024, 1025, 4097, 0)
PRIORS = ((0.0, 0.1), (0.3, 1.0), (-0.5, 3.0))


def table(kind, seed=0):
    """Tables of 1, 16, 17 and 40 entries (one to three launches of up to 16): variational and plain tensors, missing
    gradients, kl_coeff 0 and not, priors with loc != 0 and scales 0.1, 1, 3, zero-numel entries; the 40-entry table
    has a 2^21-element tensor between single-chunk tensors, more chunks than the grid has blocks."""
    if kind == "one":
        return [Entry(4097, seed, loc=0.3, scale=1.0, coeff=1e-4)]
    count = {"sixteen": 16, "seventeen": 17, "forty": 40}[kind]
    out = []
    for i in range(count):
        n = NUMELS[i % len(NUMELS)]
        if kind == "forty" and i == 20:
            n = 1 << 21
        loc, scale = PRIORS[i % 3]
        out.append(Entry(n, seed + i, variational=(i % 4 != 3), g_mu=(i % 7 != 5), g_rho=(i % 5 != 2), loc=loc,
                         scale=scale, coeff=(0.0 if i % 6 == 1 else 1e-4 * (1 + i % 3))))
    return out


HYPERS = [  # (lr, (beta1, beta2), eps, step)
    (1e-3, 0.9, 0.999, 1e-8, 1), (1e-3, 0.9, 0.999, 1e-8, 2), (1e-3, 0.9, 0.999, 1e-8, 10),
    (1e-3, 0.9, 0.999, 1e-8, 10_000), (0.0, 0.9, 0.999, 1e-8, 10), (1e-3, 0.0, 0.999, 1e-8, 3),
    (3e-2, 0.5, 0.9, 1e-6, 7), (1e-4, 0.95, 0.9999, 1e-3, 100),
]


@pytest.mark.parametrize("kind", ["one", "sixteen", "seventeen", "forty"])
@pytest.mark.parametrize("lr,b1,b2,eps,step", HYPERS)
def test_adam_kl_step_matches_fp64_adam(C, kind, lr, b1, b2, eps, step):
    """Every element of every table entry against the float64 reference, with step_host; step_dev must give the same
    bits."""
    entries = table(kind)
    hyper = (lr, b1, b2, eps)
    launch(C, entries, hyper, step, on_device=True)
    on_device = [e.outputs() for e in entries]
    for e in entries:
        e.reset()
    launch(C, entries, hyper, step, on_device=False)
    torch.cuda.synchronize()
    for e, dev in zip(entries, on_device):
        host = e.outputs()
        for k in host:
            assert torch.equal(host[k].view(torch.int32), dev[k].view(torch.int32)), f"step_dev != step_host in {k}"
        check_entry(e, hyper, step)


@pytest.mark.parametrize("offset", [1, 2, 3])
def test_adam_kl_step_misaligned_arrays(C, offset):
    """Each of the eight arrays in turn 4, 8 or 12 bytes off 16-byte alignment (the scalar path), in the same launch as
    float4-path tensors; a plain parameter with each of its four arrays off too.  Against the reference, and bit for bit
    against the same tensors at aligned addresses."""
    hyper, step = (1e-3, 0.9, 0.999, 1e-8), 5

    def build(misaligned):
        out = [Entry(4096, 100, coeff=2e-4)]                      # float4 path
        for j, k in enumerate(ARRAYS):
            out.append(Entry(1024 + 4 * j + 1, 101 + j, offsets={k: offset} if misaligned else None, loc=0.3, scale=1.0,
                             coeff=1e-4))
        for j, k in enumerate(("mu", "g_mu", "m_mu", "v_mu")):
            out.append(Entry(999, 110 + j, variational=False, offsets={k: offset} if misaligned else None))
        out.append(Entry(4096, 120, variational=False))            # float4 path
        return out

    aligned, shifted = build(False), build(True)
    for es in (aligned, shifted):
        for lo in range(0, len(es), 16):
            launch(C, es[lo: lo + 16], hyper, step, on_device=False)
    torch.cuda.synchronize()
    for a, s in zip(aligned, shifted):
        check_entry(s, hyper, step)
        for k, t in a.outputs().items():
            assert torch.equal(t.view(torch.int32), s.views[k].view(torch.int32)), f"alignment changed bits of {k}"


def test_adam_kl_step_table_order_and_launch_split(C):
    """The same 40 entries in one call (three launches), in reverse order, and one call per entry: bit-identical."""
    hyper, step = (2e-3, 0.8, 0.99, 1e-7), 4
    results = []
    for how in ("together", "reversed", "one_by_one"):
        entries = table("forty", seed=7)
        if how == "together":
            launch(C, entries, hyper, step, on_device=False)
        elif how == "reversed":
            launch(C, entries[::-1], hyper, step, on_device=False)
        else:
            for e in entries:
                launch(C, [e], hyper, step, on_device=False)
        torch.cuda.synchronize()
        for e in entries:
            e.check_guards()
        results.append([e.outputs() for e in entries])
    for other in results[1:]:
        for a, b in zip(results[0], other):
            for k in a:
                assert torch.equal(a[k].view(torch.int32), b[k].view(torch.int32)), k


def test_adam_kl_step_channels_last_and_strides(C):
    """4-d channels_last parameters with channels_last moments and gradients are taken (the update is elementwise);
    a gradient or moment in another memory order is refused before anything runs."""
    gen = torch.Generator().manual_seed(3)
    shape = (8, 32, 3, 3)

    def t(scale=1.0, shift=0.0):
        return (torch.randn(shape, generator=gen) * scale + shift).to(DEV).contiguous(memory_format=torch.channels_last)

    mu, rho, g_mu, g_rho = t(), t(1.0, -3.0), t(1e-2), t(1e-2)
    m_mu, m_rho = t(1e-2), t(1e-2)
    v_mu, v_rho = m_mu * m_mu + 1e-4, m_rho * m_rho + 1e-4
    init = [x.clone() for x in (mu, rho, g_mu, g_rho, m_mu, v_mu, m_rho, v_rho)]
    hyper, step = (1e-3, 0.9, 0.999, 1e-8), 3
    C.adam_kl_step([(mu, rho, g_mu, g_rho, m_mu, v_mu, m_rho, v_rho, 0.0, 0.1, 1e-4)], *hyper, step=step)
    # the same elements as flat contiguous arrays (memory order) through the reference
    e = Entry.__new__(Entry)
    e.n, e.variational, e.loc, e.scale, e.coeff = mu.numel(), True, 0.0, f32(0.1), f32(1e-4)
    flat = [x.permute(0, 2, 3, 1).reshape(-1) for x in init]
    e.init = dict(zip(ARRAYS, flat))
    e.views = dict(zip(ARRAYS, [x.permute(0, 2, 3, 1).reshape(-1) for x in (mu, rho, g_mu, g_rho, m_mu, v_mu, m_rho, v_rho)]))
    e.guards = {}
    check_entry(e, hyper, step)
    for bad in ("g_mu", "m_rho", "v_mu"):
        args = dict(zip(ARRAYS, [x.clone() for x in init]))
        args[bad] = args[bad].contiguous()
        with pytest.raises(ValueError):
            C.adam_kl_step([tuple(args[k] for k in ARRAYS) + (0.0, 0.1, 1e-4)], *hyper, step=step)
        assert torch.equal(args["mu"], init[0]), "a refused call changed the parameter"


# ------------------------------------------------------------------------------------------------ B: the exchange kernels
def peer_buffers(world, numel, seed):
    """`world` stand-in peer buffers on this device (the kernels only take pointers), NaN guards past `numel`."""
    gen = torch.Generator().manual_seed(seed)
    bufs = []
    for _ in range(world):
        b = torch.full((numel + 64,), float("nan"), dtype=torch.float32)
        b[:numel] = torch.randn(numel, generator=gen)
        bufs.append(b.to(DEV))
    return bufs


def rank_order_mean(bufs, numel):
    acc = bufs[0][:numel].clone()
    for b in bufs[1:]:
        acc += b[:numel]
    return acc * torch.tensor(np.float32(1) / np.float32(len(bufs)), device=DEV)


@pytest.mark.parametrize("world", range(1, 9))
def test_peer_average_is_the_rank_order_mean(C, world):
    for numel in sorted({0, 1, 3, 4, 5, 4 * world - 1, 4 * world + 1, 100_003, (1 << 20) + 3}):
        bufs = peer_buffers(world, numel, seed=numel + world)
        guards = [b[numel:].view(torch.int32).clone() for b in bufs]
        want = rank_order_mean(bufs, numel)
        for rank in range(world):
            C.peer_average([b.data_ptr() for b in bufs], rank, numel, torch.device(DEV))
        torch.cuda.synchronize()
        for r, b in enumerate(bufs):
            assert torch.equal(b[:numel].view(torch.int32), want.view(torch.int32)), (numel, r)
            assert torch.equal(b[numel:].view(torch.int32), guards[r]), (numel, r, "guard")


def peer_table(bufs, rank, seed, misaligned, coeff):
    """Entries whose gradients are views into bufs[rank] (aligned or 4 bytes off), parameters and moments with them."""
    sizes = (1, 5, 1023, 4096, 4097, 40_000)
    entries, off = [], 0
    for i, n in enumerate(sizes):
        shift = 1 if misaligned else 0
        e = Entry(n, seed + i, variational=(i != 2), offsets={k: shift for k in ("mu", "rho", "m_mu")} if misaligned
                  else None, coeff=coeff)
        for k in ("g_mu", "g_rho"):
            if e.views[k] is None:
                continue
            start = off + shift
            e.views[k] = bufs[rank][start: start + n]
            e.init[k] = e.views[k].clone()
            e.bufs[k] = None
            e.guards.pop(k)
            off = (start + n + 3) // 4 * 4
        entries.append(e)
    return entries, off


@pytest.mark.parametrize("misaligned", [False, True])
@pytest.mark.parametrize("world", range(2, 9))
def test_adam_kl_step_peers_averages_like_peer_average(C, world, misaligned):
    """bnn_adam_kl_step_peers with world stand-in buffers: with beta1 = 0, m = 0 and no KL, m after the step IS the
    averaged gradient: the rank-order float32 sum times 1/world, bit for bit, whatever the alignment.  Every rank index
    gives the same bits, and the general step (KL, beta1 > 0) equals bnn_peer_average followed by bnn_adam_kl_step."""
    total = 120_000
    for coeff, hyper, zero_m in ((0.0, (1e-3, 0.0, 0.999, 1e-8), True), (2e-4, (1e-3, 0.9, 0.999, 1e-8), False)):
        results = []
        for rank in range(world):
            bufs = peer_buffers(world, total, seed=world)
            entries, used = peer_table(bufs, rank, seed=50, misaligned=misaligned, coeff=coeff)
            assert used <= total
            if zero_m:
                for e in entries:
                    for k in ("m_mu", "m_rho"):
                        if e.views[k] is not None:
                            e.views[k].zero_()
            C.adam_kl_step([e.row() for e in entries], *hyper, step=3, peers=(rank, [b.data_ptr() for b in bufs]))
            torch.cuda.synchronize()
            for e in entries:
                e.check_guards()
            if zero_m:
                want = rank_order_mean(bufs, total)
                base = bufs[rank].data_ptr()
                for e in entries:
                    for g, m in (("g_mu", "m_mu"), ("g_rho", "m_rho")):
                        if e.views[g] is None:
                            continue
                        start = (e.views[g].data_ptr() - base) // 4
                        assert torch.equal(e.views[m].view(torch.int32), want[start: start + e.n].view(torch.int32)), \
                            (world, rank, e.n, m)
            results.append([e.outputs() for e in entries])
        for other in results[1:]:
            for a, b in zip(results[0], other):
                for k in a:
                    assert torch.equal(a[k].view(torch.int32), b[k].view(torch.int32)), f"rank changed bits of {k}"
        if zero_m:
            continue
        bufs = peer_buffers(world, total, seed=world)
        entries, _ = peer_table(bufs, 0, seed=50, misaligned=misaligned, coeff=coeff)
        for rank in range(world):
            C.peer_average([b.data_ptr() for b in bufs], rank, total, torch.device(DEV))
        C.adam_kl_step([e.row() for e in entries], *hyper, step=3)
        torch.cuda.synchronize()
        for a, e in zip(results[0], entries):
            for k, t in e.outputs().items():
                assert torch.equal(a[k].view(torch.int32), t.view(torch.int32)), f"two-hop path changed bits of {k}"


@pytest.mark.parametrize("n_items", [1, 32, 33, 70])
def test_pack_gradients_equals_cat(C, n_items):
    """bnn_pack_gradients (one launch per 32 items): sources aligned or not, None (zeros), offsets not divisible by 4,
    numel 0 to 5 and one large item; the flat buffer equals the torch.cat reference and the gaps keep their NaN."""
    gen = torch.Generator().manual_seed(n_items)
    items, pieces, off = [], [], 0
    keep = []
    for i in range(n_items):
        n = 300_001 if i == n_items // 2 else i % 6
        off += i % 3                                          # a gap of 0 to 2 words
        if i % 5 == 4:
            src = None
            pieces.append((off, torch.zeros(n)))
        else:
            shift = i % 4
            base = torch.randn(n + shift, generator=gen)
            src = base.to(DEV)[shift:]
            keep.append(src)
            pieces.append((off, base[shift:]))
        items.append((src, off, n))
        off += n
    flat = torch.full((off + 8,), float("nan"), dtype=torch.float32, device=DEV)
    want = flat.cpu().clone()
    for o, p in pieces:
        want[o: o + p.numel()] = p
    C.pack_gradients(items, flat)
    torch.cuda.synchronize()
    assert torch.equal(flat.cpu().view(torch.int32), want.view(torch.int32))
