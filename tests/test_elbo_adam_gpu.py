"""optim.ELBOAdam against torch.optim.Adam on likelihood + KLDivergence, in float64, step by step and over trajectories.

The model holds every kind of parameter ELBOAdam sorts: NormalLinear and NormalConv2d (with and without bias) weights in
the variational group, a channels_last Conv2d + BatchNorm2d trunk and a NormalLinear nested in a plain module in the
second group (kernel, rho == NULL), and a float64 parameter that goes to torch's Adam.  The reference is a float64 copy
optimized by torch.optim.Adam with the same param groups.  There is no forward pass: every step, seeded likelihood
gradients are assigned to `.grad` of both models and the reference adds the float64 autograd gradient of the oracle's
kl_divergence, so conv rounding stays out of the comparison.

Per step (`sync`), the update of every parameter must agree with the reference's to the bound of
test_adam_kernels_gpu.py and m, v to a few rounding units of their terms; then the kernel's parameters and moments are
copied into the reference so that errors do not compound.  Over whole trajectories (no copying) the parameters must stay
within 1e-3 lr per step: the mistakes looked for there (a step count that advances for skipped parameters, lost state)
are whole fractions of lr.
"""
import copy
import io

import numpy as np
import pytest
import torch
from torch.distributions import Normal

import bayesianneuralnetworks_b200 as bnn
from bayesianneuralnetworks_b200.utils.traversal import variational_tensors
from oracle import variational_oracle as orc

pytestmark = pytest.mark.gpu

DEV = "cuda"
U = 2.0 ** -24
N_BATCHES = 7


def f32(x):
    return float(np.float32(x))


# float32-exact hyper-parameters: the kernel takes them in float32 (1 - float32(0.999) is 1.3e-5 off 0.001), torch's Adam
# (the reference, and ELBOAdam's own for the float64 parameter) in float64
LR, BETAS, EPS = f32(1e-3), (f32(0.9), f32(0.999)), f32(1e-8)


class _Wrapper(torch.nn.Module):           # a plain module: the traversal does not descend into it
    def __init__(self):
        super().__init__()
        self.head = bnn.nn.NormalLinear(10, 5)


class _Net(bnn.nn.BayesianNetworkModule):
    def __init__(self):
        super().__init__(3, 10, 2)
        self.trunk = torch.nn.Sequential(torch.nn.Conv2d(3, 8, 3), torch.nn.BatchNorm2d(8))
        self.layers = torch.nn.Sequential(
            bnn.nn.NormalConv2d(8, 32, 3, prior=Normal(0.2, 1.0)),
            bnn.nn.NormalConv2d(32, 32, 3, bias=False, prior=Normal(0.0, 3.0)),
            bnn.nn.NormalLinear(32, 10))
        self.nested = _Wrapper()
        self.extra = torch.nn.Parameter(torch.randn(7, dtype=torch.float64))


def make_model(seed=0):
    torch.manual_seed(seed)
    model = _Net()
    with torch.no_grad():                 # pruning-level scales and large means next to the usual initialisation
        model.layers[2].weight.scale[0, :4] = torch.tensor([-30.0, -10.0, 0.0, 20.5])
        model.layers[2].weight.mean[1, :3] = torch.tensor([10.0, -10.0, 5.0])
    model = model.to(DEV)
    model.trunk[0].weight.data = model.trunk[0].weight.data.contiguous(memory_format=torch.channels_last)
    return model


def variational_list(model):
    """[(mean, scale, loc, scale)] in the order KLDivergence visits them."""
    out = []
    for w, module, kind in variational_tensors(model):
        prior = module.weight_prior if kind == "w" else module.bias_prior
        out.append((w.mean, w.scale, float(prior.loc), float(prior.scale)))
    return out


class Pair:
    """The ELBOAdam model and its float64 torch.optim.Adam reference, fed the same gradients."""

    def __init__(self, group_hypers=None, seed=0):
        self.model = make_model(seed)
        self.ref = copy.deepcopy(self.model).double()
        self.opt = bnn.optim.ELBOAdam(self.model, number_of_batches=N_BATCHES, lr=LR, betas=BETAS, eps=EPS)
        if group_hypers:
            for g, h in zip(self.opt.param_groups, group_hypers):
                g.update(h)
        by_name = dict(self.ref.named_parameters())
        name_of = {id(p): n for n, p in self.model.named_parameters()}
        self.ref_opt = torch.optim.Adam([{"params": [by_name[name_of[id(p)]] for p in g["params"]], "lr": g["lr"],
                                          "betas": g["betas"], "eps": g["eps"]} for g in self.opt.param_groups])
        self.params = list(self.model.named_parameters())
        self.ref_params = dict(self.ref.named_parameters())

    def set_requires_grad(self, prefix, flag):
        for n, p in self.params:
            if n.startswith(prefix):
                p.requires_grad_(flag)
                self.ref_params[n].requires_grad_(flag)

    def set_lr(self, lr):
        for g in self.opt.param_groups + self.ref_opt.param_groups:
            g["lr"] = lr

    def kernel_state(self, p):
        opt = self.opt if p.dtype == torch.float32 else self.opt._torch_adam
        return opt.state[p]

    def step(self, t, skip=(), mismatched_strides=False, sync=False):
        """One step on likelihood gradients seeded by t; parameters named in `skip` get no gradient (.grad None)."""
        gen = torch.Generator().manual_seed(1000 + t)
        lik = {}
        for n, p in self.params:
            q = self.ref_params[n]
            if not p.requires_grad or n in skip:
                p.grad = q.grad = None
                continue
            g = (torch.randn(p.shape, generator=gen, dtype=torch.float64) * 1e-2).to(p.dtype).double()   # same values
            lik[n] = g.to(DEV)
            cl = p.dim() == 4 and not p.is_contiguous() and not mismatched_strides
            p.grad = g.to(DEV, p.dtype).contiguous(memory_format=torch.channels_last if cl else torch.contiguous_format)
            q.grad = g.to(DEV).clone()
        with torch.enable_grad():                 # the reference's loss is likelihood + KLDivergence
            tensors = variational_list(self.ref)
            kl = orc.kl_divergence(tensors, N_BATCHES)
            wrt = [x for m, s, _, _ in tensors for x in (m, s) if x.requires_grad]
            kl_grads = dict(zip(map(id, wrt), torch.autograd.grad(kl, wrt))) if wrt else {}
        names = {id(q): n for n, q in self.ref_params.items()}
        kl_by_name = {names[i]: g for i, g in kl_grads.items()}
        for n, g in kl_by_name.items():
            self.ref_params[n].grad += g
        before = {n: (self.ref_params[n].detach().clone(), *self._ref_moments(n)) for n in lik}
        frozen = {n: p.detach().clone() for n, p in self.params if n not in lik}
        self.opt.step()
        self.ref_opt.step()
        for n, p in frozen.items():
            assert torch.equal(dict(self.params)[n], p), f"{n} changed without a gradient"
        if sync:
            self._check_step(before, lik, kl_by_name)

    def _ref_moments(self, n):
        st = self.ref_opt.state.get(self.ref_params[n], {})
        if "exp_avg" not in st:
            z = torch.zeros_like(self.ref_params[n])
            return z, z
        return st["exp_avg"].clone(), st["exp_avg_sq"].clone()

    def _check_step(self, before, lik, kl):
        """This step's updates, m and v against the reference's; then the reference takes the kernel's values."""
        params = dict(self.params)
        for n, (p_old, m_old, v_old) in before.items():
            p, q = params[n], self.ref_params[n]
            group = next(g for g in self.ref_opt.param_groups if any(x is q for x in g["params"]))
            lr, (b1, b2), eps = group["lr"], group["betas"], group["eps"]
            st = self.ref_opt.state[q]
            step = float(st["step"])
            g_mag = lik[n].abs() + (kl[n].abs() if n in kl else 0)
            m_tol = 16 * U * (m_old.abs() + (1 - b1) * g_mag)
            v_tol = 16 * U * (b2 * v_old + (1 - b2) * g_mag * g_mag)
            denom = st["exp_avg_sq"].sqrt() / np.sqrt(1 - b2 ** step) + eps
            upd_ref = q.detach() - p_old
            pf = p.detach().float()
            ulp = (torch.nextafter(pf.abs(), torch.full_like(pf, float("inf"))) - pf.abs()).double()
            tol = 1e-5 * upd_ref.abs() + 1e-6 * lr + ulp + lr / (1 - b1 ** step) * m_tol / denom
            ks = self.kernel_state(p)
            for what, got, want, bound in (("update", p.detach().double() - p_old, upd_ref, tol),
                                           ("m", ks["exp_avg"].double(), st["exp_avg"], m_tol),
                                           ("v", ks["exp_avg_sq"].double(), st["exp_avg_sq"], v_tol)):
                err = (got - want).abs()
                worst = float((err / bound).max())
                assert worst <= 1.0, f"{n} {what}: error {worst:.3g} x the bound at torch step {step:g}"
            with torch.no_grad():
                q.copy_(p.double())
                st["exp_avg"].copy_(ks["exp_avg"].double())
                st["exp_avg_sq"].copy_(ks["exp_avg_sq"].double())

    def max_deviation(self):
        """max |kernel - reference| over all parameters, in units of lr."""
        return max(float((p.detach().double() - self.ref_params[n].detach()).abs().max()) for n, p in self.params) / LR


SCENARIOS = ["plain", "mismatched_strides", "param_groups", "lr_by_hand", "step_lr", "lambda_lr", "freeze_trunk",
             "freeze_variational", "grad_none_on_odd_steps", "prune"]


def run(scenario, sync, steps=10):
    hypers = None
    if scenario == "param_groups":
        hypers = [dict(lr=f32(2e-3), betas=(f32(0.8), f32(0.99)), eps=f32(1e-6)),
                  dict(lr=f32(5e-4), betas=(0.5, f32(0.9)), eps=f32(1e-3))]
    pair = Pair(hypers)
    scheds = []
    if scenario == "step_lr":
        scheds = [torch.optim.lr_scheduler.StepLR(o, step_size=3, gamma=0.5) for o in (pair.opt, pair.ref_opt)]
    elif scenario == "lambda_lr":
        scheds = [torch.optim.lr_scheduler.LambdaLR(o, lambda e: 1.0 / (1 + e)) for o in (pair.opt, pair.ref_opt)]
    for t in range(steps):
        skip = ()
        if scenario == "lr_by_hand" and t == 4:
            pair.set_lr(f32(3e-3))
        if scenario == "freeze_trunk":
            pair.set_requires_grad("trunk.", t >= 5)
        if scenario == "freeze_variational":
            pair.set_requires_grad("layers.1.", not 3 <= t <= 6)
        if scenario == "grad_none_on_odd_steps" and t % 2:
            skip = ("trunk.1.weight", "trunk.1.bias")
        if scenario == "prune" and t == 5:
            bnn.prune.PruneNormal()(pair.model, 0.5)
            with torch.no_grad():
                for n, p in pair.params:
                    if n.startswith("layers."):
                        pair.ref_params[n].copy_(p.double())
        pair.step(t, skip=skip, mismatched_strides=(scenario == "mismatched_strides"), sync=sync)
        for s in scheds:
            s.step()
    return pair


@pytest.mark.parametrize("scenario", SCENARIOS)
def test_elbo_adam_each_step_matches_torch_adam(scenario):
    run(scenario, sync=True)


@pytest.mark.parametrize("scenario", SCENARIOS)
def test_elbo_adam_trajectory_matches_torch_adam(scenario):
    pair = run(scenario, sync=False)
    assert pair.max_deviation() <= 1e-3 * 10


def test_elbo_adam_state_dict_round_trip():
    """Saved after a freeze (per-parameter step counts differ), loaded through torch.save / torch.load into a fresh model
    and optimizer: continuing is bit-identical to the uninterrupted run.  A checkpoint with the single `bnn_step` count
    of older versions still loads."""
    def schedule(pair, t):
        pair.set_requires_grad("layers.1.", not 2 <= t <= 3)
        pair.step(t, skip=("trunk.1.bias",) if t == 1 else ())

    a = Pair()
    for t in range(5):
        schedule(a, t)
    buf = io.BytesIO()
    torch.save({"model": a.model.state_dict(), "opt": a.opt.state_dict()}, buf)
    order = [p for g in a.opt.param_groups for p in g["params"]]          # state_dict's parameter indices
    name_of = {id(p): n for n, p in a.params}
    steps = {name_of[id(order[i])]: float(st["step"]) for i, st in a.opt.state_dict()["state"].items()}
    assert steps["layers.0.weight.mean"] == 5.0 and steps["layers.1.weight.mean"] == 3.0
    assert steps["trunk.1.bias"] == 4.0
    for t in range(5, 9):
        schedule(a, t)
    buf.seek(0)
    saved = torch.load(buf)
    b = Pair(seed=1)
    b.model.load_state_dict(saved["model"])
    b.opt.load_state_dict(saved["opt"])
    for t in range(5, 9):
        schedule(b, t)
    for (n, p), (_, q) in zip(a.params, b.params):
        assert torch.equal(p, q), n
        for k in ("exp_avg", "exp_avg_sq", "step"):
            assert torch.equal(a.kernel_state(p)[k], b.kernel_state(q)[k]), (n, k)
    legacy = dict(saved["opt"])
    legacy["state"] = {i: {k: v for k, v in st.items() if k != "step"} for i, st in legacy["state"].items()}
    legacy["bnn_step"] = 5.0
    c = Pair(seed=1)
    c.model.load_state_dict(saved["model"])
    c.opt.load_state_dict(legacy)
    counts = {float(st["step"]) for st in c.opt.state.values() if "step" in st}
    assert counts == {5.0}
    assert len({id(st["step"]) for st in c.opt.state.values() if "step" in st}) == 1       # one cohort
    c.step(5)


@pytest.mark.parametrize("cohorts", [1, 2])
def test_elbo_adam_graph_replays_equal_eager_steps(cohorts):
    """ELBOAdam(capturable=True) with step() captured after warm-up and the gradients in static tensors: k replays are
    bit-identical to k eager steps, with one step cohort and with two (a layer frozen during the first warm-up step)."""
    def build():
        model = make_model()
        model.extra.requires_grad_(False)
        return model, bnn.optim.ELBOAdam(model, number_of_batches=N_BATCHES, lr=LR, betas=BETAS, eps=EPS, capturable=True)

    def grads(model, t):
        gen = torch.Generator().manual_seed(500 + t)
        return {n: torch.randn(p.shape, generator=gen).to(DEV).contiguous(
            memory_format=torch.channels_last if not p.is_contiguous() else torch.contiguous_format)
            for n, p in model.named_parameters() if p.requires_grad}

    (eager, opt_e), (graphed, opt_g) = build(), build()
    static = {n: torch.zeros_like(p) for n, p in graphed.named_parameters() if p.requires_grad}
    for n, p in graphed.named_parameters():
        if p.requires_grad:
            p.grad = static[n]
    for t in range(2):                            # warm-up, eager on both
        for model in (eager, graphed):
            frozen = cohorts == 2 and t == 0
            for n, p in model.named_parameters():
                if n.startswith("layers.1."):
                    p.requires_grad_(not frozen)
        for n, g in grads(eager, t).items():
            eager.get_parameter(n).grad = g
            static[n].copy_(g)
        opt_e.step()
        opt_g.step()
    assert len({id(st["step"]) for st in opt_g.state.values()}) == cohorts
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        opt_g.step()
    for t in range(2, 6):
        for n, g in grads(eager, t).items():
            eager.get_parameter(n).grad = g
            static[n].copy_(g)
        opt_e.step()
        graph.replay()
    torch.cuda.synchronize()
    for (n, p), (_, q) in zip(eager.named_parameters(), graphed.named_parameters()):
        assert torch.equal(p, q), n
        if p in opt_e.state:
            for k in ("exp_avg", "exp_avg_sq", "step"):
                assert torch.equal(opt_e.state[p][k], opt_g.state[q][k]), (n, k)
