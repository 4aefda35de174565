"""ELBOAdam — the optimizer half of the ELBO tail (SURVEY §8f-3, additive API).

The reference trains with `torch.optim.Adam(model.parameters())` on `loss = likelihood + KLDivergence(model)`
(examples/MNIST/train.py:43,57-65).  The KL term is a closed form of the variational parameters alone, so its gradient
needs no autograd: ELBOAdam applies, in ONE pass over every (mean, scale) pair the KLDivergence of the reference would
visit, `grad = d likelihood + d KL` and Adam's update (bnn_adam_kl_step).  The training loop then back-propagates the
likelihood only:

    opt = bnn.optim.ELBOAdam(model, number_of_batches=len(loader), lr=1e-3)
    preds = model(x)
    likelihood = bnn.nn.mc_mean_loss(criterion, preds, y)
    likelihood.backward()                    # (data parallel: all-reduce the gradients here, the KL part is added after)
    opt.step()                               # same parameters as Adam on likelihood + KLDivergence(n_batches)(model)
    kl = bnn.nn.KLDivergence(len(loader))(model)     # only if the value is wanted for logging (no gradient needed)

It is a `torch.optim.Optimizer`: `param_groups[0]` holds the variational tensors, `param_groups[1]` every other
parameter (deterministic layers, Bayesian layers nested in plain modules — the reference's KL does not see those
either); lr / betas / eps are read from the groups at every step, so `for g in opt.param_groups: g['lr'] = ...` and
torch's LR schedulers work in eager steps.  lr is a kernel argument: in a captured CUDA graph (ElboTrainer(graph=True))
it is the value of the captured step, and a scheduler has no effect on the replays.  CUDA float32 parameters of the
second group ride in the same kernel launch (plain Adam, `rho == NULL`); anything else goes to torch's own Adam.  Each
step agrees with torch's Adam evaluated in float64 on the same float32 inputs to 1e-5 of the update, plus 1e-6 lr, plus
one ulp of the parameter, plus what float32 rounding of the first moment allows (tests/test_adam_kernels_gpu.py).

Step counts are per parameter, as in torch's Adam: tensors with `requires_grad=False`, and deterministic parameters
whose `.grad` is None, are skipped and their count does not advance.  The counts live on the device in *cohorts*: one
0-dim float32 tensor (`state[p]['step']`) shared by every parameter that has been updated the same number of times, so
that a step in which every parameter takes part is one increment and one kernel launch per (device, hyper-parameters).
When only part of a cohort takes part, the rest keeps a copy of the count; a parameter updated for the first time
starts a cohort at 0.  A captured step advances exactly the cohorts it was captured with; capturing a step that would
start or split a cohort raises (run one eager step with the same parameters taking part first).  `state_dict()` stores
each parameter's moments and step as torch's Adam does; `load_state_dict()` regroups the counts into cohorts (and still
takes the single `bnn_step` count of older checkpoints).

Multi-GPU: `attach_peers(PeerGradients)` makes `step()` average the gradients over the ranks INSIDE the optimizer kernel
(bnn_adam_kl_step_peers: every rank reads all ranks' flat gradient buffers over NVLink), bracketed by two flag barriers —
no NCCL call, so the whole training step stays one capturable CUDA graph.
"""
import torch

from . import _C
from .nn.loss import _is_scalar_normal, _scalar_prior
from .nn.variational import WeightNormal
from .utils.traversal import apply_wb


class ELBOAdam(torch.optim.Optimizer):
    def __init__(self, model, number_of_batches=1, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, capturable=False):
        def visit(param, module=None, type=None):          # apply_wb passes module / type by keyword (utils.py:30-47)
            return (param, module.weight_prior if type == 'w' else module.bias_prior)
        found = model.traverse(lambda m: apply_wb(m, visit, pass_module=True, pass_type=True)) or []
        n = len(found)                    # loss.py:38 averages over ALL listed tensors, fused or not
        self._var = []
        self.composite = []               # tensors whose KL has no fused form: their KL gradient must come from autograd
        seen = set()
        for w, prior in found:
            if not (isinstance(w, WeightNormal) and _is_scalar_normal(prior)):
                # full-covariance tensors / tensor-valued priors: plain Adam here; add KLDivergence.composite_part(model)
                # to the loss that is back-propagated (training.ElboTrainer does)
                self.composite.append(w)
                continue
            loc, scale = _scalar_prior(prior, w.__class__.__name__)
            coeff = 1.0 / (w.mean.numel() * n * number_of_batches)      # loss.py:28,38: mean of means / n_batches
            if id(w.mean) in seen:                                       # a tensor listed twice: its KL counts twice
                for e in self._var:
                    if e["w"] is w:
                        e["coeff"] += coeff
                continue
            seen.update((id(w.mean), id(w.scale)))
            self._var.append({"w": w, "loc": loc, "scale": scale, "coeff": coeff})
        other = [p for p in model.parameters() if id(p) not in seen]
        groups = [{"params": [p for e in self._var for p in (e["w"].mean, e["w"].scale)], "variational": True}]
        if other:
            groups.append({"params": other, "variational": False})
        if not groups[0]["params"]:
            groups = groups[1:]
        if not groups:
            raise ValueError("ELBOAdam: the model has no parameters")
        super().__init__(groups, dict(lr=float(lr), betas=(float(betas[0]), float(betas[1])), eps=float(eps)))
        self.capturable = capturable
        self._torch_adam = None           # for parameters the kernel does not take (non-CUDA / non-float32)
        self._torch_adam_state = None     # its state_dict from load_state_dict(), until it is created
        self._peers = None
        self._views = None
        self.two_hop_above = 2            # peer exchange: ranks above this count average the buffers in two hops first

    # ---------------------------------------------------------------------------------------------------------------
    def attach_peers(self, peers, views=None):
        """`peers`: a parallel.PeerGradients whose flat buffer holds every gradient of this optimizer (see module doc).
        `views` ({id(param): view of peers.flat}): where each parameter's gradient sits in the flat buffer when the
        gradients are gathered into it after the backward pass (training.ElboTrainer) instead of being views of it."""
        self._peers = peers
        self._views = views

    def _moments(self, p):
        st = self.state[p]
        if "exp_avg" not in st:
            st["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
            st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
        return st["exp_avg"], st["exp_avg_sq"]

    def _kernel_ok(self, p):
        return p.is_cuda and p.dtype == torch.float32 and _C._dense(p)

    def _grad(self, p):
        if self._peers is not None and self._views is not None:
            return self._views[id(p)]
        g = p.grad
        if g is None:
            return None
        if g.stride() != p.stride():
            g = g.contiguous() if p.is_contiguous() else torch.empty_like(p).copy_(g)
        return g

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        units = []                # (parameters sharing one step count, hyper-parameters, kernel table entry)
        leftovers = []
        for group in self.param_groups:
            hyper = (group["lr"], group["betas"][0], group["betas"][1], group["eps"])
            if group.get("variational"):
                for e in self._var:
                    w = e["w"]
                    if not (w.mean.requires_grad or w.scale.requires_grad):
                        continue                      # frozen tensors are left alone, as torch's Adam leaves them
                    if w.mean.requires_grad != w.scale.requires_grad:
                        raise NotImplementedError("ELBOAdam: freeze mean and scale of a variational tensor together")
                    m_mu, v_mu = self._moments(w.mean)
                    m_rho, v_rho = self._moments(w.scale)
                    units.append(((w.mean, w.scale), hyper,
                                  (w.mean.data, w.scale.data, self._grad(w.mean), self._grad(w.scale), m_mu, v_mu, m_rho,
                                   v_rho, e["loc"], e["scale"], e["coeff"])))
            else:
                for p in group["params"]:
                    if not p.requires_grad or (p.grad is None and not (self._peers is not None and self._views is not None)):
                        continue
                    if self._kernel_ok(p):
                        m, v = self._moments(p)
                        units.append(((p,), hyper, (p.data, None, self._grad(p), None, m, v, None, None, 0.0, 1.0, 0.0)))
                    else:
                        leftovers.append((p, group))
        steps = self._advance_cohorts([ps for ps, _, _ in units])
        by_launch = {}            # (device, hyper-parameters, cohort) -> (step count, entries)
        for (ps, hyper, entry), step_dev in zip(units, steps):
            by_launch.setdefault((ps[0].device, hyper, id(step_dev)), (step_dev, []))[1].append(entry)
        peers = self._peers
        two_hop = peers is not None and peers.world > self.two_hop_above
        if peers is not None:
            peers.barrier()                               # every rank's gradients are complete
        if two_hop:
            # more than two ranks: average the flat buffers in place (every rank reduces its slice and writes it back to
            # all: (R-1)/R of the buffer per direction instead of R-1 whole buffers inbound), then the local kernel
            _C.peer_average(peers.bases, peers.rank, peers.flat.numel(), peers.device)
            peers.barrier()                               # every slice has landed in every buffer
        for (_, hyper, _), (step_dev, entries) in by_launch.items():
            _C.adam_kl_step(entries, *hyper, step_dev=step_dev,
                            peers=None if (peers is None or two_hop) else (peers.rank, peers.bases))
        if peers is not None and not two_hop:
            peers.barrier()                               # every rank has read: the buffers may be overwritten
        if leftovers:
            self._step_leftovers(leftovers)
        return loss

    def _advance_cohorts(self, units):
        """units: the tuples of parameters updated in this step (a variational tensor's mean and scale form one).
        Returns each unit's step count after this step's increment: one device tensor per cohort, shared by the
        parameters whose count it is (module doc)."""
        taking = {id(p) for ps in units for p in ps}
        cohorts = {}                              # id -> step count of the cohorts taking part
        joining = []
        for ps in units:
            c = self.state[ps[0]].get("step")
            if c is None:
                joining.append(ps)
            else:
                cohorts[id(c)] = c
        leaving = [st for p, st in self.state.items() if id(p) not in taking and "step" in st and id(st["step"]) in cohorts]
        if (joining or leaving) and torch.cuda.is_available() and torch.cuda.is_current_stream_capturing():
            raise RuntimeError("ELBOAdam: this step starts or splits a step cohort, which a CUDA graph cannot replay; "
                               "run one eager step with the same parameters taking part before capturing")
        copies = {}
        for st in leaving:                        # the count before this step's increment stays with them
            c = st["step"]
            if id(c) not in copies:
                copies[id(c)] = c.clone()
            st["step"] = copies[id(c)]
        fresh = {}                                # device -> the cohort of first updates
        for ps in joining:
            device = ps[0].device
            if device not in fresh:
                fresh[device] = torch.zeros((), device=device, dtype=torch.float32)
                cohorts[id(fresh[device])] = fresh[device]
            for p in ps:
                self.state[p]["step"] = fresh[device]
        for c in cohorts.values():
            c += 1                                # device-resident: a captured graph replays it
        return [self.state[ps[0]]["step"] for ps in units]

    def _step_leftovers(self, leftovers):
        if self._peers is not None:
            raise NotImplementedError("ELBOAdam with peer gradients needs CUDA float32 parameters")
        if self._torch_adam is None:
            groups = {}
            for p, g in leftovers:
                groups.setdefault(id(g), (g, []))[1].append(p)
            self._torch_adam = torch.optim.Adam([{"params": ps, "lr": g["lr"], "betas": g["betas"], "eps": g["eps"]}
                                                 for g, ps in groups.values()], capturable=self.capturable)
            self._torch_adam_groups = [g for g, _ in groups.values()]
            if self._torch_adam_state is not None:
                self._torch_adam.load_state_dict(self._torch_adam_state)
                self._torch_adam_state = None
        for tg, g in zip(self._torch_adam.param_groups, self._torch_adam_groups):
            tg["lr"], tg["betas"], tg["eps"] = g["lr"], g["betas"], g["eps"]
        self._torch_adam.step()

    # ---------------------------------------------------------------------------------------------------------------
    def state_dict(self):
        sd = super().state_dict()
        counts = {}                               # one read per cohort; every parameter gets its own step tensor
        for k, st in list(sd["state"].items()):
            if "step" in st:
                c = st["step"]
                if id(c) not in counts:
                    counts[id(c)] = float(c)
                sd["state"][k] = dict(st, step=torch.tensor(counts[id(c)], dtype=torch.float32))
        if self._torch_adam is not None:
            sd["bnn_torch_adam"] = self._torch_adam.state_dict()
        elif self._torch_adam_state is not None:
            sd["bnn_torch_adam"] = self._torch_adam_state
        return sd

    def load_state_dict(self, state_dict):
        state_dict = dict(state_dict)
        legacy = state_dict.pop("bnn_step", None)       # older checkpoints: one count for every updated parameter
        leftover = state_dict.pop("bnn_torch_adam", None)
        super().load_state_dict(state_dict)
        cohorts = {}                              # (device, count) -> step tensor
        for p, st in self.state.items():
            if "step" in st:
                n = float(st["step"])
            elif legacy is not None and "exp_avg" in st:
                n = float(legacy)
            else:
                continue
            if (p.device, n) not in cohorts:
                cohorts[(p.device, n)] = torch.full((), n, device=p.device, dtype=torch.float32)
            st["step"] = cohorts[(p.device, n)]
        if leftover is not None and self._torch_adam is not None:
            self._torch_adam.load_state_dict(leftover)
        else:
            self._torch_adam_state = leftover
