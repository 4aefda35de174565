#!/usr/bin/env python
"""bench.py — ELBO training throughput of the variational hot path on B200 (driver contract).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c3|c2|c4]
                    [--dump-outputs DIR]

Metric (BASELINE.json): ELBO train samples*MC/sec = (rows x Monte-Carlo samples evaluated by all ranks) / step time, where
one step is the body of the reference's training loop, examples/MNIST/train.py:55-65: zero_grad -> model(x) (S
Monte-Carlo predictions) -> KLDivergence(model) -> mean cross-entropy over the S predictions -> backward -> [gradient
exchange] -> Adam step.

Default workload = C3, the configuration BASELINE.json quotes the 1/2/4/8-GPU metric on: examples/CIFAR10/model.py:20-39
as is (NormalConv2d 128x128x3x3 on the hot path, full-covariance MultivariateNormalLinear head as a torch composite),
32x32x3 inputs, batch 512 and S = 16 per GPU, TF32.  N > 1: the data x sample grid of SURVEY §8e (2 = 1x2, 4 = 2x2,
8 = 2x4): rank (d, s) takes batch slice d and the global MC samples [16 s, 16 s + 16); per-GPU work is fixed (weak
scaling), the gradients of all ranks are averaged inside the optimizer kernel over NVLink peer memory.
Extra blocks of the same JSON line: `c2` (examples/MNIST topology, B = 256, S = 8), `c4` (4x NormalLinear(4096,4096),
B = 1024, S = 32 on one GPU, sample-sharded S = 32 / N per GPU on N), `kl_prune` (C5: KL / prune sweeps over 2^30 pairs),
`fp32` (the step in the 3xTF32 1e-5-class mode), `tf32_peak` (cuBLAS 8192^3 TF32, measured in this run: the roofline
denominator), `reference_on_gpu` (N = 1: the unmodified reference classes on the same GPU through torch),
`cpu_baseline`.

One JSON line on stdout (rank 0).  `value`: inputs resident in HBM; `e2e`: the same step fed from pinned host memory (the next
batch's copy overlaps the running step, as a pin_memory DataLoader does) with the loss read back every step; `roofline`: the dominant hot-path contraction timed live with CUDA events.
`--impl reference` times the UNMODIFIED reference (baseline/_ref, installed by baseline/install_ref.py) on the host cores.

Torch-side settings of the deterministic trunk (Conv2d / BatchNorm2d / ELU / Linear of the example models, outside the
hot path but inside the measured step): cuDNN autotuning (`--no-cudnn-benchmark`), torch.channels_last for the trunk
modules (`--nchw-trunk` = the examples' layout; its step time is reported as `nchw_trunk_ms_per_step`), allow_tf32 in
TF32 mode (SURVEY §8d).
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("NCCL_DEBUG", "WARN")   # quiet by default; a caller's NCCL_DEBUG=INFO (rank lines) is left alone
REF_DIR = os.path.join(ROOT, "baseline", "_ref")

N_BATCHES = 469          # ceil(60000 / 128), examples/MNIST/train.py:38 (any constant; SURVEY §8d)
WORKLOADS = {
    "c2": dict(name="C2 examples/MNIST/model.py topology (NormalConv2d 64x64x3x3 s2 + NormalLinear 576x10), 28x28x1",
               batch=256, samples=8, example="MNIST", cin=1),
    "c3": dict(name="C3 examples/CIFAR10/model.py:20-39 as is (NormalConv2d 128x128x3x3 on 4x4 maps + "
                    "MultivariateNormalLinear(128,10) head), 32x32x3",
               batch=512, samples=16, example="CIFAR10", cin=3),
    "c4": dict(name="C4 wide Bayesian MLP 4x NormalLinear(4096,4096)", batch=1024, samples=32, example=None, cin=4096),
}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], bf16_burst=p["bf16_tflops"], bf16_sustained=p["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def measure_tf32_peak(device, seconds=2.0):
    """cuBLAS TF32 GEMM 8192^3 (torch.matmul on fp32 operands with allow_tf32), measured the way MEASURED_PEAKS.json
    measures bf16: best of 10 single calls (burst) and back-to-back calls for `seconds` (sustained, power capped)."""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    n = 8192
    a = torch.randn(n, n, device=device)
    b = torch.randn(n, n, device=device)
    c = torch.empty(n, n, device=device)
    flops = 2.0 * n ** 3
    for _ in range(3):
        torch.matmul(a, b, out=c)
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b, out=c)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    reps = max(10, int(seconds * 1e3 / best))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        torch.matmul(a, b, out=c)
    e1.record()
    torch.cuda.synchronize()
    sustained = e0.elapsed_time(e1) / reps
    torch.backends.cuda.matmul.allow_tf32 = prev
    del a, b, c
    return {"burst_tflops": flops / best / 1e9, "sustained_tflops": flops / sustained / 1e9,
            "how": f"torch.matmul fp32 8192^3 with allow_tf32 (cuBLAS TF32): best of 10 (burst), {reps} back to back (sustained)"}


# ------------------------------------------------------------------------------------------------ models
def build_model(workload, samples, nn=None):
    """The workload's network on `nn` (default: this package's nn; the reference arm passes pytorch_bayesian.nn)."""
    from torch.nn import BatchNorm2d, Conv2d, ELU, Flatten, Linear, Sequential, Softmax
    if nn is None:
        import bayesianneuralnetworks_b200 as bnn
        nn = bnn.nn

    class Net(nn.BayesianNetworkModule):
        def __init__(self, layers, cin, cout):
            super().__init__(cin, cout, samples)
            self.layers = layers

        def _forward(self, x):
            return self.layers(x)

    if workload == "c2":        # examples/MNIST/model.py:20-33
        layers = Sequential(Conv2d(1, 32, 5, padding=2, stride=2), BatchNorm2d(32), ELU(),
                            Conv2d(32, 32, 3, padding=1, stride=1), ELU(),
                            Conv2d(32, 64, 3, padding=0, stride=2), ELU(),
                            nn.NormalConv2d(64, 64, 3, padding=1, stride=2), ELU(), Flatten(),
                            nn.NormalLinear(576, 10), Softmax(dim=-1))
        return Net(layers, 1, 10)
    if workload == "c3":        # examples/CIFAR10/model.py:20-39
        layers = Sequential(Conv2d(3, 64, 5, padding=2, stride=2), BatchNorm2d(64), ELU(),
                            Conv2d(64, 128, 5, padding=2, stride=2), ELU(),
                            Conv2d(128, 128, 5, padding=2, stride=2), ELU(),
                            Conv2d(128, 128, 3, padding=1), ELU(), Conv2d(128, 128, 3, padding=1), ELU(),
                            nn.NormalConv2d(128, 128, 3, padding=1), ELU(), Flatten(),
                            Linear(2048, 128), ELU(), nn.MultivariateNormalLinear(128, 10), Softmax(dim=-1))
        return Net(layers, 3, 10)
    layers = Sequential(nn.NormalLinear(4096, 4096), ELU(), nn.NormalLinear(4096, 4096), ELU(),
                        nn.NormalLinear(4096, 4096), ELU(), nn.NormalLinear(4096, 4096), Softmax(dim=-1))
    return Net(layers, 4096, 4096)


def synthetic_batch(workload, batch, gen):
    if workload == "c2":
        return torch.rand(batch, 1, 28, 28, generator=gen), torch.randint(0, 10, (batch,), generator=gen)
    if workload == "c3":
        return torch.rand(batch, 3, 32, 32, generator=gen), torch.randint(0, 10, (batch,), generator=gen)
    return torch.randn(batch, 4096, generator=gen), torch.randint(0, 4096, (batch,), generator=gen)


# per workload: the Bayesian layers ON THE HOT PATH as (rows per (batch row, MC sample), N, K, input elements per
# (row, sample)) — the conv layers' K is Cin*kh*kw of the implicit GEMM, their algorithmic input is the un-expanded tensor
HOT_LAYERS = {
    "c2": [(9, 64, 576, 64 * 6 * 6), (1, 10, 576, 576)],
    "c3": [(16, 128, 1152, 128 * 4 * 4)],
    "c4": [(1, 4096, 4096, 4096)] * 4,
}


def hot_flops_per_step(workload, rows):
    """Algorithmic flops of the hot-path contractions per step (SURVEY §8d): fwd 2MNK, bwd 4MNK (2MNK for a first layer
    without dX); `rows` = batch rows x MC samples."""
    if workload == "c4":
        return rows * (4 * 6 - 2) * 4096 * 4096
    return rows * 3 * sum(2 * r * n * k for r, n, k, _ in HOT_LAYERS[workload])


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed regions (B200_PROFILING.md recipe).  The sampler
    runs from before the warm-up (nvidia-smi needs ~100 ms to deliver its first line) and every line is stamped on
    arrival; `stop()` reports the samples that fall inside the marked windows — or, for a window shorter than the
    sampling period, the samples nearest to it."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.windows = index, [], None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def mark(self, t0, t1):
        self.windows.append((t0, t1))

    def summary(self, windows=None):
        windows = self.windows if windows is None else windows
        rows = [(t, r) for t, r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        inside = [r for t, r in rows if any(a - 0.05 <= t <= b + 0.05 for a, b in windows)]
        note = "inside the timed regions"
        if not inside and rows and windows:
            mid = sum(a + b for a, b in windows) / (2 * len(windows))
            inside = [r for _, r in sorted(rows, key=lambda tr: abs(tr[0] - mid))[:3]]
            note = "nearest to the timed regions (shorter than the sampling period)"
        sm = sorted(float(r[1]) for r in inside)
        reasons = set()
        for r in inside:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        mx = [float(r[2]) for r in inside if r[2].replace(".", "").isdigit()]
        pw = [float(r[3]) for r in inside if r[3].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx[0] if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(pw) if pw else None, "window": note}

    def stop(self):
        if self.proc is None:
            return
        time.sleep(0.12)
        self.proc.terminate()


# ------------------------------------------------------------------------------------------------ one workload
class Env:
    """Process-wide context of a b200 run."""

    def __init__(self, args):
        self.args = args
        self.rank = int(os.environ.get("RANK", 0))
        self.world = int(os.environ.get("WORLD_SIZE", 1))
        self.local = int(os.environ.get("LOCAL_RANK", 0))
        if self.world != args.gpus and self.world == 1 and args.gpus > 1:
            raise SystemExit("launch N>1 with torch.distributed.run (one rank per GPU)")
        torch.cuda.set_device(self.local)
        self.device = torch.device("cuda", self.local)
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.device)
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.device)      # > 126 MB L2
        self.clocks = ClockSampler(self.local)
        self.pk = peaks()

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, v):
        if self.world == 1:
            return v
        import torch.distributed as dist
        t = torch.tensor([v], device=self.device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)


def dump_outputs(out_dir, arrays, budget_bytes=64 << 20, seed=0):
    """Writes each tensor of `arrays` as out_dir/<name>.npy (float64 stays float64, other floating point types become
    float32, integers float64), at most `budget_bytes` in all.  When the arrays do not fit, every array larger than an
    even share of the budget is replaced by a fixed, seeded sample of its flattened elements: the same indices in every
    run, in ascending order."""
    os.makedirs(out_dir, exist_ok=True)
    cap = budget_bytes // (8 * len(arrays))
    sample = sum(t.numel() for t in arrays.values()) * 8 > budget_bytes
    for name, t in arrays.items():
        t = t.detach()
        if sample and t.numel() > cap:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(seed))[:cap].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        dtype = torch.float64 if t.dtype == torch.float64 or not t.is_floating_point() else torch.float32
        np.save(os.path.join(out_dir, name + ".npy"), t.to("cpu", dtype).contiguous().numpy())


def reset_training_state(model, trainer, initial):
    """Puts the model and its trainer back, in place, into the state before their first training step: parameters and
    buffers from `initial`, the optimizer's moments and step counts and the library's device-side Philox step counter to
    zero.  In-place copies keep the addresses a captured CUDA graph holds.

    Every timed step starts from this state, so what a step computes depends on its batch alone, not on the rounding of
    the steps before it: the weight and bias gradients sum their per-sample partials with atomic adds, whose order (and
    last bits) changes from run to run, and over a trajectory Adam turns such differences into whole learning-rate
    steps on gradient components that are mostly rounding.  The work of a step does not depend on these values."""
    from bayesianneuralnetworks_b200 import runtime
    opt = trainer.opt
    zeros = [t for o in (opt, getattr(opt, "_torch_adam", None)) if o is not None
             for st in o.state.values() for t in st.values() if torch.is_tensor(t)]
    zeros += list(getattr(opt, "_step_dev", {}).values())
    counter = runtime.step_counter(trainer.device)
    if counter is not None:
        zeros.append(counter)
    with torch.no_grad():
        state = model.state_dict()
        torch._foreach_copy_(list(state.values()), [initial[name] for name in state])
        torch._foreach_zero_(zeros)


def measure_step(env, workload, steps, warmup, precision, parallel_mode, with_e2e=True, with_roofline=True,
                 channels_last=True, exchange="auto", dump_dir=None):
    """Builds the workload's ElboTrainer, times `steps` device-resident steps (and, with_e2e, as many host-fed ones) and
    returns the measurements of this workload as a dict (rank 0: complete; other ranks: timing only).  With `dump_dir`,
    rank 0 writes the loss and the model state of the last device-resident step there (dump_outputs)."""
    import bayesianneuralnetworks_b200 as bnn
    from bayesianneuralnetworks_b200 import _C, parallel
    from bayesianneuralnetworks_b200.training import ElboTrainer
    args, world, device = env.args, env.world, env.device
    wl = WORKLOADS[workload]
    B, S_local = wl["batch"], wl["samples"]
    if world == 1:
        data_groups, sample_groups, scaling = 1, 1, "weak"
    elif parallel_mode == "grid":        # weak scaling: every rank keeps (B rows, S samples); SURVEY §8e
        data_groups, sample_groups = parallel.default_grid(world) if args.sample_groups == 0 else (
            world // args.sample_groups, args.sample_groups)
        scaling = "weak"
    elif parallel_mode == "sample":      # strong scaling: the S samples of ONE batch sharded over the ranks (C4)
        if S_local % world != 0:
            raise SystemExit(f"{S_local} MC samples do not split over {world} ranks")
        data_groups, sample_groups, S_local, scaling = 1, world, S_local // world, "strong"
    else:                                # plain data parallelism
        data_groups, sample_groups, scaling = world, 1, "weak"
    S_global = S_local * sample_groups
    bnn.set_precision(precision)
    torch.backends.cudnn.benchmark = not args.no_cudnn_benchmark
    tf32 = precision == "tf32"           # SURVEY §8d (C3): TF32 hot path, "deterministic trunk through torch with allow_tf32"
    torch.backends.cuda.matmul.allow_tf32 = tf32
    torch.backends.cudnn.allow_tf32 = tf32
    torch.manual_seed(0)
    model = build_model(workload, S_global).to(device)
    if channels_last:                    # torch-side knob for the deterministic trunk: cuDNN's NHWC kernels without
        for m in model.modules():        # layout conversions around each call; (mu, rho) stay row-major OIHW
            if isinstance(m, (torch.nn.Conv2d, torch.nn.BatchNorm2d)):
                m.to(memory_format=torch.channels_last)
    initial = {name: t.detach().clone() for name, t in model.state_dict().items()}
    trainer = ElboTrainer(model, N_BATCHES, lr=1e-3, graph=not args.no_graph, optimizer=args.optimizer,
                          loss_tail=args.loss_tail, exchange=exchange, sample_groups=sample_groups)
    gen = torch.Generator().manual_seed(1 + trainer.data_index)      # a data group shares its batch slice
    n_host = 8
    host = [tuple(t.pin_memory() for t in synthetic_batch(workload, B, gen)) for _ in range(n_host)]
    dev = [(x.to(device), y.to(device)) for x, y in host]

    def timed(n_steps, feed_from_host):
        """K steps, each bracketed by CUDA events on the current stream; before each step (untimed) the training state
        is reset (reset_training_state) and L2 is flushed."""
        starts = [torch.cuda.Event(enable_timing=True) for _ in range(n_steps)]
        stops = [torch.cuda.Event(enable_timing=True) for _ in range(n_steps)]
        env.barrier()
        t0, w0 = time.time(), time.perf_counter()
        last = None
        if feed_from_host:
            trainer.prefetch(*host[0])    # as a DataLoader does: the first batch is in flight before the loop starts
        for i in range(n_steps):
            reset_training_state(model, trainer, initial)
            env.flush.zero_()
            starts[i].record()
            x, y = host[i % n_host] if feed_from_host else dev[i % n_host]
            loss = trainer.step(x, y)     # host-fed: the step waits for ITS batch's pinned-host -> device copy ...
            if feed_from_host:
                trainer.prefetch(*host[(i + 1) % n_host])   # ... and the next batch's copy overlaps this step
                last = loss.item()        # device -> host read of the step's result, every step
            stops[i].record()
        env.barrier()
        wall = time.perf_counter() - w0
        env.clocks.mark(t0, time.time())
        ms = sum(a.elapsed_time(b) for a, b in zip(starts, stops))
        return ms / 1e3, wall, last, (t0, time.time()), loss

    graph_note = "eager launches"
    if trainer.use_graph:
        try:
            trainer.capture(*dev[0])
            graph_note = ("whole step captured in one CUDA graph (device-side Philox step counter), replayed per step"
                          if trainer.graph_opt is None else "forward+backward and optimizer captured as two CUDA graphs")
        except Exception as exc:      # noqa: BLE001 — fall back to eager launches, say so in the result
            if world > 1:
                raise                 # ranks must not diverge (peer barriers pair up)
            sys.stderr.write(f"CUDA graph capture failed ({exc!r}); running eagerly\n")
            trainer.graph, trainer.graph_opt, trainer.use_graph = None, None, False
            bnn.graph_safe_rng(False)
            graph_note = f"eager launches (graph capture failed: {type(exc).__name__}: {str(exc)[:120]})"
    for i in range(max(warmup, 3)):
        trainer.step(*dev[i % n_host])
    launches0 = _C.launch_count
    dev_s, dev_wall, _, window, step_loss = timed(steps, False)
    launches = _C.launch_count - launches0
    if dump_dir is not None and env.rank == 0:
        # what a caller of the last timed step holds: its loss and the model state it left behind
        dump_outputs(dump_dir, {"loss": step_loss, **{"model." + k: v for k, v in model.state_dict().items()}})
    if trainer.graph is not None:
        launches = trainer.launches_per_step * steps      # replays launch the captured kernels
    res = {"ms_per_step": None}
    e2e_s = e2e_wall = last_loss = None
    if with_e2e:
        timed(2, True)                                    # untimed: first touch of the staging path
        e2e_s, e2e_wall, last_loss, _, _ = timed(steps, True)
        e2e_s = env.max_over_ranks(e2e_s)
    dev_s = env.max_over_ranks(dev_s)
    units = B * data_groups * S_global * steps
    per_kernel, roof = None, None
    if with_roofline:
        # the dominant hot-path kernel, timed live with CUDA events on the launching stream (eager launches so that
        # every library call can be bracketed; all ranks run the same number of steps: the peer barriers pair up)
        _C.set_kernel_timing(True)
        n_prof = min(steps, 10)
        # a spin kernel in front of every profiled step lets the host enqueue the whole eager step behind it: the event
        # pairs then bracket device time only (kernels back to back, as in the replayed graph) instead of the launch
        # latency of an idle GPU, which on the 100-us kernels of C2 / C3 was ~10 % of the figure
        spin = int(2.5e-3 * 1.9e9) if workload != "c4" else 0
        for i in range(n_prof):
            env.flush.zero_()
            if spin:
                torch.cuda._sleep(spin)
            trainer._body(*dev[i % n_host])
        per_kernel = _C.kernel_timing_summary(n_prof)
        _C.set_kernel_timing(False)
        roof = roofline(workload, B * S_local, per_kernel, env.pk, precision)
    x0, y0 = host[0]
    res = {
        "workload": wl["name"], "value": units / dev_s, "unit": "samples*MC/s", "ms_per_step": 1e3 * dev_s / steps,
        "steps": steps, "scaling": scaling,
        "config": {"workload": wl["name"], "batch_per_gpu": B, "mc_samples_per_gpu": S_local,
                   "global_batch": B * data_groups, "global_mc_samples": S_global,
                   "parallelism": "single" if world == 1 else (
                       f"grid {data_groups} data x {sample_groups} sample groups: rank (d, s) = batch slice d, global MC "
                       f"samples [{S_local} s, {S_local} s + {S_local}); gradients averaged over all {world} ranks"),
                   "gradient_exchange": trainer.exchange_note, "n_batches": N_BATCHES,
                   "optimizer": "Adam (torch fused)" if args.optimizer == "adam" else
                   "bnn.optim.ELBOAdam (KL gradient + Adam for every parameter in one kernel launch)",
                   "cudnn_benchmark": not args.no_cudnn_benchmark, "trunk_allow_tf32": tf32,
                   "trunk_memory_format": "channels_last (torch Conv2d / BatchNorm2d modules only)" if channels_last
                   else "contiguous (NCHW, the examples' layout)",
                   "launch": graph_note,
                   "l2": "flushed between steps (256 MiB write, untimed); each step timed with its own CUDA event pair",
                   "training_state": "every timed step starts from the state before the first training step (parameters, "
                                     "buffers, optimizer moments, RNG step counters; restored in place, untimed)",
                   "step": "zero_grad+forward(S)+KL+CE+backward+" + ("exchange+" if world > 1 else "") + "Adam"},
        "dtype": "tf32" if tf32 else "fp32 (3xTF32 split on tcgen05)",
        "gpu_launches": launches, "wall_s": dev_wall, "clocks": env.clocks.summary([window]),
        "hot_path_algorithmic_tflops": hot_flops_per_step(workload, B * data_groups * S_global) / (dev_s / steps) / 1e12,
    }
    if with_e2e:
        res["e2e"] = {"value": units / e2e_s, "unit": "samples*MC/s",
                      "h2d_bytes_per_step": x0.numel() * x0.element_size() + y0.numel() * y0.element_size(),
                      "d2h_bytes_per_step": 4, "ms_per_step": 1e3 * e2e_s / steps, "last_loss": last_loss,
                      "wall_s": e2e_wall,
                      "input_pipeline": "every step's batch is copied from pinned host memory (ElboTrainer.prefetch: a copy "
                                        "stream, two staging buffers); the copy of batch i+1 is issued inside step i's timed "
                                        "region and overlaps it, step i+1 waits for it; loss.item() every step"}
    if with_roofline:
        res["roofline"] = roof
        res["kernels_ms_per_step"] = per_kernel
    trainer.release()
    del trainer, model, dev, host
    torch.cuda.empty_cache()
    return res


def measured_traffic(workload, name):
    """DRAM bytes per launch of `name` from the committed `ncu --set full` capture (profiles/ncu_traffic.json)."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        return json.load(open(path)).get(workload, {}).get(name, {}).get("bytes_per_launch")
    except (OSError, ValueError):
        return None


def roofline(workload, rows, per_kernel, pk, precision):
    """Dominant hot-path kernel = the libbnn_b200 CONTRACTION entry point with the largest time share of the step.
    Its roof follows from its arithmetic intensity: algorithmic flops / algorithmic bytes (operands read once, results
    written once, fp32) against the ridge point peak_tensor / peak_hbm.  Both fractions are reported.  The tensor peak
    is the TF32 cuBLAS rate MEASURED in this run (sustained; burst beside it), not an assumed fraction of bf16."""
    if not per_kernel:
        return None
    gemms = {k: v for k, v in per_kernel.items() if k.startswith("bnn_sampled_")}
    name = max(gemms or per_kernel, key=lambda k: per_kernel[k]["ms_per_step"])
    k = per_kernel[name]
    base = {"kernel": name, "launches_per_step": k["launches_per_step"],
            "avg_launch_us": 1e3 * k["ms_per_step"] / k["launches_per_step"]}
    if name not in gemms:
        return dict(base, bound="hbm", achieved=None, peak=pk["hbm"], unit="GB/s", frac=None, traffic=None)
    layers = HOT_LAYERS[workload]
    if name.endswith("dgrad") and workload == "c4":
        layers = layers[1:]                      # the first layer needs no input gradient
    flops = sum(2 * r * n * kk for r, n, kk, _ in layers) * rows
    if name.endswith("fwd"):                     # x, (mu, sigma) -> y (+ bias)
        nbytes = sum(rows * (x_in + r * n) + 2 * n * kk for r, n, kk, x_in in layers) * 4
    elif name.endswith("dgrad"):                 # dy, (mu, sigma) -> dx
        nbytes = sum(rows * (r * n + x_in) + 2 * n * kk for r, n, kk, x_in in layers) * 4
    else:                                        # dy, x, rho -> dmu, drho
        nbytes = sum(rows * (r * n + x_in) + 3 * n * kk for r, n, kk, x_in in layers) * 4
    seconds = k["ms_per_step"] * 1e-3
    tensor_peak = pk["tf32_sustained"]
    tflops, gbs = flops / seconds / 1e12, nbytes / seconds / 1e9
    intensity, ridge = flops / nbytes, tensor_peak * 1e12 / (pk["hbm"] * 1e9)
    out = dict(base, arithmetic_intensity=intensity, ridge_point=ridge,
               tensor={"achieved": tflops, "peak": tensor_peak, "unit": "TFLOP/s", "frac": tflops / tensor_peak,
                       "frac_of_burst_peak": tflops / pk["tf32_burst"]},
               hbm={"achieved": gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": gbs / pk["hbm"]},
               traffic=measured_traffic(workload, name), algorithmic_bytes_per_step=nbytes,
               algorithmic_flops_per_step=flops,
               peak_note=f"tensor peak = cuBLAS TF32 8192^3 measured in this run ({pk['tf32_sustained']:.0f} TFLOP/s "
                         f"sustained, {pk['tf32_burst']:.0f} burst); HBM peak {pk['source']}; "
                         + ("fp32 mode issues 3 TF32 MMAs per product; " if precision != "tf32" else "")
                         + "timed with CUDA events around the C-ABI call in eager steps queued behind a spin kernel (device time, "
                           "launch latency hidden)")
    side = "tensor" if intensity >= ridge else "hbm"
    out.update(bound=side, achieved=out[side]["achieved"], peak=out[side]["peak"], unit=out[side]["unit"],
               frac=out[side]["frac"])
    return out


# ------------------------------------------------------------------------------------------------ C5
def bench_kl_prune(device, pk, world=1, tensors=64):
    """C5 (BASELINE.json configs[4], SURVEY §8d/e): KL forward, KL forward+grad and the pruning sweep over 2^30
    (mu, rho) pairs — 64 tensors of 4096x4096, 8 GiB — sharded round-robin by tensor over the GPUs (64 / N tensors per
    GPU; one GPU sweeps all of them); the working set per GPU is 8 GiB / N >> L2.  Algorithmic bytes (SURVEY §8d): KL
    fwd 8 B/pair, fwd+grad 16 B/pair, prune 8 + 8p B/pair.  With several GPUs the KL legs include the one scalar
    all-reduce of the sharded sum (SURVEY §8e), prune needs no exchange; times are the max over ranks and GB/s the
    aggregate."""
    from bayesianneuralnetworks_b200 import _C
    n_t = max(1, tensors // world)
    pairs = n_t * 4096 * 4096
    gen = torch.Generator(device=device).manual_seed(5)
    mus = [(torch.rand(4096, 4096, device=device, generator=gen) * 2 - 1) / 64 for _ in range(n_t)]
    rhos = [torch.randn(4096, 4096, device=device, generator=gen) * 0.15 - 2.0 for _ in range(n_t)]
    gm = [torch.empty_like(m) for m in mus]
    gr = [torch.empty_like(m) for m in mus]
    fwd = [(m, r, None, None, 0.0, 0.1, 1.0) for m, r in zip(mus, rhos)]
    both = [(m, r, a, b, 0.0, 0.1, 1.0) for m, r, a, b in zip(mus, rhos, gm, gr)]

    def over_ranks(seconds):
        if world == 1:
            return seconds
        import torch.distributed as dist
        t = torch.tensor([seconds], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    total_buf = torch.zeros((), device=device, dtype=torch.float64)

    def kl_leg(entries):
        sums = _C.kl(entries)
        if world > 1:                       # tensor-sharded KL: one small all-reduce
            import torch.distributed as dist
            torch.sum(sums, dim=0, out=total_buf)
            dist.all_reduce(total_buf)

    def time_it(fn, reps=5, inner=8):
        """Average duration of one call: `inner` back-to-back calls between one event pair (the host-side cost of
        preparing a launch overlaps the previous kernel, as it does in a training loop; every call streams the whole
        working set, so no call finds its data in L2), best of `reps`."""
        fn()
        torch.cuda.synchronize()
        best = 1e30
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(inner):
                fn()
            b.record()
            torch.cuda.synchronize()
            best = min(best, a.elapsed_time(b) / inner)
        return over_ranks(best * 1e-3)

    def entry(bytes_per_pair, t):
        gbps = bytes_per_pair * pairs * world / t / 1e9
        return {"GBps": gbps, "frac_of_measured_hbm": gbps / (pk["hbm"] * world), "ms": t * 1e3}

    res = {"workload": "C5: 64 tensors of 4096x4096 (2^30 pairs, 8 GiB of mu/rho), sharded by tensor over the GPUs",
           "pairs_per_gpu": pairs, "tensors_per_gpu": n_t, "n_gpus": world,
           "l2": f"working set {pairs * 8 / 2 ** 30:.0f} GiB per GPU, larger than L2",
           "timing": "CUDA events; KL legs: average of 8 back-to-back calls (best of 5); prune: one call per measurement "
                     "(it modifies its input, restored untimed), best of 3"}
    res["kl_fwd"] = entry(8, time_it(lambda: kl_leg(fwd)))
    res["kl_fwd_grad"] = entry(16, time_it(lambda: kl_leg(both)))
    p = 0.75
    k = int(p * 4096 * 4096)
    del gm, gr
    saved = [(m.clone(), r.clone()) for m, r in zip(mus, rhos)]

    def restore():
        for (m, r), (sm, sr) in zip(zip(mus, rhos), saved):
            m.copy_(sm), r.copy_(sr)
        torch.cuda.synchronize()

    def best_of(fn, reps=3, prepare=None):
        best = 1e30
        for _ in range(reps):
            restore()
            if prepare is not None:
                prepare()
                torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            best = min(best, a.elapsed_time(b) * 1e-3)
        return over_ranks(best)

    # PruneNormal on tensors of this size (prune/prune.py): the ONE-sweep out-of-place kernel (bnn_prune_into: 8 B read +
    # 8 B written per pair), the outputs then replace the parameters' storage.  The output buffers are caller-owned
    # (C ABI: the library never allocates); here two spare sets alternate, allocated outside the timed region.
    state = {"mus": mus, "rhos": rhos, "turn": 0}
    spare = [[(torch.empty_like(m), torch.empty_like(r)) for m, r in zip(mus, rhos)] for _ in range(2)]

    def prune_swap(kk=k):
        out = spare[state["turn"]]
        state["turn"] ^= 1
        outs = _C.prune_into([(m, r, kk, None) for m, r in zip(state["mus"], state["rhos"])], out=out)
        state["mus"], state["rhos"] = [o[0] for o in outs], [o[1] for o in outs]

    def prune_in_place():
        _C.prune([(m, r, k, None, None) for m, r in zip(mus, rhos)])

    def restore_swap():
        restore()
        state["mus"], state["rhos"] = mus, rhos

    def best_swap(reps=3, inner=1):
        """`inner` back-to-back calls on the (unmodified) inputs between one event pair, outputs alternating between the
        two spare sets: with inner > 1 the host-side preparation of a call overlaps the previous call's kernels, the
        protocol of the KL legs.  Every call streams the whole 8 GiB / N working set."""
        best = 1e30
        for _ in range(reps):
            restore_swap()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(inner):
                prune_swap()
                state["mus"], state["rhos"] = mus, rhos
            b.record()
            torch.cuda.synchronize()
            best = min(best, a.elapsed_time(b) * 1e-3 / inner)
        return over_ranks(best)
    prune_swap()                              # warm-up (workspace allocation)
    torch.cuda.synchronize()
    res["prune_p0.75"] = entry(8 + 8 * p, best_swap(inner=2))
    res["prune_p0.75"]["single_call"] = entry(8 + 8 * p, best_swap(inner=1))
    res["prune_p0.75"]["timing"] = ("average of 2 back-to-back calls (best of 3), as for the KL legs; `single_call` = one call "
                                    "bracketed on an idle stream, including the host-side preparation of the 64-entry table")
    # the fused sweep SURVEY §8d counts at 8 + 8p B/pair: KL element sums of the (unpruned) tensors AND the pruned tensors
    # from ONE pass over (mu, rho) (bnn_prune_into with kl_sum_out)
    priors = [(0.0, 0.1)] * n_t

    def kl_prune_swap():
        out = spare[state["turn"]]
        state["turn"] ^= 1
        _C.prune_into([(m, r, k, None) for m, r in zip(mus, rhos)], out=out, kl_priors=priors)

    def time_fused(reps=3, inner=2):
        best = 1e30
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(inner):
                kl_prune_swap()
            b.record()
            torch.cuda.synchronize()
            best = min(best, a.elapsed_time(b) * 1e-3 / inner)
        return over_ranks(best)
    restore_swap()
    kl_prune_swap()
    res["kl_prune_fused_p0.75"] = entry(8 + 8 * p, time_fused())
    res["kl_prune_fused_p0.75"]["what"] = ("KL sums of the unpruned tensors + pruned outputs from one sweep (the pruning pass "
                                           "reuses the KL pass, north_star); per-GPU sums only (no all-reduce in this leg)")
    restore_swap()
    prune_in_place()
    res["prune_p0.75_in_place"] = entry(8 + 8 * p, best_of(prune_in_place))
    res["prune_p0.75_in_place"]["what"] = ("strictly in-place kernel (bnn_prune): sample + read-only interval-histogram sweep + "
                                           "apply sweep (two reads and a write: 24 B/pair of traffic)")
    # the example's sweep (examples/MNIST/prune.py:49-50): successive levels on the SAME tensors — what was pruned at
    # one level (mu = 0, rho = -30: the largest key there is) is re-selected first at the next
    restore_swap()
    sweep = []
    for level in torch.linspace(.75, 1, 6).tolist():
        kk = int(level * 4096 * 4096)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        prune_swap(kk)
        b.record()
        torch.cuda.synchronize()
        t = over_ranks(a.elapsed_time(b) * 1e-3)
        sweep.append(dict(entry(8 if kk == 4096 * 4096 else 8 + 8 * level, t), p=round(level, 2)))      # p = 1 writes only
    rhos = state["rhos"]
    pruned = sum(int((r == -30).sum()) for r in rhos)
    res["prune_sweep"] = {"levels": sweep, "all_pruned_after_p1": pruned == n_t * 4096 * 4096}
    return res


# ------------------------------------------------------------------------------------------------ reference arm
def load_reference():
    """The unmodified reference package from baseline/_ref (None when it was not installed)."""
    if not os.path.isdir(os.path.join(REF_DIR, "pytorch_bayesian")):
        return None
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import pytorch_bayesian          # noqa: F401
    import pytorch_bayesian.nn as ref_nn
    return ref_nn


def reference_model(workload, samples, ref_nn):
    """C2 / C3: the reference's own example model files, unmodified; C4: the same Sequential on the reference's classes."""
    example = WORKLOADS[workload]["example"]
    if example is None:
        return build_model(workload, samples, nn=ref_nn)
    spec = importlib.util.spec_from_file_location(f"_ref_example_{example}", os.path.join(REF_DIR, "examples", example, "model.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.BCNN(WORKLOADS[workload]["cin"], 10, samples)


def reference_step_fn(workload, B, S, device="cpu"):
    """The loop body of examples/MNIST/train.py:55-65 on the reference's own classes (kind 'reference'), or — when
    baseline/_ref is absent — on the oracle's restatement (kind 'port')."""
    ref_nn = load_reference()
    gen = torch.Generator().manual_seed(1)
    x, y = synthetic_batch(workload, B, gen)
    x, y = x.to(device), y.to(device)
    torch.manual_seed(0)
    if ref_nn is not None:
        model = reference_model(workload, S, ref_nn).to(device)
        kld = ref_nn.KLDivergence(number_of_batches=N_BATCHES)
        ce = torch.nn.CrossEntropyLoss()
        opt = torch.optim.Adam(model.parameters(), lr=1e-3)

        def run():
            opt.zero_grad()
            preds = model(x)
            if not isinstance(preds, list):
                preds = [preds]
            divergence = kld(model)
            likelihood = torch.stack([ce(p, y) for p in preds]).mean()
            loss = likelihood + divergence
            loss.backward()
            opt.step()
            return loss
        return run, "reference"
    from oracle import variational_oracle as orc
    import bayesianneuralnetworks_b200 as bnn
    model = build_model("c2" if workload == "c2" else workload, S)
    stages, cur = [], []
    for m in model.layers:
        kind = type(m).__name__
        if kind == "MultivariateNormalLinear":      # the port has no full-covariance stage: a NormalLinear head instead
            m, kind = bnn.nn.NormalLinear(128, 10), "NormalLinear"
        if kind in ("NormalConv2d", "NormalLinear"):
            if cur:
                stages.append(('torch', torch.nn.Sequential(*cur)))
                cur = []
            ps = [m.weight.mean, m.weight.scale, m.bias.mean, m.bias.scale]
            loc, scale = float(m.weight_prior.loc), float(m.weight_prior.scale)
            if kind == "NormalLinear":
                stages.append(('linear', *ps, loc, scale))
            else:
                stages.append(('conv2d', *ps, loc, scale, m.stride, m.padding, m.dilation, m.groups))
        else:
            cur.append(m)
    if cur:
        stages.append(('torch', torch.nn.Sequential(*cur)))
    step = orc.ElboStepOracle(stages, S, N_BATCHES)
    opt = torch.optim.Adam(step.parameters(), lr=1e-3)

    def run():
        opt.zero_grad()
        loss, _ = step.loss(x, y)
        loss.backward()
        opt.step()
        return loss
    return run, "port"


def cpu_sample(workload):
    wl = WORKLOADS[workload]
    B, S = wl["batch"], wl["samples"]
    if workload == "c4":            # a full C4 step is ~12 TFLOP on the CPU: time a 1-sample slice
        return B, 1, "one MC sample of the step (B=1024, S=1 of 32), scaled by samples*MC"
    return B, S, f"full step (B={B}, S={S})"


def cpu_baseline(workload, bounded_seconds):
    B, S, sample = cpu_sample(workload)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    run, kind = reference_step_fn(workload, B, S)
    run()
    t0, n = time.perf_counter(), 0
    while n < 3 or (time.perf_counter() - t0 < bounded_seconds and n < 200):
        run()
        n += 1
    dt = (time.perf_counter() - t0) / n
    return {"value": B * S / dt, "unit": "samples*MC/s", "cores": cores, "kind": kind,
            "sample": f"{sample}, {n} steps, torch {torch.__version__} CPU fp32, {torch.get_num_threads()} threads"
                      + (", unmodified reference classes from baseline/_ref" if kind == "reference" else ", oracle port"),
            "ms_per_step": dt * 1e3}


def reference_on_gpu(device, workload, steps):
    """The UNMODIFIED reference classes on the same GPU through torch (cuBLAS / cuDNN + the unfused elementwise / RNG
    launches of SURVEY §2a): the kernel sequence the fused path replaces.  Eager, allow_tf32 as in the b200 run."""
    if load_reference() is None:
        return {"unavailable": "baseline/_ref not installed"}
    wl = WORKLOADS[workload]
    B, S = wl["batch"], wl["samples"]
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.allow_tf32 = True
    run, _ = reference_step_fn(workload, B, S, device=device)
    for _ in range(2):
        run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        run()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    peak = torch.cuda.max_memory_allocated(device) / 2 ** 30
    torch.cuda.empty_cache()
    return {"ms_per_step": ms, "value": B * S / (ms * 1e-3), "unit": "samples*MC/s", "steps": steps,
            "what": f"{wl['name']}: reference classes (baseline/_ref) on cuda through torch {torch.__version__}, eager, "
                    f"allow_tf32, B={B}, S={S}", "max_memory_allocated_gib": peak}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the host cores (baseline/_ref when
    installed, else the oracle port), same config / metric / unit."""
    if int(os.environ.get("RANK", 0)) != 0:
        return
    wl = WORKLOADS[args.workload]
    B, S, sample = cpu_sample(args.workload)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    run, kind = reference_step_fn(args.workload, B, S)
    warmup = min(max(args.warmup, 1), 3)
    t0 = time.perf_counter()
    for _ in range(warmup):
        run()
    per_step = (time.perf_counter() - t0) / warmup
    steps = max(3, min(args.steps, 20, int(90.0 / max(per_step, 1e-3))))      # bounded: the whole run ends within minutes
    t0 = time.perf_counter()
    for _ in range(steps):
        run()
    dt = (time.perf_counter() - t0) / steps
    value = B * S / dt
    print(json.dumps({
        "impl": "reference", "metric": "ELBO train samples*MC/sec", "value": value, "unit": "samples*MC/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": {"workload": wl["name"], "batch_per_gpu": B, "mc_samples_per_gpu": S, "n_batches": N_BATCHES,
                   "optimizer": "Adam", "step": "zero_grad+forward(S)+KL+CE+backward+Adam"},
        "cpu_baseline": {"value": value, "unit": "samples*MC/s", "cores": cores, "kind": kind,
                         "sample": f"{sample}, {steps} steps, torch {torch.__version__} CPU fp32, "
                                   f"{torch.get_num_threads()} threads"
                                   + (", unmodified reference classes from baseline/_ref (examples/*/model.py)"
                                      if kind == "reference" else ", oracle port (baseline/_ref absent)")},
        "e2e": {"value": value, "unit": "samples*MC/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------ b200 arm
def run_b200(args):
    env = Env(args)
    from bayesianneuralnetworks_b200 import _C
    _C.lib()                          # fails loudly when the CUDA library is missing
    rank, world, device = env.rank, env.world, env.device
    env.clocks.start()
    if args.tf32_peak > 0:           # profiling runs: do not spend the profiler's launch budget on 1400 cuBLAS calls
        tf32_peak = {"burst_tflops": args.tf32_peak, "sustained_tflops": args.tf32_peak, "how": "given on the command line"}
    else:
        tf32_peak = measure_tf32_peak(device)
    env.pk.update(tf32_burst=tf32_peak["burst_tflops"], tf32_sustained=tf32_peak["sustained_tflops"])
    main_mode = {"c4": "sample"}.get(args.workload, "grid") if args.parallel == "auto" else args.parallel
    main = measure_step(env, args.workload, args.steps, args.warmup, args.precision, main_mode,
                        channels_last=not args.nchw_trunk, exchange=args.exchange, dump_dir=args.dump_outputs)
    out = {
        "metric": "ELBO train samples*MC/sec", "value": main["value"], "unit": "samples*MC/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": main["ms_per_step"],
        "higher_is_better": True, "scaling": main["scaling"], "vs_baseline": None, "dtype": main["dtype"],
        "data": "synthetic", "config": main["config"], "e2e": main["e2e"], "gpu_launches": main["gpu_launches"],
        "wall_s": {"device_resident": main["wall_s"], "e2e": main["e2e"]["wall_s"]}, "clocks": main["clocks"],
        "roofline": main["roofline"],
        "hot_path": {"algorithmic_tflops_per_s": main["hot_path_algorithmic_tflops"],
                     "kernels_ms_per_step": main["kernels_ms_per_step"]},
        "peaks": env.pk, "tf32_peak": tf32_peak,
    }
    if not args.no_extras:
        short = max(5, min(args.steps, 20))
        for wl in ("c2", "c3", "c4"):
            if wl == args.workload:
                continue
            block = measure_step(env, wl, short, 3, "tf32", "sample" if wl == "c4" else "grid")
            out[wl] = {k: block[k] for k in ("workload", "value", "unit", "ms_per_step", "steps", "scaling", "config",
                                             "dtype", "e2e", "gpu_launches", "clocks", "roofline",
                                             "hot_path_algorithmic_tflops", "kernels_ms_per_step")}
        other = "fp32" if args.precision == "tf32" else "tf32"
        alt = measure_step(env, args.workload, short, 3, other, main_mode, with_e2e=False, with_roofline=False,
                           channels_last=not args.nchw_trunk, exchange=args.exchange)
        out[other] = {"ms_per_step": alt["ms_per_step"], "value": alt["value"], "dtype": alt["dtype"], "steps": short,
                      "what": "the same workload and launch configuration in the other hot-path precision mode "
                              "(fp32 = three-term TF32 split, 1e-5 parity class; the trunk then runs without allow_tf32)"}
        if not args.nchw_trunk:
            nchw = measure_step(env, args.workload, short, 3, args.precision, main_mode, with_e2e=False,
                                with_roofline=False, channels_last=False, exchange=args.exchange)
            out["nchw_trunk_ms_per_step"] = nchw["ms_per_step"]
        out["kl_prune"] = bench_kl_prune(device, env.pk, world=world)          # every rank sweeps its shard of the tensors
        if world == 1:
            try:
                out["reference_on_gpu"] = {"c2": reference_on_gpu(device, "c2", 5), "c3": reference_on_gpu(device, "c3", 3),
                                           "c4": reference_on_gpu(device, "c4", 2)}
            except Exception as exc:      # noqa: BLE001 — a comparator, never fatal
                out["reference_on_gpu"] = {"error": f"{type(exc).__name__}: {str(exc)[:200]}"}
            if rank == 0:
                out["cpu_baseline"] = cpu_baseline(args.workload, bounded_seconds=20.0)
    env.clocks.stop()
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="tf32", choices=["tf32", "fp32"],
                    help="hot-path contraction mode: tf32 (2e-3 parity class) or fp32 = 3xTF32 split (1e-5 class)")
    ap.add_argument("--parallel", default="auto", choices=["auto", "grid", "data", "sample"],
                    help="N > 1: grid = data x sample groups, per-GPU work fixed (weak scaling; default for c2 / c3); "
                         "sample = the MC samples of one batch sharded over the ranks (strong scaling; default for c4); "
                         "data = batch sharding only")
    ap.add_argument("--sample-groups", type=int, default=0, help="sample groups of the grid (0 = 2 -> 2, 4 -> 2, 8 -> 4)")
    ap.add_argument("--exchange", default="auto", choices=["auto", "peer", "bucketed", "flat"],
                    help="gradient exchange at N > 1 (training.ElboTrainer): peer = averaged inside the optimizer kernel over "
                         "NVLink peer memory, one CUDA graph; bucketed = NCCL buckets overlapped with backward; flat = one "
                         "NCCL all-reduce between two graphs")
    ap.add_argument("--loss-tail", default="batched", choices=["batched", "loop"],
                    help="likelihood term: nn.mc_mean_loss (one CE over the S*B rows) or the reference's per-sample loop")
    ap.add_argument("--no-cudnn-benchmark", action="store_true",
                    help="leave torch.backends.cudnn.benchmark off for the deterministic torch trunk (the examples' setting)")
    ap.add_argument("--optimizer", default="elbo-adam", choices=["adam", "elbo-adam"],
                    help="elbo-adam: bnn.optim.ELBOAdam (KL gradient + Adam in one pass, likelihood-only backward; same "
                         "trajectory); adam: torch's fused Adam on likelihood + KL, the reference loop verbatim")
    ap.add_argument("--nchw-trunk", action="store_true",
                    help="leave the deterministic torch trunk in torch's default NCHW memory format (the examples' setting)")
    ap.add_argument("--no-graph", action="store_true", help="launch eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-extras", action="store_true", help="only the main workload (profiling runs)")
    ap.add_argument("--tf32-peak", type=float, default=0.0,
                    help="skip the in-run cuBLAS TF32 peak measurement and use this TFLOP/s figure (runs under a profiler)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps of the main workload, write the loss and the model state of its last step "
                         "as DIR/<name>.npy (at most 64 MiB; larger arrays as a fixed, seeded sample), for comparing two "
                         "builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
