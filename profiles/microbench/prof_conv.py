"""Profiling driver: the C3 (default) or C2 Bayesian conv layer through the implicit-GEMM path — forward, input gradient,
weight gradient — with CUDA-event times per call.  `python profiles/microbench/prof_conv.py [c3|c2] [shared|per] [nchw]`.
Under ncu: `-k regex:"contract_|wgrad_tma"`."""
import sys

import torch

sys.path.insert(0, '.')
from bayesianneuralnetworks_b200 import _C as C  # noqa: E402

which = sys.argv[1] if len(sys.argv) > 1 else "c3"
shared = (sys.argv[2] if len(sys.argv) > 2 else "shared") == "shared"
B, S, Cn, HW, stride = (512, 16, 128, 4, 1) if which == "c3" else (256, 8, 64, 6, 2)
OH = (HW + 2 - 3) // stride + 1
g = torch.Generator(device='cuda').manual_seed(0)
x = torch.randn((B if shared else S * B), HW, HW, Cn, device='cuda', generator=g)          # NHWC memory
mu = (torch.rand(Cn, Cn, 3, 3, device='cuda', generator=g) * 2 - 1) / 34
rho = torch.randn(Cn, Cn, 3, 3, device='cuda', generator=g) * 0.15 - 2
wl = C.conv_weight_layout(mu, rho)
mub = torch.zeros(Cn, device='cuda')
sigb = C.stddev(torch.full((Cn,), -2.0, device='cuda'))
geom = C.conv_geom(B, HW, HW, Cn, OH, OH, Cn, 3, 3, (stride, stride), (1, 1), (1, 1))
M, K = B * OH * OH, 9 * Cn
y = torch.empty(S * M, Cn, device='cuda')
dy = torch.randn(S * M, Cn, device='cuda', generator=g)
dx = torch.empty_like(x)
gr = torch.zeros(2, Cn * K, device='cuda')
rw, rb = C.make_rng(1, 0, 1), C.make_rng(1, 0, 2)
xss = 0 if shared else B * HW * HW * Cn


nchw = len(sys.argv) > 3 and sys.argv[3] == "nchw"        # the layers' default output layout (view P = OH*OW)
y_view = C.make_view(y.data_ptr(), Cn * OH * OH, OH * OH) if nchw else C.make_view(y.data_ptr(), Cn, 1)


def fwd():
    C.sampled_conv2d_fwd(x, xss, wl[0], wl[1], mub, sigb, None, None, y_view, M * Cn, geom, S, 0, rw, rb)


def dgrad():
    if stride == 1:
        C.sampled_conv2d_dgrad(dy, wl[0], wl[1], None, dx, xss, geom, S, 0, rw)


def wgrad():
    C.sampled_conv2d_wgrad(dy, x, xss, wl[2], None, gr[0], gr[1], geom, S, 0, rw)


import os  # noqa: E402
if os.environ.get("BNN_FORCE_VARIANT"):
    C.force_contract_variant(os.environ["BNN_FORCE_VARIANT"])
for _ in range(3):
    fwd(), dgrad(), wgrad()
torch.cuda.synchronize()
flops = 2.0 * M * Cn * K * S
for name, fn in (("fwd", fwd), ("dgrad", dgrad), ("wgrad", wgrad)):
    best = 1e9
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b))
    print(f"{which} {'shared' if shared else 'per-sample'} {name}: {best * 1e3:.1f} us  {flops / best / 1e9:.1f} TFLOP/s")

# profiling builds only (BNN_EXTRA_NVCC_FLAGS=-DBNN_PROFILE_WAITS): wait cycles of the contraction kernels' roles
import ctypes  # noqa: E402
try:
    f = C.lib().bnn_debug_wait_counters
    f.restype = ctypes.c_int
    f.argtypes = [ctypes.POINTER(ctypes.c_ulonglong), ctypes.c_int]
    buf = (ctypes.c_ulonglong * 8)()
    f(buf, 1)
    f2 = C.lib().bnn_debug_stage_counters
    f2.restype = ctypes.c_int
    f2.argtypes = [ctypes.POINTER(ctypes.c_ulonglong), ctypes.c_int]
    st = (ctypes.c_ulonglong * 8)()
    f2(st, 1)
    for name, fn in (("fwd", fwd), ("dgrad", dgrad)):
        fn()
        torch.cuda.synchronize()
        if f2(st, 1) == 0 and st[5]:
            n = st[5]
            span = (st[7] - st[6]) * 1e-3
            print(f"{name}: CTA timeline (cycles since CTA start, mean of {n} CTAs): prologue {st[0] / n:.0f} | generators done {st[1] / n:.0f} | "
                  f"accumulator complete {st[2] / n:.0f} | epilogue done {st[3] / n:.0f} | CTA end {st[4] / n:.0f} | "
                  f"first CTA start -> last CTA end {span:.1f} us")
        if f(buf, 1) == 0 and buf[5]:
            n = buf[5]
            print(f"{name}: CTAs {n}  kernel {buf[0] / n:.0f} cycles/CTA | MMA thread waits: weights {buf[1] / n * 2:.0f} (leader only) "
                  f"activations {buf[2] / n * 2:.0f} | generators wait for a free slot {buf[3] / n:.0f} | TMA thread waits {buf[4] / n:.0f}"
                  f" | uniform grid: first weight tile ready at {buf[6] / n * 2:.0f}, weight waits of k-blocks 0..4 {buf[7] / n * 2:.0f}")
except AttributeError:
    pass
