"""Forward, input gradient and weight gradient of three Bayesian volumetric decoder layers (NormalConvTranspose3d), TF32,
per pass:

  implicit   this library's kernels: the phase-decomposed transposed-filter gather over rank-5 im2col maps (forward,
             one launch per output phase), the conv view's implicit-GEMM forward (input gradient) and weight gradient —
             bnn_sampled_conv_transpose3d_*
  reference  the reference's form, which is also the layer's path for requests the kernels refuse: materialised W_s and
             one torch conv_transpose3d (or its backward) per sample
  cudnn      one fixed weight, torch conv_transpose3d batched over S*B rows with allow_tf32 — the same flops without
             sampling, a ceiling

  V1  NormalConvTranspose3d(128, 64, 2, stride=2), 16^3 -> 32^3, B = 4, S = 8 (the 3-D U-Net up-conv: k == s, p == 0,
      eight one-tap phases with K = Cin each)
  V2  NormalConvTranspose3d(64, 64, 4, stride=2, padding=1), 8^3 -> 16^3, B = 16, S = 8
  V3  NormalConvTranspose3d(64, 32, (1, 4, 4), stride=(1, 2, 2), padding=(0, 1, 1)), 8x16x16 -> 8x32x32, B = 8, S = 8

CUDA events around each pass over a window of >= 1 s per (shape, arm, pass), a 256 MiB buffer overwritten between passes
so that no operand is served from L2.  Algorithmic TFLOP/s = 2 S B Din Hin Win Cin Cout KD KH KW / t for every pass; for
V1 also the forward's output-write bound (S B OD OH OW Cout 4 bytes at the data sheet's 7.7 TB/s).  Prints one JSON
document (and writes it to --out).

    python profiles/microbench/bench_conv_transpose3d.py --out profiles/r04_bench_conv_transpose3d.json
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))

import bayesianneuralnetworks_b200 as bnn                       # noqa: E402
from bayesianneuralnetworks_b200 import _C                      # noqa: E402
from bayesianneuralnetworks_b200.nn import NormalConvTranspose3d  # noqa: E402

SHAPES = {
    "V1": dict(Cin=128, Cout=64, k=(2, 2, 2), s=(2, 2, 2), p=(0, 0, 0), size=(16, 16, 16), B=4, S=8),
    "V2": dict(Cin=64, Cout=64, k=(4, 4, 4), s=(2, 2, 2), p=(1, 1, 1), size=(8, 8, 8), B=16, S=8),
    "V3": dict(Cin=64, Cout=32, k=(1, 4, 4), s=(1, 2, 2), p=(0, 1, 1), size=(8, 16, 16), B=8, S=8),
}
HBM_BYTES_PER_S = 7.7e12           # HGX B200 data sheet, one GPU

_FLUSH = None


def flush_l2():
    global _FLUSH
    if _FLUSH is None:
        _FLUSH = torch.empty(64 << 20, device="cuda", dtype=torch.float32)
    _FLUSH.zero_()


def timed(fn, min_seconds):
    """Mean device time (ms) of fn over a window of at least min_seconds, L2 flushed before every pass."""
    for _ in range(3):
        flush_l2()
        fn()
    torch.cuda.synchronize()
    total, n = 0.0, 0
    while total < min_seconds * 1e3 or n < 5:
        flush_l2()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        total += e0.elapsed_time(e1)
        n += 1
    return total / n


def bench_shape(name, c, min_seconds):
    Cin, Cout, k, s, p, size, B, S = (c[n] for n in ("Cin", "Cout", "k", "s", "p", "size", "B", "S"))
    out_size = tuple((n - 1) * s_ - 2 * p_ + (k_ - 1) + 1 for n, k_, s_, p_ in zip(size, k, s, p))
    vox_in = size[0] * size[1] * size[2]
    flops = 2.0 * S * B * vox_in * Cin * Cout * k[0] * k[1] * k[2]
    layer = NormalConvTranspose3d(Cin, Cout, k, stride=s, padding=p).cuda()
    spec_w, spec_b = layer._draws(True, S, 0, S)
    rng_w, rng_b = spec_w.rng(), spec_b.rng()
    wl = _C.conv_weight_layout(layer.weight.mean.detach().contiguous(), layer.weight.scale.detach().contiguous())
    mu_b = layer.bias.mean.detach().contiguous()
    sigma_b = _C.stddev(layer.bias.scale.detach().contiguous())
    geom = _C.conv3d_geom(B, *out_size, Cout, *size, Cin, k, s, p, (1, 1, 1))
    M = B * vox_in
    x = torch.randn(S * B, Cin, *size, device="cuda").contiguous(memory_format=torch.channels_last_3d)
    dy = torch.randn(S * B, Cout, *out_size, device="cuda").contiguous(memory_format=torch.channels_last_3d)
    y = torch.empty(S * B, Cout, *out_size, device="cuda").contiguous(memory_format=torch.channels_last_3d)
    dx = torch.empty_like(x)
    grads = torch.zeros(2, layer.weight.mean.numel(), device="cuda")
    sb = spec_w.sample_begin

    def impl_fwd():
        assert _C.try_sampled_conv_transpose3d_fwd(x, M * Cin, wl[0], wl[1], mu_b, sigma_b, None, None, y, geom, S, sb,
                                                   rng_w, rng_b)

    def impl_dgrad():
        _C.sampled_conv_transpose3d_dgrad(dy, wl[0], wl[1], None, dx, M * Cin, geom, S, sb, rng_w)

    def impl_wgrad():
        _C.sampled_conv_transpose3d_wgrad(dy, x, M * Cin, wl[2], None, grads[0], grads[1], geom, S, sb, rng_w)

    # the reference's form: W_s materialised, one torch call per sample (cudnn, TF32 allowed)
    mu_w, rho_w = layer.weight.mean.detach(), layer.weight.scale.detach()
    sigma_w = _C.stddev(rho_w.contiguous())
    x_n, dy_n = x.contiguous(), dy.contiguous()
    sl, pl = list(s), list(p)

    def ref_fwd():
        Ws = _C.materialize(mu_w.contiguous(), sigma_w, S, sb, rng_w)
        bs = _C.materialize(mu_b, sigma_b, S, spec_b.sample_begin, rng_b)
        for i in range(S):
            F.conv_transpose3d(x_n[i * B:(i + 1) * B], Ws[i], bs[i], s, p)

    def ref_dgrad():
        Ws = _C.materialize(mu_w.contiguous(), sigma_w, S, sb, rng_w)
        for i in range(S):
            torch.ops.aten.convolution_backward(dy_n[i * B:(i + 1) * B], x_n[i * B:(i + 1) * B], Ws[i], None, sl, pl,
                                                [1, 1, 1], True, [0, 0, 0], 1, [True, False, False])

    def ref_wgrad():
        Ws, eps = _C.materialize(mu_w.contiguous(), sigma_w, S, sb, rng_w, want_eps=True)
        gm, gs = torch.zeros_like(mu_w), torch.zeros_like(mu_w)
        for i in range(S):
            g = torch.ops.aten.convolution_backward(dy_n[i * B:(i + 1) * B], x_n[i * B:(i + 1) * B], Ws[i], None, sl, pl,
                                                    [1, 1, 1], True, [0, 0, 0], 1, [False, True, False])[1]
            gm += g
            gs += g * eps[i]
        gs *= torch.sigmoid(rho_w)

    W0 = mu_w.contiguous()

    def cudnn_fwd():
        F.conv_transpose3d(x_n, W0, mu_b, s, p)

    def cudnn_dgrad():
        torch.ops.aten.convolution_backward(dy_n, x_n, W0, None, sl, pl, [1, 1, 1], True, [0, 0, 0], 1,
                                            [True, False, False])

    def cudnn_wgrad():
        torch.ops.aten.convolution_backward(dy_n, x_n, W0, None, sl, pl, [1, 1, 1], True, [0, 0, 0], 1,
                                            [False, True, False])

    # what the default NCDHW-contiguous output format adds to the implicit forward: one conversion of y
    def nchw_conversion():
        y.contiguous()

    arms = {"implicit": (impl_fwd, impl_dgrad, impl_wgrad), "reference": (ref_fwd, ref_dgrad, ref_wgrad),
            "cudnn_fixed_weight": (cudnn_fwd, cudnn_dgrad, cudnn_wgrad)}
    out = {"shape": dict(c, out_size=out_size), "flops_per_pass": flops,
           "forward_launches": len(_C.conv_transpose3d_phases(geom)), "arms": {}}
    for arm, fns in arms.items():
        out["arms"][arm] = {}
        for pas, fn in zip(("fwd", "dgrad", "wgrad"), fns):
            ms = timed(fn, min_seconds)
            out["arms"][arm][pas] = {"ms": round(ms, 4), "tflops": round(flops / ms / 1e9, 1)}
    out["nchw_output_conversion_ms"] = round(timed(nchw_conversion, min_seconds), 4)
    imp = out["arms"]["implicit"]
    out["implicit_fraction_of_cudnn"] = {pas: round(out["arms"]["cudnn_fixed_weight"][pas]["ms"] / imp[pas]["ms"], 3)
                                         for pas in imp}
    out["implicit_speedup_over_reference"] = {pas: round(out["arms"]["reference"][pas]["ms"] / imp[pas]["ms"], 2)
                                              for pas in imp}
    if name == "V1":
        y_bytes = 4.0 * S * B * out_size[0] * out_size[1] * out_size[2] * Cout
        bound_ms = y_bytes / HBM_BYTES_PER_S * 1e3
        out["fwd_output_write_bound"] = {"bytes": y_bytes, "ms_at_7.7TBps": round(bound_ms, 4),
                                         "implicit_fwd_fraction_of_bound": round(bound_ms / imp["fwd"]["ms"], 3)}
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--shapes", default="V1,V2,V3")
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_conv_transpose3d: needs a CUDA device (B200)")
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    bnn.set_precision("tf32")
    bnn.manual_seed(1)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    res = {"card": card[torch.cuda.current_device()] if card else torch.cuda.get_device_name(),
           "precision": "tf32",
           "phase_launches": "one launch of the data-gradient kernel per output phase (sd * sh * sw launches), each with "
                             "its own rank-5 im2col corners, tap list and phase output view",
           "l2": "256 MiB buffer overwritten between passes",
           "shapes": {}}
    for name in args.shapes.split(","):
        res["shapes"][name] = bench_shape(name, SHAPES[name], args.min_seconds)
    doc = json.dumps(res, indent=1)
    print(doc)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(doc + "\n")


if __name__ == "__main__":
    main()
