"""Forward, input gradient and weight gradient of two Bayesian decoder layers (NormalConvTranspose2d), TF32, per pass:

  implicit   this library's kernels: the phase-decomposed transposed-filter gather (forward, one launch per output phase),
             the conv view's implicit-GEMM forward (input gradient) and weight gradient — bnn_sampled_conv_transpose2d_*
  explicit   the explicit lowering in the same column order: bnn_sampled_gemm_dgrad + bnn_col2im_nhwc (+ sampled bias),
             bnn_im2col_nhwc + bnn_sampled_gemm_fwd / _wgrad
  reference  the reference's form: materialised W_s and one torch conv_transpose2d (or its backward) per sample
  cudnn      one fixed weight, torch conv_transpose2d batched over S*B rows with allow_tf32 — the same flops without
             sampling, a ceiling

  D1  NormalConvTranspose2d(128, 128, 4, stride=2, padding=1), 8x8 -> 16x16, B = 512, S = 16 (the C3 conv layer's scale,
      mirrored)
  D2  NormalConvTranspose2d(64, 32, 3, stride=2, padding=1, output_padding=1), 16x16 -> 32x32, B = 256, S = 8 (uneven
      phases: 4, 2, 2 and 1 taps)

CUDA events around each pass over a window of >= 1 s per (shape, arm, pass), a 256 MiB buffer overwritten between passes
so that no operand is served from L2.  Algorithmic TFLOP/s = 2 S B Hin Win Cin Cout KH KW / t for every pass.  Prints one
JSON document (and writes it to --out).

    python profiles/microbench/bench_conv_transpose.py --out profiles/r03_bench_conv_transpose.json
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
from bayesianneuralnetworks_b200.nn import NormalConvTranspose2d  # noqa: E402

SHAPES = {
    "D1": dict(Cin=128, Cout=128, k=4, s=2, p=1, op=0, H=8, B=512, S=16),
    "D2": dict(Cin=64, Cout=32, k=3, s=2, p=1, op=1, H=16, B=256, S=8),
}

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
    Cin, Cout, k, s, p, op, H, B, S = (c[n] for n in ("Cin", "Cout", "k", "s", "p", "op", "H", "B", "S"))
    OH = (H - 1) * s - 2 * p + (k - 1) + op + 1
    flops = 2.0 * S * B * H * H * Cin * Cout * k * k
    layer = NormalConvTranspose2d(Cin, Cout, k, stride=s, padding=p, output_padding=op).cuda()
    spec_w, spec_b = layer._draws(True, S, 0, S)
    rng_w, rng_b = spec_w.rng(), spec_b.rng()
    wl = _C.conv_weight_layout(layer.weight.mean.detach().contiguous(), layer.weight.scale.detach().contiguous())
    mu_b = layer.bias.mean.detach().contiguous()
    sigma_b = _C.stddev(layer.bias.scale.detach().contiguous())
    geom = _C.conv_geom(B, OH, OH, Cout, H, H, Cin, k, k, (s, s), (p, p), (1, 1))
    M, K = B * H * H, k * k * Cout
    x = torch.randn(S * B, Cin, H, H, device="cuda").contiguous(memory_format=torch.channels_last)
    dy = torch.randn(S * B, Cout, OH, OH, device="cuda").contiguous(memory_format=torch.channels_last)
    y = torch.empty(S * B, Cout, OH, OH, device="cuda").contiguous(memory_format=torch.channels_last)
    dx = torch.empty_like(x)
    grads = torch.zeros(2, Cin * K, device="cuda")
    x_rows = x.permute(0, 2, 3, 1).reshape(S * M, Cin)
    col = torch.empty(S * M, K, device="cuda")
    sb = spec_w.sample_begin

    def impl_fwd():
        assert _C.try_sampled_conv_transpose2d_fwd(x, M * Cin, wl[0], wl[1], mu_b, sigma_b, None, None, y, geom, S, sb,
                                                   rng_w, rng_b)

    def impl_dgrad():
        assert _C.try_sampled_conv_transpose2d_dgrad(dy, wl[0], wl[1], None, dx, M * Cin, geom, S, sb, rng_w)

    def impl_wgrad():
        assert _C.try_sampled_conv_transpose2d_wgrad(dy, x, M * Cin, wl[2], None, grads[0], grads[1], geom, S, sb, rng_w)

    def expl_fwd():
        _C.sampled_gemm_dgrad(_C.make_view(x_rows.data_ptr(), Cin, 1), M * Cin, wl[0], wl[1], None, col, K, M * K, M, Cin,
                              K, S, sb, rng_w, _C.PREC_TF32)
        _C.col2im_nhwc(col, y, geom, S * B)
        b = _C.materialize(mu_b, sigma_b, S, spec_b.sample_begin, rng_b)
        y.view(S, B, Cout, OH, OH).add_(b[:, None, :, None, None])

    def expl_dgrad():
        c2 = _C.im2col_nhwc(dy, geom, S * B)
        _C.sampled_gemm_fwd(c2, K, M * K, wl[0], wl[1], None, None, None, None, _C.make_view(dx.data_ptr(), Cin, 1),
                            M * Cin, M, Cin, K, S, sb, rng_w, None, _C.PREC_TF32)

    def expl_wgrad():
        c2 = _C.im2col_nhwc(dy, geom, S * B)
        _C.sampled_gemm_wgrad(_C.make_view(x_rows.data_ptr(), Cin, 1), M * Cin, c2, K, M * K, wl[2], None, grads[0],
                              grads[1], M, Cin, K, S, sb, rng_w, _C.PREC_TF32)

    # the reference's form: W_s materialised, one torch call per sample (cudnn, TF32 allowed)
    mu_w, rho_w = layer.weight.mean.detach(), layer.weight.scale.detach()
    sigma_w = _C.stddev(rho_w.contiguous())
    x_n, dy_n = x.contiguous(), dy.contiguous()

    def ref_fwd():
        Ws = _C.materialize(mu_w.contiguous(), sigma_w, S, sb, rng_w)
        bs = _C.materialize(mu_b, sigma_b, S, spec_b.sample_begin, rng_b)
        for i in range(S):
            F.conv_transpose2d(x_n[i * B:(i + 1) * B], Ws[i], bs[i], s, p, op)

    def ref_dgrad():
        Ws = _C.materialize(mu_w.contiguous(), sigma_w, S, sb, rng_w)
        for i in range(S):
            torch.ops.aten.convolution_backward(dy_n[i * B:(i + 1) * B], x_n[i * B:(i + 1) * B], Ws[i], None, [s, s],
                                                [p, p], [1, 1], True, [op, op], 1, [True, False, False])

    def ref_wgrad():
        Ws, eps = _C.materialize(mu_w.contiguous(), sigma_w, S, sb, rng_w, want_eps=True)
        gm, gs = torch.zeros_like(mu_w), torch.zeros_like(mu_w)
        for i in range(S):
            g = torch.ops.aten.convolution_backward(dy_n[i * B:(i + 1) * B], x_n[i * B:(i + 1) * B], Ws[i], None, [s, s],
                                                    [p, p], [1, 1], True, [op, op], 1, [False, True, False])[1]
            gm += g
            gs += g * eps[i]
        gs *= torch.sigmoid(rho_w)

    W0 = mu_w.contiguous()

    def cudnn_fwd():
        F.conv_transpose2d(x_n, W0, mu_b, s, p, op)

    def cudnn_dgrad():
        torch.ops.aten.convolution_backward(dy_n, x_n, W0, None, [s, s], [p, p], [1, 1], True, [op, op], 1,
                                            [True, False, False])

    def cudnn_wgrad():
        torch.ops.aten.convolution_backward(dy_n, x_n, W0, None, [s, s], [p, p], [1, 1], True, [op, op], 1,
                                            [False, True, False])

    # what the default NCHW-contiguous output format adds to the implicit forward: one conversion of y
    def nchw_conversion():
        y.contiguous()

    arms = {"implicit": (impl_fwd, impl_dgrad, impl_wgrad), "explicit": (expl_fwd, expl_dgrad, expl_wgrad),
            "reference": (ref_fwd, ref_dgrad, ref_wgrad), "cudnn_fixed_weight": (cudnn_fwd, cudnn_dgrad, cudnn_wgrad)}
    out = {"shape": dict(c, OH=OH), "flops_per_pass": flops, "arms": {}}
    for arm, fns in arms.items():
        out["arms"][arm] = {}
        for pas, fn in zip(("fwd", "dgrad", "wgrad"), fns):
            ms = timed(fn, min_seconds)
            out["arms"][arm][pas] = {"ms": round(ms, 4), "tflops": round(flops / ms / 1e9, 1)}
    out["nchw_output_conversion_ms"] = round(timed(nchw_conversion, min_seconds), 4)
    imp = out["arms"]["implicit"]
    out["implicit_fraction_of_cudnn"] = {pas: round(out["arms"]["cudnn_fixed_weight"][pas]["ms"] / imp[pas]["ms"], 3)
                                         for pas in imp}
    out["implicit_beats_explicit_and_reference"] = {
        pas: imp[pas]["ms"] < out["arms"]["explicit"][pas]["ms"] and imp[pas]["ms"] < out["arms"]["reference"][pas]["ms"]
        for pas in imp}
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--shapes", default="D1,D2")
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_conv_transpose: needs a CUDA device (B200)")
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    bnn.set_precision("tf32")
    bnn.manual_seed(1)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    res = {"card": card[torch.cuda.current_device()] if card else torch.cuda.get_device_name(),
           "precision": "tf32",
           "phase_launches": "one launch of the data-gradient kernel per output phase (sh * sw launches), each with its "
                             "own im2col corners, tap list and phase output view; phases without a tap: one bias kernel",
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
