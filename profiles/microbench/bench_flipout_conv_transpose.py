"""Flipout transposed convolution (FlipOutNormalConvTranspose2d / 3d), TF32: the layer's forward and forward + backward on
two arms, and the two sign passes alone.

  kernels    the layer's default path: two contractions of the transposed-convolution kernels (injected eps = 0) per
             pass, bnn_flipout_split / bnn_flipout_combine around them
  composite  set_flipout_conv_kernels(False): the reference's composite, conv_transpose(x, mean) + R o
             conv_transpose(x o S, stddev) with torch's cuDNN convolutions in TF32

  D1  (128 -> 128, k4 s2 p1, 8x8 -> 16x16, B 512, S 16)   the decoder workloads of bench_conv_transpose.py; the layer's
  D2  (64 -> 32, k3 s2 p1 op1, 16x16 -> 32x32, B 256, S 8)  signs are per example, so the Monte-Carlo pass is S*B rows
  V2  (64 -> 64, k4 s2 p1, 8^3 -> 16^3, B 16, S 8)          of bench_conv_transpose3d.py

The sign passes are timed on the shapes the layer gives them: split of the input (NCHW -> channels-last copy + signed
copy, 12 bytes per element) and combine into the NCHW output (two channels-last reads, one write, 12 bytes per element),
plus the layout-preserving forms (8 and 12 bytes per element); GB/s against the 6472 GB/s measured copy bandwidth
(DESIGN §4).  CUDA events over >= --min-seconds per measurement, a 256 MiB buffer overwritten before every pass so that
no operand comes from L2.  Both arms' outputs and gradients are compared at the timed sizes.  The card name and power
limit are read in the same run.

    python profiles/microbench/bench_flipout_conv_transpose.py --out profiles/r05_bench_flipout_conv_transpose.json
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))

import bayesianneuralnetworks_b200 as bnn                                          # noqa: E402
from bayesianneuralnetworks_b200 import _C                                         # noqa: E402
from bayesianneuralnetworks_b200.nn import (FlipOutNormalConvTranspose2d,          # noqa: E402
                                            FlipOutNormalConvTranspose3d)
from bayesianneuralnetworks_b200.nn.flipout import set_flipout_conv_kernels        # noqa: E402

SHAPES = {
    "D1": dict(cls=FlipOutNormalConvTranspose2d, Cin=128, Cout=128, k=4, s=2, p=1, op=0, size=(8, 8), B=512, S=16),
    "D2": dict(cls=FlipOutNormalConvTranspose2d, Cin=64, Cout=32, k=3, s=2, p=1, op=1, size=(16, 16), B=256, S=8),
    "V2": dict(cls=FlipOutNormalConvTranspose3d, Cin=64, Cout=64, k=4, s=2, p=1, op=0, size=(8, 8, 8), B=16, S=8),
}
COPY_GBS = 6472.0                  # measured HBM copy bandwidth of the B200 (MEASURED_PEAKS.json, DESIGN §4)

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


def rel_err(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))


def bench_shape(c, min_seconds):
    rows = c["S"] * c["B"]
    layer = c["cls"](c["Cin"], c["Cout"], c["k"], stride=c["s"], padding=c["p"], output_padding=c["op"]).cuda()
    x = torch.randn((rows, c["Cin"]) + c["size"], device="cuda", requires_grad=True)
    res = {"rows": rows}

    # both arms on the same signs and weights: outputs and gradients agree
    outs = {}
    for arm, on in (("kernels", True), ("composite", False)):
        set_flipout_conv_kernels(on)
        layer.zero_grad()
        x.grad = None
        y = layer(x, sample=arm == "kernels")
        g = torch.randn_like(y) if arm == "kernels" else outs["kernels"][-1]
        y.backward(g)
        outs[arm] = (y.detach(), x.grad.clone(), layer.weight.mean.grad.clone(), layer.weight.scale.grad.clone(), g)
        del y
    res["max_rel_err_kernels_vs_composite"] = {n: rel_err(a, b) for n, a, b in
                                               zip(("y", "dx", "d mean", "d scale"), outs["kernels"], outs["composite"])}
    g = outs["kernels"][-1]
    y_shape = tuple(outs["kernels"][0].shape)
    del outs

    def fwd():
        with torch.no_grad():
            layer(x)

    def fwd_bwd():
        layer(x).backward(g)

    for arm, on in (("kernels", True), ("composite", False), ("kernels", True), ("composite", False)):
        set_flipout_conv_kernels(on)                 # alternated: two windows per arm
        t = {"forward_ms": timed(fwd, min_seconds), "forward_backward_ms": timed(fwd_bwd, min_seconds)}
        for key, v in t.items():
            res.setdefault(arm, {}).setdefault(key, []).append(round(v, 4))
    set_flipout_conv_kernels(True)
    for arm in ("kernels", "composite"):
        for key in ("forward_ms", "forward_backward_ms"):
            res[arm][key + "_mean"] = round(sum(res[arm][key]) / len(res[arm][key]), 4)
    res["speedup_forward"] = round(res["composite"]["forward_ms_mean"] / res["kernels"]["forward_ms_mean"], 3)
    res["speedup_forward_backward"] = round(res["composite"]["forward_backward_ms_mean"] /
                                            res["kernels"]["forward_backward_ms_mean"], 3)

    # the sign passes alone, on this layer's tensors
    fmt = torch.channels_last if len(c["size"]) == 2 else torch.channels_last_3d
    xin = x.detach()
    sin = (torch.rand(rows, c["Cin"], device="cuda") - .5).sign()
    sout = (torch.rand(rows, c["Cout"], device="cuda") - .5).sign()
    ya = torch.randn(y_shape, device="cuda").contiguous(memory_format=fmt)
    yb = torch.randn(y_shape, device="cuda").contiguous(memory_format=fmt)
    xcl = xin.contiguous(memory_format=fmt)
    passes = {
        "split_nchw_input": (lambda: _C.flipout_split(xin, sin), 12 * xin.numel()),
        "split_channels_last_input": (lambda: _C.flipout_split(xcl, sin), 8 * xin.numel()),
        "combine_to_nchw_output": (lambda: _C.flipout_combine(ya, yb, sout, channels_last=False), 12 * ya.numel()),
        "combine_to_channels_last_output": (lambda: _C.flipout_combine(ya, yb, sout, channels_last=True), 12 * ya.numel()),
    }
    res["sign_passes"] = {}
    for name, (fn, nbytes) in passes.items():
        ms = timed(fn, min_seconds / 2)
        gbs = nbytes / (ms * 1e-3) / 1e9
        res["sign_passes"][name] = {"ms": round(ms, 4), "bytes": nbytes, "GB_per_s": round(gbs, 1),
                                    "fraction_of_copy": round(gbs / COPY_GBS, 3)}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="D1,D2,V2")
    ap.add_argument("--min-seconds", type=float, default=0.5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_flipout_conv_transpose: needs a CUDA device (B200)")
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    bnn.set_precision("tf32")
    bnn.manual_seed(1)
    torch.manual_seed(1)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    res = {"card": card[torch.cuda.current_device()] if card else torch.cuda.get_device_name(),
           "precision": "tf32",
           "l2": "256 MiB buffer overwritten before every pass",
           "copy_GB_per_s": COPY_GBS,
           "shapes": {}}
    for name in args.shapes.split(","):
        res["shapes"][name] = bench_shape(SHAPES[name], args.min_seconds)
        torch.cuda.empty_cache()
    doc = json.dumps(res, indent=1)
    print(doc)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(doc + "\n")


if __name__ == "__main__":
    main()
