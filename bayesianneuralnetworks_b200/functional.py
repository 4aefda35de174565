"""torch.autograd glue around the C ABI: each Function forwards to the CUDA library on the current
stream and implements the closed-form backward of SURVEY §3.2 with the fused kernels (eps is
regenerated from the Philox counters, never stored).  No CPU path: non-CUDA tensors raise.
"""
import math

import torch

from . import _C


class DrawSpec:
    """Which eps a launch uses: Philox (seed, tensor_id, [sample_begin, sample_begin+S)) or an
    injected tensor [S, numel] (tests).  `step_dev` (optional int64[1] device tensor) is added to the
    Philox step word inside the kernels (CUDA-graph replays, runtime.graph_safe_rng)."""
    __slots__ = ("seed", "tensor_id", "sample_begin", "step", "eps", "step_dev", "signs")

    def __init__(self, seed, tensor_id, draw_begin, eps=None, step_dev=None, signs=None):
        self.seed = seed
        self.tensor_id = tensor_id
        self.sample_begin = draw_begin & 0xFFFFFFFF
        self.step = draw_begin >> 32
        self.eps = eps
        self.step_dev = step_dev
        self.signs = signs            # (R [S, out], S [S, in]): rank-one sign noise instead of Philox normals (Flipout)

    def rng(self, elem_offset=0):
        return _C.make_rng(self.seed, self.step, self.tensor_id, elem_offset=elem_offset, step_dev=self.step_dev,
                           signs=self.signs, sample_begin=self.sample_begin)


def _check_f32_cuda(name, t):
    if t is None:
        return
    _C.require_cuda(t)
    if t.dtype != torch.float32:
        raise TypeError(f"{name}: the variational hot path computes in float32, got {t.dtype}")


def _zero_grads(w_shape, n_bias, device):
    """Zeroed accumulators [2, *w_shape] (d mean, d scale of the weight) and [2, n_bias] (of the bias) carved out of ONE
    buffer: the gradient kernels accumulate into them, so a layer's backward needs a single fill."""
    nw = 2 * math.prod(w_shape) if w_shape is not None else 0
    nb = 2 * n_bias if n_bias is not None else 0
    if nw + nb == 0:
        return None, None
    flat = torch.zeros(nw + nb, device=device, dtype=torch.float32)
    grads = flat[:nw].view((2,) + tuple(w_shape)) if nw else None
    bg = flat[nw:].view(2, n_bias) if nb else None
    return grads, bg


def _eps_slice(spec, S, numel, lo=None, hi=None):
    """Injected eps as a contiguous [S, n] block (optionally the [lo, hi) slice of every sample)."""
    if spec is None or spec.eps is None:
        return None
    e = spec.eps.reshape(S, numel)
    if lo is not None:
        e = e[:, lo:hi]
    return e.contiguous()


# ------------------------------------------------------------------------------------------------
class SampledLinear(torch.autograd.Function):
    """y[s] = x[s] W_s^T + b_s for S Monte-Carlo samples in one launch (dense.py:46-60).

    x: [R, K] with R = S*M rows (sample-major) or, when `shared`, [M, K] used by every sample.
    Returns [S*M, N]."""

    @staticmethod
    def forward(ctx, x, mu_w, rho_w, mu_b, rho_b, S, shared, spec_w, spec_b, precision):
        for n, t in (("input", x), ("weight.mean", mu_w), ("weight.scale", rho_w), ("bias.mean", mu_b),
                     ("bias.scale", rho_b)):
            _check_f32_cuda(n, t)
        x = x.contiguous()
        N, K = mu_w.shape
        if x.dim() != 2 or x.shape[1] != K:
            raise RuntimeError(f"sampled linear: input {tuple(x.shape)} does not match in_features {K}")
        rows = x.shape[0]
        M = rows if shared else rows // S
        if not shared and M * S != rows:
            raise RuntimeError(f"sampled linear: {rows} rows are not divisible by {S} Monte-Carlo samples")
        mu_w_c, rho_w_c = mu_w.contiguous(), rho_w.contiguous()
        sigma_w = _C.stddev(rho_w_c)
        has_bias = mu_b is not None
        sigma_b = _C.stddev(rho_b.contiguous()) if has_bias else None
        y = torch.empty((S * M, N), device=x.device, dtype=torch.float32)
        _C.sampled_gemm_fwd(x, K, 0 if shared else M * K, mu_w_c, sigma_w,
                            mu_b.contiguous() if has_bias else None, sigma_b,
                            _eps_slice(spec_w, S, N * K), _eps_slice(spec_b, S, N) if has_bias else None,
                            _C.make_view(y.data_ptr(), N, 1), M * N, M, N, K, S, spec_w.sample_begin,
                            spec_w.rng(), spec_b.rng() if has_bias else None, precision)
        ctx.save_for_backward(x, mu_w_c, rho_w_c, sigma_w, rho_b)
        ctx.meta = (S, shared, spec_w, spec_b, precision, M, N, K)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, mu_w, rho_w, sigma_w, rho_b = ctx.saved_tensors
        S, shared, spec_w, spec_b, precision, M, N, K = ctx.meta
        ldy = N
        if precision == _C.PREC_TF32 and N % 4 != 0:
            # the TMA-fed kernels need a 16-byte row pitch: pad the (narrow) gradient rows, e.g. a 10-class head
            ldy = (N + 3) // 4 * 4
            dy = torch.nn.functional.pad(dy, (0, ldy - N))
        dy = dy.contiguous()
        dy_view = _C.make_view(dy.data_ptr(), ldy, 1)
        eps_w = _eps_slice(spec_w, S, N * K)
        a_stride = 0 if shared else M * K
        dx = dmu_w = drho_w = dmu_b = drho_b = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            _C.sampled_gemm_dgrad(dy_view, M * ldy, mu_w, sigma_w, eps_w, dx, K, a_stride, M, N, K, S,
                                  spec_w.sample_begin, spec_w.rng(), precision)
        need_w = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
        need_b = rho_b is not None and (ctx.needs_input_grad[3] or ctx.needs_input_grad[4])
        grads, bg = _zero_grads((N, K) if need_w else None, N if need_b else None, x.device)
        if need_w:
            dmu_w, drho_w = grads[0], grads[1]
            _C.sampled_gemm_wgrad(dy_view, M * ldy, x, K, a_stride, rho_w, eps_w, dmu_w, drho_w, M, N, K, S,
                                  spec_w.sample_begin, spec_w.rng(), precision)
        if need_b:
            dmu_b, drho_b = bg[0], bg[1]
            _C.bias_grad(dy_view, M * ldy, rho_b.contiguous(), _eps_slice(spec_b, S, N), dmu_b, drho_b, M, N, S,
                         spec_b.sample_begin, spec_b.rng())
        return dx, dmu_w, drho_w, dmu_b, drho_b, None, None, None, None, None


# ------------------------------------------------------------------------------------------------
def _conv_out(size, k, s, p, d):
    return (size + 2 * p - d * (k - 1) - 1) // s + 1


_KEEP_COL_BYTES = 2 << 30      # im2col matrices up to this size are kept from forward to backward


class SampledConv2d(torch.autograd.Function):
    """y[s] = conv2d(x[s], W_s, b_s) for S samples (conv.py:65-73,112-119): im2col lowering of the
    activations per group, then the sampled GEMM writing straight into the NCHW output.

    x: [S*B, C, H, W] (sample-major) or, when `shared`, [B, C, H, W].  Returns [S*B, Cout, OH, OW]."""

    @staticmethod
    def forward(ctx, x, mu_w, rho_w, mu_b, rho_b, S, shared, spec_w, spec_b, precision, stride, padding,
                dilation, groups):
        for n, t in (("input", x), ("weight.mean", mu_w), ("weight.scale", rho_w), ("bias.mean", mu_b),
                     ("bias.scale", rho_b)):
            _check_f32_cuda(n, t)
        x = x.contiguous()
        Cout, Cg, KH, KW = mu_w.shape
        if x.dim() != 4 or x.shape[1] != Cg * groups:
            raise RuntimeError(f"sampled conv2d: input {tuple(x.shape)} does not match weight {tuple(mu_w.shape)} "
                               f"with groups={groups}")
        rows, C, H, W = x.shape
        B = rows if shared else rows // S
        if not shared and B * S != rows:
            raise RuntimeError(f"sampled conv2d: batch {rows} is not divisible by {S} Monte-Carlo samples")
        OH = _conv_out(H, KH, stride[0], padding[0], dilation[0])
        OW = _conv_out(W, KW, stride[1], padding[1], dilation[1])
        if OH <= 0 or OW <= 0:
            raise RuntimeError("sampled conv2d: empty output")
        geo = (B, C, H, W, Cout, Cg, KH, KW, OH, OW, tuple(stride), tuple(padding), tuple(dilation), groups)
        mu_w_c, rho_w_c = mu_w.contiguous(), rho_w.contiguous()
        sigma_w = _C.stddev(rho_w_c)
        has_bias = mu_b is not None
        mu_b_c = mu_b.contiguous() if has_bias else None
        sigma_b = _C.stddev(rho_b.contiguous()) if has_bias else None
        y = torch.empty((S * B, Cout, OH, OW), device=x.device, dtype=torch.float32)
        Ng, Kg, P = Cout // groups, Cg * KH * KW, OH * OW
        M = B * P
        col = torch.empty((rows * P, Kg), device=x.device, dtype=torch.float32)
        for g in range(groups):
            _C.im2col(x, col, SampledConv2d._geom(rows, geo, g))
            lo, hi = g * Ng * Kg, (g + 1) * Ng * Kg
            view = _C.make_view(y.data_ptr() + 4 * g * Ng * P, Cout * P, P)
            _C.sampled_gemm_fwd(col, Kg, 0 if shared else M * Kg, mu_w_c.view(-1)[lo:hi], sigma_w.view(-1)[lo:hi],
                                mu_b_c[g * Ng:(g + 1) * Ng] if has_bias else None,
                                sigma_b[g * Ng:(g + 1) * Ng] if has_bias else None,
                                _eps_slice(spec_w, S, Cout * Kg, lo, hi),
                                _eps_slice(spec_b, S, Cout, g * Ng, (g + 1) * Ng) if has_bias else None,
                                view, B * Cout * P, M, Ng, Kg, S, spec_w.sample_begin, spec_w.rng(lo),
                                spec_b.rng(g * Ng) if has_bias else None, precision)
        ctx.save_for_backward(x, mu_w_c, rho_w_c, sigma_w, rho_b)
        ctx.meta = (S, shared, spec_w, spec_b, precision, geo)
        # the weight gradient contracts dY with the same im2col matrix: keep it for the backward pass instead of
        # lowering x a second time (one launch and one write of the matrix less), unless it is very large
        keep = groups == 1 and (ctx.needs_input_grad[1] or ctx.needs_input_grad[2]) and col.numel() * 4 <= _KEEP_COL_BYTES
        ctx.col = col if keep else None
        return y

    @staticmethod
    def _geom(batch, geo, g):
        B, C, H, W, Cout, Cg, KH, KW, OH, OW, stride, padding, dilation, groups = geo
        return _C.bnn_conv2d_geom(batch, C, H, W, g * Cg, Cg, KH, KW, OH, OW, stride[0], stride[1],
                                  padding[0], padding[1], dilation[0], dilation[1])

    @staticmethod
    def backward(ctx, dy):
        x, mu_w, rho_w, sigma_w, rho_b = ctx.saved_tensors
        S, shared, spec_w, spec_b, precision, geo = ctx.meta
        B, C, H, W, Cout, Cg, KH, KW, OH, OW, stride, padding, dilation, groups = geo
        dy = dy.contiguous()
        rows = x.shape[0]
        Ng, Kg, P = Cout // groups, Cg * KH * KW, OH * OW
        M = B * P
        a_stride = 0 if shared else M * Kg
        # TF32: hand dY to the kernels as a row-major [S*B*P, Cout] matrix (one strided copy), which makes the
        # TMA-fed data- and weight-gradient kernels eligible; fp32 mode reads the NCHW tensor in place.
        rowmajor_dy = precision == _C.PREC_TF32 and P > 1 and Cout % 4 == 0 and Ng % 4 == 0
        if rowmajor_dy:
            dy_rows = dy.view(S * B, Cout, P).transpose(1, 2).contiguous()
        need_x = ctx.needs_input_grad[0]
        need_w = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
        need_b = rho_b is not None and (ctx.needs_input_grad[3] or ctx.needs_input_grad[4])
        dx = torch.empty_like(x) if need_x else None
        grads, bg = _zero_grads(tuple(mu_w.shape) if need_w else None, Cout if need_b else None, x.device)
        kept = ctx.col if need_w else None
        ctx.col = None
        col = kept if kept is not None else (
            torch.empty((rows * P, Kg), device=x.device, dtype=torch.float32) if need_w else None)
        dcol = torch.empty((rows * P, Kg), device=x.device, dtype=torch.float32) if need_x else None
        for g in range(groups):
            lo, hi = g * Ng * Kg, (g + 1) * Ng * Kg
            if rowmajor_dy:
                dy_view, dy_ss = _C.make_view(dy_rows.data_ptr() + 4 * g * Ng, Cout, 1), M * Cout
            else:
                dy_view, dy_ss = _C.make_view(dy.data_ptr() + 4 * g * Ng * P, Cout * P, P), B * Cout * P
            eps_w = _eps_slice(spec_w, S, Cout * Kg, lo, hi)
            geom = SampledConv2d._geom(rows, geo, g)
            if need_x:
                _C.sampled_gemm_dgrad(dy_view, dy_ss, mu_w.view(-1)[lo:hi], sigma_w.view(-1)[lo:hi], eps_w,
                                      dcol, Kg, a_stride, M, Ng, Kg, S, spec_w.sample_begin, spec_w.rng(lo),
                                      precision)
                _C.col2im(dcol, dx, geom, False)
            if need_w:
                if kept is None:
                    _C.im2col(x, col, geom)
                _C.sampled_gemm_wgrad(dy_view, dy_ss, col, Kg, a_stride, rho_w.view(-1)[lo:hi], eps_w,
                                      grads[0].view(-1)[lo:hi], grads[1].view(-1)[lo:hi], M, Ng, Kg, S,
                                      spec_w.sample_begin, spec_w.rng(lo), precision)
            if need_b:
                _C.bias_grad(dy_view, dy_ss, rho_b.contiguous()[g * Ng:(g + 1) * Ng],
                             _eps_slice(spec_b, S, Cout, g * Ng, (g + 1) * Ng), bg[0][g * Ng:(g + 1) * Ng],
                             bg[1][g * Ng:(g + 1) * Ng], M, Ng, S, spec_b.sample_begin, spec_b.rng(g * Ng))
        return (dx, grads[0] if need_w else None, grads[1] if need_w else None,
                bg[0] if need_b else None, bg[1] if need_b else None) + (None,) * 9


# ------------------------------------------------------------------------------------------------
def conv_implicit_eligible(in_channels, groups):
    """Layers whose eps stream is keyed in (o, kh, kw, c) order and that run the implicit-GEMM path (a STATIC property of
    the layer, so that forward, backward and `.sampled` agree whatever the precision mode or the input layout)."""
    return groups == 1 and in_channels % 32 == 0


_CONV_OUTPUT = {"format": "contiguous"}


def set_conv_output_format(fmt):
    """Memory format of the implicit-GEMM conv layers' OUTPUT: 'contiguous' (default: NCHW-contiguous, what the reference
    produces and what a following Flatten / view wants; the gradient that comes back is transposed to channels-last by one
    fused pass that also forms the bias gradient) or 'preserve' (torch's convention: a channels_last input gives a
    channels_last result — the choice for conv -> conv stacks kept in channels_last)."""
    if fmt not in ("contiguous", "preserve"):
        raise ValueError("conv output format must be 'contiguous' or 'preserve'")
    _CONV_OUTPUT["format"] = fmt


def conv_output_nchw(x):
    """Whether a conv layer's output is NC(D)HW-contiguous (set_conv_output_format): always under 'contiguous', and under
    'preserve' for an input that is."""
    return _CONV_OUTPUT["format"] == "contiguous" or x.is_contiguous()


def _nhwc(t):
    """(tensor whose memory is NHWC-contiguous, copied?) for a logical NCHW tensor."""
    if t.permute(0, 2, 3, 1).is_contiguous():
        return t
    return t.contiguous(memory_format=torch.channels_last)


class SampledConv2dImplicit(torch.autograd.Function):
    """y[s] = conv2d(x[s], W_s, b_s) for S samples (conv.py:65-73,112-119) WITHOUT an im2col matrix: channels-last
    activations reach the tensor cores through a TMA im2col tensor map, the weights are presented in (o, kh, kw, c) order
    (one small layout kernel per step, which also produces sigma), the input gradient of stride-1 layers is the
    transposed-filter gather, the weight gradient reads dY and x through tensor maps and is returned in OIHW order.
    TF32 mode; fp32 (3xTF32) mode, the input gradient of strided layers and every request the kernels refuse (stride > 8,
    a filter window outside the im2col descriptor's range, Cout % 32 != 0 for the input gradient or Cout % 4 != 0 for the
    weight gradient: the C entry point returns BNN_ERR_UNSUPPORTED before launching anything) lower explicitly in the
    same column order (bnn_im2col_nhwc / bnn_col2im_nhwc + the register-staged / TMA GEMM kernels).

    x: logical [S*B, C, H, W] (sample-major) or, when `shared`, [B, C, H, W]; any memory format — channels_last input gives
    a channels_last result under set_conv_output_format('preserve'); by default the result is NCHW-contiguous (written
    through the kernel's strided epilogue) and a contiguous NCHW input is converted once."""

    @staticmethod
    def forward(ctx, x, mu_w, rho_w, mu_b, rho_b, S, shared, spec_w, spec_b, precision, stride, padding, dilation):
        for n, t in (("input", x), ("weight.mean", mu_w), ("weight.scale", rho_w), ("bias.mean", mu_b),
                     ("bias.scale", rho_b)):
            _check_f32_cuda(n, t)
        Cout, C, KH, KW = mu_w.shape
        if x.dim() != 4 or x.shape[1] != C:
            raise RuntimeError(f"sampled conv2d: input {tuple(x.shape)} does not match weight {tuple(mu_w.shape)}")
        rows, _, H, W = x.shape
        B = rows if shared else rows // S
        if not shared and B * S != rows:
            raise RuntimeError(f"sampled conv2d: batch {rows} is not divisible by {S} Monte-Carlo samples")
        OH = _conv_out(H, KH, stride[0], padding[0], dilation[0])
        OW = _conv_out(W, KW, stride[1], padding[1], dilation[1])
        if OH <= 0 or OW <= 0:
            raise RuntimeError("sampled conv2d: empty output")
        nchw_out = _CONV_OUTPUT["format"] == "contiguous" or x.is_contiguous()
        x_cl = _nhwc(x)
        geom = _C.conv_geom(B, H, W, C, OH, OW, Cout, KH, KW, stride, padding, dilation)
        wl = _C.conv_weight_layout(mu_w.contiguous(), rho_w.contiguous())          # [3, numel]: mean, sigma, scale
        has_bias = mu_b is not None
        mu_b_c = mu_b.contiguous() if has_bias else None
        sigma_b = _C.stddev(rho_b.contiguous()) if has_bias else None
        P, K = OH * OW, KH * KW * C
        M = B * P
        y = torch.empty((S * B, Cout, OH, OW), device=x.device, dtype=torch.float32,
                        memory_format=torch.contiguous_format if nchw_out else torch.channels_last)
        if nchw_out:
            y_view, y_ss = _C.make_view(y.data_ptr(), Cout * P, P), B * Cout * P
        else:
            y_view, y_ss = _C.make_view(y.data_ptr(), Cout, 1), M * Cout
        eps_w = _eps_slice(spec_w, S, Cout * K)
        eps_b = _eps_slice(spec_b, S, Cout) if has_bias else None
        x_ss = 0 if shared else B * H * W * C
        done = precision == _C.PREC_TF32 and _C.try_sampled_conv2d_fwd(
            x_cl, x_ss, wl[0], wl[1], mu_b_c, sigma_b, eps_w, eps_b, y_view, y_ss, geom, S, spec_w.sample_begin,
            spec_w.rng(), spec_b.rng() if has_bias else None)
        if not done:
            col = _C.im2col_nhwc(x_cl, geom, rows)
            _C.sampled_gemm_fwd(col, K, 0 if shared else M * K, wl[0], wl[1], mu_b_c, sigma_b, eps_w, eps_b, y_view, y_ss,
                                M, Cout, K, S, spec_w.sample_begin, spec_w.rng(), spec_b.rng() if has_bias else None,
                                precision)
        ctx.save_for_backward(x_cl, wl, rho_b)
        ctx.meta = (S, shared, spec_w, spec_b, precision, geom, tuple(mu_w.shape), rows)
        return y

    @staticmethod
    def backward(ctx, dy):
        x_cl, wl, rho_b = ctx.saved_tensors
        S, shared, spec_w, spec_b, precision, geom, w_shape, rows = ctx.meta
        Cout, C, KH, KW = w_shape
        B, H, W, OH, OW = geom.B, geom.H, geom.W, geom.OH, geom.OW
        P, K = OH * OW, KH * KW * C
        M = B * P
        eps_w = _eps_slice(spec_w, S, Cout * K)
        x_ss = 0 if shared else B * H * W * C
        tf32 = precision == _C.PREC_TF32
        need_x = ctx.needs_input_grad[0]
        need_w = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
        need_b = rho_b is not None and (ctx.needs_input_grad[3] or ctx.needs_input_grad[4])
        # the gradient kernels read dY as rows [S*B*OH*OW, Cout]: free for a channels_last gradient; an NCHW-contiguous
        # one goes through ONE transposing pass that forms the bias gradient on the way
        bias_done = False
        bg_fused = None
        if dy.permute(0, 2, 3, 1).is_contiguous():
            dy_cl = dy
        else:
            dy_cl = None
            if dy.is_contiguous():
                if need_b:
                    bg_fused = torch.zeros((2, Cout), device=dy.device, dtype=torch.float32)
                dy_cl = _C.nchw_to_nhwc_bias_grad(dy, B, rho_b.contiguous() if need_b else None,
                                                  _eps_slice(spec_b, S, Cout) if need_b else None,
                                                  bg_fused[0] if need_b else None, bg_fused[1] if need_b else None,
                                                  spec_b.sample_begin if need_b else 0, spec_b.rng() if need_b else None)
                bias_done = dy_cl is not None and need_b
            if dy_cl is None:
                dy_cl = dy.contiguous(memory_format=torch.channels_last)
        dy_view, dy_ss = _C.make_view(dy_cl.data_ptr(), Cout, 1), M * Cout
        dx = None
        if need_x:
            dx = torch.empty(x_cl.shape, device=dy.device, dtype=torch.float32, memory_format=torch.channels_last)
            done = tf32 and _C.try_sampled_conv2d_dgrad(dy_cl, wl[0], wl[1], eps_w, dx, x_ss, geom, S,
                                                        spec_w.sample_begin, spec_w.rng())
            if not done:                                # strided / refused layers, fp32 mode: column gradients + gather
                dcol = torch.empty((rows * P, K), device=dy.device, dtype=torch.float32)
                _C.sampled_gemm_dgrad(dy_view, dy_ss, wl[0], wl[1], eps_w, dcol, K, 0 if shared else M * K, M, Cout, K, S,
                                      spec_w.sample_begin, spec_w.rng(), precision)
                _C.col2im_nhwc(dcol, dx, geom, rows)
        grads_p, bg = _zero_grads((Cout * K,) if need_w else None, Cout if (need_b and not bias_done) else None, dy.device)
        if bias_done:
            bg = bg_fused
        dmu = drho = None
        if need_w:
            done = tf32 and _C.try_sampled_conv2d_wgrad(dy_cl, x_cl, x_ss, wl[2], eps_w, grads_p[0], grads_p[1], geom, S,
                                                        spec_w.sample_begin, spec_w.rng())
            if not done:
                col = _C.im2col_nhwc(x_cl, geom, rows)
                _C.sampled_gemm_wgrad(dy_view, dy_ss, col, K, 0 if shared else M * K, wl[2], eps_w, grads_p[0], grads_p[1],
                                      M, Cout, K, S, spec_w.sample_begin, spec_w.rng(), precision)
            g = _C.conv_weight_unlayout(grads_p, w_shape)
            dmu, drho = g[0], g[1]
        if need_b and not bias_done:
            _C.bias_grad(dy_view, dy_ss, rho_b.contiguous(), _eps_slice(spec_b, S, Cout), bg[0], bg[1], M, Cout, S,
                         spec_b.sample_begin, spec_b.rng())
        return (dx, dmu, drho, bg[0] if need_b else None, bg[1] if need_b else None) + (None,) * 8


# ------------------------------------------------------------------------------------------------ transposed convolution
def conv_transpose_out(size, k, s, p, op, d):
    return (size - 1) * s - 2 * p + d * (k - 1) + op + 1


def _per_sample(x, S, shared):
    """The S-sample batch a kernel without a shared-operand mode reads: a shared [B, ...] input is repeated S times."""
    if not shared or S == 1:
        return x
    return x.unsqueeze(0).expand((S,) + tuple(x.shape)).reshape((S * x.shape[0],) + tuple(x.shape[1:]))


def _add_sampled_bias(y, mu_b, rho_b, S, spec_b):
    """y [S*B, C, H, W] += b_s (explicit lowering: the sampled bias materialised by the library, [S, C])."""
    b = _C.materialize(mu_b.contiguous(), _C.stddev(rho_b.contiguous()), S, spec_b.sample_begin, spec_b.rng(),
                       eps_in=_eps_slice(spec_b, S, mu_b.numel()))
    y.view((S, y.shape[0] // S) + tuple(y.shape[1:])).add_(b[:, None, :, None, None])


class SampledConvTranspose2dImplicit(torch.autograd.Function):
    """y[s] = conv_transpose2d(x[s], W_s, b_s) for S samples, W [Cin, Cout, KH, KW], for layers whose CONV VIEW (the
    convolution from y back to x with the same W read as OIHW) is implicit-eligible: groups == 1, Cout % 32 == 0.  The roles
    of SampledConv2dImplicit swap: the forward is the conv view's input gradient, computed in TF32 by the phase-decomposed
    gather (bnn_sampled_conv_transpose2d_fwd: one stride-1 gather per output phase over that phase's taps, the bias in its
    epilogue); the input gradient is the conv view's forward and the weight gradient its weight gradient.  fp32 (3xTF32)
    mode, or a request the kernels refuse (e.g. Cin % 32 != 0), lowers explicitly in the same (o, kh, kw, c) column order:
    bnn_sampled_gemm_dgrad + bnn_col2im_nhwc forward, bnn_im2col_nhwc + bnn_sampled_gemm_fwd / _wgrad backward.

    x: logical [S*B, Cin, H, W] (sample-major) or, when `shared`, [B, Cin, H, W].  The kernels write channels-last; the
    result is converted once to NCHW-contiguous unless set_conv_output_format('preserve') and x is channels_last."""

    @staticmethod
    def forward(ctx, x, mu_w, rho_w, mu_b, rho_b, S, shared, spec_w, spec_b, precision, stride, padding, output_padding,
                dilation):
        for n, t in (("input", x), ("weight.mean", mu_w), ("weight.scale", rho_w), ("bias.mean", mu_b),
                     ("bias.scale", rho_b)):
            _check_f32_cuda(n, t)
        Cin, Cout, KH, KW = mu_w.shape
        if x.dim() != 4 or x.shape[1] != Cin:
            raise RuntimeError(f"sampled conv_transpose2d: input {tuple(x.shape)} does not match weight {tuple(mu_w.shape)}")
        rows, _, H, W = x.shape
        B = rows if shared else rows // S
        if not shared and B * S != rows:
            raise RuntimeError(f"sampled conv_transpose2d: batch {rows} is not divisible by {S} Monte-Carlo samples")
        OH = conv_transpose_out(H, KH, stride[0], padding[0], output_padding[0], dilation[0])
        OW = conv_transpose_out(W, KW, stride[1], padding[1], output_padding[1], dilation[1])
        if OH <= 0 or OW <= 0:
            raise RuntimeError("sampled conv_transpose2d: empty output")
        nchw_out = _CONV_OUTPUT["format"] == "contiguous" or x.is_contiguous()
        x_cl = _nhwc(x)
        geom = _C.conv_geom(B, OH, OW, Cout, H, W, Cin, KH, KW, stride, padding, dilation)        # the conv view
        wl = _C.conv_weight_layout(mu_w.contiguous(), rho_w.contiguous())      # (o = Cin, kh, kw, c = Cout) order
        has_bias = mu_b is not None
        mu_b_c = mu_b.contiguous() if has_bias else None
        sigma_b = _C.stddev(rho_b.contiguous()) if has_bias else None
        eps_w = _eps_slice(spec_w, S, mu_w.numel())
        y = torch.empty((S * B, Cout, OH, OW), device=x.device, dtype=torch.float32, memory_format=torch.channels_last)
        done = precision == _C.PREC_TF32 and _C.try_sampled_conv_transpose2d_fwd(
            x_cl, 0 if shared else B * H * W * Cin, wl[0], wl[1], mu_b_c, sigma_b, eps_w,
            _eps_slice(spec_b, S, Cout) if has_bias else None, y, geom, S, spec_w.sample_begin, spec_w.rng(),
            spec_b.rng() if has_bias else None)
        if not done:
            M, K = B * H * W, KH * KW * Cout
            x_rows = _per_sample(x_cl, S, shared).permute(0, 2, 3, 1).reshape(S * M, Cin)
            dcol = torch.empty((S * M, K), device=x.device, dtype=torch.float32)
            _C.sampled_gemm_dgrad(_C.make_view(x_rows.data_ptr(), Cin, 1), M * Cin, wl[0], wl[1], eps_w, dcol, K, M * K, M,
                                  Cin, K, S, spec_w.sample_begin, spec_w.rng(), precision)
            _C.col2im_nhwc(dcol, y, geom, S * B)
            if has_bias:
                _add_sampled_bias(y, mu_b, rho_b, S, spec_b)
        ctx.save_for_backward(x_cl, wl, rho_b)
        ctx.meta = (S, shared, spec_w, spec_b, precision, geom, tuple(mu_w.shape), rows)
        return y.contiguous() if nchw_out else y

    @staticmethod
    def backward(ctx, dy):
        x_cl, wl, rho_b = ctx.saved_tensors
        S, shared, spec_w, spec_b, precision, geom, w_shape, rows = ctx.meta
        Cin, Cout, KH, KW = w_shape
        B, H, W, OH, OW = geom.B, geom.OH, geom.OW, geom.H, geom.W          # transposed input H x W, output OH x OW
        M, K = B * H * W, KH * KW * Cout
        eps_w = _eps_slice(spec_w, S, Cin * K)
        x_ss = 0 if shared else M * Cin
        tf32 = precision == _C.PREC_TF32
        need_x = ctx.needs_input_grad[0]
        need_w = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
        need_b = rho_b is not None and (ctx.needs_input_grad[3] or ctx.needs_input_grad[4])
        bias_done, bg_fused = False, None
        if dy.permute(0, 2, 3, 1).is_contiguous():
            dy_cl = dy
        else:
            dy_cl = None
            if dy.is_contiguous():
                if need_b:
                    bg_fused = torch.zeros((2, Cout), device=dy.device, dtype=torch.float32)
                dy_cl = _C.nchw_to_nhwc_bias_grad(dy, B, rho_b.contiguous() if need_b else None,
                                                  _eps_slice(spec_b, S, Cout) if need_b else None,
                                                  bg_fused[0] if need_b else None, bg_fused[1] if need_b else None,
                                                  spec_b.sample_begin if need_b else 0, spec_b.rng() if need_b else None)
                bias_done = dy_cl is not None and need_b
            if dy_cl is None:
                dy_cl = dy.contiguous(memory_format=torch.channels_last)
        col = None
        if (need_x or need_w) and not tf32:
            col = _C.im2col_nhwc(dy_cl, geom, S * B)
        dx = None
        if need_x:
            dx = torch.empty(x_cl.shape, device=dy.device, dtype=torch.float32, memory_format=torch.channels_last)
            done = tf32 and _C.try_sampled_conv_transpose2d_dgrad(dy_cl, wl[0], wl[1], eps_w, dx, x_ss, geom, S,
                                                                  spec_w.sample_begin, spec_w.rng())
            if not done:
                if col is None:
                    col = _C.im2col_nhwc(dy_cl, geom, S * B)
                out = dx if not shared or S == 1 else torch.empty((S * M, Cin), device=dy.device, dtype=torch.float32)
                _C.sampled_gemm_fwd(col, K, M * K, wl[0], wl[1], None, None, eps_w, None,
                                    _C.make_view(out.data_ptr(), Cin, 1), M * Cin, M, Cin, K, S, spec_w.sample_begin,
                                    spec_w.rng(), None, precision)
                if out is not dx:               # shared input: the per-sample contributions summed
                    dx.permute(0, 2, 3, 1).copy_(out.view(S, B, H, W, Cin).sum(0))
        grads_p, bg = _zero_grads((Cin * K,) if need_w else None, Cout if (need_b and not bias_done) else None, dy.device)
        if bias_done:
            bg = bg_fused
        dmu = drho = None
        if need_w:
            done = tf32 and _C.try_sampled_conv_transpose2d_wgrad(dy_cl, x_cl, x_ss, wl[2], eps_w, grads_p[0], grads_p[1],
                                                                  geom, S, spec_w.sample_begin, spec_w.rng())
            if not done:
                if col is None:
                    col = _C.im2col_nhwc(dy_cl, geom, S * B)
                x_rows = _per_sample(x_cl, S, shared).permute(0, 2, 3, 1).reshape(S * M, Cin)
                _C.sampled_gemm_wgrad(_C.make_view(x_rows.data_ptr(), Cin, 1), M * Cin, col, K, M * K, wl[2], eps_w,
                                      grads_p[0], grads_p[1], M, Cin, K, S, spec_w.sample_begin, spec_w.rng(), precision)
            g = _C.conv_weight_unlayout(grads_p, w_shape)
            dmu, drho = g[0], g[1]
        if need_b and not bias_done:
            _C.bias_grad(_C.make_view(dy_cl.data_ptr(), Cout, 1), B * OH * OW * Cout, rho_b.contiguous(),
                         _eps_slice(spec_b, S, Cout), bg[0], bg[1], B * OH * OW, Cout, S, spec_b.sample_begin, spec_b.rng())
        return (dx, dmu, drho, bg[0] if need_b else None, bg[1] if need_b else None) + (None,) * 9


class SampledConvTranspose2d(torch.autograd.Function):
    """y[s] = conv_transpose2d(x[s], W_s, b_s, groups=groups) for S samples, for layers whose conv view is not
    implicit-eligible (groups > 1, or Cout % 32 != 0 such as a 3-channel image): the NCHW lowering of SampledConv2d with the
    roles swapped — per group the column gradients of the conv view (bnn_sampled_gemm_dgrad, x in the role of dY) gathered
    by bnn_col2im; backward bnn_im2col of dy + bnn_sampled_gemm_fwd / _wgrad.  Weights keyed in storage (OIHW) order."""

    @staticmethod
    def forward(ctx, x, mu_w, rho_w, mu_b, rho_b, S, shared, spec_w, spec_b, precision, stride, padding, output_padding,
                dilation, groups):
        for n, t in (("input", x), ("weight.mean", mu_w), ("weight.scale", rho_w), ("bias.mean", mu_b),
                     ("bias.scale", rho_b)):
            _check_f32_cuda(n, t)
        Cin, Cout_g, KH, KW = mu_w.shape
        Cout = Cout_g * groups
        if x.dim() != 4 or x.shape[1] != Cin:
            raise RuntimeError(f"sampled conv_transpose2d: input {tuple(x.shape)} does not match weight {tuple(mu_w.shape)}")
        rows, _, H, W = x.shape
        B = rows if shared else rows // S
        if not shared and B * S != rows:
            raise RuntimeError(f"sampled conv_transpose2d: batch {rows} is not divisible by {S} Monte-Carlo samples")
        OH = conv_transpose_out(H, KH, stride[0], padding[0], output_padding[0], dilation[0])
        OW = conv_transpose_out(W, KW, stride[1], padding[1], output_padding[1], dilation[1])
        if OH <= 0 or OW <= 0:
            raise RuntimeError("sampled conv_transpose2d: empty output")
        geo = (B, Cin, H, W, Cout, KH, KW, OH, OW, tuple(stride), tuple(padding), tuple(dilation), groups)
        xs = _per_sample(x.contiguous(), S, shared)
        mu_w_c, rho_w_c = mu_w.contiguous(), rho_w.contiguous()
        sigma_w = _C.stddev(rho_w_c)
        Cin_g, Kg, P = Cin // groups, Cout_g * KH * KW, H * W
        M = B * P
        y = torch.empty((S * B, Cout, OH, OW), device=x.device, dtype=torch.float32)
        dcol = torch.empty((S * M, Kg), device=x.device, dtype=torch.float32)
        for g in range(groups):
            lo, hi = g * Cin_g * Kg, (g + 1) * Cin_g * Kg
            _C.sampled_gemm_dgrad(_C.make_view(xs.data_ptr() + 4 * g * Cin_g * P, Cin * P, P), B * Cin * P,
                                  mu_w_c.view(-1)[lo:hi], sigma_w.view(-1)[lo:hi], _eps_slice(spec_w, S, mu_w.numel(), lo, hi),
                                  dcol, Kg, M * Kg, M, Cin_g, Kg, S, spec_w.sample_begin, spec_w.rng(lo), precision)
            _C.col2im(dcol, y, SampledConvTranspose2d._geom(S * B, geo, g), False)
        if mu_b is not None:
            _add_sampled_bias(y, mu_b, rho_b, S, spec_b)
        ctx.save_for_backward(xs, mu_w_c, rho_w_c, sigma_w, rho_b)
        ctx.meta = (S, shared, spec_w, spec_b, precision, geo)
        return y

    @staticmethod
    def _geom(batch, geo, g):
        """bnn_conv2d_geom of group g of the conv view (input = the transposed output)."""
        B, Cin, H, W, Cout, KH, KW, OH, OW, stride, padding, dilation, groups = geo
        Cout_g = Cout // groups
        return _C.bnn_conv2d_geom(batch, Cout, OH, OW, g * Cout_g, Cout_g, KH, KW, H, W, stride[0], stride[1],
                                  padding[0], padding[1], dilation[0], dilation[1])

    @staticmethod
    def backward(ctx, dy):
        xs, mu_w, rho_w, sigma_w, rho_b = ctx.saved_tensors
        S, shared, spec_w, spec_b, precision, geo = ctx.meta
        B, Cin, H, W, Cout, KH, KW, OH, OW, stride, padding, dilation, groups = geo
        dy = dy.contiguous()
        Cin_g, Kg, P, Q = Cin // groups, (Cout // groups) * KH * KW, H * W, OH * OW
        M = B * P
        need_x = ctx.needs_input_grad[0]
        need_w = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
        need_b = rho_b is not None and (ctx.needs_input_grad[3] or ctx.needs_input_grad[4])
        dxs = torch.empty(xs.shape, device=dy.device, dtype=torch.float32) if need_x else None
        grads, bg = _zero_grads(tuple(mu_w.shape) if need_w else None, Cout if need_b else None, dy.device)
        col = torch.empty((S * M, Kg), device=dy.device, dtype=torch.float32) if (need_x or need_w) else None
        for g in range(groups):
            lo, hi = g * Cin_g * Kg, (g + 1) * Cin_g * Kg
            eps_w = _eps_slice(spec_w, S, mu_w.numel(), lo, hi)
            if need_x or need_w:
                _C.im2col(dy, col, SampledConvTranspose2d._geom(S * B, geo, g))
            if need_x:
                _C.sampled_gemm_fwd(col, Kg, M * Kg, mu_w.view(-1)[lo:hi], sigma_w.view(-1)[lo:hi], None, None, eps_w, None,
                                    _C.make_view(dxs.data_ptr() + 4 * g * Cin_g * P, Cin * P, P), B * Cin * P, M, Cin_g,
                                    Kg, S, spec_w.sample_begin, spec_w.rng(lo), None, precision)
            if need_w:
                _C.sampled_gemm_wgrad(_C.make_view(xs.data_ptr() + 4 * g * Cin_g * P, Cin * P, P), B * Cin * P, col, Kg,
                                      M * Kg, rho_w.view(-1)[lo:hi], eps_w, grads[0].view(-1)[lo:hi],
                                      grads[1].view(-1)[lo:hi], M, Cin_g, Kg, S, spec_w.sample_begin, spec_w.rng(lo),
                                      precision)
        if need_b:
            _C.bias_grad(_C.make_view(dy.data_ptr(), Cout * Q, Q), B * Cout * Q, rho_b.contiguous(),
                         _eps_slice(spec_b, S, Cout), bg[0], bg[1], B * Q, Cout, S, spec_b.sample_begin, spec_b.rng())
        dx = None
        if need_x:
            dx = dxs.view(S, B, Cin, H, W).sum(0) if shared and S > 1 else dxs
        return (dx, grads[0] if need_w else None, grads[1] if need_w else None,
                bg[0] if need_b else None, bg[1] if need_b else None) + (None,) * 10


class ConvTranspose3dRefused(Exception):
    """The 3-d implicit-GEMM kernels do not take this request; raised by SampledConvTranspose3dImplicit before anything
    is launched, so that the layer can contract materialised samples instead."""


def _ndhwc(t):
    """(tensor whose memory is NDHWC-contiguous, copied?) for a logical NCDHW tensor."""
    if t.permute(0, 2, 3, 4, 1).is_contiguous():
        return t
    return t.contiguous(memory_format=torch.channels_last_3d)


class SampledConvTranspose3dImplicit(torch.autograd.Function):
    """y[s] = conv_transpose3d(x[s], W_s, b_s) for S samples, W [Cin, Cout, KD, KH, KW], TF32, on the 3-d implicit-GEMM
    kernels (rank-5 im2col tensor maps): the forward is the conv view's input gradient, cut into sd x sh x sw phases (one
    stride-1 gather per phase, the bias in its epilogue); the input gradient is the conv view's forward and the weight
    gradient its weight gradient.  The C library checks one predicate for the three passes (Cin % 32 == 0,
    Cout % 32 == 0, stride <= 8, alignment, every corner within the rank-5 descriptor's limits); a request outside it
    raises ConvTranspose3dRefused from the forward, and once the forward has run, the backward cannot be refused.

    x: logical [S*B, Cin, D, H, W] (sample-major) or, when `shared`, [B, Cin, D, H, W]; any memory format.  The kernels
    write channels_last_3d; the result is converted once to NCDHW-contiguous unless set_conv_output_format('preserve') and
    x is channels_last_3d."""

    @staticmethod
    def forward(ctx, x, mu_w, rho_w, mu_b, rho_b, S, shared, spec_w, spec_b, stride, padding, output_padding, dilation):
        for n, t in (("input", x), ("weight.mean", mu_w), ("weight.scale", rho_w), ("bias.mean", mu_b),
                     ("bias.scale", rho_b)):
            _check_f32_cuda(n, t)
        Cin, Cout, KD, KH, KW = mu_w.shape
        if x.dim() != 5 or x.shape[1] != Cin:
            raise RuntimeError(f"sampled conv_transpose3d: input {tuple(x.shape)} does not match weight {tuple(mu_w.shape)}")
        rows, _, D, H, W = x.shape
        B = rows if shared else rows // S
        if not shared and B * S != rows:
            raise RuntimeError(f"sampled conv_transpose3d: batch {rows} is not divisible by {S} Monte-Carlo samples")
        OD, OH, OW = (conv_transpose_out(n, k, s, p, op, d) for n, k, s, p, op, d in
                      zip((D, H, W), (KD, KH, KW), stride, padding, output_padding, dilation))
        if OD <= 0 or OH <= 0 or OW <= 0:
            raise RuntimeError("sampled conv_transpose3d: empty output")
        nchw_out = conv_output_nchw(x)
        x_cl = _ndhwc(x)
        geom = _C.conv3d_geom(B, OD, OH, OW, Cout, D, H, W, Cin, (KD, KH, KW), stride, padding, dilation)   # the conv view
        wl = _C.conv_weight_layout(mu_w.contiguous(), rho_w.contiguous())      # (o = Cin, kd, kh, kw, c = Cout) order
        has_bias = mu_b is not None
        sigma_b = _C.stddev(rho_b.contiguous()) if has_bias else None
        y = torch.empty((S * B, Cout, OD, OH, OW), device=x.device, dtype=torch.float32,
                        memory_format=torch.channels_last_3d)
        if not _C.try_sampled_conv_transpose3d_fwd(
                x_cl, 0 if shared else B * D * H * W * Cin, wl[0], wl[1], mu_b.contiguous() if has_bias else None,
                sigma_b, _eps_slice(spec_w, S, mu_w.numel()), _eps_slice(spec_b, S, Cout) if has_bias else None, y,
                geom, S, spec_w.sample_begin, spec_w.rng(), spec_b.rng() if has_bias else None):
            raise ConvTranspose3dRefused()
        ctx.save_for_backward(x_cl, wl, rho_b)
        ctx.meta = (S, shared, spec_w, spec_b, geom, tuple(mu_w.shape))
        return y.contiguous() if nchw_out else y

    @staticmethod
    def backward(ctx, dy):
        x_cl, wl, rho_b = ctx.saved_tensors
        S, shared, spec_w, spec_b, geom, w_shape = ctx.meta
        Cin, Cout = w_shape[0], w_shape[1]
        B, OD, OH, OW = geom.B, geom.D, geom.H, geom.W                        # transposed output OD x OH x OW
        M = B * geom.OD * geom.OH * geom.OW
        eps_w = _eps_slice(spec_w, S, math.prod(w_shape))
        x_ss = 0 if shared else M * Cin
        need_x = ctx.needs_input_grad[0]
        need_w = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
        need_b = rho_b is not None and (ctx.needs_input_grad[3] or ctx.needs_input_grad[4])
        # the kernels read dY as NDHWC rows; an NCDHW-contiguous gradient goes through ONE transposing pass (P = D*H*W)
        # that forms the bias gradient on the way
        bias_done, bg_fused = False, None
        if dy.permute(0, 2, 3, 4, 1).is_contiguous():
            dy_cl = dy
        else:
            dy_cl = None
            if dy.is_contiguous():
                if need_b:
                    bg_fused = torch.zeros((2, Cout), device=dy.device, dtype=torch.float32)
                t = _C.nchw_to_nhwc_bias_grad(dy.view(dy.shape[0], Cout, OD, OH * OW), B,
                                              rho_b.contiguous() if need_b else None,
                                              _eps_slice(spec_b, S, Cout) if need_b else None,
                                              bg_fused[0] if need_b else None, bg_fused[1] if need_b else None,
                                              spec_b.sample_begin if need_b else 0, spec_b.rng() if need_b else None)
                if t is not None:
                    dy_cl = t.permute(0, 2, 3, 1).view(dy.shape[0], OD, OH, OW, Cout).permute(0, 4, 1, 2, 3)
                    bias_done = need_b
            if dy_cl is None:
                dy_cl = dy.contiguous(memory_format=torch.channels_last_3d)
        dx = None
        if need_x:
            dx = torch.empty(x_cl.shape, device=dy.device, dtype=torch.float32, memory_format=torch.channels_last_3d)
            _C.sampled_conv_transpose3d_dgrad(dy_cl, wl[0], wl[1], eps_w, dx, x_ss, geom, S, spec_w.sample_begin,
                                              spec_w.rng())
        grads_p, bg = _zero_grads((math.prod(w_shape),) if need_w else None, Cout if (need_b and not bias_done) else None,
                                  dy.device)
        if bias_done:
            bg = bg_fused
        dmu = drho = None
        if need_w:
            _C.sampled_conv_transpose3d_wgrad(dy_cl, x_cl, x_ss, wl[2], eps_w, grads_p[0], grads_p[1], geom, S,
                                              spec_w.sample_begin, spec_w.rng())
            g = _C.conv_weight_unlayout(grads_p, w_shape)
            dmu, drho = g[0], g[1]
        if need_b and not bias_done:
            rows_y = B * OD * OH * OW
            _C.bias_grad(_C.make_view(dy_cl.data_ptr(), Cout, 1), rows_y * Cout, rho_b.contiguous(),
                         _eps_slice(spec_b, S, Cout), bg[0], bg[1], rows_y, Cout, S, spec_b.sample_begin, spec_b.rng())
        return (dx, dmu, drho, bg[0] if need_b else None, bg[1] if need_b else None) + (None,) * 8


class FlipoutContractionRefused(Exception):
    """The transposed-convolution kernels do not take every pass of a Flipout call's geometry; raised by
    FlipoutConvTransposeImplicit before anything has launched, so that the layer evaluates its composite instead."""


class FlipoutConvTransposeImplicit(torch.autograd.Function):
    """The Flipout transposed convolution with per-example signs R [n, Cout] and S [n, Cin] (nn.flipout):

        y  = convT(x, mu) + R o convT(x o S, sigma),             sigma = 1e-10 + softplus(rho)
        dx = convT^T(g, mu) + S o convT^T(R o g, sigma),  d mu = wgrad(g, x),  d sigma = wgrad(R o g, x o S),
        d rho = d sigma * sigmoid(rho).

    x: logical [n, Cin, H, W] (the 1-d layers: H = 1) or [n, Cin, D, H, W], NC(D)HW-contiguous or channels-last; weights
    [Cin, Cout, *k].  Every contraction is one call of the transposed-convolution kernels with one sample and injected
    eps = 0 (`zero`, [1, numel]), so the kernels' weight mu + sigma * eps is the given operand exactly: mu, or sigma
    (computed once by the layout kernel) in the mean slot; the d mean slot of the sigma contraction's weight gradient is
    d sigma.  The sign products and the layout changes around the contractions are two bandwidth passes,
    bnn_flipout_split ((x, S) forward, (g, R) backward) and bnn_flipout_combine ((y_mu, y_sigma, R) forward,
    (dx_mu, dx_sigma, S) backward), which also writes the NC(D)HW output.  TF32 only.  Whether the kernels take all
    three passes of the geometry is asked once (bnn_conv_transpose{2,3}d_supported) before anything launches:
    FlipoutContractionRefused when they do not, so that the layer evaluates its composite; a refusal after that is an
    error."""

    @staticmethod
    def _passes(x, w_shape, stride, padding, output_padding, dilation):
        """(geometry of the conv view, fwd, dgrad, wgrad, memory format) of this call's rank; fwd / dgrad / wgrad return
        False when refused."""
        rows, Cin, Cout, k = x.shape[0], w_shape[0], w_shape[1], tuple(w_shape[2:])
        out = tuple(conv_transpose_out(n, kk, s, p, op, d) for n, kk, s, p, op, d in
                    zip(x.shape[2:], k, stride, padding, output_padding, dilation))
        if min(out) <= 0:
            raise RuntimeError("flipout conv_transpose: empty output")
        if x.dim() == 4:
            geom = _C.conv_geom(rows, *out, Cout, *x.shape[2:], Cin, *k, stride, padding, dilation)
            return (geom, _C.try_sampled_conv_transpose2d_fwd, _C.try_sampled_conv_transpose2d_dgrad,
                    _C.try_sampled_conv_transpose2d_wgrad, torch.channels_last, out)
        geom = _C.conv3d_geom(rows, *out, Cout, *x.shape[2:], Cin, k, stride, padding, dilation)

        def dgrad(*args):                  # the 3-d predicate is one for the three passes: the forward has checked it
            _C.sampled_conv_transpose3d_dgrad(*args)
            return True

        def wgrad(*args):
            _C.sampled_conv_transpose3d_wgrad(*args)
            return True
        return geom, _C.try_sampled_conv_transpose3d_fwd, dgrad, wgrad, torch.channels_last_3d, out

    @staticmethod
    def forward(ctx, x, mu, rho, R, S, zero, stride, padding, output_padding, dilation, nchw_out):
        for n, t in (("input", x), ("weight.mean", mu), ("weight.scale", rho), ("R", R), ("S", S)):
            _check_f32_cuda(n, t)
        if x.dim() not in (4, 5) or x.shape[1] != mu.shape[0] or mu.dim() != x.dim():
            raise RuntimeError(f"flipout conv_transpose: input {tuple(x.shape)} does not match weight {tuple(mu.shape)}")
        geom, fwd, _, _, fmt, out = FlipoutConvTransposeImplicit._passes(x, tuple(mu.shape), stride, padding,
                                                                         output_padding, dilation)
        # one predicate for the forward, input-gradient and weight-gradient kernels, asked before anything launches: in
        # 2-d the forward's phase corners (divided by the stride) admit geometries whose conv view the gradients refuse
        if not _C.conv_transpose_supported(geom):
            raise FlipoutContractionRefused()
        if x.data_ptr() % 16:                      # the kernels read 16-byte aligned tensors: a fresh copy is
            x = x.clone()
        spec = DrawSpec(0, 0, 0, eps=zero)
        rng = spec.rng()
        wl = _C.conv_weight_layout(mu.contiguous(), rho.contiguous())          # mean, sigma, scale in (o, taps, c) order
        x_cl, xs_cl = _C.flipout_split(x, S)
        shape = (x.shape[0], mu.shape[1]) + out
        y_mu = torch.empty(shape, device=x.device, dtype=torch.float32, memory_format=fmt)
        y_sigma = torch.empty(shape, device=x.device, dtype=torch.float32, memory_format=fmt)
        if not (fwd(x_cl, 0, wl[0], wl[1], None, None, zero, None, y_mu, geom, 1, 0, rng, None) and
                fwd(xs_cl, 0, wl[1], wl[1], None, None, zero, None, y_sigma, geom, 1, 0, rng, None)):
            raise RuntimeError("flipout conv_transpose: the kernels refused a forward contraction of a geometry they accept")
        ctx.save_for_backward(x_cl, xs_cl, wl, rho, R, S, zero)
        ctx.meta = (geom, tuple(mu.shape), stride, padding, output_padding, dilation, not x.is_contiguous())
        return _C.flipout_combine(y_mu, y_sigma, R, channels_last=not nchw_out)

    @staticmethod
    def backward(ctx, g):
        x_cl, xs_cl, wl, rho, R, S, zero = ctx.saved_tensors
        geom, w_shape, stride, padding, output_padding, dilation, x_channels_last = ctx.meta
        _, _, dgrad, wgrad, fmt, _ = FlipoutConvTransposeImplicit._passes(x_cl, w_shape, stride, padding, output_padding,
                                                                          dilation)
        rng = DrawSpec(0, 0, 0, eps=zero).rng()
        if g.data_ptr() % 16 or not (g.is_contiguous() or g.permute(0, *range(2, g.dim()), 1).is_contiguous()):
            g = g.clone(memory_format=torch.contiguous_format)
        g_cl, gr_cl = _C.flipout_split(g, R)
        dx = dmu = drho = None
        if ctx.needs_input_grad[0]:
            dx_mu = torch.empty(x_cl.shape, device=g.device, dtype=torch.float32, memory_format=fmt)
            dx_sigma = torch.empty(x_cl.shape, device=g.device, dtype=torch.float32, memory_format=fmt)
            if not (dgrad(g_cl, wl[0], wl[1], zero, dx_mu, 0, geom, 1, 0, rng) and
                    dgrad(gr_cl, wl[1], wl[1], zero, dx_sigma, 0, geom, 1, 0, rng)):
                raise RuntimeError("flipout conv_transpose: the kernels refused the input gradient of a call whose forward "
                                   "they ran")
            dx = _C.flipout_combine(dx_mu, dx_sigma, S, channels_last=x_channels_last)
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            # d mean, d sigma and the (zero) d scale slot both calls accumulate into
            acc = torch.zeros((3, wl.shape[1]), device=g.device, dtype=torch.float32)
            if not (wgrad(g_cl, x_cl, 0, wl[2], zero, acc[0], acc[2], geom, 1, 0, rng) and
                    wgrad(gr_cl, xs_cl, 0, wl[2], zero, acc[1], acc[2], geom, 1, 0, rng)):
                raise RuntimeError("flipout conv_transpose: the kernels refused the weight gradient of a call whose "
                                   "forward they ran")
            grads = _C.conv_weight_unlayout(acc[:2], w_shape)
            dmu, drho = grads[0], grads[1] * torch.sigmoid(rho)
        return (dx, dmu, drho) + (None,) * 8


class CudnnConvTranspose(torch.autograd.Function):
    """F.conv_transposeNd(x, w, b, ...) (N from the rank of x) with cuDNN's TF32 switched to `tf32` in the forward AND the
    backward pass (autograd runs the backward outside any context the forward was called in): the materialised-sample
    form of NormalConvTranspose3d and the composite of the Flipout transposed layers, which in fp32 mode must not round
    their operands to TF32."""

    @staticmethod
    def _tf32(flag, fn):
        prev = torch.backends.cudnn.allow_tf32
        torch.backends.cudnn.allow_tf32 = flag
        try:
            return fn()
        finally:
            torch.backends.cudnn.allow_tf32 = prev

    @staticmethod
    def forward(ctx, x, w, b, stride, padding, output_padding, groups, dilation, tf32):
        ctx.save_for_backward(x, w)
        ctx.meta = (b is not None, stride, padding, output_padding, groups, dilation, tf32)
        op = getattr(torch.nn.functional, f"conv_transpose{x.dim() - 2}d")
        return CudnnConvTranspose._tf32(tf32, lambda: op(x, w, b, stride, padding, output_padding, groups, dilation))

    @staticmethod
    def backward(ctx, gy):
        x, w = ctx.saved_tensors
        has_b, stride, padding, output_padding, groups, dilation, tf32 = ctx.meta
        mask = [ctx.needs_input_grad[0], ctx.needs_input_grad[1], has_b and ctx.needs_input_grad[2]]
        gx, gw, gb = CudnnConvTranspose._tf32(tf32, lambda: torch.ops.aten.convolution_backward(
            gy, x, w, [w.shape[1] * groups] if has_b else None, list(stride), list(padding), list(dilation), True,
            list(output_padding), groups, mask))
        return (gx, gw, gb if has_b else None) + (None,) * 6


CudnnConvTranspose3d = CudnnConvTranspose      # the name NormalConvTranspose3d's materialised-sample path was written with


# ------------------------------------------------------------------------------------------------
class Materialize(torch.autograd.Function):
    """W_s = mean + stddev * eps_s for s in [0, S) as a tensor [S, *shape] (core.py:44-45); used by
    `.sampled` and by layers without a fused contraction (NormalConv3d)."""

    @staticmethod
    def forward(ctx, mu, rho, S, spec):
        _check_f32_cuda("mean", mu)
        _check_f32_cuda("scale", rho)
        mu_c, rho_c = mu.contiguous(), rho.contiguous()
        sigma = _C.stddev(rho_c)
        out = _C.materialize(mu_c, sigma, S, spec.sample_begin, spec.rng(), eps_in=_eps_slice(spec, S, mu.numel()))
        ctx.save_for_backward(rho_c)
        ctx.meta = (S, spec)
        return out

    @staticmethod
    def backward(ctx, g):
        (rho,) = ctx.saved_tensors
        S, spec = ctx.meta
        if spec.eps is not None:
            eps = spec.eps.reshape((S,) + tuple(rho.shape))
        else:
            zero, one = torch.zeros_like(rho), torch.ones_like(rho)
            eps = _C.materialize(zero, one, S, spec.sample_begin, spec.rng())
        dmu = g.sum(0)
        drho = (g * eps).sum(0) * torch.sigmoid(rho)
        return dmu, drho, None, None


# ------------------------------------------------------------------------------------------------
class KLSum(torch.autograd.Function):
    """sum_t coeff_t * sum_i KL(N(mu_ti, sigma_ti) || N(loc_t, scale_t)) over many tensors in one
    bandwidth-bound launch (loss.py:16-38 with coeff_t = 1 / (numel_t * n_tensors * n_batches)).
    Backward is one more pass that writes coeff_t * dKL/d(mu, rho) scaled by the upstream gradient
    (read on the device, no host sync)."""

    @staticmethod
    def forward(ctx, priors, coeffs, *params):
        n = len(params) // 2
        entries = []
        for t in range(n):
            mu, rho = params[2 * t], params[2 * t + 1]
            _check_f32_cuda("mean", mu)
            _check_f32_cuda("scale", rho)
            entries.append((mu.contiguous(), rho.contiguous(), None, None, priors[t][0], priors[t][1], coeffs[t]))
        total = _C.kl(entries, want_sums=False, want_total=True)
        ctx.save_for_backward(*[e[i] for e in entries for i in (0, 1)])
        ctx.meta = (priors, coeffs)
        return total

    @staticmethod
    def backward(ctx, g):
        priors, coeffs = ctx.meta
        saved = ctx.saved_tensors
        n = len(saved) // 2
        scale = g.detach().to(torch.float32).reshape(1).contiguous()
        entries, grads = [], []
        for t in range(n):
            mu, rho = saved[2 * t], saved[2 * t + 1]
            gm, gr = torch.empty_like(mu), torch.empty_like(rho)
            grads += [gm, gr]
            entries.append((mu, rho, gm, gr, priors[t][0], priors[t][1], coeffs[t]))
        _C.kl(entries, want_sums=False, want_total=False, grad_scale=scale)
        return (None, None) + tuple(grads)


# ------------------------------------------------------------------------------------------------
class MCCrossEntropy(torch.autograd.Function):
    """Mean cross-entropy of the [S*B, C] score matrix `x` against the B labels shared by the S Monte-Carlo samples
    (examples/MNIST/train.py:59-61 with CrossEntropyLoss): one forward and one backward kernel
    (bnn_mc_cross_entropy_fwd / _bwd) instead of torch's log_softmax + nll_loss chains over a replicated target."""

    @staticmethod
    def forward(ctx, x, target, ignore_index):
        if x.stride(1) != 1 or x.stride(0) < x.shape[1]:
            x = x.contiguous()
        target = target.contiguous()
        loss, lse, count = _C.mc_cross_entropy_fwd(x, target, ignore_index)
        ctx.save_for_backward(x, target, lse, count)
        ctx.ignore_index = ignore_index
        return loss

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        x, target, lse, count = ctx.saved_tensors
        if not ctx.needs_input_grad[0]:
            return None, None, None
        g = g.detach().to(torch.float32).reshape(()).contiguous()
        return _C.mc_cross_entropy_bwd(x, target, lse, count, g, ctx.ignore_index), None, None
