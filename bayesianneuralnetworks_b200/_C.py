"""ctypes binding of libbnn_b200.so (the C ABI in include/bnn_b200.h).

Everything here takes CUDA torch tensors, checks them, and passes raw device pointers plus the
current CUDA stream across the C boundary.  There is no CPU path: a tensor that is not on a CUDA
device, or a missing/unsupported library, raises.  Status codes become `BnnError`.
"""
import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# BNN_B200_LIB: another build of the same library (profiling builds with -DBNN_PROFILE_WAITS); never a fallback
LIB_PATH = os.environ.get("BNN_B200_LIB") or os.path.join(_HERE, "libbnn_b200.so")

PREC_TF32 = 0
PREC_FP32X3 = 1

_c_f32p = ctypes.c_void_p  # raw device pointers travel as integers


class BnnError(RuntimeError):
    def __init__(self, code, where, text):
        super().__init__(f"{where}: bnn_status {code}: {text}")
        self.code = code


class bnn_rng(ctypes.Structure):
    _fields_ = [("seed", ctypes.c_uint64), ("step", ctypes.c_uint64),
                ("step_dev", ctypes.c_void_p), ("elem_offset", ctypes.c_uint64),
                ("tensor_id", ctypes.c_uint32), ("reserved", ctypes.c_uint32),
                ("row_sign", ctypes.c_void_p), ("col_sign", ctypes.c_void_p), ("rows", ctypes.c_int32),
                ("cols", ctypes.c_int32)]


class bnn_view(ctypes.Structure):
    _fields_ = [("base", ctypes.c_void_p), ("batch_stride", ctypes.c_int64),
                ("P", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class bnn_conv2d_geom(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in
                ("B", "C", "H", "W", "c0", "Cg", "KH", "KW", "OH", "OW", "sh", "sw", "ph", "pw", "dh", "dw")]


class bnn_conv2d_nhwc(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in
                ("B", "H", "W", "C", "OH", "OW", "Cout", "KH", "KW", "sh", "sw", "ph", "pw", "dh", "dw", "reserved")]


class bnn_conv3d_nhwc(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in
                ("B", "D", "H", "W", "C", "OD", "OH", "OW", "Cout", "KD", "KH", "KW", "sd", "sh", "sw", "pd", "ph", "pw",
                 "dd", "dh", "dw", "reserved")]


class bnn_kl_tensor(ctypes.Structure):
    _fields_ = [("mu", ctypes.c_void_p), ("rho", ctypes.c_void_p), ("grad_mu", ctypes.c_void_p),
                ("grad_rho", ctypes.c_void_p), ("numel", ctypes.c_int64),
                ("prior_loc", ctypes.c_float), ("prior_scale", ctypes.c_float),
                ("grad_coeff", ctypes.c_float), ("reserved", ctypes.c_float)]


class bnn_prune_tensor(ctypes.Structure):
    _fields_ = [("mu", ctypes.c_void_p), ("rho", ctypes.c_void_p), ("mask_out", ctypes.c_void_p),
                ("keys_out", ctypes.c_void_p), ("numel", ctypes.c_int64), ("k", ctypes.c_int64),
                ("flags", ctypes.c_uint32), ("reserved", ctypes.c_uint32)]


class bnn_prune_into_tensor(ctypes.Structure):
    _fields_ = [("mu", ctypes.c_void_p), ("rho", ctypes.c_void_p), ("mu_out", ctypes.c_void_p), ("rho_out", ctypes.c_void_p),
                ("mask_out", ctypes.c_void_p), ("numel", ctypes.c_int64), ("k", ctypes.c_int64),
                ("flags", ctypes.c_uint32), ("reserved", ctypes.c_uint32), ("kl_sum_out", ctypes.c_void_p),
                ("prior_loc", ctypes.c_float), ("prior_scale", ctypes.c_float)]


class bnn_adam_tensor(ctypes.Structure):
    _fields_ = [("mu", ctypes.c_void_p), ("rho", ctypes.c_void_p), ("g_mu", ctypes.c_void_p), ("g_rho", ctypes.c_void_p),
                ("m_mu", ctypes.c_void_p), ("v_mu", ctypes.c_void_p), ("m_rho", ctypes.c_void_p), ("v_rho", ctypes.c_void_p),
                ("numel", ctypes.c_int64), ("prior_loc", ctypes.c_float), ("prior_scale", ctypes.c_float),
                ("kl_coeff", ctypes.c_float), ("reserved", ctypes.c_float)]


MAX_PEERS = 8


class bnn_peer_grads(ctypes.Structure):
    _fields_ = [("world", ctypes.c_int32), ("rank", ctypes.c_int32), ("base", ctypes.c_void_p * MAX_PEERS)]


class bnn_pack_item(ctypes.Structure):
    _fields_ = [("src", ctypes.c_void_p), ("dst_offset", ctypes.c_int64), ("numel", ctypes.c_int64)]


_SIGNATURES = {
    "bnn_abi_version": (ctypes.c_int, []),
    "bnn_last_error_string": (ctypes.c_char_p, []),
    "bnn_device_supported": (ctypes.c_int, [ctypes.c_int]),
    "bnn_stddev": (ctypes.c_int, [_c_f32p, _c_f32p, ctypes.c_int64, ctypes.c_void_p]),
    "bnn_materialize": (ctypes.c_int, [_c_f32p, _c_f32p, _c_f32p, _c_f32p, _c_f32p, ctypes.c_int64,
                                       ctypes.c_int32, ctypes.c_uint32, ctypes.POINTER(bnn_rng),
                                       ctypes.c_void_p]),
    "bnn_sampled_gemm_fwd": (ctypes.c_int, [_c_f32p, ctypes.c_int64, ctypes.c_int64, _c_f32p, _c_f32p,
                                            _c_f32p, _c_f32p, _c_f32p, _c_f32p, bnn_view, ctypes.c_int64,
                                            ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                            ctypes.c_uint32, ctypes.POINTER(bnn_rng), ctypes.POINTER(bnn_rng),
                                            ctypes.c_int32, ctypes.c_void_p]),
    "bnn_sampled_gemm_dgrad": (ctypes.c_int, [bnn_view, ctypes.c_int64, _c_f32p, _c_f32p, _c_f32p, _c_f32p,
                                              ctypes.c_int64, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32,
                                              ctypes.c_int32, ctypes.c_int32, ctypes.c_uint32,
                                              ctypes.POINTER(bnn_rng), ctypes.c_int32, ctypes.c_void_p]),
    "bnn_sampled_gemm_wgrad": (ctypes.c_int, [bnn_view, ctypes.c_int64, _c_f32p, ctypes.c_int64, ctypes.c_int64,
                                              _c_f32p, _c_f32p, _c_f32p, _c_f32p, ctypes.c_int32,
                                              ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_uint32,
                                              ctypes.POINTER(bnn_rng), ctypes.c_int32, ctypes.c_void_p]),
    "bnn_bias_grad": (ctypes.c_int, [bnn_view, ctypes.c_int64, _c_f32p, _c_f32p, _c_f32p, _c_f32p,
                                     ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_uint32,
                                     ctypes.POINTER(bnn_rng), ctypes.c_void_p]),
    "bnn_im2col": (ctypes.c_int, [_c_f32p, _c_f32p, ctypes.POINTER(bnn_conv2d_geom), ctypes.c_void_p]),
    "bnn_col2im": (ctypes.c_int, [_c_f32p, _c_f32p, ctypes.POINTER(bnn_conv2d_geom), ctypes.c_int32,
                                  ctypes.c_void_p]),
    "bnn_sampled_conv2d_fwd": (ctypes.c_int, [_c_f32p, ctypes.c_int64, _c_f32p, _c_f32p, _c_f32p, _c_f32p, _c_f32p, _c_f32p,
                                              bnn_view, ctypes.c_int64, ctypes.POINTER(bnn_conv2d_nhwc), ctypes.c_int32,
                                              ctypes.c_uint32, ctypes.POINTER(bnn_rng), ctypes.POINTER(bnn_rng),
                                              ctypes.c_void_p]),
    "bnn_sampled_conv2d_dgrad": (ctypes.c_int, [_c_f32p, _c_f32p, _c_f32p, _c_f32p, _c_f32p, ctypes.c_int64,
                                                ctypes.POINTER(bnn_conv2d_nhwc), ctypes.c_int32, ctypes.c_uint32,
                                                ctypes.POINTER(bnn_rng), ctypes.c_void_p]),
    "bnn_sampled_conv2d_wgrad": (ctypes.c_int, [_c_f32p, _c_f32p, ctypes.c_int64, _c_f32p, _c_f32p, _c_f32p, _c_f32p,
                                                ctypes.POINTER(bnn_conv2d_nhwc), ctypes.c_int32, ctypes.c_uint32,
                                                ctypes.POINTER(bnn_rng), ctypes.c_void_p]),
    "bnn_sampled_conv_transpose2d_fwd": (ctypes.c_int, [_c_f32p, ctypes.c_int64, _c_f32p, _c_f32p, _c_f32p, _c_f32p, _c_f32p,
                                                        _c_f32p, _c_f32p, ctypes.POINTER(bnn_conv2d_nhwc), ctypes.c_int32,
                                                        ctypes.c_uint32, ctypes.POINTER(bnn_rng), ctypes.POINTER(bnn_rng),
                                                        ctypes.c_void_p]),
    "bnn_sampled_conv_transpose2d_dgrad": (ctypes.c_int, [_c_f32p, _c_f32p, _c_f32p, _c_f32p, _c_f32p, ctypes.c_int64,
                                                          ctypes.POINTER(bnn_conv2d_nhwc), ctypes.c_int32, ctypes.c_uint32,
                                                          ctypes.POINTER(bnn_rng), ctypes.c_void_p]),
    "bnn_sampled_conv_transpose2d_wgrad": (ctypes.c_int, [_c_f32p, _c_f32p, ctypes.c_int64, _c_f32p, _c_f32p, _c_f32p,
                                                          _c_f32p, ctypes.POINTER(bnn_conv2d_nhwc), ctypes.c_int32,
                                                          ctypes.c_uint32, ctypes.POINTER(bnn_rng), ctypes.c_void_p]),
    "bnn_debug_conv_transpose_phases": (ctypes.c_int, [ctypes.POINTER(bnn_conv2d_nhwc), ctypes.POINTER(ctypes.c_int32),
                                                       ctypes.c_int32]),
    "bnn_sampled_conv_transpose3d_fwd": (ctypes.c_int, [_c_f32p, ctypes.c_int64, _c_f32p, _c_f32p, _c_f32p, _c_f32p, _c_f32p,
                                                        _c_f32p, _c_f32p, ctypes.POINTER(bnn_conv3d_nhwc), ctypes.c_int32,
                                                        ctypes.c_uint32, ctypes.POINTER(bnn_rng), ctypes.POINTER(bnn_rng),
                                                        ctypes.c_void_p]),
    "bnn_sampled_conv_transpose3d_dgrad": (ctypes.c_int, [_c_f32p, _c_f32p, _c_f32p, _c_f32p, _c_f32p, ctypes.c_int64,
                                                          ctypes.POINTER(bnn_conv3d_nhwc), ctypes.c_int32, ctypes.c_uint32,
                                                          ctypes.POINTER(bnn_rng), ctypes.c_void_p]),
    "bnn_sampled_conv_transpose3d_wgrad": (ctypes.c_int, [_c_f32p, _c_f32p, ctypes.c_int64, _c_f32p, _c_f32p, _c_f32p,
                                                          _c_f32p, ctypes.POINTER(bnn_conv3d_nhwc), ctypes.c_int32,
                                                          ctypes.c_uint32, ctypes.POINTER(bnn_rng), ctypes.c_void_p]),
    "bnn_debug_conv_transpose3d_phases": (ctypes.c_int, [ctypes.POINTER(bnn_conv3d_nhwc), ctypes.POINTER(ctypes.c_int32),
                                                         ctypes.c_int32]),
    "bnn_conv_transpose2d_supported": (ctypes.c_int, [ctypes.POINTER(bnn_conv2d_nhwc)]),
    "bnn_conv_transpose3d_supported": (ctypes.c_int, [ctypes.POINTER(bnn_conv3d_nhwc)]),
    "bnn_conv2d_weight_layout": (ctypes.c_int, [_c_f32p, _c_f32p, _c_f32p, _c_f32p, _c_f32p, ctypes.c_int32, ctypes.c_int32,
                                                ctypes.c_int32, ctypes.c_void_p]),
    "bnn_conv2d_weight_unlayout": (ctypes.c_int, [_c_f32p, _c_f32p, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                                  ctypes.c_int32, ctypes.c_void_p]),
    "bnn_nchw_to_nhwc_bias_grad": (ctypes.c_int, [_c_f32p, _c_f32p, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32,
                                                  ctypes.c_int32, _c_f32p, _c_f32p, _c_f32p, _c_f32p, ctypes.c_uint32,
                                                  ctypes.POINTER(bnn_rng), ctypes.c_void_p]),
    "bnn_im2col_nhwc": (ctypes.c_int, [_c_f32p, _c_f32p, ctypes.POINTER(bnn_conv2d_nhwc), ctypes.c_int64, ctypes.c_void_p]),
    "bnn_col2im_nhwc": (ctypes.c_int, [_c_f32p, _c_f32p, ctypes.POINTER(bnn_conv2d_nhwc), ctypes.c_int64, ctypes.c_void_p]),
    "bnn_flipout_split": (ctypes.c_int, [_c_f32p, ctypes.c_int32, _c_f32p, _c_f32p, _c_f32p, ctypes.c_int64, ctypes.c_int32,
                                         ctypes.c_int64, ctypes.c_void_p]),
    "bnn_flipout_combine": (ctypes.c_int, [_c_f32p, _c_f32p, _c_f32p, _c_f32p, ctypes.c_int32, ctypes.c_int64, ctypes.c_int32,
                                           ctypes.c_int64, ctypes.c_void_p]),
    "bnn_kl_workspace_size": (ctypes.c_size_t, [ctypes.c_int32]),
    "bnn_kl": (ctypes.c_int, [ctypes.POINTER(bnn_kl_tensor), ctypes.c_int32, ctypes.c_void_p, _c_f32p, _c_f32p,
                              ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "bnn_prune_workspace_size": (ctypes.c_size_t, [ctypes.POINTER(bnn_prune_tensor), ctypes.c_int32]),
    "bnn_prune": (ctypes.c_int, [ctypes.POINTER(bnn_prune_tensor), ctypes.c_int32, ctypes.c_void_p,
                                 ctypes.c_size_t, ctypes.c_void_p]),
    "bnn_prune_into_workspace_size": (ctypes.c_size_t, [ctypes.POINTER(bnn_prune_into_tensor), ctypes.c_int32]),
    "bnn_prune_into": (ctypes.c_int, [ctypes.POINTER(bnn_prune_into_tensor), ctypes.c_int32, ctypes.c_void_p,
                                      ctypes.c_size_t, ctypes.c_void_p]),
    "bnn_adam_kl_step": (ctypes.c_int, [ctypes.POINTER(bnn_adam_tensor), ctypes.c_int32, ctypes.c_float, ctypes.c_float,
                                        ctypes.c_float, ctypes.c_float, _c_f32p, ctypes.c_int64, ctypes.c_void_p]),
    "bnn_adam_kl_step_peers": (ctypes.c_int, [ctypes.POINTER(bnn_adam_tensor), ctypes.c_int32, ctypes.c_float, ctypes.c_float,
                                              ctypes.c_float, ctypes.c_float, _c_f32p, ctypes.c_int64,
                                              ctypes.POINTER(bnn_peer_grads), ctypes.c_void_p]),
    "bnn_peer_average": (ctypes.c_int, [ctypes.POINTER(bnn_peer_grads), ctypes.c_int64, ctypes.c_void_p]),
    "bnn_pack_gradients": (ctypes.c_int, [ctypes.POINTER(bnn_pack_item), ctypes.c_int32, _c_f32p, ctypes.c_void_p]),
    "bnn_peer_barrier": (ctypes.c_int, [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p,
                                        ctypes.c_void_p]),
    "bnn_mc_cross_entropy_workspace_size": (ctypes.c_size_t, []),
    "bnn_mc_cross_entropy_fwd": (ctypes.c_int, [_c_f32p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64,
                                                ctypes.c_int32, ctypes.c_int64, _c_f32p, _c_f32p, _c_f32p, ctypes.c_void_p,
                                                ctypes.c_size_t, ctypes.c_void_p]),
    "bnn_mc_cross_entropy_bwd": (ctypes.c_int, [_c_f32p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64,
                                                ctypes.c_int32, ctypes.c_int64, _c_f32p, _c_f32p, _c_f32p, _c_f32p,
                                                ctypes.c_int64, ctypes.c_void_p]),
    "bnn_selftest_prune_interval": (ctypes.c_int, [_c_f32p, _c_f32p, ctypes.c_int64, _c_f32p, _c_f32p, ctypes.c_int32,
                                                   ctypes.c_void_p]),
    "bnn_debug_force_contract_variant": (ctypes.c_int, [ctypes.c_int32]),
    "bnn_debug_pair_tile_plan": (ctypes.c_int, [ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                                ctypes.POINTER(ctypes.c_int32)]),
    "bnn_debug_wgrad_plan": (ctypes.c_int, [ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                            ctypes.POINTER(ctypes.c_int32)]),
    "bnn_debug_force_wgrad_plan": (ctypes.c_int, [ctypes.c_int32, ctypes.c_int32, ctypes.c_int32]),
    "bnn_selftest_umma":(ctypes.c_int, [_c_f32p, ctypes.c_void_p]),
    "bnn_selftest_umma_mn": (ctypes.c_int, [_c_f32p, ctypes.c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None
_lib_lock = threading.Lock()
launch_count = 0          # kernels launched through this binding (bench.py reports it)


def lib():
    """The loaded library; raises (never falls back) when it is missing."""
    global _lib
    if _lib is None:
        with _lib_lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        f"{LIB_PATH} is missing: build it with `python -m bayesianneuralnetworks_b200._build` "
                        "(there is no CPU or PyTorch fallback for the variational hot path)")
                handle = ctypes.CDLL(LIB_PATH)
                for name, (res, args) in _SIGNATURES.items():
                    fn = getattr(handle, name)
                    fn.restype = res
                    fn.argtypes = args
                _lib = handle
    return _lib


def _check(code, where):
    if code != 0:
        raise BnnError(code, where, lib().bnn_last_error_string().decode("utf-8", "replace"))


_timing = None            # list of (name, start event, stop event) while kernel timing is on


def set_kernel_timing(on):
    """Bracket every library call with CUDA events on the launching stream (bench.py's live per-kernel times)."""
    global _timing
    _timing = [] if on else None


def kernel_timing_summary(steps=1):
    """{entry point: {ms_per_step, launches_per_step}} of the calls recorded since set_kernel_timing(True)."""
    torch.cuda.synchronize()
    out = {}
    for name, e0, e1 in _timing or []:
        d = out.setdefault(name, {"ms_per_step": 0.0, "launches_per_step": 0})
        d["ms_per_step"] += e0.elapsed_time(e1)
        d["launches_per_step"] += 1
    for d in out.values():
        d["ms_per_step"] /= steps
        d["launches_per_step"] /= steps
    return out


_ERR_UNSUPPORTED = 6      # BNN_ERR_UNSUPPORTED: a request outside the kernels' stated limits, refused before any launch


def _invoke(name, *args):
    """Status of one library call, bracketed with CUDA events while kernel timing is on (a refused request is not
    recorded: it launched nothing)."""
    fn = getattr(lib(), name)
    if _timing is None:
        return fn(*args)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    rc = fn(*args)
    e1.record()
    if rc != _ERR_UNSUPPORTED:
        _timing.append((name, e0, e1))
    return rc


def _call(name, *args):
    _check(_invoke(name, *args), name)


def _count(n=1):
    global launch_count
    launch_count += n


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError(
                "bayesianneuralnetworks_b200: the variational hot path runs on CUDA (sm_100a) only; got a "
                f"{t.device} tensor. Move the module and its inputs to a B200 device (no CPU fallback).")


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f32c(t, name):
    if t is None:
        return None
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    return t


def make_rng(seed, step, tensor_id, elem_offset=0, step_dev=None, signs=None, sample_begin=0):
    """signs = (row_sign [S, rows], col_sign [S, cols]) float32 CUDA tensors of +-1: rank-one sign noise (Flipout) for
    the local samples [sample_begin, sample_begin + S) — the kernels index by the global sample number."""
    r = bnn_rng()
    if signs is not None:
        row, col = signs
        require_cuda(row, col)
        _f32c(row, "row_sign"), _f32c(col, "col_sign")
        r.rows, r.cols = row.shape[-1], col.shape[-1]
        r.row_sign = row.data_ptr() - 4 * sample_begin * r.rows
        r.col_sign = col.data_ptr() - 4 * sample_begin * r.cols
    r.seed = seed & 0xFFFFFFFFFFFFFFFF
    r.step = step & 0xFFFFFFFFFFFFFFFF
    r.step_dev = None if step_dev is None else step_dev.data_ptr()
    r.elem_offset = elem_offset
    r.tensor_id = tensor_id & 0xFFFFFFFF
    r.reserved = 0
    return r


def make_view(t_base_ptr, batch_stride, P):
    v = bnn_view()
    v.base = t_base_ptr
    v.batch_stride = batch_stride
    v.P = P
    v.reserved = 0
    return v


# ---------------------------------------------------------------------------------------------
def abi_version():
    return lib().bnn_abi_version()


def device_supported(device=0):
    return lib().bnn_device_supported(int(device)) == 0


def stddev(rho, out=None):
    require_cuda(rho)
    rho = _f32c(rho, "rho")
    if out is None:
        out = torch.empty_like(rho)
    with torch.cuda.device(rho.device):
        _call("bnn_stddev", _ptr(rho), _ptr(out), rho.numel(), _stream())
    _count()
    return out


def materialize(mu, sigma, S, sample_begin, rng, eps_in=None, want_eps=False):
    """[S, *mu.shape] sampled tensors (+ the eps used when want_eps)."""
    require_cuda(mu, sigma, eps_in)
    mu, sigma, eps_in = _f32c(mu, "mu"), _f32c(sigma, "sigma"), _f32c(eps_in, "eps_in")
    out = torch.empty((S,) + tuple(mu.shape), device=mu.device, dtype=torch.float32)
    eps_out = torch.empty_like(out) if want_eps else None
    if eps_in is not None and eps_in.numel() != S * mu.numel():
        raise ValueError("eps_in must hold S * numel values")
    with torch.cuda.device(mu.device):
        _call("bnn_materialize", _ptr(mu), _ptr(sigma), _ptr(eps_in), _ptr(out), _ptr(eps_out),
                                     mu.numel(), S, sample_begin, ctypes.byref(rng), _stream())
    _count()
    return (out, eps_out) if want_eps else out


def sampled_gemm_fwd(a, lda, a_sample_stride, mu_w, sigma_w, mu_b, sigma_b, eps_w, eps_b, y_view,
                     y_sample_stride, M, N, K, S, sample_begin, rng_w, rng_b, precision):
    with torch.cuda.device(a.device):
        _call("bnn_sampled_gemm_fwd", _ptr(a), lda, a_sample_stride, _ptr(mu_w), _ptr(sigma_w),
                                          _ptr(mu_b), _ptr(sigma_b), _ptr(eps_w), _ptr(eps_b), y_view,
                                          y_sample_stride, M, N, K, S, sample_begin, ctypes.byref(rng_w),
                                          ctypes.byref(rng_b) if rng_b is not None else None, precision,
                                          _stream())
    _count()


def sampled_gemm_dgrad(dy_view, dy_sample_stride, mu_w, sigma_w, eps_w, da, lda, a_sample_stride, M, N, K,
                       S, sample_begin, rng_w, precision):
    with torch.cuda.device(da.device):
        _call("bnn_sampled_gemm_dgrad", dy_view, dy_sample_stride, _ptr(mu_w), _ptr(sigma_w), _ptr(eps_w),
                                            _ptr(da), lda, a_sample_stride, M, N, K, S, sample_begin,
                                            ctypes.byref(rng_w), precision, _stream())
    _count()


def sampled_gemm_wgrad(dy_view, dy_sample_stride, a, lda, a_sample_stride, rho_w, eps_w, dmu_w, drho_w, M, N,
                       K, S, sample_begin, rng_w, precision):
    with torch.cuda.device(a.device):
        _call("bnn_sampled_gemm_wgrad", dy_view, dy_sample_stride, _ptr(a), lda, a_sample_stride,
                                            _ptr(rho_w), _ptr(eps_w), _ptr(dmu_w), _ptr(drho_w), M, N, K, S,
                                            sample_begin, ctypes.byref(rng_w), precision, _stream())
    _count()


def bias_grad(dy_view, dy_sample_stride, rho_b, eps_b, dmu_b, drho_b, M, N, S, sample_begin, rng_b):
    with torch.cuda.device(rho_b.device):
        _call("bnn_bias_grad", dy_view, dy_sample_stride, _ptr(rho_b), _ptr(eps_b), _ptr(dmu_b),
                                   _ptr(drho_b), M, N, S, sample_begin, ctypes.byref(rng_b), _stream())
    _count()


def im2col(x, col, geom):
    with torch.cuda.device(x.device):
        _call("bnn_im2col", _ptr(x), _ptr(col), ctypes.byref(geom), _stream())
    _count()


def col2im(dcol, dx, geom, accumulate):
    with torch.cuda.device(dx.device):
        _call("bnn_col2im", _ptr(dcol), _ptr(dx), ctypes.byref(geom), 1 if accumulate else 0, _stream())
    _count()


# ---- implicit-GEMM convolution (NHWC activations, (o, kh, kw, c) weights) ------------------------------------------
def conv_geom(B, H, W, C, OH, OW, Cout, KH, KW, stride, padding, dilation):
    return bnn_conv2d_nhwc(B, H, W, C, OH, OW, Cout, KH, KW, stride[0], stride[1], padding[0], padding[1], dilation[0],
                           dilation[1], 0)


def conv_weight_layout(mu, rho):
    """OIHW mean / scale [Cout, Cg, KH, KW] -> one buffer [3, Cout*KH*KW*Cg] holding mean, sigma = 1e-10 + softplus(scale)
    and scale in (o, kh, kw, c) order."""
    require_cuda(mu, rho)
    mu, rho = _f32c(mu, "mu"), _f32c(rho, "rho")
    Cout, Cg = mu.shape[0], mu.shape[1]
    taps = mu.numel() // (Cout * Cg)
    out = torch.empty((3, mu.numel()), device=mu.device, dtype=torch.float32)
    with torch.cuda.device(mu.device):
        _call("bnn_conv2d_weight_layout", _ptr(mu), _ptr(rho), _ptr(out[0]), _ptr(out[1]), _ptr(out[2]), Cout, Cg, taps,
              _stream())
    _count()
    return out


def conv_weight_unlayout(grads_p, shape):
    """[n, numel] arrays in (o, kh, kw, c) order -> [n, Cout, Cg, KH, KW] (OIHW)."""
    Cout, Cg = shape[0], shape[1]
    taps = grads_p.shape[1] // (Cout * Cg)
    out = torch.empty((grads_p.shape[0],) + tuple(shape), device=grads_p.device, dtype=torch.float32)
    with torch.cuda.device(grads_p.device):
        _call("bnn_conv2d_weight_unlayout", _ptr(grads_p), _ptr(out), grads_p.shape[0], Cout, Cg, taps, _stream())
    _count()
    return out


def nchw_to_nhwc_bias_grad(dy, B, rho_b=None, eps_b=None, dmu_b=None, drho_b=None, sample_begin=0, rng_b=None):
    """dy: NCHW-contiguous [S*B, N, OH, OW] -> the same tensor in channels_last memory (returned as a logical NCHW tensor);
    optionally accumulates the bias gradient in the same pass.  None when the shape is not supported."""
    R, N = dy.shape[0], dy.shape[1]
    P = dy.shape[2] * dy.shape[3]
    if (N + 1) * P * 4 > 48 * 1024 or (dmu_b is not None and N > 256):
        return None
    out = torch.empty(dy.shape, device=dy.device, dtype=torch.float32, memory_format=torch.channels_last)
    with torch.cuda.device(dy.device):
        _call("bnn_nchw_to_nhwc_bias_grad", _ptr(dy), _ptr(out), R, B, N, P, _ptr(rho_b), _ptr(eps_b), _ptr(dmu_b),
              _ptr(drho_b), sample_begin, ctypes.byref(rng_b) if rng_b is not None else None, _stream())
    _count()
    return out


def _channels_last(t):
    """Whether a logical [n, C, *spatial] tensor's memory is channels-last ([n][spatial][C]) without gaps."""
    return t.permute(0, *range(2, t.dim()), 1).is_contiguous()


def _signs_for(a, sign):
    require_cuda(a, sign)
    if a.dim() < 3 or a.dtype != torch.float32 or not (a.is_contiguous() or _channels_last(a)):
        raise ValueError("a must be a float32 [n, C, *spatial] tensor, NC(D)HW-contiguous or channels-last")
    sign = _f32c(sign, "sign")
    if sign.numel() != a.shape[0] * a.shape[1] or sign.device != a.device:
        raise ValueError(f"sign must hold n x C = {a.shape[0]} x {a.shape[1]} values on {a.device}")
    return sign


def flipout_split(a, sign):
    """(a in channels-last memory, sign[n][c] * a in channels-last memory) for a logical [n, C, *spatial] tensor `a` that
    is NC(D)HW-contiguous or channels-last; the first is `a` itself when it already is channels-last.  One read of a."""
    sign = _signs_for(a, sign)
    n, C = a.shape[0], a.shape[1]
    P = a.numel() // (n * C)
    cl = _channels_last(a)
    fmt = torch.channels_last if a.dim() == 4 else torch.channels_last_3d if a.dim() == 5 else None
    def empty():
        if fmt is not None:
            return torch.empty(a.shape, device=a.device, dtype=torch.float32, memory_format=fmt)
        return torch.empty((n,) + tuple(a.shape[2:]) + (C,), device=a.device, dtype=torch.float32).movedim(-1, 1)
    a_cl = a if cl else empty()
    sa_cl = empty()
    with torch.cuda.device(a.device):
        _call("bnn_flipout_split", _ptr(a), int(cl), _ptr(sign), None if cl else _ptr(a_cl), _ptr(sa_cl), n, C, P,
              _stream())
    _count()
    return a_cl, sa_cl


def flipout_combine(a, b, sign, channels_last):
    """a + sign[n][c] * b for two channels-last logical [n, C, *spatial] tensors, written channels-last or
    NC(D)HW-contiguous; bit-identical to torch's `a + b * sign`."""
    sign = _signs_for(a, sign)
    if b.shape != a.shape or not (_channels_last(a) and _channels_last(b)) or b.dtype != torch.float32:
        raise ValueError("flipout_combine: a and b must be float32 channels-last tensors of one shape")
    require_cuda(b)
    n, C = a.shape[0], a.shape[1]
    P = a.numel() // (n * C)
    if channels_last:
        out = torch.empty_like(a)
    else:
        out = torch.empty(a.shape, device=a.device, dtype=torch.float32)
    with torch.cuda.device(a.device):
        _call("bnn_flipout_combine", _ptr(a), _ptr(b), _ptr(sign), _ptr(out), int(channels_last), n, C, P, _stream())
    _count()
    return out


def im2col_nhwc(x_nhwc_ptr_tensor, geom, n_imgs):
    K = geom.KH * geom.KW * geom.C
    col = torch.empty((n_imgs * geom.OH * geom.OW, K), device=x_nhwc_ptr_tensor.device, dtype=torch.float32)
    with torch.cuda.device(col.device):
        _call("bnn_im2col_nhwc", _ptr(x_nhwc_ptr_tensor), _ptr(col), ctypes.byref(geom), n_imgs, _stream())
    _count()
    return col


def col2im_nhwc(dcol, dx, geom, n_imgs):
    with torch.cuda.device(dx.device):
        _call("bnn_col2im_nhwc", _ptr(dcol), _ptr(dx), ctypes.byref(geom), n_imgs, _stream())
    _count()


def sampled_conv2d_fwd(x, x_sample_stride, mu_w, sigma_w, mu_b, sigma_b, eps_w, eps_b, y_view, y_sample_stride, geom, S,
                       sample_begin, rng_w, rng_b):
    with torch.cuda.device(x.device):
        _call("bnn_sampled_conv2d_fwd", _ptr(x), x_sample_stride, _ptr(mu_w), _ptr(sigma_w), _ptr(mu_b), _ptr(sigma_b),
              _ptr(eps_w), _ptr(eps_b), y_view, y_sample_stride, ctypes.byref(geom), S, sample_begin, ctypes.byref(rng_w),
              ctypes.byref(rng_b) if rng_b is not None else None, _stream())
    _count()


def sampled_conv2d_dgrad(dy, mu_w, sigma_w, eps_w, dx, x_sample_stride, geom, S, sample_begin, rng_w):
    with torch.cuda.device(dx.device):
        _call("bnn_sampled_conv2d_dgrad", _ptr(dy), _ptr(mu_w), _ptr(sigma_w), _ptr(eps_w), _ptr(dx), x_sample_stride,
              ctypes.byref(geom), S, sample_begin, ctypes.byref(rng_w), _stream())
    _count()


def sampled_conv2d_wgrad(dy, x, x_sample_stride, rho_w, eps_w, dmu_w, drho_w, geom, S, sample_begin, rng_w):
    with torch.cuda.device(x.device):
        _call("bnn_sampled_conv2d_wgrad", _ptr(dy), _ptr(x), x_sample_stride, _ptr(rho_w), _ptr(eps_w), _ptr(dmu_w),
              _ptr(drho_w), ctypes.byref(geom), S, sample_begin, ctypes.byref(rng_w), _stream())
    _count()


# The same three calls for callers with an explicit lowering to fall back on: False (nothing launched) when the kernels
# refuse the request (stride > 8, a filter window outside the im2col descriptor's range, Cout not a multiple of 32 for
# the input gradient or of 4 for the weight gradient, ...).  The C entry points are the one place that decides.
def try_sampled_conv2d_fwd(x, x_sample_stride, mu_w, sigma_w, mu_b, sigma_b, eps_w, eps_b, y_view, y_sample_stride, geom,
                           S, sample_begin, rng_w, rng_b):
    return _try_call("bnn_sampled_conv2d_fwd", x.device, _ptr(x), x_sample_stride, _ptr(mu_w), _ptr(sigma_w), _ptr(mu_b),
                     _ptr(sigma_b), _ptr(eps_w), _ptr(eps_b), y_view, y_sample_stride, ctypes.byref(geom), S, sample_begin,
                     ctypes.byref(rng_w), ctypes.byref(rng_b) if rng_b is not None else None, _stream())


def try_sampled_conv2d_dgrad(dy, mu_w, sigma_w, eps_w, dx, x_sample_stride, geom, S, sample_begin, rng_w):
    return _try_call("bnn_sampled_conv2d_dgrad", dx.device, _ptr(dy), _ptr(mu_w), _ptr(sigma_w), _ptr(eps_w), _ptr(dx),
                     x_sample_stride, ctypes.byref(geom), S, sample_begin, ctypes.byref(rng_w), _stream())


def try_sampled_conv2d_wgrad(dy, x, x_sample_stride, rho_w, eps_w, dmu_w, drho_w, geom, S, sample_begin, rng_w):
    return _try_call("bnn_sampled_conv2d_wgrad", x.device, _ptr(dy), _ptr(x), x_sample_stride, _ptr(rho_w), _ptr(eps_w),
                     _ptr(dmu_w), _ptr(drho_w), ctypes.byref(geom), S, sample_begin, ctypes.byref(rng_w), _stream())


_kl_ws = {}


def _workspace(cache, device, nbytes):
    ws = cache.get(device)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=device)
        cache[device] = ws
    return ws


def kl(entries, want_sums=True, grad_scale=None, want_total=False):
    """entries: list of (mu, rho, grad_mu|None, grad_rho|None, prior_loc, prior_scale, grad_coeff).
    Returns the per-tensor element sums (float64 device tensor), or with want_total the 0-dim float32
    sum_t grad_coeff[t] * kl_sum[t] (both as a tuple when both are requested), or None."""
    n = len(entries)
    if n == 0:
        raise ValueError("bnn_kl needs at least one tensor")
    table = (bnn_kl_tensor * n)()
    device = entries[0][0].device
    for i, (mu, rho, gmu, grho, loc, scale, coeff) in enumerate(entries):
        require_cuda(mu, rho, gmu, grho)
        _f32c(mu, "mu"), _f32c(rho, "rho"), _f32c(gmu, "grad_mu"), _f32c(grho, "grad_rho")
        if mu.device != device:
            raise ValueError("all tensors of one bnn_kl call must live on one device")
        t = table[i]
        t.mu, t.rho = mu.data_ptr(), rho.data_ptr()
        t.grad_mu = None if gmu is None else gmu.data_ptr()
        t.grad_rho = None if grho is None else grho.data_ptr()
        t.numel = mu.numel()
        t.prior_loc, t.prior_scale, t.grad_coeff, t.reserved = loc, scale, coeff, 0.0
    sums = torch.empty(n, dtype=torch.float64, device=device) if want_sums else None
    total = torch.empty((), dtype=torch.float32, device=device) if want_total else None
    nbytes = lib().bnn_kl_workspace_size(n)
    ws = _workspace(_kl_ws, device, nbytes + 256)
    base = (ws.data_ptr() + 255) & ~255
    with torch.cuda.device(device):
        _call("bnn_kl", table, n, _ptr(sums), _ptr(total), _ptr(grad_scale), ctypes.c_void_p(base), nbytes,
                            _stream())
    _count((n + 23) // 24)
    if want_sums and want_total:
        return sums, total
    return total if want_total else sums


_prune_ws = {}


PRUNE_GENERAL = 1


def prune(entries, flags=0):
    """entries: list of (mu, rho, k, mask_out|None, keys_out|None); mu/rho are modified in place.
    flags=PRUNE_GENERAL forces the general radix-select path for every tensor."""
    n = len(entries)
    if n == 0:
        return
    table = (bnn_prune_tensor * n)()
    device = entries[0][0].device
    for i, (mu, rho, k, mask, keys) in enumerate(entries):
        require_cuda(mu, rho, mask, keys)
        _f32c(mu, "mu"), _f32c(rho, "rho"), _f32c(keys, "keys_out")
        if mask is not None and (mask.dtype not in (torch.uint8, torch.bool) or not mask.is_contiguous()):
            raise TypeError("mask_out must be a contiguous uint8/bool tensor")
        t = table[i]
        t.mu, t.rho = mu.data_ptr(), rho.data_ptr()
        t.mask_out = None if mask is None else mask.data_ptr()
        t.keys_out = None if keys is None else keys.data_ptr()
        t.numel, t.k = mu.numel(), int(k)
        t.flags, t.reserved = flags, 0
    nbytes = lib().bnn_prune_workspace_size(table, n)
    ws = _workspace(_prune_ws, device, nbytes + 256)
    base = (ws.data_ptr() + 255) & ~255
    with torch.cuda.device(device):
        _call("bnn_prune", table, n, ctypes.c_void_p(base), nbytes, _stream())
    _count(14 * ((n + 23) // 24))


def prune_into(entries, flags=0, out=None, kl_priors=None):
    """Out-of-place pruning in one sweep (bnn_prune_into).  entries: list of (mu, rho, k, mask_out|None); returns the list
    of (mu_out, rho_out) tensors — the inputs are not modified.  `out`: optional list of caller-owned (mu_out, rho_out)
    pairs to write into (same shapes, not aliasing the inputs); by default every output is a fresh tensor.
    `kl_priors`: optional list of (prior_loc, prior_scale) per entry — the same sweep then also accumulates every INPUT
    tensor's KL element sum; returns (outs, sums) with sums a float64 [n] tensor (what _C.kl returns per tensor)."""
    n = len(entries)
    if n == 0:
        return [] if kl_priors is None else ([], torch.zeros(0, dtype=torch.float64))
    if kl_priors is not None and len(kl_priors) != n:
        raise ValueError("prune_into: `kl_priors` needs one (loc, scale) pair per entry")
    if out is not None and len(out) != n:
        raise ValueError("prune_into: `out` needs one (mu_out, rho_out) pair per entry")
    table = (bnn_prune_into_tensor * n)()
    device = entries[0][0].device
    outs = []
    f32 = torch.float32
    kl_sums, kl_base = None, 0
    for i, (mu, rho, k, mask) in enumerate(entries):
        if out is None:
            mu_out, rho_out = torch.empty_like(mu), torch.empty_like(rho)
        else:
            mu_out, rho_out = out[i]
            if mu_out.shape != mu.shape or rho_out.shape != rho.shape:
                raise ValueError("prune_into: output shapes must match the inputs")
        # one pass of checks per entry (this loop is on the timed path of a 64-tensor sweep)
        if not (mu.is_cuda and rho.is_cuda and mu_out.is_cuda and rho_out.is_cuda):
            require_cuda(mu, rho, mu_out, rho_out)
        if not (mu.dtype is f32 and rho.dtype is f32 and mu_out.dtype is f32 and rho_out.dtype is f32 and mu.is_contiguous()
                and rho.is_contiguous() and mu_out.is_contiguous() and rho_out.is_contiguous()):
            _f32c(mu, "mu"), _f32c(rho, "rho"), _f32c(mu_out, "mu_out"), _f32c(rho_out, "rho_out")
        outs.append((mu_out, rho_out))
        t = table[i]
        t.mu, t.rho, t.mu_out, t.rho_out = mu.data_ptr(), rho.data_ptr(), mu_out.data_ptr(), rho_out.data_ptr()
        if mask is not None:
            require_cuda(mask)
            if mask.dtype not in (torch.uint8, torch.bool) or not mask.is_contiguous():
                raise TypeError("mask_out must be a contiguous uint8/bool tensor")
            t.mask_out = mask.data_ptr()
        t.numel, t.k, t.flags = mu.numel(), int(k), flags
        if kl_priors is not None:
            if kl_sums is None:
                kl_sums = torch.zeros(n, dtype=torch.float64, device=device)
                kl_base = kl_sums.data_ptr()
            t.kl_sum_out, t.prior_loc, t.prior_scale = kl_base + 8 * i, float(kl_priors[i][0]), float(kl_priors[i][1])
    nbytes = lib().bnn_prune_into_workspace_size(table, n)
    ws = _workspace(_prune_ws, device, nbytes + 256)
    base = (ws.data_ptr() + 255) & ~255
    with torch.cuda.device(device):
        _call("bnn_prune_into", table, n, ctypes.c_void_p(base), nbytes, _stream())
    _count(15 * ((n + 23) // 24))
    return outs if kl_priors is None else (outs, kl_sums)


def adam_kl_step(entries, lr, beta1, beta2, eps, step_dev=None, step=0, peers=None):
    """entries: list of (mu, rho|None, g_mu|None, g_rho|None, m_mu, v_mu, m_rho|None, v_rho|None, prior_loc, prior_scale,
    kl_coeff); parameters and moments are updated in place (include/bnn_b200.h: bnn_adam_kl_step).  rho None = a plain
    parameter (Adam only).  peers = (rank, [base pointer of every rank's flat gradient buffer]) averages the gradients
    over the ranks inside the kernel (bnn_adam_kl_step_peers)."""
    n = len(entries)
    if n == 0:
        return
    table = (bnn_adam_tensor * n)()
    device = entries[0][0].device
    for i, (mu, rho, g_mu, g_rho, m_mu, v_mu, m_rho, v_rho, loc, scale, coeff) in enumerate(entries):
        require_cuda(mu, rho, g_mu, g_rho, m_mu, v_mu, m_rho, v_rho)
        for name, t in (("mu", mu), ("rho", rho), ("g_mu", g_mu), ("g_rho", g_rho), ("m_mu", m_mu), ("v_mu", v_mu),
                        ("m_rho", m_rho), ("v_rho", v_rho)):
            if t is not None and t.dtype != torch.float32:
                raise TypeError(f"{name} must be float32, got {t.dtype}")
            # dense storage in any dimension order (channels_last conv weights): the update is elementwise, all arrays of
            # one tensor only have to share the order
            if t is not None and not ((t.is_contiguous() and mu.is_contiguous())
                                      or (t.stride() == mu.stride() and _dense(t))):
                raise ValueError(f"{name} must be dense with the strides of the parameter")
        e = table[i]
        e.mu, e.rho = mu.data_ptr(), None if rho is None else rho.data_ptr()
        e.g_mu = None if g_mu is None else g_mu.data_ptr()
        e.g_rho = None if g_rho is None else g_rho.data_ptr()
        e.m_mu, e.v_mu = m_mu.data_ptr(), v_mu.data_ptr()
        e.m_rho, e.v_rho = (None, None) if rho is None else (m_rho.data_ptr(), v_rho.data_ptr())
        e.numel, e.prior_loc, e.prior_scale, e.kl_coeff, e.reserved = mu.numel(), loc, scale, coeff, 0.0
    if step_dev is not None:
        require_cuda(step_dev)
    with torch.cuda.device(device):
        if peers is None:
            _call("bnn_adam_kl_step", table, n, lr, beta1, beta2, eps, _ptr(step_dev), int(step), _stream())
        else:
            rank, bases = peers
            pg = bnn_peer_grads()
            pg.world, pg.rank = len(bases), rank
            for r, b in enumerate(bases):
                pg.base[r] = b
            _call("bnn_adam_kl_step_peers", table, n, lr, beta1, beta2, eps, _ptr(step_dev), int(step), ctypes.byref(pg),
                  _stream())
    _count((n + 15) // 16)


def _dense(t):
    """True when `t` covers its elements without gaps or overlap (a permutation of a contiguous tensor)."""
    sizes_strides = sorted((st, sz) for sz, st in zip(t.shape, t.stride()) if sz > 1)
    expect = 1
    for st, sz in sizes_strides:
        if st != expect:
            return False
        expect *= sz
    return True


def pack_gradients(items, flat):
    """items: list of (gradient tensor | None, offset in `flat` (floats), numel); the gradients must be dense in their
    parameter's memory order (the caller checks) — they are copied as raw memory."""
    n = len(items)
    if n == 0:
        return
    table = (bnn_pack_item * n)()
    for i, (g, off, numel) in enumerate(items):
        table[i].src = None if g is None else g.data_ptr()
        table[i].dst_offset, table[i].numel = off, numel
    with torch.cuda.device(flat.device):
        _call("bnn_pack_gradients", table, n, _ptr(flat), _stream())
    _count((n + 31) // 32)


def peer_average(bases, rank, numel, device):
    """bnn_peer_average: in-place average of the ranks' flat gradient buffers (bases = every rank's buffer as mapped here)."""
    pg = bnn_peer_grads()
    pg.world, pg.rank = len(bases), rank
    for r, b in enumerate(bases):
        pg.base[r] = b
    with torch.cuda.device(device):
        _call("bnn_peer_average", ctypes.byref(pg), int(numel), _stream())
    _count()


def peer_barrier(flag_ptrs, rank, epoch, device):
    """bnn_peer_barrier: flag_ptrs = [every rank's flag block as mapped here], epoch = local uint32/int32 [1] tensor."""
    world = len(flag_ptrs)
    arr = (ctypes.c_void_p * world)(*flag_ptrs)
    with torch.cuda.device(device):
        _call("bnn_peer_barrier", arr, world, rank, _ptr(epoch), _stream())
    _count()


_ce_ws = {}


def _check_ce(x, target):
    require_cuda(x, target)
    if x.dtype != torch.float32 or x.dim() != 2 or x.stride(1) != 1 or x.stride(0) < x.shape[1]:
        raise TypeError("x must be a float32 [rows, classes] matrix with unit column stride")
    if target.dtype != torch.int64 or target.dim() != 1 or not target.is_contiguous():
        raise TypeError("target must be a contiguous int64 vector of class indices")
    if target.numel() == 0 or x.shape[0] % target.numel() != 0:
        raise ValueError(f"{x.shape[0]} rows are not a whole number of blocks of {target.numel()} labels")


def mc_cross_entropy_fwd(x, target, ignore_index=-100):
    """(loss, lse, count) of bnn_mc_cross_entropy_fwd: x [S*B, C] float32 (row pitch x.stride(0)), target [B] int64."""
    _check_ce(x, target)
    rows, classes = x.shape
    lse = torch.empty(rows, dtype=torch.float32, device=x.device)
    out = torch.empty(2, dtype=torch.float32, device=x.device)          # loss, count
    nbytes = lib().bnn_mc_cross_entropy_workspace_size()
    ws = _ce_ws.get(x.device)
    if ws is None or ws.numel() < nbytes + 256:
        ws = torch.zeros(nbytes + 256, dtype=torch.uint8, device=x.device)      # zero once; calls leave it ready
        _ce_ws[x.device] = ws
    base = (ws.data_ptr() + 255) & ~255
    with torch.cuda.device(x.device):
        _call("bnn_mc_cross_entropy_fwd", _ptr(x), x.stride(0), _ptr(target), rows, target.numel(), classes,
              int(ignore_index), _ptr(lse), _ptr(out[0]), _ptr(out[1]), ctypes.c_void_p(base), nbytes, _stream())
    _count()
    return out[0], lse, out[1]


def mc_cross_entropy_bwd(x, target, lse, count, grad_loss, ignore_index=-100):
    """dx [S*B, C] of bnn_mc_cross_entropy_bwd (grad_loss: 0-dim float32 device tensor)."""
    _check_ce(x, target)
    require_cuda(lse, count, grad_loss)
    _f32c(lse, "lse"), _f32c(count, "count"), _f32c(grad_loss, "grad_loss")
    rows, classes = x.shape
    dx = torch.empty((rows, classes), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _call("bnn_mc_cross_entropy_bwd", _ptr(x), x.stride(0), _ptr(target), rows, target.numel(), classes,
              int(ignore_index), _ptr(lse), _ptr(count), _ptr(grad_loss), _ptr(dx), classes, _stream())
    _count()
    return dx


def selftest_prune_interval(mu, rho, variant=1):
    """(lo, hi): the certified key2 interval bnn_prune uses for every element (see include/bnn_b200.h)."""
    require_cuda(mu, rho)
    _f32c(mu, "mu"), _f32c(rho, "rho")
    lo, hi = torch.empty_like(mu), torch.empty_like(mu)
    with torch.cuda.device(mu.device):
        _call("bnn_selftest_prune_interval", _ptr(mu), _ptr(rho), mu.numel(), _ptr(lo), _ptr(hi), int(variant), _stream())
    _count()
    return lo, hi


def force_contract_variant(variant):
    """Test aid: 'pair' | 'mb4' | 'mb2' | 'mb1' | None (cost model) for the TMA-fed forward / data-gradient kernels."""
    code = {None: -1, "pair": 0, "mb1": 1, "mb2": 2, "mb4": 4}[variant]
    _check(lib().bnn_debug_force_contract_variant(code), "bnn_debug_force_contract_variant")


def wgrad_plan(M, N, K, S, sms=None):
    """Host-side plan of the TMA weight gradient (no device needed): dict of pair, n_chunks, chunk_blocks, units_per_cta
    and groups on `sms` SMs (default: those of the current device), including a forced override."""
    if sms is None:
        sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    out = (ctypes.c_int32 * 5)()
    _check(lib().bnn_debug_wgrad_plan(M, N, K, S, sms, out), "bnn_debug_wgrad_plan")
    return dict(zip(("pair", "n_chunks", "chunk_blocks", "units_per_cta", "groups"), list(out)))


def force_wgrad_plan(pair=None, n_chunks=None, units_per_cta=None):
    """Test aid: force parts of the TMA weight-gradient plan (None = the cost model's choice; all None resets).  A forced
    value the shape cannot take makes the launch raise instead of running another plan."""
    code = lambda v: -1 if v is None else int(v)
    _check(lib().bnn_debug_force_wgrad_plan(code(pair), code(n_chunks), code(units_per_cta)), "bnn_debug_force_wgrad_plan")


def selftest_umma(device="cuda", mn_major=False):
    out = torch.zeros(1, dtype=torch.float32, device=device)
    with torch.cuda.device(out.device):
        _call("bnn_selftest_umma_mn" if mn_major else "bnn_selftest_umma", _ptr(out), _stream())
    _count()
    return float(out.item())


# ---- transposed convolution (geometry = the conv view, see bnn_b200.h) ----------------------------------------------
def try_sampled_conv_transpose2d_fwd(x, x_sample_stride, mu_w, sigma_w, mu_b, sigma_b, eps_w, eps_b, y, geom, S,
                                     sample_begin, rng_w, rng_b):
    """The phase-decomposed gather; False (nothing launched) when the kernels do not take the request."""
    return _try_call("bnn_sampled_conv_transpose2d_fwd", y.device, _ptr(x), x_sample_stride, _ptr(mu_w), _ptr(sigma_w),
                     _ptr(mu_b), _ptr(sigma_b), _ptr(eps_w), _ptr(eps_b), _ptr(y), ctypes.byref(geom), S, sample_begin,
                     ctypes.byref(rng_w), ctypes.byref(rng_b) if rng_b is not None else None, _stream())


def try_sampled_conv_transpose2d_dgrad(dy, mu_w, sigma_w, eps_w, dx, x_sample_stride, geom, S, sample_begin, rng_w):
    return _try_call("bnn_sampled_conv_transpose2d_dgrad", dx.device, _ptr(dy), _ptr(mu_w), _ptr(sigma_w), _ptr(eps_w),
                     _ptr(dx), x_sample_stride, ctypes.byref(geom), S, sample_begin, ctypes.byref(rng_w), _stream())


def try_sampled_conv_transpose2d_wgrad(dy, x, x_sample_stride, rho_w, eps_w, dmu_w, drho_w, geom, S, sample_begin, rng_w):
    return _try_call("bnn_sampled_conv_transpose2d_wgrad", x.device, _ptr(dy), _ptr(x), x_sample_stride, _ptr(rho_w),
                     _ptr(eps_w), _ptr(dmu_w), _ptr(drho_w), ctypes.byref(geom), S, sample_begin, ctypes.byref(rng_w),
                     _stream())


def _try_call(name, device, *args):
    """Like _call, but BNN_ERR_UNSUPPORTED (a request outside the kernels' stated limits) returns False."""
    with torch.cuda.device(device):
        rc = _invoke(name, *args)
    if rc == _ERR_UNSUPPORTED:
        return False
    _check(rc, name)
    _count()
    return True


def conv_transpose_supported(geom):
    """Whether the transposed-convolution kernels take all three passes of this conv-view geometry (bnn_conv2d_nhwc or
    bnn_conv3d_nhwc); host only, nothing is launched.  Raises for an inconsistent geometry."""
    name = "bnn_conv_transpose3d_supported" if isinstance(geom, bnn_conv3d_nhwc) else "bnn_conv_transpose2d_supported"
    rc = getattr(lib(), name)(ctypes.byref(geom))
    if rc == _ERR_UNSUPPORTED:
        return False
    _check(rc, name)
    return True


def conv_transpose_phases(geom):
    """Host-side phase plan of bnn_sampled_conv_transpose2d_fwd: one dict per output phase (no device needed)."""
    cap = 64
    buf = (ctypes.c_int32 * (14 * cap))()
    n = lib().bnn_debug_conv_transpose_phases(ctypes.byref(geom), buf, cap)
    if n < 0:
        _check(-n, "bnn_debug_conv_transpose_phases")
    keys = ("rh", "rw", "rows_h", "rows_w", "taps_h", "taps_w", "last_h", "last_w", "tap_step_h", "tap_step_w",
            "first_h", "first_w", "in_step_h", "in_step_w")
    return [dict(zip(keys, buf[14 * i:14 * i + 14])) for i in range(min(n, cap))]


# ---- 3-d transposed convolution (NDHWC; geometry = the conv view, see bnn_b200.h) -------------------------------------
def conv3d_geom(B, D, H, W, C, OD, OH, OW, Cout, kernel, stride, padding, dilation):
    return bnn_conv3d_nhwc(B, D, H, W, C, OD, OH, OW, Cout, *kernel, *stride, *padding, *dilation, 0)


def try_sampled_conv_transpose3d_fwd(x, x_sample_stride, mu_w, sigma_w, mu_b, sigma_b, eps_w, eps_b, y, geom, S,
                                     sample_begin, rng_w, rng_b):
    """The phase-decomposed gather; False (nothing launched) when the request is outside the kernels' limits."""
    return _try_call("bnn_sampled_conv_transpose3d_fwd", y.device, _ptr(x), x_sample_stride, _ptr(mu_w), _ptr(sigma_w),
                     _ptr(mu_b), _ptr(sigma_b), _ptr(eps_w), _ptr(eps_b), _ptr(y), ctypes.byref(geom), S, sample_begin,
                     ctypes.byref(rng_w), ctypes.byref(rng_b) if rng_b is not None else None, _stream())


def sampled_conv_transpose3d_dgrad(dy, mu_w, sigma_w, eps_w, dx, x_sample_stride, geom, S, sample_begin, rng_w):
    """Raises on refusal: the forward that accepted the request checked the same predicate."""
    with torch.cuda.device(dx.device):
        _call("bnn_sampled_conv_transpose3d_dgrad", _ptr(dy), _ptr(mu_w), _ptr(sigma_w), _ptr(eps_w), _ptr(dx),
              x_sample_stride, ctypes.byref(geom), S, sample_begin, ctypes.byref(rng_w), _stream())
    _count()


def sampled_conv_transpose3d_wgrad(dy, x, x_sample_stride, rho_w, eps_w, dmu_w, drho_w, geom, S, sample_begin, rng_w):
    with torch.cuda.device(x.device):
        _call("bnn_sampled_conv_transpose3d_wgrad", _ptr(dy), _ptr(x), x_sample_stride, _ptr(rho_w), _ptr(eps_w),
              _ptr(dmu_w), _ptr(drho_w), ctypes.byref(geom), S, sample_begin, ctypes.byref(rng_w), _stream())
    _count()


def conv_transpose3d_phases(geom):
    """Host-side phase plan of bnn_sampled_conv_transpose3d_fwd: one dict per output phase (no device needed)."""
    cap = 512
    buf = (ctypes.c_int32 * (21 * cap))()
    n = lib().bnn_debug_conv_transpose3d_phases(ctypes.byref(geom), buf, cap)
    if n < 0:
        _check(-n, "bnn_debug_conv_transpose3d_phases")
    fields = ("r", "rows", "taps", "last", "tap_step", "first", "in_step")
    keys = tuple(f"{f}_{a}" for f in fields for a in "dhw")
    return [dict(zip(keys, buf[21 * i:21 * i + 21])) for i in range(min(n, cap))]
