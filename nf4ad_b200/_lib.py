"""ctypes binding of libusflow_b200.so (the C ABI in include/usflow_b200.h).

The product path has NO CPU fallback: if the shared library is missing, or a compute entry point is
called without a CUDA (sm_100) device / on a non-CUDA tensor, this module raises.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libusflow_b200.so")

USF_PREC_FP32 = 0
USF_PREC_BF16 = 1
USF_PREC_TF32X3 = 2
USF_PREC_BF16X2 = 3
USF_MAX_MLP = 8

_i64, _i32, _f32, _vp, _sz = C.c_int64, C.c_int32, C.c_float, C.c_void_p, C.c_size_t
_int = C.c_int


class LinearDesc(C.Structure):
    _fields_ = [("W", _vp), ("Wb", _vp), ("bias", _vp), ("N", _i32), ("K", _i32), ("ldw", _i32)]


class BlockDesc(C.Structure):
    _fields_ = [("G", LinearDesc), ("b_off", _i32), ("n_mlp", _i32), ("mlp", LinearDesc * USF_MAX_MLP),
                ("Da", _i32), ("Db", _i32), ("C", _i32), ("affine", _i32), ("clamp", _f32)]


class StackDesc(C.Structure):
    _fields_ = [("D", _i32), ("n_blocks", _i32), ("blocks", C.POINTER(BlockDesc)), ("G_final", LinearDesc),
                ("inverse", _i32), ("base_kind", _i32), ("loc", _vp), ("inv_scale", _vp), ("const_term", _f32),
                ("ctx_dim", _i32)]


class BlockGradDesc(C.Structure):
    _fields_ = [("G", LinearDesc), ("mlp", LinearDesc * USF_MAX_MLP)]


class StackGradDesc(C.Structure):
    _fields_ = [("n_blocks", _i32), ("blocks", C.POINTER(BlockGradDesc)), ("G_final", LinearDesc)]


# name -> (restype, argtypes); mirrors include/usflow_b200.h one to one
_PROTOS = {
    "usf_version": (_int, []),
    "usf_last_error": (C.c_char_p, []),
    "usf_device_ok": (_int, []),
    "usf_stream_create": (_int, [_int, C.POINTER(_vp)]),
    "usf_stream_destroy": (_int, [_vp]),
    "usf_lu_pack": (_int, [_vp, _vp, _i64, _vp, _vp, _vp, _vp]),
    "usf_linear": (_int, [_vp, _i64, _vp, _i64, _vp, _int, _vp, _i64, _i64, _i64, _i64, _vp]),
    "usf_lu_inverse_scratch_floats": (_i64, [_i64]),
    "usf_lu_inverse": (_int, [_vp, _vp, _i64, _vp, _vp, _vp]),
    "usf_lu_solve": (_int, [_vp, _i64, _vp, _vp, _vp, _int, _vp, _i64, _i64, _i64, _vp, _vp]),
    "usf_lu_solve_scratch_floats": (_i64, [_i64]),
    "usf_householder": (_int, [_vp, _i64, _vp, _i64, _int, _vp, _i64, _i64, _i64, _vp]),
    "usf_scale": (_int, [_vp, _i64, _vp, _int, _vp, _i64, _i64, _i64, _vp]),
    "usf_sum_log_abs": (_int, [_vp, _i64, _i64, _vp, _vp]),
    "usf_coupling": (_int, [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _f32, _int, _int, _vp, _i64, _vp, _f32, _i64, _i64, _vp]),
    "usf_base_logprob": (_int, [_int, _vp, _i64, _vp, _vp, _i64, _vp, _f32, _vp, _i64, _i64, _vp]),
    "usf_linear_bwd": (_int, [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _int, _vp,
                              _i64, _i64, _i64, _vp]),
    "usf_linear_bwd_scratch_bytes": (_sz, [_i64, _i64]),
    "usf_lu_pack_bwd": (_int, [_vp, _vp, _vp, _f32, _i64, _vp, _vp, _vp, _vp]),
    "usf_scale_bwd": (_int, [_vp, _i64, _vp, _i64, _vp, _int, _vp, _i64, _vp, _i64, _i64, _vp]),
    "usf_to_bf16": (_int, [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _i64, _vp]),
    "usf_stack_run_bf16in": (_int, [C.POINTER(StackDesc), _vp, _i64, _i64, _vp, _vp, _i64, _vp, _vp, _sz,
                                    C.POINTER(C.c_int), _vp]),
    "usf_host_f32_to_bf16": (_int, [_vp, _i64, _vp, _i64, _i64, _i64, _int]),
    "usf_host_copy_f32": (_int, [_vp, _i64, _vp, _i64, _i64, _i64, _int]),
    "usf_vae_reparam": (_int, [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _i64, _vp]),
    "usf_vae_reparam_bwd": (_int, [_vp, _i64, _vp, _vp, _i64, _vp, _i64, _vp, _i64, _i64, _i64, _vp]),
    "usf_recon_nll": (_int, [_vp, _vp, _i64, _i64, _f32, _vp, _vp]),
    "usf_recon_nll_bwd": (_int, [_vp, _vp, _vp, _i64, _i64, _f32, _vp, _vp, _vp]),
    "usf_adam_step": (_int, [_vp, _int, _vp, _f32, _f32, _f32, _f32, _f32, _int, _vp, _vp]),
    "usf_sophia_step": (_int, [_vp, _int, _vp, _f32, _f32, _f32, _f32, _f32, _f32, _int, _vp, _vp]),
    "usf_to_tf32x3": (_int, [_vp, _i64, _vp, _i64, _vp, _vp, _i64, _vp, _vp, _i64, _vp, _i64, _i64, _vp]),
    "usf_colsum": (_int, [_vp, _i64, _f32, _int, _vp, _i64, _i64, _vp]),
    "usf_gemm": (_int, [_vp, _i64, _int, _vp, _i64, _int, _vp, _i64, _int, _i64, _i64, _i64, _vp]),
    "usf_coupling_bwd": (_int, [_vp, _i64, _vp, _f32, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _f32, _int, _int, _vp, _i64,
                                _vp, _i64, _vp, _i64, _i64, _i64, _vp]),
    "usf_householder_bwd": (_int, [_vp, _i64, _vp, _i64, _vp, _i64, _int, _vp, _i64, _vp, _vp, _i64, _i64, _vp]),
    "usf_base_logprob_bwd": (_int, [_int, _vp, _vp, _i64, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _i64, _i64, _vp]),
    "usf_pack_matrix": (_int, [_vp, _i64, _vp, _vp, _int, _int, _i64, _i64, _vp, _vp, _i64, _vp]),
    "usf_stack_workspace_bytes": (_sz, [C.POINTER(StackDesc), _i64, _int]),
    "usf_stack_is_single_kernel": (_int, [C.POINTER(StackDesc), _int]),
    "usf_set_deterministic": (_int, [_int]),
    "usf_stack_run": (_int, [C.POINTER(StackDesc), _vp, _i64, _i64, _vp, _vp, _i64, _vp, _vp, _sz, _int,
                             C.POINTER(_int), _vp]),
    "usf_stack_grad_workspace_bytes": (_sz, [C.POINTER(StackDesc), C.POINTER(StackGradDesc), _i64, _int]),
    "usf_stack_log_prob_grad": (_int, [C.POINTER(StackDesc), C.POINTER(StackGradDesc), _vp, _i64, _i64, _vp, _vp, _i64,
                                       _vp, _sz, _int, C.POINTER(_int), _vp]),
    "usf_profile_begin": (_int, [_int]),
    "usf_profile_end": (_int, [C.POINTER(_f32), C.POINTER(_int), C.POINTER(_int)]),
    "usf_debug_graph_stats": (_int, [C.POINTER(C.c_longlong), C.c_char_p, _int]),
    "usf_debug_tc_timeout": (_int, [C.POINTER(_int), _int]),
    "usf_split_lo": (_int, [_vp, _i64, _vp, _i64, _i64, _i64, _vp]),
    "usf_linear_tf32x3": (_int, [_vp, _vp, _i64, _vp, _vp, _i64, _vp, _int, _vp, _vp, _i64, _i64, _i64, _i64, _vp]),
    "usf_linear_bf16": (_int, [_vp, _i64, _vp, _i64, _vp, _int, _vp, _i64, _int, _i64, _i64, _i64, _vp]),
    "usf_gemm_kernel_name": (C.c_char_p, [_int]),
}

EXPORTED = tuple(_PROTOS)
_lib = None


class USFError(RuntimeError):
    pass


def lib():
    """Loads the shared library (once).  Raises if it has not been built: there is no fallback path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise USFError(
                f"{LIB_PATH} is missing: build it with `python -m nf4ad_b200.build` "
                "(the B200 path has no CPU/PyTorch fallback)")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOS.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().usf_last_error().decode("utf-8", "replace")
        raise USFError(f"{what or 'usflow_b200'} failed (code {rc}): {msg}")


def require_cuda(*tensors):
    """Every operand is a CUDA tensor of ONE device, and that device is the current one: the library launches on the
    current device's current stream (`stream()`), so operands of another GPU would be touched through device 0's
    stream -- an illegal access or silent peer traffic.  `Flow` / `ADBenchFlow` enter `torch.cuda.device(x.device)`
    around their calls; direct callers of the layer kernels must do the same."""
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise USFError(
                "nf4ad_b200 runs on CUDA (sm_100a) tensors only and has no CPU fallback; got a "
                f"{t.device} tensor. Move the flow and its inputs to a B200 (`flow.to('cuda')`).")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise USFError(f"operands live on different GPUs ({dev} and {t.device})")
    if dev is not None and dev.index != torch.cuda.current_device():
        raise USFError(
            f"operands live on {dev} but the current CUDA device is cuda:{torch.cuda.current_device()}: wrap the call "
            f"in `with torch.cuda.device({dev.index}):` (Flow / ADBenchFlow do this themselves)")


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def new_stream(device, priority=0):
    """A stream of its own on `device` (torch's `Stream()` hands out a pool of 32 per device round-robin: the ~20 side
    streams of a training step plus whatever else the process created would alias, and two aliased chains run one after
    the other).  `priority`: 0 default, negative = more urgent.  Wrapped as an `ExternalStream`; lives as long as the
    process."""
    device = torch.device(device)
    handle = _vp()
    with torch.cuda.device(device):
        check(lib().usf_stream_create(int(priority), C.byref(handle)), "usf_stream_create")
    return torch.cuda.ExternalStream(handle.value, device=device)


_STREAM_POOL = {}


def pooled_stream(device, name, priority=0):
    """The process-wide stream `name` of `device`, created on first use.  Flows and trainers come and go (one per
    hyper-parameter trial); the streams they fork their weight-space work onto are shared per device instead of being
    created per object, so a long sweep does not accumulate thousands of CUDA streams."""
    device = torch.device(device)
    key = (device.index if device.index is not None else torch.cuda.current_device(), name)
    st = _STREAM_POOL.get(key)
    if st is None:
        st = _STREAM_POOL[key] = new_stream(device, priority)
    return st


def stream():
    """torch's current stream of the current device (`require_cuda` has checked that the operands live there)."""
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# Packed-weight caches (`Flow._compiled`) are keyed by the parameters' (id, _version) pairs.  Updates that bypass
# torch's version counters -- `FusedAdam` writing through raw pointers, a CUDA-graph replay of a whole training step
# -- bump this epoch instead; it is part of every flow's key.
_WEIGHTS_EPOCH = [0]


def bump_weights_epoch():
    _WEIGHTS_EPOCH[0] += 1


def weights_epoch():
    return _WEIGHTS_EPOCH[0]


def f32c(t):
    """fp32, last-dim-contiguous 2-D view (no copy when already so)."""
    if t.dtype != torch.float32:
        t = t.float()
    if t.dim() >= 1 and t.stride(-1) != 1:
        t = t.contiguous()
    return t
