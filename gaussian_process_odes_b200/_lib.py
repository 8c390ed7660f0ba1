"""ctypes binding of ``libgpode_b200.so`` (C ABI declared in ``include/gpode_b200.h``).

There is no CPU or PyTorch fallback: if the shared library is missing or a call fails, an exception is raised.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgpode_b200.so")

c_float_p = ctypes.c_void_p  # device pointers travel as plain addresses
c_stream = ctypes.c_void_p


class GpodeCache(ctypes.Structure):
    """``gpode_cache_t`` of include/gpode_b200.h."""
    _fields_ = [("D", ctypes.c_int32), ("M", ctypes.c_int32), ("S", ctypes.c_int32),
                ("omega", ctypes.c_void_p), ("phase", ctypes.c_void_p), ("w", ctypes.c_void_p),
                ("Z", ctypes.c_void_p), ("nu", ctypes.c_void_p), ("ell", ctypes.c_void_p), ("var", ctypes.c_void_p)]


class GpodeShoot(ctypes.Structure):
    """``gpode_shoot_t`` of include/gpode_b200.h."""
    _fields_ = [("S_mc", ctypes.c_int32), ("N", ctypes.c_int32), ("T", ctypes.c_int32), ("D_obs", ctypes.c_int32),
                ("laplace", ctypes.c_int32), ("ys", ctypes.c_void_p), ("W", ctypes.c_void_p), ("bias", ctypes.c_void_p),
                ("lik_var", ctypes.c_void_p), ("cons_scale", ctypes.c_void_p), ("row_lo", ctypes.c_int64),
                ("row_hi", ctypes.c_int64)]


_I, _L, _P, _D, _F = ctypes.c_int, ctypes.c_int64, ctypes.c_void_p, ctypes.c_double, ctypes.c_float
_CP = ctypes.POINTER(GpodeCache)

# name -> (restype, argtypes); every symbol include/gpode_b200.h declares
SIGNATURES = {
    "gpode_abi_version": (_I, []),
    "gpode_last_error": (ctypes.c_char_p, []),
    "gpode_packed_floats": (_L, [_I, _I, _I]),
    "gpode_pack_cache": (_I, [_CP, _P, _P]),
    "gpode_vf_fwd": (_I, [_P, _I, _I, _I, _P, _P, _L, _P]),
    "gpode_vf_bwd": (_I, [_P, _I, _I, _I, _P, _P, _P, _P, _P, _L, _P]),
    "gpode_rk4_fwd": (_I, [_P, _I, _I, _I, _P, _P, _I, _L, _P, _P, _P]),
    "gpode_rk4_bwd": (_I, [_P, _I, _I, _I, _P, _I, _L, _P, _P, _P, _P, _P, _P, _P]),
    "gpode_param_grad": (_I, [_P, _I, _I, _I, _P, _P, _L, _P, _P]),
    "gpode_acc_floats": (_L, [_I, _I]),
    "gpode_vrow_floats": (_L, [_I, _L]),
    "gpode_grads_finalize": (_I, [_CP, _P, _P, _P, _P, _P, _P]),
    "gpode_whiten_fwd": (_I, [_CP, _P, _F, _P, _P, _P, _P]),
    "gpode_whiten_bwd": (_I, [_CP, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "gpode_kl_fwd": (_I, [_P, _P, _I, _I, _P, _P]),
    "gpode_kl_bwd": (_I, [_P, _P, _I, _I, _P, _P, _P, _P]),
    "gpode_inducing_sample_fwd": (_I, [_P, _P, _P, _I, _I, _P, _P]),
    "gpode_inducing_sample_bwd": (_I, [_P, _P, _I, _I, _P, _P]),
    "gpode_dopri5_work_floats": (_L, [_I, _L]),
    "gpode_state_fwd": (_I, [_P, _P, _P, _I, _L, _I, _F, _P, _P, _P]),
    "gpode_state_bwd": (_I, [_P, _P, _I, _L, _I, _F, _P, _P, _P, _P, _P]),
    "gpode_loglik_sum": (_I, [_P, _P, _P, _P, _P, _I, _L, _I, _I, _P, _P, _P, _P, _P]),
    "gpode_constraint_sum": (_I, [_P, _P, _P, _L, _I, _I, _I, _P, _P, _P, _P, _P]),
    "gpode_side_work_doubles": (_L, []),
    "gpode_set_option": (_I, [ctypes.c_char_p, _I]),
    "gpode_get_option": (_I, [ctypes.c_char_p]),
    "gpode_shoot_work_doubles": (_L, []),
    "gpode_packed_large_bwd_floats": (_L, [_I, _I, _I]),
    "gpode_acc_large_floats": (_L, [_I, _I]),
    "gpode_pack_cache_large_bwd": (_I, [_CP, _P, _P]),
    "gpode_vf_bwd_large": (_I, [_P, _I, _I, _I, _P, _P, _P, _P, _P, _L, _P]),
    "gpode_grads_finalize_large": (_I, [_CP, _P, _L, _P, _P, _P, _P, _P]),
    "gpode_rk4_fwd_large_dev": (_I, [_P, _CP, _P, _P, _I, _L, _P, _P, _P, _P]),
    "gpode_rk4_bwd_large": (_I, [_P, _CP, _P, _I, _L, _P, _P, _P, _P, _P, _P, _P]),
    "gpode_dopri5_large_work_floats": (_L, [_I, _L]),
    "gpode_dopri5_fwd_large": (_I, [_P, _CP, _P, _P, _I, _L, _D, _D, _P, _P, _P, _I, _P]),
    "gpode_dopri5_fwd_large_ckpt": (_I, [_P, _CP, _P, _P, _I, _L, _D, _D, _P, _P, _P, _I, _P, _I, _P]),
    "gpode_dopri5_bwd_large": (_I, [_P, _CP, _P, _I, _L, _P, _P, _I, _I, _P, _P, _P, _P]),
    "gpode_shoot_fwd": (_I, [_P, _I, _I, _I, ctypes.POINTER(GpodeShoot), _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "gpode_shoot_bwd": (_I, [_P, _I, _I, _I, ctypes.POINTER(GpodeShoot), _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "gpode_shoot_bwd_vrows": (_L, [_I, _I, _I, _L]),
    "gpode_shoot_large_work_doubles": (_L, [_I, _L]),
    "gpode_shoot_fwd_large": (_I, [_P, _CP, ctypes.POINTER(GpodeShoot), _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "gpode_shoot_bwd_large": (_I, [_P, _CP, ctypes.POINTER(GpodeShoot), _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "gpode_acc_header_floats": (_L, []),
    "gpode_probe_fp32_fma": (_I, [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double), _P, _P]),
    "gpode_dopri5_ckpt_floats": (_L, [_I, _L, _I, _I]),
    "gpode_dopri5_fwd": (_I, [_P, _I, _I, _I, _P, _P, _I, _L, _D, _D, _P, _P, _P, _P, _I, _P]),
    "gpode_dopri5_bwd": (_I, [_P, _I, _I, _I, _P, _I, _L, _P, _P, _I, _I, _P, _P, _P, _P]),
    "gpode_dopri5_bwd_dev": (_I, [_P, _I, _I, _I, _P, _I, _L, _P, _P, _I, _P, _P, _P, _P, _P]),
    "gpode_param_grad_dev": (_I, [_P, _I, _I, _I, _P, _P, _L, _P, _L, _P, _P]),
    "gpode_packed_large_floats": (_L, [_I, _I, _I]),
    "gpode_rbf_fwd_large": (_I, [_P, _I, _I, _I, _P, _P, _P, _P, _L, _P]),
    "gpode_pack_cache_large": (_I, [_CP, _P, _P]),
    "gpode_rff_fwd_large": (_I, [_P, _I, _I, _P, _P, _L, _P]),
    "gpode_vf_fwd_large_add_rbf": (_I, [_CP, _P, _P, _P, _L, _P]),
    "gpode_pack_cache_sets": (_I, [_CP, _I, _P, _P]),
    "gpode_whiten_fwd_sets": (_I, [_CP, _P, _F, _I, _P, _P, _P, _P]),
    "gpode_vf_fwd_sets": (_I, [_P, _I, _I, _I, _I, _L, _P, _P, _P]),
    "gpode_rk4_fwd_sets": (_I, [_P, _I, _I, _I, _I, _L, _P, _P, _I, _P, _P]),
    "gpode_dopri5_fwd_sets": (_I, [_P, _I, _I, _I, _I, _L, _P, _P, _I, _D, _D, _P, _P, _P, _P]),
    "gpode_pack_cache_large_sets": (_I, [_CP, _I, _P, _P]),
    "gpode_vf_fwd_large_sets": (_I, [_P, _CP, _I, _L, _P, _P, _P, _P]),
    "gpode_rk4_fwd_large_sets": (_I, [_P, _CP, _I, _L, _P, _P, _I, _P, _P, _P]),
    "gpode_dopri5_large_sets_work_floats": (_L, [_I, _I, _L]),
    "gpode_dopri5_fwd_large_sets": (_I, [_P, _CP, _I, _L, _P, _P, _I, _D, _D, _P, _P, _P, _I, _P]),
    "gpode_whiten_blocked_work_doubles": (_L, [_I, _I, _I]),
    "gpode_whiten_fwd_blocked": (_I, [_CP, _P, _F, _P, _P, _P, _P, _P]),
    "gpode_whiten_fwd_sets_blocked": (_I, [_CP, _P, _F, _I, _P, _P, _P, _P, _P]),
    "gpode_whiten_bwd_blocked": (_I, [_CP, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
}

_lib = None


class GpodeError(RuntimeError):
    pass


def load():
    """Load the shared library (once). Raises if it has not been built -- no fallback exists."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GpodeError(
            "%s is missing: build it with `python -m gaussian_process_odes_b200.build` "
            "(or __graft_entry__.build()). The GPODE hot path has no CPU / PyTorch fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch, fail loudly
        fn.restype, fn.argtypes = res, args
    if lib.gpode_abi_version() != 2:
        raise GpodeError("libgpode_b200.so ABI version %d, expected 2" % lib.gpode_abi_version())
    _lib = lib
    return lib


def set_option(name, value):
    """Process-wide kernel-selection option (``gpode_set_option``): bwd_mma, fwd_mma."""
    check(load().gpode_set_option(name.encode(), int(value)))


def get_option(name):
    return load().gpode_get_option(name.encode())


def check(rc):
    if rc != 0:
        msg = load().gpode_last_error().decode("utf-8", "replace")
        raise GpodeError("gpode_b200 call failed (rc=%d): %s" % (rc, msg))


def stream_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device address of a contiguous float32/float64/int32 CUDA tensor (or NULL for None)."""
    if t is None:
        return ctypes.c_void_p(0)
    if not t.is_cuda:
        raise GpodeError("gpode_b200 needs CUDA tensors, got device %s (there is no CPU path)" % t.device)
    if not t.is_contiguous():
        raise GpodeError("gpode_b200 needs contiguous tensors")
    return ctypes.c_void_p(t.data_ptr())


def f32(t, name="tensor"):
    """Detached contiguous float32 CUDA view of ``t`` (raises instead of silently moving/casting)."""
    if t.dtype != torch.float32:
        raise GpodeError("%s must be float32, got %s" % (name, t.dtype))
    if not t.is_cuda:
        raise GpodeError("%s must live on a CUDA device, got %s (there is no CPU path)" % (name, t.device))
    return t.detach().contiguous()


# ---- launch accounting and optional per-call CUDA-event timing (used by bench.py) --------------------------------
# kernels enqueued by one C-ABI call (memsets / memcpys not counted)
KERNELS_PER_CALL = {
    "gpode_pack_cache": 1, "gpode_vf_fwd": 1, "gpode_vf_bwd": 1, "gpode_rk4_fwd": 1, "gpode_rk4_bwd": 1,
    "gpode_param_grad": 1, "gpode_grads_finalize": 1, "gpode_whiten_fwd": 1, "gpode_whiten_bwd": 1,
    "gpode_kl_fwd": 1, "gpode_kl_bwd": 1, "gpode_inducing_sample_fwd": 1, "gpode_inducing_sample_bwd": 1, "gpode_dopri5_fwd": 1, "gpode_dopri5_bwd": 1, "gpode_state_fwd": 1,
    "gpode_state_bwd": 1, "gpode_loglik_sum": 2, "gpode_constraint_sum": 2,
    "gpode_pack_cache_large": 1, "gpode_rbf_fwd_large": 1, "gpode_rff_fwd_large": 1,
    "gpode_vf_fwd_large_add_rbf": 1, "gpode_dopri5_bwd_dev": 1, "gpode_param_grad_dev": 1,
    "gpode_pack_cache_sets": 1, "gpode_whiten_fwd_sets": 2, "gpode_vf_fwd_sets": 1, "gpode_rk4_fwd_sets": 1,
    "gpode_dopri5_fwd_sets": 1, "gpode_shoot_fwd": 2, "gpode_shoot_bwd": 1,
    "gpode_pack_cache_large_bwd": 2, "gpode_vf_bwd_large": 2, "gpode_grads_finalize_large": 2,
    # per RK4 step: forward 4 evaluations x 2 kernels + 4 stage kernels; adjoint 4 VJPs + 8 element-wise kernels
    "gpode_rk4_fwd_large_dev": 12, "gpode_rk4_bwd_large": 16,
    # start: 2 evaluations (2 kernels each) + 6 small kernels; every attempt of the device-side loop launches 21 more
    "gpode_dopri5_fwd_large": 10 + 21, "gpode_dopri5_fwd_large_ckpt": 10 + 21,
    # batched prediction above D = 8: the same counts, all draws in each launch; dopri5 adds the "any draw left" kernel
    "gpode_pack_cache_large_sets": 1, "gpode_vf_fwd_large_sets": 2, "gpode_rk4_fwd_large_sets": 12,
    "gpode_dopri5_fwd_large_sets": 10 + 22,
    # per accepted step: 6 VJPs (2 kernels each) + 7 element-wise kernels; once: the VJP at x0 + the grad_x0 kernel
    "gpode_dopri5_bwd_large": 19 + 3,
    # shooting step above D = 8: one RK4 interval + the epilogue and its ordered sum; seed kernel + adjoint + pull kernel
    "gpode_shoot_fwd_large": 12 + 2, "gpode_shoot_bwd_large": 1 + 16 + 1,
}
assert all(isinstance(v, int) for v in KERNELS_PER_CALL.values()), "KERNELS_PER_CALL holds launch counts"
assert set(KERNELS_PER_CALL) <= set(SIGNATURES), sorted(set(KERNELS_PER_CALL) - set(SIGNATURES))
LAUNCH_COUNT = {}
_PROFILE = None  # None, or {name: [(start_event, end_event), ...]}


def profile_start():
    global _PROFILE
    _PROFILE = {}


def profile_stop(raw=False):
    """-> {name: (calls, total_ms)} (``raw``: {name: [ms of every call, in call order]}); synchronises the device."""
    global _PROFILE
    rec, _PROFILE = _PROFILE, None
    torch.cuda.synchronize()
    if raw:
        return {k: [a.elapsed_time(b) for a, b in v] for k, v in (rec or {}).items()}
    return {k: (len(v), sum(a.elapsed_time(b) for a, b in v)) for k, v in (rec or {}).items()}


def reset_launch_count():
    LAUNCH_COUNT.clear()


def total_launches():
    return sum(LAUNCH_COUNT.values())


def whiten_blocked_launches(M, bwd=False):
    """Kernels enqueued by gpode_whiten_{fwd,fwd_sets,bwd}_blocked at this M (csrc/whiten_blocked.cu): with
    P = ceil(M / 64) panels, the Cholesky and every triangular solve take 2 P - 1 launches; the forward adds four
    element-wise kernels to one Cholesky and two solves, the backward five to four solves."""
    per = 2 * ((M + 63) // 64) - 1
    return 5 + 4 * per if bwd else 4 + 3 * per


def call(name, *args, launches=None):
    """Invoke one C-ABI entry point on the current stream, check its return code, count its kernel launches
    (``launches`` for the entry points whose count depends on the shape)."""
    fn = getattr(load(), name)
    LAUNCH_COUNT[name] = LAUNCH_COUNT.get(name, 0) + (KERNELS_PER_CALL[name] if launches is None else launches)
    if _PROFILE is None:
        check(fn(*args))
        return
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    check(fn(*args))
    e1.record()
    _PROFILE.setdefault(name, []).append((e0, e1))
