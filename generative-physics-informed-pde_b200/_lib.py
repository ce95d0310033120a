"""ctypes binding of libgpde_b200.so (C ABI declared in include/gpde_b200.h).

There is NO fallback: if the shared library is missing or a symbol cannot be resolved the import of
the hot-path modules fails loudly (``GpdeLibraryError``).  torch is used only for device memory,
streams and autograd plumbing; every number on the hot path is produced by the kernels in csrc/.
"""
import ctypes
import os

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libgpde_b200.so")

c_i32, c_i64, c_sz, c_vp, c_f64 = ctypes.c_int, ctypes.c_int64, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_double
PP = ctypes.POINTER(ctypes.c_void_p)


class GpdeLibraryError(RuntimeError):
    pass


# name -> (restype, argtypes); must list every symbol of include/gpde_b200.h (tests check this)
SIGNATURES = {
    "gpde_version": (c_i32, []),
    "gpde_last_error": (ctypes.c_char_p, []),
    "gpde_rom_plan_create": (c_i32, [PP, c_i32, c_i32, c_vp, c_vp, c_i32, c_i32]),
    "gpde_rom_plan_destroy": (c_i32, [c_vp]),
    "gpde_rom_plan_info": (c_i32, [c_vp, c_vp]),
    "gpde_rom_factor_bytes": (c_sz, [c_vp, c_i64]),
    "gpde_rom_forward_f64": (c_i32, [c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gpde_rom_forward_f32": (c_i32, [c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gpde_rom_adjoint_f64": (c_i32, [c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gpde_rom_adjoint_f32": (c_i32, [c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gpde_rom_stiffness_f64": (c_i32, [c_vp, c_vp, c_vp, c_i32, c_i64, c_vp]),
    "gpde_prolong_plan_create": (c_i32, [PP, c_i32, c_i32, c_vp, c_i32]),
    "gpde_prolong_plan_destroy": (c_i32, [c_vp]),
    "gpde_prolong_apply_f64": (c_i32, [c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gpde_prolong_apply_T_f64": (c_i32, [c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gpde_prolong_apply_f32": (c_i32, [c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gpde_prolong_apply_T_f32": (c_i32, [c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gpde_prolong_loglik_f64": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gpde_prolong_loglik_f32": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gpde_prolong_moments_f64": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i32, c_vp]),
    "gpde_prolong_moments_f32": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i32, c_vp]),
    "gpde_vo_plan_create": (c_i32, [PP, c_i32, c_i32, c_vp, c_vp, c_vp, c_i32, c_vp, c_i32, c_vp, c_i32,
                                    c_vp, c_i32]),
    "gpde_vo_plan_destroy": (c_i32, [c_vp]),
    "gpde_vo_plan_info": (c_i32, [c_vp, c_vp]),
    "gpde_vo_plan_kernel_path": (c_i32, [c_vp, c_i32, c_i32]),
    "gpde_vo_workspace_bytes": (c_sz, [c_vp, c_i64, c_i32]),
    "gpde_vo_residual_f64": (c_i32, [c_vp, c_vp, c_i64, c_i32, c_vp, c_vp, c_i64, c_vp, c_i64, c_i32, c_vp, c_vp,
                                     c_vp, c_i32, c_i64, c_vp]),
    "gpde_vo_residual_f32": (c_i32, [c_vp, c_vp, c_i64, c_i32, c_vp, c_vp, c_i64, c_vp, c_i64, c_i32, c_vp, c_vp,
                                     c_vp, c_i32, c_i64, c_vp]),
    "gpde_vo_pack_weights_f64": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_vp, c_vp]),
    "gpde_vo_pack_weights_f32": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_vp, c_vp]),
    "gpde_vo_posterior_f64": (c_i32, [c_vp, c_vp, c_i64, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gpde_vo_posterior_blocked_workspace_bytes": (c_sz, [c_vp, c_i64, c_i32]),
    "gpde_vo_posterior_blocked_f64": (c_i32, [c_vp, c_vp, c_i64, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                              c_vp, c_vp, c_sz, c_i64, c_vp]),
    "gpde_vo_moments_f64": (c_i32, [c_vp, c_vp, c_i64, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gpde_vo_energy_step_f64": (c_i32, [c_vp, c_vp, c_i64, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64,
                                        c_vp]),
    "gpde_vo_energy_step_blocked_f64": (c_i32, [c_vp, c_vp, c_i64, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                                c_vp, c_sz, c_i64, c_vp]),
    "gpde_vo_residual_T_f64": (c_i32, [c_vp, c_vp, c_i64, c_i32, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gpde_vo_residual_T_f32": (c_i32, [c_vp, c_vp, c_i64, c_i32, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gpde_vo_residual_grad_f64": (c_i32, [c_vp, c_vp, c_i64, c_i32, c_vp, c_vp, c_i64, c_vp, c_i64, c_i32, c_vp, c_vp,
                                          c_vp, c_vp, c_i64, c_vp]),
    "gpde_vo_residual_grad_f32": (c_i32, [c_vp, c_vp, c_i64, c_i32, c_vp, c_vp, c_i64, c_vp, c_i64, c_i32, c_vp, c_vp,
                                          c_vp, c_vp, c_i64, c_vp]),
    "gpde_cg_init_f64": (c_i32, [c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_f64, c_i32, c_i64, c_i32, c_vp]),
    "gpde_cg_step_f64": (c_i32, [c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_i64, c_i32, c_vp]),
}

_lib = None


def load():
    """Loads the shared library once and declares every signature.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GpdeLibraryError(
            "%s not found: build it with `python generative-physics-informed-pde_b200/build.py` "
            "(or __graft_entry__.build()).  There is no CPU/PyTorch fallback for the hot path." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            raise GpdeLibraryError("symbol %s missing from %s (stale build?)" % (name, LIB_PATH))
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().gpde_last_error()
        raise GpdeLibraryError("%s failed (%d): %s" % (what, rc, msg.decode() if msg else "?"))


def ptr(t, device=None):
    """Device/host pointer of a contiguous tensor (or NULL).  With ``device`` the tensor must live on that CUDA
    device: a CPU tensor or a tensor of another GPU would make the kernel dereference a foreign pointer (sticky
    illegal-address fault); the reference raises a clean torch device-mismatch error in that situation, so do we."""
    if t is None:
        return None
    if device is not None:
        if not t.is_cuda or t.device != device:
            raise RuntimeError("Expected all tensors to be on the same device, but found a tensor on %s "
                               "(the physics-layer plan lives on %s)" % (t.device, device))
    assert t.is_contiguous(), "non-contiguous tensor passed to the C ABI"
    return ctypes.c_void_p(t.data_ptr())


def stream_of(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(device, what):
    device = torch.device(device)
    if device.type != "cuda":
        raise GpdeLibraryError(
            "%s runs only on a CUDA device (sm_100a kernels, no CPU fallback); got device %r" % (what, device))
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    return device


def suffix(dtype):
    if dtype == torch.float64:
        return "f64"
    if dtype == torch.float32:
        return "f32"
    raise TypeError("the physics layer supports float64 and float32, got %r" % (dtype,))
