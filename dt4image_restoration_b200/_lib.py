"""ctypes binding of ``csrc/libpnp_b200.so`` (C-ABI declared in ``include/pnp_b200.h``).

There is no fallback: if the library is missing or ``pnp_init`` fails (no sm_100a device) every
operator raises.  PyTorch is used only for device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libpnp_b200.so")

_lib = None
_inited = False
_init_device = None          # CUDA device index pnp_init ran on (twiddle tables, kernel attributes are per device)
_lock = threading.Lock()

c_void_p, c_int, c_ll, c_size_t, c_char_p = C.c_void_p, C.c_int, C.c_longlong, C.c_size_t, C.c_char_p

# name -> (restype, argtypes); mirrors include/pnp_b200.h one to one
SIGNATURES = {
    "pnp_init": (c_int, []),
    "pnp_last_error": (c_char_p, []),
    "pnp_num_sms": (c_int, []),
    "pnp_abi_version": (c_int, []),
    "pnp_psnr": (c_int, [c_void_p, c_void_p, c_ll, c_void_p, c_int, c_int, c_void_p]),
    "pnp_psnr_allgather": (c_int, [c_void_p, c_void_p, c_ll, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                   c_void_p, C.c_uint, C.c_uint, c_void_p, c_int, c_int, c_void_p]),
    "pnp_ssim_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "pnp_ssim": (c_int, [c_void_p, c_void_p, c_ll, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "pnp_fft2c": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "pnp_simulate_measurements": (c_int, [c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_int, c_void_p, c_void_p, c_void_p,
                                          c_void_p, c_int, c_int, c_int, c_void_p]),
    "pnp_cartesian_masks": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p]),
    "pnp_radial_masks": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "pnp_variable_density_masks": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int,
                                           c_void_p]),
    "pnp_residual_real": (c_int, [c_void_p, c_void_p, c_void_p, c_ll, c_void_p]),
    "pnp_prox_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "pnp_prox_dual": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_ll, c_void_p, c_int, c_void_p, c_void_p,
                              c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "pnp_prox_prepared_supported": (c_int, [c_int, c_int]),
    "pnp_prox_prepared_bytes": (c_int, [c_int, c_int, c_int, c_void_p, c_void_p]),
    "pnp_prox_prepare": (c_int, [c_void_p, c_void_p, c_ll, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "pnp_prox_dual_prepared": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_ll, c_void_p, c_int, c_void_p, c_void_p,
                                       c_void_p, c_int, c_int, c_int, c_void_p]),
    "pnp_prox_prepared_kind_async": (c_int, [c_void_p, c_ll, c_int, c_int, c_int, c_void_p, c_void_p]),
    "pnp_prox_dual_prepared_kind": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_ll, c_void_p, c_int, c_void_p,
                                            c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "pnp_step_prepared_kind": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_ll, c_void_p, c_int,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "pnp_step_prepared_active": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_ll, c_void_p, c_int,
                                         c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "pnp_step_prepared": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_ll, c_void_p, c_int,
                                  c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "pnp_unet_num_params": (c_size_t, []),
    "pnp_unet_packed_bytes": (c_size_t, []),
    "pnp_unet_pack_weights": (c_int, [c_void_p, c_void_p, c_void_p]),
    "pnp_unet_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "pnp_unet_plan_create": (c_int, [C.POINTER(c_void_p), c_void_p, c_void_p, c_size_t, c_int, c_int, c_int]),
    "pnp_unet_plan_destroy": (None, [c_void_p]),
    "pnp_unet_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "pnp_unet_profile": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, C.POINTER(C.c_float),
                                 C.POINTER(c_int), C.POINTER(c_int), C.POINTER(c_int)]),
    "pnp_unet_num_launches": (c_int, [c_void_p]),
    "pnp_unet_micro_batch": (c_int, [c_void_p]),
    "pnp_unet_set_workspace_cap": (c_size_t, [c_size_t]),
    "pnp_unet_set_splitk": (c_int, [c_int]),
    "pnp_unet_plan_tensor": (c_int, [c_void_p, c_char_p, C.POINTER(c_size_t), C.POINTER(c_int), C.POINTER(c_int),
                                     C.POINTER(c_int)]),
    "pnp_unet_forward_ops": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "pnp_unet_op_describe": (c_int, [c_void_p, c_int, C.POINTER(c_ll)]),
    "pnp_conv3x3_packed_bytes": (c_size_t, [c_int, c_int]),
    "pnp_conv3x3_bf16": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                 c_int, c_int, c_int, c_void_p]),
    "pnp_policy_packed_floats": (c_size_t, [c_int, c_int]),
    "pnp_policy_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                C.c_float, C.c_float, C.c_float, c_int, c_int, c_int, c_int, c_void_p]),
    "pnp_policy_encoder_packed_floats": (c_size_t, []),
    "pnp_policy_observe": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "pnp_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_ll, c_void_p, c_int, c_void_p,
                         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
}


class PnpError(RuntimeError):
    pass


def load() -> C.CDLL:
    """dlopen the library and declare every prototype (no CUDA call is made)."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise PnpError(
                    f"{LIB_PATH} is missing: build it with `python -m dt4image_restoration_b200.build` "
                    "(there is no CPU fallback)")
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def lib() -> C.CDLL:
    """Loaded AND initialised library (needs a B200)."""
    global _inited
    l = load()
    if not _inited:
        with _lock:
            if not _inited:
                rc = l.pnp_init()
                if rc != 0:
                    raise PnpError(f"pnp_init failed ({rc}): {l.pnp_last_error().decode()}")
                global _init_device
                try:
                    import torch
                    _init_device = torch.cuda.current_device()
                except Exception:
                    _init_device = None
                _inited = True
    return l


def check_device(device) -> None:
    """One process drives ONE GPU (one process per GPU, as torchrun launches them): the library's device-side tables and
    kernel attributes are set up by ``pnp_init`` on the device that was current at the first call, and every launch goes to
    the current device's stream.  A tensor on another device, or a changed current device, would silently compute with an
    empty twiddle table or launch on the wrong GPU - so it is an error."""
    import torch
    lib()
    idx = torch.device(device).index
    cur = torch.cuda.current_device()
    if idx is None:
        idx = cur
    if _init_device is not None and (idx != _init_device or cur != _init_device):
        raise PnpError(f"libpnp_b200 was initialised on cuda:{_init_device}; got a tensor on cuda:{idx} with current device "
                       f"cuda:{cur}.  Use one process per GPU and call torch.cuda.set_device(local_rank) before the first "
                       f"operation (there is no multi-device dispatch inside one process)")


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().pnp_last_error().decode()
        raise PnpError(f"{what or 'libpnp_b200'} failed with code {rc}: {msg}")


def stream_ptr() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream
