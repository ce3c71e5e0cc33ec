"""ctypes binding of libmcedm_b200.so (the C ABI declared in include/mcedm_b200.h).

The library is built in-tree by ``mcedm_b200.build``.  There is no fallback: if the shared object is
missing, or a call fails, a RuntimeError is raised with the library's own message.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# MCEDM_LIB: another build of the same library, e.g. the parent commit's, for an A/B comparison
LIB_PATH = os.environ.get("MCEDM_LIB") or os.path.join(_HERE, "lib", "libmcedm_b200.so")

_vp = C.c_void_p
_i = C.c_int
_u = C.c_uint
_f = C.c_float
_d = C.c_double
_ip = C.POINTER(C.c_int)
_vpp = C.POINTER(C.c_void_p)
_llp = C.POINTER(C.c_longlong)

# name -> argtypes; every function returns int (0 = ok) unless listed in _RESTYPES
_PROTOTYPES = {
    "mcedm_abi_version": [],
    "mcedm_check_watchdog": [_vp],
    "mcedm_conv_igemm": [_vpp, _i, _ip, _ip, _ip, _i, _vp, _vp, _i, _i, _i, _i, _vp, _i, _vp, _i, _vp, _i, _vp],
    "mcedm_conv_rows": [_vpp, _i, _vpp, _i, _vp, _vp, _i, _i, _i, _vp, _i, _vp, _i, _vp, _i, _vp],
    "mcedm_gn_coef": [_vp, _i, _vp, _vp, _vp, _i, _i, _f, _i, _i, _i, _vp, _vp, _vp],
    "mcedm_gn_apply16": [_vp, _i, _i, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _i, _vp],
    "mcedm_gn_apply16_dropout": [_vp, _i, _i, _vp, _i, _i, _i, _i, _i, _vp, _u, _f, _i, _vp, _i, _vp],
    "mcedm_dropout_bwd16": [_vp, _i, _i, _i, _i, _i, _u, _f, _i, _vp, _i, _vp],
    "mcedm_conv_rows_fused": [_vpp, _vpp, _i, _vpp, _i, _vp, _vp, _i, _i, _i, _i, _i, _vp, _i, _vp, _i, _i, _i, _vp, _i,
                              _vp],
    "mcedm_conv_head_fused": [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _i, _vp],
    "mcedm_conv_flat_fused": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _i, _vp, _i, _i, _i, _i, _vp, _i, _vp],
    "mcedm_conv_igemm16": [_vpp, _i, _ip, _ip, _ip, _i, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _i, _i, _i, _vp, _i, _vp],
    "mcedm_conv_in_tc16": [_vp, _i, _vp, _i, _vp, _vp, _i, _i, _vp, _vp, _i, _vp],
    "mcedm_conv_in16": [_vp, _i, _vp, _i, _vp, _vp, _i, _i, _i, _vp, _vp, _i, _vp],
    "mcedm_gn_apply_split": [_vp, _vp, _vp, _vp, _vp, _i, _i, _f, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp],
    "mcedm_split16": [_vp, C.c_longlong, _vp, _vp, _vp],
    "mcedm_attention_f32": [_vp, _i, _i, _vp, _vp],
    "mcedm_gn_stats": [_vp, C.c_longlong, _vp, _vp],
    "mcedm_gn_apply": [_vp, _vp, _vp, _vp, _vp, _i, _i, _f, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _vp],
    "mcedm_gn_bwd_ctas_per_img": [_i, _i, _i],
    "mcedm_gn_bwd": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _f, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _vp, _i, _vp,
                     _vp, _vp, _i, _i, _vp, _vp, _vp],
    "mcedm_gn_bwd16_ctas_per_img": [_i, _i, _i],
    "mcedm_gn_bwd16": [_vp, _i, _i, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp,
                       _vp, _i, _vp, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp],
    "mcedm_reduce_rows": [_vp, _i, C.c_longlong, _i, C.c_longlong, _vp, _i, _f, _vp],
    "mcedm_reduce_rows_batched": [_vp, _i, _i, _vp],
    "mcedm_wgrad_reduce_batched": [_vp, _i, _vp],
    "mcedm_edm_loss": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, C.c_longlong, _vp, _vp, C.c_longlong, _vp, _i, _vp],
    "mcedm_edm_noise_in": [_vp, _vp, _vp, _vp, _vp, _i, C.c_longlong, _vp, _vp, _vp],
    "mcedm_mcedm_prep": [_vp, _vp, _vp, _vp, _f, _f, _f, _f, _i, C.c_longlong, _vp, _vp, _vp, _vp],
    "mcedm_mcedm_prep_rows": [_vp, _vp, _vp, _vp, _f, _f, _f, _f, _i, _i, _i, _vp, _vp, _vp, _vp, _vp],
    "mcedm_nchw_to_nhwc_pad": [_vp, _i, _vp, _i, _i, _i, _i, _vp, _i, _vp],
    "mcedm_colsum_bf16": [_vp, C.c_longlong, _i, _i, _vp, _i, _vp],
    "mcedm_nchw_to_nhwc_pad16": [_vp, _i, _vp, _i, _i, _i, _i, _vp, _i, _f, _i, _vp],
    "mcedm_colsum16": [_vp, C.c_longlong, _i, _i, _vp, _i, _i, _vp],
    "mcedm_emb_mlp_bwd": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "mcedm_sumsq_partial": [_vp, C.c_longlong, _vp, _i, _vp],
    "mcedm_adam_step": [_vp, _vp, _vp, _vp, C.c_longlong, _f, _f, _f, _f, _f, _i, _vp, _i, _f, _f, _vp, _vp],
    "mcedm_ema_update": [_vp, _vp, C.c_longlong, _f, _vp],
    "mcedm_grad_accumulate": [_vp, _vp, C.c_longlong, _f, _i, _vp],
    "mcedm_nchw_to_nhwc_pad16_scaled": [_vp, _i, _vp, _i, _i, _i, _i, _vp, _i, _vp, _i, _vp],
    "mcedm_grad_unscale": [_vp, C.c_longlong, _vp, _vp],
    "mcedm_adam_step_dyn": [_vp, _vp, _vp, _vp, C.c_longlong, _f, _f, _f, _f, _f, _vp, _vp, _i, _f, _f, _vp, _vp, _vp],
    "mcedm_loss_scale_update": [_vp, _vp, _vp, _vp, _f, _f, _i, _vp],
    "mcedm_pack_gather": [_vp, _vp, _vp, C.c_longlong, C.c_longlong, _i, _vp, _vp, _vp],
    "mcedm_wgrad_ctas": [_i, _i, _i],
    "mcedm_conv_wgrad": [_vp, _i, _i, _i, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp],
    "mcedm_conv_wgrad16": [_vp, _i, _i, _i, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _i, _vp],
    "mcedm_conv_wgrad16_fused": [_vp, _i, _i, _i, _vp, _i, _i, _i, _vp, _i, _i, _i, _i, _i, _vp, _i, _vp],
    "mcedm_wgrad_reduce": [_vp, _i, _i, _vp, _i, _i, _i, _i, _i, _i, _i, _vp],
    "mcedm_flat_geometry": [_i, _i, _ip, _ip],
    "mcedm_conv_flat": [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _i, _vp, _i, _vp],
    "mcedm_attention": [_vp, _i, _i, _vp, _vp, _i, _vp],
    "mcedm_attention_bwd": [_vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp],
    "mcedm_attention_bwd16": [_vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _i, _vp],
    "mcedm_emb_mlp": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp],
    "mcedm_conv_in": [_vp, _i, _vp, _i, _vp, _vp, _i, _i, _i, _vp, _vp, _vp],
    "mcedm_head_to_nchw": [_vp, _i, _i, _i, _i, _i, _vp, _vp],
    "mcedm_edm_init": [_vp, _vp, _i, _vp, _d, _i, _i, _i, _i, _vp, _vp],
    "mcedm_edm_churn": [_vp, _vp, _vp, _d, _f, C.c_longlong, _vp, _vp, _vp],
    "mcedm_edm_euler": [_vp, _vp, _vp, _d, _d, _f, _f, _f, C.c_longlong, _vp, _vp, _vp, _vp, _vp],
    "mcedm_edm_correct": [_vp, _vp, _vp, _vp, _vp, _d, _d, _f, _f, C.c_longlong, _vp, _vp, _vp],
    "mcedm_edm_precond_in": [_vp, _vp, _i, _i, C.c_longlong, _vp, _vp],
    "mcedm_edm_precond_out": [_vp, _vp, _vp, _vp, _i, _i, C.c_longlong, _vp, _vp],
    "mcedm_edm_denoised": [_vp, _vp, _f, _f, C.c_longlong, _vp, _vp],
    "mcedm_edm_euler_guided": [_vp, _vp, _vp, _vp, _d, _d, _f, C.c_longlong, _vp, _vp, _vp, _vp],
    "mcedm_edm_correct_guided": [_vp, _vp, _vp, _vp, _vp, _vp, _d, _d, C.c_longlong, _vp, _vp],
    "mcedm_edm_churn_cfg": [_vp, _vp, _vp, _d, _f, C.c_longlong, _vp, _vp, _vp],
    "mcedm_edm_euler_cfg": [_vp, _vp, _vp, _d, _d, _f, _f, _f, _d, C.c_longlong, _vp, _vp, _vp, _vp, _vp],
    "mcedm_edm_correct_cfg": [_vp, _vp, _vp, _vp, _vp, _d, _d, _f, _f, _d, C.c_longlong, _vp, _vp, _vp],
    "mcedm_edm_denoised_cfg": [_vp, _vp, _f, _f, _d, C.c_longlong, _vp, _vp],
    "mcedm_edm_precond_out_cfg": [_vp, _vp, _vp, _vp, _i, _d, _i, C.c_longlong, _vp, _vp, _vp],
    "mcedm_edm_vp_init": [_vp, _vp, _vp, _f, _f, _d, C.c_longlong, _vp, _vp],
    "mcedm_edm_repaint_blend": [_vp, _vp, _vp, _f, _f, C.c_longlong, _vp, _vp],
    "mcedm_ddim_init": [_vp, _vp, _vp, _f, _f, C.c_longlong, _vp, _vp],
    "mcedm_ddim_x0": [_vp, _vp, _vp, _vp, _f, _f, C.c_longlong, _vp, _vp, _vp],
    "mcedm_ddim_next": [_vp, _vp, _vp, _vp, _vp, _vp, _f, _f, _f, C.c_longlong, _vp, _vp],
    "mcedm_swe_fv_loss": [_vp, _i, _llp, _vp, _i, _llp, _i, _f, _f, _f, _f, _vp, _i, _i, _i, _f, _f, _f, _vp, _vp, _vp,
                          _vp],
    "mcedm_swe_fv_grad": [_vp, _i, _llp, _vp, _i, _llp, _i, _f, _f, _f, _f, _vp, _i, _i, _i, _f, _f, _f, _i, _vp, _vp],
    "mcedm_darcy_loss": [_vp, _i, _llp, _vp, _i, _llp, _i, _f, _f, _f, _f, _i, _i, _f, _vp, _vp, _vp, _vp],
    "mcedm_gn_stats16": [_vp, C.c_longlong, _i, _i, _i, _vp, _vp],
    "mcedm_gn_coef_groups": [_vp, _i, C.c_longlong, _vp, _vp, _i, _f, _vp, _i, _i, _vp, _vp],
    "mcedm_decimate16": [_vp, _i, _i, _i, _i, _i, _vp, _i, _i, _vp],
    "mcedm_ddpm_temb": [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp],
    "mcedm_masked_mae_mean": [_vp, _i, _i, C.c_longlong, _i, _vp, _vp, _vp, _i, _vp, _i, _i, _vp, _vp, _i, _vp, _vp, _i,
                              _vp, _vp],
    "mcedm_corr_minmax": [_vp, _vp, _i, C.c_longlong, _i, _vp, _vp, _vp, _vp],
    "mcedm_saturation_count": [_llp, _i, _vp],
    "mcedm_debug_rows": [_vp],
}
_RESTYPES = {"mcedm_last_error": C.c_char_p}
# checker / probe kernels: libmcedm_b200_check.so (include/mcedm_b200_check.h), loaded by tests and scripts only
_CHECK_PROTOTYPES = {
    "mcedm_probe_mma_rate": [_i, _i, _vp, _vp],
    "mcedm_probe_mma_queue": [_i, _i, _i, _vp, _vp],
    "mcedm_probe_umma": [_vp, _i, _vp, _i, _i, _i, _vp, _vp],
    "mcedm_conv_direct_ref": [_vpp, _i, _vp, _i, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _i, _vp],
    "mcedm_attention_ref": [_vp, _i, _i, _vp, _vp],
}
CHECK_LIB_PATH = os.path.join(_HERE, "lib", "libmcedm_b200_check.so")

_lib = None
# number of kernel launches issued through the C ABI by this process (every successful call below launches
# exactly one kernel; graph replays are added by the engine); bench.py reports it as gpu_launches
LAUNCHES = [0]
# op_fmt of fp16 stores without saturation (include/mcedm_b200.h MCEDM_FMT_F16_INF): dynamic loss scaling's gradients
FMT_F16_INF = 3


class McedmError(RuntimeError):
    pass


def exported_names():
    """Every symbol include/mcedm_b200.h declares (used by the CPU-side ABI test)."""
    return sorted(list(_PROTOTYPES) + list(_RESTYPES))


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise McedmError(
                f"{LIB_PATH} is missing: build it with `python -m mcedm_b200.build` "
                "(there is no CPU or PyTorch fallback for the sm_100a kernels)")
        l = C.CDLL(LIB_PATH)
        for name, args in _PROTOTYPES.items():
            fn = getattr(l, name)
            fn.argtypes = args
            fn.restype = C.c_int
        for name, res in _RESTYPES.items():
            fn = getattr(l, name)
            fn.argtypes = []
            fn.restype = res
        if l.mcedm_abi_version() != 1:
            raise McedmError("libmcedm_b200.so ABI version mismatch; rebuild with `python -m mcedm_b200.build`")
        _lib = l
    return _lib


_check_lib = None


def check_exported_names():
    """Every symbol include/mcedm_b200_check.h declares."""
    return sorted(_CHECK_PROTOTYPES)


def check_lib():
    """The checker / probe library (test infrastructure): not needed, and never loaded, by the product path."""
    global _check_lib
    if _check_lib is None:
        if not os.path.exists(CHECK_LIB_PATH):
            raise McedmError(f"{CHECK_LIB_PATH} is missing: build it with `python -m mcedm_b200.build`")
        l = C.CDLL(CHECK_LIB_PATH)
        for name, args in _CHECK_PROTOTYPES.items():
            fn = getattr(l, name)
            fn.argtypes = args
            fn.restype = C.c_int
        l.mcedm_last_error.argtypes = []
        l.mcedm_last_error.restype = C.c_char_p
        _check_lib = l
    return _check_lib


def check(rc: int, what: str = "", lib_=None):
    LAUNCHES[0] += 1
    if rc != 0:
        msg = (lib_ or lib()).mcedm_last_error()
        raise McedmError(f"{what or 'mcedm call'} failed (rc={rc}): {msg.decode() if msg else '?'}")


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def int_array(vals):
    return (C.c_int * len(vals))(*[int(v) for v in vals])


def ll_array(vals):
    return (C.c_longlong * len(vals))(*[int(v) for v in vals])


def ptr_array(tensors):
    return (C.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def check_watchdog():
    check(lib().mcedm_check_watchdog(stream_ptr()), "watchdog")
    LAUNCHES[0] -= 1
