"""ctypes binding of libipdm_b200.so (the C ABI declared in include/ipdm_b200.h).

Fails loudly when the shared object is missing or does not export a declared symbol: the
product path never falls back to PyTorch or CPU code.
"""
import ctypes
import os
import re
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libipdm_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "ipdm_b200.h")

c_float_p = ctypes.POINTER(ctypes.c_float)
c_double_p = ctypes.POINTER(ctypes.c_double)
vp = ctypes.c_void_p


class UNetConfig(ctypes.Structure):
    _fields_ = [("in_channels", ctypes.c_int), ("model_channels", ctypes.c_int), ("out_channels", ctypes.c_int),
                ("num_res_blocks", ctypes.c_int), ("num_heads", ctypes.c_int), ("n_mult", ctypes.c_int),
                ("channel_mult", ctypes.c_double * 8), ("n_attn", ctypes.c_int),
                ("attention_resolutions", ctypes.c_int * 8), ("precision", ctypes.c_int), ("max_t", ctypes.c_int)]


class GuidedParams(ctypes.Structure):
    _fields_ = [("mode", ctypes.c_int), ("n_iters", ctypes.c_int), ("t_start", ctypes.c_int * 8), ("clip", ctypes.c_int),
                ("lambda_ratio", ctypes.c_double), ("eta", ctypes.c_double), ("constant_guidance_set", ctypes.c_int),
                ("constant_guidance", ctypes.c_double), ("kernel_size", ctypes.c_int), ("amplitude", ctypes.c_double),
                ("curve_kind", ctypes.c_int), ("timesteps", ctypes.c_int), ("schedule_power", ctypes.c_double),
                ("seed", ctypes.c_uint64)]


_SIGNATURES = {
    "ipdm_last_error": (ctypes.c_char_p, []),
    "ipdm_abi_version": (ctypes.c_int, []),
    "ipdm_launch_count": (ctypes.c_ulonglong, []),
    "ipdm_launch_count_reset": (None, []),
    "ipdm_profile_enable": (None, [ctypes.c_int]),
    "ipdm_profile_collect": (ctypes.c_int, [c_double_p, c_double_p, ctypes.POINTER(ctypes.c_longlong)]),
    "ipdm_debug_fold_pack": (ctypes.c_int, [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp, ctypes.POINTER(ctypes.c_int),
                                            ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]),
    "ipdm_debug_phase_pack": (ctypes.c_int, [vp, ctypes.c_int, ctypes.c_int, vp, ctypes.POINTER(ctypes.c_int)]),
    "ipdm_profile_roofline": (ctypes.c_int, [ctypes.c_int, ctypes.c_double, ctypes.c_double, c_double_p, c_double_p, c_double_p]),
    "ipdm_fbp_plan_create": (ctypes.c_int, [ctypes.POINTER(vp), ctypes.c_int]),
    "ipdm_fbp_plan_destroy": (ctypes.c_int, [vp]),
    "ipdm_fbp_filter": (ctypes.c_int, [vp, vp, vp, ctypes.c_int, ctypes.c_int, vp]),
    "ipdm_fbp_backproject": (ctypes.c_int, [vp, vp, vp, ctypes.c_int, ctypes.c_int, vp]),
    "ipdm_fbp_forward": (ctypes.c_int, [vp, vp, vp, ctypes.c_int, ctypes.c_int, vp]),
    "ipdm_fbp_convert_host": (ctypes.c_int, [vp, vp, vp, ctypes.c_int, ctypes.c_int]),
    "ipdm_fbp_tables": (ctypes.c_int, [vp, vp, vp, vp, vp]),
    "ipdm_fbp_project": (ctypes.c_int, [vp, vp, vp, ctypes.c_int, ctypes.c_int, vp]),
    "ipdm_fbp_project_adjoint": (ctypes.c_int, [vp, vp, vp, ctypes.c_int, ctypes.c_int, vp]),
    "ipdm_fbp_sart_tv": (ctypes.c_int, [vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_int,
                                        ctypes.c_float, ctypes.c_float, ctypes.c_int, vp]),
    "ipdm_fbp_tv_descent": (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_float, vp]),
    "ipdm_fbp_pwls": (ctypes.c_int, [vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_float,
                                     ctypes.c_float, ctypes.c_int, vp]),
    "ipdm_fbp_pwls_penalty": (ctypes.c_int, [vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_float, vp]),
    "ipdm_low_dose_noise": (ctypes.c_int, [vp, vp, vp, ctypes.c_int, ctypes.c_size_t, ctypes.c_float, ctypes.c_int, ctypes.c_uint64, vp,
                                           vp]),
    "ipdm_cosine_beta_schedule": (ctypes.c_int, [ctypes.c_int, ctypes.c_double, c_double_p]),
    "ipdm_schedule_at": (ctypes.c_int, [ctypes.c_int, ctypes.c_double, ctypes.c_int, c_double_p]),
    "ipdm_lincomb": (ctypes.c_int, [vp, ctypes.c_float, vp, ctypes.c_float, vp, ctypes.c_float, vp, ctypes.c_size_t, vp]),
    "ipdm_clamp": (ctypes.c_int, [vp, ctypes.c_float, ctypes.c_float, ctypes.c_size_t, vp]),
    "ipdm_sampler_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "ipdm_sampler_step": (ctypes.c_int, [vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_float_p, ctypes.c_float,
                                         vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_uint64, ctypes.c_uint64, vp, vp]),
    "ipdm_sampler_step_ddim": (ctypes.c_int, [vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_float_p, ctypes.c_float,
                                              ctypes.c_int, ctypes.c_int, ctypes.c_uint64, ctypes.c_uint64, vp, vp]),
    "ipdm_set_noise_epoch": (ctypes.c_int, [ctypes.c_uint64, vp]),
    "ipdm_q_sample": (ctypes.c_int, [vp, vp, vp, ctypes.c_float, ctypes.c_float, ctypes.c_size_t, ctypes.c_int, ctypes.c_uint64,
                                     ctypes.c_uint64, vp]),
    "ipdm_delta_lambda_map": (ctypes.c_int, [vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float,
                                             ctypes.c_int, vp, vp]),
    "ipdm_delta_lambda_map_img": (ctypes.c_int, [vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float,
                                                 ctypes.c_int, vp, vp]),
    "ipdm_delta_exp_max": (ctypes.c_int, [vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float, vp, vp]),
    "ipdm_lambda_step_map": (ctypes.c_int, [vp, vp, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, vp]),
    "ipdm_lambda_curve_host": (ctypes.c_int, [vp, vp, ctypes.c_size_t, ctypes.c_int]),
    "ipdm_sharpen3x3": (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp]),
    "ipdm_unet_create": (ctypes.c_int, [ctypes.POINTER(vp), ctypes.POINTER(UNetConfig), vp, ctypes.c_size_t]),
    "ipdm_unet_destroy": (ctypes.c_int, [vp]),
    "ipdm_unet_param_count": (ctypes.c_longlong, [ctypes.POINTER(UNetConfig)]),
    "ipdm_unet_forward": (ctypes.c_int, [vp, vp, ctypes.c_int, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp]),
    "ipdm_unet_flops": (ctypes.c_double, [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "ipdm_guided_noise_count": (ctypes.c_int, [ctypes.POINTER(GuidedParams)]),
    "ipdm_guided_workspace_bytes": (ctypes.c_size_t, [ctypes.POINTER(GuidedParams), ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "ipdm_guided_process": (ctypes.c_int, [vp, ctypes.POINTER(GuidedParams), vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                           vp, vp]),
    "ipdm_guided_process_resume": (ctypes.c_int, [vp, ctypes.POINTER(GuidedParams), vp, vp, vp, vp, ctypes.c_uint64, vp, ctypes.c_int,
                                                  ctypes.c_int, ctypes.c_int, vp, vp]),
    "ipdm_debug_conv": (ctypes.c_int, [vp, ctypes.c_int, ctypes.c_int, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                       vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp, vp, ctypes.c_int,
                                       vp, ctypes.c_int, ctypes.c_int, vp]),
    "ipdm_debug_conv_time": (ctypes.c_int, [ctypes.c_int] * 12 + [c_float_p, c_double_p]),
    "ipdm_debug_groupnorm": (ctypes.c_int, [vp, ctypes.c_int, ctypes.c_int, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                            ctypes.c_int, vp, vp, ctypes.c_int, vp, vp, vp, ctypes.c_int, vp]),
    "ipdm_debug_attention": (ctypes.c_int, [vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp]),
    "ipdm_metrics_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "ipdm_psnr_ssim": (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp, vp]),
    "ipdm_miu2pixel": (ctypes.c_int, [vp, vp, ctypes.c_size_t, ctypes.c_float, ctypes.c_float, vp]),
    "ipdm_debug_attention_bf16": (ctypes.c_int, [vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp]),
    "ipdm_debug_upsample": (ctypes.c_int, [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, ctypes.c_int, ctypes.c_int, vp]),
}


def declared_symbols():
    """Every `ipdm_*` function name declared in include/ipdm_b200.h."""
    with open(HEADER_PATH) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    return sorted(set(re.findall(r"\b(ipdm_[a-z0-9_]+)\s*\(", text)))


def build(verbose=False):
    """Compile csrc/*.cu for sm_100a into libipdm_b200.so (nvcc cross-compiles without a GPU)."""
    out = subprocess.run(["bash", os.path.join(_HERE, "csrc", "build.sh")], capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError("building libipdm_b200.so failed:\n" + out.stdout[-4000:] + out.stderr[-4000:])
    if verbose:
        print(out.stdout[-2000:])
    return SO_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise RuntimeError(f"{SO_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(there is no CPU or PyTorch fallback for the IPDM hot path)")
        handle = ctypes.CDLL(SO_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)          # AttributeError if the .so does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().ipdm_last_error()
        raise RuntimeError(f"{what} failed with code {rc}: {msg.decode() if msg else ''}")
