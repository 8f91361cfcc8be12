"""Tensor-level wrappers over the C ABI (include/ipdm_b200.h).

PyTorch is plumbing here: it owns device memory and the CUDA stream; every arithmetic step of the
hot path runs in libipdm_b200.so.  All functions validate device / dtype / contiguity in Python
and enqueue on `torch.cuda.current_stream()`; none of them synchronises with the host.
"""
import ctypes
import math

import numpy as np
import torch

from . import _lib
from ._lib import GuidedParams, UNetConfig, check

N_VIEWS, N_DET, N_PIX = 2000, 912, 512
SART_DEFAULTS = dict(iterations=5, subsets=100, relaxation=1.0)     # the sart_* options of Config/default_config.py
# the TV options of SART-TV (ntv, tv_alpha, tv_eps, sart_init of Config/default_config.py); ntv = 0 with the zero start is plain SART
SART_TV_DEFAULTS = dict(ntv=0, tv_alpha=0.2, tv_eps=1e-4, init="zero")
SART_INITS = ("zero", "fbp")
# the pwls_* options of convertor="PWLS" (pwls_beta, pwls_delta in 1/cm of Config/default_config.py; DESIGN 8 has the study)
PWLS_DEFAULTS = dict(beta=1e6, delta=0.0002)
PWLS_DOSE = 0.25             # the dose `FBPPlan.pwls` weights the rays for when none is given (the default of the dose option)
PRECISIONS = {"tf32": 0, "bf16": 1, "fp32": 2}


def _require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("the IPDM B200 path needs a CUDA device (sm_100a); there is no CPU fallback")


def _dev(t, name="tensor"):
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
        raise ValueError(f"{name} must be a contiguous float32 CUDA tensor")
    return ctypes.c_void_p(t.data_ptr())


def _opt(t, name="tensor"):
    return None if t is None else _dev(t, name)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _real(v, name, rule, ok):
    """float(v); ValueError "<name> must be <rule>" unless v is a finite real number (a bool or a str is not) with ok(v)."""
    if isinstance(v, bool) or not isinstance(v, (int, float, np.integer, np.floating)) or not (math.isfinite(v) and ok(v)):
        raise ValueError(f"{name} must be {rule}, got {v!r}")
    return float(v)


def _sweeps(who, iterations, subsets, init):
    """(int, int, str): the sweeps, subsets and start every iterative convertor takes; ValueError unless iterations >= 1, subsets
    divides 2000 and init is "zero" or "fbp"."""
    if isinstance(iterations, bool) or int(iterations) != iterations or iterations < 1:
        raise ValueError(f"{who} iterations must be an integer >= 1, got {iterations!r}")
    if isinstance(subsets, bool) or int(subsets) != subsets or not 1 <= subsets <= N_VIEWS or N_VIEWS % int(subsets):
        raise ValueError(f"{who} subsets must be an integer dividing {N_VIEWS}, got {subsets!r}")
    if init not in SART_INITS:
        raise ValueError(f"{who} init must be one of {SART_INITS}, got {init!r}")
    return int(iterations), int(subsets), str(init)


def launch_count():
    return int(_lib.lib().ipdm_launch_count())


def launch_count_reset():
    _lib.lib().ipdm_launch_count_reset()


PROF_FAMILIES = ("conv_tc", "attention", "conv_direct", "groupnorm", "upsample", "fbp_filter", "fbp_backproject", "sampler",
                 "conv_halo_persistent")


def profile_enable(on=True):
    _lib.lib().ipdm_profile_enable(int(bool(on)))


def profile_collect():
    """{family: (milliseconds, work, launches)}; work is FLOPs for conv_tc / conv_halo_persistent / attention, bytes otherwise."""
    k = len(PROF_FAMILIES)
    ms, work, n = (ctypes.c_double * k)(), (ctypes.c_double * k)(), (ctypes.c_longlong * k)()
    check(_lib.lib().ipdm_profile_collect(ms, work, n), "ipdm_profile_collect")
    return {f: (ms[i], work[i], int(n[i])) for i, f in enumerate(PROF_FAMILIES)}


def profile_roofline(family, peak_tflops, peak_gbs):
    """(roof_ms, ms, bytes) of one FLOP-counted family: the time its launches would take with each one at its own roof
    (max of FLOPs / tensor peak and algorithmic bytes / HBM peak), their measured time, and their algorithmic bytes."""
    roof, ms, by = ctypes.c_double(), ctypes.c_double(), ctypes.c_double()
    check(_lib.lib().ipdm_profile_roofline(PROF_FAMILIES.index(family), ctypes.c_double(peak_tflops * 1e12), ctypes.c_double(peak_gbs * 1e9),
                                           ctypes.byref(roof), ctypes.byref(ms), ctypes.byref(by)), "ipdm_profile_roofline")
    return roof.value, ms.value, by.value


# ---------------------------------------------------------------------------------------------
# FBP convertor
# ---------------------------------------------------------------------------------------------
class FBPPlan:
    """Device-side plan of the fan-beam FBP (reference: Recon/FBP_kernel.py FBP)."""

    def __init__(self, max_batch=0):
        _require_cuda()
        self._h = ctypes.c_void_p()
        check(_lib.lib().ipdm_fbp_plan_create(ctypes.byref(self._h), int(max_batch)), "ipdm_fbp_plan_create")

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None and getattr(_lib, "_lib", None) is not None:
            _lib._lib.ipdm_fbp_plan_destroy(self._h)
            self._h = None

    @staticmethod
    def _check_sino(s):
        if s.dim() != 3 or tuple(s.shape[1:]) != (N_VIEWS, N_DET):
            raise ValueError(f"sinogram must be [B,{N_VIEWS},{N_DET}], got {tuple(s.shape)}")

    def forward(self, sino, flip=True, out=None):
        """[B,2000,912] device -> [B,512,512] device."""
        self._check_sino(sino)
        b = sino.shape[0]
        out = torch.empty(b, N_PIX, N_PIX, device=sino.device, dtype=torch.float32) if out is None else out
        check(_lib.lib().ipdm_fbp_forward(self._h, _dev(sino, "sino"), _dev(out, "out"), b, int(bool(flip)), _stream()), "ipdm_fbp_forward")
        return out

    def filter(self, sino, flip=True):
        self._check_sino(sino)
        q = torch.empty_like(sino)
        check(_lib.lib().ipdm_fbp_filter(self._h, _dev(sino), _dev(q), sino.shape[0], int(bool(flip)), _stream()), "ipdm_fbp_filter")
        return q

    def backproject(self, q, flip=True):
        self._check_sino(q)
        out = torch.empty(q.shape[0], N_PIX, N_PIX, device=q.device, dtype=torch.float32)
        check(_lib.lib().ipdm_fbp_backproject(self._h, _dev(q), _dev(out), q.shape[0], int(bool(flip)), _stream()), "ipdm_fbp_backproject")
        return out

    def convert_host(self, pj, flip=True):
        """`FBP.convert` semantics: host ndarray in, host ndarray out (copies inside the call)."""
        pj = np.ascontiguousarray(pj, dtype=np.float32)
        if pj.ndim == 2:
            pj = pj[None]
        if pj.shape[1:] != (N_VIEWS, N_DET):
            raise ValueError(f"sinogram must be [B,{N_VIEWS},{N_DET}], got {pj.shape}")
        out = np.empty((pj.shape[0], N_PIX, N_PIX), dtype=np.float32)
        check(_lib.lib().ipdm_fbp_convert_host(self._h, pj.ctypes.data_as(ctypes.c_void_p), out.ctypes.data_as(ctypes.c_void_p),
                                               pj.shape[0], int(bool(flip))), "ipdm_fbp_convert_host")
        return out

    def project(self, img, flip=True, out=None):
        """Forward projection (Joseph's method, the geometry of `forward`): mu image [B,512,512] device (1/cm) -> line integrals
        [B,2000,912] device.  flip as for `forward`, so forward(project(x, flip), flip) approximates x."""
        if img.dim() != 3 or tuple(img.shape[1:]) != (N_PIX, N_PIX):
            raise ValueError(f"image must be [B,{N_PIX},{N_PIX}], got {tuple(img.shape)}")
        b = img.shape[0]
        out = torch.empty(b, N_VIEWS, N_DET, device=img.device, dtype=torch.float32) if out is None else out
        if tuple(out.shape) != (b, N_VIEWS, N_DET):
            raise ValueError(f"out must be [{b},{N_VIEWS},{N_DET}], got {tuple(out.shape)}")
        check(_lib.lib().ipdm_fbp_project(self._h, _dev(img, "img"), _dev(out, "out"), b, int(bool(flip)), _stream()), "ipdm_fbp_project")
        return out

    def _image_out(self, sino, out):
        """out, or a new [B,512,512] device image, for the sinogram sino [B,2000,912]; ValueError unless both have these shapes and
        out is not sino."""
        self._check_sino(sino)
        b = sino.shape[0]
        out = torch.empty(b, N_PIX, N_PIX, device=sino.device, dtype=torch.float32) if out is None else out
        if tuple(out.shape) != (b, N_PIX, N_PIX):
            raise ValueError(f"out must be [{b},{N_PIX},{N_PIX}], got {tuple(out.shape)}")
        if out.data_ptr() == sino.data_ptr():
            raise ValueError("out must not alias sino")
        return out

    def project_adjoint(self, sino, flip=True, out=None):
        """Exact adjoint (transpose) of `project`: [B,2000,912] device -> [B,512,512] device, the same weights and flip frames, so
        <project(x), y> = <x, project_adjoint(y)> up to fp32 rounding.  Deterministic and slice by slice."""
        out = self._image_out(sino, out)
        check(_lib.lib().ipdm_fbp_project_adjoint(self._h, _dev(sino, "sino"), _dev(out, "out"), sino.shape[0], int(bool(flip)),
                                                  _stream()), "ipdm_fbp_project_adjoint")
        return out

    @staticmethod
    def check_sart_args(iterations=SART_DEFAULTS["iterations"], subsets=SART_DEFAULTS["subsets"], relaxation=SART_DEFAULTS["relaxation"],
                        ntv=SART_TV_DEFAULTS["ntv"], tv_alpha=SART_TV_DEFAULTS["tv_alpha"], tv_eps=SART_TV_DEFAULTS["tv_eps"],
                        init=SART_TV_DEFAULTS["init"]):
        """ValueError unless iterations >= 1, subsets divides 2000, 0 < relaxation < 2, ntv is an integer >= 0, tv_alpha and tv_eps
        are finite and > 0 and init is "zero" or "fbp"; returns them as (int, int, float, int, float, float, str)."""
        iterations, subsets, init = _sweeps("SART", iterations, subsets, init)
        relaxation = _real(relaxation, "SART relaxation", "in (0, 2)", lambda v: 0 < v < 2)
        if isinstance(ntv, bool) or not isinstance(ntv, (int, np.integer)) or ntv < 0:
            raise ValueError(f"SART-TV ntv must be an integer >= 0, got {ntv!r}")
        tv_alpha = _real(tv_alpha, "SART-TV tv_alpha", "finite and > 0", lambda v: v > 0)
        tv_eps = _real(tv_eps, "SART-TV tv_eps", "finite and > 0", lambda v: v > 0)
        return iterations, subsets, relaxation, int(ntv), tv_alpha, tv_eps, init

    @staticmethod
    def check_tv_args(ntv=SART_TV_DEFAULTS["ntv"], tv_alpha=SART_TV_DEFAULTS["tv_alpha"], tv_eps=SART_TV_DEFAULTS["tv_eps"],
                      init=SART_TV_DEFAULTS["init"]):
        """The SART-TV part of `check_sart_args`: (ntv, tv_alpha, tv_eps, init) as (int, float, float, str)."""
        return FBPPlan.check_sart_args(ntv=ntv, tv_alpha=tv_alpha, tv_eps=tv_eps, init=init)[3:]

    def sart(self, sino, flip=True, iterations=SART_DEFAULTS["iterations"], subsets=SART_DEFAULTS["subsets"],
             relaxation=SART_DEFAULTS["relaxation"], out=None, ntv=SART_TV_DEFAULTS["ntv"], tv_alpha=SART_TV_DEFAULTS["tv_alpha"],
             tv_eps=SART_TV_DEFAULTS["tv_eps"], init=SART_TV_DEFAULTS["init"]):
        """Ordered-subset SART, regularised to SART-TV by ntv > 0 (see include/ipdm_b200.h ipdm_fbp_sart_tv): line integrals
        [B,2000,912] device -> mu image [B,512,512] device in the frame of `forward` for the same flip.  The start is 0, or
        max(0, forward(sino)) for init="fbp"; every sweep is followed by ntv TV steps of length tv_alpha |x - x_prev| (tv_eps in 1/cm
        smooths the TV).  The first call for a subset count builds the plan's tables and synchronises; later calls allocate nothing
        (CUDA-graph safe)."""
        iterations, subsets, relaxation, ntv, tv_alpha, tv_eps, init = self.check_sart_args(iterations, subsets, relaxation, ntv,
                                                                                            tv_alpha, tv_eps, init)
        out = self._image_out(sino, out)
        check(_lib.lib().ipdm_fbp_sart_tv(self._h, _dev(sino, "sino"), _dev(out, "out"), sino.shape[0], int(bool(flip)), iterations,
                                          subsets, ctypes.c_float(relaxation), ntv, ctypes.c_float(tv_alpha), ctypes.c_float(tv_eps),
                                          int(init == "fbp"), _stream()), "ipdm_fbp_sart_tv")
        return out

    @staticmethod
    def check_pwls_args(iterations=SART_DEFAULTS["iterations"], subsets=SART_DEFAULTS["subsets"], dose=PWLS_DOSE,
                        beta=PWLS_DEFAULTS["beta"], delta=PWLS_DEFAULTS["delta"], init=SART_TV_DEFAULTS["init"]):
        """ValueError unless iterations >= 1, subsets divides 2000, 0 < dose <= 1, beta is finite and >= 0, delta is finite and > 0
        and init is "zero" or "fbp"; returns them as (int, int, float, float, float, str)."""
        iterations, subsets, init = _sweeps("PWLS", iterations, subsets, init)
        dose = _real(dose, "PWLS dose", "in (0, 1]", lambda v: 0 < v <= 1)
        beta = _real(beta, "PWLS beta", "finite and >= 0", lambda v: v >= 0)
        delta = _real(delta, "PWLS delta", "finite and > 0", lambda v: v > 0)
        return iterations, subsets, dose, beta, delta, init

    def pwls(self, sino, flip=True, iterations=SART_DEFAULTS["iterations"], subsets=SART_DEFAULTS["subsets"], dose=PWLS_DOSE,
             beta=PWLS_DEFAULTS["beta"], delta=PWLS_DEFAULTS["delta"], init=SART_TV_DEFAULTS["init"], out=None):
        """Penalised weighted least squares by ordered-subset SQS (see include/ipdm_b200.h ipdm_fbp_pwls): line integrals
        [B,2000,912] device at dose `dose` -> mu image [B,512,512] device in the frame of `forward` for the same flip.  The weights
        are the inverse variances of the rays at that dose; beta scales the hyperbola penalty, delta (1/cm) is its edge scale;
        subsets and sweeps as in `sart`; init="fbp" starts from max(0, forward(sino)).  The first call builds the plan's row sums and
        synchronises; later calls allocate nothing (CUDA-graph safe)."""
        iterations, subsets, dose, beta, delta, init = self.check_pwls_args(iterations, subsets, dose, beta, delta, init)
        out = self._image_out(sino, out)
        check(_lib.lib().ipdm_fbp_pwls(self._h, _dev(sino, "sino"), _dev(out, "out"), sino.shape[0], int(bool(flip)), iterations, subsets,
                                       ctypes.c_float(dose), ctypes.c_float(beta), ctypes.c_float(delta), int(init == "fbp"), _stream()),
              "ipdm_fbp_pwls")
        return out

    def pwls_penalty(self, img, delta=PWLS_DEFAULTS["delta"], flip=True):
        """(grad R, d^R) of the PWLS penalty of a [B,512,512] device image, [B,512,512] device each in the image's frame: the
        regulariser of `pwls` on its own (include/ipdm_b200.h ipdm_fbp_pwls_penalty)."""
        if img.dim() != 3 or tuple(img.shape[1:]) != (N_PIX, N_PIX):
            raise ValueError(f"image must be [B,{N_PIX},{N_PIX}], got {tuple(img.shape)}")
        delta = _real(delta, "PWLS delta", "finite and > 0", lambda v: v > 0)
        grad, curv = torch.empty_like(img), torch.empty_like(img)
        check(_lib.lib().ipdm_fbp_pwls_penalty(self._h, _dev(img, "img"), _dev(grad, "grad"), _dev(curv, "curv"), img.shape[0],
                                               int(bool(flip)), ctypes.c_float(delta), _stream()), "ipdm_fbp_pwls_penalty")
        return grad, curv

    def tv_descent(self, img, steps, step, eps=SART_TV_DEFAULTS["tv_eps"], flip=True):
        """`steps` TV steps of length `step` (the same for every slice) on a [B,512,512] device image, in place: the regulariser of
        SART-TV on its own (include/ipdm_b200.h ipdm_fbp_tv_descent).  Returns img."""
        if img.dim() != 3 or tuple(img.shape[1:]) != (N_PIX, N_PIX):
            raise ValueError(f"image must be [B,{N_PIX},{N_PIX}], got {tuple(img.shape)}")
        if isinstance(steps, bool) or int(steps) != steps or steps < 0:
            raise ValueError(f"TV steps must be an integer >= 0, got {steps!r}")
        step = _real(step, "TV step", "finite and >= 0", lambda v: v >= 0)
        eps = _real(eps, "TV eps", "finite and > 0", lambda v: v > 0)
        check(_lib.lib().ipdm_fbp_tv_descent(self._h, _dev(img, "img"), img.shape[0], int(bool(flip)), int(steps), ctypes.c_float(step),
                                             ctypes.c_float(eps), _stream()), "ipdm_fbp_tv_descent")
        return img

    def tables(self):
        theta = np.empty(N_VIEWS, np.float64)
        nda, h, wcos = np.empty(N_DET, np.float32), np.empty(2 * N_DET - 1, np.float32), np.empty(N_DET, np.float32)
        check(_lib.lib().ipdm_fbp_tables(self._h, *(a.ctypes.data_as(ctypes.c_void_p) for a in (theta, nda, h, wcos))), "ipdm_fbp_tables")
        return dict(theta=theta, nda=nda, h_RL=h, wcos=wcos)


# ---------------------------------------------------------------------------------------------
# schedules (host, fp64)
# ---------------------------------------------------------------------------------------------
SCHEDULE_FIELDS = ("betas", "alphas_cumprod", "sqrt_alphas_cumprod", "sqrt_one_minus_alphas_cumprod",
                   "sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod", "posterior_variance",
                   "posterior_log_variance_clipped", "posterior_mean_coef1", "posterior_mean_coef2")


def cosine_beta_schedule(timesteps, schedule_power=1.0):
    out = np.empty(int(timesteps), np.float64)
    check(_lib.lib().ipdm_cosine_beta_schedule(int(timesteps), float(schedule_power), out.ctypes.data_as(_lib.c_double_p)),
          "ipdm_cosine_beta_schedule")
    return out


def schedule_at(timesteps, schedule_power, t):
    out = (ctypes.c_double * 10)()
    check(_lib.lib().ipdm_schedule_at(int(timesteps), float(schedule_power), int(t), out), "ipdm_schedule_at")
    return dict(zip(SCHEDULE_FIELDS, list(out)))


def step_coefficients(timesteps, schedule_power, t):
    s = schedule_at(timesteps, schedule_power, t)
    f = np.float32
    return [f(s["sqrt_alphas_cumprod"]), f(s["sqrt_one_minus_alphas_cumprod"]), f(s["sqrt_recip_alphas_cumprod"]),
            f(s["sqrt_recipm1_alphas_cumprod"]), f(s["posterior_mean_coef1"]), f(s["posterior_mean_coef2"]),
            f(math.exp(0.5 * float(f(s["posterior_log_variance_clipped"]))))]


def lambda_curve_host(x, kind):
    x = np.ascontiguousarray(x, dtype=np.float32)
    y = np.empty_like(x)
    check(_lib.lib().ipdm_lambda_curve_host(x.ctypes.data_as(ctypes.c_void_p), y.ctypes.data_as(ctypes.c_void_p), x.size,
                                            0 if kind == "proj" else 1), "ipdm_lambda_curve_host")
    return y


# ---------------------------------------------------------------------------------------------
# sampler ops
# ---------------------------------------------------------------------------------------------
def _workspace(nbytes, device):
    return torch.empty((int(nbytes) + 3) // 4, dtype=torch.float32, device=device)


def lincomb(a, x, b, y, c=0.0, z=None, out=None):
    out = torch.empty_like(x) if out is None else out
    check(_lib.lib().ipdm_lincomb(_dev(out), float(a), _dev(x), float(b), _dev(y), float(c), _opt(z), x.numel(), _stream()), "ipdm_lincomb")
    return out


def clamp_(x, lo=-math.inf, hi=math.inf):
    check(_lib.lib().ipdm_clamp(_dev(x), float(lo), float(hi), x.numel(), _stream()), "ipdm_clamp")
    return x


def set_noise_epoch(epoch):
    """Stream-ordered update of the device-resident half of the Philox key (fresh noise per CUDA-graph replay)."""
    check(_lib.lib().ipdm_set_noise_epoch(int(epoch) & (2 ** 64 - 1), _stream()), "ipdm_set_noise_epoch")


def q_sample(x, a, b, noise=None, seed=0, call_id=0, out=None):
    bsz = x.shape[0]
    out = torch.empty_like(x) if out is None else out
    check(_lib.lib().ipdm_q_sample(_dev(x), _opt(noise), _dev(out), float(a), float(b), x.numel() // bsz, bsz, int(seed), int(call_id),
                                   _stream()), "ipdm_q_sample")
    return out


def low_dose_noise(sino, dose, seed=0, slice_ids=None, noise=None, clip=True, out=None):
    """Dose-reduction noise of the reference's add_noise (Utils/Low_dose_CT_simulate.py:38-44) on line integrals sino [B,...]
    (device): p + sqrt((1-f) e^p (1 + (1+f) Ne e^p / (f N0)) / (f N0)) * n with f = dose, clamped at 0 iff clip.  n is the tape
    `noise` (shaped like sino) or in-kernel Philox keyed by (seed, slice id, element / 4); slice_ids (B ints, default 0..B-1) are
    dataset indices, so a slice draws the same noise whatever batch it is in.  out may be sino (in place)."""
    if sino.dim() < 2:
        raise ValueError(f"sino must be [B,...], got {tuple(sino.shape)}")
    if not 0.0 < float(dose) <= 1.0:
        raise ValueError(f"dose must be in (0, 1], got {dose}")
    b = sino.shape[0]
    out = torch.empty_like(sino) if out is None else out
    if out.shape != sino.shape:
        raise ValueError(f"out must be shaped like sino {tuple(sino.shape)}, got {tuple(out.shape)}")
    if noise is not None and noise.shape != sino.shape:
        raise ValueError(f"noise must be shaped like sino {tuple(sino.shape)}, got {tuple(noise.shape)}")
    ids = None
    if slice_ids is not None:
        ids = torch.as_tensor([int(i) for i in slice_ids], dtype=torch.int64).to(sino.device)
        if ids.numel() != b or bool((ids < 0).any()):
            raise ValueError(f"slice_ids must hold {b} non-negative ids, got {list(slice_ids)}")
    check(_lib.lib().ipdm_low_dose_noise(_dev(sino, "sino"), _opt(noise, "noise"), _dev(out, "out"), b, sino.numel() // b, float(dose),
                                         int(bool(clip)), int(seed) & (2 ** 64 - 1), None if ids is None else ctypes.c_void_p(ids.data_ptr()),
                                         _stream()), "ipdm_low_dose_noise")
    return out


def sampler_step(x_t, x0c, eps, coef7, lam, noise=None, clip=False, t_nonzero=True, ks=4, seed=0, call_id=0, out=None):
    """One guided reverse step (see ipdm_sampler_step); `lam` is a float or a [B,h/ks,w/ks] tensor."""
    b, h, w = x_t.shape[0], x_t.shape[-2], x_t.shape[-1]
    out = torch.empty_like(x_t) if out is None else out
    ws = _workspace(_lib.lib().ipdm_sampler_workspace_bytes(b, h, w), x_t.device)
    coef = (ctypes.c_float * 7)(*[float(c) for c in coef7])
    lam_map = lam if isinstance(lam, torch.Tensor) else None
    check(_lib.lib().ipdm_sampler_step(_dev(x_t), _dev(x0c), _dev(eps), _opt(noise), _dev(out), b, h, w, coef,
                                       0.0 if lam_map is not None else float(lam), _opt(lam_map), int(ks), int(bool(clip)),
                                       int(bool(t_nonzero)), int(seed), int(call_id), _dev(ws), _stream()), "ipdm_sampler_step")
    return out


def ddim_coefficients(timesteps, schedule_power, t, t_prev, ddim_eta=0.0):
    """coef8 of ipdm_sampler_step_ddim for the pair (t, t_prev), from the fp64 schedule tables cast to fp32 like the reference's
    `_extract(...).float()` (Model/model.py ddim_sample :688-712)."""
    f = schedule_at(timesteps, schedule_power, int(t))
    fp = schedule_at(timesteps, schedule_power, int(t_prev))
    a_t, a_p = np.float32(f["alphas_cumprod"]), np.float32(fp["alphas_cumprod"])
    one = np.float32(1.0)
    sig_dir = np.float32(ddim_eta) * np.sqrt((one - a_p) / (one - a_t) * (one - a_t / a_p))
    coef_e = np.sqrt(one - a_p - sig_dir * sig_dir)
    sigma = np.float32(ddim_eta) * np.float32(f["posterior_variance"])
    return [float(f["sqrt_alphas_cumprod"]), float(f["sqrt_one_minus_alphas_cumprod"]), float(one / np.sqrt(a_t)),
            float(np.sqrt(one - a_t) / np.sqrt(a_t)), float(np.sqrt(a_p)), 0.0, float(sigma), float(coef_e)]


def sampler_step_ddim(x_t, x0c, eps, coef8, lam, noise=None, clip=True, with_noise=False, seed=0, call_id=0, out=None):
    """One guided DDIM step (see ipdm_sampler_step_ddim); `lam` is the scalar condition_lambda."""
    b, h, w = x_t.shape[0], x_t.shape[-2], x_t.shape[-1]
    out = torch.empty_like(x_t) if out is None else out
    ws = _workspace(_lib.lib().ipdm_sampler_workspace_bytes(b, h, w), x_t.device)
    coef = (ctypes.c_float * 8)(*[float(c) for c in coef8])
    check(_lib.lib().ipdm_sampler_step_ddim(_dev(x_t), _dev(x0c), _dev(eps), _opt(noise), _dev(out), b, h, w, coef, float(lam),
                                            int(bool(clip)), int(bool(with_noise)), int(seed), int(call_id), _dev(ws), _stream()),
          "ipdm_sampler_step_ddim")
    return out


def delta_lambda_map(x, img, ks=4, amplitude=7.0, kind="proj", return_median=False):
    b, h, w = x.shape[0], x.shape[-2], x.shape[-1]
    out = torch.empty(b, h // ks, w // ks, device=x.device, dtype=torch.float32)
    med = torch.empty(b, device=x.device, dtype=torch.float32)
    ws = _workspace(_lib.lib().ipdm_sampler_workspace_bytes(b, h, w), x.device)
    check(_lib.lib().ipdm_delta_lambda_map(_dev(x), _dev(img), _dev(out), _dev(med), b, h, w, int(ks), float(amplitude),
                                           0 if kind == "proj" else 1, _dev(ws), _stream()), "ipdm_delta_lambda_map")
    return (out, med) if return_median else out


def delta_lambda_map_img(x, img, ks=4, amplitude=7.0):
    """Image-domain lambda-exponent map (Model/model.py:591-595): pool |miu2pixel(x) - miu2pixel(img)| first, median of the pooled map."""
    b, h, w = x.shape[0], x.shape[-2], x.shape[-1]
    out = torch.empty(b, h // ks, w // ks, device=x.device, dtype=torch.float32)
    pooled = torch.empty_like(out)
    ws = _workspace(_lib.lib().ipdm_sampler_workspace_bytes(b, h, w), x.device)
    check(_lib.lib().ipdm_delta_lambda_map_img(_dev(x), _dev(img), _dev(out), None, _dev(pooled), b, h, w, int(ks), float(amplitude), 1,
                                               _dev(ws), _stream()), "ipdm_delta_lambda_map_img")
    return out


def delta_exp_max(x, img, ks=4, amplitude=7.0):
    """Per-slice max of exp(amplitude * relu(avgpool(|x - img| - median))) as a CUDA tensor [B] (adaptive schedule selection, :596-613)."""
    b, h, w = x.shape[0], x.shape[-2], x.shape[-1]
    out = torch.empty(b, device=x.device, dtype=torch.float32)
    ws = _workspace(_lib.lib().ipdm_sampler_workspace_bytes(b, h, w), x.device)
    check(_lib.lib().ipdm_delta_exp_max(_dev(x), _dev(img), _dev(out), b, h, w, int(ks), float(amplitude), _dev(ws), _stream()), "ipdm_delta_exp_max")
    return out


def lambda_step_map(lam_exp, i, ts):
    out = torch.empty_like(lam_exp)
    check(_lib.lib().ipdm_lambda_step_map(_dev(lam_exp), _dev(out), lam_exp.numel(), int(i), int(ts), _stream()), "ipdm_lambda_step_map")
    return out


def sharpen3x3(img, N):
    """tensor_sharpen (Utils/train_test_utils.py:868-878) per slice; img [B,1,H,W] or [B,H,W]."""
    b, h, w = img.shape[0], img.shape[-2], img.shape[-1]
    out = torch.empty_like(img)
    check(_lib.lib().ipdm_sharpen3x3(_dev(img), _dev(out), b, h, w, int(N), _stream()), "ipdm_sharpen3x3")
    return out


# ---------------------------------------------------------------------------------------------
# UNet
# ---------------------------------------------------------------------------------------------
# ---------------------------------------------------------------------------------------------
# image-quality metrics (SURVEY N1; reference: metric_calculate, Utils/train_test_utils.py:789-799)
# ---------------------------------------------------------------------------------------------
def miu2pixel(mu, hu_range=(-1024.0, 3072.0), out=None):
    """Dataset/npz_data_loader.py:20-36 on the device: mu -> HU -> [hu_lo, hu_hi] window mapped to [0,1], clipped; NaN -> 0.5."""
    _require_cuda()
    out = torch.empty_like(mu) if out is None else out
    check(_lib.lib().ipdm_miu2pixel(_dev(mu, "mu"), _dev(out, "out"), mu.numel(), float(hu_range[0]), float(hu_range[1]), _stream()), "ipdm_miu2pixel")
    return out


def psnr_ssim(test, ref, win_size=11):
    """[B,H,W] (or [B,1,H,W]) images in pixel units -> float64 CUDA tensor [B,2] = (PSNR dB, SSIM) with skimage's definitions
    for data_range=1, win_size=11 (uniform window, K1=.01, K2=.03, sample covariance, map cropped by win//2)."""
    _require_cuda()
    if test.dim() == 4:
        test, ref = test[:, 0], ref[:, 0]
    if test.dim() != 3 or test.shape != ref.shape:
        raise ValueError(f"psnr_ssim: shapes {tuple(test.shape)} / {tuple(ref.shape)} must be equal [B,H,W]")
    test, ref = test.contiguous(), ref.contiguous()
    b, h, w = test.shape
    out = torch.empty(b, 2, device=test.device, dtype=torch.float64)
    ws = _workspace(int(_lib.lib().ipdm_metrics_workspace_bytes(b, h, w)), test.device)
    check(_lib.lib().ipdm_psnr_ssim(_dev(test, "test"), _dev(ref, "ref"), b, h, w, int(win_size), ctypes.c_void_p(out.data_ptr()),
                                    ctypes.c_void_p(ws.data_ptr()), _stream()), "ipdm_psnr_ssim")
    return out


def unet_config(in_channels, model_channels, out_channels, num_res_blocks, attention_resolutions, channel_mult, num_heads,
                precision="tf32", max_t=64):
    cfg = UNetConfig()
    cfg.in_channels, cfg.model_channels, cfg.out_channels = int(in_channels), int(model_channels), int(out_channels)
    cfg.num_res_blocks, cfg.num_heads = int(num_res_blocks), int(num_heads)
    cfg.n_mult = len(channel_mult)
    for i, m in enumerate(channel_mult):
        cfg.channel_mult[i] = float(m)
    cfg.n_attn = len(attention_resolutions)
    for i, a in enumerate(attention_resolutions):
        cfg.attention_resolutions[i] = int(a)
    if precision not in PRECISIONS:
        raise ValueError(f"precision must be one of {sorted(PRECISIONS)}")
    cfg.precision = PRECISIONS[precision]
    cfg.max_t = int(max_t)
    return cfg


class UNetHandle:
    """Packed weights + execution plans of one UNet on the current device."""

    def __init__(self, cfg, state_dict, device=None):
        _require_cuda()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        flat = torch.cat([v.detach().reshape(-1).to(torch.float32).cpu() for v in state_dict.values()]).contiguous()
        expect = int(_lib.lib().ipdm_unet_param_count(ctypes.byref(cfg)))
        if flat.numel() != expect:
            raise ValueError(f"state_dict holds {flat.numel()} values, the architecture needs {expect}")
        self.cfg = cfg
        self._h = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            check(_lib.lib().ipdm_unet_create(ctypes.byref(self._h), ctypes.byref(cfg), ctypes.c_void_p(flat.data_ptr()), flat.numel()),
                  "ipdm_unet_create")

    def _on_device(self, x, name):
        if x.device != self.device:
            raise ValueError(f"{name} lives on {x.device}, the UNet handle on {self.device}")
        return torch.cuda.device(self.device)

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None and getattr(_lib, "_lib", None) is not None:
            _lib._lib.ipdm_unet_destroy(self._h)
            self._h = None

    def forward(self, x, t, out=None):
        """eps[B,1,H,W] = UNet(x[B,1,H,W], t) with one integer timestep for the whole batch."""
        b, h, w = x.shape[0], x.shape[-2], x.shape[-1]
        out = torch.empty_like(x) if out is None else out
        with self._on_device(x, "x"):
            check(_lib.lib().ipdm_unet_forward(self._h, _dev(x, "x"), int(t), _dev(out, "out"), b, h, w, _stream()), "ipdm_unet_forward")
        return out

    def flops(self, b, h, w):
        with torch.cuda.device(self.device):                     # builds (and keeps) the plan of this shape
            return float(_lib.lib().ipdm_unet_flops(self._h, int(b), int(h), int(w)))


# ---------------------------------------------------------------------------------------------
# guided process
# ---------------------------------------------------------------------------------------------
def guided_params(mode, t_start, clip, lambda_ratio, eta, constant_guidance, kernel_size, amplitude, schedule_power,
                  timesteps=1000, seed=0):
    p = GuidedParams()
    p.mode = 0 if mode == "proj" else 1
    if t_start is None:
        raise ValueError("guided_params needs an explicit t_start list (the adaptive branch picks one on the host first, Model/model.py)")
    if not 1 <= len(t_start) <= 8:
        raise ValueError("t_start must hold 1..8 entries")
    p.n_iters = len(t_start)
    for i, t in enumerate(t_start):
        p.t_start[i] = int(t)
    p.clip = int(bool(clip))
    p.lambda_ratio, p.eta = float(lambda_ratio), float(eta)
    p.constant_guidance_set = int(constant_guidance is not None)
    p.constant_guidance = float(constant_guidance) if constant_guidance is not None else 0.0
    p.kernel_size, p.amplitude = int(kernel_size), float(amplitude)
    p.curve_kind = 0 if mode == "proj" else 1
    p.timesteps, p.schedule_power = int(timesteps), float(schedule_power)
    p.seed = int(seed)
    return p


def guided_noise_count(p):
    return int(_lib.lib().ipdm_guided_noise_count(ctypes.byref(p)))


def guided_process(unet, p, img, ldct=None, noise=None, out=None):
    """Runs ipdm_guided_process. img [B,1,H,W]; noise None (Philox) or [count,B,1,H,W];
    returns [n_iters+1 (or 1), B, 1, H, W]."""
    b, h, w = img.shape[0], img.shape[-2], img.shape[-1]
    n_out = p.n_iters + 1 if p.n_iters > 1 else 1
    if noise is not None and noise.shape[0] < guided_noise_count(p):
        raise ValueError(f"noise tape holds {noise.shape[0]} draws, the process consumes {guided_noise_count(p)}")
    out = torch.empty((n_out, b, 1, h, w), device=img.device, dtype=torch.float32) if out is None else out
    with unet._on_device(img, "img"):
        ws = _workspace(_lib.lib().ipdm_guided_workspace_bytes(ctypes.byref(p), b, h, w), img.device)
        check(_lib.lib().ipdm_guided_process(unet._h, ctypes.byref(p), _dev(img, "img"), _opt(ldct, "ldct"), _opt(noise, "noise"),
                                             _dev(out), b, h, w, _dev(ws), _stream()), "ipdm_guided_process")
    return out


def guided_process_resume(unet, p, img, lam_exp, call_base, ldct=None, noise=None):
    """Runs ipdm_guided_process_resume: iterations 1.. of an adaptive-lambda process whose probing iteration produced `lam_exp`
    [B,H/ks,W/ks]; noise None or the tape of the continuation [count,B,1,H,W]; returns [n_iters+1, B, 1, H, W]."""
    b, h, w = img.shape[0], img.shape[-2], img.shape[-1]
    if noise is not None and noise.shape[0] < guided_noise_count(p):
        raise ValueError(f"noise tape holds {noise.shape[0]} draws, the continuation consumes {guided_noise_count(p)}")
    out = torch.empty((p.n_iters + 1, b, 1, h, w), device=img.device, dtype=torch.float32)
    with unet._on_device(img, "img"):
        ws = _workspace(_lib.lib().ipdm_guided_workspace_bytes(ctypes.byref(p), b, h, w), img.device)
        check(_lib.lib().ipdm_guided_process_resume(unet._h, ctypes.byref(p), _dev(img, "img"), _opt(ldct, "ldct"), _opt(noise, "noise"),
                                                    _dev(lam_exp, "lam_exp"), int(call_base), _dev(out), b, h, w, _dev(ws), _stream()),
              "ipdm_guided_process_resume")
    return out
