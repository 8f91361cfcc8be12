"""Shim for the reference's Windows-only ART extension (Recon/TASART2DNSL0.pyd, out of scope).

Its source is not available, so neither its NSL0 regulariser nor its area-integral projector is ported.  The nearest thing this
build has is convertor="SART" with ntv > 0: ordered-subset SART on a Joseph projector with TV steps between the sweeps
(ASD-POCS on a smoothed isotropic TV, include/ipdm_b200.h ipdm_fbp_sart_tv), which is a different algorithm.

Utils/train_test_utils.py of the reference imports `recons_torch` / `proj_torch` unconditionally
(:19) and wraps `proj_torch` in a partial (:233); both names exist here and fail loudly when called.
"""


def _unavailable(name):
    def fn(*args, **kwargs):
        raise RuntimeError(f"{name}: the ART convertor / area-integral projector (TASART2DNSL0.pyd, Windows + CUDA 11.0) is "
                           "out of scope of the B200 build; use convertor='FBP'")
    fn.__name__ = name
    return fn


recons_torch = _unavailable("recons_torch")
proj_torch = _unavailable("proj_torch")
