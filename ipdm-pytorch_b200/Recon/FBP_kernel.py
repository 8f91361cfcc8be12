"""Host-side mirror of the reference's Recon/FBP_kernel.py: class FBP with `convert`.

`FBP(device).convert(pj, flip=True)` keeps the reference contract (:86-122): ndarray or Tensor
[B,2000,912] / [2000,912] in, the same kind out, [B,512,512] float32 ON THE HOST.  The arithmetic
(cosine weighting, ramp filter, pixel-driven fan-beam backprojection) runs in libipdm_b200.so;
`convert_device` is the additive zero-copy entry the progressive pipeline uses.

Additive: `project(img, flip=True)` / `project_device(img)`, the forward projector in the same geometry
(Joseph's method, see include/ipdm_b200.h ipdm_fbp_project).  It is not the reference's `proj_torch`
(an area-integral projector with a lookup table, Recon/TASART2DNSL0.py), so the two do not agree sample
for sample.

Additive: `sart(pj, flip=True, **kw)` / `sart_device(pj)`, an iterative convertor (ordered-subset SART on the projector and its
exact adjoint, SART-TV with ntv > 0, include/ipdm_b200.h ipdm_fbp_sart_tv) with `convert`'s contract.  It is not the reference's
ART convertor (TASART2DNSL0.pyd: SART with an NSL0-TV step and the area-integral projector): its TV steps are ASD-POCS steps on a
smoothed isotropic TV, not the NSL0 formula.

Additive: `pwls(pj, flip=True, **kw)` / `pwls_device(pj)`, a statistically weighted iterative convertor (penalised weighted
least squares with dose-aware weights, solved by ordered-subset SQS, include/ipdm_b200.h ipdm_fbp_pwls) with `convert`'s contract.
"""
import numpy as np
import torch

from _ipdm_boot import engine as _eng


class FBP:
    def __init__(self, device="cuda:0"):
        if str(device) == "cpu":
            raise RuntimeError("FBP: the B200 build has no CPU path (the reference's numba CPU twin is the test oracle only)")
        self.device = torch.device(device)
        with torch.cuda.device(self.device):
            self._plan = _eng.FBPPlan()
        t = self._plan.tables()
        # geometry attributes of the reference object (FBP_kernel.py:32-56)
        self.os_, self.od, self.T, self.da = 59.5, 108.56 - 59.5, 0.0010125, 0.0010125
        self.D, self.N, self.M = 59.5, 912, 2000
        self.theta, self.nda, self.h_RL = t["theta"], t["nda"], t["h_RL"][:, None]

    def convert_device(self, pj, flip=True):
        """[B,2000,912] CUDA tensor -> [B,512,512] CUDA tensor, no host copy, current stream."""
        with torch.cuda.device(self.device):
            return self._plan.forward(pj.contiguous().float(), flip=flip)

    def project_device(self, img, flip=True):
        """[B,512,512] CUDA mu image -> [B,2000,912] CUDA line integrals, no host copy, current stream."""
        with torch.cuda.device(self.device):
            return self._plan.project(img.contiguous().float(), flip=flip)

    def _on_host(self, device_call, a, flip, **kw):
        """`convert`'s contract around a device call: ndarray or Tensor, one slice or a batch, in; the same kind out, float32 on
        the host."""
        as_tensor = isinstance(a, torch.Tensor)
        x = a.detach().float() if as_tensor else torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32))
        x = x[None] if x.dim() == 2 else x
        out = device_call(x.to(self.device), flip, **kw).cpu()
        return out if as_tensor else out.numpy()

    def project(self, img, flip=True):
        """`convert`'s contract in the other direction: ndarray or Tensor [B,512,512] / [512,512] in, the same kind out,
        [B,2000,912] float32 on the host."""
        return self._on_host(self.project_device, img, flip)

    def sart_device(self, pj, flip=True, **kw):
        """Iterative convertor: [B,2000,912] CUDA line integrals -> [B,512,512] CUDA image by ordered-subset SART (keywords
        iterations, subsets, relaxation, and ntv, tv_alpha, tv_eps, init of SART-TV; see engine.FBPPlan.sart), no host copy,
        current stream."""
        with torch.cuda.device(self.device):
            return self._plan.sart(pj.contiguous().float(), flip=flip, **kw)

    def sart(self, pj, flip=True, **kw):
        """`convert`'s contract with SART instead of FBP: ndarray or Tensor [B,2000,912] / [2000,912] in, the same kind out,
        [B,512,512] float32 on the host."""
        return self._on_host(self.sart_device, pj, flip, **kw)

    def pwls_device(self, pj, flip=True, **kw):
        """Statistically weighted convertor: [B,2000,912] CUDA line integrals -> [B,512,512] CUDA image by PWLS / OS-SQS (keywords
        iterations, subsets, dose, beta, delta, init; see engine.FBPPlan.pwls), no host copy, current stream."""
        with torch.cuda.device(self.device):
            return self._plan.pwls(pj.contiguous().float(), flip=flip, **kw)

    def pwls(self, pj, flip=True, **kw):
        """`convert`'s contract with PWLS instead of FBP: ndarray or Tensor [B,2000,912] / [2000,912] in, the same kind out,
        [B,512,512] float32 on the host."""
        return self._on_host(self.pwls_device, pj, flip, **kw)

    def convert(self, pj, flip=True):
        as_tensor = isinstance(pj, torch.Tensor)
        if as_tensor and pj.is_cuda:
            x = pj.detach().float()
            x = x[None] if x.dim() == 2 else x
            return self.convert_device(x.contiguous(), flip).cpu()
        arr = pj.detach().cpu().numpy() if as_tensor else np.asarray(pj)
        with torch.cuda.device(self.device):
            out = self._plan.convert_host(arr, flip)
        return torch.from_numpy(out) if as_tensor else out
