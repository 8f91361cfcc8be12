"""TEST INFRASTRUCTURE ONLY -- python face of oracle/project_oracle.c.

fp64 Joseph forward projector in the geometry of the reference FBP (the rays synthetic.fan_sinogram
traces).  Only tests/ may import this module.
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "project_oracle.c")
D, DX = 59.5, 42.0 / 512
# the flags of oracle/Makefile; some images wrap gcc without libgomp: OpenMP first, then without
_CFLAGS = ["-O2", "-fPIC", "-shared", "-ffp-contract=off", "-Wall"]

_lib = None


def build():
    """Compiles project_oracle.c into oracle/_build (or a temporary directory when the tree is read-only); returns the .so path."""
    out_dir = os.path.join(_HERE, "_build")
    try:
        os.makedirs(out_dir, exist_ok=True)
        if not os.access(out_dir, os.W_OK):
            raise PermissionError(out_dir)
    except OSError:
        out_dir = tempfile.mkdtemp(prefix="project_oracle_")
    so = os.path.join(out_dir, "libproject_oracle.so")
    if os.path.exists(so) and os.path.getmtime(so) >= os.path.getmtime(_SRC):
        return so
    for cc in (["/usr/bin/gcc"], ["gcc"]):
        for extra in (["-fopenmp"], ["-Wno-unknown-pragmas"]):
            try:
                if subprocess.run(cc + _CFLAGS + extra + ["-o", so, _SRC, "-lm"]).returncode == 0:
                    return so
            except OSError:                                    # no such compiler
                pass
    raise RuntimeError("could not compile oracle/project_oracle.c")


def _load():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
    return _lib


def project(img, flip=True, views=None):
    """[B,512,512] or [512,512] f32 mu image -> [B,n_views,912] f64 line integrals, all 2000 views or the indices `views`."""
    from ipdm_pytorch_b200 import synthetic as S
    img = np.ascontiguousarray(img, dtype=np.float32)
    if img.ndim == 2:
        img = img[None]
    assert img.shape[1:] == (512, 512), img.shape
    theta = S.view_angles()
    theta = np.ascontiguousarray(theta if views is None else theta[np.asarray(views)], dtype=np.float64)
    alpha = np.ascontiguousarray(S.detector_angles().astype(np.float64) + 0.5 * S.DET_PITCH)
    out = np.empty((img.shape[0], theta.size, 912), dtype=np.float64)
    dp = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    _load().project_oracle(img.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), dp(out), ctypes.c_int(img.shape[0]), ctypes.c_int(theta.size),
                           ctypes.c_int(1 if flip else 0), dp(theta), dp(alpha), ctypes.c_double(D), ctypes.c_double(DX))
    return out
