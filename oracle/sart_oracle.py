"""TEST INFRASTRUCTURE ONLY -- python face of oracle/sart_oracle.c.

fp64 adjoint of the Joseph forward projector (oracle/project_oracle.py) and fp64 ordered-subset SART, in the geometry of the
reference FBP.  Only tests/ may import this module.
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "sart_oracle.c")
D, DX = 59.5, 42.0 / 512
# the flags of oracle/Makefile; some images wrap gcc without libgomp: OpenMP first, then without
_CFLAGS = ["-O2", "-fPIC", "-shared", "-ffp-contract=off", "-Wall"]

_lib = None


def build():
    """Compiles sart_oracle.c into oracle/_build (or a temporary directory when the tree is read-only); returns the .so path."""
    out_dir = os.path.join(_HERE, "_build")
    try:
        os.makedirs(out_dir, exist_ok=True)
        if not os.access(out_dir, os.W_OK):
            raise PermissionError(out_dir)
    except OSError:
        out_dir = tempfile.mkdtemp(prefix="sart_oracle_")
    so = os.path.join(out_dir, "libsart_oracle.so")
    if os.path.exists(so) and os.path.getmtime(so) >= os.path.getmtime(_SRC):
        return so
    for cc in (["/usr/bin/gcc"], ["gcc"]):
        for extra in (["-fopenmp"], ["-Wno-unknown-pragmas"]):
            try:
                if subprocess.run(cc + _CFLAGS + extra + ["-o", so, _SRC, "-lm"]).returncode == 0:
                    return so
            except OSError:                                    # no such compiler
                pass
    raise RuntimeError("could not compile oracle/sart_oracle.c")


def _load():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
    return _lib


def _geometry(views=None):
    from ipdm_pytorch_b200 import synthetic as S
    theta = S.view_angles()
    theta = np.ascontiguousarray(theta if views is None else theta[np.asarray(views)], dtype=np.float64)
    alpha = np.ascontiguousarray(S.detector_angles().astype(np.float64) + 0.5 * S.DET_PITCH)
    return theta, alpha


_dp = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def adjoint(sino, flip=True, views=None):
    """[B,n_views,912] or [n_views,912] sinogram -> [B,512,512] f64 A^T sino, over all 2000 views or the indices `views` (the rows
    of sino are those views, in that order)."""
    sino = np.ascontiguousarray(sino, dtype=np.float64)
    if sino.ndim == 2:
        sino = sino[None]
    theta, alpha = _geometry(views)
    assert sino.shape[1:] == (theta.size, 912), sino.shape
    out = np.empty((sino.shape[0], 512, 512), dtype=np.float64)
    _load().adjoint_oracle(_dp(sino), _dp(out), ctypes.c_int(sino.shape[0]), ctypes.c_int(theta.size), ctypes.c_int(1 if flip else 0),
                           _dp(theta), _dp(alpha), ctypes.c_double(D), ctypes.c_double(DX))
    return out


def visit_step(subsets):
    return int(_load().sart_visit_step(ctypes.c_int(int(subsets))))


def sart(sino, flip=True, iterations=5, subsets=20, relaxation=1.0, history=False):
    """[B,2000,912] or [2000,912] line integrals (taken as f32, as the device takes them) -> [B,512,512] f64 image after
    `iterations` sweeps of ordered-subset SART (ipdm_fbp_sart_tv with ntv = 0); with history=True also [B,iterations,512,512],
    the iterate after every sweep."""
    sino = np.ascontiguousarray(sino, dtype=np.float32)
    if sino.ndim == 2:
        sino = sino[None]
    assert sino.shape[1:] == (2000, 912), sino.shape
    assert 2000 % subsets == 0 and iterations >= 1
    theta, alpha = _geometry()
    b = sino.shape[0]
    out = np.empty((b, 512, 512), dtype=np.float64)
    hist = np.empty((b, iterations, 512, 512), dtype=np.float64) if history else None
    _load().sart_oracle(sino.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), _dp(out), None if hist is None else _dp(hist),
                        ctypes.c_int(b), ctypes.c_int(1 if flip else 0), ctypes.c_int(int(iterations)), ctypes.c_int(int(subsets)),
                        ctypes.c_double(relaxation), _dp(theta), _dp(alpha), ctypes.c_double(D), ctypes.c_double(DX))
    return (out, hist) if history else out
