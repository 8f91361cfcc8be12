"""TEST INFRASTRUCTURE ONLY -- python face of oracle/pwls_oracle.c.

fp64 penalised weighted least squares (dose-aware weights, hyperbola edge-preserving penalty) and its ordered-subset SQS solver,
in the geometry of the reference FBP and on the Joseph matrix of oracle/sart_oracle.c.  Only tests/ and tools/ may import this
module.
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

from . import sart_oracle as _sart

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "pwls_oracle.c")
_DEPS = (_SRC, os.path.join(_HERE, "sart_oracle.c"))            # pwls_oracle.c includes sart_oracle.c
_lib = None


def build():
    """Compiles pwls_oracle.c into oracle/_build (or a temporary directory when the tree is read-only); returns the .so path."""
    out_dir = os.path.join(_HERE, "_build")
    try:
        os.makedirs(out_dir, exist_ok=True)
        if not os.access(out_dir, os.W_OK):
            raise PermissionError(out_dir)
    except OSError:
        out_dir = tempfile.mkdtemp(prefix="pwls_oracle_")
    so = os.path.join(out_dir, "libpwls_oracle.so")
    if os.path.exists(so) and os.path.getmtime(so) >= max(os.path.getmtime(d) for d in _DEPS):
        return so
    for cc in (["/usr/bin/gcc"], ["gcc"]):
        for extra in (["-fopenmp"], ["-Wno-unknown-pragmas"]):
            try:
                if subprocess.run(cc + _sart._CFLAGS + extra + ["-o", so, _SRC, "-lm"]).returncode == 0:
                    return so
            except OSError:                                    # no such compiler
                pass
    raise RuntimeError("could not compile oracle/pwls_oracle.c")


def _load():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
    return _lib


_dp = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
_fp = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
_i = lambda v: ctypes.c_int(int(v))
_d = ctypes.c_double


def _images(img):
    img = np.array(img, dtype=np.float64, order="C", copy=True)
    if img.ndim == 2:
        img = img[None]
    assert img.shape[1:] == (512, 512), img.shape
    return img


def _sinos(sino):
    sino = np.ascontiguousarray(sino, dtype=np.float32)
    if sino.ndim == 2:
        sino = sino[None]
    assert sino.shape[1:] == (2000, 912), sino.shape
    return sino


def _geom():
    theta, alpha = _sart._geometry()
    return _dp(theta), _dp(alpha), _d(_sart.D), _d(_sart.DX), (theta, alpha)


def weights(sino, dose):
    """w = 1 / sigma^2(max(b, 0)) of every bin of a sinogram (taken as f32), f64, the same shape."""
    b = np.ascontiguousarray(sino, dtype=np.float32)
    w = np.empty(b.shape, np.float64)
    _load().pwls_weights_oracle(_fp(b), _dp(w), ctypes.c_long(b.size), _d(dose))
    return w


def penalty(img, delta, flip=True):
    """[B,512,512] / [512,512] image (frame flip) -> (R [B], grad R [B,512,512], d^R [B,512,512]), f64, the same frame."""
    x = _images(img)
    b = x.shape[0]
    val, g, c = np.empty(b), np.empty_like(x), np.empty_like(x)
    _load().pwls_penalty_oracle(_dp(x), _dp(val), _dp(g), _dp(c), _i(b), _i(flip), _d(delta))
    return val, g, c


def denominator(sino, dose, flip=True):
    """D^L = A^T (w o A 1) of every slice: [B,2000,912] / [2000,912] -> [B,512,512] f64 (frame flip)."""
    s = _sinos(sino)
    out = np.empty((s.shape[0], 512, 512))
    th, al, D, dx, keep = _geom()
    _load().pwls_denom_oracle(_fp(s), _dp(out), _i(s.shape[0]), _i(flip), _d(dose), th, al, D, dx)
    return out


def data_term(sino, img, dose, flip=True, grad=False):
    """L(x) = 1/2 sum w (A x - b)^2 per slice [B]; with grad=True also grad L = A^T (w o (A x - b)) [B,512,512] (frame flip)."""
    s, x = _sinos(sino), _images(img)
    assert s.shape[0] == x.shape[0]
    val = np.empty(s.shape[0])
    g = np.empty_like(x) if grad else None
    th, al, D, dx, keep = _geom()
    _load().pwls_data_oracle(_fp(s), _dp(x), _dp(val), None if g is None else _dp(g), _i(s.shape[0]), _i(flip), _d(dose), th, al, D, dx)
    return (val, g) if grad else val


def objective(sino, img, dose, beta, delta, flip=True):
    """Phi(x) = L(x) + beta R(x) per slice [B], f64."""
    return data_term(sino, img, dose, flip) + beta * penalty(img, delta, flip)[0]


def pwls(sino, flip=True, iterations=5, subsets=100, dose=0.25, beta=1e4, delta=0.005, init="zero", x0=None, history=False):
    """OS-SQS for PWLS (ipdm_fbp_pwls): [B,2000,912] / [2000,912] line integrals (taken as f32) -> [B,512,512] f64 after
    `iterations` sweeps.  init="zero" starts at 0; init="fbp" at max(0, FBP(sino)) of the fp32 FBP oracle, or at max(0, x0) when x0
    ([B,512,512], frame flip) is given.  With history=True also [B,iterations,512,512], the iterate after every sweep."""
    s = _sinos(sino)
    assert 2000 % subsets == 0 and iterations >= 1 and init in ("zero", "fbp")
    b = s.shape[0]
    if init == "fbp":
        if x0 is None:
            from . import fbp_oracle
            x0 = fbp_oracle.convert(s, flip)
        x0 = np.ascontiguousarray(x0, dtype=np.float64).reshape(b, 512, 512)
    else:
        x0 = None
    out = np.empty((b, 512, 512))
    hist = np.empty((b, iterations, 512, 512)) if history else None
    th, al, D, dx, keep = _geom()
    _load().pwls_oracle(_fp(s), None if x0 is None else _dp(x0), _dp(out), None if hist is None else _dp(hist), _i(b), _i(flip),
                        _i(iterations), _i(subsets), _d(dose), _d(beta), _d(delta), th, al, D, dx)
    return (out, hist) if history else out
