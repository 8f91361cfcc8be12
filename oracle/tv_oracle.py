"""TEST INFRASTRUCTURE ONLY -- python face of oracle/tv_oracle.c.

fp64 gradient of the eps-smoothed isotropic total variation, fp64 TV steps, and fp64 SART-TV (ordered-subset SART of
oracle/sart_oracle.c with a start image and TV steps between the sweeps), in the geometry of the reference FBP.  Only tests/ and
tools/ may import this module.
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

from . import sart_oracle as _sart

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "tv_oracle.c")
_DEPS = (_SRC, os.path.join(_HERE, "sart_oracle.c"))            # tv_oracle.c includes sart_oracle.c
_lib = None


def build():
    """Compiles tv_oracle.c into oracle/_build (or a temporary directory when the tree is read-only); returns the .so path."""
    out_dir = os.path.join(_HERE, "_build")
    try:
        os.makedirs(out_dir, exist_ok=True)
        if not os.access(out_dir, os.W_OK):
            raise PermissionError(out_dir)
    except OSError:
        out_dir = tempfile.mkdtemp(prefix="tv_oracle_")
    so = os.path.join(out_dir, "libtv_oracle.so")
    if os.path.exists(so) and os.path.getmtime(so) >= max(os.path.getmtime(d) for d in _DEPS):
        return so
    for cc in (["/usr/bin/gcc"], ["gcc"]):
        for extra in (["-fopenmp"], ["-Wno-unknown-pragmas"]):
            try:
                if subprocess.run(cc + _sart._CFLAGS + extra + ["-o", so, _SRC, "-lm"]).returncode == 0:
                    return so
            except OSError:                                    # no such compiler
                pass
    raise RuntimeError("could not compile oracle/tv_oracle.c")


def _load():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
    return _lib


_dp = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def _images(img):
    img = np.array(img, dtype=np.float64, order="C", copy=True)
    if img.ndim == 2:
        img = img[None]
    assert img.shape[1:] == (512, 512), img.shape
    return img


def tv_grad(img, eps=1e-4, flip=True):
    """[B,512,512] or [512,512] image (frame flip) -> [B,512,512] f64 gradient of TV_eps, the same frame."""
    x = _images(img)
    g = np.empty_like(x)
    _load().tv_grad_oracle(_dp(x), _dp(g), ctypes.c_int(x.shape[0]), ctypes.c_int(1 if flip else 0), ctypes.c_double(eps))
    return g


def tv_value(img, eps=1e-4, flip=True):
    """TV_eps of one [512,512] image (frame flip), f64, with the differences taken in the native frame."""
    x = np.asarray(img, np.float64)
    x = x[:, ::-1] if flip else x
    dx = np.zeros_like(x)
    dy = np.zeros_like(x)
    dx[:, :-1] = x[:, 1:] - x[:, :-1]
    dy[:-1, :] = x[1:, :] - x[:-1, :]
    return float(np.sqrt(dx * dx + dy * dy + eps * eps).sum())


def tv_descent(img, steps, step, eps=1e-4, flip=True):
    """`steps` TV steps x <- max(0, x - step g / |g|) on every slice of a [B,512,512] / [512,512] image -> [B,512,512] f64."""
    x = _images(img)
    _load().tv_descent_oracle(_dp(x), ctypes.c_int(x.shape[0]), ctypes.c_int(1 if flip else 0), ctypes.c_int(int(steps)),
                              ctypes.c_double(step), ctypes.c_double(eps))
    return x


def sart(sino, flip=True, iterations=5, subsets=20, relaxation=1.0, history=False, ntv=0, tv_alpha=0.1, tv_eps=1e-4, init="zero",
         x0=None):
    """SART-TV (ipdm_fbp_sart_tv): [B,2000,912] / [2000,912] line integrals (taken as f32) -> [B,512,512] f64 after `iterations`
    sweeps, each followed by `ntv` TV steps of length tv_alpha |x - x_prev|.  init="zero" starts at 0; init="fbp" starts at
    max(0, FBP(sino)) of the fp32 FBP oracle, or at max(0, x0) when x0 ([B,512,512], frame flip) is given.  With history=True also
    [B,iterations,512,512], the iterate after every sweep."""
    sino = np.ascontiguousarray(sino, dtype=np.float32)
    if sino.ndim == 2:
        sino = sino[None]
    assert sino.shape[1:] == (2000, 912), sino.shape
    assert 2000 % subsets == 0 and iterations >= 1 and ntv >= 0 and init in ("zero", "fbp")
    b = sino.shape[0]
    if init == "fbp":
        if x0 is None:
            from . import fbp_oracle
            x0 = fbp_oracle.convert(sino, flip)
        x0 = np.ascontiguousarray(x0, dtype=np.float64).reshape(b, 512, 512)
    else:
        x0 = None
    theta, alpha = _sart._geometry()
    out = np.empty((b, 512, 512), dtype=np.float64)
    hist = np.empty((b, iterations, 512, 512), dtype=np.float64) if history else None
    _load().sart_tv_oracle(sino.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), None if x0 is None else _dp(x0), _dp(out),
                           None if hist is None else _dp(hist), ctypes.c_int(b), ctypes.c_int(1 if flip else 0),
                           ctypes.c_int(int(iterations)), ctypes.c_int(int(subsets)), ctypes.c_double(relaxation), ctypes.c_int(int(ntv)),
                           ctypes.c_double(tv_alpha), ctypes.c_double(tv_eps), _dp(theta), _dp(alpha), ctypes.c_double(_sart.D),
                           ctypes.c_double(_sart.DX))
    return (out, hist) if history else out
