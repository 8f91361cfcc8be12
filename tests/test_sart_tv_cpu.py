"""CPU: the fp64 C restatement of the TV steps and of SART-TV (oracle/tv_oracle.c) -- the TV gradient is the gradient of TV_eps,
SART-TV without TV steps is the plain SART reference, and the recommended SART-TV setting beats plain SART and FBP at dose 0.25 --
and the TV options of convertor="SART"."""
import numpy as np
import pytest

from test_sart_cpu import BODY

FD_TOL = 2e-6                  # |g - central difference| / max |g|: measured 2.5e-9 (random, eps 1e-2) and 1.3e-7 .. 2.5e-7 (phantom,
                               # eps 1e-3, flat regions where n ~ eps) with h = 1e-5; the O((h / eps)^2) truncation term dominates, x8
RECOMMENDED = dict(ntv=20, tv_alpha=0.2, init="fbp")


def _terms(x, eps):
    """sqrt(dx^2 + dy^2 + eps^2) per pixel of a native image: TV_eps is their sum."""
    dx = np.zeros_like(x)
    dy = np.zeros_like(x)
    dx[:, :-1] = x[:, 1:] - x[:, :-1]
    dy[:-1, :] = x[1:, :] - x[:-1, :]
    return np.sqrt(dx * dx + dy * dy + eps * eps)


def _fd_error(x, eps, flip, pixels, h=1e-5):
    """Worst |g - (TV(x + h e) - TV(x - h e)) / 2h| over `pixels`, relative to max |g|.  Only the terms of a pixel's 3 x 3
    neighbourhood change, so the difference is summed from the per-term differences (no cancellation against the whole sum)."""
    from oracle import tv_oracle as T
    g = T.tv_grad(x, eps, flip)[0]
    nat = lambda a: a[:, ::-1] if flip else a
    worst = 0.0
    for i, j in pixels:
        e = np.zeros_like(x)
        e[i, j] = h
        fd = float((_terms(nat(x + e), eps) - _terms(nat(x - e), eps)).sum()) / (2 * h)
        worst = max(worst, abs(fd - g[i, j]))
    return worst / float(np.abs(g).max())


def _pixels(rng):
    edges = [(0, 0), (0, 511), (511, 0), (511, 511), (0, 200), (511, 300), (200, 0), (300, 511), (1, 1), (510, 510)]
    return edges + [tuple(int(v) for v in p) for p in rng.integers(0, 512, (30, 2))]


@pytest.mark.parametrize("flip", [True, False])
def test_oracle_tv_gradient_matches_finite_differences(flip):
    import ipdm_pytorch_b200.synthetic as S
    rng = np.random.default_rng(11)
    x = rng.random((512, 512))
    e_rand = _fd_error(x, 1e-2, flip, _pixels(rng))
    ph = S.rasterize(S.phantom_ellipses(0)).astype(np.float64)
    # the phantom's edges, where the gradient is largest, plus the random and border pixels
    gi, gj = np.nonzero(np.abs(np.diff(ph, axis=1)) > 0.01)
    pick = rng.choice(gi.size, 30, replace=False)
    e_ph = _fd_error(ph, 1e-3, flip, _pixels(rng) + list(zip(gi[pick].tolist(), gj[pick].tolist())))
    print(f"TV gradient vs central differences (flip={int(flip)}): random {e_rand:.2e}, phantom {e_ph:.2e}")
    assert e_rand <= FD_TOL and e_ph <= FD_TOL, (e_rand, e_ph)


def test_oracle_tv_descent_lowers_tv_and_mirrors():
    from oracle import tv_oracle as T
    rng = np.random.default_rng(5)
    x = np.clip(0.2 + 0.02 * rng.standard_normal((512, 512)), 0, None)
    y = T.tv_descent(x, 3, 0.5, 1e-4, flip=False)[0]
    assert T.tv_value(y, 1e-4, False) < T.tv_value(x, 1e-4, False)
    assert float(np.linalg.norm(y - x)) <= 3 * 0.5 * (1 + 1e-12)     # each step moves by at most t (the clamp only shortens it)
    ym = T.tv_descent(np.ascontiguousarray(x[:, ::-1]), 3, 0.5, 1e-4, flip=True)[0]
    assert np.array_equal(ym, y[:, ::-1])
    assert np.array_equal(T.tv_descent(x, 0, 0.5)[0], x)


def test_oracle_sart_tv_without_tv_is_plain_sart():
    """ntv = 0 from the zero start is the plain SART reference (oracle/sart_oracle.c), exactly, in both frames."""
    import ipdm_pytorch_b200.synthetic as S
    from oracle import project_oracle as P, sart_oracle as Q, tv_oracle as T
    b = P.project(S.rasterize(S.phantom_ellipses(0)))[0].astype(np.float32)
    for flip in (True, False):
        bb = b if flip else np.ascontiguousarray(b[:, ::-1])
        assert np.array_equal(T.sart(bb, flip, 2, 20, 1.0, ntv=0, init="zero"), Q.sart(bb, flip, 2, 20, 1.0)), flip


def test_oracle_sart_tv_beats_sart_and_fbp_at_low_dose():
    """Dose 0.25 (synthetic.add_noise, default_rng(7), clipped at 0), S = 100, 5 sweeps.  Measured body RMSE after sweep 5:
    plain SART 0.0097, SART-TV at the recommended setting 0.0039, FBP 0.0150 1/cm."""
    import ipdm_pytorch_b200.synthetic as S
    from Config.default_config import default_cfg
    from oracle import fbp_oracle, project_oracle as P, sart_oracle as Q, tv_oracle as T
    img = S.rasterize(S.phantom_ellipses(0))
    b = np.maximum(S.add_noise(P.project(img)[0], 0.25, np.random.default_rng(7)), 0).astype(np.float32)
    o = default_cfg([])
    body = img > BODY
    rmse = lambda r: float(np.sqrt(((r - img)[body] ** 2).mean()))
    fbp = fbp_oracle.convert(b[None])[0]
    plain = Q.sart(b, True, o.sart_iterations, o.sart_subsets, o.sart_relaxation)[0]
    _, hist = T.sart(b, True, o.sart_iterations, o.sart_subsets, o.sart_relaxation, history=True, tv_eps=o.tv_eps, x0=fbp[None],
                     **RECOMMENDED)
    tv = [rmse(h) for h in hist[0]]
    print("SART-TV body RMSE per sweep:", " ".join(f"{r:.5f}" for r in tv), f"| SART {rmse(plain):.5f} | FBP {rmse(fbp):.5f} 1/cm")
    assert tv[-1] < rmse(plain) and tv[-1] < rmse(fbp)
    assert all(b1 < a1 for a1, b1 in zip(tv, tv[1:])), tv
    assert float(hist.min()) >= 0.0


def test_sart_tv_options_parse():
    from Config.default_config import default_cfg
    from ipdm_pytorch_b200 import engine
    o = default_cfg([])
    assert (o.ntv, o.tv_alpha, o.tv_eps, o.sart_init) == (0, 0.2, 1e-4, "zero")
    assert engine.SART_TV_DEFAULTS == dict(ntv=o.ntv, tv_alpha=o.tv_alpha, tv_eps=o.tv_eps, init=o.sart_init)
    o = default_cfg(["--ntv", "20", "--tv_alpha", "0.1", "--tv_eps", "1e-3", "--sart_init", "fbp"])
    assert (o.ntv, o.tv_alpha, o.tv_eps, o.sart_init) == (20, 0.1, 1e-3, "fbp")
    assert o.convertor == "TV" and default_cfg([]).ntv == 0    # the reference's defaults are untouched


@pytest.mark.parametrize("bad", [dict(ntv=-1), dict(ntv=2.5), dict(ntv=True), dict(ntv="3"), dict(tv_alpha=0.0), dict(tv_alpha=-0.1),
                                 dict(tv_alpha=float("inf")), dict(tv_alpha=float("nan")), dict(tv_eps=0.0), dict(tv_eps=float("nan")),
                                 dict(init="FBP"), dict(init=None)])
def test_sart_tv_argument_checks(bad):
    from ipdm_pytorch_b200 import engine
    args = dict(engine.SART_TV_DEFAULTS, **bad)
    with pytest.raises(ValueError):
        engine.FBPPlan.check_tv_args(**args)
    with pytest.raises(ValueError):
        engine.FBPPlan.check_sart_args(**args)
    with pytest.raises(ValueError):
        engine.FBPPlan.check_sart_args(**engine.SART_DEFAULTS, **args)
    assert engine.FBPPlan.check_tv_args(**engine.SART_TV_DEFAULTS) == (0, 0.2, 1e-4, "zero")
    assert engine.FBPPlan.check_sart_args(**engine.SART_TV_DEFAULTS) == (5, 100, 1.0, 0, 0.2, 1e-4, "zero")
