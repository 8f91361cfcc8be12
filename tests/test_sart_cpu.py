"""CPU: the fp64 C restatement of the adjoint projector and of ordered-subset SART (oracle/sart_oracle.c) -- the adjoint is the
transpose of the fp64 projector (oracle/project_oracle.c), SART lowers the ray-weighted data residual at every sweep and ends below
FBP's -- and the sart_* options."""
import math

import numpy as np
import pytest

DOT_TOL = 1e-12                # |<Ax, y> - <x, A^T y>| / (|Ax| |y|): measured 0 / 8.6e-18 (16 views, flip 1 / 0) and 6.6e-19 /
                               # 2.2e-19 (all views) in fp64; far below this bound, which only reordered fp64 sums could approach
BODY = 0.05                    # 1/cm: the body mask of test_project_cpu.py


def weighted_residual(sino, img, flip=True):
    """|(b - A x) / sqrt(R)| over the rays with R = A 1 > 0 (fp64 projector, x taken as f32): the norm SART minimises."""
    from oracle import project_oracle as P
    R = P.project(np.ones((512, 512), np.float32), flip)[0]
    m = R > 0
    r = np.asarray(sino, np.float64) - P.project(np.asarray(img, np.float32), flip)[0]
    return float(np.linalg.norm(r[m] / np.sqrt(R[m])))


@pytest.fixture(scope="module")
def phantom():
    import ipdm_pytorch_b200.synthetic as S
    from oracle import project_oracle as P
    img = S.rasterize(S.phantom_ellipses(0))
    return img, P.project(img)[0].astype(np.float32)          # noise-free Joseph projection of the raster, flip = 1


@pytest.mark.parametrize("flip", [True, False])
@pytest.mark.parametrize("subset", [True, False], ids=["16views", "allviews"])
def test_oracle_adjoint_is_the_transpose_of_the_oracle_projector(flip, subset):
    from oracle import project_oracle as P, sart_oracle as Q
    rng = np.random.default_rng(1 + 2 * int(flip) + int(subset))
    views = np.arange(0, 2000, 125) + 7 if subset else None
    x = rng.random((512, 512)).astype(np.float32)
    y = rng.standard_normal((16 if subset else 2000, 912))
    ax = P.project(x, flip, views)[0]
    aty = Q.adjoint(y, flip, views)[0]
    err = abs(float((ax * y).sum()) - float((x * aty).sum())) / (np.linalg.norm(ax) * np.linalg.norm(y))
    print(f"oracle dot test (flip={int(flip)}, {'16 views' if subset else 'all views'}): {err:.2e}")
    assert err <= DOT_TOL, err


def test_visit_order():
    """Subsets are visited at the step p in [1, S) coprime to S closest to 0.382 S (smaller on a tie), p = 1 when S <= 2."""
    from oracle import sart_oracle as Q
    def step(S):
        if S <= 2:
            return 1
        return min((q for q in range(1, S) if math.gcd(q, S) == 1), key=lambda q: (abs(q - 0.382 * S), q))
    for S in (1, 2, 4, 5, 8, 10, 16, 20, 25, 40, 50, 80, 100, 125, 200, 400, 500, 1000, 2000):
        assert Q.visit_step(S) == step(S), S
    assert [Q.visit_step(S) for S in (20, 100)] == [7, 39]


def test_oracle_sart_converges_below_fbp(phantom):
    """SART at the default options on noise-free data.  Measured with S = 100, 5 sweeps, lambda = 1: weighted residual 8.26, 3.77,
    2.43, 1.81, 1.45 after sweeps 1..5 against 4.58 for the FBP oracle; body RMSE 0.0180, 0.0118, 0.0094, 0.0080, 0.0070 1/cm
    against 0.0043 for FBP (x0 = 0: 5 sweeps have not reached the FBP image's fine detail, while the data fit is 3x closer)."""
    from Config.default_config import default_cfg
    from oracle import fbp_oracle, sart_oracle as Q
    img, b = phantom
    o = default_cfg([])
    _, hist = Q.sart(b, True, o.sart_iterations, o.sart_subsets, o.sart_relaxation, history=True)
    res = [weighted_residual(b, h) for h in hist[0]]
    fbp = fbp_oracle.convert(b[None])[0]
    body = img > BODY
    rmse = lambda r: float(np.sqrt(((r - img)[body] ** 2).mean()))
    print("weighted residual per sweep:", " ".join(f"{r:.3f}" for r in res), f"| FBP {weighted_residual(b, fbp):.3f}")
    print("body RMSE per sweep:", " ".join(f"{rmse(h):.5f}" for h in hist[0]), f"| FBP {rmse(fbp):.5f} 1/cm")
    assert all(b1 < a1 for a1, b1 in zip(res, res[1:])), res
    assert res[-1] < weighted_residual(b, fbp)
    assert float(hist.min()) >= 0.0


def test_sart_options_parse():
    from Config.default_config import default_cfg
    from ipdm_pytorch_b200 import engine
    o = default_cfg([])
    assert (o.sart_iterations, o.sart_subsets, o.sart_relaxation) == (5, 100, 1.0)
    assert engine.SART_DEFAULTS == dict(iterations=o.sart_iterations, subsets=o.sart_subsets, relaxation=o.sart_relaxation)
    o = default_cfg(["--sart_iterations", "3", "--sart_subsets", "10", "--sart_relaxation", "0.5"])
    assert (o.sart_iterations, o.sart_subsets, o.sart_relaxation) == (3, 10, 0.5)
    assert o.convertor == "TV" and o.ntv == 0                  # the reference's defaults are untouched


@pytest.mark.parametrize("bad", [dict(iterations=0), dict(iterations=1.5), dict(subsets=7), dict(subsets=0), dict(subsets=4000),
                                 dict(relaxation=0.0), dict(relaxation=2.0), dict(relaxation=float("nan")), dict(relaxation=True),
                                 dict(relaxation="0.5")])
def test_sart_argument_checks(bad):
    from ipdm_pytorch_b200 import engine
    args = dict(engine.SART_DEFAULTS, **bad)
    with pytest.raises(ValueError):
        engine.FBPPlan.check_sart_args(**args)
