"""CPU: the fp64 C restatement of the forward projector (oracle/project_oracle.c) against the analytic line integrals of the
phantom, through the FBP oracle, and the factored noise formula of ipdm_low_dose_noise against synthetic.add_noise."""
import numpy as np
import pytest

from conftest import rel_l2

# Bounds measured on the CPU (slice-0 phantom), with the margin stated next to each.
RASTER_VS_ANALYTIC = 4e-3      # measured 2.81e-3 (16-view subset) and 2.95e-3 (all views): x1.4.  The 2x-oversampled raster is
                               # not the ellipses: edges are smeared over a pixel, which sets this distance, not the projector
FBP_BODY_EXCESS = 1e-3         # body RMSE of FBP(projection of the raster) minus that of FBP(analytic): measured 3.6e-4 (0.00427 vs
                               # 0.00391 1/cm), x2.8


@pytest.fixture(scope="module")
def phantom():
    import ipdm_pytorch_b200.synthetic as S
    ell = S.phantom_ellipses(0)
    return ell, S.rasterize(ell)


def test_oracle_projection_of_the_raster_matches_the_analytic_integrals(phantom):
    """16 views 22.5 deg apart (offset by 7 views so that no ray family is axis-aligned): every octant, both dominant axes."""
    import ipdm_pytorch_b200.synthetic as S
    from oracle import project_oracle as P
    ell, img = phantom
    views = np.arange(0, 2000, 125) + 7
    want = S.fan_sinogram(ell, views=S.view_angles()[views])
    got = P.project(img, flip=True, views=views)[0]
    err = rel_l2(got, want)
    print(f"oracle projection of the raster vs analytic line integrals: rel-L2 {err:.3e}")
    assert err < RASTER_VS_ANALYTIC, err
    # flip = 0: native image in, native sinogram out -- the same numbers with both axes reversed
    native = P.project(np.ascontiguousarray(img[:, ::-1]), flip=False, views=views)[0]
    np.testing.assert_array_equal(native[:, ::-1], got)


def test_fbp_of_the_oracle_projection_reconstructs_the_raster(phantom):
    """Frame or orientation mistakes of the projector would reconstruct a mirrored or rotated body."""
    import ipdm_pytorch_b200.synthetic as S
    from oracle import fbp_oracle, project_oracle as P
    ell, img = phantom
    rec_p = fbp_oracle.convert(P.project(img).astype(np.float32))[0]
    rec_a = fbp_oracle.convert(S.fan_sinogram(ell).astype(np.float32))[0]
    body = img > 0.05
    rmse = lambda r: float(np.sqrt(((r - img)[body] ** 2).mean()))
    print(f"body RMSE: FBP(oracle projection) {rmse(rec_p):.5f}, FBP(analytic) {rmse(rec_a):.5f} 1/cm")
    assert rmse(rec_a) < 0.006
    assert rmse(rec_p) < rmse(rec_a) + FBP_BODY_EXCESS


@pytest.mark.parametrize("dose", [0.1, 0.25, 0.5])
def test_factored_noise_formula_equals_add_noise(dose):
    """ipdm_low_dose_noise evaluates p + sqrt(ka e^p (1 + kc e^p)) n with ka = (1-f)/(f N0), kc = (1+f) Ne/(f N0) (csrc/project.cu);
    in fp64 that is synthetic.add_noise (Low_dose_CT_simulate.py:38-44) on the same normals."""
    import ipdm_pytorch_b200.synthetic as S
    p = np.linspace(0.0, 9.0, 4096).reshape(64, 64)
    want = S.add_noise(p, dose, np.random.default_rng(3))
    n = np.random.default_rng(3).standard_normal(p.shape)
    ka, kc = (1 - dose) / (dose * 1.4e5), (1 + dose) * 5.8 / (dose * 1.4e5)
    got = p + np.sqrt(ka * np.exp(p) * (1 + kc * np.exp(p))) * n
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()


def test_simulate_low_dose_option_defaults_off():
    from Config.default_config import default_cfg
    assert default_cfg([]).simulate_low_dose is False
    assert default_cfg(["--simulate_low_dose", "1"]).simulate_low_dose is True
