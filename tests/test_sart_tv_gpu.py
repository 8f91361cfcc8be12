"""GPU: the TV steps (ipdm_fbp_tv_descent) and SART-TV (ipdm_fbp_sart_tv) against their fp64 C restatement (oracle/tv_oracle.c),
bit-for-bit frame mirroring, determinism and batch invariance, the low-dose convergence claim with the device operators, and
convertor="SART" with TV steps in the progressive pipeline (eager and CUDA graph)."""
import numpy as np
import pytest
import torch

from conftest import rel_l2
from test_sart_cpu import BODY
from test_sart_gpu import _model

pytestmark = pytest.mark.gpu
# Bounds measured on one B200, with the margin stated next to each.
TV_ORACLE_TOL = 1e-5         # rel-L2 of 5 fp32 TV steps vs fp64 (noisy phantom, both frames): measured 4.8e-7, x20
# rel-L2 of SART-TV (2 sweeps, S = 20, ntv = 5, dose 0.25) vs fp64, both frames, per start.  From the FBP start: measured 4.3e-7, x12.
# From 0 the first sweep's image is smooth, with neighbour differences near eps over wide areas, where g = grad TV_eps changes by
# up to 1/eps per unit of x; the first TV steps are long (t = 0.2 |x1|), so rounding is amplified: in fp64 alone, a 1e-6 relative
# perturbation of the sinogram moves plain SART by 3.5e-7 and SART-TV from 0 by 5.2e-4 (from the FBP start by 7.1e-7).  Measured
# 9.3e-4 (fp32 vs fp64, ~1400 x SART's own 7e-7), x3.2; still well below the 2.9e-2 the TV steps move the image.
SART_TV_ORACLE_TOL = dict(fbp=5e-6, zero=3e-3)
RECOMMENDED = dict(ntv=20, tv_alpha=0.2, init="fbp")


@pytest.fixture(scope="module")
def plan(cuda):
    from ipdm_pytorch_b200 import engine
    return engine.FBPPlan(max_batch=16)


@pytest.fixture(scope="module")
def phantom():
    import ipdm_pytorch_b200.synthetic as S
    from oracle import project_oracle as P
    img = S.rasterize(S.phantom_ellipses(0))
    b0 = P.project(img)[0]
    noisy = np.maximum(S.add_noise(b0, 0.25, np.random.default_rng(7)), 0).astype(np.float32)
    return img, b0.astype(np.float32), noisy


def _dev(a, cuda):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(cuda)


def _noisy_image(seed=3):
    import ipdm_pytorch_b200.synthetic as S
    img = S.rasterize(S.phantom_ellipses(0))
    rng = np.random.default_rng(seed)
    return np.maximum(img + 0.01 * rng.standard_normal(img.shape), 0).astype(np.float32)


def test_tv_descent_matches_the_oracle_and_mirrors(plan, cuda):
    from oracle import tv_oracle as T
    x = _noisy_image()
    got = {}
    for flip in (False, True):
        xin = x if not flip else np.ascontiguousarray(x[:, ::-1])
        d = _dev(xin, cuda)[None].contiguous()
        got[flip] = plan.tv_descent(d, 5, 2.0, 1e-4, flip=flip).cpu().numpy()[0]
        want = T.tv_descent(xin, 5, 2.0, 1e-4, flip=flip)[0]
        err = rel_l2(got[flip], want)
        print(f"TV steps vs fp64 oracle (flip={int(flip)}): rel-L2 {err:.2e}, moved {rel_l2(want, xin):.2e}")
        assert err <= TV_ORACLE_TOL, err
        assert rel_l2(want, xin) > 100 * TV_ORACLE_TOL            # the steps did something
    assert np.array_equal(got[True], got[False][:, ::-1])
    zero = torch.zeros(1, 512, 512, device=cuda)                   # |g| = 0: no change
    assert float(plan.tv_descent(zero, 3, 1.0).abs().max()) == 0.0


def test_tv_and_sart_tv_determinism_and_batch_invariance(plan, phantom, cuda):
    g = torch.Generator(device=cuda).manual_seed(9)
    x = torch.rand(16, 512, 512, device=cuda, generator=g)
    a1 = plan.tv_descent(x.clone(), 4, 3.0)
    assert torch.equal(a1, plan.tv_descent(x.clone(), 4, 3.0))
    for k in (0, 7, 15):
        assert torch.equal(plan.tv_descent(x[k:k + 1].clone(), 4, 3.0)[0], a1[k]), k
    b = _dev(phantom[2], cuda)
    sb = torch.stack([b * (1 + 0.05 * k) for k in range(16)])
    kw = dict(iterations=1, subsets=20, ntv=5, tv_alpha=0.2, init="fbp")
    s1 = plan.sart(sb, **kw)
    assert torch.equal(s1, plan.sart(sb, **kw))
    for k in (0, 9, 15):
        assert torch.equal(plan.sart(sb[k:k + 1].contiguous(), **kw)[0], s1[k]), k
    for bad in (dict(ntv=-1), dict(tv_alpha=0.0), dict(tv_eps=float("nan")), dict(init="x")):
        with pytest.raises(ValueError):
            plan.sart(sb[:1].contiguous(), **bad)
    for bad in (dict(steps=-1), dict(step=float("inf")), dict(step=True), dict(eps=0.0)):
        with pytest.raises(ValueError):
            plan.tv_descent(x[:1].clone(), **dict(dict(steps=1, step=1.0, eps=1e-4), **bad))


@pytest.mark.parametrize("init", ["zero", "fbp"])
@pytest.mark.parametrize("flip", [True, False])
def test_sart_tv_matches_the_oracle(plan, phantom, cuda, flip, init):
    """The fp64 run starts from the device's own FBP image (init="fbp"), so the comparison holds SART-TV, not FBP, to fp64."""
    from oracle import tv_oracle as T
    b = phantom[2] if flip else np.ascontiguousarray(phantom[2][:, ::-1])
    bd = _dev(b, cuda)[None]
    kw = dict(iterations=2, subsets=20, relaxation=1.0, ntv=5, tv_alpha=0.2, tv_eps=1e-4, init=init)
    got = plan.sart(bd, flip=flip, **kw).cpu().numpy()[0]
    x0 = plan.forward(bd, flip=flip).cpu().numpy() if init == "fbp" else None
    want = T.sart(b, flip=flip, x0=x0, **kw)[0]
    plain = T.sart(b, flip=flip, **dict(kw, ntv=0))[0]
    err = rel_l2(got, want)
    print(f"SART-TV vs fp64 oracle (flip={int(flip)}, init={init}): rel-L2 {err:.2e}; TV moved the image by {rel_l2(want, plain):.2e}")
    assert err <= SART_TV_ORACLE_TOL[init], err
    assert rel_l2(want, plain) > 1e-2                            # the TV steps matter: measured 2.9e-2 (zero), 3.1e-2 (fbp)


def test_sart_tv_beats_sart_and_fbp_on_the_device(plan, phantom, cuda):
    """The CPU test's low-dose claim with the device operators, on the same noisy sinogram (dose 0.25, default_rng(7))."""
    from ipdm_pytorch_b200 import engine
    img, _, noisy = phantom
    bd = _dev(noisy, cuda)[None]
    body = torch.from_numpy(img > BODY).to(cuda)
    ref = _dev(img, cuda)
    rmse = lambda x: float(((x[0] - ref)[body] ** 2).mean().sqrt())
    d = engine.SART_DEFAULTS
    tv = [rmse(plan.sart(bd, **dict(d, iterations=k), **RECOMMENDED)) for k in range(1, d["iterations"] + 1)]
    plain, fbp = rmse(plan.sart(bd)), rmse(plan.forward(bd))
    print("device SART-TV body RMSE per sweep:", " ".join(f"{r:.5f}" for r in tv), f"| SART {plain:.5f} | FBP {fbp:.5f} 1/cm")
    assert tv[-1] < plain and tv[-1] < fbp
    assert all(b1 < a1 for a1, b1 in zip(tv, tv[1:])), tv


TV_OPTS = dict(sart_iterations=2, sart_subsets=20, ntv=5, tv_alpha=0.2, sart_init="fbp")


def test_progressive_pass_with_sart_tv(cuda, tmp_path):
    import ipdm_pytorch_b200.synthetic as S
    model = _model(tmp_path, TV_OPTS)
    ld = torch.from_numpy(np.stack([S.make_slice(s)[0] for s in (0, 1)]))[:, None]
    model.data_sample_load(ldct=None, ldproj=ld, fdproj=None, fdct=None)
    out = model.progressive_denoiser(save_proj_state=True)
    assert torch.isfinite(out).all()
    last = torch.from_numpy(model.proj_denoise_result[-1][:, 0]).to(cuda).float()
    want = model._fbp.sart_device(last, iterations=2, subsets=20, ntv=5, tv_alpha=0.2, tv_eps=1e-4, init="fbp").cpu().numpy()
    rec = model.proj_denoise_convert2img_result["iter_1"][:, 0]
    assert np.isfinite(rec).all() and np.array_equal(rec, want)
    plain = model._fbp.sart_device(last, iterations=2, subsets=20).cpu().numpy()
    assert not np.array_equal(rec, plain)


def test_cuda_graph_replay_equals_eager_with_sart_tv(cuda, tmp_path):
    import ipdm_pytorch_b200.synthetic as S
    model = _model(tmp_path, TV_OPTS)
    ld = torch.from_numpy(np.stack([S.make_slice(s)[0] for s in (0, 1)]))[:, None]
    model.data_sample_load(ldct=None, ldproj=ld, fdproj=None, fdct=None)
    eager1 = model.progressive_denoiser()
    eager2 = model.progressive_denoiser()
    model.update_opt(dict(cuda_graph=True, noise_seed=5))
    g1 = model.progressive_denoiser()
    g2 = model.progressive_denoiser()
    assert torch.equal(g1, eager1) and torch.equal(g2, eager2) and not torch.equal(g1, g2)
    model.update_opt(dict(ntv=3, noise_seed=5))                   # a TV option re-captures
    assert model._graph is None
    g3 = model.progressive_denoiser()
    model.update_opt(dict(cuda_graph=False, noise_seed=5))
    assert torch.equal(g3, model.progressive_denoiser()) and not torch.equal(g3, g1)


def test_bad_sart_tv_options_raise(cuda, tmp_path):
    import ipdm_pytorch_b200.synthetic as S
    model = _model(tmp_path, TV_OPTS)
    ld = torch.from_numpy(S.make_slice(0)[0])[None, None]
    model.data_sample_load(ldct=None, ldproj=ld, fdproj=None, fdct=None)
    for bad in (dict(ntv=-2), dict(tv_alpha=0.0), dict(tv_eps=-1e-4), dict(sart_init="ones")):
        model.update_opt(dict(bad, noise_seed=5))
        with pytest.raises(ValueError):
            model.progressive_denoiser()
        with pytest.raises(ValueError):
            model.convertor(np.zeros((2000, 912), np.float32))
        model.update_opt(dict(TV_OPTS, tv_eps=1e-4))
    host = model.convertor(S.make_slice(0)[0])
    assert isinstance(host, np.ndarray) and host.shape == (1, 512, 512) and np.isfinite(host).all()
