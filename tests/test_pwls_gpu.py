"""GPU: the PWLS penalty (ipdm_fbp_pwls_penalty) and PWLS / OS-SQS (ipdm_fbp_pwls) against their fp64 C restatement
(oracle/pwls_oracle.c), bit-for-bit frame mirroring, determinism and batch invariance, one plan shared by every convertor at
changing batches, the objective's descent with one subset and the low-dose claim with the device operators, and convertor="PWLS" in the progressive pipeline (eager, CUDA graph,
simulate_low_dose)."""
import numpy as np
import pytest
import torch

from conftest import rel_l2
from test_sart_cpu import BODY
from test_sart_gpu import _model

pytestmark = pytest.mark.gpu
# Bounds measured on one B200, with the margin stated next to each.
PENALTY_TOL = 1e-6           # rel-L2 of fp32 grad R and d^R vs fp64 (noisy phantom, both frames): measured 5.5e-8 / 5.3e-8, x18
# rel-L2 of PWLS (2 sweeps, S = 20, dose 0.25, beta 3e4, delta 0.005) vs fp64, both frames: measured 6.4e-7 from the FBP start (x15)
# and 8.7e-7 from 0 (x11); the penalty moves the image by 3.4e-2 / 6.1e-3, far above either
PWLS_ORACLE_TOL = dict(fbp=1e-5, zero=1e-5)
KW = dict(dose=0.25, beta=3e4, delta=0.005)
# the same comparison at the shipped defaults (beta 1e6, delta 2e-4) from the FBP start; see test_pwls_matches_the_oracle_at_the_defaults
DEFAULTS_ORACLE_TOL = 1e-5


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
    noisy = {d: np.maximum(S.add_noise(b0, d, np.random.default_rng(7)), 0).astype(np.float32) for d in (0.25, 0.1)}
    return img, b0.astype(np.float32), noisy


def _dev(a, cuda):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(cuda)


def test_penalty_matches_the_oracle_and_mirrors(plan, cuda):
    import ipdm_pytorch_b200.synthetic as S
    from oracle import pwls_oracle as W
    img = S.rasterize(S.phantom_ellipses(0))
    x = np.maximum(img + 0.01 * np.random.default_rng(3).standard_normal(img.shape), 0).astype(np.float32)
    got = {}
    for flip in (False, True):
        xin = x if not flip else np.ascontiguousarray(x[:, ::-1])
        g, c = plan.pwls_penalty(_dev(xin, cuda)[None].contiguous(), 0.005, flip=flip)
        got[flip] = (g.cpu().numpy()[0], c.cpu().numpy()[0])
        _, wg, wc = W.penalty(xin, 0.005, flip)
        eg, ec = rel_l2(got[flip][0], wg[0]), rel_l2(got[flip][1], wc[0])
        print(f"penalty vs fp64 oracle (flip={int(flip)}): grad rel-L2 {eg:.2e}, curvature rel-L2 {ec:.2e}")
        assert eg <= PENALTY_TOL and ec <= PENALTY_TOL, (eg, ec)
    assert np.array_equal(got[True][0], got[False][0][:, ::-1]) and np.array_equal(got[True][1], got[False][1][:, ::-1])
    for bad in (0.0, "0.1"):
        with pytest.raises(ValueError):
            plan.pwls_penalty(_dev(x, cuda)[None].contiguous(), bad)


@pytest.mark.parametrize("init", ["zero", "fbp"])
@pytest.mark.parametrize("flip", [True, False])
def test_pwls_matches_the_oracle(plan, phantom, cuda, flip, init):
    """The fp64 run starts from the device's own FBP image (init="fbp"), so the comparison holds PWLS, not FBP, to fp64."""
    from oracle import pwls_oracle as W
    b = phantom[2][0.25] if flip else np.ascontiguousarray(phantom[2][0.25][:, ::-1])
    bd = _dev(b, cuda)[None]
    kw = dict(iterations=2, subsets=20, init=init, **KW)
    got = plan.pwls(bd, flip=flip, **kw).cpu().numpy()[0]
    x0 = plan.forward(bd, flip=flip).cpu().numpy() if init == "fbp" else None
    want = W.pwls(b, flip=flip, x0=x0, **kw)[0]
    wls = W.pwls(b, flip=flip, x0=x0, **dict(kw, beta=0.0))[0]
    err = rel_l2(got, want)
    print(f"PWLS vs fp64 oracle (flip={int(flip)}, init={init}): rel-L2 {err:.2e}; the penalty moved the image by {rel_l2(want, wls):.2e}")
    assert err <= PWLS_ORACLE_TOL[init], err
    assert rel_l2(want, wls) > 300 * PWLS_ORACLE_TOL[init]


def test_pwls_matches_the_oracle_at_the_defaults(plan, phantom, cuda):
    """The shipped delta puts the penalty in its near-TV regime (|x_j - x_k| >> delta at most edges), both frames, from the FBP
    start the defaults recommend.  There the problem is well conditioned: in fp64 alone, a 1e-6 relative perturbation of the
    sinogram moves the 2-sweep image by 2.1e-7.  From 0 it is not (6.2e-3 for the same perturbation, against 6.8e-2 that the
    penalty moves the image), so the zero start is held to fp64 at the settings of test_pwls_matches_the_oracle instead."""
    from ipdm_pytorch_b200 import engine
    from oracle import pwls_oracle as W
    kw = dict(iterations=2, subsets=20, init="fbp", dose=0.25, **engine.PWLS_DEFAULTS)
    for flip in (True, False):
        b = phantom[2][0.25] if flip else np.ascontiguousarray(phantom[2][0.25][:, ::-1])
        bd = _dev(b, cuda)[None]
        got = plan.pwls(bd, flip=flip, **kw).cpu().numpy()[0]
        x0 = plan.forward(bd, flip=flip).cpu().numpy()
        want = W.pwls(b, flip=flip, x0=x0, **kw)[0]
        wls = W.pwls(b, flip=flip, x0=x0, **dict(kw, beta=0.0))[0]
        err = rel_l2(got, want)
        print(f"PWLS at the defaults vs fp64 oracle (flip={int(flip)}): rel-L2 {err:.2e}; the penalty moved the image by "
              f"{rel_l2(want, wls):.2e}")
        assert err <= DEFAULTS_ORACLE_TOL, err
        assert rel_l2(want, wls) > 1000 * DEFAULTS_ORACLE_TOL


def test_pwls_mirrors_and_is_deterministic_and_batch_invariant(plan, phantom, cuda):
    b = _dev(phantom[2][0.25], cuda)
    kw = dict(iterations=1, subsets=20, init="fbp", **KW)
    one = plan.pwls(b[None], flip=True, **kw)
    mirrored = plan.pwls(b.flip(-1)[None].contiguous(), flip=False, **kw)
    assert torch.equal(one, mirrored.flip(-1))
    sb = torch.stack([b * (1 + 0.05 * k) for k in range(16)])
    s1 = plan.pwls(sb, **kw)
    assert torch.equal(s1, plan.pwls(sb, **kw))
    for k in (0, 9, 15):
        assert torch.equal(plan.pwls(sb[k:k + 1].contiguous(), **kw)[0], s1[k]), k
    for bad in (dict(dose=0.0), dict(beta=-1.0), dict(delta=float("nan")), dict(init="x"), dict(subsets=7)):
        with pytest.raises(ValueError):
            plan.pwls(sb[:1].contiguous(), **dict(kw, **bad))


def test_one_plan_serves_every_convertor_at_growing_and_shrinking_batches(phantom, cuda):
    """A plan's per-call scratch is laid out for each call's batch and kept across convertors: calls interleaved on one plan, at
    batches that grow and shrink, give bit for bit what the same call gives on a fresh plan."""
    from ipdm_pytorch_b200 import engine
    b = _dev(phantom[2][0.25], cuda)
    sb = torch.stack([b * (1 + 0.05 * k) for k in range(16)])
    x = torch.rand(1, 512, 512, device=cuda, generator=torch.Generator(device=cuda).manual_seed(5))
    sart_tv = dict(ntv=20, tv_alpha=0.2, init="fbp")                # the recommended SART-TV setting
    calls = [lambda p: p.sart(sb, **sart_tv),
             lambda p: p.pwls(sb[:4], init="fbp", **engine.PWLS_DEFAULTS),
             lambda p: p.tv_descent(x.clone(), 5, 1.0),
             lambda p: p.sart(sb[:2]),
             lambda p: p.sart(sb[:3], **sart_tv),
             lambda p: p.pwls(sb, **engine.PWLS_DEFAULTS)]
    shared = engine.FBPPlan()
    for k, call in enumerate(calls):
        assert torch.equal(call(shared), call(engine.FBPPlan())), k


@pytest.mark.parametrize("beta", [0.0, 3e4])
def test_objective_falls_at_every_sweep_on_the_device(plan, phantom, cuda, beta):
    """S = 1: every update minimises a separable majoriser of Phi, so Phi (fp64, of the device's iterates) falls at every sweep.
    Measured on one B200: 4.0586e9, 1.3002e9, 5.3760e8, 2.7752e8 (beta = 0) and 4.0586e9, 1.4761e9, 6.3839e8, 3.2178e8 (beta = 3e4);
    the beta = 0 values are within 4e-7 of the fp64 iterates' own."""
    from oracle import pwls_oracle as W
    b = phantom[2][0.25]
    bd = _dev(b, cuda)[None]
    phi = [float(W.objective(b, np.zeros((512, 512)), 0.25, beta, 0.005)[0])]
    for k in (1, 2, 3):
        x = plan.pwls(bd, iterations=k, subsets=1, dose=0.25, beta=beta, delta=0.005).cpu().numpy()
        phi.append(float(W.objective(b, x, 0.25, beta, 0.005)[0]))
    print(f"device Phi with S = 1, beta = {beta:g}:", " ".join(f"{p:.8g}" for p in phi))
    assert all(p1 < p0 for p0, p1 in zip(phi, phi[1:])), phi


@pytest.mark.parametrize("dose", [0.25, 0.1])
def test_pwls_beats_sart_and_fbp_on_the_device(plan, phantom, cuda, dose):
    """The CPU test's low-dose claim with the device operators, on the same noisy sinograms (default_rng(7))."""
    from ipdm_pytorch_b200 import engine
    img, _, noisy = phantom
    bd = _dev(noisy[dose], cuda)[None]
    body = torch.from_numpy(img > BODY).to(cuda)
    ref = _dev(img, cuda)
    rmse = lambda x: float(((x[0] - ref)[body] ** 2).mean().sqrt())
    got = rmse(plan.pwls(bd, dose=dose, init="fbp", **engine.PWLS_DEFAULTS))
    plain, fbp = rmse(plan.sart(bd)), rmse(plan.forward(bd))
    print(f"device, dose {dose}: PWLS {got:.5f} | SART {plain:.5f} | FBP {fbp:.5f} 1/cm")
    assert got < plain and got < fbp


PWLS_OPTS = dict(convertor="PWLS", sart_iterations=2, sart_subsets=20, sart_init="fbp")


def _pwls_kw(o, dose=None):
    return dict(iterations=o.sart_iterations, subsets=o.sart_subsets, dose=o.dose if dose is None else dose, beta=o.pwls_beta,
                delta=o.pwls_delta, init=o.sart_init)


def test_progressive_pass_with_pwls(cuda, tmp_path):
    import ipdm_pytorch_b200.synthetic as S
    model = _model(tmp_path, PWLS_OPTS)
    ld = torch.from_numpy(np.stack([S.make_slice(s)[0] for s in (0, 1)]))[:, None]
    model.data_sample_load(ldct=None, ldproj=ld, fdproj=None, fdct=None)
    out = model.progressive_denoiser(save_proj_state=True)
    assert torch.isfinite(out).all()
    last = torch.from_numpy(model.proj_denoise_result[-1][:, 0]).to(cuda).float()
    last = last * 10 if model.opt.clip_proj else last
    want = model._fbp.pwls_device(last, **_pwls_kw(model.opt)).cpu().numpy()
    rec = model.proj_denoise_convert2img_result["iter_1"][:, 0]
    assert np.isfinite(rec).all() and np.array_equal(rec, want)
    sart = model._fbp.sart_device(last, iterations=2, subsets=20, init="fbp").cpu().numpy()
    assert not np.array_equal(rec, sart)


def test_cuda_graph_replay_equals_eager_with_pwls(cuda, tmp_path):
    import ipdm_pytorch_b200.synthetic as S
    model = _model(tmp_path, PWLS_OPTS)
    ld = torch.from_numpy(np.stack([S.make_slice(s)[0] for s in (0, 1)]))[:, None]
    model.data_sample_load(ldct=None, ldproj=ld, fdproj=None, fdct=None)
    eager1 = model.progressive_denoiser()
    eager2 = model.progressive_denoiser()
    model.update_opt(dict(cuda_graph=True, noise_seed=5))
    g1 = model.progressive_denoiser()
    g2 = model.progressive_denoiser()
    assert torch.equal(g1, eager1) and torch.equal(g2, eager2) and not torch.equal(g1, g2)
    model.update_opt(dict(pwls_beta=1e4, noise_seed=5))          # a PWLS option re-captures
    assert model._graph is None
    g3 = model.progressive_denoiser()
    model.update_opt(dict(cuda_graph=False, noise_seed=5))
    assert torch.equal(g3, model.progressive_denoiser()) and not torch.equal(g3, g1)


def test_simulate_low_dose_converts_at_its_own_dose(cuda, tmp_path):
    import ipdm_pytorch_b200.synthetic as S
    model = _model(tmp_path, PWLS_OPTS)
    fd = torch.from_numpy(S.rasterize(S.phantom_ellipses(1)))[None, None].to(cuda)
    assert model.opt.dose != 0.1
    ldproj, ldct = model.simulate_low_dose(fd, dose=0.1)
    s = ldproj[:, 0] * 10 if model.opt.clip_proj else ldproj[:, 0]
    want = model._fbp.pwls_device(s, **_pwls_kw(model.opt, 0.1))
    assert torch.equal(ldct[:, 0], want)
    assert not torch.equal(ldct[:, 0], model._fbp.pwls_device(s, **_pwls_kw(model.opt)))


def test_bad_pwls_options_raise(cuda, tmp_path):
    import ipdm_pytorch_b200.synthetic as S
    model = _model(tmp_path, PWLS_OPTS)
    ld = torch.from_numpy(S.make_slice(0)[0])[None, None]
    model.data_sample_load(ldct=None, ldproj=ld, fdproj=None, fdct=None)
    for bad in (dict(pwls_beta=-1.0), dict(pwls_delta=0.0), dict(dose=0.0), dict(sart_subsets=7), dict(sart_init="ones")):
        model.update_opt(dict(bad, noise_seed=5))
        with pytest.raises(ValueError):
            model.progressive_denoiser()
        with pytest.raises(ValueError):
            model.convertor(np.zeros((2000, 912), np.float32))
        model.update_opt(dict(PWLS_OPTS, pwls_beta=3e4, pwls_delta=0.005, dose=0.25))
    host = model.convertor(S.make_slice(0)[0])
    assert isinstance(host, np.ndarray) and host.shape == (1, 512, 512) and np.isfinite(host).all()
