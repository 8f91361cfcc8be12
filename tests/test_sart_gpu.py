"""GPU: the adjoint projector (ipdm_fbp_project_adjoint) against its fp64 C restatement and bit for bit against the forward
projector's weights, ordered-subset SART (ipdm_fbp_sart) against its fp64 restatement, and convertor="SART" in the progressive
pipeline (eager, CUDA graph, simulate_low_dose evaluation loop)."""
import json
import os

import numpy as np
import pytest
import torch

from conftest import PKG, rel_l2
from test_sart_cpu import BODY

pytestmark = pytest.mark.gpu
# Bounds measured on one B200, with the margin stated next to each.
ADJ_ORACLE_TOL = 1e-5        # rel-L2 of A^T y, fp32 weights and sums vs fp64: measured 1.02e-6 (both frames), x10 (the projector's bound)
DOT_TOL = 1e-6               # |<Ax, y> - <x, A^T y>| / (|Ax| |y|) with fp32 sums: measured 2.0e-10 .. 4.2e-10
ENTRY_TOL = 2e-4             # per-entry |A_gpu - A_fp64| / max of the row.  Not a rounding bound of the sums: fp32 u = u0 + (m - 255.5) g
                             # carries up to ~ulp(512) = 6e-5 of absolute error into an interpolation weight, so a single entry cannot be held
                             # to 1e-6; the bit-for-bit test below holds the adjoint to the projector's own fp32 weights instead
SART_ORACLE_TOL = 1e-5       # rel-L2 of the fp32 SART image vs fp64: measured 7.2e-7 (2 sweeps, S = 20, both frames), 1.4e-6 (1 sweep,
                             # S = 1), x7


@pytest.fixture(scope="module")
def plan(cuda):
    from ipdm_pytorch_b200 import engine
    return engine.FBPPlan(max_batch=16)


@pytest.fixture(scope="module")
def phantom():
    import ipdm_pytorch_b200.synthetic as S
    from oracle import project_oracle as P
    img = S.rasterize(S.phantom_ellipses(0))
    return img, P.project(img)[0].astype(np.float32)


def _dev(a, cuda):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(cuda)


@pytest.mark.parametrize("flip", [True, False])
def test_adjoint_matches_the_oracle(plan, phantom, cuda, flip):
    from oracle import sart_oracle as Q
    y = phantom[1] if flip else np.ascontiguousarray(phantom[1][:, ::-1])
    got = plan.project_adjoint(_dev(y, cuda)[None], flip=flip).cpu().numpy()[0]
    want = Q.adjoint(y, flip=flip)[0]
    err = rel_l2(got, want)
    print(f"adjoint vs fp64 oracle (flip={int(flip)}): rel-L2 {err:.2e}")
    assert err <= ADJ_ORACLE_TOL, err


def _rays():
    """32 rays (v, k) in the sinogram's flip=1 frame: random ones, both fan edges, and views near 45 / 135 deg, where the
    dominant axis switches inside one view."""
    rng = np.random.default_rng(7)
    rays = [(int(v), int(k)) for v, k in zip(rng.integers(0, 2000, 16), rng.integers(0, 912, 16))]
    rays += [(int(v), 0) for v in rng.integers(0, 2000, 3)] + [(int(v), 911) for v in rng.integers(0, 2000, 3)]
    rays += [(v, int(k)) for v, k in zip((249, 250, 251, 252, 749, 750, 751, 1250, 1251, 1750), rng.integers(300, 612, 10))]
    return rays


def test_adjoint_rows_match_the_oracle_entry_by_entry(plan, cuda):
    """A^T e_r is row r of A.  Every entry the fp64 row has above 10 x ENTRY_TOL must be present on the GPU and the other way round
    (a missed candidate ray drops whole entries), and all entries agree to ENTRY_TOL of the row's largest."""
    from oracle import sart_oracle as Q
    rays = _rays()
    y = torch.zeros(len(rays), 2000, 912, device=cuda)
    for n, (v, k) in enumerate(rays):
        y[n, v, k] = 1.0
    rows = plan.project_adjoint(y).cpu().numpy()
    worst, hit = 0.0, 0
    for n, (v, k) in enumerate(rays):
        e = np.zeros((1, 912))
        e[0, k] = 1.0
        want = Q.adjoint(e, flip=True, views=[v])[0]
        got = rows[n].astype(np.float64)
        top = float(want.max())
        if top == 0.0:                                         # a fan-edge ray that misses the grid in this view: an empty row
            assert not got.any(), (v, k)
            continue
        hit += 1
        assert np.all(got[want > 10 * ENTRY_TOL * top] != 0), (v, k)
        assert np.all(want[got > 10 * ENTRY_TOL * top] != 0), (v, k)
        err = float(np.abs(got - want).max()) / top
        worst = max(worst, err)
        assert err <= ENTRY_TOL, (v, k, err)
    print(f"adjoint rows vs fp64 rows ({hit} of {len(rays)} rays touch the grid): worst entry error {worst:.2e} of the row maximum")
    assert hit >= 20


def test_adjoint_entries_are_the_projector_weights_bit_for_bit(plan, cuda):
    """Column p of A from the projector (a one-hot image: each ray's sum has one non-zero term, so it is the weight exactly) against
    entry p of the adjoint's rows for the rays that touch p and their neighbours, which must be exactly 0 where the projector says 0."""
    torch.manual_seed(0)
    for (i, j) in [(0, 0), (3, 508), (255, 256), (100, 31), (400, 470)]:
        e = torch.zeros(1, 512, 512, device=cuda)
        e[0, i, j] = 1.0
        col = plan.project(e)[0]
        hit = torch.nonzero(col).cpu()
        assert hit.shape[0] > 0
        pick = hit[torch.randperm(hit.shape[0])[:24]]
        rays = [(int(v), int(k)) for v, k in pick] + [(int(v), int(min(k + 3, 911))) for v, k in pick[:8]]
        y = torch.zeros(len(rays), 2000, 912, device=cuda)
        for n, (v, k) in enumerate(rays):
            y[n, v, k] = 1.0
        rows = plan.project_adjoint(y)
        got = rows[:, i, j]
        want = torch.stack([col[v, k] for v, k in rays])
        assert torch.equal(got, want), (i, j)


def test_dot_test_on_the_device(plan, cuda):
    g = torch.Generator(device=cuda).manual_seed(3)
    for flip in (True, False):
        x = torch.rand(2, 512, 512, device=cuda, generator=g)
        y = torch.randn(2, 2000, 912, device=cuda, generator=g)
        ax, aty = plan.project(x, flip=flip), plan.project_adjoint(y, flip=flip)
        for b in range(2):
            lhs = float((ax[b].double() * y[b].double()).sum())
            rhs = float((x[b].double() * aty[b].double()).sum())
            err = abs(lhs - rhs) / (float(ax[b].double().norm()) * float(y[b].double().norm()))
            print(f"device dot test (flip={int(flip)}): {err:.2e}")
            assert err <= DOT_TOL, err


def test_determinism_batch_invariance_and_linearity(plan, phantom, cuda):
    g = torch.Generator(device=cuda).manual_seed(4)
    y = torch.randn(16, 2000, 912, device=cuda, generator=g)
    a1, a2 = plan.project_adjoint(y), plan.project_adjoint(y)
    assert torch.equal(a1, a2)
    for k in (0, 5, 15):
        assert torch.equal(plan.project_adjoint(y[k:k + 1].contiguous())[0], a1[k]), k
    assert float(plan.project_adjoint(torch.zeros_like(y[:1])).abs().max()) == 0.0
    lin = plan.project_adjoint((0.5 * y[0] + 2.0 * y[1])[None].contiguous())
    assert rel_l2(lin.cpu().numpy(), (0.5 * a1[0] + 2.0 * a1[1]).cpu().numpy()[None]) < 1e-5
    b = _dev(phantom[1], cuda)
    sb = torch.stack([b * (1 + 0.05 * k) for k in range(16)])
    s1 = plan.sart(sb, iterations=1, subsets=20)
    assert torch.equal(s1, plan.sart(sb, iterations=1, subsets=20))
    for k in (0, 9, 15):
        assert torch.equal(plan.sart(sb[k:k + 1].contiguous(), iterations=1, subsets=20)[0], s1[k]), k
    with pytest.raises(ValueError):
        plan.project_adjoint(torch.zeros(1, 1000, 912, device=cuda))
    for bad in (dict(iterations=0), dict(subsets=7), dict(relaxation=2.0), dict(relaxation=0.0)):
        with pytest.raises(ValueError):
            plan.sart(sb[:1].contiguous(), **bad)


@pytest.mark.parametrize("flip,iterations,subsets", [(True, 2, 20), (False, 2, 20), (True, 1, 1)])
def test_sart_matches_the_oracle(plan, phantom, cuda, flip, iterations, subsets):
    from oracle import sart_oracle as Q
    b = phantom[1] if flip else np.ascontiguousarray(phantom[1][:, ::-1])
    got = plan.sart(_dev(b, cuda)[None], flip=flip, iterations=iterations, subsets=subsets, relaxation=1.0).cpu().numpy()[0]
    want = Q.sart(b, flip=flip, iterations=iterations, subsets=subsets, relaxation=1.0)[0]
    err = rel_l2(got, want)
    print(f"SART vs fp64 oracle (flip={int(flip)}, {iterations} sweeps, S={subsets}): rel-L2 {err:.2e}")
    assert err <= SART_ORACLE_TOL, err


def test_sart_converges_below_fbp_on_the_device(plan, phantom, cuda):
    """The CPU test's convergence claims with the device operators: the weighted residual falls at every sweep (a call with k
    sweeps returns the k-th iterate) and ends below that of the FBP image."""
    from ipdm_pytorch_b200 import engine
    img, b = phantom
    bd = _dev(b, cuda)[None]
    R = plan.project(torch.ones(1, 512, 512, device=cuda))[0].double()
    m = R > 0
    wres = lambda x: float(((bd[0].double() - plan.project(x)[0].double())[m] / R[m].sqrt()).norm())
    d = engine.SART_DEFAULTS
    xs = [plan.sart(bd, iterations=k, subsets=d["subsets"], relaxation=d["relaxation"]) for k in range(1, d["iterations"] + 1)]
    res = [wres(x) for x in xs]
    fbp = plan.forward(bd)
    body = torch.from_numpy(img > BODY).to(cuda)
    ref = _dev(img, cuda)
    rmse = lambda x: float(((x[0] - ref)[body] ** 2).mean().sqrt())
    print("device weighted residual per sweep:", " ".join(f"{r:.3f}" for r in res), f"| FBP {wres(fbp):.3f}")
    print("device body RMSE per sweep:", " ".join(f"{rmse(x):.5f}" for x in xs), f"| FBP {rmse(fbp):.5f} 1/cm")
    assert all(b1 < a1 for a1, b1 in zip(res, res[1:])), res
    assert res[-1] < wres(fbp)
    assert torch.equal(plan.sart(bd), xs[-1])                # the defaults


def _model(tmp_path, extra=None):
    from Config.default_config import default_cfg
    from Utils.train_test_utils import progressive_domain_denoiser
    opt = default_cfg(["--load_option_path", os.path.join(PKG, "Config/Mayo-Config/test_progressive_option.json"), "--device", "cuda:0"])
    opt.load_img_model_path = opt.load_proj_model_path = None
    opt.test_dataset_path_FD_img = opt.test_dataset_path_LD_img = opt.test_dataset_path_FD_proj = opt.test_dataset_path_LD_proj = None
    torch.manual_seed(0)
    model = progressive_domain_denoiser(opt, result_save_path=str(tmp_path))
    cfg = dict(convertor="SART", save_it_state_img=False, save_it_state_proj=False, ultra_img_denoise=False, t_start_proj=[2, 1],
               t_start_img=[2, 1], noise_seed=5)
    cfg.update(extra or {})
    model.update_opt(cfg)
    return model


@pytest.mark.parametrize("clip_proj", [False, True])
def test_progressive_pass_with_sart(cuda, tmp_path, monkeypatch, clip_proj):
    """proj stage -> SART -> image stage: the reconstruction is FBP.sart_device of the stage's last iterate (x G = 10 with clip_proj)
    and the sharpen filter is not applied (the shipped Mayo options have fbp_sharpen on)."""
    import ipdm_pytorch_b200.synthetic as S
    import Utils.train_test_utils as U
    seen = []
    real = U.tensor_sharpen
    monkeypatch.setattr(U, "tensor_sharpen", lambda x, N=60: (seen.append(N), real(x, N))[1])
    model = _model(tmp_path, dict(clip_proj=clip_proj, sart_iterations=2, sart_subsets=20))
    assert model.opt.fbp_sharpen
    ld = torch.from_numpy(np.stack([S.make_slice(s)[0] for s in (0, 1)]))[:, None]
    model.data_sample_load(ldct=None, ldproj=ld, fdproj=None, fdct=None)
    out = model.progressive_denoiser(save_proj_state=True)
    assert torch.isfinite(out).all() and seen == [-1]
    last = torch.from_numpy(model.proj_denoise_result[-1][:, 0]).to(cuda).float()
    want = model._fbp.sart_device(last * 10 if clip_proj else last, iterations=2, subsets=20).cpu().numpy()
    rec = model.proj_denoise_convert2img_result["iter_1"][:, 0]
    assert np.isfinite(rec).all() and np.array_equal(rec, want)
    model.update_opt(dict(convertor="FBP"))                    # FBP is unchanged: sharpened again
    model.progressive_denoiser()
    assert seen[-1] == 42


def test_cuda_graph_replay_equals_eager_with_sart(cuda, tmp_path):
    import ipdm_pytorch_b200.synthetic as S
    model = _model(tmp_path)
    ld = torch.from_numpy(np.stack([S.make_slice(s)[0] for s in (0, 1)]))[:, None]
    model.data_sample_load(ldct=None, ldproj=ld, fdproj=None, fdct=None)
    eager1 = model.progressive_denoiser()
    eager2 = model.progressive_denoiser()
    model.update_opt(dict(cuda_graph=True, noise_seed=5))
    g1 = model.progressive_denoiser()
    g2 = model.progressive_denoiser()
    assert torch.equal(g1, eager1) and torch.equal(g2, eager2) and not torch.equal(g1, g2)
    model.update_opt(dict(sart_iterations=1, noise_seed=5))     # an option of the convertor re-captures, no re-init needed
    assert model._graph is None
    g3 = model.progressive_denoiser()
    model.update_opt(dict(cuda_graph=False, noise_seed=5))
    assert torch.equal(g3, model.progressive_denoiser()) and not torch.equal(g3, g1)


def test_bad_sart_options_raise(cuda, tmp_path):
    import ipdm_pytorch_b200.synthetic as S
    model = _model(tmp_path)
    ld = torch.from_numpy(S.make_slice(0)[0])[None, None]
    model.data_sample_load(ldct=None, ldproj=ld, fdproj=None, fdct=None)
    for bad in (dict(sart_subsets=7), dict(sart_iterations=0), dict(sart_relaxation=2.5)):
        model.update_opt(dict(bad, noise_seed=5))
        with pytest.raises(ValueError):
            model.progressive_denoiser()
        with pytest.raises(ValueError):
            model.convertor(np.zeros((2000, 912), np.float32))
        model.update_opt(dict(sart_subsets=100, sart_iterations=5, sart_relaxation=1.0))
    host = model.convertor(S.make_slice(0)[0])                 # convert's host contract: 2-D ndarray in, [1,512,512] ndarray out
    assert isinstance(host, np.ndarray) and host.shape == (1, 512, 512) and np.isfinite(host).all()


def _dataset(root):
    import ipdm_pytorch_b200.synthetic as S
    for sid in range(3):
        d = root / "fdimg" / "P001"
        d.mkdir(parents=True, exist_ok=True)
        np.save(d / f"S{sid:03d}.npy", S.rasterize(S.phantom_ellipses(sid)))
    return str(root / "fdimg")


def _run(fdimg, out, bs):
    from Config.default_config import default_cfg
    from Utils.train_test_utils import progressive_domain_denoiser
    opt = default_cfg(["--load_option_path", os.path.join(PKG, "Config/Mayo-Config/test_progressive_option.json"), "--device", "cuda:0"])
    opt.load_img_model_path = opt.load_proj_model_path = None
    opt.test_dataset_path_FD_img, opt.test_dataset_path_FD_proj = fdimg, None
    opt.test_dataset_path_LD_img = opt.test_dataset_path_LD_proj = None
    opt.data_type = "siemens"
    torch.manual_seed(0)
    model = progressive_domain_denoiser(opt, result_save_path=str(out))
    model.update_opt(dict(convertor="SART", save_it_state_img=False, save_it_state_proj=False, ultra_img_denoise=False,
                          t_start_proj=[2, 1], t_start_img=[2, 1], test_batch_size=bs, test_numbers=-1, noise_seed=11,
                          simulate_low_dose=True))
    model.fit()
    per_slice = []
    for sid in range(3):
        with open(os.path.join(model.save_root_path, "Save_Iter_0", "P001", f"S{sid:03d}", "metric.json")) as f:
            per_slice.append(json.load(f))
    return per_slice


def test_evaluation_loop_simulates_low_dose_with_sart(cuda, tmp_path):
    """simulate_low_dose's ldct goes through the selected convertor: finite metrics, and the same numbers at batch 1 and 2."""
    fdimg = _dataset(tmp_path / "data")
    one = _run(fdimg, tmp_path / "bs1", 1)
    two = _run(fdimg, tmp_path / "bs2", 2)
    for sid in range(3):
        for m in ("psnr_iter_0", "ssim_iter_0"):
            assert np.isfinite(one[sid]["LDCT"][m]) and abs(one[sid]["LDCT"][m] - two[sid]["LDCT"][m]) <= 1e-9, (sid, m)
        assert np.isfinite(one[sid]["deProg"]["psnr_iter_1"]) and np.isfinite(one[sid]["deProg"]["ssim_iter_1"])
