"""GPU: forward projector (ipdm_fbp_project) against its fp64 C restatement and the analytic line integrals, the low-dose noise
(ipdm_low_dose_noise) against synthetic.add_noise, and the simulate_low_dose evaluation loop."""
import json
import os

import numpy as np
import pytest
import torch

from conftest import PKG, rel_l2
from test_project_cpu import FBP_BODY_EXCESS, RASTER_VS_ANALYTIC

pytestmark = pytest.mark.gpu
ORACLE_TOL = 1e-5          # fp32 weights and sums of <= 512 samples vs fp64


@pytest.fixture(scope="module")
def plan(cuda):
    from ipdm_pytorch_b200 import engine
    return engine.FBPPlan(max_batch=16)


@pytest.fixture(scope="module")
def phantom():
    import ipdm_pytorch_b200.synthetic as S
    ell = S.phantom_ellipses(0)
    return S.rasterize(ell), S.fan_sinogram(ell)


@pytest.mark.parametrize("flip", [True, False])
def test_projector_matches_the_oracle(plan, phantom, cuda, flip):
    from oracle import project_oracle as P
    img = phantom[0] if flip else np.ascontiguousarray(phantom[0][:, ::-1])        # flip = 0 takes the native frame
    got = plan.project(torch.from_numpy(img)[None].to(cuda), flip=flip).cpu().numpy()[0]
    want = P.project(img, flip=flip)[0]
    err = rel_l2(got, want)
    print(f"projector vs fp64 oracle (flip={int(flip)}): rel-L2 {err:.2e}")
    assert err <= ORACLE_TOL, err


def test_projection_and_reconstruction_of_the_phantom(plan, phantom, cuda):
    img, analytic = phantom
    x = torch.from_numpy(img)[None].to(cuda)
    sino = plan.project(x)
    e = rel_l2(sino.cpu().numpy()[0], analytic)
    assert e < RASTER_VS_ANALYTIC, e
    rec_p = plan.forward(sino).cpu().numpy()[0]
    rec_a = plan.forward(torch.from_numpy(analytic.astype(np.float32))[None].to(cuda)).cpu().numpy()[0]
    body = img > 0.05
    rmse = lambda r: float(np.sqrt(((r - img)[body] ** 2).mean()))
    print(f"projection vs analytic rel-L2 {e:.3e}; body RMSE FBP(project) {rmse(rec_p):.5f}, FBP(analytic) {rmse(rec_a):.5f}")
    assert rmse(rec_a) < 0.006 and rmse(rec_p) < rmse(rec_a) + FBP_BODY_EXCESS


def test_linearity_zero_and_batch_invariance(plan, cuda):
    import ipdm_pytorch_b200.synthetic as S
    a = torch.from_numpy(S.rasterize(S.phantom_ellipses(0))).to(cuda)
    b = torch.from_numpy(S.rasterize(S.phantom_ellipses(1))).to(cuda)
    pa, pb = plan.project(a[None]), plan.project(b[None])
    assert float(plan.project(torch.zeros_like(a)[None]).abs().max()) == 0.0
    two = plan.project(torch.stack([b, a]))
    assert torch.equal(two[0], pb[0]) and torch.equal(two[1], pa[0])
    sixteen = plan.project(torch.stack([a, b] * 8))
    for k in range(16):
        assert torch.equal(sixteen[k], (pa if k % 2 == 0 else pb)[0]), k
    lin = plan.project((0.5 * a + 2.0 * b)[None].contiguous())
    assert rel_l2(lin.cpu().numpy(), (0.5 * pa + 2.0 * pb).cpu().numpy()) < 1e-5
    with pytest.raises(ValueError):
        plan.project(torch.zeros(1, 256, 256, device=cuda))


@pytest.mark.parametrize("dose", [0.1, 0.25, 0.5])
def test_noise_tape_matches_add_noise(phantom, cuda, dose):
    import ipdm_pytorch_b200.synthetic as S
    from ipdm_pytorch_b200 import engine
    p = phantom[1].astype(np.float32)
    want = S.add_noise(p.astype(np.float64), dose, np.random.default_rng(11))
    tape = np.random.default_rng(11).standard_normal(p.shape).astype(np.float32)
    sino = torch.from_numpy(p)[None].to(cuda)
    got = engine.low_dose_noise(sino, dose, noise=torch.from_numpy(tape)[None].to(cuda), clip=False).cpu().numpy()[0]
    err = rel_l2(got, want)
    assert err <= 1e-6, err
    clipped = engine.low_dose_noise(sino, dose, noise=torch.from_numpy(tape)[None].to(cuda), clip=True).cpu().numpy()[0]
    assert clipped.min() == 0.0 and rel_l2(clipped, np.clip(want, 0, None)) <= 1e-6


def test_philox_noise_keys_and_statistics(cuda):
    from ipdm_pytorch_b200 import engine
    s = torch.full((2, 2000, 912), 2.0, device=cuda)
    a = engine.low_dose_noise(s, 0.25, seed=7, slice_ids=[5, 9], clip=False)
    assert torch.equal(a, engine.low_dose_noise(s, 0.25, seed=7, slice_ids=[5, 9], clip=False))          # deterministic
    assert not torch.equal(a, engine.low_dose_noise(s, 0.25, seed=8, slice_ids=[5, 9], clip=False))      # seed is in the key
    assert not torch.equal(a[0], a[1])                                                                   # slice id is in the key
    alone = engine.low_dose_noise(s[1:].contiguous(), 0.25, seed=7, slice_ids=[9], clip=False)
    assert torch.equal(alone[0], a[1])                                                                   # not the batch position
    default = engine.low_dose_noise(s, 0.25, seed=7, clip=False)                                         # NULL ids: 0..B-1
    assert torch.equal(default[1], engine.low_dose_noise(s, 0.25, seed=7, slice_ids=[0, 1], clip=False)[1])
    inplace = s.clone()
    engine.low_dose_noise(inplace, 0.25, seed=7, slice_ids=[5, 9], clip=False, out=inplace)             # out may alias sino
    assert torch.equal(inplace, a)
    f, ex = 0.25, np.exp(2.0)
    sigma = np.sqrt((1 - f) * ex * (1 + (1 + f) * 5.8 * ex / (f * 1.4e5)) / (f * 1.4e5))
    z = (a[0].double() - 2.0) / sigma
    n = z.numel()
    mean, var = float(z.mean()), float(z.var())
    print(f"standardised residual over {n} bins: mean {mean:+.2e}, variance {var:.5f}")
    assert abs(mean) < 5 / np.sqrt(n) and abs(var - 1) < 5 * np.sqrt(2 / n)


def test_clip_is_honoured(cuda):
    from ipdm_pytorch_b200 import engine
    s = torch.zeros(1, 2000, 912, device=cuda)
    raw = engine.low_dose_noise(s, 0.25, seed=1, clip=False)
    assert float(raw.min()) < 0
    clipped = engine.low_dose_noise(s, 0.25, seed=1, clip=True)
    assert torch.equal(clipped, raw.clamp(min=0))
    with pytest.raises(ValueError):
        engine.low_dose_noise(s, 0.0)


def _dataset(root, kinds):
    import ipdm_pytorch_b200.synthetic as S
    for sid in range(3):
        ell = S.phantom_ellipses(sid)
        arrays = dict(fdimg=S.rasterize(ell), fdproj=S.fan_sinogram(ell).astype(np.float32))
        for k in kinds:
            d = root / k / "P001"
            d.mkdir(parents=True, exist_ok=True)
            np.save(d / f"S{sid:03d}.npy", arrays[k])
    return {k: str(root / k) for k in kinds}


def _run(roots, out, bs, extra=None):
    from Config.default_config import default_cfg
    from Utils.train_test_utils import progressive_domain_denoiser
    opt = default_cfg(["--load_option_path", os.path.join(PKG, "Config/Mayo-Config/test_progressive_option.json"), "--device", "cuda:0"])
    opt.load_img_model_path = opt.load_proj_model_path = None
    opt.test_dataset_path_FD_img, opt.test_dataset_path_FD_proj = roots.get("fdimg"), roots.get("fdproj")
    opt.test_dataset_path_LD_img = opt.test_dataset_path_LD_proj = None
    opt.data_type = "siemens"
    for k, v in (extra or {}).items():               # before the dataset is built: clip_proj also sets its units
        setattr(opt, k, v)
    torch.manual_seed(0)
    model = progressive_domain_denoiser(opt, result_save_path=str(out))
    cfg = dict(convertor="FBP", save_it_state_img=False, save_it_state_proj=False, ultra_img_denoise=False, t_start_proj=[2, 1],
               t_start_img=[2, 1], test_batch_size=bs, test_numbers=-1, noise_seed=11, simulate_low_dose=True)
    model.update_opt(cfg)
    model.fit()
    per_slice = []
    for sid in range(3):
        with open(os.path.join(model.save_root_path, "Save_Iter_0", "P001", f"S{sid:03d}", "metric.json")) as f:
            per_slice.append(json.load(f))
    with open(os.path.join(model.save_root_path, "Save_Iter_0", "metric.json")) as f:
        total = json.load(f)
    return model, per_slice, total


def test_evaluation_loop_simulates_low_dose_from_full_dose_images(cuda, tmp_path):
    """A dataset with full-dose images only: test() projects them, adds the noise at opt.dose, and evaluates as usual."""
    roots = _dataset(tmp_path / "data", ["fdimg"])
    _, one, total = _run(roots, tmp_path / "bs1", 1)
    _, two, _ = _run(roots, tmp_path / "bs2", 2)
    for sid in range(3):
        for m in ("psnr_iter_0", "ssim_iter_0"):
            assert np.isfinite(one[sid]["LDCT"][m]) and abs(one[sid]["LDCT"][m] - two[sid]["LDCT"][m]) <= 1e-9, (sid, m)
        assert np.isfinite(one[sid]["deProg"]["psnr_iter_1"]) and np.isfinite(one[sid]["deProg"]["ssim_iter_1"])
    assert np.isfinite(total["LDCT"]["psnr_iter_0"]) and "psnr_iter_1_std" in total["deProg"]


def test_evaluation_loop_adds_noise_to_full_dose_projections(cuda, tmp_path):
    """With full-dose sinograms in the dataset the projector is skipped: the LD input is their noisy copy (clip_proj: in the dataset's
    /10 units on both sides)."""
    from ipdm_pytorch_b200 import engine
    roots = _dataset(tmp_path / "data", ["fdimg", "fdproj"])
    model, per_slice, _ = _run(roots, tmp_path / "out", 2, dict(clip_proj=True))
    assert all(np.isfinite(m["LDCT"]["psnr_iter_0"]) for m in per_slice)
    fd = torch.from_numpy(np.load(os.path.join(roots["fdproj"], "P001", "S002.npy")))[None].to(cuda)    # the last batch: slice 2
    want = engine.low_dose_noise(fd, model.opt.dose, seed=model._stage_seed(3), slice_ids=[2]) / 10
    assert tuple(model.ldproj.shape) == (1, 1, 2000, 912)
    assert rel_l2(model.ldproj[0].cpu().numpy(), want.cpu().numpy()) < 1e-6
