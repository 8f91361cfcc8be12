"""TEST INFRASTRUCTURE ONLY -- writes tests/golden/*.npz by running the UNMODIFIED reference.

Run in the build container (needs /root/reference):

    python oracle/make_golden.py small      # schedule, small UNet / guided-process cases, one FBP slice (~2 min)
    python oracle/make_golden.py sparse     # sparse (DDIM) guided sampler on the small fields (SURVEY N3)
    python oracle/make_golden.py imgadaptive  # image-domain adaptive lambda (SURVEY N4)
    python oracle/make_golden.py adaptive   # adaptive t_start=None schedule selection, both domains (SURVEY N3)
    python oracle/make_golden.py full       # one full 2000x912 -> 512x512 progressive slice (~12 min on 8 cores)

Every case fixes (weights seed, input seed, noise-tape seed); tests re-create the
inputs from the same seeds (ipdm-pytorch_b200/synthetic.py) and compare the CUDA
path and the oracle restatement against the arrays stored here.
"""
import glob
import importlib.util
import io
import json
import os
import sys
import tempfile
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
GOLD = os.path.join(REPO, "tests", "golden")
sys.path.insert(0, HERE)

from ref_harness import NoiseTape, build_denoiser, load_reference  # noqa: E402


def _synthetic():
    spec = importlib.util.spec_from_file_location("ipdm_synthetic", os.path.join(REPO, "ipdm-pytorch_b200", "synthetic.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


SYN = _synthetic()

PROJ_CFG = dict(in_channels=1, model_channels=64, out_channels=1, attention_resolutions=[16, 32],
                channel_mult=[0.0625, 0.125, 0.25, 2, 2, 4, 4])
IMG_CFG = dict(in_channels=1, model_channels=64, out_channels=1, attention_resolutions=[8, 16],
               channel_mult=[1, 1, 2, 2, 4, 4])


def small_proj_input(seed, h=100, w=76):
    """Sinogram-like positive field [1,1,h,w]; shared by tests (same formula there)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    d = torch.arange(w, dtype=torch.float32)[None, :]
    v = torch.arange(h, dtype=torch.float32)[:, None]
    base = 3.0 * torch.exp(-((d - w / 2) / (w / 3.5)) ** 2) * (1 + 0.1 * torch.sin(2 * np.pi * v / h))
    x = base + 0.08 * torch.randn(h, w, generator=g)
    return x.clamp(min=0)[None, None].contiguous()


def small_img_input(seed, n=64):
    """mu-image-like field [1,1,n,n] around mu_water; shared by tests."""
    import torch
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.linspace(-1, 1, n), torch.linspace(-1, 1, n), indexing="ij")
    body = ((xx / 0.8) ** 2 + (yy / 0.6) ** 2 <= 1).float()
    x = 0.19 * body + 0.012 * body * torch.sin(6 * xx) + 0.004 * torch.randn(n, n, generator=g)
    return x.clamp(min=0)[None, None].contiguous()


def tape(shape, count, seed):
    return SYN.noise_tape(shape, count, seed)


def case_schedule(MM):
    out = {}
    for name, p in (("proj", 5), ("img", 1)):
        gd = MM.GaussianDiffusion(timesteps=1000, beta_schedule="cosine", schedule_power=p)
        for attr in ("betas", "alphas_cumprod", "sqrt_alphas_cumprod", "sqrt_one_minus_alphas_cumprod",
                     "sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod", "posterior_variance",
                     "posterior_log_variance_clipped", "posterior_mean_coef1", "posterior_mean_coef2"):
            out[f"{name}_{attr}"] = getattr(gd, attr).numpy()[:64].astype(np.float64)
    out["lambda_cosine_15"] = MM.cosine_beta_schedule(15, schedule_power=1).numpy().astype(np.float64)
    out["lambda_cosine_5_p10"] = MM.cosine_beta_schedule(5, schedule_power=10).numpy().astype(np.float64)
    return out


def case_curves(TT):
    x = np.linspace(0.5, 4.0, 701).astype(np.float32)
    return dict(x=x, proj=TT.proj_curv_init()(x), img=TT.curve_init()(x))


def case_unet_small(MM):
    import torch
    out = {}
    for name, cfg, seed, shape, t in (("proj", PROJ_CFG, 0, (1, 1, 100, 76), 7), ("img", IMG_CFG, 1, (1, 1, 64, 64), 3)):
        torch.manual_seed(seed)
        net = MM.UNetModel(**cfg).eval()
        g = torch.Generator().manual_seed(100 + seed)
        x = torch.randn(shape, generator=g)
        with torch.no_grad():
            y = net(x, torch.full((1,), t, dtype=torch.long))
        out[f"{name}_y"] = y.numpy()
        out[f"{name}_nparams"] = np.int64(sum(p.numel() for p in net.parameters()))
        out[f"{name}_wsum"] = np.float64(sum(p.double().sum().item() for p in net.parameters()))
    return out


def case_grp_small(MM, TT):
    """guided_reverse_process on small fields, both domains, shipped hyper-parameters."""
    import torch
    out = {}
    torch.manual_seed(0)
    pnet = MM.UNetModel(**PROJ_CFG).eval()
    pgd = MM.GaussianDiffusion(1000, "cosine", schedule_power=5)
    for sid in (0, 1):
        x = small_proj_input(200 + sid)
        with NoiseTape(tape(x.shape, 48, 300 + sid)) as nt:
            res, _, ns = pgd.guided_reverse_process(
                model=pnet, img=x, t_start=[15, 15, 15], clip=False, lambda_ratio=1, eta=0.5,
                lambda_curve=TT.proj_curv_init(), mode="proj", constant_guidance=None, kernel_size_proj=4,
                amplitude_proj=7, only_convertor=False, normal=False, transformer=None)
        assert nt.used == 48 and ns is None and len(res) == 4
        out[f"proj{sid}"] = np.stack([r.numpy()[0, 0] for r in res])
    torch.manual_seed(1)
    inet = MM.UNetModel(**IMG_CFG).eval()
    igd = MM.GaussianDiffusion(1000, "cosine", schedule_power=1)
    for sid in (0, 1):
        x = small_img_input(400 + sid)
        common = dict(model=inet, clip=True, lambda_ratio=10, save_states=False, lambda_curve=TT.curve_init(),
                      noise_strength=None, ldct=x, kernel_size_img=4, amplitude_img=30, only_convertor=False,
                      normal=False, transformer=None)
        with NoiseTape(tape(x.shape, 48 + 18, 500 + sid)) as nt:
            res, _, _ = igd.guided_reverse_process(img=x, t_start=[15, 15, 15], eta=0.7, constant_guidance=0.45, **common)
            res2, _, _ = igd.guided_reverse_process(img=res[-1], t_start=[5, 5, 5], eta=0.6, constant_guidance=0.6, **common)
        assert nt.used == 66
        out[f"img{sid}"] = np.stack([r.numpy()[0, 0] for r in res + res2])
    return out


def case_sparse_small(MM):
    """sparse_guided_reverse_process (DDIM, model.py:654-759) on the small fields with the arguments proj_denoiser / img_denoiser
    pass (train_test_utils.py:445-453, :505-514) and the notebook's cell-3 schedules."""
    import torch
    out = {}
    torch.manual_seed(0)
    pnet = MM.UNetModel(**PROJ_CFG).eval()
    pgd = MM.GaussianDiffusion(1000, "cosine", schedule_power=5)
    for sid in (0, 1):
        x = small_proj_input(200 + sid)
        with NoiseTape(tape(x.shape, 7, 700 + sid)) as nt:
            res = pgd.sparse_guided_reverse_process(model=pnet, condition=x, t_start=[15, 15, 5], condition_lambda_max=0.49,
                                                    condition_lambda_min=0.35, clip_denoised=False, ddim_timesteps=[1, 2, 3], eta=0.5)
        assert nt.used == 7 and len(res) == 3
        out[f"proj{sid}"] = np.stack([r.numpy()[0, 0] for r in res])
    torch.manual_seed(1)
    inet = MM.UNetModel(**IMG_CFG).eval()
    igd = MM.GaussianDiffusion(1000, "cosine", schedule_power=1)
    for sid in (0, 1):
        x = small_img_input(400 + sid)
        with NoiseTape(tape(x.shape, 7, 800 + sid)) as nt:
            res = igd.sparse_guided_reverse_process(model=inet, condition=x, t_start=[18, 18, 5], condition_lambda_max=0.5,
                                                    condition_lambda_min=0.3, clip_denoised=True, ddim_timesteps=[1, 2, 3], eta=0.7)
        assert nt.used == 7
        out[f"img{sid}"] = np.stack([r.numpy()[0, 0] for r in res])
    return out


def case_img_adaptive_small(MM, TT):
    """Image-domain guided process with constant_guidance=None (the argparse default): scalar cosine lambda in iteration 0, the
    per-pixel lambda map built from |miu2pixel(x) - miu2pixel(img)| afterwards (model.py:575-595, SURVEY N4)."""
    import torch
    out = {}
    torch.manual_seed(1)
    inet = MM.UNetModel(**IMG_CFG).eval()
    igd = MM.GaussianDiffusion(1000, "cosine", schedule_power=1)
    for sid in (0, 1):
        x = small_img_input(400 + sid)
        with NoiseTape(tape(x.shape, 30, 900 + sid)) as nt:
            res, _, _ = igd.guided_reverse_process(model=inet, img=x, t_start=[10, 9, 8], clip=True, lambda_ratio=10, eta=0.7, save_states=False,
                                                   mode="img", constant_guidance=None, lambda_curve=TT.curve_init(), noise_strength=None, ldct=x,
                                                   kernel_size_img=4, amplitude_img=20, only_convertor=False, normal=False, transformer=None)
        assert nt.used == 30 and len(res) == 4
        out[f"img{sid}"] = np.stack([r.numpy()[0, 0] for r in res])
    return out


def case_adaptive_schedule_small(MM, TT):
    """t_start=None (the argparse default; Model/model.py:531-535, 582-613, 639-640): probing iteration with t_start = 20, then the
    schedule is picked from max(exp(amplitude * delta-map)) in the projection domain (three slices with amplitude_proj = 7 (shipped), 3, 15 so that
    the reference itself lands in three different classes) and from `noise_strength` in the image domain (SURVEY N3, second half)."""
    import torch
    out = {}
    torch.manual_seed(0)
    pnet = MM.UNetModel(**PROJ_CFG).eval()
    pgd = MM.GaussianDiffusion(1000, "cosine", schedule_power=5)
    for sid, amp in ((0, 7), (1, 3), (2, 15)):
        x = small_proj_input(200 + sid)
        with NoiseTape(tape(x.shape, 21 + 75 + 3, 1100 + sid)) as nt:
            res, _, ns = pgd.guided_reverse_process(
                model=pnet, img=x, t_start=None, clip=False, lambda_ratio=1, eta=0.5, lambda_curve=TT.proj_curv_init(), mode="proj",
                constant_guidance=None, kernel_size_proj=4, amplitude_proj=amp, only_convertor=False, normal=False, transformer=None)
        want = {"high": 75, "mid": 53, "low": 45}[ns]
        assert nt.used == 21 + want + 3 and len(res) == 4, (nt.used, ns, len(res))
        out[f"proj{sid}"] = np.stack([r.numpy()[0, 0] for r in res])
        out[f"proj{sid}_class"] = np.array(ns)
        out[f"proj{sid}_amplitude"] = np.float32(amp)
        print(f"adaptive proj slice {sid} (amplitude {amp}): class {ns}, {nt.used} noise draws", flush=True)
    torch.manual_seed(1)
    inet = MM.UNetModel(**IMG_CFG).eval()
    igd = MM.GaussianDiffusion(1000, "cosine", schedule_power=1)
    for sid, ns in ((0, "mid"), (1, None), (2, "high")):
        x = small_img_input(400 + sid)
        with NoiseTape(tape(x.shape, 21 + 45 + 3, 1200 + sid)) as nt:
            res, _, _ = igd.guided_reverse_process(model=inet, img=x, t_start=None, clip=True, lambda_ratio=10, eta=0.7, save_states=False,
                                                   mode="img", constant_guidance=None, lambda_curve=TT.curve_init(), noise_strength=ns, ldct=x,
                                                   kernel_size_img=4, amplitude_img=20, only_convertor=False, normal=False, transformer=None)
        assert len(res) == 4
        out[f"img{sid}"] = np.stack([r.numpy()[0, 0] for r in res])
        out[f"img{sid}_class"] = np.array("none" if ns is None else ns)
        print(f"adaptive img slice {sid}: noise_strength {ns}, {nt.used} noise draws", flush=True)
    return out


def case_fbp(RF):
    import numba
    numba.set_num_threads(1)
    fbp = RF.FBP(device="cpu")
    ld, nd, img = SYN.make_slice(0)
    t0 = time.time()
    rec = fbp.convert(ld[None])          # includes JIT
    t1 = time.time()
    rec = fbp.convert(ld[None])
    t2 = time.time()
    rec_nd = fbp.convert(nd[None])
    out = dict(ld=rec[0], nd_sub=rec_nd[0, 1::4, 2::4].copy(), h_RL=fbp.h_RL[:, 0].copy(), nda=fbp.nda.copy(),
               theta=fbp.theta.copy(), r_sub=fbp.r[1::4, 2::4].copy(), phi_sub=fbp.phi[1::4, 2::4].copy(),
               seconds_warm=np.float64(t2 - t1), seconds_cold=np.float64(t1 - t0))
    # the two table files the reference ships: theta must equal arange(0, 360, .18) deg (SURVEY D2)
    st = np.fromfile(os.path.join(os.environ.get("IPDM_REFERENCE_ROOT", "/root/reference"), "Recon/Simens_theta.txt"), "float32")
    out["simens_theta_maxabs_rad"] = np.float64(np.abs(st.astype(np.float64) / 180 * np.pi - fbp.theta).max())
    err = rec_nd[0] - img
    body = img > 0.05
    out["nd_rmse_in_body"] = np.float64(np.sqrt((err[body] ** 2).mean()))
    return out


def sub(a):
    """Strided sample + moments of a full-size field (keeps fixtures small)."""
    a = np.asarray(a, dtype=np.float32)
    return dict(sub=a[..., 1::4, 2::4].copy(), sum=np.float64(a.astype(np.float64).sum()),
                sumsq=np.float64((a.astype(np.float64) ** 2).sum()))


def case_full_slice():
    import torch
    tmp = tempfile.mkdtemp(prefix="ipdm_ref_")
    model = build_denoiser(tmp, seed=0)
    ld, nd, img = SYN.make_slice(0)
    ldproj = torch.from_numpy(ld)[None, None]
    ldct = torch.zeros(1, 1, 512, 512)
    tp = tape((1, 1, 2000, 912), 48, 9527) + tape((1, 1, 512, 512), 66, 19527)
    stamps = {}
    with NoiseTape(tp) as nt:
        model.data_sample_load(ldct=ldct, ldproj=ldproj, fdproj=None, fdct=torch.from_numpy(img)[None, None])
        model.temp_clear()
        t0 = time.time()
        res = model.progressive_denoiser(save_proj_state=True)
        stamps["total_s"] = time.time() - t0
    assert nt.used == 114, nt.used
    out = {}
    for k in range(4):
        for kk, v in sub(model.proj_denoise_result[f"iter_{k + 1}"][0, 0]).items():
            out[f"proj_iter{k + 1}_{kk}"] = v
    for kk, v in sub(model.proj_denoise_convert2img_result["iter_1"][0, 0]).items():
        out[f"fbp_img_{kk}"] = v
    for kk, v in sub(res[0, 0].numpy()).items():
        out[f"final_{kk}"] = v
    out["final"] = res[0, 0].numpy()
    out["total_s"] = np.float64(stamps["total_s"])
    out["threads"] = np.int64(torch.get_num_threads())
    return out


def case_img_stage_512():
    """Image-domain stage alone at 512x512 (60 UNet forwards): input = sharpened reference FBP of the low-dose slice."""
    import torch
    tmp = tempfile.mkdtemp(prefix="ipdm_ref_")
    model = build_denoiser(tmp, seed=0)
    ld, nd, img = SYN.make_slice(0)
    rec = model.convertor(torch.from_numpy(ld)[None])[:, None]             # reference FBP.convert, CPU tensor [1,1,512,512]
    x = TTsharpen(rec, 42)
    with NoiseTape(tape((1, 1, 512, 512), 66, 19527)) as nt:
        t0 = time.time()
        res = model.img_denoiser(x, noise_strength=None, save_state=True)
        total = time.time() - t0
    assert nt.used == 66
    out = dict(x=x[0, 0].numpy(), final=res[0, 0].numpy(), total_s=np.float64(total))
    for k in range(1, 9):
        out[f"iter{k}_sub"] = model.progressive_denoise_result[f"iter_{k}"][0, 0][1::4, 2::4].copy()
    return out


def TTsharpen(x, n):
    MM, RF, TT, CFG = load_reference()
    return TT.tensor_sharpen(x, n)


FILE_LIMIT = 1_000_000           # bytes per stored file: a full-size case is split over several files


def _npz_bytes(key, value):
    buf = io.BytesIO()
    np.savez_compressed(buf, **{key: value})
    return buf.getbuffer().nbytes


def save(name, d):
    """Writes the arrays of one case as <name>.npz, <name>.1.npz, ... (first fit, each file under FILE_LIMIT); the tests'
    golden(name) merges them.  Every array is stored whole."""
    os.makedirs(GOLD, exist_ok=True)
    for stale in glob.glob(os.path.join(GOLD, glob.escape(name) + ".[0-9]*.npz")):
        os.remove(stale)
    parts, sizes = [], []
    for key, value in d.items():
        n = _npz_bytes(key, value)
        assert n < FILE_LIMIT, (name, key, n)
        i = next((i for i, s in enumerate(sizes) if s + n < FILE_LIMIT), len(parts))
        if i == len(parts):
            parts.append({})
            sizes.append(0)
        parts[i][key] = value
        sizes[i] += n
    for i, part in enumerate(parts):
        path = os.path.join(GOLD, name + (f".{i}" if i else "") + ".npz")
        np.savez_compressed(path, **part)
        assert os.path.getsize(path) < FILE_LIMIT, path
        print(f"wrote {path} ({os.path.getsize(path) / 1024:.0f} KiB)", flush=True)


def main():
    what = sys.argv[1] if len(sys.argv) > 1 else "small"
    cwd = os.getcwd()
    if what == "small":
        MM, RF, TT, CFG = load_reference()
        save("schedule", case_schedule(MM))
        save("curves", case_curves(TT))
        save("unet_small", case_unet_small(MM))
        save("grp_small", case_grp_small(MM, TT))
        save("fbp_slice0", case_fbp(RF))
    elif what == "sparse":
        MM, RF, TT, CFG = load_reference()
        save("sparse_small", case_sparse_small(MM))
    elif what == "imgadaptive":
        MM, RF, TT, CFG = load_reference()
        save("img_adaptive_small", case_img_adaptive_small(MM, TT))
    elif what == "adaptive":
        MM, RF, TT, CFG = load_reference()
        save("adaptive_schedule_small", case_adaptive_schedule_small(MM, TT))
    elif what == "fbp":
        MM, RF, TT, CFG = load_reference()
        save("fbp_slice0", case_fbp(RF))
    elif what == "full":
        save("full_slice0", case_full_slice())
    elif what == "img512":
        save("img_stage512", case_img_stage_512())
    os.chdir(cwd)


if __name__ == "__main__":
    main()
