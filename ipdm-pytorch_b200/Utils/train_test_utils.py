"""Host-side mirror of the reference's inference orchestrator (Utils/train_test_utils.py).

`progressive_domain_denoiser` keeps the reference's constructor, option handling
(`update_opt` / `reset_opt`, :202-211), per-slice entry points (`data_sample_load` :569-594,
`proj_denoiser` :421-480, `img_denoiser` :482-550, `progressive_denoiser` :552-567) and result
attributes (`ResultTempDict`s of numpy arrays keyed `iter_k`), so `main.py` and notebook cells 0-2
drive it unchanged.  Differences, all additive:
  * batches of B >= 1 slices are accepted everywhere; statistics are per slice (SURVEY D3);
  * `progressive_denoiser(..., noise=(proj_tape, img_tape))` injects caller noise for parity runs;
  * `simulate_low_dose` makes low-dose inputs from full-dose images or sinograms on the device, and the
    option of the same name makes `test()` use it instead of reading low-dose files;
  * `convertor="SART"` (ordered-subset SART on the device, `sart_*` options) is a second convertor next to FBP;
  * between the projection stage, the convertor, the sharpen filter and the image stage the
    data stays on the GPU (the reference crosses to the host three times, SURVEY 3.2);
  * training (`train`, the train branch of `fit`), figures and skimage/piq metrics are out of scope.
"""
import copy
import functools
import json
import os
import os.path as osp
from datetime import datetime
from typing import Optional

import numpy as np
import torch
import torch.distributed as dist
from torch import Tensor

from _ipdm_boot import engine as _eng
from Config.default_config import cfg_load
from Dataset.npz_data_loader import Siemens_dataset_npz, miu2pixel
from Model.model import GaussianDiffusion, UNetModel
from Recon.FBP_kernel import FBP
from Recon.TASART2DNSL0 import proj_torch, recons_torch
from Utils.loggerx import LoggerX


class DotDict(dict):
    def __setattr__(self, key, value):
        self[key] = value

    def __getattr__(self, key):
        value = self[key]
        return DotDict(value) if isinstance(value, dict) else value


class ResultTempDict(DotDict):
    def __getitem__(self, item):
        if isinstance(item, str):
            return super().__getitem__(item)
        if isinstance(item, int):
            if item > 0:
                return self[f"iter_{item}"]
            if item == -1:
                return self[f"iter_{len(self)}"]
        raise KeyError(item)


_CURVES = {"img": ([1, 1.1, 1.2, 1.3, 1.4, 1.5, 1.6, 1.7], [20, 17.5, 15, 12, 8.5, 5, 2, 1],
                   [1.7, 1.8, 2.0, 2.2, 2.35, 2.5, 3], [1, 0.7, 0.5, 0.3, 0.2, 0.1, 0.05]),
           "proj": ([1, 1.1, 1.2, 1.3, 1.4, 1.5, 1.6, 1.7], [20, 17.5, 15, 12, 8.5, 7.5, 5, 4],
                    [1.7, 1.8, 2.0, 2.2, 2.35, 2.5, 3, 3.5], [4, 3, 2, 1, 0.5, 0.3, 0.1, 0.01])}


def weight_lambda(x, f1, f2):
    if x < 1:
        return f1(1)
    if x <= 1.7:
        return f1(x)
    if x <= 2.75:
        return f2(x)
    return f2(2.75)


def _curve(kind):
    """Host callable ndarray -> float32 ndarray; the device pipeline evaluates the same polynomials in-kernel."""
    return functools.partial(_eng.lambda_curve_host, kind=kind)


def curve_init():
    return _curve("img")


def proj_curv_init():
    return _curve("proj")


def tensor_sharpen(img_in, N=60):
    """3x3 sharpen of every slice of [B,1,H,W] (reference :868-878 at B = 1); CUDA tensors only."""
    if N == -1:
        return img_in
    return _eng.sharpen3x3(img_in.contiguous().float(), N)


class progressive_domain_denoiser:
    def __init__(self, opt, result_save_path=None):
        self.trans_ldproj = self.trans_ldimg = None
        self.opt = opt
        self.opt_temp = copy.deepcopy(opt)
        stamp = "{0:%Y-%m-%dT%H-%M-%S/}".format(datetime.now())
        if result_save_path is None:
            save_root = osp.join(osp.dirname(osp.abspath(__file__)), 'ModelTrainLog/', '{}_{}/{}'.format(opt.model_name, opt.run_name, stamp))
        else:
            save_root = osp.join(result_save_path, '{}_{}'.format(opt.model_name, opt.run_name))
        self.logger = LoggerX(save_root, opt)
        self.rank = dist.get_rank() if (dist.is_available() and dist.is_initialized()) else 0
        self.logger.save_option(self.opt)
        if "train" in self.opt.mode:
            raise NotImplementedError("training modes are outside the B200 inference path; use the reference to train")
        self.optimizer = self.proj_model = self.img_model = None
        if self.opt.mode in ["test_proj", "test_prog"]:
            self.init_proj_model()
        self.init_convertor(opt.convertor)
        if self.opt.mode in ["test_img", "test_prog"]:
            self.init_img_model()
        self.logger.modules = [self.proj_model, self.img_model, self.optimizer]
        self.logger.module_names = ["proj_model", "img_model", "optimizer"]
        self.load_model()
        self.init_data_loader()
        self.fdct = self.fdproj = self.ldct = self.ldct_np = self.ldproj = self.ldproj_np = None
        self.proj_denoise_result = ResultTempDict()
        self.proj_denoise_convert2img_result = ResultTempDict()
        self.img_denoise_result = ResultTempDict()
        self.progressive_denoise_result = ResultTempDict()
        self.noise_strength = None
        self.img_lambda_curve = curve_init()
        self.proj_lambda_curve = proj_curv_init()
        self.metric_instance = DotDict(LDCT=DotDict(), deProj=DotDict(), deImg=DotDict(), deProg=DotDict(), deProj2img=DotDict())
        self.metric_total = DotDict()
        self.metric_each_sample = []
        self.save_root_path = osp.join(save_root, 'save_test_results')
        os.makedirs(self.save_root_path, exist_ok=True)

    # ---- options ---------------------------------------------------------------------------
    def update_opt(self, ultra_cfg=None):
        if ultra_cfg is not None:
            self._drop_graph()                                   # a captured pass freezes every option as kernel arguments
            cfg_load(ultra_cfg, self.opt.__dict__)
            self.logger.save_option(self.opt)
            if "convertor" in ultra_cfg.keys():
                self.init_convertor(ultra_cfg["convertor"])
            if "precision" in ultra_cfg.keys():
                for m in (self.proj_model, self.img_model):
                    if m is not None:
                        m.set_precision(self.opt.precision)
            if "noise_seed" in ultra_cfg.keys():
                self._noise_calls = 0                            # same seed => same noise sequence from here on

    def reset_opt(self):
        self._drop_graph()
        self.opt = copy.deepcopy(self.opt_temp)

    def _drop_graph(self):
        """Forget the captured CUDA graph: it holds raw pointers into the FBP plan, both UNet handles and their arenas."""
        self.__dict__["_graph"] = None

    # ---- in-kernel noise keys ----------------------------------------------------------------
    def _stage_seed(self, stage):
        """Philox key of one stage (0 proj, 1 img, 2 ultra, 3 low-dose simulation): a hash of (noise_seed, stage), so that neighbouring seeds (e.g. the
        per-rank seeds of bench.py) never share a stream with another stage."""
        z = (int(getattr(self.opt, "noise_seed", 0)) * 0x9E3779B97F4A7C15 + (stage + 1) * 0xBF58476D1CE4E5B9) & (2 ** 64 - 1)
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & (2 ** 64 - 1)
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & (2 ** 64 - 1)
        return z ^ (z >> 31)

    def _next_noise_epoch(self):
        """Every call of a denoiser entry point draws fresh noise, as the reference's randn_like does: the device-resident half of
        the Philox key is a per-model call counter (reset by update_opt(dict(noise_seed=...)))."""
        self._noise_calls = getattr(self, "_noise_calls", 0) + 1
        _eng.set_noise_epoch(self._noise_calls)

    # ---- models / convertor ----------------------------------------------------------------
    def _make_unet(self, suffix):
        o = self.opt
        net = UNetModel(in_channels=getattr(o, "in_channels_" + suffix), model_channels=getattr(o, "model_channels_" + suffix),
                        out_channels=getattr(o, "out_channels_" + suffix),
                        attention_resolutions=getattr(o, "attention_resolutions_" + suffix),
                        channel_mult=getattr(o, "channel_mult_" + suffix)).to(o.device)
        net.set_precision(getattr(o, "precision", "tf32"))
        return net.eval()

    def init_img_model(self):
        self.img_model = self._make_unet("img")
        self.img_device = next(self.img_model.parameters()).device
        self.img_dtype = next(self.img_model.parameters()).dtype
        self.img_gaussian_diffusion = GaussianDiffusion(timesteps=self.opt.timesteps_img, beta_schedule='cosine',
                                                        schedule_power=self.opt.schedule_power_img)

    def init_proj_model(self):
        self.proj_model = self._make_unet("proj")
        self.proj_device = self.opt.device
        self.proj_dtype = next(self.proj_model.parameters()).dtype
        self.proj_gaussian_diffusion = GaussianDiffusion(timesteps=self.opt.timesteps_proj, beta_schedule='cosine',
                                                         schedule_power=self.opt.schedule_power_proj)

    def init_convertor(self, convertor):
        self._drop_graph()
        self._fbp, self._fbp_cap = None, 0
        if convertor == "FBP":
            self._fbp = FBP(device=self.opt.device)
            self.convertor = self._fbp.convert
        elif convertor == "SART":
            self._fbp = FBP(device=self.opt.device)
            self.convertor = lambda pj, flip=True: self._fbp.sart(pj, flip, **self._sart_kw())
        else:
            def _unsupported(*a, **k):
                raise RuntimeError(f"convertor={convertor!r} is not available in the B200 build (only 'FBP' and 'SART'; the ART "
                                   "extension TASART2DNSL0.pyd is Windows-only): call update_opt(dict(convertor='FBP'))")
            self.convertor = _unsupported
        self.projection = functools.partial(proj_torch, lut_area=None, betas=None)

    def load_model(self):
        self._drop_graph()
        o = self.opt
        if o.resume_epochs_img > 0 and o.load_img_model_path is not None and self.img_model is not None:
            self.logger.load_checkpoints(o.resume_epochs_img, o.load_img_model_path)
        if o.resume_epochs_proj > 0 and o.load_proj_model_path is not None and self.proj_model is not None:
            self.logger.load_checkpoints(o.resume_epochs_proj, o.load_proj_model_path)

    def init_data_loader(self):
        o = self.opt
        self.test_dataset = Siemens_dataset_npz(ldimg_path=o.test_dataset_path_LD_img, fdimg_path=o.test_dataset_path_FD_img,
                                                ldproj_path=o.test_dataset_path_LD_proj, fdproj_path=o.test_dataset_path_FD_proj,
                                                proj_clip=o.clip_proj, img_clip=o.clip_img, data_type=o.data_type)
        self.test_loader = torch.utils.data.DataLoader(dataset=self.test_dataset, batch_size=o.test_batch_size, shuffle=False,
                                                       collate_fn=self.test_dataset.collate)

    # ---- temporaries -----------------------------------------------------------------------
    def temp_clear(self):
        self.proj_temp_clear()
        self.img_temp_clear()
        self.metric_clear()
        self.noise_strength = None

    def metric_clear(self):
        self.metric_instance = DotDict(LDCT=DotDict(), deProj=DotDict(), deImg=DotDict(), deProg=DotDict(), deProj2img=DotDict())

    def proj_temp_clear(self):
        self.proj_denoise_convert2img_result = ResultTempDict()
        self.proj_denoise_result = ResultTempDict()

    def img_temp_clear(self):
        self.img_denoise_result = ResultTempDict()
        self.progressive_denoise_result = ResultTempDict()

    # ---- stages (device resident) ------------------------------------------------------------
    def _proj_stage(self, x, noise=None):
        o = self.opt
        if o.sample_method_proj == "sparse":                                   # reference :445-453 (SURVEY N3)
            return self.proj_gaussian_diffusion.sparse_guided_reverse_process(
                model=self.proj_model, condition=x.type(self.proj_dtype), t_start=o.t_start_proj, condition_lambda_max=0.49,
                condition_lambda_min=0.35, clip_denoised=o.clip_proj, ddim_timesteps=o.ddim_timesteps_proj, eta=o.eta_proj,
                noise=noise, seed=self._stage_seed(0))
        res, _, ns = self.proj_gaussian_diffusion.guided_reverse_process(
            model=self.proj_model, img=x.type(self.proj_dtype), t_start=o.t_start_proj, clip=o.clip_proj,
            lambda_ratio=o.lambda_ratio_proj, eta=o.eta_proj, lambda_curve=self.proj_lambda_curve, mode="proj",
            constant_guidance=o.constant_guidance_proj, kernel_size_proj=o.kernel_size_proj, amplitude_proj=o.amplitude_proj,
            only_convertor=o.benchmark_test, normal=o.normal, transformer=self.trans_ldproj, noise=noise,
            seed=self._stage_seed(0))
        self.noise_strength = ns
        return res

    def _reserve_fbp(self, batch):
        if self._fbp is None:
            self.convertor(None)
        if batch > getattr(self, "_fbp_cap", 0):                     # the plan re-allocates its filtered-sinogram workspace for a larger batch
            if not torch.cuda.is_current_stream_capturing():
                self._drop_graph()
            self._fbp_cap = int(batch)

    def _sart_kw(self):
        """The sart_* options, read at call time (update_opt needs no re-init)."""
        o = self.opt
        return dict(iterations=o.sart_iterations, subsets=o.sart_subsets, relaxation=o.sart_relaxation)

    def _convert_device(self, sino):
        """[B,1,2000,912] device -> [B,1,512,512] device through the FBP plan: SART when opt.convertor is 'SART', FBP otherwise."""
        self._reserve_fbp(sino.shape[0])
        G = 10 if self.opt.clip_proj else 1
        s = sino[:, 0].float()
        s = s * G if G != 1 else s
        if self.opt.convertor == "SART":
            return self._fbp.sart_device(s, **self._sart_kw())[:, None]
        return self._fbp.convert_device(s)[:, None]

    def simulate_low_dose(self, fd, dose=None, slice_ids=None):
        """Low-dose inputs at `dose` (default opt.dose) from a full-dose batch: a sinogram [B,1,2000,912] gets the dose-reduction
        noise of the reference's Low_dose_CT_simulate.add_noise; a mu image [B,1,512,512] is forward-projected (FBP geometry,
        Joseph's method) first.  Returns (ldproj [B,1,2000,912], ldct [B,1,512,512] = ldproj through the convertor, no sharpen), both on the
        device.  The noise is drawn in line-integral units from Philox keyed by (a hash of noise_seed, slice id, bin), slice ids
        default to 0..B-1; with clip_proj, sinograms are in the dataset's units (line integrals / 10) on the way in and out."""
        o = self.opt
        fd = fd.to(o.device).float()
        if fd.dim() != 4 or fd.shape[1] != 1:
            raise ValueError(f"simulate_low_dose: expected [B,1,2000,912] or [B,1,512,512], got {tuple(fd.shape)}")
        G = 10 if o.clip_proj else 1
        self._reserve_fbp(fd.shape[0])
        if tuple(fd.shape[2:]) == (_eng.N_PIX, _eng.N_PIX):
            sino = self._fbp.project_device(fd[:, 0])
        elif tuple(fd.shape[2:]) == (_eng.N_VIEWS, _eng.N_DET):
            sino = fd[:, 0] * G                                                # always a fresh buffer: the noise is added in place
        else:
            raise ValueError(f"simulate_low_dose: expected [B,1,2000,912] or [B,1,512,512], got {tuple(fd.shape)}")
        _eng.low_dose_noise(sino, o.dose if dose is None else dose, seed=self._stage_seed(3), slice_ids=slice_ids, clip=True, out=sino)
        ldproj = (sino / G if G != 1 else sino)[:, None]
        return ldproj, self._convert_device(ldproj)

    def _img_stage(self, x, noise=None, noise_strength=None):
        o = self.opt
        x = x.type(self.img_dtype).to(self.img_device).contiguous()
        common = dict(model=self.img_model, clip=o.clip_img, lambda_ratio=o.lambda_ratio_img, save_states=o.save_states_img,
                      lambda_curve=self.img_lambda_curve, noise_strength=noise_strength, ldct=x, kernel_size_img=o.kernel_size_img,
                      amplitude_img=o.amplitude_img, only_convertor=o.benchmark_test, normal=o.normal, transformer=self.trans_ldimg,
                      mode="img")
        if o.sample_method_img == "sparse":                                    # reference :505-514 (SURVEY N3)
            n_count = 1 + sum(o.ddim_timesteps_img[:len(o.t_start_img)])
            result = self.img_gaussian_diffusion.sparse_guided_reverse_process(
                model=self.img_model, condition=x, t_start=o.t_start_img, condition_lambda_max=0.5, condition_lambda_min=0.3,
                clip_denoised=True, ddim_timesteps=o.ddim_timesteps_img, eta=o.eta_img,
                noise=None if noise is None else noise[:n_count], seed=self._stage_seed(1))
        else:
            if o.t_start_img is not None:
                n_count = sum(o.t_start_img) + len(o.t_start_img)
            elif noise is not None:                                            # adaptive schedule (t_start_img=None) with a noise tape
                cls = set(noise_strength) if isinstance(noise_strength, (list, tuple)) else {noise_strength}
                if len(cls) != 1:
                    raise ValueError("a noise tape with t_start_img=None needs one noise_strength class for the whole batch (the tape order is per slice)")
                n_count = 21 + sum(GaussianDiffusion._ADAPTIVE_IMG[cls.pop() or "low"][0]) + 3
            result, _, _ = self.img_gaussian_diffusion.guided_reverse_process(
                img=x, t_start=o.t_start_img, eta=o.eta_img, constant_guidance=o.constant_guidance_img,
                noise=None if noise is None else noise[:n_count], seed=self._stage_seed(1), **common)
        if o.ultra_img_denoise:
            n_ultra = None if noise is None else noise[n_count:]
            extra, _, _ = self.img_gaussian_diffusion.guided_reverse_process(
                img=result[-1], t_start=[5, 5, 5], eta=0.6, constant_guidance=0.6, noise=n_ultra,
                seed=self._stage_seed(2), **common)
            result = result + extra
        return result

    # ---- reference entry points --------------------------------------------------------------
    def proj_denoiser(self, x: Tensor, convert=True, save_state=True, save_proj_state=False, return_idx=-1, noise=None):
        if noise is None:
            self._next_noise_epoch()
        result = self._proj_stage(x, noise)
        self.proj_temp_clear()
        if save_proj_state:
            for k, r in enumerate(result):
                self.proj_denoise_result[f"iter_{k + 1}"] = r.cpu().numpy()
        if save_state:
            if convert:
                for k, r in enumerate(result):
                    self.proj_denoise_convert2img_result[f"iter_{k + 1}"] = self._convert_device(r).cpu().numpy()
                return torch.from_numpy(self.proj_denoise_convert2img_result[f"iter_{len(result)}"]), self.noise_strength
            for k, r in enumerate(result):
                self.proj_denoise_result[f"iter_{k + 1}"] = r.cpu().numpy()
            return result[return_idx], self.noise_strength
        if convert:
            self.proj_denoise_convert2img_result["iter_1"] = self._convert_device(result[return_idx]).cpu().numpy()
            return torch.from_numpy(self.proj_denoise_convert2img_result["iter_1"]), self.noise_strength
        self.proj_denoise_result["iter_1"] = result[return_idx].cpu().numpy()
        return result[return_idx], self.noise_strength

    def img_denoiser(self, x, return_idx=-1, noise_strength=None, mode="progressive", sharpen_num=45, save_state=True, noise=None):
        if noise is None:
            self._next_noise_epoch()
        result = self._img_stage(x, noise, noise_strength)
        self.img_temp_clear()
        store = self.progressive_denoise_result if mode == "progressive" else self.img_denoise_result
        if save_state:
            for k, r in enumerate(result):
                store[f"iter_{k + 1}"] = r.cpu().numpy()
        else:
            store["iter_1"] = result[return_idx].cpu().numpy()
        return result[return_idx]

    def _graph_key(self, sharpen_num):
        """Everything a captured pass freezes: the whole option table, the input shape, and the identity + weights of the FBP plan and of
        both UNet handles (their device pointers are baked into the graph)."""
        opts = json.dumps({k: v for k, v in sorted(vars(self.opt).items())}, sort_keys=True, default=str)
        nets = tuple((id(m.cuda_handle()), m._weights_key()) for m in (self.proj_model, self.img_model))
        return (tuple(self.ldproj.shape), str(self.ldproj.device), int(sharpen_num), opts, id(self._fbp), nets)

    def _progressive_graphed(self, sharpen_num):
        """Whole progressive pass as ONE CUDA graph (north_star item 4): captured after an eager warm-up that builds every plan and
        workspace, replayed with fresh Philox noise (device-resident epoch) and a refreshed input.  Exactly one graph is kept: any
        change of an option, the batch shape, the convertor, the precision or the weights drops it and re-captures, so a replay never
        touches freed plans, arenas or workspaces; the cache entry keeps the captured objects alive."""
        key = self._graph_key(sharpen_num)
        ent = self.__dict__.get("_graph")
        if ent is None or ent["key"] != key:
            self._drop_graph()
            static_in = self.ldproj.clone()
            self._progressive_eager(static_in, sharpen_num, None, None)            # warm-up: plans, workspaces, attributes
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                outs = self._progressive_eager(static_in, sharpen_num, None, None)
            ent = dict(key=key, graph=g, static_in=static_in, outs=outs,
                       keep=(self._fbp, self.proj_model.cuda_handle(), self.img_model.cuda_handle()))
            self._graph = ent
        ent["static_in"].copy_(self.ldproj, non_blocking=True)
        ent["graph"].replay()
        return ent["outs"]                           # graph-static memory: the caller copies what it hands out

    def _progressive_eager(self, ldproj, sharpen_num, pn, inn):
        o = self.opt
        result = self._proj_stage(ldproj, pn)
        recs = [self._convert_device(r) for r in result] if o.save_it_state_proj else [self._convert_device(result[-1])]
        sharpen = sharpen_num if (o.convertor == "FBP" and o.fbp_sharpen) else -1
        x = tensor_sharpen(recs[-1], sharpen)
        out = self._img_stage(x, inn, self.noise_strength)
        return result, recs, out

    def progressive_denoiser(self, save_proj_state=False, convert=True, sharpen_num=42, noise=None):
        """proj stage -> FBP -> sharpen -> img stage, all on the GPU; returns [B,1,512,512] on the device."""
        o = self.opt
        if noise is None:
            self._next_noise_epoch()                                   # eager and graph replays alike: call k of a model uses epoch k
        if getattr(o, "cuda_graph", False) and noise is None and convert:
            result, recs, out = self._progressive_graphed(sharpen_num)
            self.proj_temp_clear()
            self.img_temp_clear()
            if save_proj_state:
                for k, r in enumerate(result):
                    self.proj_denoise_result[f"iter_{k + 1}"] = r.cpu().numpy()
            for k, r in enumerate(recs):
                self.proj_denoise_convert2img_result[f"iter_{k + 1}"] = r.cpu().numpy()
            for k, r in enumerate(out if o.save_it_state_img else out[-1:]):
                self.progressive_denoise_result[f"iter_{k + 1}"] = r.cpu().numpy()
            return out[-1].clone()                                     # the next replay overwrites the graph's own output buffer
        pn, inn = (None, None) if noise is None else noise
        result = self._proj_stage(self.ldproj, pn)
        self.proj_temp_clear()
        if save_proj_state:
            for k, r in enumerate(result):
                self.proj_denoise_result[f"iter_{k + 1}"] = r.cpu().numpy()
        if not convert:
            raise NotImplementedError("progressive_denoiser(convert=False) feeds a sinogram to the image model in the reference")
        if o.save_it_state_proj:
            recs = [self._convert_device(r) for r in result]
            for k, r in enumerate(recs):
                self.proj_denoise_convert2img_result[f"iter_{k + 1}"] = r.cpu().numpy()
            rec = recs[-1]
        else:
            rec = self._convert_device(result[-1])
            self._rec_device = rec
        sharpen = sharpen_num if (o.convertor == "FBP" and o.fbp_sharpen) else -1
        x = tensor_sharpen(rec, sharpen)
        out = self._img_stage(x, inn, self.noise_strength)
        self.img_temp_clear()
        if not o.save_it_state_proj:
            self.proj_denoise_convert2img_result["iter_1"] = rec.cpu().numpy()
        if o.save_it_state_img:
            for k, r in enumerate(out):
                self.progressive_denoise_result[f"iter_{k + 1}"] = r.cpu().numpy()
        else:
            self.progressive_denoise_result["iter_1"] = out[-1].cpu().numpy()
        return out[-1]

    def data_sample_load(self, ldct=Optional[Tensor], ldproj=Optional[Tensor], fdproj=Optional[np.ndarray], fdct=Optional[np.ndarray]):
        if self.opt.normal:
            raise NotImplementedError("normal=True (Yeo-Johnson) is off in every shipped config")
        if isinstance(ldct, torch.Tensor):
            self.ldct = ldct.to(self.opt.device)
            self.ldct_np = miu2pixel(ldct.squeeze().cpu().numpy())
        if isinstance(ldproj, torch.Tensor):
            self.ldproj = ldproj.to(self.opt.device, non_blocking=True).float().contiguous()
            self.ldproj_np = ldproj.squeeze().cpu().numpy()
        if isinstance(fdct, torch.Tensor):
            self.fdct = miu2pixel(fdct).squeeze().numpy()
        if isinstance(fdproj, torch.Tensor):
            self.fdproj = fdproj.squeeze().numpy()

    # ---- results ---------------------------------------------------------------------------
    def save_path_load(self, epoch, patient_name, slice_name):
        self.save_path = osp.join(self.save_root_path, f'Save_Iter_{epoch}', f'{patient_name}', f'{slice_name}')
        os.makedirs(self.save_path, exist_ok=True)

    def result_data_save(self, data_save=True):
        os.makedirs(self.save_path, exist_ok=True)
        if data_save:
            for ftype, fdata in (("prog_denoise_result", self.progressive_denoise_result), ("proj_denoise_result", self.proj_denoise_result),
                                 ("img_denoise_result", self.img_denoise_result), ("proj_denoise_result_2img", self.proj_denoise_convert2img_result)):
                if len(fdata) > 0:
                    np.savez_compressed(osp.join(self.save_path, f'{ftype}.npz'), **fdata)
        with open(osp.join(self.save_path, 'metric.json'), 'w') as f:
            f.write(json.dumps(self.metric_instance, sort_keys=False, indent=4, separators=(',', ': ')))

    def result_figure_save(self, mode="progressive", display=True, only_metric=False):
        """Metric part of the reference's result_figure_save (:596-763): LDCT at it=0 and every stored iterate of the stage, in the
        reference's order and key names.  The matplotlib figures themselves are reporting and out of scope."""
        if self.fdct is None:
            return
        store = {"progressive": (self.progressive_denoise_result, "deProg"), "dimg": (self.img_denoise_result, "deImg"),
                 "dproj2img": (self.proj_denoise_convert2img_result, "deProj2img")}[mode]
        if self.ldct_np is not None:
            self.metric_calculate(mode="LDCT", it=0, denoise_result=self.ldct_np)
        n_it = len([k for k in store[0] if isinstance(k, str) and k.startswith("iter_")]) or len(store[0])
        for i in range(1, n_it + 1):
            r_it = n_it + 1 - i
            key = f"iter_{r_it}" if f"iter_{r_it}" in store[0] else r_it
            self.metric_calculate(mode=store[1], it=r_it, denoise_result=miu2pixel(np.array(store[0][key]).squeeze()))

    def metric_calculate(self, mode="LDCT", **kwargs):
        """PSNR / SSIM of `denoise_result` (pixel units, [H,W] or [B,H,W]) against the full-dose image, on the device with the
        reference's definitions (:789-799: skimage compare_psnr(data_range=1), compare_ssim(win_size=11, data_range=1), NaN -> 0.5).
        fsim / vif / nqm are piq / NQM reporting metrics outside this path and are skipped."""
        from ipdm_pytorch_b200 import engine
        i = kwargs["it"]
        ld = kwargs["denoise_result"]
        ld = ld if isinstance(ld, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(ld, dtype=np.float32))
        fd = torch.from_numpy(np.ascontiguousarray(self.fdct, dtype=np.float32))
        ld, fd = ld.reshape(-1, *ld.shape[-2:]), fd.reshape(-1, *fd.shape[-2:])
        if fd.shape[0] == 1 and ld.shape[0] > 1:
            fd = fd.expand_as(ld)
        vals = engine.psnr_ssim(ld.to(self.opt.device).float().contiguous(), fd.to(self.opt.device).contiguous(), win_size=11).cpu().numpy()
        grp = self.metric_instance.setdefault(mode, DotDict()) if hasattr(self.metric_instance, "setdefault") else self.metric_instance[mode]
        if 'psnr' in self.opt.metrics:
            grp["psnr_iter_{}".format(i)] = float(vals[:, 0].mean())
        if 'ssim' in self.opt.metrics:
            grp["ssim_iter_{}".format(i)] = float(vals[:, 1].mean())

    def metric_update(self):
        self.metric_each_sample.append(self.metric_instance)

    def metric_total_save(self, epoch):
        keys = {}
        for m in self.metric_each_sample:
            for grp, d in m.items():
                for k, v in d.items():
                    keys.setdefault((grp, k), []).append(v)
        total = DotDict()
        for (grp, k), vals in keys.items():
            total.setdefault(grp, DotDict())[k] = float(np.mean(vals))
            total[grp][k + "_std"] = float(np.std(vals))
        self.metric_total = total
        os.makedirs(osp.join(self.save_root_path, f'Save_Iter_{epoch}'), exist_ok=True)
        with open(osp.join(self.save_root_path, f'Save_Iter_{epoch}', 'metric.json'), 'w') as f:
            f.write(json.dumps(self.metric_total, sort_keys=False, indent=4, separators=(',', ': ')))

    # ---- evaluation loop (reference test() :274-315, fit() :326-348) ---------------------------
    # SURVEY N2: `test_batch_size` slices go through the path together (the reference loops one slice at a time; batching is exact
    # here because every statistic is per slice), and the files of the NEXT batch are read and pinned on a worker thread while the
    # GPU works on the current one.  Results, metrics and save paths stay per slice, as the reference writes them.
    def _fetch_batch(self, ids):
        cols = self.test_dataset.collate([self.test_dataset[int(i)] for i in ids])
        pin = torch.cuda.is_available()
        return tuple(None if c is None else (c.contiguous().pin_memory() if pin else c.contiguous()) for c in cols)

    def _run_batch(self, epoch, ids, cols):
        ld_img, fd_proj, fd_img, ld_proj = cols
        if getattr(self.opt, "simulate_low_dose", False):                    # LD files on disk, if any, are not used
            fd = fd_proj if fd_proj is not None else fd_img
            if fd is None:
                raise ValueError("simulate_low_dose needs full-dose projections or images in the test dataset")
            ld_proj, ld_img = self.simulate_low_dose(fd, slice_ids=[int(i) for i in ids])
        self.temp_clear()
        self.data_sample_load(ldct=ld_img, ldproj=ld_proj, fdproj=fd_proj, fdct=fd_img)
        if self.opt.mode == "test_proj":
            self.proj_denoiser(self.ldproj)
            fig_mode = "dproj2img"
        elif self.opt.mode == "test_img":
            self.img_denoiser(self.ldct, mode="img_only")
            fig_mode = "dimg"
        else:
            self.progressive_denoiser()
            fig_mode = "progressive"
        names = ("progressive_denoise_result", "proj_denoise_result", "img_denoise_result", "proj_denoise_convert2img_result")
        full = {n: getattr(self, n) for n in names}
        per_slice = {n: getattr(self, n) for n in ("fdct", "ldct_np", "fdproj", "ldproj_np")}
        nb = len(ids)
        for j, idx in enumerate(ids):
            for n, d in full.items():                           # views of slice j, shaped like the reference's B = 1 results
                setattr(self, n, ResultTempDict({k: v[j:j + 1] for k, v in d.items()}))
            for n, v in per_slice.items():
                setattr(self, n, v[j] if (v is not None and nb > 1 and getattr(v, "ndim", 0) >= 3) else v)
            self.metric_clear()
            self.save_path_load(epoch, self.test_dataset.patient_name[idx], self.test_dataset.slice_name[idx])
            self.result_figure_save(mode=fig_mode, display=False)
            self.result_data_save(data_save=self.opt.test_result_data_save)
            self.metric_update()
        for n, d in full.items():
            setattr(self, n, d)
        for n, v in per_slice.items():
            setattr(self, n, v)

    @torch.no_grad()
    def test(self, epoch):
        from concurrent.futures import ThreadPoolExecutor
        n = len(self.test_dataset)
        if self.opt.test_numbers <= 0:
            self.opt.test_numbers = n
        if n == 0:
            print("test dataset is empty: nothing to do")
            return
        np.random.seed(9527)
        ids = np.sort(np.random.choice(n, self.opt.test_numbers, replace=False))
        bs = max(1, int(getattr(self.opt, "test_batch_size", 1)))
        batches = [ids[k:k + bs] for k in range(0, len(ids), bs)]
        with ThreadPoolExecutor(max_workers=1) as pool:
            fut = pool.submit(self._fetch_batch, batches[0])
            for k, b in enumerate(batches):
                cols = fut.result()
                if k + 1 < len(batches):
                    fut = pool.submit(self._fetch_batch, batches[k + 1])      # disk -> pinned host overlaps the GPU work below
                self._run_batch(epoch, b, cols)
        self.metric_total_save(epoch)

    def fit(self):
        if 'test' in self.opt.mode:
            self.test(0)
        else:
            raise NotImplementedError("training is outside the B200 inference path")
