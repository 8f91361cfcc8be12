#!/usr/bin/env python
"""Benchmark of the IPDM domain-progressive inference path (BASELINE.json metric: slices/sec).

    python bench.py --gpus N --steps K --warmup W            # this build (libipdm_b200.so), one rank per GPU
    python bench.py --impl reference --gpus N --steps K ...   # the reference algorithm on the host CPU (oracle port)
    python bench.py ... --dump-outputs DIR                    # also save the last timed step's result, to compare two builds

A "step" is one pass of the whole hot path over one batch of synthetic slices per GPU:
projection-domain guided process (t_start_proj) -> FBP -> sharpen -> image-domain guided process
(t_start_img) -> "ultra" pass [5,5,5], i.e. `progressive_denoiser` of the reference with
convertor="FBP", ultra_img_denoise=True on 2000x912 sinograms -> 512x512 images.
`value` is timed with inputs resident in HBM; `e2e` goes through the reference-facing API
(`progressive_domain_denoiser.data_sample_load` + `.progressive_denoiser`) from pinned host buffers
to a host result.  Slices are sharded across ranks with no collective on the data path (weak
scaling); the only collective is the final gather of the [B,1,512,512] results.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(REPO, "ipdm-pytorch_b200")
for p in (REPO, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

HBM_FALLBACK_GBS, TENSOR_FALLBACK_TFLOPS = 6650.0, 1590.0        # /opt/skills/guides/B200_PROFILING.md
# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel from an `ncu --set full` capture
CONV_TC_NCU_TRAFFIC = dict(bytes_per_launch=2.748e9,
                           note="profiles/r02_conv_halo_fused_ncu_full.md: conv_halo_fused_kernel<128,8,bf16>, 16 x 500x228, GroupNorm+SiLU -> 128->128 3x3 "
                                "+residual: 1.868 GB read + 0.880 GB written per launch; algorithmic bytes of that layer 2.80 GB (raw fp32 input 0.93 + fp32 "
                                "residual 0.93 + fp32 output 0.93).  The unfused conv_halo_persistent_kernel<128,6> moves 2.28 GB per launch.")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=16, help="slices per GPU per step (BASELINE.json configs[2]: batch 16 on one B200)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "tf32", "fp32"],
                    help="UNet operand precision (configs[2]: bf16 UNet, fp32 sampler state); tf32 / fp32 are the parity modes")
    ap.add_argument("--t_start_proj", type=int, nargs="+", default=[15, 15, 15])
    ap.add_argument("--t_start_img", type=int, nargs="+", default=[15, 15, 15])
    ap.add_argument("--skip_cpu_baseline", action="store_true")
    ap.add_argument("--skip_cpu_whole_slice", action="store_true", help="do not run the one unsampled whole slice on the host (~150 s)")
    ap.add_argument("--skip_extras", action="store_true", help="only the headline line: no modes / c1 / cuda_graph / C4 / C5 sub-reports")
    ap.add_argument("--cuda_graph", type=int, default=0, help="1: capture the whole progressive pass in one CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (rank 0's denoised images, float32) as DIR/denoised_images.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory, images):
    """Saves the [B,1,512,512] result of the last timed step; beyond DUMP_LIMIT_BYTES only the leading slices are kept."""
    import numpy as np
    per_slice = images[0].numel() * 4
    images = images[:max(1, DUMP_LIMIT_BYTES // per_slice)]
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "denoised_images.npy"), images.float().cpu().numpy())


def peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return dict(hbm=d["hbm_gbs"], tensor=d.get("bf16_tflops_sustained", d["bf16_tflops"]), which="measured (MEASURED_PEAKS.json; sustained bf16)")
    return dict(hbm=HBM_FALLBACK_GBS, tensor=TENSOR_FALLBACK_TFLOPS, which="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower() == "active" for r in self.rows)]
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons, samples=len(sm))


# -------------------------------------------------------------------------------------------------
# CPU legs (oracle port): the reference algorithm on the host cores, bounded sample
# -------------------------------------------------------------------------------------------------
_CPU = {}


def _cpu_setup():
    """Oracle networks, inputs and tables of the CPU legs (built once per process; weights are the same seed-0 random init)."""
    if not _CPU:
        import torch
        from oracle import ipdm_oracle as O
        torch.set_num_threads(len(os.sched_getaffinity(0)))
        torch.manual_seed(0)
        g = torch.Generator().manual_seed(0)
        _CPU.update(O=O, pnet=O.UNetOracle(**O.PROJ_UNET).eval(), inet=O.UNetOracle(**O.IMG_UNET).eval(), g=g,
                    xp=3 * torch.rand(1, 1, 2000, 912, generator=g), xi=0.2 * torch.rand(1, 1, 512, 512, generator=g),
                    ptab=O.Tables(1000, 5), itab=O.Tables(1000, 1), cores=torch.get_num_threads())
    return _CPU


CPU_SAMPLE_PROJ, CPU_SAMPLE_IMG = 3, 4           # forwards + reverse steps per bounded sample


def cpu_sample_fraction(t_start_proj, t_start_img):
    """Fraction of ONE slice a bounded sample covers: 3 of the sum(t_start_proj) projection steps and 4 of the sum(t_start_img)+15
    image steps.  For the shipped lists (45 + 60 steps) both are exactly 1/15 of the slice; otherwise the time-weighted mean is used."""
    return CPU_SAMPLE_PROJ / sum(t_start_proj), CPU_SAMPLE_IMG / (sum(t_start_img) + 15)


def cpu_reference_sample(t_start_proj, t_start_img):
    """One bounded sample of the reference algorithm (oracle port) on the host cores: 3 projection-domain reverse steps (UNet forward at
    2000x912 + p_sample_condition) and 4 image-domain ones at 512x512, i.e. 1/15 of one slice of the shipped configuration.  The
    FBP (1 per slice, ~1 % of a slice) and the once-per-process delta-map / curve are NOT in the sample (they are in the whole-slice
    run), so the sample slightly favours the reference.  Returns the measured seconds and the slices/s it implies."""
    import torch
    c = _cpu_setup()
    O = c["O"]
    t0 = time.perf_counter()
    x = c["xp"]
    for k in range(CPU_SAMPLE_PROJ):
        t = 7 + k
        eps = c["pnet"](x, torch.full((1,), t, dtype=torch.long))
        x = O.p_sample_condition(c["ptab"], eps, x, c["xp"], t, 0.4, False, torch.randn(x.shape, generator=c["g"]))
    t_proj = time.perf_counter() - t0
    t1 = time.perf_counter()
    x = c["xi"]
    for k in range(CPU_SAMPLE_IMG):
        t = 7 + k
        eps = c["inet"](x, torch.full((1,), t, dtype=torch.long))
        x = O.p_sample_condition(c["itab"], eps, x, c["xi"], t, 0.45, True, torch.randn(x.shape, generator=c["g"]))
    t_img = time.perf_counter() - t1
    fp, fi = cpu_sample_fraction(t_start_proj, t_start_img)
    per_slice = t_proj / fp + t_img / fi
    sample_s = t_proj + t_img
    return dict(sample_s=sample_s, per_slice_s=per_slice, slice_fraction=sample_s / per_slice, t_proj_step=t_proj / CPU_SAMPLE_PROJ,
                t_img_step=t_img / CPU_SAMPLE_IMG, cores=c["cores"],
                sample=f"{CPU_SAMPLE_PROJ} proj reverse steps at 2000x912 ({t_proj / CPU_SAMPLE_PROJ:.2f} s each: UNet forward + guided step) + "
                       f"{CPU_SAMPLE_IMG} img reverse steps at 512x512 ({t_img / CPU_SAMPLE_IMG:.2f} s each) of the oracle port (torch CPU fp32), "
                       f"= {sample_s / per_slice:.4f} of one slice ({sum(t_start_proj)} + {sum(t_start_img) + 15} steps per slice; FBP and delta-map "
                       f"not sampled)")


def cpu_reference_whole_slice(t_start_proj, t_start_img):
    """ONE whole slice of the reference algorithm on the host, nothing extrapolated: projection stage (incl. the delta-map / lambda
    curve / per-step lambda maps on the host), FBP (C oracle, OpenMP), sharpen, image stage + ultra pass."""
    import torch
    from ipdm_pytorch_b200 import synthetic
    c = _cpu_setup()
    O = c["O"]
    x = torch.from_numpy(synthetic.cheap_sinogram(1, seed=100))[:, None].contiguous()
    g = torch.Generator().manual_seed(1)
    n_p, n_i = sum(t_start_proj) + len(t_start_proj), sum(t_start_img) + len(t_start_img) + 18
    pn = [torch.randn(1, 1, 2000, 912, generator=g) for _ in range(n_p)]
    inn = [torch.randn(1, 1, 512, 512, generator=g) for _ in range(n_i)]
    t0 = time.perf_counter()
    st = {}
    out = O.progressive_denoise(c["pnet"], c["inet"], x, pn, inn, t_start_proj=tuple(t_start_proj), t_start_img=tuple(t_start_img),
                                ultra=True, stages=st)
    dt = time.perf_counter() - t0
    assert tuple(out.shape) == (1, 1, 512, 512)
    return dt


def run_reference(args, rank, world):
    """Reference arm: the reference algorithm's CPU implementation (oracle port; the Python reference itself cannot travel to the GPU
    box) on all host cores.  One step = one bounded sample (1/15 of a slice, ~10 s) and `ms_per_step` is its MEASURED duration, so
    steps x ms_per_step is the real timed region; `value` = slices per second that sample implies.  During warm-up one WHOLE slice
    is run once, unsampled, and reported beside the sampled figure."""
    if rank != 0:
        return
    whole = None
    if args.warmup > 0 and not args.skip_cpu_whole_slice:
        whole = cpu_reference_whole_slice(args.t_start_proj, args.t_start_img)
    vals, secs, last = [], [], None
    for i in range(args.warmup + args.steps):
        last = cpu_reference_sample(args.t_start_proj, args.t_start_img)
        if i >= args.warmup:
            vals.append(last["per_slice_s"]); secs.append(last["sample_s"])
    per_slice = sum(vals) / len(vals)
    v = 1.0 / per_slice
    cfg = base_config(args, args.batch, world)
    cfg.update(note="reference algorithm on the host CPU (oracle port: torch CPU UNet + C FBP), one slice at a time (the reference cannot batch): "
                    "the batch of the workload is B x one slice; each step is a bounded sample of one slice")
    cpu = dict(value=v, unit="slices/s", cores=last["cores"], kind="port", sample=last["sample"], sampled_s_per_slice=per_slice)
    if whole is not None:
        cpu.update(whole_slice_s=whole, whole_slice_value=1.0 / whole, sampled_over_whole=per_slice / whole,
                   whole_note="one complete slice (45 + 60 forwards, delta-map, lambda maps, FBP, sharpen), run once during warm-up")
    line = dict(metric="ipdm_progressive_slices_per_sec", value=v, unit="slices/s", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * sum(secs) / len(secs), higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                impl="reference", config=cfg, cpu_baseline=cpu,
                e2e=dict(value=v, unit="slices/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0,
                slices_per_step=last["slice_fraction"])
    print(json.dumps(line))


def workload_name(args, batch):
    return (f"IPDM progressive inference, convertor=FBP, t_start_proj={args.t_start_proj}, t_start_img={args.t_start_img} + ultra [5,5,5], "
            f"{batch} slice(s)/GPU/step, sinogram 2000x912 -> image 512x512, random-init UNets (28.4M + 29.1M params)")


def base_config(args, batch, world):
    """`config` keys shared by both arms (the driver compares them)."""
    return dict(workload=workload_name(args, batch), global_batch=world * batch, parallelism=f"slice-sharded x{world}, no data-path collective")


# -------------------------------------------------------------------------------------------------
# B200 arm
# -------------------------------------------------------------------------------------------------
def run_b200(args, rank, world, local_rank):
    import numpy as np
    import torch
    import torch.distributed as dist
    from Config.default_config import default_cfg
    from ipdm_pytorch_b200 import engine, synthetic
    from Utils.train_test_utils import progressive_domain_denoiser

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    B = args.batch
    import contextlib
    import io
    import tempfile
    with contextlib.redirect_stdout(io.StringIO()):          # the reference's option loader prints; stdout carries ONE JSON line
        opt = default_cfg(["--load_option_path", os.path.join(PKG, "Config/Mayo-Config/test_progressive_option.json"), "--device", f"cuda:{local_rank}"])
    opt.load_img_model_path = opt.load_proj_model_path = None
    for k in ("test_dataset_path_FD_img", "test_dataset_path_LD_img", "test_dataset_path_FD_proj", "test_dataset_path_LD_proj"):
        setattr(opt, k, None)
    torch.manual_seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        model = progressive_domain_denoiser(opt, result_save_path=tempfile.mkdtemp(prefix="ipdm_bench_"))
        model.update_opt(dict(convertor="FBP", save_it_state_img=False, save_it_state_proj=False, ultra_img_denoise=True,
                              t_start_proj=args.t_start_proj, t_start_img=args.t_start_img, precision=args.precision, noise_seed=1234 + rank,
                              cuda_graph=bool(args.cuda_graph)))
    # synthetic slices of this rank's shard (weak scaling: B per GPU), pinned on the host
    host = torch.from_numpy(synthetic.cheap_sinogram(B, seed=100 + rank))[:, None].contiguous().pin_memory()
    host_out = torch.empty(B, 1, 512, 512).pin_memory()
    resident = host.to(dev)

    def step_resident():
        model.ldproj = resident
        return model.progressive_denoiser()

    gathered_shape = []

    def step_e2e():
        """The call a user makes: pinned host tensors -> data_sample_load (H2D inside) -> progressive_denoiser -> host result; with
        N > 1 ranks the final gather of the [B,1,512,512] results (the only collective of the path) is part of the step."""
        model.data_sample_load(ldct=None, ldproj=host, fdproj=None, fdct=None)
        out = model.progressive_denoiser()
        if world > 1:
            from ipdm_pytorch_b200.sharding import gather_slices
            full = gather_slices(out.contiguous(), world * B)
            gathered_shape[:] = list(full.shape)
            if rank == 0:
                host_full.copy_(full, non_blocking=True)
        else:
            host_out.copy_(out, non_blocking=True)
        return out

    host_full = torch.empty(world * B, 1, 512, 512).pin_memory() if (world > 1 and rank == 0) else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            out = fn()
        b.record()
        barrier()
        ms = a.elapsed_time(b)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms, out

    engine.launch_count_reset()
    for w_i in range(args.warmup):
        step_resident()
        if w_i == 0:
            launches_first_step = engine.launch_count()          # graph mode: the kernels recorded by the capture pass = kernels per replay
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    engine.launch_count_reset()
    ms, out = timed(step_resident, args.steps)
    launches = engine.launch_count()
    if args.cuda_graph and launches == 0 and args.warmup > 0:
        launches = launches_first_step * args.steps                  # replays do not pass through the host-side launch counter
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)           # before any later call can reuse the result's memory
    step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)
    if world > 1:
        assert gathered_shape and gathered_shape[0] == world * B

    # ---- sub-reports: the other BASELINE configs and precision modes (short: 1 warm-up + 1-2 steps each) ----
    extras = {}
    if not args.skip_extras:
        def sub(batch, steps, host_src=None, **opts):
            """slices/s of `steps` resident steps at `batch` slices per GPU after one warm-up step, with `opts` applied to the model."""
            with contextlib.redirect_stdout(io.StringIO()):
                model.update_opt(dict(opts))
            src = resident if host_src is None else host_src
            model.ldproj = src[:batch].contiguous()
            fn = lambda: model.progressive_denoiser()
            fn()
            m, _ = timed(fn, steps)
            return dict(slices_per_s=world * batch * steps / (m / 1e3), ms_per_step=m / steps, slices_per_gpu_per_step=batch, steps=steps, warmup=1)

        base = dict(precision=args.precision, cuda_graph=bool(args.cuda_graph), t_start_proj=args.t_start_proj, t_start_img=args.t_start_img)
        if world == 1:
            extras["modes"] = {
                "tf32": dict(sub(B, 2, precision="tf32"), note="tf32 mode: kind::tf32 tensor-core layers, exact CUDA-core thin layers (what the reference does on its own GPU)"),
                "fp32": dict(sub(B, 1, precision="fp32"), note="fp32 mode: 3xTF32 split, the mode that meets the 1 HU parity bar"),
            }
            extras["c1_single_slice_fp32"] = dict(sub(1, 2, precision="fp32"), note="BASELINE configs[0]: one slice, fp32 mode, default lists, ultra on")
            extras["c1_single_slice_bf16"] = sub(1, 2, precision="bf16")
            extras["cuda_graph"] = dict(sub(B, 2, precision=args.precision, cuda_graph=True), note="whole progressive pass replayed as ONE CUDA graph (capture in the warm-up step)")
            with contextlib.redirect_stdout(io.StringIO()):
                model.update_opt(base)
        else:
            # BASELINE configs[3]: t_start_proj=[15,12,10,10] + image stage, a FIXED global batch of 64 slices split over the ranks (strong scaling)
            per_rank = 64 // world
            micro = min(per_rank, 16)
            c4_host = torch.from_numpy(synthetic.cheap_sinogram(micro, seed=300 + rank))[:, None].contiguous().to(dev)
            with contextlib.redirect_stdout(io.StringIO()):
                model.update_opt(dict(t_start_proj=[15, 12, 10, 10]))

            def c4_step():
                for _ in range(per_rank // micro):
                    model.ldproj = c4_host
                    o = model.progressive_denoiser()
                return o
            c4_step()
            m, _ = timed(c4_step, 1)
            extras["c4_strong_global64"] = dict(slices_per_s=64 / (m / 1e3), ms_per_step=m, global_batch=64, slices_per_gpu=per_rank, micro_batch=micro, scaling="strong",
                                                t_start_proj=[15, 12, 10, 10], steps=1, warmup=1,
                                                note="BASELINE configs[3]: 64 slices in total, 64/N per GPU in micro-batches of <= 16; time = max over ranks")
            with contextlib.redirect_stdout(io.StringIO()):
                model.update_opt(base)
            if world == 8:
                # BASELINE configs[4]: a 512-slice volume over 8 GPUs = 64 slices per GPU in 4 micro-batches of 16, then ONE gather of the volume
                from ipdm_pytorch_b200.sharding import gather_slices
                vol_out = torch.empty(64, 1, 512, 512, device=dev)

                def c5_step():
                    for k in range(4):
                        model.ldproj = resident
                        vol_out[k * 16:(k + 1) * 16] = model.progressive_denoiser()
                    return gather_slices(vol_out, 512)
                m, full = timed(c5_step, 1)
                extras["c5_volume512_8gpu"] = dict(slices_per_s=512 / (m / 1e3), ms=m, slices=512, gathered_shape=list(full.shape), steps=1,
                                                   note="BASELINE configs[4]: 512 slices, 64 per GPU in micro-batches of 16, final all-gather of the 512 MiB volume inside the timed region")

    if rank != 0:
        return
    value = world * B * args.steps / (ms / 1e3)
    e2e = world * B * args.steps / (ms_e2e / 1e3)
    # per-family profile of ONE extra step (CUDA events around every launch, on the launching stream)
    engine.profile_enable(True)
    step_resident()
    prof = engine.profile_collect()
    engine.profile_enable(False)
    pk = peaks()
    tc_ms, tc_flops, tc_n = prof["conv_halo_persistent"]                  # the dominant kernel of the step
    fam_ms = tc_ms + prof["conv_tc"][0]
    fam_flops = tc_flops + prof["conv_tc"][1]
    total_prof_ms = sum(v[0] for v in prof.values())
    kind = {"bf16": "kind::f16 (bf16 operands, fp32 accumulate)", "tf32": "kind::tf32", "fp32": "kind::tf32 x3 (3xTF32 split)"}[args.precision]
    if args.precision == "fp32" or not tc_ms:                              # the 3xTF32 mode runs the one-tile kernel: report the family
        tc_ms, tc_flops, tc_n = fam_ms, fam_flops, tc_n + prof["conv_tc"][2]
        kname = f"conv_tc_kernel<N,S,SPLIT> (tcgen05 {kind} implicit-GEMM conv)"
    else:
        kname = (f"conv_halo_fused_kernel<N,NB,op,NA> / conv_halo_persistent_kernel<N,NB> (tcgen05 {kind} implicit-GEMM 3x3 conv, halo reuse, persistent; "
                 "the fused form applies GroupNorm+SiLU on the operand path and runs the upsample convs as four output-parity phases)")
    roof = dict(bound="tensor", kernel=kname, achieved=tc_flops / (tc_ms * 1e-3) / 1e12 if tc_ms else None,
                peak=pk["tensor"], unit="TFLOP/s", traffic=CONV_TC_NCU_TRAFFIC["bytes_per_launch"] if args.precision == "bf16" else None,
                traffic_note=CONV_TC_NCU_TRAFFIC["note"], peak_source=pk["which"],
                note="achieved = layer FLOPs (2*pixels*taps*K*C_out with K padded to the operand stride; discarded tile columns not counted; an upsample conv counts as the 3x3 conv on the upsampled image it replaces, of which 16/36 is issued) of every launch of this kernel in one profiled step / their summed "
                     "CUDA-event time on the launching stream; peak is dense bf16 (a kind::tf32 MMA runs at half that rate, so 0.5 is the "
                     "ceiling in tf32 mode).  conv_tc_family_* = the same over ALL tensor-core conv kernels (adds 1x1 / stride-2 / N=16 / qkv "
                     "layers, most of which are HBM-bound)",
                share_of_step=tc_ms / total_prof_ms if total_prof_ms else None, launches_per_step=tc_n,
                conv_tc_family_achieved=fam_flops / (fam_ms * 1e-3) / 1e12 if fam_ms else None,
                conv_tc_family_share_of_step=fam_ms / total_prof_ms if total_prof_ms else None)
    roof["frac"] = roof["achieved"] / roof["peak"] if roof["achieved"] else None
    if args.precision != "fp32" and prof["conv_halo_persistent"][0]:
        # the family straddles the ridge (128/256-channel layers tensor-bound, 64-channel image layers HBM-bound with their fp32 residual
        # stream): time the launches would take with EACH at its own roof / their measured time
        r_ms, m_ms, r_bytes = engine.profile_roofline("conv_halo_persistent", pk["tensor"] * (0.5 if args.precision == "tf32" else 1.0), pk["hbm"])
        roof["mixed"] = dict(frac=r_ms / m_ms if m_ms else None, roof_ms=round(r_ms, 2), measured_ms=round(m_ms, 2), algorithmic_gb=round(r_bytes / 1e9, 1),
                             note="sum over the launches of this kernel of max(FLOPs / tensor peak, algorithmic bytes / HBM peak), divided by their "
                                  "measured time: the fraction of the per-launch roofline (tensor OR HBM, whichever binds that layer)")
    families = {}
    for k, (m, w, n) in prof.items():
        unit = "TFLOP/s" if k in ("conv_tc", "conv_halo_persistent", "attention") else "GB/s"
        rate = (w / (m * 1e-3) / (1e12 if unit == "TFLOP/s" else 1e9)) if m else None
        families[k] = dict(ms=round(m, 3), launches=n, rate=None if rate is None else round(rate, 2), unit=unit,
                           frac_of_peak=None if rate is None else round(rate / (pk["tensor"] if unit == "TFLOP/s" else pk["hbm"]), 4))
    p_flops = model.proj_model.cuda_handle().flops(B, 2000, 912)
    i_flops = model.img_model.cuda_handle().flops(B, 512, 512)
    step_flops = sum(args.t_start_proj) * p_flops + (sum(args.t_start_img) + 15) * i_flops
    line = dict(metric="ipdm_progressive_slices_per_sec", value=value, unit="slices/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
                ms_per_step=ms / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype={"tf32": "tf32 (fp32 state, tcgen05 kind::tf32, fp32 accumulate)", "fp32": "f32 (3xTF32)", "bf16": "bf16"}[args.precision],
                data="synthetic",
                config=dict(base_config(args, B, world),
                            l2="working set (activation arena of several GB per step) >> 126 MB L2; no explicit flush needed",
                            noise="in-kernel Philox4x32-10", cuda_graph=bool(args.cuda_graph), unet_tflop_per_step=step_flops / 1e12),
                e2e=dict(value=e2e, unit="slices/s", h2d_bytes_per_step=int(world * host.numel() * 4), d2h_bytes_per_step=int(world * host_out.numel() * 4),
                         ms_per_step=ms_e2e / args.steps),
                gpu_launches=int(launches), clocks=clocks, roofline=roof, kernel_families=families,
                unet_effective_tflops=step_flops * args.steps / (ms * 1e-3) / 1e12)
    line["e2e"]["note"] = ("data_sample_load(pinned host sinograms) + progressive_denoiser + D2H of the result" +
                           ("; the final all-gather of the results over NCCL is inside the timed region" if world > 1 else ""))
    line.update(extras)
    line["fbp_batch64"] = fbp_batch64(dev, pk)
    if not args.skip_cpu_baseline and world == 1:             # rank 0 at N=1 only
        cpu_reference_sample(args.t_start_proj, args.t_start_img)                       # warm-up (thread pools, oneDNN primitives)
        c = cpu_reference_sample(args.t_start_proj, args.t_start_img)
        line["cpu_baseline"] = dict(value=1.0 / c["per_slice_s"], unit="slices/s", cores=c["cores"], kind="port", sample=c["sample"],
                                    sampled_s_per_slice=c["per_slice_s"])
        if not args.skip_cpu_whole_slice:
            whole = cpu_reference_whole_slice(args.t_start_proj, args.t_start_img)
            line["cpu_baseline"].update(whole_slice_s=whole, whole_slice_value=1.0 / whole, sampled_over_whole=c["per_slice_s"] / whole,
                                        whole_note="one complete slice on the host (45 + 60 forwards, delta-map, lambda maps, FBP, sharpen), nothing extrapolated")
    print(json.dumps(line))


def fbp_batch64(dev, pk):
    """BASELINE.json configs[1]: the FBP convertor alone on 64 sinograms (fan-beam weight + ramp filter + pixel-driven backprojection).
    Algorithmic HBM bytes per slice: sinogram read + filtered write + filtered read + image write; the backprojection itself is bound
    by the 2000 x 512 x 512 pixel-view updates per slice (gather + interpolate from L1/shared), not by HBM."""
    import torch
    from ipdm_pytorch_b200 import engine, synthetic
    n = 64
    sino = torch.from_numpy(synthetic.cheap_sinogram(4, seed=7)).to(dev).repeat(n // 4, 1, 1).contiguous()
    plan = engine.FBPPlan(max_batch=n)
    out = torch.empty(n, 512, 512, device=dev)
    for _ in range(2):
        plan.forward(sino, out=out)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(5):
        plan.forward(sino, out=out)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 5
    bytes_alg = n * (3 * 2000 * 912 * 4 + 512 * 512 * 4)
    return dict(workload="FBP convertor alone, 64 sinograms 2000x912 -> 512x512", ms=round(ms, 3), slices_per_s=round(n / (ms * 1e-3), 1),
                algorithmic_gb_s=round(bytes_alg / (ms * 1e-3) / 1e9, 1), frac_of_hbm=round(bytes_alg / (ms * 1e-3) / 1e9 / pk["hbm"], 4),
                pixel_view_updates_per_s=round(n * 2000 * 512 * 512 / (ms * 1e-3) / 1e9, 1), updates_unit="G/s")


def main():
    args = parse()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        if rank == 0:
            # torchrun exports OMP_NUM_THREADS=1; the reference arm uses every host core it is allowed to run on
            os.environ["OMP_NUM_THREADS"] = str(len(os.sched_getaffinity(0)))
            run_reference(args, rank, world)
        return
    import torch
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_b200(args, rank, world, local_rank)
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
