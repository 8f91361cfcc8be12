"""Timing of the low-dose simulation kernels: python tools/bench_project.py [batch ...]  (default 16 64).

CUDA events around ipdm_fbp_project (transpose + projector) and ipdm_low_dose_noise (in-kernel Philox) after a warm-up of the same
shape.  Each timed call reads and writes buffers of its own, rotated so that one round of them exceeds the 126 MB L2: inputs come
from HBM, not from the previous call's cache lines.  Samples are counted from the geometry (rays x grid columns / rows where the
ray has a non-zero tap); bytes are the compulsory ones (projector: image read + sinogram written; noise: sinogram read + written).
"""
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import numpy as np
import torch

from ipdm_pytorch_b200 import engine, synthetic as S

NV, ND, NP = engine.N_VIEWS, engine.N_DET, engine.N_PIX
L2_BYTES = 126 << 20


def samples_per_slice():
    """Joseph samples with a tap inside the grid, summed over the 2000 x 912 rays (fp64, the kernel's parametrisation)."""
    th = S.view_angles()[:, None]
    al = (S.detector_angles().astype(np.float64) + 0.5 * S.DET_PITCH)[None, :]
    c, s = np.cos(th - al), np.sin(th - al)
    p = 59.5 * np.sin(al) / (42.0 / 512)
    xm = np.abs(c) >= np.abs(s)
    a, o = np.where(xm, c, s), np.where(xm, s, c)
    u0, g = np.where(xm, 255.5 - p / a, 255.5 + p / a), o / a
    m = np.arange(NP, dtype=np.float64)
    total = 0
    for v in range(NV):                                        # u(m) in [-1, 512) <=> at least one tap inside the grid
        u = u0[v][:, None] + (m[None, :] - 255.5) * g[v][:, None]
        total += int(((u >= -1) & (u < 512)).sum())
    return total


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.TimeoutExpired):
        return "unknown (nvidia-smi not readable)"


def timed(fn, n_sets, iters):
    for k in range(n_sets):                                    # warm-up: every buffer set once
        fn(k)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for i in range(iters):
        fn(i % n_sets)
    t1.record()
    t1.synchronize()
    return t0.elapsed_time(t1) / iters


def main():
    if not torch.cuda.is_available():
        raise SystemExit("bench_project.py measures the B200 kernels: it needs a CUDA device")
    batches = [int(b) for b in sys.argv[1:]] or [16, 64]
    dev = torch.device("cuda:0")
    plan = engine.FBPPlan(max_batch=max(batches))
    n_samp = samples_per_slice()
    print(f"card: {card()}")
    print(f"Joseph samples per slice: {n_samp / 1e9:.3f} G over {NV * ND} rays ({n_samp / (NV * ND):.0f} per ray)")
    print("| kernel | B | ms / call | ms / slice | G samples/s | GB/s (compulsory) |\n|---|---:|---:|---:|---:|---:|")
    img0 = torch.from_numpy(S.rasterize(S.phantom_ellipses(0))).to(dev)
    for b in batches:
        per_set = 4 * b * (NP * NP + NV * ND)
        n_sets = max(2, -(-2 * L2_BYTES // per_set))
        imgs = [(img0 * (1 + 0.01 * k)).expand(b, NP, NP).contiguous() for k in range(n_sets)]
        sinos = [torch.empty(b, NV, ND, device=dev) for _ in range(n_sets)]
        iters = max(10, 2000 // b)
        ms = timed(lambda k: plan.project(imgs[k], out=sinos[k]), n_sets, iters)
        print(f"| projector (transpose + Joseph) | {b} | {ms:.3f} | {ms / b:.3f} | {n_samp * b / ms / 1e6:.1f} | "
              f"{4 * b * (NP * NP + NV * ND) / ms / 1e6:.0f} |")
        outs = [torch.empty_like(s) for s in sinos]
        ms = timed(lambda k: engine.low_dose_noise(sinos[k], 0.25, seed=1, out=outs[k]), n_sets, iters)
        print(f"| low-dose noise (Philox) | {b} | {ms:.3f} | {ms / b:.4f} | - | {8 * b * NV * ND / ms / 1e6:.0f} |")
        del imgs, sinos, outs
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
