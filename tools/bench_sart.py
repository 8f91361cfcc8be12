"""Timing of the iterative convertor: python tools/bench_sart.py [batch ...]  (default 16 64).

CUDA events around ipdm_fbp_project_adjoint, plain SART (ipdm_fbp_sart_tv at the default options, ntv = 0), one TV step
(ipdm_fbp_tv_descent), SART-TV at the recommended setting (ipdm_fbp_sart_tv, ntv = 20, tv_alpha = 0.2, FBP start), PWLS at its defaults (ipdm_fbp_pwls, the sweeps
and subsets of SART, dose 0.25, FBP start) and the PWLS penalty alone (ipdm_fbp_pwls_penalty) after a warm-up of the same shape,
which also builds SART's geometry tables.  Each timed call reads and writes buffers of its own, rotated so that one round of them exceeds the
126 MB L2: inputs come from HBM, not from the previous call's cache lines.  Weight updates are counted from the geometry: the
non-zero entries of A (Joseph taps inside the grid), which the adjoint applies once each.  The TV step's rate is taken on its
compulsory bytes, 16 per pixel: x read and written, g written and read; the penalty's on 12 per pixel: x read, grad R and d^R
written.
"""
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tools"))
import numpy as np
import torch

from bench_project import L2_BYTES, card, timed
from ipdm_pytorch_b200 import engine, synthetic as S

NV, ND, NP = engine.N_VIEWS, engine.N_DET, engine.N_PIX
SART_TV = dict(ntv=20, tv_alpha=0.2, init="fbp")           # the recommended SART-TV setting (DESIGN 8)
TV_BYTES_PER_PIXEL = 16
PENALTY_BYTES_PER_PIXEL = 12
PWLS = dict(dose=0.25, init="fbp", **engine.PWLS_DEFAULTS)


def entries_per_slice():
    """Non-zero entries of A: taps floor(u), floor(u) + 1 inside [0, 512) of every sample, summed over the 2000 x 912 rays (fp64)."""
    th = S.view_angles()[:, None]
    al = (S.detector_angles().astype(np.float64) + 0.5 * S.DET_PITCH)[None, :]
    c, s = np.cos(th - al), np.sin(th - al)
    p = 59.5 * np.sin(al) / (42.0 / 512)
    xm = np.abs(c) >= np.abs(s)
    a, o = np.where(xm, c, s), np.where(xm, s, c)
    u0, g = np.where(xm, 255.5 - p / a, 255.5 + p / a), o / a
    m = np.arange(NP, dtype=np.float64)
    total = 0
    for v in range(NV):
        k = np.floor(u0[v][:, None] + (m[None, :] - 255.5) * g[v][:, None])
        total += int(((k >= 0) & (k < NP)).sum() + ((k + 1 >= 0) & (k + 1 < NP)).sum())
    return total


def main():
    if not torch.cuda.is_available():
        raise SystemExit("bench_sart.py measures the B200 kernels: it needs a CUDA device")
    batches = [int(b) for b in sys.argv[1:]] or [16, 64]
    dev = torch.device("cuda:0")
    plan = engine.FBPPlan(max_batch=max(batches))
    n_upd = entries_per_slice()
    d = engine.SART_DEFAULTS
    print(f"card: {card()}")
    print(f"non-zero entries of A per slice: {n_upd / 1e9:.3f} G; SART defaults: {d}")
    print("| operation | B | ms / call | ms / slice | G weight-updates/s |\n|---|---:|---:|---:|---:|")
    ell = S.phantom_ellipses(0)
    sino0 = torch.from_numpy(S.fan_sinogram(ell).astype(np.float32)).to(dev)
    for b in batches:
        per_set = 4 * b * (NP * NP + NV * ND)
        n_sets = max(2, -(-2 * L2_BYTES // per_set))
        sinos = [(sino0 * (1 + 0.01 * k)).expand(b, NV, ND).contiguous() for k in range(n_sets)]
        imgs = [torch.empty(b, NP, NP, device=dev) for _ in range(n_sets)]
        iters = max(10, 1000 // b)
        ms = timed(lambda k: plan.project_adjoint(sinos[k], out=imgs[k]), n_sets, iters)
        print(f"| adjoint (A^T y) | {b} | {ms:.3f} | {ms / b:.3f} | {n_upd * b / ms / 1e6:.1f} |")
        ms = timed(lambda k: plan.project(imgs[k], out=sinos[k]), n_sets, iters)
        print(f"| projector (A x), for reference | {b} | {ms:.3f} | {ms / b:.3f} | {n_upd * b / ms / 1e6:.1f} |")
        ms_sart = timed(lambda k: plan.sart(sinos[k], out=imgs[k], **d), n_sets, max(3, 64 // b))
        print(f"| SART, {d['iterations']} sweeps x {d['subsets']} subsets | {b} | {ms_sart:.3f} | {ms_sart / b:.3f} | "
              f"{2 * d['iterations'] * n_upd * b / ms_sart / 1e6:.1f} |")
        ms = timed(lambda k: plan.sart(sinos[k], out=imgs[k], **d, **SART_TV), n_sets, max(3, 64 // b))
        print(f"| SART-TV {SART_TV}: {ms / ms_sart - 1:+.1%} over SART | {b} | {ms:.3f} | {ms / b:.3f} | "
              f"{2 * d['iterations'] * n_upd * b / ms / 1e6:.1f} |")
        ms = timed(lambda k: plan.pwls(sinos[k], out=imgs[k], iterations=d["iterations"], subsets=d["subsets"], **PWLS), n_sets,
                   max(3, 64 // b))
        print(f"| PWLS {PWLS}: {ms / ms_sart:.2f}x plain SART | {b} | {ms:.3f} | {ms / b:.3f} | "
              f"{2 * d['iterations'] * n_upd * b / ms / 1e6:.1f} |")
        del sinos, imgs
        n_img = max(2, -(-2 * L2_BYTES // (4 * b * NP * NP)))
        xs = [torch.rand(b, NP, NP, device=dev) for _ in range(n_img)]
        ms = timed(lambda k: plan.tv_descent(xs[k], 1, 1e-4), n_img, max(50, 4000 // b))
        print(f"| one TV step (gradient + update): {TV_BYTES_PER_PIXEL * b * NP * NP / ms / 1e6:.0f} GB/s on its compulsory bytes "
              f"| {b} | {ms:.4f} | {ms / b:.4f} | - |")
        ms = timed(lambda k: plan.pwls_penalty(xs[k]), n_img, max(50, 4000 // b))
        print(f"| PWLS penalty (grad R, d^R): {PENALTY_BYTES_PER_PIXEL * b * NP * NP / ms / 1e9:.2f} TB/s on its compulsory bytes "
              f"| {b} | {ms:.4f} | {ms / b * 1e3:.2f} us | - |")
        del xs
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
