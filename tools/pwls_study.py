"""Parameter study of PWLS / OS-SQS on the fp64 reference implementation (oracle/pwls_oracle.c), CPU only:
python tools/pwls_study.py [--quick]

The setup of tools/sart_tv_study.py: slice-0 ellipse raster, its Joseph projection (oracle/project_oracle.c), then noise-free data
and the dose-reduction noise of synthetic.add_noise at doses 0.25 and 0.1 (default_rng(7), clipped at 0).  S = 100 subsets, 5
sweeps, FBP start; beta x delta grid (the weights use the data's dose; noise-free data is weighted as dose 1).  Prints D^L inside
the body, then one markdown row per run: the body RMSE (1/cm, pixels of the raster above 0.05) after every sweep.  For the chosen
point (CHOSEN, engine.PWLS_DEFAULTS) it also prints the run from 0, 10 sweeps at dose 0.1 next to plain SART's 10 sweeps, and
Phi after every sweep; at the end, the grid point with the least sum of the 5-sweep body RMSE at the two doses.  --quick runs the
chosen point only.
"""
import os
import sys
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "ipdm-pytorch_b200"))
import numpy as np

import ipdm_pytorch_b200.synthetic as S
from oracle import fbp_oracle, project_oracle as P, pwls_oracle as W, sart_oracle as Q

SUBSETS, SWEEPS, BODY = 100, 5, 0.05
BETAS = (3e3, 1e4, 3e4, 1e5, 3e5, 1e6, 3e6)
DELTAS = (0.0001, 0.0002, 0.0005, 0.001, 0.002, 0.005, 0.01)
CHOSEN = dict(beta=1e6, delta=0.0002)         # engine.PWLS_DEFAULTS


def main():
    quick = "--quick" in sys.argv[1:]
    img = S.rasterize(S.phantom_ellipses(0))
    b0 = P.project(img)[0]
    body = img > BODY
    rmse = lambda r: float(np.sqrt(((r - img)[body] ** 2).mean()))
    grid = [] if quick else [(be, de) for de in DELTAS for be in BETAS]
    c = CHOSEN
    final = {}
    t0 = time.time()
    for name, dose in (("dose 0.25", 0.25), ("dose 0.1", 0.1), ("noise-free", None)):
        b = b0 if dose is None else np.maximum(S.add_noise(b0, dose, np.random.default_rng(7)), 0)
        b = b.astype(np.float32)
        f = dose or 1.0
        fbp = fbp_oracle.convert(b[None])[0]
        dl = W.denominator(b, f)[0]
        print(f"\n### {name} (weights at dose {f}): FBP {rmse(fbp):.4f}; D^L in the body: median {np.median(dl[body]):.3g}, "
              f"range {dl[body].min():.3g} .. {dl[body].max():.3g}\n\n| beta | delta | start | body RMSE after sweeps 1..{SWEEPS} (1/cm) |"
              "\n|---:|---:|---|---|", flush=True)
        for beta, delta in grid:
            _, hist = W.pwls(b, True, SWEEPS, SUBSETS, f, beta, delta, init="fbp", x0=fbp[None], history=True)
            final[name, beta, delta] = rmse(hist[0, -1])
            print(f"| {beta:g} | {delta:g} | fbp | {', '.join(f'{rmse(h):.4f}' for h in hist[0])} |", flush=True)
        _, hist = W.pwls(b, True, SWEEPS, SUBSETS, f, c["beta"], c["delta"], init="zero", history=True)
        print(f"| {c['beta']:g} | {c['delta']:g} | zero | {', '.join(f'{rmse(h):.4f}' for h in hist[0])} |", flush=True)
        n = 10 if dose == 0.1 else SWEEPS
        _, hist = W.pwls(b, True, n, SUBSETS, f, c["beta"], c["delta"], init="fbp", x0=fbp[None], history=True)
        phi = [float(W.objective(b, h, f, c["beta"], c["delta"])[0]) for h in hist[0]]
        print(f"\nchosen point, FBP start, {n} sweeps: body RMSE {', '.join(f'{rmse(h):.4f}' for h in hist[0])}\n"
              f"Phi after every sweep: {', '.join(f'{p:.6g}' for p in phi)}", flush=True)
        if dose == 0.1:
            _, hs = Q.sart(b, True, 10, SUBSETS, 1.0, history=True)
            print(f"plain SART, 10 sweeps: body RMSE {', '.join(f'{rmse(h):.4f}' for h in hs[0])}", flush=True)
    if grid:
        score = {(be, de): final["dose 0.25", be, de] + final["dose 0.1", be, de] for be, de in grid}
        be, de = min(score, key=score.get)
        edge = be in (BETAS[0], BETAS[-1]) or de in (DELTAS[0], DELTAS[-1])
        print(f"\nbest grid point (sum of the 5-sweep body RMSE at doses 0.25 and 0.1): beta {be:g}, delta {de:g}"
              f"{' -- ON THE EDGE of the grid' if edge else ''}", flush=True)
    print(f"\n{time.time() - t0:.0f} s", flush=True)


if __name__ == "__main__":
    main()
