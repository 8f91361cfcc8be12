"""Parameter study of SART-TV on the fp64 reference implementation (oracle/tv_oracle.c), CPU only:
python tools/sart_tv_study.py [--quick]

Slice-0 ellipse raster, its Joseph projection (oracle/project_oracle.c), then noise-free data and the dose-reduction noise of
synthetic.add_noise at doses 0.25 and 0.1 (default_rng(7), clipped at 0).  S = 100 subsets, lambda = 1, eps = 1e-4 1/cm, 5 sweeps;
ntv in {0, 5, 10, 20} x alpha in {0.05, 0.1, 0.2}, each from x0 = 0 and from x0 = max(0, FBP).  Prints one markdown row per run:
the body RMSE (1/cm, pixels of the raster above 0.05) after every sweep.  --quick runs ntv = 20, alpha = 0.1 only.
"""
import os
import sys
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "ipdm-pytorch_b200"))
import numpy as np

import ipdm_pytorch_b200.synthetic as S
from oracle import fbp_oracle, project_oracle as P, tv_oracle as T

SUBSETS, SWEEPS, LAMBDA, EPS, BODY = 100, 5, 1.0, 1e-4, 0.05


def main():
    quick = "--quick" in sys.argv[1:]
    img = S.rasterize(S.phantom_ellipses(0))
    b0 = P.project(img)[0]
    body = img > BODY
    rmse = lambda r: float(np.sqrt(((r - img)[body] ** 2).mean()))
    grid = [(20, 0.1)] if quick else [(0, 0.0)] + [(n, a) for n in (5, 10, 20) for a in (0.05, 0.1, 0.2)]
    t0 = time.time()
    for name, dose in (("noise-free", None), ("dose 0.25", 0.25), ("dose 0.1", 0.1)):
        b = b0 if dose is None else np.maximum(S.add_noise(b0, dose, np.random.default_rng(7)), 0)
        b = b.astype(np.float32)
        fbp = fbp_oracle.convert(b[None])[0]
        print(f"\n### {name}: FBP {rmse(fbp):.4f}\n\n| ntv | alpha | start | body RMSE after sweeps 1..{SWEEPS} (1/cm) |\n|---:|---:|---|---|",
              flush=True)
        for init in ("zero", "fbp"):
            for ntv, alpha in grid:
                _, hist = T.sart(b, True, SWEEPS, SUBSETS, LAMBDA, history=True, ntv=ntv, tv_alpha=alpha or 0.1, tv_eps=EPS, init=init,
                                 x0=fbp[None] if init == "fbp" else None)
                r = ", ".join(f"{rmse(h):.4f}" for h in hist[0])
                print(f"| {ntv} | {alpha if ntv else '-'} | {init} | {r} |", flush=True)
    print(f"\n{time.time() - t0:.0f} s", flush=True)


if __name__ == "__main__":
    main()
