"""Device-resident timing of kernel C with a λ-map (the patch operator's up-sampled λ, MAP instantiations):
`python tools/time_pdps_map.py [iters]` prints ms/iteration and Gpixel-iter/s at T = 2, 3, 4 in strict and fast
arithmetic.  Same shape and conventions as tools/time_pdps.py (BPLTV_PREC, BPLTV_SHAPE)."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bpldenoising_b200 as bp  # noqa: E402

iters = int(sys.argv[1]) if len(sys.argv) > 1 else 240
prec = int(os.environ.get("BPLTV_PREC", "64"))
M, N, O = (int(v) for v in os.environ.get("BPLTV_SHAPE", "512,512,64").split(","))
t, f = bp.synthetic_dataset(M, N, O, seed=20240601)
lam = np.array([[0.05, 0.1], [0.08, 0.12]])    # 2 × 2 patch λ, up-sampled to an M × N map by the library
with bp.Context([0], prec) as ctx:
    ctx.set_dataset((t, f))
    for arith, an in ((bp.STRICT, "strict"), (bp.FAST, "fast")):
        for depth in (2, 3, 4):
            best = 1e30
            for rep in range(3):
                ctx.denoise(None, lam, bp.pdps_opts(maxiter=iters, kernel=bp.KERNEL_TBLOCK, tblock=depth, arith=arith))
                best = min(best, ctx.stats()["ms_pdps"])
            print("prec %d map %-6s T=%d  %.4f ms/iter  %.1f Gpixel-iter/s" %
                  (prec, an, depth, best / iters, M * N * O * iters / best / 1e6), flush=True)
