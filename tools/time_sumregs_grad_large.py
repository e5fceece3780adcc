"""Times the sum-of-regularisers gradients of one image at sizes whose nested-dissection fronts may outgrow shared
memory (288², 384², 512²): sumregs_gradient (scalar and 2×2×3 patch) and scalar sumregs_gradient_reg.  The time is
the library's `ms_gradient` (device events around the gradient phase), best and median of REPS calls after one
warm-up call; the bytes per image are the device memory the first gradient call of a fresh context allocated.
The GPU's name, power limit, clocks and active throttle reasons are printed before and after.

    python tools/time_sumregs_grad_large.py [REPS] [SIZES...]        (defaults: 3; 288 384 512)
"""
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bpldenoising_b200 as bp  # noqa: E402
import torch  # noqa: E402

X = np.array([0.03, 0.02, 0.04])
XP = np.stack([np.array([[0.03, 0.05], [0.02, 0.04]]) * s for s in (1.0, 0.7, 1.3)], axis=2)
VARIANTS = [("sumregs_gradient scalar", X, False), ("sumregs_gradient 2x2 patch", XP, False),
            ("sumregs_gradient_reg scalar", X, True)]


def gpu_state(tag):
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks_throttle_reasons.active"
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True)
    print("%s: %s [%s]" % (tag, out.stdout.strip().splitlines()[0] if out.stdout else out.stderr.strip(), q), flush=True)


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
    sizes = [int(a) for a in sys.argv[2:]] or [288, 384, 512]
    torch.cuda.init()
    gpu_state("before")
    for n in sizes:
        t, f = bp.synthetic_dataset(n, n, 1, seed=3)
        with bp.Context([0], 64) as c:
            c.set_dataset((t, f))
            u = np.asfortranarray(c.sumregs_denoise(f, X, bp.sumregs_pdps_opts(maxiter=300)))
        for name, x, reg in VARIANTS:
            with bp.Context([0], 64) as c:
                c.set_dataset((t, f))
                free0 = torch.cuda.mem_get_info()[0]
                try:
                    c.sumregs_gradient(x, u, regularised=reg)
                except bp.BpltvError as e:
                    print("%dx%d %-28s refused: %s" % (n, n, name, e), flush=True)
                    continue
                used = free0 - torch.cuda.mem_get_info()[0]
                ms = []
                for _ in range(reps):
                    c.sumregs_gradient(x, u, regularised=reg)
                    ms.append(c.stats()["ms_gradient"])
                st = c.stats()
                print("%dx%d %-28s best %9.1f ms  median %9.1f ms  %.2f GB/image  relres %.1e  %d launches" %
                      (n, n, name, min(ms), float(np.median(ms)), used / 1e9, st["solver_max_relres"],
                       st["kernel_launches"]), flush=True)
    gpu_state("after")


if __name__ == "__main__":
    main()
