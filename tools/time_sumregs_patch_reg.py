"""Times the patch sumregs_gradient_reg (2×2×3 λ, rows scaled per operator) of one image on the band LU and on the LU of
the nested-dissection fronts (BPLTV_SUMREGS_PATCH_REG_ND=1): both at 128² (cameraman_128_5 and synthetic), 256², 384²
and 430², the fronts alone at 512², 768² and 1024² (beyond the band LU).  The time is the library's `ms_gradient`
(device events around the gradient phase), best and median of REPS calls after one warm-up call; the bytes per image
are the device memory the first gradient call of a fresh context allocated.  The GPU's name, power limit, clocks and
active throttle reasons are printed before and after.

    python tools/time_sumregs_patch_reg.py [REPS] [SIZES...]        (defaults: 5; 128 256 384 430 512 768 1024)
"""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bpldenoising_b200 as bp  # noqa: E402
import torch  # noqa: E402

X = np.array([0.03, 0.02, 0.04])
XP = np.stack([np.array([[0.03, 0.05], [0.02, 0.04]]) * s for s in (1.0, 0.7, 1.3)], axis=2)
BAND_MAX = 430


def gpu_state(tag):
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks_throttle_reasons.active"
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True)
    print("%s: %s [%s]" % (tag, out.stdout.strip().splitlines()[0] if out.stdout else out.stderr.strip(), q), flush=True)


def images(sizes):
    for n in sizes:
        if n == 128:
            z = np.load(os.path.join(ROOT, "tests", "golden", "datasets.npz"))
            t = z["cameraman_128_5/true"].astype(np.float64) / z["cameraman_128_5/true_div"].astype(np.float64)
            f = z["cameraman_128_5/data"].astype(np.float64) / z["cameraman_128_5/data_div"].astype(np.float64)
            yield "128x128 cameraman", np.asfortranarray(t[:, :, :1]), np.asfortranarray(f[:, :, :1])
        t, f = bp.synthetic_dataset(n, n, 1, seed=3)
        yield "%dx%d synthetic" % (n, n), t, f


def time_one(label, solver, t, f, u, reps):
    os.environ["BPLTV_SUMREGS_PATCH_REG_ND"] = "1" if solver == "nd-lu" else "0"
    bp.reload_env()
    with bp.Context([0], 64) as c:
        c.set_dataset((t, f))
        free0 = torch.cuda.mem_get_info()[0]
        try:
            c.sumregs_gradient(XP, u, regularised=True)
        except bp.BpltvError as e:
            print("%-20s %-8s refused: %s" % (label, solver, e), flush=True)
            return
        used = free0 - torch.cuda.mem_get_info()[0]
        ms = []
        for _ in range(reps):
            c.sumregs_gradient(XP, u, regularised=True)
            ms.append(c.stats()["ms_gradient"])
        st = c.stats()
        print("%-20s %-8s best %9.2f ms  median %9.2f ms  %.2f GB/image  relres %.1e  %d launches" %
              (label, solver, min(ms), float(np.median(ms)), used / 1e9, st["solver_max_relres"], st["kernel_launches"]),
              flush=True)


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    sizes = [int(a) for a in sys.argv[2:]] or [128, 256, 384, 430, 512, 768, 1024]
    torch.cuda.init()
    gpu_state("before")
    for label, t, f in images(sizes):
        with bp.Context([0], 64) as c:
            c.set_dataset((t, f))
            u = np.asfortranarray(c.sumregs_denoise(f, X, bp.sumregs_pdps_opts(maxiter=300)))
        for solver in (("band-lu", "nd-lu") if t.shape[0] <= BAND_MAX else ("nd-lu",)):
            time_one(label, solver, t, f, u, reps)
    os.environ.pop("BPLTV_SUMREGS_PATCH_REG_ND", None)
    gpu_state("after")


if __name__ == "__main__":
    main()
