#!/usr/bin/env python
"""bench.py — the hot path's headline measurement.

Workload (config.workload): BASELINE.json configs[3], the HBM-streaming case the
roofline ceilings of BASELINE.md are quoted on — a synthetic batch of 64 noisy
512×512 images PER GPU, fixed scalar λ = 0.1, exactly 1000 accelerated PDPS
iterations in fp64, followed by the upper-level loss 0.5‖u-ū‖² (and, at N>1, the
NCCL all-reduce of that loss across ranks: the path's only exchange step).
A "step" is one such pass = 64·512·512·1000 = 16.78 Gpixel-iterations per GPU.

  value  — Gpixel-iter/s, whole job (all ranks), inputs resident in HBM.
  e2e    — the same metric through the reference-facing call `denoise(data, x)` with
           HOST (pinned) buffers: H2D of the noisy stack and D2H of the denoised
           stack inside the timed region.
  --impl reference — the reference algorithm on the box's host cores (the C oracle
           port, OpenMP over images; Julia is not installed anywhere: DESIGN.md).
  --dump-outputs DIR — what the last timed step handed back (rank 0): DIR/costgrad.npy, the [loss, gradient] pair,
           and DIR/u_sample.npy, the denoised stack at 2^22 fixed, seeded positions of its column-major M×N×O
           layout (the whole stack is 128 MiB), both float64.  The inputs are seeded, so two builds run with the same
           arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

M = N = 512
O_PER_GPU = 64
ITERS = 1000
LAM = 0.1
METRIC = "tv_pdps_gpixel_iter_per_s"
UNIT = "Gpixel-iter/s"
ALG_BYTES_PER_PIXEL_ITER_F64 = 56  # read x,y1,y2,f + write x,y1,y2 (SURVEY §8d)


def _config(n_gpus):
    return {
        "workload": "BASELINE configs[3]: synthetic 64x512x512 noisy images per GPU, scalar lambda=0.1, "
                    "1000 accelerated PDPS iterations (tau0=5, sigma0=0.99/5) + loss 0.5||u-u_true||^2",
        "images_per_gpu": O_PER_GPU, "image": [M, N], "iterations": ITERS, "lambda": LAM,
        "arith": "strict (one IEEE op per reference operator; bit-identical to the oracle) unless --arith fast",
        "kernel": "auto: temporally blocked streaming kernel, 4 iterations per HBM pass (fp64; strict fp32: 2)",
        "l2": "working set 7 planes x 128 MiB = 896 MiB per GPU >> 126 MB L2 (no flush needed)",
        "parallelism": f"images sharded over {n_gpus} GPU(s), one NCCL all-reduce of [loss, gradient] per step, issued by libbpltv itself (bpltv_comm_init)",
    }


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def __exit__(self, *exc):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if p[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm)}


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except (KeyError, ValueError):
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel_family, depth):
    """dram bytes per launch of the dominant kernel from the committed ncu capture — only if that capture is of the
    kernel this run dispatched (same family, same temporal depth); otherwise None."""
    p = os.path.join(ROOT, "profiles", "ncu_top_kernel.json")
    if os.path.exists(p):
        try:
            rec = json.load(open(p))
        except ValueError:
            return None
        name = rec.get("kernel", "")
        # pdps_tblock_kernel<double, VEC, T, ...>: the third template argument is the depth
        args_ = [a.strip() for a in name[name.find("<") + 1:name.rfind(">")].split(",")] if "<" in name else []
        if name.startswith(kernel_family) and args_[:1] == ["double"] and (kernel_family != "pdps_tblock_kernel" or
                                                                            (len(args_) > 2 and args_[2] == str(depth))):
            return rec.get("dram_bytes_per_launch")
    return None


def host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_reference_step(orc, f_sample, iters, threads, fused=False):
    t0 = time.perf_counter()
    orc.pdps(f_sample, LAM, maxiter=iters, nthreads=threads, fused=fused)
    dt = time.perf_counter() - t0
    return f_sample.size * iters / dt / 1e9, dt


def _leaf_datasets_module():
    """bpldenoising_b200/datasets.py executed as a stand-alone module: the reference arm must not import the package
    (its __init__ loads libbpltv.so — the library under test has no business in the baseline's process)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("_bpltv_datasets_leaf", os.path.join(ROOT, "bpldenoising_b200", "datasets.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def run_reference(args):
    """The reference algorithm on the host cores: the C port of the recursion (oracle/bpltv_oracle.c), all threads.
    Each step is the FULL workload (64 images × 1000 iterations) when the whole run fits ~4 minutes, otherwise the full
    batch for a proportionally reduced iteration count (the rate does not depend on the iteration count).  `value` is the
    faster of two bit-identical variants: the faithful one (separate passes, like the reference's broadcasts) and a
    fused single-sweep one (what a tuned CPU code would do)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import oracle as orc
    orc.build()
    assert "bpldenoising_b200" not in sys.modules
    synthetic_dataset = _leaf_datasets_module().synthetic_dataset
    cores = host_threads()   # torchrun exports OMP_NUM_THREADS=1: ask for the cores explicitly
    _, f = synthetic_dataset(M, N, O_PER_GPU, seed=20240601)
    # probe both variants on a short run
    probe = {}
    for fused in (False, True):
        cpu_reference_step(orc, f, 5, cores, fused)
        probe[fused] = cpu_reference_step(orc, f, 25, cores, fused)[0]
    fused = probe[True] >= probe[False]
    n_steps = args.warmup + args.steps
    full_s = f.size * ITERS / (probe[fused] * 1e9)
    budget_s = 230.0
    iters = ITERS if full_s * n_steps <= budget_s else max(50, int(ITERS * budget_s / (full_s * n_steps)))
    vals = []
    for k in range(n_steps):
        v, dt = cpu_reference_step(orc, f, iters, cores, fused)
        if k >= args.warmup:
            vals.append((v, dt))
    value = statistics.mean(v for v, _ in vals)
    ms = statistics.mean(dt for _, dt in vals) * 1e3
    full = iters == ITERS
    sample = (f"all {O_PER_GPU} images (512x512) x {iters} of the {ITERS} iterations per step"
              + (" = the full step" if full else " (rate extrapolates to the full step: per-iteration cost is constant)")
              + f", OpenMP over images, {cores} threads; C port of the reference recursion (oracle/bpltv_oracle.c, gcc -O3), "
              + ("fused single-sweep variant" if fused else "separate passes as in the reference's broadcasts")
              + "; not Julia (not installed; its solver packages are un-vendored)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms if full else ms * ITERS / iters,
        "ms_per_step_is": "measured" if full else f"extrapolated from {iters} iterations per step",
        "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": _config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "variant": "fused" if fused else "unfused",
                         "probe_unfused": probe[False], "probe_fused": probe[True]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="bpltv", choices=["bpltv", "reference"])
    ap.add_argument("--arith", default="strict", choices=["strict", "fast"])
    ap.add_argument("--no-extras", action="store_true", help="skip the learn_eval wall-time extras")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's outputs as DIR/<name>.npy (costgrad, u_sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    import bpldenoising_b200 as bp

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    W = max(args.warmup, 3)
    K = args.steps

    truth, noisy = bp.synthetic_dataset(M, N, O_PER_GPU, seed=20240601 + rank)
    ctx = bp.Context([local], 64)
    arith = bp.STRICT if args.arith == "strict" else bp.FAST
    popts = bp.pdps_opts(maxiter=ITERS, arith=arith)
    eopts = bp.eval_opts(popts, force_branch=3)  # solve + loss (fixed λ: no gradient in this config)

    # ---- device-resident leg (value) ---------------------------------------------
    # column-major M×N×O on the host == contiguous (O,N,M) torch tensor
    d_truth = torch.from_numpy(np.ascontiguousarray(truth.transpose(2, 1, 0))).to(dev)
    d_noisy = torch.from_numpy(np.ascontiguousarray(noisy.transpose(2, 1, 0))).to(dev)
    d_costgrad = torch.zeros(2, dtype=torch.float64, device=dev)
    # ONE explicit stream carries the kernels, the timing events and the NCCL all-reduce.  (The
    # legacy default stream has handle 0, which the C ABI reads as "use the context's own stream":
    # events recorded on it would not see the kernels.)
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.synchronize()
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0
    ctx.set_dataset_device(d_truth.data_ptr(), d_noisy.data_ptr(), M, N, O_PER_GPU, stream)

    # N > 1: the context joins the job's NCCL communicator INSIDE libbpltv (bpltv_comm_init; torch.distributed only carries
    # the 128-byte id): every learn_eval then ends in the library's own ncclAllReduce of [loss, gradient] on `stream`
    collective = "none (one rank)"
    lib_comm = False
    if world > 1:
        from bpldenoising_b200.parallel import join_job
        try:
            join_job(ctx)
            lib_comm = True
            collective = "ncclAllReduce issued by libbpltv (bpltv_comm_init)"
        except Exception as e:      # noqa: BLE001 - keep the scaling run alive and say what happened
            # every rank fails or succeeds together (the id broadcast is collective, the NCCL binding is the same file)
            collective = f"torch.distributed all_reduce (library communicator unavailable: {type(e).__name__}: {e})"

    def step(d_u_ptr=0):
        ctx.learn_eval_device(LAM, 0.1, d_costgrad.data_ptr(), eopts, d_u_ptr=d_u_ptr, stream=stream)
        if world > 1 and not lib_comm:
            dist.all_reduce(d_costgrad)

    # --dump-outputs: the last timed step also hands back the denoised stack (one device-to-device copy of it)
    d_u = torch.empty((O_PER_GPU, N, M), dtype=torch.float64, device=dev) if args.dump_outputs else None

    for _ in range(W):
        step()
    launches_per_step = ctx.stats()["kernel_launches"]
    kernel_used = ctx.stats()["pdps_kernel_used"]
    depth = max(1, ctx.stats()["tblock_depth"])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        e0.record(tstream)
        for k in range(K):
            step(d_u.data_ptr() if d_u is not None and k == K - 1 else 0)
        e1.record(tstream)
        torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms_total = e0.elapsed_time(e1)
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_per_step = ms_total / K
    pix_iter_per_step = float(M) * N * O_PER_GPU * ITERS
    value = pix_iter_per_step * world / (ms_per_step * 1e-3) / 1e9
    loss = float(d_costgrad[0].item())   # after the all-reduce: the loss of the whole job
    if d_u is not None and rank == 0:
        dump_outputs(args.dump_outputs, d_costgrad.cpu().numpy(), d_u.cpu().numpy())
        del d_u

    # ---- the same leg in the fast arithmetic mode (FMA, rsqrt; within 1e-10 of the oracle) ----
    value_other = None
    if not args.no_extras:
        other = bp.FAST if arith == bp.STRICT else bp.STRICT
        eo2 = bp.eval_opts(bp.pdps_opts(maxiter=ITERS, arith=other), force_branch=3)
        for _ in range(2):
            ctx.learn_eval_device(LAM, 0.1, d_costgrad.data_ptr(), eo2, stream=stream)
        torch.cuda.synchronize()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(tstream)
        for _ in range(3):
            ctx.learn_eval_device(LAM, 0.1, d_costgrad.data_ptr(), eo2, stream=stream)
        f1.record(tstream)
        torch.cuda.synchronize()
        value_other = pix_iter_per_step / (f0.elapsed_time(f1) / 3 * 1e-3) / 1e9  # per GPU

    # ---- fp32 build-only mode: same workload, float planes (28 B per pixel-iteration) -----
    value_f32 = None
    if not args.no_extras:
        c32 = bp.Context([local], 32)
        d_t32, d_n32 = d_truth.float(), d_noisy.float()
        c32.set_dataset_device(d_t32.data_ptr(), d_n32.data_ptr(), M, N, O_PER_GPU, stream)
        for _ in range(2):
            c32.learn_eval_device(LAM, 0.1, d_costgrad.data_ptr(), eopts, stream=stream)
        torch.cuda.synchronize()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(tstream)
        for _ in range(3):
            c32.learn_eval_device(LAM, 0.1, d_costgrad.data_ptr(), eopts, stream=stream)
        f1.record(tstream)
        torch.cuda.synchronize()
        value_f32 = pix_iter_per_step / (f0.elapsed_time(f1) / 3 * 1e-3) / 1e9
        c32.close()
        del d_t32, d_n32

    # ---- roofline of the dominant kernel ------------------------------------------------
    # AUTO dispatches the streaming solve to kernel C (pdps_tblock_kernel): one launch = `depth`
    # PDPS iterations for ONE pass over HBM (depth = 1 would be kernel A, pdps_march_kernel).
    peak, peak_src = hbm_peak()
    # per-launch duration measured live: K steps × ITERS/depth launches back to back on this
    # stream; the loss reduction (2 tiny launches per step) is < 0.1 % of the step
    n_launch = ITERS // depth + ITERS % depth
    launch_ms = ms_per_step / n_launch
    # ALGORITHMIC bytes of one launch = 56 B per pixel-iteration (SURVEY §8d) × the pixel-
    # iterations it performs.  With temporal blocking this exceeds what the launch moves
    # through HBM (≈ 56 B per pixel per launch), so `frac` may legitimately exceed 1 — the
    # single-pass roofline is what kernel A is bound by; `frac_dram` is the share of the HBM
    # peak the launch actually uses (ncu dram bytes ÷ launch time).
    alg_bytes = ALG_BYTES_PER_PIXEL_ITER_F64 * float(M) * N * O_PER_GPU * depth
    achieved = alg_bytes / (launch_ms * 1e-3) / 1e9
    kname = {2: "pdps_march_kernel<double,VEC=2>", 4: "pdps_tblock_kernel<double,VEC=2,T=%d>" % depth}.get(
        kernel_used, "kernel id %d" % kernel_used)
    traffic = ncu_traffic({2: "pdps_march_kernel", 4: "pdps_tblock_kernel"}.get(kernel_used, "?"), depth)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "peak_source": peak_src, "kernel": kname,
                "iterations_per_launch": depth, "algorithmic_bytes_per_launch": alg_bytes, "launch_ms": launch_ms,
                "frac_dram": (traffic / (launch_ms * 1e-3) / 1e9 / peak) if traffic else None,
                "note": "frac = algorithmic bytes (56 B x pixel-iterations of the launch) / time / peak; > 1 means "
                        "the temporally blocked kernel beats the single-pass HBM roofline; frac_dram = measured "
                        "dram bytes per launch (ncu) / time / peak"}

    # ---- end-to-end leg through the reference-facing call with host buffers ----------
    h_in = torch.empty((O_PER_GPU, N, M), dtype=torch.float64).pin_memory()
    h_out = torch.empty((O_PER_GPU, N, M), dtype=torch.float64).pin_memory()
    h_in.copy_(torch.from_numpy(np.ascontiguousarray(noisy.transpose(2, 1, 0))))
    np_in = h_in.numpy().transpose(2, 1, 0)    # Fortran-ordered M×N×O views of the pinned buffers
    np_out = h_out.numpy().transpose(2, 1, 0)
    for _ in range(2):
        ctx.denoise(np_in, LAM, popts, out=np_out)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        u = ctx.denoise(np_in, LAM, popts, out=np_out)   # blocking: H2D + solve + D2H
        _ = float(u[0, 0, 0])                             # the result is read on the host
    t1 = time.perf_counter()
    e2e_ms = (t1 - t0) * 1e3 / K
    st = ctx.stats()
    t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    e2e_val = pix_iter_per_step * world / (e2e_ms * 1e-3) / 1e9
    nbytes = M * N * O_PER_GPU * 8
    e2e = {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": nbytes,
           "ms_per_step": e2e_ms, "device_ms": {"upload": st["ms_upload"], "pdps": st["ms_pdps"],
                                                 "download": st["ms_download"]},
           "copies": "inside the timed call: H2D and D2H of image chunks run on a second stream under the first and the last "
                     "passes of the solve (libbpltv PipeIO), so device_ms.pdps contains them and upload/download read ~0; "
                     "BPLTV_PIPE_IO=0 gives the serial upload -> solve -> download"}

    # the same call with PAGEABLE host arrays (what a Julia caller passes: plain Array{Float64,3})
    pg_in = np.asfortranarray(np.array(noisy, copy=True))
    pg_out = np.zeros_like(pg_in, order="F")
    for _ in range(2):
        ctx.denoise(pg_in, LAM, popts, out=pg_out)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(max(2, K // 2)):
        u = ctx.denoise(pg_in, LAM, popts, out=pg_out)
        _ = float(u[0, 0, 0])
    pg_ms = (time.perf_counter() - t0) * 1e3 / max(2, K // 2)
    stp = ctx.stats()
    t = torch.tensor([pg_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    pg_ms = float(t.item())
    e2e["pageable"] = {"value": pix_iter_per_step * world / (pg_ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": pg_ms,
                       "device_ms": {"upload": stp["ms_upload"], "pdps": stp["ms_pdps"], "download": stp["ms_download"]},
                       "note": "pageable numpy arrays as the caller's buffers; the headline e2e uses pinned ones"}
    del pg_in, pg_out

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": dict(_config(world), collective=collective), "roofline": roofline, "e2e": e2e,
        "gpu_launches": int(launches_per_step * K), "loss": loss,
    }
    if value_f32 is not None:
        line["per_gpu_value_fp32"] = {"value": value_f32, "unit": UNIT, "arith": args.arith,
                                      "frac_of_hbm_peak": value_f32 * 28.0 / peak}
    if value_other is not None:
        line["per_gpu_value_other_arith"] = {"arith": "fast" if arith == bp.STRICT else "strict", "value": value_other,
                                              "unit": UNIT, "frac_of_hbm_peak": value_other * 1e9 * ALG_BYTES_PER_PIXEL_ITER_F64 / 1e9 / peak}

    # ---- BASELINE configs[4] ("config 5") at every N: one bilevel learning step on 1024 synthetic 256×256 images,
    # sharded by image over the ranks, ONE all-reduce of [loss, gradient] per evaluation; strong scaling (total work fixed)
    if not args.no_extras:
        try:
            line["config5"] = config5_extra(bp, torch, dist, dev, tstream, world, rank, local)
        except Exception as e:
            line["config5"] = {"error": f"{type(e).__name__}: {e}"}
        if world == 1 and torch.cuda.device_count() > 1:
            try:
                line["multi_device_context"] = multi_device_extra(bp, torch.cuda.device_count())
            except Exception as e:
                line["multi_device_context"] = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        line["clocks"] = clk.summary()
        # ---- CPU baseline: the oracle port on this box's host cores (bounded sample) ----
        from oracle import oracle as orc
        orc.build()
        cores = host_threads()
        n_img = max(1, min(cores, O_PER_GPU))
        f_s = np.asfortranarray(noisy[:, :, np.arange(n_img) % O_PER_GPU])
        iters_s = 200
        v_unf, dt_unf = cpu_reference_step(orc, f_s, iters_s, cores)
        v_fus, dt_fus = cpu_reference_step(orc, f_s, iters_s, cores, fused=True)
        v_one, dt_one = cpu_reference_step(orc, np.asfortranarray(noisy[:, :, :1]), iters_s, 1)
        line["cpu_baseline"] = {
            "value": max(v_unf, v_fus), "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{n_img} images 512x512 x {iters_s} iterations, OpenMP over images, gcc -O3: faithful separate "
                      f"passes {v_unf:.3f} ({dt_unf:.1f} s), fused single sweep {v_fus:.3f} ({dt_fus:.1f} s), bit-identical; "
                      f"1 thread / 1 image: {v_one:.4f} {UNIT} ({dt_one:.1f} s). C restatement of the reference "
                      "recursion (oracle/bpltv_oracle.c) — Julia is not installed",
            "unfused_value": v_unf, "fused_value": v_fus, "single_thread_value": v_one,
        }
        # ---- extras: learn_eval wall time on the reference-shaped configs (N=1 only) ------
        if world == 1 and not args.no_extras:
            try:
                line["learn_eval"] = learn_eval_extras(bp)
            except Exception as e:   # the extras must never cost the headline line
                line["learn_eval"] = {"error": f"{type(e).__name__}: {e}"}
        print(json.dumps(line))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def dump_outputs(out_dir, costgrad, u_onm):
    """`u_onm`: the denoised stack as the contiguous (O, N, M) array, i.e. the column-major M×N×O layout."""
    os.makedirs(out_dir, exist_ok=True)
    u = u_onm.ravel()
    idx = np.sort(np.random.default_rng(20240601).choice(u.size, size=min(u.size, 1 << 22), replace=False))
    np.save(os.path.join(out_dir, "costgrad.npy"), np.asarray(costgrad, dtype=np.float64))
    np.save(os.path.join(out_dir, "u_sample.npy"), u[idx].astype(np.float64))


def config5_extra(bp, torch, dist, dev, tstream, world, rank, local, total=1024, n=256, iters=5000):
    """BASELINE.json configs[4]: tv_op_learning_function on `total` synthetic n×n images, both gradient branches
    (Δ = 0.1 → gradient, Δ = 1e-7 → gradient_reg) and the loss alone, images sharded `shard_range(total, world, rank)`.
    Each evaluation = one learn_eval_device, which ends in the library's NCCL all-reduce of [loss, gradient]; CUDA-event
    time, max over ranks.
    The gradient's share is the difference to the loss-only evaluation."""
    from bpldenoising_b200.parallel import shard_range
    b, c = shard_range(total, world, rank)
    truth, noisy = bp.synthetic_dataset(n, n, c, seed=20240602 + 1000 * rank)
    d_t = torch.from_numpy(np.ascontiguousarray(truth.transpose(2, 1, 0))).to(dev)
    d_n = torch.from_numpy(np.ascontiguousarray(noisy.transpose(2, 1, 0))).to(dev)
    cg = torch.zeros(2, dtype=torch.float64, device=dev)
    out = {"images_total": total, "image": [n, n], "iterations": iters, "images_per_rank": c, "ranks": world,
           "scaling": "strong", "lambda": LAM}
    with bp.Context([local], 64) as c5:
        lib_comm = False
        if world > 1:
            from bpldenoising_b200.parallel import join_job
            try:
                join_job(c5)          # [loss, gradient] summed by the library's own ncclAllReduce
                lib_comm = True
            except Exception:         # noqa: BLE001 - the headline leg has recorded why
                pass
        out["collective"] = "libbpltv ncclAllReduce" if lib_comm else ("torch.distributed all_reduce" if world > 1 else "none")
        c5.set_dataset_device(d_t.data_ptr(), d_n.data_ptr(), n, n, c, tstream.cuda_stream)
        for name, Delta, branch in (("loss_only", 0.1, 3), ("gradient", 0.1, 0), ("gradient_reg", 1e-7, 0)):
            eo = bp.eval_opts(bp.pdps_opts(maxiter=iters), force_branch=branch)
            ms = None
            for rep in range(2):     # the first evaluation allocates workspaces
                torch.cuda.synchronize()
                if world > 1:
                    dist.barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(tstream)
                c5.learn_eval_device(LAM, Delta, cg.data_ptr(), eo, stream=tstream.cuda_stream)
                if world > 1 and not lib_comm:
                    dist.all_reduce(cg)
                e1.record(tstream)
                torch.cuda.synchronize()
                t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
                if world > 1:
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
            out[name] = {"seconds": ms * 1e-3, "loss": float(cg[0].item()), "grad": float(cg[1].item()),
                         "kernel_launches": c5.stats()["kernel_launches"]}
        for name in ("gradient", "gradient_reg"):
            out[name]["gradient_share_seconds"] = out[name]["seconds"] - out["loss_only"]["seconds"]
        out["gpixel_iter_per_s_loss_only"] = total * n * n * iters / out["loss_only"]["seconds"] / 1e9
    del d_t, d_n
    return out


def multi_device_extra(bp, ndev):
    """The in-library multi-device path (bpltv_create with several device ids: what a single Julia process uses) against
    a one-device context on the same data: identical images, loss and gradient to rounding of the host-side sum."""
    ds = _reference_datasets()
    t, f = (a[:, :, :5].copy(order="F") for a in ds["faces_train_128_10"])
    res = {"devices": ndev}
    with bp.Context([0], 64) as c1, bp.Context(list(range(ndev)), 64) as cn:
        c1.set_dataset((t, f)); cn.set_dataset((t, f))
        eo = bp.eval_opts(bp.pdps_opts(maxiter=1000))
        for name, Delta in (("gradient", 0.1), ("gradient_reg", 1e-7)):
            u1, cost1, g1 = c1.learn_eval(0.07, Delta, eo)
            un, costn, gn = cn.learn_eval(0.07, Delta, eo)
            res[name] = {"max_abs_du": float(np.abs(u1 - un).max()), "rel_dcost": abs(cost1 - costn) / abs(cost1),
                         "rel_dgrad": abs(g1 - gn) / abs(g1), "n_devices_used": cn.stats()["n_devices"]}
    return res


def _reference_datasets():
    """The reference's own datasets (packed from its PNGs into tests/golden/datasets.npz by
    tools/make_dataset_fixtures.py; /root/reference does not exist on the GPU box)."""
    z = np.load(os.path.join(ROOT, "tests", "golden", "datasets.npz"))
    out = {}
    for key in z.files:
        if key.endswith("/true"):
            name = key[:-5]
            out[name] = (np.asfortranarray(z[name + "/true"].astype(np.float64) / z[name + "/true_div"]),
                         np.asfortranarray(z[name + "/data"].astype(np.float64) / z[name + "/data_div"]))
    return out


def learn_eval_extras(bp):
    """BASELINE configs 1-3 on the reference's own datasets: wall time of one
    tv_op_learning_function evaluation (5000 PDPS iterations + cost + λ-gradient) and of the full
    bilevel learn run through the host restatement of the reference's trust-region driver
    (bpldenoising_b200/trbox.py ← TRBox.jl:192-273); config 2's validation solve."""
    from bpldenoising_b200 import trbox
    ds = _reference_datasets()
    out = {}
    for name, dsname, x, Delta in (("config1_cameraman_128_5_scalar", "cameraman_128_5", 0.1, 0.1),
                                   ("config2_faces_train_128_10_scalar", "faces_train_128_10", 0.1, 0.1),
                                   ("config3_circle_128_10_patch2x2", "circle_128_10", 1e-4 * np.ones((2, 2)), 1e-4)):
        data = ds[dsname]
        with bp.Context([0], 64) as c:
            c.set_dataset(data)
            c.learn_eval(x, Delta)  # warm-up (allocations)
            c.learn_eval(x, 1e-9)   # … of the regularised branch too (Δ ≤ Δt): the learn run below reaches it
            ts = []
            for _ in range(3):
                t0 = time.perf_counter()
                _, cost, g = c.learn_eval(x, Delta)
                ts.append((time.perf_counter() - t0) * 1e3)
            st = c.stats()
            out[name] = {"images": int(data[0].shape[2]), "ms": min(ts), "ms_pdps": st["ms_pdps"],
                         "ms_gradient": st["ms_gradient"], "cost": cost, "grad": np.asarray(g).ravel().tolist()}
            # best of two runs: the first one still pays for buffers that grow with the data (the number of adjoint
            # unknowns follows λ); a warmed context repeats the run to within 1 % (tools/dbg_learn_run.py)
            runs = [trbox.bilevel_learn(data, lambda xx, d_, D: bp.tv_op_learning_function(xx, d_, D, ctx=c), x,
                                        dict(Delta0=Delta)) for _ in range(2)]
            res = min(runs, key=lambda r: r.seconds)
            out[name]["learn_run"] = {"seconds": res.seconds, "seconds_first_run": runs[0].seconds, "evaluations": res.evaluations,
                                      "final_cost": res.log[-1].function_value,
                                      "x": np.asarray(res.x).ravel().tolist()}
            if dsname == "faces_train_128_10":   # "validated on faces_val_128_10": TVDenoise = 10000 iterations
                t0 = time.perf_counter()
                val = bp.validate_tv_parameter(float(res.x), ds["faces_val_128_10"], ctx=c)
                out[name]["validation"] = {"seconds": time.perf_counter() - t0, "cost": val["cost"],
                                           "mean_psnr": val["mean_psnr"], "mean_ssim": val["mean_ssim"]}
    # the reference-form gradient on the host cores in the same run: the literal sparse systems of
    # TVLearningFunctionVec.jl:98-161 through SciPy's SuperLU (oracle/oracle.py), one image, one thread
    from oracle import oracle as orc
    t1, f1 = ds["cameraman_128_5"]
    with bp.Context([0], 64) as c:
        u1 = c.denoise(f1, 0.1)
    cpu = {}
    for name, fn in (("gradient", orc.gradient_scalar), ("gradient_reg", orc.gradient_reg_scalar)):
        t0 = time.perf_counter()
        gval = fn(0.1, u1[:, :, 0], t1[:, :, 0])
        cpu[name] = {"seconds_per_image": time.perf_counter() - t0, "grad": float(gval)}
    out["cpu_port_gradient_cameraman_128_5"] = cpu

    # sum-of-regularisers interface (SURVEY §8f row 1): one sumregs_learning_function evaluation on the
    # reference's cameraman dataset at α₀ = [0.001, 0.001, 0.001], both gradient branches
    data = ds["cameraman_128_5"]
    with bp.Context([0], 64) as c:
        c.set_dataset(data)
        x0 = np.array([0.001, 0.001, 0.001])
        xp = 0.001 * np.ones((2, 2, 3))      # α₀ of the patch experiment (BPLDenoising.jl:462)

        def best_of_3(x, Delta):
            # the first evaluation of a branch in a context allocates its workspace and loads its kernels
            best = None
            for rep in range(3):
                t0 = time.perf_counter()
                _, cost, g = c.sumregs_learn_eval(x, Delta)
                st = c.stats()
                r = {"ms": (time.perf_counter() - t0) * 1e3, "ms_pdps": st["ms_pdps"], "ms_gradient": st["ms_gradient"],
                     "cost": cost, "grad": np.asarray(g).ravel().tolist(), "best_of": 3}
                if best is None or r["ms"] < best["ms"]:
                    best = r
            return best

        rec = {}
        # scalar parameter: Δ₀ = 0.01 > Δt → sumregs_gradient; Δ ≤ Δt = 1e-3 → sumregs_gradient_reg (:8-20)
        rec["sumregs_gradient"] = best_of_3(x0, 0.01)
        rec["sumregs_gradient_reg"] = best_of_3(x0, 1e-4)
        # patch parameter 2×2×3, both branches; the regularised one is the row-scaled system of
        # SumRegsLearningFunction.jl:246 (node-space band LU)
        rec["patch_sumregs_gradient"] = best_of_3(xp, 0.1)
        rec["patch_sumregs_gradient_reg"] = best_of_3(xp, 1e-4)
        # the reference's two sum-of-regularisers experiments (BPLDenoising.jl:432-481: cameraman_128_5, one sample,
        # 20 trust-region iterations) through the host restatement of the driver; best of two runs (warmed context)
        for key, fn in (("learn_run_scalar", trbox.scalar_bilevel_sumregs_learn), ("learn_run_patch", trbox.patch_bilevel_sumregs_learn)):
            runs = [fn(data, ctx=c) for _ in range(2)]
            res = min(runs, key=lambda r: r.seconds)
            rec[key] = {"seconds": res.seconds, "seconds_first_run": runs[0].seconds, "evaluations": res.evaluations,
                        "final_cost": res.log[-1].function_value, "x": np.asarray(res.x).ravel().tolist()}
        out["sumregs_cameraman_128_5"] = rec

    # λ-sweep (generate_scalar_tv_cost, /root/reference/src/BPLDenoising.jl:92-130): 64 parameters ×
    # 1 image 128×128 × 10000 iterations, batched into one launch vs the reference's loop of solves
    data = bp.synthetic_dataset(128, 128, 1, seed=7)
    rng_ = np.geomspace(0.005, 0.5, 64)
    with bp.Context([0], 64) as c:
        bp.generate_scalar_tv_cost(data, rng_[:2], ctx=c)
        t0 = time.perf_counter()
        costs = bp.generate_scalar_tv_cost(data, rng_, ctx=c)
        t_batched = time.perf_counter() - t0
        st = c.stats()
        t0 = time.perf_counter()
        for lam_ in rng_[:8]:
            c.sweep([float(lam_)], bp.pdps_opts(maxiter=10000))
        t_loop = (time.perf_counter() - t0) * 8
        out["cost_curve_64x1x128x128_10000its"] = {
            "seconds_batched": t_batched, "seconds_looped_estimate": t_loop, "kernel": st["pdps_kernel_used"],
            "gpixel_iter_per_s": 64 * 16384 * 10000 / t_batched / 1e9, "argmin_lambda": float(rng_[int(np.argmin(costs))])}
    return out


if __name__ == "__main__":
    sys.exit(main())
