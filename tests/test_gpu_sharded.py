"""The sharded path of the host-pointer entry points, run on one GPU.

bpltv_create accepts a repeated device id, and each entry is its own shard: a context over [0, 0] has two shards on
device 0, each with its own stream, buffers, gradient workspaces and pinned staging slots, and goes through the same
per-device passes as a context over two GPUs.  Every entry point of such a context must return the bits of a one-device
context (cost and gradient up to the order of the host sums over the devices).  The fields of stats() that do not depend
on timing are pinned for both contexts, with which of the timed fields are set.  O = 5 splits the images 3 + 2, O = 1
leaves the second shard without images."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MN = 32
MAXITER = 200
XP = np.array([[0.05, 0.08], [0.06, 0.04]])                  # 2×2 patch λ
X3 = np.array([0.02, 0.03, 0.01])                            # sum-of-regularisers λ
XP3 = np.stack([0.5 * XP, 0.7 * XP, 0.2 * XP], axis=2)        # 2×2×3
MS = ("ms_upload", "ms_pdps", "ms_cost", "ms_gradient", "ms_download", "ms_total")


def _stats_key(s):
    """(n_devices, pdps_iterations, pixel_iterations, tblock_depth, pdps_kernel_used, kernel_launches,
    solver_iterations, solver_max_relres > 0, which ms_* fields are set)"""
    return (s["n_devices"], s["pdps_iterations"], s["pixel_iterations"], s["tblock_depth"], s["pdps_kernel_used"],
            s["kernel_launches"], s["solver_iterations"], s["solver_max_relres"] > 0,
            "".join("+" if s[k] > 0 else "0" for k in MS))


def _run(bp, prec, devices, O):
    """Every host-pointer entry point once per variant; returns [(case, outputs, stats)] in call order."""
    t, f = bp.synthetic_dataset(MN, MN, O, seed=7)
    out = []
    with bp.Context(devices, prec) as c:
        def rec(case, **res):
            out.append((case, res, c.stats()))

        po = bp.pdps_opts(maxiter=MAXITER)
        rec("denoise_stack_scalar", u=c.denoise(f, 0.07, po))
        before = c.stats()
        c.set_dataset((t, f))
        assert c.stats() == before, "set_dataset changed the stats"
        rec("denoise_stack_patch", u=c.denoise(f, XP, po))
        rec("denoise_resident_scalar", u=c.denoise(None, 0.07, po))
        rec("denoise_resident_patch", u=c.denoise(None, XP, po))
        for lam, lname in ((0.07, "scalar"), (XP, "patch")):
            for Delta, bname in ((0.1, "nonreg"), (1e-8, "reg")):
                u, cost, g = c.learn_eval(lam, Delta, bp.eval_opts(po))
                rec("learn_eval_%s_%s" % (lname, bname), u=u, cost=cost, grad=g)
            u, cost, _ = c.learn_eval(lam, 0.1, bp.eval_opts(po, force_branch=3))
            rec("learn_eval_%s_loss" % lname, u=u, cost=cost)
            u = c.denoise(None, lam, po)
            for reg in (True, False):
                rec("gradient_%s_%s" % (lname, "reg" if reg else "nonreg"), grad=c.gradient(lam, u, reg))
        for params, lname in (([0.03, 0.07, 0.15], "scalar"), ([XP, 2 * XP], "patch")):
            cost, sq, u = c.sweep(params, bp.pdps_opts(maxiter=MAXITER), return_u=True, return_sqerr=True)
            rec("sweep_" + lname, u=u, sqerr=sq, cost=cost)
        spo = bp.sumregs_pdps_opts(maxiter=MAXITER)
        rec("sumregs_denoise_stack", u=c.sumregs_denoise(f, X3, spo))
        rec("sumregs_denoise_resident", u=c.sumregs_denoise(None, XP3, spo))
        for lam, lname in ((X3, "scalar"), (XP3, "patch")):
            for Delta, bname in ((0.01, "nonreg"), (1e-4, "reg")):
                u, cost, g = c.sumregs_learn_eval(lam, Delta, bp.sumregs_eval_opts(spo))
                rec("sumregs_learn_eval_%s_%s" % (lname, bname), u=u, cost=cost, grad=g)
        u = c.sumregs_denoise(None, X3, spo)
        for reg in (True, False):
            rec("sumregs_gradient_%s" % ("reg" if reg else "nonreg"), grad=c.sumregs_gradient(X3, u, reg))
    return out


def _assert_same_results(one, two):
    assert [case for case, _, _ in one] == [case for case, _, _ in two]
    for (case, r1, _), (_, r2, _) in zip(one, two):
        for k in ("u", "sqerr"):
            if k in r1:
                assert np.array_equal(r1[k], r2[k]), (case, k)
        if "cost" in r1:
            assert np.allclose(r1["cost"], r2["cost"], rtol=1e-13, atol=0), (case, r1["cost"], r2["cost"])
        if "grad" in r1:
            assert np.allclose(r1["grad"], r2["grad"], rtol=1e-12, atol=0), (case, r1["grad"], r2["grad"])


def _matches(key, pin):
    """None in a pin: the field is not pinned"""
    return tuple(None if p is None else k for k, p in zip(key, pin)) == tuple(pin)


def _assert_stats(runs, pins):
    for ndev, run in runs.items():
        got = {case: _stats_key(s) for case, _, s in run}
        assert set(got) == set(pins), ndev
        for case, pin in pins.items():
            assert _matches(got[case], pin[ndev - 1]), (ndev, case, got[case], pin[ndev - 1])


@pytest.mark.parametrize("O", [5, 2, 1])
@pytest.mark.parametrize("prec", [64, 32])
def test_two_shards_on_one_gpu_match_one_shard(bp, prec, O):
    runs = {1: _run(bp, prec, [0], O), 2: _run(bp, prec, [0, 0], O)}
    _assert_same_results(runs[1], runs[2])
    _assert_stats(runs, PINS[prec, O])


def _run_pipelined(bp, prec):
    """denoise with pinned caller buffers, 16 images of 64², x⁰ = 0 and x⁰ = f; returns {(ndev, init_mode): (u, stats)}"""
    torch = pytest.importorskip("torch")
    O = 16
    _, f = bp.synthetic_dataset(64, 64, O, seed=11)
    h_in = torch.empty((O, 64, 64), dtype=torch.float64).pin_memory()
    h_out = torch.empty((O, 64, 64), dtype=torch.float64).pin_memory()
    np_in = h_in.numpy().transpose(2, 1, 0)      # Fortran-ordered M×N×O views of the pinned buffers
    np_out = h_out.numpy().transpose(2, 1, 0)
    np_in[...] = f
    os.environ["BPLTV_PIPE_MIN_MB"] = "0"
    os.environ["BPLTV_PIPE_CHUNKS"] = "4"
    bp.reload_env()
    res = {}
    try:
        for devices in ([0], [0, 0]):
            with bp.Context(devices, prec) as c:
                for init_mode in (0, 1):
                    np_out[...] = -1.0
                    c.denoise(np_in, 0.1, bp.pdps_opts(maxiter=120, kernel=bp.KERNEL_TBLOCK, init_mode=init_mode),
                              out=np_out)
                    res[len(devices), init_mode] = (np_out.copy(), c.stats())
    finally:
        del os.environ["BPLTV_PIPE_MIN_MB"], os.environ["BPLTV_PIPE_CHUNKS"]
        bp.reload_env()
    return res


@pytest.mark.parametrize("prec", [64, 32])
def test_pipelined_copies_on_both_shards(bp, prec):
    """In fp64 each shard of 8 images runs its own pipelined copies in 4 chunks, as
    test_pipelined_host_copies_do_not_change_the_result runs them on one device (the launch count shows it); fp32
    takes the serial path."""
    res = _run_pipelined(bp, prec)
    for init_mode in (0, 1):
        assert np.array_equal(res[1, init_mode][0], res[2, init_mode][0]), init_mode
        for ndev in (1, 2):
            got = _stats_key(res[ndev, init_mode][1])
            assert _matches(got, PIPE_PINS[prec][ndev - 1]), (ndev, init_mode, got)


# stats of a run on one B200: PINS[prec, O][case] = (one shard, two shards), fields as in _stats_key
PINS = {
    (64, 5): {
        'denoise_stack_scalar': ((1, 200, 1024000, 1, 3, 1, 0, False, '++00++'), (2, 200, 1024000, 1, 3, 2, 0, False, '++00++')),
        'denoise_stack_patch': ((1, 200, 1024000, 1, 3, 2, 0, False, '++00++'), (2, 200, 1024000, 1, 3, 4, 0, False, '++00++')),
        'denoise_resident_scalar': ((1, 200, 1024000, 1, 3, 1, 0, False, '++00++'), (2, 200, 1024000, 1, 3, 2, 0, False, '++00++')),
        'denoise_resident_patch': ((1, 200, 1024000, 1, 3, 2, 0, False, '++00++'), (2, 200, 1024000, 1, 3, 4, 0, False, '++00++')),
        'learn_eval_scalar_nonreg': ((1, 200, 1024000, 1, 3, 48, 0, True, '0+++++'), (2, 200, 1024000, 1, 3, 96, 0, True, '0+++++')),
        'learn_eval_scalar_reg': ((1, 200, 1024000, 1, 3, 45, 0, True, '0+++++'), (2, 200, 1024000, 1, 3, 90, 0, True, '0+++++')),
        'learn_eval_scalar_loss': ((1, 200, 1024000, 1, 3, 3, 0, False, '0+++++'), (2, 200, 1024000, 1, 3, 6, 0, False, '0+++++')),
        'gradient_scalar_reg': ((1, 0, 0, 0, 0, 42, 0, True, '000+00'), (2, 0, 0, 0, 0, 84, 0, True, '000+00')),
        'gradient_scalar_nonreg': ((1, 0, 0, 0, 0, 45, 0, True, '000+00'), (2, 0, 0, 0, 0, 90, 0, True, '000+00')),
        'learn_eval_patch_nonreg': ((1, 200, 1024000, 1, 3, 49, 0, True, '0+++++'), (2, 200, 1024000, 1, 3, 98, 0, True, '0+++++')),
        'learn_eval_patch_reg': ((1, 200, 1024000, 1, 3, 46, 0, True, '0+++++'), (2, 200, 1024000, 1, 3, 92, 0, True, '0+++++')),
        'learn_eval_patch_loss': ((1, 200, 1024000, 1, 3, 4, 0, False, '0+++++'), (2, 200, 1024000, 1, 3, 8, 0, False, '0+++++')),
        'gradient_patch_reg': ((1, 0, 0, 0, 0, 43, 0, True, '000+00'), (2, 0, 0, 0, 0, 86, 0, True, '000+00')),
        'gradient_patch_nonreg': ((1, 0, 0, 0, 0, 46, 0, True, '000+00'), (2, 0, 0, 0, 0, 92, 0, True, '000+00')),
        'sweep_scalar': ((1, 200, 3072000, 1, 3, 3, 0, False, '+++0++'), (2, 200, 3072000, 1, 3, 6, 0, False, '+++0++')),
        'sweep_patch': ((1, 200, 2048000, 1, 3, 3, 0, False, '+++0++'), (2, 200, 2048000, 1, 3, 6, 0, False, '+++0++')),
        'sumregs_denoise_stack': ((1, 200, 1024000, 1, 0, 1, 0, False, '++00++'), (2, 200, 1024000, 1, 0, 2, 0, False, '++00++')),
        'sumregs_denoise_resident': ((1, 200, 1024000, 1, 0, 2, 0, False, '++00++'), (2, 200, 1024000, 1, 0, 4, 0, False, '++00++')),
        'sumregs_learn_eval_scalar_nonreg': ((1, 200, 1024000, 1, 0, 49, 0, True, '0+++++'), (2, 200, 1024000, 1, 0, 98, 0, True, '0+++++')),
        'sumregs_learn_eval_scalar_reg': ((1, 200, 1024000, 1, 0, 45, 0, True, '0+++++'), (2, 200, 1024000, 1, 0, 90, 0, True, '0+++++')),
        'sumregs_learn_eval_patch_nonreg': ((1, 200, 1024000, 1, 0, 50, 0, True, '0+++++'), (2, 200, 1024000, 1, 0, 100, 0, True, '0+++++')),
        'sumregs_learn_eval_patch_reg': ((1, 200, 1024000, 1, 0, 9, 0, True, '0+++++'), (2, 200, 1024000, 1, 0, 18, 0, True, '0+++++')),
        'sumregs_gradient_reg': ((1, 0, 0, 1, 0, 44, 0, True, '0+++++'), (2, 0, 0, 1, 0, 88, 0, True, '0+++++')),
        'sumregs_gradient_nonreg': ((1, 0, 0, 1, 0, 48, 0, True, '0+++++'), (2, 0, 0, 1, 0, 96, 0, True, '0+++++')),
    },
    (64, 2): {
        'denoise_stack_scalar': ((1, 200, 409600, 1, 3, 1, 0, False, '++00++'), (2, 200, 409600, 1, 3, 2, 0, False, '++00++')),
        'denoise_stack_patch': ((1, 200, 409600, 1, 3, 2, 0, False, '++00++'), (2, 200, 409600, 1, 3, 4, 0, False, '++00++')),
        'denoise_resident_scalar': ((1, 200, 409600, 1, 3, 1, 0, False, '++00++'), (2, 200, 409600, 1, 3, 2, 0, False, '++00++')),
        'denoise_resident_patch': ((1, 200, 409600, 1, 3, 2, 0, False, '++00++'), (2, 200, 409600, 1, 3, 4, 0, False, '++00++')),
        'learn_eval_scalar_nonreg': ((1, 200, 409600, 1, 3, 48, 0, True, '0+++++'), (2, 200, 409600, 1, 3, 96, 0, True, '0+++++')),
        'learn_eval_scalar_reg': ((1, 200, 409600, 1, 3, 45, 0, True, '0+++++'), (2, 200, 409600, 1, 3, 90, 0, True, '0+++++')),
        'learn_eval_scalar_loss': ((1, 200, 409600, 1, 3, 3, 0, False, '0+++++'), (2, 200, 409600, 1, 3, 6, 0, False, '0+++++')),
        'gradient_scalar_reg': ((1, 0, 0, 0, 0, 42, 0, True, '000+00'), (2, 0, 0, 0, 0, 84, 0, True, '000+00')),
        'gradient_scalar_nonreg': ((1, 0, 0, 0, 0, 45, 0, True, '000+00'), (2, 0, 0, 0, 0, 90, 0, True, '000+00')),
        'learn_eval_patch_nonreg': ((1, 200, 409600, 1, 3, 49, 0, True, '0+++++'), (2, 200, 409600, 1, 3, 98, 0, True, '0+++++')),
        'learn_eval_patch_reg': ((1, 200, 409600, 1, 3, 46, 0, True, '0+++++'), (2, 200, 409600, 1, 3, 92, 0, True, '0+++++')),
        'learn_eval_patch_loss': ((1, 200, 409600, 1, 3, 4, 0, False, '0+++++'), (2, 200, 409600, 1, 3, 8, 0, False, '0+++++')),
        'gradient_patch_reg': ((1, 0, 0, 0, 0, 43, 0, True, '000+00'), (2, 0, 0, 0, 0, 86, 0, True, '000+00')),
        'gradient_patch_nonreg': ((1, 0, 0, 0, 0, 46, 0, True, '000+00'), (2, 0, 0, 0, 0, 92, 0, True, '000+00')),
        'sweep_scalar': ((1, 200, 1228800, 1, 3, 3, 0, False, '+++0++'), (2, 200, 1228800, 1, 3, 6, 0, False, '+++0++')),
        'sweep_patch': ((1, 200, 819200, 1, 3, 3, 0, False, '+++0++'), (2, 200, 819200, 1, 3, 6, 0, False, '+++0++')),
        'sumregs_denoise_stack': ((1, 200, 409600, 1, 0, 1, 0, False, '++00++'), (2, 200, 409600, 1, 0, 2, 0, False, '++00++')),
        'sumregs_denoise_resident': ((1, 200, 409600, 1, 0, 2, 0, False, '++00++'), (2, 200, 409600, 1, 0, 4, 0, False, '++00++')),
        'sumregs_learn_eval_scalar_nonreg': ((1, 200, 409600, 1, 0, 49, 0, True, '0+++++'), (2, 200, 409600, 1, 0, 98, 0, True, '0+++++')),
        'sumregs_learn_eval_scalar_reg': ((1, 200, 409600, 1, 0, 45, 0, True, '0+++++'), (2, 200, 409600, 1, 0, 90, 0, True, '0+++++')),
        'sumregs_learn_eval_patch_nonreg': ((1, 200, 409600, 1, 0, 50, 0, True, '0+++++'), (2, 200, 409600, 1, 0, 100, 0, True, '0+++++')),
        'sumregs_learn_eval_patch_reg': ((1, 200, 409600, 1, 0, 9, 0, True, '0+++++'), (2, 200, 409600, 1, 0, 18, 0, True, '0+++++')),
        'sumregs_gradient_reg': ((1, 0, 0, 1, 0, 44, 0, True, '0+++++'), (2, 0, 0, 1, 0, 88, 0, True, '0+++++')),
        'sumregs_gradient_nonreg': ((1, 0, 0, 1, 0, 48, 0, True, '0+++++'), (2, 0, 0, 1, 0, 96, 0, True, '0+++++')),
    },
    (64, 1): {
        'denoise_stack_scalar': ((1, 200, 204800, 1, 3, 1, 0, False, '++00++'), (2, 200, 204800, None, None, 1, 0, False, '++00++')),
        'denoise_stack_patch': ((1, 200, 204800, 1, 3, 2, 0, False, '++00++'), (2, 200, 204800, None, None, 3, 0, False, '++00++')),
        'denoise_resident_scalar': ((1, 200, 204800, 1, 3, 1, 0, False, '++00++'), (2, 200, 204800, None, None, 1, 0, False, '++00++')),
        'denoise_resident_patch': ((1, 200, 204800, 1, 3, 2, 0, False, '++00++'), (2, 200, 204800, None, None, 3, 0, False, '++00++')),
        'learn_eval_scalar_nonreg': ((1, 200, 204800, 1, 3, 48, 0, True, '0+++++'), (2, 200, 204800, None, None, 48, 0, True, '0+++++')),
        'learn_eval_scalar_reg': ((1, 200, 204800, 1, 3, 45, 0, True, '0+++++'), (2, 200, 204800, None, None, 45, 0, True, '0+++++')),
        'learn_eval_scalar_loss': ((1, 200, 204800, 1, 3, 3, 0, False, '0+++++'), (2, 200, 204800, None, None, 3, 0, False, '0+++++')),
        'gradient_scalar_reg': ((1, 0, 0, 0, 0, 42, 0, True, '000+00'), (2, 0, 0, None, None, 42, 0, True, '000+00')),
        'gradient_scalar_nonreg': ((1, 0, 0, 0, 0, 45, 0, True, '000+00'), (2, 0, 0, None, None, 45, 0, True, '000+00')),
        'learn_eval_patch_nonreg': ((1, 200, 204800, 1, 3, 49, 0, True, '0+++++'), (2, 200, 204800, None, None, 50, 0, True, '0+++++')),
        'learn_eval_patch_reg': ((1, 200, 204800, 1, 3, 46, 0, True, '0+++++'), (2, 200, 204800, None, None, 47, 0, True, '0+++++')),
        'learn_eval_patch_loss': ((1, 200, 204800, 1, 3, 4, 0, False, '0+++++'), (2, 200, 204800, None, None, 5, 0, False, '0+++++')),
        'gradient_patch_reg': ((1, 0, 0, 0, 0, 43, 0, True, '000+00'), (2, 0, 0, None, None, 43, 0, True, '000+00')),
        'gradient_patch_nonreg': ((1, 0, 0, 0, 0, 46, 0, True, '000+00'), (2, 0, 0, None, None, 46, 0, True, '000+00')),
        'sweep_scalar': ((1, 200, 614400, 1, 3, 3, 0, False, '+++0++'), (2, 200, 614400, None, None, 3, 0, False, '+++0++')),
        'sweep_patch': ((1, 200, 409600, 1, 3, 3, 0, False, '+++0++'), (2, 200, 409600, None, None, 3, 0, False, '+++0++')),
        'sumregs_denoise_stack': ((1, 200, 204800, 1, 0, 1, 0, False, '++00++'), (2, 200, 204800, None, None, 1, 0, False, '++00++')),
        'sumregs_denoise_resident': ((1, 200, 204800, 1, 0, 2, 0, False, '++00++'), (2, 200, 204800, None, None, 3, 0, False, '++00++')),
        'sumregs_learn_eval_scalar_nonreg': ((1, 200, 204800, 1, 0, 49, 0, True, '0+++++'), (2, 200, 204800, None, None, 49, 0, True, '0+++++')),
        'sumregs_learn_eval_scalar_reg': ((1, 200, 204800, 1, 0, 45, 0, True, '0+++++'), (2, 200, 204800, None, None, 45, 0, True, '0+++++')),
        'sumregs_learn_eval_patch_nonreg': ((1, 200, 204800, 1, 0, 50, 0, True, '0+++++'), (2, 200, 204800, None, None, 51, 0, True, '0+++++')),
        'sumregs_learn_eval_patch_reg': ((1, 200, 204800, 1, 0, 9, 0, True, '0+++++'), (2, 200, 204800, None, None, 10, 0, True, '0+++++')),
        'sumregs_gradient_reg': ((1, 0, 0, 1, 0, 44, 0, True, '0+++++'), (2, 0, 0, None, None, 44, 0, True, '0+++++')),
        'sumregs_gradient_nonreg': ((1, 0, 0, 1, 0, 48, 0, True, '0+++++'), (2, 0, 0, None, None, 48, 0, True, '0+++++')),
    },
    (32, 5): {
        'denoise_stack_scalar': ((1, 200, 1024000, 1, 3, 3, 0, False, '++00++'), (2, 200, 1024000, 1, 3, 6, 0, False, '++00++')),
        'denoise_stack_patch': ((1, 200, 1024000, 1, 3, 4, 0, False, '++00++'), (2, 200, 1024000, 1, 3, 8, 0, False, '++00++')),
        'denoise_resident_scalar': ((1, 200, 1024000, 1, 3, 2, 0, False, '++00++'), (2, 200, 1024000, 1, 3, 4, 0, False, '++00++')),
        'denoise_resident_patch': ((1, 200, 1024000, 1, 3, 3, 0, False, '++00++'), (2, 200, 1024000, 1, 3, 6, 0, False, '++00++')),
        'learn_eval_scalar_nonreg': ((1, 200, 1024000, 1, 3, 49, 0, True, '0+++++'), (2, 200, 1024000, 1, 3, 98, 0, True, '0+++++')),
        'learn_eval_scalar_reg': ((1, 200, 1024000, 1, 3, 46, 0, True, '0+++++'), (2, 200, 1024000, 1, 3, 92, 0, True, '0+++++')),
        'learn_eval_scalar_loss': ((1, 200, 1024000, 1, 3, 4, 0, False, '0+++++'), (2, 200, 1024000, 1, 3, 8, 0, False, '0+++++')),
        'gradient_scalar_reg': ((1, 0, 0, 0, 0, 43, 0, True, '000+00'), (2, 0, 0, 0, 0, 86, 0, True, '000+00')),
        'gradient_scalar_nonreg': ((1, 0, 0, 0, 0, 46, 0, True, '000+00'), (2, 0, 0, 0, 0, 92, 0, True, '000+00')),
        'learn_eval_patch_nonreg': ((1, 200, 1024000, 1, 3, 50, 0, True, '0+++++'), (2, 200, 1024000, 1, 3, 100, 0, True, '0+++++')),
        'learn_eval_patch_reg': ((1, 200, 1024000, 1, 3, 47, 0, True, '0+++++'), (2, 200, 1024000, 1, 3, 94, 0, True, '0+++++')),
        'learn_eval_patch_loss': ((1, 200, 1024000, 1, 3, 5, 0, False, '0+++++'), (2, 200, 1024000, 1, 3, 10, 0, False, '0+++++')),
        'gradient_patch_reg': ((1, 0, 0, 0, 0, 44, 0, True, '000+00'), (2, 0, 0, 0, 0, 88, 0, True, '000+00')),
        'gradient_patch_nonreg': ((1, 0, 0, 0, 0, 47, 0, True, '000+00'), (2, 0, 0, 0, 0, 94, 0, True, '000+00')),
        'sweep_scalar': ((1, 200, 3072000, 1, 3, 6, 0, False, '+++0++'), (2, 200, 3072000, 1, 3, 12, 0, False, '+++0++')),
        'sweep_patch': ((1, 200, 2048000, 1, 3, 5, 0, False, '+++0++'), (2, 200, 2048000, 1, 3, 10, 0, False, '+++0++')),
        'sumregs_denoise_stack': ((1, 200, 1024000, 1, 0, 3, 0, False, '++00++'), (2, 200, 1024000, 1, 0, 6, 0, False, '++00++')),
        'sumregs_denoise_resident': ((1, 200, 1024000, 1, 0, 3, 0, False, '++00++'), (2, 200, 1024000, 1, 0, 6, 0, False, '++00++')),
        'sumregs_learn_eval_scalar_nonreg': ((1, 200, 1024000, 1, 0, 50, 0, True, '0+++++'), (2, 200, 1024000, 1, 0, 100, 0, True, '0+++++')),
        'sumregs_learn_eval_scalar_reg': ((1, 200, 1024000, 1, 0, 46, 0, True, '0+++++'), (2, 200, 1024000, 1, 0, 92, 0, True, '0+++++')),
        'sumregs_learn_eval_patch_nonreg': ((1, 200, 1024000, 1, 0, 51, 0, True, '0+++++'), (2, 200, 1024000, 1, 0, 102, 0, True, '0+++++')),
        'sumregs_learn_eval_patch_reg': ((1, 200, 1024000, 1, 0, 10, 0, True, '0+++++'), (2, 200, 1024000, 1, 0, 20, 0, True, '0+++++')),
        'sumregs_gradient_reg': ((1, 0, 0, 1, 0, 45, 0, True, '0+++++'), (2, 0, 0, 1, 0, 90, 0, True, '0+++++')),
        'sumregs_gradient_nonreg': ((1, 0, 0, 1, 0, 49, 0, True, '0+++++'), (2, 0, 0, 1, 0, 98, 0, True, '0+++++')),
    },
    (32, 2): {
        'denoise_stack_scalar': ((1, 200, 409600, 1, 3, 3, 0, False, '++00++'), (2, 200, 409600, 1, 3, 6, 0, False, '++00++')),
        'denoise_stack_patch': ((1, 200, 409600, 1, 3, 4, 0, False, '++00++'), (2, 200, 409600, 1, 3, 8, 0, False, '++00++')),
        'denoise_resident_scalar': ((1, 200, 409600, 1, 3, 2, 0, False, '++00++'), (2, 200, 409600, 1, 3, 4, 0, False, '++00++')),
        'denoise_resident_patch': ((1, 200, 409600, 1, 3, 3, 0, False, '++00++'), (2, 200, 409600, 1, 3, 6, 0, False, '++00++')),
        'learn_eval_scalar_nonreg': ((1, 200, 409600, 1, 3, 49, 0, True, '0+++++'), (2, 200, 409600, 1, 3, 98, 0, True, '0+++++')),
        'learn_eval_scalar_reg': ((1, 200, 409600, 1, 3, 46, 0, True, '0+++++'), (2, 200, 409600, 1, 3, 92, 0, True, '0+++++')),
        'learn_eval_scalar_loss': ((1, 200, 409600, 1, 3, 4, 0, False, '0+++++'), (2, 200, 409600, 1, 3, 8, 0, False, '0+++++')),
        'gradient_scalar_reg': ((1, 0, 0, 0, 0, 43, 0, True, '000+00'), (2, 0, 0, 0, 0, 86, 0, True, '000+00')),
        'gradient_scalar_nonreg': ((1, 0, 0, 0, 0, 46, 0, True, '000+00'), (2, 0, 0, 0, 0, 92, 0, True, '000+00')),
        'learn_eval_patch_nonreg': ((1, 200, 409600, 1, 3, 50, 0, True, '0+++++'), (2, 200, 409600, 1, 3, 100, 0, True, '0+++++')),
        'learn_eval_patch_reg': ((1, 200, 409600, 1, 3, 47, 0, True, '0+++++'), (2, 200, 409600, 1, 3, 94, 0, True, '0+++++')),
        'learn_eval_patch_loss': ((1, 200, 409600, 1, 3, 5, 0, False, '0+++++'), (2, 200, 409600, 1, 3, 10, 0, False, '0+++++')),
        'gradient_patch_reg': ((1, 0, 0, 0, 0, 44, 0, True, '000+00'), (2, 0, 0, 0, 0, 88, 0, True, '000+00')),
        'gradient_patch_nonreg': ((1, 0, 0, 0, 0, 47, 0, True, '000+00'), (2, 0, 0, 0, 0, 94, 0, True, '000+00')),
        'sweep_scalar': ((1, 200, 1228800, 1, 3, 6, 0, False, '+++0++'), (2, 200, 1228800, 1, 3, 12, 0, False, '+++0++')),
        'sweep_patch': ((1, 200, 819200, 1, 3, 5, 0, False, '+++0++'), (2, 200, 819200, 1, 3, 10, 0, False, '+++0++')),
        'sumregs_denoise_stack': ((1, 200, 409600, 1, 0, 3, 0, False, '++00++'), (2, 200, 409600, 1, 0, 6, 0, False, '++00++')),
        'sumregs_denoise_resident': ((1, 200, 409600, 1, 0, 3, 0, False, '++00++'), (2, 200, 409600, 1, 0, 6, 0, False, '++00++')),
        'sumregs_learn_eval_scalar_nonreg': ((1, 200, 409600, 1, 0, 50, 0, True, '0+++++'), (2, 200, 409600, 1, 0, 100, 0, True, '0+++++')),
        'sumregs_learn_eval_scalar_reg': ((1, 200, 409600, 1, 0, 46, 0, True, '0+++++'), (2, 200, 409600, 1, 0, 92, 0, True, '0+++++')),
        'sumregs_learn_eval_patch_nonreg': ((1, 200, 409600, 1, 0, 51, 0, True, '0+++++'), (2, 200, 409600, 1, 0, 102, 0, True, '0+++++')),
        'sumregs_learn_eval_patch_reg': ((1, 200, 409600, 1, 0, 10, 0, True, '0+++++'), (2, 200, 409600, 1, 0, 20, 0, True, '0+++++')),
        'sumregs_gradient_reg': ((1, 0, 0, 1, 0, 45, 0, True, '0+++++'), (2, 0, 0, 1, 0, 90, 0, True, '0+++++')),
        'sumregs_gradient_nonreg': ((1, 0, 0, 1, 0, 49, 0, True, '0+++++'), (2, 0, 0, 1, 0, 98, 0, True, '0+++++')),
    },
    (32, 1): {
        'denoise_stack_scalar': ((1, 200, 204800, 1, 3, 3, 0, False, '++00++'), (2, 200, 204800, None, None, 3, 0, False, '++00++')),
        'denoise_stack_patch': ((1, 200, 204800, 1, 3, 4, 0, False, '++00++'), (2, 200, 204800, None, None, 5, 0, False, '++00++')),
        'denoise_resident_scalar': ((1, 200, 204800, 1, 3, 2, 0, False, '++00++'), (2, 200, 204800, None, None, 2, 0, False, '++00++')),
        'denoise_resident_patch': ((1, 200, 204800, 1, 3, 3, 0, False, '++00++'), (2, 200, 204800, None, None, 4, 0, False, '++00++')),
        'learn_eval_scalar_nonreg': ((1, 200, 204800, 1, 3, 49, 0, True, '0+++++'), (2, 200, 204800, None, None, 49, 0, True, '0+++++')),
        'learn_eval_scalar_reg': ((1, 200, 204800, 1, 3, 46, 0, True, '0+++++'), (2, 200, 204800, None, None, 46, 0, True, '0+++++')),
        'learn_eval_scalar_loss': ((1, 200, 204800, 1, 3, 4, 0, False, '0+++++'), (2, 200, 204800, None, None, 4, 0, False, '0+++++')),
        'gradient_scalar_reg': ((1, 0, 0, 0, 0, 43, 0, True, '000+00'), (2, 0, 0, None, None, 43, 0, True, '000+00')),
        'gradient_scalar_nonreg': ((1, 0, 0, 0, 0, 46, 0, True, '000+00'), (2, 0, 0, None, None, 46, 0, True, '000+00')),
        'learn_eval_patch_nonreg': ((1, 200, 204800, 1, 3, 50, 0, True, '0+++++'), (2, 200, 204800, None, None, 51, 0, True, '0+++++')),
        'learn_eval_patch_reg': ((1, 200, 204800, 1, 3, 47, 0, True, '0+++++'), (2, 200, 204800, None, None, 48, 0, True, '0+++++')),
        'learn_eval_patch_loss': ((1, 200, 204800, 1, 3, 5, 0, False, '0+++++'), (2, 200, 204800, None, None, 6, 0, False, '0+++++')),
        'gradient_patch_reg': ((1, 0, 0, 0, 0, 44, 0, True, '000+00'), (2, 0, 0, None, None, 44, 0, True, '000+00')),
        'gradient_patch_nonreg': ((1, 0, 0, 0, 0, 47, 0, True, '000+00'), (2, 0, 0, None, None, 47, 0, True, '000+00')),
        'sweep_scalar': ((1, 200, 614400, 1, 3, 6, 0, False, '+++0++'), (2, 200, 614400, None, None, 6, 0, False, '+++0++')),
        'sweep_patch': ((1, 200, 409600, 1, 3, 5, 0, False, '+++0++'), (2, 200, 409600, None, None, 5, 0, False, '+++0++')),
        'sumregs_denoise_stack': ((1, 200, 204800, 1, 0, 3, 0, False, '++00++'), (2, 200, 204800, None, None, 3, 0, False, '++00++')),
        'sumregs_denoise_resident': ((1, 200, 204800, 1, 0, 3, 0, False, '++00++'), (2, 200, 204800, None, None, 4, 0, False, '++00++')),
        'sumregs_learn_eval_scalar_nonreg': ((1, 200, 204800, 1, 0, 50, 0, True, '0+++++'), (2, 200, 204800, None, None, 50, 0, True, '0+++++')),
        'sumregs_learn_eval_scalar_reg': ((1, 200, 204800, 1, 0, 46, 0, True, '0+++++'), (2, 200, 204800, None, None, 46, 0, True, '0+++++')),
        'sumregs_learn_eval_patch_nonreg': ((1, 200, 204800, 1, 0, 51, 0, True, '0+++++'), (2, 200, 204800, None, None, 52, 0, True, '0+++++')),
        'sumregs_learn_eval_patch_reg': ((1, 200, 204800, 1, 0, 10, 0, True, '0+++++'), (2, 200, 204800, None, None, 11, 0, True, '0+++++')),
        'sumregs_gradient_reg': ((1, 0, 0, 1, 0, 45, 0, True, '0+++++'), (2, 0, 0, None, None, 45, 0, True, '0+++++')),
        'sumregs_gradient_nonreg': ((1, 0, 0, 1, 0, 49, 0, True, '0+++++'), (2, 0, 0, None, None, 49, 0, True, '0+++++')),
    },
}
PIPE_PINS = {
    64: ((1, 120, 7864320, 2, 4, 96, 0, False, '++00++'), (2, 120, 7864320, 2, 4, 192, 0, False, '++00++')),
    32: ((1, 120, 7864320, 2, 4, 62, 0, False, '++00++'), (2, 120, 7864320, 2, 4, 124, 0, False, '++00++')),
}
