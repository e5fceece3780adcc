"""Adjoint solves whose nested-dissection fronts outgrow shared memory (bpldenoising_b200/csrc/nd_solver.cuh, the
large-front variants: the factorisation's panel and the solves' front vector in global memory).

On small images BPLTV_ND_LARGE_KB sends every level (or the upper ones) to the variants: the gradients must be the
bits of the shared-memory kernels.  On images that neither the shared-memory fronts nor the band solvers take, the
calls must succeed with a backward error at rounding level and match the CPU checkers."""
import os
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

X = np.array([0.03, 0.02, 0.04])
XP = np.stack([np.array([[0.03, 0.05], [0.02, 0.04]]) * s for s in (1.0, 0.7, 1.3)], axis=2)     # 2×2 patches × 3


@pytest.fixture(scope="module")
def sr():
    from oracle import sumregs
    return sumregs


def _with_env(bp, name, value, fn):
    os.environ[name] = value
    bp.reload_env()
    try:
        return fn()
    finally:
        del os.environ[name]
        bp.reload_env()


def _denoised(bp, c, n, O=1, seed=3, maxiter=300):
    t, f = bp.synthetic_dataset(n, n, O, seed=seed)
    c.set_dataset((t, f))
    return t, f, np.asfortranarray(c.sumregs_denoise(f, X, bp.sumregs_pdps_opts(maxiter=maxiter)))


def _crop(datasets, name, n, k, off=20):
    t, f = datasets[name]
    return (np.asfortranarray(t[off:off + n, off:off + n, :k]), np.asfortranarray(f[off:off + n, off:off + n, :k]))


@pytest.mark.parametrize("n", [48, 128])
def test_large_front_variants_give_the_bits_of_the_shared_memory_kernels(bp, datasets, n):
    """sumregs_gradient (scalar and 2×2×3 patch), scalar sumregs_gradient_reg and the TV gradients (same planner) with
    every level, and with only the levels beyond 40 KB, on the large-front variants"""
    if n == 48:
        t, f = _crop(datasets, "faces_train_128_10", 48, k=2)
    else:
        t, f = bp.synthetic_dataset(128, 128, 1, seed=5)
    with bp.Context([0], 64) as c:
        c.set_dataset((t, f))
        u = np.asfortranarray(c.sumregs_denoise(f, X, bp.sumregs_pdps_opts(maxiter=300)))
        utv = np.asfortranarray(c.denoise(f, 0.07, bp.pdps_opts(maxiter=300)))

        def run():
            return (c.sumregs_gradient(X, u, regularised=False), c.sumregs_gradient(XP, u, regularised=False),
                    c.sumregs_gradient(X, u, regularised=True), c.gradient(0.07, utv, False), c.gradient(0.07, utv, True))
        ref = run()
        assert all(np.all(np.isfinite(g)) for g in ref)
        for kb in ("0", "40"):
            got = _with_env(bp, "BPLTV_ND_LARGE_KB", kb, run)
            for k, (a, b) in enumerate(zip(got, ref)):
                assert np.array_equal(a, b), (kb, k, a, b)


@pytest.mark.parametrize("n", [288, 512])
def test_sumregs_gradient_beyond_the_band_cholesky(bp, sr, n):
    """sumregs_gradient beyond the band Cholesky (n ≤ 136): at 512² its fronts exceed shared memory; at 288² a front of
    this image comes within the kernels' static shared memory of the opt-in maximum (a kernel-attribute error before).
    The scalar regularised branch still runs on the shared-memory fronts at both sizes."""
    with bp.Context([0], 64) as c:
        t, f, u = _denoised(bp, c, n)
        for x in (X, XP):
            g = c.sumregs_gradient(x, u, regularised=False)
            st = c.stats()
            assert np.all(np.isfinite(g)) and st["solver_max_relres"] <= 1e-9, (g, st)
        gr = c.sumregs_gradient(X, u, regularised=True)
        st = c.stats()
        assert np.all(np.isfinite(gr)) and st["solver_max_relres"] <= 1e-9, (gr, st)


def test_sumregs_gradient_reg_448_matches_the_literal_solve(bp, sr):
    """448², just above the band LU's limit (n ≤ 430), on the node form's shared-memory fronts: the refined literal
    node-space solve of oracle/sumregs.py"""
    with bp.Context([0], 64) as c:
        t, f, u = _denoised(bp, c, 448)
        g = c.sumregs_gradient(X, u, regularised=True)
        st = c.stats()
    assert st["solver_max_relres"] <= 1e-9, st
    lit = sr.sumregs_gradient_reg(X, u[:, :, 0], t[:, :, 0], refine=3)
    assert np.all(np.abs(g - lit) <= 1e-9 * np.abs(lit).max()), (g, lit)


def test_sumregs_gradient_matches_the_compliance_form_checker_beyond_shared_memory(bp, sr):
    """288² with every level on the large-front variants (BPLTV_ND_LARGE_KB = 0): the largest size at which the
    compliance-form checker runs in reasonable time on the CPU (about a minute; 256² about half that)"""
    with bp.Context([0], 64) as c:
        t, f, u = _denoised(bp, c, 288)
        g = _with_env(bp, "BPLTV_ND_LARGE_KB", "0", lambda: c.sumregs_gradient(X, u, regularised=False))
        st = c.stats()
    assert st["solver_max_relres"] <= 1e-9, st
    du = sr.sumregs_gradient_dual("nonreg", X, u[:, :, 0], t[:, :, 0])
    assert np.all(np.abs(g - du) <= 1e-10 * np.abs(du).max()), (g, du)


def test_sumregs_gradient_at_512_in_fp32(bp):
    with bp.Context([0], 32) as c:
        t, f, u = _denoised(bp, c, 512)
        g = c.sumregs_gradient(X, u, regularised=False)
        st = c.stats()
    assert np.all(np.isfinite(g)) and st["solver_max_relres"] <= 1e-9, (g, st)


def test_sumregs_learn_eval_at_512_through_both_branches_and_shards(bp):
    """the trust-region evaluation at 512² in the non-regularised (Δ > Δt) and the regularised branch; a context that
    runs the two images as two shards on one GPU gives the same cost and gradient"""
    t, f = bp.synthetic_dataset(512, 512, 2, seed=11)
    res = {}
    for devs in ([0], [0, 0]):
        with bp.Context(devs, 64) as c:
            c.set_dataset((t, f))
            for delta in (0.01, 1e-4):
                _, cost, g = c.sumregs_learn_eval(X, delta, return_u=False)
                assert np.all(np.isfinite(g)) and c.stats()["solver_max_relres"] <= 1e-9
                res[len(devs), delta] = (cost, g)
    for delta in (0.01, 1e-4):
        (c1, g1), (c2, g2) = res[1, delta], res[2, delta]
        assert abs(c2 - c1) <= 1e-13 * abs(c1) and np.all(np.abs(g2 - g1) <= 1e-12 * np.abs(g1).max()), (delta, g1, g2)
    assert not np.allclose(res[1, 0.01][1], res[1, 1e-4][1])


def test_tv_gradient_at_1024(bp):
    """1024²: the TV multiplier form's fronts exceed shared memory and the band Cholesky refuses the size"""
    t, f = bp.synthetic_dataset(1024, 1024, 1, seed=7)
    with bp.Context([0], 64) as c:
        c.set_dataset((t, f))
        u = np.asfortranarray(c.denoise(f, 0.07, bp.pdps_opts(maxiter=200)))
        for reg in (False, True):
            g = c.gradient(0.07, u, reg)
            st = c.stats()
            assert np.all(np.isfinite(g)) and st["solver_max_relres"] <= 1e-9, (reg, g, st)


def test_sumregs_gradient_that_does_not_fit_names_its_size(bp):
    """2048², flat everywhere (six multipliers per pixel): the factor alone needs more than the device has — the call
    returns BPLTV_ERR_ALLOC with the size one image needs, not the band Cholesky's size limit"""
    n = 2048
    t, _ = bp.synthetic_dataset(n, n, 1, seed=1)
    u = np.asfortranarray(np.full((n, n, 1), 0.5))
    with bp.Context([0], 64) as c:
        c.set_dataset((t, t))
        with pytest.raises(bp.BpltvError) as e:
            c.sumregs_gradient(X, u, regularised=False)
    assert e.value.code == -6 and re.search(r"[\d.]+(e\+\d+)? GB per image", str(e.value)), str(e.value)
