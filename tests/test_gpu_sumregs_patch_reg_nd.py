"""The patch sumregs_gradient_reg (SumRegsLearningFunction.jl:195-262: rows scaled by a different λ-map per operator, not
symmetric) on the LU form of the nested-dissection fronts (bpldenoising_b200/csrc/nd_solver.cuh, nd_lu_factor_*).

The band LU keeps every shape it takes (≤ 430²) with its bits; the fronts' LU takes the larger images, and
BPLTV_SUMREGS_PATCH_REG_ND=1 sends small ones to it as well, where it must agree with the band LU, the refined
literal solve and the scalar variant.  solver_max_relres is the band LU's relative residual ‖r − Mp‖/‖r‖ after the last
refinement step (at γ = 1e8 up to ≈ 1e-9 at rounding level); a solve that fails the backward-error test comes back as
NaN.  The CPU counterpart is tests/test_emu_nd_lu.py."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

X = np.array([0.03, 0.02, 0.04])
XP = np.stack([np.array([[0.03, 0.05], [0.02, 0.04]]) * s for s in (1.0, 0.7, 1.3)], axis=2)      # 2×2 patches × 3
XQ = np.stack([np.array([[0.03, 0.05], [0.02, 0.04], [0.06, 0.01]]) * s for s in (1.0, 0.7, 1.3)], axis=2)  # 3×2


@pytest.fixture(scope="module")
def sr():
    from oracle import sumregs
    return sumregs


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    return oracle


def _with_env(bp, env, fn):
    for k, v in env.items():
        os.environ[k] = v
    bp.reload_env()
    try:
        return fn()
    finally:
        for k in env:
            del os.environ[k]
        bp.reload_env()


def _nd(bp, fn):
    return _with_env(bp, {"BPLTV_SUMREGS_PATCH_REG_ND": "1"}, fn)


def _crop(datasets, name, n, k, off=20):
    t, f = datasets[name]
    return (np.asfortranarray(t[off:off + n, off:off + n, :k]), np.asfortranarray(f[off:off + n, off:off + n, :k]))


def _maps(orc, x, n):
    return [orc.patch_upsample(x[:, :, k], n, n) for k in range(3)]


def _denoised(bp, c, t, f, x=X, maxiter=300):
    c.set_dataset((t, f))
    return np.asfortranarray(c.sumregs_denoise(f, x, bp.sumregs_pdps_opts(maxiter=maxiter)))


def test_default_stays_on_the_band_lu(bp, datasets):
    """without the switch, the patch regularised branch at 128² is the band LU's: its bits and its launch count"""
    t, f = _crop(datasets, "cameraman_128_5", 128, k=2, off=0)
    with bp.Context([0], 64) as c:
        u = _denoised(bp, c, t, f)
        g = c.sumregs_gradient(XP, u, regularised=True)
        launches = c.stats()["kernel_launches"]
        gb = c.sumregs_gradient(XP, u, regularised=True, opts=bp.sumregs_eval_opts(solver=1))
        assert np.array_equal(g, gb) and c.stats()["kernel_launches"] == launches


@pytest.mark.parametrize("case", ["40", "37-3x2", "128"])
def test_fronts_lu_on_small_images(bp, sr, orc, datasets, case):
    """with the switch: the refined literal solve, the band LU, image-order sums, and the large-front variants' bits"""
    if case == "128":
        t, f = _crop(datasets, "cameraman_128_5", 128, k=1, off=0)
        x = XP
    else:
        n = int(case.split("-")[0])
        t, f = _crop(datasets, "faces_train_128_10", n, k=3, off=30)
        x = XQ if case.endswith("3x2") else XP
    n = t.shape[0]
    with bp.Context([0], 64) as c:
        u = _denoised(bp, c, t, f)
        g = _nd(bp, lambda: c.sumregs_gradient(x, u, regularised=True))
        st = c.stats()
        band = c.sumregs_gradient(x, u, regularised=True, opts=bp.sumregs_eval_opts(solver=1))
        assert st["solver_max_relres"] <= 1e-8, st
        assert np.all(np.abs(g - band) <= 1e-9 * np.abs(band).max()), (g, band)
        for kb in ("0", "40"):
            gk = _with_env(bp, {"BPLTV_SUMREGS_PATCH_REG_ND": "1", "BPLTV_ND_LARGE_KB": kb},
                           lambda: c.sumregs_gradient(x, u, regularised=True))
            assert np.array_equal(gk, g), (kb, gk, g)
        if u.shape[2] > 1:
            parts = []
            for i in range(u.shape[2]):
                c.set_dataset((t[:, :, i:i + 1], f[:, :, i:i + 1]))
                parts.append(_nd(bp, lambda: c.sumregs_gradient(x, np.asfortranarray(u[:, :, i:i + 1]), regularised=True)))
            acc = parts[0]
            for p in parts[1:]:
                acc = acc + p
            assert np.array_equal(acc, g), (acc, g)
    maps = _maps(orc, x, n)
    lit = sum(sr.sumregs_gradient_reg(maps, u[:, :, i], t[:, :, i], grid_shape=x.shape[:2], refine=3) for i in range(u.shape[2]))
    assert np.all(np.abs(g - lit) <= 1e-9 * np.abs(lit).max()), (g, lit)


def test_uniform_maps_match_the_scalar_variant(bp, datasets):
    """equal patches per operator: the symmetric system of the scalar sumregs_gradient_reg, on the Cholesky of the fronts"""
    t, f = _crop(datasets, "faces_train_128_10", 64, k=2)
    xu = np.broadcast_to(X, (2, 2, 3)).copy()
    with bp.Context([0], 64) as c:
        u = _denoised(bp, c, t, f)
        opts = bp.sumregs_eval_opts(gamma_patch=1e3)        # the scalar variant's γ (:117)
        g = _nd(bp, lambda: c.sumregs_gradient(xu, u, regularised=True, opts=opts))
        gs = c.sumregs_gradient(X, u, regularised=True)
    g = g.sum(axis=(0, 1))
    assert np.all(np.abs(g - gs) <= 1e-10 * np.abs(gs).max()), (g, gs)


def test_beyond_the_band_lu_448_matches_the_literal_solve(bp, sr, orc):
    """448², above the band LU's limit (n ≤ 430), without the switch; and 512²"""
    with bp.Context([0], 64) as c:
        t, f = bp.synthetic_dataset(448, 448, 1, seed=3)
        u = _denoised(bp, c, t, f)
        g = c.sumregs_gradient(XP, u, regularised=True)
        st = c.stats()
        t5, f5 = bp.synthetic_dataset(512, 512, 1, seed=4)
        u5 = _denoised(bp, c, t5, f5)
        g5 = c.sumregs_gradient(XQ, u5, regularised=True)
        st5 = c.stats()
    assert st["solver_max_relres"] <= 1e-8, st
    assert np.all(np.isfinite(g5)) and st5["solver_max_relres"] <= 1e-8, (g5, st5)
    lit = sr.sumregs_gradient_reg(_maps(orc, XP, 448), u[:, :, 0], t[:, :, 0], grid_shape=(2, 2), refine=3)
    assert np.all(np.abs(g - lit) <= 1e-9 * np.abs(lit).max()), (g, lit)


def test_learn_eval_at_512_through_the_regularised_branch_and_shards(bp):
    """the trust-region evaluation at Δ = 1e-4 < Δt takes the patch regularised branch; two shards on one GPU agree"""
    t, f = bp.synthetic_dataset(512, 512, 2, seed=11)
    res = {}
    for devs in ([0], [0, 0]):
        with bp.Context(devs, 64) as c:
            c.set_dataset((t, f))
            _, cost, g = c.sumregs_learn_eval(XP, 1e-4, return_u=False)
            assert np.all(np.isfinite(g)) and c.stats()["solver_max_relres"] <= 1e-8
            res[len(devs)] = (cost, g)
    (c1, g1), (c2, g2) = res[1], res[2]
    assert abs(c2 - c1) <= 1e-13 * abs(c1) and np.all(np.abs(g2 - g1) <= 1e-12 * np.abs(g1).max()), (g1, g2)


@pytest.mark.parametrize("prec,n", [(32, 512), (64, 1024)])
def test_fp32_and_the_largest_size(bp, prec, n):
    """an fp32 context at 512², and 1024², whose fronts need the global-memory panels"""
    t, f = bp.synthetic_dataset(n, n, 1, seed=7)
    with bp.Context([0], prec) as c:
        u = _denoised(bp, c, t, f, maxiter=200)
        g = c.sumregs_gradient(XP, u, regularised=True)
        st = c.stats()
    assert np.all(np.isfinite(g)) and st["solver_max_relres"] <= 1e-8, (g, st)
