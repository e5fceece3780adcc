"""CPU check of the LU form of the nested-dissection solver (bpldenoising_b200/csrc/nd_solver.cuh: nd_lu_factor_*), which
takes the row-scaled patch sum-of-regularisers system (I + Σ_k diag(a_k) G_kᵀ(B_k − C_k) G_k) p = ū − u of
sumregs_gradient_reg (SumRegsLearningFunction.jl:195-262).  The device code runs on the thread emulation
(tests/emu/emu_cuda.h) through tests/emu/emu_nd_lu.cpp, in the launch order of run_gradient3_nd_reg: the result must
match the oracle's literal solve, reduce to the Cholesky of the same fronts when the maps are uniform, give the same
bits for every cluster size and with the panels in global memory, and report a vanished pivot as a breakdown followed
by NaN.  The GPU counterpart is tests/test_gpu_sumregs_patch_reg_nd.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle as orc
from oracle import sumregs as sr

HERE = os.path.dirname(os.path.abspath(__file__))
EMU = os.path.join(HERE, "emu")
CSRC = os.path.join(HERE, "..", "bpldenoising_b200", "csrc")

ALL = 0          # large_limit: every level on the large-front variants
NONE = -1        # none
WIDE = 1 << 30   # smem_limit: 16-column block steps everywhere
NARROW = 0       # 8-column block steps everywhere


@pytest.fixture(scope="module")
def lib():
    out = os.path.join(EMU, "_build", "libemu_nd_lu.so")
    srcs = [os.path.join(EMU, "emu_nd_lu.cpp"), os.path.join(EMU, "emu_cuda.h")] + \
           [os.path.join(CSRC, f) for f in ("nd_symbolic.h", "nd_solver.cuh", "nd_sumregs.cuh", "lu_band.cuh",
                                            "sumregs_stencils.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        subprocess.run(["g++", "-std=c++20", "-O1", "-pthread", "-fPIC", "-shared", "-DBPLTV_EMU", "-ffp-contract=off",
                        "-o", out, srcs[0]], check=True)
    lib = C.CDLL(out)
    lib.emu_nd_lu_gradient_reg.restype = C.c_int
    return lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))


def _case(n, seed):
    rng = np.random.default_rng(seed)
    t = np.round(rng.random((n, n)) * 255) / 255
    u = np.asfortranarray(t + 0.05 * rng.standard_normal((n, n)))
    u[:3, :3] = u[0, 0]                      # exactly flat blocks: γ·I tensors
    u[n - 4:, n - 5:] = u[n - 1, n - 1]
    return np.asfortranarray(t), u


def _lam(grid, seed):
    rng = np.random.default_rng(seed)
    return 0.02 + 0.06 * rng.random(tuple(grid) + (3,))


def _maps(lam, n):
    return [orc.patch_upsample(lam[:, :, k], n, n) for k in range(3)]


def _run(lib, u, t, lam=None, scalar=None, gamma=1e8, csize=1, smem_limit=WIDE, large=NONE, zero_row=-1, small=0,
         refine=3):
    """lam: m×n×3 patch values (LU form) or None with `scalar` (Cholesky form)"""
    n = u.shape[0]
    lm, ln = (lam.shape[0], lam.shape[1]) if lam is not None else (1, 1)
    maps = None if lam is None else np.concatenate([m.flatten(order="F") for m in _maps(lam, n)])
    out, stats, p = np.zeros(3 * lm * ln), np.zeros(8), np.zeros(n * n)
    rc = lib.emu_nd_lu_gradient_reg(n, _ptr(u.flatten(order="F")), _ptr(t.flatten(order="F")),
                                    _ptr(None if scalar is None else np.asarray(scalar, dtype=np.float64)), _ptr(maps),
                                    lm, ln, C.c_double(gamma), refine, 4, int(small), csize, C.c_longlong(smem_limit),
                                    C.c_longlong(large), zero_row, _ptr(out), _ptr(stats), _ptr(p))
    assert rc == 0
    return out, stats, p


def _oracle_layout(gx):
    """m×n×3 → [operator][patch], patch index i + m·j (the library's layout)"""
    return np.concatenate([gx[:, :, k].flatten(order="F") for k in range(3)])


@pytest.mark.parametrize("n", [16, 24, 40])
@pytest.mark.parametrize("grid", [(2, 2), (3, 2)])
def test_patch_maps_match_the_literal_solve(lib, n, grid):
    t, u = _case(n, 7 + n)
    lam = _lam(grid, n + grid[0])
    got, stats, _ = _run(lib, u, t, lam)
    assert stats[1] == 0 and stats[6] == 1, stats
    lit = _oracle_layout(sr.sumregs_gradient_reg(_maps(lam, n), u, t, grid, gamma=1e8, refine=3))
    # the bar of the band LU's emulation test (tests/test_emu_lu.py): at γ = 1e8 the patch holding the flat block is
    # only as accurate as refinement with an fp64 residual makes it, and the band LU lands at the same distance (1.2e-9
    # on the 16² 2×2 case, within 3e-16 of this result on every case here)
    assert np.all(np.abs(got - lit) <= 2e-9 * np.abs(lit).max()), (got, lit)


@pytest.mark.parametrize("n", [16, 24])
def test_uniform_maps_match_the_cholesky(lib, n):
    """equal patches per operator: the system is symmetric, and the LU reproduces the Cholesky of the same fronts"""
    t, u = _case(n, 31 + n)
    x = np.array([0.05, 0.04, 0.06])
    lam = np.broadcast_to(x, (2, 2, 3)).copy()
    got, stats, _ = _run(lib, u, t, lam, gamma=1e3)
    chol, cstats, _ = _run(lib, u, t, None, scalar=x, gamma=1e3, refine=3)
    assert stats[1] == 0 and cstats[1] == 0
    g = got.reshape(3, 4).sum(axis=1)
    assert np.all(np.abs(g - chol) <= 1e-10 * np.abs(chol).max()), (g, chol)


@pytest.mark.parametrize("smem_limit", [WIDE, NARROW])
def test_bits_do_not_depend_on_the_cluster_or_the_panel_place(lib, smem_limit):
    """the same bits for 1, 2 and 4 CTAs per front, and with the panels in global memory, at NB = 16 and NB = 8"""
    t, u = _case(40, 3)
    lam = _lam((3, 2), 11)
    ref = _run(lib, u, t, lam, csize=1, smem_limit=smem_limit)
    assert ref[1][1] == 0 and ref[1][4] == 0
    assert (ref[1][3] == ref[1][2]) == (smem_limit == NARROW) and (ref[1][3] == 0) == (smem_limit == WIDE), ref[1]
    runs = [_run(lib, u, t, lam, csize=c, smem_limit=smem_limit) for c in (2, 4)]
    runs += [_run(lib, u, t, lam, csize=c, smem_limit=smem_limit, large=ALL) for c in (1, 2)]
    assert runs[-1][1][4] == ref[1][2], runs[-1][1]        # every level on the global-memory panels
    for got in runs:
        assert np.array_equal(got[0], ref[0]) and np.array_equal(got[2], ref[2])
        assert got[1][0] == ref[1][0]


def test_small_level_solves_give_the_same_result(lib):
    """the bottom levels' warp-per-front solves run on L and Uᵀ as well (the factorisation stays on the per-CTA kernel)"""
    t, u = _case(40, 5)
    lam = _lam((2, 2), 4)
    a = _run(lib, u, t, lam, small=0)
    b = _run(lib, u, t, lam, small=1)
    assert np.all(np.abs(a[0] - b[0]) <= 1e-12 * np.abs(a[0]).max())


def test_zero_pivot_breaks_down_to_nan(lib):
    t, u = _case(24, 9)
    lam = _lam((2, 2), 2)
    got, stats, _ = _run(lib, u, t, lam, zero_row=24 * 5 + 7)
    assert stats[1] != 0
    assert np.all(np.isnan(got)), got
