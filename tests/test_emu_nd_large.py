"""CPU check of the large-front variants of the nested-dissection solver (bpldenoising_b200/csrc/nd_solver.cuh:
nd_factor_*large*, nd_fwd/bwd_large_kernel), which keep the factorisation's panel and the solves' front vector in global
memory for fronts beyond shared memory.  The device code runs on the thread emulation (tests/emu/emu_cuda.h) through
tests/emu/emu_nd_large.cpp, which sends every level whose shared-memory kernels would take more than
`large_limit` bytes to the variants, as nd_level_large does on the device.  On small crops the variants must give the
bits of the shared-memory kernels at the same block width, alone and shared by a cluster, in node space (W = 2,
scalar sumregs_gradient_reg) and in multiplier space (sumregs_gradient), and match the oracle's literal solves.
The GPU counterpart is tests/test_gpu_sumregs_large.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import sumregs as sr

HERE = os.path.dirname(os.path.abspath(__file__))
EMU = os.path.join(HERE, "emu")
CSRC = os.path.join(HERE, "..", "bpldenoising_b200", "csrc")

ALL = 0          # large_limit: every generic level on the variants
NONE = -1        # none


@pytest.fixture(scope="module")
def lib():
    out = os.path.join(EMU, "_build", "libemu_nd_large.so")
    srcs = [os.path.join(EMU, "emu_nd_large.cpp"), os.path.join(EMU, "emu_cuda.h")] + \
           [os.path.join(CSRC, f) for f in ("nd_symbolic.h", "nd_solver.cuh", "nd_sumregs.cuh", "lu_band.cuh",
                                            "sumregs_stencils.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        subprocess.run(["g++", "-std=c++20", "-O1", "-pthread", "-fPIC", "-shared", "-DBPLTV_EMU", "-ffp-contract=off",
                        "-o", out, srcs[0]], check=True)
    lib = C.CDLL(out)
    lib.emu_nd_large_gradient_reg.restype = C.c_int
    lib.emu_nd_large_gradient_mult.restype = C.c_int
    return lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))


def _case(n, seed):
    rng = np.random.default_rng(seed)
    t = np.round(rng.random((n, n)) * 255) / 255
    u = np.asfortranarray(t + 0.05 * rng.standard_normal((n, n)))
    u[:3, :3] = u[0, 0]                      # exactly flat blocks: γ·I tensors / two multipliers per operator
    u[n - 4:, n - 5:] = u[n - 1, n - 1]
    return np.asfortranarray(t), u


X = np.array([0.05, 0.04, 0.06])


def _reg(lib, u, t, large, csize=1, small=1, refine=1):
    n = u.shape[0]
    out, stats, p = np.zeros(3), np.zeros(8), np.zeros(n * n)
    rc = lib.emu_nd_large_gradient_reg(n, _ptr(u.flatten(order="F")), _ptr(t.flatten(order="F")), _ptr(X), C.c_double(1e3),
                                     refine, 4, int(small), csize, C.c_longlong(large), _ptr(out), _ptr(stats), _ptr(p), None)
    assert rc == 0
    return out, stats, p


def _mult(lib, u, t, large, csize=1, smem_limit=1 << 30, refine=1):
    n = u.shape[0]
    out, stats, p = np.zeros(3), np.zeros(8), np.zeros(n * n)
    rc = lib.emu_nd_large_gradient_mult(n, _ptr(u.flatten(order="F")), _ptr(t.flatten(order="F")), _ptr(X), None, 1, 1,
                                      C.c_double(1e-12), C.c_double(sr.EPS), refine, 4, csize, C.c_longlong(smem_limit),
                                      C.c_longlong(large), _ptr(out), _ptr(stats), _ptr(p))
    assert rc == 0
    return out, stats, p


def _same(a, b):
    ga, sa, pa = a
    gb, sb, pb = b
    assert np.array_equal(ga, gb) and np.array_equal(pa, pb), (ga, gb)
    assert sa[0] == sb[0] and sa[1] == sb[1] and sa[2] == sb[2]


@pytest.mark.parametrize("csize", [1, 2, 3])
def test_node_form_large_fronts_give_the_same_bits(lib, csize):
    """scalar sumregs_gradient_reg (node space, W = 2): every generic level, or only the upper ones, on the variants"""
    t, u = _case(24, 5)
    ref = _reg(lib, u, t, NONE, csize=csize, small=0)
    assert ref[1][6] == 0 and ref[1][7] == 0
    for large in (ALL, 14000):
        got = _reg(lib, u, t, large, csize=csize, small=0)
        if large == ALL:
            assert got[1][6] == got[1][4] and got[1][7] == got[1][4], got[1]     # every level
        else:
            assert 0 < got[1][6] < got[1][4], got[1]                             # the upper levels only
        _same(got, ref)


@pytest.mark.parametrize("csize", [1, 2])
@pytest.mark.parametrize("smem_limit", [1 << 30, 20000])
def test_multiplier_form_large_fronts_give_the_same_bits(lib, csize, smem_limit):
    """sumregs_gradient (multiplier space): 16-column block steps, and 8-column ones on the upper levels (smem_limit)"""
    t, u = _case(13, 17)
    ref = _mult(lib, u, t, NONE, csize=csize, smem_limit=smem_limit)
    assert ref[1][6] == 0 and (ref[1][5] > 0) == (smem_limit < 1 << 30)
    for large in (ALL, 16000):      # 16000: the upper levels only
        got = _mult(lib, u, t, large, csize=csize, smem_limit=smem_limit)
        assert got[1][6] > 0 and (got[1][7] > 0) == (large == ALL) and got[1][5] == ref[1][5], got[1]
        _same(got, ref)


def test_node_form_large_fronts_match_the_literal_solve(lib):
    t, u = _case(20, 60)
    got, stats, _ = _reg(lib, u, t, ALL, csize=2, small=0)
    lit = sr.sumregs_gradient_reg(X, u, t, refine=3)
    assert stats[1] == 0 and stats[6] > 0
    assert np.all(np.abs(got - lit) <= 1e-9 * np.abs(lit).max()), (got, lit)


def test_multiplier_form_large_fronts_match_the_oracle(lib):
    t, u = _case(16, 83)
    got, stats, _ = _mult(lib, u, t, ALL, csize=2)
    assert stats[2] == 0 and stats[6] > 0
    du = sr.sumregs_gradient_dual("nonreg", X, u, t)
    assert np.all(np.abs(got - du) <= 1e-10 * np.abs(du).max()), (got, du)
    lit = sr.sumregs_gradient(X, u, t, refine=3)
    assert np.all(np.abs(got - lit) <= 1e-6 * np.abs(lit).max()), (got, lit)
