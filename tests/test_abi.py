"""C-ABI boundary checks that need no GPU: the library loads, exports every symbol
include/bpltv.h declares, its defaults are the reference's parameters, and it refuses
to run without a CUDA device (no CPU fallback)."""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest

from conftest import ROOT


def test_exports_match_header(bp):
    hdr = open(os.path.join(ROOT, "include", "bpltv.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = sorted(set(re.findall(r"\b(bpltv_[a-z_]+)\s*\(", hdr)))
    assert declared, "no declarations found"
    L = bp._lib.load()
    for name in declared:
        assert hasattr(L, name), f"{name} declared in bpltv.h but not exported"
    assert sorted(bp._lib.EXPORTS) == declared
    assert L.bpltv_version() == 100


def test_defaults_are_the_reference_parameters(bp):
    o = bp.pdps_opts()
    # /root/reference/src/TVLearningFunctionVec.jl:33-43
    assert (o.tau0, o.sigma0, o.rho, o.accel, o.maxiter) == (5.0, 0.99 / 5, 0.0, 1, 5000)
    assert abs(o.opnorm - 8 ** 0.5) < 1e-15 and o.init_mode == 0 and o.arith == bp.STRICT
    e = bp.eval_opts()
    assert (e.delta_t, e.gamma, e.act_tol) == (1e-6, 1e8, 1e-12)  # :14, :142, :109
    o2 = bp.pdps_opts(maxiter=10000, verbose_iter=10001, ρ=0.5)
    assert o2.maxiter == 10000 and o2.rho == 0.5
    with pytest.raises(TypeError):
        bp.pdps_opts(bogus=1)


def test_struct_layout_matches_c(bp):
    # sizes the C compiler computes for the header's structs (natural alignment)
    assert C.sizeof(bp._lib.PdpsOpts) == 4 * 8 + 10 * 4
    assert C.sizeof(bp._lib.EvalOpts) == C.sizeof(bp._lib.PdpsOpts) + 5 * 8 + 8 * 4 == 144
    assert bp._lib.EvalOpts.gamma_patch.offset == 128      # static_assert'ed on the C side (bpltv_api.cu)
    assert C.sizeof(bp._lib.Stats) == 6 * 8 + 4 * 8 + 8 + 8 * 4


def test_no_cpu_fallback():
    # a process that sees no device, also on a GPU machine: CUDA_VISIBLE_DEVICES is read once, at CUDA's initialisation
    code = ("import bpldenoising_b200 as bp\n"
            "try:\n    bp.Context()\nexcept bp.BpltvError as e:\n    print(e.code, e)\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=300,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.startswith("-3 ") and "no CPU fallback" in r.stdout, r.stdout


def test_argument_errors_before_any_device_work(bp):
    L = bp._lib.load()
    h = C.c_void_p()
    assert L.bpltv_create(None, 1, 48, C.byref(h)) == -1
    assert b"precision" in L.bpltv_last_error()
    assert L.bpltv_create(None, 0, 64, C.byref(h)) == -1
    assert L.bpltv_destroy(None) == 0


def test_product_does_not_import_the_oracle():
    # the oracle is test infrastructure: nothing under bpldenoising_b200/ may use it
    pkg = os.path.join(ROOT, "bpldenoising_b200")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, fn), encoding="utf-8").read()
                assert "import oracle" not in txt and "from oracle" not in txt and "liboracle" not in txt, fn
