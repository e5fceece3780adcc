"""Kernel C's projection scales a pixel inside the λ-ball by BallScale(α², α) instead of selecting: that factor is exactly 1.

RN(√RN(α²)) = α for every binary floating-point α > 0 whose square neither overflows nor underflows (Boldo 2015), so
RN(α / RN(√RN(α²))) = 1, and the chain only sees α in BallScale's fast range 2⁻²⁰⁰ ≤ α < 2²⁰⁰ (2⁻³⁰ ≤ α < 2³⁰ in fp32).
numpy's sqrt, multiply and divide are the correctly rounded IEEE operations, as on the GPU.
"""
import numpy as np
import pytest


def _alphas(dtype, lo, hi, n=2_000_000, seed=3):
    rng = np.random.default_rng(seed)
    a = np.exp2(rng.uniform(lo, hi, n)).astype(dtype)
    # significands with their upper bits all ones / all zeros, one ulp around powers of two
    p = np.exp2(np.arange(lo, hi, dtype=np.float64)).astype(dtype)
    edge = np.concatenate([p, np.nextafter(p, dtype(0)), np.nextafter(p, dtype(np.inf)),
                           np.nextafter(np.nextafter(p, dtype(0)), dtype(0))])
    a = np.concatenate([a, edge])
    return a[(a >= dtype(2.0 ** lo)) & (a < dtype(2.0 ** hi))]


@pytest.mark.parametrize("dtype,lo,hi", [(np.float64, -200, 200), (np.float32, -30, 30)])
def test_scale_of_alpha_squared_is_one(dtype, lo, hi):
    a = _alphas(dtype, lo, hi)
    s = np.sqrt(a * a)
    assert s.dtype == dtype
    assert np.array_equal(s, a)
    assert np.all(a / s == dtype(1))


def test_image_range_alphas():
    # the λ values the project's configurations use, and a dense sweep around them
    a = np.concatenate([np.array([0.01, 0.05, 0.08, 0.1, 0.5, 1.0, 2.0]), np.linspace(1e-4, 10.0, 1_000_001)])
    for dt in (np.float64, np.float32):
        x = a.astype(dt)
        assert np.array_equal(np.sqrt(x * x), x)
