"""Host build of the per-element batch-statistics arithmetic (pumiumtally_b200/csrc/batch_stats.cuh): the
running sums S1, S2 that Engine::end_batch accumulates on the device, and the mean and standard deviation of
the mean read out of them, against numpy.  Needs g++, no GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from helpers import ROOT

_TU = r"""
#include "batch_stats.cuh"
extern "C" void batch_stats(const double *x, int64_t nb, int64_t ne, const double *vol, double *mean, double *sd) {
  for (int64_t e = 0; e < ne; ++e) {
    double s1 = NAN, s2 = NAN;  // the first batch must not read the sums
    for (int64_t b = 0; b < nb; ++b) ptb::batch_accumulate(x[b * ne + e], s1, s2, b == 0);
    mean[e] = ptb::batch_mean(s1, double(nb), vol[e]);
    sd[e] = ptb::batch_std_dev(s1, s2, double(nb), vol[e]);
  }
}
extern "C" double batch_rel(double mean, double sd) { return ptb::batch_relative_error(mean, sd); }
"""


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    d = tmp_path_factory.mktemp("batch_stats")
    src, so = d / "bs.cpp", d / "bs.so"
    src.write_text(_TU)
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-shared", "-fPIC", "-I",
                           os.path.join(ROOT, "pumiumtally_b200", "csrc"), str(src), "-o", str(so)])
    L = C.CDLL(str(so))
    dp = C.POINTER(C.c_double)
    L.batch_stats.argtypes = [dp, C.c_int64, C.c_int64, dp, dp, dp]
    L.batch_stats.restype = None
    L.batch_rel.argtypes = [C.c_double, C.c_double]
    L.batch_rel.restype = C.c_double
    return L


def _run(lib, x, vol):
    x = np.ascontiguousarray(x, dtype=np.float64)
    vol = np.ascontiguousarray(vol, dtype=np.float64)
    nb, ne = x.shape
    mean, sd = np.empty(ne), np.empty(ne)
    dp = C.POINTER(C.c_double)
    lib.batch_stats(x.ctypes.data_as(dp), nb, ne, vol.ctypes.data_as(dp), mean.ctypes.data_as(dp), sd.ctypes.data_as(dp))
    return mean, sd


def _numpy(x, vol):
    n = x.shape[0]
    return np.mean(x, axis=0) / vol, np.std(x, axis=0, ddof=1) / np.sqrt(n) / vol


def _check(lib, x, vol):
    mean, sd = _run(lib, x, vol)
    want_m, want_s = _numpy(x, vol)
    np.testing.assert_allclose(mean, want_m, rtol=1e-15, atol=0)
    assert (sd >= 0).all() and np.isfinite(sd).all()
    np.testing.assert_array_less(np.abs(sd - want_s), 1e-9 * want_s + 1e-12 * np.abs(want_m) + 1e-300)
    return mean, sd


def test_one_batch_has_a_mean_and_no_standard_deviation(lib):
    rng = np.random.default_rng(1)
    x, vol = rng.random((1, 500)) * 10, rng.random(500) + 0.1
    mean, sd = _run(lib, x, vol)
    np.testing.assert_allclose(mean, x[0] / vol, rtol=1e-15, atol=0)
    assert np.isnan(sd).all()


@pytest.mark.parametrize("n", [2, 3, 6, 40])
def test_positive_scores_against_numpy(lib, n):
    rng = np.random.default_rng(n)
    x = rng.gamma(2.0, 3.0, (n, 2000))
    _check(lib, x, rng.random(2000) + 0.05)


def test_negative_scores_against_numpy(lib):
    rng = np.random.default_rng(7)
    x = -rng.gamma(2.0, 3.0, (5, 1000))  # a tally of a signed quantity: every value below zero
    mean, sd = _check(lib, x, rng.random(1000) + 0.05)
    assert (mean < 0).all()


def test_zero_mean_and_all_zero_elements(lib):
    x = np.array([[1.0, 0.0, 2.5], [-1.0, 0.0, -2.5]])
    mean, sd = _run(lib, x, np.ones(3))
    np.testing.assert_array_equal(mean, [0.0, 0.0, 0.0])
    np.testing.assert_array_equal(sd, [1.0, 0.0, 2.5])  # np.std(ddof=1) / sqrt(2) of +-a is a
    assert lib.batch_rel(0.0, 1.0) < 0  # zero-mean pairs are left out of the trigger
    assert lib.batch_rel(-2.0, 1.0) == 0.5


def test_identical_batches_give_a_rounding_residue_not_nan(lib):
    rng = np.random.default_rng(3)
    row = rng.random(3000) * 10 ** rng.uniform(-5, 5, 3000)
    for n in (2, 3, 7, 100):
        mean, sd = _run(lib, np.tile(row, (n, 1)), np.ones(3000))
        assert np.isfinite(sd).all() and (sd >= 0).all()
        assert (sd <= 1e-7 * np.abs(mean)).all(), (n, np.max(sd / mean))


def test_cancellation_in_the_sum_of_squares(lib):
    """1e4 batches of values around 1e6 with a relative spread of 1e-4: S2/n and (S1/n)^2 agree to about 8
    digits, and each of the 1e4 additions to S2 (~1e16) rounds by up to half an ulp (~1), so the variance
    (~1e4 per batch) keeps only about 1e-6 of relative accuracy in the standard deviation -- the price of
    plain running sums, which is what a running tally can keep per element.  Hence 1e-5 here instead of
    1e-9."""
    rng = np.random.default_rng(11)
    x = 1e6 * (1.0 + 1e-4 * rng.standard_normal((10_000, 64)))
    mean, sd = _run(lib, x, np.ones(64))
    want_m, want_s = _numpy(x, np.ones(64))
    np.testing.assert_allclose(mean, want_m, rtol=1e-15, atol=0)
    assert np.isfinite(sd).all() and (sd >= 0).all()
    np.testing.assert_allclose(sd, want_s, rtol=1e-5)
