"""The per-DOF envelope on the CPU: the device's per-record terms (eskf_math.cuh dof_terms) through a host harness against
numpy, and ``consistency.summarise_dofs`` against scipy."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from dvi_ekf_b200.consistency import summarise_dofs
from tests.dof_reference import PAIRS, USED, dof_terms, envelope

dp = ctypes.POINTER(ctypes.c_double)


def _p(a):
    return a.ctypes.data_as(dp)


@pytest.fixture(scope="module")
def hc(tmp_path_factory):
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostcheck", "dof_check.cpp")
    lib_path = str(tmp_path_factory.mktemp("hostcheck") / "libdofcheck.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", lib_path, src], check=True)
    lib = ctypes.CDLL(lib_path)
    lib.hc_dof_terms.argtypes = [dp, dp, dp, ctypes.POINTER(ctypes.c_int32), ctypes.c_int64, dp]
    lib.hc_dof_terms.restype = None
    assert lib.hc_dof_used() == USED
    return lib


def _terms(hc, nis, eps, B, masks):
    nis, eps = np.ascontiguousarray(nis, dtype=float), np.ascontiguousarray(eps, dtype=float)
    B = np.ascontiguousarray(B, dtype=float).reshape(len(nis), 36)
    masks = np.ascontiguousarray(np.broadcast_to(masks, (len(nis),)), dtype=np.int32)
    out = np.empty((len(nis), USED))
    hc.hc_dof_terms(_p(nis), _p(eps), _p(B), masks.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), len(nis), _p(out))
    return out


def _blocks(rng, n):
    """n random SPD 6x6 blocks with a relative asymmetry of 1e-11 (as the filter's P has), scaled over 8 decades"""
    A = rng.normal(size=(n, 6, 6))
    B = A @ A.transpose(0, 2, 1) + 0.1 * np.eye(6)
    B *= 1 + 1e-11 * rng.normal(size=B.shape)
    return B * 10.0 ** rng.uniform(-6, 2, (n, 1, 1))


def test_terms_every_frozen_mask(hc):
    """random blocks and errors (about a third outside 1 sigma) under all 64 masks: the same bits as numpy"""
    rng = np.random.default_rng(11)
    n = 50
    for mask in range(64):
        B = _blocks(rng, n)
        eps = rng.normal(size=(n, 6)) * np.sqrt(np.diagonal(B, axis1=1, axis2=2)) * 1.5
        nis = rng.chisquare(7, n)
        got = _terms(hc, nis, eps, B, mask)
        ref = dof_terms(nis, eps, B, mask)
        assert np.array_equal(got, ref), (mask, np.argwhere(got != ref)[:5])
        assert (got[:, 0] == 1).all() and (got[:, 1] == 0).all()
        for i in range(6):
            if (mask >> i) & 1:
                assert (got[:, 2 + 7 * i:9 + 7 * i] == 0).all()
        for p, (i, j) in enumerate(PAIRS):
            if (mask >> i) & 1 or (mask >> j) & 1:
                assert (got[:, 44 + p] == 0).all() and (got[:, 59 + p] == 0).all()
        if mask == 0:
            assert 0 < got[:, 2 + 4].mean() < 1  # the 1-sigma counts are really exercised


@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf])
def test_non_finite_values_exclude(hc, bad):
    """a non-finite NIS, error or any entry of the block excludes the filter when it concerns an estimated DOF (or pair),
    and changes nothing when it concerns a frozen one"""
    rng = np.random.default_rng(12)
    B0 = _blocks(rng, 1)[0]
    e0 = rng.normal(size=6) * np.sqrt(np.diag(B0))
    cases = []  # (nis, eps, B, mask, excluded)
    cases.append((bad, e0, B0, 0, True))
    for i in range(6):
        e = e0.copy()
        e[i] = bad
        cases.append((7.0, e, B0, 0, True))
        cases.append((7.0, e, B0, 1 << i, False))
    for i in range(6):
        for j in range(6):
            B = B0.copy()
            B[i, j] = bad
            cases.append((7.0, e0, B, 0, True))
            cases.append((7.0, e0, B, 1 << j, False))  # frozen j: the entry is in a frozen DOF's row or column
            if i != j:
                cases.append((7.0, e0, B, 63 & ~((1 << i) | (1 << j)) | (1 << i), False))  # only j estimated
    for nis, e, B, mask, excl in cases:
        got = _terms(hc, [nis], e[None], B[None], mask)[0]
        ref = dof_terms([nis], e[None], B[None], mask)[0]
        assert np.array_equal(got, ref), (nis, mask)
        assert got[1] == float(excl) and got[0] == float(not excl), (nis, mask, got[:2])
        if excl:
            assert (got[2:] == 0).all()


def test_zero_and_negative_variance_exclude(hc):
    rng = np.random.default_rng(13)
    B0 = _blocks(rng, 1)[0]
    e0 = rng.normal(size=6)
    for v in (0.0, -0.0, -1e-30, -3.0):
        for i in range(6):
            B = B0.copy()
            B[i, i] = v
            assert _terms(hc, [7.0], e0[None], B[None], 0)[0, 1] == 1.0
            assert _terms(hc, [7.0], e0[None], B[None], 1 << i)[0, 0] == 1.0  # frozen: not looked at
    P = np.zeros((6, 6))  # P0 = 0
    assert _terms(hc, [7.0], e0[None], P[None], 0)[0, 1] == 1.0
    assert _terms(hc, [7.0], e0[None], P[None], 63)[0, 0] == 1.0  # d = 0: only the NIS decides


def test_coverage_boundaries_count_as_inside(hc):
    """eps^2 == k^2 B_ii exactly (3^2 = 9 B with B = 9, 2.25, 1): inside at k and above"""
    B = np.diag([9.0, 2.25, 1.0, 9.0 * (1 + 2 ** -52), 2.25 * (1 - 2 ** -53), 1.0 - 2 ** -53])
    eps = np.full(6, 3.0)
    t = _terms(hc, [7.0], eps[None], B[None], 0)[0]
    cov = t[2:44].reshape(6, 7)[:, 4:7]
    assert cov.tolist() == [[1, 1, 1], [0, 1, 1], [0, 0, 1], [1, 1, 1], [0, 0, 1], [0, 0, 0]]
    assert np.array_equal(t, dof_terms([7.0], eps[None], B[None], 0)[0])


def _sample(rng, N, E, frozen_mask, bias=0.0, infl=1.0):
    """nis [N,E], dofs [N,E,6], B [N,E,6,6], gt: a synthetic ensemble whose errors are infl x the claimed sigma"""
    B = _blocks(rng, N * E).reshape(N, E, 6, 6)
    L = np.linalg.cholesky(0.5 * (B + B.transpose(0, 1, 3, 2)))
    gt = rng.normal(size=6)
    dofs = gt + bias + infl * np.einsum("neij,nej->nei", L, rng.normal(size=(N, E, 6)))
    return rng.chisquare(7, (N, E)), dofs, B, gt


def test_summary_against_scipy():
    from scipy.special import erf
    from scipy.stats import binom, chi2

    rng = np.random.default_rng(21)
    N, E, mask = 400, 5, 0b000100  # DOF 2 frozen
    frozen = [(mask >> i) & 1 for i in range(6)]
    nis, dofs, B, gt = _sample(rng, N, E, mask, bias=0.1, infl=2.0)
    nis[:7, 1] = np.nan  # 7 filters excluded at epoch 1
    nis[:, 3] = np.nan  # M = 0 at epoch 3
    nis[1:, 4] = np.nan  # M = 1 at epoch 4
    s = summarise_dofs(envelope(nis, dofs, B, gt, mask), frozen, alpha=0.1)
    assert s["count"].tolist() == [N, N - 7, N, 0, 1] and s["excluded"].tolist() == [0, 7, 0, N, N - 1]
    for e in range(E):
        ok = np.isfinite(nis[:, e])
        m = ok.sum()
        for key in ("bias", "rmse", "std", "sigma_filter", "inflation", "anees_dof"):
            assert np.isnan(s[key][e, 2]), key  # frozen
        if m == 0:
            for key in ("bias", "rmse", "std", "sigma_filter", "inflation", "anees_dof", "coverage", "err_second_moment",
                        "filter_cov", "anees_interval", "coverage_interval"):
                assert np.isnan(s[key][e]).all(), key
            continue
        eps = dofs[ok, e] - gt
        var = B[ok, e][:, np.arange(6), np.arange(6)]
        keep = [0, 1, 3, 4, 5]
        np.testing.assert_allclose(s["bias"][e, keep], eps[:, keep].mean(0), rtol=1e-12)
        np.testing.assert_allclose(s["rmse"][e, keep], np.sqrt((eps[:, keep] ** 2).mean(0)), rtol=1e-12)
        np.testing.assert_allclose(s["sigma_filter"][e, keep], np.sqrt(var[:, keep].mean(0)), rtol=1e-12)
        np.testing.assert_allclose(s["inflation"][e, keep], s["rmse"][e, keep] / s["sigma_filter"][e, keep], rtol=1e-15)
        np.testing.assert_allclose(s["anees_dof"][e, keep], (eps[:, keep] ** 2 / var[:, keep]).mean(0), rtol=1e-12)
        if m >= 2:
            np.testing.assert_allclose(s["std"][e, keep], eps[:, keep].std(0, ddof=1), rtol=1e-9)
        else:
            assert np.isnan(s["std"][e]).all()
        assert np.allclose(s["anees_interval"][e], [chi2.ppf(0.05, m) / m, chi2.ppf(0.95, m) / m], rtol=1e-14)
        p = erf(np.arange(1, 4) / np.sqrt(2))
        assert np.allclose(s["coverage_expected"], p, rtol=1e-15)
        for k in range(3):
            inside = (eps[:, keep] ** 2 <= (k + 1) ** 2 * var[:, keep]).mean(0)
            assert np.array_equal(s["coverage"][e, keep, k], inside)
            assert np.array_equal(s["coverage_interval"][e, k], [binom.ppf(0.05, m, p[k]) / m, binom.ppf(0.95, m, p[k]) / m])
        em = np.einsum("ni,nj->ij", eps, eps) / m
        fc = (B[ok, e] + B[ok, e].transpose(0, 2, 1)).sum(0) / (2 * m)
        for ref, key in ((em, "err_second_moment"), (fc, "filter_cov")):
            got = s[key][e]
            assert np.isnan(got[2]).all() and np.isnan(got[:, 2]).all()
            np.testing.assert_allclose(got[np.ix_(keep, keep)], ref[np.ix_(keep, keep)], rtol=1e-11, atol=1e-13 * np.abs(ref).max())
    assert 1.5 < np.nanmean(s["inflation"][0]) < 2.5  # the synthetic errors are 2 x the claimed sigma, plus the bias


def test_summary_of_two_shards_is_that_of_one():
    """shards add their dof_sum (all-reduce); the summary of the sum is that of the whole job"""
    rng = np.random.default_rng(22)
    nis, dofs, B, gt = _sample(rng, 600, 4, 0)
    nis[rng.random(nis.shape) < 0.02] = np.nan
    whole = envelope(nis, dofs, B, gt, 0)
    split = envelope(nis[:250], dofs[:250], B[:250], gt, 0) + envelope(nis[250:], dofs[250:], B[250:], gt, 0)
    sw, ss = summarise_dofs(whole, [0] * 6), summarise_dofs(split, [0] * 6)
    for key, v in sw.items():
        np.testing.assert_allclose(ss[key], v, rtol=1e-12, atol=1e-15)
    for key in ("count", "excluded", "coverage"):
        assert np.array_equal(ss[key], sw[key])
    # a consistent synthetic filter (whose variances span 8 decades, so that RMSE / mean sigma says little): per-DOF ANEES
    # near 1, coverage near erf(k / sqrt 2)
    assert np.all(np.abs(sw["anees_dof"] - 1) < 0.3)
    assert np.all(np.abs(sw["coverage"] - sw["coverage_expected"]) < 0.06)
