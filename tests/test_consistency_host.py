"""Filter consistency on the CPU: the NIS and NEES arithmetic of the device (eskf_cov3.cuh upd3_nis, eskf_math.cuh nees_dofs)
through the tests/hostcheck harness against numpy and the oracle, and the Python summary / tuning objective."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from dvi_ekf_b200.consistency import candidate_objective, summarise_consistency
from tests.consistency_oracle import RecordingOracle as BatchOracle
from tests.helpers import mandala_scenario

dp = ctypes.POINTER(ctypes.c_double)


def _p(a):
    return a.ctypes.data_as(dp)


@pytest.fixture(scope="module")
def hc(tmp_path_factory):
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostcheck", "consistency_check.cpp")
    lib_path = str(tmp_path_factory.mktemp("hostcheck") / "libconsistencycheck.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", lib_path, src], check=True)
    lib = ctypes.CDLL(lib_path)
    lib.hc_nis3.argtypes = [dp, dp, dp, dp, dp, ctypes.c_double, dp]
    lib.hc_nis3.restype = ctypes.c_double
    lib.hc_nees.argtypes = [dp, dp, ctypes.POINTER(ctypes.c_int32), ctypes.c_int64, dp]
    lib.hc_nees.restype = None
    return lib


def _nees(hc, B, eps, masks):
    B, eps = np.ascontiguousarray(B, dtype=float), np.ascontiguousarray(eps, dtype=float)
    masks = np.ascontiguousarray(masks, dtype=np.int32)
    out = np.empty(len(B))
    hc.hc_nees(_p(B), _p(eps), masks.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), len(B), _p(out))
    return out


def _ref_nees(B, e, mask):
    keep = [i for i in range(6) if not (mask >> i) & 1]
    if not keep:
        return np.nan
    Bs = B.reshape(6, 6)[np.ix_(keep, keep)]
    return float(e[keep] @ np.linalg.solve(Bs, e[keep]))


def _spd(rng, cond):
    Q, _ = np.linalg.qr(rng.normal(size=(6, 6)))
    return (Q * np.logspace(0, -np.log10(cond), 6)) @ Q.T


@pytest.mark.parametrize("cond", [1e1, 1e4, 1e8, 1e12])
def test_nees_against_numpy_solve(hc, cond):
    """SPD blocks up to condition 1e12, exactly symmetric and with a relative asymmetry of 1e-11 (as the reference's P
    has), all DOFs estimated: the LU solve agrees with np.linalg.solve to the conditioning of the block"""
    rng = np.random.default_rng(int(np.log10(cond)))
    n = 200
    B = np.array([_spd(rng, cond) for _ in range(n)])
    B[n // 2:] *= 1 + 1e-11 * rng.normal(size=(n - n // 2, 6, 6))  # slightly asymmetric
    B *= 10.0 ** rng.uniform(-6, 2, (n, 1, 1))
    eps = rng.normal(size=(n, 6)) * np.sqrt(np.abs(np.diagonal(B, axis1=1, axis2=2)))
    got = _nees(hc, B.reshape(n, 36), eps, np.zeros(n))
    ref = np.array([_ref_nees(B[i], eps[i], 0) for i in range(n)])
    rel = np.abs(got / ref - 1)
    assert rel.max() < 100 * np.finfo(float).eps * cond, rel.max()


def test_nees_every_frozen_mask(hc):
    """all 64 masks: the estimated DOFs' sub-block only, NaN when all six are frozen"""
    rng = np.random.default_rng(5)
    masks = np.arange(64)
    B = np.array([_spd(rng, 1e3) for _ in masks]).reshape(64, 36)
    eps = rng.normal(size=(64, 6))
    got = _nees(hc, B, eps, masks)
    ref = np.array([_ref_nees(B[i], eps[i], int(m)) for i, m in enumerate(masks)])
    assert np.isnan(got[63]) and np.isnan(ref[63])
    assert np.all(np.abs(got[:63] / ref[:63] - 1) < 1e-12), np.abs(got[:63] / ref[:63] - 1).max()
    # a frozen DOF's row, column and error do not enter: garbage there changes nothing
    Bg, eg = B.reshape(64, 6, 6).copy(), eps.copy()
    for i, m in enumerate(masks):
        for k in range(6):
            if (m >> k) & 1:
                Bg[i, k, :] = Bg[i, :, k] = np.nan
                eg[i, k] = np.inf
    assert np.array_equal(_nees(hc, Bg.reshape(64, 36), eg, masks), got, equal_nan=True)


def test_nees_singular_and_non_finite_blocks(hc):
    rng = np.random.default_rng(9)
    B = _spd(rng, 1e2)
    eps = rng.normal(size=6)
    cases = []
    Z = np.zeros((6, 6))
    cases.append(Z)  # P0 = 0
    S = B.copy()
    S[2] = S[4]
    S[:, 2] = S[:, 4]  # two identical rows: exactly singular
    cases.append(S)
    for bad in (np.nan, np.inf, -np.inf):
        X = B.copy()
        X[3, 1] = bad
        cases.append(X)
    got = _nees(hc, np.array(cases).reshape(len(cases), 36), np.repeat(eps[None], len(cases), 0), np.zeros(len(cases)))
    assert np.isnan(got).all(), got
    # a frozen DOF's singular row does not make the block singular
    assert np.isfinite(_nees(hc, S.reshape(1, 36), eps[None], [1 << 2]))[0]


@pytest.mark.parametrize("frozen", [(1,) * 6, (0,) * 6])
def test_nis_lockstep_against_oracle(hc, golden, frozen):
    """upd3_nis on the record the register-tile update builds (hc_nis3 follows hc_update3 up to the gain) against the batch
    oracle's r inv(S) r, 30 epochs in lock step; the first update is the prior >> R case (cond(S) 1.4e7).
    The host replay inverts with inv7, the device with inv7_group3: tests/test_gpu_consistency.py covers that."""
    sc = mandala_scenario(golden, n_frames=31, ifv=10, frozen_dofs=frozen)
    bo = BatchOracle(sc.cfg, sc.x0, sc.P0, sc.u0, sc.Qd, sc.Rd, sc.sig_om)
    k, worst, conds = 0, 0.0, []
    for e in range(len(sc.n_prop)):
        for _ in range(sc.n_prop[e]):
            bo.propagate(sc.dt[k], sc.om_acc[k, :3], sc.om_acc[k, 3:])
            k += 1
        x, P = bo.x[0].copy(), bo.P[0].copy()
        u = np.hstack((bo.om_old[0], bo.acc_old[0]))
        Ro = bo.R_old[0].reshape(9).copy()
        got = hc.hc_nis3(_p(x), _p(P), _p(u), _p(Ro), _p(sc.cam_meas[e].copy()), sc.notch_meas[e], _p(sc.Rd))
        bo.update(sc.cam_meas[e, :3], sc.cam_meas[e, 3:], sc.notch_meas[e])
        r, S = bo.res[0], bo.S[0]
        ref = float(r @ np.linalg.inv(S) @ r)
        conds.append(np.linalg.cond(S))
        worst = max(worst, abs(got / ref - 1))
    print(f"MEASURED host NIS vs oracle, frozen={frozen}: worst relative {worst:.2e}, max cond(S) {max(conds):.1e}")
    assert worst < 5e-13, worst  # measured 1.4e-13 (all DOFs frozen) / 2.0e-14 (estimated)


def test_summary_intervals_match_scipy():
    from scipy.stats import chi2

    rng = np.random.default_rng(3)
    E, d = 12, 4
    es = np.zeros((E, 8))
    es[:, 0] = rng.integers(0, 500, E)
    es[0, 0] = 0  # an epoch without a finite NIS
    es[:, 1] = es[:, 0] * rng.uniform(5, 9, E)
    es[:, 3] = rng.integers(1, 500, E)
    es[:, 4] = es[:, 3] * rng.uniform(3, 5, E)
    es[:, 6] = rng.integers(0, 3, E)
    s = summarise_consistency(es, d, alpha=0.1)
    for e in range(E):
        m = es[e, 0]
        if m == 0:
            assert np.isnan(s["anis"][e]) and np.isnan(s["nis_interval"][e]).all()
            continue
        assert s["anis"][e] == es[e, 1] / m
        assert np.allclose(s["nis_interval"][e], [chi2.ppf(0.05, 7 * m) / m, chi2.ppf(0.95, 7 * m) / m], rtol=1e-14)
        mn = es[e, 3]
        assert np.allclose(s["nees_interval"][e], [chi2.ppf(0.05, d * mn) / mn, chi2.ppf(0.95, d * mn) / mn], rtol=1e-14)
    inside = [(s["nis_interval"][e, 0] <= s["anis"][e] <= s["nis_interval"][e, 1]) for e in range(1, E)]
    assert s["nis_inside"] == np.mean(inside)
    assert s["skipped_total"] == es[:, 6].sum()
    s0 = summarise_consistency(es, 0)
    assert np.isnan(s0["anees"]).all() and np.isnan(s0["nees_inside"]) and np.array_equal(s0["anis"], s["anis"], equal_nan=True)


def test_summary_of_two_shards_is_that_of_one():
    """shards add their epoch sums (all-reduce); the summary of the sum is that of the whole job"""
    rng = np.random.default_rng(4)
    nis = rng.chisquare(7, (1000, 9))
    nees = rng.chisquare(6, (1000, 9))
    nis[rng.random(nis.shape) < 0.01] = np.nan

    def sums(a, b):
        fa, fb = np.isfinite(a), np.isfinite(b)
        z = lambda v, f: np.where(f, v, 0.0)
        return np.stack([fa.sum(0), z(a, fa).sum(0), z(a * a, fa).sum(0), fb.sum(0), z(b, fb).sum(0), z(b * b, fb).sum(0),
                         (~fa | ~fb).sum(0), np.zeros(a.shape[1])], axis=1)

    whole = summarise_consistency(sums(nis, nees), 6)
    split = summarise_consistency(sums(nis[:400], nees[:400]) + sums(nis[400:], nees[400:]), 6)
    for key, v in whole.items():
        np.testing.assert_allclose(split[key], v, rtol=1e-12)
    assert 0.5 < whole["nis_inside"] <= 1.0 and 0.5 < whole["nees_inside"] <= 1.0  # chi-square samples are consistent


def test_candidate_objective_with_nans():
    """[m r, E] -> per candidate |ln(mean of the finite values / dim)|, +inf for a candidate without one"""
    m, r, E = 3, 2, 4
    v = np.arange(1.0, 1 + m * r * E).reshape(m * r, E)
    v[0, 1] = np.nan
    v[3, :] = np.inf
    v[4:, :] = np.nan
    got = candidate_objective(v, m, 7)
    c0 = np.delete(v[:2].ravel(), 1)
    c1 = v[2]
    assert got[0] == abs(np.log(c0.mean() / 7)) and got[1] == abs(np.log(c1.mean() / 7)) and got[2] == np.inf
