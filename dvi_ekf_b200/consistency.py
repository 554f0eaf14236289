"""Filter consistency from the per-epoch sums of ``BatchFilter.get_consistency`` (include/eskf.h, eskf_get_consistency).

A filter whose covariance matches the errors it makes has E[NIS] = 7 (the measurement dimension) and E[NEES] = d (the
number of estimated DOFs).  Over M independent Monte-Carlo runs the averages ANIS = sum(NIS) / M and ANEES = sum(NEES) / M
are chi-square distributed with M * 7 (M * d) degrees of freedom, divided by M: the two-sided acceptance interval below is
the usual test of that hypothesis per epoch.
"""
from __future__ import annotations

import numpy as np

from ._lib import NDOFSUM

NIS_DIM = 7  # measurement dimension (camera position, orientation, notch)


def _interval(count, dim, alpha):
    from scipy.stats import chi2

    lo, hi = np.full(len(count), np.nan), np.full(len(count), np.nan)
    ok = count > 0
    if dim > 0 and ok.any():
        m = count[ok]
        lo[ok] = chi2.ppf(alpha / 2, m * dim) / m
        hi[ok] = chi2.ppf(1 - alpha / 2, m * dim) / m
    return np.stack([lo, hi], axis=1)


def summarise_consistency(epoch_sum, dim_dofs: int, alpha: float = 0.05) -> dict:
    """Summary of ``epoch_sum`` [E, 8] (one handle's, or the all-reduced sum of several shards'), ``dim_dofs`` the number of
    estimated DOFs d.  Returns a dict of numpy arrays / floats:

    - ``anis``, ``anees`` [E]: average NIS / NEES of the finite values of each epoch (NaN where there is none, and for the
      NEES when d = 0);
    - ``nis_interval``, ``nees_interval`` [E, 2]: the (1 - alpha) acceptance interval of that average,
      ``[chi2.ppf(alpha/2, M n), chi2.ppf(1 - alpha/2, M n)] / M`` with M the epoch's count and n = 7 or d;
    - ``nis_inside``, ``nees_inside``: fraction of the epochs with a count whose average lies inside its interval (NaN if
      there is no such epoch);
    - ``n_nis``, ``n_nees`` [E]: the counts; ``skipped`` [E]: filters whose value is NaN at the epoch (a dropped measurement
      is not counted); ``skipped_total``;
    - ``dropped`` [E]: filters whose measurement was dropped (``BatchFilter.run(drop_prob=...)``; 0 without dropout).
    """
    s = np.asarray(epoch_sum, dtype=float).reshape(-1, 8)
    d = int(dim_dofs)
    if not 0 <= d <= 6:
        raise ValueError("dim_dofs must be 0..6")
    out = {"n_nis": s[:, 0].copy(), "n_nees": s[:, 3].copy(), "skipped": s[:, 6].copy(), "skipped_total": float(s[:, 6].sum()),
           "dropped": s[:, 7].copy()}
    for key, cnt, tot, dim in (("nis", s[:, 0], s[:, 1], NIS_DIM), ("nees", s[:, 3], s[:, 4], d)):
        avg = np.full(len(s), np.nan)
        if dim > 0:
            np.divide(tot, cnt, out=avg, where=cnt > 0)
        iv = _interval(cnt, dim, alpha)
        has = (cnt > 0) & (dim > 0)
        inside = (avg >= iv[:, 0]) & (avg <= iv[:, 1])
        out["a" + key] = avg
        out[key + "_interval"] = iv
        out[key + "_inside"] = float(inside[has].mean()) if has.any() else float("nan")
    return out


def candidate_objective(values, n_candidates: int, dim: int):
    """Tuning objective per candidate from a [m * r, E] array of NIS or NEES values (candidate c owns the r consecutive rows
    c r .. c r + r - 1): ``|ln(mean / dim)|`` over every finite value of the candidate's runs and epochs, 0 for a consistent
    filter; ``+inf`` for a candidate without a finite value.  Returns [m]."""
    v = np.asarray(values, dtype=float).reshape(n_candidates, -1)
    fin = np.isfinite(v)
    cnt = fin.sum(axis=1)
    tot = np.where(fin, v, 0.0).sum(axis=1)
    out = np.full(n_candidates, np.inf)
    ok = cnt > 0
    with np.errstate(divide="ignore"):
        out[ok] = np.abs(np.log(tot[ok] / cnt[ok] / dim))
    return out


_PAIRS = [(i, j) for i in range(6) for j in range(i + 1, 6)]  # the pair order of the dof_sum row, (0,1), (0,2), ..., (4,5)


def summarise_dofs(dof_sum, frozen_dofs, alpha: float = 0.05) -> dict:
    """Per-DOF Monte-Carlo envelope from ``dof_sum`` [E, 80] (``BatchFilter.get_dof_envelope`` of one handle, or the
    all-reduced sum of several shards'; layout in include/eskf.h, eskf_get_dof_envelope); ``frozen_dofs`` six flags (the
    config's ``frozen_dofs``).  With M the contributing filters of an epoch, eps = dofs - gt_dofs and B_ii the filter's
    variance of DOF i, returns a dict of numpy arrays (NaN for frozen DOFs and for epochs with M = 0):

    - ``bias`` [E,6] = mean eps; ``rmse`` [E,6] = sqrt(mean eps^2); ``std`` [E,6], the sample std of eps (NaN when M < 2);
    - ``sigma_filter`` [E,6] = sqrt(mean B_ii), the filter's claimed sigma; ``inflation`` [E,6] = rmse / sigma_filter, the
      factor by which that sigma is too small (1 for a consistent filter);
    - ``anees_dof`` [E,6] = mean eps^2 / B_ii, 1 in expectation, and ``anees_interval`` [E,2], its (1 - alpha) chi-square
      acceptance interval ``[chi2.ppf(alpha/2, M), chi2.ppf(1 - alpha/2, M)] / M``;
    - ``coverage`` [E,6,3]: fraction of the filters with |eps| <= k sigma, k = 1, 2, 3; ``coverage_expected`` [3] =
      erf(k / sqrt 2); ``coverage_interval`` [E,3,2], the binomial acceptance interval
      ``[binom.ppf(alpha/2, M, p_k), binom.ppf(1 - alpha/2, M, p_k)] / M``;
    - ``err_second_moment`` [E,6,6] = sum eps eps^T / M (the ensemble's error correlation, bias included) and
      ``filter_cov`` [E,6,6] = sum B / M (the filter's claimed one, symmetrised);
    - ``count`` [E] = M and ``excluded`` [E], the filters left out at the epoch; ``dropped`` [E], the filters whose measurement
      was dropped (they contribute their prior).
    """
    from scipy.special import erf
    from scipy.stats import binom, chi2

    s = np.asarray(dof_sum, dtype=float).reshape(-1, NDOFSUM)
    fr = np.asarray(frozen_dofs, dtype=bool).reshape(6)
    E = len(s)
    m = s[:, 0].copy()
    has = m > 0
    mm = np.where(has, m, 1.0)[:, None]  # (a divisor that is only used where M > 0)
    dof = s[:, 2:44].reshape(E, 6, 7)
    est = np.where(has[:, None] & ~fr[None, :], 1.0, np.nan)  # 1 for an estimated DOF of an epoch with M > 0, else NaN
    s1, s2, sb, sr = dof[:, :, 0], dof[:, :, 1], dof[:, :, 2], dof[:, :, 3]
    bias = s1 / mm * est
    msq = s2 / mm * est
    with np.errstate(invalid="ignore", divide="ignore"):
        var = np.where(m[:, None] >= 2, np.maximum(s2 - s1 * s1 / mm, 0.0) / np.maximum(mm - 1, 1.0), np.nan) * est
    sig = np.sqrt(sb / mm) * est
    out = {"count": m, "excluded": s[:, 1].copy(), "dropped": s[:, 74].copy(), "bias": bias, "rmse": np.sqrt(msq), "std": np.sqrt(var), "sigma_filter": sig}
    with np.errstate(invalid="ignore", divide="ignore"):
        out["inflation"] = out["rmse"] / sig
    out["anees_dof"] = sr / mm * est
    iv = np.full((E, 2), np.nan)
    if has.any():
        iv[has, 0] = chi2.ppf(alpha / 2, m[has]) / m[has]
        iv[has, 1] = chi2.ppf(1 - alpha / 2, m[has]) / m[has]
    out["anees_interval"] = iv
    k = np.arange(1, 4)
    p = erf(k / np.sqrt(2.0))
    out["coverage"] = dof[:, :, 4:7] / mm[:, :, None] * est[:, :, None]
    out["coverage_expected"] = p
    civ = np.full((E, 3, 2), np.nan)
    if has.any():
        mh = m[has][:, None]
        civ[has, :, 0] = binom.ppf(alpha / 2, mh, p[None]) / mh
        civ[has, :, 1] = binom.ppf(1 - alpha / 2, mh, p[None]) / mh
    out["coverage_interval"] = civ
    mask2 = est[:, :, None] * est[:, None, :]
    for key, diag, off in (("err_second_moment", s2, s[:, 44:59]), ("filter_cov", sb, s[:, 59:74])):
        a = np.zeros((E, 6, 6))
        a[:, np.arange(6), np.arange(6)] = diag
        for c, (i, j) in enumerate(_PAIRS):
            a[:, i, j] = a[:, j, i] = off[:, c]
        out[key] = a / mm[:, :, None] * mask2
    return out
