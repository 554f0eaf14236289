"""Filter consistency from the per-epoch sums of ``BatchFilter.get_consistency`` (include/eskf.h, eskf_get_consistency).

A filter whose covariance matches the errors it makes has E[NIS] = 7 (the measurement dimension) and E[NEES] = d (the
number of estimated DOFs).  Over M independent Monte-Carlo runs the averages ANIS = sum(NIS) / M and ANEES = sum(NEES) / M
are chi-square distributed with M * 7 (M * d) degrees of freedom, divided by M: the two-sided acceptance interval below is
the usual test of that hypothesis per epoch.
"""
from __future__ import annotations

import numpy as np

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
    - ``n_nis``, ``n_nees`` [E]: the counts; ``skipped`` [E]: filters whose value is NaN at the epoch; ``skipped_total``.
    """
    s = np.asarray(epoch_sum, dtype=float).reshape(-1, 8)
    d = int(dim_dofs)
    if not 0 <= d <= 6:
        raise ValueError("dim_dofs must be 0..6")
    out = {"n_nis": s[:, 0].copy(), "n_nees": s[:, 3].copy(), "skipped": s[:, 6].copy(), "skipped_total": float(s[:, 6].sum())}
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
