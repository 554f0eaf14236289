"""The per-DOF envelope of eskf_get_dof_envelope in numpy (TEST INFRASTRUCTURE): the terms of one record as include/eskf.h
defines them, and their sums per epoch."""
import numpy as np

NDOFSUM, USED = 80, 74
PAIRS = [(i, j) for i in range(6) for j in range(i + 1, 6)]


def dof_terms(nis, eps, B, mask):
    """[n, 74] terms of n records: nis [n], eps [n, 6], B [n, 6, 6], one frozen mask (bit i: DOF i frozen)"""
    nis, eps, B = np.asarray(nis, dtype=float), np.asarray(eps, dtype=float), np.asarray(B, dtype=float)
    n = len(nis)
    est = np.array([not (mask >> i) & 1 for i in range(6)])
    dg = B[:, np.arange(6), np.arange(6)]
    ok = np.isfinite(nis)
    with np.errstate(invalid="ignore"):
        for i in np.flatnonzero(est):
            ok &= np.isfinite(eps[:, i]) & np.isfinite(dg[:, i]) & (dg[:, i] > 0)
    for i, j in PAIRS:
        if est[i] and est[j]:
            ok &= np.isfinite(B[:, i, j]) & np.isfinite(B[:, j, i])
    t = np.zeros((n, USED))
    t[:, 0], t[:, 1] = ok, ~ok
    use = ok[:, None] & est[None, :]
    e = np.where(use, eps, 0.0)
    b = np.where(use, dg, 1.0)
    e2 = e * e
    with np.errstate(invalid="ignore", over="ignore"):
        cols = [e, e2, np.where(use, b, 0.0), np.where(use, e2 / b, 0.0),
                use & (e2 <= b), use & (e2 <= 4.0 * b), use & (e2 <= 9.0 * b)]
    t[:, 2:44] = np.stack(cols, axis=2).reshape(n, 42)
    for p, (i, j) in enumerate(PAIRS):
        uj = use[:, i] & est[j]
        t[:, 44 + p] = np.where(uj, eps[:, i] * eps[:, j], 0.0)
        with np.errstate(invalid="ignore", over="ignore"):
            t[:, 59 + p] = np.where(uj, 0.5 * (B[:, i, j] + B[:, j, i]), 0.0)
    return t


def envelope(nis, dofs, B, gt, mask, absolute=False):
    """dof_sum [E, 80] of nis [N, E], dofs [N, E, 6], B [N, E, 6, 6] against gt (6); ``absolute``: the sums of |term|,
    the scale of the rounding of a sum"""
    nis, dofs, B = np.asarray(nis), np.asarray(dofs), np.asarray(B)
    N, E = nis.shape
    out = np.zeros((E, NDOFSUM))
    for e in range(E):
        t = dof_terms(nis[:, e], dofs[:, e] - np.asarray(gt, dtype=float), B[:, e], mask)
        out[e, :USED] = (np.abs(t) if absolute else t).sum(axis=0)
    return out


COUNTS = [0, 1] + [2 + 7 * i + k for i in range(6) for k in (4, 5, 6)]  # the integer columns: compared exactly


def assert_envelope_close(got, ref, scale, rtol, cols=slice(0, NDOFSUM)):
    """counts exact; every other column within rtol of the sum of the absolute terms (``envelope(..., absolute=True)``)"""
    got, ref, scale = np.asarray(got)[:, cols], np.asarray(ref)[:, cols], np.asarray(scale)[:, cols]
    idx = np.arange(NDOFSUM)[cols]
    cnt = np.isin(idx, COUNTS)
    assert np.array_equal(got[:, cnt], ref[:, cnt]), np.argwhere(got[:, cnt] != ref[:, cnt])[:5]
    err = np.abs(got[:, ~cnt] - ref[:, ~cnt])
    bad = err > rtol * scale[:, ~cnt]
    assert not bad.any(), (np.argwhere(bad)[:5], (err / np.maximum(scale[:, ~cnt], 1e-300)).max())
