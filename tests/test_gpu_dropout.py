"""Simulated frame loss (eskf_set_meas_dropout, ``BatchFilter.run(drop_prob=...)``) on the stacked Monte-Carlo workload of
tests/test_gpu_paths.py: four trajectories x 13 filters, all six DOFs estimated, ragged n_prop, noise read back with
eskf_noise_dump.  The drop probability is 0.3 everywhere except one epoch at 1 and one at 0; the mask comes from
``engine.dropout_mask`` and the batch oracle skips exactly those updates.  The canonical cell (pre-pass, F = 28, stacked,
consistency on) is held to the oracle and every other cell, segmentation, shard and group to its bits."""
import ctypes as C

import numpy as np
import pytest

from tests.consistency_oracle import RecordingOracle
from tests.helpers import cov_err, model_kwargs, state_err
from tests.test_gpu_consistency import FLOOR, TOL_NEES, TOL_NIS, _oracle_values
from tests.test_gpu_noise import CAM_STD, IMU_STD, _noisy_streams
from tests.test_gpu_paths import (FPT, GT, K_SPREAD, N_PROP, NAMES, PATHS, SEED, SHAPES, TOL_COV, TOL_STAT, TOL_STATE, Workload,
                                  _assert_bounded, _update_mse)

pytestmark = pytest.mark.gpu

E_ONE, E_ZERO = 2, 4  # the epoch every filter loses, and the one no filter loses


def _prob(E, n_traj=4):
    p = np.full((n_traj, E), 0.3)
    p[:, E_ONE], p[:, E_ZERO] = 1.0, 0.0
    return p


class DropOracle(RecordingOracle):
    """the batch oracle that skips the updates of the rows in ``drop`` (state and covariance stay at the prior)"""

    drop = None

    def update(self, cam_pos, cam_q, notch):
        x, P = self.x.copy(), self.P.copy()
        out = super().update(cam_pos, cam_q, notch)
        self.x[self.drop], self.P[self.drop] = x[self.drop], P[self.drop]
        return out


def _reference(wl, mask):
    """final x / P, statistics rows, nis / nees [n, E] (NaN nis where dropped, the prior's NEES there) and the twin oracle's
    spreads, on the kernels' noise, skipping the masked updates"""
    from dvi_ekf_b200.engine import NOISE_CAM, NOISE_IMU, noise_samples

    n, T, E = wl.n, wl.T, wl.E
    zi = noise_samples(SEED, 0, n, 0, T, NOISE_IMU)
    zc = noise_samples(SEED, 0, n, 0, E, NOISE_CAM)
    r = dict(x=np.empty((n, 26)), P=np.empty((n, 24, 24)), stats=np.zeros((n, 16)), spread=np.empty((n, 2)),
             trace=np.full((n, T, 26), np.nan), last=np.full((n, E), -1),
             nis=np.empty((n, E)), nees=np.empty((n, E)), s_nis=np.zeros((n, E)), s_nees=np.zeros((n, E)))
    for j, sc in enumerate(wl.scs):
        rows = slice(j * FPT, (j + 1) * FPT)
        oa, cam, notch = np.empty((FPT, T, 6)), np.empty((FPT, E, 7)), np.empty((FPT, E))
        for i, g in enumerate(range(j * FPT, (j + 1) * FPT)):
            oa[i], cam[i], notch[i] = (sc.om_acc, sc.cam_meas, sc.notch_meas) if g == 0 else _noisy_streams(sc, zi[g], zc[g])
        bo = DropOracle(sc.cfg, wl.x0[rows], sc.P0, wl.u0[rows], sc.Qd, sc.Rd, sc.sig_om)
        tw = DropOracle(sc.cfg, wl.x0[rows] * (1 + 1e-15), sc.P0, wl.u0[rows], sc.Qd, sc.Rd, sc.sig_om)
        k, mse = 0, []
        for e in range(E):
            for _ in range(N_PROP[j, e]):
                for b in (bo, tw):
                    b.propagate(sc.dt[k], oa[:, k, :3], oa[:, k, 3:])
                r["trace"][rows, k] = bo.x
                k += 1
            vals = []
            for b in (bo, tw):
                b.drop = mask[rows, e]
                b.update(cam[:, e, :3], cam[:, e, 3:], notch[:, e])
                vals.append(_oracle_values(b, GT, (0,) * 6))
            (ni, ne), (ti, te) = vals
            if k > 0:  # the update overwrites the row of the epoch's last step (a dropped one leaves the propagated state)
                r["trace"][rows, k - 1] = bo.x
                r["last"][rows, e] = k - 1
            r["nis"][rows, e] = np.where(mask[rows, e], np.nan, ni)
            r["nees"][rows, e] = ne
            with np.errstate(invalid="ignore"):
                r["s_nis"][rows, e] = np.where(mask[rows, e], 0.0, np.abs(ti / ni - 1))
            r["s_nees"][rows, e] = np.abs(te / ne - 1)
            mse.append(_update_mse(bo.x, wl.cam_ref[j, e], wl.imu_ref[j, e]))
        r["x"][rows], r["P"][rows] = bo.x, bo.P
        d2 = np.square(bo.x[:, 10:16] - GT)
        mse = np.array(mse)
        r["stats"][rows, 0:6] = d2
        r["stats"][rows, 6] = d2.mean(axis=1)
        r["stats"][rows, 7] = mse[-1]
        r["stats"][rows, 8] = mse.sum(axis=0)
        r["stats"][rows, 9] = E - mask[rows].sum(axis=1)
        r["stats"][rows, 11] = 1.0
        r["spread"][rows] = [(state_err(tw.x[i], bo.x[i]), cov_err(tw.P[i], bo.P[i], sc.Rd)) for i in range(FPT)]
    return r


def _run(wl, prob="default", F=28, path="prepass", n_traj=4, lo=0, hi=None, trace=False, jac=False, cons=True, modulus=0,
         segments=None, groups=0, noise_free0=True):
    """one run (or the segments [b0, b1), [b1, b2), ...) of filters lo..hi-1 of the workload with drop_prob = prob; every
    output the run and the getters give"""
    from dvi_ekf_b200 import BatchFilter

    hi = wl.n if hi is None else hi
    n, sc0 = hi - lo, wl.sc0
    if isinstance(prob, str):
        prob = _prob(wl.E, n_traj)
    with BatchFilter(n, **model_kwargs(sc0.cfg)) as bf:
        bf.set_tuning(F)
        if path == "inkernel":
            bf.set_prepass_budget(0)
        bf.set_noise(sc0.Qd[None], sc0.Rd[None], sc0.sig_om[None])
        bf.set_state(wl.x0[lo:hi], sc0.P0[None], wl.u0[lo:hi], None)
        if jac:
            bf.keep_jacobians(True)
        if cons:
            bf.keep_consistency(True)
        if groups:
            bf.set_groups(groups)
        tr = np.full((n, wl.T, 26), np.nan) if trace else None
        kw = dict(**(wl.streams if n_traj > 1 else wl.streams0), n_traj=n_traj, filters_per_traj=FPT if n_traj > 1 else None,
                  seed=SEED, filter_id0=lo, imu_noise_std=IMU_STD, cam_noise_std=CAM_STD, noise_free_filter0=noise_free0,
                  trace=tr, gt_dofs=GT, noise_id_modulus=modulus, drop_prob=prob)
        out = {}
        if segments is None:
            out["stats"], out["sum"] = bf.run(**kw)
            if cons:
                out["nis"], out["nees"], out["esum"] = bf.get_consistency()
                out["dofs"], out["var"] = bf.get_dof_history()
                out["env"] = bf.get_dof_envelope()
            if groups:
                _, out["gstats"], out["gesum"], out["genv"] = bf.get_group_sums(True, cons, cons)
        else:
            parts = {k: [] for k in ("nis", "nees", "esum", "dofs", "var", "env")}
            for e0, e1, st, sm in bf.run_segments(**kw, boundaries=segments):
                out["stats"], out["sum"] = st, sm
                if cons and e1 > e0:
                    for k, v in zip(("nis", "nees", "esum"), bf.get_consistency()):
                        parts[k].append(v)
                    for k, v in zip(("dofs", "var"), bf.get_dof_history()):
                        parts[k].append(v)
                    parts["env"].append(bf.get_dof_envelope())
            if cons:
                for k in ("nis", "nees", "dofs", "var"):
                    out[k] = np.concatenate(parts[k], axis=1)
                for k in ("esum", "env"):
                    out[k] = np.concatenate(parts[k], axis=0)
        out["x"], out["P"], out["u"], out["R"], out["status"] = bf.get_state()
        out["trace"] = tr
        if jac:
            out["jac"] = bf.get_jacobians()
        out["launches"] = bf.launch_count
    return out


def _mask(wl, prob=None, lo=0, n=None, n_traj=4, modulus=0, noise_free0=True):
    from dvi_ekf_b200.engine import dropout_mask

    prob = _prob(wl.E, n_traj) if prob is None else prob
    return dropout_mask(prob, SEED, lo, wl.n - lo if n is None else n, (0, wl.E), n_traj=n_traj,
                        filters_per_traj=FPT if n_traj > 1 else None, noise_id_modulus=modulus, noise_free_filter0=noise_free0)


KEYS = ("x", "P", "u", "R", "status", "stats", "sum", "nis", "nees", "esum", "dofs", "var", "env")


def _same(out, base, rows=slice(None), keys=KEYS, what=""):
    for k in keys:
        if k in ("sum", "esum", "env"):
            assert out[k].tobytes() == base[k].tobytes(), (what, k)
        else:
            assert out[k].tobytes() == base[k][rows].tobytes(), (what, k)


@pytest.fixture(scope="module")
def wl(golden):
    return Workload(golden)


@pytest.fixture(scope="module")
def mask(wl):
    m = _mask(wl)
    assert m[:, E_ONE].all() and not m[:, E_ZERO].any()
    assert 0.15 < m[:, [e for e in range(wl.E) if e not in (E_ONE, E_ZERO)]].mean() < 0.45
    assert not m[0, [e for e in range(wl.E) if e != E_ONE]].any()  # noise-free filter 0: only the p = 1 epoch
    return m


@pytest.fixture(scope="module")
def canon(wl):
    return _run(wl, trace=True, jac=True)


@pytest.fixture(scope="module")
def plain(wl):
    """the same run without dropout"""
    return _run(wl, prob=None, trace=True)


def test_against_the_oracle(wl, mask, canon):
    """state, covariance, statistics rows, NIS and NEES against the batch oracle that skips the masked updates"""
    ref = _reference(wl, mask)
    err = np.zeros((wl.n, 3))
    for f in range(wl.n):
        s, sr = canon["stats"][f], ref["stats"][f]
        err[f] = (state_err(canon["x"][f], ref["x"][f]), cov_err(canon["P"][f], ref["P"][f], wl.sc0.Rd),
                  max(np.abs(s[0:7] - sr[0:7]).max() / np.abs(sr[0:7]).max(), abs(s[7] - sr[7]) / abs(sr[7]),
                      abs(s[8] - sr[8]) / abs(sr[8])))
        assert np.array_equal(s[9:], sr[9:]), (f, s[9:12], sr[9:12])
    # traj_trans_x at the tolerances of the parity tests; the ill-conditioned three at FLOOR + K_SPREAD x the twin's spread
    spread = ref["spread"][:, [0, 1, 0]]
    for j, nm in enumerate(NAMES):
        rows = slice(j * FPT, (j + 1) * FPT)
        print(f"MEASURED dropout vs oracle, state / P / statistics {nm}: worst "
              f"{' / '.join(f'{v:.2e}' for v in err[rows].max(axis=0))}, oracle spread {spread[rows].max():.2e}")
    bound = np.where(np.arange(wl.n)[:, None] < FPT, np.array([TOL_STATE, TOL_COV, TOL_STAT])[None], FLOOR) + K_SPREAD * spread
    assert (err <= bound).all(), np.argwhere(err > bound)[:5]
    for key, tol in (("nis", TOL_NIS), ("nees", TOL_NEES)):
        fin = np.isfinite(ref[key])
        assert np.array_equal(np.isfinite(canon[key]), fin), key
        e = np.where(fin, np.abs(canon[key] / np.where(fin, ref[key], 1.0) - 1), 0.0)
        for j, nm in enumerate(NAMES):
            rows = slice(j * FPT, (j + 1) * FPT)
            print(f"MEASURED dropout {key} {nm}: worst relative {e[rows].max():.2e}, oracle spread {ref['s_' + key][rows].max():.2e}")
        bound = np.where(np.arange(wl.n)[:, None] < FPT, tol, FLOOR + K_SPREAD * ref["s_" + key])
        assert (e <= bound).all(), (key, np.argwhere(e > bound)[:5])


def test_exact_effects_of_the_mask(wl, mask, canon, plain):
    """applied updates, status words, NaN pattern of the NIS, the prior in the records, trace rows, and the dropped counts"""
    E, n = wl.E, wl.n
    assert np.array_equal(canon["stats"][:, 9], E - mask.sum(axis=1))
    assert np.array_equal(canon["status"], plain["status"]) and (canon["status"] == 0).all()
    assert np.array_equal(np.isnan(canon["nis"]), mask | np.isnan(plain["nis"]))
    assert np.isfinite(canon["nees"]).all()
    ref = _reference(wl, mask)
    err = np.zeros((n, 1))
    for f in range(n):
        for e in np.nonzero(mask[f])[0]:
            k = ref["last"][f, e]
            if k < 0:
                continue
            # the trace row of the epoch's last step keeps the propagated state, and the record the prior DOFs
            err[f, 0] = max(err[f, 0], state_err(canon["trace"][f, k], ref["trace"][f, k]))
            if not (ref["last"][f, e + 1:] == k).any():  # (a later epoch of 0 steps writes the same row)
                assert canon["dofs"][f, e].tobytes() == canon["trace"][f, k, 10:16].tobytes(), (f, e)
    _assert_bounded("dropout trace rows at dropped epochs vs the propagated oracle state", err, (TOL_STATE,), ref["spread"][:, 0])
    es, env = canon["esum"], canon["env"]
    assert np.array_equal(es[:, 7], mask.sum(axis=0)) and np.array_equal(env[:, 74], mask.sum(axis=0))
    assert np.array_equal(es[:, 0], (~mask).sum(axis=0)) and np.array_equal(es[:, 3], np.full(E, n))
    assert (es[:, 6] == 0).all()  # a dropped measurement is not a failure
    assert np.array_equal(env[:, 0], np.full(E, n))  # every filter contributes, the dropped ones their prior
    assert (env[:, 75:] == 0).all() and (plain["esum"][:, 7] == 0).all() and (plain["env"][:, 74] == 0).all()
    from dvi_ekf_b200.consistency import summarise_consistency, summarise_dofs

    assert np.array_equal(summarise_consistency(es, 6)["dropped"], mask.sum(axis=0))
    assert np.array_equal(summarise_dofs(env, (0,) * 6)["dropped"], mask.sum(axis=0))


@pytest.mark.parametrize("export", [False, True], ids=["plain", "export"])
@pytest.mark.parametrize("F", SHAPES)
@pytest.mark.parametrize("path", PATHS)
def test_every_cell_is_bit_identical_to_canonical(wl, canon, path, F, export):
    """pre-pass / in-kernel x every CTA shape x trace and Jacobians off / on, stacked and trajectory 0 alone"""
    out = _run(wl, F=F, path=path, trace=export, jac=export)
    _same(out, canon, what=(path, F, export))
    if export:
        assert out["trace"].tobytes() == canon["trace"].tobytes()
    one = _run(wl, F=F, path=path, trace=export, jac=export, n_traj=1, hi=FPT)
    _same(one, canon, rows=slice(0, FPT), keys=("x", "P", "u", "R", "status", "stats", "nis", "nees", "dofs", "var"),
          what=(path, F, export, "single"))


@pytest.mark.parametrize("path", PATHS)
def test_segments_and_checkpoint_restart(wl, canon, path):
    """1, 2, 3 and E segments give the bits of one launch; so does a restart from a checkpoint on a new handle"""
    from dvi_ekf_b200 import BatchFilter

    E = wl.E
    for b in ([0, E], [0, 3, E], [0, 1, 5, E], list(range(E + 1))):
        out = _run(wl, path=path, segments=b)
        _same(out, canon, what=(path, b))
    sc0 = wl.sc0
    kw = dict(**wl.streams, n_traj=4, filters_per_traj=FPT, seed=SEED, imu_noise_std=IMU_STD, cam_noise_std=CAM_STD,
              noise_free_filter0=True, gt_dofs=GT, drop_prob=_prob(E))
    with BatchFilter(wl.n, **model_kwargs(sc0.cfg)) as bf:
        if path == "inkernel":
            bf.set_prepass_budget(0)
        bf.set_noise(sc0.Qd[None], sc0.Rd[None], sc0.sig_om[None])
        bf.set_state(wl.x0, sc0.P0[None], wl.u0, None)
        _, _, carry = bf.run(epochs=(0, 3), **kw)
        x, P, u, R, _ = bf.get_state()
    with BatchFilter(wl.n, **model_kwargs(sc0.cfg)) as bf:
        if path == "inkernel":
            bf.set_prepass_budget(0)
        bf.set_noise(sc0.Qd[None], sc0.Rd[None], sc0.sig_om[None])
        bf.set_state(x.copy(), P.copy(), u.copy(), R.copy())
        st, sm, _ = bf.run(epochs=(3, E), carry=np.array(carry), **kw)
        out = dict(zip(("x", "P", "u", "R", "status"), bf.get_state()), stats=st, sum=sm)
    _same(out, canon, keys=("x", "P", "u", "R", "status", "stats", "sum"), what=(path, "restart"))


def test_shards_and_groups(wl, canon):
    """two shards split at a trajectory boundary give the rows of one handle; grouped sums (one group per trajectory) equal
    the sums of a handle holding only that trajectory"""
    a = _run(wl, hi=2 * FPT)
    b = _run(wl, lo=2 * FPT)
    for k in ("x", "P", "status", "stats", "nis", "nees", "dofs"):
        assert np.concatenate((a[k], b[k])).tobytes() == canon[k].tobytes(), k
    assert np.array_equal(a["esum"][:, [0, 3, 6, 7]] + b["esum"][:, [0, 3, 6, 7]], canon["esum"][:, [0, 3, 6, 7]])
    g = _run(wl, groups=FPT)
    _same(g, canon, keys=("x", "P", "status", "stats", "nis", "nees"), what="groups")
    for j in range(len(NAMES)):
        alone = _run(wl, lo=j * FPT, hi=(j + 1) * FPT)
        assert g["gstats"][j].tobytes() == alone["sum"].tobytes(), j
        assert g["gesum"][j].tobytes() == alone["esum"].tobytes(), j
        assert g["genv"][j].tobytes() == alone["env"].tobytes(), j


def test_p_zero_is_bit_identical_to_no_dropout(wl, plain):
    """dropout set with p = 0 everywhere (the export instantiation): every output as without dropout"""
    out = _run(wl, prob=0.0, trace=True)
    _same(out, plain, what="p = 0")
    assert out["trace"].tobytes() == plain["trace"].tobytes()


def test_p_one_applies_no_update(wl):
    """p = 1 everywhere: no update, row [9] = 0, status 0, x and P of propagation only, nis all NaN, epoch_sum[7] = N"""
    m = np.ones((wl.n, wl.E), bool)
    out = _run(wl, prob=1.0)
    ref = _reference(wl, m)
    assert (out["stats"][:, 9] == 0).all() and (out["status"] == 0).all()
    assert np.isnan(out["nis"]).all() and np.array_equal(out["esum"][:, 7], np.full(wl.E, wl.n))
    err = np.array([(state_err(out["x"][f], ref["x"][f]), cov_err(out["P"][f], ref["P"][f], wl.sc0.Rd)) for f in range(wl.n)])
    _assert_bounded("p = 1 vs propagation-only oracle, state / P", err, (TOL_STATE, TOL_COV), ref["spread"])


def test_noise_id_modulus_shares_and_nests_masks(wl):
    """noise_id_modulus = r: filters with the same noise id share a mask, the masks nest over p, the noise-free filter 0 drops
    only at p = 1; a run with the modulus loses exactly those updates"""
    r = 5
    ms = [_mask(wl, prob=np.full((4, wl.E), p), modulus=r) for p in (0.1, 0.3, 0.5)]
    ids = np.arange(wl.n) % r
    for m in ms:
        for g in range(r):
            assert (m[ids == g] == m[np.argmax(ids == g)]).all()
        assert not m[ids == 0].any()
    for lo_, hi_ in zip(ms, ms[1:]):
        assert not (lo_ & ~hi_).any()
    p = _prob(wl.E)
    m = _mask(wl, prob=p, modulus=r)
    assert m[ids == 0][:, E_ONE].all() and not m[ids == 0][:, [e for e in range(wl.E) if e != E_ONE]].any()
    out = _run(wl, modulus=r)
    assert np.array_equal(out["stats"][:, 9], wl.E - m.sum(axis=1))
    assert np.array_equal(np.isnan(out["nis"]), m)
    # without noise_free_filter0, id 0 draws like the others
    m1 = _mask(wl, prob=p, modulus=r, noise_free0=False)
    assert np.array_equal(_run(wl, modulus=r, noise_free0=False)["stats"][:, 9], wl.E - m1.sum(axis=1))


def test_generator_statistics():
    """10^6 uniforms from the read-back: KS against U(0, 1), lag-1 correlations across epochs and filters, the dropped fraction
    at p = 0.3 inside its binomial 99.9 % interval, and the device bits equal to the host harness"""
    import ctypes
    import os
    import subprocess
    import tempfile

    from scipy.stats import binom, kstest

    from dvi_ekf_b200.engine import NOISE_DROP, dropout_mask, noise_samples

    nf, ne = 1000, 1000
    z = noise_samples(99, 0, nf, 5, ne, NOISE_DROP)
    assert (z[:, :, 1:] == 0).all()
    u = z[:, :, 0]
    assert (u > 0).all() and (u < 1).all()
    ks = kstest(u.ravel(), "uniform")
    c_ep = np.corrcoef(u[:, :-1].ravel(), u[:, 1:].ravel())[0, 1]
    c_f = np.corrcoef(u[:-1].ravel(), u[1:].ravel())[0, 1]
    m = dropout_mask(0.3, 99, 0, nf, (5, 5 + ne), noise_free_filter0=False)
    lo, hi = binom.ppf(0.0005, u.size, 0.3), binom.ppf(0.9995, u.size, 0.3)
    print(f"MEASURED dropout uniforms: KS p = {ks.pvalue:.3f}, lag-1 corr epochs {c_ep:.2e} filters {c_f:.2e}, "
          f"dropped {m.sum()} in [{lo:.0f}, {hi:.0f}]")
    assert ks.pvalue > 1e-3 and abs(c_ep) < 5e-3 and abs(c_f) < 5e-3 and lo <= m.sum() <= hi
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostcheck", "dropout_check.cpp")
    with tempfile.TemporaryDirectory() as d:
        lib_path = os.path.join(d, "libdropoutcheck.so")
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", lib_path, src], check=True)
        lib = ctypes.CDLL(lib_path)
        f64p = ctypes.POINTER(ctypes.c_double)
        lib.hc_drop_uniforms.argtypes = [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_int64, ctypes.c_uint64, ctypes.c_int64, f64p]
        for seed, id0, e0 in ((99, 0, 5), (2 ** 40 + 1, 2 ** 33, 2 ** 32 - 3)):
            host = np.empty((64, 16))
            lib.hc_drop_uniforms(seed, id0, 64, e0, 16, host.ctypes.data_as(f64p))
            assert host.tobytes() == noise_samples(seed, id0, 64, e0, 16, NOISE_DROP)[:, :, 0].copy().tobytes()


def test_error_paths(wl, monkeypatch):
    """a shape that does not match the streams and variant 1: ESKF_EINVAL with nothing launched and the state unchanged; the
    setter refuses bad values (host and device arrays); eskf_propagate / eskf_update ignore the setting"""
    import torch

    from dvi_ekf_b200 import BatchFilter
    from dvi_ekf_b200._lib import EskfError

    sc0 = wl.sc0
    kw = dict(**wl.streams, n_traj=4, filters_per_traj=FPT, seed=SEED, imu_noise_std=IMU_STD, cam_noise_std=CAM_STD, gt_dofs=GT)
    with BatchFilter(wl.n, **model_kwargs(sc0.cfg)) as bf:
        bf.set_noise(sc0.Qd[None], sc0.Rd[None], sc0.sig_om[None])
        bf.set_state(wl.x0, sc0.P0[None], wl.u0, None)
        before = bf.get_state()
        for shape in ((4, wl.E + 1), (1, wl.E), (3, wl.E)):
            bf.set_meas_dropout(np.zeros(shape), *shape)
            n0 = bf.launch_count
            with monkeypatch.context() as mp:
                mp.setattr(bf, "set_meas_dropout", lambda *a, **k: None)
                with pytest.raises(EskfError, match="dropout"):
                    bf.run(**kw)
                with pytest.raises(EskfError, match="dropout"):
                    bf.run(**kw, epochs=(0, 2))
            assert bf.launch_count == n0
            assert all(a.tobytes() == b.tobytes() for a, b in zip(bf.get_state(), before))
        for bad in (np.nan, -0.5, 1.5, np.inf):
            p = np.full((4, wl.E), 0.2)
            p[1, 3] = bad
            with pytest.raises(ValueError):
                bf.set_meas_dropout(p, 4, wl.E)
            with pytest.raises(EskfError, match="probability"):  # the C setter's own check, host and device arrays
                check_raw = bf._lib.eskf_set_meas_dropout
                from dvi_ekf_b200._lib import check

                check(check_raw(bf._h, p.ctypes.data_as(C.c_void_p), 4, wl.E, 0), "eskf_set_meas_dropout")
            t = torch.tensor(p, device="cuda")
            with pytest.raises(EskfError, match="probability"):
                check(check_raw(bf._h, C.c_void_p(t.data_ptr()), 4, wl.E, 1), "eskf_set_meas_dropout")
        # a device array of valid values is taken (and a run with it matches the host array's)
        bf.set_meas_dropout(torch.tensor(_prob(wl.E), device="cuda"), 4, wl.E)
        # eskf_propagate / eskf_update ignore it: the same bits as on a handle without dropout
        bf.set_state(wl.x0[:1].repeat(wl.n, 0), sc0.P0[None], wl.u0[:1].repeat(wl.n, 0), None)
        bf.propagate(sc0.dt[:10], sc0.om_acc[:10])
        bf.update(sc0.cam_meas[0], sc0.notch_meas[0])
        got = bf.get_state()
    with BatchFilter(wl.n, **model_kwargs(sc0.cfg)) as bf:
        bf.set_noise(sc0.Qd[None], sc0.Rd[None], sc0.sig_om[None])
        bf.set_state(wl.x0[:1].repeat(wl.n, 0), sc0.P0[None], wl.u0[:1].repeat(wl.n, 0), None)
        bf.propagate(sc0.dt[:10], sc0.om_acc[:10])
        bf.update(sc0.cam_meas[0], sc0.notch_meas[0])
        assert all(a.tobytes() == b.tobytes() for a, b in zip(bf.get_state(), got))
    with BatchFilter(8, variant=1, **model_kwargs(sc0.cfg)) as bf:
        bf.set_noise(sc0.Qd[None], sc0.Rd[None], sc0.sig_om[None])
        bf.set_state(wl.x0[:8], sc0.P0[None], wl.u0[:8], None)
        n0 = bf.launch_count
        with pytest.raises(EskfError, match="default kernel"):
            bf.run(**wl.streams0, seed=SEED, gt_dofs=GT, drop_prob=0.3)
        assert bf.launch_count == n0
        bf.run(**wl.streams0, seed=SEED, gt_dofs=GT)  # (without dropout variant 1 runs)


def test_device_resident_probabilities_and_streams(wl, canon):
    """drop_prob as a CUDA tensor with device-resident streams: the bits of the canonical cell"""
    import torch

    from dvi_ekf_b200 import BatchFilter

    sc0 = wl.sc0
    dev = lambda a, dt=torch.float64: torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device="cuda")
    s = {k: dev(v, torch.int32 if k == "n_prop" else torch.float64) for k, v in wl.streams.items()}
    with BatchFilter(wl.n, **model_kwargs(sc0.cfg)) as bf:
        bf.set_noise(sc0.Qd[None], sc0.Rd[None], sc0.sig_om[None])
        bf.set_state(wl.x0, sc0.P0[None], wl.u0, None)
        bf.keep_consistency(True)
        st, sm = bf.run(**s, n_traj=4, filters_per_traj=FPT, seed=SEED, imu_noise_std=IMU_STD, cam_noise_std=CAM_STD, gt_dofs=GT,
                        drop_prob=dev(_prob(wl.E)), stats_on_device=True)
        x, P, _, _, status = bf.get_state()
        nis = bf.get_consistency()[0]
    assert st.cpu().numpy().tobytes() == canon["stats"].tobytes() and x.tobytes() == canon["x"].tobytes()
    assert P.tobytes() == canon["P"].tobytes() and nis.tobytes() == canon["nis"].tobytes()


def test_simulator(tmp_path, monkeypatch):
    """batch.cam_dropout 0.2: Simulator.run(consistency=True) sets ``dropped`` in both summaries; 0 passes no drop_prob (the
    launches of a run without frame loss), and cam_dropout= overrides the config"""
    import os

    import yaml

    from dvi_ekf_b200 import engine
    from dvi_ekf_b200.config import Config
    from dvi_ekf_b200.filter import Simulator

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    base = yaml.safe_load(open(os.path.join(root, "config.yaml")))
    base["simulation"]["num_kf_runs"] = 64

    def sim(p):
        d = dict(base, batch=dict(base.get("batch") or {}, cam_dropout=p))
        f = tmp_path / f"c{p}.yaml"
        f.write_text(yaml.safe_dump(d))
        return Simulator(Config(str(f)))

    calls = []
    orig = engine.BatchFilter.run

    def spy(self, *a, **k):
        n0 = self.launch_count
        out = orig(self, *a, **k)
        calls.append((k.get("drop_prob"), self.launch_count - n0))
        return out

    monkeypatch.setattr(engine.BatchFilter, "run", spy)
    s2 = sim(0.2)
    s2.run(consistency=True, verbose=False)
    E = len(s2.streams.n_prop)
    assert calls[-1][0] == 0.2
    dr = s2.consistency["dropped"]
    assert dr.shape == (E,) and np.array_equal(dr, s2.dof_envelope["dropped"])
    assert 0.1 * 63 * E < dr.sum() < 0.3 * 63 * E
    assert s2.stats[0, 9] == E and (s2.stats[1:, 9] < E).any()  # run 0 (noise free) loses no frame
    s0 = sim(0.0)
    s0.run(consistency=True, verbose=False)
    assert calls[-1][0] is None and (s0.consistency["dropped"] == 0).all()
    s0.run(consistency=True, verbose=False, cam_dropout=0.2)
    assert calls[-1][0] == 0.2 and calls[-1][1] == calls[-2][1]  # (the same launches: frame loss only selects the kernel)
    assert np.array_equal(s0.consistency["dropped"], dr)
