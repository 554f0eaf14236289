"""The innovation gate (eskf_set_innovation_gate, ``BatchFilter.run(nis_gate=...)``) and simulated outlier frames
(eskf_set_meas_outliers, ``run(outlier_prob=..., outlier_std=...)``) on the stacked Monte-Carlo workload of
tests/test_gpu_paths.py: four trajectories x 13 filters, all six DOFs estimated, ragged n_prop, noise read back with
eskf_noise_dump.  The outlier probability is 0.3 everywhere except one epoch at 1 and one at 0; the mask and the offsets come
from ``engine.outlier_mask``.  The runs are held to the batch oracle fed the corrupted measurements (and gated by its own NIS),
and every kernel cell, segmentation, shard and group to the bits of the canonical cell (pre-pass, F = 28, stacked,
consistency on)."""
import ctypes as C

import numpy as np
import pytest

from oracle.eskf_oracle import quat_about_axis, quat_mul
from tests.consistency_oracle import RecordingOracle
from tests.helpers import cov_err, model_kwargs, state_err
from tests.test_gpu_consistency import FLOOR, TOL_NEES, TOL_NIS, _oracle_values
from tests.test_gpu_dropout import E_ONE, E_ZERO, _prob, _same
from tests.test_gpu_noise import CAM_STD, IMU_STD, _noisy_streams
from tests.test_gpu_paths import (FPT, GT, K_SPREAD, N_PROP, NAMES, PATHS, SEED, SHAPES, TOL_COV, TOL_STAT, TOL_STATE, Workload,
                                  _update_mse)

pytestmark = pytest.mark.gpu

OUT_STD = np.array([2.0, 2.0, 2.0, 0.1, 0.1, 0.1, 0.2])  # cm, rad, rad: gross errors, twenty camera noise sigmas
# Without a gate, twenty-sigma errors drive the ill-conditioned trajectories into numerical divergence: the oracle's own
# twin then differs from it by 1e12 in P, beyond what any parity bound can speak for.  The ungated comparison with the
# oracle uses errors of five camera sigmas, which keep every filter in the regime the parity protocol covers; the gated
# runs keep the twenty-sigma errors, which the gate rejects.
MILD_STD = OUT_STD / 4


class GateOracle(RecordingOracle):
    """the batch oracle with the gate: rows whose NIS exceeds ``thr`` keep the prior (``rej`` records them)"""

    thr = None
    rej = None

    def update(self, cam_pos, cam_q, notch):
        x, P = self.x.copy(), self.P.copy()
        out = super().update(cam_pos, cam_q, notch)
        nis = np.einsum("ni,ni->n", self.res, np.linalg.solve(self.S, self.res[..., None])[..., 0])
        self.rej = np.zeros(len(nis), bool) if self.thr is None else nis > self.thr
        self.x[self.rej], self.P[self.rej] = x[self.rej], P[self.rej]
        return out


def _corrupt(cam, notch, z, std=OUT_STD):
    """cam_offset (eskf_math.cuh) in numpy: the outlier offset of one measurement, std * z"""
    cam, notch = cam.copy(), float(notch)
    cam[:3] += std[:3] * z[:3]
    dth = std[3:6] * z[3:6]
    dq = quat_about_axis(np.linalg.norm(dth), dth)
    nq = np.linalg.norm(cam[3:])
    cam[3:] = quat_mul(cam[3:], dq) * nq
    return cam, notch + std[6] * z[6]


def _omask(wl, prob=None, modulus=0, noise_free0=True):
    from dvi_ekf_b200.engine import outlier_mask

    prob = _prob(wl.E) if prob is None else prob
    return outlier_mask(prob, SEED, 0, wl.n, (0, wl.E), n_traj=4, filters_per_traj=FPT, noise_id_modulus=modulus,
                        noise_free_filter0=noise_free0)


def _reference(wl, omask, off, thr=None, std=OUT_STD):
    """final x / P, statistics rows, nis / nees [n, E], the rejection mask and the twin oracles' spreads, on the kernels'
    noise with the masked measurements offset by std * off and, with ``thr`` [n], the gate.

    The device and numpy evaluate the offset's rotation with different sines and cosines, so the corrupted measurements
    the two filters see differ in their last bits.  On the ill-conditioned trajectories a gross error makes the filter far
    more sensitive to that difference than to one in its initial state, so the spread is the larger of two twins': one
    started from x0 (1 + 1e-15), one fed the corrupted measurements (1 + 1e-15)."""
    from dvi_ekf_b200.engine import NOISE_CAM, NOISE_IMU, noise_samples

    n, T, E = wl.n, wl.T, wl.E
    zi = noise_samples(SEED, 0, n, 0, T, NOISE_IMU)
    zc = noise_samples(SEED, 0, n, 0, E, NOISE_CAM)
    r = dict(x=np.empty((n, 26)), P=np.empty((n, 24, 24)), stats=np.zeros((n, 16)), spread=np.empty((n, 2)),
             nis=np.empty((n, E)), nees=np.empty((n, E)), s_nis=np.zeros((n, E)), s_nees=np.zeros((n, E)),
             rej=np.zeros((n, E), bool), margin=np.full((n, E), np.inf))
    for j, sc in enumerate(wl.scs):
        rows = slice(j * FPT, (j + 1) * FPT)
        oa, cam, notch = np.empty((FPT, T, 6)), np.empty((FPT, E, 7)), np.empty((FPT, E))
        for i, g in enumerate(range(j * FPT, (j + 1) * FPT)):
            oa[i], cam[i], notch[i] = (sc.om_acc, sc.cam_meas, sc.notch_meas) if g == 0 else _noisy_streams(sc, zi[g], zc[g])
            for e in np.nonzero(omask[g])[0]:
                cam[i, e], notch[i, e] = _corrupt(cam[i, e], notch[i, e], off[g, e], std)
        cam_m, notch_m = cam.copy(), notch.copy()  # (the measurement twin's input: the corrupted measurements perturbed)
        m = omask[rows]
        cam_m[m] *= 1 + 1e-15
        notch_m[m] *= 1 + 1e-15
        bo = GateOracle(sc.cfg, wl.x0[rows], sc.P0, wl.u0[rows], sc.Qd, sc.Rd, sc.sig_om)
        tw = GateOracle(sc.cfg, wl.x0[rows] * (1 + 1e-15), sc.P0, wl.u0[rows], sc.Qd, sc.Rd, sc.sig_om)
        tm = GateOracle(sc.cfg, wl.x0[rows], sc.P0, wl.u0[rows], sc.Qd, sc.Rd, sc.sig_om)
        for b in (bo, tw, tm):
            b.thr = None if thr is None else thr[rows]
        k, mse = 0, []
        for e in range(E):
            for _ in range(N_PROP[j, e]):
                for b in (bo, tw, tm):
                    b.propagate(sc.dt[k], oa[:, k, :3], oa[:, k, 3:])
                k += 1
            vals = []
            for b, c, nt in ((bo, cam, notch), (tw, cam, notch), (tm, cam_m, notch_m)):
                b.update(c[:, e, :3], c[:, e, 3:], nt[:, e])
                vals.append(_oracle_values(b, GT, (0,) * 6))
            (ni, ne), (ti, te), (mi, me) = vals
            r["nis"][rows, e], r["nees"][rows, e], r["rej"][rows, e] = ni, ne, bo.rej
            r["s_nis"][rows, e] = np.maximum(np.abs(ti / ni - 1), np.abs(mi / ni - 1))
            r["s_nees"][rows, e] = np.maximum(np.abs(te / ne - 1), np.abs(me / ne - 1))
            if thr is not None:
                r["margin"][rows, e] = np.abs(ni / thr[rows] - 1)
            mse.append(_update_mse(bo.x, wl.cam_ref[j, e], wl.imu_ref[j, e]))
        r["x"][rows], r["P"][rows] = bo.x, bo.P
        d2 = np.square(bo.x[:, 10:16] - GT)
        mse = np.array(mse)
        r["stats"][rows, 0:6] = d2
        r["stats"][rows, 6] = d2.mean(axis=1)
        r["stats"][rows, 7] = mse[-1]
        r["stats"][rows, 8] = mse.sum(axis=0)
        r["stats"][rows, 9] = E - r["rej"][rows].sum(axis=1)
        r["stats"][rows, 11] = 1.0
        r["spread"][rows] = [(max(state_err(t.x[i], bo.x[i]) for t in (tw, tm)), max(cov_err(t.P[i], bo.P[i], sc.Rd) for t in (tw, tm)))
                             for i in range(FPT)]
    return r


def _bound(wl, ref, key, tol):
    """the tolerance of the NIS or NEES of every (filter, epoch): ``tol`` on traj_trans_x, FLOOR on the ill-conditioned
    three, plus K_SPREAD x the twins' spread -- the form of the state bound.  (Gross errors make even traj_trans_x sensitive:
    its twins' states differ by 6e-9 in the gated run, so its NIS cannot be held to a bound without the spread.)"""
    return np.where(np.arange(wl.n)[:, None] < FPT, tol, FLOOR) + K_SPREAD * ref["s_" + key]


def _run(wl, thr=None, prob="default", std=OUT_STD, F=28, path="prepass", n_traj=4, lo=0, hi=None, trace=False, jac=False,
         cons=True, modulus=0, segments=None, groups=0, drop=None):
    """one run (or its segments) of filters lo..hi-1 with nis_gate = thr[lo:hi] (thr [n] or a scalar) and outlier_prob = prob;
    every output the run and the getters give"""
    from dvi_ekf_b200 import BatchFilter

    hi = wl.n if hi is None else hi
    n, sc0 = hi - lo, wl.sc0
    if isinstance(prob, str):
        prob = _prob(wl.E, n_traj)
    if thr is not None and np.ndim(thr):
        thr = np.asarray(thr)[lo:hi]
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
                  seed=SEED, filter_id0=lo, imu_noise_std=IMU_STD, cam_noise_std=CAM_STD, noise_free_filter0=True,
                  trace=tr, gt_dofs=GT, noise_id_modulus=modulus, drop_prob=drop, nis_gate=thr, outlier_prob=prob,
                  outlier_std=std if prob is not None else None)
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
                if e1 > e0:
                    for k, v in zip(("nis", "nees", "esum"), bf.get_consistency()):
                        parts[k].append(v)
                    for k, v in zip(("dofs", "var"), bf.get_dof_history()):
                        parts[k].append(v)
                    parts["env"].append(bf.get_dof_envelope())
            for k in ("nis", "nees", "dofs", "var"):
                out[k] = np.concatenate(parts[k], axis=1)
            for k in ("esum", "env"):
                out[k] = np.concatenate(parts[k], axis=0)
        out["x"], out["P"], out["u"], out["R"], out["status"] = bf.get_state()
        out["trace"] = tr
        if jac:
            out["jac"] = bf.get_jacobians()
    return out


@pytest.fixture(scope="module")
def wl(golden):
    return Workload(golden)


@pytest.fixture(scope="module")
def omask(wl):
    m, off = _omask(wl)
    assert m[1:, E_ONE].all() and not m[:, E_ZERO].any() and not m[0].any()  # (filter 0: noise free, never corrupted)
    assert 0.15 < m[:, [e for e in range(wl.E) if e not in (E_ONE, E_ZERO)]].mean() < 0.45
    return m, off


@pytest.fixture(scope="module")
def ungated(wl, omask):
    return _reference(wl, *omask)


@pytest.fixture(scope="module")
def gate(wl, omask, ungated):
    """per-filter thresholds (a base scaled by 1, 1.01, 1.02 by filter) with some updates rejected, none all, and every
    oracle NIS of the gated run farther from its threshold than the NIS tolerance: (thr [n], gated reference)"""
    fin = ungated["nis"][np.isfinite(ungated["nis"])]
    for q in (0.7, 0.75, 0.8, 0.65, 0.85, 0.6, 0.9):
        thr = np.quantile(fin, q) * (1 + 0.01 * (np.arange(wl.n) % 3))
        ref = _reference(wl, *omask, thr=thr)
        if 0 < ref["rej"].sum() < wl.n * wl.E // 2 and (ref["margin"] > _bound(wl, ref, "nis", TOL_NIS)).all():
            print(f"MEASURED gate threshold: quantile {q} of the outlier run's NIS, base {thr[0]:.4g}, "
                  f"{int(ref['rej'].sum())} of {wl.n * wl.E} updates rejected, smallest margin {ref['margin'].min():.2e}")
            return thr, ref
    pytest.fail("no threshold candidate keeps every oracle NIS off its knife edge")


@pytest.fixture(scope="module")
def canon(wl, gate):
    return _run(wl, thr=gate[0], trace=True, jac=True)


def _check_against(wl, out, ref, what):
    err = np.zeros((wl.n, 3))
    for f in range(wl.n):
        s, sr = out["stats"][f], ref["stats"][f]
        err[f] = (state_err(out["x"][f], ref["x"][f]), cov_err(out["P"][f], ref["P"][f], wl.sc0.Rd),
                  max(np.abs(s[0:7] - sr[0:7]).max() / np.abs(sr[0:7]).max(), abs(s[7] - sr[7]) / abs(sr[7]),
                      abs(s[8] - sr[8]) / abs(sr[8])))
        assert np.array_equal(s[9:], sr[9:]), (what, f, s[9:12], sr[9:12])
    spread = ref["spread"][:, [0, 1, 0]]
    for j, nm in enumerate(NAMES):
        rows = slice(j * FPT, (j + 1) * FPT)
        print(f"MEASURED {what} vs oracle, state / P / statistics {nm}: worst "
              f"{' / '.join(f'{v:.2e}' for v in err[rows].max(axis=0))}, oracle spread {spread[rows].max():.2e}")
    bound = np.where(np.arange(wl.n)[:, None] < FPT, np.array([TOL_STATE, TOL_COV, TOL_STAT])[None], FLOOR) + K_SPREAD * spread
    assert (err <= bound).all(), (what, np.argwhere(err > bound)[:5])
    for key, tol in (("nis", TOL_NIS), ("nees", TOL_NEES)):
        fin = np.isfinite(ref[key])
        assert np.array_equal(np.isfinite(out[key]), fin), (what, key)
        e = np.where(fin, np.abs(out[key] / np.where(fin, ref[key], 1.0) - 1), 0.0)
        bound = _bound(wl, ref, key, tol)
        print(f"MEASURED {what} {key}: worst relative {e.max():.2e}")
        assert (e <= bound).all(), (what, key, np.argwhere(e > bound)[:5])


def test_outliers_against_the_oracle(wl, omask):
    """outliers only (five camera sigmas): the batch oracle fed the measurements the read-back corrupts"""
    out = _run(wl, std=MILD_STD)
    assert (out["status"] == 0).all()
    _check_against(wl, out, _reference(wl, *omask, std=MILD_STD), "outliers")
    # until a filter's first outlier its run is that of the run without outliers, bit for bit; at it, the gross error
    # shows in the NIS
    plain = _run(wl, prob=None)
    m = omask[0]
    first = np.where(m.any(axis=1), np.argmax(m, axis=1), wl.E)
    for f in range(wl.n):
        assert out["nis"][f, :first[f]].tobytes() == plain["nis"][f, :first[f]].tobytes(), f
    hit = np.nonzero(m.any(axis=1))[0]
    assert (out["nis"][hit, first[hit]] > plain["nis"][hit, first[hit]]).mean() > 0.9


def test_gate_against_the_oracle(wl, gate, canon):
    """gate and outliers: the gated oracle; the rejection masks are equal, and the trace keeps the propagated state"""
    thr, ref = gate
    _check_against(wl, canon, ref, "gate + outliers")
    rej = canon["nis"] > thr[:, None]
    assert np.array_equal(rej, ref["rej"])
    assert (canon["status"] == 0).all() and np.isfinite(canon["nis"]).all()
    assert np.array_equal(canon["stats"][:, 9], wl.E - rej.sum(axis=1))


def test_counts_identity_and_getters_answer_from_the_run(wl, gate, canon):
    """dof_sum[75] = count of nis > thr per epoch; rejected = epochs - dropped - row [9] for every healthy filter; epoch_sum
    counts the rejected NIS and prior NEES; a set_innovation_gate after the run changes no getter output"""
    from dvi_ekf_b200 import BatchFilter
    from dvi_ekf_b200.consistency import summarise_dofs

    thr = gate[0]
    rej = canon["nis"] > thr[:, None]
    env, es = canon["env"], canon["esum"]
    assert np.array_equal(env[:, 75], rej.sum(axis=0)) and rej.sum() > 0
    assert (env[:, 76:] == 0).all() and (env[:, 74] == 0).all()
    assert np.array_equal(summarise_dofs(env, (0,) * 6)["rejected"], rej.sum(axis=0))
    assert np.array_equal(es[:, 0], np.full(wl.E, wl.n)) and np.array_equal(es[:, 3], np.full(wl.E, wl.n))
    assert (es[:, 6] == 0).all() and (es[:, 7] == 0).all()
    assert np.array_equal(env[:, 0], np.full(wl.E, wl.n))
    healthy = canon["status"] == 0
    assert np.array_equal(rej.sum(axis=1)[healthy], (wl.E - canon["stats"][:, 9])[healthy])
    # with dropout as well: rejected = E - dropped - row [9]
    from dvi_ekf_b200.engine import dropout_mask

    dp = np.full((4, wl.E), 0.2)
    dm = dropout_mask(dp, SEED, 0, wl.n, (0, wl.E), n_traj=4, filters_per_traj=FPT)
    both = _run(wl, thr=thr, drop=dp)
    rj = both["nis"] > thr[:, None]
    assert not (rj & dm).any() and np.array_equal(both["env"][:, 74], dm.sum(axis=0))
    assert np.array_equal(both["env"][:, 75], rj.sum(axis=0))
    h = both["status"] == 0
    assert np.array_equal(rj.sum(axis=1)[h], (wl.E - dm.sum(axis=1) - both["stats"][:, 9])[h])
    # getters after a later set_innovation_gate
    sc0 = wl.sc0
    with BatchFilter(wl.n, **model_kwargs(sc0.cfg)) as bf:
        bf.set_noise(sc0.Qd[None], sc0.Rd[None], sc0.sig_om[None])
        bf.set_state(wl.x0, sc0.P0[None], wl.u0, None)
        bf.keep_consistency(True)
        bf.set_groups(FPT)
        bf.run(**wl.streams, n_traj=4, filters_per_traj=FPT, seed=SEED, imu_noise_std=IMU_STD, cam_noise_std=CAM_STD, gt_dofs=GT,
               nis_gate=thr, outlier_prob=_prob(wl.E), outlier_std=OUT_STD)
        before = [bf.get_dof_envelope(), *bf.get_consistency(), *bf.get_group_sums(False, True, True)[1:]]
        for later in (0.0, np.inf, None):
            bf.set_innovation_gate(later)
            after = [bf.get_dof_envelope(), *bf.get_consistency(), *bf.get_group_sums(False, True, True)[1:]]
            for a, b in zip(after, before):
                assert (a is None and b is None) or a.tobytes() == b.tobytes(), later
    assert before[0].tobytes() == canon["env"].tobytes()


@pytest.mark.parametrize("export", [False, True], ids=["plain", "export"])
@pytest.mark.parametrize("F", SHAPES)
@pytest.mark.parametrize("path", PATHS)
def test_every_cell_is_bit_identical_to_canonical(wl, gate, canon, path, F, export):
    """pre-pass / in-kernel x every CTA shape x trace and Jacobians off / on, stacked and trajectory 0 alone"""
    thr = gate[0]
    out = _run(wl, thr=thr, F=F, path=path, trace=export, jac=export)
    _same(out, canon, what=(path, F, export))
    if export:
        assert out["trace"].tobytes() == canon["trace"].tobytes()
    one = _run(wl, thr=thr, F=F, path=path, trace=export, jac=export, n_traj=1, hi=FPT)
    _same(one, canon, rows=slice(0, FPT), keys=("x", "P", "u", "R", "status", "stats", "nis", "nees", "dofs", "var"),
          what=(path, F, export, "single"))


@pytest.mark.parametrize("path", PATHS)
def test_segments_and_checkpoint_restart(wl, gate, canon, path):
    """1, 2, 3 and E segments give the bits of one launch; so does a restart from a checkpoint on a new handle, which sets
    the gate and the outliers again"""
    from dvi_ekf_b200 import BatchFilter

    thr, E = gate[0], wl.E
    for b in ([0, E], [0, 3, E], [0, 1, 5, E], list(range(E + 1))):
        _same(_run(wl, thr=thr, path=path, segments=b), canon, what=(path, b))
    sc0 = wl.sc0
    kw = dict(**wl.streams, n_traj=4, filters_per_traj=FPT, seed=SEED, imu_noise_std=IMU_STD, cam_noise_std=CAM_STD,
              noise_free_filter0=True, gt_dofs=GT, nis_gate=thr, outlier_prob=_prob(E), outlier_std=OUT_STD)
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


def test_shards_and_groups(wl, gate, canon):
    """two shards split at a trajectory boundary, each with its threshold slice, give the rows of one handle; grouped sums
    (one group per trajectory), dof_sum[75] included, equal the sums of a handle holding only that trajectory"""
    thr = gate[0]
    a = _run(wl, thr=thr, hi=2 * FPT)
    b = _run(wl, thr=thr, lo=2 * FPT)
    for k in ("x", "P", "status", "stats", "nis", "nees", "dofs"):
        assert np.concatenate((a[k], b[k])).tobytes() == canon[k].tobytes(), k
    assert np.array_equal(a["env"][:, 75] + b["env"][:, 75], canon["env"][:, 75])
    assert np.array_equal(a["esum"][:, [0, 3, 6, 7]] + b["esum"][:, [0, 3, 6, 7]], canon["esum"][:, [0, 3, 6, 7]])
    g = _run(wl, thr=thr, groups=FPT)
    _same(g, canon, keys=("x", "P", "status", "stats", "nis", "nees"), what="groups")
    rej = canon["nis"] > thr[:, None]
    for j in range(len(NAMES)):
        alone = _run(wl, thr=thr, lo=j * FPT, hi=(j + 1) * FPT)
        assert g["gstats"][j].tobytes() == alone["sum"].tobytes(), j
        assert g["gesum"][j].tobytes() == alone["esum"].tobytes(), j
        assert g["genv"][j].tobytes() == alone["env"].tobytes(), j
        assert np.array_equal(g["genv"][j][:, 75], rej[j * FPT:(j + 1) * FPT].sum(axis=0)), j


def test_settings_that_switch_the_feature_off(wl):
    """gate +inf everywhere and p = 0: the bits of the same export run without either; threshold 0: the x, P and nees of
    dropout p = 1, with row [9] = 0, no status bit and a finite nis"""
    base = _run(wl, prob=None, trace=True)
    off = _run(wl, thr=np.inf, prob=0.0, trace=True)
    _same(off, base, what="gate +inf, p = 0")
    assert off["trace"].tobytes() == base["trace"].tobytes()
    zero = _run(wl, thr=0.0, prob=None)
    p1 = _run(wl, prob=None, drop=1.0)
    for k in ("x", "P", "nees", "dofs", "var"):
        assert zero[k].tobytes() == p1[k].tobytes(), k
    assert (zero["stats"][:, 9] == 0).all() and (zero["status"] == 0).all() and np.isfinite(zero["nis"]).all()
    assert np.array_equal(zero["env"][:, 75], np.full(wl.E, wl.n)) and np.array_equal(zero["env"][:, 1:74], p1["env"][:, 1:74])


def test_generator_statistics_and_shared_draws(wl):
    """the read-back: u uniform on (0, 1), the offsets standard normal, the device uniform equal to the host harness's bits;
    noise_id_modulus shares masks and offsets, and a run with it corrupts exactly those measurements"""
    import os
    import subprocess
    import tempfile

    from scipy.stats import kstest

    from dvi_ekf_b200.engine import NOISE_OUTLIER, noise_samples

    z = noise_samples(99, 0, 1000, 5, 1000, NOISE_OUTLIER)
    u, off = z[:, :, 0], z[:, :, 1:]
    assert (u > 0).all() and (u < 1).all()
    ks_u, ks_z = kstest(u.ravel(), "uniform"), kstest(off.ravel()[::7], "norm")
    c_uz = np.corrcoef(u.ravel(), off[:, :, 0].ravel())[0, 1]
    print(f"MEASURED outlier draws: KS u p = {ks_u.pvalue:.3f}, KS offsets p = {ks_z.pvalue:.3f}, mean {off.mean():.2e}, "
          f"std {off.std():.4f}, corr(u, z0) {c_uz:.2e}")
    assert ks_u.pvalue > 1e-3 and ks_z.pvalue > 1e-3 and abs(off.mean()) < 5e-3 and abs(off.std() - 1) < 5e-3 and abs(c_uz) < 5e-3
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostcheck", "outlier_check.cpp")
    with tempfile.TemporaryDirectory() as d:
        lib_path = os.path.join(d, "liboutliercheck.so")
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", lib_path, src], check=True)
        lib = C.CDLL(lib_path)
        f64p = C.POINTER(C.c_double)
        lib.hc_outlier_uniforms.argtypes = [C.c_uint64, C.c_uint64, C.c_int64, C.c_uint64, C.c_int64, f64p]
        for seed, id0, e0 in ((99, 0, 5), (2 ** 40 + 1, 2 ** 33, 2 ** 32 - 3)):
            host = np.empty((64, 16))
            lib.hc_outlier_uniforms(seed, id0, 64, e0, 16, host.ctypes.data_as(f64p))
            assert host.tobytes() == noise_samples(seed, id0, 64, e0, 16, NOISE_OUTLIER)[:, :, 0].copy().tobytes()
    r = 5
    ids = np.arange(wl.n) % r
    ms = [_omask(wl, prob=np.full((4, wl.E), p), modulus=r) for p in (0.1, 0.3, 0.5)]
    for m, o in ms:
        for g in range(r):
            assert (m[ids == g] == m[np.argmax(ids == g)]).all()
            assert (o[ids == g] == o[np.argmax(ids == g)]).all()
        assert not m[ids == 0].any()
    for (lo_, _), (hi_, _) in zip(ms, ms[1:]):
        assert not (lo_ & ~hi_).any()
    assert all(o.tobytes() == ms[0][1].tobytes() for _, o in ms)
    shared = _run(wl, modulus=r)
    plain = _run(wl, prob=None, modulus=r)
    m = _omask(wl, modulus=r)[0]
    first = np.argmax(m, axis=1)  # (before a filter's first outlier nothing differs)
    for f in range(wl.n):
        e = first[f] if m[f].any() else wl.E
        assert shared["nis"][f, :e].tobytes() == plain["nis"][f, :e].tobytes(), f
        if m[f].any():
            assert shared["nis"][f, e] != plain["nis"][f, e], f


def test_error_paths(wl):
    """a table whose shape differs from the streams' and variant 1: ESKF_EINVAL with nothing launched and the state
    unchanged; the C setters refuse bad values (host and device arrays); eskf_propagate / eskf_update ignore the settings"""
    import torch

    from dvi_ekf_b200 import BatchFilter
    from dvi_ekf_b200._lib import EskfError, check

    sc0 = wl.sc0
    kw = dict(**wl.streams, n_traj=4, filters_per_traj=FPT, seed=SEED, imu_noise_std=IMU_STD, cam_noise_std=CAM_STD, gt_dofs=GT)
    sd = OUT_STD.ctypes.data_as(C.c_void_p)
    with BatchFilter(wl.n, **model_kwargs(sc0.cfg)) as bf:
        bf.set_noise(sc0.Qd[None], sc0.Rd[None], sc0.sig_om[None])
        bf.set_state(wl.x0, sc0.P0[None], wl.u0, None)
        before = bf.get_state()
        raw = bf._lib.eskf_set_meas_outliers
        for shape in ((4, wl.E + 1), (1, wl.E), (3, wl.E)):
            p = np.zeros(shape)
            check(raw(bf._h, p.ctypes.data_as(C.c_void_p), shape[0], shape[1], sd, 0), "eskf_set_meas_outliers")
            n0 = bf.launch_count
            for seg in (None, (0, 2)):
                with pytest.raises(EskfError, match="outlier"):
                    _raw_run(bf, kw, seg)
            assert bf.launch_count == n0
            assert all(a.tobytes() == b.tobytes() for a, b in zip(bf.get_state(), before))
        check(raw(bf._h, None, 0, 0, None, 0), "eskf_set_meas_outliers")
        p = np.full((4, wl.E), 0.2)
        for bad_p, bad_s, match in ((np.nan, OUT_STD, "probability"), (1.5, OUT_STD, "probability"),
                                    (0.2, np.r_[OUT_STD[:6], np.nan], "std"), (0.2, np.r_[-1.0, OUT_STD[1:]], "std"),
                                    (0.2, np.r_[OUT_STD[:6], np.inf], "std")):
            q = p.copy()
            q[1, 3] = bad_p
            s_ = np.ascontiguousarray(bad_s, dtype=np.float64)
            with pytest.raises(EskfError, match=match):
                check(raw(bf._h, q.ctypes.data_as(C.c_void_p), 4, wl.E, s_.ctypes.data_as(C.c_void_p), 0), "eskf_set_meas_outliers")
            t = torch.tensor(q, device="cuda")
            with pytest.raises(EskfError, match=match):
                check(raw(bf._h, C.c_void_p(t.data_ptr()), 4, wl.E, s_.ctypes.data_as(C.c_void_p), 1), "eskf_set_meas_outliers")
        g = bf._lib.eskf_set_innovation_gate
        for bad in (np.array([np.nan]), np.array([-1.0]), np.r_[np.ones(wl.n - 1), np.nan]):
            with pytest.raises(EskfError, match="threshold"):
                check(g(bf._h, bad.ctypes.data_as(C.c_void_p), len(bad), 0), "eskf_set_innovation_gate")
            t = torch.tensor(bad, device="cuda")
            with pytest.raises(EskfError, match="threshold"):
                check(g(bf._h, C.c_void_p(t.data_ptr()), len(bad), 1), "eskf_set_innovation_gate")
        with pytest.raises(EskfError, match="n must be 1 or n_filters"):
            check(g(bf._h, np.ones(3).ctypes.data_as(C.c_void_p), 3, 0), "eskf_set_innovation_gate")
        with pytest.raises(ValueError):
            bf.set_innovation_gate(np.r_[np.ones(wl.n - 1), -1.0])
        # device thresholds are taken; eskf_propagate / eskf_update ignore both settings
        bf.set_innovation_gate(torch.zeros(wl.n, dtype=torch.float64, device="cuda"))
        bf.set_meas_outliers(torch.ones((4, wl.E), dtype=torch.float64, device="cuda"), OUT_STD, 4, wl.E)
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
            bf.run(**wl.streams0, seed=SEED, gt_dofs=GT, nis_gate=10.0)
        with pytest.raises(EskfError, match="default kernel"):
            bf.run(**wl.streams0, seed=SEED, gt_dofs=GT, outlier_prob=0.3, outlier_std=OUT_STD)
        assert bf.launch_count == n0
        bf.run(**wl.streams0, seed=SEED, gt_dofs=GT)  # (without either, variant 1 runs)


def _raw_run(bf, s, seg):
    """eskf_run / eskf_run_epochs through the C ABI with the handle's current settings (BatchFilter.run sets them from its
    arguments first)"""
    orig_o, orig_g, orig_d = bf.set_meas_outliers, bf.set_innovation_gate, bf.set_meas_dropout
    bf.set_meas_outliers = lambda *a, **k: None
    bf.set_innovation_gate = lambda *a, **k: None
    bf.set_meas_dropout = lambda *a, **k: None
    try:
        bf.run(**s, epochs=seg)
    finally:
        bf.set_meas_outliers, bf.set_innovation_gate, bf.set_meas_dropout = orig_o, orig_g, orig_d


def test_simulator(tmp_path, monkeypatch):
    """batch.nis_gate / cam_outlier_prob / cam_outlier_std feed Simulator.run; absent they pass nothing (the launches of a
    run without either), and nis_gate= / cam_outliers= override the config"""
    import os

    import yaml

    from dvi_ekf_b200 import engine
    from dvi_ekf_b200.config import Config
    from dvi_ekf_b200.filter import Simulator

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    base = yaml.safe_load(open(os.path.join(root, "config.yaml")))
    base["simulation"]["num_kf_runs"] = 64

    def sim(**b):
        d = dict(base, batch=dict(base.get("batch") or {}, **b))
        f = tmp_path / "c.yaml"
        f.write_text(yaml.safe_dump(d))
        return Simulator(Config(str(f)))

    calls = []
    orig = engine.BatchFilter.run

    def spy(self, *a, **k):
        n0 = self.launch_count
        out = orig(self, *a, **k)
        calls.append((k.get("nis_gate"), k.get("outlier_prob"), self.launch_count - n0))
        return out

    monkeypatch.setattr(engine.BatchFilter, "run", spy)
    std = [1.0, 1.0, 1.0, 0.05, 0.05, 0.05, 0.1]
    s = sim(nis_gate=50.0, cam_outlier_prob=0.2, cam_outlier_std=std)
    s.run(consistency=True, verbose=False)
    E = len(s.streams.n_prop)
    assert calls[-1][:2] == (50.0, 0.2)
    rej = s.dof_envelope["rejected"]
    assert rej.shape == (E,) and rej.sum() > 0
    s0 = sim()
    s0.run(consistency=True, verbose=False)
    assert calls[-1][:2] == (None, None) and (s0.dof_envelope["rejected"] == 0).all()
    s0.run(consistency=True, verbose=False, nis_gate=50.0, cam_outliers=(0.2, std))
    assert calls[-1][:2] == (50.0, 0.2) and calls[-1][2] == calls[-2][2]
    assert np.array_equal(s0.dof_envelope["rejected"], rej)
