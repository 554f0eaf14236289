"""Filter consistency of eskf_run (eskf_keep_consistency: NIS of every update, NEES of the estimated DOFs after it) against
the batch oracle, through every path of eskf_kernel3 that files it.

The workload is the stacked Monte-Carlo workload of tests/test_gpu_paths.py: four trajectories x 13 filters, all six DOFs
estimated from perturbed values, ragged n_prop (epochs of 0..2 steps, a trajectory that stops 28 steps early), noise read
back with eskf_noise_dump.  With all DOFs estimated the recursion is ill-conditioned on three of the trajectories (see the
header of that file): there the bound is a floor plus K_SPREAD times the spread of a twin oracle started 1e-15 away."""
import numpy as np
import pytest

from tests.consistency_oracle import RecordingOracle as BatchOracle
from oracle.eskf_oracle import OracleConfig
from tests.helpers import Scenario, model_kwargs, mandala_scenario
from tests.test_gpu_noise import CAM_STD, IMU_STD, _noisy_streams
from tests.test_gpu_paths import FPT, GT, K_SPREAD, N_PROP, NAMES, SEED, SHAPES, Workload

pytestmark = pytest.mark.gpu

# relative bounds, ~3x the worst value measured on a B200 (1000 W), printed with -s as "MEASURED ...": NIS / NEES on
# traj_trans_x 1.25e-10 / 2.4e-10 (cond(S) up to 1e8 at the first update: the kernel's left inverse of S costs nothing there);
# d = 3 and the tuner objective 2.5e-12 .. 6.9e-12
TOL_NIS, TOL_NEES = 4e-10, 7e-10
# the other three trajectories: FLOOR + K_SPREAD x the twin oracle's spread (measured: 1.0 .. 3.0 x the largest spread)
FLOOR = 1e-6
TOL_SUM = 1e-12


def _oracle_values(bo, gt, frozen):
    """NIS of the oracle's last update and NEES of its estimated DOFs after it, per filter"""
    nis = np.einsum("ni,ni->n", bo.res, np.linalg.solve(bo.S, bo.res[..., None])[..., 0])
    keep = [i for i in range(6) if not frozen[i]]
    if not keep:
        return nis, np.full(len(nis), np.nan)
    eps = (bo.x[:, 10:16] - gt)[:, keep]
    B = bo.P[:, 9:15, 9:15][:, keep][:, :, keep]
    return nis, np.einsum("ni,ni->n", eps, np.linalg.solve(B, eps[..., None])[..., 0])


def _cons_reference(wl):
    """nis, nees [n, E] of the batch oracle on the kernels' noise, and their relative spread under a 1e-15 perturbation"""
    from dvi_ekf_b200.engine import NOISE_CAM, NOISE_IMU, noise_samples

    n, T, E = wl.n, wl.T, wl.E
    zi = noise_samples(SEED, 0, n, 0, T, NOISE_IMU)
    zc = noise_samples(SEED, 0, n, 0, E, NOISE_CAM)
    out = {k: np.empty((n, E)) for k in ("nis", "nees", "s_nis", "s_nees")}
    for j, sc in enumerate(wl.scs):
        rows = slice(j * FPT, (j + 1) * FPT)
        oa, cam, notch = np.empty((FPT, T, 6)), np.empty((FPT, E, 7)), np.empty((FPT, E))
        for i, g in enumerate(range(j * FPT, (j + 1) * FPT)):
            oa[i], cam[i], notch[i] = (sc.om_acc, sc.cam_meas, sc.notch_meas) if g == 0 else _noisy_streams(sc, zi[g], zc[g])
        bo = BatchOracle(sc.cfg, wl.x0[rows], sc.P0, wl.u0[rows], sc.Qd, sc.Rd, sc.sig_om)
        tw = BatchOracle(sc.cfg, wl.x0[rows] * (1 + 1e-15), sc.P0, wl.u0[rows], sc.Qd, sc.Rd, sc.sig_om)
        k = 0
        for e in range(E):
            for _ in range(N_PROP[j, e]):
                for b in (bo, tw):
                    b.propagate(sc.dt[k], oa[:, k, :3], oa[:, k, 3:])
                k += 1
            vals = []
            for b in (bo, tw):
                b.update(cam[:, e, :3], cam[:, e, 3:], notch[:, e])
                vals.append(_oracle_values(b, GT, (0,) * 6))
            (ni, ne), (ti, te) = vals
            out["nis"][rows, e], out["nees"][rows, e] = ni, ne
            out["s_nis"][rows, e], out["s_nees"][rows, e] = np.abs(ti / ni - 1), np.abs(te / ne - 1)
    return out


def _run(wl, F=28, path="prepass", n_traj=4, trace=False, jac=False, cons=True, lo=0, hi=None):
    """one eskf_run of filters lo..hi-1 of the workload (n_traj = 1: trajectory 0 alone) with consistency on / off, trace rows
    and the Jacobian record on / off"""
    from dvi_ekf_b200 import BatchFilter

    hi = wl.n if hi is None else hi
    n, sc0 = hi - lo, wl.sc0
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
        tr = np.full((n, wl.T, 26), np.nan) if trace else None
        st, sm = bf.run(**(wl.streams if n_traj > 1 else wl.streams0), n_traj=n_traj, filters_per_traj=FPT if n_traj > 1 else None,
                        seed=SEED, filter_id0=lo, imu_noise_std=IMU_STD, cam_noise_std=CAM_STD, noise_free_filter0=True, trace=tr,
                        gt_dofs=GT)
        x, P, u, R, status = bf.get_state()
        out = dict(x=x, P=P, u=u, R=R, status=status, stats=st, sum=sm)
        if cons:
            out["nis"], out["nees"], out["esum"] = bf.get_consistency()
    return out


def _sums(nis, nees, with_nees=True):
    """epoch_sum as include/eskf.h defines it, in numpy"""
    fa, fb = np.isfinite(nis), np.isfinite(nees)
    z = lambda v, f: np.where(f, v, 0.0)
    bad = ~fa | (~fb if with_nees else False)
    return np.stack([fa.sum(0), z(nis, fa).sum(0), z(nis * nis, fa).sum(0), fb.sum(0), z(nees, fb).sum(0),
                     z(nees * nees, fb).sum(0), bad.sum(0), np.zeros(nis.shape[1])], axis=1)


def _check_esum(out, with_nees=True):
    ref = _sums(out["nis"], out["nees"], with_nees)
    es = out["esum"]
    for c in (0, 3, 6, 7):
        assert np.array_equal(es[:, c], ref[:, c]), (c, es[:, c], ref[:, c])
    for c in (1, 2, 4, 5):
        assert np.allclose(es[:, c], ref[:, c], rtol=TOL_SUM, atol=0), (c, es[:, c], ref[:, c])


@pytest.fixture(scope="module")
def wl(golden):
    return Workload(golden)


@pytest.fixture(scope="module")
def cref(wl):
    return _cons_reference(wl)


@pytest.fixture(scope="module")
def canon(wl):
    return _run(wl)


@pytest.fixture(scope="module")
def canon1(wl):
    """trajectory 0 alone, pre-pass, F = 28"""
    out = _run(wl, n_traj=1, hi=FPT)
    _check_esum(out)
    return out


def test_parity_against_oracle(wl, cref, canon):
    """canonical cell (pre-pass, F = 28, stacked): NIS and NEES of every (filter, epoch) against the batch oracle fed the
    same noise; epoch_sum against the sums of the returned values"""
    assert canon["nis"].shape == (wl.n, wl.E) and canon["esum"].shape == (wl.E, 8)
    assert np.isfinite(canon["nis"]).all() and np.isfinite(canon["nees"]).all()
    for key, tol in (("nis", TOL_NIS), ("nees", TOL_NEES)):
        err = np.abs(canon[key] / cref[key] - 1)
        spread = cref["s_" + key]
        for j, nm in enumerate(NAMES):
            rows = slice(j * FPT, (j + 1) * FPT)
            print(f"MEASURED {key} {nm}: worst relative {err[rows].max():.2e}, oracle spread {spread[rows].max():.2e}, "
                  f"ANIS/ANEES {np.mean(canon[key][rows]):.3g}")
        bound = np.where(np.arange(wl.n)[:, None] < FPT, tol, FLOOR + K_SPREAD * spread)
        assert (err <= bound).all(), (key, np.argwhere(err > bound)[:5])
    _check_esum(canon)
    ref_sum = _sums(cref["nis"], cref["nees"])
    rel = np.abs(canon["esum"][:, [1, 4]] / ref_sum[:, [1, 4]] - 1)
    print(f"MEASURED epoch_sum vs oracle sums: worst relative {rel.max():.2e}")


@pytest.mark.parametrize("path", ("prepass", "inkernel"))
@pytest.mark.parametrize("F", SHAPES)
@pytest.mark.parametrize("n_traj", (4, 1), ids=["stacked", "traj0"])
def test_every_cell_bit_identical_and_unchanged(wl, canon, canon1, path, F, n_traj):
    """pre-pass / in-kernel statistics x every CTA shape x stacked / trajectory 0 alone x trace on / off x Jacobian record
    on / off: nis, nees and epoch_sum bit-identical to the canonical cell (trajectory 0 alone: its rows, and the epoch sums
    of trajectory 0 alone at F = 28); everything else the run leaves (x, P, u_old, R_old, status, statistics rows,
    stats_sum) bit-identical to the same cell with consistency off"""
    hi = wl.n if n_traj > 1 else FPT
    for trace in (False, True):
        for jac in (False, True):
            on = _run(wl, F, path, n_traj, trace, jac, True, hi=hi)
            off = _run(wl, F, path, n_traj, trace, jac, False, hi=hi)
            for key in ("x", "P", "u", "R", "status", "stats", "sum"):
                assert on[key].tobytes() == off[key].tobytes(), (trace, jac, key)
            for key in ("nis", "nees"):
                assert on[key].tobytes() == canon[key][:hi].tobytes(), (trace, jac, key)
            assert on["esum"].tobytes() == (canon if n_traj > 1 else canon1)["esum"].tobytes(), (trace, jac)


def test_sharding(wl, canon):
    """two shards at filter_id0 = 0 and N / 2 (a trajectory boundary): the rows of one handle bit for bit, epoch sums that
    add up to the whole handle's"""
    a = _run(wl, hi=wl.n // 2)
    b = _run(wl, lo=wl.n // 2)
    for key in ("nis", "nees"):
        assert np.concatenate([a[key], b[key]]).tobytes() == canon[key].tobytes()
    tot = a["esum"] + b["esum"]
    assert np.allclose(tot, canon["esum"], rtol=TOL_SUM, atol=0)
    assert np.array_equal(tot[:, [0, 3, 6]], canon["esum"][:, [0, 3, 6]])


def _single(golden, frozen, n, P0=None, Rd=None, Qd=None, oracle=True):
    """noise-free traj_trans_x run of n filters (initial DOFs of filter i > 0 perturbed where estimated) with consistency
    on, and (oracle) the batch oracle of the same filters"""
    from dvi_ekf_b200 import BatchFilter

    cfg = OracleConfig(max_vals=8, interframe_vals=10, frozen_dofs=frozen)
    sc = Scenario(golden["traj_trans_x"][:8], cfg)
    rng = np.random.default_rng(1)
    x0 = np.repeat(sc.x0[None], n, 0)
    est = ~np.array(frozen, dtype=bool)
    x0[1:, 10:16] += np.where(est, np.hstack((rng.normal(0, 0.03, (n - 1, 3)), rng.normal(0, 2.0, (n - 1, 3)))), 0.0)
    P = np.repeat(sc.P0[None], n, 0) if P0 is None else P0
    R = np.repeat(sc.Rd[None], n, 0) if Rd is None else Rd
    E = len(sc.n_prop)
    with BatchFilter(n, **model_kwargs(cfg)) as bf:
        bf.set_noise(sc.Qd[None] if Qd is None else Qd, R, sc.sig_om[None])
        bf.set_state(x0, P, sc.u0[None], None)
        bf.keep_consistency()
        bf.run(sc.dt, sc.om_acc, sc.n_prop, sc.cam_meas, sc.notch_meas, gt_dofs=GT)
        nis, nees, es = bf.get_consistency()
        status = bf.get_state()[4]
    if not oracle:
        return dict(nis=nis, nees=nees, esum=es, status=status)
    bo = BatchOracle(cfg, x0, P, sc.u0, sc.Qd, R, sc.sig_om)
    rn, re = np.empty((n, E)), np.empty((n, E))
    k = 0
    for e in range(E):
        for _ in range(sc.n_prop[e]):
            bo.propagate(sc.dt[k], sc.om_acc[k, :3], sc.om_acc[k, 3:])
            k += 1
        bo.update(sc.cam_meas[e, :3], sc.cam_meas[e, 3:], sc.notch_meas[e])
        rn[:, e], re[:, e] = _oracle_values(bo, GT, frozen)
    return dict(nis=nis, nees=nees, esum=es, status=status, rnis=rn, rnees=re)


def test_three_estimated_dofs(golden):
    """frozen (1, 1, 1, 0, 0, 0): d = 3, the NEES of the translational DOFs against the oracle"""
    r = _single(golden, (1, 1, 1, 0, 0, 0), 8)
    en, ee = np.abs(r["nis"] / r["rnis"] - 1).max(), np.abs(r["nees"] / r["rnees"] - 1).max()
    print(f"MEASURED d = 3 vs oracle: NIS {en:.2e}, NEES {ee:.2e}")
    assert en < TOL_NIS and ee < TOL_NEES
    assert r["esum"][:, 3].tolist() == [8.0] * r["nis"].shape[1]


def test_all_frozen(golden):
    """config.yaml freezes all six DOFs: NEES NaN and not counted, NIS valid"""
    r = _single(golden, (1,) * 6, 4)
    assert np.isnan(r["nees"]).all() and np.isfinite(r["nis"]).all()
    assert np.abs(r["nis"] / r["rnis"] - 1).max() < TOL_NIS
    es = r["esum"]
    assert (es[:, 3:6] == 0).all() and (es[:, 6] == 0).all() and (es[:, 0] == 4).all()


def test_singular_filter_is_nan_and_counted(golden):
    """one filter with P0 = 0, Q = 0 and R = 0 (singular S at every update, never applied): NaN at every epoch, counted in
    [6]; the other filters have the values of a run without it"""
    n = 5
    cfg = OracleConfig(max_vals=8, interframe_vals=10, frozen_dofs=(0,) * 6)
    sc = Scenario(golden["traj_trans_x"][:8], cfg)
    P = np.repeat(sc.P0[None], n, 0)
    R = np.repeat(sc.Rd[None], n, 0)
    Q = np.repeat(sc.Qd[None], n, 0)
    P[2], R[2], Q[2] = 0.0, 0.0, 0.0
    good = _single(golden, (0,) * 6, n, Qd=Q, oracle=False)
    bad = _single(golden, (0,) * 6, n, P0=P, Rd=R, Qd=Q, oracle=False)
    assert bad["status"][2] & 1 and np.all(np.delete(bad["status"], 2) == 0)
    assert np.isnan(bad["nis"][2]).all() and np.isnan(bad["nees"][2]).all()
    others = [0, 1, 3, 4]
    assert bad["nis"][others].tobytes() == good["nis"][others].tobytes()
    assert bad["nees"][others].tobytes() == good["nees"][others].tobytes()
    assert (bad["esum"][:, 6] == 1).all() and (bad["esum"][:, 0] == n - 1).all() and (bad["esum"][:, 3] == n - 1).all()


def test_zero_epochs_errors_and_variant(golden):
    """E = 0 gives empty arrays; get_consistency before any run and the first kernel (variant 1) raise"""
    from dvi_ekf_b200 import BatchFilter
    from dvi_ekf_b200._lib import EskfError

    sc = mandala_scenario(golden, n_frames=4, ifv=2)
    with BatchFilter(3, **model_kwargs(sc.cfg)) as bf:
        bf.set_noise(sc.Qd[None], sc.Rd[None], sc.sig_om[None])
        bf.set_state(sc.x0[None], sc.P0[None], sc.u0[None], None)
        with pytest.raises(EskfError, match="no eskf_run"):
            bf.get_consistency()
        bf.keep_consistency()
        with pytest.raises(EskfError, match="no eskf_run"):
            bf.get_consistency()
        bf.propagate(sc.dt[:2], sc.om_acc[:2])  # (the single-step verbs file nothing)
        with pytest.raises(EskfError):
            bf.get_consistency()
        bf.run(sc.dt, sc.om_acc, np.zeros(0, np.int32), np.zeros((0, 7)), np.zeros(0))
        nis, nees, es = bf.get_consistency()
        assert nis.shape == (3, 0) and nees.shape == (3, 0) and es.shape == (0, 8)
        with pytest.raises(EskfError):
            bf.set_variant(1)
    with BatchFilter(3, variant=1, **model_kwargs(sc.cfg)) as bf:
        with pytest.raises(EskfError, match="default kernel"):
            bf.keep_consistency()


def test_records_that_do_not_fit_are_refused_before_anything_runs(golden):
    """65,536 filters x 4,000,000 epochs would need 92 TB of records: ESKF_ENOMEM, the state is untouched, and the handle
    still runs (and keeps the results of its last run readable until then)"""
    from dvi_ekf_b200 import BatchFilter
    from dvi_ekf_b200._lib import EskfError

    sc = mandala_scenario(golden, n_frames=4, ifv=2)
    n, E = 1 << 16, 4_000_000
    with BatchFilter(n, **model_kwargs(sc.cfg)) as bf:
        bf.set_noise(sc.Qd[None], sc.Rd[None], sc.sig_om[None])
        bf.set_state(sc.x0[None], sc.P0[None], sc.u0[None], None)
        bf.keep_consistency()
        bf.run(sc.dt, sc.om_acc, sc.n_prop, sc.cam_meas, sc.notch_meas)
        first = bf.get_consistency()
        x0, _, _, _, st0 = bf.get_state()
        with pytest.raises(EskfError, match=r"code -3"):
            bf.run(sc.dt[:1], sc.om_acc[:1], np.zeros(E, np.int32), np.zeros((E, 7)), np.zeros(E))
        x1, _, _, _, st1 = bf.get_state()
        assert x1.tobytes() == x0.tobytes() and st1.tobytes() == st0.tobytes()
        again = bf.get_consistency()
        assert all(a.tobytes() == b.tobytes() for a, b in zip(first, again))
        bf.run(sc.dt, sc.om_acc, sc.n_prop, sc.cam_meas, sc.notch_meas)
        assert np.isfinite(bf.get_consistency()[0]).all()


def test_tuner_objective_matches_oracle(golden, tmp_path):
    """Simulator.evaluate_candidates(metric="nis" / "nees") for 2 candidates x 3 runs with all six DOFs estimated, against
    the batch oracle on the noise the kernels drew (the set-up of test_gpu_configs.py::test_tuner_objective_matches_oracle)"""
    import os

    import yaml

    from dvi_ekf_b200 import Config, Simulator
    from dvi_ekf_b200.consistency import candidate_objective
    from dvi_ekf_b200.engine import NOISE_CAM, NOISE_IMU, noise_samples
    from oracle.eskf_oracle import quat_about_axis, quat_mul

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    y = yaml.safe_load(open(os.path.join(root, "config.yaml")))
    frames, ifv, r = 14, 5, 3
    y["simulation"].update(do_fast_sim=False, frozen_dofs=[0] * 6)
    y["camera"]["total_frames"] = frames
    y["imu"]["interframe_vals"] = ifv
    fp = tmp_path / "config.yaml"
    fp.write_text(yaml.safe_dump(y))
    cfg = Config(str(fp))
    sim = Simulator(cfg)
    b = cfg.batch
    base = np.array([*cfg.process_noise_rw_std, *cfg.meas_noise_std], dtype=float)
    X = np.array([base, base * np.linspace(0.5, 2.0, 14)])
    f_nis = sim.evaluate_candidates(X, runs_per_candidate=r, metric="nis")
    f_nees = sim.evaluate_candidates(X, runs_per_candidate=r, metric="nees")

    sc = mandala_scenario(golden, n_frames=frames, ifv=ifv, frozen_dofs=(0,) * 6)
    s = sim.streams
    T, E = len(sc.dt), len(sc.n_prop)
    imu_std = np.hstack((cfg.imu.stdev_omega, cfg.imu.stdev_accel))
    cam_std = np.array(cfg.meas_noise_std)
    zi = noise_samples(b.seed, 0, r, 0, T, NOISE_IMU)
    zc = noise_samples(b.seed, 0, r, 0, E, NOISE_CAM)
    gt = np.asarray(cfg.gt_imu_dofs, dtype=float)
    x0 = np.repeat(s.x0[None], r, 0)
    oa, cam, notch = np.repeat(s.om_acc[None], r, 0), np.repeat(s.cam[None], r, 0), np.repeat(s.notch[None], r, 0)
    for j in range(1, r):  # run 0 of every candidate: nominal initial state, noise free
        rng = np.random.default_rng([b.seed, j])
        x0[j, 10:13] += rng.normal(0.0, np.deg2rad(b.dof_ic_std_deg), 3)
        x0[j, 13:16] += rng.normal(0.0, b.dof_ic_std_cm, 3)
        oa[j] += imu_std[None, :] * zi[j][:, :6]
        for e in range(E):
            cam[j, e, :3] += cam_std[:3] * zc[j][e, :3]
            dth = cam_std[3:6] * zc[j][e, 3:6]
            nq = np.linalg.norm(cam[j, e, 3:])
            cam[j, e, 3:] = quat_mul(cam[j, e, 3:], quat_about_axis(np.linalg.norm(dth), dth)) * nq
            notch[j, e] += cam_std[6] * zc[j][e, 6]
    rn, re = np.empty((2 * r, E)), np.empty((2 * r, E))
    for c in range(2):
        bo = BatchOracle(sc.cfg, x0, sc.P0, s.u0, np.hstack((np.zeros(6), np.square(X[c, 0:7]))), np.square(X[c, 7:14]), sim.kf.stdev_nom)
        k = 0
        for e in range(E):
            for _ in range(s.n_prop[e]):
                bo.propagate(s.dt[k], oa[:, k, :3], oa[:, k, 3:])
                k += 1
            bo.update(cam[:, e, :3], cam[:, e, 3:], notch[:, e])
            rn[c * r:(c + 1) * r, e], re[c * r:(c + 1) * r, e] = _oracle_values(bo, gt, (0,) * 6)
    o_nis, o_nees = candidate_objective(rn, 2, 7), candidate_objective(re, 2, 6)
    en, ee = np.abs(f_nis - o_nis).max(), np.abs(f_nees - o_nees).max()
    print(f"MEASURED tuner objective vs oracle: nis {en:.2e} ({f_nis}), nees {ee:.2e} ({f_nees})")
    assert en < TOL_NIS and ee < TOL_NEES
    assert abs(f_nis[0] - f_nis[1]) > 1e-3  # the candidates really differ
    cfg.frozen_dofs = [1] * 6
    with pytest.raises(ValueError, match="nees"):
        sim.evaluate_candidates(X, runs_per_candidate=r, metric="nees")


def test_config2_calibration_full_size(golden):
    """config 2 calibration: mandala0_mono, 1390 steps, 139 updates, 4096 filters, all six DOFs estimated from perturbed
    values, Monte-Carlo noise.  epoch_sum finite with counts that add up to N; the noise-free filter 0 against a single
    free-running oracle; the ANIS / ANEES curve printed with -s (the reference's filter, not the engine: DESIGN.md section 6)"""
    from bench import SEED as BSEED
    from bench import Workload as BenchWorkload
    from dvi_ekf_b200 import BatchFilter
    from dvi_ekf_b200.consistency import summarise_consistency
    from dvi_ekf_b200.sharding import mc_initial_states

    wl = BenchWorkload()
    s = wl.s
    n = 4096
    gt = np.asarray(wl.cfg.gt_imu_dofs, dtype=float)
    model = dict(wl.model, frozen_dofs=(0,) * 6)
    with BatchFilter(n, **model) as bf:
        bf.set_noise(wl.Qd[None], wl.Rd[None], wl.sig_om[None])
        bf.set_state(mc_initial_states(s.x0, n, 0, BSEED), wl.P0[None], s.u0[None], None)
        bf.keep_consistency()
        bf.run(s.dt, s.om_acc, s.n_prop, s.cam, s.notch, seed=BSEED, imu_noise_std=wl.imu_std, cam_noise_std=wl.cam_std,
               gt_dofs=tuple(gt))
        nis, nees, es = bf.get_consistency()
    E = len(s.n_prop)
    assert nis.shape == (n, E) and np.isfinite(es).all()
    assert (es[:, 0] + es[:, 6] >= n).all() and (es[:, 0] <= n).all() and (es[:, 3] <= n).all()
    assert np.array_equal(es[:, 6], (~np.isfinite(nis) | ~np.isfinite(nees)).sum(0))
    _check_esum(dict(nis=nis, nees=nees, esum=es))
    cfg = OracleConfig(max_vals=140, interframe_vals=10, frozen_dofs=(0,) * 6)
    bo = BatchOracle(cfg, np.stack([s.x0, s.x0 * (1 + 1e-15)]), wl.P0, s.u0, wl.Qd, wl.Rd, wl.sig_om)
    rn, re = np.empty((2, E)), np.empty((2, E))
    k = 0
    for e in range(E):
        for _ in range(s.n_prop[e]):
            bo.propagate(s.dt[k], s.om_acc[k, :3], s.om_acc[k, 3:])
            k += 1
        bo.update(s.cam[e, :3], s.cam[e, 3:], s.notch[e])
        rn[:, e], re[:, e] = _oracle_values(bo, gt, (0,) * 6)
    en, ee = np.abs(nis[0] / rn[0] - 1), np.abs(nees[0] / re[0] - 1)
    sn, se = np.abs(rn[1] / rn[0] - 1), np.abs(re[1] / re[0] - 1)
    for nm, err, spr in (("NIS", en, sn), ("NEES", ee, se)):
        late = np.flatnonzero(err > 1e-6)
        print(f"MEASURED config 2 filter 0 {nm} vs free-running oracle: worst {err.max():.2e} (oracle spread {spr.max():.2e}); "
              f"epochs 0..9 {err[:10].max():.2e}; first epoch above 1e-6: {late[0] if len(late) else None}; worst ratio to the "
              f"spread {(err / np.maximum(spr, 1e-16)).max():.1f}")
    summ = summarise_consistency(es, 6)
    for e in (0, 1, 9, 49, 99, E - 1):
        print(f"MEASURED config 2 epoch {e}: ANIS {summ['anis'][e]:.4g} {summ['nis_interval'][e].round(3)}, "
              f"ANEES {summ['anees'][e]:.4g} {summ['nees_interval'][e].round(3)}, skipped {summ['skipped'][e]:.0f}")
    print(f"MEASURED config 2: epochs inside the 95 % interval: NIS {summ['nis_inside']:.2f}, NEES {summ['nees_inside']:.2f}; "
          f"ANIS over all epochs {np.nanmean(nis):.4g}, ANEES {np.nanmean(nees):.4g}")
    # the first ten epochs, before the all-DOF recursion amplifies rounding (measured 3.5e-11 / 2.1e-11; the relative error first
    # exceeds 1e-6 at epoch 67 / 78, where the oracle's own spread has grown to the same order), then the spread bound
    assert en[:10].max() < 1e-10 and ee[:10].max() < 1e-10
    assert (en <= FLOOR + K_SPREAD * sn).all() and (ee <= FLOOR + K_SPREAD * se).all()
