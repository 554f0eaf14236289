"""Per-DOF history and Monte-Carlo envelope (eskf_get_dof_history / eskf_get_dof_envelope) against the batch oracle and
numpy, through every path of eskf_kernel3 that files the consistency records.

The workload is the stacked Monte-Carlo workload of tests/test_gpu_paths.py (four trajectories x 13 filters, all six DOFs
estimated from perturbed values, ragged n_prop, noise read back with eskf_noise_dump).  On the three ill-conditioned
trajectories the oracle bound is a floor plus K_SPREAD times the spread of a twin oracle started 1e-15 away, as in
tests/test_gpu_consistency.py."""
import numpy as np
import pytest

from oracle.eskf_oracle import OracleConfig
from tests.consistency_oracle import RecordingOracle as BatchOracle
from tests.dof_reference import COUNTS, NDOFSUM, PAIRS, assert_envelope_close, envelope
from tests.helpers import Scenario, mandala_scenario, model_kwargs
from tests.test_gpu_consistency import FLOOR, TOL_SUM, _oracle_values
from tests.test_gpu_noise import CAM_STD, IMU_STD, _noisy_streams
from tests.test_gpu_paths import FPT, GT, K_SPREAD, N_PROP, NAMES, SEED, SHAPES, Workload

pytestmark = pytest.mark.gpu

# ~3x the worst value measured on a B200 (1000 W), printed with -s as "MEASURED ...": the history on traj_trans_x against
# the oracle, relative (DOFs: to the largest |value| of their rotation / translation triple; variances: to themselves),
# measured 1.1e-10 / 1.3e-10; the envelope of trajectory 0 alone against the one of the oracle's values, relative to the
# sums of the absolute terms, measured 7.2e-11
TOL_DOFS, TOL_VAR = 3.5e-10, 4e-10
TOL_ENV_ORACLE = 2.5e-10
KEYS = ("x", "P", "u", "R", "status", "stats", "sum", "nis", "nees", "esum", "trace")


def _dof_err(got, ref):
    """[..., 6] error relative to the largest |ref| of the rotation / translation triple"""
    out = np.empty(got.shape)
    for s in (slice(0, 3), slice(3, 6)):
        den = np.maximum(np.abs(ref[..., s]).max(axis=-1, keepdims=True), 1e-12)
        out[..., s] = np.abs(got[..., s] - ref[..., s]) / den
    return out


def _dof_reference(wl):
    """the batch oracle on the kernels' noise after every update: nis [n, E], dofs and var [n, E, 6], B [n, E, 6, 6], and the
    relative spread of dofs / var under a 1e-15 perturbation of the initial state"""
    from dvi_ekf_b200.engine import NOISE_CAM, NOISE_IMU, noise_samples

    n, T, E = wl.n, wl.T, wl.E
    zi = noise_samples(SEED, 0, n, 0, T, NOISE_IMU)
    zc = noise_samples(SEED, 0, n, 0, E, NOISE_CAM)
    out = dict(nis=np.empty((n, E)), dofs=np.empty((n, E, 6)), var=np.empty((n, E, 6)), B=np.empty((n, E, 6, 6)),
               s_dofs=np.empty((n, E, 6)), s_var=np.empty((n, E, 6)))
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
            for b in (bo, tw):
                b.update(cam[:, e, :3], cam[:, e, 3:], notch[:, e])
            out["nis"][rows, e] = _oracle_values(bo, GT, (0,) * 6)[0]
            out["dofs"][rows, e] = bo.x[:, 10:16]
            out["B"][rows, e] = bo.P[:, 9:15, 9:15]
            out["var"][rows, e] = np.diagonal(bo.P[:, 9:15, 9:15], axis1=1, axis2=2)
            out["s_dofs"][rows, e] = _dof_err(tw.x[:, 10:16], bo.x[:, 10:16])
            out["s_var"][rows, e] = np.abs(np.diagonal(tw.P[:, 9:15, 9:15], axis1=1, axis2=2) / out["var"][rows, e] - 1)
    return out


def _run(wl, F=28, path="prepass", n_traj=4, trace=False, jac=False, getters=True, lo=0, hi=None):
    """one eskf_run of filters lo..hi-1 of the workload with consistency on; with ``getters`` the per-DOF history and
    (twice) the envelope are read BEFORE everything else the run returned"""
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
        bf.keep_consistency(True)
        tr = np.full((n, wl.T, 26), np.nan) if trace else None
        st, sm = bf.run(**(wl.streams if n_traj > 1 else wl.streams0), n_traj=n_traj, filters_per_traj=FPT if n_traj > 1 else None,
                        seed=SEED, filter_id0=lo, imu_noise_std=IMU_STD, cam_noise_std=CAM_STD, noise_free_filter0=True, trace=tr,
                        gt_dofs=GT)
        out = dict(stats=st, sum=sm, trace=tr)
        if getters:
            out["dofs"], out["var"] = bf.get_dof_history()
            out["env"] = bf.get_dof_envelope()
            out["env2"] = bf.get_dof_envelope()
        out["x"], out["P"], out["u"], out["R"], out["status"] = bf.get_state()
        out["nis"], out["nees"], out["esum"] = bf.get_consistency()
    return out


@pytest.fixture(scope="module")
def wl(golden):
    return Workload(golden)


@pytest.fixture(scope="module")
def dref(wl):
    return _dof_reference(wl)


@pytest.fixture(scope="module")
def canon(wl):
    return _run(wl)


@pytest.fixture(scope="module")
def canon1(wl):
    """trajectory 0 alone, pre-pass, F = 28"""
    return _run(wl, n_traj=1, hi=FPT)


def _engine_envelope(out, B=None):
    """the envelope of a run's own history and nis in numpy; B [n, E, 6, 6] for the off-diagonal entries (zeros without)"""
    n, E = out["nis"].shape
    if B is None:
        B = np.zeros((n, E, 6, 6))
    B = B.copy()
    B[:, :, np.arange(6), np.arange(6)] = out["var"]
    return envelope(out["nis"], out["dofs"], B, GT, 0), envelope(out["nis"], out["dofs"], B, GT, 0, absolute=True)


def test_history_against_oracle(wl, dref, canon):
    """canonical cell: dofs and var of every (filter, epoch) against the batch oracle fed the same noise"""
    assert canon["dofs"].shape == (wl.n, wl.E, 6) and canon["var"].shape == (wl.n, wl.E, 6)
    assert np.isfinite(canon["dofs"]).all() and (canon["var"] > 0).all()
    err = dict(dofs=_dof_err(canon["dofs"], dref["dofs"]), var=np.abs(canon["var"] / dref["var"] - 1))
    for key, tol in (("dofs", TOL_DOFS), ("var", TOL_VAR)):
        spread = dref["s_" + key]
        for j, nm in enumerate(NAMES):
            rows = slice(j * FPT, (j + 1) * FPT)
            print(f"MEASURED dof history {key} {nm}: worst relative {err[key][rows].max():.2e}, oracle spread "
                  f"{spread[rows].max():.2e}")
        bound = np.where(np.arange(wl.n)[:, None, None] < FPT, tol, FLOOR + K_SPREAD * spread)
        assert (err[key] <= bound).all(), (key, np.argwhere(err[key] > bound)[:5])


def test_history_is_the_trace_row_of_the_update(wl, canon):
    """traj_trans_x (10 steps per epoch): the DOFs of epoch e are x[10:16] of the trace row of its last step, bit for bit"""
    out = _run(wl, trace=True)
    last = np.cumsum(N_PROP[0]) - 1
    assert out["dofs"][:FPT].tobytes() == np.ascontiguousarray(out["trace"][:FPT][:, last, 10:16]).tobytes()
    assert out["dofs"].tobytes() == canon["dofs"].tobytes()


def test_device_outputs_match_host(canon, wl):
    """get_dof_history / get_dof_envelope into CUDA tensors: the bits of the host copies"""
    from dvi_ekf_b200 import BatchFilter

    sc0 = wl.sc0
    with BatchFilter(wl.n, **model_kwargs(sc0.cfg)) as bf:
        bf.set_tuning(28)
        bf.set_noise(sc0.Qd[None], sc0.Rd[None], sc0.sig_om[None])
        bf.set_state(wl.x0, sc0.P0[None], wl.u0, None)
        bf.keep_consistency(True)
        bf.run(**wl.streams, n_traj=4, filters_per_traj=FPT, seed=SEED, imu_noise_std=IMU_STD, cam_noise_std=CAM_STD,
               noise_free_filter0=True, gt_dofs=GT)
        d, v = bf.get_dof_history(device=True)
        env = bf.get_dof_envelope(device=True)
        assert d.is_cuda and env.is_cuda
        assert d.cpu().numpy().tobytes() == canon["dofs"].tobytes() and v.cpu().numpy().tobytes() == canon["var"].tobytes()
        assert env.cpu().numpy().tobytes() == canon["env"].tobytes()


def test_envelope_against_numpy(wl, dref, canon, canon1):
    """the envelope against numpy on the engine's own history and nis: counts exact, sums to TOL_SUM of the absolute sums;
    the pair sums of the block at the last epoch against get_state's P (the last update is the last thing every
    trajectory does); trajectory 0 alone once more against the envelope of the oracle's values"""
    env = canon["env"]
    assert env.shape == (wl.E, NDOFSUM) and (env[:, 74:] == 0).all()
    assert (env[:, 0] == wl.n).all() and (env[:, 1] == 0).all()
    ref, scale = _engine_envelope(canon)
    assert_envelope_close(env, ref, scale, TOL_SUM, cols=slice(0, 59))
    B = np.zeros((wl.n, wl.E, 6, 6))
    B[:, -1] = canon["P"][:, 9:15, 9:15]
    ref, scale = _engine_envelope(canon, B)
    assert_envelope_close(env[-1:], ref[-1:], scale[-1:], TOL_SUM)
    o = {k: dref[k][:FPT] for k in ("nis", "dofs", "B")}
    oref = envelope(o["nis"], o["dofs"], o["B"], GT, 0)
    oscale = envelope(o["nis"], o["dofs"], o["B"], GT, 0, absolute=True)
    rel = np.abs(canon1["env"] - oref) / np.maximum(oscale, 1e-300)
    print(f"MEASURED envelope of traj_trans_x vs the oracle's: worst relative {rel.max():.2e}")
    assert_envelope_close(canon1["env"], oref, oscale, TOL_ENV_ORACLE)


@pytest.mark.parametrize("path", ("prepass", "inkernel"))
@pytest.mark.parametrize("F", SHAPES)
@pytest.mark.parametrize("n_traj", (4, 1), ids=["stacked", "traj0"])
def test_every_cell_bit_identical_and_unchanged(wl, canon, canon1, path, F, n_traj):
    """pre-pass / in-kernel statistics x every CTA shape x stacked / trajectory 0 alone x trace on / off x Jacobian record
    on / off: the history bit-identical to the canonical cell (trajectory 0 alone: its rows), the envelope to the canonical
    run of the same filters, twice; everything else the run returned bit-identical to the same run without the getters"""
    hi = wl.n if n_traj > 1 else FPT
    for trace in (False, True):
        for jac in (False, True):
            on = _run(wl, F, path, n_traj, trace, jac, True, hi=hi)
            off = _run(wl, F, path, n_traj, trace, jac, False, hi=hi)
            for key in KEYS:
                a, b = on[key], off[key]
                assert (a is None and b is None) or a.tobytes() == b.tobytes(), (trace, jac, key)
            for key in ("dofs", "var"):
                assert on[key].tobytes() == canon[key][:hi].tobytes(), (trace, jac, key)
            ref = (canon if n_traj > 1 else canon1)["env"]
            assert on["env"].tobytes() == ref.tobytes() and on["env2"].tobytes() == ref.tobytes(), (trace, jac)


def test_sharding(wl, dref, canon):
    """two shards at filter_id0 = 0 and N / 2 (a trajectory boundary): the histories concatenate bit for bit, the envelopes
    add up to the whole handle's (counts exact)"""
    a = _run(wl, hi=wl.n // 2)
    b = _run(wl, lo=wl.n // 2)
    for key in ("dofs", "var"):
        assert np.concatenate([a[key], b[key]]).tobytes() == canon[key].tobytes()
    scale = envelope(dref["nis"], dref["dofs"], dref["B"], GT, 0, absolute=True)
    assert_envelope_close(a["env"] + b["env"], canon["env"], scale, TOL_SUM)


def _single(golden, frozen, n, P0=None, Rd=None, Qd=None):
    """noise-free traj_trans_x run of n filters (initial DOFs of filter i > 0 perturbed where estimated) with consistency on"""
    from dvi_ekf_b200 import BatchFilter

    cfg = OracleConfig(max_vals=8, interframe_vals=10, frozen_dofs=frozen)
    sc = Scenario(golden["traj_trans_x"][:8], cfg)
    rng = np.random.default_rng(1)
    x0 = np.repeat(sc.x0[None], n, 0)
    est = ~np.array(frozen, dtype=bool)
    x0[1:, 10:16] += np.where(est, np.hstack((rng.normal(0, 0.03, (n - 1, 3)), rng.normal(0, 2.0, (n - 1, 3)))), 0.0)
    with BatchFilter(n, **model_kwargs(cfg)) as bf:
        bf.set_noise(sc.Qd[None] if Qd is None else Qd, np.repeat(sc.Rd[None], n, 0) if Rd is None else Rd, sc.sig_om[None])
        bf.set_state(x0, np.repeat(sc.P0[None], n, 0) if P0 is None else P0, sc.u0[None], None)
        bf.keep_consistency()
        bf.run(sc.dt, sc.om_acc, sc.n_prop, sc.cam_meas, sc.notch_meas, gt_dofs=GT)
        nis, nees, es = bf.get_consistency()
        dofs, var = bf.get_dof_history()
        env = bf.get_dof_envelope()
        status = bf.get_state()[4]
    return dict(nis=nis, nees=nees, esum=es, dofs=dofs, var=var, env=env, status=status)


def test_one_estimated_dof(golden):
    """frozen_mask = 31: the NEES is eps_5^2 / B_55, so the envelope's sum of it is epoch_sum[:, 4] and M epoch_sum[:, 3]"""
    r = _single(golden, (1, 1, 1, 1, 1, 0), 8)
    env, es = r["env"], r["esum"]
    assert np.array_equal(env[:, 0], es[:, 3]) and (env[:, 0] == 8).all()
    rel = np.abs(env[:, 2 + 7 * 5 + 3] / es[:, 4] - 1)
    assert rel.max() < 1e-13, rel.max()


def test_three_and_zero_estimated_dofs(golden):
    """d = 3 (rotations frozen): their entries and every pair involving one are 0, the summary NaN for them; d = 0: every
    sum 0 and M the finite NIS"""
    from dvi_ekf_b200.consistency import summarise_dofs

    frozen = (1, 1, 1, 0, 0, 0)
    r = _single(golden, frozen, 8)
    env = r["env"]
    zero = [2 + 7 * i + k for i in range(3) for k in range(7)]
    zero += [44 + p for p, (i, j) in enumerate(PAIRS) if i < 3] + [59 + p for p, (i, j) in enumerate(PAIRS) if i < 3]
    assert (env[:, zero] == 0).all()
    assert (env[:, [2 + 7 * i + 2 for i in range(3, 6)]] > 0).all()  # sum of the translations' variances
    s = summarise_dofs(env, frozen)
    for key in ("bias", "rmse", "std", "sigma_filter", "inflation", "anees_dof"):
        assert np.isnan(s[key][:, :3]).all() and np.isfinite(s[key][:, 3:]).all(), key
    assert np.isnan(s["err_second_moment"][:, :3]).all() and np.isfinite(s["filter_cov"][:, 3:, 3:]).all()
    r0 = _single(golden, (1,) * 6, 4)
    assert (r0["env"][:, 2:] == 0).all() and np.array_equal(r0["env"][:, 0], r0["esum"][:, 0]) and (r0["env"][:, 1] == 0).all()


def test_singular_filter_is_excluded_and_counted(golden):
    """one filter with P0 = Q = R = 0 (the update is never applied, its NIS is NaN): excluded at every epoch, counted in
    [1], and the envelope is the numpy reduction over the other filters' history"""
    n = 5
    cfg = OracleConfig(max_vals=8, interframe_vals=10, frozen_dofs=(0,) * 6)
    sc = Scenario(golden["traj_trans_x"][:8], cfg)
    P, R, Q = np.repeat(sc.P0[None], n, 0), np.repeat(sc.Rd[None], n, 0), np.repeat(sc.Qd[None], n, 0)
    P[2], R[2], Q[2] = 0.0, 0.0, 0.0
    r = _single(golden, (0,) * 6, n, P0=P, Rd=R, Qd=Q)
    assert r["status"][2] & 1 and np.isnan(r["nis"][2]).all()
    env = r["env"]
    assert (env[:, 1] == 1).all() and (env[:, 0] == n - 1).all()
    others = [0, 1, 3, 4]
    sub = {k: r[k][others] for k in ("nis", "dofs", "var")}
    ref, scale = _engine_envelope(sub)
    ref[:, 1] = 1.0  # (the excluded filter)
    assert_envelope_close(env, ref, scale, TOL_SUM, cols=slice(0, 59))


def test_errors_zero_epochs_and_memory(golden):
    """EINVAL before any run, after keep_consistency(False) and with the first kernel; E = 0 gives empty arrays; a run
    refused with ESKF_ENOMEM leaves the history and envelope of the last run readable, unchanged"""
    from dvi_ekf_b200 import BatchFilter
    from dvi_ekf_b200._lib import EskfError

    sc = mandala_scenario(golden, n_frames=4, ifv=2)
    with BatchFilter(3, **model_kwargs(sc.cfg)) as bf:
        bf.set_noise(sc.Qd[None], sc.Rd[None], sc.sig_om[None])
        bf.set_state(sc.x0[None], sc.P0[None], sc.u0[None], None)
        for get in (bf.get_dof_history, bf.get_dof_envelope):
            with pytest.raises(EskfError, match="no eskf_run"):
                get()
        bf.keep_consistency()
        bf.run(sc.dt, sc.om_acc, np.zeros(0, np.int32), np.zeros((0, 7)), np.zeros(0))
        d, v = bf.get_dof_history()
        assert d.shape == (3, 0, 6) and v.shape == (3, 0, 6) and bf.get_dof_envelope().shape == (0, NDOFSUM)
        bf.run(sc.dt, sc.om_acc, sc.n_prop, sc.cam_meas, sc.notch_meas)
        assert bf.get_dof_envelope()[:, 0].tolist() == [3.0] * len(sc.n_prop)
        bf.keep_consistency(False)
        for get in (bf.get_dof_history, bf.get_dof_envelope):
            with pytest.raises(EskfError, match="no eskf_run"):
                get()
    with BatchFilter(3, variant=1, **model_kwargs(sc.cfg)) as bf:
        for get in (bf.get_dof_history, bf.get_dof_envelope):
            with pytest.raises(EskfError):
                get()
    n, E = 1 << 16, 4_000_000
    with BatchFilter(n, **model_kwargs(sc.cfg)) as bf:
        bf.set_noise(sc.Qd[None], sc.Rd[None], sc.sig_om[None])
        bf.set_state(sc.x0[None], sc.P0[None], sc.u0[None], None)
        bf.keep_consistency()
        bf.run(sc.dt, sc.om_acc, sc.n_prop, sc.cam_meas, sc.notch_meas)
        first = (*bf.get_dof_history(), bf.get_dof_envelope())
        with pytest.raises(EskfError, match=r"code -3"):
            bf.run(sc.dt[:1], sc.om_acc[:1], np.zeros(E, np.int32), np.zeros((E, 7)), np.zeros(E))
        again = (*bf.get_dof_history(), bf.get_dof_envelope())
        assert all(a.tobytes() == b.tobytes() for a, b in zip(first, again))


def test_host_history_in_chunks(golden):
    """64 filters x 12,000 epochs: a host copy of the history takes two chunks of the staging buffer (58 rows of 32 MiB
    per array, then 6); the same bits as the device copy, which is one launch"""
    from dvi_ekf_b200 import BatchFilter

    sc = mandala_scenario(golden, n_frames=4, ifv=2, frozen_dofs=(0,) * 6)
    E, n = 12000, 64
    rng = np.random.default_rng(3)
    x0 = np.repeat(sc.x0[None], n, 0)
    x0[:, 13:16] += rng.normal(0, 1.0, (n, 3))
    cam = np.repeat(sc.cam_meas[:1], E, 0)
    n_prop = np.zeros(E, np.int32)
    n_prop[0] = 1
    with BatchFilter(n, **model_kwargs(sc.cfg)) as bf:
        bf.set_noise(sc.Qd[None], sc.Rd[None], sc.sig_om[None])
        bf.set_state(x0, sc.P0[None], sc.u0[None], None)
        bf.keep_consistency()
        bf.run(sc.dt[:1], sc.om_acc[:1], n_prop, cam, np.repeat(sc.notch_meas[:1], E))
        dh, vh = bf.get_dof_history()
        dd, vd = bf.get_dof_history(device=True)
    assert dh.shape == (n, E, 6) and np.isfinite(dh[:, 0]).all()
    assert dh.tobytes() == dd.cpu().numpy().tobytes() and vh.tobytes() == vd.cpu().numpy().tobytes()
    assert len(np.unique(dh[:, 0, 5])) == n  # every row really is its own filter's


def test_config2_calibration_full_size(golden):
    """config 2 calibration: mandala0_mono, 139 updates, 4096 filters, all six DOFs estimated from perturbed values,
    Monte-Carlo noise.  Every filter counted once per epoch, every summary value finite; the per-DOF inflation printed
    with -s (the reference's filter, not the engine: DESIGN.md section 2)"""
    from bench import SEED as BSEED
    from bench import Workload as BenchWorkload
    from dvi_ekf_b200 import BatchFilter
    from dvi_ekf_b200.consistency import summarise_dofs
    from dvi_ekf_b200.sharding import mc_initial_states

    wl = BenchWorkload()
    s = wl.s
    n = 4096
    gt = np.asarray(wl.cfg.gt_imu_dofs, dtype=float)
    with BatchFilter(n, **dict(wl.model, frozen_dofs=(0,) * 6)) as bf:
        bf.set_noise(wl.Qd[None], wl.Rd[None], wl.sig_om[None])
        bf.set_state(mc_initial_states(s.x0, n, 0, BSEED), wl.P0[None], s.u0[None], None)
        bf.keep_consistency()
        bf.run(s.dt, s.om_acc, s.n_prop, s.cam, s.notch, seed=BSEED, imu_noise_std=wl.imu_std, cam_noise_std=wl.cam_std,
               gt_dofs=tuple(gt))
        env = bf.get_dof_envelope()
        dofs, var = bf.get_dof_history()
        nis = bf.get_consistency()[0]
    E = len(s.n_prop)
    assert env.shape == (E, NDOFSUM) and np.array_equal(env[:, 0] + env[:, 1], np.full(E, float(n)))
    ref = envelope(nis, dofs, np.einsum("nei,ij->neij", var, np.eye(6)), gt, 0)
    assert np.array_equal(env[:, COUNTS], ref[:, COUNTS])
    summ = summarise_dofs(env, (0,) * 6)
    for key in ("bias", "rmse", "std", "sigma_filter", "inflation", "anees_dof", "coverage", "err_second_moment", "filter_cov"):
        assert np.isfinite(summ[key]).all(), key
    for e in (0, E - 1):
        print(f"MEASURED config 2 epoch {e}: inflation per DOF {np.array2string(summ['inflation'][e], precision=3)}, "
              f"ANEES per DOF {np.array2string(summ['anees_dof'][e], precision=3)}, 1-sigma coverage "
              f"{np.array2string(summ['coverage'][e, :, 0], precision=3)}, M {summ['count'][e]:.0f}")


def test_simulator_run_sets_the_envelope(tmp_path):
    """Simulator.run(consistency=True) on a short config with all six DOFs estimated sets ``dof_envelope``, the
    summarise_dofs of the run: every filter counted once per epoch"""
    import os

    import yaml

    from dvi_ekf_b200 import Config, Simulator

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    y = yaml.safe_load(open(os.path.join(root, "config.yaml")))
    y["simulation"].update(do_fast_sim=False, frozen_dofs=[0] * 6)
    y["camera"]["total_frames"] = 14
    y["imu"]["interframe_vals"] = 5
    fp = tmp_path / "config.yaml"
    fp.write_text(yaml.safe_dump(y))
    sim = Simulator(Config(str(fp)))
    sim.run(n_filters=16, consistency=True, verbose=False)
    s = sim.dof_envelope
    E = len(sim.streams.n_prop)
    assert s["bias"].shape == (E, 6) and ((s["count"] + s["excluded"]) == 16).all() and (s["count"] > 0).all()
    assert np.isfinite(s["inflation"]).all()
