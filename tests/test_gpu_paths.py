"""The stacked, in-kernel-statistics and export paths of eskf_kernel3 against the oracle.

``eskf_run`` on eskf_kernel3 is sixteen instantiations -- CTA shape F in {28, 16, 8, 4} x MODE (bit 0: export, i.e. FilterTraj
rows or the Jacobian record; bit 1: stacked trajectories) -- and two data paths: the Monte-Carlo streams and the update-MSE
statistics in pre- / post-pass kernels, or everything inside the persistent kernel (``set_prepass_budget(0)``, what a batch
whose buffers do not fit runs).  One small stacked workload goes through all of them: four trajectories of the same length,
13 filters each (a ragged last CTA at every shape), every filter with its own perturbed initial DOFs and all six DOFs
estimated, Monte-Carlo noise, and a different n_prop per trajectory.  The reference is the batch oracle fed the noise the
kernels drew (read back with eskf_noise_dump), computed once; the canonical cell (pre-pass, F = 28, no export) is held to
it and every other cell to the canonical cell's bits."""
import numpy as np
import pytest

from oracle.batch_oracle import BatchOracle
from oracle.eskf_oracle import OracleConfig, euler_xyz_deg
from tests.helpers import Scenario, cov_err, model_kwargs, state_err
from tests.test_gpu_noise import CAM_STD, IMU_STD, _noisy_streams

pytestmark = pytest.mark.gpu

NAMES = ["traj_trans_x", "traj_rot_z", "traj_from_prop", "traj_mandala0_gt"]
FRAMES, IFV, FPT = 8, 10, 13  # 70 IMU steps, 7 epochs; 13 filters per trajectory is a multiple of no CTA shape
N_PROP = np.array([[10, 10, 10, 10, 10, 10, 10],  # regular, even
                   [11, 9, 13, 7, 9, 11, 10],  # odd counts: the covariance role re-orients explicitly before the update
                   [3, 0, 1, 2, 0, 17, 47],  # epochs of 0, 1 and 2 steps: the deferred statistics have to catch up
                   [10, 10, 5, 1, 0, 7, 9]], dtype=np.int32)  # 42 of the 70 steps: the stream outlasts the trajectory
SEED = 2718
GT = np.array([0, 0, 0, 0, 0, 20.0])
SHAPES = (28, 16, 8, 4)
PATHS = ("prepass", "inkernel")
# free-running bounds (70 noisy steps, all DOFs estimated), ~3x the worst value measured on a B200 (1000 W), printed with -s
# as "MEASURED ...": state / covariance / Jacobians on traj_trans_x 1.9e-10 / 1.6e-10 / 7.7e-11
TOL_STATE, TOL_COV, TOL_JAC = 6e-10, 5e-10, 2.5e-10
TOL_STAT = 1e-8  # relative, statistics rows (as tests/test_gpu_stats.py)
# where the oracle's own spread (Workload.reference) is larger, K_SPREAD times that spread is added: the other three
# trajectories measured 8 .. 630 times their spread (spreads 5e-8 .. 8e-3)
K_SPREAD = 2000.0


def _update_mse(x, cam_ref, imu_ref):
    """Filter.calculate_update_mse (Filter.py:397-418) of every row of x [n, 26]"""
    s_cam = np.sum(np.square(cam_ref - np.hstack((x[:, 19:22], euler_xyz_deg(x[:, 22:26])))), axis=1)
    s_imu = np.sum(np.square(np.hstack((x[:, 3:6], euler_xyz_deg(x[:, 6:10]))) - imu_ref), axis=1)
    return (s_cam + s_imu) / 12


class Workload:
    def __init__(self, golden):
        cfg = OracleConfig(max_vals=FRAMES, interframe_vals=IFV, frozen_dofs=(0,) * 6)
        self.scs = [Scenario(golden[nm][:FRAMES], cfg) for nm in NAMES]
        sc0 = self.sc0 = self.scs[0]
        self.T, self.E = len(sc0.dt), len(sc0.n_prop)
        assert all(len(s.dt) == self.T and len(s.n_prop) == self.E for s in self.scs)
        assert all(np.array_equal(s.Qd, sc0.Qd) and np.array_equal(s.Rd, sc0.Rd) and np.array_equal(s.P0, sc0.P0) for s in self.scs)
        self.steps = N_PROP.sum(axis=1)  # steps each trajectory executes
        assert N_PROP.shape == (len(NAMES), self.E) and self.steps.max() == self.T and self.steps[3] < self.T
        self.n = FPT * len(NAMES)
        rng = np.random.default_rng(17)
        self.x0 = np.concatenate([np.repeat(s.x0[None], FPT, 0) for s in self.scs])
        self.x0[:, 10:13] += rng.normal(0.0, np.deg2rad(2.0), (self.n, 3))
        self.x0[:, 13:16] += rng.normal(0.0, 2.0, (self.n, 3))
        self.u0 = np.concatenate([np.repeat(s.u0[None], FPT, 0) for s in self.scs])
        # the references of the error statistics: the noise-free camera pose, and velocity / Euler angles of the IMU reference
        # trajectory at the regular epoch ends
        ends = np.cumsum(sc0.n_prop) - 1
        self.cam_ref = np.array([np.hstack((s.cam_meas[:, :3], euler_xyz_deg(s.cam_meas[:, 3:]))) for s in self.scs])
        self.imu_ref = np.array([s.imu_ref_rows[ends][:, 4:10] for s in self.scs])
        cat = lambda f: np.concatenate([f(s) for s in self.scs])
        self.streams = dict(dt=cat(lambda s: s.dt), om_acc=cat(lambda s: s.om_acc), n_prop=N_PROP.reshape(-1),
                            cam=cat(lambda s: s.cam_meas), notch=cat(lambda s: s.notch_meas),
                            cam_ref=self.cam_ref.reshape(-1, 6), imu_ref=self.imu_ref.reshape(-1, 6))
        self.streams0 = dict(dt=sc0.dt, om_acc=sc0.om_acc, n_prop=N_PROP[0], cam=sc0.cam_meas, notch=sc0.notch_meas,
                             cam_ref=self.cam_ref[0], imu_ref=self.imu_ref[0])
        self.ref = self.reference()

    def reference(self, modulus=0):
        """The batch oracle, one per trajectory, on the noise of the kernels' id rule: global filter g draws the samples of id
        g (g % modulus with a modulus), id 0 is noise free.  Final states, statistics rows, FilterTraj rows (NaN where the
        kernel writes nothing) and Fx / Fi of every filter's last executed step.  With all six DOFs estimated the recursion is
        ill-conditioned on some of these trajectories (the oracle itself moves by up to 1e-7 when its initial state moves by
        1e-15): a twin oracle started 1e-15 away gives every filter's spread, the scale of what the reference determines."""
        from dvi_ekf_b200.engine import NOISE_CAM, NOISE_IMU, noise_samples

        n, T, E = self.n, self.T, self.E
        ids = np.arange(n) % modulus if modulus else np.arange(n)
        zi = noise_samples(SEED, 0, int(ids.max()) + 1, 0, T, NOISE_IMU)
        zc = noise_samples(SEED, 0, int(ids.max()) + 1, 0, E, NOISE_CAM)
        r = dict(x=np.empty((n, 26)), P=np.empty((n, 24, 24)), u=np.empty((n, 6)), R=np.empty((n, 9)),
                 stats=np.zeros((n, 16)), trace=np.full((n, T, 26), np.nan), Fx=np.empty((n, 24, 24)), Fi=np.empty((n, 24, 13)),
                 spread=np.empty((n, 2)))
        for j, sc in enumerate(self.scs):
            rows = slice(j * FPT, (j + 1) * FPT)
            oa, cam, notch = np.empty((FPT, T, 6)), np.empty((FPT, E, 7)), np.empty((FPT, E))
            for i, g in enumerate(ids[rows]):
                oa[i], cam[i], notch[i] = (sc.om_acc, sc.cam_meas, sc.notch_meas) if g == 0 else _noisy_streams(sc, zi[g], zc[g])
            bo = BatchOracle(sc.cfg, self.x0[rows], sc.P0, self.u0[rows], sc.Qd, sc.Rd, sc.sig_om)
            tw = BatchOracle(sc.cfg, self.x0[rows] * (1 + 1e-15), sc.P0, self.u0[rows], sc.Qd, sc.Rd, sc.sig_om)
            k, mse = 0, []
            for e in range(E):
                for _ in range(N_PROP[j, e]):
                    for b in (bo, tw):
                        b.propagate(sc.dt[k], oa[:, k, :3], oa[:, k, 3:])
                    r["trace"][rows, k] = bo.x
                    k += 1
                for b in (bo, tw):
                    b.update(cam[:, e, :3], cam[:, e, 3:], notch[:, e])
                if k > 0:  # FilterTraj.append_updated_states: the update overwrites the row of the epoch's last step
                    r["trace"][rows, k - 1] = bo.x
                mse.append(_update_mse(bo.x, self.cam_ref[j, e], self.imu_ref[j, e]))
            assert k == self.steps[j]
            r["x"][rows], r["P"][rows], r["Fx"][rows], r["Fi"][rows] = bo.x, bo.P, bo.Fx, bo.Fi
            r["u"][rows] = np.hstack((bo.om_old, bo.acc_old))
            r["R"][rows] = bo.R_old.reshape(FPT, 9)
            d2 = np.square(bo.x[:, 10:16] - GT)
            mse = np.array(mse)
            r["stats"][rows, 0:6] = d2
            r["stats"][rows, 6] = d2.mean(axis=1)
            r["stats"][rows, 7] = mse[-1]
            r["stats"][rows, 8] = mse.sum(axis=0)
            r["stats"][rows, 9] = E
            r["stats"][rows, 11] = 1.0
            r["spread"][rows] = [(state_err(tw.x[i], bo.x[i]), cov_err(tw.P[i], bo.P[i], sc.Rd)) for i in range(FPT)]
        return r

    def run(self, F, path, export, lo=0, hi=None, n_traj=4, modulus=0):
        """filters lo..hi-1 of the workload (a shard starting at global id lo) through one eskf_run; n_traj = 1: trajectory 0
        alone (the single-trajectory instantiations)"""
        from dvi_ekf_b200 import BatchFilter

        hi = self.n if hi is None else hi
        n, sc0 = hi - lo, self.sc0
        with BatchFilter(n, **model_kwargs(sc0.cfg)) as bf:
            bf.set_tuning(F)
            if path == "inkernel":
                bf.set_prepass_budget(0)
            bf.set_noise(sc0.Qd[None], sc0.Rd[None], sc0.sig_om[None])
            bf.set_state(self.x0[lo:hi], sc0.P0[None], self.u0[lo:hi], None)
            trace = np.full((n, self.T, 26), np.nan) if export else None
            if export:
                bf.keep_jacobians(True)
            st, sm = bf.run(**(self.streams if n_traj > 1 else self.streams0), n_traj=n_traj,
                            filters_per_traj=FPT if n_traj > 1 else None, seed=SEED, filter_id0=lo, imu_noise_std=IMU_STD,
                            cam_noise_std=CAM_STD, noise_free_filter0=True, noise_id_modulus=modulus, trace=trace, gt_dofs=GT)
            x, P, u, R, status = bf.get_state()
            jac = bf.get_jacobians() if export else None
        return dict(x=x, P=P, u=u, R=R, status=status, stats=st, sum=sm, trace=trace, jac=jac)


@pytest.fixture(scope="module")
def wl(golden):
    return Workload(golden)


@pytest.fixture(scope="module")
def canon(wl):
    return wl.run(28, "prepass", False)


def _against_oracle(out, ref, rd, lo=0):
    """per filter: state (x, u_old, R_old), covariance and relative statistics error of a run against the oracle; the
    statistics rows' counters exactly ([9] updates = E, [10] status 0, [11] healthy)"""
    err = np.zeros((len(out["x"]), 3))
    for i in range(len(out["x"])):
        f = lo + i
        s, sr = out["stats"][i], ref["stats"][f]
        err[i] = (max(state_err(out["x"][i], ref["x"][f]), np.abs(out["u"][i] - ref["u"][f]).max(),
                      np.abs(out["R"][i] - ref["R"][f]).max()),
                  cov_err(out["P"][i], ref["P"][f], rd),
                  max(np.abs(s[0:7] - sr[0:7]).max() / np.abs(sr[0:7]).max(),  # DOF terms, norm-wise like the state
                      abs(s[7] - sr[7]) / abs(sr[7]), abs(s[8] - sr[8]) / abs(sr[8])))
        assert np.array_equal(s[9:], sr[9:]), (f, s[9:12])
    assert np.all(out["status"] == 0)
    return err


def _assert_bounded(what, err, tols, spread):
    """err [n, m] <= tol + K_SPREAD * spread (the oracle's own spread of each filter: [n] or [n, m]); prints the worst error and the worst
    ratio to the spread per trajectory"""
    spread = spread if spread.ndim == 2 else spread[:, None]
    bound = np.asarray(tols)[None, :] + K_SPREAD * spread
    for j in range(len(err) // FPT + (len(err) % FPT > 0)):
        rows = slice(j * FPT, (j + 1) * FPT)
        ratio = (err[rows] / np.maximum(spread[rows], 1e-300)).max()
        print(f"MEASURED {what} {NAMES[j]}: worst {' / '.join(f'{v:.2e}' for v in err[rows].max(axis=0))}, "
              f"oracle spread {spread[rows].max():.2e}, worst ratio to the spread {ratio:.1f}")
    assert (err <= bound).all(), (what, np.argwhere(err > bound)[:5])


def _check_sum(out):
    """stats_sum: the masked sum of the rows (every filter healthy here)"""
    st, sm = out["stats"], out["sum"]
    n = len(st)
    assert np.allclose(sm[:10], st[:, :10].sum(axis=0), rtol=1e-12, atol=0), (sm[:10], st[:, :10].sum(axis=0))
    assert sm[10] == 0 and sm[11] == n and sm[12] == 0


def _check_export(wl, out, lo=0):
    """FilterTraj rows against the oracle's per-step states, untouched rows past the trajectory's steps, and Fx / Fi of the
    filter's last executed step.  Returns the worst row and Jacobian error per filter."""
    ref = wl.ref
    Fx, Fi = out["jac"]
    err = np.zeros((len(out["x"]), 2))
    for i in range(len(out["x"])):
        f = lo + i
        steps = wl.steps[f // FPT]
        tr = out["trace"][i]
        assert np.isnan(tr[steps:]).all(), (f, steps)  # the caller's fill survives where the trajectory has no step
        assert np.isfinite(tr[:steps]).all(), f
        err[i, 0] = max(state_err(tr[k], ref["trace"][f, k]) for k in range(steps))
        err[i, 1] = max(np.abs(Fx[i] - ref["Fx"][f]).max() / max(1.0, np.abs(ref["Fx"][f]).max()),
                        np.abs(Fi[i] - ref["Fi"][f]).max() / max(1.0, np.abs(ref["Fi"][f]).max()))
    return err


def _assert_same_bits(out, base, rows=slice(None), what=""):
    for key in ("x", "P", "u", "R", "status", "stats"):
        assert out[key].tobytes() == base[key][rows].tobytes(), (what, key)


def test_canonical_cell_matches_oracle(wl, canon):
    """pre-pass, F = 28, no export (MODE 2): every filter's x, P, u_old, R_old and statistics row against the oracle"""
    err = _against_oracle(canon, wl.ref, wl.sc0.Rd)
    _assert_bounded("stacked run vs oracle, state / P / statistics", err, (TOL_STATE, TOL_COV, TOL_STAT), wl.ref["spread"][:, [0, 1, 0]])
    _check_sum(canon)
    # the filters really saw different inputs: noise, initial DOFs, trajectories
    x = canon["x"]
    assert np.abs(x[1] - x[2]).max() > 1e-6 and np.abs(x[FPT] - x[0]).max() > 1e-3


@pytest.mark.parametrize("export", [False, True], ids=["plain", "export"])
@pytest.mark.parametrize("F", SHAPES)
@pytest.mark.parametrize("path", PATHS)
def test_stacked_cell_is_bit_identical_to_canonical(wl, canon, path, F, export):
    """pre-pass / in-kernel x every CTA shape x export off / on (MODE 2 and MODE 3): the same bits as the canonical cell in
    x, P, u_old, R_old, status, the statistics rows and stats_sum; in export mode the FilterTraj rows and the Jacobians of
    every filter's last executed step against the oracle (trajectory 3 stops 28 steps before the end of the stream)"""
    out = wl.run(F, path, export)
    _assert_same_bits(out, canon, what=(path, F, export))
    assert out["sum"].tobytes() == canon["sum"].tobytes()
    if export:
        _assert_bounded(f"stacked export {path} F={F}, FilterTraj rows / Jacobians", _check_export(wl, out), (TOL_STATE, TOL_JAC),
                        wl.ref["spread"][:, 0])


@pytest.mark.parametrize("export", [False, True], ids=["plain", "export"])
@pytest.mark.parametrize("F", (28, 4))
@pytest.mark.parametrize("path", PATHS)
def test_single_trajectory_cell_is_bit_identical_to_canonical(wl, canon, path, F, export):
    """trajectory 0 alone (MODE 0 and MODE 1): its 13 filters with the bits they have in the stacked canonical cell"""
    out = wl.run(F, path, export, hi=FPT, n_traj=1)
    _assert_same_bits(out, canon, rows=slice(0, FPT), what=(path, F, export))
    _check_sum(out)
    if export:
        _assert_bounded(f"single-trajectory export {path} F={F}, FilterTraj rows / Jacobians", _check_export(wl, out),
                        (TOL_STATE, TOL_JAC), wl.ref["spread"][:FPT, 0])


@pytest.mark.parametrize("F", SHAPES)
def test_partially_covered_last_trajectory(wl, canon, F):
    """N = 2 fpt + 5: the third trajectory holds only 5 of its 13 filters (the grid launches no CTA for the missing 8):
    the rows are those of the same filters in the full run"""
    n = 2 * FPT + 5
    out = wl.run(F, "prepass", False, hi=n)
    _assert_same_bits(out, canon, rows=slice(0, n), what=F)
    _check_sum(out)


@pytest.mark.parametrize("path", PATHS)
def test_shard_at_a_trajectory_boundary(wl, canon, path):
    """filter_id0 = fpt: trajectories 1..3 of the streams, global noise ids 13..51 -- the rows of the full run"""
    out = wl.run(28, path, False, lo=FPT)
    _assert_same_bits(out, canon, rows=slice(FPT, None), what=path)
    _check_sum(out)


def test_noise_id_modulus_on_the_stacked_paths(wl):
    """noise_id_modulus = 3 (common random numbers: filter g draws the noise of id g % 3, so every third filter is noise free)
    on the stacked pre-pass and in-kernel paths: both give the same bits, and the oracle fed the ids g % 3 agrees"""
    ref = wl.reference(modulus=3)
    pp = wl.run(28, "prepass", False, modulus=3)
    ik = wl.run(8, "inkernel", False, modulus=3)
    _assert_same_bits(ik, pp, what="modulus")
    assert ik["sum"].tobytes() == pp["sum"].tobytes()
    _assert_bounded("noise_id_modulus 3 vs oracle, state / P / statistics", _against_oracle(pp, ref, wl.sc0.Rd),
                    (TOL_STATE, TOL_COV, TOL_STAT), ref["spread"][:, [0, 1, 0]])
    assert np.abs(ref["x"][4:] - wl.ref["x"][4:]).max() > 1e-6  # the ids really changed the noise
