"""eskf_run against the oracle at orientations, residual angles and frame timings the packaged trajectories never reach
(the host replay of the same scenarios: tests/test_rotated_host.py).

* All 37 turned worlds of tests/helpers.py (world_rotations / RotatedScenario) in ONE stacked launch, 5 filters each (a
  ragged CTA at every shape), every filter with a slightly moved initial position and velocity: final x and P, every
  FilterTraj row (quaternions compared with their sign: the reference forces w >= 0) and statistics rows [6..9] with the
  update MSE against the turned references, whose Euler angles wrap (roll-wrap) and come within 0.06 deg of gimbal lock
  (eight cube rotations).  Pre-pass and in-kernel statistics, CTA shapes 28 and 4: bit-identical.  Variant 1 and the
  Monte-Carlo path on subsets.
* eskf_update with camera measurements 180 deg from q_cam: ESKF_STATUS_ASIN_DOMAIN, and the same inside eskf_run.
* eskf_prepass on jittered frame stamps, and eskf_run on its device-resident streams."""
import numpy as np
import pytest

from oracle.batch_oracle import BatchOracle
from tests.helpers import RotatedScenario, Scenario, cov_err, mandala_scenario, model_kwargs, state_err, world_rotations
from tests.test_gpu_noise import CAM_STD, IMU_STD, _noisy_streams
from tests.test_gpu_paths import _update_mse
from tests.test_rotated_host import ULP1, asin_domain_inputs, jittered_camera, oracle_update, residual_norms

pytestmark = pytest.mark.gpu

FRAMES, IFV, FPT = 21, 10, 5  # 200 IMU steps, 20 epochs per world
SEED = 1618
GT = np.array([0, 0, 0, 0, 0, 20.0])
# bounds at ~3x the worst value measured on an NVIDIA B200 (power limit 1000 W), printed with -s as "MEASURED ...": state 6.9e-11
# (Monte-Carlo, y150 .. cube13), covariance 8.6e-12 (Monte-Carlo), statistics 2.7e-9 (cube13: pitch within 0.06 deg of
# gimbal lock, where roll and yaw move 1 / cos(pitch) times faster than the state), FilterTraj rows 1.8e-10 (random7).  The
# oracle's own spread (its response to a one-ulp change of the initial state, a twin oracle) is printed beside them: 1e-12 ..
# 1.1e-11 for the state in every world.
TOL_STATE, TOL_COV, TOL_STAT, TOL_TRACE = 2e-10, 3e-11, 8e-9, 5.5e-10
NOISY = ["x-60", "y150", "z150", "roll-wrap", "cube13"]


class World:
    """The stacked workload and its batch-oracle reference (one row block of FPT filters per world)."""

    def __init__(self, golden, names=None, noise=False):
        sc = mandala_scenario(golden, n_frames=FRAMES, ifv=IFV)
        allw = world_rotations(sc)
        self.names = list(allw) if names is None else names
        self.rs = [RotatedScenario(sc, allw[nm], nm) for nm in self.names]
        self.sc, self.noise = sc, noise
        self.T, self.E, self.nt = len(sc.dt), len(sc.n_prop), len(self.names)
        self.n = FPT * self.nt
        rng = np.random.default_rng(31)
        self.x0 = np.concatenate([np.repeat(r.x0[None], FPT, 0) for r in self.rs])
        self.x0[:, 0:3] += rng.normal(0.0, 1e-3, (self.n, 3))
        self.x0[:, 3:6] += rng.normal(0.0, 1e-4, (self.n, 3))
        cat = lambda f: np.concatenate([f(r) for r in self.rs])
        self.streams = dict(dt=np.tile(sc.dt, self.nt), om_acc=np.tile(sc.om_acc, (self.nt, 1)), n_prop=np.tile(sc.n_prop, self.nt),
                            cam=cat(lambda r: r.cam_meas), notch=cat(lambda r: r.notch_meas), cam_ref=cat(lambda r: r.cam_ref),
                            imu_ref=cat(lambda r: r.imu_ref))
        self.ref = self.reference()

    def reference(self):
        from dvi_ekf_b200.engine import NOISE_CAM, NOISE_IMU, noise_samples

        n, T, E, sc = self.n, self.T, self.E, self.sc
        oa = np.broadcast_to(sc.om_acc, (n, T, 6)).copy()
        cam = np.repeat(np.stack([r.cam_meas for r in self.rs]), FPT, 0)
        notch = np.repeat(np.stack([r.notch_meas for r in self.rs]), FPT, 0)
        if self.noise:
            zi = noise_samples(SEED, 0, n, 0, T, NOISE_IMU)
            zc = noise_samples(SEED, 0, n, 0, E, NOISE_CAM)
            for g in range(1, n):  # global filter 0 is noise free
                oa[g], cam[g], notch[g] = _noisy_streams(self.rs[g // FPT], zi[g], zc[g])
        cam_ref = np.repeat(np.stack([r.cam_ref for r in self.rs]), FPT, 0)
        imu_ref = np.repeat(np.stack([r.imu_ref for r in self.rs]), FPT, 0)
        bo = BatchOracle(sc.cfg, self.x0, sc.P0, sc.u0, sc.Qd, sc.Rd, sc.sig_om)
        tw = BatchOracle(sc.cfg, self.x0 * (1 + ULP1), sc.P0, sc.u0, sc.Qd, sc.Rd, sc.sig_om)
        trace = np.empty((n, T, 26))
        k, mse = 0, []
        for e in range(E):
            for _ in range(sc.n_prop[e]):
                for b in (bo, tw):
                    b.propagate(sc.dt[k], oa[:, k, :3], oa[:, k, 3:])
                trace[:, k] = bo.x
                k += 1
            for b in (bo, tw):
                b.update(cam[:, e, :3], cam[:, e, 3:], notch[:, e])
            trace[:, k - 1] = bo.x
            mse.append(_update_mse(bo.x, cam_ref[:, e], imu_ref[:, e]))
        mse = np.array(mse)
        d2 = np.square(bo.x[:, 10:16] - GT)
        stats = np.stack([d2.mean(axis=1), mse[-1], mse.sum(axis=0), np.full(n, float(E))], -1)
        spread = np.array([(state_err(tw.x[i], bo.x[i]), cov_err(tw.P[i], bo.P[i], sc.Rd)) for i in range(n)])
        return dict(x=bo.x, P=bo.P, trace=trace, stats=stats, spread=spread)

    def run(self, F=28, path="prepass", trace=False):
        from dvi_ekf_b200 import BatchFilter

        sc = self.sc
        with BatchFilter(self.n, **model_kwargs(sc.cfg)) as bf:
            bf.set_tuning(F)
            if path == "inkernel":
                bf.set_prepass_budget(0)
            bf.set_noise(sc.Qd[None], sc.Rd[None], sc.sig_om[None])
            bf.set_state(self.x0, sc.P0[None], sc.u0[None], None)
            tr = np.full((self.n, self.T, 26), np.nan) if trace else None
            noise = dict(seed=SEED, imu_noise_std=IMU_STD, cam_noise_std=CAM_STD) if self.noise else {}
            st, sm = bf.run(**self.streams, n_traj=self.nt, filters_per_traj=FPT, trace=tr, gt_dofs=GT, **noise)
            x, P, u, R, status = bf.get_state()
        return dict(x=x, P=P, u=u, R=R, status=status, stats=st, sum=sm, trace=tr)

    def errors(self, out):
        """per filter: state, covariance, statistics [6..8] (relative), FilterTraj rows (or 0 without trace)"""
        ref, err = self.ref, np.zeros((self.n, 4))
        assert np.all(out["status"] == 0)
        assert np.array_equal(out["stats"][:, 9], ref["stats"][:, 3])
        for i in range(self.n):
            s, sr = out["stats"][i, 6:9], ref["stats"][i, :3]
            err[i, 0] = state_err(out["x"][i], ref["x"][i])
            err[i, 1] = cov_err(out["P"][i], ref["P"][i], self.sc.Rd)
            err[i, 2] = (np.abs(s - sr) / np.abs(sr)).max()
            if out["trace"] is not None:
                err[i, 3] = max(state_err(out["trace"][i, k], ref["trace"][i, k]) for k in range(self.T))
        return err

    def check(self, what, err, tols):
        spread = self.ref["spread"][:, [0, 1, 0, 0]]
        bound = np.asarray(tols)[None, :]
        for j, nm in enumerate(self.names):
            rows = slice(j * FPT, (j + 1) * FPT)
            print(f"MEASURED {what} {nm}: state / P / stats / trace {' / '.join(f'{v:.1e}' for v in err[rows].max(axis=0))}, "
                  f"oracle spread {spread[rows].max():.1e}")
        print(f"MEASURED {what} worst over worlds: {' / '.join(f'{v:.2e}' for v in err.max(axis=0))}")
        bad = np.argwhere(err > bound)
        assert not len(bad), (what, [(self.names[i // FPT], i, c, err[i, c], bound[0, c]) for i, c in bad[:6]])


@pytest.fixture(scope="module")
def world(golden):
    return World(golden)


@pytest.fixture(scope="module")
def canon(world):
    return world.run(28, "prepass", trace=True)


def test_turned_worlds_stacked_run_matches_oracle(world, canon):
    """one stacked launch of all 37 worlds, pre-pass statistics, F = 28, FilterTraj rows: x, P, statistics and every row"""
    world.check("turned worlds, stacked", world.errors(canon), (TOL_STATE, TOL_COV, TOL_STAT, TOL_TRACE))
    assert np.all(np.isfinite(canon["trace"]))
    q = canon["trace"][:, :, 6:10]
    assert (q[:, :, 3] >= 0).all() and (canon["trace"][:, :, 25] >= 0).all()  # the w >= 0 convention, row by row


@pytest.mark.parametrize("path,F,trace", [("inkernel", 28, True), ("prepass", 4, False), ("inkernel", 4, False)])
def test_turned_worlds_paths_and_shapes_are_bit_identical(world, canon, path, F, trace):
    """in-kernel statistics (set_prepass_budget(0)) and CTA shape 4: the canonical run's bits, statistics rows included"""
    out = world.run(F, path, trace=trace)
    for key in ("x", "P", "u", "R", "status", "stats", "sum") + (("trace",) if trace else ()):
        assert out[key].tobytes() == canon[key].tobytes(), (path, F, key)


def test_turned_worlds_variant1(golden):
    """the first kernel (eskf_kernel) on the worlds that leave Markley branch 0 / 3 and wrap, one launch per world"""
    from dvi_ekf_b200 import BatchFilter

    names = ["x-60", "y150", "z150", "roll-wrap", "cube12"]
    w = World(golden, names)
    err = np.zeros((w.n, 4))
    for j in range(len(names)):
        rows = slice(j * FPT, (j + 1) * FPT)
        sc, r = w.sc, w.rs[j]
        with BatchFilter(FPT, variant=1, **model_kwargs(sc.cfg)) as bf:
            bf.set_noise(sc.Qd[None], sc.Rd[None], sc.sig_om[None])
            bf.set_state(w.x0[rows], sc.P0[None], sc.u0[None], None)
            st, _ = bf.run(sc.dt, sc.om_acc, sc.n_prop, r.cam_meas, r.notch_meas, cam_ref=r.cam_ref, imu_ref=r.imu_ref, gt_dofs=GT)
            x, P, _, _, status = bf.get_state()
        assert np.all(status == 0)
        for i in range(FPT):
            f = j * FPT + i
            s, sr = st[i, 6:9], w.ref["stats"][f, :3]
            err[f, :3] = (state_err(x[i], w.ref["x"][f]), cov_err(P[i], w.ref["P"][f], sc.Rd), (np.abs(s - sr) / np.abs(sr)).max())
    w.check("turned worlds, variant 1", err, (TOL_STATE, TOL_COV, TOL_STAT, 0.0))


def test_turned_worlds_monte_carlo(golden):
    """five worlds stacked with Monte-Carlo noise on; the oracle fed the noise the kernels drew (eskf_noise_dump)"""
    w = World(golden, NOISY, noise=True)
    out = w.run(28, "prepass")
    w.check("turned worlds, Monte-Carlo", w.errors(out), (TOL_STATE, TOL_COV, TOL_STAT, 0.0))
    assert np.abs(out["x"][1] - out["x"][2]).max() > 1e-6  # the filters saw different noise


# ---- residual at 180 deg ------------------------------------------------------------------------------------------------


def test_asin_domain_eskf_update(golden):
    """4096 filters, one eskf_update: 2048 measurements exactly 180 deg from q_cam about seeded axes, 2048 at 90 .. 179.9 deg.
    A filter with ESKF_STATUS_ASIN_DOMAIN has an oracle |v| within 4 ulp of 1, and at least one is flagged; its status word
    is ESKF_STATUS_ASIN_DOMAIN | ESKF_STATUS_UPDATE_SKIPPED (include/eskf.h), its state and P are the prior and its K is 0.
    The band's filters are all applied and match the oracle at 1e-9.  (Unflagged 180-deg updates are not compared: the
    residual's direction there is the sign of a rounding error, tests/test_rotated_host.py.)"""
    from dvi_ekf_b200 import BatchFilter
    from dvi_ekf_b200._lib import STATUS_ASIN_DOMAIN, STATUS_UPDATE_SKIPPED

    sc = mandala_scenario(golden, n_frames=3, ifv=1)
    a = asin_domain_inputs(sc.cfg, 2048, 97)
    b = asin_domain_inputs(sc.cfg, 2048, 98, band=True)
    xs, Ps, us, cam = (np.concatenate(v) for v in zip(a, b))
    n = len(xs)
    with BatchFilter(n, **model_kwargs(sc.cfg)) as bf:
        bf.set_noise(sc.Qd[None], sc.Rd[None], sc.sig_om[None])
        bf.set_state(xs, Ps, us, None)
        K = bf.update(cam, np.zeros(n), want_gain=True)
        x, P, _, _, status = bf.get_state()
    flagged = (status & STATUS_ASIN_DOMAIN) != 0
    assert flagged.any() and not flagged[2048:].any()
    assert np.all(status[flagged] == STATUS_ASIN_DOMAIN | STATUS_UPDATE_SKIPPED) and np.all(status[~flagged] == 0)
    assert np.array_equal(x[flagged], xs[flagged]) and np.array_equal(P[flagged], Ps[flagged]) and not K[flagged].any()
    for i in np.flatnonzero(flagged):
        nv_o, _ = residual_norms(xs[i, 22:26], cam[i, 3:])
        assert nv_o >= 1.0 - 4 * ULP1 / 2, (i, nv_o)
    worst = 0.0
    for i in range(2048, n):
        ref = oracle_update(sc.cfg, sc.probe, xs[i], Ps[i], us[i], cam[i])
        assert ref is not None
        worst = max(worst, state_err(x[i], ref[0]), cov_err(P[i], ref[1], sc.Rd))
    print(f"MEASURED asin domain on the device: {int(flagged.sum())} of 2048 180-deg filters flagged; band vs oracle {worst:.2e}")
    assert worst < 1e-9


def test_asin_domain_inside_eskf_run(golden):
    """the 180-deg inputs as 2048 stacked one-filter trajectories, one epoch of 0 IMU steps: a flagged filter has status 3,
    no applied update (row [9] = 0), is counted by stats_sum[10] and not by [11], and its NIS is NaN; an unflagged one has
    status 0 and a finite NIS"""
    from dvi_ekf_b200 import BatchFilter
    from dvi_ekf_b200._lib import STATUS_ASIN_DOMAIN

    sc = mandala_scenario(golden, n_frames=3, ifv=1)
    xs, Ps, us, cam = asin_domain_inputs(sc.cfg, 2048, 97)
    n = len(xs)
    with BatchFilter(n, **model_kwargs(sc.cfg)) as bf:
        bf.set_noise(sc.Qd[None], sc.Rd[None], sc.sig_om[None])
        bf.set_state(xs, Ps, us, None)
        bf.keep_consistency(True)
        st, sm = bf.run(np.full(n, 0.1), np.zeros((n, 6)), np.zeros(n, dtype=np.int32), cam, np.zeros(n),
                        cam_ref=np.zeros((n, 6)), imu_ref=np.zeros((n, 6)), n_traj=n, filters_per_traj=1, gt_dofs=GT)
        x, P, _, _, status = bf.get_state()
        nis = bf.get_consistency()[0]
    flagged = (status & STATUS_ASIN_DOMAIN) != 0
    print(f"MEASURED asin domain inside eskf_run: {int(flagged.sum())} of {n} flagged")
    assert flagged.any() and np.all(status[flagged] == 3) and np.all(status[~flagged] == 0)
    for i in np.flatnonzero(flagged):
        assert residual_norms(xs[i, 22:26], cam[i, 3:])[0] >= 1.0 - 2 * ULP1
    assert np.array_equal(x[flagged], xs[flagged]) and np.array_equal(P[flagged], Ps[flagged])
    assert np.all(st[flagged, 9] == 0) and np.all(st[~flagged, 9] == 1) and np.all(st[flagged, 10] == 3)
    assert sm[10] == flagged.sum() and sm[11] == (~flagged & np.isfinite(st[:, :10]).all(axis=1)).sum()
    assert np.isnan(nis[flagged, 0]).all() and np.isfinite(nis[~flagged, 0]).all()


# ---- irregular frame stamps ---------------------------------------------------------------------------------------------


@pytest.mark.parametrize("world_name", [None, "roll-wrap", "y150"])
def test_irregular_stamps_gpu_prepass(golden, world_name):
    """eskf_prepass on jittered stamps (an epoch of 0 IMU steps, a 3x gap), in the plain and two turned worlds (the camera's
    Euler angles wrap inside the gradient in roll-wrap): n_prop exactly that of the oracle and of the product's numpy
    pre-pass, the other streams within the bounds of tests/test_gpu_prepass.py"""
    from dvi_ekf_b200.camera import Camera, build_streams
    from dvi_ekf_b200.prepass import build_streams_gpu
    from oracle.eskf_oracle import OracleConfig

    G = None if world_name is None else world_rotations(mandala_scenario(golden, n_frames=30, ifv=10))[world_name]
    t, xyz, q = jittered_camera(golden, G=G)
    sc = Scenario(np.hstack((t[:, None], xyz, q)), OracleConfig(max_vals=len(t), interframe_vals=IFV))
    host = build_streams(Camera(t, xyz, q, scale=10.0), IFV, sc.cfg.length, sc.cfg.angle)
    dev = build_streams_gpu(t, xyz, q, IFV, sc.cfg.length, sc.cfg.angle, scale=10.0)
    T = len(host.dt)
    assert dev.n_steps == T == len(sc.dt)
    npd = dev.n_prop.cpu().numpy()
    assert np.array_equal(npd, host.n_prop) and np.array_equal(npd, sc.n_prop) and (npd == 0).any()

    def close(a, b, tol, what):
        a, b = np.asarray(a), np.asarray(b)
        err = np.abs(a - b).max() / max(np.abs(b).max(), 1e-12)
        assert err < tol, (what, err)

    g = lambda v: v.cpu().numpy()
    close(g(dev.dt)[:T], host.dt, 1e-12, "dt")
    close(g(dev.om_acc)[:T, :3], host.om_acc[:, :3], 1e-10, "om")
    close(g(dev.om_acc)[:T, 3:], host.om_acc[:, 3:], 1e-10, "acc")
    close(g(dev.om_acc)[:T], sc.om_acc, 1e-10, "om_acc vs oracle")
    close(g(dev.cam), host.cam, 1e-15, "cam")
    close(g(dev.cam_ref), host.cam_ref, 1e-12, "cam_ref")
    close(g(dev.imu_ref), host.imu_ref, 1e-10, "imu_ref")
    close(g(dev.imu_ref_rows)[:T], sc.imu_ref_rows, 1e-10, "imu_ref_rows")
    close(g(dev.x0), sc.x0, 1e-12, "x0")
    close(g(dev.u0), sc.u0, 1e-10, "u0")


def test_irregular_stamps_run_on_device_streams(golden):
    """jittered stamps -> eskf_prepass -> eskf_run without a host copy of the streams, against the oracle on its own streams
    (varying dt, an epoch of 0 steps, a 3x gap)"""
    import torch

    from dvi_ekf_b200 import BatchFilter
    from dvi_ekf_b200.prepass import build_streams_gpu
    from oracle.eskf_oracle import OracleConfig

    t, xyz, q = jittered_camera(golden)
    sc = Scenario(np.hstack((t[:, None], xyz, q)), OracleConfig(max_vals=len(t), interframe_vals=IFV))
    ds = build_streams_gpu(t, xyz, q, IFV, sc.cfg.length, sc.cfg.angle, scale=10.0)
    T = ds.n_steps
    dd = lambda v: torch.tensor(np.ascontiguousarray(v), dtype=torch.float64, device=ds.dt.device)
    with BatchFilter(4, **model_kwargs(sc.cfg)) as bf:
        bf.set_noise(sc.Qd[None], sc.Rd[None], sc.sig_om[None])
        bf.set_state(ds.x0[None].contiguous(), dd(sc.P0[None]), ds.u0[None].contiguous(), None)
        bf.run(ds.dt[:T].contiguous(), ds.om_acc[:T].contiguous(), ds.n_prop, ds.cam, ds.notch, cam_ref=ds.cam_ref,
               imu_ref=ds.imu_ref, stats_on_device=True)
        xg, Pg, _, _, st = bf.get_state()
    kf = sc.new_oracle()
    k = 0
    for e in range(len(sc.n_prop)):
        for _ in range(sc.n_prop[e]):
            kf.propagate(sc.dt[k], sc.om_acc[k, :3], sc.om_acc[k, 3:])
            k += 1
        assert kf.update(sc.cam_meas[e, :3], sc.cam_meas[e, 3:], sc.notch_meas[e]) is not None
    xr, Pr, _, _ = kf.get_vectors()
    assert np.all(st == 0)
    ws, wP = state_err(xg[0], xr), cov_err(Pg[0], Pr, sc.Rd)
    print(f"MEASURED jittered stamps on device-resident streams ({T} steps): state {ws:.2e} P {wP:.2e}")
    assert ws < 8e-12 and wP < 1.5e-13  # measured 2.5e-12 / 4.2e-14 (B200, 1000 W)
