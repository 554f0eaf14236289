"""``Filter`` / ``Simulator``: the reference's Python interface in front of the CUDA engine.

Same names, argument meaning and error behaviour as dvi_ekf/filter/Filter.py:28-476 and
dvi_ekf/filter/Simulator.py:24-252 for the hot path (plots, the differential-evolution tuner and the
file-based IMU generator are out of scope).  A single ``Filter`` is a batch of one; ``Simulator.run``
executes all ``num_kf_runs`` runs as ONE batched launch (``Filter.run`` for every Monte-Carlo seed).
"""
from __future__ import annotations

import os
from dataclasses import dataclass
from typing import List, Optional, Tuple

import numpy as np

from . import rotations as rot
from .camera import Camera, Streams, build_streams, load_notch, load_trajectory
from .config import Config
from .consistency import NIS_DIM, candidate_objective, summarise_consistency, summarise_dofs
from .engine import BatchFilter
from .probe import GT_IMU_DOFS
from .sharding import summarise_stats


@dataclass(frozen=True)
class State:
    """dvi_ekf/filter/state.py:11-29."""

    SIZE = 26
    p: np.ndarray
    v: np.ndarray
    q: rot.Quaternion
    dofs: np.ndarray
    notch_dofs: np.ndarray
    p_cam: np.ndarray
    q_cam: rot.Quaternion

    @staticmethod
    def from_vector(x) -> "State":
        x = np.asarray(x, dtype=float)
        return State(x[0:3].copy(), x[3:6].copy(), rot.Quaternion(x[6:10]), x[10:16].copy(), x[16:19].copy(),
                     x[19:22].copy(), rot.Quaternion(x[22:26]))

    def as_vector(self) -> np.ndarray:
        return np.hstack((self.p, self.v, self.q.xyzw, self.dofs, self.notch_dofs, self.p_cam, self.q_cam.xyzw))


@dataclass(frozen=True)
class VisualMeasurementPoint:
    """dvi_ekf/models/measurement_point/VisualMeasurementPoint.py:11-31 (q is NOT normalised)."""

    t: float
    x: float
    y: float
    z: float
    q: rot.Quaternion

    @property
    def pos(self):
        return np.array([self.x, self.y, self.z])

    @property
    def vec(self):
        return np.hstack((self.pos, self.q.xyzw))


class FilterTraj:
    """dvi_ekf/models/trajectory/FilterTraj.py: 30 labelled columns, one row per IMU step, the row of an
    update instant overwritten by the updated state."""

    labels_imu = ["x", "y", "z", "vx", "vy", "vz", "rx", "ry", "rz", "qw", "qx", "qy", "qz"]
    labels_imu_dofs = ["dof1", "dof2", "dof3", "dof4", "dof5", "dof6"]
    labels_camera = ["xc", "yc", "zc", "rx_degc", "ry_degc", "rz_degc", "qwc", "qxc", "qyc", "qzc"]
    labels = ["t", *labels_imu, *labels_imu_dofs, *labels_camera]

    def __init__(self, name="kf"):
        self.name = name
        self.reset()

    def reset(self):
        self.rows: List[np.ndarray] = []

    @staticmethod
    def row(t, s: State) -> np.ndarray:
        """_get_euler_measurement_array (FilterTraj.py:12-32)."""
        return np.array([t, *s.p, *s.v, *s.q.euler_xyz_deg, *s.q.wxyz, *np.rad2deg(s.dofs[:3]), *s.dofs[3:], *s.p_cam,
                         *s.q_cam.euler_xyz_deg, *s.q_cam.wxyz])

    def append_propagated_states(self, t, state):
        self.rows.append(self.row(t, state))

    def append_updated_states(self, t, state):
        self.rows[-1] = self.row(t, state)

    def __getattr__(self, label):
        if label in FilterTraj.labels:
            return [r[FilterTraj.labels.index(label)] for r in self.rows]
        raise AttributeError(label)

    @property
    def num_values(self):
        return len(self.rows)


def save_trajectory(rows, filename):
    """tools/files.py:68-82: ``%.6f`` time, `` %.9f`` values, trailing space."""
    with open(filename, "w+") as f:
        for r in rows:
            f.write(f"{r[0]:.6f}" + "".join(f" {v:.9f}" for v in r[1:]) + " \n")


class _ImuView:
    """the attributes of dvi_ekf.models.Imu.Imu that Filter users touch"""

    def __init__(self, sim):
        self.stdev_na = np.array(sim.config.imu.stdev_accel)
        self.stdev_nom = np.array(sim.config.imu.stdev_omega)
        self.cam = sim.camera_interp
        self.ref_rows: List[np.ndarray] = []
        self.om = sim.streams.u0[:3].copy()
        self.acc = sim.streams.u0[3:].copy()

    class _Ref:
        labels = ["t", "x", "y", "z", "vx", "vy", "vz", "rx", "ry", "rz", "qw", "qx", "qy", "qz"]

    @property
    def ref(self):
        r = _ImuView._Ref()
        r.rows = self.ref_rows
        return r


class Filter:
    """Error-State Kalman Filter (dvi_ekf/filter/Filter.py:28).  State and covariance live on the GPU."""

    def __init__(self, sim: "Simulator"):
        assert sim.config.dofs_updated
        self.run_id: Optional[int] = None
        self._config = sim.config
        self._sim = sim
        self._dt = 0.0
        self.show_progress = True
        self.num_meas, self.num_noise = 7, 13
        self._frozen_dofs = [bool(fr) for fr in self._config.frozen_dofs]
        self.imu = _ImuView(sim)
        self.stdev_na, self.stdev_nom = self.imu.stdev_na, self.imu.stdev_nom
        self._engine = BatchFilter(1, scope_length=self._config.model.length, cam_angle_rad=self._config.model.angle,
                                   frozen_dofs=self._config.frozen_dofs, zero_frozen_dofs=not sim.legacy_golden,
                                   device=sim.device)
        self.H = np.zeros([self.num_meas, 24])
        self.H[0:6, 18:24] = np.eye(6)
        self.H[6, 15] = 1
        self._engine.keep_jacobians(True)  # Fx / Fi of the last IMU step are read out on demand (properties below)
        self._propagated = False
        self.traj = FilterTraj("kf")
        self.update_noise_matrices()  # with _dt = 0: Q[0:6] = 0 (Filter.py:40,68-72)
        self._engine.set_state(sim.x0.as_vector()[None], sim.cov0[None], sim.streams.u0[None], None)
        self.traj.append_propagated_states(self._config.min_t, sim.x0)
        self.mse = 0
        self.update_mse = 0

    # ---- state views -------------------------------------------------------
    @property
    def Fx(self):
        """Filter.py:249-259: the error-state transition matrix of the last propagate (None before the first one, as in
        the reference, which creates the attribute there)."""
        return self._engine.get_jacobians()[0][0] if self._propagated else None

    @property
    def Fi(self):
        """Filter.py:261-268: the noise Jacobian of the last propagate."""
        return self._engine.get_jacobians()[1][0] if self._propagated else None

    @property
    def _states(self) -> State:
        return State.from_vector(self._engine.get_state()[0][0])

    @property
    def _P(self) -> np.ndarray:
        return self._engine.get_state()[1][0]

    @property
    def om_old(self):
        return self._engine.get_state()[2][0, :3]

    @property
    def acc_old(self):
        return self._engine.get_state()[2][0, 3:]

    @property
    def R_WB_old(self):
        return self._engine.get_state()[3][0].reshape(3, 3)

    # ---- Filter.py:95-117 --------------------------------------------------------
    def reset(self, x0: State, cov0, notch0=None):
        self._dt = 0.0
        self._engine.set_state(x0.as_vector()[None], np.asarray(cov0, dtype=float)[None], self._sim.streams.u0[None], None)
        self.imu.ref_rows = []
        self.traj.reset()
        self.traj.append_propagated_states(self._config.min_t, x0)
        self.mse = 0

    def update_noise_matrices(self):
        Q = np.eye(self.num_noise)
        Q[0:3, 0:3] = self._dt ** 2 * self.stdev_na ** 2 * np.eye(3)
        Q[3:6, 3:6] = self._dt ** 2 * self.stdev_nom ** 2 * np.eye(3)
        Q[6:13, 6:13] = np.diag(self._config.process_noise_rw_var)
        self.Q = Q
        self.R = np.diag(self._config.meas_noise_var)
        self._engine.set_noise(np.diag(Q)[None].copy(), np.diag(self.R)[None].copy(), self.stdev_nom[None].copy())

    # ---- Filter.py:144-230 -------------------------------------------------------
    def run(self, camera: Camera, k: int, run_desc_str: str = "") -> None:
        """Filter.run (Filter.py:144-168): every epoch of the camera trajectory, as ONE launch of the persistent kernel in
        trace mode (eskf_streams_t.trace_x: the nominal state after every IMU step, the updated state at the update
        instants -- the rows FilterTraj keeps).  ``camera`` must be the simulator's camera (the streams were built from
        it); epoch-by-epoch stepping with another camera goes through ``run_one_epoch``."""
        self.run_id = k
        s = self._sim.streams
        if camera is not self._sim.camera:  # a foreign camera object: the reference's loop, one launch per call
            old_t = self._config.min_t
            for i, t in enumerate(camera.t[1:]):
                self.run_one_epoch(old_t, t, i + 1, camera)
                self.calculate_update_mse(i + 1, camera)
                old_t = t
            return
        T, E = len(s.dt), len(s.n_prop)
        trace = np.zeros((1, T, 26))
        st, _ = self._engine.run(s.dt, s.om_acc, s.n_prop, s.cam, s.notch, cam_ref=s.cam_ref, imu_ref=s.imu_ref,
                                 gt_dofs=self._config.gt_imu_dofs, trace=trace)
        for kk in range(T):
            self.imu.ref_rows.append(s.imu_ref_rows[kk])
            self.traj.append_propagated_states(s.t_imu[kk], State.from_vector(trace[0, kk]))
        if T:
            self._dt = float(s.dt[T - 1])
            self.imu.om, self.imu.acc = s.om_acc[T - 1, :3].copy(), s.om_acc[T - 1, 3:].copy()
            self._propagated = True
        if int(st[0, 9]) != E:  # Filter.py:358-361: the reference prints and carries on with the next epoch
            print("ERROR: Singular matrix!")
            print("Stopping simulation.")
        self.update_mse = float(st[0, 7])  # Filter.calculate_update_mse of the last epoch (Filter.py:397-418)

    def run_one_epoch(self, old_t: float, t: float, i_cam: int, camera: Camera) -> None:
        self.propagate_imu(old_t, t)
        self.update(t, camera_at_index(camera, i_cam), camera.get_notch_vec_at(i_cam)[0])

    def propagate_imu(self, t0: float, tn: float):
        s = self._sim.streams
        sel = np.nonzero((s.t_imu > t0) & (s.t_imu <= tn))[0]
        if len(sel):
            self._propagate_range(int(sel[0]), len(sel))

    def _propagate_range(self, k0: int, n: int):
        s = self._sim.streams
        for k in range(k0, k0 + n):
            self.imu.ref_rows.append(s.imu_ref_rows[k])
            self._dt = float(s.dt[k])
            self.propagate(s.t_imu[k], s.om_acc[k, :3], s.om_acc[k, 3:])

    def propagate(self, t, om, acc):
        """One IMU step with the current ``self._dt`` (Filter.py:219-230)."""
        oa = np.hstack((np.asarray(om, dtype=float).reshape(3), np.asarray(acc, dtype=float).reshape(3)))
        self._engine.propagate(np.array([self._dt]), oa[None])
        self._propagated = True
        self.imu.om, self.imu.acc = oa[:3].copy(), oa[3:].copy()
        self.traj.append_propagated_states(t, self._states)

    # ---- Filter.py:351-395 ---------------------------------------------------------
    def update(self, t: float, camera: VisualMeasurementPoint, ang_notch: float):
        st0 = int(self._engine.get_state()[4][0])
        K = self._engine.update(np.hstack((camera.pos, camera.q.xyzw)), float(ang_notch), want_gain=True)
        # decided from THIS call (the engine's status word is sticky until the next reset): a skipped update leaves the
        # gain buffer at zero
        if not np.any(K[0]):
            st = int(self._engine.get_state()[4][0])
            if (st & ~st0) & 2 or ((st & 2) and not (st & 1)):
                # math.asin raises ValueError in the reference (Quaternion.py:150-160) -- reported, not raised, here
                print("ERROR: rotation residual outside the domain of asin!")
            else:
                print("ERROR: Singular matrix!")  # Filter.py:358-361
            print("Stopping simulation.")
            return None
        self.traj.append_updated_states(t, self._states)
        return K[0]

    # ---- metrics (Filter.py:397-455) -------------------------------------------------------
    def calculate_update_mse(self, i_cam, camera):
        kf = self.traj.rows[-1]
        camera = camera.rotated if camera.rotated is not None else camera  # Filter.py:398
        cam_ref = np.hstack((camera.p[:, i_cam], camera.r_deg[i_cam]))
        s_cam = np.sum(np.square(cam_ref - kf[20:26]))
        s_imu = np.sum(np.square(kf[4:10] - self.imu.ref_rows[-1][4:10]))
        self.update_mse = (s_cam + s_imu) / 12

    def calculate_dof_metric(self):
        res = self._states.dofs - self._config.gt_imu_dofs
        return float(np.dot(res, res) / 6)

    def save(self):
        self._config.mse = self.mse
        kf_fp = os.path.join(str(self._config.traj_path), f"kf_best_{self._config.traj_name}.txt")
        save_trajectory(self.traj.rows, kf_fp)
        save_trajectory(self.imu.ref_rows, kf_fp.replace("kf_best", "imu_ref"))


def camera_at_index(camera: Camera, i: int) -> VisualMeasurementPoint:
    """VisualTraj.at_index (VisualTrajectory.py:120-134): scaled position, RAW quaternion."""
    return VisualMeasurementPoint(camera.t[i], camera.p[0, i], camera.p[1, i], camera.p[2, i], rot.Quaternion(camera.q_raw[i]))


class Simulator:
    """dvi_ekf/filter/Simulator.py:24: builds camera / IMU streams / x0 / cov0, owns the filter."""

    def __init__(self, config: Config, device: Optional[int] = None):
        self._config = config
        self.device = config.batch.device if device is None else int(device)
        self.legacy_golden = config.batch.legacy_golden
        config.update_dofs(None)
        self._update_config(config)
        self.kf = Filter(self)
        self._optim_std = [*config.process_noise_rw_std, *config.meas_noise_std]
        self.mode = config.sim.mode
        self.num_kf_runs = config.sim.num_kf_runs
        self.show_run_progress = True
        self.mses: List[float] = []
        self.mse_best = 1e10
        self.mse_avg: Optional[float] = None
        self._kf_best = None
        self.stats = None
        self.consistency = None  # summary of the last run(consistency=True)
        self.dof_envelope = None  # per-DOF envelope of the last run(consistency=True)

    @property
    def config(self):
        return self._config

    @property
    def cov0(self) -> np.ndarray:
        return self._cov0.copy()

    @property
    def optim_std(self):
        return self._optim_std

    @optim_std.setter
    def optim_std(self, val):
        """Simulator.py:76-86, reproduced literally (including the ``val[7:8]`` slice and the un-refreshed
        ``*_var`` vectors the reference's noise matrices are built from)."""
        self._optim_std = val
        self.config.process_noise_rw_std = val[0:7]
        self.config.meas_noise_std = val[7:8]
        self.kf.update_noise_matrices()

    def _trajectory(self, cfg: Config, traj_fp: str, max_vals: Optional[int]) -> Tuple[Camera, Streams]:
        """(Camera, Streams) of one camera trajectory (a path, or a name of data/trajs.npz) cut to ``max_vals`` frames"""
        t, xyz, q, i0 = load_trajectory(str(traj_fp), max_vals=max_vals, start_frame=cfg.camera.start_frame, with_start_index=True)
        mode = "zyx_legacy" if self.legacy_golden else "xyz"
        # with_notch: true (SURVEY 8f rank 4; unrunnable at the reference's HEAD, quirk Q12): the notch rows are cut like the
        # camera rows (VisualTrajectory.py:66-70) and the camera generates its rotated twin (Camera.py:131-134)
        notch = load_notch(str(cfg.notch_fp), max_vals=len(t), start_index=i0) if cfg.with_notch else None
        if notch is not None and len(notch) != len(t):
            raise ValueError(f"notch trajectory has {len(notch)} rows for {len(t)} camera frames")  # VisualTrajectory.py:70
        camera = Camera(t, xyz, q, scale=cfg.camera.scale, euler_mode=mode, notch=notch)
        streams = build_streams(camera, cfg.interframe_vals, cfg.model.length, cfg.model.angle, gt_dofs=cfg.gt_imu_dofs,
                                ic_dofs=cfg.ic_imu_dofs)
        return camera, streams

    def _update_config(self, cfg: Config) -> None:
        self.camera, self.streams = self._trajectory(cfg, cfg.traj_fp, cfg.max_vals)
        cfg.max_vals, cfg.min_t, cfg.max_t = self.camera.max_vals, self.camera.min_t, self.camera.max_t
        cfg.total_data_pts = (self.camera.max_vals - 1) * cfg.interframe_vals + 1
        self.camera_interp = (self.camera.rotated or self.camera).interpolate(cfg.interframe_vals)  # Imu.create (Imu.py:87-90)
        self.x0 = State.from_vector(self.streams.x0)
        self._cov0 = cfg.cov0_matrix

    # ---- batched tuner (SURVEY 8f rank 3; Simulator.optimise, Simulator.py:163-245) -------------------------
    OPTIM_BOUNDS = ((0, 10), (0, 10), (0, 10), (0, np.deg2rad(5)), (0, np.deg2rad(5)), (0, np.deg2rad(5)), (0, np.deg2rad(5)),
                    (0, 0.2), (0, 0.2), (0, 0.2), (0, np.deg2rad(10)), (0, np.deg2rad(10)), (0, np.deg2rad(10)),
                    (0, np.deg2rad(1)))  # random walks p(3) r(3) notch'' | measurement p_cam(3) r_cam(3) notch

    def evaluate_candidates(self, X, runs_per_candidate: Optional[int] = None, metric: str = "dof"):
        """Objective of ``Simulator.optimise`` for a whole POPULATION in one launch.  ``X`` is [M,14]: the optimisation
        variables of the reference (random-walk std of the 6 DOFs and of the notch acceleration, measurement std of the
        camera position, orientation and notch) -- unlike the reference's setter (Simulator.py:76-86, which keeps only
        ``val[7:8]`` and never refreshes the variances) all 14 take effect.  Every candidate runs ``runs_per_candidate``
        Monte-Carlo filters (run 0 of each candidate is noise free); returns per candidate, [M], the mean DOF MSE
        (``metric="dof"``, Filter.calculate_dof_metric), the mean update MSE (``"update"``) or the filter's inconsistency
        ``|ln(ANIS / 7)|`` (``"nis"``) / ``|ln(ANEES / d)|`` (``"nees"``, d estimated DOFs), the averages taken over every finite
        value of the candidate's runs and epochs (``consistency.candidate_objective``; +inf without one)."""
        X = np.atleast_2d(np.asarray(X, dtype=float))
        if X.shape[1] != 14:
            raise ValueError("candidates must have 14 columns: rw_std (7), meas_std (7)")
        if metric not in ("dof", "update", "nis", "nees"):
            raise ValueError(f"unknown metric {metric!r}: dof, update, nis or nees")
        cfg, s, b = self.config, self.streams, self.config.batch
        dim_dofs = 6 - sum(1 for f in cfg.frozen_dofs if f)
        if metric == "nees" and dim_dofs == 0:
            raise ValueError("metric 'nees' needs at least one estimated DOF (frozen_dofs freezes all six)")
        m, r = len(X), int(runs_per_candidate or self.num_kf_runs)
        n = m * r
        Qd = np.zeros((n, 13))
        Qd[:, 6:13] = np.repeat(np.square(X[:, 0:7]), r, 0)
        Rd = np.repeat(np.square(X[:, 7:14]), r, 0)
        x0 = np.repeat(s.x0[None], n, 0)
        for i in range(n):
            if i % r:  # the same perturbed initial conditions and noise seeds for every candidate (common random numbers)
                rng = np.random.default_rng([b.seed, i % r])
                x0[i, 10:13] += rng.normal(0.0, np.deg2rad(b.dof_ic_std_deg), 3)
                x0[i, 13:16] += rng.normal(0.0, b.dof_ic_std_cm, 3)
        imu_std = np.hstack((cfg.imu.stdev_omega, cfg.imu.stdev_accel)) if b.imu_noise else None
        cam_std = np.array(cfg.meas_noise_std) if b.cam_noise else None
        with BatchFilter(n, scope_length=cfg.model.length, cam_angle_rad=cfg.model.angle, frozen_dofs=cfg.frozen_dofs,
                         zero_frozen_dofs=not self.legacy_golden, device=self.device) as bf:
            bf.set_noise(Qd, Rd, self.kf.stdev_nom[None].copy())
            bf.set_state(x0, self._cov0[None], s.u0[None], None)
            if metric in ("nis", "nees"):
                bf.keep_consistency()
            # noise keyed by the run id INSIDE the candidate (noise_id_modulus = r): every candidate sees the same
            # r noise realisations, so candidates differ only by their parameters
            st, _ = bf.run(s.dt, s.om_acc, s.n_prop, s.cam, s.notch, cam_ref=s.cam_ref, imu_ref=s.imu_ref,
                           gt_dofs=cfg.gt_imu_dofs, seed=b.seed, imu_noise_std=imu_std, cam_noise_std=cam_std,
                           noise_free_filter0=True, noise_id_modulus=r, **self._dropout_kwargs())
            if metric in ("nis", "nees"):
                nis, nees, _ = bf.get_consistency()
                return candidate_objective(nis if metric == "nis" else nees, m, NIS_DIM if metric == "nis" else dim_dofs)
        col = 6 if metric == "dof" else 8
        vals = st[:, col].reshape(m, r)
        if metric != "dof":
            vals = vals / max(1, len(s.n_prop))
        return vals.mean(axis=1)

    def optimise(self, maxiter: int = 1, popsize: int = 1, runs_per_candidate: Optional[int] = None, seed: Optional[int] = None,
                 metric: str = "dof"):
        """``Simulator.optimise`` (Simulator.py:163-245): differential evolution over the 14 noise parameters, with the
        objective of a whole generation evaluated by ONE batched launch (scipy ``vectorized=True``,
        ``updating="deferred"``).  ``metric`` is that of ``evaluate_candidates``: "dof" or "update" minimise an error,
        "nis" / "nees" the distance of ANIS / ANEES from 7 / d (the usual objective for tuning Q and R: a filter whose
        covariance matches its errors).  Returns the scipy result; the best parameters become ``optim_std``."""
        from scipy.optimize import differential_evolution

        def fun(x):  # x: (14, S) for a population of S members
            return self.evaluate_candidates(np.asarray(x).T, runs_per_candidate, metric)

        ret = differential_evolution(fun, self.OPTIM_BOUNDS, strategy="best1bin", maxiter=maxiter, popsize=popsize, seed=seed,
                                     vectorized=True, updating="deferred", polish=False)
        self._optim_std = list(ret.x)
        self._dof_mse = float(ret.fun)
        return ret

    def run_once(self) -> None:
        self.kf.run(self.camera, 0, "KF run")
        self.mse_best = self.kf.mse
        print(f"\t MSE: {self.mse_best:.2E}")

    def reset_kf(self) -> None:
        self.kf = Filter(self)

    def _mc_x0(self, x0_row, n: int):
        """[n, 26] initial states of Monte-Carlo runs 0 .. n-1: run 0 nominal, run i's DOFs perturbed by the draws of
        (batch seed, i)"""
        b = self.config.batch
        x0 = np.repeat(np.asarray(x0_row)[None], n, 0)
        for i in range(1, n):
            rng = np.random.default_rng([b.seed, i])
            x0[i, 10:13] += rng.normal(0.0, np.deg2rad(b.dof_ic_std_deg), 3)
            x0[i, 13:16] += rng.normal(0.0, b.dof_ic_std_cm, 3)
        return x0

    def _batch(self, n: int, x0, u0, consistency: bool, groups: int = 0) -> BatchFilter:
        """a BatchFilter of n filters with the filter's noise matrices, cov0, the given x0 / u0 rows, consistency on or off
        and filter groups of ``groups``"""
        cfg = self.config
        bf = BatchFilter(n, scope_length=cfg.model.length, cam_angle_rad=cfg.model.angle, frozen_dofs=cfg.frozen_dofs,
                         zero_frozen_dofs=not self.legacy_golden, device=self.device)
        try:
            bf.set_noise(np.diag(self.kf.Q)[None].copy(), np.diag(self.kf.R)[None].copy(), self.kf.stdev_nom[None].copy())
            bf.set_state(x0, self._cov0[None], u0, None)
            if consistency:
                bf.keep_consistency()
            if groups:
                bf.set_groups(groups)
        except Exception:
            bf.close()
            raise
        return bf

    def _dropout_kwargs(self, cam_dropout: Optional[float] = None) -> dict:
        """``drop_prob`` of BatchFilter.run for the frame-loss probability ``cam_dropout`` (None: ``batch.cam_dropout``); nothing
        at 0, so that a run without frame loss keeps the production kernel"""
        p = self.config.batch.cam_dropout if cam_dropout is None else float(cam_dropout)
        if not 0.0 <= p <= 1.0:
            raise ValueError(f"cam_dropout must be a probability in [0, 1], not {p}")
        return {"drop_prob": p} if p > 0 else {}

    def _run_kwargs(self, cam_ref, imu_ref, cam_dropout: Optional[float] = None) -> dict:
        """the keyword arguments of BatchFilter.run for a Monte-Carlo run (``batch:`` section)"""
        cfg, b = self.config, self.config.batch
        imu_std = np.hstack((cfg.imu.stdev_omega, cfg.imu.stdev_accel)) if b.imu_noise else None
        cam_std = np.array(cfg.meas_noise_std) if b.cam_noise else None
        return dict(cam_ref=cam_ref, imu_ref=imu_ref, gt_dofs=cfg.gt_imu_dofs, seed=b.seed, imu_noise_std=imu_std,
                    cam_noise_std=cam_std, **self._dropout_kwargs(cam_dropout))

    def _stacked_trajectories(self, names, n_filters: int, frames: Optional[int] = None, consistency: bool = False):
        """(BatchFilter, run keyword arguments) of the stacked launch of ``run_trajectories``: the named trajectories built as
        ``__init__`` builds ``config.traj_name``, cut to ``frames`` frames (None: the shortest one's), ``n_filters`` filters
        each, groups of ``n_filters``.  ``bf.run(**kw)`` runs it; the caller closes the handle.  (Also the hook through which
        tools/trajectory_study.py times the launch and the getters.)"""
        names = [str(nm) for nm in names]
        if not names or len(set(names)) != len(names):
            raise ValueError("names must be one or more distinct trajectory names")
        n = int(n_filters)
        if n <= 0:
            raise ValueError("n_filters must be positive")
        cfg = self.config
        avail = min(len(load_trajectory(nm, start_frame=cfg.camera.start_frame)[0]) for nm in names)
        frames = avail if frames is None else int(frames)
        if not 2 <= frames <= avail:
            raise ValueError(f"frames must be 2 .. {avail} (the shortest trajectory's frame count), not {frames}")
        ss = [self._trajectory(cfg, nm, frames)[1] for nm in names]
        T = max(len(s.dt) for s in ss)
        pad = lambda a: np.concatenate((a, np.zeros((T - len(a), *a.shape[1:]))))  # (steps past sum(n_prop): never read)
        cat = lambda f: np.ascontiguousarray(np.concatenate([f(s) for s in ss]))
        bf = self._batch(n * len(names), cat(lambda s: self._mc_x0(s.x0, n)), cat(lambda s: np.repeat(s.u0[None], n, 0)),
                         consistency, groups=n)
        kw = self._run_kwargs(cat(lambda s: s.cam_ref), cat(lambda s: s.imu_ref))
        kw.update(dt=cat(lambda s: pad(s.dt)), om_acc=cat(lambda s: pad(s.om_acc)), n_prop=cat(lambda s: s.n_prop),
                  cam=cat(lambda s: s.cam), notch=cat(lambda s: s.notch), n_traj=len(names), filters_per_traj=n,
                  noise_free_filter0=True, noise_id_modulus=n)
        return bf, kw

    def run_trajectories(self, names, n_filters: int, frames: Optional[int] = None, consistency: bool = False) -> dict:
        """One Monte-Carlo study over several trajectories (names as ``load_trajectory`` takes them, e.g. ``trans_x``), in ONE
        stacked launch: every trajectory cut to ``frames`` camera frames (None: the shortest one's), ``n_filters`` filters
        each.  Filter j of every trajectory is run j of ``run``: the same perturbed initial DOFs and the noise of id j
        (run 0 noise free), so trajectories are compared on common random numbers, and each trajectory's filters give the
        bits ``run(n_filters)`` of a simulator configured with it alone gives.  Returns, and keeps as
        ``trajectory_results``, per name: ``stats`` (``sharding.summarise_stats`` of its filters) and, with ``consistency``,
        ``consistency`` and ``dof_envelope`` (``summarise_consistency`` / ``summarise_dofs`` of its filters).  The
        per-filter statistics rows are kept as ``stats`` ([len(names) * n_filters, 16], trajectory-major)."""
        cfg = self.config
        bf, kw = self._stacked_trajectories(names, n_filters, frames, consistency)
        with bf:
            st, _ = bf.run(**kw)
            _, gst, gcons, gdof = bf.get_group_sums(stats=True, consistency=consistency, dof_envelope=consistency)
        dim = 6 - sum(1 for f in cfg.frozen_dofs if f)
        res = {}
        for k, nm in enumerate(str(v) for v in names):
            res[nm] = {"stats": summarise_stats(gst[k])}
            if consistency:
                res[nm]["consistency"] = summarise_consistency(gcons[k], dim)
                res[nm]["dof_envelope"] = summarise_dofs(gdof[k], cfg.frozen_dofs)
        self.stats = st
        self.trajectory_results = res
        return res

    def run(self, disp_config=False, save_best=False, verbose=True, n_filters: Optional[int] = None, consistency: bool = False,
            segment_epochs: Optional[int] = None, cam_dropout: Optional[float] = None):
        """Simulator.run (Simulator.py:121-158) as ONE batched launch: ``num_kf_runs`` (or ``n_filters``)
        independent filters, run 0 noise free (the reference's deterministic run), the others with
        Monte-Carlo IMU / camera noise and DOF initial-condition perturbations (``batch:`` section).
        ``consistency``: ``self.consistency`` becomes ``consistency.summarise_consistency`` of the run (ANIS / ANEES per
        epoch and their chi-square intervals), ``self.dof_envelope`` ``consistency.summarise_dofs`` of it (bias, RMSE,
        claimed sigma, inflation, per-DOF ANEES and coverage per DOF and epoch).
        ``segment_epochs`` k: the same run in launches of k epochs (``BatchFilter.run_segments``), with the same results; the
        consistency records then take the memory of k epochs, not of the whole run, and their per-epoch rows are joined.
        ``cam_dropout``: the probability that a filter loses a camera frame (``BatchFilter.run(drop_prob=...)``; run 0, the
        noise-free one, loses none); None takes ``batch.cam_dropout`` (default 0: no frame loss)."""
        cfg, s = self.config, self.streams
        n = int(n_filters or self.num_kf_runs)
        with self._batch(n, self._mc_x0(s.x0, n), s.u0[None], consistency) as bf:
            kw = self._run_kwargs(s.cam_ref, s.imu_ref, cam_dropout)
            E = len(s.n_prop)
            if segment_epochs and E:
                k = int(segment_epochs)
                if k <= 0:
                    raise ValueError("segment_epochs must be positive")
                esum, env = [], []
                for _, _, st, sm in bf.run_segments(s.dt, s.om_acc, s.n_prop, s.cam, s.notch, [*range(0, E, k), E], **kw):
                    if consistency:  # per-epoch rows: joining the segments' rows is exact
                        esum.append(bf.get_consistency()[2])
                        env.append(bf.get_dof_envelope())
                if consistency:
                    esum, env = np.concatenate(esum), np.concatenate(env)
            else:
                st, sm = bf.run(s.dt, s.om_acc, s.n_prop, s.cam, s.notch, **kw)
                if consistency:
                    esum, env = bf.get_consistency()[2], bf.get_dof_envelope()
            self.final_states = bf.get_state()[0]
            if consistency:
                self.consistency = summarise_consistency(esum, 6 - sum(1 for f in cfg.frozen_dofs if f))
                self.dof_envelope = summarise_dofs(env, cfg.frozen_dofs)
        self.stats = st
        # Simulator.py:138-158 appends ``kf.mse`` of every run -- which is 0 at the reference's HEAD, because the call that
        # would set it is commented out (Filter.py:92,167-168).  ``mses`` / ``mse_best`` / ``mse_avg`` keep exactly that
        # behaviour; the DOF metric the author meant (Filter.calculate_dof_metric, Filter.py:452-455) of every run is in
        # ``dof_mses`` / ``dof_mse_best`` / ``dof_mse_avg`` (INTEGRATION.md, "Deviations").
        self.mses = [float(self.kf.mse)] * n
        self.mse_best = min(self.mse_best, min(self.mses))
        self.mse_avg = sum(self.mses) / len(self.mses)
        self.dof_mses = [float(v) for v in st[:, 6]]
        self.dof_mse_best = min(self.dof_mses)
        self.dof_mse_avg = sum(self.dof_mses) / len(self.dof_mses)
        if verbose:
            print(f"\tOptimvars: {self.optim_std}")
            print(f"\tDOF MSE: {self.mse_avg:.2E}")
            print(f"\tDOF MSE (Filter.calculate_dof_metric, mean of {n} runs): {self.dof_mse_avg:.2E}")
        return st, sm
