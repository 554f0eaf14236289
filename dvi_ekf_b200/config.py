"""``Config``: the reference's config.yaml, loaded without pydantic-v1.

Mirrors dvi_ekf/tools/config.py:214-272 attribute for attribute (same names,
same unit conversions: every angle given in degrees in the YAML is converted to
radians) so the same file drives the reference and this engine.  An optional
``batch:`` section (ignored by the reference) configures the Monte-Carlo /
sweep extensions.
"""
from __future__ import annotations

import math
import os
from types import SimpleNamespace
from typing import Optional

import numpy as np
import yaml


class Config:
    def __init__(self, filepath):
        with open(filepath) as f:
            cfg = yaml.safe_load(f)
        s, c, i, m, fl = cfg["simulation"], cfg["camera"], cfg["imu"], cfg["model"], cfg["filter"]
        self.filepath = str(filepath)
        # --- simulation (config.py:16-54) ---
        self.sim = SimpleNamespace(
            mode=s.get("mode", "run"), img_path=s.get("img_path"), traj_path=s.get("traj_path", "."),
            traj_name=s["traj_name"], notch_traj_name=s.get("notch_traj_name"), num_kf_runs=int(s.get("num_kf_runs", 1)),
            frozen_dofs=list(s["frozen_dofs"]), do_plot=bool(s.get("do_plot", False)), do_fast_sim=bool(s.get("do_fast_sim", False)))
        self.sim.traj_fp = os.path.join(self.sim.traj_path, f"{self.sim.traj_name}.csv")
        self.sim.notch_fp = os.path.join(self.sim.traj_path, f"{self.sim.notch_traj_name}.csv")
        # --- camera (config.py:57-94) ---
        noise = c["noise"]
        total = c.get("total_frames")
        self.camera = SimpleNamespace(
            start_frame=c.get("start_frame"), total_frames=None if total == "all" else total, scale=c.get("scale", 1),
            with_notch=bool(c.get("with_notch", False)),
            noise=SimpleNamespace(position=list(noise["position"]), theta=np.deg2rad(noise["theta"]).tolist(),
                                  notch=float(np.deg2rad(noise["notch"]))))
        self.camera.noise.vec = np.hstack((self.camera.noise.position, self.camera.noise.theta, self.camera.noise.notch))
        # --- imu (config.py:96-120) ---
        rate, grav = float(i["noise_sample_rate"]), float(i["gravity"])
        self.imu = SimpleNamespace(
            interframe_vals=int(i["interframe_vals"]), noise_sample_rate=rate, gravity=grav,
            noise_gyro=0.005 * math.sqrt(rate),
            stdev_omega=[float(np.deg2rad(0.005 * math.sqrt(rate)))] * 3,
            stdev_accel=np.array([400 * 1e-6 * grav * math.sqrt(rate)] * 3))
        # --- model (config.py:123-133) ---
        self.model = SimpleNamespace(length=float(m["length"]), angle=float(np.deg2rad(m["angle"])))
        # --- filter (config.py:136-211) ---
        def states(d):
            rad = lambda k: np.deg2rad(d[k]).tolist()
            ns = SimpleNamespace(imu_pos=list(d["imu_pos"]), imu_vel=list(d["imu_vel"]), imu_theta=rad("imu_theta"),
                                 dofs_rot=rad("dofs_rot"), dofs_trans=list(d["dofs_trans"]), notch=rad("notch"),
                                 camera_pos=list(d["camera_pos"]), camera_theta=rad("camera_theta"))
            ns.vec = np.hstack((ns.imu_pos, ns.imu_vel, ns.imu_theta, ns.dofs_rot, ns.dofs_trans, ns.notch, ns.camera_pos,
                                ns.camera_theta))
            return ns

        ic = fl["ic"]
        pn = fl["process_noise"]["dofs"]
        noise_dofs = SimpleNamespace(translation=list(pn["translation"]), rotation=np.deg2rad(pn["rotation"]).tolist(),
                                     notch_accel=float(np.deg2rad(pn["notch_accel"])))
        noise_dofs.vec = np.hstack((noise_dofs.rotation, noise_dofs.translation, noise_dofs.notch_accel))
        self.filter = SimpleNamespace(ic=SimpleNamespace(cov0=states(ic["cov0"]), x0=states(ic["x0"])), noise_dofs=noise_dofs)
        self.filter.ic.cov0_matrix = np.square(np.diag(self.filter.ic.cov0.vec))

        # --- derived (config.py:234-272) ---
        self.interframe_vals = self.imu.interframe_vals
        self.cov0_matrix = self.filter.ic.cov0_matrix
        self.with_notch = self.camera.with_notch
        self.max_vals = self.camera.total_frames
        self.min_t: Optional[float] = None
        self.max_t: Optional[float] = None
        self.total_data_pts: Optional[int] = None
        if self.sim.do_fast_sim:  # config.py:246-248
            self.interframe_vals = 1
            self.max_vals = 10
        self.frozen_dofs = self.sim.frozen_dofs
        self.gt_joint_dofs = None
        self.gt_imu_dofs = None
        self.ic_imu_dofs = None
        self._dofs_updated = False
        self.process_noise_rw_std = self.filter.noise_dofs.vec / self.interframe_vals
        self.process_noise_rw_var = np.square(self.process_noise_rw_std)
        self.meas_noise_std = self.camera.noise.vec
        self.meas_noise_var = np.square(self.meas_noise_std)
        self.img_path, self.traj_path = self.sim.img_path, self.sim.traj_path
        self.traj_name, self.notch_traj_name = self.sim.traj_name, self.sim.notch_traj_name
        self.traj_fp, self.notch_fp = self.sim.traj_fp, self.sim.notch_fp
        self.mse = None
        self.do_plot = self.sim.do_plot
        # --- engine extensions (not read by the reference) ---
        b = cfg.get("batch") or {}
        self.batch = SimpleNamespace(
            seed=int(b.get("seed", 1234)), imu_noise=bool(b.get("imu_noise", True)), cam_noise=bool(b.get("cam_noise", True)),
            dof_ic_std_deg=float(b.get("dof_ic_std_deg", 3.0)), dof_ic_std_cm=float(b.get("dof_ic_std_cm", 3.0)),
            legacy_golden=bool(b.get("legacy_golden", False)), device=int(b.get("device", 0)),
            cam_dropout=float(b.get("cam_dropout", 0.0)),  # probability that a Monte-Carlo filter loses a camera frame
            # innovation gate: NIS threshold of every camera update (absent or null: no gate)
            nis_gate=None if b.get("nis_gate") is None else float(b.get("nis_gate")),
            # simulated outlier frames: probability per frame and the offsets' 7 standard deviations (units of meas_noise_std)
            cam_outlier_prob=float(b.get("cam_outlier_prob", 0.0)),
            cam_outlier_std=None if b.get("cam_outlier_std") is None else [float(v) for v in b.get("cam_outlier_std")])
        if not 0.0 <= self.batch.cam_dropout <= 1.0:
            raise ValueError(f"batch.cam_dropout must be a probability in [0, 1], not {self.batch.cam_dropout}")
        if self.batch.nis_gate is not None and not self.batch.nis_gate >= 0.0:
            raise ValueError(f"batch.nis_gate must be a NIS threshold >= 0 (or null for no gate), not {self.batch.nis_gate}")
        if not 0.0 <= self.batch.cam_outlier_prob <= 1.0:
            raise ValueError(f"batch.cam_outlier_prob must be a probability in [0, 1], not {self.batch.cam_outlier_prob}")
        sd = self.batch.cam_outlier_std
        if sd is not None and not (len(sd) == 7 and all(v >= 0.0 and v != float("inf") for v in sd)):
            raise ValueError(f"batch.cam_outlier_std must be 7 finite values >= 0, not {sd}")
        if self.batch.cam_outlier_prob > 0 and sd is None:
            raise ValueError("batch.cam_outlier_prob > 0 requires batch.cam_outlier_std (7 values)")

    @property
    def dofs_updated(self) -> bool:
        return self._dofs_updated

    def update_dofs(self, probe=None) -> None:
        """config.py:278-283 with SimpleProbe's constraints (Probe.py:385-388) and utils.generate_imudof_ic
        (tools/utils.py:41-42: the IC equals the ground truth)."""
        from .probe import GT_IMU_DOFS

        self.gt_imu_dofs = GT_IMU_DOFS.copy()
        self.gt_joint_dofs = [np.hstack((GT_IMU_DOFS, 0.0, 0.0)), np.zeros(8), np.zeros(8)]
        self.ic_imu_dofs = self.gt_imu_dofs.copy()
        self._dofs_updated = True
