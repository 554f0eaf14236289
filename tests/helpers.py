"""Shared test helpers: oracle-driven scenarios and the parity metrics.

Parity metric (DESIGN.md, "Parity protocol"): state groups are compared
norm-wise (max |diff| / max |ref| per group p, v, q, dofs, notch, p_cam,
q_cam); covariance blocks are compared per 3x3 block, normalised by the
geometric mean of the two diagonal blocks' largest entries -- never per tiny
entry.  Directly measured blocks after an update additionally get an absolute
floor of 1e-7 * sqrt(R_i R_j): when the prior is >> R the reference's own FP64
arithmetic only determines those entries to ~1e-8 (it computes 1 - K with
K = 1 - O(1e-12); see tests/test_conditioning.py).
"""
import os

import numpy as np

from oracle.eskf_oracle import (
    OracleConfig,
    OracleFilter,
    Probe,
    State,
    build_streams,
    camera_from_arrays,
    camera_gen_rotated,
    quat_normalise,
)

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
LEGACY_COLS = [0, 1, 2, 3, 7, 8, 9, 10, 11, 12, 13]  # all but the velocity columns (an older velocity definition)


def legacy_imu_ref(kp):
    """The reference's legacy imu_ref_mandala0_mono_upd_Kp<kp>_Km1.000.txt [rows, 14], decoded bit-exactly from
    tests/golden/imu_ref_legacy.npz (see make_golden.py); the velocity columns 4:7 are not stored and read as NaN."""
    with np.load(os.path.join(GOLDEN_DIR, "imu_ref_legacy.npz")) as z:
        n = np.cumsum(z[f"Kp{kp}"], axis=0)
    out = np.full((len(n), 14), np.nan)
    out[:, LEGACY_COLS] = n / 1e9
    return out


GROUPS = {"p": (0, 3), "v": (3, 6), "q": (6, 10), "dofs": (10, 16), "notch": (16, 19), "pc": (19, 22), "qc": (22, 26)}
HSET = [18, 19, 20, 21, 22, 23, 15]


def state_err(x, xr, floor=1e-12):
    """worst group-wise relative error; groups whose reference is (near) zero use an absolute floor"""
    worst = 0.0
    for s, e in GROUPS.values():
        den = max(np.abs(xr[s:e]).max(), floor)
        worst = max(worst, np.abs(x[s:e] - xr[s:e]).max() / den)
    return worst


def cov_err(P, Pr, rd=None):
    """worst 3x3-block error of P vs Pr; rd (7) enables the measured-block floor"""
    d = np.abs(np.diag(Pr))
    floor = np.zeros(24)
    if rd is not None:
        for m, h in enumerate(HSET):
            floor[h] = rd[m]
    worst = 0.0
    for i in range(8):
        for j in range(8):
            si, sj = slice(3 * i, 3 * i + 3), slice(3 * j, 3 * j + 3)
            den = np.sqrt(d[si].max() * d[sj].max())
            fl = 1e-7 * np.sqrt(floor[si].max() * floor[sj].max())
            diff = np.abs(P[si, sj] - Pr[si, sj]).max()
            diff = max(0.0, diff - fl)
            worst = max(worst, diff / max(den, 1e-300))
    return worst


def model_kwargs(cfg: OracleConfig):
    return dict(scope_length=cfg.length, cam_angle_rad=cfg.angle, frozen_dofs=tuple(cfg.frozen_dofs),
                zero_frozen_dofs=cfg.zero_frozen_dofs)


class Scenario:
    """Everything needed to run one trajectory through the oracle and the engine."""

    def __init__(self, traj, cfg: OracleConfig, notch=None):
        self.cfg = cfg
        self.probe = Probe(cfg.length, cfg.angle)
        self.cam = camera_from_arrays(traj[:, 0], traj[:, 1:4], traj[:, 4:8], cfg, notch=notch)
        # with_notch: true -- the rotated camera is the IMU source / initial state / error reference (Camera.py:172-208)
        self.rotated = camera_gen_rotated(self.cam, cfg) if notch is not None else None
        (self.x0s, self.u0, self.dt, self.om_acc, self.n_prop, self.cam_meas, self.notch_meas,
         self.imu_ref_rows) = build_streams(self.cam, cfg, self.probe, self.rotated)
        self.x0 = self.x0s.as_vector()
        self.P0 = cfg.cov0_matrix
        kf = self.new_oracle()
        self.Qd = np.diag(kf.Q).copy()
        self.Rd = np.diag(kf.R).copy()
        self.sig_om = kf.stdev_nom.copy()
        self.R_old0 = kf.R_WB_old.reshape(9).copy()

    def new_oracle(self, x0=None, P0=None, u0=None):
        x = self.x0s if x0 is None else State.from_vector(x0)
        u = self.u0 if u0 is None else u0
        return OracleFilter(self.cfg, x, self.P0 if P0 is None else P0, u[:3], u[3:], self.probe)


def mandala_scenario(golden, n_frames=10, ifv=1, with_notch=False, **cfg_kw):
    cfg = OracleConfig(max_vals=n_frames, interframe_vals=ifv, **cfg_kw)
    notch = golden["notch_notch90"][:n_frames] if with_notch else None
    return Scenario(golden["traj_mandala0_mono"][:n_frames], cfg, notch=notch)


def random_filter_inputs(rng, n, cfg: OracleConfig, frozen=False):
    """n random-but-plausible (state, P, u_old) triples (SURVEY section 8d)."""
    xs, Ps, us = [], [], []
    for _ in range(n):
        dofs = np.zeros(6) if frozen else np.hstack((rng.normal(0, 0.3, 3), rng.normal(0, 3, 2), 20 + rng.normal(0, 3)))
        notch = rng.normal(0, 0.2, 3) * np.array([1.0, 0.1, 0.01])
        x = np.hstack((rng.normal(0, 30, 3), rng.normal(0, 1, 3), quat_normalise(rng.normal(0, 1, 4)), dofs, notch,
                       rng.normal(0, 10, 3), quat_normalise(rng.normal(0, 1, 4))))
        A = rng.normal(0, 1, (24, 24))
        sd = np.sqrt(np.diag(cfg.cov0_matrix)) * np.exp(rng.normal(0, 0.5, 24))
        Pm = (A @ A.T / 24 + np.eye(24)) * np.outer(sd, sd)
        xs.append(x)
        Ps.append(Pm)
        us.append(np.hstack((rng.normal(0, 0.05, 3), rng.normal(0, 0.5, 3))))
    return np.array(xs), np.array(Ps), np.array(us)
