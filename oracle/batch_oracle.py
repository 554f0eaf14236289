"""Batch-vectorised numpy restatement of the VI-ESKF path (leading axis = filters).

TEST INFRASTRUCTURE / CPU BASELINE ONLY -- see ``oracle/__init__.py``.  Same
algorithm as ``oracle/eskf_oracle.py`` (generic DH chain, geometric Jacobian,
dense 24x24 matmuls exactly as the reference executes them, LAPACK inverse),
but every operation carries a batch axis so that numpy's C loops / BLAS do the
work.  This is the strongest honest CPU implementation of the reference
algorithm we can time next to the GPU (the real reference rebuilds three CasADi
functions per IMU step and is orders of magnitude slower).  Validated against
the single-filter oracle in tests/test_batch_oracle.py.
"""
from __future__ import annotations

import math

import numpy as np

from .eskf_oracle import OracleConfig

HSET = [18, 19, 20, 21, 22, 23, 15]


def _skew(v):
    z = np.zeros(v.shape[:-1])
    return np.stack(
        [np.stack([z, -v[..., 2], v[..., 1]], -1), np.stack([v[..., 2], z, -v[..., 0]], -1), np.stack([-v[..., 1], v[..., 0], z], -1)],
        -2,
    )


def _qnorm(q):
    q = q / np.sqrt(np.sum(q * q, -1, keepdims=True))
    return np.where(q[..., 3:4] < 0, -q, q)


def _qmul(a, b):
    aw, av, bw, bv = a[..., 3:4], a[..., :3], b[..., 3:4], b[..., :3]
    w = aw * bw - np.sum(av * bv, -1, keepdims=True)
    v = aw * bv + bw * av + np.cross(av, bv)
    return _qnorm(np.concatenate([v, w], -1))


def _q2R(q):
    x, y, z, w = q[..., 0], q[..., 1], q[..., 2], q[..., 3]
    x2, y2, z2, w2 = x * x, y * y, z * z, w * w
    xy, zw, xz, yw, yz, xw = x * y, z * w, x * z, y * w, y * z, x * w
    return np.stack(
        [
            np.stack([x2 - y2 - z2 + w2, 2 * (xy - zw), 2 * (xz + yw)], -1),
            np.stack([2 * (xy + zw), -x2 + y2 - z2 + w2, 2 * (yz - xw)], -1),
            np.stack([2 * (xz - yw), 2 * (yz + xw), -x2 - y2 + z2 + w2], -1),
        ],
        -2,
    )


def _markley(M):
    """scipy-1.10.1 Rotation.from_matrix on a stack of raw matrices + Quaternion.normalise."""
    d = np.stack([M[:, 0, 0], M[:, 1, 1], M[:, 2, 2], M[:, 0, 0] + M[:, 1, 1] + M[:, 2, 2]], -1)
    choice = np.argmax(d, -1)  # first maximum, like _argmax4
    tr = d[:, 3]
    q = np.empty((M.shape[0], 4))
    m = choice == 3
    q[m] = np.stack([M[m, 2, 1] - M[m, 1, 2], M[m, 0, 2] - M[m, 2, 0], M[m, 1, 0] - M[m, 0, 1], 1 + tr[m]], -1)
    for i in range(3):
        m = choice == i
        if not np.any(m):
            continue
        j, k = (i + 1) % 3, (i + 2) % 3
        qq = np.empty((int(m.sum()), 4))
        qq[:, i] = 1 - tr[m] + 2 * M[m, i, i]
        qq[:, j] = M[m, j, i] + M[m, i, j]
        qq[:, k] = M[m, k, i] + M[m, i, k]
        qq[:, 3] = M[m, k, j] - M[m, j, k]
        q[m] = qq
    return _qnorm(q)


def _about_axis(angle, axis):
    qlen = np.sqrt(np.sum(axis * axis, -1))
    f = np.where(qlen > 4 * np.finfo(float).eps, np.sin(angle / 2) / np.where(qlen > 0, qlen, 1.0), 1.0)
    return _qnorm(np.concatenate([axis * f[:, None], np.cos(angle / 2)[:, None]], -1))


class BatchProbe:
    """Batched numeric DH chain (Probe.py:147-167) with geometric Jacobian."""

    def __init__(self, length, angle):
        hp = math.pi / 2
        self.links = [(True, hp, 0.0, hp), (True, -hp, 0.0, -hp), (True, 0.0, 0.0, 0.0), (False, 0.0, 0.0, hp),
                      (False, hp, 0.0, hp), (False, -hp, 0.0, hp), (True, 0.0, float(length), float(angle)), (True, 0.0, 0.0, 0.0)]
        self.base = np.array([[-1.0, 0, 0, 0], [0, 1, 0, 0], [0, 0, -1.0, 0], [0, 0, 0, 1]])

    def fwkin(self, dofs, notch):
        n = dofs.shape[0]
        q = np.concatenate([dofs, notch[:, :1], np.zeros((n, 1))], -1)
        T = np.broadcast_to(self.base, (n, 4, 4)).copy()
        zs, os_ = [], []
        for i, (rev, th, d, al) in enumerate(self.links):
            zs.append(T[:, :3, 2].copy())
            os_.append(T[:, :3, 3].copy())
            A = np.zeros((n, 4, 4))
            ang = q[:, i] + th if rev else np.full(n, th)
            dd = np.full(n, d) if rev else q[:, i]
            c, s, ca, sa = np.cos(ang), np.sin(ang), math.cos(al), math.sin(al)
            A[:, 0, 0], A[:, 0, 1], A[:, 0, 2] = c, -s * ca, s * sa
            A[:, 1, 0], A[:, 1, 1], A[:, 1, 2] = s, c * ca, -c * sa
            A[:, 2, 1], A[:, 2, 2], A[:, 2, 3], A[:, 3, 3] = sa, ca, dd, 1.0
            T = T @ A
        p = T[:, :3, 3]
        R = T[:, :3, :3]
        Jv = np.stack([np.cross(zs[i], p - os_[i]) if self.links[i][0] else zs[i] for i in range(7)], -1)  # N,3,7
        Jw = np.stack([zs[i] if self.links[i][0] else np.zeros_like(zs[i]) for i in range(7)], -1)
        om = zs[6] * notch[:, 1:2]
        return p, R, om, Jv, Jw


class BatchOracle:
    """N filters advanced in lock-step with dense batched linear algebra (Filter.py:219-395)."""

    def __init__(self, cfg: OracleConfig, x0, P0, u0, Qd=None, Rd=None, sig_om=None):
        self.cfg = cfg
        x0 = np.atleast_2d(np.asarray(x0, dtype=float))
        n = x0.shape[0]
        self.n = n
        self.x = x0.copy()
        P0 = np.asarray(P0, dtype=float)
        self.P = np.broadcast_to(P0, (n, 24, 24)).copy()
        u0 = np.broadcast_to(np.asarray(u0, dtype=float), (n, 6))
        self.om_old, self.acc_old = u0[:, :3].copy(), u0[:, 3:].copy()
        self.R_old = _q2R(self.x[:, 6:10])
        self.probe = BatchProbe(cfg.length, cfg.angle)
        self.frozen = np.array([bool(f) for f in cfg.frozen_dofs])
        rw = np.square(cfg.process_noise_rw_std)
        self.Qd = np.broadcast_to(np.hstack((np.zeros(6), rw)) if Qd is None else np.asarray(Qd, dtype=float), (n, 13))
        self.Rd = np.broadcast_to(np.square(cfg.meas_noise_std) if Rd is None else np.asarray(Rd, dtype=float), (n, 7))
        self.sig_om = np.broadcast_to(np.asarray(cfg.stdev_omega) if sig_om is None else np.asarray(sig_om, dtype=float), (n, 3))
        self.H = np.zeros((7, 24))
        self.H[0:6, 18:24] = np.eye(6)
        self.H[6, 15] = 1
        self.status = np.zeros(n, dtype=np.int32)

    def propagate(self, dt, om, acc):
        n, x = self.n, self.x
        om = np.broadcast_to(np.asarray(om, dtype=float), (n, 3))
        acc = np.broadcast_to(np.asarray(acc, dtype=float), (n, 3))
        dofs, notch = x[:, 10:16], x[:, 16:19]
        p_p, R_p, om_p, _, _ = self.probe.fwkin(dofs, notch)
        R_WB, R_WC = _q2R(x[:, 6:10]), _q2R(x[:, 22:26])
        om_avg = (self.om_old + om) / 2
        R_next = R_WB + R_WB @ _skew(dt * om_avg)
        acc_avg = (np.einsum("nij,nj->ni", R_WB, self.acc_old) + np.einsum("nij,nj->ni", R_next, acc)) / 2
        p = x[:, 0:3] + dt * x[:, 3:6] + (dt ** 2 / 2) * acc_avg
        v = x[:, 3:6] + dt * acc_avg
        notch_n = np.stack([notch[:, 0] + dt * notch[:, 1], notch[:, 1] + dt * notch[:, 2], notch[:, 2]], -1)
        p_cam = x[:, 19:22] + dt * x[:, 3:6] + dt * np.einsum("nij,nj->ni", R_WB, np.cross(om_avg, p_p))
        om_c = np.einsum("nji,nj->ni", R_p, self.om_old + om_p)
        R_WC_next = R_WC + R_WC @ _skew(dt * om_c)
        dofs_n = dofs.copy()
        if self.cfg.zero_frozen_dofs:
            dofs_n[:, self.frozen] = 0.0
        self.x = np.concatenate([p, v, _markley(R_next), dofs_n, notch_n, p_cam, _markley(R_WC_next)], -1)

        # error Jacobians with the buffered R_old / om_old / acc_old and the post-predict dofs
        Ro = self.R_old
        p_p, R_p, om_p, Jv, Jw = self.probe.fwkin(dofs_n, notch_n)
        Fx = np.broadcast_to(np.eye(24), (n, 24, 24)).copy()
        Fx[:, 0:3, 3:6] = dt * np.eye(3)
        Fx[:, 3:6, 6:9] = -Ro @ _skew(self.acc_old) * dt
        Om = _qnorm(np.concatenate([0.5 * dt * self.om_old, np.ones((n, 1))], -1))
        Fx[:, 6:9, 6:9] = np.swapaxes(_q2R(Om), 1, 2)
        Fx[:, 15, 16] += dt
        Fx[:, 16, 17] += dt
        om_tr = self.om_old - self.sig_om
        w = p_p + np.cross(om_tr, p_p)
        dw_dq = (np.eye(3) + _skew(om_tr)) @ Jv
        a = np.einsum("nji,nj->ni", R_p, om_tr + om_p)
        b = np.einsum("nji,nj->ni", R_p, self.om_old + om_p)
        u_tot = om_tr + om_p
        da = -np.cross(Jw, u_tot[:, :, None], axis=1)
        d_om_p = np.cross(Jw, om_p[:, :, None], axis=1)
        d_om_p[:, :, 6] = 0.0
        da_dq = np.einsum("nji,njk->nik", R_p, da + d_om_p)
        J = np.zeros((n, 6, 22))
        J[:, 0:3, 3:6] = dt * np.eye(3)
        J[:, 0:3, 6:9] = -dt * Ro @ _skew(w)
        J[:, 0:3, 9:16] = dt * Ro @ dw_dq
        J[:, 0:3, 16:19] = np.eye(3)
        J[:, 3:6, 9:16] = dt * da_dq
        J[:, 3:6, 19:22] = np.eye(3) - 0.5 * dt * _skew(a + b)
        Fx[:, 18:24, 0:22] = J
        Fi = np.zeros((n, 24, 13))
        Fi[:, 3:15, 0:12] = np.eye(12)
        Fi[:, 17, 12] = 1
        Fi[:, 18:21, 3:6] = dt * Ro @ _skew(p_p)
        Fi[:, 21:24, 3:6] = -dt * np.swapaxes(R_p, 1, 2)
        self.P = Fx @ self.P @ np.swapaxes(Fx, 1, 2) + (Fi * self.Qd[:, None, :]) @ np.swapaxes(Fi, 1, 2)
        self.Fx, self.Fi = Fx, Fi  # Filter.Fx / Filter.Fi of the last step
        self.om_old, self.acc_old = om.copy(), acc.copy()
        self.R_old = _q2R(self.x[:, 6:10])

    def update(self, cam_pos, cam_q, notch):
        n, x, P, H = self.n, self.x, self.P, self.H
        cam_pos = np.broadcast_to(np.asarray(cam_pos, dtype=float), (n, 3))
        cam_q = np.broadcast_to(np.asarray(cam_q, dtype=float), (n, 4))
        notch = np.broadcast_to(np.asarray(notch, dtype=float), (n,))
        Rm = np.zeros((n, 7, 7))
        Rm[:, np.arange(7), np.arange(7)] = self.Rd
        S = H @ P @ H.T + Rm
        K = P @ H.T @ np.linalg.inv(S)
        nq = np.stack([np.zeros(n), np.zeros(n), np.sin(notch / 2), np.cos(notch / 2)], -1)
        qm = _qmul(nq, cam_q)
        err_q = _qmul(qm * np.array([-1.0, -1.0, -1.0, 1.0]), x[:, 22:26])
        nv = np.sqrt(np.sum(err_q[:, :3] ** 2, -1))
        ang = np.arcsin(nv)
        f = np.where(ang == 0.0, 0.0, ang / np.where(nv > 0, nv, 1.0))
        res = np.concatenate([cam_pos - x[:, 19:22], err_q[:, :3] * f[:, None], (notch - x[:, 16])[:, None]], -1)
        d = np.einsum("nij,nj->ni", K, res)
        th, thc = d[:, 6:9], d[:, 21:24]
        dq = _about_axis(np.sqrt(np.sum(th * th, -1)), th)
        dqc = _about_axis(np.sqrt(np.sum(thc * thc, -1)), th)  # axis = theta (quirk Q4)
        dd = d[:, 9:15].copy()
        dd[:, self.frozen] = 0.0
        self.x = np.concatenate([x[:, 0:3] + d[:, 0:3], x[:, 3:6] + d[:, 3:6], _qmul(x[:, 6:10], dq), x[:, 10:16] + dd,
                                 x[:, 16:19] + d[:, 15:18], x[:, 19:22] + d[:, 18:21], _qmul(x[:, 22:26], dqc)], -1)
        M = np.eye(24) - K @ H
        P = M @ P @ np.swapaxes(M, 1, 2) + (K * self.Rd[:, None, :]) @ np.swapaxes(K, 1, 2)
        G = np.broadcast_to(np.eye(24), (n, 24, 24)).copy()
        G[:, 6:9, 6:9] = np.eye(3) - _skew(0.5 * th)
        G[:, 21:24, 21:24] = np.eye(3) - _skew(0.5 * thc)
        self.P = G @ P @ np.swapaxes(G, 1, 2)
        return K

    def run(self, dt, om_acc, n_prop, cam, notch):
        k = 0
        for e in range(len(n_prop)):
            for _ in range(int(n_prop[e])):
                self.propagate(dt[k], om_acc[k, :3], om_acc[k, 3:])
                k += 1
            self.update(cam[e, :3], cam[e, 3:], notch[e])
        return k
