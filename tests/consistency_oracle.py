"""The batch oracle with the innovation covariance and residual of its last update kept, for the NIS (TEST INFRASTRUCTURE)."""
import numpy as np

from oracle.batch_oracle import BatchOracle, _qmul


class RecordingOracle(BatchOracle):
    """``BatchOracle`` that also keeps ``S = H P H^T + R`` and the residual ``res`` of its last update (Filter.py:355-375),
    formed by the same expressions as ``BatchOracle.update``."""

    def update(self, cam_pos, cam_q, notch):
        n, x, P, H = self.n, self.x, self.P, self.H
        cam_pos = np.broadcast_to(np.asarray(cam_pos, dtype=float), (n, 3))
        cam_q = np.broadcast_to(np.asarray(cam_q, dtype=float), (n, 4))
        nt = np.broadcast_to(np.asarray(notch, dtype=float), (n,))
        Rm = np.zeros((n, 7, 7))
        Rm[:, np.arange(7), np.arange(7)] = self.Rd
        S = H @ P @ H.T + Rm
        nq = np.stack([np.zeros(n), np.zeros(n), np.sin(nt / 2), np.cos(nt / 2)], -1)
        qm = _qmul(nq, cam_q)
        err_q = _qmul(qm * np.array([-1.0, -1.0, -1.0, 1.0]), x[:, 22:26])
        nv = np.sqrt(np.sum(err_q[:, :3] ** 2, -1))
        ang = np.arcsin(nv)
        f = np.where(ang == 0.0, 0.0, ang / np.where(nv > 0, nv, 1.0))
        self.S = S
        self.res = np.concatenate([cam_pos - x[:, 19:22], err_q[:, :3] * f[:, None], (nt - x[:, 16])[:, None]], -1)
        return super().update(cam_pos, cam_q, notch)
