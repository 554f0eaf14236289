"""The device arithmetic (eskf_math.cuh through the CPU harness tests/hostcheck) at orientations, residual angles and frame
timings the packaged trajectories never reach.

Every packaged trajectory keeps the IMU quaternion's w between 0.38 and 0.94, takes one branch of Markley's method
(quat_from_matrix) for q and one for q_cam, never wraps an Euler angle and has uniform frame stamps.  Here:

* the mandala trajectory in 37 turned worlds (tests/helpers.py world_rotations, RotatedScenario), replayed step by step in
  lock step with the oracle at 1e-9: all four Markley branches for q and for q_cam, w-sign flips, an Euler wrap;
* camera measurements 180 deg away from q_cam, where |v| of the residual quaternion is 1 up to rounding and math.asin of the
  reference may raise (ESKF_STATUS_ASIN_DOMAIN), and a band of residual angles from 90 to 179.9 deg;
* jittered frame stamps with an epoch of no IMU sample and a 3x gap, through the oracle's and the product's pre-pass;
* the Euler angles of the update MSE near gimbal lock, where the kernels' formula and the installed scipy part ways."""
import ctypes

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

from oracle.eskf_oracle import OracleConfig, OracleFilter, quat_mul
from tests.helpers import (RotatedScenario, Scenario, cov_err, mandala_scenario, markley_branch, random_filter_inputs,
                           state_err, world_rotations)

TOL = 1e-9
ULP1 = np.finfo(float).eps  # one ulp of 1.0 (spacing above 1; below 1 it is half of this)
dp = ctypes.POINTER(ctypes.c_double)


def _p(a):
    return a.ctypes.data_as(dp)


@pytest.fixture(scope="module")
def hc():
    from dvi_ekf_b200 import build

    lib = ctypes.CDLL(build.build_hostcheck())
    lib.hc_propagate3.argtypes = [dp, dp, dp, dp, dp, ctypes.c_double, dp, dp, dp, dp]
    lib.hc_propagate3.restype = None
    lib.hc_update3.argtypes = [dp, dp, dp, dp, dp, dp, ctypes.c_double, dp, dp]
    lib.hc_update3.restype = ctypes.c_int
    return lib


def _model(cfg):
    mask = sum(1 << i for i, f in enumerate(cfg.frozen_dofs) if f)
    return np.array([cfg.length, cfg.angle, float(mask), 1.0 if cfg.zero_frozen_dofs else 0.0])


class _Recording(OracleFilter):
    """The oracle, noting the Markley branch of every matrix it turns into a quaternion (q and q_cam alternate) and whether
    the raw quaternion had w < 0, i.e. whether the w >= 0 convention flipped its sign."""

    def _mat2quat(self, M):
        from oracle.eskf_oracle import quat_from_matrix_scipy110

        self.branches.append(markley_branch(M))
        self.flips += int(quat_from_matrix_scipy110(M)[3] < 0)
        return super()._mat2quat(M)


@pytest.fixture(scope="module")
def replays(hc, golden):
    """Every turned world in lock step: per-step worst state / covariance / gain error of hc_propagate3 + hc_update3 against
    the oracle started from the same state, and the branches and sign flips the run visited."""
    sc = mandala_scenario(golden, n_frames=25, ifv=10)
    model = _model(sc.cfg)
    out = {}
    for name, G in world_rotations(sc).items():
        rs = RotatedScenario(sc, G, name)
        kf = rs.new_oracle(cls=_Recording)
        kf.branches, kf.flips = [], 0
        ws = wP = wK = 0.0
        k = 0
        for e in range(len(rs.n_prop)):
            for _ in range(rs.n_prop[e]):
                x, P, u, Ro = [a.copy() for a in kf.get_vectors()]
                kf.propagate(rs.dt[k], rs.om_acc[k, :3], rs.om_acc[k, 3:])
                oa = rs.om_acc[k].copy()
                hc.hc_propagate3(_p(model), _p(x), _p(P), _p(u), _p(Ro), rs.dt[k], _p(oa), _p(rs.Qd), _p(rs.sig_om), None)
                xr, Pr, ur, Rr = kf.get_vectors()
                ws = max(ws, state_err(x, xr), np.abs(Ro - Rr).max(), np.abs(u - ur).max())
                wP = max(wP, cov_err(P, Pr))
                k += 1
            x, P, u, Ro = [a.copy() for a in kf.get_vectors()]
            K = kf.update(rs.cam_meas[e, :3], rs.cam_meas[e, 3:], rs.notch_meas[e])
            assert K is not None, (name, e)
            cm = rs.cam_meas[e].copy()
            Kd = np.zeros((24, 7))
            assert hc.hc_update3(_p(model), _p(x), _p(P), _p(u), _p(Ro), _p(cm), rs.notch_meas[e], _p(rs.Rd), _p(Kd)) == 1, (name, e)
            xr, Pr, _, _ = kf.get_vectors()
            ws = max(ws, state_err(x, xr))
            if e > 0:
                wP = max(wP, cov_err(P, Pr, rs.Rd))
            wK = max(wK, np.abs(Kd - K).max() / np.abs(K).max())
        out[name] = dict(ws=ws, wP=wP, wK=wK, q=set(kf.branches[0::2]), qc=set(kf.branches[1::2]), flips=kf.flips,
                         cam_ref=rs.cam_ref, x0=rs.x0)
    return out


def test_turned_worlds_replay_in_lock_step(replays):
    """hc_propagate3 / hc_update3 (the building blocks of eskf_kernel3) against the oracle in every turned world, 240 steps
    and 24 updates each: the 1e-9 bound of tests/test_hostcheck.py.  The covariance after the FIRST update is not checked, as
    in test_hostcheck.py::test_lockstep_random_tunings: the prior is up to 5e15 times R there and the reference does not
    determine the result (tests/test_conditioning.py); in some turned worlds a one-ulp change of the oracle's own prior moves
    its DOF block by 1.4e-7."""
    for n, r in replays.items():
        print(f"MEASURED lock step {n}: state {r['ws']:.1e} P {r['wP']:.1e} K {r['wK']:.1e}")
    bad = {n: (r["ws"], r["wP"], r["wK"]) for n, r in replays.items() if not (r["ws"] < TOL and r["wP"] < TOL and r["wK"] < 1e-7)}
    assert not bad, bad


def test_turned_worlds_cover_every_branch(replays):
    """What the turned worlds are for: all four Markley branches for q and for q_cam in a whole run (the packaged
    trajectories reach branch 0 for q and 3 for q_cam only), the w >= 0 flip during a run, an initial q at exactly 180 deg
    from the identity (w = 0), and a camera roll that wraps through +-180 deg between two updates."""
    assert set().union(*(r["q"] for r in replays.values())) == {0, 1, 2, 3}
    assert set().union(*(r["qc"] for r in replays.values())) == {0, 1, 2, 3}
    assert replays["y150"]["q"] == {2} and replays["y150"]["qc"] == {1}
    assert replays["z150"]["q"] == {1} and replays["z150"]["qc"] == {2}
    assert abs(replays["x-60"]["x0"][9]) < 1e-15 and replays["x-60"]["flips"] > 0
    assert sum(r["flips"] > 0 for r in replays.values()) >= 8
    roll = replays["roll-wrap"]["cam_ref"][:, 3]
    assert np.abs(np.diff(roll)).max() > 300.0  # a jump of ~360 deg: the wrap lies between two frames
    assert np.abs(roll).max() > 179.0
    assert np.abs(np.diff(replays["identity"]["cam_ref"][:, 3])).max() < 10.0


# ---- residual at 180 deg: the domain of asin --------------------------------------------------------------------------


def _dev_normalise(q):
    """quat_normalise of eskf_math.cuh, operation for operation: q * (sign / |q|)"""
    d = np.sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3])
    return q * ((-1.0 if q[3] < 0.0 else 1.0) / d)


def _dev_mul(a, b):
    """quat_mul of eskf_math.cuh, operation for operation"""
    w = a[3] * b[3] - (a[0] * b[0] + a[1] * b[1] + a[2] * b[2])
    c = (a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0])
    return _dev_normalise(np.array([a[3] * b[0] + b[3] * a[0] + c[0], a[3] * b[1] + b[3] * a[1] + c[1],
                                    a[3] * b[2] + b[3] * a[2] + c[2], w]))


def residual_norms(q_cam, cam_q):
    """|v| of the residual quaternion conj(notch * cam_q) * q_cam for a zero notch angle: (the oracle's value, the value of
    eskf_math.cuh's update_residual restated operation for operation without contraction -- what the g++ build computes)"""
    from oracle.eskf_oracle import quat_conj

    e = quat_mul(quat_conj(quat_mul(np.array([0.0, 0.0, 0.0, 1.0]), cam_q)), q_cam)
    qm = _dev_mul(np.array([0.0, 0.0, 0.0, 1.0]), cam_q)
    ed = _dev_mul(qm * np.array([-1.0, -1.0, -1.0, 1.0]), q_cam)
    return float(np.linalg.norm(e[:3])), float(np.sqrt(ed[0] * ed[0] + ed[1] * ed[1] + ed[2] * ed[2]))


def asin_domain_inputs(cfg, n, seed, band=False):
    """n random filter states (tests/helpers.py random_filter_inputs) and camera measurements whose rotation is q_cam turned
    by exactly 180 deg about a seeded axis (|v| = 1 up to rounding), or with band=True by an angle drawn from 90 .. 179.9 deg.
    The raw measured quaternion is scaled by a seeded norm (the residual normalises it).  Notch measurement 0."""
    rng = np.random.default_rng(seed)
    xs, Ps, us = random_filter_inputs(rng, n, cfg, frozen=True)
    cam = np.empty((n, 7))
    for i in range(n):
        u = rng.normal(size=3)
        u /= np.linalg.norm(u)
        half = np.deg2rad(rng.uniform(90.0, 179.9)) / 2 if band else np.pi / 2
        a = np.array([*(np.sin(half) * u), np.cos(half)])
        cam[i, :3] = xs[i, 19:22] + rng.normal(0.0, 0.05, 3)
        cam[i, 3:] = quat_mul(xs[i, 22:26], a) * rng.uniform(0.5, 2.0)
    return xs, Ps, us, cam


def oracle_update(cfg, probe, x, P, u, cam):
    """Filter.update on one filter: (x+, P+, K), or None where math.asin raises (|v| > 1)"""
    from oracle.eskf_oracle import State

    kf = OracleFilter(cfg, State.from_vector(x), P, u[:3], u[3:], probe)
    try:
        K = kf.update(cam[:3], cam[3:], 0.0)
    except ValueError:
        return None
    return kf.x.as_vector(), kf.P, K


@pytest.mark.parametrize("band", [False, True], ids=["180deg", "90-179.9deg"])
def test_asin_domain_host(hc, golden, band):
    """hc_update3 on measurements 180 deg from q_cam: it skips (returns 0, x and P untouched) exactly where its own |v|,
    restated here operation for operation, exceeds 1; the oracle raises exactly where ITS |v| exceeds 1.  The two disagree
    input by input, and only within 2 ulp of |v| = 1: the kernels normalise a quaternion by multiplying with the reciprocal
    of its norm (eskf_math.cuh quat_normalise), the reference divides, and at 180 deg that last-bit difference decides the
    test of |v| against 1.  Neither side is the better answer there: the reference's own outcome is the rounding of its
    operations.  Where both apply a 180-deg update the results are not compared: the residual's direction is the sign of
    the rounding error of w (the w >= 0 convention), and asin at 1 turns one ulp of |v| into 1e-8 of the angle.  In the band
    of 90 .. 179.9 deg no input is near the domain's edge and every update agrees with the oracle at 1e-9."""
    sc = mandala_scenario(golden, n_frames=3, ifv=1)
    model = _model(sc.cfg)
    n = 3000
    xs, Ps, us, cam = asin_domain_inputs(sc.cfg, n, 97 if not band else 98, band)
    flagged = raised = differ = 0
    worst = 0.0
    for i in range(n):
        nv_o, nv_d = residual_norms(xs[i, 22:26], cam[i, 3:])
        x, P, Ro = xs[i].copy(), Ps[i].copy(), np.eye(3).reshape(9)
        Kd = np.zeros((24, 7))
        r = hc.hc_update3(_p(model), _p(x), _p(P), _p(us[i].copy()), _p(Ro), _p(cam[i].copy()), 0.0, _p(sc.Rd), _p(Kd))
        ref = oracle_update(sc.cfg, sc.probe, xs[i], Ps[i], us[i], cam[i])
        assert (r == 0) == (nv_d > 1.0), (i, nv_d)
        assert (ref is None) == (nv_o > 1.0), (i, nv_o)
        if r == 0:
            flagged += 1
            assert np.array_equal(x, xs[i]) and np.array_equal(P, Ps[i]) and not Kd.any()
        raised += ref is None
        if (r == 0) != (ref is None):
            differ += 1
            assert abs(nv_o - 1.0) <= 2 * ULP1, (i, nv_o)
        if band and r == 1 and ref is not None:
            worst = max(worst, state_err(x, ref[0]), cov_err(P, ref[1], sc.Rd))
    print(f"MEASURED asin domain, {n} inputs ({'band' if band else '180 deg'}): hc_update3 skips {flagged}, the oracle raises "
          f"{raised}, they differ on {differ}" + (f"; updates vs oracle {worst:.2e}" if band else ""))
    assert worst < TOL
    if band:
        assert flagged == raised == 0
    else:
        assert flagged > 0 and raised > 0


# ---- irregular frame stamps ---------------------------------------------------------------------------------------------


def jittered_camera(golden, name="traj_mandala0_mono", frames=30, seed=3, G=None):
    """Frame stamps t_k = k + U(-0.3, 0.3) (seeded), then two frames 0.02 apart (closer than one IMU interval of ~0.1:
    an epoch without IMU sample) and one gap of 3 intervals.  The positions and raw quaternions are the trajectory's rows.
    With G: xyz turned by G and the raw quaternions by its quaternion, their signs kept continuous (the interpolation
    reads the raw components).  Returns t, xyz, q."""
    a = golden[name][:frames]
    rng = np.random.default_rng(seed)
    t = np.arange(frames, dtype=float) + rng.uniform(-0.3, 0.3, frames)
    t[0] = 0.0
    t[12] = t[11] + 0.02
    t[20:] += 2.0  # frames 19 -> 20: about 3 s
    xyz, q = a[:, 1:4].copy(), a[:, 4:8].copy()
    if G is not None:
        g = Rotation.from_matrix(G).as_quat()
        xyz = xyz @ np.asarray(G).T
        q = np.array([quat_mul(g, qi) * np.linalg.norm(qi) for qi in q])
        for i in range(1, len(q)):
            if q[i] @ q[i - 1] < 0:
                q[i] = -q[i]
    assert np.all(np.diff(t) > 0)
    return t, xyz, q


@pytest.mark.parametrize("world", [None, "roll-wrap", "y150"])
def test_irregular_stamps_product_prepass_matches_oracle(golden, world):
    """The oracle's build_streams and the product's numpy pre-pass (dvi_ekf_b200.camera) on jittered stamps: n_prop exactly
    equal (float comparisons of interpolated instants against frame stamps, Camera.py:320-347), an epoch of 0 steps and a
    long one present; the other streams within the bounds of tests/test_prepass_host.py.  (np.gradient takes t[1] - t[0]
    as the spacing of every frame, as the reference does: the derived rates are what the reference computes, not the true
    ones.)  In the turned worlds the Euler angles of the camera wrap inside the gradient (roll-wrap)."""
    from dvi_ekf_b200.camera import Camera, build_streams

    sc0 = mandala_scenario(golden, n_frames=30, ifv=10)
    G = None if world is None else world_rotations(sc0)[world]
    t, xyz, q = jittered_camera(golden, G=G)
    ifv = 10
    sc = Scenario(np.hstack((t[:, None], xyz, q)), OracleConfig(max_vals=len(t), interframe_vals=ifv))
    s = build_streams(Camera(t, xyz, q, scale=10.0), ifv, sc.cfg.length, sc.cfg.angle)
    assert np.array_equal(s.n_prop, sc.n_prop) and len(s.dt) == len(sc.dt)
    assert (sc.n_prop == 0).any() and sc.n_prop.max() >= 3 * np.median(sc.n_prop)
    assert np.ptp(sc.dt) > 0.05  # the first step of an epoch runs from the frame stamp to the next interpolated instant

    def close(x, y, tol, what):
        err = np.abs(np.asarray(x) - np.asarray(y)).max() / max(np.abs(y).max(), 1e-12)
        assert err < tol, (what, err)

    close(s.x0, sc.x0, 1e-13, "x0")
    close(s.u0, sc.u0, 1e-10, "u0")
    close(s.dt, sc.dt, 1e-15, "dt")
    close(s.om_acc[:, :3], sc.om_acc[:, :3], 1e-10, "om")
    close(s.om_acc[:, 3:], sc.om_acc[:, 3:], 1e-10, "acc")
    close(s.cam, sc.cam_meas, 1e-15, "cam")
    close(s.imu_ref_rows, sc.imu_ref_rows, 1e-10, "imu_ref_rows")
    if world == "roll-wrap":
        eul = Rotation.from_quat(q).as_euler("xyz", degrees=True)
        assert np.abs(np.diff(eul[:, 0])).max() > 300.0  # the wrap is inside the camera data


# ---- Euler angles near gimbal lock --------------------------------------------------------------------------------------


def kernel_euler_xyz_deg(q):
    """The kernels' Euler angles (eskf_kernel.cuh euler_xyz_deg, eskf_kernel3.cuh flush_stats, the post-pass of eskf_api.cu):
    atan2(R21, R22), -asin(clamp(R20)), atan2(R10, R00), in degrees; q [n,4] xyzw"""
    from tests.helpers import quat_to_matrix

    R = np.array([quat_to_matrix(qi) for qi in q])
    return np.rad2deg(np.stack([np.arctan2(R[:, 2, 1], R[:, 2, 2]), -np.arcsin(np.clip(R[:, 2, 0], -1, 1)),
                                np.arctan2(R[:, 1, 0], R[:, 0, 0])], -1))


def test_euler_angles_near_gimbal_lock():
    """The deviation DESIGN.md records: the kernels' xyz Euler angles against the installed scipy's as_euler("xyz"), the
    oracle's Euler function.  Away from pitch +-90 deg they agree to rounding; the difference grows as 1 / cos(pitch); within
    about 1e-6 deg of gimbal lock scipy takes its degenerate branch and sets the third angle to 0, so the two describe the same
    rotation with roll and yaw traded (up to a full turn apart).  The parity tests therefore stay at |pitch| <= 89.99 deg."""
    rng = np.random.default_rng(12)
    out = {}
    for off in (None, 1e-2, 1e-4, 1e-6):
        n = 2000
        if off is None:
            q = Rotation.random(n, random_state=5).as_quat()
        else:
            e = np.stack([rng.uniform(-180, 180, n), np.where(rng.random(n) < 0.5, -1, 1) * (90.0 - off),
                          rng.uniform(-180, 180, n)], -1)
            q = Rotation.from_euler("xyz", e, degrees=True).as_quat()
        d = np.abs(kernel_euler_xyz_deg(q) - Rotation.from_quat(q).as_euler("xyz", degrees=True))
        d = np.minimum(d, 360.0 - d)  # the same angle across the +-180 deg seam
        out[off] = d.max()
    print("MEASURED kernel Euler angles vs scipy, largest difference (deg): "
          + ", ".join(f"{'random' if k is None else f'pitch 90 - {k:g}'}: {v:.1e}" for k, v in out.items()))
    assert out[None] < 1e-11 and out[1e-2] < 1e-8 and out[1e-4] < 1e-6
    assert out[1e-6] > 1.0  # inside the band: the other branch of the degenerate decomposition
