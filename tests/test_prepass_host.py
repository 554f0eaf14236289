"""The product's numpy pre-pass (dvi_ekf_b200.camera.build_streams: camera-derived data, interpolation, synthetic IMU,
reference rows -- Camera.py:84-170,299-347, Interpolator.py:25-88, Imu.py:141-226, tools/utils.py:54-75) against the oracle's
restatement of the same flow, NOTCH FREE (the with_notch flow: tests/test_notch_flow.py), on every trajectory of data/trajs
and at the interpolation factors of the BASELINE configurations; and directly against the reference's imu_ref artefacts."""
import numpy as np
import pytest

from oracle.eskf_oracle import OracleConfig
from tests.helpers import Scenario, legacy_imu_ref

ROUND_FLOOR = 5.0e-10  # the artefacts are printed with 9 decimals (files.py:68-82)


def _close(x, y, tol, what):
    err = np.abs(np.asarray(x) - np.asarray(y)).max() / max(np.abs(y).max(), 1e-12)
    assert err < tol, (what, err)


@pytest.mark.parametrize("name,frames,ifv", [("traj_mandala0_mono", 10, 1), ("traj_mandala0_mono", 140, 10), ("traj_mandala0_gt", 115, 33),
                                             ("traj_trans_x", 60, 10), ("traj_rot_z", 60, 33), ("traj_from_prop", 50, 5)])
def test_product_prepass_matches_the_oracle_notch_free(golden, name, frames, ifv):
    from dvi_ekf_b200.camera import Camera, build_streams

    a = golden[name][:frames]
    sc = Scenario(a, OracleConfig(max_vals=frames, interframe_vals=ifv))
    s = build_streams(Camera(a[:, 0], a[:, 1:4], a[:, 4:8], scale=10.0), ifv, sc.cfg.length, sc.cfg.angle)
    assert np.array_equal(s.n_prop, sc.n_prop) and len(s.dt) == len(sc.dt)
    _close(s.x0, sc.x0, 1e-13, "x0")
    _close(s.u0, sc.u0, 1e-10, "u0")
    _close(s.dt, sc.dt, 1e-15, "dt")
    _close(s.om_acc[:, :3], sc.om_acc[:, :3], 1e-10, "om")
    _close(s.om_acc[:, 3:], sc.om_acc[:, 3:], 1e-10, "acc")
    _close(s.cam, sc.cam_meas, 1e-15, "cam")
    _close(s.notch, sc.notch_meas, 1e-15, "notch")
    _close(s.imu_ref_rows, sc.imu_ref_rows, 1e-10, "imu_ref_rows")


def test_product_prepass_reproduces_the_reference_imu_ref_file(golden):
    """imu_ref_mandala0_mono.txt (9 x 14), what Filter.save writes next to kf_best_*.txt (Filter.py:457-465), from the numpy
    pre-pass with the legacy camera-omega convention."""
    from dvi_ekf_b200.camera import Camera, build_streams

    a = golden["traj_mandala0_mono"][:10]
    s = build_streams(Camera(a[:, 0], a[:, 1:4], a[:, 4:8], scale=10.0, euler_mode="zyx_legacy"), 1, 50.0, np.deg2rad(30.0))
    ref = golden["imu_ref_mandala0_mono"]
    assert s.imu_ref_rows.shape == ref.shape == (9, 14)
    assert np.abs(s.imu_ref_rows - ref).max() <= ROUND_FLOOR


@pytest.mark.parametrize("kp, ifv, nfr", [("0.006", 10, 140), ("0.01", 50, 140), ("2.0", 50, 70), ("1.0", 5, 70)])
def test_product_prepass_reproduces_the_legacy_imu_ref_files(golden, kp, ifv, nfr):
    from dvi_ekf_b200.camera import Camera, build_streams

    a = golden["traj_mandala0_mono"][:nfr]
    s = build_streams(Camera(a[:, 0], a[:, 1:4], a[:, 4:8], scale=10.0, euler_mode="zyx_legacy"), ifv, 50.0, np.deg2rad(30.0))
    ref = legacy_imu_ref(kp)
    assert s.imu_ref_rows.shape == ref.shape and np.all(s.n_prop == ifv)
    cols = [0, 1, 2, 3, 7, 8, 9, 10, 11, 12, 13]  # (velocity columns: an older velocity definition, tests/test_oracle_golden.py)
    assert np.abs(s.imu_ref_rows[:, cols] - ref[:, cols]).max() <= ROUND_FLOOR
