"""Pins the numpy oracle against the reference's own numeric artefacts
(data/trajs/kf_best_mandala0_mono.txt, imu_ref_mandala0_mono*.txt)."""
import numpy as np
import pytest

from oracle.eskf_oracle import (
    OracleConfig,
    Probe,
    build_streams,
    camera_from_arrays,
    run_reference_flow,
)
from tests.helpers import legacy_imu_ref

# the golden files are written with 9 decimals (tools/files.py:68-82)
ROUND_FLOOR = 5.0e-10 + 1e-15


def _run(golden, cfg, n=10):
    tr = golden["traj_mandala0_mono"][:n]
    return run_reference_flow(tr[:, 0], tr[:, 1:4], tr[:, 4:8], cfg)


def test_legacy_preset_reproduces_kf_best(golden):
    r = _run(golden, OracleConfig.legacy_golden())
    ref = golden["kf_best_mandala0_mono"]
    assert r.kf_rows.shape == ref.shape == (10, 30)
    assert np.abs(r.kf_rows - ref).max() <= ROUND_FLOOR


def test_legacy_preset_reproduces_imu_ref(golden):
    r = _run(golden, OracleConfig.legacy_golden())
    ref = golden["imu_ref_mandala0_mono"]
    assert r.imu_ref_rows.shape == ref.shape == (9, 14)
    assert np.abs(r.imu_ref_rows - ref).max() <= ROUND_FLOOR


@pytest.mark.parametrize(
    "kw, lo",
    [
        (dict(markley=False), 1e-3),  # Q1: SVD-orthogonalising from_matrix
        (dict(fix_q2=True), 10.0),  # Q2: v_tr = p_tr
        (dict(fix_q3=True), 1.0),  # Q3: Jacobian column mis-alignment
        (dict(fix_q4=True), 1.0),  # Q4: dqc axis = theta
    ],
)
def test_quirks_are_load_bearing(golden, kw, lo):
    """Flipping any single quirk breaks the golden match by orders of
    magnitude, i.e. the golden file really pins them."""
    r = _run(golden, OracleConfig.legacy_golden(**kw))
    assert np.abs(r.kf_rows - golden["kf_best_mandala0_mono"]).max() > lo


def test_head_deltas_vs_golden(golden):
    """HEAD differs from the golden revision by exactly Q7 and Q11."""
    ref = golden["kf_best_mandala0_mono"]
    q7 = _run(golden, OracleConfig(euler_mode="zyx_legacy"))
    assert np.abs(q7.kf_rows - ref).max() == pytest.approx(20.0, abs=1e-9)  # dof6 zeroed
    q11 = _run(golden, OracleConfig(zero_frozen_dofs=False))
    d = np.abs(q11.kf_rows - ref).max()
    assert 1e-3 < d < 1e-1


def test_head_mode_final_row(golden):
    """HEAD-mode expectation for config 1 (SURVEY section 8c)."""
    r = _run(golden, OracleConfig())
    last = r.kf_rows[-1]
    np.testing.assert_allclose(last[1:4], [-0.203684503, -40.582872809, -34.345751962], atol=5e-9)
    np.testing.assert_allclose(last[4:7], [-0.024313107, 0.170609201, -0.103690214], atol=5e-9)
    np.testing.assert_allclose(last[10:14], [0.514775575, -0.857321201, 0.002532295, -0.000231132], atol=5e-9)
    assert np.all(last[14:20] == 0.0)
    np.testing.assert_allclose(last[20:23], [0.046807223, 0.695593986, 0.240214951], atol=5e-9)
    np.testing.assert_allclose(last[26:30], [0.999882719, 0.015057016, 0.000728335, -0.002702629], atol=5e-9)


@pytest.mark.parametrize("kp, ifv, nfr", [("0.006", 10, 140), ("0.01", 50, 140), ("2.0", 50, 70), ("1.0", 5, 70)])
def test_legacy_imu_ref_pins_interpolation_path(golden, kp, ifv, nfr):
    """The interframe>1 pose / interpolation path (Interpolator + f_imu with
    the ground-truth probe) reproduces the legacy imu_ref files; their
    velocity columns come from an older velocity definition and are skipped."""
    tr = golden["traj_mandala0_mono"][:nfr]
    cfg = OracleConfig.legacy_golden(max_vals=nfr, interframe_vals=ifv)
    cam = camera_from_arrays(tr[:, 0], tr[:, 1:4], tr[:, 4:8], cfg)
    out = build_streams(cam, cfg, Probe(cfg.length, cfg.angle))
    rows, n_prop = out[-1], out[4]
    ref = legacy_imu_ref(kp)
    assert rows.shape == ref.shape
    assert np.all(n_prop == ifv)
    cols = [0, 1, 2, 3, 7, 8, 9, 10, 11, 12, 13]
    assert np.abs(rows[:, cols] - ref[:, cols]).max() <= ROUND_FLOOR
