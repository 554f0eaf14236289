"""SURVEY 8f rank 1: the GPU pre-pass (eskf_prepass) against the numpy pre-pass of the product (dvi_ekf_b200.camera,
itself pinned by the oracle's build_streams and the reference's imu_ref_* golden files), and the filter run on
device-resident streams that never touched the host."""
import numpy as np
import pytest

from tests.helpers import cov_err, legacy_imu_ref, mandala_scenario, model_kwargs, state_err

pytestmark = pytest.mark.gpu

LENGTH, ANGLE = 50.0, np.deg2rad(30.0)


def _both(golden, name, frames, ifv, scale=10.0, euler_mode="xyz"):
    from dvi_ekf_b200.camera import Camera, build_streams
    from dvi_ekf_b200.prepass import build_streams_gpu

    a = golden[name][:frames]
    t, xyz, q = a[:, 0].copy(), a[:, 1:4].copy(), a[:, 4:8].copy()
    host = build_streams(Camera(t, xyz, q, scale=scale, euler_mode=euler_mode), ifv, LENGTH, ANGLE)
    dev = build_streams_gpu(t, xyz, q, ifv, LENGTH, ANGLE, scale=scale, euler_mode=euler_mode)
    return host, dev


@pytest.mark.parametrize("name,frames,ifv,mode", [("traj_mandala0_mono", 140, 10, "xyz"), ("traj_mandala0_mono", 10, 1, "zyx_legacy"),
                                                  ("traj_rot_z", 60, 33, "xyz"), ("traj_from_prop", 50, 5, "xyz"),
                                                  ("traj_mandala0_gt", 115, 33, "xyz")])
def test_gpu_prepass_matches_the_numpy_prepass(golden, name, frames, ifv, mode):
    host, dev = _both(golden, name, frames, ifv, euler_mode=mode)
    T = len(host.dt)
    assert dev.n_steps == T
    assert np.array_equal(dev.n_prop.cpu().numpy(), host.n_prop)

    def close(a, b, tol, what):
        a, b = np.asarray(a), np.asarray(b)
        err = np.abs(a - b).max() / max(np.abs(b).max(), 1e-12)
        assert err < tol, (what, err)

    g = lambda x: x.cpu().numpy()
    close(g(dev.dt)[:T], host.dt, 1e-12, "dt")
    close(g(dev.t_imu)[:T], host.t_imu, 1e-14, "t_imu")
    close(g(dev.om_acc)[:T, :3], host.om_acc[:, :3], 1e-10, "om")  # second differences of Euler angles: ~1e-13 abs
    close(g(dev.om_acc)[:T, 3:], host.om_acc[:, 3:], 1e-10, "acc")
    close(g(dev.cam), host.cam, 1e-15, "cam")
    close(g(dev.notch), host.notch, 1e-15, "notch")
    close(g(dev.cam_ref), host.cam_ref, 1e-12, "cam_ref")
    close(g(dev.imu_ref), host.imu_ref, 1e-10, "imu_ref")
    close(g(dev.imu_ref_rows)[:T], host.imu_ref_rows, 1e-10, "imu_ref_rows")
    close(g(dev.x0), host.x0, 1e-12, "x0")
    close(g(dev.u0), host.u0, 1e-10, "u0")


def test_filter_on_device_resident_streams(golden):
    """trajectory -> eskf_prepass -> eskf_run without a host copy of the streams; result = the oracle on its own streams"""
    from dvi_ekf_b200 import BatchFilter
    from dvi_ekf_b200.prepass import build_streams_gpu

    frames, ifv = 20, 10
    sc = mandala_scenario(golden, n_frames=frames, ifv=ifv)
    a = golden["traj_mandala0_mono"][:frames]
    ds = build_streams_gpu(a[:, 0], a[:, 1:4], a[:, 4:8], ifv, sc.cfg.length, sc.cfg.angle, scale=10.0)
    T = ds.n_steps
    assert T == len(sc.dt)
    import torch

    n = 8
    dev = ds.dt.device
    dd = lambda x: torch.tensor(np.ascontiguousarray(x), dtype=torch.float64, device=dev)
    with BatchFilter(n, **model_kwargs(sc.cfg)) as bf:
        bf.set_noise(sc.Qd[None], sc.Rd[None], sc.sig_om[None])
        bf.set_state(ds.x0[None].contiguous(), dd(sc.P0[None]), ds.u0[None].contiguous(), None)
        bf.run(ds.dt[:T].contiguous(), ds.om_acc[:T].contiguous(), ds.n_prop, ds.cam, ds.notch, cam_ref=ds.cam_ref, imu_ref=ds.imu_ref,
               stats_on_device=True)
        xg, Pg, ug, Rg, st = bf.get_state()
    kf = sc.new_oracle()
    k = 0
    for e in range(len(sc.n_prop)):
        for _ in range(sc.n_prop[e]):
            kf.propagate(sc.dt[k], sc.om_acc[k, :3], sc.om_acc[k, 3:])
            k += 1
        kf.update(sc.cam_meas[e, :3], sc.cam_meas[e, 3:], sc.notch_meas[e])
    xr, Pr, ur, Rr = kf.get_vectors()
    assert np.all(st == 0)
    # inputs agree to ~1e-12 (two implementations of the pre-pass); 190 free-running steps
    print(f"MEASURED device-resident streams (190 free-running steps): state {state_err(xg[0], xr):.2e} P {cov_err(Pg[0], Pr, sc.Rd):.2e}")
    assert state_err(xg[0], xr) < 5e-12 and cov_err(Pg[0], Pr, sc.Rd) < 5e-13  # measured 8.1e-13 / 3.4e-14


ROUND_FLOOR = 5.0e-10  # the artefacts are printed with 9 decimals (files.py:68-82)


def test_gpu_prepass_reproduces_the_reference_imu_ref_file(golden):
    """eskf_prepass pinned to the reference's own artefact: its imu_ref rows (Imu.eval_expr_single / ImuRefTraj,
    Imu.py:141-226) for the default main.py run are data/trajs/imu_ref_mandala0_mono.txt (9 x 14), to the file's rounding."""
    _, dev = _both(golden, "traj_mandala0_mono", 10, 1, euler_mode="zyx_legacy")
    rows = dev.imu_ref_rows.cpu().numpy()[: dev.n_steps]
    ref = golden["imu_ref_mandala0_mono"]
    assert rows.shape == ref.shape == (9, 14)
    assert np.abs(rows - ref).max() <= ROUND_FLOOR, np.abs(rows - ref).max()


@pytest.mark.parametrize("kp, ifv, nfr", [("0.006", 10, 140), ("0.01", 50, 140), ("2.0", 50, 70), ("1.0", 5, 70)])
def test_gpu_prepass_reproduces_the_legacy_imu_ref_files(golden, kp, ifv, nfr):
    """The interpolation path at interframe_vals > 1 (Interpolator.py:25-88: np.linspace / np.interp / slerp, then f_imu
    with the ground-truth probe) on the DEVICE against the four legacy imu_ref_*_upd_* artefacts -- the same column set as
    tests/test_oracle_golden.py (their velocity columns come from an older velocity definition)."""
    _, dev = _both(golden, "traj_mandala0_mono", nfr, ifv, euler_mode="zyx_legacy")
    rows = dev.imu_ref_rows.cpu().numpy()[: dev.n_steps]
    ref = legacy_imu_ref(kp)
    assert rows.shape == ref.shape
    assert np.all(dev.n_prop.cpu().numpy() == ifv)
    cols = [0, 1, 2, 3, 7, 8, 9, 10, 11, 12, 13]
    assert np.abs(rows[:, cols] - ref[:, cols]).max() <= ROUND_FLOOR, np.abs(rows[:, cols] - ref[:, cols]).max()
