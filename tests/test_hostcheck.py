"""Device arithmetic on the CPU: dvi_ekf_b200/csrc/eskf_math.cuh compiled with g++ (tests/hostcheck) and
replayed lane by lane, checked against the numpy oracle in lock-step at 1e-9 (norm-wise per state group /
covariance block, tests/helpers.py).  Covers the first kernel's path (hc_propagate) and the building blocks of
the warp-specialised kernel (hc_propagate3: split scalar roles, register tile, transposition)."""
import ctypes
import os

import numpy as np
import pytest

from tests.helpers import cov_err, mandala_scenario, random_filter_inputs, state_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 1e-9
dp = ctypes.POINTER(ctypes.c_double)


def _p(a):
    return a.ctypes.data_as(dp)


@pytest.fixture(scope="module")
def hc():
    from dvi_ekf_b200 import build

    lib = ctypes.CDLL(build.build_hostcheck())
    for name in ("hc_propagate", "hc_propagate3"):
        getattr(lib, name).argtypes = [dp, dp, dp, dp, dp, ctypes.c_double, dp, dp, dp, dp]
        getattr(lib, name).restype = None
    for name in ("hc_update", "hc_update3"):
        getattr(lib, name).argtypes = [dp, dp, dp, dp, dp, dp, ctypes.c_double, dp, dp]
        getattr(lib, name).restype = ctypes.c_int
    return lib


def _model(cfg):
    mask = sum(1 << i for i, f in enumerate(cfg.frozen_dofs) if f)
    return np.array([cfg.length, cfg.angle, float(mask), 1.0 if cfg.zero_frozen_dofs else 0.0])


@pytest.mark.parametrize("fn,ufn", [("hc_propagate", "hc_update"), ("hc_propagate3", "hc_update3")])
def test_lockstep_trajectory(hc, golden, fn, ufn):
    sc = mandala_scenario(golden, n_frames=30, ifv=10)
    kf = sc.new_oracle()
    model = _model(sc.cfg)
    step = getattr(hc, fn)
    k = 0
    ws = wP = 0.0
    for e in range(len(sc.n_prop)):
        for _ in range(sc.n_prop[e]):
            x, P, u, Ro = [a.copy() for a in kf.get_vectors()]
            kf.propagate(sc.dt[k], sc.om_acc[k, :3], sc.om_acc[k, 3:])
            oa = sc.om_acc[k].copy()
            step(_p(model), _p(x), _p(P), _p(u), _p(Ro), sc.dt[k], _p(oa), _p(sc.Qd), _p(sc.sig_om), None)
            xr, Pr, ur, Rr = kf.get_vectors()
            ws = max(ws, state_err(x, xr), np.abs(Ro - Rr).max(), np.abs(u - ur).max())
            wP = max(wP, cov_err(P, Pr))
            k += 1
        x, P, u, Ro = [a.copy() for a in kf.get_vectors()]
        K = kf.update(sc.cam_meas[e, :3], sc.cam_meas[e, 3:], sc.notch_meas[e])
        cm = sc.cam_meas[e].copy()
        Kd = np.zeros((24, 7))
        assert getattr(hc, ufn)(_p(model), _p(x), _p(P), _p(u), _p(Ro), _p(cm), sc.notch_meas[e], _p(sc.Rd), _p(Kd)) == 1
        xr, Pr, _, _ = kf.get_vectors()
        ws = max(ws, state_err(x, xr))
        wP = max(wP, cov_err(P, Pr, sc.Rd))
        assert np.abs(Kd - K).max() / np.abs(K).max() < 1e-7
    assert ws < TOL and wP < TOL, (ws, wP)


@pytest.mark.parametrize("imu_q", [False, True])
def test_v3_blocks_equal_v1_path_on_random_states(hc, golden, imu_q):
    """hc_propagate3 (kernel-3 building blocks) against hc_propagate (v1 path) and the oracle on random, non-frozen
    states with non-zero notch rates; with and without IMU noise in Q (Filter.py:110-117)."""
    sc = mandala_scenario(golden, n_frames=10, ifv=1, frozen_dofs=(0, 0, 0, 0, 0, 0))
    rng = np.random.default_rng(7)
    xs, Ps, us = random_filter_inputs(rng, 200, sc.cfg)
    model = _model(sc.cfg)
    qd = sc.Qd.copy()
    if imu_q:
        qd[0:6] = np.array([3e-4, 3e-4, 3e-4, 2e-5, 2e-5, 2e-5])
    w12 = ws = wP = 0.0
    for i in range(len(xs)):
        dt = float(rng.uniform(0.01, 1.0))
        oa = np.hstack((rng.normal(0, 0.05, 3), rng.normal(0, 0.5, 3)))
        kf = sc.new_oracle(xs[i], Ps[i], us[i])
        kf.Q = np.diag(qd)
        x0, P0, u0, R0 = [a.copy() for a in kf.get_vectors()]
        kf.propagate(dt, oa[:3], oa[3:])
        xr, Pr, ur, Rr = kf.get_vectors()
        outs = []
        for fn in (hc.hc_propagate, hc.hc_propagate3):
            x, P, u, Ro = x0.copy(), P0.copy(), u0.copy(), R0.copy()
            fn(_p(model), _p(x), _p(P), _p(u), _p(Ro), dt, _p(oa.copy()), _p(qd), _p(sc.sig_om), None)
            outs.append((x, P, u, Ro))
            ws = max(ws, state_err(x, xr), np.abs(Ro - Rr).max())
            wP = max(wP, cov_err(P, Pr))
        w12 = max(w12, state_err(outs[1][0], outs[0][0]), cov_err(outs[1][1], outs[0][1]))
    assert ws < TOL and wP < TOL, (ws, wP)
    assert w12 < 1e-12, w12


@pytest.mark.parametrize("fn,ufn", [("hc_propagate", "hc_update"), ("hc_propagate3", "hc_update3")])
def test_free_running_low_process_noise(hc, golden, fn, ufn):
    """Regression: 40 free-running epochs with the DOF random walks 10x smaller than config.yaml (a point of the BASELINE
    config-3 tuning grid).  A version of the register-tile path that did not exchange the identity rows 9:15 of Fx between
    its two passes (lanes 3 and 4 kept their own tile, "P is symmetric") passed every lock-step and default-tuning test
    and blew up here: the asymmetry of the stored covariance grew tenfold per epoch (1e-14 -> 1e-6 after 12 updates,
    covariance error 1e+4) while the oracle stays put.  Both device paths must stay with the oracle."""
    sc = mandala_scenario(golden, n_frames=41, ifv=10)
    model = _model(sc.cfg)
    Qd = sc.Qd.copy()
    Qd[6:12] *= 0.01
    kf = sc.new_oracle()
    kf.Q = np.diag(Qd)
    x, P, u, Ro = [a.copy() for a in kf.get_vectors()]
    k = 0
    for e in range(len(sc.n_prop)):
        for _ in range(sc.n_prop[e]):
            kf.propagate(sc.dt[k], sc.om_acc[k, :3], sc.om_acc[k, 3:])
            oa = sc.om_acc[k].copy()
            getattr(hc, fn)(_p(model), _p(x), _p(P), _p(u), _p(Ro), sc.dt[k], _p(oa), _p(Qd), _p(sc.sig_om), None)
            k += 1
        assert kf.update(sc.cam_meas[e, :3], sc.cam_meas[e, 3:], sc.notch_meas[e]) is not None
        cm = sc.cam_meas[e].copy()
        Kd = np.zeros((24, 7))
        assert getattr(hc, ufn)(_p(model), _p(x), _p(P), _p(u), _p(Ro), _p(cm), sc.notch_meas[e], _p(sc.Rd), _p(Kd)) == 1
    xr, Pr, _, _ = kf.get_vectors()
    asym = np.abs(P - P.T).max() / np.abs(P).max()
    assert state_err(x, xr) < 1e-7 and cov_err(P, Pr, sc.Rd) < 1e-7 and asym < 1e-11, (state_err(x, xr), cov_err(P, Pr, sc.Rd), asym)


@pytest.mark.parametrize("fn,ufn", [("hc_propagate", "hc_update"), ("hc_propagate3", "hc_update3")])
def test_free_running_unfrozen_dofs(hc, golden, fn, ufn):
    """The calibration use case: all six DOFs estimated (config.yaml freezes them), perturbed initial DOFs, 40 epochs."""
    sc = mandala_scenario(golden, n_frames=41, ifv=10, frozen_dofs=[False] * 6)
    model = _model(sc.cfg)
    x0 = sc.x0.copy()
    x0[10:13] += np.deg2rad([2.0, -3.0, 1.5])
    x0[13:16] += [2.0, -1.0, 3.0]
    kf = sc.new_oracle(x0=x0)
    x, P, u, Ro = [a.copy() for a in kf.get_vectors()]
    k = 0
    for e in range(len(sc.n_prop)):
        for _ in range(sc.n_prop[e]):
            kf.propagate(sc.dt[k], sc.om_acc[k, :3], sc.om_acc[k, 3:])
            oa = sc.om_acc[k].copy()
            getattr(hc, fn)(_p(model), _p(x), _p(P), _p(u), _p(Ro), sc.dt[k], _p(oa), _p(sc.Qd), _p(sc.sig_om), None)
            k += 1
        assert kf.update(sc.cam_meas[e, :3], sc.cam_meas[e, 3:], sc.notch_meas[e]) is not None
        cm = sc.cam_meas[e].copy()
        Kd = np.zeros((24, 7))
        assert getattr(hc, ufn)(_p(model), _p(x), _p(P), _p(u), _p(Ro), _p(cm), sc.notch_meas[e], _p(sc.Rd), _p(Kd)) == 1
    xr, Pr, _, _ = kf.get_vectors()
    assert np.abs(xr[10:16] - x0[10:16]).max() > 0.1  # the DOFs really move
    assert state_err(x, xr) < 1e-8 and cov_err(P, Pr, sc.Rd) < 1e-8, (state_err(x, xr), cov_err(P, Pr, sc.Rd))


@pytest.mark.parametrize("fn,ufn", [("hc_propagate", "hc_update"), ("hc_propagate3", "hc_update3")])
def test_lockstep_ill_conditioned_tuning(hc, golden, fn, ufn):
    """A point of the BASELINE config-3 grid (DOF random walks x 0.12 / 0.018, measurement noise x 398 / 4) where the
    REFERENCE's covariance is asymmetric at 2.6e-11 after the first update and reading the other triangle moves the next
    update by 3e-8: the register-tile path must consume the matrix in the reference's orientation (S is filed transposed,
    eskf_cov3.cuh).  Lock step over 20 epochs; the first update is the prior >> R case of tests/test_conditioning.py."""
    sc = mandala_scenario(golden, n_frames=21, ifv=10)
    model = _model(sc.cfg)
    Qd, Rd = sc.Qd.copy(), sc.Rd.copy()
    Qd[6:9] *= 0.018478497974222907 ** 2
    Qd[9:12] *= 0.11659144011798317 ** 2
    Rd[0:3] *= 398.1071705534977 ** 2
    Rd[3:6] *= 3.981071705534973 ** 2
    kf = sc.new_oracle()
    kf.Q, kf.R = np.diag(Qd), np.diag(Rd)
    k = 0
    ws = wP = asym = 0.0
    for e in range(len(sc.n_prop)):
        for _ in range(sc.n_prop[e]):
            x, P, u, Ro = [a.copy() for a in kf.get_vectors()]
            kf.propagate(sc.dt[k], sc.om_acc[k, :3], sc.om_acc[k, 3:])
            oa = sc.om_acc[k].copy()
            getattr(hc, fn)(_p(model), _p(x), _p(P), _p(u), _p(Ro), sc.dt[k], _p(oa), _p(Qd), _p(sc.sig_om), None)
            xr, Pr, _, _ = kf.get_vectors()
            ws, wP = max(ws, state_err(x, xr)), max(wP, cov_err(P, Pr))
            k += 1
        x, P, u, Ro = [a.copy() for a in kf.get_vectors()]
        asym = max(asym, np.abs(P - P.T).max() / np.abs(P).max())
        assert kf.update(sc.cam_meas[e, :3], sc.cam_meas[e, 3:], sc.notch_meas[e]) is not None
        cm = sc.cam_meas[e].copy()
        Kd = np.zeros((24, 7))
        assert getattr(hc, ufn)(_p(model), _p(x), _p(P), _p(u), _p(Ro), _p(cm), sc.notch_meas[e], _p(Rd), _p(Kd)) == 1
        xr, Pr, _, _ = kf.get_vectors()
        if e > 0:
            ws, wP = max(ws, state_err(x, xr)), max(wP, cov_err(P, Pr, Rd))
        else:
            assert state_err(x, xr) < TOL and cov_err(P, Pr, Rd) < 1e-6
    assert asym > 1e-12  # the reference's own covariance is not symmetric here
    assert ws < 1e-11 and wP < 1e-11, (ws, wP)


@pytest.mark.parametrize("fn,ufn", [("hc_propagate", "hc_update"), ("hc_propagate3", "hc_update3")])
def test_lockstep_random_tunings(hc, golden, fn, ufn):
    """Sixteen random points of the BASELINE config-3 tuning space (DOF random walks x 1e-2 .. 1e2, camera measurement noise
    x 1e-3 .. 1e3), six epochs each in lock step.  The first update of every run (prior >> R, with these scales up to 1e21)
    is excluded from the covariance check: the reference does not determine it (tests/test_conditioning.py; both device
    paths differ from the oracle by the same 0.2 there)."""
    sc = mandala_scenario(golden, n_frames=7, ifv=10)
    model = _model(sc.cfg)
    rng = np.random.default_rng(11)
    wps = wpP = wus = wuP = 0.0
    for _ in range(16):
        a, b = 10 ** rng.uniform(-2, 2, 2)
        c, d = 10 ** rng.uniform(-3, 3, 2)
        Qd, Rd = sc.Qd.copy(), sc.Rd.copy()
        Qd[6:9] *= b ** 2
        Qd[9:12] *= a ** 2
        Rd[0:3] *= c ** 2
        Rd[3:6] *= d ** 2
        kf = sc.new_oracle()
        kf.Q, kf.R = np.diag(Qd), np.diag(Rd)
        k = 0
        for e in range(len(sc.n_prop)):
            for _ in range(sc.n_prop[e]):
                x, P, u, Ro = [v.copy() for v in kf.get_vectors()]
                kf.propagate(sc.dt[k], sc.om_acc[k, :3], sc.om_acc[k, 3:])
                oa = sc.om_acc[k].copy()
                getattr(hc, fn)(_p(model), _p(x), _p(P), _p(u), _p(Ro), sc.dt[k], _p(oa), _p(Qd), _p(sc.sig_om), None)
                xr, Pr, _, _ = kf.get_vectors()
                wps, wpP = max(wps, state_err(x, xr)), max(wpP, cov_err(P, Pr))
                k += 1
            x, P, u, Ro = [v.copy() for v in kf.get_vectors()]
            assert kf.update(sc.cam_meas[e, :3], sc.cam_meas[e, 3:], sc.notch_meas[e]) is not None
            cm = sc.cam_meas[e].copy()
            Kd = np.zeros((24, 7))
            assert getattr(hc, ufn)(_p(model), _p(x), _p(P), _p(u), _p(Ro), _p(cm), sc.notch_meas[e], _p(Rd), _p(Kd)) == 1
            xr, Pr, _, _ = kf.get_vectors()
            if e > 0:
                wus, wuP = max(wus, state_err(x, xr)), max(wuP, cov_err(P, Pr, Rd))
    assert wps < TOL and wpP < TOL, (wps, wpP)
    assert wus < 1e-11 and wuP < 1e-11, (wus, wuP)


def test_stacked_cta_mapping_covers_every_filter_once(hc):
    """The CTA mapping of stacked trajectories (stacked_grid / stacked_cta, eskf_math.cuh), exhaustively: every CTA shape,
    filters_per_traj 1..70, 1..4 trajectories, shards starting at trajectory 0, 1 or 2 and every batch size the streams
    cover.  Every filter belongs to exactly one CTA, every CTA holds 1..F existing filters of ONE trajectory, the trajectory
    the kernel derives from the CTA's first global id exists, and the grid launches no CTA without filters (when N is not a
    multiple of filters_per_traj, ceil(N / fpt) * ceil(fpt / F) CTAs would read parameter rows past the batch)."""
    fn = hc.hc_stacked_sweep
    i64 = ctypes.c_int64
    fn.argtypes = [ctypes.c_int, i64, i64, i64, ctypes.POINTER(i64), i64]
    fn.restype = i64
    geometries = 0
    for F in (28, 16, 8, 4):
        for fpt in range(1, 71):
            cpt = -(-fpt // F)
            for n_traj in range(1, 5):
                for id0 in (0, fpt, 2 * fpt):
                    if id0 >= n_traj * fpt:
                        continue
                    cap = (n_traj * fpt - id0) * (n_traj * cpt + 1)
                    buf = np.empty((cap, 7), dtype=np.int64)
                    r = fn(F, fpt, n_traj, id0, buf.ctypes.data_as(ctypes.POINTER(i64)), cap)
                    assert r > 0
                    N, grid, blk, f0, nf, traj, tl = buf[:r].T
                    where = f"F={F} fpt={fpt} n_traj={n_traj} filter_id0={id0}"
                    bad = (nf < 1) | (nf > F) | (f0 < 0) | (f0 + nf > N)
                    assert not bad.any(), (where, "empty / oversized / out-of-range CTA", buf[:r][bad][:3])
                    bad = ((id0 + f0) // fpt != (id0 + f0 + nf - 1) // fpt) | (traj >= n_traj) | (traj != id0 // fpt + tl)
                    assert not bad.any(), (where, "CTA straddles trajectories / no such trajectory", buf[:r][bad][:3])
                    # exactly-once coverage: per batch size, the CTAs sorted by first filter tile 0..N-1 without gap or overlap
                    o = np.lexsort((f0, N))
                    N, f0, nf, blk, grid = N[o], f0[o], nf[o], blk[o], grid[o]
                    first = np.r_[True, N[1:] != N[:-1]]
                    last = np.r_[N[1:] != N[:-1], True]
                    assert (f0[first] == 0).all() and (f0[last] + nf[last] == N[last]).all(), where
                    assert (f0[1:][~first[1:]] == (f0 + nf)[:-1][~first[1:]]).all(), where
                    counts = np.diff(np.r_[np.flatnonzero(first), len(N)])
                    assert (counts == grid[first]).all(), where  # the grid is the number of CTAs that hold filters
                    geometries += 1
    assert geometries == 4 * 70 * 9


def test_streaming_pass2_is_bit_identical(hc, golden):
    """fx3_apply_stream (pass 2 fused with the transposed reload, eskf_cov3.cuh) performs the same operations in the same
    order per accumulator as the reload followed by fx3_apply_inplace: identical bits on random tiles and records."""
    hc.hc_pass2_both.argtypes = [dp, dp, dp, dp]
    hc.hc_pass2_both.restype = None
    rng = np.random.default_rng(11)
    for _ in range(50):
        T = rng.normal(size=(24, 24)) * 10.0 ** rng.integers(-6, 6, size=(24, 24))
        fx3 = rng.normal(size=90)
        a, b = np.empty((8, 24, 3)), np.empty((8, 24, 3))
        hc.hc_pass2_both(_p(T), _p(fx3), _p(a), _p(b))
        assert np.array_equal(a, b)
