"""A trajectory in epoch segments (eskf_run_epochs, BatchFilter.run(epochs=...), run_segments) against one eskf_run.

Everything is compared BIT FOR BIT with the one-launch run of the same handle geometry: state, covariance, u_old, R_old and
status; every statistics column and stats_sum; the FilterTraj rows; the Jacobian record of the last segment; and each
segment's consistency rows, per-DOF history and envelope rows against the rows of the whole run.  The workload is the stacked
Monte-Carlo one of tests/test_gpu_paths.py: four trajectories with a different n_prop each, epochs of 0, 1 and 2 steps, one
trajectory that stops 28 steps before the stream ends."""
import ctypes as C

import numpy as np
import pytest

from oracle.eskf_oracle import OracleConfig
from tests.helpers import Scenario, mandala_scenario, model_kwargs
from tests.test_gpu_noise import CAM_STD, IMU_STD
from tests.test_gpu_paths import FPT, GT, N_PROP, SEED, Workload

pytestmark = pytest.mark.gpu

SHAPES = (28, 16, 8, 4)
# 1, 2, 3 and E segments; boundaries on both sides of the 0-step epochs (trajectory 2: epochs 1 and 4, trajectory 3: epoch 4)
SPLITS = ([0, 7], [0, 4, 7], [0, 1, 2, 7], [0, 4, 5, 7], list(range(8)))


class SegWorkload(Workload):
    def reference(self, modulus=0):  # (compared with one eskf_run, not with the oracle)
        return None


@pytest.fixture(scope="module")
def wl(golden):
    return SegWorkload(golden)


def _handle(wl, n, F=28, path="prepass", export=False, lo=0, x0=None, cons=None):
    from dvi_ekf_b200 import BatchFilter

    sc0 = wl.sc0
    bf = BatchFilter(n, **model_kwargs(sc0.cfg))
    bf.set_tuning(F)
    if path == "inkernel":
        bf.set_prepass_budget(0)
    bf.set_noise(sc0.Qd[None], sc0.Rd[None], sc0.sig_om[None])
    bf.set_state(wl.x0[lo:lo + n] if x0 is None else x0, sc0.P0[None], wl.u0[lo:lo + n], None)
    if export:
        bf.keep_jacobians(True)
    if export if cons is None else cons:
        bf.keep_consistency()
    return bf


def _kw(wl, n_traj, lo, trace, modulus=0, noise_free0=True):
    return dict(**(wl.streams if n_traj > 1 else wl.streams0), n_traj=n_traj, filters_per_traj=FPT if n_traj > 1 else None,
                seed=SEED, filter_id0=lo, imu_noise_std=IMU_STD, cam_noise_std=CAM_STD, noise_free_filter0=noise_free0,
                noise_id_modulus=modulus, trace=trace, gt_dofs=GT)


def _collect(bf, out, cons):
    if cons:
        nis, nees, es = bf.get_consistency()
        dofs, var = bf.get_dof_history()
        for k, v in dict(nis=nis, nees=nees, esum=es, dofs=dofs, var=var, env=bf.get_dof_envelope()).items():
            out.setdefault(k, []).append(v)


def _finish(bf, out, export):
    x, P, u, R, status = bf.get_state()
    out.update(x=x, P=P, u=u, R=R, status=status)
    if export:
        out["jac"] = bf.get_jacobians()
    for k, ax in (("nis", 1), ("nees", 1), ("esum", 0), ("dofs", 1), ("var", 1), ("env", 0)):
        if k in out:
            out[k] = np.concatenate(out[k], axis=ax)
    return out


def run_cell(wl, F, path, export, n_traj=4, splits=None, lo=0, hi=None, **kw):
    """one eskf_run (splits None) or the same trajectory in segments [splits[i], splits[i + 1]); trace, Jacobian record and
    consistency with ``export``"""
    hi = (wl.n if n_traj > 1 else FPT) if hi is None else hi
    n = hi - lo
    trace = np.full((n, wl.T, 26), np.nan) if export else None
    out = {}
    with _handle(wl, n, F, path, export, lo) as bf:
        if splits is None:
            out["stats"], out["sum"] = bf.run(**_kw(wl, n_traj, lo, trace, **kw))
            _collect(bf, out, export)
        else:
            for _, _, st, sm in bf.run_segments(boundaries=splits, **_kw(wl, n_traj, lo, trace, **kw)):
                out["stats"], out["sum"] = st, sm
                _collect(bf, out, export)
            out["carry"] = bf.last_carry
        out["trace"] = trace
        return _finish(bf, out, export)


def _same(a, b, what=""):
    keys = [k for k in a if k in b and k != "carry"]
    for k in keys:
        if k == "jac":
            assert all(x.tobytes() == y.tobytes() for x, y in zip(a[k], b[k])), (what, k)
        elif a[k] is not None:
            assert a[k].shape == b[k].shape and a[k].tobytes() == b[k].tobytes(), (what, k)
    return keys


@pytest.mark.parametrize("n_traj", [4, 1])
@pytest.mark.parametrize("export", [False, True])
@pytest.mark.parametrize("path", ["prepass", "inkernel"])
@pytest.mark.parametrize("F", SHAPES)
def test_segments_are_bit_identical_to_one_launch(wl, F, path, export, n_traj):
    whole = run_cell(wl, F, path, export, n_traj)
    for splits in SPLITS:
        seg = run_cell(wl, F, path, export, n_traj, splits=splits)
        keys = _same(seg, whole, splits)
        assert {"x", "P", "u", "R", "status", "stats", "sum"} <= set(keys)
        if export:
            assert {"trace", "jac", "nis", "nees", "esum", "dofs", "var", "env"} <= set(keys)
        assert np.all(seg["status"] == 0) and (seg["stats"][:, 9] == wl.E).all()
        c = seg["carry"]
        assert (c[:, 2] == seg["stats"][:, 9]).all() and (c[:, 3] == 0).all()
        assert ((c[:, 0] + c[:, 1]) / 12.0).tobytes() == seg["stats"][:, 8].tobytes()


@pytest.mark.parametrize("path", ["prepass", "inkernel"])
def test_noise_id_modulus_and_noisy_filter0(wl, path):
    for kw in (dict(modulus=5), dict(noise_free0=False), dict(modulus=3, noise_free0=False)):
        whole = run_cell(wl, 28, path, True, **kw)
        for splits in (SPLITS[2], SPLITS[4]):
            _same(run_cell(wl, 28, path, True, splits=splits, **kw), whole, (kw, splits))


def test_trace_rows_outside_the_segment_keep_the_callers_content(wl):
    """a segment writes exactly the rows of its steps, [k0[t], k1[t]) of segment_steps, and nothing else -- but for the row
    k0[t] - 1 when it begins with an epoch of 0 steps: that update overwrites the last step's row, as in one launch"""
    from dvi_ekf_b200.engine import segment_steps

    sentinel = -12345.0
    for e0, e1 in ((0, 2), (2, 3), (4, 5), (5, 7)):
        trace = np.full((wl.n, wl.T, 26), sentinel)
        with _handle(wl, wl.n, export=True) as bf:
            if e0:
                bf.run(epochs=(0, e0), **_kw(wl, 4, 0, None))
            bf.run(epochs=(e0, e1), carry=bf.last_carry, **_kw(wl, 4, 0, trace))
        k0, k1 = segment_steps(N_PROP, wl.T, e0, e1)
        for t in range(4):
            rows = trace[t * FPT:(t + 1) * FPT]
            written = (rows != sentinel).all(axis=2).all(axis=0)
            untouched = (rows == sentinel).all(axis=2).all(axis=0)
            assert (written | untouched).all()
            expect = np.arange(k0[t] - 1 if k0[t] > 0 and N_PROP[t, e0] == 0 else k0[t], k1[t])
            assert np.array_equal(np.nonzero(written)[0], expect), (e0, e1, t)


def test_checkpoint_restart_on_a_new_handle(wl):
    """after segment 1: state, carry and epoch to host arrays, continue on a new handle -- bit-identical to the uninterrupted
    run; the same for two shards split at a trajectory boundary"""
    for lo, hi in ((0, wl.n), (0, 2 * FPT), (2 * FPT, wl.n)):
        n = hi - lo
        for path in ("prepass", "inkernel"):
            whole = run_cell(wl, 28, path, True, lo=lo, hi=hi)
            trace = np.full((n, wl.T, 26), np.nan)
            out = {}
            with _handle(wl, n, 28, path, True, lo) as bf:
                _, _, carry = bf.run(epochs=(0, 3), **_kw(wl, 4, lo, trace))
                _collect(bf, out, True)
                x, P, u, R, _ = bf.get_state()
                ckpt = dict(x=x.copy(), P=P.copy(), u=u.copy(), R=R.copy(), carry=np.array(carry), epoch=3)
            with _handle(wl, n, 28, path, True, lo, x0=ckpt["x"]) as bf:
                bf.set_state(ckpt["x"], ckpt["P"], ckpt["u"], ckpt["R"])
                out["stats"], out["sum"], _ = bf.run(epochs=(ckpt["epoch"], wl.E), carry=ckpt["carry"], **_kw(wl, 4, lo, trace))
                _collect(bf, out, True)
                out["trace"] = trace
                _finish(bf, out, False)
            del whole["jac"]  # (the new handle filed the record of its own last step: compared in the cells above)
            _same(out, whole, (lo, hi, path))
            if (lo, hi) != (0, wl.n):  # a shard's rows are those of the same filters in the whole batch
                full = run_cell(wl, 28, path, True)
                assert out["stats"].tobytes() == full["stats"][lo:hi].tobytes()
                assert out["x"].tobytes() == full["x"][lo:hi].tobytes()


def _singular(golden):
    cfg = OracleConfig(max_vals=8, interframe_vals=10, frozen_dofs=(0,) * 6)
    sc = Scenario(golden["traj_trans_x"][:8], cfg)
    n = 5
    P, R, Q = (np.repeat(a[None], n, 0) for a in (sc.P0, sc.Rd, sc.Qd))
    P[2], R[2], Q[2] = 0.0, 0.0, 0.0
    return sc, n, P, R, Q


def test_sticky_status_survives_a_restart(golden):
    """a filter whose S is singular at every update keeps its status bit through set_state on a new handle, and the masked
    stats_sum counts it as the one-launch run does"""
    from dvi_ekf_b200 import BatchFilter

    sc, n, P, R, Q = _singular(golden)
    kw = dict(dt=sc.dt, om_acc=sc.om_acc, n_prop=sc.n_prop, cam=sc.cam_meas, notch=sc.notch_meas, gt_dofs=GT,
              cam_ref=np.zeros((len(sc.n_prop), 6)), imu_ref=np.zeros((len(sc.n_prop), 6)))
    E = len(sc.n_prop)

    def handle():
        bf = BatchFilter(n, **model_kwargs(sc.cfg))
        bf.set_noise(Q, R, sc.sig_om[None])
        return bf

    with handle() as bf:
        bf.set_state(sc.x0[None], P, sc.u0[None], None)
        st_w, sm_w = bf.run(**kw)
        state_w = bf.get_state()
    with handle() as bf:
        bf.set_state(sc.x0[None], P, sc.u0[None], None)
        _, _, carry = bf.run(epochs=(0, 2), **kw)
        x, P1, u, R1, status = bf.get_state()
    assert status[2] & 1 and carry[2, 3] == status[2]
    with handle() as bf:
        bf.set_state(x, P1, u, R1)
        assert bf.get_state()[4][2] == 0  # (set_state clears the status word: the carry restores it)
        st, sm, _ = bf.run(epochs=(2, E), carry=carry, **kw)
        state = bf.get_state()
    assert all(a.tobytes() == b.tobytes() for a, b in zip(state, state_w))
    assert st.tobytes() == st_w.tobytes() and sm.tobytes() == sm_w.tobytes()
    assert sm[10] == 1 and sm[11] == n - 1 and st[2, 10] == state[4][2]


def test_a_segment_takes_the_prepass_path_where_the_whole_run_would_not(wl):
    """with a pre-pass budget the whole run exceeds and a short segment fits, the segment runs the pre- and post-pass kernels
    (eskf_launch_count) and the result is bit-identical to the whole run"""
    n = wl.n
    # the whole run's pre-pass: [T, N, 6] + [E, N, 8] + [E, N, 14] doubles; the first segment: 12 steps (11 and the one staged
    # ahead), 1 epoch
    whole_b = n * (wl.T * 6 + wl.E * 22) * 8
    seg_b = n * (12 * 6 + 22) * 8
    budget = (whole_b + seg_b) // 2
    assert seg_b < budget < whole_b
    kw = _kw(wl, 4, 0, None)
    ref = run_cell(wl, 28, "prepass", False)  # (default budget: the whole run takes the pre-pass path)
    with _handle(wl, n) as bf:
        bf.set_prepass_budget(budget)
        c0 = bf.launch_count
        bf.run(**kw)
        assert bf.launch_count - c0 == 3  # the persistent kernel and the statistics reduction: no pre- / post-pass
    with _handle(wl, n) as bf:
        bf.set_prepass_budget(budget)
        c0 = bf.launch_count
        bf.run(epochs=(0, 1), **kw)
        # segment bases, pre-pass (2), persistent kernel, post-pass (2), reduction (2)
        assert bf.launch_count - c0 == 8
        st, sm, _ = bf.run(epochs=(1, wl.E), carry=bf.last_carry, **kw)
        x, P, u, R, status = bf.get_state()
    assert st.tobytes() == ref["stats"].tobytes() and sm.tobytes() == ref["sum"].tobytes()
    assert x.tobytes() == ref["x"].tobytes() and P.tobytes() == ref["P"].tobytes()


def test_consistency_of_a_few_epochs_of_a_run_too_long_for_its_records(golden):
    """65,536 filters x 4,000,000 epochs (mostly 0 steps): eskf_run with consistency is ESKF_ENOMEM; eskf_run_epochs over the
    first epochs runs, and its records are those of a short run of the same epochs"""
    from dvi_ekf_b200 import BatchFilter
    from dvi_ekf_b200._lib import EskfError

    sc = mandala_scenario(golden, n_frames=4, ifv=2)
    n, E, e = 1 << 16, 4_000_000, len(sc.n_prop)
    npr, cam, notch = np.zeros(E, np.int32), np.zeros((E, 7)), np.zeros(E)
    npr[:e], cam[:e], notch[:e] = sc.n_prop, sc.cam_meas, sc.notch_meas
    outs = []
    for long in (True, False):
        with BatchFilter(n, **model_kwargs(sc.cfg)) as bf:
            bf.set_noise(sc.Qd[None], sc.Rd[None], sc.sig_om[None])
            bf.set_state(sc.x0[None], sc.P0[None], sc.u0[None], None)
            bf.keep_consistency()
            if long:
                with pytest.raises(EskfError, match=r"code -3"):
                    bf.run(sc.dt, sc.om_acc, npr, cam, notch)
                bf.run(sc.dt, sc.om_acc, npr, cam, notch, epochs=(0, e))
            else:
                bf.run(sc.dt, sc.om_acc, sc.n_prop, sc.cam_meas, sc.notch_meas)
            outs.append((*bf.get_consistency(), bf.get_dof_envelope(), bf.get_state()[0]))
    assert outs[0][0].shape == (n, e)
    assert np.isfinite(outs[0][0]).all()
    assert all(a.tobytes() == b.tobytes() for a, b in zip(*outs))


def test_argument_rules(wl, monkeypatch):
    """bad ranges are ESKF_EINVAL; an empty range launches nothing, passes the carry through and writes no statistics;
    variant 1 is ESKF_EINVAL; every refused call leaves the handle unchanged"""
    import dvi_ekf_b200.engine as eng
    from dvi_ekf_b200 import BatchFilter
    from dvi_ekf_b200._lib import NCARRY, NSTAT, EskfError

    n = wl.n
    kw = _kw(wl, 4, 0, None)
    with pytest.raises(ValueError, match="epoch range"):
        eng.check_run_geometry(n, 4, FPT, 0, wl.T, wl.E, epochs=(3, 2))
    with _handle(wl, n, export=True) as bf:
        bf.run(epochs=(0, 2), **kw)
        nis0 = bf.get_consistency()[0]
        before, c0 = bf.get_state(), bf.launch_count
        monkeypatch.setattr(eng, "check_run_geometry", lambda *a, **k: None)  # the library's own checks
        for e0, e1 in ((-1, 2), (3, 2), (0, wl.E + 1), (wl.E + 1, wl.E + 1)):
            with pytest.raises(EskfError, match=r"code -1.*epoch range"):
                bf.run(epochs=(e0, e1), **kw)
            assert bf.launch_count == c0
            assert all(a.tobytes() == b.tobytes() for a, b in zip(bf.get_state(), before))
            assert bf.get_consistency()[0].tobytes() == nis0.tobytes()
        monkeypatch.undo()

        # an empty range, through the C entry point with sentinel outputs
        grabbed = {}
        orig = bf._run_epochs

        def raw(s, e0, e1, carry, want, dev):
            cin = np.arange(n * NCARRY, dtype=np.float64).reshape(n, NCARRY)
            cout, st, sm = np.full((n, NCARRY), 7.0), np.full((n, NSTAT), 7.0), np.full(NSTAT, 7.0)
            p = lambda a: a.ctypes.data_as(C.c_void_p)
            c1 = bf.launch_count
            grabbed["rc"] = bf._lib.eskf_run_epochs(bf._h, C.byref(s), 3, 3, p(cin), p(cout), p(st), p(sm), 0)
            grabbed["launches"] = bf.launch_count - c1
            grabbed["pass"] = cout.tobytes() == cin.tobytes()
            grabbed["untouched"] = (st == 7.0).all() and (sm == 7.0).all()
            grabbed["rc0"] = bf._lib.eskf_run_epochs(bf._h, C.byref(s), 3, 3, None, p(cout), None, None, 0)
            grabbed["zeros"] = (cout == 0.0).all()
            return orig(s, e0, e1, carry, want, dev)

        bf._run_epochs = raw
        bf.run(epochs=(2, 2), **kw)
        assert grabbed == dict(rc=0, launches=0, **{"pass": True}, untouched=True, rc0=0, zeros=True)
        bf._run_epochs = orig
        _, _, c = bf.run(epochs=(2, 2), carry=np.ones((n, NCARRY)), **kw)
        assert (c == 1.0).all() and bf.get_consistency()[0].shape == (n, 0)
        assert all(a.tobytes() == b.tobytes() for a, b in zip(bf.get_state(), before))
    with BatchFilter(n, variant=1, **model_kwargs(wl.sc0.cfg)) as bf:
        bf.set_noise(wl.sc0.Qd[None], wl.sc0.Rd[None], wl.sc0.sig_om[None])
        bf.set_state(wl.x0, wl.sc0.P0[None], wl.u0, None)
        before, c0 = bf.get_state(), bf.launch_count
        with pytest.raises(EskfError, match="default kernel"):
            bf.run(epochs=(0, 2), **kw)
        assert bf.launch_count == c0 and all(a.tobytes() == b.tobytes() for a, b in zip(bf.get_state(), before))


def test_device_resident_streams(wl):
    """CUDA tensors: the segment's step counts are read back to size the pre-pass; bit-identical to one launch"""
    import torch

    dev = torch.device("cuda", 0)
    t = lambda a: torch.tensor(np.ascontiguousarray(a), device=dev)
    s = {k: t(v) for k, v in wl.streams.items()}
    kw = dict(**s, n_traj=4, filters_per_traj=FPT, seed=SEED, imu_noise_std=IMU_STD, cam_noise_std=CAM_STD, gt_dofs=GT,
              stats_on_device=True)
    outs = []
    for splits in (None, SPLITS[3]):
        with _handle(wl, wl.n) as bf:
            if splits is None:
                st, sm = bf.run(**kw)
            else:
                for _, _, st, sm in bf.run_segments(boundaries=splits, **kw):
                    assert torch.is_tensor(bf.last_carry) and bf.last_carry.is_cuda
            outs.append((st.cpu().numpy(), sm.cpu().numpy(), *bf.get_state()))
    assert all(a.tobytes() == b.tobytes() for a, b in zip(*outs))


def test_stopping_run_segments_keeps_the_last_finished_segment(wl):
    """a caller who stops iterating after two segments holds the state of epochs [0, 4): that of one eskf_run of the
    trajectory cut after epoch 4"""
    kw = _kw(wl, 4, 0, None)
    with _handle(wl, wl.n) as bf:
        gen = bf.run_segments(boundaries=[0, 2, 4, 7], **kw)
        done = [next(gen)[:2] for _ in range(2)]
        gen.close()  # (nothing more runs)
        assert done == [(0, 2), (2, 4)]
        seg, st = bf.get_state(), bf.last_carry
    cut = dict(kw, n_prop=np.ascontiguousarray(N_PROP[:, :4]).reshape(-1), cam=wl.streams["cam"].reshape(4, wl.E, 7)[:, :4].reshape(-1, 7),
               notch=wl.streams["notch"].reshape(4, wl.E)[:, :4].reshape(-1),
               cam_ref=wl.cam_ref[:, :4].reshape(-1, 6), imu_ref=wl.imu_ref[:, :4].reshape(-1, 6))
    with _handle(wl, wl.n) as bf:
        stats, _ = bf.run(**cut)
        ref = bf.get_state()
    assert all(a.tobytes() == b.tobytes() for a, b in zip(seg, ref))
    assert (st[:, 2] == stats[:, 9]).all() and ((st[:, 0] + st[:, 1]) / 12.0).tobytes() == stats[:, 8].tobytes()


def test_simulator_run_in_segments(tmp_path):
    """Simulator.run(segment_epochs=k) gives what Simulator.run() gives, with consistency=True as well"""
    import os

    import yaml

    from dvi_ekf_b200 import Config, Simulator

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    y = yaml.safe_load(open(os.path.join(root, "config.yaml")))
    y["simulation"].update(do_fast_sim=False, frozen_dofs=[0] * 6)
    y["camera"]["total_frames"] = 14
    y["imu"]["interframe_vals"] = 5
    fp = tmp_path / "config.yaml"
    fp.write_text(yaml.safe_dump(y))
    sim = Simulator(Config(str(fp)))
    for consistency in (False, True):
        res = []
        for k in (None, 4, 1):
            st, sm = sim.run(n_filters=16, consistency=consistency, verbose=False, segment_epochs=k)
            res.append((st, sm, sim.final_states.copy(), sim.consistency, sim.dof_envelope))
        for r in res[1:]:
            assert r[0].tobytes() == res[0][0].tobytes() and r[1].tobytes() == res[0][1].tobytes()
            assert r[2].tobytes() == res[0][2].tobytes()
            if consistency:
                for a, b in ((r[3], res[0][3]), (r[4], res[0][4])):
                    assert a.keys() == b.keys()
                    for key in a:
                        va, vb = np.asarray(a[key]), np.asarray(b[key])
                        assert va.tobytes() == vb.tobytes(), key
