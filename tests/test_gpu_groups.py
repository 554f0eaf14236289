"""Filter groups (eskf_set_groups / eskf_get_group_sums, BatchFilter.set_groups / get_group_sums) on the stacked Monte-Carlo
workload of tests/test_gpu_paths.py: four trajectories x 13 filters, all six DOFs estimated.

A group's row is reduced over the same blocks and trees as the ungrouped sum of a handle that holds exactly that group's
filters, so one group per trajectory is compared BIT FOR BIT with a shard that runs the trajectory alone; smaller groups
(partial first and last ones, groups that straddle trajectories) against numpy on the run's own rows.  Grouping changes
nothing else a run returns."""
import os

import numpy as np
import pytest

from tests.dof_reference import COUNTS, NDOFSUM, envelope
from tests.helpers import model_kwargs
from tests.test_gpu_noise import CAM_STD, IMU_STD
from tests.test_gpu_paths import FPT, GT, SEED, Workload

pytestmark = pytest.mark.gpu


class GroupWorkload(Workload):
    def reference(self, modulus=0):  # (compared with ungrouped runs and numpy, not with the oracle)
        return None


@pytest.fixture(scope="module")
def wl(golden):
    return GroupWorkload(golden)


def run(wl, groups=0, F=28, path="prepass", lo=0, hi=None, n_traj=4, cons=True, stats=True, splits=None):
    """one eskf_run (or segments [splits[i], splits[i + 1])) of filters lo..hi-1 with groups of ``groups``; returns everything
    it returned and, after it, the ungrouped and the grouped getters' outputs"""
    from dvi_ekf_b200 import BatchFilter

    hi = (wl.n if n_traj > 1 else FPT) if hi is None else hi
    n, sc0 = hi - lo, wl.sc0
    out = {}
    with BatchFilter(n, **model_kwargs(sc0.cfg)) as bf:
        bf.set_tuning(F)
        if path == "inkernel":
            bf.set_prepass_budget(0)
        bf.set_noise(sc0.Qd[None], sc0.Rd[None], sc0.sig_om[None])
        bf.set_state(wl.x0[lo:hi], sc0.P0[None], wl.u0[lo:hi], None)
        if cons:
            bf.keep_consistency()
        bf.set_groups(groups)
        kw = dict(**(wl.streams if n_traj > 1 else wl.streams0), n_traj=n_traj, filters_per_traj=FPT if n_traj > 1 else None,
                  seed=SEED, filter_id0=lo, imu_noise_std=IMU_STD, cam_noise_std=CAM_STD, noise_free_filter0=True, gt_dofs=GT,
                  want_stats=stats)
        c0 = bf.launch_count
        if splits is None:
            r = bf.run(**kw)
            out["stats"], out["sum"] = r if stats else (None, None)
        else:
            for e0, e1 in zip(splits, splits[1:]):
                out["stats"], out["sum"], out["carry"] = bf.run(epochs=(e0, e1), carry=out.get("carry"), **kw)
                if cons:
                    g = bf.get_group_sums(stats=False, consistency=True, dof_envelope=True)
                    out.setdefault("seg", []).append((e0, e1, g[2], g[3]))
        out["launches"] = bf.launch_count - c0
        bf.set_groups(7)  # (changes nothing the getters return: the run recorded its groups)
        out["x"], out["P"], out["u"], out["R"], out["status"] = bf.get_state()
        if cons:
            out["nis"], out["nees"], out["esum"] = bf.get_consistency()
            out["dofs"], out["var"] = bf.get_dof_history()
            out["env"] = bf.get_dof_envelope()
        out["group0"], out["gstats"], out["gesum"], out["genv"] = bf.get_group_sums(stats=groups > 0 and stats,
                                                                                       consistency=cons, dof_envelope=cons)
    return out


def _same(a, b, what, keys=("x", "P", "u", "R", "status", "stats", "sum", "nis", "nees", "esum", "env", "dofs", "var")):
    for k in keys:
        if a.get(k) is not None or b.get(k) is not None:
            assert a[k].tobytes() == b[k].tobytes(), (what, k)


@pytest.mark.parametrize("F", (28, 4))
@pytest.mark.parametrize("path", ("prepass", "inkernel"))
def test_one_group_per_trajectory_is_a_shard_of_that_trajectory(wl, path, F):
    whole = run(wl, FPT, F, path)
    assert whole["group0"] == 0 and whole["gstats"].shape == (4, 16) and whole["genv"].shape == (4, wl.E, NDOFSUM)
    for k in range(4):
        shard = run(wl, 0, F, path, lo=k * FPT, hi=(k + 1) * FPT)
        assert whole["gstats"][k].tobytes() == shard["sum"].tobytes(), (path, F, k)
        assert whole["gesum"][k].tobytes() == shard["esum"].tobytes(), (path, F, k)
        assert whole["genv"][k].tobytes() == shard["env"].tobytes(), (path, F, k)
        assert shard["group0"] == 0 and shard["gesum"][0].tobytes() == shard["esum"].tobytes()


def test_one_group_is_the_ungrouped_sum(wl):
    base = run(wl, 0)
    assert base["group0"] == 0 and base["gstats"] is None and base["gesum"].shape == (1, wl.E, 8)
    assert base["gesum"][0].tobytes() == base["esum"].tobytes() and base["genv"][0].tobytes() == base["env"].tobytes()
    for g in (wl.n, wl.n + 1, 1000):
        out = run(wl, g)
        _same(out, base, g)
        assert out["gstats"].shape == (1, 16) and out["gstats"][0].tobytes() == base["sum"].tobytes()
        assert out["gesum"][0].tobytes() == base["esum"].tobytes() and out["genv"][0].tobytes() == base["env"].tobytes()


def _masked_rows(st, status):
    """per-filter contributions to stats_sum: the row [0:10] of a healthy filter, and the counts [10], [11], [12]"""
    fin = np.isfinite(st[:, :10]).all(axis=1)
    ok = fin & (status == 0)
    c = np.zeros((len(st), 16))
    c[:, :10] = np.where(ok[:, None], st[:, :10], 0.0)
    c[:, 10], c[:, 11], c[:, 12] = status != 0, ok, ~fin
    return c


def _cons_terms(nis, nees):
    """[N, E, 8] per-filter terms of epoch_sum (d = 6)"""
    fa, fc = np.isfinite(nis), np.isfinite(nees)
    a, c = np.where(fa, nis, 0.0), np.where(fc, nees, 0.0)
    return np.stack([fa, a, a * a, fc, c, c * c, ~fa | ~fc, 0 * a], axis=2).astype(float)


def _dof_terms(out):
    """[N, E, 59] per-filter terms of the envelope columns that need only the diagonal of the DOF block"""
    n, E = out["nis"].shape
    t = np.empty((n, E, NDOFSUM))
    for f in range(n):
        B = np.zeros((E, 6, 6))
        B[:, np.arange(6), np.arange(6)] = out["var"][f]
        t[f] = envelope(out["nis"][f:f + 1], out["dofs"][f:f + 1], B[None], GT, 0)
    return t[:, :, :59]


def _by_group(terms, id0, g):
    gid = (id0 + np.arange(len(terms))) // g
    out = np.zeros((gid[-1] - gid[0] + 1, *terms.shape[1:]))
    np.add.at(out, gid - gid[0], terms)
    return gid[0], out


def _close(got, ref, count_cols, what, scale=None):
    """counts exact, every other entry within 1e-12 of ``scale`` (the sum of the absolute terms; default |ref|)"""
    cnt = np.zeros(got.shape[-1], bool)
    cnt[count_cols] = True
    assert np.array_equal(got[..., cnt], ref[..., cnt]), what
    scale = np.maximum(np.abs(ref if scale is None else scale)[..., ~cnt], 1e-300)
    err = np.abs(got[..., ~cnt] - ref[..., ~cnt])
    assert (err <= 1e-12 * scale).all(), (what, (err / scale).max())


DOF_COUNTS = [c for c in COUNTS if c < 59]


@pytest.mark.parametrize("g", (5, 1))
def test_small_groups_against_numpy(wl, g):
    out = run(wl, g)
    G = -(-wl.n // g)
    assert out["group0"] == 0 and out["gstats"].shape == (G, 16) and out["gesum"].shape == (G, wl.E, 8)
    for key, terms, counts in (("gstats", _masked_rows(out["stats"], out["status"]), [10, 11, 12]),
                               ("gesum", _cons_terms(out["nis"], out["nees"]), [0, 3, 6, 7]),
                               ("genv", _dof_terms(out), DOF_COUNTS)):
        _, ref = _by_group(terms, 0, g)
        _close(out[key][..., :ref.shape[-1]], ref, counts, (key, g), _by_group(np.abs(terms), 0, g)[1])
    assert not out["genv"][..., 74:].any()
    # per epoch, the counts over all groups are the ungrouped counts; the other sums within rounding
    for key, ukey, counts in (("gstats", "sum", [10, 11, 12]), ("gesum", "esum", [0, 3, 6, 7]), ("genv", "env", COUNTS)):
        _close(out[key].sum(axis=0), out[ukey], counts, (key, "total", g), np.abs(out[key]).sum(axis=0))


def test_two_shards_that_cut_a_group(wl):
    """trajectory 0 alone (n_traj = 1, as tuning candidates are), groups of 5: filters 0..12 are groups 0, 1, 2; shards
    [0, 7) and [7, 13) cut group 1"""
    from dvi_ekf_b200.sharding import place_group_rows

    whole = run(wl, 5, n_traj=1)
    parts = [run(wl, 5, n_traj=1, lo=lo, hi=hi) for lo, hi in ((0, 7), (7, FPT))]
    assert [p["group0"] for p in parts] == [0, 1] and [len(p["gstats"]) for p in parts] == [2, 2]
    for key, counts in (("gstats", [10, 11, 12]), ("gesum", [0, 3, 6, 7]), ("genv", COUNTS)):
        placed = [place_group_rows(p[key], p["group0"], 3) for p in parts]
        _close(placed[0] + placed[1], whole[key], counts, key, np.abs(placed[0]) + np.abs(placed[1]))
    for p, rows in zip(parts, (slice(0, 7), slice(7, FPT))):  # (the filters themselves are those of the whole run)
        assert p["stats"].tobytes() == whole["stats"][rows].tobytes()


@pytest.mark.parametrize("path", ("prepass", "inkernel"))
def test_segments(wl, path):
    whole = run(wl, FPT, path=path)
    seg = run(wl, FPT, path=path, splits=[0, 4, 7])
    assert seg["gstats"].tobytes() == whole["gstats"].tobytes()
    _same(seg, whole, path, keys=("x", "P", "stats", "sum"))
    for e0, e1, gesum, genv in seg["seg"]:
        assert gesum.tobytes() == np.ascontiguousarray(whole["gesum"][:, e0:e1]).tobytes(), (e0, e1)
        assert genv.tobytes() == np.ascontiguousarray(whole["genv"][:, e0:e1]).tobytes(), (e0, e1)


@pytest.mark.parametrize("path", ("prepass", "inkernel"))
def test_grouping_changes_nothing_else(wl, path):
    off = run(wl, 0, path=path)
    for g in (FPT, 5):
        on = run(wl, g, path=path)
        _same(on, off, (path, g))
        assert on["launches"] == off["launches"] + 2  # the grouped statistics reduction
    segs = [run(wl, g, path=path, splits=[0, 3, 7]) for g in (0, FPT)]
    _same(segs[1], segs[0], ("segments", path), keys=("x", "P", "stats", "sum", "carry", "nis", "nees", "esum", "env"))
    assert segs[1]["launches"] == segs[0]["launches"] + 2 * 2
    nostats = [run(wl, g, path=path, stats=False) for g in (0, FPT)]
    assert nostats[1]["launches"] == nostats[0]["launches"]  # no statistics rows: nothing to reduce


def test_error_paths(wl):
    from dvi_ekf_b200 import BatchFilter
    from dvi_ekf_b200._lib import EskfError

    sc0 = wl.sc0
    kw = dict(**wl.streams, n_traj=4, filters_per_traj=FPT, seed=SEED, imu_noise_std=IMU_STD, cam_noise_std=CAM_STD, gt_dofs=GT)
    with BatchFilter(wl.n, **model_kwargs(sc0.cfg)) as bf:
        with pytest.raises(ValueError):
            bf.set_groups(-1)
        assert bf._lib.eskf_set_groups(bf._h, -1) == -1  # (the library's own check)
        bf.set_noise(sc0.Qd[None], sc0.Rd[None], sc0.sig_om[None])
        bf.set_state(wl.x0, sc0.P0[None], wl.u0, None)
        with pytest.raises(EskfError, match="code -1.*no statistics"):  # before any run
            bf.get_group_sums()
        bf.set_groups(FPT)
        bf.run(want_stats=False, **kw)  # a run without statistics rows
        with pytest.raises(EskfError, match="code -1.*no statistics"):
            bf.get_group_sums()
        with pytest.raises(EskfError, match="code -1.*keep_consistency"):  # consistency rows without records
            bf.get_group_sums(stats=False, consistency=True)
        with pytest.raises(EskfError, match="code -1.*keep_consistency"):
            bf.get_group_sums(stats=False, dof_envelope=True)
        assert bf.get_group_sums(stats=False)[0] == 0
        bf.set_groups(0)
        bf.run(**kw)  # statistics, but no groups
        with pytest.raises(EskfError, match="code -1.*without groups"):
            bf.get_group_sums()
    with BatchFilter(FPT, variant=1, **model_kwargs(sc0.cfg)) as bf:
        bf.set_noise(sc0.Qd[None], sc0.Rd[None], sc0.sig_om[None])
        bf.set_state(wl.x0[:FPT], sc0.P0[None], wl.u0[:FPT], None)
        bf.set_groups(5)
        bf.run(**wl.streams0, seed=SEED, imu_noise_std=IMU_STD, cam_noise_std=CAM_STD, gt_dofs=GT)
        assert bf.get_group_sums()[1].shape == (3, 16)  # the statistics of the first kernel are grouped too
        with pytest.raises(EskfError, match="code -1"):
            bf.get_group_sums(stats=False, consistency=True)


def _config(tmp_path, name, frames):
    import yaml

    from dvi_ekf_b200 import Config

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    y = yaml.safe_load(open(os.path.join(root, "config.yaml")))
    y["simulation"].update(do_fast_sim=False, frozen_dofs=[0] * 6, traj_name=name)
    y["camera"]["total_frames"] = frames
    y["imu"]["interframe_vals"] = 5
    fp = tmp_path / f"config_{name}.yaml"
    fp.write_text(yaml.safe_dump(y))
    return Config(str(fp))


def test_simulator_run_trajectories(tmp_path):
    """three trajectories in one stacked launch against Simulator.run of each trajectory alone: the same bits"""
    from dvi_ekf_b200 import Simulator
    from dvi_ekf_b200._lib import NSTAT

    names = ["trans_x", "rot_x", "mandala0_mono"]
    sim = Simulator(_config(tmp_path, "mandala0_mono", "all"))
    res = sim.run_trajectories(names, 16, consistency=True)
    assert list(res) == names and sim.trajectory_results is res and sim.stats.shape == (48, NSTAT)
    stacked = sim.stats
    for k, nm in enumerate(names):
        one = Simulator(_config(tmp_path, nm, 60))
        st, sm = one.run(n_filters=16, consistency=True, verbose=False)
        assert stacked[16 * k:16 * (k + 1)].tobytes() == st.tobytes(), nm
        for key, ref in (("stats", None), ("consistency", one.consistency), ("dof_envelope", one.dof_envelope)):
            got = res[nm][key]
            if key == "stats":
                from dvi_ekf_b200.sharding import summarise_stats

                ref = summarise_stats(sm)
            assert got.keys() == ref.keys()
            for f in got:
                assert np.asarray(got[f]).tobytes() == np.asarray(ref[f]).tobytes(), (nm, key, f)
    with pytest.raises(ValueError, match="frames"):
        sim.run_trajectories(names, 4, frames=61)
