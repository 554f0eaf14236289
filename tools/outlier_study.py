"""The innovation gate (``BatchFilter.run(nis_gate=...)``) and simulated outlier frames (``run(outlier_prob=...,
outlier_std=...)``) on the config-2 calibration workload (mandala0_mono, 140 frames x 10 IMU samples, all six DOFs estimated
from perturbed values, Monte-Carlo noise), and the false-rejection rate of the gate on config 2 as config.yaml sets it.

1. Cost: eskf_run at each size five ways -- the production instantiation (nothing set), dropout set with p = 0 (the
   export instantiation, for reference), the gate at +inf everywhere, the gate at chi2(7) 0.999, and outliers at p = 0.1
   with that gate -- timed with CUDA events, the handles interleaved run by run; the median of the runs.
2. Science: ONE stacked launch, one copy of the calibration trajectory per cell of outlier p in {0, 0.05, 0.2} x gate in
   {off, chi2 0.99, 0.999, 0.99999}, filters_per_traj = n, noise_id_modulus = n and one filter group per copy, consistency
   on: every cell sees the same noise, initial DOFs and outlier offsets, and the outlier masks nest over p.  Per cell: frames
   corrupted, updates rejected, ANIS / ANEES over all epochs, and per DOF the RMSE and inflation at epochs 1, 10, 50, 138.
3. False rejections at p = 0: the fraction of updates the gate rejects without any outlier, on the calibration workload
   (from the sweep) and on config 2 as config.yaml sets it (DOFs frozen; Simulator.run with nis_gate=).

Prints the card and its power limit.

    python tools/outlier_study.py [--filters 4096 65536] [--reps 7] [--study-filters 4096] [--out results/outlier_study.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench import SEED, Workload, mc_initial_states  # noqa: E402
from dvi_ekf_b200 import BatchFilter  # noqa: E402
from dvi_ekf_b200.consistency import nis_gate_threshold, summarise_dofs  # noqa: E402
from tools.consistency_cost import card  # noqa: E402
from tools.dof_envelope import DOF_NAMES  # noqa: E402

WAYS = ("production", "dropout p=0", "gate +inf", "gate 0.999", "p=0.1 + gate")
STUDY_P = (0.0, 0.05, 0.2)
STUDY_GATE = (None, 0.99, 0.999, 0.99999)


def outlier_std(wl):
    """gross errors: twenty camera noise sigmas on every channel"""
    return 20.0 * np.asarray(wl.cam_std, dtype=np.float64)


def measure(wl, n, reps):
    s = wl.s
    dev = torch.device("cuda", 0)
    t = lambda x, dt=torch.float64: torch.tensor(np.ascontiguousarray(x), dtype=dt, device=dev)
    d = dict(dt=t(s.dt), oa=t(s.om_acc), npr=t(s.n_prop, torch.int32), cam=t(s.cam), notch=t(s.notch), cam_ref=t(s.cam_ref),
             imu_ref=t(s.imu_ref))
    x0, P0, u0 = t(mc_initial_states(s.x0, n, 0)), t(wl.P0[None]), t(s.u0[None])
    gt = tuple(wl.cfg.gt_imu_dofs)
    E = len(s.n_prop)
    g999 = nis_gate_threshold(0.999)
    kws = {"production": {}, "dropout p=0": dict(drop_prob=t(np.zeros(E))), "gate +inf": dict(nis_gate=np.inf),
           "gate 0.999": dict(nis_gate=g999),
           "p=0.1 + gate": dict(nis_gate=g999, outlier_prob=t(np.full(E, 0.1)), outlier_std=outlier_std(wl))}
    bfs = {}
    for w in WAYS:
        bf = BatchFilter(n, **dict(wl.model, frozen_dofs=(0,) * 6))
        bf.set_noise(wl.Qd[None], wl.Rd[None], wl.sig_om[None])
        bfs[w] = bf
    times = {w: [] for w in WAYS}

    def run(w):
        bf = bfs[w]
        bf.set_state(x0, P0, u0, None)
        bf.sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        st, _ = bf.run(d["dt"], d["oa"], d["npr"], d["cam"], d["notch"], cam_ref=d["cam_ref"], imu_ref=d["imu_ref"],
                       stats_on_device=True, seed=SEED, imu_noise_std=wl.imu_std, cam_noise_std=wl.cam_std, gt_dofs=gt, **kws[w])
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), st

    outs = {w: run(w)[1] for w in WAYS}  # warm-up: module load, first launches of both instantiations
    # the gate at +inf rejects nothing: the statistics rows are those of the production run, bit for bit
    assert outs["gate +inf"].cpu().numpy().tobytes() == outs["production"].cpu().numpy().tobytes()
    applied = {w: float(outs[w][1:, 9].mean().item()) / E for w in ("gate 0.999", "p=0.1 + gate")}
    for r in range(reps):
        order = WAYS if r % 2 == 0 else WAYS[::-1]
        for w in order:
            times[w].append(run(w)[0])
    for bf in bfs.values():
        bf.close()
    return {w: float(np.median(v)) for w, v in times.items()}, times, applied


def study(wl, n):
    """one stacked launch, one copy of the calibration trajectory per (p, gate) cell; per-group consistency and envelope"""
    s = wl.s
    cells = [(p, g) for p in STUDY_P for g in STUDY_GATE]
    k = len(cells)
    E = len(s.n_prop)
    rep = lambda a: np.ascontiguousarray(np.concatenate([a] * k))
    thr = np.concatenate([np.full(n, np.inf if g is None else nis_gate_threshold(g)) for _, g in cells])
    with BatchFilter(n * k, **dict(wl.model, frozen_dofs=(0,) * 6)) as bf:
        bf.set_noise(wl.Qd[None], wl.Rd[None], wl.sig_om[None])
        bf.set_state(rep(mc_initial_states(s.x0, n, 0)), wl.P0[None], s.u0[None], None)
        bf.keep_consistency()
        bf.set_groups(n)
        bf.run(rep(s.dt), rep(s.om_acc), rep(s.n_prop), rep(s.cam), rep(s.notch), cam_ref=rep(s.cam_ref), imu_ref=rep(s.imu_ref),
               n_traj=k, filters_per_traj=n, noise_id_modulus=n, seed=SEED, imu_noise_std=wl.imu_std, cam_noise_std=wl.cam_std,
               gt_dofs=tuple(wl.cfg.gt_imu_dofs), nis_gate=thr, outlier_prob=np.repeat(np.array([p for p, _ in cells])[:, None], E, 1),
               outlier_std=outlier_std(wl))
        _, _, gcons, gdof = bf.get_group_sums(stats=False, consistency=True, dof_envelope=True)
    from dvi_ekf_b200.engine import outlier_mask

    m, _ = outlier_mask(np.repeat(np.array([p for p, _ in cells])[:, None], E, 1), SEED, 0, n * k, (0, E), n_traj=k,
                        filters_per_traj=n, noise_id_modulus=n)
    epochs = [e for e in (1, 10, 50, 138) if e < E]
    rows = []
    for j, (p, g) in enumerate(cells):
        es, dm = gcons[j], summarise_dofs(gdof[j], (0,) * 6)
        anis = float(es[:, 1].sum() / max(es[:, 0].sum(), 1))
        anees = float(es[:, 4].sum() / max(es[:, 3].sum(), 1))
        corrupted = int(m[j * n:(j + 1) * n].sum())
        rejected = float(dm["rejected"].sum())
        gname = "off" if g is None else f"chi2 {g} ({nis_gate_threshold(g):.2f})"
        print(f"p = {p}, gate {gname}: frames corrupted {corrupted} of {n * E}, updates rejected {rejected:.0f} "
              f"({rejected / (n * E) * 100:.1f} %), ANIS {anis:.4g} (7 if consistent), ANEES {anees:.4g} (6)")
        print(f"  {'epoch':<7}{'DOF':<13}{'RMSE':>11}{'inflation':>11}")
        r = dict(p=p, gate=g, corrupted=corrupted, rejected=rejected, anis=anis, anees=anees, dofs=[])
        for e in epochs:
            for i, dn in enumerate(DOF_NAMES):
                v = dict(epoch=e, dof=dn, rmse=float(dm["rmse"][e, i]), inflation=float(dm["inflation"][e, i]))
                r["dofs"].append(v)
                print(f"  {e:<7}{dn:<13}{v['rmse']:>11.3g}{v['inflation']:>11.3g}")
        rows.append(r)
    return rows


def false_rejections_config_yaml(n):
    """the gate's rejected fraction without outliers on config 2 as config.yaml sets it (Simulator.run(nis_gate=...))"""
    from dvi_ekf_b200.config import Config
    from dvi_ekf_b200.filter import Simulator

    sim = Simulator(Config(os.path.join(ROOT, "config.yaml")))
    out = {}
    for g in (0.99, 0.999, 0.99999):
        sim.run(consistency=True, verbose=False, n_filters=n, nis_gate=nis_gate_threshold(g))
        E = len(sim.streams.n_prop)
        rej = float(sim.dof_envelope["rejected"].sum())
        out[str(g)] = dict(rejected=rej, fraction=rej / (n * E), epochs=E)
        print(f"config.yaml, gate chi2 {g} ({nis_gate_threshold(g):.2f}), p = 0: {rej:.0f} of {n * E} updates rejected "
              f"({rej / (n * E) * 100:.2f} %)")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--filters", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--study-filters", type=int, default=4096, help="filters per cell of the sweep")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, power = card()
    wl = Workload()
    print(f"card {name}, power limit {power}")
    res = dict(card=name, power_limit=power, workload="config 2 calibration, mandala0_mono 1390 steps / 139 updates", sizes={})
    for n in a.filters:
        med, raw, applied = measure(wl, n, a.reps)
        res["sizes"][n] = dict(median_ms=med, all_ms=raw, applied_fraction=applied)
        base = med["production"]
        print(f"N={n} (median of {a.reps}, CUDA events): " +
              ", ".join(f"{w} {med[w]:.3f} ms ({(med[w] / base - 1) * 100:+.1f} %)" for w in WAYS) +
              f"; applied: gate 0.999 {applied['gate 0.999'] * 100:.1f} %, p = 0.1 + gate {applied['p=0.1 + gate'] * 100:.1f} %")
    res["study"] = dict(filters_per_cell=a.study_filters, rows=study(wl, a.study_filters))
    res["false_rejections_config_yaml"] = false_rejections_config_yaml(a.study_filters)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
