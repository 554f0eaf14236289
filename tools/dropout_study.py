"""Simulated frame loss (``BatchFilter.run(drop_prob=...)``, eskf_set_meas_dropout) on the config-2 calibration workload
(mandala0_mono, 140 frames x 10 IMU samples, all six DOFs estimated from perturbed values, Monte-Carlo noise).

1. Cost: eskf_run at each size three ways -- dropout off (the production instantiation), dropout set with p = 0 everywhere
   (the export instantiation, no frame lost) and p = 0.2 -- timed with CUDA events, the three handles interleaved run by run;
   the median of the runs.
2. Science: ONE stacked launch of the calibration trajectory repeated for p in {0, 0.1, 0.3, 0.5}, filters_per_traj = n,
   noise_id_modulus = n and one filter group per copy, consistency on: every copy sees the same noise and initial DOFs, and
   the masks nest (a frame lost at p is lost at every larger p).  Per p: ANIS / ANEES over all epochs, frames lost, and per
   DOF the RMSE, inflation and 1-sigma coverage at epochs 1, 10, 50 and the last.

Prints the card and its power limit.

    python tools/dropout_study.py [--filters 4096 65536] [--reps 7] [--study-filters 4096] [--out results/dropout_study.json]
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
from dvi_ekf_b200.consistency import summarise_consistency, summarise_dofs  # noqa: E402
from tools.consistency_cost import card  # noqa: E402
from tools.dof_envelope import DOF_NAMES  # noqa: E402

WAYS = ("off", "p=0", "p=0.2")
STUDY_P = (0.0, 0.1, 0.3, 0.5)


def measure(wl, n, reps):
    s = wl.s
    dev = torch.device("cuda", 0)
    t = lambda x, dt=torch.float64: torch.tensor(np.ascontiguousarray(x), dtype=dt, device=dev)
    d = dict(dt=t(s.dt), oa=t(s.om_acc), npr=t(s.n_prop, torch.int32), cam=t(s.cam), notch=t(s.notch), cam_ref=t(s.cam_ref),
             imu_ref=t(s.imu_ref))
    x0, P0, u0 = t(mc_initial_states(s.x0, n, 0)), t(wl.P0[None]), t(s.u0[None])
    gt = tuple(wl.cfg.gt_imu_dofs)
    E = len(s.n_prop)
    prob = {"off": None, "p=0": t(np.zeros(E)), "p=0.2": t(np.full(E, 0.2))}
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
                       stats_on_device=True, seed=SEED, imu_noise_std=wl.imu_std, cam_noise_std=wl.cam_std, gt_dofs=gt,
                       drop_prob=prob[w])
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), st

    outs = {w: run(w)[1] for w in WAYS}  # warm-up: module load, first launches of both instantiations
    # p = 0 loses nothing: the statistics rows are those of the run without dropout, bit for bit
    assert outs["p=0"].cpu().numpy().tobytes() == outs["off"].cpu().numpy().tobytes()
    applied = float(outs["p=0.2"][1:, 9].mean().item()) / E
    for r in range(reps):
        order = WAYS if r % 2 == 0 else WAYS[::-1]
        for w in order:
            times[w].append(run(w)[0])
    for bf in bfs.values():
        bf.close()
    return {w: float(np.median(v)) for w, v in times.items()}, times, applied


def study(wl, n):
    """one stacked launch, copy j of the calibration trajectory with p = STUDY_P[j]; per-group consistency and envelope"""
    s = wl.s
    k = len(STUDY_P)
    E = len(s.n_prop)
    rep = lambda a: np.ascontiguousarray(np.concatenate([a] * k))
    with BatchFilter(n * k, **dict(wl.model, frozen_dofs=(0,) * 6)) as bf:
        bf.set_noise(wl.Qd[None], wl.Rd[None], wl.sig_om[None])
        bf.set_state(rep(mc_initial_states(s.x0, n, 0)), wl.P0[None], s.u0[None], None)
        bf.keep_consistency()
        bf.set_groups(n)
        bf.run(rep(s.dt), rep(s.om_acc), rep(s.n_prop), rep(s.cam), rep(s.notch), cam_ref=rep(s.cam_ref), imu_ref=rep(s.imu_ref),
               n_traj=k, filters_per_traj=n, noise_id_modulus=n, seed=SEED, imu_noise_std=wl.imu_std, cam_noise_std=wl.cam_std,
               gt_dofs=tuple(wl.cfg.gt_imu_dofs), drop_prob=np.repeat(np.array(STUDY_P)[:, None], E, 1))
        _, _, gcons, gdof = bf.get_group_sums(stats=False, consistency=True, dof_envelope=True)
    epochs = [e for e in (1, 10, 50, E - 1) if e < E]
    rows = []
    for j, p in enumerate(STUDY_P):
        es, sm, dm = gcons[j], summarise_consistency(gcons[j], 6), summarise_dofs(gdof[j], (0,) * 6)
        anis = float(es[:, 1].sum() / max(es[:, 0].sum(), 1))
        anees = float(es[:, 4].sum() / max(es[:, 3].sum(), 1))
        lost = float(sm["dropped"].sum())
        print(f"p = {p}: ANIS {anis:.4g} (7 if consistent), ANEES {anees:.4g} (6), frames lost {lost:.0f} of {n * E} "
              f"({lost / (n * E) * 100:.1f} %)")
        print(f"  {'epoch':<7}{'DOF':<13}{'RMSE':>11}{'inflation':>11}{'1-sig cov':>11}")
        r = dict(p=p, anis=anis, anees=anees, frames_lost=lost, dofs=[])
        for e in epochs:
            for i, dn in enumerate(DOF_NAMES):
                v = dict(epoch=e, dof=dn, rmse=float(dm["rmse"][e, i]), inflation=float(dm["inflation"][e, i]),
                         coverage1=float(dm["coverage"][e, i, 0]))
                r["dofs"].append(v)
                print(f"  {e:<7}{dn:<13}{v['rmse']:>11.3g}{v['inflation']:>11.3g}{v['coverage1']:>11.3f}")
        rows.append(r)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--filters", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--study-filters", type=int, default=4096, help="filters per copy of the trajectory in the study")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, power = card()
    wl = Workload()
    print(f"card {name}, power limit {power}")
    res = dict(card=name, power_limit=power, workload="config 2 calibration, mandala0_mono 1390 steps / 139 updates", sizes={})
    for n in a.filters:
        med, raw, applied = measure(wl, n, a.reps)
        res["sizes"][n] = dict(median_ms=med, all_ms=raw, applied_fraction_p02=applied)
        print(f"N={n} (median of {a.reps}, CUDA events): off {med['off']:.3f} ms, p = 0 set {med['p=0']:.3f} ms "
              f"({(med['p=0'] / med['off'] - 1) * 100:+.1f} %), p = 0.2 {med['p=0.2']:.3f} ms "
              f"({(med['p=0.2'] / med['off'] - 1) * 100:+.1f} %; {applied * 100:.1f} % of the updates applied)")
    res["study"] = dict(filters_per_copy=a.study_filters, rows=study(wl, a.study_filters))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
