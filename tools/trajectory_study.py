"""Which motion makes which calibration DOF observable: one Monte-Carlo study over the six canonical motions (trans_x/y/z,
rot_x/y/z) and mandala0_mono, cut to their common 60 frames (10 IMU samples per frame), all six DOFs estimated from perturbed
values, 4,096 filters per trajectory, Monte-Carlo noise, consistency on -- ONE stacked launch with one filter group per
trajectory (Simulator.run_trajectories).  Prints the card and its power limit, per trajectory and DOF at the first and the
last epoch: bias, RMSE, the filter's claimed sigma, inflation, per-DOF ANEES and 1-sigma coverage; and the time of the run,
of the ungrouped envelope getter (eskf_get_dof_envelope), of the grouped one (eskf_get_group_sums with the envelope) with one
group per trajectory, and of the grouped one with groups of 8 (tuning-candidate sized), timed with CUDA events as the median
of interleaved calls.  The table describes the reference's filter, not the engine.

    python tools/trajectory_study.py [--filters 4096] [--reps 7] [--out results/trajectory_study.json]
"""
import argparse
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import yaml  # noqa: E402

from dvi_ekf_b200 import Config, Simulator  # noqa: E402
from tools.consistency_cost import card  # noqa: E402
from tools.dof_envelope import DOF_NAMES  # noqa: E402

NAMES = ("trans_x", "trans_y", "trans_z", "rot_x", "rot_y", "rot_z", "mandala0_mono")
FRAMES = 60


def simulator(tmp):
    """config.yaml with the calibration variant: all six DOFs estimated, full trajectories, 10 IMU samples per frame"""
    y = yaml.safe_load(open(os.path.join(ROOT, "config.yaml")))
    y["simulation"].update(do_fast_sim=False, frozen_dofs=[0] * 6)
    y["camera"]["total_frames"] = "all"
    fp = os.path.join(tmp, "config.yaml")
    with open(fp, "w") as f:
        yaml.safe_dump(y, f)
    return Simulator(Config(fp))


def measure(sim, n, reps):
    """median times [ms]: the run, the ungrouped and grouped envelope getters with one group per trajectory, then (after a
    run with groups of 8) the ungrouped and the grouped getter at g = 8; interleaved call by call"""
    bf, kw = sim._stacked_trajectories(NAMES, n, frames=FRAMES, consistency=True)
    dev = torch.device("cuda", 0)
    for k in ("dt", "om_acc", "n_prop", "cam", "notch", "cam_ref", "imu_ref"):
        kw[k] = torch.tensor(np.ascontiguousarray(kw[k]), device=dev)
    kw["n_prop"] = kw["n_prop"].to(torch.int32)
    x0 = bf.get_state(device=True)[:4]

    def timed(fn):
        bf.sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def run():
        bf.set_state(*x0)
        bf.run(stats_on_device=True, **kw)

    envelope = lambda: bf.get_dof_envelope(device=True)
    grouped = lambda: bf.get_group_sums(stats=False, dof_envelope=True, device=True)
    times = {}
    with bf:
        for phase, calls in ((n, dict(run=run, envelope=envelope, grouped_per_trajectory=grouped)),
                             (8, dict(envelope_g8_records=envelope, grouped_g8=grouped))):
            bf.set_groups(phase)
            run()
            for fn in calls.values():  # warm-up: module load, first launches, allocations
                fn()
            for k in calls:
                times[k] = []
            for _ in range(reps):
                for k, fn in calls.items():
                    times[k].append(timed(fn))
            if phase == n:
                env = bf.get_dof_envelope()
                genv = bf.get_group_sums(stats=False, dof_envelope=True)[3]
                # the groups add up to the ungrouped envelope (counts exactly)
                assert np.array_equal(genv.sum(axis=0)[:, :2], env[:, :2])
    return {k: float(np.median(v)) for k, v in times.items()}, times


def table(res, E):
    rows = []
    for nm in NAMES:
        sm = res[nm]["dof_envelope"]
        for e in (0, E - 1):
            print(f"{nm}, epoch {e} (M = {sm['count'][e]:.0f}, excluded {sm['excluded'][e]:.0f}; per-DOF ANEES 95 % interval "
                  f"[{sm['anees_interval'][e, 0]:.3f}, {sm['anees_interval'][e, 1]:.3f}])")
            print(f"  {'DOF':<13}{'bias':>11}{'RMSE':>11}{'filter sig':>11}{'inflation':>11}{'ANEES_i':>11}{'1-sig cov':>11}")
            for i, dn in enumerate(DOF_NAMES):
                r = dict(trajectory=nm, epoch=e, dof=dn, bias=float(sm["bias"][e, i]), rmse=float(sm["rmse"][e, i]),
                         sigma_filter=float(sm["sigma_filter"][e, i]), inflation=float(sm["inflation"][e, i]),
                         anees=float(sm["anees_dof"][e, i]), coverage1=float(sm["coverage"][e, i, 0]))
                rows.append(r)
                print(f"  {dn:<13}{r['bias']:>11.3g}{r['rmse']:>11.3g}{r['sigma_filter']:>11.3g}{r['inflation']:>11.3g}"
                      f"{r['anees']:>11.3g}{r['coverage1']:>11.3f}")
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--filters", type=int, default=4096, help="filters per trajectory")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, power = card()
    print(f"card {name}, power limit {power}")
    with tempfile.TemporaryDirectory() as tmp:
        sim = simulator(tmp)
    res = sim.run_trajectories(NAMES, a.filters, frames=FRAMES, consistency=True)
    E = len(res[NAMES[0]]["consistency"]["anis"])
    out = dict(card=name, power_limit=power, filters_per_trajectory=a.filters, trajectories=list(NAMES), frames=FRAMES,
               epochs=E, table=table(res, E))
    med, raw = measure(sim, a.filters, a.reps)
    out.update(median_ms=med, all_ms=raw)
    n = a.filters * len(NAMES)
    print(f"{len(NAMES)} trajectories x {a.filters} filters = {n} filters, {E} epochs (median of {a.reps}, CUDA events):")
    print(f"  run (set_state + eskf_run, consistency on, groups of {a.filters}) {med['run']:.3f} ms")
    for k in ("envelope", "grouped_per_trajectory", "envelope_g8_records", "grouped_g8"):
        print(f"  {k:<24} {med[k]:.4f} ms ({med[k] / med['run'] * 100:.2f} % of the run)")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
