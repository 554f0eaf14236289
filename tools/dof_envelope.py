"""Per-DOF consistency of the config-2 calibration and the cost of its getters (eskf_get_dof_envelope,
eskf_get_dof_history): eskf_run on the config-2 calibration workload (mandala0_mono, 140 frames x 10 IMU samples, all six
DOFs estimated from perturbed values, Monte-Carlo noise, statistics on the device) with consistency on.  Prints the card,
its power limit, a per-DOF table at epochs 1, 10, 50 and the last (bias, RMSE, filter sigma, inflation, per-DOF ANEES
and its 95 % interval, 1-sigma coverage) at the first size, and the time of each getter, timed with CUDA events as the
median of interleaved calls, also as a fraction of the consistency run.  The table describes the reference's filter, not
the engine.

    python tools/dof_envelope.py [--filters 4096 65536] [--reps 7] [--out results/dof_envelope.json]
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
from dvi_ekf_b200.consistency import summarise_dofs  # noqa: E402
from tools.consistency_cost import card  # noqa: E402

DOF_NAMES = ("rot x [rad]", "rot y [rad]", "rot z [rad]", "trans x [cm]", "trans y [cm]", "trans z [cm]")


def measure(wl, n, reps):
    """median times [ms] of the consistency run and of each getter, interleaved call by call; and the envelope"""
    s = wl.s
    dev = torch.device("cuda", 0)
    t = lambda x, dt=torch.float64: torch.tensor(np.ascontiguousarray(x), dtype=dt, device=dev)
    d = dict(dt=t(s.dt), oa=t(s.om_acc), npr=t(s.n_prop, torch.int32), cam=t(s.cam), notch=t(s.notch), cam_ref=t(s.cam_ref),
             imu_ref=t(s.imu_ref))
    x0, P0, u0 = t(mc_initial_states(s.x0, n, 0)), t(wl.P0[None]), t(s.u0[None])
    bf = BatchFilter(n, **dict(wl.model, frozen_dofs=(0,) * 6))
    bf.set_noise(wl.Qd[None], wl.Rd[None], wl.sig_om[None])
    bf.keep_consistency()

    def timed(fn):
        bf.sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def run():
        bf.set_state(x0, P0, u0, None)
        bf.run(d["dt"], d["oa"], d["npr"], d["cam"], d["notch"], cam_ref=d["cam_ref"], imu_ref=d["imu_ref"], stats_on_device=True,
               seed=SEED, imu_noise_std=wl.imu_std, cam_noise_std=wl.cam_std, gt_dofs=tuple(wl.cfg.gt_imu_dofs))

    calls = dict(run=run, envelope=lambda: bf.get_dof_envelope(device=True),
                 history_device=lambda: bf.get_dof_history(device=True), history_host=bf.get_dof_history)
    times = {k: [] for k in calls}
    for fn in calls.values():  # warm-up: module load, first launches, allocations
        fn()
    for _ in range(reps):
        for k, fn in calls.items():
            times[k].append(timed(fn))
    env = bf.get_dof_envelope()
    bf.close()
    return {k: float(np.median(v)) for k, v in times.items()}, times, env


def table(env, E):
    sm = summarise_dofs(env, (0,) * 6)
    rows = []
    for e in sorted({1, 10, 50, E - 1}):
        if e >= E:
            continue
        print(f"epoch {e} (M = {sm['count'][e]:.0f}, excluded {sm['excluded'][e]:.0f}; per-DOF ANEES 95 % interval "
              f"[{sm['anees_interval'][e, 0]:.3f}, {sm['anees_interval'][e, 1]:.3f}], expected 1-sigma coverage "
              f"{sm['coverage_expected'][0]:.3f})")
        print(f"  {'DOF':<13}{'bias':>11}{'RMSE':>11}{'filter sig':>11}{'inflation':>11}{'ANEES_i':>11}{'1-sig cov':>11}")
        for i, nm in enumerate(DOF_NAMES):
            r = dict(epoch=e, dof=nm, bias=float(sm["bias"][e, i]), rmse=float(sm["rmse"][e, i]),
                     sigma_filter=float(sm["sigma_filter"][e, i]), inflation=float(sm["inflation"][e, i]),
                     anees=float(sm["anees_dof"][e, i]), anees_interval=sm["anees_interval"][e].tolist(),
                     coverage1=float(sm["coverage"][e, i, 0]))
            rows.append(r)
            print(f"  {nm:<13}{r['bias']:>11.3g}{r['rmse']:>11.3g}{r['sigma_filter']:>11.3g}{r['inflation']:>11.3g}"
                  f"{r['anees']:>11.3g}{r['coverage1']:>11.3f}")
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--filters", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, power = card()
    wl = Workload()
    E = len(wl.s.n_prop)
    res = dict(card=name, power_limit=power, workload="config 2 calibration, mandala0_mono 1390 steps / 139 updates", sizes={})
    print(f"card {name}, power limit {power}")
    for i, n in enumerate(a.filters):
        med, raw, env = measure(wl, n, a.reps)
        res["sizes"][n] = dict(median_ms=med, all_ms=raw)
        line = ", ".join(f"{k} {v:.4f} ms ({v / med['run'] * 100:.2f} % of the run)" for k, v in med.items() if k != "run")
        print(f"N={n}: consistency run {med['run']:.3f} ms; {line} (median of {a.reps})")
        if i == 0:
            res["table"] = dict(n=n, rows=table(env, E))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
