"""Cost of filter consistency (eskf_keep_consistency): eskf_run on the config-2 calibration workload (mandala0_mono, 140
frames x 10 IMU samples, all six DOFs estimated from perturbed values, Monte-Carlo noise, statistics on the device) with
consistency off and on, timed with CUDA events, the two handles interleaved run by run.  "On" runs the export
instantiation of the persistent kernel and the consistency post-pass.  Prints the card, its power limit, the median times
and the ANIS / ANEES of the run at the first size.

    python tools/consistency_cost.py [--filters 4096 65536] [--reps 7] [--out results/consistency_cost.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench import SEED, Workload, mc_initial_states  # noqa: E402
from dvi_ekf_b200 import BatchFilter  # noqa: E402
from dvi_ekf_b200.consistency import summarise_consistency  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def measure(wl, n, reps):
    s = wl.s
    dev = torch.device("cuda", 0)
    t = lambda x, dt=torch.float64: torch.tensor(np.ascontiguousarray(x), dtype=dt, device=dev)
    d = dict(dt=t(s.dt), oa=t(s.om_acc), npr=t(s.n_prop, torch.int32), cam=t(s.cam), notch=t(s.notch), cam_ref=t(s.cam_ref),
             imu_ref=t(s.imu_ref))
    x0, P0, u0 = t(mc_initial_states(s.x0, n, 0)), t(wl.P0[None]), t(s.u0[None])
    gt = tuple(wl.cfg.gt_imu_dofs)
    model = dict(wl.model, frozen_dofs=(0,) * 6)
    bfs = {}
    for on in (False, True):
        bf = BatchFilter(n, **model)
        bf.set_noise(wl.Qd[None], wl.Rd[None], wl.sig_om[None])
        if on:
            bf.keep_consistency()
        bfs[on] = bf
    times = {False: [], True: []}

    def run(on):
        bf = bfs[on]
        bf.set_state(x0, P0, u0, None)
        bf.sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        bf.run(d["dt"], d["oa"], d["npr"], d["cam"], d["notch"], cam_ref=d["cam_ref"], imu_ref=d["imu_ref"], stats_on_device=True,
               seed=SEED, imu_noise_std=wl.imu_std, cam_noise_std=wl.cam_std, gt_dofs=gt)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    for on in (False, True):  # warm-up: module load, first launches of both instantiations
        run(on)
    for r in range(reps):
        for on in ((False, True) if r % 2 == 0 else (True, False)):
            times[on].append(run(on))
    _, _, es = bfs[True].get_consistency()
    for bf in bfs.values():
        bf.close()
    return {k: float(np.median(v)) for k, v in times.items()}, {k: v for k, v in times.items()}, es


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--filters", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, power = card()
    wl = Workload()
    res = dict(card=name, power_limit=power, workload="config 2 calibration, mandala0_mono 1390 steps / 139 updates", sizes={})
    print(f"card {name}, power limit {power}")
    for i, n in enumerate(a.filters):
        med, raw, es = measure(wl, n, a.reps)
        cost = med[True] / med[False] - 1
        res["sizes"][n] = dict(off_ms=med[False], on_ms=med[True], cost=cost, off_all=raw[False], on_all=raw[True])
        print(f"N={n}: consistency off {med[False]:.3f} ms, on {med[True]:.3f} ms (median of {a.reps}): +{cost * 100:.1f} %")
        if i == 0:
            sm = summarise_consistency(es, 6)
            fin = es[:, 0] > 0
            anis = float(es[fin, 1].sum() / es[fin, 0].sum())
            anees = float(es[:, 4].sum() / max(es[:, 3].sum(), 1))
            res["consistency"] = dict(n=n, anis_all=anis, anees_all=anees, nis_inside=sm["nis_inside"], nees_inside=sm["nees_inside"],
                                      anis_first=float(sm["anis"][0]), anees_first=float(sm["anees"][0]),
                                      anis_last=float(sm["anis"][-1]), anees_last=float(sm["anees"][-1]),
                                      skipped_total=sm["skipped_total"])
            print(f"N={n}: ANIS {anis:.4g} (7 if consistent), ANEES {anees:.4g} (6), over all epochs; epochs inside the 95 % "
                  f"interval: NIS {sm['nis_inside']:.2f}, NEES {sm['nees_inside']:.2f}; first / last epoch ANIS "
                  f"{sm['anis'][0]:.4g} / {sm['anis'][-1]:.4g}, ANEES {sm['anees'][0]:.4g} / {sm['anees'][-1]:.4g}; "
                  f"skipped {sm['skipped_total']:.0f}")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
