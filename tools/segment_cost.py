"""Cost of running a trajectory in epoch segments (BatchFilter.run_segments / eskf_run_epochs) against one eskf_run, timed with
CUDA events (device-resident streams and statistics), the variants interleaved run by run:

  * config 2 (mandala0_mono, 140 frames x 10 IMU samples, Monte-Carlo noise) and its calibration variant (all six DOFs
    estimated from perturbed values) at --filters filters: one eskf_run, and 7 and 139 segments -- the cost per boundary;
  * config 5 (--big filters of config 2): one launch, which keeps the Monte-Carlo generator in the persistent kernel because
    the pre-pass buffers of the whole run exceed the default budget, against segments of --big-seg epochs whose buffers fit;
  * consistency on config 5: one eskf_run (ESKF_ENOMEM where its records do not fit), and the same in segments.

Prints the card and its power limit first.

    python tools/segment_cost.py [--filters 4096] [--reps 7] [--big 1048576] [--big-seg 35] [--out results/segment_cost.json]
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
from dvi_ekf_b200._lib import EskfError  # noqa: E402
from tools.consistency_cost import card  # noqa: E402


def streams(wl):
    s = wl.s
    dev = torch.device("cuda", 0)
    t = lambda x, dt=torch.float64: torch.tensor(np.ascontiguousarray(x), dtype=dt, device=dev)
    return dict(dt=t(s.dt), om_acc=t(s.om_acc), n_prop=t(s.n_prop, torch.int32), cam=t(s.cam), notch=t(s.notch),
                cam_ref=t(s.cam_ref), imu_ref=t(s.imu_ref)), t


def timed(bf, reset, fn):
    reset()
    bf.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def bounds(E, k):
    """k segments of (nearly) equal epoch counts"""
    return sorted(set(int(round(v)) for v in np.linspace(0, E, k + 1)))


def compare(wl, n, reps, calibration, variants, consistency=False, budget=None):
    """median ms per variant: None = one eskf_run, k = k segments (or a list of boundaries); the final stats_sum of each
    variant is checked bit for bit against the one-launch run"""
    d, t = streams(wl)
    E = len(wl.s.n_prop)
    model = dict(wl.model, frozen_dofs=(0,) * 6) if calibration else wl.model
    x0 = t(mc_initial_states(wl.s.x0, n, 0))
    P0, u0 = t(wl.P0[None]), t(wl.s.u0[None])
    kw = dict(stats_on_device=True, seed=SEED, imu_noise_std=wl.imu_std, cam_noise_std=wl.cam_std,
              gt_dofs=tuple(wl.cfg.gt_imu_dofs) if calibration else (0, 0, 0, 0, 0, 20.0))
    bf = BatchFilter(n, **model)
    bf.set_noise(wl.Qd[None], wl.Rd[None], wl.sig_om[None])
    if budget is not None:
        bf.set_prepass_budget(budget)
    if consistency:
        bf.keep_consistency()
    reset = lambda: bf.set_state(x0, P0, u0, None)

    def one(v):
        if v is None:
            return bf.run(**d, **kw)[1]
        sm = None
        for _, _, _, sm in bf.run_segments(boundaries=bounds(E, v) if isinstance(v, int) else v, **d, **kw):
            pass
        return sm

    times, sums = {v: [] for v in variants}, {}
    for v in variants:  # warm-up: module load, first launches
        _, sums[v] = timed(bf, reset, lambda: one(v))
    for r in range(reps):
        for v in (variants if r % 2 == 0 else variants[::-1]):
            times[v].append(timed(bf, reset, lambda: one(v))[0])
    same = {str(v): bool(sums[v].cpu().numpy().tobytes() == sums[variants[0]].cpu().numpy().tobytes()) for v in variants}
    bf.close()
    torch.cuda.empty_cache()
    return {str(v): dict(median_ms=float(np.median(times[v])), all_ms=times[v]) for v in variants}, same


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--filters", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--big", type=int, default=1 << 20)
    ap.add_argument("--big-seg", type=int, default=35)
    ap.add_argument("--big-reps", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, power = card()
    print(f"card {name}, power limit {power}")
    wl = Workload()
    E = len(wl.s.n_prop)
    res = dict(card=name, power_limit=power, epochs=E, steps=int(len(wl.s.dt)))
    for calib in (False, True):
        tag = "config2_calibration" if calib else "config2"
        r, same = compare(wl, a.filters, a.reps, calib, [None, 7, E])
        res[tag] = dict(filters=a.filters, times=r, bit_identical=same)
        base = r["None"]["median_ms"]
        for k in ("7", str(E)):
            per = (r[k]["median_ms"] - base) / (int(k) - 1)
            print(f"{tag} N={a.filters}: one launch {base:.3f} ms, {k} segments {r[k]['median_ms']:.3f} ms "
                  f"({per * 1e3:.1f} us per boundary), stats_sum bit-identical: {same[k]}")
    nseg = -(-E // a.big_seg)
    r, same = compare(wl, a.big, a.big_reps, False, [None, nseg])
    res["config5"] = dict(filters=a.big, segment_epochs=a.big_seg, times=r, bit_identical=same)
    print(f"config5 N={a.big}: one launch {r['None']['median_ms']:.1f} ms, {nseg} segments of <= {a.big_seg} epochs "
          f"{r[str(nseg)]['median_ms']:.1f} ms (median of {a.big_reps}), stats_sum bit-identical: {same[str(nseg)]}")
    try:
        r1, _ = compare(wl, a.big, 1, False, [None], consistency=True)
        res["config5_consistency_one_launch"] = r1
        print(f"config5 consistency, one launch: {r1['None']['median_ms']:.1f} ms")
    except EskfError as e:
        res["config5_consistency_one_launch"] = str(e)
        print(f"config5 consistency, one launch: {e}")
    r2, _ = compare(wl, a.big, 1, False, [nseg], consistency=True)
    res["config5_consistency_segments"] = r2
    print(f"config5 consistency, {nseg} segments: {r2[str(nseg)]['median_ms']:.1f} ms (one run after warm-up)")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
