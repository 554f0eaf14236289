#!/usr/bin/env python
"""Benchmark of the batched VI-ESKF hot path (BASELINE.json metric: ESKF filter-steps/sec).

One "step" of this benchmark = one pass of the hot path over one batch: every filter of the batch runs
the whole default simulated trajectory (mandala0_mono, 140 camera frames, 10 IMU samples per frame:
1390 x Filter.propagate + 139 x Filter.update) inside ONE persistent kernel launch.  One *filter-step*
(the metric's unit) = one Filter.propagate on one filter.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--filters F] [--impl ours|reference] [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed pass computed (per-filter statistics, the reduced statistics vector, final
state x and covariance P) as DIR/<name>.npy, so that two builds can be compared output for output on identical inputs.

N > 1 is launched by torchrun (one rank per GPU); every rank runs its own shard of the Monte-Carlo batch
(weak scaling: --filters is per GPU; Philox noise is keyed by the GLOBAL filter id) and the only
collective is the all-reduce of the 16-entry error-statistics vector, inside the timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

# stdout carries ONE JSON line: NCCL prints its "NCCL version ..." banner to stdout at the levels VERSION (set on the GPU
# boxes) and WARN; the level is switched off before anything loads NCCL (an explicit INFO / TRACE of the user is left alone)
if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
    os.environ["NCCL_DEBUG"] = "NONE"

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "eskf_filter_steps_per_sec"
UNIT = "filter-steps/s"
N_FRAMES, IFV = 140, 10
# algorithmic FP64 flops per filter-step, SURVEY.md section 8(d) / BASELINE.md section 5 (ifv = 10)
F_MIN_PER_STEP = 9031 + 29587 / IFV  # structure-aware lower bound  (11,990)
F_DENSE_PER_STEP = 78960 + 160767 / IFV  # reference-as-executed dense matmuls (95,037)
SEED = 1234


class Workload:
    """Config 2 of BASELINE.md: the default simulated trajectory (full variant: 140 frames, 10 IMU samples per
    frame), HEAD behaviour, built by the PRODUCT's host pre-pass (dvi_ekf_b200.camera) from config.yaml."""

    def __init__(self):
        from dvi_ekf_b200.camera import Camera, build_streams, load_trajectory
        from dvi_ekf_b200.config import Config

        cfg = Config(os.path.join(ROOT, "config.yaml"))
        cfg.update_dofs()
        self.cfg = cfg
        t, xyz, q = load_trajectory("mandala0_mono", max_vals=N_FRAMES)
        cam = Camera(t, xyz, q, scale=cfg.camera.scale)
        self.s = build_streams(cam, IFV, cfg.model.length, cfg.model.angle)
        self.P0 = cfg.cov0_matrix
        rw = cfg.filter.noise_dofs.vec / IFV  # config.py:258 with interframe_vals = 10
        self.Qd = np.hstack((np.zeros(6), np.square(rw)))  # Q[0:6] = 0: Filter.py:40,68-72
        self.Rd = np.square(cfg.meas_noise_std)
        self.sig_om = np.array(cfg.imu.stdev_omega)
        self.imu_std = np.hstack((cfg.imu.stdev_omega, cfg.imu.stdev_accel))  # config.py:105-120
        self.cam_std = np.array(cfg.meas_noise_std)  # config.yaml:20-23
        self.model = dict(scope_length=cfg.model.length, cam_angle_rad=cfg.model.angle, frozen_dofs=cfg.frozen_dofs,
                          zero_frozen_dofs=True)


def mc_initial_states(x0_row, n, first_id):
    from dvi_ekf_b200.sharding import mc_initial_states as _mc

    return _mc(x0_row, n, first_id, SEED)


# ----------------------------------------------------------------------------------------------
# CPU arm: the batch-vectorised numpy oracle (a port: the reference itself needs casadi /
# roboticstoolbox, which are not installable here -- DESIGN.md)


def _cpu_worker(args):
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    n, n_epochs, seed = args
    from oracle.batch_oracle import BatchOracle
    from tests.helpers import mandala_scenario

    sc = mandala_scenario(np.load(os.path.join(ROOT, "tests", "golden", "reference_golden.npz")), n_frames=N_FRAMES, ifv=IFV)
    rng = np.random.default_rng(seed)
    x0 = np.repeat(sc.x0[None], n, 0)
    x0[:, 10:13] += rng.normal(0.0, np.deg2rad(3.0), (n, 3))
    bo = BatchOracle(sc.cfg, x0, sc.P0, sc.u0)
    t0 = time.perf_counter()
    steps = bo.run(sc.dt, sc.om_acc, sc.n_prop[:n_epochs], sc.cam_meas, sc.notch_meas)
    return n * steps, time.perf_counter() - t0


def cpu_sample(procs, filters_per_proc, n_epochs):
    """Runs the batch oracle on `procs` host processes; returns (filter-steps, seconds)."""
    import multiprocessing as mp

    jobs = [(filters_per_proc, n_epochs, 100 + i) for i in range(procs)]
    t0 = time.perf_counter()
    if procs == 1:
        res = [_cpu_worker(jobs[0])]
    else:
        with mp.get_context("spawn").Pool(procs) as pool:
            res = pool.map(_cpu_worker, jobs)
    wall = time.perf_counter() - t0
    work = sum(r[0] for r in res)
    busy = max(r[1] for r in res)  # slowest worker, excludes interpreter start-up
    return work, busy, wall


def workload_config(n, T, E, world, fpc):
    """`config` of the JSON line: the same for both arms (the reference arm times a bounded sample of it)."""
    return {
        "workload": f"config2: {n} Monte-Carlo filters per GPU (Philox noise seeds, DOF IC perturbation) on the default "
                    f"simulated trajectory mandala0_mono, {N_FRAMES} frames x {IFV} IMU samples "
                    f"({T} propagates + {E} updates per filter per pass)",
        "filters_per_gpu": n, "filter_steps_per_pass": int(n) * T * world,
        "l2": "flushed between timed iterations (256 MiB memset)", "filters_per_cta": fpc or "auto",
        "parallelism": f"filters sharded over {world} GPU(s)",
    }


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    fpp, n_epochs = 256, 32  # bounded sample per step: cores x 256 filters x 32 epochs (320 propagates + 32 updates)
    for _ in range(a.warmup):
        cpu_sample(cores, 32, 1)
    times, work = [], 0
    for _ in range(a.steps):
        w, busy, _ = cpu_sample(cores, fpp, n_epochs)
        times.append(busy)
        work = w
    ms = 1e3 * float(np.mean(times))
    val = work / (ms * 1e-3)
    sample = f"{cores} procs x {fpp} filters x {n_epochs} epochs ({n_epochs * IFV} propagates + {n_epochs} updates) per step"
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": dict(workload_config(a.filters, (N_FRAMES - 1) * IFV, N_FRAMES - 1, 1, a.fpc), sample=sample),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "numpy batch-vectorised port of the reference algorithm (oracle/batch_oracle.py); the reference itself "
                "cannot be installed here (casadi, roboticstoolbox, spatialmath absent; pydantic v2) and would be slower",
    }
    print(json.dumps(line), flush=True)
    return 0


# ----------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md recipe), sampled through NVML every
    few milliseconds from a thread of this process (the timed region of the default run lasts a few hundred ms,
    shorter than the start-up of an `nvidia-smi -lms` child)."""

    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}

    def __init__(self, index, period_s=0.004):
        self.index, self.period = index, period_s
        self.sm, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self.thr = None
        self.err = None

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.index
            if vis:
                try:
                    idx = int(vis.split(",")[self.index])
                except Exception:
                    pass
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.thr = threading.Thread(target=self._loop, daemon=True)
            self.thr.start()
        except Exception as e:  # no NVML: reported, not fatal
            self.err = f"NVML unavailable: {e}"

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                for name, bit in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception as e:
                self.err = str(e)
                break
            time.sleep(self.period)

    def stop(self):
        self._stop.set()
        if self.thr:
            self.thr.join(timeout=1.0)
        out = {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
               "reasons": sorted(self.reasons), "samples": len(self.sm)}
        if self.err:
            out["note"] = self.err
        return out


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback"


def ncu_traffic():
    """dram bytes per launch of the dominant kernel from the committed ncu capture, if any."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            try:
                return json.load(open(p))
            except Exception:
                pass
    return None


DUMP_BYTES = 64 << 20
DUMP_SEED = 20240


def dump_rows(n, bytes_per_row, budget):
    """Rows of the per-filter outputs that --dump-outputs writes: all of them if they fit the budget, else a fixed seeded
    sample (sorted), the same from run to run for the same n."""
    cap = budget // bytes_per_row
    if n <= cap:
        return None
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=cap, replace=False))


def last_pass_outputs(bf, st, sm, budget):
    """The arrays a caller of the timed pass receives: per-filter statistics [N,16] and the reduced vector [16] from run(),
    the final state x [N,26] and covariance P [N,24,24] from get_state(); a seeded row sample above `budget` bytes."""
    import torch

    x, P, _, _, _ = bf.get_state(device=True)
    rows = dump_rows(bf.n, (st.shape[1] + x.shape[1] + P.shape[1] * P.shape[2]) * 8, budget - sm.numel() * 8)
    per = {"stats": st, "x": x, "P": P}
    if rows is not None:
        idx = torch.from_numpy(rows).to(st.device)
        per = {k: v.index_select(0, idx) for k, v in per.items()}
    out = {k: v.cpu().numpy() for k, v in per.items()}
    out["stats_sum"] = sm.cpu().numpy()
    return out


def _guard(launch, dev):
    """One launch of a secondary workload: an exception on THIS rank (bad geometry, out of memory) must not leave the other
    ranks waiting in the all-reduce that follows, so the launch is caught here and answered with a NaN vector; the
    collective then still runs on every rank and the figure of the workload comes out as NaN."""
    import torch

    try:
        return launch()
    except Exception as e:
        print(f"bench.py: secondary workload failed on this rank: {type(e).__name__}: {e}", file=sys.stderr, flush=True)
        return torch.full((16,), float("nan"), dtype=torch.float64, device=dev)


def _timed(fn, reset, reps, barrier, flush):
    """mean device time [ms] of `reps` calls of fn (CUDA events on torch's current stream, which is the handle's stream);
    one untimed warm-up call; `reset` (state reload) and the L2 flush sit outside the events"""
    import torch

    reset()
    fn()
    barrier()
    ms = []
    for _ in range(reps):
        reset()
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        barrier()
        ms.append(e0.elapsed_time(e1))
    return float(np.mean(ms)), out


CONFIG4_TRAJS = ["mandala0_mono", "mandala0_gt", "trans_x", "trans_y", "trans_z", "rot_x", "rot_y", "rot_z", "from_prop"]
CONFIG4_SEEDS, CONFIG4_IFV, CONFIG4_FRAMES = 1024, 33, 200


def secondary_plan(rank, world, filters_per_gpu):
    """Who runs what in the secondary workloads: the launch geometry of every rank (filters, first GLOBAL filter id, stacked
    trajectories), a pure function so that tests/test_multi_gpu.py can hold it against the argument checks of eskf_run for
    every world size without a GPU (a plan that is valid on rank 0 only would leave the other ranks of a torchrun job
    waiting in the all-reduce)."""
    from dvi_ekf_b200.sharding import shard_of

    f3, n3 = shard_of(16 ** 4, rank, world)
    f5, n5 = shard_of(1 << 20, rank, world)
    seeds = CONFIG4_SEEDS // world
    return {
        "config3": dict(n=n3, filter_id0=f3, n_traj=1, filters_per_traj=n3, total=16 ** 4),
        # all nine trajectories x this rank's share of the seeds; LOCAL ids (the stacked streams are indexed by the global id:
        # trajectory = id // filters_per_traj), independent noise per rank through the Philox key
        "config4": dict(n=len(CONFIG4_TRAJS) * seeds, filter_id0=0, n_traj=len(CONFIG4_TRAJS), filters_per_traj=seeds,
                        seed_offset=rank, total=len(CONFIG4_TRAJS) * seeds * world),
        "config5": dict(n=n5, filter_id0=f5, n_traj=1, filters_per_traj=n5, total=1 << 20),
        "calibration": dict(n=filters_per_gpu, filter_id0=rank * filters_per_gpu, n_traj=1, filters_per_traj=filters_per_gpu,
                            total=filters_per_gpu * world),
    }


def secondary_workloads(a, wl, dev, local, rank, world, dist, flush, barrier):
    """BASELINE.json configs 3, 4, 5 and the calibration (all DOFs estimated) variant of config 2, timed in the same run
    as the headline, with the same clock sampler running.  Every rank works on its shard; the figures are max-over-ranks
    device times.  Returns {name: {...}} on every rank (identical after the MAX all-reduce of the times)."""
    import torch

    from dvi_ekf_b200 import BatchFilter
    from dvi_ekf_b200.prepass import build_streams_gpu
    from dvi_ekf_b200.sharding import allreduce_stats, shard_of, summarise_stats

    sc = wl.s
    T, E = len(sc.dt), len(sc.n_prop)
    t64 = lambda x, dtype=torch.float64: torch.tensor(np.ascontiguousarray(x), dtype=dtype, device=dev)
    d = dict(dt=t64(sc.dt), oa=t64(sc.om_acc), npr=t64(sc.n_prop, torch.int32), cam=t64(sc.cam), notch=t64(sc.notch),
             cam_ref=t64(sc.cam_ref), imu_ref=t64(sc.imu_ref))
    P0, u0 = t64(wl.P0[None]), t64(sc.u0[None])
    out = {}

    def record(name, ms, n_total, steps_per_filter, ifv, scaling, what, stats=None, reps=0):
        if dist is not None:
            tt = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = float(tt[0])
        fs = float(n_total) * steps_per_filter
        out[name] = {"workload": what, "filters_total": int(n_total), "filter_steps_per_pass": fs, "ms_per_pass": ms,
                     "value": fs / (ms * 1e-3), "unit": UNIT, "scaling": scaling, "timed_passes": reps,
                     "flops_per_filter_step": 9031 + 29587 / ifv}
        if stats is not None:
            out[name]["stats"] = stats

    # ---- config 3: 16^4 tuning grid, per-filter Q / R, noise-free streams (Simulator.py:163-245, config.yaml:76-82) ----
    plan = secondary_plan(rank, world, a.filters)
    g = 16
    n3 = g ** 4
    first, cnt = plan["config3"]["filter_id0"], plan["config3"]["n"]
    ga, gb, gc, gd = np.meshgrid(np.logspace(-2, 2, g), np.logspace(-2, 2, g), np.logspace(-3, 3, g), np.logspace(-3, 3, g),
                                 indexing="ij")
    sl = slice(first, first + cnt)
    ga, gb, gc, gd = ga.ravel()[sl], gb.ravel()[sl], gc.ravel()[sl], gd.ravel()[sl]
    Qd = np.repeat(wl.Qd[None], cnt, 0)
    Qd[:, 6:9] *= gb[:, None] ** 2
    Qd[:, 9:12] *= ga[:, None] ** 2
    Rd = np.repeat(wl.Rd[None], cnt, 0)
    Rd[:, 0:3] *= gc[:, None] ** 2
    Rd[:, 3:6] *= gd[:, None] ** 2
    x0 = t64(sc.x0[None])
    with BatchFilter(cnt, device=local, **wl.model) as bf:
        bf.set_noise(Qd, Rd, wl.sig_om[None])

        def run3():
            sm = _guard(lambda: bf.run(d["dt"], d["oa"], d["npr"], d["cam"], d["notch"], cam_ref=d["cam_ref"],
                                       imu_ref=d["imu_ref"], stats_on_device=True, filter_id0=first)[1], dev)
            allreduce_stats(sm)
            return sm

        ms, sm = _timed(run3, lambda: bf.set_state(x0, P0, u0, None), 3, barrier, flush)
    record("config3", ms, n3, T, IFV, "strong", f"{n3}-filter tuning grid (16^4 over DOF random walks and camera measurement "
           f"noise, per-filter Q / R), noise-free streams, mandala0_mono {N_FRAMES} frames x {IFV}; sharded over {world} GPU(s), "
           "all-reduce of the statistics inside", summarise_stats(sm.cpu().numpy()), 3)

    # ---- config 4: nine data/trajs trajectories x 1024 seeds, 33 IMU samples per frame, 200 frames, device pre-pass ----
    from dvi_ekf_b200.camera import load_trajectory

    names = CONFIG4_TRAJS
    base, ifv4, frames, seeds_total = 50, CONFIG4_IFV, CONFIG4_FRAMES, CONFIG4_SEEDS
    # every rank: all nine trajectories x its share of the seeds.  (The stacked-trajectory streams are indexed by the GLOBAL
    # filter id -- trajectory = id / filters_per_traj -- so a rank keeps local ids 0 .. 9 * seeds and draws its own noise
    # realisations from a rank-specific Philox key instead of an id offset.)
    seeds = plan["config4"]["filters_per_traj"]
    idx = np.resize(np.concatenate((np.arange(base), np.arange(base - 2, 0, -1))), frames)  # there and back again
    tt = np.arange(frames) / 30.0
    ds = []
    for nm in names:
        t_, xyz, q = load_trajectory(nm, max_vals=base)
        ds.append(build_streams_gpu(tt, xyz[idx].copy(), q[idx].copy(), ifv4, wl.cfg.model.length, wl.cfg.model.angle,
                                    scale=wl.cfg.camera.scale, device=local))
    T4, E4 = ds[0].n_steps, frames - 1
    cat = lambda f: torch.cat([f(x) for x in ds]).contiguous()
    w = dict(dt=cat(lambda x: x.dt[:T4]), oa=cat(lambda x: x.om_acc[:T4]), npr=cat(lambda x: x.n_prop), cam=cat(lambda x: x.cam),
             notch=cat(lambda x: x.notch), cam_ref=cat(lambda x: x.cam_ref), imu_ref=cat(lambda x: x.imu_ref),
             x0=torch.cat([x.x0[None].repeat(seeds, 1) for x in ds]).contiguous(),
             u0=torch.cat([x.u0[None].repeat(seeds, 1) for x in ds]).contiguous())
    n4 = plan["config4"]["n"]
    with BatchFilter(n4, device=local, **wl.model) as bf:
        bf.set_noise(wl.Qd[None], wl.Rd[None], wl.sig_om[None])

        def run4():
            sm = _guard(lambda: bf.run(w["dt"], w["oa"], w["npr"], w["cam"], w["notch"], cam_ref=w["cam_ref"],
                                       imu_ref=w["imu_ref"], n_traj=len(names), filters_per_traj=seeds, stats_on_device=True,
                                       seed=SEED + plan["config4"]["seed_offset"], filter_id0=plan["config4"]["filter_id0"],
                                       imu_noise_std=wl.imu_std, cam_noise_std=wl.cam_std)[1], dev)
            allreduce_stats(sm)
            return sm

        ms, sm = _timed(run4, lambda: bf.set_state(w["x0"], P0, w["u0"], None), 3, barrier, flush)
    record("config4", ms, n4 * world, T4, ifv4, "strong", f"{len(names)} data/trajs trajectories x {seeds_total} noise seeds, "
           f"30 Hz camera / {ifv4} IMU samples per frame, {frames} frames ({T4} propagates + {E4} updates per filter), streams "
           f"from the device pre-pass; seeds sharded over {world} GPU(s)", summarise_stats(sm.cpu().numpy()), 3)
    del w, ds

    # ---- config 5: 1,048,576 Monte-Carlo filters, sharded; NCCL all-reduce of the calibration statistics inside ----
    n5 = plan["config5"]["total"]
    first, cnt = plan["config5"]["filter_id0"], plan["config5"]["n"]
    gen = torch.Generator(device=dev).manual_seed(7 + rank)
    x5 = t64(sc.x0).repeat(cnt, 1)
    x5[:, 10:13] += torch.randn((cnt, 3), generator=gen, dtype=torch.float64, device=dev) * np.deg2rad(3.0)
    x5[:, 13:16] += torch.randn((cnt, 3), generator=gen, dtype=torch.float64, device=dev) * 3.0
    with BatchFilter(cnt, device=local, **wl.model) as bf:
        bf.set_noise(wl.Qd[None], wl.Rd[None], wl.sig_om[None])

        def run5():
            sm = _guard(lambda: bf.run(d["dt"], d["oa"], d["npr"], d["cam"], d["notch"], cam_ref=d["cam_ref"],
                                       imu_ref=d["imu_ref"], stats_on_device=True, seed=SEED, filter_id0=first,
                                       imu_noise_std=wl.imu_std, cam_noise_std=wl.cam_std)[1], dev)
            allreduce_stats(sm)
            return sm

        ms, sm = _timed(run5, lambda: bf.set_state(x5, P0, u0, None), 2, barrier, flush)
    record("config5", ms, n5, T, IFV, "strong", f"{n5} Monte-Carlo filters (Philox noise seeds, DOF IC perturbation) on "
           f"mandala0_mono {N_FRAMES} frames x {IFV}, {cnt} filters per GPU on {world} GPU(s), all-reduce of the calibration "
           "statistics inside", summarise_stats(sm.cpu().numpy()), 2)
    del x5
    torch.cuda.empty_cache()

    # ---- calibration: config 2 with all six DOFs ESTIMATED (config.yaml freezes them; HEAD zeroes frozen DOFs, quirk Q7) ----
    nc = a.filters
    model = dict(wl.model, frozen_dofs=(0,) * 6)
    xc = t64(mc_initial_states(sc.x0, nc, rank * nc))
    with BatchFilter(nc, device=local, **model) as bf:
        bf.set_noise(wl.Qd[None], wl.Rd[None], wl.sig_om[None])

        def runc():
            sm = _guard(lambda: bf.run(d["dt"], d["oa"], d["npr"], d["cam"], d["notch"], cam_ref=d["cam_ref"],
                                       imu_ref=d["imu_ref"], stats_on_device=True, seed=SEED, filter_id0=rank * nc,
                                       imu_noise_std=wl.imu_std, cam_noise_std=wl.cam_std,
                                       gt_dofs=tuple(wl.cfg.gt_imu_dofs))[1], dev)
            allreduce_stats(sm)
            return sm

        ms, sm = _timed(runc, lambda: bf.set_state(xc, P0, u0, None), 5, barrier, flush)
    record("calibration", ms, nc * world, T, IFV, "weak", f"config 2 with all six calibration DOFs estimated (none frozen): {nc} "
           f"filters per GPU, per-filter DOF initial-condition perturbation N(0, 3 deg) / N(0, 3 cm), Philox noise; dof_rmse is the "
           "calibration RMSE against the ground-truth DOFs", summarise_stats(sm.cpu().numpy()), 5)
    return out


def run_ours(a):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    wl = Workload()
    sc = wl.s
    T, E = len(sc.dt), len(sc.n_prop)

    # CPU baseline first (rank 0, single-GPU runs only; before CUDA is initialised in this process)
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        cores = os.cpu_count() or 1
        fpp, n_ep = 512, E  # bounded sample: 512 filters per core over the whole trajectory (10-30 s of CPU work)
        work, busy, wall = cpu_sample(cores, fpp, n_ep)
        cpu = {"value": work / busy, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{cores} procs x {fpp} filters x {n_ep} epochs of the same trajectory "
                         f"({work} filter-steps in {busy:.1f} s; numpy batch oracle, oracle/batch_oracle.py)"}

    import torch

    from dvi_ekf_b200 import BatchFilter
    from dvi_ekf_b200.engine import fp64_peak_tflops
    from dvi_ekf_b200.sharding import allreduce_stats, summarise_stats

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        from datetime import timedelta

        # (a rank that dies must take the job down within minutes, not after NCCL's default ten)
        dist.init_process_group("nccl", device_id=dev, timeout=timedelta(seconds=240))
    n = a.filters
    first_id = rank * n
    imu_std, cam_std = wl.imu_std, wl.cam_std

    def dt64(x, dtype=torch.float64):
        return torch.tensor(np.ascontiguousarray(x), dtype=dtype, device=dev)

    # references for the update-MSE statistic (Filter.calculate_update_mse, Filter.py:397-418)
    cam_ref, imu_ref = sc.cam_ref, sc.imu_ref
    x0_host = mc_initial_states(sc.x0, n, first_id)
    d = dict(dt=dt64(sc.dt), oa=dt64(sc.om_acc), npr=dt64(sc.n_prop, torch.int32), cam=dt64(sc.cam),
             notch=dt64(sc.notch), cam_ref=dt64(cam_ref), imu_ref=dt64(imu_ref), x0=dt64(x0_host),
             P0=dt64(wl.P0[None]), u0=dt64(sc.u0[None]))
    bf = BatchFilter(n, device=local, **wl.model)
    bf.set_tuning(a.fpc)
    bf.set_noise(wl.Qd[None], wl.Rd[None], wl.sig_om[None])
    run_kw = dict(gt_dofs=(0, 0, 0, 0, 0, 20.0), seed=SEED, filter_id0=first_id, imu_noise_std=imu_std,
                  cam_noise_std=cam_std, noise_free_filter0=True)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # 256 MiB > 126 MB L2

    def one_pass():
        st, sm = bf.run(d["dt"], d["oa"], d["npr"], d["cam"], d["notch"], cam_ref=d["cam_ref"], imu_ref=d["imu_ref"],
                        stats_on_device=True, **run_kw)
        allreduce_stats(sm)  # the only collective of the job (NCCL, 16 doubles); no-op on one GPU
        return st, sm

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def reset():
        bf.set_state(d["x0"], d["P0"], d["u0"], None)
        flush.zero_()  # evict L2 between timed iterations

    for _ in range(max(a.warmup, 3)):
        reset()
        one_pass()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = bf.launch_count
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    launches_timed = 0
    barrier()
    t_wall0 = time.perf_counter()
    for i in range(a.steps):
        reset()
        lb = bf.launch_count
        ev[i][0].record()
        st, sm = one_pass()
        ev[i][1].record()
        launches_timed += bf.launch_count - lb
    barrier()
    t_wall = time.perf_counter() - t_wall0
    ms_steps = [e0.elapsed_time(e1) for e0, e1 in ev]
    ms = float(np.mean(ms_steps))
    # keep the hardware busy for the clock sampler a little longer on very short runs
    clocks = sampler.stop() if rank == 0 else None
    stats_sum = sm.cpu().numpy()
    # read out before the end-to-end passes below overwrite the filters' state
    dumped = last_pass_outputs(bf, st, sm, DUMP_BYTES // world) if a.dump_outputs else None

    # ---- end-to-end through the C ABI with HOST buffers (pinned), copies inside the timed region ----
    def pinned(x, dtype=np.float64):
        t = torch.from_numpy(np.ascontiguousarray(x, dtype=dtype)).pin_memory()
        return t.numpy(), t

    keep = []
    hp = {}
    for k, v in dict(dt=sc.dt, oa=sc.om_acc, cam=sc.cam, notch=sc.notch, cam_ref=cam_ref, imu_ref=imu_ref,
                     x0=x0_host, P0=wl.P0[None], u0=sc.u0[None]).items():
        hp[k], t = pinned(v)
        keep.append(t)
    hp["npr"], t = pinned(sc.n_prop, np.int32)
    keep.append(t)
    h2d = sum(hp[k].nbytes for k in ("dt", "oa", "npr", "cam", "notch", "cam_ref", "imu_ref", "x0", "P0", "u0"))
    d2h = n * 16 * 8 + 16 * 8

    st_pin = torch.empty((n, 16), dtype=torch.float64).pin_memory()
    sm_pin = torch.empty((16,), dtype=torch.float64).pin_memory()
    x_pin = torch.empty((n, 26), dtype=torch.float64).pin_memory()
    P_pin = torch.empty((n, 24, 24), dtype=torch.float64).pin_memory()

    def e2e_pass(full_readback=False):
        bf.set_state(hp["x0"], hp["P0"], hp["u0"], None)
        if dist is None:
            st_h, sm_h = bf.run(hp["dt"], hp["oa"], hp["npr"], hp["cam"], hp["notch"], cam_ref=hp["cam_ref"],
                                imu_ref=hp["imu_ref"], **run_kw)
        else:
            # host streams in, statistics left on the device: the reduced vector is all-reduced where it is and crosses
            # the bus once (round 1 copied it down, up and down again)
            st_d, sm_d = bf.run(hp["dt"], hp["oa"], hp["npr"], hp["cam"], hp["notch"], cam_ref=hp["cam_ref"],
                                imu_ref=hp["imu_ref"], stats_on_device=True, **run_kw)
            dist.all_reduce(sm_d)
            st_pin.copy_(st_d, non_blocking=True)
            sm_pin.copy_(sm_d, non_blocking=True)
            torch.cuda.synchronize()
            st_h, sm_h = st_pin.numpy(), sm_pin.numpy()
        if full_readback:  # a caller that wants Filter._states / Filter._P of every filter, not only the error statistics
            xd, Pd, _, _, _ = bf.get_state(device=True)
            x_pin.copy_(xd, non_blocking=True)
            P_pin.copy_(Pd, non_blocking=True)
            torch.cuda.synchronize()
        return st_h, sm_h

    def e2e_time(full_readback):
        for _ in range(2):
            e2e_pass(full_readback)
        barrier()
        ts = []
        for _ in range(a.steps):
            flush.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e2e_pass(full_readback)  # returns after the D2H read of the statistics (and of x, P with full_readback)
            ts.append(1e3 * (time.perf_counter() - t0))
        barrier()
        return float(np.mean(ts))

    e2e_t = e2e_time(False)
    e2e_full_t = e2e_time(True)
    d2h_full = d2h + n * (26 + 576) * 8

    # ---- BASELINE configs 3 / 4 / 5 and the calibration variant, same run, same clock sampler ----
    secondary = None
    if not a.no_configs:
        sampler2 = ClockSampler(local)
        if rank == 0:
            sampler2.start()
        try:
            secondary = secondary_workloads(a, wl, dev, local, rank, world, dist, flush, barrier)
        except Exception as e:  # the headline line must not depend on the secondary workloads
            secondary = {"error": f"{type(e).__name__}: {e}"}
        clocks2 = sampler2.stop() if rank == 0 else None

    # max over ranks
    if dist is not None:
        tt = torch.tensor([ms, e2e_t, e2e_full_t], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms, e2e_t, e2e_full_t = float(tt[0]), float(tt[1]), float(tt[2])
    total_steps = float(n) * T * world
    value = total_steps / (ms * 1e-3)
    e2e_val = total_steps / (e2e_t * 1e-3)

    if rank == 0:
        peak_tf = fp64_peak_tflops(local)
        peaks, which = measured_peaks()
        per_launch_flops = float(n) * T * F_MIN_PER_STEP
        ach = per_launch_flops / (ms * 1e-3) * 1e-12
        # state in / out + statistics row per filter, the shared streams, and the per-filter Monte-Carlo streams the pre-pass
        # leaves in HBM for the persistent kernel (48 B per filter-step, 64 B per filter-update read, 112 B snapshot written)
        alg_bytes = (float(n) * (2 * (576 + 26 + 6 + 9) * 8 + 16 * 8) + (T * 7 + E * 21) * 8
                     + float(n) * (T * 48 + E * (64 + 112)))
        tr = ncu_traffic()
        roofline = {
            "bound": "fp64",
            "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
            "peak_source": "eskf_fp64_peak(): pure-DFMA kernel timed in this run (MEASURED_PEAKS.json has no FP64 figure; "
                           "nominal 37 TFLOP/s at 1965 MHz)",
            "flops_per_filter_step": F_MIN_PER_STEP,
            "dense_equiv": {"achieved": float(n) * T * F_DENSE_PER_STEP / (ms * 1e-3) * 1e-12,
                            "flops_per_filter_step": F_DENSE_PER_STEP},
            "hbm": {"algorithmic_bytes_per_launch": alg_bytes, "achieved_gbs": alg_bytes / (ms * 1e-3) * 1e-9,
                    "peak_gbs": peaks.get("hbm_gbs"), "peak_source": which + " (MEASURED_PEAKS.json)"},
            "traffic": (tr or {}).get("dram_bytes_per_launch"),
            "kernel": "eskf::eskf_kernel3<F> (one launch per pass)",
        }
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": workload_config(n, T, E, world, a.fpc),
            "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": e2e_t,
                    "result": "per-filter error statistics [N,16] + the reduced vector (the result of a Monte-Carlo job: "
                              "calibration RMSE, update MSE); the final x, P stay on the device -- see e2e_full_readback"},
            "e2e_full_readback": {"value": total_steps / (e2e_full_t * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                                  "d2h_bytes_per_step": int(d2h_full), "ms_per_step": e2e_full_t,
                                  "result": "statistics + final state x [N,26] and covariance P [N,24,24] of every filter"},
            "gpu_launches": int(launches_timed),
            "roofline": roofline,
            "cpu_baseline": cpu,
            "wall_s_timed_loop": t_wall,
            "stats": summarise_stats(stats_sum),
        }
        if secondary is not None:
            for v in secondary.values():
                if isinstance(v, dict):
                    v["achieved_tflops"] = v["value"] * v["flops_per_filter_step"] * 1e-12
                    v["frac"] = v["achieved_tflops"] / (peak_tf * world)  # of the FP64 peak of ALL GPUs of the job
            line["configs"] = secondary
            line["configs_clocks"] = clocks2
        print(json.dumps(line), flush=True)
    if dumped is not None:
        os.makedirs(a.dump_outputs, exist_ok=True)
        suffix = f"_rank{rank}" if world > 1 else ""
        for k, v in dumped.items():
            np.save(os.path.join(a.dump_outputs, f"{k}{suffix}.npy"), v)
    bf.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--filters", type=int, default=4096, help="filters per GPU (BASELINE config 2: 4096)")
    ap.add_argument("--fpc", type=int, default=0, help="filters per CTA (0 = automatic)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the secondary workloads (BASELINE configs 3 / 4 / 5, calibration)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed pass as DIR/<name>.npy (float64; "
                    "a seeded sample of the filters above 64 MiB in all); with N > 1 every rank writes <name>_rank<r>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if a.impl == "reference":
        return run_reference_arm(a)
    return run_ours(a)


if __name__ == "__main__":
    sys.exit(main())
