"""Multi-GPU plumbing of the Monte-Carlo batch (SURVEY.md section 8e): filters are independent, so the batch is cut
into contiguous shards, one per rank (one process per GPU); the only exchange is the all-reduce of the
ESKF_NSTAT-entry statistics vector after the trajectory kernel.  Noise and initial-condition perturbations are
keyed by the GLOBAL filter id, so an N-GPU run reproduces the 1-GPU results filter by filter."""
from __future__ import annotations

import numpy as np

NSTAT = 16


def shard_of(n_total: int, rank: int, world: int):
    """(first global filter id, number of filters) of `rank`: contiguous blocks, the remainder spread over the
    first ranks."""
    if not (0 <= rank < world):
        raise ValueError("rank out of range")
    base, rem = divmod(int(n_total), int(world))
    count = base + (1 if rank < rem else 0)
    first = rank * base + min(rank, rem)
    return first, count


def mc_initial_states(x0_row, n: int, first_id: int, seed: int):
    """DOF initial-condition perturbation N(0, 3 deg) / N(0, 3 cm) (the commented intent at
    dvi_ekf/tools/utils.py:28-33), drawn per GLOBAL filter id; global filter 0 keeps the nominal state."""
    x0 = np.repeat(np.asarray(x0_row, dtype=float)[None], n, 0)
    for i in range(n):
        gid = first_id + i
        if gid == 0:
            continue
        rng = np.random.default_rng([seed, gid])
        x0[i, 10:13] += rng.normal(0.0, np.deg2rad(3.0), 3)
        x0[i, 13:16] += rng.normal(0.0, 3.0, 3)
    return x0


def allreduce_stats(stats_sum, group=None):
    """Sum of the per-rank statistics vectors (eskf_run's stats_sum), in place; a torch tensor on the device the
    process group works on (NCCL: the GPU; gloo: the CPU).  No-op without an initialised process group.  It serves any
    per-rank sum the same way: the consistency epoch sums (``get_consistency``) and the per-DOF envelope ``dof_sum``
    (``get_dof_envelope``, for ``consistency.summarise_dofs``) as well, and the per-group sums of ``get_group_sums`` once
    ``place_group_rows`` has put every rank's rows at their global groups."""
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized():
        import torch

        nvtx = stats_sum.is_cuda  # NVTX range on the timeline of a profiler (SURVEY section 5)
        if nvtx:
            torch.cuda.nvtx.range_push("eskf: all-reduce of the error statistics")
        try:
            dist.all_reduce(stats_sum, op=dist.ReduceOp.SUM, group=group)
        finally:
            if nvtx:
                torch.cuda.nvtx.range_pop()
    return stats_sum


def place_group_rows(rows, group0: int, n_groups_total: int):
    """A shard's per-group rows (``BatchFilter.get_group_sums``: row k is global group ``group0 + k``) scattered into a zero
    array of the job's ``n_groups_total`` groups, ``[n_groups_total, ...]``, so that ``allreduce_stats`` adds the ranks'
    arrays.  A group cut by a shard boundary is a partial row in both shards; the addition gives its sums.  numpy in, numpy
    out; a torch tensor gives a tensor on its device."""
    n, g0, total = len(rows), int(group0), int(n_groups_total)
    if g0 < 0 or g0 + n > total:
        raise ValueError(f"rows of groups [{g0}, {g0 + n}) do not fit in {total} groups")
    if type(rows).__module__.startswith("torch"):
        import torch

        out = torch.zeros((total, *rows.shape[1:]), dtype=rows.dtype, device=rows.device)
    else:
        rows = np.asarray(rows)
        out = np.zeros((total, *rows.shape[1:]), dtype=rows.dtype)
    out[g0:g0 + n] = rows
    return out


def summarise_stats(stats_sum):
    """Error statistics of the whole job from the reduced vector (include/eskf.h): sums over the HEALTHY filters (finite
    row, status 0) in [0:10] -- [0:6] (dofs - gt)^2, [6] DOF metric, [7] last update_mse, [8] update_mse summed over the
    epochs, [9] applied updates -- and the counts [10] filters with a non-zero status word, [11] healthy filters (the
    divisor of every mean), [12] filters with non-finite results."""
    s = np.asarray(stats_sum, dtype=float)
    n = s[11]
    d = n if n > 0 else float("nan")
    return {"dof_rmse": [float(np.sqrt(v / d)) for v in s[:6]], "dof_metric_mean": float(s[6] / d),
            "mean_update_mse_last": float(s[7] / d), "filters": float(n), "updates_applied": float(s[9]),
            "filters_flagged": float(s[10]), "filters_nonfinite": float(s[12])}
