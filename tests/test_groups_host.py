"""Filter groups on the CPU: the block map of the grouped reductions (eskf_math.cuh group_blocks / group_block /
group_row0) through a host harness, exhaustively; ``sharding.place_group_rows`` with shards that split a group, added through
gloo at world size 2; and the argument checks of ``BatchFilter.set_groups`` / ``get_group_sums``."""
import ctypes
import os
import socket
import subprocess

import numpy as np
import pytest

from dvi_ekf_b200.sharding import place_group_rows

i64p = ctypes.POINTER(ctypes.c_int64)


@pytest.fixture(scope="module")
def hc(tmp_path_factory):
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostcheck", "group_check.cpp")
    lib_path = str(tmp_path_factory.mktemp("hostcheck") / "libgroupcheck.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", lib_path, src], check=True)
    lib = ctypes.CDLL(lib_path)
    lib.hc_group_map.argtypes = [ctypes.c_int64] * 4 + [i64p, ctypes.c_int64]
    lib.hc_group_map.restype = ctypes.c_int64
    lib.hc_group_first_blocks.argtypes = [ctypes.c_int64] * 5 + [i64p]
    lib.hc_group_first_blocks.restype = None
    return lib


def _check(hc, N, id0, g, rpb):
    cap = N + N // max(1, min(rpb, N)) + 2 * (N // max(g, 1)) + 4
    buf = np.empty((cap, 3), dtype=np.int64)
    nblk = hc.hc_group_map(N, id0, g, rpb, buf.ctypes.data_as(i64p), cap)
    where = f"N={N} id0={id0} g={g} rpb={rpb}"
    assert nblk > 0, where
    r0, r1, k = buf[:nblk].T
    assert ((r1 - r0 >= 1) & (r1 - r0 <= rpb)).all(), (where, "empty or oversized block")
    # every row exactly once, blocks in row order (so a group's blocks come in row order and groups follow each other)
    assert r0[0] == 0 and r1[-1] == N and np.array_equal(r0[1:], r1[:-1]), where
    # no block straddles a group; the local group is the global group of the block's rows minus the first one's
    if g > 0:
        assert np.array_equal((id0 + r0) // g, (id0 + r1 - 1) // g), (where, "block straddles a group")
        assert np.array_equal(k, (id0 + r0) // g - id0 // g), where
        G = (id0 + N - 1) // g - id0 // g + 1
        # each group's blocks start at the group's first row
        starts = np.r_[True, k[1:] != k[:-1]]
        assert np.array_equal(r0[starts] + id0, np.maximum(np.arange(G) + id0 // g, 0) * g + np.r_[id0 % g, np.zeros(G - 1, int)]), where
    else:
        assert (k == 0).all()
        G = 1
    assert np.array_equal(np.unique(k), np.arange(G)), where
    first = np.empty(G + 1, dtype=np.int64)
    hc.hc_group_first_blocks(N, id0, g, rpb, G, first.ctypes.data_as(i64p))
    assert first[0] == 0 and first[-1] == nblk, where
    for j in range(G):
        assert (k[first[j]:first[j + 1]] == j).all(), (where, "group_row0 does not give the group's blocks")
    return nblk, buf[:nblk]


def _today(N, rpb):
    """the blocks of the ungrouped reduction: ceil(N / rpb) blocks of rows b rpb .. min(N, (b + 1) rpb) - 1"""
    b = np.arange(-(-N // rpb))
    return np.stack([b * rpb, np.minimum(N, (b + 1) * rpb), 0 * b], axis=1)


def test_block_map_exhaustively(hc):
    count = 0
    for N in range(1, 201):
        for rpb in (*range(1, 10), 4096):
            for g in (0, *range(1, 41), N + 1, 2 * N + 3):
                ids = {0} if g == 0 else {0, g, 2 * g, g - 1, 3 * g - 1, 1, g // 2, 5 * g + g // 3}
                for id0 in sorted(i for i in ids if i >= 0):
                    nblk, blocks = _check(hc, N, id0, g, rpb)
                    if g == 0 or (id0 % g == 0 and g >= N):  # one group: the layout of the ungrouped reduction
                        assert np.array_equal(blocks, _today(N, rpb)), (N, id0, g, rpb)
                    count += 1
    assert count > 100_000


def test_large_counts(hc):
    """a million filters in groups of 8 and of 4096 (trajectories), and shards that start inside a group"""
    for N, id0, g in ((1 << 20, 0, 8), (1 << 20, 3, 8), (9 * 4096, 0, 4096), (5000, 4093, 4096), (4097, 0, 0)):
        nblk, blocks = _check(hc, N, id0, g, 4096)
        G = (id0 + N - 1) // g - id0 // g + 1 if g else 1
        assert nblk == sum(-(-(min(N, (id0 // g + j + 1) * g - id0) - max(0, (id0 // g + j) * g - id0)) // 4096) for j in range(G)) if g else nblk == 2


def test_place_group_rows():
    rows = np.arange(6.0).reshape(3, 2)
    out = place_group_rows(rows, 2, 6)
    assert out.shape == (6, 2) and np.array_equal(out[2:5], rows) and not out[[0, 1, 5]].any()
    for g0, total in ((-1, 6), (4, 6)):
        with pytest.raises(ValueError, match="do not fit"):
            place_group_rows(rows, g0, total)
    torch = pytest.importorskip("torch")
    t = place_group_rows(torch.from_numpy(rows), 1, 4)
    assert torch.is_tensor(t) and np.array_equal(t.numpy()[1:4], rows)


def _grouped(values, id0, g):
    """group rows of per-filter values [n, w] of filters id0 .. id0 + n - 1: (group0, [G, w]), summed in numpy"""
    gid = (id0 + np.arange(len(values))) // g
    g0 = gid[0]
    out = np.zeros((gid[-1] - g0 + 1, values.shape[1]))
    np.add.at(out, gid - g0, values)
    return g0, out


def _worker(rank, world, port, q):
    import torch
    import torch.distributed as dist

    from dvi_ekf_b200.sharding import allreduce_stats, shard_of

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    vals = np.random.default_rng(3).normal(size=(45, 4))
    first, count = shard_of(45, rank, world)  # 23 + 22 filters: the boundary cuts group 3 of groups of 7
    g0, rows = _grouped(vals[first:first + count], first, 7)
    t = torch.from_numpy(place_group_rows(rows, g0, 7))
    allreduce_stats(t)
    q.put((rank, first, g0, len(rows), t.numpy().copy()))
    dist.barrier()
    dist.destroy_process_group()


def test_world_size_2_gloo_adds_a_split_group():
    import torch.multiprocessing as mp

    world = 2
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=240) for _ in range(world)), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert [(r[1], r[2], r[3]) for r in res] == [(0, 0, 4), (23, 3, 4)]  # group 3 (filters 21..27) is in both shards
    _, whole = _grouped(np.random.default_rng(3).normal(size=(45, 4)), 0, 7)
    for r in res:
        assert np.allclose(r[4], whole, rtol=1e-13, atol=1e-15)


class _StubLib:
    """the two C entry points, recording their arguments: G = 3 groups from group 5, E = 4 epochs"""

    def __init__(self):
        self.calls = []

    def eskf_set_groups(self, h, g):
        self.calls.append(("set", g))
        return 0

    def eskf_get_group_sums(self, h, st, es, ds, g0, G, E, mem):
        self.calls.append(("get", st is not None, es is not None, ds is not None, mem))
        for p, v in ((g0, 5), (G, 3), (E, 4)):
            if p is not None:
                p._obj.value = v
        return 0


def _stub_filter():
    from dvi_ekf_b200.engine import BatchFilter

    bf = BatchFilter.__new__(BatchFilter)
    bf._lib, bf._h, bf.n, bf.device = _StubLib(), None, 10, 0
    return bf


def test_engine_argument_checks():
    bf = _stub_filter()
    for bad, err in ((-1, ValueError), (2.5, TypeError), (True, TypeError)):
        with pytest.raises(err):
            bf.set_groups(bad)
    bf.set_groups(0)
    bf.set_groups(np.int64(13))
    assert bf._lib.calls == [("set", 0), ("set", 13)]
    bf._lib.calls.clear()
    g0, st, es, ds = bf.get_group_sums()
    assert g0 == 5 and st.shape == (3, 16) and es is None and ds is None
    g0, st, es, ds = bf.get_group_sums(stats=False, consistency=True, dof_envelope=True)
    assert st is None and es.shape == (3, 4, 8) and ds.shape == (3, 4, 80)
    # a query without outputs first, then only the arrays asked for, in host memory
    assert bf._lib.calls == [("get", False, False, False, 0), ("get", True, False, False, 0),
                             ("get", False, False, False, 0), ("get", False, True, True, 0)]
