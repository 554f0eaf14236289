"""Simulated frame loss on the CPU: the dropout draw of eskf_rng.cuh (philox4x32_10, unit_open32, drop_uniform, meas_dropped)
through a host harness -- Random123's known-answer vectors, the uniform's range, the rule's edge cases, the noise-free
reference filter, the nesting of masks over p and the high counter bits of large epochs -- and the host side of
``BatchFilter.run(drop_prob=...)``: broadcasting and validation (``engine.drop_prob_array``), the mask rule
(``engine.mask_from_uniforms``) and the ``batch.cam_dropout`` key of the config."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from dvi_ekf_b200.engine import drop_prob_array, mask_from_uniforms

u32p, f64p = ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(ctypes.c_double)
u64 = ctypes.c_uint64


@pytest.fixture(scope="module")
def hc(tmp_path_factory):
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostcheck", "dropout_check.cpp")
    lib_path = str(tmp_path_factory.mktemp("hostcheck") / "libdropoutcheck.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", lib_path, src], check=True)
    lib = ctypes.CDLL(lib_path)
    lib.hc_philox.argtypes = [u32p, ctypes.c_uint32, ctypes.c_uint32, u32p]
    lib.hc_philox.restype = None
    lib.hc_drop_uniforms.argtypes = [u64, u64, ctypes.c_int64, u64, ctypes.c_int64, f64p]
    lib.hc_drop_uniforms.restype = None
    lib.hc_unit_open32.argtypes = [ctypes.c_uint32]
    lib.hc_unit_open32.restype = ctypes.c_double
    lib.hc_meas_dropped.argtypes = [ctypes.c_double, u64, u64, u64, ctypes.c_int]
    lib.hc_meas_dropped.restype = ctypes.c_int
    return lib


def _philox(hc, ctr, k0, k1):
    c = np.array(ctr, dtype=np.uint32)
    out = np.empty(4, dtype=np.uint32)
    hc.hc_philox(c.ctypes.data_as(u32p), k0, k1, out.ctypes.data_as(u32p))
    return [int(v) for v in out]


def _uniforms(hc, seed, id0, n_ids, e0, n_epochs):
    out = np.empty((n_ids, n_epochs))
    hc.hc_drop_uniforms(seed, id0, n_ids, e0, n_epochs, out.ctypes.data_as(f64p))
    return out


def test_philox_known_answer_vectors(hc):
    """Random123's known-answer vectors of Philox4x32-10"""
    assert _philox(hc, [0, 0, 0, 0], 0, 0) == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    assert _philox(hc, [0xFFFFFFFF] * 4, 0xFFFFFFFF, 0xFFFFFFFF) == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]
    assert _philox(hc, [0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], 0xA4093822, 0x299F31D0) == \
        [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]


def test_uniform_range_and_extreme_words(hc):
    """u = (x + 1/2) 2^-32: the extreme words give 2^-33 and 1 - 2^-33, exactly, strictly inside (0, 1)"""
    assert hc.hc_unit_open32(0) == 2.0 ** -33
    assert hc.hc_unit_open32(0xFFFFFFFF) == 1.0 - 2.0 ** -33
    assert hc.hc_unit_open32(0x80000000) == 0.5 + 2.0 ** -33
    u = _uniforms(hc, 99, 0, 200, 0, 500)
    assert (u > 0).all() and (u < 1).all()
    # every u is x 2^-32 + 2^-33 for an integer x: exact in double precision
    x = (u - 2.0 ** -33) * 2.0 ** 32
    assert np.array_equal(x, np.round(x))


def test_uniform_is_word0_of_the_documented_counter(hc):
    """counter (e lo, 3 * 16 + (e hi << 8), id lo, id hi), key (seed lo, seed hi): the layout of normal4 with kind 3, draw 0"""
    for seed, gid, e in ((0, 0, 0), (2718, 5, 17), (2 ** 40 + 3, 2 ** 33 + 9, 123456), (7, 1, 2 ** 32 + 5), (1, 2, 2 ** 35 - 1)):
        ctr = [e & 0xFFFFFFFF, (3 * 16 + ((e >> 32) << 8)) & 0xFFFFFFFF, gid & 0xFFFFFFFF, gid >> 32]
        x = _philox(hc, ctr, seed & 0xFFFFFFFF, seed >> 32)[0]
        assert _uniforms(hc, seed, gid, 1, e, 1)[0, 0] == hc.hc_unit_open32(x), (seed, gid, e)


def test_rule_edges(hc):
    """p = 0 never drops, p = 1 always drops, u == p does not drop (strict u < p)"""
    u = _uniforms(hc, 31, 0, 50, 0, 40)
    for i in range(50):
        for k in range(40):
            assert hc.hc_meas_dropped(0.0, 31, i, k, 0) == 0
            assert hc.hc_meas_dropped(1.0, 31, i, k, 0) == 1
            assert hc.hc_meas_dropped(u[i, k], 31, i, k, 0) == 0  # u < u is false
            assert hc.hc_meas_dropped(np.nextafter(u[i, k], 2.0), 31, i, k, 0) == 1
    assert mask_from_uniforms(u, u, np.zeros(50, bool)).sum() == 0


def test_noise_free_reference_filter(hc):
    """with nf0 (noise_free_filter0 and id 0) only p == 1 drops, whatever u"""
    u = _uniforms(hc, 5, 0, 1, 0, 1000)[0]
    for k in range(1000):
        for p in (0.0, 0.3, 0.999999, np.nextafter(1.0, 0.0)):
            assert hc.hc_meas_dropped(p, 5, 0, k, 1) == 0
        assert hc.hc_meas_dropped(1.0, 5, 0, k, 1) == 1
    assert (u < 0.999999).sum() > 990  # (it would have dropped nearly every one)
    p = np.array([[0.0, 0.5, 1.0, 0.999]])
    m = mask_from_uniforms(np.full((2, 4), 1e-9), np.repeat(p, 2, 0), np.array([True, False]))
    assert m.tolist() == [[False, False, True, False], [False, True, True, True]]


def test_masks_nest_over_p(hc):
    """within one noise id, p1 <= p2 drops a subset of what p2 drops"""
    ps = [0.0, 0.05, 0.1, 0.3, 0.3000001, 0.5, 0.9, 1.0]
    masks = [np.array([[hc.hc_meas_dropped(p, 77, i, k, 0) for k in range(300)] for i in range(20)], bool) for p in ps]
    for a, b in zip(masks, masks[1:]):
        assert not (a & ~b).any()
    assert masks[0].sum() == 0 and masks[-1].all()
    assert 0.2 < masks[3].mean() < 0.4


def test_high_epoch_bits(hc):
    """epochs at or above 2^32 put their high bits into counter word 1: epoch 2^32 + k differs from epoch k, and the
    uniform matches the Philox block of that counter"""
    lo = _uniforms(hc, 11, 3, 1, 0, 64)[0]
    hi = _uniforms(hc, 11, 3, 1, 2 ** 32, 64)[0]
    assert not np.array_equal(lo, hi)
    for e in (2 ** 32, 2 ** 32 + 1, 3 * 2 ** 32 + 7, 2 ** 40 + 11):
        ctr = [e & 0xFFFFFFFF, (3 * 16 + ((e >> 32) << 8)) & 0xFFFFFFFF, 3, 0]
        assert _uniforms(hc, 11, 3, 1, e, 1)[0, 0] == hc.hc_unit_open32(_philox(hc, ctr, 11, 0)[0]), e


def test_drop_prob_broadcasting():
    """a scalar, [E] or [n_traj, E] broadcast to [n_traj, E], C-contiguous float64"""
    a = drop_prob_array(0.25, 3, 5)
    assert a.shape == (3, 5) and a.dtype == np.float64 and a.flags.c_contiguous and (a == 0.25).all()
    row = np.linspace(0, 1, 5)
    b = drop_prob_array(row, 3, 5)
    assert b.shape == (3, 5) and (b == row[None]).all()
    c = np.random.default_rng(0).uniform(size=(3, 5))
    assert np.array_equal(drop_prob_array(c, 3, 5), c)
    assert drop_prob_array([0, 1], 1, 2).tolist() == [[0.0, 1.0]]
    assert drop_prob_array(0.5, 2, 0).shape == (2, 0)


@pytest.mark.parametrize("bad, match", [
    (np.nan, "finite"), ([0.1, np.nan, 0.2], "finite"), (np.inf, "finite"), (-0.01, r"\[0, 1\]"), (1.0000001, r"\[0, 1\]"),
    ([0.5, 0.5], "shape"), (np.zeros((2, 3)), "shape"), (np.zeros((3, 4)), "shape"), (np.zeros((1, 1, 3)), "shape"),
])
def test_drop_prob_validation(bad, match):
    with pytest.raises(ValueError, match=match):
        drop_prob_array(bad, 3, 3)


def test_config_cam_dropout(tmp_path):
    """batch.cam_dropout: absent = 0, a probability, anything else is refused"""
    import yaml

    from dvi_ekf_b200.config import Config

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    base = yaml.safe_load(open(os.path.join(root, "config.yaml")))
    base.pop("batch", None)

    def load(batch):
        d = dict(base)
        if batch is not None:
            d["batch"] = batch
        p = tmp_path / "c.yaml"
        p.write_text(yaml.safe_dump(d))
        return Config(str(p))

    assert load(None).batch.cam_dropout == 0.0
    assert load({"seed": 3}).batch.cam_dropout == 0.0
    assert load({"cam_dropout": 0.2}).batch.cam_dropout == 0.2
    for bad in (-0.1, 1.5, float("nan")):
        with pytest.raises(ValueError, match="cam_dropout"):
            load({"cam_dropout": bad})
