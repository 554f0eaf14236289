"""Simulated outlier frames and the innovation gate on the CPU: the outlier draw of eskf_rng.cuh (outlier_uniform,
meas_outlier and the kind-4 normals) through a host harness against Random123's known-answer vectors and an independent
numpy Philox -- the uniform's range, the rule's edge cases, the noise-free reference filter, the nesting of masks over p with
offsets that do not depend on p, the high counter bits of large epochs -- and the host side of the Python interface: the
argument checks of ``BatchFilter.run(nis_gate=..., outlier_prob=..., outlier_std=...)``, the config keys and
``consistency.nis_gate_threshold``."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from dvi_ekf_b200.engine import drop_prob_array, mask_from_uniforms, nis_gate_array, outlier_std_array

u32p, f64p = ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(ctypes.c_double)
u64 = ctypes.c_uint64
M32 = 0xFFFFFFFF


@pytest.fixture(scope="module")
def hc(tmp_path_factory):
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostcheck", "outlier_check.cpp")
    lib_path = str(tmp_path_factory.mktemp("hostcheck") / "liboutliercheck.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", lib_path, src], check=True)
    lib = ctypes.CDLL(lib_path)
    lib.hc_philox.argtypes = [u32p, ctypes.c_uint32, ctypes.c_uint32, u32p]
    lib.hc_philox.restype = None
    lib.hc_outlier_uniforms.argtypes = [u64, u64, ctypes.c_int64, u64, ctypes.c_int64, f64p]
    lib.hc_outlier_uniforms.restype = None
    lib.hc_outlier_normals.argtypes = [u64, u64, u64, f64p]
    lib.hc_outlier_normals.restype = None
    lib.hc_unit_open32.argtypes = [ctypes.c_uint32]
    lib.hc_unit_open32.restype = ctypes.c_double
    lib.hc_meas_outlier.argtypes = [ctypes.c_double, u64, u64, u64, ctypes.c_int]
    lib.hc_meas_outlier.restype = ctypes.c_int
    return lib


def np_philox(ctr, k0, k1):
    """Philox4x32-10 (Salmon et al., SC'11) written independently of eskf_rng.cuh, on Python integers"""
    c = [int(v) & M32 for v in ctr]
    k0, k1 = int(k0) & M32, int(k1) & M32
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c[0], 0xCD9E8D57 * c[2]
        c = [((p1 >> 32) ^ c[1] ^ k0) & M32, p1 & M32, ((p0 >> 32) ^ c[3] ^ k1) & M32, p0 & M32]
        k0, k1 = (k0 + 0x9E3779B9) & M32, (k1 + 0xBB67AE85) & M32
    return c


def ctr(e, draw, gid):
    """the counter of kind 4 and `draw` at epoch e and noise id gid"""
    return [e & M32, (4 * 16 + draw + ((e >> 32) << 8)) & M32, gid & M32, (gid >> 32) & M32]


def np_box_muller(a, b):
    """box_muller32 in float32, as the host build evaluates it"""
    u1 = np.float32(a) * np.float32(2.3283064365386963e-10) + np.float32(1.1641532182693481e-10)
    th = np.float32(np.int32(np.uint32(b).astype(np.int32))) * np.float32(1.4629180792671596e-9)
    r = np.sqrt(np.float32(-2.0) * np.log(u1))
    return float(r * np.cos(th)), float(r * np.sin(th))


def _philox(hc, c, k0, k1):
    a = np.array(c, dtype=np.uint32)
    out = np.empty(4, dtype=np.uint32)
    hc.hc_philox(a.ctypes.data_as(u32p), k0, k1, out.ctypes.data_as(u32p))
    return [int(v) for v in out]


def _uniforms(hc, seed, id0, n_ids, e0, n_epochs):
    out = np.empty((n_ids, n_epochs))
    hc.hc_outlier_uniforms(seed, id0, n_ids, e0, n_epochs, out.ctypes.data_as(f64p))
    return out


def _normals(hc, seed, gid, e):
    out = np.empty(8)
    hc.hc_outlier_normals(seed, gid, e, out.ctypes.data_as(f64p))
    return out


def test_philox_known_answer_vectors(hc):
    """Random123's known-answer vectors of Philox4x32-10, through the harness and the numpy Philox alike"""
    kat = (([0, 0, 0, 0], 0, 0, [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]),
           ([M32] * 4, M32, M32, [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]),
           ([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], 0xA4093822, 0x299F31D0,
            [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]))
    for c, k0, k1, want in kat:
        assert _philox(hc, c, k0, k1) == want
        assert np_philox(c, k0, k1) == want


def test_uniform_is_word0_of_draw2(hc):
    """u = unit_open32(word 0) of the Philox block of kind 4, draw 2, drop_uniform's counter layout, keyed by the seed"""
    for seed, gid, e in ((0, 0, 0), (2718, 5, 17), (2 ** 40 + 3, 2 ** 33 + 9, 123456), (7, 1, 2 ** 32 + 5), (1, 2, 2 ** 35 - 1)):
        x = np_philox(ctr(e, 2, gid), seed & M32, seed >> 32)[0]
        assert _uniforms(hc, seed, gid, 1, e, 1)[0, 0] == (x + 0.5) * 2.0 ** -32 == hc.hc_unit_open32(x), (seed, gid, e)


def test_offsets_are_normal8_of_kind4(hc):
    """the offsets z[0..6] are Box-Muller of draws 0 and 1 of kind 4 (normal8); the host harness and numpy agree to float32
    rounding of the host's libm"""
    for seed, gid, e in ((99, 0, 0), (2718, 5, 17), (2 ** 40 + 3, 2 ** 33 + 9, 2 ** 32 + 1)):
        a = np_philox(ctr(e, 0, gid), seed & M32, seed >> 32)
        b = np_philox(ctr(e, 1, gid), seed & M32, seed >> 32)
        want = [*np_box_muller(a[0], a[1]), *np_box_muller(a[2], a[3]), *np_box_muller(b[0], b[1]), *np_box_muller(b[2], b[3])]
        got = _normals(hc, seed, gid, e)
        np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-6)


def test_uniform_range(hc):
    """u lies strictly inside (0, 1) and is x 2^-32 + 2^-33 for an integer x"""
    assert hc.hc_unit_open32(0) == 2.0 ** -33 and hc.hc_unit_open32(M32) == 1.0 - 2.0 ** -33
    u = _uniforms(hc, 99, 0, 200, 0, 500)
    assert (u > 0).all() and (u < 1).all()
    x = (u - 2.0 ** -33) * 2.0 ** 32
    assert np.array_equal(x, np.round(x))
    assert 0.48 < u.mean() < 0.52


def test_rule_edges(hc):
    """p = 0 never corrupts, p = 1 always, u == p does not (strict u < p)"""
    u = _uniforms(hc, 31, 1, 50, 0, 40)
    for i in range(50):
        for k in range(40):
            assert hc.hc_meas_outlier(0.0, 31, 1 + i, k, 0) == 0
            assert hc.hc_meas_outlier(1.0, 31, 1 + i, k, 0) == 1
            assert hc.hc_meas_outlier(u[i, k], 31, 1 + i, k, 0) == 0
            assert hc.hc_meas_outlier(np.nextafter(u[i, k], 2.0), 31, 1 + i, k, 0) == 1
    assert mask_from_uniforms(u, u, np.zeros(50, bool)).sum() == 0


def test_noise_free_reference_filter(hc):
    """with nf0 (noise_free_filter0 and id 0) no outlier at all, even at p = 1"""
    for k in range(500):
        for p in (0.0, 0.3, 1.0):
            assert hc.hc_meas_outlier(p, 5, 0, k, 1) == 0
    assert hc.hc_meas_outlier(1.0, 5, 0, 3, 0) == 1  # (without nf0, id 0 draws like any other)


def test_masks_nest_and_offsets_do_not_depend_on_p(hc):
    """within one noise id, p1 <= p2 corrupts a subset of what p2 corrupts; the offsets are a function of (seed, id, epoch)"""
    ps = [0.0, 0.05, 0.2, 0.2000001, 0.5, 1.0]
    masks = [np.array([[hc.hc_meas_outlier(p, 77, i, k, 0) for k in range(300)] for i in range(20)], bool) for p in ps]
    for a, b in zip(masks, masks[1:]):
        assert not (a & ~b).any()
    assert masks[0].sum() == 0 and masks[-1].all() and 0.1 < masks[2].mean() < 0.3
    z1, z2 = _normals(hc, 77, 3, 12), _normals(hc, 77, 3, 12)
    assert z1.tobytes() == z2.tobytes() and not np.array_equal(z1, _normals(hc, 77, 3, 13))


def test_high_epoch_bits(hc):
    """epochs at or above 2^32 put their high bits into counter word 1"""
    lo = _uniforms(hc, 11, 3, 1, 0, 64)[0]
    hi = _uniforms(hc, 11, 3, 1, 2 ** 32, 64)[0]
    assert not np.array_equal(lo, hi)
    for e in (2 ** 32, 2 ** 32 + 1, 3 * 2 ** 32 + 7, 2 ** 40 + 11):
        assert _uniforms(hc, 11, 3, 1, e, 1)[0, 0] == hc.hc_unit_open32(np_philox(ctr(e, 2, 3), 11, 0)[0]), e


def test_outlier_prob_checks():
    """outlier probabilities are checked and broadcast like the dropout table, with their own name in the message"""
    assert drop_prob_array(0.1, 2, 3, "outlier_prob").shape == (2, 3)
    for bad, match in ((np.nan, "outlier_prob must be finite"), (-0.1, r"\[0, 1\]"), (1.5, r"\[0, 1\]"),
                       (np.zeros((3, 3)), "outlier_prob must be a scalar")):
        with pytest.raises(ValueError, match=match):
            drop_prob_array(bad, 2, 3, "outlier_prob")


@pytest.mark.parametrize("bad", [None, [1.0] * 6, [1.0] * 8, [1.0] * 6 + [np.nan], [1.0] * 6 + [np.inf], [-1.0] + [1.0] * 6,
                                 np.ones((7, 1))])
def test_outlier_std_checks(bad):
    with pytest.raises(ValueError, match="outlier_std"):
        outlier_std_array(bad)


def test_outlier_std_accepts():
    s = outlier_std_array([0, 1, 2, 3, 4, 5, 6])
    assert s.dtype == np.float64 and s.shape == (7,) and s.flags.c_contiguous


def test_nis_gate_checks():
    """a scalar or [N]; >= 0 and not NaN; +inf passes (that filter is never gated)"""
    assert nis_gate_array(3.0, 5).tolist() == [3.0]
    assert nis_gate_array([1, 2, 3, np.inf, 0], 5).tolist() == [1, 2, 3, np.inf, 0]
    assert nis_gate_array(np.inf, 5).tolist() == [np.inf]
    for bad, match in ((np.nan, "NaN"), (-1.0, ">= 0"), ([1.0, np.nan, 1, 1, 1], "NaN"), ([1.0, 2.0], "shape"),
                       (np.ones((5, 1)), "shape"), ([-np.inf] * 5, ">= 0")):
        with pytest.raises(ValueError, match=match):
            nis_gate_array(bad, 5)


def test_nis_gate_threshold_matches_scipy():
    from scipy.stats import chi2

    from dvi_ekf_b200.consistency import nis_gate_threshold

    for p in (0.9, 0.99, 0.999, 0.99999):
        assert nis_gate_threshold(p) == chi2.ppf(p, 7)
        assert nis_gate_threshold(p, 3) == chi2.ppf(p, 3)
    assert abs(nis_gate_threshold(0.999) - 24.3219) < 1e-3
    assert nis_gate_threshold(1.0) == np.inf
    with pytest.raises(ValueError):
        nis_gate_threshold(1.5)


def test_config_keys(tmp_path):
    """batch.nis_gate (absent / null = off), batch.cam_outlier_prob (default 0) and batch.cam_outlier_std (7 values, required
    with p > 0)"""
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

    b = load(None).batch
    assert b.nis_gate is None and b.cam_outlier_prob == 0.0 and b.cam_outlier_std is None
    b = load({"nis_gate": None, "cam_outlier_prob": 0.1, "cam_outlier_std": [1, 1, 1, 0.1, 0.1, 0.1, 0.2]}).batch
    assert b.nis_gate is None and b.cam_outlier_prob == 0.1 and b.cam_outlier_std == [1, 1, 1, 0.1, 0.1, 0.1, 0.2]
    assert load({"nis_gate": 24.3}).batch.nis_gate == 24.3
    assert load({"nis_gate": float("inf")}).batch.nis_gate == float("inf")
    for bad, match in (({"nis_gate": -1.0}, "nis_gate"), ({"nis_gate": float("nan")}, "nis_gate"),
                       ({"cam_outlier_prob": 1.5}, "cam_outlier_prob"), ({"cam_outlier_prob": float("nan")}, "cam_outlier_prob"),
                       ({"cam_outlier_prob": 0.1}, "cam_outlier_std"), ({"cam_outlier_std": [1.0] * 6}, "cam_outlier_std"),
                       ({"cam_outlier_std": [1.0] * 6 + [-1.0]}, "cam_outlier_std"),
                       ({"cam_outlier_std": [1.0] * 6 + [float("nan")]}, "cam_outlier_std")):
        with pytest.raises(ValueError, match=match):
            load(bad)
