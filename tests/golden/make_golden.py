"""Packs the reference's numeric artefacts for the hot path into two fixtures.

Run with the reference's trajectory directory (dvi-ekf/data/trajs, read-only):

    python tests/golden/make_golden.py <dvi-ekf>/data/trajs

Inputs:
  * camera trajectories (t x y z qx qy qz qw): mandala0_mono.csv and the
    space-separated *.txt files without header;
  * kf_best_mandala0_mono.txt / imu_ref_mandala0_mono.txt -- the only numeric
    pins of Filter.propagate/update (FilterTraj / ImuRefTraj rows written by
    Filter.save, dvi_ekf/filter/Filter.py:457-465);
  * the legacy imu_ref_mandala0_mono_upd_Kp*_Km1.000.txt files, which pin the
    interframe>1 interpolation / IMU-reference pose path;
  * notch90.csv, the notch trajectory config.yaml names (an INPUT of the
    with_notch flow; the reference holds no output for it).
Output: tests/golden/reference_golden.npz (float64 arrays, compressed) and
tests/golden/imu_ref_legacy.npz (the legacy files, read back by
tests.helpers.legacy_imu_ref): their 9-decimal values as int64 in units of
1e-9, differenced along the rows, LZMA-compressed -- a quarter of the size of
the float64 arrays and bit-exact after decoding.  Their velocity columns 4:7
come from an older velocity definition, no test compares them, and they are
not stored.
"""
import io
import os
import sys
import zipfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "reference_golden.npz")
OUT_LEGACY = os.path.join(HERE, "imu_ref_legacy.npz")
LEGACY_COLS = [0, 1, 2, 3, 7, 8, 9, 10, 11, 12, 13]


def encode_legacy(a):
    n = np.round(a[:, LEGACY_COLS] * 1e9).astype(np.int64)
    assert np.array_equal(n / 1e9, a[:, LEGACY_COLS]), "not a 9-decimal file"
    return np.vstack((n[:1], np.diff(n, axis=0)))


def save_npz_lzma(path, arrays):
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_LZMA) as z:
        for k, v in arrays.items():
            b = io.BytesIO()
            np.save(b, v)
            z.writestr(k + ".npy", b.getvalue())


def main():
    if len(sys.argv) != 2 or not os.path.isdir(sys.argv[1]):
        sys.exit("usage: make_golden.py <dvi-ekf>/data/trajs")
    ref = sys.argv[1]
    out = {}
    out["traj_mandala0_mono"] = np.loadtxt(os.path.join(ref, "mandala0_mono.csv"), delimiter=",", skiprows=1)
    for name in ["mandala0_gt", "trans_x", "trans_y", "trans_z", "rot_x", "rot_y", "rot_z", "from_prop"]:
        out[f"traj_{name}"] = np.loadtxt(os.path.join(ref, f"{name}.txt"))
    out["kf_best_mandala0_mono"] = np.loadtxt(os.path.join(ref, "kf_best_mandala0_mono.txt"))
    out["imu_ref_mandala0_mono"] = np.loadtxt(os.path.join(ref, "imu_ref_mandala0_mono.txt"))
    # notch trajectory of config.yaml (notch_traj_name: notch90): "notch,notch_d,notch_dd" per camera frame, comma separated
    out["notch_notch90"] = np.loadtxt(os.path.join(ref, "notch90.csv"), delimiter=",")
    np.savez_compressed(OUT, **out)
    legacy = {}
    for kp in ["0.006", "0.01", "2.0", "1.0"]:
        a = np.loadtxt(os.path.join(ref, f"imu_ref_mandala0_mono_upd_Kp{kp}_Km1.000.txt"))
        legacy[f"Kp{kp}"] = encode_legacy(a)
    save_npz_lzma(OUT_LEGACY, legacy)
    for k, v in {**out, **legacy}.items():
        print(f"{k:34s} {v.shape}")
    for p in (OUT, OUT_LEGACY):
        print("wrote", p, os.path.getsize(p), "bytes")


if __name__ == "__main__":
    main()
