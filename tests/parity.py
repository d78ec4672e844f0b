"""Comparison helpers shared by the parity tests."""
import numpy as np

T_TOL = 1e-3   # K   (BASELINE.json north_star: surface/ground temperatures within 1e-3 K)
S_TOL = 1e-3   # mm  (storage terms within 1e-3 mm water equivalent)
STORAGES = ("SnowOut", "WaterOut", "IceOut", "DepositOut", "Ice2Out")


def bit_mismatch(a, b):
    """Elementwise: True where two float64 arrays differ as bit patterns.  Zeros must carry the same sign;
    any two NaNs are equal (the device and x86 produce different NaN payloads for invalid operations)."""
    a = np.ascontiguousarray(a, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    return (a.view(np.uint64) != b.view(np.uint64)) & ~(np.isnan(a) & np.isnan(b))


def same_bits(a, b):
    """Two float64 arrays of one shape are equal bit for bit (under the NaN rule of bit_mismatch)."""
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and not bit_mismatch(a, b).any()


def compare(out_a, out_b):
    """Per-point comparison of two output dicts name -> [npoints, n].  Returns a dict with the max
    temperature / storage differences over matching points, the mismatch fraction (points with any
    value beyond tolerance: threshold-induced state flips), the index of the worst point and the number of
    values that differ as bit patterns (bit_identical: none does)."""
    dT = np.abs(out_a["TsurfOut"] - out_b["TsurfOut"])
    dS = np.zeros_like(dT)
    for n in STORAGES:
        dS = np.maximum(dS, np.abs(out_a[n] - out_b[n]))
    bad = (dT.max(axis=1) > T_TOL) | (dS.max(axis=1) > S_TOL)
    good = ~bad
    differing = 0
    for n in ("TsurfOut",) + STORAGES:
        differing += int(bit_mismatch(out_a[n], out_b[n]).sum())
    res = {
        "bit_identical": differing == 0,
        "differing_values": differing,
        "npoints": int(dT.shape[0]),
        "mismatch_points": int(bad.sum()),
        "mismatch_fraction": float(bad.mean()),
        "max_dT_all": float(dT.max()),
        "max_dS_all": float(dS.max()),
        "max_dT_matching": float(dT[good].max()) if good.any() else 0.0,
        "max_dS_matching": float(dS[good].max()) if good.any() else 0.0,
        "worst_point": int(np.argmax(dT.max(axis=1) + dS.max(axis=1))),
    }
    if bad.any():
        w = np.where(bad)[0][0]
        d = np.maximum(dT[w] / T_TOL, dS[w] / S_TOL)
        res["first_bad_point"] = int(w)
        res["first_bad_step"] = int(np.argmax(d > 1.0))
    return res
