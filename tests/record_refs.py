"""Plain restatements of the two examples' record interpolations, one variable of one point at a time, and a
generator of adversarial record grids.  Shared by test_host_logic.py and test_record_interpolation.py.

example1 (JsonSource.cpp:49-176) is forcing_mode 1 and expansion rule 1; example2 (AsciiSource.cpp:223-345)
is forcing_mode 2 and expansion rule 2.  Both loops are written from the reference's structure, not from the
library's code, and neither calls the oracle."""
import math

import numpy as np

RECORD_VARS = ("tair", "tdew", "VZ", "Rhz", "prec", "SW", "LW", "SW_dir", "LW_net", "TSurfObs", "PrecPhase")
V = {name: v for v, name in enumerate(RECORD_VARS)}
PHASE, LWNET, RHZ, PREC = V["PrecPhase"], V["LW_net"], V["Rhz"], V["prec"]


def interpolate_like_json_source(raw, rawtime, simtime, miss=-100.0, phase=False):
    """Literal restatement of examples/example1/src/JsonSource.cpp:49-176 for one variable.  A value is valid
    when it is > miss (NaN is not).  The precipitation phase (phase=True) takes the record itself at a record
    time and the NEXT record in between; it is left at -9999 (an int there) where the loop assigns nothing."""
    out = np.full(len(simtime), -9999.0 if phase else -9999.9)
    raw_pos = sim_pos = 0
    if rawtime[0] < simtime[0]:
        raw_pos = 0
        while raw_pos < len(rawtime) and not rawtime[raw_pos] >= simtime[0]:
            raw_pos += 1
        raw_pos -= 1
    elif simtime[0] < rawtime[0]:
        while sim_pos < len(simtime) and not simtime[sim_pos] >= rawtime[0]:
            sim_pos += 1
    while raw_pos + 1 < len(rawtime) and sim_pos < len(simtime):
        if abs(simtime[sim_pos] - rawtime[raw_pos]) < 0.01:
            if raw[raw_pos] > miss:
                out[sim_pos] = raw[raw_pos]
            sim_pos += 1
        elif abs(simtime[sim_pos] - rawtime[raw_pos + 1]) < 0.01:
            raw_pos += 1
        elif phase:
            if raw[raw_pos + 1] > miss:
                out[sim_pos] = raw[raw_pos + 1]
            sim_pos += 1
        else:
            if raw[raw_pos] > miss and raw[raw_pos + 1] > miss:
                out[sim_pos] = raw[raw_pos] + (simtime[sim_pos] - rawtime[raw_pos]) * (
                    raw[raw_pos + 1] - raw[raw_pos]) / (rawtime[raw_pos + 1] - rawtime[raw_pos])
            sim_pos += 1
    return out


def _std_min(a, b):
    return b if b < a else a


def _std_max(a, b):
    return b if a < b else a


def interpolate_like_ascii_source(raw, record_step, dt, sim_len, kind=0, fill=-9999.9):
    """examples/example2/src/AsciiSource.cpp:223-345 for one variable of one point: AsciiSource::Impl::interpolate
    (:223-281) called by the per-time loop of GetWeather (:292-345).  Record k lies at model step record_step[k]
    (time = step * dt seconds).  A value is missing when NaN or < -9000 (read_file leaves NaN for -9999).
    NFmiMetTime::DifferenceInMinutes is taken as whole minutes, truncated; for a dt that does not divide 60 this
    truncation is an assumption shared with the library and the oracle, not verified against the reference.
    kind 0 plain, 1 relative humidity (std::max(0.0, std::min(100.0, v)), :322-323), 2 precipitation (> 100
    dropped, :326-327), 3 precipitation phase (stored into an int: truncation toward zero, :345)."""
    def missing(x):
        return math.isnan(x) or x < -9000.0

    def minutes(steps):
        return int(steps * dt) // 60

    rs = [int(s) for s in record_step]
    raw = [float(x) for x in raw]
    n = len(rs)
    out = np.full(sim_len, fill)
    for t in range(sim_len):
        if n < 1 or t < rs[0] or t > rs[n - 1]:          # :307-308 outside the data's time interval
            continue
        pos = 0                                          # :313-316 first position where time >= t
        while pos < n and rs[pos] < t:
            pos += 1
        value = math.nan
        if rs[pos] == t and not missing(raw[pos]):       # :228-233 an exact valid hit
            value = raw[pos]
        elif pos != 0:                                   # :235-236 nothing before the first record
            value2 = math.nan                            # :240-250 first valid value at or after
            pos2 = pos
            while pos2 < n:
                value2 = raw[pos2]
                if not missing(value2):
                    break
                pos2 += 1
            if not missing(value2):
                pos1 = pos - 1                           # :254-264 first valid value before (stops at 0)
                while True:
                    value1 = raw[pos1]
                    if pos1 == 0 or not missing(value1):
                        break
                    pos1 -= 1
                if not missing(value1):                  # :268-279 whole-minute weights, at most 180 minutes
                    gap = minutes(rs[pos2] - rs[pos1])
                    if 0 < gap <= 180:
                        gap1 = minutes(t - rs[pos1])
                        value = (float(gap - gap1) * value1 + float(gap1) * value2) / float(gap)
        if kind == 1 and not missing(value):
            value = _std_max(0.0, _std_min(100.0, value))
        if kind == 2 and value > 100:
            value = math.nan
        if not missing(value):
            out[t] = float(int(value)) if kind == 3 else value
    return out


def json_source_fields(rec, record_step, sim_len, dt):
    """rec [n_records, 11, npoints] -> example1's per-step forcing [sim_len, 11, npoints]."""
    rawtime = [int(s) * int(dt) for s in record_step]
    simtime = [i * int(dt) for i in range(sim_len)]
    out = np.empty((sim_len, rec.shape[1], rec.shape[2]))
    for v in range(rec.shape[1]):
        miss = -1000.0 if v == LWNET else -100.0
        for p in range(rec.shape[2]):
            out[:, v, p] = interpolate_like_json_source(rec[:, v, p], rawtime, simtime, miss, phase=(v == PHASE))
    return out


def ascii_source_fields(rec, record_step, sim_len, dt):
    """rec [n_records, 11, npoints] -> example2's per-step forcing [sim_len, 11, npoints]."""
    kinds = {RHZ: 1, PREC: 2, PHASE: 3}
    out = np.empty((sim_len, rec.shape[1], rec.shape[2]))
    for v in range(rec.shape[1]):
        fill = -9999.0 if v == PHASE else -9999.9
        for p in range(rec.shape[2]):
            out[:, v, p] = interpolate_like_ascii_source(rec[:, v, p], record_step, dt, sim_len, kinds.get(v, 0), fill)
    return out


# ---- adversarial record grids -------------------------------------------------------------------------

DTS = (20.0, 30.0, 45.0, 60.0, 90.0, 120.0)


def steps_for_minutes(minutes, dt):
    """The fewest model steps whose whole-minute length is `minutes` or more."""
    return int(math.ceil(minutes * 60.0 / dt))


def record_grids(dt, sim_len, seed=0):
    """dict name -> record_step (int32) for a run of sim_len steps at time step dt: spacings of one step, irregular
    spacings and hour-plus gaps (180 minutes exactly and the next reachable length above), first records at step 0,
    before it and after it, last records at sim_len - 1, at sim_len and far beyond, and a two-record grid."""
    rng = np.random.default_rng(seed)
    hour, g180, g181 = steps_for_minutes(60, dt), steps_for_minutes(180, dt), steps_for_minutes(181, dt)
    assert g181 * dt // 60 > 180 >= g180 * dt // 60 >= 180

    def walk(first, spacings, last):
        rs = [first]
        for s in spacings:
            if rs[-1] + s >= last:
                break
            rs.append(rs[-1] + s)
        rs.append(last)
        return np.array(rs, dtype=np.int32)

    mixed = [1, 1, 2, g180, 1, g181, 3, 5, hour, 7, 1, hour + 1]
    irregular = [int(x) for x in rng.integers(1, 2 * hour, size=64)]
    return {
        "hourly_from_0": walk(0, [hour] * 64, sim_len + hour),
        "mixed_from_0_to_last_step": walk(0, mixed + irregular, sim_len - 1),
        "mixed_from_negative_to_sim_len": walk(-3, [2] + mixed + irregular, sim_len),
        "irregular_from_negative_far_beyond": walk(-hour - 1, [hour + 1, 1] + irregular[::-1], sim_len + 100000),
        "one_step_spacing": walk(0, [1] * 40 + [g180] + [1] * 8 + [g181] + [1] * 8, sim_len + 1),
        "two_records": np.array([0, sim_len + 7], dtype=np.int32),
        "two_records_negative_to_last_step": np.array([-5, sim_len - 1], dtype=np.int32),
        "after_step_0": walk(6, [1, hour, g180, 2] + irregular, sim_len + hour),
    }


def _one_ulp_below(x):
    return float(np.nextafter(x, -np.inf))


def _one_ulp_above(x):
    return float(np.nextafter(x, np.inf))


def grid_values(n_records, npoints, seed):
    """Records [n_records, 11, npoints] with the edge values of both rules sprinkled over plausible weather:
    missing as -9999.9 and NaN; -100 (missing for example1) and -1000 for LW_net (missing there; -100 is valid
    for LW_net); -9000 (valid for example2) and one ulp below (missing for both); Rhz at and beyond its clamp
    bounds and -0.0; precipitation of 100 and one ulp above; negative non-integer phases (example2 interpolates
    the phase, then truncates); tiny values and -0.0 for the air and dew point temperatures.  Example1's phase
    records are whole numbers, as in its input."""
    rng = np.random.default_rng(seed)
    r = np.empty((n_records, 11, npoints))
    shape = (n_records, npoints)
    r[:, V["tair"]] = rng.normal(-1.0, 4.0, shape)
    r[:, V["tdew"]] = r[:, V["tair"]] - rng.uniform(0.0, 4.0, shape)
    r[:, V["VZ"]] = rng.uniform(0.0, 12.0, shape)
    r[:, V["Rhz"]] = rng.uniform(40.0, 100.0, shape)
    r[:, V["prec"]] = np.where(rng.random(shape) < 0.3, rng.exponential(1.0, shape), 0.0)
    r[:, V["SW"]] = rng.uniform(0.0, 300.0, shape)
    r[:, V["LW"]] = rng.uniform(200.0, 350.0, shape)
    r[:, V["SW_dir"]] = 0.5 * r[:, V["SW"]]
    r[:, V["LW_net"]] = rng.uniform(-120.0, 20.0, shape)
    r[:, V["TSurfObs"]] = r[:, V["tair"]] - 1.0
    r[:, PHASE] = rng.integers(1, 4, shape)
    edges = {
        "tair": [-9999.9, np.nan, -100.0, _one_ulp_above(-100.0), -9000.0, _one_ulp_below(-9000.0), -0.0, 0.0,
                 1e-300, 3e-300, -1e-300],
        "tdew": [-9999.9, np.nan, -100.0, -0.0, 1e-300, 2.5e-300, -9000.0],
        "VZ": [-9999.9, np.nan, -9000.0, _one_ulp_below(-9000.0)],
        "Rhz": [-0.0, 0.0, 100.0, _one_ulp_above(100.0), 140.0, -5.0, -9999.9, np.nan, -9000.0],
        "prec": [100.0, _one_ulp_above(100.0), 250.0, -9999.9, np.nan],
        "SW": [-9999.9, np.nan, -100.0],
        "LW": [-9999.9, np.nan],
        "SW_dir": [-100.0, -9999.9],
        "LW_net": [-1000.0, _one_ulp_above(-1000.0), -100.0, -9999.9, np.nan, -9000.0],
        "TSurfObs": [-9999.9, np.nan, -100.0],
        "PrecPhase": [-9999.0, np.nan, -100.0],
    }
    for name, vals in edges.items():
        hit = rng.random(shape) < 0.12
        r[:, V[name]][hit] = rng.choice(np.array(vals, dtype=np.float64), size=int(hit.sum()))
    return r


def with_fractional_phases(rec, seed):
    """Example2's phase input: interpolated as a double, so non-integer and negative values are in its domain."""
    rng = np.random.default_rng(seed)
    out = rec.copy()
    ph = out[:, PHASE]
    frac = rng.random(ph.shape) < 0.3
    ph[frac] = rng.choice(np.array([-0.5, -1.5, -0.25, 0.75, 2.5, -2.0]), size=int(frac.sum()))
    return out
