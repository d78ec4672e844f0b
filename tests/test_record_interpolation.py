"""Coarse-record interpolation against plain restatements of both examples' rules (tests/record_refs.py), bit for
bit, on adversarial record grids: spacings of one step, irregular spacings, hour-plus gaps, first records before,
at and after step 0, last records at and beyond the end of the run, two-record grids, missing values of every
form and at the exact thresholds, at time steps of 20 to 120 s.

The implementations under test: the step kernel's in-flight interpolation (forcing_mode 1: coarse_refill /
fetch_coarse), rs_expand_records_kernel rules 1 and 2 (roadsurf_expand_records; rule 2 is forcing_mode 2), and the
host derivation roadsurf_read_input_derive_records.  Every comparison is bitwise (parity.same_bits: zeros carry
their sign)."""
import datetime as _dt
import functools

import numpy as np
import pytest

import record_refs as rr
from parity import same_bits
from roadsurf_b200 import abi, lib, synth

NPTS = 12
START = _dt.datetime(2019, 12, 2, 0, 0, 0)
REQUIRED = [rr.V[n] for n in ("tair", "Rhz", "prec", "SW", "LW", "VZ")]   # roadrunner.cpp:167-195


def _sim_len(dt):
    return rr.steps_for_minutes(400, dt) + 1


@functools.lru_cache(maxsize=None)
def _grids(dt):
    return rr.record_grids(dt, _sim_len(dt), seed=int(dt))


@functools.lru_cache(maxsize=None)
def _case(dt, name, nvar=11):
    """(record_step, records [n_records, nvar, NPTS], example1's fields, example2's fields) of one grid; the 12th
    variable (the output-depth plane) gets the surface observations' values."""
    rs = _grids(dt)[name]
    rec = rr.grid_values(len(rs), NPTS, seed=int(dt) * 100 + len(rs))
    if nvar == 12:
        rec = np.concatenate([rec, rec[:, rr.V["TSurfObs"]:rr.V["TSurfObs"] + 1][:, :, ::-1]], axis=1)
    rec2 = rr.with_fractional_phases(rec, seed=len(rs))
    sim_len = _sim_len(dt)
    ex1 = rr.json_source_fields(rec, rs, sim_len, dt) if rs[0] <= 0 else None
    return rs, rec, ex1, rec2, rr.ascii_source_fields(rec2, rs, sim_len, dt)


# ---- the references (CPU) -------------------------------------------------------------------------------

def test_json_source_restatement_by_hand():
    miss = -9999.9
    simtime = [0, 30, 60, 90, 120, 150, 180]
    got = rr.interpolate_like_json_source([1.0, 3.0, 0.0], [0, 60, 150], simtime)
    assert same_bits(got, [1.0, 2.0, 3.0, 2.0, 1.0, miss, miss])        # nothing at / after the last record
    # a grid that starts after the first step leaves the steps before it missing
    got = rr.interpolate_like_json_source([1.0, 3.0], [60, 120], [0, 30, 60, 90, 120])
    assert same_bits(got, [miss, miss, 1.0, 2.0, miss])
    # a first record before the first step: the first interval is entered part-way
    assert same_bits(rr.interpolate_like_json_source([0.0, 4.0, 0.0], [-60, 60, 90], [0, 30, 60]), [2.0, 3.0, 4.0])
    # -100 is missing (> -100 is valid), except for LW_net whose threshold is -1000; NaN is missing
    got = rr.interpolate_like_json_source([1.0, -100.0, 3.0, 5.0], [0, 60, 120, 180], [0, 30, 60, 90, 120, 150])
    assert same_bits(got, [1.0, miss, miss, miss, 3.0, 4.0])
    got = rr.interpolate_like_json_source([1.0, -100.0, 3.0], [0, 60, 120], [0, 30, 60], miss=-1000.0)
    assert same_bits(got, [1.0, -49.5, -100.0])
    got = rr.interpolate_like_json_source([1.0, -1000.0, 3.0], [0, 60, 120], [0, 30, 60, 90], miss=-1000.0)
    assert same_bits(got, [1.0, miss, miss, miss])
    assert same_bits(rr.interpolate_like_json_source([np.nan, 2.0, 4.0], [0, 60, 120], [0, 30, 60, 90]),
                     [miss, miss, 2.0, 3.0])
    # -0.0 is a value: kept with its sign at its record time
    assert same_bits(rr.interpolate_like_json_source([-0.0, 2.0], [0, 60], [0, 30]), [-0.0, 1.0])
    # the phase: the record at its time, the NEXT record in between, -9999 where missing
    got = rr.interpolate_like_json_source([1.0, 2.0, -9999.0, 3.0], [0, 60, 120, 180], [0, 30, 60, 90, 120, 150, 180],
                                          phase=True)
    assert same_bits(got, [1.0, 2.0, 2.0, -9999.0, -9999.0, 3.0, -9999.0])


def test_ascii_source_restatement_by_hand():
    f = -9999.9
    ia = rr.interpolate_like_ascii_source
    # nearest VALID records on either side, whole-minute weights; an exact hit on a missing record interpolates
    got = ia([10.0, 20.0, np.nan, 40.0], [0, 1, 4, 7], 60.0, 9)
    assert same_bits(got, [10.0, 20.0, 140.0 / 6, (4 * 20.0 + 2 * 40.0) / 6, 30.0, (2 * 20.0 + 4 * 40.0) / 6,
                           (20.0 + 5 * 40.0) / 6, 40.0, f])
    # 180 minutes apart is interpolated, 181 is not
    assert same_bits(ia([0.0, 18.0], [0, 180], 60.0, 181)[[0, 90, 180]], [0.0, 9.0, 18.0])
    assert same_bits(ia([0.0, 18.0], [0, 181], 60.0, 182)[[0, 90, 181]], [0.0, f, 18.0])
    # before the first record and after the last nothing; a missing first record: the backward search stops at 0
    assert same_bits(ia([5.0, 7.0], [2, 4], 60.0, 6), [f, f, 5.0, 6.0, 7.0, f])
    assert same_bits(ia([np.nan, 5.0, 7.0], [0, 2, 4], 60.0, 5), [f, f, 5.0, 6.0, 7.0])
    assert same_bits(ia([-9999.0, 5.0, np.nan, 9.0], [0, 2, 4, 6], 60.0, 7), [f, f, 5.0, 6.0, 7.0, 8.0, 9.0])
    # whole minutes at a time step that does not divide 60: 45 s -> 0, 90 s -> 1, 135 s -> 2 minutes
    assert same_bits(ia([3.0, 6.0], [0, 4], 45.0, 5), [3.0, 3.0, 4.0, 5.0, 6.0])
    assert same_bits(ia([3.0, 6.0], [0, 3], 20.0, 4), [3.0, 3.0, 3.0, 6.0])
    # -9000 is a value, one ulp below it is missing
    below = float(np.nextafter(-9000.0, -np.inf))
    assert same_bits(ia([-9000.0, 0.0], [0, 2], 60.0, 3), [-9000.0, -4500.0, 0.0])
    assert same_bits(ia([below, 0.0], [0, 2], 60.0, 3), [f, f, 0.0])
    # relative humidity clamped to [0, 100], -0 becomes +0; precipitation above 100 is dropped
    got = ia([-0.0, 140.0, -5.0, 100.0], [0, 1, 2, 3], 60.0, 4, kind=1)
    assert same_bits(got, [0.0, 100.0, 0.0, 100.0])
    above = float(np.nextafter(100.0, np.inf))
    assert same_bits(ia([100.0, above], [0, 1], 60.0, 2, kind=2), [100.0, f])
    # the phase is interpolated, then stored into an int: truncation toward zero, and +0 for (-1, 0)
    got = ia([-0.5, -1.5, 2.7, -2.0, 0.0], [0, 1, 2, 3, 5], 60.0, 5, kind=3, fill=-9999.0)
    assert same_bits(got, [0.0, -1.0, 2.0, -2.0, -1.0])


@pytest.mark.parametrize("dt", rr.DTS)
def test_restatements_agree_with_synth_and_the_oracle(dt, oracle):
    """The literal JsonSource loop against synth.interpolate_records (the vectorised form the other suites use) on
    every grid it covers, and the AsciiSource loop against the oracle's restatement on every grid."""
    sim_len = _sim_len(dt)
    for name in _grids(dt):
        rs, rec, ex1, rec2, ex2 = _case(dt, name)
        if rs[0] <= 0:
            r = synth.Records(NPTS, len(rs))
            for v, n in enumerate(rr.RECORD_VARS):
                setattr(r, n, np.ascontiguousarray(rec[:, v, :].T))
            r.record_step = rs
            fields = synth.interpolate_records(r, sim_len, dt)
            for v, n in enumerate(rr.RECORD_VARS):
                assert same_bits(fields[n].astype(np.float64), ex1[:, v, :].T), (name, n)
        else:
            with pytest.raises(ValueError):                # (synth covers grids from step 0 or before only)
                synth.interpolate_records(_records_with_steps(rs), sim_len, dt)
        kinds = {rr.RHZ: 1, rr.PREC: 2, rr.PHASE: 3}
        for v in range(11):
            for p in range(NPTS):
                want = oracle.interpolate_example2(rec2[:, v, p], rs, dt, sim_len, kinds.get(v, 0),
                                                   -9999.0 if v == rr.PHASE else -9999.9)
                assert same_bits(ex2[:, v, p], want), (name, v, p)


def _records_with_steps(rs):
    r = synth.Records(1, len(rs))
    r.record_step = rs
    return r


def _derivable(rec, seed):
    """The grid's records with the required inputs made valid for most points, so that the derivation has
    something to derive: points 0-2 keep their missing required values and fail the screening."""
    rng = np.random.default_rng(seed)
    r = rec.copy()
    n = r.shape[0]
    for v, lo, hi in ((rr.V["tair"], -8.0, 4.0), (rr.V["Rhz"], 50.0, 100.0), (rr.V["prec"], 0.0, 2.0),
                      (rr.V["SW"], 0.0, 200.0), (rr.V["LW"], 200.0, 320.0), (rr.V["VZ"], 0.0, 10.0)):
        r[:, v, 3:] = rng.uniform(lo, hi, (n, r.shape[2] - 3))
    return r


@pytest.mark.parametrize("dt", rr.DTS)
def test_host_derivation_equals_read_input_on_json_source_arrays(dt):
    """roadsurf_read_input_derive_records on every grid against synth.read_input_derive (examples/example1
    roadrunner.cpp:157-278) on arrays interpolated by the literal JsonSource loop, plus read_input's screening:
    a point is active when no required input is missing at any step.  A grid that starts after step 0 leaves the
    first steps missing, so read_input rejects every point; the library rejects the grid."""
    sim_len = _sim_len(dt)
    settings = abi.default_settings(sim_len, 1, 1, dt, 15, coupling_minutes=60)
    fstep = sim_len // 3
    for name in _grids(dt):
        rs, rec0, _, _, _ = _case(dt, name)
        rec = _derivable(rec0, seed=len(rs))
        fields = rr.json_source_fields(rec, rs, sim_len, dt)
        x = fields[:, REQUIRED, :]
        ok = ~(np.isnan(x) | (x < -9000.0)).any(axis=(0, 1))
        local = np.full((lib.L_NLOCAL, NPTS), 123.0)
        latest = np.full(NPTS, fstep + 1, dtype=np.int32)
        if rs[0] > 0:
            assert not ok.any(), name
            with pytest.raises(lib.RoadSurfError, match="record_step"):
                lib.read_input_derive_records(rec, rs, settings, fstep, local, latest_obs_index=latest)
            continue
        lib.read_input_derive_records(rec, rs, settings, fstep, local, latest_obs_index=latest)
        assert np.array_equal(local[lib.L_ACTIVE] != 0, ok), (name, local[lib.L_ACTIVE], ok)
        pa = abi.PointArrays(NPTS, sim_len)
        for v, n in enumerate(rr.RECORD_VARS):
            if n == "PrecPhase":
                pa.PrecPhase[:] = fields[:, v, :].T.astype(np.int32)
            else:
                getattr(pa, n)[:] = fields[:, v, :].T
        synth.read_input_derive(pa, settings, fstep)
        for p in np.nonzero(ok)[0]:
            lp = pa.local[p]
            want = [lp.tair_relax, lp.VZ_relax, lp.RH_relax, lp.couplingTsurf, lp.couplingIndexI, lp.InitLenI]
            got = local[[lib.L_TAIR_RELAX, lib.L_VZ_RELAX, lib.L_RH_RELAX, lib.L_COUPLING_TSURF,
                         lib.L_COUPLING_INDEX, lib.L_INIT_LEN], p]
            assert same_bits(got, np.array(want, dtype=np.float64)), (name, int(p), got, want)
        if name == "hourly_from_0":
            assert ok[3:].all() and (local[lib.L_COUPLING_INDEX, 3:] > 0).any(), name


# ---- the expansion kernel (GPU) -------------------------------------------------------------------------

def _model(rslib, dt, sim_len, **kw):
    settings = abi.default_settings(sim_len, 0, 0, dt, 15, **kw)
    params = abi.default_parameters(dt)
    rslib.set_model(settings, params)
    return settings, params


def _records_batch(rslib, rs, rec, sim_len, **kw):
    import torch
    npts = rec.shape[2]
    db = rslib.DeviceBatch(npts, sim_len, n_records=len(rs), coarse=True, nvar=rec.shape[1], **kw)
    host = np.zeros(tuple(db.forcing.shape))
    host[:, :, :npts] = rec
    db.forcing.copy_(torch.from_numpy(host))
    db.record_step.copy_(torch.from_numpy(np.asarray(rs, dtype=np.int32)))
    return db


@pytest.mark.gpu
@pytest.mark.parametrize("dt", rr.DTS)
def test_expansion_kernel_equals_both_restatements(rslib, dt):
    """rs_expand_records_kernel, rule 1 and rule 2, all 12 variables, npoints < ld: the full run and sub-ranges
    [b, e] whose first step lies on a record step, one step before and one step after it."""
    sim_len = _sim_len(dt)
    _model(rslib, dt, sim_len)
    for name in _grids(dt):
        rs, rec, ex1, rec2, ex2 = _case(dt, name, nvar=12)
        inner = [int(s) for s in rs if 2 <= s < sim_len - 40]
        k = inner[len(inner) // 2] if inner else sim_len // 2
        ranges = [(1, sim_len), (k + 1, k + 37), (k, k + 3), (k + 2, sim_len)]   # (1-based step = index + 1)
        for rule, records, want in ((1, rec, ex1), (2, rec2, ex2)):
            if want is None:
                continue                      # example1's grids start at or before step 0 (checked elsewhere)
            db = _records_batch(rslib, rs, records, sim_len)
            assert db.ld > NPTS
            for b, e in ranges:
                got = db.expand(rule, b, e).cpu().numpy()
                assert same_bits(got[:, :, :NPTS], want[b - 1:e]), (name, rule, b, e, _first_diff(got[:, :, :NPTS],
                                                                                               want[b - 1:e]))


def _first_diff(a, b):
    from parity import bit_mismatch
    bad = np.argwhere(bit_mismatch(a, b))
    if not len(bad):
        return None
    i = tuple(bad[0])
    return dict(at=[int(x) for x in i], got=float(a[i]).hex(), want=float(b[i]).hex(), count=len(bad))


@pytest.mark.gpu
def test_expansion_of_more_than_65535_steps_in_one_call(rslib):
    """rs_launch_expand caps grid.y at 65535 and strides over the rest: 70 001 steps in one call at ld = 32 against
    the vectorised example1 rule (rule 1) and against calls that each fit one pass (rule 2)."""
    dt, sim_len, npts = 30.0, 70_001, 5
    _model(rslib, dt, sim_len)
    rs = np.arange(-1, sim_len + 240, 120, dtype=np.int32)
    rs[5:9] += np.array([1, 2, -3, 0], dtype=np.int32)           # a few irregular intervals
    rec = rr.grid_values(len(rs), npts, seed=65535)
    db = _records_batch(rslib, rs, rec, sim_len)
    assert db.ld == 32 and sim_len > 65535
    r = synth.Records(npts, len(rs))
    for v, n in enumerate(rr.RECORD_VARS):
        setattr(r, n, np.ascontiguousarray(rec[:, v, :].T))
    r.record_step = rs
    fields = synth.interpolate_records(r, sim_len, dt)
    got = db.expand(1, 1, sim_len).cpu().numpy()
    assert got.shape[0] == sim_len
    for v, n in enumerate(rr.RECORD_VARS):
        assert same_bits(got[:, v, :npts], fields[n].astype(np.float64).T), (n, _first_diff(got[:, v, :npts],
                                                                                          fields[n].astype(np.float64).T))
    db2 = _records_batch(rslib, rs, rr.with_fractional_phases(rec, seed=1), sim_len)
    got = db2.expand(2, 1, sim_len).cpu().numpy()
    parts = np.concatenate([db2.expand(2, 1, 40_000).cpu().numpy(), db2.expand(2, 40_001, sim_len).cpu().numpy()])
    assert same_bits(got[:, :, :npts], parts[:, :, :npts])
    assert (got[65_535:, rr.V["tair"], :npts] > -9000).any()
    tail = rr.ascii_source_fields(rr.with_fractional_phases(rec, seed=1)[-6:], rs[-6:], sim_len, dt)[-200:]
    assert same_bits(got[-200:, :, :npts], tail)


# ---- the step kernel's in-flight interpolation (GPU) ------------------------------------------------------

# Subnormal records: the quotient dt_a * (vb - va) / span is subnormal there, outside div_const's exact domain
# (DESIGN.md section 4), and the step kernel's value differs from the IEEE quotient's by one ulp at some steps.
# (va, vb) at record steps 0 and 4, DT = 30 s; the kernel's and IEEE's values at steps 1, 2, 3.
SUBNORMAL_PINNED = [
    ("0x0.00c9e1a79e2a2p-1022", "0x0.0032b4aa7762fp-1022",
     ("0x0.00a4166854785p-1022", "0x0.007e4b290ac69p-1022", "0x0.00587fe9c114cp-1022"),
     ("0x0.00a4166854785p-1022", "0x0.007e4b290ac68p-1022", "0x0.00587fe9c114cp-1022")),
    ("0x0.0084aaead28d1p-1022", "0x0.00dd9a6bc2fp-1022",
     ("0x0.009ae6cb0ea5dp-1022", "0x0.00b122ab4abe8p-1022", "0x0.00c75e8b86d74p-1022"),
     ("0x0.009ae6cb0ea5dp-1022", "0x0.00b122ab4abe9p-1022", "0x0.00c75e8b86d74p-1022")),
    ("0x0.002d56010d508p-1022", "0x0.00a91fc011602p-1022",
     ("0x0.004c4870ce546p-1022", "0x0.006b3ae08f585p-1022", "0x0.008a2d50505c3p-1022"),
     ("0x0.004c4870ce546p-1022", "0x0.006b3ae08f585p-1022", "0x0.008a2d50505c4p-1022")),
]

PLANE_TAIR, PLANE_TDEW = lib.O_NAMES.__len__(), lib.O_NAMES.__len__() + 1     # extended output planes


def _in_kernel_records(rec, seed):
    """Adversarial air and dew point temperatures (missing, thresholds, tiny values, -0.0) over otherwise valid
    weather, so that the points run until a missing or out-of-range Tair / Tdew stops them."""
    rng = np.random.default_rng(seed)
    r = _derivable(rec, seed)
    n, _, npts = r.shape
    r[:, rr.V["tdew"], 3:] = np.where(rng.random((n, npts - 3)) < 0.9, r[:, rr.V["tair"], 3:] - 1.0,
                                      rec[:, rr.V["tdew"], 3:])
    r[:, rr.V["tair"], 6:] = np.where(rng.random((n, npts - 6)) < 0.5, rec[:, rr.V["tair"], 6:], r[:, rr.V["tair"], 6:])
    r[:, rr.V["SW_dir"]] = 0.0
    r[:, rr.V["LW_net"]] = -50.0
    r[:, rr.V["TSurfObs"]] = r[:, rr.V["tair"]] - 0.5
    r[:, rr.PHASE] = np.where(np.isnan(r[:, rr.PHASE]), -9999.0, r[:, rr.PHASE])
    return r


def _tiny_cases(n_records):
    """Extra points whose Tair / Tdew records are tiny normal numbers (1e-300 apart): inside the exact domain."""
    rng = np.random.default_rng(n_records)
    t = rng.uniform(1.0, 4.0, (n_records, 2, 4)) * 1e-300 * rng.choice([-1.0, 1.0], (n_records, 2, 4))
    return t


def _stop_reference(fields, sim_len):
    """First forcing index < sim_len - 1 at which CheckValues (src/InputOutput.f90:45-84) rejects the step, or -1."""
    ta, td = fields[:, rr.V["tair"]], fields[:, rr.V["tdew"]]
    bad = (ta < -90.0) | (ta > 100.0) | (td < -90) | (td > 100.0)
    for v, lo, hi in ((rr.V["Rhz"], -0.1, 120.0), (rr.V["VZ"], -1.0, 100.0), (rr.V["SW"], -0.1, 4000.0),
                      (rr.V["LW"], -0.1, 1000.0), (rr.V["prec"], -0.1, 500.0)):
        x = fields[:, v].copy()
        if v == rr.V["VZ"]:                  # Initialization raises VZ(1) to 0.4 first (src/Initialization.f90:121-123)
            x[0] = np.where(x[0] < 0.4, 0.4, x[0])
        bad |= (x < lo) | (x > hi)
    bad = bad[:sim_len - 1]
    return np.where(bad.any(axis=0), np.argmax(bad, axis=0), -1)


IN_KERNEL_VARIANTS = {
    "n15": dict(dt=30.0),
    "run_time_layers": dict(dt=45.0, nlayers=10),
    "output_depth": dict(dt=20.0, depth=True),
    "latency0_spread0": dict(dt=60.0, latency=0, spread=0),
    "latency1_spread0": dict(dt=90.0, latency=1, spread=0),
    "latency0_spread1": dict(dt=120.0, latency=0, spread=1),
    "latency1_spread1": dict(dt=30.0, latency=1, spread=1),
    "coupling_compacted": dict(dt=30.0, coupling=True, state=True),
    "coupling_one_launch": dict(dt=60.0, coupling=True, state=False),
    "chunked": dict(dt=30.0, chunked=True),
}


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(IN_KERNEL_VARIANTS))
def test_in_kernel_interpolation_is_example1s_rule(rslib, variant):
    """forcing_mode 1 with the extended outputs at out_stride 1: the Tair / Tdew planes are the forcing the step
    kernel used at each step (nothing rewrites f.Tair / f.Tdew between the fetch and store_outputs; relaxation
    works on a copy), so they must equal the literal JsonSource loop at every step of every point -- through the
    refill path at each record, the shared-memory fast path in between, the refill after coupling rewinds and in
    resumed launches.  Points stop exactly at the reference's first rejected step.  The expansion pass (rule 1) on
    the same records gives the same planes."""
    import torch
    cfg = IN_KERNEL_VARIANTS[variant]
    dt = cfg["dt"]
    sim_len = _sim_len(dt)
    coupled = cfg.get("coupling", False)
    kw = dict(coupling_minutes=60) if coupled else {}
    if cfg.get("depth"):
        kw["tsurf_output_depth"] = 0.02
    settings = abi.default_settings(sim_len, int(coupled), 0, dt, cfg.get("nlayers", 15), **kw)
    params = abi.default_parameters(dt)
    rslib.set_model(settings, params)
    time_fields = torch.from_numpy(synth.time_axis(START, sim_len, dt))
    try:
        if "latency" in cfg:
            rslib.set_option("latency_body", cfg["latency"])
            rslib.set_option("spread_small", cfg["spread"])
        for name, rs in _grids(dt).items():
            if rs[0] > 0:
                continue
            rs_, rec0, _, _, _ = _case(dt, name)
            rec = _in_kernel_records(rec0, seed=len(rs))
            tiny = _tiny_cases(len(rs))
            rec = np.concatenate([rec, np.zeros((len(rs), 11, 4))], axis=2)
            rec[:, :, NPTS:] = rec[:, :, :4]
            rec[:, rr.V["tair"]:rr.V["tdew"] + 1, NPTS:] = tiny
            npts = rec.shape[2]
            fields = rr.json_source_fields(rec, rs, sim_len, dt)
            db = _records_batch(rslib, rs, rec, sim_len, extended_outputs=True, coupling=coupled,
                                state=cfg.get("state", False) or cfg.get("chunked", False), nlayers=cfg.get("nlayers", 15))
            db.time_fields.copy_(time_fields)
            L = db.local.cpu().numpy()
            L[lib.L_LAT, :npts], L[lib.L_LON, :npts] = 62.0, 25.0
            cidx = sim_len // 2
            if coupled:
                L[lib.L_COUPLING_INDEX, :npts] = cidx
                L[lib.L_COUPLING_TSURF, :npts] = -1.5
                db.coupling_window_end = cidx if db.state is not None else 0
            db.local.copy_(torch.from_numpy(L))
            db.out.fill_(7.0)
            before = rslib.last_launch()["launches_total"]
            if cfg.get("chunked"):
                k = [int(s) for s in rs if 3 <= s < sim_len - 3]
                r0 = k[len(k) // 2] if k else sim_len // 2
                # launches whose first step reads forcing index r0 - 1, r0 (a record step), r0 + 1 and r0 + 2
                cuts = sorted({1, r0, r0 + 1, r0 + 2, r0 + 3, min(r0 + 50, sim_len), sim_len + 1})
                if len(k) > 1:
                    cuts = sorted(set(cuts) | {k[-1] + 1})
                for b, e in zip(cuts[:-1], cuts[1:]):
                    db.run(step_begin=b, step_end=e - 1)
            else:
                db.run()
            torch.cuda.synchronize()
            if coupled:                                   # lane compaction splits the run into several launches
                assert (rslib.last_launch()["launches_total"] - before > 2) == cfg["state"], variant
            out = db.out.cpu().numpy()
            got = np.stack([out[PLANE_TAIR, :, :npts], out[PLANE_TDEW, :, :npts]], axis=1)
            want = fields[:, rr.V["tair"]:rr.V["tdew"] + 1, :]
            assert same_bits(got, want), (variant, name, _first_diff(got, want))
            # the expansion pass, rule 1, on the same records
            ex = db.expand(1, 1, sim_len).cpu().numpy()[:, :11, :npts]
            assert same_bits(ex, fields), (variant, name, _first_diff(ex, fields))
            # where the points stopped
            status = db.status.cpu().numpy()[:npts]
            stop = _stop_reference(fields, sim_len)
            assert np.array_equal((status & rslib.ST_BAD_INPUT) != 0, stop >= 0), (variant, name, status, stop)
            if not coupled:
                ts = out[0, :, :npts]
                first_missing = np.where((ts == -9999.0).any(axis=0), np.argmax(ts == -9999.0, axis=0), -1)
                want_stop = np.where((stop >= 0) & (stop + 1 < sim_len), stop + 1, -1)
                assert np.array_equal(first_missing, want_stop), (variant, name, first_missing, want_stop)
            else:
                assert (status & rslib.ST_COUPLING_USED).any(), (variant, name)
    finally:
        rslib.set_option("latency_body", -1)
        rslib.set_option("spread_small", 1)


@pytest.mark.gpu
def test_in_kernel_interpolation_of_subnormal_records_is_pinned(rslib):
    """Outside div_const's domain: subnormal quotients follow the operation sequence, so the step kernel's
    interpolated value can be one ulp away from the IEEE quotient's (the expansion pass and the references divide).
    Pinned here as data, and the expansion pass still equals the IEEE value."""
    import torch
    dt, sim_len = 30.0, 6
    settings, params = _model(rslib, dt, sim_len)
    rs = np.array([0, 4, 8], dtype=np.int32)
    n = len(SUBNORMAL_PINNED)
    rec = np.zeros((3, 11, n))
    rec[:, rr.V["VZ"]], rec[:, rr.V["Rhz"]], rec[:, rr.V["LW"]], rec[:, rr.V["LW_net"]] = 3.0, 80.0, 300.0, -50.0
    rec[:, rr.PHASE], rec[:, rr.V["TSurfObs"]] = 1.0, -9999.9
    for p, (va, vb, _, _) in enumerate(SUBNORMAL_PINNED):
        rec[0, 0:2, p] = float.fromhex(va)
        rec[1, 0:2, p] = float.fromhex(vb)
        rec[2, 0:2, p] = float.fromhex(vb)
    db = _records_batch(rslib, rs, rec, sim_len, extended_outputs=True)
    db.time_fields.copy_(torch.from_numpy(synth.time_axis(START, sim_len, dt)))
    db.run()
    torch.cuda.synchronize()
    out = db.out.cpu().numpy()
    ex = db.expand(1, 1, sim_len).cpu().numpy()
    differ = 0
    for p, (va, vb, kern, ieee) in enumerate(SUBNORMAL_PINNED):
        kern = np.array([float.fromhex(x) for x in kern])
        ieee = np.array([float.fromhex(x) for x in ieee])
        ref = rr.interpolate_like_json_source([float.fromhex(va), float.fromhex(vb), float.fromhex(vb)], [0, 120, 240],
                                              [30 * i for i in range(sim_len)])
        assert same_bits(ref[1:4], ieee), p
        for plane in (PLANE_TAIR, PLANE_TDEW):
            assert same_bits(out[plane, 1:4, p], kern), (p, [float(x).hex() for x in out[plane, 1:4, p]])
        assert same_bits(ex[1:4, 0, p], ieee) and same_bits(ex[1:4, 1, p], ieee), p
        differ += int((kern != ieee).sum())
    assert differ == n


@pytest.mark.gpu
def test_in_kernel_interpolation_in_a_launch_of_the_512_and_128_thread_split(rslib):
    """One launch of more than 8 rounds of 512-thread blocks on the device's SMs with a remainder: the whole rounds
    run the 512-thread variant, the remainder the 128-thread tail.  The points are copies of a small distinct set;
    the Tair / Tdew planes of every copy must equal the reference of its original, compared on the device."""
    import torch
    dt = 30.0
    sim_len = 121
    _model(rslib, dt, sim_len)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    nb = 8 * sms + sms // 3
    P = nb * 512 - 100
    assert P >= 606_208 or sms < 148
    rs = np.array([-7, -6, 1, 2, 3, 40, 41, 100, 121, 200], dtype=np.int32)
    base = 256
    rec = _in_kernel_records(rr.grid_values(len(rs), base, seed=606), seed=7)
    fields = rr.json_source_fields(rec, rs, sim_len, dt)
    stop = _stop_reference(fields, sim_len)
    small = _records_batch(rslib, rs, rec, sim_len)
    big = rslib.DeviceBatch(P, sim_len, n_records=len(rs), coarse=True, extended_outputs=True)
    idx = torch.arange(big.ld, device="cuda") % base
    big.forcing.copy_(small.forcing[:, :, idx])
    big.record_step.copy_(small.record_step)
    big.time_fields.copy_(torch.from_numpy(synth.time_axis(START, sim_len, dt)))
    big.local[lib.L_LAT] = 62.0
    big.local[lib.L_LON] = 25.0
    before = rslib.last_launch()["launches_total"]
    big.run()
    torch.cuda.synchronize()
    li = rslib.last_launch()
    rem = nb % sms
    assert li["block"] == 512 and li["grid"] == nb - rem and 0 < rem and 4 * rem <= 3 * sms, (li, nb, sms)
    assert li["launches_total"] - before == 2          # the solar table and the step kernel (main part + tail)
    want = torch.from_numpy(np.ascontiguousarray(fields[:, rr.V["tair"]:rr.V["tdew"] + 1, :].transpose(1, 0, 2))).cuda()
    got = big.out[PLANE_TAIR:PLANE_TDEW + 1, :, :P]
    same = got.view(torch.int64) == want[:, :, idx[:P]].view(torch.int64)
    assert bool(same.all()), int((~same).sum())
    # the tail's points too: the last block of the launch
    assert bool(same[:, :, (nb - rem) * 512:].all())
    bad = (big.status[:P] & rslib.ST_BAD_INPUT) != 0
    assert torch.equal(bad, torch.from_numpy(stop >= 0).cuda()[idx[:P]])


# ---- forcing_mode 2 end to end (GPU) -----------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("dt", (30.0, 45.0, 60.0))
def test_forcing_mode_2_equals_mode_0_on_example2s_arrays(rslib, dt):
    """forcing_mode 2 in chunks of expand_steps that do not divide sim_len, with chunk boundaries on record steps and
    next to them, against forcing_mode 0 (pinned to the oracle elsewhere) on the AsciiSource restatement's arrays:
    all outputs and the status words, bit for bit."""
    import torch
    sim_len = _sim_len(dt)
    hour = rr.steps_for_minutes(60, dt)
    rs = _grids(dt)["hourly_from_0"]
    rec = rr.with_fractional_phases(_derivable(rr.grid_values(len(rs), 64, seed=int(dt)), seed=3), seed=4)
    rec[:, rr.V["tdew"]] = np.where(rec[:, rr.V["tdew"]] > -9000, np.minimum(rec[:, rr.V["tdew"]],
                                                                             rec[:, rr.V["tair"]] - 0.5), rec[:, rr.V["tdew"]])
    rec[5, rr.V["SW"], 40:44] = np.nan                 # missing in the middle of the run: those points stop
    ex2 = rr.ascii_source_fields(rec, rs, sim_len, dt)
    settings, params = _model(rslib, dt, sim_len)
    tf = torch.from_numpy(synth.time_axis(START, sim_len, dt))
    npts = rec.shape[2]
    full = rslib.DeviceBatch(npts, sim_len)
    host = np.zeros(tuple(full.forcing.shape))
    host[:, :, :npts] = ex2
    full.forcing.copy_(torch.from_numpy(host))
    full.time_fields.copy_(tf)
    full.local[lib.L_LAT] = 62.0
    full.local[lib.L_LON] = 25.0
    full.run()
    torch.cuda.synchronize()
    want = full.out.cpu().numpy()[:, :, :npts]
    want_status = full.status.cpu().numpy()[:npts]
    assert (want_status & rslib.ST_BAD_INPUT).any() and not (want_status & rslib.ST_BAD_INPUT).all()
    for E in (hour - 1, hour, hour + 1):
        assert sim_len % E != 0
        db = _records_batch(rslib, rs, rec, sim_len, rule=2, expand_steps=E, state=True)
        db.time_fields.copy_(tf)
        db.local.copy_(full.local)
        db.run()
        torch.cuda.synchronize()
        assert same_bits(db.out.cpu().numpy()[:, :, :npts], want), (E, _first_diff(db.out.cpu().numpy()[:, :, :npts], want))
        assert np.array_equal(db.status.cpu().numpy()[:npts], want_status), E


@pytest.mark.gpu
def test_ensemble_device_entry_checks_the_record_grid(rslib):
    """roadsurf_run_ensemble_device reads record_step back to place the fork: it checks the grid there too."""
    import torch
    dt, sim_len = 30.0, 241
    _model(rslib, dt, sim_len)
    for rs in (np.array([2, 60, 120, 180, 300], dtype=np.int32), np.array([0, 60, 60, 180, 300], dtype=np.int32)):
        rec = _in_kernel_records(rr.grid_values(len(rs), 8, seed=1), seed=2)
        shared = _records_batch(rslib, rs, rec, sim_len, state=True)
        shared.time_fields.copy_(torch.from_numpy(synth.time_axis(START, sim_len, dt)))
        ens = rslib.EnsembleBatch(shared, 2, 122)
        with pytest.raises(lib.RoadSurfError, match="record_step"):
            ens.run()
