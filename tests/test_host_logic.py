"""Host-side logic that surrounds the kernel: forcing interpolation, read_input derivations,
point sharding (world_size-2 gloo) and the synthetic generator."""
import os
import subprocess
import sys
import textwrap

import numpy as np

from record_refs import interpolate_like_json_source
from roadsurf_b200 import abi, sharding, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_interpolation_matches_json_source_semantics():
    rec = synth.draw_records(3, 5, seed=9, start=synth.FORECAST_START)
    rec.tair[1, 2] = -9999.9          # a missing record blanks both neighbouring intervals
    sim_len = 1 + 3 * 120
    fields = synth.interpolate_records(rec, sim_len)
    rawtime = [int(s) * 30 for s in rec.record_step]
    simtime = [i * 30 for i in range(sim_len)]
    for p in range(3):
        want = interpolate_like_json_source(rec.tair[p], rawtime, simtime)
        assert np.array_equal(fields["tair"][p], want)
        want = interpolate_like_json_source(rec.LW_net[p], rawtime, simtime, miss=-1000.0)
        assert np.array_equal(fields["LW_net"][p], want)
    # precipitation phase: the record itself at record times, otherwise the NEXT record
    assert fields["PrecPhase"].dtype == np.int32
    assert np.array_equal(fields["PrecPhase"][:, 0], rec.PrecPhase[:, 0].astype(np.int32))
    assert np.array_equal(fields["PrecPhase"][:, 1], rec.PrecPhase[:, 1].astype(np.int32))
    assert np.array_equal(fields["PrecPhase"][:, 120], rec.PrecPhase[:, 1].astype(np.int32))
    assert (fields["tair"][1, 121:360] < -9000).all() and fields["tair"][1, 120] > -100


def test_read_input_derivations_follow_the_example():
    """examples/example1/src/roadrunner.cpp:157-278."""
    arrays, settings, params, rec = synth.make_case(3, 6, seed=4, analysis_hours=6, use_coupling=1,
                                                    use_relaxation=1)
    for p in range(3):
        lp = arrays.local[p]
        assert lp.InitLenI == 721                       # GetLatestObsIndex: count of observed steps
        assert lp.tair_relax == arrays.tair[p, 721]     # first pure-forecast value
        assert lp.couplingIndexI == 720                 # 0-based index of the last observation...
        assert (arrays.TSurfObs[p, 361:721] < -9000).all()   # ...blanked over the coupling window
        assert arrays.TSurfObs[p, 360] > -100 and lp.couplingTsurf > -100
    # without observations nothing is derived and the library disables both features per point
    arrays, settings, params, rec = synth.make_case(2, 2, seed=4, use_coupling=1, use_relaxation=1)
    assert arrays.local[0].couplingIndexI == -9999 and arrays.local[0].tair_relax < -9000


def test_time_axis_and_case_shape():
    arrays, settings, params, rec = synth.make_case(2, 24, seed=1)
    assert settings.SimLen == arrays.sim_len == 2881        # 1 + 24 h * 120 (SURVEY.md section 8)
    t = arrays.time
    assert tuple(t[:, 0]) == (2019, 12, 2, 0, 0, 0) and tuple(t[:, 1]) == (2019, 12, 2, 0, 0, 30)
    assert tuple(t[:, -1]) == (2019, 12, 3, 0, 0, 0)
    arrays, settings, params, rec = synth.make_case(2, 48, seed=1, analysis_hours=6)
    assert settings.SimLen == 6481 and tuple(arrays.time[:, 0]) == (2019, 12, 1, 18, 0, 0)
    assert (arrays.Rhz <= 100).all() and (arrays.SW >= 0).all() and (arrays.SW_dir <= arrays.SW + 1e-12).all()


def test_point_arrays_pointers_address_rows():
    arrays, settings, params, rec = synth.make_case(3, 2, seed=2)
    ins = arrays.input_pointers()
    for p in range(3):
        assert ins[p].inputLen == arrays.sim_len
        assert ins[p].c_tair[5] == arrays.tair[p, 5] and ins[p].c_PrecPhase[7] == arrays.PrecPhase[p, 7]
        assert ins[p].c_hour[130] == 1 and ins[p].c_local_horizons[359] == arrays.local_horizons[p, 359]
    outs = arrays.output_pointers()
    outs[2].c_TsurfOut[3] = 1.25
    assert arrays.out["TsurfOut"][2, 3] == 1.25
    cp = arrays.copy()
    cp.tair[0, 0] += 1.0
    assert cp.tair[0, 0] != arrays.tair[0, 0] and cp.local[1].lat == arrays.local[1].lat


def test_shard_ranges_partition_the_points():
    for n in (0, 1, 7, 100000, 10**7, 51 * 10**6):
        for w in (1, 2, 4, 8):
            parts = [sharding.shard_range(n, r, w) for r in range(w)]
            assert parts[0][0] == 0 and parts[-1][1] == n
            assert all(parts[i][1] == parts[i + 1][0] for i in range(w - 1))
            sizes = [b - a for a, b in parts]
            assert max(sizes) - min(sizes) <= 1


def test_two_rank_gloo_reduction_and_sharding(tmp_path):
    """The N>1 host path of bench.py on CPU: two gloo ranks shard the points, time their shard and
    reduce max-over-ranks / sum-over-ranks."""
    script = tmp_path / "worker.py"
    script.write_text(textwrap.dedent(f"""
        import os, sys, json
        sys.path.insert(0, {ROOT!r})
        import torch.distributed as dist
        from roadsurf_b200 import sharding
        dist.init_process_group("gloo")
        r, w = dist.get_rank(), dist.get_world_size()
        a, b = sharding.shard_range(1001, r, w)
        sharding.barrier()
        tmax = sharding.reduce_over_ranks(10.0 + r, "max")
        total = sharding.reduce_over_ranks(b - a, "sum")
        if r == 0:
            print(json.dumps(dict(world=w, tmax=tmax, total=total, mine=[a, b])))
        dist.destroy_process_group()
    """))
    import socket
    with socket.socket() as sock:                      # a free port: a fixed one can be taken by another run
        sock.bind(("127.0.0.1", 0))
        port = str(sock.getsockname()[1])
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=port)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", port, str(script)],
                       capture_output=True, text=True, env=env, timeout=240)
    assert r.returncode == 0, r.stderr[-2000:]
    import json
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1]
    res = json.loads(line)
    assert res == dict(world=2, tmax=11.0, total=1001.0, mine=[0, 500])


def test_default_settings_and_copy_semantics():
    s = abi.default_settings(100)
    assert (s.DTSecs, s.NLayers, s.coupling_minutes, s.couplingEffectReduction, s.outputStep) == (
        30.0, 15, 180, 14400.0, 60)
    assert s.force_tsurf == 0 and s.tsurfOutputDepth < 0


def test_library_read_input_derive_matches_the_example_logic():
    """roadsurf_read_input_derive (C, host only, no GPU needed) against the Python restatement of
    examples/example1/src/roadrunner.cpp:157-278 used by the synthetic cases."""
    from roadsurf_b200 import lib
    arrays, settings, params, rec = synth.make_case(40, 6, seed=8, analysis_hours=6, use_coupling=1,
                                                    use_relaxation=1)
    # undo the derivation made by make_case: rebuild the un-derived inputs from the records
    fresh, settings, params = synth.case_from_records(rec, 6, 6, 1, 1)
    want_local = [(lp.InitLenI, lp.tair_relax, lp.VZ_relax, lp.RH_relax, lp.couplingIndexI, lp.couplingTsurf)
                  for lp in fresh.local]
    want_obs = fresh.TSurfObs.copy()
    raw, _, _ = synth.case_from_records(rec, 6, 6, 0, 0)       # no derivation: use flags are off
    raw.TSurfObs[3, :] = -9999.9                                # a point without any surface observation
    raw.tair[5, 100] = float("nan")                             # a point with missing required input
    ok = lib.read_input_derive(raw, settings, 720, latest_obs_index=np.full(40, 721))
    assert ok[5] == 0 and ok.sum() == 39
    for p in range(40):
        lp = raw.local[p]
        got = (lp.InitLenI, lp.tair_relax, lp.VZ_relax, lp.RH_relax, lp.couplingIndexI, lp.couplingTsurf)
        if p == 5:
            continue
        if p == 3:
            assert lp.couplingIndexI == -9999 and lp.couplingTsurf == -9999.9 and lp.InitLenI == 721
            continue
        assert got == want_local[p], p
        assert np.array_equal(raw.TSurfObs[p], want_obs[p]), p


def test_read_input_derive_from_records_equals_derivation_on_interpolated_arrays():
    """roadsurf_read_input_derive_records (coarse records, nothing materialised) against
    roadsurf_read_input_derive on the time-interpolated full-resolution arrays: same InitLenI,
    relaxation targets, coupling index / observation and screening verdicts, bit for bit.  Cases:
    observations ending at different records, a gap in the middle of the observations, none at all,
    an isolated last observation, missing required inputs at a record / only between records."""
    from roadsurf_b200 import lib
    npts, hours, ana = 48, 5, 6
    arrays, settings, params, rec = synth.make_case(npts, hours, seed=9, analysis_hours=ana, use_coupling=1,
                                                     use_relaxation=1, obs_bias=False)
    rec.TSurfObs[1, :] = -9999.9                    # no observations
    rec.TSurfObs[2, 5:] = -9999.9                   # observations end two records early
    rec.TSurfObs[3, 3] = -9999.9                    # a gap in the middle
    rec.TSurfObs[4, ana] = -9999.9                  # last analysis record missing
    rec.TSurfObs[6, :ana] = -9999.9                 # only the last observation record is valid
    rec.TSurfObs[7, :] = -9999.9
    rec.TSurfObs[7, 1] = -3.25                      # one isolated early observation (< coupling span)
    rec.tair[8, 4] = -9999.9                        # required input missing at a record
    rec.VZ[9, rec.nrec - 1] = float("nan")          # ... at the last record (only the extrapolated tail needs it)
    rec.SW[10, 0] = -9999.9                         # ... at the first record
    raw, settings, params = synth.case_from_records(rec, hours, ana, 0, 0, coupling_minutes=90)
    settings.use_coupling, settings.use_relaxation = 1, 1
    forecast_step = ana * 120
    latest = np.full(npts, forecast_step + 1, dtype=np.int32)
    latest[11] = -9999
    ok = lib.read_input_derive(raw, settings, forecast_step, latest_obs_index=latest)

    forcing = np.zeros((rec.nrec, 11, npts))
    for v, name in enumerate(synth.RECORD_VARS):
        forcing[:, v, :] = getattr(rec, name).T
    local = np.full((lib.L_NLOCAL, npts), 123.0)
    wend = lib.read_input_derive_records(forcing, rec.record_step.astype(np.int32), settings, forecast_step, local,
                                         latest_obs_index=latest)
    assert np.array_equal(local[lib.L_ACTIVE] != 0, ok != 0), (local[lib.L_ACTIVE], ok)
    assert ok[8] == 0 and ok[10] == 0 and ok.sum() < npts
    ends = set()
    for p in range(npts):
        if not ok[p]:
            continue
        lp = raw.local[p]
        want = (lp.tair_relax, lp.VZ_relax, lp.RH_relax, lp.couplingTsurf, lp.couplingIndexI, lp.InitLenI)
        got = tuple(local[[lib.L_TAIR_RELAX, lib.L_VZ_RELAX, lib.L_RH_RELAX, lib.L_COUPLING_TSURF,
                           lib.L_COUPLING_INDEX, lib.L_INIT_LEN], p])
        assert got == want, (p, got, want)
        if lp.couplingIndexI > 0:
            ends.add(lp.couplingIndexI)
    assert len(ends) > 1 and wend == 0                       # windows differ in this batch
    assert raw.local[1].couplingIndexI == -9999 and raw.local[7].couplingIndexI == -9999
    assert raw.local[6].couplingIndexI == forecast_step and raw.local[2].couplingIndexI == 4 * 120

    # a batch with one common window reports it
    common = np.arange(npts) >= 12
    local2 = np.full((lib.L_NLOCAL, int(common.sum())), 0.0)
    wend2 = lib.read_input_derive_records(np.ascontiguousarray(forcing[:, :, common]), rec.record_step.astype(np.int32),
                                          settings, forecast_step, local2)
    assert wend2 == forecast_step


def test_c_abi_defaults_equal_the_python_mirror_of_the_examples_defaults():
    """roadsurf_default_parameters / roadsurf_default_settings (C) against abi.default_parameters /
    default_settings (Python): both restate examples/example1/src/InputParameters.{h,cpp} and
    InputSettings.h; byte-identical structs for several time steps."""
    import ctypes as C
    from roadsurf_b200 import lib
    L = lib.load()
    for dt in (30.0, 60.0, 7.5):
        p = abi.InputParameters()
        C.memset(C.byref(p), 0xAB, C.sizeof(p))
        L.roadsurf_default_parameters(C.byref(p), dt)
        assert bytes(p) == bytes(abi.default_parameters(dt)), dt
        s = abi.InputSettings()
        C.memset(C.byref(s), 0xAB, C.sizeof(s))
        L.roadsurf_default_settings(C.byref(s), 2881, dt)
        assert bytes(s) == bytes(abi.default_settings(2881, dt=dt)), dt


def test_read_input_derive_from_records_randomised_missing_patterns():
    """Random holes in the observation and forcing records (seeded): the record-based derivation keeps
    agreeing with the derivation on the interpolated arrays, field by field and bit for bit."""
    from roadsurf_b200 import lib
    rng = np.random.default_rng(2024)
    npts, hours, ana = 64, 4, 5
    for trial in range(12):
        arrays, settings, params, rec = synth.make_case(npts, hours, seed=100 + trial, analysis_hours=ana,
                                                         use_coupling=1, use_relaxation=1, obs_bias=False)
        holes = rng.random(rec.TSurfObs.shape) < 0.25
        rec.TSurfObs[holes] = -9999.9
        for name in ("tair", "VZ", "Rhz", "prec", "SW", "LW"):
            v = getattr(rec, name)
            bad = rng.random(v.shape) < 0.004
            v[bad] = -9999.9 if trial % 2 else float("nan")
        span_min = int(rng.choice([30, 60, 90, 180]))
        raw, settings, params = synth.case_from_records(rec, hours, ana, 0, 0, coupling_minutes=span_min)
        settings.use_coupling, settings.use_relaxation = 1, 1
        fstep = ana * 120
        latest = rng.integers(-1, raw.sim_len, size=npts).astype(np.int32)
        ok = lib.read_input_derive(raw, settings, fstep, latest_obs_index=latest)
        forcing = np.zeros((rec.nrec, 11, npts))
        for v, name in enumerate(synth.RECORD_VARS):
            forcing[:, v, :] = getattr(rec, name).T
        local = np.zeros((lib.L_NLOCAL, npts))
        lib.read_input_derive_records(forcing, rec.record_step.astype(np.int32), settings, fstep, local,
                                      latest_obs_index=latest)
        assert np.array_equal(local[lib.L_ACTIVE] != 0, ok != 0), trial
        for p in np.where(ok != 0)[0]:
            lp = raw.local[p]
            want = (lp.tair_relax, lp.VZ_relax, lp.RH_relax, lp.couplingTsurf, lp.couplingIndexI, lp.InitLenI)
            got = tuple(local[[lib.L_TAIR_RELAX, lib.L_VZ_RELAX, lib.L_RH_RELAX, lib.L_COUPLING_TSURF,
                               lib.L_COUPLING_INDEX, lib.L_INIT_LEN], p])
            assert got == want, (trial, int(p), got, want)


def test_records_ending_inside_the_run_fail_the_screening_like_read_input():
    """JsonSource's interpolation leaves every step at or after its last raw record missing
    (JsonSource.cpp:85), and read_input then rejects the point (roadrunner.cpp:167-195).  The coarse-record
    derivation does the same, and agrees with the derivation on arrays interpolated by the example's rule
    (roadsurf_b200/example1.py::interpolate)."""
    from roadsurf_b200 import example1, lib
    npts, hours = 5, 4
    arrays, settings, params, rec = synth.make_case(npts, hours, seed=12)
    forcing = np.zeros((rec.nrec, 11, npts))
    for v, name in enumerate(synth.RECORD_VARS):
        forcing[:, v, :] = getattr(rec, name).T
    rs = rec.record_step.astype(np.int32)
    local = np.zeros((lib.L_NLOCAL, npts))
    lib.read_input_derive_records(forcing, rs, settings, 0, local)
    assert (local[lib.L_ACTIVE] == 1).all()                  # records reach beyond the last step: fine
    for cut in (1, 2):                                       # last record == last step, and before it
        f2, r2 = np.ascontiguousarray(forcing[:rec.nrec - cut]), np.ascontiguousarray(rs[:rec.nrec - cut])
        assert r2[-1] <= settings.SimLen - 1
        lib.read_input_derive_records(f2, r2, settings, 0, local)
        assert (local[lib.L_ACTIVE] == 0).all(), cut
        # the example's own rule: the tail of the interpolated series is missing
        simtime = 30 * np.arange(settings.SimLen)
        tair = example1.interpolate(30 * r2.astype(np.int64), f2[:, 0, 0], simtime)
        assert (tair[int(r2[-1]):] < -9000).all() and tair[int(r2[-1]) - 1] > -100
        fields_tail = synth.interpolate_records(_short_records(rec, cut), settings.SimLen)["tair"][0]
        assert np.array_equal(fields_tail, tair)


def _short_records(rec, cut):
    short = synth.Records(rec.npoints, rec.nrec - cut)
    for v in synth.RECORD_VARS:
        setattr(short, v, getattr(rec, v)[:, :rec.nrec - cut].copy())
    short.record_step = rec.record_step[:rec.nrec - cut]
    return short


def test_read_input_derive_covers_example2s_relaxation_rule():
    """example2's read_input (examples/example2/src/roadrunner.cpp:139-264) differs from example1's only in the
    relaxation block: InitLenI = secs/DT + 1 from the TIME of the latest air-temperature observation, targets at
    the 0-based index InitLenI (:223-231).  Restated here directly and compared with the library called the way
    the header says (latest_obs_index = secs/DT + 1), point by point, with per-point observation times."""
    from roadsurf_b200 import lib
    rng = np.random.default_rng(5)
    arrays, settings, params, rec = synth.make_case(24, 6, seed=11, analysis_hours=6, use_coupling=1, use_relaxation=1)
    raw, _, _ = synth.case_from_records(rec, 6, 6, 0, 0)
    dt, sim_len = settings.DTSecs, settings.SimLen
    forecast_step = 720
    obs_secs = rng.integers(3 * 3600, 6 * 3600, size=24) // 30 * 30      # seconds after start_time, per point
    obs_secs[7] = -1                                                      # a point without air-temperature observations
    span = int(settings.coupling_minutes * 60 / dt)
    want = []
    for p in range(24):
        init_len = 1 + int(forecast_step * dt / dt)                       # :162-164
        tr = vr = rr = -9999.9
        if obs_secs[p] >= 0:                                              # :220-231
            init_len = int(obs_secs[p] / dt) + 1
            tr, vr, rr = raw.tair[p, init_len], raw.VZ[p, init_len], raw.Rhz[p, init_len]
        obs = raw.TSurfObs[p]
        i = sim_len - 1                                                   # :234-259
        while i >= 0 and (np.isnan(obs[i]) or obs[i] < -9000 or obs[i] < -100):
            i -= 1
        ci, ct = -9999, -9999.9
        if i >= span:
            ci, ct = i, obs[i]
        want.append((init_len, tr, vr, rr, ci, ct))
    idx = np.where(obs_secs >= 0, obs_secs // 30 + 1, -1).astype(np.int32)
    ok = lib.read_input_derive(raw, settings, forecast_step, latest_obs_index=idx)
    assert ok.all()
    for p in range(24):
        lp = raw.local[p]
        assert (lp.InitLenI, lp.tair_relax, lp.VZ_relax, lp.RH_relax, lp.couplingIndexI, lp.couplingTsurf) == want[p], p
        if want[p][4] > 0:                                                # blanked over (i - span, i]
            assert (raw.TSurfObs[p, want[p][4] - span + 1: want[p][4] + 1] == -9999.9).all()
