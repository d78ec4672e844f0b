"""Parity of the CUDA path against the CPU oracle, through the C ABI (roadsurf_run_batch,
runsimulation, roadsurf_run_device).  All tests need a GPU.

BASELINE.json's tolerance is 1e-3 K / 1e-3 mm with threshold flips counted; since the kernel evaluates
exp / log as the host libm does, the CUDA path is BIT-IDENTICAL to the oracle, and that is what every
comparison here asserts: every output value of every point and step, the -9999.0 fill, the status
words, and the ground-layer temperatures.  The `exact` fixture fails (it does not skip) on a box whose
libm is not the mirrored one.
"""
import numpy as np
import pytest

from golden_io import CASE_NAMES, load_case
from parity import S_TOL, T_TOL, compare, same_bits
from roadsurf_b200 import abi, synth

pytestmark = pytest.mark.gpu


def _run_both(rslib, oracle, arrays, settings, params, ngpus=1):
    ref = arrays.copy()
    st_gpu = rslib.run_batch(arrays, settings, params, ngpus=ngpus)
    st_cpu, steps = oracle.run_batch(ref, settings, params, nthreads=8)
    return compare(arrays.out, ref.out), st_gpu, st_cpu, ref, steps


@pytest.fixture(autouse=True)
def _exact_everywhere(exact):
    """Every test of this module asserts bit-identity: fail loudly where the host libm cannot give it."""


def _assert_parity(r, max_mismatch=0.0):
    """Bit-identity (the `max_mismatch` argument of the tolerance era is ignored)."""
    assert r["bit_identical"], r
    assert r["mismatch_fraction"] == 0.0 and r["max_dT_all"] == 0.0 and r["max_dS_all"] == 0.0, r


def test_plain_forecast_matches_oracle(rslib, oracle):
    """c2-like: multi-point, no coupling, 30 % of the points with sky-view radiation."""
    arrays, settings, params, _ = synth.make_case(300, 24, seed=21)
    r, sg, sc, ref, steps = _run_both(rslib, oracle, arrays, settings, params)
    _assert_parity(r)
    assert np.array_equal(sg, sc)
    stats = rslib.last_batch_stats()
    assert stats["executed_steps"] == steps == 300 * arrays.sim_len
    assert rslib.last_launch()["regs_per_thread"] > 0


def test_coupling_and_relaxation_match_oracle(rslib, oracle):
    """c3-like: 6 h analysis + 24 h forecast with coupling to the last observation + relaxation."""
    arrays, settings, params, _ = synth.make_case(400, 24, seed=22, analysis_hours=6, use_coupling=1,
                                                   use_relaxation=1)
    r, sg, sc, ref, steps = _run_both(rslib, oracle, arrays, settings, params)
    _assert_parity(r)
    assert np.array_equal(sg, sc) and (sg & rslib.ST_COUPLING_USED).all()
    # coupling did its job: surface temperature at the window end is near the observation
    end = arrays.local[0].couplingIndexI - 1
    ok = ~((sg & rslib.ST_COUPLING_FAILED) > 0)
    obs = np.array([arrays.local[p].couplingTsurf for p in range(arrays.npoints)])
    assert np.max(np.abs(arrays.out["TsurfOut"][ok, end] - obs[ok])) < 0.11
    # the lockstep re-runs cost more steps than the per-point re-runs, never fewer
    assert rslib.last_batch_stats()["executed_steps"] == steps


@pytest.mark.parametrize("name", CASE_NAMES)
def test_golden_fixtures(rslib, name):
    arrays, settings, params, golden, status, stride, steps = load_case(name)
    st = rslib.run_batch(arrays, settings, params, ngpus=1)
    assert np.array_equal(st, status)
    got = {k: arrays.out[k][:, ::stride] for k in golden}
    _assert_parity(compare(got, golden), max_mismatch=0.34)


def test_runsimulation_single_point_drop_in(rslib, oracle):
    """The reference's own entry point and signature (examples/example1/src/Simulation.f90:4-6)."""
    arrays, settings, params, _ = synth.make_case(3, 6, seed=23, analysis_hours=6, use_coupling=1,
                                                   use_relaxation=1, sky_view_fraction=1.0)
    ref = arrays.copy()
    for p in range(3):
        rslib.runsimulation(arrays, settings, params, point=p)
    oracle.run_batch(ref, settings, params)
    _assert_parity(compare(arrays.out, ref.out), max_mismatch=0.34)


def test_empty_ragged_and_tiny_batches(rslib, oracle):
    arrays, settings, params, _ = synth.make_case(1, 1, seed=24)
    empty = abi.PointArrays(0, arrays.sim_len)
    assert len(rslib.run_batch(empty, settings, params)) == 0          # npoints = 0
    for npts in (1, 31, 33, 97):                                       # not multiples of the warp size
        arrays, settings, params, _ = synth.make_case(npts, 2, seed=25 + npts)
        r, sg, sc, _, _ = _run_both(rslib, oracle, arrays, settings, params)
        _assert_parity(r, max_mismatch=0.2)
        assert np.array_equal(sg, sc)
    # SimLen = 1 (only the "last value" step runs) and SimLen = 2
    for sim_len in (1, 2):
        arrays, settings, params, _ = synth.make_case(5, 1, seed=26)
        settings.SimLen = sim_len
        short = abi.PointArrays(5, sim_len)
        for n in abi.INPUT_DOUBLE_FIELDS:
            getattr(short, n[2:])[:] = getattr(arrays, n[2:])[:, :sim_len]
        short.PrecPhase[:] = arrays.PrecPhase[:, :sim_len]
        short.time[:] = arrays.time[:, :sim_len]
        short.local_horizons[:] = arrays.local_horizons
        for p in range(5):
            short.local[p] = arrays.local[p]
        r, sg, sc, _, _ = _run_both(rslib, oracle, short, settings, params)
        assert r["max_dT_all"] < 1e-9 and r["max_dS_all"] < 1e-9 and np.array_equal(sg, sc)


def test_bad_input_stops_the_point_and_leaves_missing_values(rslib, oracle):
    """CheckValues (src/InputOutput.f90:45-84): the loop stops, later outputs stay -9999.0."""
    arrays, settings, params, _ = synth.make_case(40, 6, seed=27)
    arrays.tair[3, 100] = 150.0       # out of range at step 101
    arrays.VZ[7, 0] = -5.0            # clamped to 0.4 by Initialization before it is checked
    arrays.SW[9, 300] = np.nan        # NaN compares false: not caught by the range check
    arrays.Rhz[11, 1] = 130.0
    r, sg, sc, ref, _ = _run_both(rslib, oracle, arrays, settings, params)
    assert np.array_equal(sg, sc)
    assert sg[3] & rslib.ST_FAILED and sg[3] & rslib.ST_BAD_INPUT and sg[11] & rslib.ST_FAILED
    assert not (sg[7] & rslib.ST_FAILED)
    for k in arrays.out:
        # identical pattern of computed / missing values, bit-exact fill
        assert np.array_equal(arrays.out[k] == -9999.0, ref.out[k] == -9999.0), k
        assert np.array_equal(np.isnan(arrays.out[k]), np.isnan(ref.out[k])), k
    assert (arrays.out["TsurfOut"][3, 101:] == -9999.0).all() and arrays.out["TsurfOut"][3, 100] != -9999.0
    assert (arrays.out["TsurfOut"][11, 2:] == -9999.0).all()
    good = [p for p in range(40) if p not in (3, 9, 11)]
    sub = lambda o: {k: v[good] for k, v in o.items()}
    _assert_parity(compare(sub(arrays.out), sub(ref.out)), max_mismatch=0.2)


def test_missing_observations_and_mixed_coupling_windows(rslib, oracle):
    """Per-point coupling windows: different observation times, points without observations and
    points whose window starts at step 1 share one batch (grouped into warps by the library)."""
    arrays, settings, params, _ = synth.make_case(150, 6, seed=28, analysis_hours=6, use_coupling=1,
                                                   use_relaxation=1)
    rng = np.random.default_rng(5)
    for p in range(150):
        lp = arrays.local[p]
        kind = p % 5
        if kind == 1:                                   # no surface observation: coupling off
            lp.couplingTsurf, lp.couplingIndexI = -9999.9, -9999
        elif kind == 2:                                 # earlier observation time
            lp.couplingIndexI = int(rng.integers(400, 700))
        elif kind == 3:                                 # window clipped at the start of the run
            lp.couplingIndexI = int(rng.integers(50, 360))
        elif kind == 4:                                 # relaxation switched off by a bad target
            lp.tair_relax = -9999.9
    r, sg, sc, ref, steps = _run_both(rslib, oracle, arrays, settings, params)
    assert np.array_equal(sg, sc)
    assert not (sg[1::5] & rslib.ST_COUPLING_USED).any() and (sg[0::5] & rslib.ST_COUPLING_USED).all()
    _assert_parity(r, max_mismatch=0.1)
    assert rslib.last_batch_stats()["groups"] == 1


def test_time_axis_per_point_is_grouped(rslib, oracle):
    arrays, settings, params, _ = synth.make_case(70, 3, seed=29, sky_view_fraction=1.0)
    import datetime as dt
    tpp = np.repeat(arrays.time[None], 70, axis=0).copy()
    summer = synth.time_axis(dt.datetime(2020, 6, 20, 9, 0, 0), arrays.sim_len, 30.0)
    tpp[35:] = summer                                   # half of the points run on a June morning
    arrays.time_per_point = tpp
    r, sg, sc, ref, _ = _run_both(rslib, oracle, arrays, settings, params)
    assert rslib.last_batch_stats()["groups"] == 2 and np.array_equal(sg, sc)
    _assert_parity(r, max_mismatch=0.1)
    # the sun is up in June: the shadowing code really ran and changed the result
    assert np.abs(arrays.out["TsurfOut"][35:, -1] - arrays.out["TsurfOut"][:35, -1]).max() > 1e-3


def test_output_depth_force_tsurf_and_layer_count_variants(rslib, oracle):
    # per-step depth array
    arrays, settings, params, _ = synth.make_case(40, 3, seed=30, analysis_hours=2)
    arrays.Depth[:, :] = 0.04
    arrays.Depth[::3, 100:] = 0.0
    arrays.Depth[1::3, :] = 5.0        # deeper than the last layer
    _assert_parity(_run_both(rslib, oracle, arrays, settings, params)[0], max_mismatch=0.1)
    # run-constant tsurfOutputDepth, forced surface temperature, NLayers != 15 (generic kernel)
    for kw, nl in ((dict(tsurf_output_depth=0.06), 15), (dict(force_tsurf=1), 15),
                   (dict(tsurf_output_depth=0.0), 12), ({}, 20), ({}, 4)):
        arrays, settings, params, _ = synth.make_case(40, 3, seed=31, analysis_hours=2, nlayers=nl,
                                                       settings_kw=kw)
        r, sg, sc, _, _ = _run_both(rslib, oracle, arrays, settings, params)
        _assert_parity(r, max_mismatch=0.1)
        assert np.array_equal(sg, sc)
        assert rslib.last_launch()["nlayers"] == nl


def test_parameter_overrides_reach_the_kernel(rslib, oracle):
    arrays, settings, _, _ = synth.make_case(64, 6, seed=32)
    params = abi.default_parameters(30.0, Emiss=0.9, ZMom=0.2, AlbSnow=0.7, freezing_limit_normal=-0.5,
                                    ice_melting_limit_normal=0.4, TClimG=4.0, Albedo_surroundings=0.3)
    r, sg, sc, ref, _ = _run_both(rslib, oracle, arrays, settings, params)
    _assert_parity(r, max_mismatch=0.1)
    base = arrays.copy()
    rslib.run_batch(base, settings, abi.default_parameters(30.0))
    assert np.abs(base.out["TsurfOut"] - arrays.out["TsurfOut"]).max() > 1e-2


def test_device_resident_coarse_forcing_and_strided_output(rslib, oracle):
    """Coarse hourly records interpolated on the device (N1) + output every 120th step (N2) against
    the oracle fed with host-interpolated full-resolution arrays."""
    import torch
    arrays, settings, params, rec = synth.make_case(200, 12, seed=33)
    ref = arrays.copy()
    st_cpu, _ = oracle.run_batch(ref, settings, params, nthreads=8)
    rslib.set_model(settings, params)
    for stride in (1, 120):
        db = rslib.DeviceBatch(200, arrays.sim_len, n_records=rec.nrec, coarse=True, horizons=True,
                               out_stride=stride)
        db.load_records(rec)
        db.time_fields.copy_(torch.from_numpy(arrays.time))
        db.load_local(arrays.local, arrays.local_horizons)
        db.out.fill_(7.0)
        db.run()
        torch.cuda.synchronize()
        got = db.outputs()
        want = {k: v[:, ::stride] for k, v in ref.out.items()}
        _assert_parity(compare(got, want), max_mismatch=0.1)
        assert np.array_equal(db.status.cpu().numpy()[:200], st_cpu)
        cnt = db.counters.cpu().numpy()
        assert cnt[rslib.CNT_EXECUTED_STEPS] == 200 * arrays.sim_len
    assert got["TsurfOut"].shape == (200, 13)


def test_device_resident_full_resolution_matches_batch_entry(rslib):
    """Same inputs through the SoA device entry and through roadsurf_run_batch: bit-identical."""
    import torch
    arrays, settings, params, _ = synth.make_case(100, 3, seed=34, analysis_hours=2, use_coupling=1,
                                                   use_relaxation=1, settings_kw=dict(coupling_minutes=60))
    rslib.set_model(settings, params)
    db = rslib.DeviceBatch(100, arrays.sim_len, horizons=True, coupling=True)
    db.load_point_arrays(arrays)
    db.run()
    torch.cuda.synchronize()
    got = db.outputs()
    rslib.run_batch(arrays, settings, params)
    for k in got:
        assert np.array_equal(got[k], arrays.out[k]), k


def test_point_order_does_not_matter(rslib):
    """Indexing is bit-exact: permuting the points permutes the outputs and nothing else."""
    arrays, settings, params, _ = synth.make_case(130, 4, seed=35, analysis_hours=4, use_coupling=1,
                                                   use_relaxation=1)
    perm = np.random.default_rng(1).permutation(130)
    shuffled = abi.PointArrays(130, arrays.sim_len)
    for n in abi.INPUT_DOUBLE_FIELDS:
        getattr(shuffled, n[2:])[:] = getattr(arrays, n[2:])[perm]
    shuffled.PrecPhase[:] = arrays.PrecPhase[perm]
    shuffled.local_horizons[:] = arrays.local_horizons[perm]
    shuffled.time[:] = arrays.time
    for q, p in enumerate(perm):
        shuffled.local[q] = arrays.local[int(p)]
    rslib.run_batch(arrays, settings, params)
    rslib.run_batch(shuffled, settings, params)
    for k in arrays.out:
        assert np.array_equal(shuffled.out[k], arrays.out[k][perm]), k


def test_full_size_properties_c4_shard(rslib, oracle):
    """BASELINE config 4 at one GPU's share (10^7 / 8 points, 24 h, hourly forcing, hourly output):
    size-independent properties + sampled parity.  Replicated points must give identical results
    wherever they sit in the grid; a random sample is checked against the oracle."""
    import torch
    base_n, P = 2048, 1_250_000
    arrays, settings, params, rec = synth.make_case(base_n, 24, seed=36)
    rslib.set_model(settings, params)
    small = rslib.DeviceBatch(base_n, arrays.sim_len, n_records=rec.nrec, coarse=True, horizons=True,
                              out_stride=120)
    small.load_records(rec)
    small.time_fields.copy_(torch.from_numpy(arrays.time))
    small.load_local(arrays.local, arrays.local_horizons)
    big = rslib.DeviceBatch(P, arrays.sim_len, n_records=rec.nrec, coarse=True, horizons=True, out_stride=120)
    idx = torch.arange(big.ld, device="cuda") % base_n
    big.forcing.copy_(small.forcing[:, :, idx])
    big.record_step.copy_(small.record_step)
    big.time_fields.copy_(small.time_fields)
    big.local.copy_(small.local[:, idx])
    big.local[rslib.L_ACTIVE, P:] = 0
    big.horizons.copy_(small.horizons[:, idx])
    big.run()
    small.run()
    torch.cuda.synchronize()
    out_big, out_small = big.out[:, :, :P], small.out[:, :, :base_n]
    assert torch.equal(out_big, out_small[:, :, idx[:P]])                 # replication invariance
    assert int(big.counters[rslib.CNT_EXECUTED_STEPS]) == P * arrays.sim_len
    assert int((big.status[:P] != 0).sum()) == 0 and int((big.status[P:] != rslib.ST_NOT_RUN).sum()) == 0
    big.run()                                                             # idempotent re-run
    torch.cuda.synchronize()
    assert torch.equal(big.out[:, :, :P], out_small[:, :, idx[:P]])
    # sampled parity against the oracle
    sample = np.random.default_rng(2).choice(base_n, 128, replace=False)
    sub = abi.PointArrays(128, arrays.sim_len)
    for n in abi.INPUT_DOUBLE_FIELDS:
        getattr(sub, n[2:])[:] = getattr(arrays, n[2:])[sample]
    sub.PrecPhase[:] = arrays.PrecPhase[sample]
    sub.local_horizons[:] = arrays.local_horizons[sample]
    sub.time[:] = arrays.time
    for q, p in enumerate(sample):
        sub.local[q] = arrays.local[int(p)]
    oracle.run_batch(sub, settings, params, nthreads=8)
    got_all = small.outputs()
    got = {k: v[sample] for k, v in got_all.items()}
    want = {k: v[:, ::120] for k, v in sub.out.items()}
    _assert_parity(compare(got, want), max_mismatch=0.1)


def test_branch_free_division_primitives_are_ieee_exact(rslib):
    """The kernel replaces `a / b` by a reciprocal seed + Newton + remainder correction without the
    compiler's exponent-range test: every result must equal the IEEE quotient bit for bit."""
    tested, bad = rslib.selftest_arith(400_000_000, seed=2024)
    assert tested >= 400_000_000 and bad == [0, 0, 0], (tested, bad)


def test_tma_staged_forcing_ring_gives_identical_results(rslib):
    """Full-resolution forcing through the per-warp TMA/mbarrier ring in shared memory (option
    "forcing_staging") against the default direct loads: bit-identical, including coupling rewinds
    that restart the ring, per-step depth (12 planes) and the generic layer-count kernel."""
    cases = [dict(analysis_hours=4, use_coupling=1, use_relaxation=1), dict(), dict(nlayers=9)]
    for kw in cases:
        arrays, settings, params, _ = synth.make_case(200, 6, seed=41, **kw)
        if not kw:
            arrays.Depth[:, 50:] = 0.05
        staged = arrays.copy()
        try:
            rslib.set_option("forcing_staging", 1)
            st1 = rslib.run_batch(staged, settings, params)
            smem_staged = rslib.last_launch()["smem_bytes"]
        finally:
            rslib.set_option("forcing_staging", 0)
        st0 = rslib.run_batch(arrays, settings, params)
        # the staged variant adds the per-warp tile ring to the per-lane cold-state slots
        assert smem_staged > rslib.last_launch()["smem_bytes"] > 0
        assert np.array_equal(st0, st1)
        for k in arrays.out:
            assert np.array_equal(arrays.out[k], staged.out[k]), (kw, k)


def test_runsimulation_is_reentrant_from_host_threads(rslib, oracle):
    """The reference is called concurrently from N host threads, one point each
    (examples/example1/src/roadrunner.cpp:454-496); the drop-in must give the same answers."""
    import threading
    arrays, settings, params, _ = synth.make_case(24, 3, seed=42, analysis_hours=2, use_coupling=1,
                                                   use_relaxation=1, settings_kw=dict(coupling_minutes=60))
    ref = arrays.copy()
    rslib.run_batch(ref, settings, params)
    errors = []

    def work(lo, hi):
        try:
            for p in range(lo, hi):
                rslib.runsimulation(arrays, settings, params, point=p)
        except Exception as e:  # pragma: no cover
            errors.append(e)
    threads = [threading.Thread(target=work, args=(k * 6, k * 6 + 6)) for k in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors
    for k in arrays.out:
        assert np.array_equal(arrays.out[k], ref.out[k]), k


def test_concurrent_runsimulation_calls_are_combined_into_batches(rslib):
    """Concurrent single-point calls are run as batches by a leader thread (one point per launch
    would sit at the single-warp latency): same answers, calls with different settings are kept
    apart, and the 64 calls of ten threads are served in far fewer than 64 batches."""
    import threading
    a1, s1, p1, _ = synth.make_case(48, 3, seed=52, analysis_hours=2, use_coupling=1, use_relaxation=1,
                                    settings_kw=dict(coupling_minutes=60))
    a2, s2, p2, _ = synth.make_case(16, 3, seed=53)                     # other settings: no coupling
    r1, r2 = a1.copy(), a2.copy()
    rslib.run_batch(r1, s1, p1)
    rslib.run_batch(r2, s2, p2)
    errors = []
    import ctypes as C
    L = rslib.load()
    # the ctypes argument structs are built once: rebuilding them per call (rslib.runsimulation does) costs
    # milliseconds under the GIL, staggers the ten threads by more than a batch takes, and the test would then
    # measure Python, not the library's gathering of concurrent callers
    ptrs = {id(a): (a.input_pointers(), a.output_pointers()) for a in (a1, a2)}

    def work(arrays, settings, params, pts):
        try:
            ins, outs = ptrs[id(arrays)]
            for p in pts:
                L.runsimulation(C.byref(outs[p]), C.byref(ins[p]), C.byref(settings), C.byref(params),
                                C.byref(arrays.local[p]))
        except Exception as e:  # pragma: no cover
            errors.append(e)
    threads = [threading.Thread(target=work, args=(a1, s1, p1, range(k * 6, k * 6 + 6))) for k in range(8)]
    threads += [threading.Thread(target=work, args=(a2, s2, p2, range(k * 8, k * 8 + 8))) for k in range(2)]
    calls0, batches0 = rslib.runsimulation_counters()
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    calls, batches = rslib.runsimulation_counters()
    assert not errors
    for k in a1.out:
        assert np.array_equal(a1.out[k], r1.out[k]), k
        assert np.array_equal(a2.out[k], r2.out[k]), k
    assert calls - calls0 == 64
    assert batches - batches0 <= 40, batches - batches0      # ten callers at a time, two kinds of settings


def test_time_chunked_launches_resume_from_soa_state(rslib):
    """A run split into time chunks (state written as SoA planes at the end of a launch and loaded
    by the next one; each chunk given only its own slice of forcing and of the output tensor) is
    bit-identical to the single launch, with the coupling window inside the first chunk."""
    import torch
    arrays, settings, params, _ = synth.make_case(96, 8, seed=43, analysis_hours=4, use_coupling=1,
                                                   use_relaxation=1)
    rslib.set_model(settings, params)
    whole = rslib.DeviceBatch(96, arrays.sim_len, horizons=True, coupling=True, state=True)
    whole.load_point_arrays(arrays)
    whole.run()
    torch.cuda.synchronize()
    want, want_status = whole.out.clone(), whole.status.clone()
    want_steps = int(whole.counters[rslib.CNT_EXECUTED_STEPS])

    chunked = rslib.DeviceBatch(96, arrays.sim_len, horizons=True, coupling=True, state=True)
    chunked.load_point_arrays(arrays)
    chunked.out.fill_(123.0)
    cend = arrays.local[0].couplingIndexI
    bounds = [1, cend + 40, cend + 700, arrays.sim_len + 1]       # chunk k = steps [b[k], b[k+1]-1]
    got = torch.empty_like(want)
    for k in range(3):
        b, e = bounds[k], bounds[k + 1] - 1
        forcing = chunked.forcing[b - 1:e].clone()                # only this chunk's records
        out = torch.full((rslib.O_NVAR, e - b + 1, chunked.ld), 55.0, dtype=torch.float64, device="cuda")
        chunked.run(step_begin=b, step_end=e, forcing=forcing, forcing_step0=b, out=out, out_slot0=b - 1)
        torch.cuda.synchronize()
        got[:, b - 1:e] = out
    assert torch.equal(got, want)
    assert torch.equal(chunked.status, want_status)
    assert int(chunked.counters[rslib.CNT_EXECUTED_STEPS]) == want_steps
    assert torch.equal(chunked.state, whole.state)

    # a chunk boundary inside the coupling window is refused per point, not silently accepted
    bad = rslib.DeviceBatch(96, arrays.sim_len, horizons=True, coupling=True, state=True)
    bad.load_point_arrays(arrays)
    bad.run(step_begin=1, step_end=cend - 10)
    torch.cuda.synchronize()
    assert (bad.status[:96].cpu().numpy() & rslib.ST_BAD_WINDOW).all()

    # coarse forcing + strided output, two chunks
    arrays2, settings2, params2, rec = synth.make_case(64, 6, seed=44)
    rslib.set_model(settings2, params2)

    def coarse_batch():
        db = rslib.DeviceBatch(64, arrays2.sim_len, n_records=rec.nrec, coarse=True, horizons=True,
                               out_stride=120, state=True)
        db.load_records(rec)
        db.time_fields.copy_(torch.from_numpy(arrays2.time))
        db.load_local(arrays2.local, arrays2.local_horizons)
        return db
    one, two = coarse_batch(), coarse_batch()
    one.run()
    two.run(step_begin=1, step_end=300)
    two.run(step_begin=301, step_end=arrays2.sim_len)
    torch.cuda.synchronize()
    assert torch.equal(one.out, two.out) and torch.equal(one.state, two.state)


def test_batches_larger_than_the_device_budget_are_split(rslib):
    """roadsurf_run_batch processes a batch in several device batches when it does not fit the
    memory budget; forced here with a 64-point cap.  Mixed coupling windows keep their warp padding."""
    arrays, settings, params, _ = synth.make_case(300, 4, seed=45, analysis_hours=4, use_coupling=1,
                                                   use_relaxation=1, settings_kw=dict(coupling_minutes=120))
    for p in range(0, 300, 3):
        arrays.local[p].couplingIndexI = 400 + (p % 7)
    split = arrays.copy()
    st0 = rslib.run_batch(arrays, settings, params)
    try:
        rslib.set_option("max_points_per_device_batch", 64)
        st1 = rslib.run_batch(split, settings, params)
    finally:
        rslib.set_option("max_points_per_device_batch", 0)
    assert np.array_equal(st0, st1)
    for k in arrays.out:
        assert np.array_equal(arrays.out[k], split.out[k]), k
    # one common window: every device batch runs the compacted coupling passes on its own state planes
    uni, settings_u, params_u, _ = synth.make_case(300, 4, seed=48, analysis_hours=4, use_coupling=1,
                                                    use_relaxation=1, settings_kw=dict(coupling_minutes=120))
    uni_split, uni_single = uni.copy(), uni.copy()
    st_u = rslib.run_batch(uni, settings_u, params_u)
    try:
        rslib.set_option("max_points_per_device_batch", 96)
        st_us = rslib.run_batch(uni_split, settings_u, params_u)
        rslib.set_option("max_points_per_device_batch", 0)
        rslib.set_option("coupling_compaction_passes", 0)          # whole warps repeat the window
        st_u1 = rslib.run_batch(uni_single, settings_u, params_u)
    finally:
        rslib.set_option("max_points_per_device_batch", 0)
        rslib.set_option("coupling_compaction_passes", 6)
    assert np.array_equal(st_u, st_us) and np.array_equal(st_u, st_u1)
    for k in uni.out:
        assert np.array_equal(uni.out[k], uni_split.out[k]), k
        assert np.array_equal(uni.out[k], uni_single.out[k]), k
    # pooled work buffers can be released and are re-created on demand
    rslib.release_workspace()
    again = arrays.copy()
    assert np.array_equal(rslib.run_batch(again, settings, params), st0)
    assert np.array_equal(again.out["TsurfOut"], arrays.out["TsurfOut"])


def test_multi_gpu_sharding_inside_the_library(rslib):
    """ngpus > 1: contiguous point shards on several devices from the library's own host threads.
    Needs two visible GPUs; bit-identical to the single-GPU result."""
    if rslib.load().roadsurf_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    arrays, settings, params, _ = synth.make_case(333, 4, seed=46, analysis_hours=4, use_coupling=1,
                                                   use_relaxation=1, settings_kw=dict(coupling_minutes=120))
    two = arrays.copy()
    st0 = rslib.run_batch(arrays, settings, params, ngpus=1)
    st1 = rslib.run_batch(two, settings, params, ngpus=2)
    assert np.array_equal(st0, st1)
    for k in arrays.out:
        assert np.array_equal(arrays.out[k], two.out[k]), k

    # the host structure-of-arrays entry shards the same way (coarse records, coupling, strided output)
    import torch
    arr, settings, params, rec = synth.make_case(777, 5, seed=49, analysis_hours=3, use_coupling=1,
                                                 use_relaxation=1, obs_bias=False,
                                                 settings_kw=dict(coupling_minutes=60))
    forcing = np.zeros((rec.nrec, 11, 777))
    for v, name in enumerate(synth.RECORD_VARS):
        forcing[:, v, :] = getattr(rec, name).T
    local = np.zeros((rslib.L_NLOCAL, 777))
    for p in range(777):
        lp = arr.local[p]
        local[:, p] = (lp.tair_relax, lp.VZ_relax, lp.RH_relax, lp.couplingTsurf, lp.lat, lp.lon, lp.sky_view,
                       lp.couplingIndexI, lp.InitLenI, 1.0)
    hor = np.ascontiguousarray(arr.local_horizons.T)
    n_out = (arr.sim_len + 59) // 60
    outs = []
    for ng in (1, 2):
        out = np.full((rslib.O_NVAR, n_out, 777), 5.0)
        st = np.zeros(777, dtype=np.int32)
        rslib.run_host_soa(settings, params, forcing, arr.time, local, out, record_step=rec.record_step.astype(np.int32),
                           horizons=hor, status=st, out_stride=60, ngpus=ng,
                           coupling_window_end=arr.local[0].couplingIndexI)
        outs.append((out, st))
    assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1])
    assert (outs[0][0] != 5.0).all()


@pytest.mark.gpu
def test_extended_output_set_with_start_offset(rslib, oracle):
    """example2's stored set (examples/example2/src/QueryDataTools.cpp:270-341): outputs from a start
    position at a stride, plus the Tair / Tdew inputs of those steps and the dew point deficit
    Tsurf - Tdew (-9999 where either operand is missing).  One point fails its input check mid-run."""
    import torch
    npts, start, stride = 96, 37, 60
    arrays, settings, params, _ = synth.make_case(npts, 6, seed=47, analysis_hours=3, use_coupling=1,
                                                   use_relaxation=1, settings_kw=dict(coupling_minutes=60))
    arrays.tair[5, 900] = 250.0          # CheckValues stops point 5 at step 901
    arrays.tdew[7, start + 2 * stride] = -9999.9
    ref = arrays.copy()
    oracle.run_batch(ref, settings, params, nthreads=8)
    rslib.set_model(settings, params)
    sel = slice(start, None, stride)

    def check(got):
        assert np.array_equal(got["Tair"], arrays.tair[:, sel])
        assert np.array_equal(got["Tdew"], arrays.tdew[:, sel])
        ts, td = got["TsurfOut"], arrays.tdew[:, sel]
        ok = (ts > -9000) & (td > -9000)
        assert np.array_equal(got["DewPointDeficit"], np.where(ok, ts - td, -9999.0))
        assert (got["DewPointDeficit"][5, 900 // stride + 1:] == -9999.0).all()
        assert got["DewPointDeficit"][7, 2] == -9999.0
        _assert_parity(compare({k: got[k] for k in ref.out}, {k: v[:, sel] for k, v in ref.out.items()}),
                       max_mismatch=0.1)

    db = rslib.DeviceBatch(npts, arrays.sim_len, horizons=True, coupling=True, state=True, out_stride=stride,
                           out_start=start, extended_outputs=True)
    db.load_point_arrays(arrays)
    db.out.fill_(3.0)
    db.run()
    torch.cuda.synchronize()
    assert db.out.shape[0] == rslib.O_NVAR_EXT and db.n_out == len(range(start, arrays.sim_len, stride))
    check(db.outputs())

    # the same in two time chunks, each with a chunk-local output tensor
    want = db.out.clone()
    cend = arrays.local[0].couplingIndexI
    cut = cend + 100                                    # chunk 1 = steps [1, cut], chunk 2 the rest
    slots1 = len(range(start, cut, stride))             # 0-based steps start, start+stride, ... < cut
    ch = rslib.DeviceBatch(npts, arrays.sim_len, horizons=True, coupling=True, state=True, out_stride=stride,
                           out_start=start, extended_outputs=True)
    ch.load_point_arrays(arrays)
    o1 = torch.full((rslib.O_NVAR_EXT, slots1, ch.ld), 5.0, dtype=torch.float64, device="cuda")
    o2 = torch.full((rslib.O_NVAR_EXT, db.n_out - slots1, ch.ld), 5.0, dtype=torch.float64, device="cuda")
    ch.run(step_begin=1, step_end=cut, out=o1, out_slot0=0)
    ch.run(step_begin=cut + 1, step_end=arrays.sim_len, out=o2, out_slot0=slots1)
    torch.cuda.synchronize()
    assert torch.equal(torch.cat([o1, o2], dim=1), want)


@pytest.mark.gpu
@pytest.mark.parametrize("passes", [1, 3, 30])
def test_coupling_lane_compaction_is_bit_identical(rslib, passes):
    """The run split at the coupling window end, with compacted passes over the points that want
    another iteration and the stragglers finishing inside the last launch, against the single
    launch in which whole warps repeat the window: outputs, status words, per-point state and the
    number of executed point-steps are identical.  Includes points without coupling, a point that
    fails its input check inside the window and one that fails right after it."""
    import torch
    npts = 777
    arrays, settings, params, _ = synth.make_case(npts, 5, seed=51, analysis_hours=4, use_coupling=1,
                                                   use_relaxation=1, settings_kw=dict(coupling_minutes=90))
    cend = arrays.local[0].couplingIndexI
    for p in (3, 40, 41):                      # uncoupled points among coupled ones
        arrays.local[p].couplingTsurf = -9999.9
        arrays.local[p].couplingIndexI = -9999
    arrays.tair[10, cend - 50] = 250.0         # fails inside the window (0-based index = step - 1)
    arrays.tair[11, cend] = 250.0              # fails CheckValues(window end + 1)
    arrays.tair[12, cend + 30] = 250.0         # fails later
    rslib.set_model(settings, params)

    def run(compaction):
        db = rslib.DeviceBatch(npts, arrays.sim_len, horizons=True, coupling=True, state=True)
        db.load_point_arrays(arrays)
        assert db.coupling_window_end == cend
        if not compaction:
            db.coupling_window_end = 0
        db.out.fill_(9.0)
        db.run()
        torch.cuda.synchronize()
        return db

    rslib.set_option("coupling_compaction_passes", passes)
    try:
        got = run(True)
        launches = rslib.last_launch()["launches_total"]
    finally:
        rslib.set_option("coupling_compaction_passes", 6)
    want = run(False)
    assert rslib.last_launch()["launches_total"] - launches == 2      # solar table + one run kernel
    assert torch.equal(got.out, want.out)
    assert torch.equal(got.status, want.status)
    assert torch.equal(got.state[:, :npts], want.state[:, :npts])
    assert int(got.counters[rslib.CNT_EXECUTED_STEPS]) == int(want.counters[rslib.CNT_EXECUTED_STEPS])
    assert int(got.counters[rslib.CNT_FAILED_POINTS]) == int(want.counters[rslib.CNT_FAILED_POINTS]) == 3
    st = want.status[:npts].cpu().numpy()
    assert (st & rslib.ST_COUPLING_USED).astype(bool).sum() == npts - 3

    # a point whose window differs from the asserted one is refused, not silently mis-run
    bad = rslib.DeviceBatch(npts, arrays.sim_len, horizons=True, coupling=True, state=True)
    bad.load_point_arrays(arrays)
    bad.local[rslib.L_COUPLING_INDEX, 5] = cend - 7
    bad.run()
    torch.cuda.synchronize()
    st = bad.status[:npts].cpu().numpy()
    assert st[5] & rslib.ST_BAD_WINDOW and not (np.delete(st, 5) & rslib.ST_BAD_WINDOW).any()


@pytest.mark.gpu
def test_replicated_coupled_points_agree_anywhere_in_a_large_batch(rslib):
    """Config-3-like property test at a size where the compacted passes span many warps: 1536 distinct
    coupled points tiled to 30 000 (plus a ragged tail).  Every replica, wherever the compaction put
    it in any pass, must reproduce the result of the small single-launch run bit for bit."""
    import torch
    base, P = 1536, 30_011
    arrays, settings, params, _ = synth.make_case(base, 8, seed=61, analysis_hours=4, use_coupling=1,
                                                   use_relaxation=1)
    rslib.set_model(settings, params)
    small = rslib.DeviceBatch(base, arrays.sim_len, horizons=True, coupling=True)   # no state: one launch
    small.load_point_arrays(arrays)
    small.run()
    big = rslib.DeviceBatch(P, arrays.sim_len, horizons=True, coupling=True, state=True)
    idx = torch.arange(big.ld, device="cuda") % base
    for t0 in range(0, arrays.sim_len, 512):
        big.forcing[t0:t0 + 512] = small.forcing[t0:t0 + 512][:, :, idx]
    big.time_fields.copy_(small.time_fields)
    big.local.copy_(small.local[:, idx])
    big.local[rslib.L_ACTIVE, P:] = 0
    big.horizons.copy_(small.horizons[:, idx])
    big.coupling_window_end = arrays.local[0].couplingIndexI
    big.run()
    torch.cuda.synchronize()
    assert rslib.last_launch()["launches_total"] > 0
    assert torch.equal(big.out[:, :, :P], small.out[:, :, idx[:P]])
    assert torch.equal(big.status[:P], small.status[idx[:P]])
    passes_small = int(small.counters[rslib.CNT_COUPLING_PASSES]) / (small.ld / 32)
    passes_big = int(big.counters[rslib.CNT_COUPLING_PASSES]) / (big.ld / 32)
    assert passes_big < 0.6 * passes_small, (passes_big, passes_small)   # the compaction did compact
    assert int(big.counters[rslib.CNT_EXECUTED_STEPS]) * base == pytest.approx(
        int(small.counters[rslib.CNT_EXECUTED_STEPS]) * P, rel=0.02)


@pytest.mark.gpu
def test_coarse_records_with_coupling_blank_the_observations_in_the_kernel(rslib, oracle):
    """Hourly records + coupling on the device: the kernel interpolates in time (JsonSource.cpp:49-176)
    and blanks TSurfObs over the coupling window as read_input does after the interpolation
    (roadrunner.cpp:263-274).  Must equal the run on the host-interpolated, host-blanked
    full-resolution arrays bit for bit, with and without lane compaction, and match the oracle."""
    import torch
    npts = 400
    arrays, settings, params, rec = synth.make_case(npts, 6, seed=71, analysis_hours=5, use_coupling=1,
                                                     use_relaxation=1, obs_bias=False,
                                                     settings_kw=dict(coupling_minutes=120))
    ref = arrays.copy()
    st_cpu, _ = oracle.run_batch(ref, settings, params, nthreads=8)
    rslib.set_model(settings, params)
    full = rslib.DeviceBatch(npts, arrays.sim_len, horizons=True, coupling=True)
    full.load_point_arrays(arrays)
    full.run()

    def coarse(state):
        db = rslib.DeviceBatch(npts, arrays.sim_len, n_records=rec.nrec, coarse=True, horizons=True,
                               coupling=True, state=state)
        db.load_records(rec)
        db.time_fields.copy_(torch.from_numpy(arrays.time))
        db.load_local(arrays.local, arrays.local_horizons)
        db.run()
        torch.cuda.synchronize()
        return db

    one = coarse(False)                       # single launch
    assert one.coupling_window_end == 0
    many = coarse(True)                       # split at the window end, compacted passes
    assert many.coupling_window_end == arrays.local[0].couplingIndexI
    assert torch.equal(one.out, full.out) and torch.equal(one.status, full.status)
    assert torch.equal(many.out, full.out) and torch.equal(many.status, full.status)
    assert int(many.counters[rslib.CNT_EXECUTED_STEPS]) == int(full.counters[rslib.CNT_EXECUTED_STEPS])
    _assert_parity(compare(many.outputs(), ref.out), max_mismatch=0.05)
    assert np.array_equal(many.status.cpu().numpy()[:npts], st_cpu)


@pytest.mark.gpu
def test_host_soa_entry_matches_device_entry(rslib):
    """roadsurf_run_host_soa (host structure-of-arrays in, strided outputs back, chunk-pipelined
    copies) against the device-resident entry on the same data: coarse records with coupling
    (window asserted -> compacted passes, and not asserted -> single launch), ragged point count."""
    import torch
    npts = 1000 + 13
    arrays, settings, params, rec = synth.make_case(npts, 6, seed=73, analysis_hours=4, use_coupling=1,
                                                     use_relaxation=1, obs_bias=False,
                                                     settings_kw=dict(coupling_minutes=90))
    rslib.set_model(settings, params)
    db = rslib.DeviceBatch(npts, arrays.sim_len, n_records=rec.nrec, coarse=True, horizons=True,
                           coupling=True, out_stride=120)
    db.load_records(rec)
    db.time_fields.copy_(torch.from_numpy(arrays.time))
    db.load_local(arrays.local, arrays.local_horizons)
    db.run()
    torch.cuda.synchronize()
    want, want_status = db.out[:, :, :npts].cpu(), db.status[:npts].cpu()
    h = dict(forcing=db.forcing[:, :, :npts].cpu().contiguous(), time_fields=db.time_fields.cpu(),
             local=db.local[:, :npts].cpu().contiguous(), horizons=db.horizons[:, :npts].cpu().contiguous(),
             record_step=db.record_step.cpu())
    for wend in (0, arrays.local[0].couplingIndexI):
        out = torch.full((rslib.O_NVAR, db.n_out, npts), 4.0, dtype=torch.float64)
        status = torch.zeros(npts, dtype=torch.int32)
        rslib.run_host_soa(settings, params, h["forcing"], h["time_fields"], h["local"], out,
                           record_step=h["record_step"], horizons=h["horizons"], status=status, out_stride=120,
                           coupling_window_end=wend)
        assert torch.equal(out, want), wend
        assert torch.equal(status, want_status), wend
        launches = rslib.last_batch_stats()["kernel_launches"]
        assert (launches > 10) == (wend > 0), (wend, launches)


@pytest.mark.gpu
def test_bit_identical_to_the_oracle_where_the_host_libm_is_the_one_the_kernel_mirrors(rslib, oracle):
    """With exp / log evaluated as the host libm does, the CUDA path reproduces the CPU restatement
    bit for bit: no tolerance, no flips -- plain forecast with sky-view points, and analysis +
    forecast with coupling and relaxation.  (The `exact` fixture fails the test where this process's
    libm is another version.)"""
    for kw in (dict(npoints=600, hours=24, seed=81),
               dict(npoints=600, hours=30, seed=82, analysis_hours=6, use_coupling=1, use_relaxation=1)):
        arrays, settings, params, _ = synth.make_case(**kw)
        ref = arrays.copy()
        st_gpu = rslib.run_batch(arrays, settings, params)
        st_cpu, _ = oracle.run_batch(ref, settings, params, nthreads=8)
        assert np.array_equal(st_gpu, st_cpu)
        for k in ref.out:
            assert np.array_equal(arrays.out[k], ref.out[k]), (kw, k)


@pytest.mark.gpu
def test_point_order_permutation_does_not_change_results(rslib):
    """RsDeviceBatch.order (roadsurf_order_points: sky-view points gathered at one end of the launch)
    changes which thread runs which point and nothing else: coarse forcing, and full-resolution
    forcing with coupling (order + lane compaction together)."""
    import torch
    arrays, settings, params, rec = synth.make_case(1000 + 7, 6, seed=91, sky_view_fraction=0.3)
    rslib.set_model(settings, params)
    db = rslib.DeviceBatch(arrays.npoints, arrays.sim_len, n_records=rec.nrec, coarse=True, horizons=True,
                           out_stride=60)
    db.load_records(rec)
    db.time_fields.copy_(torch.from_numpy(arrays.time))
    db.load_local(arrays.local, arrays.local_horizons)
    db.run()
    torch.cuda.synchronize()
    want, want_status = db.out.clone(), db.status.clone()
    db.build_order()
    order = db.order.cpu().numpy()
    sky = db.local[rslib.L_SKY_VIEW].cpu().numpy() < 1.0
    sky[arrays.npoints:] = False
    assert sorted(order.tolist()) == list(range(db.ld))                       # a permutation
    assert sky[order[:int(sky.sum())]].all() and not sky[order[int(sky.sum()):]].any()
    db.out.fill_(1.0)
    db.run()
    torch.cuda.synchronize()
    assert torch.equal(db.out, want) and torch.equal(db.status, want_status)

    arrays, settings, params, _ = synth.make_case(500, 4, seed=92, analysis_hours=3, use_coupling=1,
                                                   use_relaxation=1, settings_kw=dict(coupling_minutes=60))
    rslib.set_model(settings, params)
    outs = []
    for ordered in (False, True):
        fb = rslib.DeviceBatch(500, arrays.sim_len, horizons=True, coupling=True, state=True)
        fb.load_point_arrays(arrays)
        if ordered:
            fb.build_order()
        fb.run()
        torch.cuda.synchronize()
        outs.append((fb.out.clone(), fb.status.clone(), int(fb.counters[rslib.CNT_EXECUTED_STEPS])))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1]) and outs[0][2] == outs[1][2]


def _coarse_run_with_state(rslib, arrays, rec, coupling, out_stride=1):
    """Device-resident coarse-record run that keeps the final per-point state planes."""
    import torch
    db = rslib.DeviceBatch(arrays.npoints, arrays.sim_len, n_records=rec.nrec, coarse=True, horizons=True,
                           coupling=coupling, state=True, out_stride=out_stride)
    db.load_records(rec)
    db.time_fields.copy_(torch.from_numpy(arrays.time))
    db.load_local(arrays.local, arrays.local_horizons)
    db.run()
    torch.cuda.synchronize()
    return db


def _assert_outputs_and_ground_state_exact(rslib, oracle, arrays, settings, params, rec, coupling):
    """Outputs, status words AND the ground temperature profile Tmp(0:N+1) + surface state at the end of
    the run, all bit for bit (north star: "surface and ground temperatures")."""
    n, nl = arrays.npoints, settings.NLayers
    ref = arrays.copy()
    st_cpu, tmp_cpu, surf_cpu = oracle.run_batch_state(ref, settings, params, nthreads=8)
    rslib.set_model(settings, params)
    db = _coarse_run_with_state(rslib, arrays, rec, coupling)
    got = db.outputs()
    for k in ref.out:
        assert same_bits(got[k], ref.out[k]), k
    assert np.array_equal(db.status.cpu().numpy()[:n], st_cpu)
    state = db.state.cpu().numpy()
    ok = (st_cpu & rslib.ST_FAILED) == 0
    assert ok.sum() > 0.9 * n
    # a failed point stops before its last step: its state is not the end-of-run state on either side
    assert same_bits(state[:nl + 2, :n].T[ok], tmp_cpu[ok]), "ground temperatures Tmp(0:N+1)"
    assert same_bits(state[nl + 2:nl + 12, :n].T[ok], surf_cpu[ok]), "surface state"
    return db, ref


def test_48h_coupled_forecast_config3_like_exact_including_ground_temperatures(rslib, oracle):
    """Config 3's shape at 1024 points: 6 h analysis + 48 h forecast (6481 steps of 30 s), coupling to the
    last observation + relaxation, 30 % sky-view points; from hourly records on the device against the
    oracle on host-interpolated arrays."""
    arrays, settings, params, rec = synth.make_case(1024, 48, seed=301, analysis_hours=6, use_coupling=1,
                                                    use_relaxation=1, obs_bias=False)
    assert arrays.sim_len == 6481
    db, ref = _assert_outputs_and_ground_state_exact(rslib, oracle, arrays, settings, params, rec, True)
    assert (db.status.cpu().numpy()[:1024] & rslib.ST_COUPLING_USED).all()
    # the same through the reference-facing batched entry (full-resolution host arrays)
    st = rslib.run_batch(arrays, settings, params)
    for k in ref.out:
        assert same_bits(arrays.out[k], ref.out[k]), k


def test_74h_example1_span_401_points_exact(rslib, oracle):
    """Configs 1-2's shape: example1's 48 h analysis + 26 h forecast (8881 steps) for its 401 stations,
    coupling + relaxation."""
    arrays, settings, params, rec = synth.make_case(401, 26, seed=302, analysis_hours=48, use_coupling=1,
                                                    use_relaxation=1, obs_bias=False)
    assert arrays.sim_len == 8881
    _assert_outputs_and_ground_state_exact(rslib, oracle, arrays, settings, params, rec, True)


def test_ground_temperatures_match_for_other_layer_counts(rslib, oracle):
    """Run-time layer counts go through the generic kernel: profile compared layer by layer."""
    for nl in (4, 12, 20):
        arrays, settings, params, rec = synth.make_case(96, 6, seed=310 + nl, nlayers=nl)
        ref = arrays.copy()
        st_cpu, tmp_cpu, _ = oracle.run_batch_state(ref, settings, params, nthreads=4)
        rslib.set_model(settings, params)
        import torch
        db = rslib.DeviceBatch(96, arrays.sim_len, nlayers=nl, horizons=True, state=True)
        db.load_point_arrays(arrays)
        db.run()
        torch.cuda.synchronize()
        assert same_bits(db.state.cpu().numpy()[:nl + 2, :96].T, tmp_cpu), nl


def test_records_that_end_inside_the_run_are_not_extrapolated(rslib, oracle):
    """The reference's interpolation stops at its last raw record (JsonSource.cpp:85): steps at and after it
    stay missing, so the point fails CheckValues there -- on the device exactly as in the oracle fed with
    host-interpolated arrays.  (read_input would reject such a point before the run; so does
    roadsurf_read_input_derive_records, tests/test_host_logic.py.)"""
    import torch
    arrays, settings, params, rec = synth.make_case(64, 6, seed=320)
    short = synth.Records(64, rec.nrec - 3)            # records end 2 h before the end of the run
    for v in synth.RECORD_VARS:
        setattr(short, v, getattr(rec, v)[:, :rec.nrec - 3].copy())
    short.lat, short.lon, short.sky_view, short.horizons = rec.lat, rec.lon, rec.sky_view, rec.horizons
    short.record_step = rec.record_step[:rec.nrec - 3]
    fields = synth.interpolate_records(short, arrays.sim_len)
    assert (fields["tair"][:, int(short.record_step[-1]):] < -9000).all()
    ref = arrays.copy()
    for name, val in fields.items():
        getattr(ref, name)[...] = val
    st_cpu, _ = oracle.run_batch(ref, settings, params, nthreads=4)
    assert (st_cpu & rslib.ST_BAD_INPUT).all()
    rslib.set_model(settings, params)
    db = rslib.DeviceBatch(64, arrays.sim_len, n_records=short.nrec, coarse=True, horizons=True)
    db.load_records(short)
    db.time_fields.copy_(torch.from_numpy(arrays.time))
    db.load_local(arrays.local, arrays.local_horizons)
    db.run()
    torch.cuda.synchronize()
    got = db.outputs()
    # The step AT the last record is still executed, on the missing values -9999.9 (CheckValues only stops
    # the next loop trip, Simulation.f90:58-59).  Its output is garbage on both sides, and the one place
    # where the two are not bit-identical: exp / log arguments that far outside the physical range leave
    # the mirrored libm fast path (rs_libm.h) for the device library, 1 ulp apart per call.
    last = int(short.record_step[-1])
    for k in ref.out:
        same = (got[k] == ref.out[k]) | (np.isnan(got[k]) & np.isnan(ref.out[k]))
        same[:, last] |= np.isclose(got[k][:, last], ref.out[k][:, last], rtol=1e-6, atol=0.0, equal_nan=True)
        bad = np.argwhere(~same)
        assert same.all(), (k, bad[:5].tolist(), [(got[k][tuple(b)], ref.out[k][tuple(b)]) for b in bad[:5]], last)
    assert np.array_equal(db.status.cpu().numpy()[:64], st_cpu)
    assert (got["TsurfOut"][:, last + 1:] == -9999.0).all() and (got["TsurfOut"][:, last - 1] > -100).all()


def test_model_switch_waits_for_asynchronous_kernels_in_flight(rslib):
    """The device's model lives in constant memory.  roadsurf_run_device is asynchronous: replacing the
    model (roadsurf_set_model, or a host entry with other settings) while its kernels run must not change
    their results -- the library waits for them before it overwrites the symbol."""
    import torch
    arrays, settings, params, rec = synth.make_case(40000, 6, seed=330)
    params_b = abi.default_parameters(30.0)
    params_b.Emiss, params_b.AlbDry, params_b.ZMom = 0.90, 0.2, 0.3

    def batch():
        db = rslib.DeviceBatch(arrays.npoints, arrays.sim_len, n_records=rec.nrec, coarse=True, horizons=True)
        db.load_records(rec)
        db.time_fields.copy_(torch.from_numpy(arrays.time))
        db.load_local(arrays.local, arrays.local_horizons)
        return db
    a, b = batch(), batch()
    rslib.set_model(settings, params)
    a.run()
    torch.cuda.synchronize()
    want_a = a.out.clone()
    rslib.set_model(settings, params_b)
    b.run()
    torch.cuda.synchronize()
    want_b = b.out.clone()
    assert not torch.equal(want_a, want_b)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    for _ in range(3):
        a.out.fill_(0.0)
        b.out.fill_(0.0)
        rslib.set_model(settings, params)
        a.run(s1)                                   # tens of milliseconds of kernel time, not waited for
        rslib.set_model(settings, params_b)         # must block until a's kernels are done
        b.run(s2)
        torch.cuda.synchronize()
        assert torch.equal(a.out, want_a) and torch.equal(b.out, want_b)


def test_prepared_statics_give_the_same_results_with_less_upload(rslib):
    """roadsurf_prepare_statics keeps the horizon table (and the sky-view point order) of a grid on the
    device: later roadsurf_run_host_soa calls upload forcing records only and produce the same bits."""
    import torch
    npts = 70000 + 5                    # two pipeline chunks, ragged
    arrays, settings, params, rec = synth.make_case(256, 6, seed=340)
    rslib.set_model(settings, params)
    small = rslib.DeviceBatch(256, arrays.sim_len, n_records=rec.nrec, coarse=True, horizons=True, out_stride=120)
    small.load_records(rec)
    small.time_fields.copy_(torch.from_numpy(arrays.time))
    small.load_local(arrays.local, arrays.local_horizons)
    idx = (torch.arange(npts, device="cuda") * 7) % 256
    forcing = small.forcing[:, :, idx].cpu().contiguous()
    local = small.local[:, idx].cpu().contiguous()
    hor = small.horizons[:, idx].cpu().contiguous()
    tf, rs = small.time_fields.cpu(), small.record_step.cpu()
    n_out = small.n_out

    def run(**kw):
        out = torch.full((rslib.O_NVAR, n_out, npts), 3.0, dtype=torch.float64)
        status = torch.zeros(npts, dtype=torch.int32)
        rslib.run_host_soa(settings, params, forcing, tf, local, out, record_step=rs, status=status,
                           out_stride=120, **kw)
        return out, status, rslib.last_batch_stats()
    want, want_status, st0 = run(horizons=hor)
    handle = rslib.prepare_statics(local, hor, ngpus=1)
    try:
        for _ in range(2):
            got, got_status, st1 = run(statics=handle)
            assert torch.equal(got, want) and torch.equal(got_status, want_status)
        assert st0["h2d_bytes"] - st1["h2d_bytes"] == 360 * 8 * npts
        # the handle belongs to one grid size
        with pytest.raises(rslib.RoadSurfError):
            rslib.run_host_soa(settings, params, forcing[:, :, :1000].contiguous(), tf, local[:, :1000].contiguous(),
                               torch.zeros((rslib.O_NVAR, n_out, 1000), dtype=torch.float64), record_step=rs,
                               out_stride=120, statics=handle)
    finally:
        rslib.release_statics(handle)
    # results agree with the device-resident run of the same points
    small.run()
    torch.cuda.synchronize()
    assert torch.equal(want.cuda(), small.out[:, :, idx])


def _stepwise(rslib, arrays, settings, params, chunk=1, stop_when_failed=True):
    """Drive a session the way examples/example1/src/Simulation.f90 drives the library: one step per loop
    trip, outputs fetched after every step, the loop ends when the (single) point has failed."""
    sess = rslib.Session(arrays, settings, params, chunk=chunk)
    launches0 = rslib.last_launch()["launches_total"]
    try:
        i = 1
        status = np.zeros(arrays.npoints, dtype=np.int32)
        while i < settings.SimLen:
            sess.step(i)
            status = sess.fetch(i)
            if stop_when_failed and arrays.npoints == 1 and (status[0] & rslib.ST_FAILED):
                break
            i += 1
        else:
            sess.step(settings.SimLen)            # lastValues + the final step (Simulation.f90:100-115)
            status = sess.fetch(settings.SimLen)
        return status, rslib.last_launch()["launches_total"] - launches0
    finally:
        sess.close()


def test_stepwise_session_equals_the_single_launch(rslib):
    """roadsurf_step (one launch per model step on the resumable path, state resident on the device) against
    roadsurf_run_batch: bit-identical outputs and status words -- plain forecast with sky-view points and a
    point that fails in the middle; a coupled run, whose window is indivisible; run-ahead chunks."""
    arrays, settings, params, _ = synth.make_case(40, 2, seed=350)
    arrays.tair[3, 100] = 333.0                                       # CheckValues fails point 3 at step 101
    ref = arrays.copy()
    st_ref = rslib.run_batch(ref, settings, params)
    for chunk in (1, 37):
        work = arrays.copy()
        st, launches = _stepwise(rslib, work, settings, params, chunk=chunk)
        for k in ref.out:
            assert np.array_equal(work.out[k], ref.out[k], equal_nan=True), (chunk, k)
        assert np.array_equal(st, st_ref)
        assert (launches >= settings.SimLen) if chunk == 1 else (launches < 12)
    assert st_ref[3] & rslib.ST_FAILED and (ref.out["TsurfOut"][3, 101:] == -9999.0).all()

    arrays, settings, params, _ = synth.make_case(33, 1, seed=351, analysis_hours=2, use_coupling=1, use_relaxation=1,
                                                   settings_kw=dict(coupling_minutes=60))
    ref = arrays.copy()
    st_ref = rslib.run_batch(ref, settings, params)
    work = arrays.copy()
    st, launches = _stepwise(rslib, work, settings, params)
    for k in ref.out:
        assert np.array_equal(work.out[k], ref.out[k], equal_nan=True), k
    assert np.array_equal(st, st_ref) and (st & rslib.ST_COUPLING_USED).all()
    window = 60 * 60 // 30
    assert settings.SimLen - window - 2 <= launches <= settings.SimLen - window + 2   # the window was one launch


def test_stepwise_single_point_like_the_fortran_main(rslib, oracle):
    """One point, one step per call, stop at failure: the call pattern of the Fortran main against the oracle."""
    arrays, settings, params, _ = synth.make_case(1, 1, seed=352, sky_view_fraction=1.0)
    arrays.SW[0, 60] = -50.0
    ref = arrays.copy()
    st_cpu, _ = oracle.run_batch(ref, settings, params)
    st, _ = _stepwise(rslib, arrays, settings, params)
    for k in ref.out:
        assert np.array_equal(arrays.out[k], ref.out[k], equal_nan=True), k
    assert st[0] == st_cpu[0] and (st[0] & rslib.ST_FAILED)


def _example2_arrays(oracle, arrays, rec, dt=30.0):
    """Per-step arrays as example2's AsciiSource would interpolate the raw records (oracle restatement)."""
    kinds = {"Rhz": 1, "prec": 2, "PrecPhase": 3}
    out = arrays.copy()
    for name in synth.RECORD_VARS:
        dst = getattr(out, name)
        for p in range(arrays.npoints):
            fill = -9999.0 if name == "PrecPhase" else -9999.9
            v = oracle.interpolate_example2(getattr(rec, name)[p], rec.record_step, dt, arrays.sim_len,
                                            kinds.get(name, 0), fill)
            dst[p] = v.astype(dst.dtype)
    return out


def test_example2_interpolation_mode_matches_the_oracle(rslib, oracle):
    """forcing_mode 2: coarse records interpolated by example2's rule (AsciiSource.cpp:223-345: per variable
    the nearest valid records, at most 180 minutes apart, whole-minute weights) in an expansion pass ahead
    of the step kernel -- against the oracle fed with arrays interpolated on the host by the restatement of
    that rule.  One chunk and several chunks (resumable path); the expansion pass itself is also compared
    value by value, for both rules."""
    import torch
    npts = 96
    arrays, settings, params, rec = synth.make_case(npts, 6, seed=360)
    rec.VZ[5:20, 3] = np.nan                     # one record missing: interpolated across a 120-minute gap
    rec.prec[10:30, 2:4] = -9999.0               # two missing: 180 minutes, still allowed
    rec.SW[40:44, 2:5] = np.nan                  # three missing: 240 minutes -> stays missing -> the point fails
    rec.Rhz[50:60, 4] = 140.0                    # clamped to 100
    rec.prec[61, 5] = 250.0                      # dropped (> 100): neighbours 4 and 6 bracket it
    ex2 = _example2_arrays(oracle, arrays, rec)
    ref = ex2.copy()
    st_cpu, _ = oracle.run_batch(ref, settings, params, nthreads=8)
    assert (st_cpu[40:44] & rslib.ST_BAD_INPUT).all() and not (st_cpu[:40] & rslib.ST_FAILED).any()
    rslib.set_model(settings, params)
    for expand_steps, state in ((0, False), (100, True)):
        db = rslib.DeviceBatch(npts, arrays.sim_len, n_records=rec.nrec, coarse=True, horizons=True, rule=2,
                               expand_steps=expand_steps, state=state)
        db.load_records(rec)
        db.time_fields.copy_(torch.from_numpy(arrays.time))
        db.load_local(arrays.local, arrays.local_horizons)
        db.run()
        torch.cuda.synchronize()
        got = db.outputs()
        for k in ref.out:
            same = (got[k] == ref.out[k]) | (np.isnan(got[k]) & np.isnan(ref.out[k]))
            # (the step executed on missing inputs is garbage on both sides, see the records-end test)
            fail_step = np.argmax(ex2.SW < -9000, axis=1)
            for p in range(40, 44):
                same[p, fail_step[p]] = True
            assert same.all(), (expand_steps, k, np.argwhere(~same)[:5].tolist())
        assert np.array_equal(db.status.cpu().numpy()[:npts], st_cpu)
    # the expansion pass, value by value
    full = db.expand(2, 1, arrays.sim_len).cpu().numpy()
    for v, name in enumerate(synth.RECORD_VARS):
        want = getattr(ex2, name).astype(np.float64)
        assert np.array_equal(full[:, v, :npts].T, want, equal_nan=True), name
    fields = synth.interpolate_records(rec, arrays.sim_len)
    rule1 = db.expand(1, 1, arrays.sim_len).cpu().numpy()
    for v, name in enumerate(synth.RECORD_VARS):
        ok = ~np.isnan(fields[name].astype(np.float64))           # (NaN records: example1's rule has no NaN notion)
        assert np.array_equal(rule1[:, v, :npts].T[ok], fields[name].astype(np.float64)[ok]), name


def test_solar_geometry_decisions_equal_the_hosts_over_a_year(rslib, oracle):
    """The solar geometry is the one place where the kernel still calls the device library's sin / cos / acos /
    atan2 (exp and log mirror the host libm).  What the model takes from it are two decisions: the horizon index
    NINT(azimuth) and `horizon > elevation` (src/ModRadiation.f90:41-49).  A year of half-hourly times x 600
    locations over the reference's lat/lon box (1.05e7 evaluations): sun-up / sun-down pattern and NINT(azimuth)
    must equal the oracle's everywhere; elevation to 1e-12 degrees (a shadow decision could only flip for a horizon
    angle within that distance of the elevation; measured 4e-14) and azimuth to 1e-7 degrees (acos is ill
    conditioned near due north / south; measured 7e-9, against the 0.5 degree that would move an index)."""
    import datetime as dt
    import torch
    n, npts = 17520, 600
    tf = synth.time_axis(dt.datetime(2019, 1, 1), n, 1800.0)
    rng = np.random.Generator(np.random.PCG64(5))
    lat, lon = rng.uniform(59.8, 69.9, npts), rng.uniform(20.0, 31.0, npts)
    e_cpu, a_cpu = oracle.sun_position_batch(tf, lat, lon, nthreads=8)
    e_gpu, a_gpu = rslib.sun_position(torch.from_numpy(tf).cuda(), torch.from_numpy(lat).cuda(), torch.from_numpy(lon).cuda())
    e_gpu, a_gpu = e_gpu.cpu().numpy(), a_gpu.cpu().numpy()
    assert not np.isnan(e_cpu).any() and not np.isnan(e_gpu).any()          # nobody would `stop`
    up_cpu, up_gpu = e_cpu > 0, e_gpu > 0
    assert np.array_equal(up_cpu, up_gpu)
    assert 0.25 < up_cpu.mean() < 0.6
    assert np.array_equal(np.rint(a_cpu[up_cpu]), np.rint(a_gpu[up_cpu])), "a horizon index differs"
    de, da = np.abs(e_cpu - e_gpu)[up_cpu].max(), np.abs(a_cpu - a_gpu)[up_cpu].max()
    print(f"solar geometry, {up_cpu.sum()} sun-up evaluations: max |d elevation| = {de:.2e} deg, max |d azimuth| = {da:.2e} deg, "
          f"bit-identical elevations: {(e_cpu == e_gpu)[up_cpu].mean():.4f}")
    assert de < 1e-12 and da < 1e-7


def test_guard_planes_around_every_written_tensor_stay_intact(rslib):
    """Stand-in for compute-sanitizer (closed on this pool): out, state, scratch, status, solar table and the
    expansion work space are carved out of larger buffers filled with a sentinel; coupled run with lane compaction
    (index lists), ragged point count, point order, chunked launches, forcing_mode 2 -- no write may land outside."""
    import torch
    SENT, G = -7.25e300, 4096

    def guarded(t):
        buf = torch.full((t.numel() + 2 * G,), SENT if t.dtype == torch.float64 else -77, dtype=t.dtype, device=t.device)
        view = buf[G:G + t.numel()].view(t.shape)
        view.copy_(t)
        return buf, view

    def intact(bufs):
        for name, buf in bufs.items():
            s = SENT if buf.dtype == torch.float64 else -77
            assert bool((buf[:G] == s).all()) and bool((buf[-G:] == s).all()), f"write outside {name}"

    npts = 1000 + 7
    arrays, settings, params, rec = synth.make_case(npts, 4, seed=370, analysis_hours=3, use_coupling=1, use_relaxation=1,
                                                    obs_bias=False, settings_kw=dict(coupling_minutes=60))
    rslib.set_model(settings, params)
    for mode in ("compaction+order", "chunks", "example2"):
        db = rslib.DeviceBatch(npts, arrays.sim_len, n_records=rec.nrec, coarse=True, horizons=True, coupling=True, state=True,
                               out_stride=7, rule=2 if mode == "example2" else 1, expand_steps=arrays.sim_len)
        db.load_records(rec)
        db.time_fields.copy_(torch.from_numpy(arrays.time))
        db.load_local(arrays.local, arrays.local_horizons)
        bufs = {}
        for name in ("out", "state", "scratch", "status", "solar") + (("expand_workspace",) if mode == "example2" else ()):
            bufs[name], view = guarded(getattr(db, name))
            setattr(db, name, view)
        if mode == "compaction+order":
            db.build_order()
            db.run()
        elif mode == "chunks":
            db.coupling_window_end = 0
            wend = arrays.local[0].couplingIndexI
            db.run(step_begin=1, step_end=wend + 1)
            db.run(step_begin=wend + 2, step_end=arrays.sim_len)
        else:
            db.coupling_window_end = 0
            db.run()
        torch.cuda.synchronize()
        intact(bufs)
        assert (db.status[:npts] & rslib.ST_NOT_RUN).sum() == 0


def test_opt_in_write_back_reproduces_the_references_input_mutations(rslib, oracle):
    """The reference mutates its INPUT arrays (VZ(1) clamp, SW_dir <= SW per visited step, sky-view rewrite of
    SW / SW_dir / LW per executed step, restored and re-applied by coupling re-runs).  With the option
    "write_back_inputs" the caller's arrays after roadsurf_run_batch equal the oracle's after its run, bit for
    bit; without it (the default) they are untouched."""
    arrays, settings, params, _ = synth.make_case(200, 3, seed=380, analysis_hours=3, use_coupling=1, use_relaxation=1,
                                                   sky_view_fraction=0.5, settings_kw=dict(coupling_minutes=60))
    arrays.VZ[:50, 0] = 0.1                        # clamped to 0.4 by Initialization
    arrays.SW_dir[:, 100:140] += 500.0             # above SW: clamped by CheckValues
    arrays.tair[7, 300] = 500.0                    # point 7 fails at step 301: nothing after it is touched
    ref, untouched = arrays.copy(), arrays.copy()
    st_cpu, _ = oracle.run_batch(ref, settings, params, nthreads=8)
    rslib.run_batch(untouched, settings, params)
    for k in ("VZ", "SW", "SW_dir", "LW"):
        assert np.array_equal(getattr(untouched, k), getattr(arrays, k)), k
    rslib.set_option("write_back_inputs", 1)
    try:
        st = rslib.run_batch(arrays, settings, params)
    finally:
        rslib.set_option("write_back_inputs", 0)
    assert np.array_equal(st, st_cpu)
    for k in ref.out:
        assert np.array_equal(arrays.out[k], ref.out[k], equal_nan=True), k
    changed = 0
    for k in ("VZ", "SW", "SW_dir", "LW", "tair", "LW_net", "prec"):
        assert np.array_equal(getattr(arrays, k), getattr(ref, k), equal_nan=True), k
        changed += int((getattr(arrays, k) != getattr(untouched, k)).sum())
    assert changed > 1000
    assert np.array_equal(arrays.SW_dir[7, 301:], untouched.SW_dir[7, 301:])      # beyond the failure: as given


def test_latency_body_and_throughput_body_give_identical_results(rslib, oracle):
    """The step kernel has two bodies (option "latency_body"): grids of at most one block per SM run the latency
    body by default.  Both, forced in turn on the same coupled + sky-view case, must equal the oracle bit for bit --
    so neither body is only covered by the grid sizes the other tests happen to use."""
    arrays, settings, params, _ = synth.make_case(300, 12, seed=77, analysis_hours=6, use_coupling=1, use_relaxation=1)
    ref = arrays.copy()
    st_ref, _ = oracle.run_batch(ref, settings, params, nthreads=8)
    try:
        for spread in (0, 1):       # one point per warp (the default for batches this small) or 32
            rslib.set_option("spread_small", spread)
            for mode in (0, 1, -1):
                rslib.set_option("latency_body", mode)
                work = arrays.copy()
                st = rslib.run_batch(work, settings, params)
                assert np.array_equal(st, st_ref), (spread, mode)
                _assert_parity(compare(work.out, ref.out))
                li = rslib.last_launch()
                assert (li["regs_per_thread"] > 168) == (mode != 0), (mode, li)      # the latency body has no register cap
                assert li["grid"] == (80 if spread else 3), li                       # 320 slots: 4 or 128 points per block
    finally:
        rslib.set_option("latency_body", -1)
        rslib.set_option("spread_small", 1)


def test_other_time_steps_are_bit_identical_too(rslib, oracle):
    """DTSecs enters the per-run constants (layer update factors, correctly rounded reciprocals, the coupling span,
    wear and evaporation per step): 60 s and 20 s, with and without coupling / relaxation, against the oracle."""
    for dt, kw in ((60.0, dict(analysis_hours=3, use_coupling=1, use_relaxation=1, settings_kw=dict(coupling_minutes=60))),
                   (20.0, dict()),
                   (120.0, dict(analysis_hours=2, use_relaxation=1))):
        arrays, settings, params, _ = synth.make_case(96, 6, seed=int(dt), dt=dt, **kw)
        assert settings.DTSecs == dt
        r, st_gpu, st_cpu, _, _ = _run_both(rslib, oracle, arrays, settings, params)
        _assert_parity(r)
        assert np.array_equal(st_gpu, st_cpu), dt


def test_extreme_inputs_are_bit_identical_too(rslib, oracle):
    """Storage caps and snow / ice transitions under heavy precipitation, a 40-degree surface, six places around
    the globe on a leap day, the turn of the year (tests/extreme_cases.py; the two CPU restatements agree on them)."""
    from extreme_cases import extreme_cases
    for name, arrays, settings, params in extreme_cases():
        r, st_gpu, st_cpu, _, _ = _run_both(rslib, oracle, arrays, settings, params)
        assert r["bit_identical"] and np.array_equal(st_gpu, st_cpu), (name, r)


def test_randomised_parameters_and_settings_fuzz(rslib, oracle):
    """Twelve random configurations: every one of the 69 InputParameters scaled by a random factor in [0.8, 1.25]
    (sign-preserving; the integer-valued hours and missing-value markers kept), random layer count, output depth,
    coupling window and decay, relaxation on / off -- GPU against the oracle, bit for bit, status words included."""
    rng = np.random.default_rng(20191207)
    keep = {"NightOn", "NightOff", "MissValI", "MissValR"}
    for trial in range(12):
        base = abi.default_parameters(30.0)
        over = {n: getattr(base, n) * rng.uniform(0.8, 1.25) for n, _ in base._fields_ if n not in keep}
        params = abi.default_parameters(30.0, **over)
        nl = int(rng.choice([15, 15, 6, 10, 24]))
        coupled = bool(rng.integers(0, 2))
        skw = dict(coupling_minutes=int(rng.choice([30, 60, 180])), coupling_effect_reduction=float(rng.choice([3600.0, 14400.0])))
        if rng.integers(0, 3) == 0:
            skw["tsurf_output_depth"] = float(rng.choice([0.0, 0.02, 0.3]))
        arrays, settings, _, _ = synth.make_case(64, 4, seed=100 + trial, nlayers=nl, analysis_hours=4 if coupled else 0,
                                                 use_coupling=int(coupled), use_relaxation=int(rng.integers(0, 2)) if coupled else 0,
                                                 sky_view_fraction=float(rng.choice([0.0, 0.3, 1.0])), settings_kw=skw)
        r, st_gpu, st_cpu, _, _ = _run_both(rslib, oracle, arrays, settings, params)
        assert r["bit_identical"] and np.array_equal(st_gpu, st_cpu), (trial, nl, coupled, skw, r)


def test_irregular_record_grid_with_missing_records_inside(rslib, oracle):
    """Coarse mode on an IRREGULAR record grid (gaps of 1 step to several hours, a record exactly on a model step and
    in between) with records missing inside the series: optional variables (TSurfObs, PrecPhase, LW_net / SW_dir of
    points without sky view) stay missing between their neighbours, a missing required value stops the point at the
    first step that sees it -- the device-side interpolation against the oracle on host-interpolated arrays."""
    import torch
    arrays, settings, params, rec = synth.make_case(96, 12, seed=330, sky_view_fraction=0.5)
    rng = np.random.default_rng(9)
    # an irregular subset of model steps as record times: keep the hourly values but move the times
    rs = np.unique(np.concatenate([[0, 1, 2, 121, 500, 501], rng.integers(3, arrays.sim_len + 200, size=rec.nrec - 8),
                                   [arrays.sim_len + 300, arrays.sim_len + 301]])).astype(np.int32)[:rec.nrec]
    assert len(rs) == rec.nrec and rs[-1] > arrays.sim_len - 1
    irr = synth.Records(96, rec.nrec)
    for v in synth.RECORD_VARS:
        setattr(irr, v, getattr(rec, v).copy())
    irr.lat, irr.lon, irr.sky_view, irr.horizons = rec.lat, rec.lon, rec.sky_view, rec.horizons
    irr.record_step = rs
    irr.TSurfObs[:, 3:] = -9999.9                       # observations only at the very start
    irr.PrecPhase[::3, 4] = -9999                       # unknown phase for one record: interpretation from Tair
    irr.tair[5, 6] = -9999.9                            # point 5: a required value missing inside the series
    irr.LW[7, rec.nrec // 2] = -9999.9                  # point 7: likewise, later
    fields = synth.interpolate_records(irr, arrays.sim_len)
    ref = arrays.copy()
    for name, val in fields.items():
        getattr(ref, name)[...] = val
    st_cpu, _ = oracle.run_batch(ref, settings, params, nthreads=4)
    assert (st_cpu[[5, 7]] & rslib.ST_BAD_INPUT).all() and (np.delete(st_cpu, [5, 7]) & rslib.ST_FAILED == 0).all()
    rslib.set_model(settings, params)
    db = rslib.DeviceBatch(96, arrays.sim_len, n_records=irr.nrec, coarse=True, horizons=True)
    db.load_records(irr)
    db.time_fields.copy_(torch.from_numpy(arrays.time))
    db.load_local(arrays.local, arrays.local_horizons)
    db.run()
    torch.cuda.synchronize()
    got = db.outputs()
    assert np.array_equal(db.status.cpu().numpy()[:96], st_cpu)
    for k in ref.out:
        same = (got[k] == ref.out[k]) | (np.isnan(got[k]) & np.isnan(ref.out[k]))
        for p in (5, 7):                                # the one step executed on missing values (see the test above)
            t = int(np.argmax(ref.out[k][p] == -9999.0)) - 1
            same[p, t] |= np.isclose(got[k][p, t], ref.out[k][p, t], rtol=1e-6, atol=0.0, equal_nan=True)
        assert same.all(), (k, np.argwhere(~same)[:5].tolist())


def test_batch_sizes_across_the_points_per_warp_choices(rslib, oracle):
    """rs_launch_run maps small batches to 1, 2, 4, 8 or 16 points per warp (the other lanes are ghosts) and larger
    ones to 32: coupled batches whose sizes land in each of those choices -- and whose compacted coupling passes
    therefore read their index lists through each mapping -- against the oracle, bit for bit."""
    for npts in (31, 593, 1300, 2500, 5000, 9500, 20000):
        arrays, settings, params, _ = synth.make_case(npts, 2, seed=500 + npts, analysis_hours=2, use_coupling=1,
                                                       use_relaxation=1, settings_kw=dict(coupling_minutes=45))
        r, st_gpu, st_cpu, _, _ = _run_both(rslib, oracle, arrays, settings, params)
        assert r["bit_identical"] and np.array_equal(st_gpu, st_cpu), (npts, r)
    assert (st_gpu & rslib.ST_COUPLING_USED).any()
