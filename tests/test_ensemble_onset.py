"""Ensemble event onset (include/roadsurf_b200.h part 3, after RsEnsembleAreas): the probability that an event has
begun by each member slot.  For station p, event e, member m and slot s < S, the member is valid when every plane the
conditions name holds a valid value at every slot of [0, s], and hits when it is valid and the conjunction holds at one
slot or more of [0, s]; onset[e][s][p] = hits / valid, -9999.0 where no member is valid.  Areas: valid at every station
of the area, a hit at one station or more.  This equals the event (area event) rule at slot 0 with window s + 1."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from parity import same_bits
from roadsurf_b200 import abi, lib, synth
from test_ensemble import QUANTILES, _Case, _host_case
from test_ensemble_areas import FREEZE2, _bad_areas, _random_areas, _tiny, areas_reference
from test_ensemble_events import (DEWDEFICIT, OPS, ROAD_EVENTS, TS, WATER, _bad_specs, _device_ensemble,
                                  _random_events, events_reference)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RS_ERR_BAD_ARGUMENT = -2


# ---- NumPy restatement ------------------------------------------------------------------------------------------

def first_slots(member_out, npoints, members, events, n_slots=None):
    """Per (event, station, member): X, the first slot where a named plane is invalid (S if none), and O, the first
    slot before X where the conditions all hold (S if none); both [n_events, P, M]."""
    S = member_out.shape[1] if n_slots is None else n_slots
    x = member_out[:, :S, :npoints * members].reshape(member_out.shape[0], S, npoints, members)
    X = np.full((len(events), npoints, members), S)
    O = np.full((len(events), npoints, members), S)
    for j, (conds, _) in enumerate(events):
        bad = ~np.logical_and.reduce([(x[pl] == x[pl]) & (x[pl] > -9000.0) for pl, _, _ in conds])    # [S, P, M]
        with np.errstate(invalid="ignore"):
            both = np.logical_and.reduce([OPS[op](x[pl], v) for pl, op, v in conds])
        X[j] = np.where(bad.any(axis=0), bad.argmax(axis=0), S)
        before = both & (np.arange(S)[:, None, None] < X[j])
        O[j] = np.where(before.any(axis=0), before.argmax(axis=0), S)
    return O, X


def _ratio(valid, hit):
    n, c = valid.sum(axis=-1), hit.sum(axis=-1)
    return np.where(n == 0, -9999.0, c / np.maximum(n, 1))


def onset_reference(member_out, npoints, members, events, n_slots=None):
    """onset [n_events, S, P]: valid(s) <=> X > s, hit(s) <=> valid and O <= s."""
    O, X = first_slots(member_out, npoints, members, events, n_slots)
    S = member_out.shape[1] if n_slots is None else n_slots
    s = np.arange(S)[None, :, None, None]
    valid = X[:, None] > s
    return _ratio(valid, valid & (O[:, None] <= s))


def area_onset_reference(member_out, npoints, members, events, areas, n_slots=None):
    """area_onset [n_events, S, n_areas]: per member the minimum X and the minimum O over the area's stations."""
    O, X = first_slots(member_out, npoints, members, events, n_slots)
    S = member_out.shape[1] if n_slots is None else n_slots
    s = np.arange(S)[None, :, None]
    out = np.zeros((len(events), S, len(areas)))
    for a, st in enumerate(areas):
        st = np.asarray(st)
        xa, oa = X[:, st].min(axis=1)[:, None], O[:, st].min(axis=1)[:, None]       # [E, 1, M]
        valid = xa > s
        out[..., a] = _ratio(valid, valid & (oa <= s))
    return out


def test_restatement_known_answers():
    """Hand-computed on the 3 stations x 2 members x 4 slots of test_ensemble_areas: station 0's member 1 is cut off
    from slot 2 by a NaN; station 2 did not run, so every area holding it is -9999.0."""
    x = _tiny()
    areas = [[0], [1], [0, 1], [2], [1, 2]]
    O, X = first_slots(x, 3, 2, [FREEZE2])
    assert X[0].tolist() == [[4, 2], [4, 4], [0, 0]] and O[0].tolist() == [[1, 4], [2, 0], [4, 4]]
    on = onset_reference(x, 3, 2, [FREEZE2])[0]
    assert list(on[:, 0]) == [0.0, 0.5, 1.0, 1.0]
    assert list(on[:, 1]) == [0.5, 0.5, 1.0, 1.0]
    assert (on[:, 2] == -9999.0).all()
    ar = area_onset_reference(x, 3, 2, [FREEZE2], areas)[0]
    assert same_bits(ar[:, 0], on[:, 0]) and same_bits(ar[:, 1], on[:, 1])
    assert list(ar[:, 2]) == [0.5, 1.0, 1.0, 1.0]      # member 1 hits at station 1 at slot 0, member 0 at station 0 at 1
    assert (ar[:, 3] == -9999.0).all() and (ar[:, 4] == -9999.0).all()


def _identity_tensor(seed, P=12, M=7, S=30):
    rng = np.random.Generator(np.random.PCG64(seed))
    x = np.round(rng.normal(0.0, 1.0, (3, S, P * M + 4)), 1) + 0.0
    x[rng.random(x.shape) < 0.01] = np.nan
    x[:, :, 2 * M:3 * M] = -9999.0
    return x


def test_restatement_is_the_event_rule_over_the_growing_window():
    """onset[e][s] equals the station events (and area events) at slot 0 with window s + 1, for every s."""
    P, M, S = 12, 7, 30
    x = _identity_tensor(11, P, M, S)
    conds = [[(0, "<", 0.0), (1, ">", -0.5)], [(2, ">=", 0.5)], [(1, "<=", 0.0), (0, ">", 0.1), (2, "<", 1.0)]]
    areas = [[0], [3, 4, 9], list(range(P)), [1, 2], [5, 6, 7, 8, 10, 11]]
    on = onset_reference(x, P, M, [(c, 1) for c in conds])
    ar = area_onset_reference(x, P, M, [(c, 1) for c in conds], areas)
    for s in range(S):
        ev = [(c, s + 1) for c in conds]
        assert same_bits(on[:, s], events_reference(x, P, M, ev)[:, 0]), s
        assert same_bits(ar[:, s], areas_reference(x, P, M, ev, areas)[:, 0]), s
    assert ((on > 0.0) & (on < 1.0)).any() and (on == -9999.0).any()


def _prototype_argtypes(name):
    """The ctypes argument list that the prototype of `name` in the header asks for."""
    with open(os.path.join(ROOT, "include", "roadsurf_b200.h")) as f:
        text = f.read()
    args = re.search(r"\bint\s+" + name + r"\(([^)]*)\);", text).group(1)
    out = []
    for a in (" ".join(a.split()) for a in args.split(",")):
        if a.startswith("int ") and "*" not in a:
            out.append(C.c_int)
        elif a.startswith("const RsHostBatch*"):
            out.append(C.POINTER(lib.RsHostBatch))
        elif a.startswith("const RsEnsembleStatsSpec*"):
            out.append(C.POINTER(lib.RsEnsembleStatsSpec))
        elif a.startswith("const RsEnsembleAreas*"):
            out.append(C.POINTER(lib.RsEnsembleAreas))
        elif a.startswith("const InputSettings*"):
            out.append(C.POINTER(abi.InputSettings))
        elif a.startswith("const InputParameters*"):
            out.append(C.POINTER(abi.InputParameters))
        else:
            assert re.match(r"(const )?(double|int|void)\* \w+$", a), a
            out.append(C.c_void_p)
    return out


def test_ctypes_argument_lists_match_the_header():
    handle = lib.load()
    for name in ("roadsurf_ensemble_onset", "roadsurf_run_ensemble_host_soa_onset"):
        assert name in lib.EXPORTS
        want = _prototype_argtypes(name)
        assert list(getattr(handle, name).argtypes) == want, name
    assert len(_prototype_argtypes("roadsurf_ensemble_onset")) == 12
    assert len(_prototype_argtypes("roadsurf_run_ensemble_host_soa_onset")) == 16
    assert b" 0.4 " in handle.roadsurf_version()


def test_bad_arguments_are_rejected_before_device_work():
    """Through roadsurf_ensemble_onset and roadsurf_run_ensemble_host_soa_onset (a well-placed fork): onset outputs
    with a spec without events, area_onset without areas, areas without an area output, the device entry without
    outputs, every malformed area set and every malformed spec return RS_ERR_BAD_ARGUMENT with a message."""
    handle = lib.load()
    P, M = 3, 4
    member_out = np.zeros((lib.O_NVAR, 5, 32))
    good = lib.ensemble_areas([[0, 2], [1]])
    buf = np.zeros(1 << 12)
    b = buf.ctypes.data
    spec = lib.stats_spec(events=[([(TS, "<", 0.0), (WATER, ">", 0.1)], 3)])
    no_events = lib.stats_spec(QUANTILES, [(TS, "<", 0.0)])

    def device(sp, onset, areas, area_onset):
        return handle.roadsurf_ensemble_onset(member_out.ctypes.data, lib.O_NVAR, 5, 32, P, M, C.byref(sp), onset, 32,
                                              None if areas is None else C.byref(areas), area_onset, None)
    dcases = [(spec, None, None, None, b"both NULL"), (spec, None, good, None, b"both NULL"),
              (spec, b, good, None, b"null area pointer"), (spec, None, None, b, b"null area pointer"),
              (no_events, b, None, None, b"at least one event"), (no_events, None, good, b, b"at least one event")]
    dcases += [(spec, b, a, b, what) for a, what in _bad_areas(P) if a is not None]
    dcases += [(sp, b, None, None, what) for sp, what in _bad_specs(lib.O_NVAR)]
    for sp, onset, areas, area_onset, what in dcases:
        assert device(sp, onset, areas, area_onset) == RS_ERR_BAD_ARGUMENT, what
        assert what in handle.roadsurf_last_error(), what
    # ld < npoints with onset planes
    assert handle.roadsurf_ensemble_onset(member_out.ctypes.data, lib.O_NVAR, 5, 32, P, M, C.byref(spec), b, 2, None,
                                          None, None) == RS_ERR_BAD_ARGUMENT

    base, pa, settings, params, start = _host_case(P=P)
    F = 2 * 120 + 2
    forcing = np.ascontiguousarray(np.stack([getattr(base, v).T for v in synth.RECORD_VARS], axis=1))
    local = np.zeros((lib.L_NLOCAL, P))
    r_f = lib.fork_record(base.record_step, F)
    mrec = np.zeros((base.nrec - r_f - 1, 11, P * M))
    hb = lib.RsHostBatch(npoints=P, sim_len=pa.sim_len, forcing_mode=1, n_records=base.nrec, nvar=11, out_stride=1,
                         forcing=forcing.ctypes.data, record_step=base.record_step.ctypes.data,
                         time_fields=pa.time.ctypes.data, local=local.ctypes.data)
    stats, prob = np.zeros(1 << 16), np.zeros(1 << 16)

    def host(sp, areas, area_prob, onset, area_onset):
        return handle.roadsurf_run_ensemble_host_soa_onset(
            C.byref(hb), mrec.ctypes.data, M, F, None, C.byref(sp), stats.ctypes.data, prob.ctypes.data, None, None,
            None if areas is None else C.byref(areas), area_prob, onset, area_onset, C.byref(settings), C.byref(params))
    hcases = [(spec, good, None, None, None, b"null area pointer"), (spec, good, None, b, None, b"null area pointer"),
              (spec, None, b, None, None, b"null area pointer"), (spec, None, None, b, b, b"null area pointer"),
              (no_events, None, None, b, None, b"at least one event"),
              (no_events, good, None, None, b, b"at least one event"), (no_events, good, b, None, None, b"at least one event")]
    hcases += [(spec, a, None, b, b, what) for a, what in _bad_areas(P) if a is not None]
    hcases += [(spec, a, b, None, None, what) for a, what in _bad_areas(P) if a is not None]
    hcases += [(sp, None, None, b, None, what) for sp, what in _bad_specs(lib.O_NVAR)]
    for sp, areas, area_prob, onset, area_onset, what in hcases:
        assert host(sp, areas, area_prob, onset, area_onset) == RS_ERR_BAD_ARGUMENT, what
        assert what in handle.roadsurf_last_error(), what
    if handle.roadsurf_device_count() == 0:
        # good outputs pass the checks and then find no device
        assert host(spec, good, None, b, b) == -1 and host(spec, None, None, b, None) == -1


# ---- GPU --------------------------------------------------------------------------------------------------------

def _kernel_tensor(M, seed):
    """The tensors of test_events_kernel_equals_the_restatement: 2 003 slots, NaN and -9999.0 holes in half the lanes,
    station 3 all missing."""
    rng = np.random.Generator(np.random.PCG64(seed + M))
    P, S, out_nvar = min(150, max(5, 2400 // M)), 2003, lib.O_NVAR
    ldm = (P * M + 31) // 32 * 32
    x = np.round(rng.normal(0.0, 2.0, (out_nvar, S, ldm)), 1) + 0.0
    holes = (rng.random(x.shape) < 0.0005) & (rng.random(ldm) < 0.5)
    x[holes & (rng.random(x.shape) < 0.5)] = np.nan
    x[holes & ~np.isnan(x)] = -9999.0
    x[:, :, 3 * M:4 * M] = -9999.0
    return rng, x, P, S


@pytest.mark.gpu
@pytest.mark.parametrize("M", [1, 2, 31, 51, 128])
def test_onset_kernels_equal_the_restatement(rslib, M):
    """Eight events with all four comparisons and thresholds drawn from member values (ties), one of them never met
    (below the plane's minimum); bit for bit against the restatement, per station and per area."""
    import torch
    rng, x, P, S = _kernel_tensor(M, 300)
    events, _ = _random_events(rng, x, P, M, S)
    v3 = x[3, :S, :P * M]
    events[6] = ([(3, "<", float(v3[(v3 == v3) & (v3 > -9000.0)].min()))], 1)
    areas = _random_areas(rng, P, 3)
    want = onset_reference(x, P, M, events)
    want_a = area_onset_reference(x, P, M, events, areas)
    xd = torch.from_numpy(x).cuda()
    spec = lib.stats_spec((), (), events)
    on, ar = rslib.ensemble_onset(xd, P, M, spec, rslib.ensemble_areas(areas))
    on, ar = on.cpu().numpy(), ar.cpu().numpy()
    assert on.shape == (len(events), S, P) and ar.shape == (len(events), S, len(areas))
    for j in range(len(events)):
        assert same_bits(on[j], want[j]), (M, j)
        assert same_bits(ar[j], want_a[j]), (M, j)
    only, none = rslib.ensemble_onset(xd, P, M, spec)
    assert none is None and same_bits(only.cpu().numpy(), on)
    assert (want[6] == 0.0).any() and (want == -9999.0).any() and (M == 1 or ((want > 0.0) & (want < 1.0)).any())
    assert (want[:, -1] == 0.0).any()                  # stations that never hit


@pytest.mark.gpu
def test_onset_equals_the_merged_event_kernels_at_slot_zero(rslib):
    """onset[e][s] equals roadsurf_ensemble_stats' event plane and roadsurf_ensemble_area_events at slot 0 of the
    same conditions with window s + 1, around the 64-slot tiles of the area kernels and at a random sample of s;
    several specs of 8 events."""
    import torch
    rng = np.random.Generator(np.random.PCG64(77))
    P, M, S = 70, 31, 260
    x = np.round(rng.normal(0.5, 2.0, (lib.O_NVAR, S, P * M)), 1) + 0.0
    x[(rng.random(x.shape) < 0.0004)] = np.nan
    x[:, :, 5 * M:6 * M] = -9999.0
    xd = torch.from_numpy(x).cuda()
    area_lists = _random_areas(rng, P, 5)
    areas = rslib.ensemble_areas(area_lists)
    sample = sorted(set([0, 1, 62, 63, 64, 65, S - 1] + rng.choice(S, 6, replace=False).tolist()))
    for spec_seed in range(3):
        events, _ = _random_events(np.random.Generator(np.random.PCG64(spec_seed)), x, P, M, S)
        on, ar = rslib.ensemble_onset(xd, P, M, lib.stats_spec((), (), events), areas)
        on, ar = on.cpu().numpy(), ar.cpu().numpy()
        for s in sample:
            sp = lib.stats_spec((), (), [(c, s + 1) for c, _ in events])
            _, prob = rslib.ensemble_stats(xd, P, M, sp)
            area_prob = rslib.ensemble_area_events(xd, P, M, sp, areas)
            assert same_bits(on[:, s], prob.cpu().numpy()[:, 0]), (spec_seed, s)
            assert same_bits(ar[:, s], area_prob.cpu().numpy()[:, 0]), (spec_seed, s)
        assert ((on > 0.0) & (on < 1.0)).any()


@pytest.mark.gpu
def test_device_entry_then_onset_equals_the_restatement(rslib):
    """roadsurf_run_ensemble_device with out_nvar = RS_O_NVAR_EXT (coarse records, coupling + relaxation), then
    roadsurf_ensemble_onset on its member_out, hoar-frost events on the dew-point-deficit plane included."""
    P, M = 60, 5
    c = _Case(P, M, 3, 6, seed=4606)
    spec = lib.stats_spec(QUANTILES, [(TS, "<", 0.0)], ROAD_EVENTS)
    assert any(cd[0] == DEWDEFICIT for conds, _ in ROAD_EVENTS for cd in conds)
    ens = _device_ensemble(rslib, c, spec)
    ens.run()
    area_lists = [[7], [0, 1, 2, 3], list(range(0, P, 3)), list(range(P)), [59, 12, 33, 12]]
    on, ar = rslib.ensemble_onset(ens.member_out, P, M, spec, rslib.ensemble_areas(area_lists))
    mo = ens.member_out.cpu().numpy()
    want = onset_reference(mo, P, M, ROAD_EVENTS, ens.n_slots)
    assert same_bits(on.cpu().numpy()[:, :ens.n_slots], want)
    assert same_bits(ar.cpu().numpy()[:, :ens.n_slots], area_onset_reference(mo, P, M, ROAD_EVENTS, area_lists,
                                                                              ens.n_slots))
    assert ((want > 0.0) & (want < 1.0)).any()


@pytest.mark.gpu
def test_host_entry_onset_in_station_chunks(rslib):
    """roadsurf_run_ensemble_host_soa_onset in one and in eight station chunks, areas straddling the chunks: onset and
    area_onset equal the device entry on the device ensemble's member_out; stats, prob and area_prob are bitwise those
    of the call without onset; d2h_bytes grows by exactly onset and area_onset; the onset kernels add two launches per
    chunk and one; an onset-only call (prob and area_prob NULL) runs no events or area event kernel."""
    P, M = 50, 6
    c = _Case(P, M, 3, 6, seed=4707)
    events = [e for e in ROAD_EVENTS if all(cd[0] < lib.O_NVAR for cd in e[0])]
    spec = lib.stats_spec(QUANTILES, [(TS, "<", 0.0)], events)
    ens = _device_ensemble(rslib, c, spec, extended=False)
    ens.run()
    area_lists = [[0], [49], [5, 6, 7, 8], list(range(3, 30)), list(range(P)), [48, 1, 20, 34, 6, 13],
                  list(range(0, P, 7)), [44, 45, 46, 47, 48, 49, 0]]
    areas = rslib.ensemble_areas(area_lists)
    want_on, want_ar = rslib.ensemble_onset(ens.member_out, P, M, spec, areas)
    want_on, want_ar = want_on.cpu().numpy(), want_ar.cpu().numpy()
    mo = ens.member_out.cpu().numpy()
    assert same_bits(want_on, onset_reference(mo, P, M, events, ens.n_slots))
    assert same_bits(want_ar, area_onset_reference(mo, P, M, events, area_lists, ens.n_slots))
    sh = ens.shared
    forcing = sh.forcing[:, :, :P].cpu().numpy().copy()
    local = sh.local[:, :P].cpu().numpy().copy()
    hor = sh.horizons[:, :P].cpu().numpy().copy()
    mrec = synth.member_record_tensor(c.mrecs, c.r_f)
    A, E = len(area_lists), len(events)

    def run(**kw):
        res = rslib.run_ensemble_host_soa(c.settings, c.params, forcing, c.base.record_step.astype(np.int32),
                                          c.pa.time, local, mrec, M, c.F, spec, horizons=hor, out_stride=60,
                                          coupling_window_end=sh.coupling_window_end,
                                          latest_obs_index=np.full(P, c.forecast_step + 1, dtype=np.int32), **kw)
        return res, rslib.last_batch_stats()
    for cap in (0, 7 * M):
        rslib.set_option("max_points_per_device_batch", cap)
        try:
            plain, st0 = run(areas=areas)
            res, st1 = run(areas=areas, onset=True)
            only, st2 = run(areas=areas, onset=True, prob=False, area_prob=False)
            station, st3 = run(onset=True)
        finally:
            rslib.set_option("max_points_per_device_batch", 0)
        groups = 1 if cap == 0 else 8
        assert st0["groups"] == st1["groups"] == st2["groups"] == st3["groups"] == groups
        n_m = res["stats"].shape[2]
        assert res["onset"].shape == (E, n_m, P) and res["area_onset"].shape == (E, n_m, A)
        for r in (res, only):
            assert same_bits(r["onset"], want_on), cap
            assert same_bits(r["area_onset"], want_ar), cap
            assert same_bits(r["stats"], plain["stats"])
        assert same_bits(station["onset"], want_on) and "area_onset" not in station
        assert same_bits(res["prob"], plain["prob"]) and same_bits(res["area_prob"], plain["area_prob"])
        assert "prob" not in only and "area_prob" not in only
        assert st1["d2h_bytes"] == st0["d2h_bytes"] + 8 * E * n_m * (P + A)
        assert st1["kernel_launches"] == st0["kernel_launches"] + 2 * groups + 1
        # no station events kernel (one per chunk), no area event kernels (one per chunk and one)
        assert st2["kernel_launches"] == st1["kernel_launches"] - groups - (groups + 1)
        assert st2["d2h_bytes"] == st1["d2h_bytes"] - 8 * (spec.n_prob * n_m * P + E * n_m * A)


@pytest.mark.gpu
def test_onset_is_written_inside_its_planes_only(rslib):
    """onset and area_onset pre-filled with a sentinel, longer than their planes and with ld > npoints; the spec's
    event array filled beyond n_events: exactly the first n_events planes, the npoints columns of each row and
    n_events * S * n_areas values are written."""
    import torch
    rng = np.random.Generator(np.random.PCG64(8))
    P, M, S, ld = 40, 9, 70, 64
    x = np.round(rng.normal(0.0, 2.0, (lib.O_NVAR, S, P * M)), 1) + 0.0
    events = [([(TS, "<", 0.0)], 2), ([(WATER, ">", 0.0), (TS, "<=", 1.0)], 5), ([(2, ">=", 0.0)], 1)]
    spec = lib.stats_spec((), (), events)
    spec.n_events = 2
    area_lists = [[0, 5], list(range(P)), [39]]
    areas = lib.ensemble_areas(area_lists)
    n_on, n_ar = 2 * S * ld, 2 * S * 3
    on = torch.full((n_on + 1000,), 777.0, dtype=torch.float64, device="cuda")
    ar = torch.full((n_ar + 1000,), 777.0, dtype=torch.float64, device="cuda")
    xd = torch.from_numpy(x).cuda()
    lib._check(lib.load().roadsurf_ensemble_onset(xd.data_ptr(), lib.O_NVAR, S, P * M, P, M, C.byref(spec),
                                                  on.data_ptr(), ld, C.byref(areas), ar.data_ptr(), None))
    torch.cuda.synchronize()
    o, a = on.cpu().numpy(), ar.cpu().numpy()
    assert (o[n_on:] == 777.0).all() and (a[n_ar:] == 777.0).all() and (a[:n_ar] != 777.0).all()
    planes = o[:n_on].reshape(2, S, ld)
    assert (planes[..., P:] == 777.0).all() and (planes[..., :P] != 777.0).all()
    assert same_bits(planes[..., :P], onset_reference(x, P, M, events[:2]))
    assert same_bits(a[:n_ar].reshape(2, S, 3), area_onset_reference(x, P, M, events[:2], area_lists))
