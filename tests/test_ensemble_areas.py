"""Ensemble area event probabilities (RsEnsembleAreas, include/roadsurf_b200.h part 3): the probability that an event
of the spec occurs anywhere in a group of stations.  For area A, event e, member m and slot s < S, the member is valid
when it is valid for e at s (the station rule of RsEnsembleEvent) at every station of A, and hits when it is valid and
hits e at s at one station of A or more; area_prob[e][s][a] = hits / valid, -9999.0 where no member is valid."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from parity import same_bits
from roadsurf_b200 import lib, synth
from test_ensemble import QUANTILES, _Case, _host_case
from test_ensemble_events import (DEWDEFICIT, ROAD_EVENTS, TS, WATER, _bad_specs, _device_ensemble, _random_events,
                                  events_reference)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RS_ERR_BAD_ARGUMENT = -2


# ---- NumPy restatement ------------------------------------------------------------------------------------------

def member_outcomes(member_out, npoints, members, events, n_slots=None):
    """Per member: valid, hit [n_events, S, P, M] by the station rule.  events_reference over one-member "stations"
    (every lane its own station) gives 1.0 where the member hits, 0.0 where it is valid without a hit and -9999.0
    where it is not valid."""
    p = events_reference(member_out, npoints * members, 1, events, n_slots)
    p = p.reshape(len(events), p.shape[1], npoints, members)
    return p != -9999.0, p == 1.0


def areas_reference(member_out, npoints, members, events, areas, n_slots=None):
    """area_prob [n_events, S, n_areas] as the header defines it: valid ANDed and hit ORed over each area's stations."""
    valid, hit = member_outcomes(member_out, npoints, members, events, n_slots)
    out = np.zeros(valid.shape[:2] + (len(areas),))
    for a, stations in enumerate(areas):
        st = np.asarray(stations)
        v = valid[:, :, st, :].all(axis=2)                     # [E, S, M]
        h = v & hit[:, :, st, :].any(axis=2)
        n, c = v.sum(axis=-1), h.sum(axis=-1)
        out[..., a] = np.where(n == 0, -9999.0, c / np.maximum(n, 1))
    return out


def _tiny():
    """3 stations x 2 members x 4 slots, planes 0 (surface temperature) and 1 (water 0.5 everywhere); station 2 did not
    run (all -9999)."""
    nan = np.nan
    t = np.array([[[1, -1, 1, 1], [1, 1, nan, 1]],          # station 0, members 0 and 1
                  [[1, 1, -1, 1], [-1, -1, -1, -1]],        # station 1
                  [[-9999.0] * 4, [-9999.0] * 4]])          # station 2
    w = np.where(t == -9999.0, -9999.0, 0.5)
    out = np.stack([t, w])                                  # [plane, station, member, slot]
    return np.ascontiguousarray(out.transpose(0, 3, 1, 2).reshape(2, 4, 6))


FREEZE2 = ([(0, "<", 0.0), (1, ">", 0.1)], 2)


def test_restatement_known_answers():
    """Hand-computed, window 2 (W(3) = [3] is truncated at the last slot):
    - area {0, 1}, s = 1: member 0 hits at station 0 (slot 1) and at station 1 (slot 2): one hit, not two;
      member 1 is invalid at station 0 (NaN at slot 2), which removes it from the area although station 1 hits;
    - s = 3: member 0 hits nowhere, member 1 hits at station 1: 1/2;
    - station 2 did not run: every area holding it is -9999.0, the overlapping {1, 2} too."""
    x = _tiny()
    areas = [[0], [1], [0, 1], [2], [1, 2]]
    p = areas_reference(x, 3, 2, [FREEZE2], areas)[0]
    assert list(p[:, 0]) == [0.5, 1.0, 0.0, 0.0]
    assert list(p[:, 1]) == [0.5, 1.0, 1.0, 0.5]
    assert list(p[:, 2]) == [1.0, 1.0, 1.0, 0.5]
    assert (p[:, 3] == -9999.0).all() and (p[:, 4] == -9999.0).all()
    # at s = 0 each station alone gives 1/2, the area 1: the members hit at different stations
    assert p[0, 2] > max(p[0, 0], p[0, 1])


def test_restatement_identities():
    """One-station areas equal the station events; repeated stations and their order change nothing."""
    rng = np.random.Generator(np.random.PCG64(11))
    P, M, S = 12, 7, 30
    x = np.round(rng.normal(0.0, 1.0, (3, S, P * M + 4)), 1) + 0.0
    x[rng.random(x.shape) < 0.03] = np.nan
    events = [([(0, "<", 0.0), (1, ">", -0.5)], 3), ([(2, ">=", 0.5)], 1), ([(1, "<=", 0.0)], S + 2)]
    ones = areas_reference(x, P, M, events, [[p] for p in range(P)])
    assert same_bits(ones, events_reference(x, P, M, events))
    base = [[0, 3, 4, 9], list(range(P)), [5, 6]]
    again = [[9, 4, 0, 3, 4, 9, 0], list(range(P))[::-1] * 2, [6, 5, 5]]
    assert same_bits(areas_reference(x, P, M, events, base), areas_reference(x, P, M, events, again))


def test_ensemble_areas_builds_offsets_and_stations():
    a = lib.ensemble_areas([[3, 1], [0], range(5, 8)])
    assert a.n_areas == 3
    assert list(a.offsets_array) == [0, 2, 3, 6] and list(a.stations_array) == [3, 1, 0, 5, 6, 7]
    assert a.offsets == a.offsets_array.ctypes.data and a.stations == a.stations_array.ctypes.data


def test_ctypes_mirror_matches_the_c_header():
    probe = r"""
#include <stdio.h>
#include <stddef.h>
#include "roadsurf_b200.h"
#define S(t) printf("sizeof " #t " %zu\n", sizeof(t))
#define O(t, f) printf("offsetof " #t "." #f " %zu\n", offsetof(t, f))
int main(void) {
  S(RsEnsembleAreas);
  O(RsEnsembleAreas, n_areas); O(RsEnsembleAreas, offsets); O(RsEnsembleAreas, stations);
  return 0;
}
"""
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "probe.c"), os.path.join(d, "probe")
        with open(src, "w") as f:
            f.write(probe)
        subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), src, "-o", exe], check=True)
        lines = subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split("\n")
    seen = 0
    for line in filter(None, lines):
        kind, name, val = line.split()
        if kind == "sizeof":
            assert C.sizeof(getattr(lib, name)) == int(val), name
        else:
            t, f = name.split(".")
            assert getattr(getattr(lib, t), f).offset == int(val), name
        seen += 1
    assert seen == 4


def _bad_areas(npoints):
    """(areas or None, what the error message names) for every malformed area set over npoints stations."""
    def raw(n, offsets, stations):
        o, s = np.asarray(offsets, dtype=np.int32), np.asarray(stations, dtype=np.int32)
        a = lib.RsEnsembleAreas(n_areas=n, offsets=o.ctypes.data if len(o) else None,
                                stations=s.ctypes.data if len(s) else None)
        a.keep = (o, s)
        return a
    return [(None, b"null area pointer"),
            (raw(1, [], [0]), b"null area pointer"), (raw(1, [0, 1], []), b"null area pointer"),
            (raw(0, [0], [0]), b"n_areas"), (raw(-1, [0], [0]), b"n_areas"),
            (raw(1, [1, 2], [0, 1]), b"offsets[0]"),
            (raw(3, [0, 2, 2, 3], [0, 1, 2]), b"strictly increasing"), (raw(2, [0, 3, 2], [0, 1, 2]), b"strictly increasing"),
            (raw(2, [0, 1, 3], [0, 1, -1]), b"outside [0, npoints)"),
            (raw(2, [0, 1, 3], [0, npoints, 1]), b"outside [0, npoints)")]


def test_bad_areas_and_specs_are_rejected_before_device_work():
    """Through roadsurf_ensemble_area_events and roadsurf_run_ensemble_host_soa_areas (a well-placed fork): every
    malformed area set, a spec without events, and every malformed spec return RS_ERR_BAD_ARGUMENT with a message."""
    handle = lib.load()
    P, M = 3, 4
    member_out = np.zeros((lib.O_NVAR, 5, 32))
    good = lib.ensemble_areas([[0, 2], [1]])
    area_prob = np.zeros(1 << 12)
    spec = lib.stats_spec(events=[([(TS, "<", 0.0), (WATER, ">", 0.1)], 3)])
    no_events = lib.stats_spec(QUANTILES, [(TS, "<", 0.0)])
    cases = [(spec, a, what) for a, what in _bad_areas(P)] + [(no_events, good, b"at least one event")]
    cases += [(sp, good, what) for sp, what in _bad_specs(lib.O_NVAR)]
    for sp, areas, what in cases:
        rc = handle.roadsurf_ensemble_area_events(member_out.ctypes.data, lib.O_NVAR, 5, 32, P, M, C.byref(sp),
                                                  None if areas is None else C.byref(areas), area_prob.ctypes.data,
                                                  None)
        assert rc == RS_ERR_BAD_ARGUMENT and what in handle.roadsurf_last_error(), what

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

    def host(sp, areas, area_prob_ptr):
        return handle.roadsurf_run_ensemble_host_soa_areas(C.byref(hb), mrec.ctypes.data, M, F, None, C.byref(sp),
                                                           stats.ctypes.data, prob.ctypes.data, None, None,
                                                           None if areas is None else C.byref(areas), area_prob_ptr,
                                                           C.byref(settings), C.byref(params))
    for sp, areas, what in cases:
        assert host(sp, areas, area_prob.ctypes.data) == RS_ERR_BAD_ARGUMENT, what
        assert what in handle.roadsurf_last_error(), what
    # areas without area_prob
    assert host(spec, good, None) == RS_ERR_BAD_ARGUMENT and b"null area pointer" in handle.roadsurf_last_error()
    if handle.roadsurf_device_count() == 0:
        # good areas pass the checks and then find no device, as does the call without areas
        assert host(spec, good, area_prob.ctypes.data) == -1 and host(spec, None, None) == -1


# ---- GPU --------------------------------------------------------------------------------------------------------

def _random_areas(rng, P, missing):
    """One-station areas (the all-missing station among them), ragged random areas (overlapping), an area of every
    station and one of every station but the missing one, one larger than a segment of 16 stations."""
    areas = [[0], [missing], [P - 1], [P // 2]]
    for size in (2, 3, 5, 7, 11, 17, 33):
        if size < P:
            areas.append(sorted(rng.choice(P, size, replace=False).tolist()))
    areas.append(list(range(P)))
    areas.append([p for p in range(P) if p != missing])
    areas.append(list(range(P // 3, P)))
    return areas


@pytest.mark.gpu
@pytest.mark.parametrize("M", [1, 2, 31, 51, 128])
def test_area_kernel_equals_the_restatement(rslib, M):
    """The tensors of test_events_kernel_equals_the_restatement: 2 003 slots (32 tiles of 64 slots), windows 1, 3,
    24, S and S + 5 whose look-ahead crosses tile ends, NaN and -9999.0 holes in half the lanes, an all-missing
    station.  Bit for bit against the restatement; one-station areas equal the station event planes written by
    roadsurf_ensemble_stats in the same run; a repeated, reordered copy of an area gives the same result."""
    import torch
    rng = np.random.Generator(np.random.PCG64(100 + M))
    P, S, out_nvar = min(150, max(5, 2400 // M)), 2003, lib.O_NVAR
    ldm = (P * M + 31) // 32 * 32
    x = np.round(rng.normal(0.0, 2.0, (out_nvar, S, ldm)), 1) + 0.0
    holes = (rng.random(x.shape) < 0.02) & (rng.random(ldm) < 0.5)
    x[holes & (rng.random(x.shape) < 0.5)] = np.nan
    x[holes & ~np.isnan(x)] = -9999.0
    x[:, :, 3 * M:4 * M] = -9999.0
    events, _ = _random_events(rng, x, P, M, S)
    areas = _random_areas(rng, P, 3)
    shuffled = list(areas[-3]) * 2
    rng.shuffle(shuffled)
    areas.append(shuffled)
    want = areas_reference(x, P, M, events, areas)
    xd = torch.from_numpy(x).cuda()
    spec = lib.stats_spec((), (), events)
    got = rslib.ensemble_area_events(xd, P, M, spec, rslib.ensemble_areas(areas)).cpu().numpy()
    assert got.shape == (len(events), S, len(areas))
    for j in range(len(events)):
        assert same_bits(got[j], want[j]), (M, j)
    _, prob = rslib.ensemble_stats(xd, P, M, spec)
    prob = prob.cpu().numpy()
    for a in range(4):
        assert same_bits(got[:, :, a], prob[:, :, areas[a][0]]), (M, a)
    assert same_bits(got[:, :, -1], got[:, :, -4])
    assert (want == -9999.0).any() and (M == 1 or ((want > 0.0) & (want < 1.0)).any())


@pytest.mark.gpu
def test_area_prob_is_written_inside_its_planes_only(rslib):
    """area_prob pre-filled with a sentinel and longer than [n_events][S][n_areas], the spec's event array filled
    beyond n_events: the kernels write exactly the first n_events * S * n_areas values."""
    import torch
    rng = np.random.Generator(np.random.PCG64(7))
    P, M, S = 40, 9, 70
    x = np.round(rng.normal(0.0, 2.0, (lib.O_NVAR, S, P * M)), 1) + 0.0
    events = [([(TS, "<", 0.0)], 2), ([(WATER, ">", 0.0), (TS, "<=", 1.0)], 5), ([(2, ">=", 0.0)], 1)]
    spec = lib.stats_spec((), (), events)
    spec.n_events = 2
    areas = lib.ensemble_areas([[0, 5], list(range(P)), [39]])
    n = 2 * S * 3
    buf = torch.full((n + 1000,), 777.0, dtype=torch.float64, device="cuda")
    xd = torch.from_numpy(x).cuda()
    lib._check(lib.load().roadsurf_ensemble_area_events(xd.data_ptr(), lib.O_NVAR, S, P * M, P, M, C.byref(spec),
                                                        C.byref(areas), buf.data_ptr(), None))
    torch.cuda.synchronize()
    b = buf.cpu().numpy()
    assert (b[n:] == 777.0).all() and (b[:n] != 777.0).all()
    want = areas_reference(x, P, M, events[:2], [[0, 5], list(range(P)), [39]])
    assert same_bits(b[:n].reshape(2, S, 3), want)


@pytest.mark.gpu
def test_device_entry_then_area_events_equal_the_restatement(rslib):
    """roadsurf_run_ensemble_device with out_nvar = RS_O_NVAR_EXT (coarse records, coupling + relaxation), then
    roadsurf_ensemble_area_events on its member_out: equal to the restatement, the hoar-frost events on the
    dew-point-deficit plane included, and one-station areas equal the run's own event planes."""
    P, M = 60, 5
    c = _Case(P, M, 3, 6, seed=4606)
    spec = lib.stats_spec(QUANTILES, [(TS, "<", 0.0)], ROAD_EVENTS)
    assert any(cd[0] == DEWDEFICIT for conds, _ in ROAD_EVENTS for cd in conds)
    ens = _device_ensemble(rslib, c, spec)
    ens.run()
    assert ens.n_out_members == ens.n_slots
    areas = [[7], [0, 1, 2, 3], list(range(0, P, 3)), list(range(P)), [59, 12, 33, 12], list(range(20, 45))]
    got = rslib.ensemble_area_events(ens.member_out, P, M, spec, rslib.ensemble_areas(areas)).cpu().numpy()
    want = areas_reference(ens.member_out.cpu().numpy(), P, M, ROAD_EVENTS, areas, ens.n_slots)
    assert same_bits(got, want)
    assert ((want > 0.0) & (want < 1.0)).any()
    _, prob = ens.stats()
    assert same_bits(got[:, :, 0], prob[1:, :, 7])


@pytest.mark.gpu
def test_host_entry_areas_in_station_chunks(rslib):
    """roadsurf_run_ensemble_host_soa_areas in one and in eight station chunks (areas straddle the chunk boundaries):
    area_prob equals roadsurf_ensemble_area_events on the device entry's member_out; stats and prob are bitwise those
    of the call without areas; d2h_bytes grows by exactly area_prob; the area kernels add one launch per chunk and
    one; with prob NULL area_prob is unchanged and no station events kernel runs."""
    P, M = 50, 6
    c = _Case(P, M, 3, 6, seed=4707)
    events = [e for e in ROAD_EVENTS if all(cd[0] < lib.O_NVAR for cd in e[0])]
    spec = lib.stats_spec(QUANTILES, [(TS, "<", 0.0)], events)
    ens = _device_ensemble(rslib, c, spec, extended=False)
    ens.run()
    area_lists = [[0], [49], [5, 6, 7, 8], list(range(3, 30)), list(range(P)), [48, 1, 20, 34, 6, 13],
                  list(range(0, P, 7)), [44, 45, 46, 47, 48, 49, 0]]
    areas = rslib.ensemble_areas(area_lists)
    want = rslib.ensemble_area_events(ens.member_out, P, M, spec, areas).cpu().numpy()
    assert same_bits(want, areas_reference(ens.member_out.cpu().numpy(), P, M, events, area_lists, ens.n_slots))
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
            plain, st0 = run()
            res, st1 = run(areas=areas)
            bare, st2 = run(areas=areas, prob=False)
        finally:
            rslib.set_option("max_points_per_device_batch", 0)
        groups = 1 if cap == 0 else 8
        assert st0["groups"] == st1["groups"] == st2["groups"] == groups
        n_m = res["stats"].shape[2]
        assert res["area_prob"].shape == (E, n_m, A)
        assert same_bits(res["area_prob"], want), cap
        assert same_bits(res["stats"], plain["stats"]) and same_bits(res["prob"], plain["prob"])
        assert st1["d2h_bytes"] == st0["d2h_bytes"] + 8 * E * n_m * A
        assert st1["kernel_launches"] == st0["kernel_launches"] + groups + 1
        assert "prob" not in bare and same_bits(bare["area_prob"], want) and same_bits(bare["stats"], plain["stats"])
        assert st2["kernel_launches"] == st1["kernel_launches"] - groups     # one station events kernel per chunk
