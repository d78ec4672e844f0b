"""Ensemble event probabilities (RsEnsembleEvent, include/roadsurf_b200.h part 3): compound conditions over a window
of member output slots, reduced on the device.  For station p, member m, slot s < S and event e, the member is valid
when every plane the conditions name holds a valid value at every slot of W(s) = [s, min(s + window, S) - 1], and hits
when the conjunction of the conditions holds at one slot or more of W(s); prob[n_thresholds + e][s][p] = hits / valid,
-9999.0 where no member is valid."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from parity import same_bits
from roadsurf_b200 import lib, synth
from test_ensemble import QUANTILES, _Case, _host_case, _relax_of, stats_reference

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OPS = {"<": np.less, "<=": np.less_equal, ">": np.greater, ">=": np.greater_equal}
TS, WATER, DEWDEFICIT = lib.O_NAMES.index("TsurfOut"), lib.O_NAMES.index("WaterOut"), 8
RS_ERR_BAD_ARGUMENT = -2


# ---- NumPy restatement ------------------------------------------------------------------------------------------

def events_reference(member_out, npoints, members, events, n_slots=None):
    """member_out [out_nvar, >= S, >= P * M] (lane p * M + m), events [(conditions, window), ...] ->
    prob [n_events, S, P] as the header defines it.  Counts of invalid and of hit slots per window come from
    prefix sums along the slots."""
    S = member_out.shape[1] if n_slots is None else n_slots
    x = member_out[:, :S, :npoints * members].reshape(member_out.shape[0], S, npoints, members)
    valid = (x == x) & (x > -9000.0)
    prob = np.zeros((len(events), S, npoints))
    zero = np.zeros((1, npoints, members), dtype=np.int64)
    for j, (conds, window) in enumerate(events):
        bad = ~np.logical_and.reduce([valid[plane] for plane, _, _ in conds])          # [S, P, M]
        with np.errstate(invalid="ignore"):
            both = np.logical_and.reduce([OPS[op](x[plane], value) for plane, op, value in conds])
        n_bad = np.concatenate([zero, np.cumsum(bad, axis=0)])
        n_both = np.concatenate([zero, np.cumsum(both, axis=0)])
        first = np.arange(S)
        end = np.minimum(first + window, S)                                                 # W(s) = [s, end)
        ok = (n_bad[end] - n_bad[first]) == 0
        hit = ok & ((n_both[end] - n_both[first]) > 0)
        n, c = ok.sum(axis=-1), hit.sum(axis=-1)
        prob[j] = np.where(n == 0, -9999.0, c / np.maximum(n, 1))
    return prob


def _tiny():
    """2 stations x 3 members x 5 slots, planes 0 (surface temperature) and 1 (water)."""
    nan = np.nan
    t = np.array([[[1, -1, 1, 1, -1], [1, 1, 1, 1, 1], [-1, nan, -1, -1, 0]],              # station 0, members 0..2
                  [[0, 0, -9999.0, 0, 0], [nan, 0, 0, 0, 0], [0, 0, 0, -9999.9, 0]]])      # station 1
    w = np.full_like(t, 0.5)
    w[0, 0, 2] = 0.0
    w[0, 2, 3] = 0.0                                  # station 0, member 2: T < 0 at slot 3 but no water
    out = np.stack([t, w])                            # [plane, station, member, slot]
    return np.ascontiguousarray(out.transpose(0, 3, 1, 2).reshape(2, 5, 6))


def test_restatement_known_answers():
    """Hand-computed: AND across two planes, an invalid value removing a member from every window that holds it,
    windows truncated at the last slot, n = 0 -> -9999.0, LT against LE on a tie."""
    x = _tiny()
    freeze = ([(0, "<", 0.0), (1, ">", 0.1)], 2)
    le, lt = ([(0, "<=", 0.0)], 5), ([(0, "<", 0.0)], 5)
    p = events_reference(x, 2, 3, [freeze, le, lt])
    third, half, two3 = 1.0 / 3.0, 0.5, 2.0 / 3.0
    # station 0: member 2 is invalid at slot 1, so out of W(0) and W(1); W(4) = [4] is truncated
    assert list(p[0, :, 0]) == [half, half, third, third, third]
    assert list(p[1, :, 0]) == [half, half, two3, two3, two3]
    assert list(p[2, :, 0]) == [half, half, two3, two3, third]        # slot 4: member 2's 0.0 is <= 0, not < 0
    # station 1: no member is valid over W(0) = [0, 4]; afterwards every valid member has T == 0
    assert list(p[0, :, 1]) == [0.0] * 5
    assert list(p[1, :, 1]) == [-9999.0, 1.0, 1.0, 1.0, 1.0]
    assert list(p[2, :, 1]) == [-9999.0, 0.0, 0.0, 0.0, 0.0]


def test_restatement_window_one_is_the_threshold():
    rng = np.random.Generator(np.random.PCG64(3))
    x = np.round(rng.normal(0.0, 1.0, (3, 7, 40)), 1) + 0.0
    x[rng.random(x.shape) < 0.2] = np.nan
    thresholds = [(0, "<", 0.0), (1, "<=", 0.3), (2, ">", -0.2), (2, ">=", 0.1)]
    _, want = stats_reference(x, 8, 5, (), thresholds)
    got = events_reference(x, 8, 5, [([t], 1) for t in thresholds])
    assert same_bits(got, want)


def test_stats_spec_builds_events():
    sp = lib.stats_spec((0.5,), [(0, "<", 0.0)], [([(TS, "<", 0.0), (WATER, ">", 0.2)], 6), ([(2, ">=", 1.5)], 1)])
    assert (sp.n_quantiles, sp.n_thresholds, sp.n_events, sp.n_prob) == (1, 1, 2, 3)
    e = sp.events[0]
    assert (e.n_conditions, e.window) == (2, 6)
    assert [(c.plane, c.op, c.value) for c in e.conditions[:2]] == [(TS, lib.ENS_LT, 0.0), (WATER, lib.ENS_GT, 0.2)]
    assert (sp.events[1].conditions[0].op, sp.events[1].window) == (lib.ENS_GE, 1)
    with pytest.raises(ValueError):
        lib.stats_spec(events=[([(0, "<", 0.0)], 1)] * 9)
    with pytest.raises(ValueError):
        lib.stats_spec(events=[([], 1)])


def test_ctypes_mirrors_match_the_c_header():
    probe = r"""
#include <stdio.h>
#include <stddef.h>
#include "roadsurf_b200.h"
#define S(t) printf("sizeof " #t " %zu\n", sizeof(t))
#define O(t, f) printf("offsetof " #t "." #f " %zu\n", offsetof(t, f))
int main(void) {
  S(RsEnsembleEvent); S(RsEnsembleStatsSpec); S(RsEnsembleBatch);
  O(RsEnsembleEvent, n_conditions); O(RsEnsembleEvent, window); O(RsEnsembleEvent, conditions);
  O(RsEnsembleStatsSpec, quantiles); O(RsEnsembleStatsSpec, thresholds); O(RsEnsembleStatsSpec, n_events);
  O(RsEnsembleStatsSpec, events);
  O(RsEnsembleBatch, spec); O(RsEnsembleBatch, stats); O(RsEnsembleBatch, prob);
  printf("const RS_ENS_MAX_EVENTS %d\n", RS_ENS_MAX_EVENTS);
  printf("const RS_ENS_MAX_CONDITIONS %d\n", RS_ENS_MAX_CONDITIONS);
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
        val = int(val)
        if kind == "sizeof":
            assert C.sizeof(getattr(lib, name)) == val, name
        elif kind == "offsetof":
            t, f = name.split(".")
            assert getattr(getattr(lib, t), f).offset == val, name
        else:
            assert {"RS_ENS_MAX_EVENTS": lib.ENS_MAX_EVENTS, "RS_ENS_MAX_CONDITIONS": lib.ENS_MAX_CONDITIONS}[name] == val
        seen += 1
    assert seen == 15


def _bad_specs(out_nvar):
    """(spec, what the error message names) for every malformed event."""
    def spec(**ev):
        sp = lib.stats_spec(QUANTILES, [(0, "<", 0.0)], [([(TS, "<", 0.0), (WATER, ">", 0.1)], 3)])
        for k, v in ev.items():
            if k == "n_events":
                sp.n_events = v
            elif k in ("plane", "op"):
                setattr(sp.events[0].conditions[1], k, v)
            else:
                setattr(sp.events[0], k, v)
        return sp
    return [(spec(n_events=-1), b"8 events"), (spec(n_events=9), b"8 events"),
            (spec(n_conditions=0), b"conditions"), (spec(n_conditions=5), b"conditions"),
            (spec(window=0), b"window"), (spec(window=-3), b"window"),
            (spec(plane=-1), b"plane"), (spec(plane=out_nvar), b"plane"),
            (spec(op=-1), b"comparison"), (spec(op=4), b"comparison")]


def test_bad_event_specs_are_rejected_before_device_work():
    """Through roadsurf_ensemble_stats (stats and prob NULL: a good spec returns RS_OK without a launch) and through
    the host entry (a well-placed fork), every bad spec returns RS_ERR_BAD_ARGUMENT with a message."""
    handle = lib.load()
    member_out = np.zeros((lib.O_NVAR_EXT, 5, 32))
    for out_nvar in (lib.O_NVAR, lib.O_NVAR_EXT):
        for sp, what in _bad_specs(out_nvar):
            rc = handle.roadsurf_ensemble_stats(member_out.ctypes.data, out_nvar, 5, 32, 2, 3, C.byref(sp), None, None,
                                                32, None)
            assert rc == RS_ERR_BAD_ARGUMENT and what in handle.roadsurf_last_error(), (out_nvar, what)
    # the extended planes are legal where out_nvar == RS_O_NVAR_EXT
    dew = lib.stats_spec(events=[([(TS, "<", 0.0), (DEWDEFICIT, "<", 0.0)], 1)])
    assert handle.roadsurf_ensemble_stats(member_out.ctypes.data, lib.O_NVAR_EXT, 5, 32, 2, 3, C.byref(dew), None, None,
                                          32, None) == 0
    assert handle.roadsurf_ensemble_stats(member_out.ctypes.data, lib.O_NVAR, 5, 32, 2, 3, C.byref(dew), None, None,
                                          32, None) == RS_ERR_BAD_ARGUMENT

    base, pa, settings, params, start = _host_case()
    P, M = base.npoints, 4
    F = 2 * 120 + 2
    forcing = np.ascontiguousarray(np.stack([getattr(base, v).T for v in synth.RECORD_VARS], axis=1))
    local = np.zeros((lib.L_NLOCAL, P))
    r_f = lib.fork_record(base.record_step, F)
    mrec = np.zeros((base.nrec - r_f - 1, 11, P * M))
    hb = lib.RsHostBatch(npoints=P, sim_len=pa.sim_len, forcing_mode=1, n_records=base.nrec, nvar=11, out_stride=1,
                         forcing=forcing.ctypes.data, record_step=base.record_step.ctypes.data,
                         time_fields=pa.time.ctypes.data, local=local.ctypes.data)
    stats, prob = np.zeros(1 << 16), np.zeros(1 << 16)
    # the host entry's outputs are RS_O_NVAR planes: the dew-point deficit is not one of them
    for sp, what in _bad_specs(lib.O_NVAR) + [(dew, b"plane")]:
        rc = handle.roadsurf_run_ensemble_host_soa(C.byref(hb), mrec.ctypes.data, M, F, None, C.byref(sp),
                                                   stats.ctypes.data, prob.ctypes.data, None, None, C.byref(settings),
                                                   C.byref(params))
        assert rc == RS_ERR_BAD_ARGUMENT and what in handle.roadsurf_last_error(), what


# ---- GPU --------------------------------------------------------------------------------------------------------

def _random_events(rng, x, P, M, S):
    """Eight events over windows {1, 3, 24, S, S + 5} and all four ops, their values drawn from valid member values
    (ties), with one single-condition window-1 event per threshold of the returned list."""
    valid = np.argwhere((x[:, :S, :P * M] == x[:, :S, :P * M]) & (x[:, :S, :P * M] > -9000.0))

    def cond(plane, op):
        s, lane = valid[valid[:, 0] == plane][rng.integers(0, (valid[:, 0] == plane).sum())][1:]
        return (plane, op, float(x[plane, s, lane]))
    events = [([cond(0, "<")], 1),
              ([cond(0, "<="), cond(1, ">")], 3),
              ([cond(2, ">="), cond(3, "<"), cond(4, "<=")], 24),
              ([cond(5, ">"), cond(0, ">="), cond(1, "<"), cond(2, "<=")], S),
              ([cond(1, "<=")], S + 5),
              ([cond(0, ">"), cond(0, "<")], 24),
              ([cond(3, ">=")], 1),
              ([cond(4, "<"), cond(5, ">=")], 3)]
    thresholds = [events[0][0][0], events[6][0][0]]
    return events, thresholds


@pytest.mark.gpu
@pytest.mark.parametrize("M", [1, 2, 31, 51, 128])
def test_events_kernel_equals_the_restatement(rslib, M):
    """2 003 slots, ragged station counts, NaN and -9999.0 in half the lanes, an all-missing station; a one-condition
    window-1 event equals its threshold plane in the same call.  With windows up to S + 5 a thread scans all slots;
    the second call, windows up to 24 over these few stations, splits the slots into tiles whose look-ahead crosses
    the tile ends."""
    import torch
    rng = np.random.Generator(np.random.PCG64(100 + M))
    P, S, out_nvar = min(150, max(5, 2400 // M)), 2003, lib.O_NVAR
    ldm = (P * M + 31) // 32 * 32
    x = np.round(rng.normal(0.0, 2.0, (out_nvar, S, ldm)), 1) + 0.0
    holes = (rng.random(x.shape) < 0.02) & (rng.random(ldm) < 0.5)
    x[holes & (rng.random(x.shape) < 0.5)] = np.nan
    x[holes & ~np.isnan(x)] = -9999.0
    x[:, :, 3 * M:4 * M] = -9999.0
    events, thresholds = _random_events(rng, x, P, M, S)
    want = events_reference(x, P, M, events)
    xd = torch.from_numpy(x).cuda()
    _, prob = rslib.ensemble_stats(xd, P, M, lib.stats_spec((), thresholds, events))
    prob = prob.cpu().numpy()
    assert prob.shape == (len(thresholds) + len(events), S, P)
    for j in range(len(events)):
        assert same_bits(prob[len(thresholds) + j], want[j]), (M, j)
    assert same_bits(prob[2], prob[0]) and same_bits(prob[2 + 6], prob[1])
    short = [j for j, (_, w) in enumerate(events) if w <= 24]
    _, tiled = rslib.ensemble_stats(xd, P, M, lib.stats_spec((), (), [events[j] for j in short]))
    assert same_bits(tiled.cpu().numpy(), want[short]), M
    assert (want == -9999.0).any() and (M == 1 or ((want > 0.0) & (want < 1.0)).any())


def _device_ensemble(rslib, c, spec, order=False, extended=True, extra_slots=0, out_stride=60):
    """_Case through roadsurf_run_ensemble_device, with the extended output planes."""
    import torch
    rslib.set_model(c.settings, c.params)
    sh = rslib.DeviceBatch(c.P, c.sim_len, n_records=c.base.nrec, coarse=True, horizons=True, coupling=True,
                           state=True, out_stride=out_stride, extended_outputs=extended)
    sh.load_records(c.base)
    sh.time_fields.copy_(torch.from_numpy(c.pa.time))
    sh.load_local(c.station_local, c.pa.local_horizons)
    ens = rslib.EnsembleBatch(sh, c.M, c.F, spec, member_relax=True, extra_slots=extra_slots)
    ens.load_member_records(c.mrecs)
    ens.set_member_relax(_relax_of(c.lane_local))
    if order:
        ens.run()
        torch.cuda.synchronize()
        ens.build_member_order()
    return ens


ROAD_EVENTS = [([(TS, "<", 0.0), (WATER, ">", 0.0)], 6),       # wet road freezing within the next 3 h
               ([(TS, "<", 0.0), (DEWDEFICIT, "<", 0.0)], 1),  # hoar frost risk
               ([(TS, "<", 0.0), (DEWDEFICIT, "<", 0.0)], 6),
               ([(TS, "<=", -1.0)], 4)]


@pytest.mark.gpu
def test_device_entry_events_equal_the_restatement_of_its_member_out(rslib):
    """Coarse records, coupling + relaxation, example1's shape, out_nvar = RS_O_NVAR_EXT: the event planes equal the
    restatement applied to the run's own member_out, and are unchanged with a member_order."""
    import torch
    P, M = 60, 5
    c = _Case(P, M, 3, 6, seed=4606)
    spec = lib.stats_spec(QUANTILES, [(TS, "<", 0.0)], ROAD_EVENTS)
    ens = _device_ensemble(rslib, c, spec)
    ens.run()
    torch.cuda.synchronize()
    _, prob = ens.stats()
    assert prob.shape == (1 + len(ROAD_EVENTS), ens.n_slots, P)
    want = events_reference(ens.member_out.cpu().numpy(), P, M, ROAD_EVENTS, ens.n_slots)
    assert same_bits(prob[1:], want)
    assert ((want > 0.0) & (want < 1.0)).any()
    ordered = _device_ensemble(rslib, c, spec, order=True)
    assert ordered.member_order is not None
    ordered.run()
    torch.cuda.synchronize()
    assert torch.equal(ordered.member_out, ens.member_out)
    assert same_bits(ordered.stats()[1], prob)


@pytest.mark.gpu
def test_host_entry_events_equal_the_device_entry_in_station_chunks(rslib):
    """roadsurf_run_ensemble_host_soa without member_out, in one and in several station chunks: its event planes equal
    the device entry's, and d2h_bytes counts the grown probability tensor."""
    P, M = 50, 6
    c = _Case(P, M, 3, 6, seed=4707)
    events = [e for e in ROAD_EVENTS if all(cd[0] < lib.O_NVAR for cd in e[0])]
    spec = lib.stats_spec(QUANTILES, [(TS, "<", 0.0)], events)
    ens = _device_ensemble(rslib, c, spec, extended=False)
    ens.run()
    want_s, want_p = ens.stats()
    sh = ens.shared
    forcing = sh.forcing[:, :, :P].cpu().numpy().copy()
    local = sh.local[:, :P].cpu().numpy().copy()
    hor = sh.horizons[:, :P].cpu().numpy().copy()
    mrec = synth.member_record_tensor(c.mrecs, c.r_f)
    n_m = want_s.shape[2]
    for cap in (0, 7 * M):
        rslib.set_option("max_points_per_device_batch", cap)
        try:
            res = rslib.run_ensemble_host_soa(c.settings, c.params, forcing, c.base.record_step.astype(np.int32),
                                              c.pa.time, local, mrec, M, c.F, spec, horizons=hor, out_stride=60,
                                              coupling_window_end=sh.coupling_window_end,
                                              latest_obs_index=np.full(P, c.forecast_step + 1, dtype=np.int32))
        finally:
            rslib.set_option("max_points_per_device_batch", 0)
        st = rslib.last_batch_stats()
        assert st["groups"] == (1 if cap == 0 else 8)
        assert "member_out" not in res and res["prob"].shape == (1 + len(events), n_m, P)
        assert same_bits(res["prob"], want_p), cap
        assert st["d2h_bytes"] == 8 * P * n_m * ((lib.ENS_NFIXED + len(QUANTILES)) * lib.O_NVAR + 1 + len(events))


@pytest.mark.gpu
def test_event_planes_stay_inside_the_member_slots_and_their_planes(rslib):
    """n_out_members two larger than the member slots, prob_t pre-filled with two spare planes: the events write
    their planes over the member slots only."""
    import torch
    P, M = 40, 5
    c = _Case(P, M, 3, 6, seed=4808)
    spec = lib.stats_spec((), [(TS, "<", 0.0)], ROAD_EVENTS)
    ens = _device_ensemble(rslib, c, spec, extra_slots=2)
    n, k = ens.n_slots, spec.n_prob
    ens.prob_t = torch.full((k + 2, ens.n_out_members, ens.shared.ld), 777.0, dtype=torch.float64, device="cuda")
    ens.run()
    torch.cuda.synchronize()
    prob = ens.prob_t.cpu().numpy()
    assert (prob[:, n:] == 777.0).all() and (prob[k:] == 777.0).all()
    assert (prob[:k, :n, :P] != 777.0).all()
    want = events_reference(ens.member_out.cpu().numpy(), P, M, ROAD_EVENTS, n)
    assert same_bits(prob[1:k, :n, :P], want)
