"""Ensemble runs (include/roadsurf_b200.h, part 3): the shared analysis, the fork into member lanes and the
ensemble statistics.  The contract: an ensemble over P stations and M members equals, bit for bit, P * M
independent runs in which lane p * M + m reads station p's forcing before the fork step F and member m's
from F on -- every output slot, status word and end-of-run state plane."""
import ctypes as C
import datetime as dt
import os
import subprocess
import tempfile

import numpy as np
import pytest

from parity import same_bits
from roadsurf_b200 import abi, lib, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
QUANTILES = (0.0, 0.1, 0.5, 0.9, 1.0)
THRESHOLDS = ((lib.O_NAMES.index("TsurfOut"), "<", 0.0), (lib.O_NAMES.index("IceOut"), ">", 0.0),
              (lib.O_NAMES.index("SnowOut"), ">=", 0.5), (8, "<", 0.0))   # 8: RS_O_DEWDEFICIT


# ---- NumPy restatement of the statistics kernel ---------------------------------------------------------

def stats_reference(member_out, npoints, members, quantiles=(), thresholds=()):
    """member_out [out_nvar, n_out, >= P * M] (lane p * M + m) -> (stats [5 + nq, out_nvar, n_out, P],
    prob [nt, n_out, P]), as the header defines them."""
    out_nvar, n_out, _ = member_out.shape
    x = member_out[:, :, :npoints * members].reshape(out_nvar, n_out, npoints, members)
    valid = (x == x) & (x > -9000.0)
    n = valid.sum(axis=-1)
    dn = n.astype(np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        acc = np.zeros(x.shape[:-1])
        for m in range(members):          # left to right in member order from +0.0
            acc = acc + np.where(valid[..., m], x[..., m], 0.0)
        mean = acc / dn
        ss = np.zeros(x.shape[:-1])
        for m in range(members):
            d = x[..., m] - mean
            ss = ss + np.where(valid[..., m], d * d, 0.0)
        std = np.sqrt(ss / dn)
        mn = np.where(valid, x, np.inf).min(axis=-1)
        mx = np.where(valid, x, -np.inf).max(axis=-1)
        ys = np.sort(np.where(valid, x, np.inf), axis=-1)
        planes = [dn, mean, std, mn, mx]
        for q in quantiles:
            h = (dn - 1.0) * q
            i = np.floor(np.maximum(h, 0.0)).astype(np.int64)
            t = h - i
            yi = np.take_along_axis(ys, i[..., None], -1)[..., 0]
            yn = np.take_along_axis(ys, np.minimum(i + 1, members - 1)[..., None], -1)[..., 0]
            planes.append(np.where((t == 0.0) | (i == n - 1), yi, yi + t * (yn - yi)))
        stats = np.stack(planes)
        stats[1:, n == 0] = -9999.0
        prob = np.zeros((len(thresholds), n_out, npoints))
        ops = {"<": np.less, "<=": np.less_equal, ">": np.greater, ">=": np.greater_equal}
        for j, (plane, op, value) in enumerate(thresholds):
            hit = (ops[op](x[plane], value) & valid[plane]).sum(axis=-1)
            prob[j] = np.where(n[plane] == 0, -9999.0, hit / dn[plane])
    return stats, prob


def test_restatement_known_answers():
    """Hand-computed results: NaN and -9999.0 are not members, n = 0 gives -9999.0, n = 1, ties."""
    nan = float("nan")
    vals = np.array([
        [3.0, nan, 1.0, -9999.0, 2.0],        # n = 3: 1 2 3
        [nan, nan, -9999.0, -9999.9, nan],    # n = 0
        [5.0, -9999.0, nan, nan, nan],        # n = 1
        [1.0, 1.0, 2.0, 2.0, 2.0],            # ties
    ])
    out = vals.reshape(1, 1, -1)              # one plane, one slot, 4 stations of 5 members
    st, pr = stats_reference(out, 4, 5, (0.0, 0.25, 0.5, 1.0), ((0, "<", 2.0), (0, ">=", 2.0)))
    s = st[:, 0, 0, :]
    assert list(s[0]) == [3.0, 0.0, 1.0, 5.0]
    assert s[1, 0] == 2.0 and s[2, 0] == np.sqrt(2.0 / 3.0) and s[3, 0] == 1.0 and s[4, 0] == 3.0
    assert list(s[5:, 0]) == [1.0, 1.5, 2.0, 3.0]
    assert (s[1:, 1] == -9999.0).all() and list(pr[:, 0, 1]) == [-9999.0, -9999.0]
    assert list(s[1:, 2]) == [5.0, 0.0, 5.0, 5.0, 5.0, 5.0, 5.0, 5.0]
    assert s[1, 3] == 8.0 / 5.0 and list(s[5:, 3]) == [1.0, 1.0, 2.0, 2.0]
    assert list(pr[:, 0, 0]) == [1.0 / 3.0, 2.0 / 3.0] and list(pr[:, 0, 3]) == [0.4, 0.6]


def test_ctypes_mirrors_match_the_c_header():
    probe = r"""
#include <stdio.h>
#include <stddef.h>
#include "roadsurf_b200.h"
#define S(t) printf("sizeof " #t " %zu\n", sizeof(t))
#define O(t, f) printf("offsetof " #t "." #f " %zu\n", offsetof(t, f))
int main(void) {
  S(RsEnsembleThreshold); S(RsEnsembleStatsSpec); S(RsEnsembleBatch);
  O(RsEnsembleThreshold, value); O(RsEnsembleStatsSpec, quantiles); O(RsEnsembleStatsSpec, thresholds);
  O(RsEnsembleBatch, members); O(RsEnsembleBatch, fork_step); O(RsEnsembleBatch, ld_members);
  O(RsEnsembleBatch, member_forcing); O(RsEnsembleBatch, member_relax); O(RsEnsembleBatch, member_local);
  O(RsEnsembleBatch, member_horizons); O(RsEnsembleBatch, member_state); O(RsEnsembleBatch, member_scratch);
  O(RsEnsembleBatch, member_status); O(RsEnsembleBatch, member_out); O(RsEnsembleBatch, n_out_members);
  O(RsEnsembleBatch, member_order); O(RsEnsembleBatch, spec); O(RsEnsembleBatch, stats); O(RsEnsembleBatch, prob);
  printf("const RS_ST_BAD_FORK %d\n", RS_ST_BAD_FORK);
  printf("const RS_ENS_MAX_MEMBERS %d\n", RS_ENS_MAX_MEMBERS);
  return 0;
}
"""
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "probe.c"), os.path.join(d, "probe")
        with open(src, "w") as f:
            f.write(probe)
        subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), src, "-o", exe], check=True)
        lines = subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split("\n")
    for line in filter(None, lines):
        kind, name, val = line.split()
        val = int(val)
        if kind == "sizeof":
            assert C.sizeof(getattr(lib, name)) == val, name
        elif kind == "offsetof":
            t, f = name.split(".")
            assert getattr(getattr(lib, t), f).offset == val, name
        else:
            assert {"RS_ST_BAD_FORK": lib.ST_BAD_FORK, "RS_ENS_MAX_MEMBERS": lib.ENS_MAX_MEMBERS}[name] == val


def _host_case(P=3, analysis_hours=2, hours=2, seed=5):
    start = synth.FORECAST_START - dt.timedelta(hours=analysis_hours)
    nrec = analysis_hours + hours + 2
    base = synth.draw_records(P, nrec, seed, start)
    base.TSurfObs[:, analysis_hours + 1:] = -9999.9
    pa, settings, params = synth.case_from_records(base, hours, analysis_hours, 1, 1)
    return base, pa, settings, params, start


def test_host_entry_checks_the_fork_without_a_gpu():
    """Argument errors are reported before any device work."""
    base, pa, settings, params, start = _host_case()
    P, M = base.npoints, 4
    forcing = np.ascontiguousarray(np.stack([getattr(base, v).T for v in synth.RECORD_VARS], axis=1))
    local = np.zeros((lib.L_NLOCAL, P))
    spec = lib.stats_spec(QUANTILES)
    handle = lib.load()

    def call(F, members=M, mode=1):
        r_f = lib.fork_record(base.record_step, F)
        mrec = np.zeros((max(1, base.nrec - r_f - 1), 11, P * members))
        hb = lib.RsHostBatch(npoints=P, sim_len=pa.sim_len, forcing_mode=mode, n_records=base.nrec, nvar=11,
                             out_stride=1, forcing=forcing.ctypes.data, record_step=base.record_step.ctypes.data,
                             time_fields=pa.time.ctypes.data, local=local.ctypes.data)
        stats = np.zeros(1 << 16)
        return handle.roadsurf_run_ensemble_host_soa(C.byref(hb), mrec.ctypes.data, members, F, None, C.byref(spec),
                                                     stats.ctypes.data, None, None, None, C.byref(settings),
                                                     C.byref(params))

    fs = 2 * 120
    assert call(fs + 5) == -2 and b"record time" in handle.roadsurf_last_error()        # RS_ERR_BAD_ARGUMENT
    assert call(fs + 2, mode=2) == -4                                                   # RS_ERR_UNSUPPORTED
    assert call(fs + 2, members=129) == -2 and b"128" in handle.roadsurf_last_error()
    assert call(fs + 2, mode=0) == -4
    if handle.roadsurf_device_count() == 0:
        # a well-placed fork passes the checks and then finds no device
        assert call(fs + 2) == -1 and call(fs + 1) == -1


def test_device_entry_checks_without_a_gpu():
    """Mode 2 and the member count are rejected before the device is touched."""
    handle = lib.load()
    sd = lib.RsDeviceBatch(npoints=10, ld=32, sim_len=100, forcing_mode=2, n_records=5, nvar=11)
    eb = lib.RsEnsembleBatch(shared=sd, members=4, fork_step=50, ld_members=64)
    assert handle.roadsurf_run_ensemble_device(C.byref(eb), None) == -4
    sd.forcing_mode = 1
    eb = lib.RsEnsembleBatch(shared=sd, members=200, fork_step=50, ld_members=2048)
    assert handle.roadsurf_run_ensemble_device(C.byref(eb), None) == -2


def test_member_records_equal_the_base_up_to_the_fork_record():
    base, pa, settings, params, start = _host_case(P=5)
    r_f = 2
    mrecs = synth.member_records(base, 3, r_f, 5, start)
    for m, r in enumerate(mrecs):
        for v in synth.RECORD_VARS:
            a, b = getattr(r, v), getattr(base, v)
            assert np.array_equal(a[:, :r_f + 1], b[:, :r_f + 1]), (m, v)
        assert np.array_equal(r.TSurfObs, base.TSurfObs)
        assert not np.array_equal(r.tair[:, r_f + 1:], base.tair[:, r_f + 1:])
    assert not np.array_equal(mrecs[0].tair, mrecs[1].tair)
    t = synth.member_record_tensor(mrecs, r_f)
    assert t.shape == (base.nrec - r_f - 1, 11, 15)
    assert np.array_equal(t[:, 0, 3 * 2 + 1], mrecs[1].tair[2, r_f + 1:])
    lanes = synth.lane_records(mrecs)
    assert np.array_equal(lanes.tair[4 * 3 + 2], mrecs[2].tair[4])


# ---- GPU -------------------------------------------------------------------------------------------------

def _lane_local(locals_m, P, M):
    """LocalParameters of lane p * M + m = member m's local of station p."""
    arr = (abi.LocalParameters * (P * M))()
    size = C.sizeof(abi.LocalParameters)
    for m, loc in enumerate(locals_m):
        for p in range(P):
            C.memmove(C.addressof(arr) + (p * M + m) * size, C.addressof(loc) + p * size, size)
    return arr


def _relax_of(local_arr):
    return np.array([[lp.tair_relax, lp.VZ_relax, lp.RH_relax] for lp in local_arr]).T.copy()


class _Case:
    """example1's shape: analysis + forecast, coupling + relaxation, hourly records, F = forecast step + 2."""

    def __init__(self, P, M, analysis_hours, hours, seed, use_coupling=1, use_relaxation=1):
        self.P, self.M = P, M
        self.start = synth.FORECAST_START - dt.timedelta(hours=analysis_hours)
        nrec = analysis_hours + hours + 2
        self.base = synth.draw_records(P, nrec, seed, self.start)
        self.base.TSurfObs[:, analysis_hours + 1:] = -9999.9
        self.forecast_step = analysis_hours * 120
        self.F = self.forecast_step + 2
        self.r_f = lib.fork_record(self.base.record_step, self.F)
        self.mrecs = synth.member_records(self.base, M, self.r_f, seed, self.start)
        self.kw = (hours, analysis_hours, use_coupling, use_relaxation)
        self.pa, self.settings, self.params = synth.case_from_records(self.base, *self.kw)
        self.pas = [synth.case_from_records(r, *self.kw)[0] for r in self.mrecs]
        self.sim_len = self.pa.sim_len
        self.lane_local = _lane_local([p.local for p in self.pas], P, M)
        self.station_local = self.pa.local

    def ensemble(self, rslib, spec, order=False, out_stride=1):
        import torch
        rslib.set_model(self.settings, self.params)
        sh = rslib.DeviceBatch(self.P, self.sim_len, n_records=self.base.nrec, coarse=True, horizons=True,
                               coupling=True, state=True, out_stride=out_stride)
        sh.load_records(self.base)
        sh.time_fields.copy_(torch.from_numpy(self.pa.time))
        sh.load_local(self.station_local, self.pa.local_horizons)
        ens = rslib.EnsembleBatch(sh, self.M, self.F, spec, member_relax=True)
        ens.load_member_records(self.mrecs)
        ens.set_member_relax(_relax_of(self.lane_local))
        if order:
            ens.run()
            torch.cuda.synchronize()
            ens.build_member_order()
        ens.run()
        torch.cuda.synchronize()
        return ens

    def independent(self, rslib, out_stride=1):
        import torch
        rslib.set_model(self.settings, self.params)
        lanes = synth.lane_records(self.mrecs)
        db = rslib.DeviceBatch(self.P * self.M, self.sim_len, n_records=self.base.nrec, coarse=True, horizons=True,
                               coupling=True, state=True, out_stride=out_stride)
        db.load_records(lanes)
        db.time_fields.copy_(torch.from_numpy(self.pa.time))
        db.load_local(self.lane_local, lanes.horizons)
        db.run()
        torch.cuda.synchronize()
        return db


def _assert_equivalent(ens, db, lanes=None):
    """Every output slot, status word and state plane of the ensemble lanes equal the independent runs'."""
    P, M = ens.shared.npoints, ens.members
    n = P * M
    lanes = np.arange(n) if lanes is None else np.asarray(lanes)
    s0 = ens.slot0
    ind = db.out.cpu().numpy()
    pre = ens.shared.out.cpu().numpy()[:, :s0, :P]
    assert same_bits(ind[:, :s0, lanes], pre[:, :, lanes // M]), "slots before the fork"
    mo = ens.member_out.cpu().numpy()
    assert same_bits(ind[:, s0:, lanes], mo[:, :ind.shape[1] - s0, lanes]), "member slots"
    assert np.array_equal(db.status.cpu().numpy()[lanes], ens.member_status.cpu().numpy()[lanes])
    assert same_bits(db.state.cpu().numpy()[:, lanes], ens.member_state.cpu().numpy()[:, lanes]), "state planes"


@pytest.mark.gpu
def test_coarse_ensemble_equals_independent_runs_and_the_oracle(rslib, oracle, exact):
    """P = 97 (ragged), M = 7, 6 h analysis + 12 h forecast, coupling + relaxation, 30 % sky-view points,
    F = forecast step + 2.  Also: a station that fails before F fails in all its members; a member with a
    missing forecast record fails alone and drops out of n_valid; relaxation edge cases; RS_ST_BAD_FORK."""
    P, M = 97, 7
    c = _Case(P, M, 6, 12, seed=4101)
    assert c.pa.sim_len == 1 + 18 * 120 and (c.base.sky_view < 1).mean() > 0.15
    oracle_ref = []
    for pa_m in c.pas:   # the oracle on unmodified members (stations 0..7 are compared below)
        ref = pa_m.copy()
        st, _ = oracle.run_batch(ref, c.settings, c.params, nthreads=8)
        oracle_ref.append((ref.out, st))
    # station 10 fails in the shared part: a missing air temperature record in the analysis
    c.base.tair[10, 2] = -9999.9
    for r in c.mrecs:
        r.tair[10, 2] = -9999.9
    # member 2 of station 11 misses a forecast record
    c.mrecs[2].tair[11, c.r_f + 3] = -9999.9
    # relaxation: station 12's own targets are invalid, its members' are valid; member 4 of station 13 invalid
    local = (abi.LocalParameters * P)()
    C.memmove(local, c.station_local, C.sizeof(c.station_local))
    local[12].tair_relax = 250.0
    c.lane_local[13 * M + 4].VZ_relax = -5.0
    # station 14 relaxes inside the shared part (InitLenI <= F - 2): member 0 keeps the station's targets
    local[14].InitLenI = c.F - 3
    for m in range(M):
        lp = c.lane_local[14 * M + m]
        lp.InitLenI = c.F - 3
        if m == 0:
            lp.tair_relax, lp.VZ_relax, lp.RH_relax = local[14].tair_relax, local[14].VZ_relax, local[14].RH_relax
    c.station_local = local
    spec = lib.stats_spec(QUANTILES, THRESHOLDS[:3])
    ens = c.ensemble(rslib, spec)
    db = c.independent(rslib)
    status = ens.member_status.cpu().numpy()[:P * M]
    bad = np.arange(14 * M + 1, 15 * M)
    assert ((status[bad] & (lib.ST_BAD_FORK | lib.ST_NOT_RUN)) == lib.ST_BAD_FORK | lib.ST_NOT_RUN).all()
    assert not (np.delete(status, bad) & lib.ST_BAD_FORK).any()
    assert (ens.member_out.cpu().numpy()[:, :, bad] == -9999.0).all()
    good = np.setdiff1d(np.arange(P * M), bad)
    _assert_equivalent(ens, db, good)
    assert (status[10 * M:11 * M] & lib.ST_FAILED).all() and len(set(status[10 * M:11 * M])) == 1
    fail11 = (status[11 * M:12 * M] & lib.ST_FAILED) != 0
    assert fail11.tolist() == [m == 2 for m in range(M)]
    assert (status & lib.ST_COUPLING_USED).sum() > 0.5 * P * M
    stats, prob = ens.stats()
    ts = lib.O_NAMES.index("TsurfOut")
    assert stats[lib.ENS_NVALID, ts, -1, 11] == M - 1 and stats[lib.ENS_NVALID, ts, -1, 0] == M
    assert (stats[lib.ENS_NVALID, ts, :, 10] == 0).all() and (stats[1:, ts, :, 10] == -9999.0).all()
    want_s, want_p = stats_reference(ens.member_out.cpu().numpy(), P, M, QUANTILES, THRESHOLDS[:3])
    assert np.array_equal(stats, want_s, equal_nan=True) and np.array_equal(prob, want_p)
    # the oracle: members of stations 0..7, every step
    got = ens.member_outputs()
    pre = ens.shared.outputs()
    for m, (ref_out, st) in enumerate(oracle_ref):
        for k, name in enumerate(lib.O_NAMES):
            full = np.concatenate([pre[name][:8, :ens.slot0], got[name][:8, m]], axis=1)
            assert np.array_equal(full, ref_out[name][:8]), (m, name)
        assert np.array_equal(status[np.arange(8) * M + m], st[:8])


@pytest.mark.gpu
def test_full_resolution_ensemble_off_record_strided_extended(rslib, exact):
    """forcing_mode 0, F off any record time, output every 120th step from out_start 30, RS_O_NVAR_EXT."""
    import torch
    P, M = 45, 5
    c = _Case(P, M, 3, 6, seed=4202, use_coupling=1, use_relaxation=0)
    F = c.forecast_step + 47
    lanes = abi.PointArrays(P * M, c.sim_len)
    for name in [n[2:] for n in abi.INPUT_DOUBLE_FIELDS] + ["PrecPhase"]:
        a = getattr(lanes, name)
        for m, pa_m in enumerate(c.pas):
            a[m::M, :F - 1] = getattr(c.pa, name)[:, :F - 1]
            a[m::M, F - 1:] = getattr(pa_m, name)[:, F - 1:]
    lanes.time[:] = c.pa.time
    lanes.local_horizons[:] = np.repeat(c.pa.local_horizons, M, axis=0)
    lane_local = _lane_local([c.pa.local] * M, P, M)
    rslib.set_model(c.settings, c.params)
    kw = dict(horizons=True, coupling=True, state=True, out_stride=120, out_start=30, extended_outputs=True)
    sh = rslib.DeviceBatch(P, c.sim_len, **kw)
    sh.load_point_arrays(c.pa)
    ens = rslib.EnsembleBatch(sh, M, F, lib.stats_spec(QUANTILES, THRESHOLDS))
    ens.load_member_forcing(lanes)
    ens.run()
    db = rslib.DeviceBatch(P * M, c.sim_len, **kw)
    db.load_point_arrays(lanes)
    db.load_local(lane_local, lanes.local_horizons)
    db.run()
    torch.cuda.synchronize()
    _assert_equivalent(ens, db)
    stats, prob = ens.stats()
    want_s, want_p = stats_reference(ens.member_out.cpu().numpy(), P, M, QUANTILES, THRESHOLDS)
    assert np.array_equal(stats, want_s, equal_nan=True) and np.array_equal(prob, want_p)
    assert stats.shape[1] == lib.O_NVAR_EXT


@pytest.mark.gpu
@pytest.mark.parametrize("M", [1, 2, 7, 32, 51, 128])
def test_statistics_kernel_equals_the_restatement(rslib, M):
    """Crafted member tensors with NaN, -9999.0, ties and all-missing stations."""
    import torch
    rng = np.random.Generator(np.random.PCG64(M))
    P, n_out, out_nvar = 37, 5, lib.O_NVAR_EXT
    ldm = (P * M + 31) // 32 * 32
    x = np.round(rng.normal(0.0, 2.0, (out_nvar, n_out, ldm)), 1) + 0.0   # ties; no -0.0
    x[rng.random(x.shape) < 0.1] = np.nan
    x[rng.random(x.shape) < 0.1] = -9999.0
    x[:, :, 3 * M:4 * M] = -9999.0
    spec = lib.stats_spec(QUANTILES, THRESHOLDS)
    stats, prob = rslib.ensemble_stats(torch.from_numpy(x).cuda(), P, M, spec)
    want_s, want_p = stats_reference(x, P, M, QUANTILES, THRESHOLDS)
    assert np.array_equal(stats.cpu().numpy(), want_s, equal_nan=True)
    assert np.array_equal(prob.cpu().numpy(), want_p)


@pytest.mark.gpu
def test_host_entry_equals_the_device_entry_in_station_chunks(rslib, exact):
    """roadsurf_run_ensemble_host_soa derives the member relaxation targets itself (from latest_obs_index and the
    members' records, also where the station's records after r_f are missing); with max_points_per_device_batch it
    runs several station chunks.  Bit-identical to the device entry."""
    P, M = 50, 6
    c = _Case(P, M, 3, 6, seed=4303)
    spec = lib.stats_spec(QUANTILES, THRESHOLDS[:3])
    ens = c.ensemble(rslib, spec, out_stride=60)
    want_s, want_p = ens.stats()
    sh = ens.shared
    forcing = sh.forcing[:, :, :P].cpu().numpy().copy()
    forcing[c.r_f + 1:] = -9999.9   # the station records after r_f never reach a result: they may be missing
    local = sh.local[:, :P].cpu().numpy().copy()
    hor = sh.horizons[:, :P].cpu().numpy().copy()
    mrec = synth.member_record_tensor(c.mrecs, c.r_f)
    for cap in (0, 7 * M):
        rslib.set_option("max_points_per_device_batch", cap)
        try:
            res = rslib.run_ensemble_host_soa(c.settings, c.params, forcing, c.base.record_step.astype(np.int32),
                                              c.pa.time, local, mrec, M, c.F, spec, horizons=hor, out_stride=60,
                                              coupling_window_end=sh.coupling_window_end, member_out=True,
                                              member_status=True,
                                              latest_obs_index=np.full(P, c.forecast_step + 1, dtype=np.int32))
        finally:
            rslib.set_option("max_points_per_device_batch", 0)
        assert rslib.last_batch_stats()["groups"] == (1 if cap == 0 else 8)
        n_m = want_s.shape[2]
        assert np.array_equal(res["stats"], want_s[:, :6, :n_m], equal_nan=True), cap
        assert np.array_equal(res["prob"], want_p), cap
        assert np.array_equal(res["member_out"], ens.member_out.cpu().numpy()[:, :n_m, :P * M]), cap
        assert np.array_equal(res["member_status"], ens.member_status.cpu().numpy()[:P * M]), cap


@pytest.mark.gpu
def test_member_order_and_a_single_member(rslib, exact):
    """A member_order from roadsurf_order_points changes nothing; M = 1 with the station's own records is
    the plain run."""
    import torch
    P, M = 70, 4
    c = _Case(P, M, 3, 6, seed=4404)
    spec = lib.stats_spec(QUANTILES)
    a = c.ensemble(rslib, spec)
    b = c.ensemble(rslib, spec, order=True)
    assert b.member_order is not None
    for t in ("member_out", "member_status", "member_state"):
        assert torch.equal(getattr(a, t), getattr(b, t)), t
    assert all(np.array_equal(x, y, equal_nan=True) for x, y in zip(a.stats(), b.stats()))
    one = _Case(P, 1, 3, 6, seed=4404)
    one.mrecs = [one.base]
    one.pas = [one.pa]
    one.lane_local = _lane_local([one.pa.local], P, 1)
    ens = one.ensemble(rslib, spec)
    plain = one.independent(rslib)
    _assert_equivalent(ens, plain)


@pytest.mark.gpu
def test_member_slot_dimension_larger_than_the_member_slots(rslib, exact):
    """n_out_members one larger than the output slots of [F, sim_len] (through the C ABI): the member launch and the
    statistics use it as the slot stride, the statistics cover the real slots only and equal the tight layout's."""
    import torch
    P, M = 40, 5
    c = _Case(P, M, 3, 6, seed=4505)
    spec = lib.stats_spec(QUANTILES, THRESHOLDS[:3])
    tight = c.ensemble(rslib, spec, out_stride=60)
    rslib.set_model(c.settings, c.params)
    sh = tight.shared
    wide = rslib.EnsembleBatch(sh, M, c.F, spec, member_relax=True, extra_slots=1)
    wide.load_member_records(c.mrecs)
    wide.set_member_relax(_relax_of(c.lane_local))
    wide.stats_t.fill_(777.0)
    wide.prob_t.fill_(777.0)
    wide.run()
    torch.cuda.synchronize()
    n = tight.n_slots
    assert wide.n_out_members == n + 1 and wide.member_out.shape[1] == n + 1
    assert torch.equal(wide.member_out[:, :n], tight.member_out)
    for a, b in zip(wide.stats(), tight.stats()):
        assert np.array_equal(a, b, equal_nan=True)
    want_s, want_p = stats_reference(wide.member_out[:, :n].cpu().numpy(), P, M, QUANTILES, THRESHOLDS[:3])
    got_s, got_p = wide.stats()
    assert np.array_equal(got_s, want_s, equal_nan=True) and np.array_equal(got_p, want_p)
    assert (wide.stats_t[:, :, n].cpu().numpy() == 777.0).all() and (wide.prob_t[:, n].cpu().numpy() == 777.0).all()
