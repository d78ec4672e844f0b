"""Ensemble window extremes (include/roadsurf_b200.h part 3, after RsEnsembleAreas): statistics of each member's minimum
or maximum of one plane over a window of member slots.  For station p, extreme x, member m and slot s < S, the member is
valid when the plane holds a valid value at every slot of W(s) = [s, min(s + window, S) - 1], and its value is the
minimum (maximum) over W(s) in the order of the int64 map b >= 0 ? b : b ^ 0x7fff...ff of the bits (-0.0 below +0.0);
ext_stats[j][x][s][p] are the statistics of `stats` over the valid members' values.  Areas: valid at every station, the
minimum (maximum) over the stations."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from parity import same_bits
from roadsurf_b200 import abi, lib, synth
from test_ensemble import QUANTILES, _Case, _host_case, stats_reference
from test_ensemble_areas import _bad_areas, _random_areas, _tiny, areas_reference
from test_ensemble_events import DEWDEFICIT, ROAD_EVENTS, TS, WATER, _bad_specs, _device_ensemble, events_reference

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RS_ERR_BAD_ARGUMENT = -2
ICE, SNOW = lib.O_NAMES.index("IceOut"), lib.O_NAMES.index("SnowOut")
MISSING = -9999.0


# ---- NumPy restatement ------------------------------------------------------------------------------------------

def _key(x):
    """The header's order-preserving map of a double's bits to int64 (an involution on negative bit patterns)."""
    b = np.ascontiguousarray(x, dtype=np.float64).view(np.int64)
    return np.where(b >= 0, b, b ^ np.int64(0x7FFFFFFFFFFFFFFF))


def _unkey(k):
    return np.where(k >= 0, k, k ^ np.int64(0x7FFFFFFFFFFFFFFF)).astype(np.int64).view(np.float64)


def window_values(member_out, npoints, members, extremes, n_slots=None):
    """[n_extremes, S, P, M]: each member's minimum (maximum) over W(s), MISSING where W(s) holds an invalid value.
    A direct loop over the offsets of the window in key space; where window >= S every W(s) is the suffix [s, S)."""
    S = member_out.shape[1] if n_slots is None else n_slots
    lanes = npoints * members
    out = np.zeros((len(extremes), S, lanes))
    for j, (plane, kind, window) in enumerate(extremes):
        x = member_out[plane, :S, :lanes]
        valid = (x == x) & (x > -9000.0)
        fn = np.minimum if kind == "min" else np.maximum
        k = _key(np.where(valid, x, 0.0))
        if window >= S:
            ok = np.logical_and.accumulate(valid[::-1], axis=0)[::-1]
            acc = fn.accumulate(k[::-1], axis=0)[::-1]
        else:
            ok, acc = valid.copy(), k.copy()
            for d in range(1, window):                  # W(s) = [s, s + window - 1], cut at S
                ok[:S - d] &= valid[d:]
                acc[:S - d] = fn(acc[:S - d], k[d:])
        out[j] = np.where(ok, _unkey(acc), MISSING)
    return out.reshape(len(extremes), S, npoints, members)


def extremes_reference(member_out, npoints, members, extremes, quantiles=(), n_slots=None):
    """ext_stats [5 + nq, n_extremes, S, P]: stats_reference over the window values."""
    v = window_values(member_out, npoints, members, extremes, n_slots)
    return stats_reference(v.reshape(v.shape[0], v.shape[1], -1), npoints, members, quantiles)[0]


def area_values(member_out, npoints, members, extremes, areas, n_slots=None):
    """[n_extremes, S, n_areas, M]: valid at every station of the area, the minimum (maximum) over its stations."""
    v = window_values(member_out, npoints, members, extremes, n_slots)
    out = np.zeros(v.shape[:2] + (len(areas), members))
    for a, st in enumerate(areas):
        w = v[:, :, np.asarray(st), :]                                    # [X, S, stations, M]
        k = _key(w)
        for j, (_, kind, _) in enumerate(extremes):
            kk = k[j].min(axis=1) if kind == "min" else k[j].max(axis=1)
            out[j, :, a] = np.where((w[j] != MISSING).all(axis=1), _unkey(kk), MISSING)
    return out


def area_extremes_reference(member_out, npoints, members, extremes, areas, quantiles=(), n_slots=None):
    """area_ext_stats [5 + nq, n_extremes, S, n_areas]."""
    v = area_values(member_out, npoints, members, extremes, areas, n_slots)
    return stats_reference(v.reshape(v.shape[0], v.shape[1], -1), len(areas), members, quantiles)[0]


def _tiny_signed():
    """_tiny of test_ensemble_areas (3 stations x 2 members x 4 slots; station 0's member 1 has a NaN at slot 2,
    station 2 did not run) with signed zeros: station 0 member 0 is [1, -1, 1, -0.0], station 1 member 0
    [1, 1, +0.0, -0.0]."""
    x = _tiny()
    x[0, 3, 0] = -0.0
    x[0, 2, 2], x[0, 3, 2] = 0.0, -0.0
    return x


def test_restatement_known_answers():
    """Hand-computed, window 2 (W(3) = [3] is cut at the last slot)."""
    x = _tiny_signed()
    v = window_values(x, 3, 2, [(0, "min", 2), (0, "max", 2)])
    nan_cut = [1.0, MISSING, MISSING, 1.0]                          # station 0 member 1: the NaN at slot 2
    assert v[0, :, 0, 0].tolist() == [-1.0, -1.0, 0.0, 0.0] and np.signbit(v[0, 2:, 0, 0]).all()
    assert v[0, :, 0, 1].tolist() == nan_cut and v[1, :, 0, 1].tolist() == nan_cut
    # the tie of W(2) = {+0.0, -0.0} at station 1: -0.0 for the minimum, +0.0 for the maximum
    assert v[0, :, 1, 0].tolist() == [1.0, 0.0, 0.0, 0.0] and np.signbit(v[0, :, 1, 0]).tolist() == [0, 0, 1, 1]
    assert v[1, :, 1, 0].tolist() == [1.0, 1.0, 0.0, -0.0] and np.signbit(v[1, :, 1, 0]).tolist() == [0, 0, 0, 1]
    assert (v[:, :, 2] == MISSING).all()
    st = extremes_reference(x, 3, 2, [(0, "min", 2)], (0.5,))[:, 0]         # [planes, S, P]
    assert st[lib.ENS_NVALID, :, 0].tolist() == [2.0, 1.0, 1.0, 2.0]
    assert st[lib.ENS_MIN, 2, 0] == 0.0 and np.signbit(st[lib.ENS_MIN, 2, 0])
    assert not np.signbit(st[lib.ENS_MEAN, 2, 0])                          # +0.0 + -0.0 from +0.0
    assert st[lib.ENS_MEAN, 0, 0] == 0.0 and st[lib.ENS_MAX, 0, 0] == 1.0 and st[lib.ENS_NFIXED, 3, 0] == 0.5
    assert st[lib.ENS_NVALID, 0, 2] == 0.0 and (st[1:, :, 2] == MISSING).all()
    areas = [[0], [0, 1], [2], [1, 2]]
    av = area_values(x, 3, 2, [(0, "min", 2)], areas)[0]                     # [S, A, M]
    assert av[:, 1, 0].tolist() == [-1.0, -1.0, 0.0, 0.0] and np.signbit(av[2:, 1, 0]).all()
    assert av[:, 1, 1].tolist() == [-1.0, MISSING, MISSING, -1.0]
    ar = area_extremes_reference(x, 3, 2, [(0, "min", 2)], areas, (0.5,))[:, 0]
    assert same_bits(ar[..., 0], st[..., 0])
    assert ar[lib.ENS_NVALID, :, 1].tolist() == [2.0, 1.0, 1.0, 2.0]
    assert (ar[lib.ENS_NVALID, :, 2:] == 0.0).all() and (ar[1:, :, 2:] == MISSING).all()


def _identity_tensor(seed, P=12, M=7, S=30):
    rng = np.random.Generator(np.random.PCG64(seed))
    x = np.round(rng.normal(0.0, 1.0, (3, S, P * M + 4)), 1) + 0.0
    x[rng.random(x.shape) < 0.3] *= -0.0
    x[rng.random(x.shape) < 0.01] = np.nan
    x[:, :, 2 * M:3 * M] = MISSING
    return x


def test_restatement_identities():
    """(1) window 1 is the `stats` plane; (2) one-station areas are the station values, repeats and order change
    nothing; (3) the fraction of valid members whose minimum is < v (maximum > v) is the event probability of
    {plane, <, v} ({plane, >, v}) with the same window, per station and per area."""
    P, M, S = 12, 7, 30
    x = _identity_tensor(11, P, M, S)
    stats = stats_reference(x, P, M, QUANTILES)[0]
    for plane in range(3):
        for kind in ("min", "max"):
            assert same_bits(extremes_reference(x, P, M, [(plane, kind, 1)], QUANTILES)[:, 0], stats[:, plane])
    ext = [(0, "min", 3), (1, "max", 1), (2, "min", S), (0, "max", S + 4), (1, "min", 7)]
    ones = area_extremes_reference(x, P, M, ext, [[p] for p in range(P)], QUANTILES)
    assert same_bits(ones, extremes_reference(x, P, M, ext, QUANTILES))
    base = [[0, 3, 4, 9], list(range(P)), [5, 6]]
    again = [[9, 4, 0, 3, 4, 9, 0], list(range(P))[::-1] * 2, [6, 5, 5]]
    assert same_bits(area_extremes_reference(x, P, M, ext, base, QUANTILES),
                     area_extremes_reference(x, P, M, ext, again, QUANTILES))
    areas = [[0], [3, 4, 9], list(range(P)), [1, 2], [5, 6, 7, 8, 10, 11]]
    sv, av = window_values(x, P, M, ext), area_values(x, P, M, ext, areas)
    for j, (plane, kind, window) in enumerate(ext):
        for value in (-0.5, 0.0, 0.3):
            op = "<" if kind == "min" else ">"
            ev = [([(plane, op, value)], window)]
            for v, want in ((sv[j], events_reference(x, P, M, ev)[0]), (av[j], areas_reference(x, P, M, ev, areas)[0])):
                valid = v != MISSING
                n, c = valid.sum(axis=-1), (valid & ((v < value) if kind == "min" else (v > value))).sum(axis=-1)
                assert same_bits(np.where(n == 0, MISSING, c / np.maximum(n, 1)), want), (j, value)


def test_ensemble_extremes_builds_the_struct():
    ext = lib.ensemble_extremes([(TS, "min", 6), (ICE, "max", 3), (2, lib.ENS_WMAX, 1)])
    assert ext.n_extremes == 3
    assert [(e.plane, e.kind, e.window) for e in ext.extremes[:3]] == [(TS, 0, 6), (ICE, 1, 3), (2, 1, 1)]
    for bad in ([], [(TS, "mn", 6)], [(TS, 2, 6)], [(TS, -1, 6)]):
        with pytest.raises(ValueError):
            lib.ensemble_extremes(bad)


def test_ctypes_mirrors_match_the_c_header():
    probe = r"""
#include <stdio.h>
#include <stddef.h>
#include "roadsurf_b200.h"
#define S(t) printf("sizeof " #t " %zu\n", sizeof(t))
#define O(t, f) printf("offsetof " #t "." #f " %zu\n", offsetof(t, f))
int main(void) {
  S(RsEnsembleExtreme); S(RsEnsembleExtremes);
  O(RsEnsembleExtreme, plane); O(RsEnsembleExtreme, kind); O(RsEnsembleExtreme, window);
  O(RsEnsembleExtremes, n_extremes); O(RsEnsembleExtremes, extremes);
  printf("const ENS_MAX_EXTREMES %d\nconst ENS_WMIN %d\nconst ENS_WMAX %d\n", RS_ENS_MAX_EXTREMES, RS_ENS_WMIN,
         RS_ENS_WMAX);
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
        elif kind == "const":
            assert getattr(lib, name) == int(val), name
        else:
            t, f = name.split(".")
            assert getattr(getattr(lib, t), f).offset == int(val), name
        seen += 1
    assert seen == 10


def _prototype_argtypes(name):
    """The ctypes argument list that the prototype of `name` in the header asks for."""
    with open(os.path.join(ROOT, "include", "roadsurf_b200.h")) as f:
        text = f.read()
    args = re.search(r"\bint\s+" + name + r"\(([^)]*)\);", text).group(1)
    structs = {"RsHostBatch": lib.RsHostBatch, "RsEnsembleStatsSpec": lib.RsEnsembleStatsSpec,
               "RsEnsembleAreas": lib.RsEnsembleAreas, "RsEnsembleExtremes": lib.RsEnsembleExtremes,
               "InputSettings": abi.InputSettings, "InputParameters": abi.InputParameters}
    out = []
    for a in (" ".join(a.split()) for a in args.split(",")):
        m = re.match(r"const (\w+)\* \w+$", a)
        if a.startswith("int ") and "*" not in a:
            out.append(C.c_int)
        elif m and m.group(1) in structs:
            out.append(C.POINTER(structs[m.group(1)]))
        else:
            assert re.match(r"(const )?(double|int|void)\* \w+$", a), a
            out.append(C.c_void_p)
    return out


def test_ctypes_argument_lists_match_the_header():
    handle = lib.load()
    for name, n in (("roadsurf_ensemble_extremes", 13), ("roadsurf_run_ensemble_host_soa_extremes", 19)):
        assert name in lib.EXPORTS
        want = _prototype_argtypes(name)
        assert len(want) == n and list(getattr(handle, name).argtypes) == want, name


def _bad_extremes(out_nvar):
    """(extremes, what the error message names) for every malformed extremes set."""
    def ext(n=None, **kw):
        x = lib.ensemble_extremes([(TS, "min", 6), (ICE, "max", 2)])
        if n is not None:
            x.n_extremes = n
        for k, v in kw.items():
            setattr(x.extremes[1], k, v)
        return x
    return [(ext(0), b"1 to 8 extremes"), (ext(9), b"1 to 8 extremes"), (ext(-1), b"1 to 8 extremes"),
            (ext(kind=2), b"kind"), (ext(kind=-1), b"kind"), (ext(window=0), b"window"), (ext(window=-2), b"window"),
            (ext(plane=-1), b"plane"), (ext(plane=out_nvar), b"plane")]


def _host_args(P, M):
    base, pa, settings, params, start = _host_case(P=P)
    F = 2 * 120 + 2
    forcing = np.ascontiguousarray(np.stack([getattr(base, v).T for v in synth.RECORD_VARS], axis=1))
    local = np.zeros((lib.L_NLOCAL, P))
    r_f = lib.fork_record(base.record_step, F)
    mrec = np.zeros((base.nrec - r_f - 1, 11, P * M))
    hb = lib.RsHostBatch(npoints=P, sim_len=pa.sim_len, forcing_mode=1, n_records=base.nrec, nvar=11, out_stride=1,
                         forcing=forcing.ctypes.data, record_step=base.record_step.ctypes.data,
                         time_fields=pa.time.ctypes.data, local=local.ctypes.data)
    return hb, F, mrec, settings, params, (forcing, local, base, pa)


def test_bad_arguments_are_rejected_before_device_work():
    """Through roadsurf_ensemble_extremes and roadsurf_run_ensemble_host_soa_extremes (a well-placed fork): every
    malformed extremes set, outputs without ext, ext without an output, area_ext_stats without areas, the device
    entry's areas without area_ext_stats, malformed area sets and malformed specs return RS_ERR_BAD_ARGUMENT with a
    message.  The dew-point-deficit plane is legal through the device entry only.  Areas with area_ext_stats alone
    need no events."""
    handle = lib.load()
    P, M = 3, 4
    member_out = np.zeros((lib.O_NVAR_EXT, 5, 32))
    good = lib.ensemble_areas([[0, 2], [1]])
    buf = np.zeros(1 << 14)
    b = buf.ctypes.data
    spec = lib.stats_spec(QUANTILES)
    ext = lib.ensemble_extremes([(TS, "min", 6), (ICE, "max", 2)])
    dew = lib.ensemble_extremes([(DEWDEFICIT, "min", 3)])

    def device(sp, x, xs, areas, axs, out_nvar=lib.O_NVAR, n_out=5):
        return handle.roadsurf_ensemble_extremes(member_out.ctypes.data, out_nvar, n_out, 32, P, M, C.byref(sp),
                                                 None if x is None else C.byref(x), xs, 32,
                                                 None if areas is None else C.byref(areas), axs, None)
    dcases = [(spec, None, b, None, None, b"null extremes pointer"), (spec, None, None, good, b, b"null extremes pointer"),
              (spec, None, None, None, None, b"null extremes pointer"),
              (spec, ext, None, None, None, b"both NULL"), (spec, ext, None, good, None, b"both NULL"),
              (spec, ext, b, None, b, b"null area pointer"), (spec, ext, b, good, None, b"null area pointer")]
    dcases += [(spec, x, b, None, None, what) for x, what in _bad_extremes(lib.O_NVAR)]
    dcases += [(spec, ext, b, a, b, what) for a, what in _bad_areas(P) if a is not None]
    dcases += [(sp, ext, b, None, None, what) for sp, what in _bad_specs(lib.O_NVAR)]
    dcases += [(spec, dew, b, None, None, b"plane")]
    for sp, x, xs, areas, axs, what in dcases:
        assert device(sp, x, xs, areas, axs) == RS_ERR_BAD_ARGUMENT, what
        assert what in handle.roadsurf_last_error(), what
    for x, what in _bad_extremes(lib.O_NVAR_EXT):
        assert device(spec, x, b, None, None, lib.O_NVAR_EXT) == RS_ERR_BAD_ARGUMENT and what in handle.roadsurf_last_error()
    # ld < npoints with ext_stats
    assert handle.roadsurf_ensemble_extremes(member_out.ctypes.data, lib.O_NVAR, 5, 32, P, M, C.byref(spec),
                                             C.byref(ext), b, 2, None, None, None) == RS_ERR_BAD_ARGUMENT
    # good arguments pass every check (n_out = 0: nothing to do): the extended plane, areas with a spec without events
    assert device(spec, dew, b, None, None, lib.O_NVAR_EXT, n_out=0) == 0
    assert device(spec, ext, None, good, b, n_out=0) == 0 and device(spec, ext, b, good, b, n_out=0) == 0

    hb, F, mrec, settings, params, keep = _host_args(P, M)
    stats, prob = np.zeros(1 << 16), np.zeros(1 << 16)
    ev_spec = lib.stats_spec(QUANTILES, (), [([(TS, "<", 0.0), (WATER, ">", 0.1)], 3)])

    def host(sp, areas, area_prob, onset, area_onset, x, xs, axs):
        return handle.roadsurf_run_ensemble_host_soa_extremes(
            C.byref(hb), mrec.ctypes.data, M, F, None, C.byref(sp), stats.ctypes.data, prob.ctypes.data, None, None,
            None if areas is None else C.byref(areas), area_prob, onset, area_onset,
            None if x is None else C.byref(x), xs, axs, C.byref(settings), C.byref(params))
    hcases = [(spec, None, None, None, None, None, b, None, b"null extremes pointer"),
              (spec, good, None, None, None, None, None, b, b"null extremes pointer"),
              (spec, None, None, None, None, ext, None, None, b"both NULL"),
              (spec, good, b, None, None, ext, None, None, b"both NULL"),
              (spec, None, None, None, None, ext, b, b, b"null area pointer"),
              (spec, good, None, None, None, ext, b, None, b"null area pointer"),
              (spec, good, b, None, None, ext, b, None, b"at least one event"),       # area_prob still needs events
              (spec, None, None, None, None, dew, b, None, b"plane")]
    hcases += [(spec, None, None, None, None, x, b, None, what) for x, what in _bad_extremes(lib.O_NVAR)]
    hcases += [(spec, a, None, None, None, ext, None, b, what) for a, what in _bad_areas(P) if a is not None]
    hcases += [(sp, None, None, None, None, ext, b, None, what) for sp, what in _bad_specs(lib.O_NVAR)]
    for sp, areas, area_prob, onset, area_onset, x, xs, axs, what in hcases:
        assert host(sp, areas, area_prob, onset, area_onset, x, xs, axs) == RS_ERR_BAD_ARGUMENT, what
        assert what in handle.roadsurf_last_error(), what
    if handle.roadsurf_device_count() == 0:
        # good outputs pass the checks and then find no device; an extremes-only call with areas needs no events
        assert host(spec, good, None, None, None, ext, b, b) == -1 and host(spec, None, None, None, None, ext, b, None) == -1
        assert host(ev_spec, good, b, b, b, ext, None, b) == -1


# ---- GPU --------------------------------------------------------------------------------------------------------

def _kernel_tensor(M, seed):
    """About 2 000 slots, NaN and -9999.0 holes in half the lanes, signed zeros, +inf and -inf, an all-missing
    station (3)."""
    rng = np.random.Generator(np.random.PCG64(seed + M))
    P, S, out_nvar = min(150, max(5, 2400 // M)), 2003, lib.O_NVAR
    ldm = (P * M + 31) // 32 * 32
    x = np.round(rng.normal(0.0, 2.0, (out_nvar, S, ldm)), 0) + 0.0
    x[rng.random(x.shape) < 0.5] *= -1.0                      # about half the zeros are -0.0
    x[rng.random(x.shape) < 0.0005] = np.inf
    x[rng.random(x.shape) < 0.0002] = -np.inf
    holes = (rng.random(x.shape) < 0.0005) & (rng.random(ldm) < 0.5)
    x[holes & (rng.random(x.shape) < 0.5)] = np.nan
    x[holes & ~np.isnan(x)] = MISSING
    x[:, :, 3 * M:4 * M] = MISSING
    return rng, x, P, S


def _device_stats(rslib, values, members, quantiles):
    """roadsurf_ensemble_stats over restated values [n <= 9, S, columns, M] as a member tensor (padded to the nine
    extended planes with MISSING): [5 + nq, n, S, columns]."""
    import torch
    n, S, cols = values.shape[:3]
    t = np.full((lib.O_NVAR_EXT, S, cols * members), MISSING)
    t[:n] = values.reshape(n, S, -1)
    stats, _ = rslib.ensemble_stats(torch.from_numpy(t).cuda(), cols, members, lib.stats_spec(quantiles))
    return stats.cpu().numpy()[:, :n]


def _zero(a):
    """-0.0 -> +0.0: NumPy's min and sort do not keep member order among -0.0 / +0.0 ties, the statistics kernel does."""
    return np.asarray(a) + 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("M", [1, 7, 30, 32, 33, 128])
def test_extremes_kernels_equal_the_restatement(rslib, M):
    """Windows 1, 2, 63, 64, 65, S and S + 7 in both kinds over the six planes, in two calls of 7 extremes; per station
    and per area, bit for bit the statistics kernel over the restated window values, and the NumPy restatement (the sign
    of a zero aside where members tie at -0.0 / +0.0: stats_reference does not keep their member order)."""
    import torch
    rng, x, P, S = _kernel_tensor(M, 500)
    windows = [1, 2, 63, 64, 65, S, S + 7]
    calls = [[(j % lib.O_NVAR, kind, w) for j, w in enumerate(windows)] for kind in ("min", "max")]
    area_lists = _random_areas(rng, P, 3)
    areas = rslib.ensemble_areas(area_lists)
    xd = torch.from_numpy(x).cuda()
    spec = lib.stats_spec(QUANTILES)
    for ext in calls:
        xs, ar = rslib.ensemble_extremes_device(xd, P, M, spec, rslib.ensemble_extremes(ext), areas)
        xs, ar = xs.cpu().numpy(), ar.cpu().numpy()
        want = extremes_reference(x, P, M, ext, QUANTILES)
        want_a = area_extremes_reference(x, P, M, ext, area_lists, QUANTILES)
        dev = _device_stats(rslib, window_values(x, P, M, ext), M, QUANTILES)
        dev_a = _device_stats(rslib, area_values(x, P, M, ext, area_lists), M, QUANTILES)
        assert xs.shape == want.shape == dev.shape and ar.shape == want_a.shape == dev_a.shape
        for j in range(len(ext)):
            assert same_bits(xs[:, j], dev[:, j]) and same_bits(ar[:, j], dev_a[:, j]), (M, ext[j])
            assert same_bits(_zero(xs[:, j]), _zero(want[:, j])), (M, ext[j])
            assert same_bits(_zero(ar[:, j]), _zero(want_a[:, j])), (M, ext[j])
        if M == 1:                                          # no ties: the restatement holds for the signs too
            assert same_bits(xs, want) and same_bits(ar, want_a)
        assert (want[lib.ENS_NVALID] == 0.0).any() and (want[lib.ENS_MAX] == np.inf).any()
        assert (want_a[lib.ENS_NVALID] == 0.0).any() and (M == 1 or (want_a[lib.ENS_NVALID] == M).any())


@pytest.mark.gpu
def test_window_one_equals_the_statistics_planes(rslib):
    """Extremes of window 1 over the six planes equal roadsurf_ensemble_stats' planes bit for bit."""
    import torch
    rng, x, P, S = _kernel_tensor(30, 600)
    xd = torch.from_numpy(x[:, :300]).contiguous().cuda()
    spec = lib.stats_spec(QUANTILES)
    stats, _ = rslib.ensemble_stats(xd, P, 30, spec)
    ext = [(p, "min" if p % 2 else "max", 1) for p in range(lib.O_NVAR)]
    xs, none = rslib.ensemble_extremes_device(xd, P, 30, spec, rslib.ensemble_extremes(ext))
    assert none is None and same_bits(xs.cpu().numpy(), stats.cpu().numpy())


EXTREMES = [(TS, "min", 6), (TS, "min", 12), (ICE, "max", 6), (SNOW, "max", 6)]


@pytest.mark.gpu
def test_device_entry_then_extremes_equal_the_restatement(rslib):
    """roadsurf_run_ensemble_device with out_nvar = RS_O_NVAR_EXT (coarse records, coupling + relaxation), then
    roadsurf_ensemble_extremes on its member_out, a dew-point-deficit extreme included."""
    P, M = 60, 5
    c = _Case(P, M, 3, 6, seed=4606)
    spec = lib.stats_spec(QUANTILES, [(TS, "<", 0.0)], ROAD_EVENTS)
    ens = _device_ensemble(rslib, c, spec)
    ens.run()
    ext = EXTREMES + [(DEWDEFICIT, "min", 3), (DEWDEFICIT, "max", 1)]
    area_lists = [[7], [0, 1, 2, 3], list(range(0, P, 3)), list(range(P)), [59, 12, 33, 12]]
    xs, ar = rslib.ensemble_extremes_device(ens.member_out, P, M, spec, rslib.ensemble_extremes(ext),
                                            rslib.ensemble_areas(area_lists))
    mo = ens.member_out.cpu().numpy()
    n = ens.n_slots
    want = extremes_reference(mo, P, M, ext, QUANTILES, n)
    assert same_bits(xs.cpu().numpy()[:, :, :n], want)
    assert same_bits(ar.cpu().numpy()[:, :, :n], area_extremes_reference(mo, P, M, ext, area_lists, QUANTILES, n))
    assert (want[lib.ENS_STD] > 0.0).any()


@pytest.mark.gpu
def test_host_entry_extremes_in_station_chunks(rslib):
    """roadsurf_run_ensemble_host_soa_extremes in one and in eight station chunks, areas straddling the chunks:
    ext_stats and area_ext_stats equal the restatement of the device ensemble's member_out; stats, prob, area_prob,
    onset and area_onset are bitwise those of the call without extremes; d2h_bytes grows by exactly ext_stats and
    area_ext_stats; the extremes add three launches per chunk and two; an extremes-only call (stats and prob NULL, areas
    with a spec without events) adds the same to a call with neither."""
    P, M = 50, 6
    c = _Case(P, M, 3, 6, seed=4707)
    events = [e for e in ROAD_EVENTS if all(cd[0] < lib.O_NVAR for cd in e[0])]
    spec = lib.stats_spec(QUANTILES, [(TS, "<", 0.0)], events)
    ens = _device_ensemble(rslib, c, spec, extended=False)
    ens.run()
    area_lists = [[0], [49], [5, 6, 7, 8], list(range(3, 30)), list(range(P)), [48, 1, 20, 34, 6, 13],
                  list(range(0, P, 7)), [44, 45, 46, 47, 48, 49, 0]]
    areas = rslib.ensemble_areas(area_lists)
    ext = rslib.ensemble_extremes(EXTREMES)
    mo = ens.member_out.cpu().numpy()
    want = extremes_reference(mo, P, M, EXTREMES, QUANTILES, ens.n_slots)
    want_a = area_extremes_reference(mo, P, M, EXTREMES, area_lists, QUANTILES, ens.n_slots)
    sh = ens.shared
    forcing = sh.forcing[:, :, :P].cpu().numpy().copy()
    local = sh.local[:, :P].cpu().numpy().copy()
    hor = sh.horizons[:, :P].cpu().numpy().copy()
    mrec = synth.member_record_tensor(c.mrecs, c.r_f)
    A, X, rows = len(area_lists), len(EXTREMES), lib.ENS_NFIXED + len(QUANTILES)
    no_events = lib.stats_spec(QUANTILES)

    def run(sp=spec, **kw):
        res = rslib.run_ensemble_host_soa(c.settings, c.params, forcing, c.base.record_step.astype(np.int32),
                                          c.pa.time, local, mrec, M, c.F, sp, horizons=hor, out_stride=60,
                                          coupling_window_end=sh.coupling_window_end,
                                          latest_obs_index=np.full(P, c.forecast_step + 1, dtype=np.int32), **kw)
        return res, rslib.last_batch_stats()
    results = {}
    for cap in (0, 7 * M):
        rslib.set_option("max_points_per_device_batch", cap)
        try:
            plain, st0 = run(areas=areas, onset=True)
            res, st1 = run(areas=areas, onset=True, extremes=ext)
            neither, st2 = run(stats=False, prob=False)
            only, st3 = run(no_events, areas=areas, stats=False, prob=False, area_prob=False, extremes=ext)
        finally:
            rslib.set_option("max_points_per_device_batch", 0)
        groups = 1 if cap == 0 else 8
        assert st0["groups"] == st1["groups"] == st2["groups"] == st3["groups"] == groups
        n_m = res["stats"].shape[2]
        assert n_m == ens.n_slots
        assert res["ext_stats"].shape == (rows, X, n_m, P) and res["area_ext_stats"].shape == (rows, X, n_m, A)
        for r in (res, only):
            assert same_bits(r["ext_stats"], want), cap
            assert same_bits(r["area_ext_stats"], want_a), cap
        for k in ("stats", "prob", "area_prob", "onset", "area_onset"):
            assert same_bits(res[k], plain[k]), k
        assert set(only) == {"ext_stats", "area_ext_stats"} and set(neither) == set()
        grow = 8 * rows * X * n_m * (P + A)
        assert st1["d2h_bytes"] == st0["d2h_bytes"] + grow and st3["d2h_bytes"] == st2["d2h_bytes"] + grow
        assert st1["kernel_launches"] == st0["kernel_launches"] + 3 * groups + 2
        assert st3["kernel_launches"] == st2["kernel_launches"] + 3 * groups + 2
        results[cap] = res
    assert same_bits(results[0]["ext_stats"], results[7 * M]["ext_stats"])
    assert ((want_a[lib.ENS_STD] > 0.0) & (want_a[lib.ENS_NVALID] == M)).any()


@pytest.mark.gpu
def test_extremes_are_written_inside_their_planes_only(rslib):
    """ext_stats and area_ext_stats pre-filled with a sentinel, longer than their planes and with ld > npoints; the
    extremes array filled beyond n_extremes: exactly the planes of n_extremes extremes, the npoints columns of each row
    and their area values are written."""
    import torch
    rng = np.random.Generator(np.random.PCG64(8))
    P, M, S, ld = 40, 9, 70, 64
    x = np.round(rng.normal(0.0, 2.0, (lib.O_NVAR, S, P * M)), 1) + 0.0
    full = [(TS, "min", 5), (ICE, "max", 80), (2, "min", 1)]
    ext = lib.ensemble_extremes(full)
    ext.n_extremes = 2
    spec = lib.stats_spec((0.25, 0.5))
    area_lists = [[0, 5], list(range(P)), [39]]
    areas = lib.ensemble_areas(area_lists)
    rows = lib.ENS_NFIXED + 2
    n_xs, n_ar = rows * 2 * S * ld, rows * 2 * S * 3
    xs = torch.full((n_xs + 1000,), 777.0, dtype=torch.float64, device="cuda")
    ar = torch.full((n_ar + 1000,), 777.0, dtype=torch.float64, device="cuda")
    xd = torch.from_numpy(x).cuda()
    lib._check(lib.load().roadsurf_ensemble_extremes(xd.data_ptr(), lib.O_NVAR, S, P * M, P, M, C.byref(spec),
                                                     C.byref(ext), xs.data_ptr(), ld, C.byref(areas), ar.data_ptr(),
                                                     None))
    torch.cuda.synchronize()
    o, a = xs.cpu().numpy(), ar.cpu().numpy()
    assert (o[n_xs:] == 777.0).all() and (a[n_ar:] == 777.0).all() and (a[:n_ar] != 777.0).all()
    planes = o[:n_xs].reshape(rows, 2, S, ld)
    assert (planes[..., P:] == 777.0).all() and (planes[..., :P] != 777.0).all()
    assert same_bits(planes[..., :P], extremes_reference(x, P, M, full[:2], (0.25, 0.5)))
    assert same_bits(a[:n_ar].reshape(rows, 2, S, 3), area_extremes_reference(x, P, M, full[:2], area_lists, (0.25, 0.5)))


# ---- long segments ----------------------------------------------------------------------------------------------

def _segment_length(area_lists, n_extremes, chunks):
    """The stations per segment the library plans for the area extremes (segment_length in rs_host.cu): about 2^15
    (segment, extreme) work items per chunk, between 1 and 64."""
    memberships = sum(len(set(a)) for a in area_lists)
    return min(64, max(1, memberships * n_extremes // (chunks << 15)))


def _many_areas(rng, P, n, lo, hi):
    """n random areas of lo to hi distinct stations in random order, some with a station repeated."""
    areas = []
    for k in range(n):
        a = rng.choice(P, int(rng.integers(lo, hi + 1)), replace=False).tolist()
        areas.append(a + a[:1] if k % 5 == 0 else a)
    return areas


LONG_EXTREMES = [(0, "min", 1), (0, "max", 2), (1, "min", 5), (2, "max", 3), (3, "min", 200), (4, "max", 40),
                 (5, "min", 7), (0, "min", 64)]


@pytest.mark.gpu
def test_area_extremes_in_long_segments_equal_the_restatement(rslib):
    """8 extremes over 300 areas of 80 to 140 of 150 stations: about 33 000 memberships, so that a segment holds 7
    stations and the accumulate kernel combines them in key space before its atomics.  NaN and -9999.0 holes, an
    all-missing station; bit for bit against the restatement (no signed zeros, so no -0.0 / +0.0 ties)."""
    import torch
    rng = np.random.Generator(np.random.PCG64(909))
    P, M, S = 150, 7, 300
    x = np.round(rng.normal(0.0, 2.0, (lib.O_NVAR, S, P * M)), 1) + 0.0
    x[x == 0.0] = 0.05
    holes = (rng.random(x.shape) < 0.001) & (rng.random(P * M) < 0.5)
    x[holes & (rng.random(x.shape) < 0.5)] = np.nan
    x[holes & ~np.isnan(x)] = MISSING
    x[:, :, 9 * M:10 * M] = MISSING
    area_lists = _many_areas(rng, P, 300, 80, 140)
    assert _segment_length(area_lists, len(LONG_EXTREMES), 1) >= 7
    xs, ar = rslib.ensemble_extremes_device(torch.from_numpy(x).cuda(), P, M, lib.stats_spec(QUANTILES),
                                            rslib.ensemble_extremes(LONG_EXTREMES), rslib.ensemble_areas(area_lists))
    want_a = area_extremes_reference(x, P, M, LONG_EXTREMES, area_lists, QUANTILES)
    assert same_bits(xs.cpu().numpy(), extremes_reference(x, P, M, LONG_EXTREMES, QUANTILES))
    assert same_bits(ar.cpu().numpy(), want_a)
    assert (want_a[lib.ENS_NVALID] == 0.0).any() and (want_a[lib.ENS_NVALID] == M).any()
    assert len(np.unique(want_a[lib.ENS_MEAN])) > 100                    # the areas' results differ


@pytest.mark.gpu
def test_host_entry_area_extremes_in_long_segments(rslib):
    """The host entry with 8 extremes over 1 500 areas of 40 to 50 of 50 stations (about 67 000 memberships): segments
    of 16 stations in one chunk and of 2 in eight chunks.  The device entry on the device ensemble's member_out and the
    host entry in both chunkings give area_ext_stats and ext_stats bit for bit equal to the statistics kernel over the
    restated values, and equal to the NumPy restatement (bit for bit where member_out holds no -0.0, else up to the
    sign of a zero where members tie at -0.0 / +0.0)."""
    P, M = 50, 6
    c = _Case(P, M, 3, 6, seed=4808)
    spec = lib.stats_spec(QUANTILES)
    ens = _device_ensemble(rslib, c, spec, extended=False)
    ens.run()
    rng = np.random.Generator(np.random.PCG64(4808))
    area_lists = _many_areas(rng, P, 1500, 40, 50)
    X = len(LONG_EXTREMES)
    assert _segment_length(area_lists, X, 1) >= 16 and _segment_length(area_lists, X, 8) >= 2
    areas = rslib.ensemble_areas(area_lists)
    ext = rslib.ensemble_extremes(LONG_EXTREMES)
    mo = ens.member_out.cpu().numpy()
    n = ens.n_slots
    want = extremes_reference(mo, P, M, LONG_EXTREMES, QUANTILES, n)
    want_a = area_extremes_reference(mo, P, M, LONG_EXTREMES, area_lists, QUANTILES, n)
    dev = _device_stats(rslib, window_values(mo, P, M, LONG_EXTREMES, n), M, QUANTILES)
    dev_a = _device_stats(rslib, area_values(mo, P, M, LONG_EXTREMES, area_lists, n), M, QUANTILES)
    signed_zero = bool((np.signbit(mo[:, :n, :P * M]) & (mo[:, :n, :P * M] == 0.0)).any())

    def check(got, got_a, what):
        assert same_bits(got, dev) and same_bits(got_a, dev_a), what
        assert same_bits(_zero(got), _zero(want)) and same_bits(_zero(got_a), _zero(want_a)), what
        if not signed_zero:
            assert same_bits(got, want) and same_bits(got_a, want_a), what
    xs, ar = rslib.ensemble_extremes_device(ens.member_out, P, M, spec, ext, areas)
    check(xs.cpu().numpy()[:, :, :n], ar.cpu().numpy()[:, :, :n], "device entry")
    sh = ens.shared
    for cap, groups in ((0, 1), (7 * M, 8)):
        rslib.set_option("max_points_per_device_batch", cap)
        try:
            res = rslib.run_ensemble_host_soa(c.settings, c.params, sh.forcing[:, :, :P].cpu().numpy().copy(),
                                              c.base.record_step.astype(np.int32), c.pa.time,
                                              sh.local[:, :P].cpu().numpy().copy(),
                                              synth.member_record_tensor(c.mrecs, c.r_f), M, c.F, spec,
                                              horizons=sh.horizons[:, :P].cpu().numpy().copy(), out_stride=60,
                                              coupling_window_end=sh.coupling_window_end,
                                              latest_obs_index=np.full(P, c.forecast_step + 1, dtype=np.int32),
                                              areas=areas, stats=False, prob=False, area_prob=False, extremes=ext)
            st = rslib.last_batch_stats()
        finally:
            rslib.set_option("max_points_per_device_batch", 0)
        assert st["groups"] == groups
        check(res["ext_stats"], res["area_ext_stats"], cap)
    assert len(np.unique(want_a[lib.ENS_MEAN])) > 100                    # the areas' results differ
