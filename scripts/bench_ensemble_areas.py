"""Ensemble area event probabilities (RsEnsembleAreas) on one GPU: the two area kernels against the station events
kernel on the same member tensor, and the host entry with area probabilities alone against member_out.  Prints one
JSON line per shape.

  ex1-ens, c3-ens: the shapes of scripts/bench_ensemble.py (M = 30, an output slot every 120 steps = 1 h), the member
  tensor and the 4 events of scripts/bench_ensemble_events.py (3 conditions, window 6 h).
  Areas: routes of 50 stations drawn at random (a random permutation of the stations cut into routes, so that a
  route's member lanes are not adjacent and the routes partition the stations), plus 20 districts of 5 % of the
  stations each, drawn independently (they overlap each other and the routes).  So every station is in about two
  areas.

  - kernel times: torch.profiler (CUDA activities) over --reps calls after a warm-up, mean per launch of the
    accumulate and the finalize kernel, and of the station events kernel (roadsurf_ensemble_stats, stats NULL) on the
    same member tensor; separately, CUDA events around one whole roadsurf_ensemble_area_events call (the host's
    planning, the plan's upload, the accumulator reset and both kernels), best of --reps;
  - bytes the area kernels must read: each referenced plane once per (event, area membership), n_conditions x S x M x 8
    bytes per membership and event, plus area_prob written, over the two kernels' time, against a device-to-device copy
    measured in the same process; the same once-per-event bound for the station events kernel;
  - host entry: wall clock around roadsurf_run_ensemble_host_soa_areas with areas alone (prob NULL, no member_out)
    and with member_out instead of areas, best of 2 after a warm-up call, and d2h_bytes of each.
The card's name and power limit are read in the same process.  Usage:
  python scripts/bench_ensemble_areas.py [--shape ex1-ens|c3-ens|all] [--members 30] [--stations N] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import bench_ensemble  # noqa: E402
from bench_ensemble_events import EVENTS, copy_peak_gbs, member_forcing_on_device  # noqa: E402
from roadsurf_b200 import lib  # noqa: E402

ROUTE = 50
DISTRICTS, DISTRICT_FRACTION = 20, 0.05


def make_areas(P, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    perm = rng.permutation(P)
    routes = [perm[k:k + ROUTE] for k in range(0, P, ROUTE)]
    size = max(1, int(round(DISTRICT_FRACTION * P)))
    districts = [rng.choice(P, size, replace=False) for _ in range(DISTRICTS)]
    return routes + districts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shape", default="all")
    ap.add_argument("--members", type=int, default=30)
    ap.add_argument("--stations", type=int, default=0, help="override the station count")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    handle = lib.load()
    if handle.roadsurf_device_count() < 1:
        raise SystemExit("no CUDA device visible")
    shapes = list(bench_ensemble.SHAPES) if args.shape == "all" else [args.shape]
    name = bench_ensemble.card()
    peak = copy_peak_gbs(torch)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

    def timed(fn, reps):
        fn()
        torch.cuda.synchronize()
        best = float("inf")
        for _ in range(reps):
            ev[0].record()
            fn()
            ev[1].record()
            torch.cuda.synchronize()
            best = min(best, ev[0].elapsed_time(ev[1]))
        return best

    for shape in shapes:
        P, M = args.stations or bench_ensemble.SHAPES[shape]["stations"], args.members
        c = bench_ensemble.build(shape, P, M, member_records=False)
        spec = lib.stats_spec(events=EVENTS)
        area_lists = make_areas(P, seed=11)
        areas = lib.ensemble_areas(area_lists)
        A, E = len(area_lists), len(EVENTS)
        memberships = int(sum(len(a) for a in area_lists))
        lib.set_model(c["settings"], c["params"])
        sh = lib.DeviceBatch(P, c["sim_len"], n_records=c["base"].nrec, coarse=True, horizons=True, coupling=True,
                             state=True, out_stride=120)
        sh.load_records(c["base"])
        sh.time_fields.copy_(torch.from_numpy(c["time"]))
        sh.local[:, :P] = torch.from_numpy(c["local"])
        sh.horizons[:, :P] = torch.from_numpy(c["horizons"])
        sh.coupling_window_end = c["wend"]
        ens = lib.EnsembleBatch(sh, M, c["F"], spec)
        member_forcing_on_device(torch, ens, sh, c["r_f"], P, M, seed=7)
        ens.run()
        torch.cuda.synchronize()
        S, ldm, ld = ens.n_slots, ens.ld_members, sh.ld
        mo = ens.member_out
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        f64 = dict(dtype=torch.float64, device="cuda")
        prob_e = torch.empty((E, S, ld), **f64)
        area_prob = torch.empty((E, S, A), **f64)

        def run_areas():
            lib._check(handle.roadsurf_ensemble_area_events(mo.data_ptr(), lib.O_NVAR, S, ldm, P, M, C.byref(spec),
                                                            C.byref(areas), area_prob.data_ptr(), stream))

        def run_events():
            lib._check(handle.roadsurf_ensemble_stats(mo.data_ptr(), lib.O_NVAR, S, ldm, P, M, C.byref(spec),
                                                      None, prob_e.data_ptr(), ld, stream))
        t_call = timed(run_areas, args.reps)
        timed(run_events, 1)
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(args.reps):
                run_areas()
                run_events()
            torch.cuda.synchronize()
        kt = {}
        for k in prof.key_averages():
            for tag in ("rs_ens_area_accumulate_kernel", "rs_ens_area_finalize_kernel", "rs_ens_events_kernel"):
                if tag in k.key:
                    kt[tag] = (getattr(k, "device_time", None) or k.cuda_time) / 1e3   # mean per launch, ms
        t_acc, t_fin = kt["rs_ens_area_accumulate_kernel"], kt["rs_ens_area_finalize_kernel"]
        t_areas, t_events = t_acc + t_fin, kt["rs_ens_events_kernel"]
        conds = sum(len(cd) for cd, _ in EVENTS)
        area_bytes = 8 * (conds * S * M * memberships + E * S * A)
        ev_bytes = 8 * (conds * S * P * M + E * S * P)
        ap_dev = area_prob.cpu().numpy()
        del prob_e, area_prob

        # host entry: area probabilities alone, against member_out
        mrec = ens.member_forcing[1:, :, :P * M].contiguous().cpu().numpy()
        hargs = (c["settings"], c["params"], c["forcing"], c["base"].record_step.astype(np.int32), c["time"],
                 c["local"], mrec, M, c["F"], spec)
        hkw = dict(horizons=c["horizons"], out_stride=120, coupling_window_end=c["wend"],
                   latest_obs_index=np.full(P, c["F"] - 1, dtype=np.int32))
        del ens, mo, sh
        torch.cuda.empty_cache()

        def host(reps=2, **kw):
            lib.run_ensemble_host_soa(*hargs, **hkw, **kw)
            best, res, st = float("inf"), None, None
            for _ in range(reps):
                res = None
                t0 = time.perf_counter()
                res = lib.run_ensemble_host_soa(*hargs, **hkw, **kw)
                t = (time.perf_counter() - t0) * 1e3
                if t < best:
                    best, st = t, lib.last_batch_stats()
            return best, st, res
        t_host_ar, st_ar, _ = host(areas=areas, prob=False)
        t_host_mo, st_mo, _ = host(member_out=True)
        del mrec
        lib.release_workspace()
        line = dict(shape=shape, card=name, stations=P, members=M, member_slots=S, n_events=E,
                    conditions_per_event=3, window=6, routes=len(area_lists) - DISTRICTS, route_stations=ROUTE,
                    districts=DISTRICTS, district_stations=int(round(DISTRICT_FRACTION * P)), n_areas=A,
                    memberships=memberships, member_out_gb=8 * lib.O_NVAR * S * P * M / 1e9, copy_peak_gbs=peak,
                    accumulate_kernel_ms=t_acc, finalize_kernel_ms=t_fin, area_kernels_ms=t_areas,
                    area_call_ms=t_call, events_kernel_ms=t_events, areas_over_events=t_areas / t_events,
                    area_bytes_bound=area_bytes, area_gbs=area_bytes / t_areas / 1e6,
                    area_share_of_copy_peak=area_bytes / t_areas / 1e6 / peak,
                    events_bytes_bound=ev_bytes, events_gbs=ev_bytes / t_events / 1e6,
                    area_prob_fraction_in_0_1=float(((ap_dev > 0) & (ap_dev < 1)).mean()),
                    host_areas_only_ms=t_host_ar, host_areas_only_d2h_bytes=st_ar["d2h_bytes"],
                    host_areas_only_phases=st_ar,
                    host_member_out_ms=t_host_mo, host_member_out_d2h_bytes=st_mo["d2h_bytes"],
                    host_member_out_phases=st_mo)
        print(json.dumps(line), flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
