"""Ensemble event onset (roadsurf_ensemble_onset) on one GPU: the onset kernels against the event kernels on the same
member tensor, and the host entry with onset and area onset alone against member_out.  Prints one JSON line per shape.

  ex1-ens, c3-ens: the shapes, member tensor, 4 events of 3 conditions and areas of scripts/bench_ensemble_areas.py.

  - kernel times: torch.profiler (CUDA activities) over --reps calls after a warm-up, mean per launch of
    rs_ens_onset_kernel (onset planes and the workspace) and of the two area onset kernels; in the same window the
    station events kernel (roadsurf_ensemble_stats, stats NULL) and the two area event kernels
    (roadsurf_ensemble_area_events) on the same member tensor;
  - read bound of the station onset kernel: each referenced plane once per event over all S slots,
    n_conditions x S x P x M x 8 bytes per event (a scan that stops at X reads less), plus the onset planes and the
    workspace written; of the area onset kernels: the workspace {O, X} once per (event, area membership), 8 x M bytes,
    plus area_onset written.  Rates are against a device-to-device copy measured in the same process;
  - host entry: wall clock around roadsurf_run_ensemble_host_soa_onset with onset and area onset alone (prob and
    area_prob NULL, no member_out) and with member_out alone, best of 2 after a warm-up call, and d2h_bytes of each.
The card's name and power limit are read in the same process.  Usage:
  python scripts/bench_ensemble_onset.py [--shape ex1-ens|c3-ens|all] [--members 30] [--stations N] [--out FILE]
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
from bench_ensemble_areas import DISTRICTS, make_areas  # noqa: E402
from bench_ensemble_events import EVENTS, copy_peak_gbs, member_forcing_on_device  # noqa: E402
from roadsurf_b200 import lib  # noqa: E402

KERNELS = ("rs_ens_onset_kernel", "rs_ens_area_onset_accumulate_kernel", "rs_ens_area_onset_finalize_kernel",
           "rs_ens_events_kernel", "rs_ens_area_accumulate_kernel", "rs_ens_area_finalize_kernel")


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
        onset = torch.empty((E, S, ld), **f64)
        area_onset = torch.empty((E, S, A), **f64)

        def run_onset():
            lib._check(handle.roadsurf_ensemble_onset(mo.data_ptr(), lib.O_NVAR, S, ldm, P, M, C.byref(spec),
                                                      onset.data_ptr(), ld, C.byref(areas), area_onset.data_ptr(),
                                                      stream))

        def run_events():
            lib._check(handle.roadsurf_ensemble_stats(mo.data_ptr(), lib.O_NVAR, S, ldm, P, M, C.byref(spec),
                                                      None, prob_e.data_ptr(), ld, stream))
            lib._check(handle.roadsurf_ensemble_area_events(mo.data_ptr(), lib.O_NVAR, S, ldm, P, M, C.byref(spec),
                                                            C.byref(areas), area_prob.data_ptr(), stream))
        run_onset()
        run_events()
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(args.reps):
                run_onset()
                run_events()
            torch.cuda.synchronize()
        kt = {}
        for k in prof.key_averages():
            for tag in KERNELS:
                if tag in k.key:
                    kt[tag] = (getattr(k, "device_time", None) or k.cuda_time) / 1e3   # mean per launch, ms
        t_on = kt["rs_ens_onset_kernel"]
        t_area_on = kt["rs_ens_area_onset_accumulate_kernel"] + kt["rs_ens_area_onset_finalize_kernel"]
        t_events = kt["rs_ens_events_kernel"]
        t_area_ev = kt["rs_ens_area_accumulate_kernel"] + kt["rs_ens_area_finalize_kernel"]
        conds = sum(len(cd) for cd, _ in EVENTS)
        on_bytes = 8 * (conds * S * P * M + E * S * P + E * P * M)
        area_on_bytes = 8 * (E * M * memberships + E * S * A)
        on_dev = onset[:, :, :P].cpu().numpy()
        # the identity at the last slot: onset equals the event at slot 0 with window S
        full = lib.stats_spec(events=[(cd, S) for cd, _ in EVENTS])
        lib._check(handle.roadsurf_ensemble_stats(mo.data_ptr(), lib.O_NVAR, S, ldm, P, M, C.byref(full), None,
                                                  prob_e.data_ptr(), ld, stream))
        torch.cuda.synchronize()
        identity_last_slot = bool(np.array_equal(prob_e[:, 0, :P].cpu().numpy().view(np.int64),
                                                 on_dev[:, S - 1].view(np.int64)))
        del prob_e, area_prob, onset, area_onset

        mrec = ens.member_forcing[1:, :, :P * M].contiguous().cpu().numpy()
        hargs = (c["settings"], c["params"], c["forcing"], c["base"].record_step.astype(np.int32), c["time"],
                 c["local"], mrec, M, c["F"], spec)
        hkw = dict(horizons=c["horizons"], out_stride=120, coupling_window_end=c["wend"],
                   latest_obs_index=np.full(P, c["F"] - 1, dtype=np.int32))
        del ens, mo, sh
        torch.cuda.empty_cache()

        def host(reps=2, **kw):
            lib.run_ensemble_host_soa(*hargs, **hkw, **kw)
            best, st = float("inf"), None
            for _ in range(reps):
                t0 = time.perf_counter()
                res = lib.run_ensemble_host_soa(*hargs, **hkw, **kw)
                t = (time.perf_counter() - t0) * 1e3
                del res
                if t < best:
                    best, st = t, lib.last_batch_stats()
            return best, st
        t_host_on, st_on = host(areas=areas, prob=False, area_prob=False, onset=True)
        t_host_mo, st_mo = host(prob=False, member_out=True)
        del mrec
        lib.release_workspace()
        line = dict(shape=shape, card=name, stations=P, members=M, member_slots=S, n_events=E,
                    conditions_per_event=3, n_areas=A, routes=A - DISTRICTS, districts=DISTRICTS,
                    memberships=memberships, copy_peak_gbs=peak,
                    onset_kernel_ms=t_on, events_kernel_ms=t_events, onset_over_events=t_on / t_events,
                    onset_bytes_bound=on_bytes, onset_gbs=on_bytes / t_on / 1e6,
                    onset_share_of_copy_peak=on_bytes / t_on / 1e6 / peak,
                    area_onset_accumulate_ms=kt["rs_ens_area_onset_accumulate_kernel"],
                    area_onset_finalize_ms=kt["rs_ens_area_onset_finalize_kernel"], area_onset_kernels_ms=t_area_on,
                    area_event_kernels_ms=t_area_ev, area_onset_bytes_bound=area_on_bytes,
                    area_onset_gbs=area_on_bytes / t_area_on / 1e6,
                    onset_fraction_in_0_1=float(((on_dev > 0) & (on_dev < 1)).mean()),
                    identity_last_slot=identity_last_slot,
                    host_onset_only_ms=t_host_on, host_onset_only_d2h_bytes=st_on["d2h_bytes"],
                    host_onset_only_phases=st_on,
                    host_member_out_ms=t_host_mo, host_member_out_d2h_bytes=st_mo["d2h_bytes"],
                    host_member_out_phases=st_mo)
        print(json.dumps(line), flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
