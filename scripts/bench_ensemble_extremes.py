"""Ensemble window extremes (roadsurf_ensemble_extremes) on one GPU: the extremes kernels against the statistics kernel
on the same member tensor, and the host entry with extremes alone against member_out.  Prints one JSON line per shape.

  ex1-ens, c3-ens: the shapes, member tensor and areas of scripts/bench_ensemble_onset.py; four extremes (Tsurf minimum
  over 6 and over 12 slots, Ice and Snow maximum over 6 slots) with the quantiles 0, 0.1, 0.5, 0.9 and 1.

  - kernel times: torch.profiler (CUDA activities) over --reps calls after a warm-up, mean per launch of
    rs_ens_window_extremes_kernel, of the statistics kernel on its output and of the two area kernels and the
    statistics launch on the area accumulators (the three statistics launches of a rep are told apart by their order);
    in the same window the statistics kernel on the six planes of member_out (roadsurf_ensemble_stats, prob NULL);
  - byte bound of the window kernel (window_bytes_bound, window_gbs): the least any kernel must move, each extreme's
    plane read once over all S slots and its work space written once, 2 x S x P x M x 8 bytes per extreme.  The
    van Herk / Gil-Werman passes move 5 x 8 bytes per value and extreme (two reads of the value, two writes and one read
    of the work space), so the rate against this bound understates the bandwidth the kernel draws by 2.5 times.  Of the
    area accumulate kernel: the work space once per (extreme, area membership), S x M x 8 bytes.  Rates are against a
    device-to-device copy measured in the same process;
  - host entry: wall clock around roadsurf_run_ensemble_host_soa_extremes with extremes alone (stats, prob and the
    area event outputs NULL, no member_out) and with member_out alone (stats NULL), best of 2 after a warm-up call, and
    d2h_bytes of each.
The card's name and power limit are read in the same process.  Usage:
  python scripts/bench_ensemble_extremes.py [--shape ex1-ens|c3-ens|all] [--members 30] [--stations N] [--out FILE]
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
from bench_ensemble_events import EVENTS, ICE, SNOW, TS, copy_peak_gbs, member_forcing_on_device  # noqa: E402
from roadsurf_b200 import lib  # noqa: E402

QUANTILES = (0.0, 0.1, 0.5, 0.9, 1.0)
EXTREMES = [(TS, "min", 6), (TS, "min", 12), (ICE, "max", 6), (SNOW, "max", 6)]
KERNELS = ("rs_ens_window_extremes_kernel", "rs_ens_area_extremes_accumulate_kernel",
           "rs_ens_area_extremes_finalize_kernel", "rs_ens_stats_kernel")


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
        spec = lib.stats_spec(QUANTILES)
        ext = lib.ensemble_extremes(EXTREMES)
        area_lists = make_areas(P, seed=11)
        areas = lib.ensemble_areas(area_lists)
        A, X, rows = len(area_lists), len(EXTREMES), lib.ENS_NFIXED + len(QUANTILES)
        memberships = int(sum(len(a) for a in area_lists))
        lib.set_model(c["settings"], c["params"])
        sh = lib.DeviceBatch(P, c["sim_len"], n_records=c["base"].nrec, coarse=True, horizons=True, coupling=True,
                             state=True, out_stride=120)
        sh.load_records(c["base"])
        sh.time_fields.copy_(torch.from_numpy(c["time"]))
        sh.local[:, :P] = torch.from_numpy(c["local"])
        sh.horizons[:, :P] = torch.from_numpy(c["horizons"])
        sh.coupling_window_end = c["wend"]
        ens = lib.EnsembleBatch(sh, M, c["F"], lib.stats_spec(events=EVENTS))
        member_forcing_on_device(torch, ens, sh, c["r_f"], P, M, seed=7)
        ens.run()
        torch.cuda.synchronize()
        S, ldm, ld = ens.n_slots, ens.ld_members, sh.ld
        mo = ens.member_out
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        f64 = dict(dtype=torch.float64, device="cuda")
        ext_stats = torch.empty((rows, X, S, ld), **f64)
        area_ext_stats = torch.empty((rows, X, S, A), **f64)
        stats = torch.empty((rows, lib.O_NVAR, S, ld), **f64)

        def run_extremes():
            lib._check(handle.roadsurf_ensemble_extremes(mo.data_ptr(), lib.O_NVAR, S, ldm, P, M, C.byref(spec),
                                                         C.byref(ext), ext_stats.data_ptr(), ld, C.byref(areas),
                                                         area_ext_stats.data_ptr(), stream))

        def run_stats():
            lib._check(handle.roadsurf_ensemble_stats(mo.data_ptr(), lib.O_NVAR, S, ldm, P, M, C.byref(spec),
                                                      stats.data_ptr(), None, ld, stream))
        run_extremes()
        run_stats()
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(args.reps):
                run_extremes()
                run_stats()
            torch.cuda.synchronize()
        # per launch; the statistics kernel runs three times per rep, in this order: on the station extremes, on the
        # area extremes, on member_out
        kt, stats_launches = {}, []
        for evt in sorted(prof.events(), key=lambda e: e.time_range.start):
            if evt.device_type != torch.autograd.DeviceType.CUDA:
                continue
            for tag in KERNELS:
                if tag in evt.name:
                    t = evt.time_range.elapsed_us() / 1e3
                    if tag == "rs_ens_stats_kernel":
                        stats_launches.append(t)
                    else:
                        kt.setdefault(tag, []).append(t)
        kt = {k: float(np.mean(v)) for k, v in kt.items()}
        # launch order per rep: station extremes stats, area extremes stats, member_out stats
        sl = np.asarray(stats_launches).reshape(args.reps, 3)
        t_ext_stats, t_area_stats, t_mo_stats = (float(v) for v in sl.mean(axis=0))
        t_win = kt["rs_ens_window_extremes_kernel"]
        t_area = kt["rs_ens_area_extremes_accumulate_kernel"] + kt["rs_ens_area_extremes_finalize_kernel"] + t_area_stats
        win_bytes = 8 * X * S * P * M * 2
        area_bytes = 8 * X * S * M * memberships
        xs = ext_stats[..., :P].cpu().numpy()
        del ext_stats, area_ext_stats, stats

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
        t_host_x, st_x = host(areas=areas, stats=False, prob=False, area_prob=False, extremes=ext)
        t_host_mo, st_mo = host(stats=False, prob=False, member_out=True)
        del mrec
        lib.release_workspace()
        line = dict(shape=shape, card=name, stations=P, members=M, member_slots=S, n_extremes=X,
                    extremes=EXTREMES, quantiles=QUANTILES, n_areas=A, routes=A - DISTRICTS, districts=DISTRICTS,
                    memberships=memberships, copy_peak_gbs=peak,
                    window_kernel_ms=t_win, window_bytes_bound=win_bytes, window_gbs=win_bytes / t_win / 1e6,
                    window_share_of_copy_peak=win_bytes / t_win / 1e6 / peak,
                    ext_stats_kernel_ms=t_ext_stats, member_out_stats_kernel_ms=t_mo_stats,
                    area_accumulate_ms=kt["rs_ens_area_extremes_accumulate_kernel"],
                    area_finalize_ms=kt["rs_ens_area_extremes_finalize_kernel"], area_stats_kernel_ms=t_area_stats,
                    area_kernels_ms=t_area, area_bytes_bound=area_bytes,
                    area_accumulate_gbs=area_bytes / kt["rs_ens_area_extremes_accumulate_kernel"] / 1e6,
                    tsurf_min12_median_mean=float(np.mean(xs[lib.ENS_NFIXED + 2, 1][xs[0, 1] > 0])),
                    host_extremes_only_ms=t_host_x, host_extremes_only_d2h_bytes=st_x["d2h_bytes"],
                    host_extremes_only_phases=st_x,
                    host_member_out_ms=t_host_mo, host_member_out_d2h_bytes=st_mo["d2h_bytes"],
                    host_member_out_phases=st_mo)
        print(json.dumps(line), flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
