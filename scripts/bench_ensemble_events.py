"""Ensemble event probabilities (RsEnsembleEvent) on one GPU: the events kernel against the statistics kernel on the
same member tensor, and the host entry's transfer with event probabilities only against member_out.  Prints one
JSON line per shape.

  ex1-ens, c3-ens: the shapes of scripts/bench_ensemble.py (M = 30, an output slot every 120 steps = 1 h).

The member tensor is the output of one device-resident ensemble run.  The members' forcing is made on the device: the
stations' records after the fork record with a per-member offset of air and dew-point temperature (N(0, 1.5) K) and a
per-member, per-record factor on precipitation (lognormal, sigma 0.3).  The events: 4 events x 3 conditions x
window 6 (6 h) over the six model output planes.

  - kernel times: CUDA events around one launch, best of --reps after one warm-up launch; the statistics kernel with
    bench_ensemble.py's spec (3 quantiles, 2 thresholds), the events kernel alone (stats NULL);
  - bytes bound of the events kernel: the referenced planes read once (planes x S x P*M x 8) plus the probabilities
    written (n_events x S x P x 8), over kernel time, against a device-to-device copy measured in the same process;
    ex1-ens's member tensor (8 MB) fits in L2, c3-ens's (7 GB) does not;
  - host entry: wall clock around roadsurf_run_ensemble_host_soa with the event spec, without and with member_out,
    best of 2 after a warm-up call, and roadsurf_last_batch_stats().d2h_bytes.
The card's name and power limit are read in the same process.  Usage:
  python scripts/bench_ensemble_events.py [--shape ex1-ens|c3-ens|all] [--members 30] [--stations N] [--out FILE]
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
from roadsurf_b200 import lib  # noqa: E402

TS, SNOW, WATER, ICE, DEPOSIT, ICE2 = range(6)
EVENTS = [([(TS, "<", 0.0), (WATER, ">", 0.05), (ICE, "<", 0.05)], 6),       # wet road freezing
          ([(TS, "<", 0.0), (SNOW, ">", 0.1), (WATER, "<=", 0.05)], 6),      # snow on a frozen road
          ([(TS, "<", -1.0), (ICE, ">", 0.0), (ICE2, ">=", 0.0)], 6),
          ([(TS, "<", 0.0), (DEPOSIT, ">", 0.0), (ICE, "<=", 0.05)], 6)]
STATS_SPEC = dict(quantiles=(0.1, 0.5, 0.9), thresholds=((TS, "<", 0.0), (ICE, ">", 0.0)))


def copy_peak_gbs(torch, nbytes=4 << 30, reps=5):
    """Device-to-device copy rate, bytes read + written per second (GB/s), best of `reps`."""
    a = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda")
    b = torch.empty_like(a)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    b.copy_(a)
    best = float("inf")
    for _ in range(reps):
        ev[0].record()
        b.copy_(a)
        ev[1].record()
        torch.cuda.synchronize()
        best = min(best, ev[0].elapsed_time(ev[1]))
    del a, b
    return 2 * nbytes / best / 1e6


def member_forcing_on_device(torch, ens, sh, r_f, P, M, seed):
    """Records r_f + 1 ... of the stations into every member lane, perturbed per member (slot 0 is the library's)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    rec = sh.forcing[r_f + 1:, :, :P].repeat_interleave(M, dim=2)
    dt = torch.randn(P * M, generator=g, device="cuda", dtype=torch.float64) * 1.5
    rec[:, 0] += dt                                     # tair
    rec[:, 1] += dt                                     # tdew
    f = torch.exp(torch.randn(rec[:, 4].shape, generator=g, device="cuda", dtype=torch.float64) * 0.3)
    rec[:, 4] = torch.where(rec[:, 4] > 0, rec[:, 4] * f, rec[:, 4])   # precipitation
    ens.member_forcing[1:, :, :P * M] = rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shape", default="all")
    ap.add_argument("--members", type=int, default=30)
    ap.add_argument("--stations", type=int, default=0, help="override the station count")
    ap.add_argument("--reps", type=int, default=5)
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
        events_spec = lib.stats_spec(events=EVENTS)
        stats_spec = lib.stats_spec(**STATS_SPEC)
        lib.set_model(c["settings"], c["params"])
        sh = lib.DeviceBatch(P, c["sim_len"], n_records=c["base"].nrec, coarse=True, horizons=True, coupling=True,
                             state=True, out_stride=120)
        sh.load_records(c["base"])
        sh.time_fields.copy_(torch.from_numpy(c["time"]))
        sh.local[:, :P] = torch.from_numpy(c["local"])
        sh.horizons[:, :P] = torch.from_numpy(c["horizons"])
        sh.coupling_window_end = c["wend"]
        ens = lib.EnsembleBatch(sh, M, c["F"], events_spec)
        member_forcing_on_device(torch, ens, sh, c["r_f"], P, M, seed=7)
        ens.run()
        torch.cuda.synchronize()
        S, ldm, ld = ens.n_slots, ens.ld_members, sh.ld
        mo = ens.member_out
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        f64 = dict(dtype=torch.float64, device="cuda")
        stats = torch.empty((lib.ENS_NFIXED + 3, lib.O_NVAR, S, ld), **f64)
        prob_t = torch.empty((2, S, ld), **f64)
        prob_e = torch.empty((len(EVENTS), S, ld), **f64)

        def run_stats():
            lib._check(handle.roadsurf_ensemble_stats(mo.data_ptr(), lib.O_NVAR, S, ldm, P, M, C.byref(stats_spec),
                                                      stats.data_ptr(), prob_t.data_ptr(), ld, stream))

        def run_events():
            lib._check(handle.roadsurf_ensemble_stats(mo.data_ptr(), lib.O_NVAR, S, ldm, P, M, C.byref(events_spec),
                                                      None, prob_e.data_ptr(), ld, stream))
        t_stats = timed(run_stats, args.reps)
        t_events = timed(run_events, args.reps)
        same_as_run = bool(torch.equal(prob_e[:, :, :P], ens.prob_t[:, :S, :P]))
        planes = len({cd[0] for conds, _ in EVENTS for cd in conds})
        ev_bytes = 8 * (planes * S * P * M + len(EVENTS) * S * P)
        st_bytes = 8 * (lib.O_NVAR * S * P * M + stats[..., :P].numel() + prob_t[..., :P].numel())
        probs = prob_e[:, :, :P].cpu().numpy()
        del stats, prob_t, prob_e

        # host entry: event probabilities only, against member_out as well
        mrec = ens.member_forcing[1:, :, :P * M].contiguous().cpu().numpy()
        hargs = (c["settings"], c["params"], c["forcing"], c["base"].record_step.astype(np.int32), c["time"],
                 c["local"], mrec, M, c["F"], events_spec)
        hkw = dict(horizons=c["horizons"], out_stride=120, coupling_window_end=c["wend"],
                   latest_obs_index=np.full(P, c["F"] - 1, dtype=np.int32))
        del ens, mo, sh
        torch.cuda.empty_cache()

        def host(member_out, reps=2):
            lib.run_ensemble_host_soa(*hargs, member_out=member_out, **hkw)
            best, res, st = float("inf"), None, None
            for _ in range(reps):
                res = None
                t0 = time.perf_counter()
                res = lib.run_ensemble_host_soa(*hargs, member_out=member_out, **hkw)
                t = (time.perf_counter() - t0) * 1e3
                if t < best:
                    best, st = t, lib.last_batch_stats()
            return best, st, res["prob"]
        t_host_ev, st_ev, prob_ev = host(False)
        t_host_mo, st_mo, prob_mo = host(True)
        del mrec
        lib.release_workspace()
        line = dict(shape=shape, card=name, stations=P, members=M, member_slots=S, n_events=len(EVENTS),
                    conditions_per_event=3, window=6, referenced_planes=planes,
                    member_out_gb=8 * lib.O_NVAR * S * P * M / 1e9, copy_peak_gbs=peak,
                    stats_kernel_ms=t_stats, events_kernel_ms=t_events, events_over_stats=t_events / t_stats,
                    stats_gbs=st_bytes / t_stats / 1e6,
                    events_bytes_bound=ev_bytes, events_gbs=ev_bytes / t_events / 1e6,
                    events_share_of_copy_peak=ev_bytes / t_events / 1e6 / peak,
                    events_equal_device_entry=same_as_run,
                    event_prob_fraction_in_0_1=float(((probs > 0) & (probs < 1)).mean()),
                    host_events_only_ms=t_host_ev, host_events_only_d2h_bytes=st_ev["d2h_bytes"],
                    host_events_only_phases=st_ev,
                    host_member_out_ms=t_host_mo, host_member_out_d2h_bytes=st_mo["d2h_bytes"],
                    host_member_out_phases=st_mo,
                    host_event_planes_identical=bool(np.array_equal(prob_ev, prob_mo)))
        print(json.dumps(line), flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
