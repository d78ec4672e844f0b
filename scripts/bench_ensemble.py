"""Ensemble runs on one GPU: shared analysis + fork + member forecast + statistics against the same P * M
lanes run as independent points.  Prints one JSON line per shape.

  ex1-ens  401 stations x SimLen 8881 (48 h analysis + 26 h forecast, 30 s steps), coupling + relaxation,
           hourly records, M = 30
  c3-ens   1e5 stations x SimLen 6481 (6 h analysis + 48 h forecast), coupling + relaxation, M = 30

Times are CUDA-event (device-resident runs) or wall-clock around synchronous calls (host entries).  The
card's name and power limit are read in the same process.  Usage:
  python scripts/bench_ensemble.py [--shape ex1-ens|c3-ens|all] [--members 30] [--stations N] [--out FILE]
"""
import argparse
import datetime as dt
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from roadsurf_b200 import lib, synth  # noqa: E402

SHAPES = {"ex1-ens": dict(stations=401, analysis_hours=48, hours=26),
          "c3-ens": dict(stations=100_000, analysis_hours=6, hours=48)}
COPY_PEAK_GBS = 6542.0  # measured device-to-device copy rate of the B200 (README)


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def build(shape, P, M, seed=2024, member_records=True):
    cfg = SHAPES[shape]
    ah, hours = cfg["analysis_hours"], cfg["hours"]
    start = synth.FORECAST_START - dt.timedelta(hours=ah)
    nrec = ah + hours + 2
    base = synth.draw_records(P, nrec, seed, start)
    base.TSurfObs[:, ah + 1:] = -9999.9
    fs = ah * 120
    F = fs + 2
    r_f = lib.fork_record(base.record_step, F)
    mrecs = synth.member_records(base, M, r_f, seed, start) if member_records else None
    sim_len = 1 + (ah + hours) * 120
    settings = synth.abi.default_settings(sim_len, 1, 1)
    params = synth.abi.default_parameters()
    forcing = np.ascontiguousarray(np.stack([getattr(base, v).T for v in synth.RECORD_VARS], axis=1))
    local = np.zeros((lib.L_NLOCAL, P))
    local[lib.L_LAT], local[lib.L_LON], local[lib.L_SKY_VIEW] = base.lat, base.lon, base.sky_view
    wend = lib.read_input_derive_records(forcing, base.record_step.astype(np.int32), settings, fs, local,
                                         np.full(P, fs + 1, dtype=np.int32))
    time_fields = synth.time_axis(start, sim_len, 30.0)
    return dict(base=base, mrecs=mrecs, F=F, r_f=r_f, settings=settings, params=params, forcing=forcing,
                local=local, wend=wend, time=time_fields, horizons=np.ascontiguousarray(base.horizons.T),
                sim_len=sim_len)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shape", default="all")
    ap.add_argument("--members", type=int, default=30)
    ap.add_argument("--stations", type=int, default=0, help="override the station count")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    if lib.load().roadsurf_device_count() < 1:
        raise SystemExit("no CUDA device visible")
    shapes = list(SHAPES) if args.shape == "all" else [args.shape]
    name = card()
    lines = []
    for shape in shapes:
        P, M = args.stations or SHAPES[shape]["stations"], args.members
        c = build(shape, P, M)
        spec = lib.stats_spec((0.1, 0.5, 0.9), ((0, "<", 0.0), (3, ">", 0.0)))
        lib.set_model(c["settings"], c["params"])
        sh = lib.DeviceBatch(P, c["sim_len"], n_records=c["base"].nrec, coarse=True, horizons=True, coupling=True,
                             state=True, out_stride=120)
        sh.load_records(c["base"])
        sh.time_fields.copy_(torch.from_numpy(c["time"]))
        sh.local[:, :P] = torch.from_numpy(c["local"])
        sh.horizons[:, :P] = torch.from_numpy(c["horizons"])
        sh.coupling_window_end = c["wend"]
        ens = lib.EnsembleBatch(sh, M, c["F"], spec)
        ens.load_member_records(c["mrecs"])
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]

        def timed(fn, reps=3):
            fn()
            torch.cuda.synchronize()
            ts = []
            for _ in range(reps):
                ev[0].record()
                fn()
                ev[1].record()
                torch.cuda.synchronize()
                ts.append(ev[0].elapsed_time(ev[1]))
            return min(ts)

        # device-resident: the whole ensemble, and the prefix alone (a plain launch of the stations [1, F - 1])
        t_total = timed(lambda: ens.run())
        t_prefix = timed(lambda: sh.run(step_begin=1, step_end=c["F"] - 1))
        t_nostats = timed(lambda: ens.run(stats=False))
        mo = ens.member_out
        t_stats = timed(lambda: lib.ensemble_stats(mo, P, M, spec))
        # member-major thread order: thread m * P + p runs lane p * M + m
        t_idx = torch.arange(P * M, device="cuda", dtype=torch.int64)
        order = torch.arange(ens.ld_members, device="cuda", dtype=torch.int32)
        order[:P * M] = ((t_idx % P) * M + t_idx // P).to(torch.int32)
        out_sm = ens.member_out.clone()
        ens.member_order = order
        t_member_major = timed(lambda: ens.run(stats=False))
        same_order = bool(torch.equal(out_sm, ens.member_out))
        ens.member_order = None
        ldm = ens.ld_members
        fork_bytes = 8 * (ldm * (lib.state_nplanes(15) * 2 + lib.scratch_nplanes(15) * 2 + 360 * 2 + lib.L_NLOCAL * 2
                                 + 11 * 2) + 4 * ldm * 2)
        stats_bytes = 8 * (mo.numel() + ens.stats_t.numel() + ens.prob_t.numel())
        # host entries: ensemble, and the same lanes as independent points
        mrec = synth.member_record_tensor(c["mrecs"], c["r_f"])
        t0 = time.perf_counter()
        res = lib.run_ensemble_host_soa(c["settings"], c["params"], c["forcing"], c["base"].record_step.astype(np.int32),
                                        c["time"], c["local"], mrec, M, c["F"], spec, horizons=c["horizons"],
                                        out_stride=120, coupling_window_end=c["wend"], member_out=True,
                                        member_status=True, latest_obs_index=np.full(P, c["F"] - 1, dtype=np.int32))
        t_host_ens = (time.perf_counter() - t0) * 1e3
        ens_host_stats = lib.last_batch_stats()
        lanes = synth.lane_records(c["mrecs"])
        lforcing = np.ascontiguousarray(np.stack([getattr(lanes, v).T for v in synth.RECORD_VARS], axis=1))
        llocal = np.repeat(c["local"], M, axis=1)
        llocal[:3] = -9999.9
        # member relaxation targets as the ensemble derives them: read_input's rule on the lane records
        lib.read_input_derive_records(lforcing, c["base"].record_step.astype(np.int32), c["settings"],
                                      c["F"] - 2, llocal, np.full(P * M, c["F"] - 1, dtype=np.int32))
        llocal[lib.L_ACTIVE] = np.repeat(c["local"][lib.L_ACTIVE], M)
        n_out = (c["sim_len"] + 119) // 120
        out = np.zeros((lib.O_NVAR, n_out, P * M))
        status = np.zeros(P * M, dtype=np.int32)
        t0 = time.perf_counter()
        lib.run_host_soa(c["settings"], c["params"], lforcing, c["time"], llocal, out,
                         record_step=c["base"].record_step.astype(np.int32),
                         horizons=np.repeat(c["horizons"], M, axis=1), status=status, out_stride=120, ngpus=1,
                         coupling_window_end=c["wend"])
        t_host_ind = (time.perf_counter() - t0) * 1e3
        s0 = ens.slot0
        identical = bool(np.array_equal(out[:, s0:], res["member_out"], equal_nan=True)
                         and np.array_equal(status, res["member_status"]))
        line = dict(shape=shape, card=name, stations=P, members=M, sim_len=c["sim_len"], fork_step=c["F"],
                    device_total_ms=t_total, prefix_ms=t_prefix, stats_ms=t_stats,
                    fork_plus_members_ms=t_nostats - t_prefix, member_major_fork_plus_members_ms=t_member_major - t_prefix,
                    member_major_identical=same_order,
                    stats_gbs=stats_bytes / t_stats / 1e6, stats_share_of_copy_peak=stats_bytes / t_stats / 1e6 / COPY_PEAK_GBS,
                    fork_bytes=fork_bytes, host_ensemble_ms=t_host_ens, host_ensemble_phases=ens_host_stats,
                    host_independent_ms=t_host_ind, independent_bit_identical=identical,
                    member_tensor_gb=8 * (ens.member_forcing.numel() + ens.member_out.numel() + ens.member_state.numel()
                                          + ens.member_horizons.numel() + ens.member_local.numel()
                                          + ens.member_scratch.numel()) / 1e9)
        print(json.dumps(line), flush=True)
        lines.append(line)
        del ens, sh
        torch.cuda.empty_cache()
        lib.release_workspace()
    if args.out:
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
