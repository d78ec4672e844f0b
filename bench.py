#!/usr/bin/env python
"""Benchmark of the RoadSurf per-point simulation loop on B200.

    python bench.py --gpus N --steps K --warmup W [--impl reference]
                    [--workload c4|c3|c5] [--scaling weak|strong] [--inproc] [--dump-outputs DIR]

Workloads (BASELINE.json configs; `config.workload` in the output names the one that ran):
  c4 (default)  "synthetic 10^7-point km-scale road grid, 24 h forecast, sharded across 1/2/4/8 B200":
                SimLen 2881 steps of 30 s, 15 ground layers, hourly forcing records interpolated on the
                device, hourly outputs, 30 % of the points with sky-view / shadow radiation.
                weak (default): every GPU runs one 1.25e6-point shard (10^7 / 8), so at N = 8 the job is
                exactly the named configuration; at N = 1 the FULL 10^7-point configuration (it fits one
                B200: ~65 GB) is also run once and reported as `full_config`.
                strong: the 10^7 points are split over the N GPUs.
  c3            "synthetic 10^5-point national road network, 48 h forecast ... with Coupling/Relaxation":
                6 h analysis + 48 h forecast (SimLen 6481), coupling window 180 min, from hourly records;
                weak = one 10^5-point replica per GPU, strong = 10^5 points split over the GPUs.
  c5            "51-member ensemble x 10^6 points (5.1e7 point-runs), 48 h, full 8xB200 box": SimLen 5761;
                weak = 5.1e7 / 8 = 6.375e6 point-runs per GPU.
One bench "step" = one full pass over the rank's points (one launch of the step kernel, several for c3).

metric  road-point-timesteps/s = points * SimLen / seconds (nominal model steps).
value   kernel-resident throughput: inputs already in HBM when the timed region starts.
e2e     same metric through the C ABI with HOST buffers (roadsurf_run_host_soa): pinned host
        records -> H2D -> kernel -> D2H of the hourly outputs, all inside the timed region; the grid's
        horizon table is resident on the device (roadsurf_prepare_statics), as for repeated forecasts.
--impl reference  the reference's CPU path: the C++ restatement of the Fortran loop (oracle/, compiled with
        the reference's own -Ofast flag set; oracle/_ref -- the gfortran build -- is used instead when
        it exists) on all host cores, on the first 10240 points of the very workload the GPU arm runs.
--inproc  one process drives all N GPUs through the library's own `ngpus` argument
        (roadsurf_run_host_soa(..., ngpus=N)) and compares the result with the one-GPU run.
--dump-outputs DIR  after the timed steps, write what the last one computed as DIR/<name>.npy (float64):
        every output variable [points, hourly slots], the status words [points], for the coupled workloads
        (c3, c2) the end-of-run state planes [points, planes] (ground-layer temperatures first), and the
        indices of the points written [points].  Points are a fixed, seeded sample of rank 0's points (with
        --inproc: of all points), all of them when they fit 64 MB.  The inputs depend on the arguments alone,
        so two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "road_point_timesteps_per_sec"
UNIT = "point-steps/s"
CPU_SAMPLE = 10240

WORKLOADS = {
    "c4": dict(total=10_000_000, per_gpu=1_250_000, hours=24, analysis=0, coupling=False,
               name="c4: synthetic km-scale road grid, 24 h forecast, 10^7 points over 8 GPUs"),
    "c3": dict(total=100_000, per_gpu=100_000, hours=48, analysis=6, coupling=True,
               name="c3: synthetic national road network, 10^5 points, 6 h analysis + 48 h forecast, coupling + relaxation"),
    "c2": dict(total=401, per_gpu=401, hours=26, analysis=48, coupling=True,
               name="c2: example1's shape, 401 stations, 48 h analysis + 26 h forecast, coupling + relaxation "
                    "(latency-bound: a warp per point)"),
    "c5": dict(total=51_000_000, per_gpu=6_375_000, hours=48, analysis=0, coupling=False,
               name="c5: 51-member ensemble x 10^6 points (flattened member x point), 48 h forecast"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=("ours", "reference"))
    ap.add_argument("--workload", default="c4", choices=tuple(WORKLOADS))
    ap.add_argument("--scaling", default="weak", choices=("weak", "strong"))
    ap.add_argument("--inproc", action="store_true")
    ap.add_argument("--points-per-gpu", type=int, default=0, help="override the per-GPU point count")
    ap.add_argument("--hours", type=int, default=0, help="override the forecast length")
    ap.add_argument("--cpu-sample-points", type=int, default=CPU_SAMPLE)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-full-config", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU paths only")
    return args


def rank_points(args, world):
    w = WORKLOADS[args.workload]
    if args.points_per_gpu:
        return args.points_per_gpu
    if args.scaling == "strong":
        return (w["total"] + world - 1) // world
    return w["per_gpu"]


def workload_config(args, world, extra=None):
    w = WORKLOADS[args.workload]
    hours = args.hours or w["hours"]
    cfg = {"workload": w["name"], "scaling_mode": args.scaling, "points_per_gpu": rank_points(args, world),
           "sim_len": 1 + (w["analysis"] + hours) * 120, "dt_s": 30.0, "nlayers": 15,
           "forcing": "hourly records, device-side linear interpolation", "output": "every 120th step (hourly)",
           "sky_view_fraction": 0.3, "coupling": w["coupling"], "relaxation": w["coupling"],
           "point_order": "sky-view points scattered at random in the input; gathered per launch by "
                          "roadsurf_order_points (inside the timed step)",
           "l2": "inputs + outputs of a step (GBs) exceed the 126 MB L2; no flush needed"}
    if extra:
        cfg.update(extra)
    return cfg


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.proc = index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.samples.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=2)
        sm = sorted(int(s[0]) for s in self.samples if s and s[0].isdigit())
        mx = [int(s[1]) for s in self.samples if len(s) > 1 and s[1].isdigit()]
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        reasons = [n for k, n in enumerate(names) if any(len(s) > 3 + k and s[3 + k] == "Active" for s in self.samples)]
        power = [float(s[2]) for s in self.samples if len(s) > 2 and s[2].replace(".", "", 1).isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "power_w_max": max(power) if power else None}


# ----------------------------------------------------------------------------------------------------
# workloads
# ----------------------------------------------------------------------------------------------------
class Workload:
    """One rank's share of a named configuration: a coarse-record device batch + how to step it."""

    def __init__(self, args, rank, world, device, data_only=False):
        """data_only: generate the workload's data and nothing else (the reference arm: libroadsurf_b200.so is
        never loaded there, torch is used for the random numbers only)."""
        import torch
        from roadsurf_b200 import abi, lib, synth, synth_torch
        self.torch, self.lib, self.data_only = torch, lib, data_only
        w = WORKLOADS[args.workload]
        self.name, self.args = args.workload, args
        self.P = rank_points(args, world)
        self.hours = args.hours or w["hours"]
        self.analysis = w["analysis"]
        self.sim_len = 1 + (self.analysis + self.hours) * 120
        self.coupled = w["coupling"]
        self.seed = 20191206 + rank
        nrec = self.analysis + self.hours + 2
        if self.coupled:
            self.settings = abi.default_settings(self.sim_len)
            self.settings.use_coupling = self.settings.use_relaxation = 1
        else:
            self.settings = abi.default_settings(self.sim_len)
        self.params = abi.default_parameters(30.0)
        if not data_only:
            lib.set_model(self.settings, self.params)
        self.db = lib.DeviceBatch(self.P, self.sim_len, n_records=nrec, coarse=True, horizons=True, out_stride=120,
                                  coupling=self.coupled, state=self.coupled)
        start = synth.FORECAST_START - __import__("datetime").timedelta(hours=self.analysis)
        synth_torch.fill_device_batch_chunked(self.db, seed=self.seed, start=start)
        self.window_end = 0
        if self.coupled:
            self._derive_coupled()

    def _derive_coupled(self):
        """What read_input derives per point (relaxation targets, coupling index / observation), computed by
        the library from the hourly records; observations = air temperature - 1 + noise during the analysis."""
        torch, lib, db = self.torch, self.lib, self.db
        g = torch.Generator(device=db.forcing.device)
        g.manual_seed(self.seed + 77)
        obs = db.forcing[:, lib.F_NAMES.index("tair")] - 1.0 + 0.5 * torch.randn(db.forcing.shape[0], db.ld, generator=g,
                                                                               dtype=torch.float64, device=db.forcing.device)
        obs[self.analysis + 1:] = -9999.9
        db.forcing[:, lib.F_NAMES.index("TSurfObs")] = obs
        if self.data_only:
            return                      # (cpu_case re-derives the per-point parameters on the host, in Python)
        forcing = db.forcing[:, :, :self.P].cpu().contiguous()
        local = db.local[:, :self.P].cpu().contiguous()
        forecast_step = self.analysis * 120
        latest = __import__("numpy").full(self.P, forecast_step + 1, dtype="int32")
        self.window_end = lib.read_input_derive_records(forcing, db.record_step.cpu(), self.settings, forecast_step, local,
                                                        latest_obs_index=latest)
        db.local[:, :self.P] = local.to(db.local.device)
        db.coupling_window_end = self.window_end

    def step(self, stream):
        # one pass: the library gathers the sky-view points at one end of the launch (the permutation is
        # rebuilt every step here, as a caller with changing statics would; it is static per grid)
        self.db.build_order(stream)
        self.db.run(stream)

    def host_buffers(self):
        torch, lib, db, P = self.torch, self.lib, self.db, self.P
        pin = dict(pin_memory=True)
        h = {"forcing": torch.empty((db.n_records, db.nvar, P), dtype=torch.float64, **pin),
             "local": torch.empty((lib.L_NLOCAL, P), dtype=torch.float64, **pin),
             "horizons": torch.empty((360, P), dtype=torch.float64, **pin),
             "out": torch.empty((lib.O_NVAR, db.n_out, P), dtype=torch.float64, **pin),
             "status": torch.empty(P, dtype=torch.int32, **pin)}
        h["forcing"].copy_(db.forcing[:, :, :P])
        h["local"].copy_(db.local[:, :P])
        h["horizons"].copy_(db.horizons[:, :P])
        h["tf"], h["rs"] = db.time_fields.cpu(), db.record_step.cpu()
        return h

    def cpu_case(self, npts):
        """The first `npts` points of this rank's workload in the reference's host layout."""
        from roadsurf_b200 import synth, synth_torch
        rec = synth_torch.records_sample(self.db, npts)
        arrays, settings, params = synth.case_from_records(rec, self.hours, self.analysis, int(self.coupled),
                                                           int(self.coupled))
        return arrays, settings, params


def cpu_arm(arrays, settings, params, steps, warmup, threads, fast=True, backend="port"):
    """Times the CPU implementation on `threads` host threads over the sample; returns rate + last outputs."""
    from oracle import pyoracle
    n = arrays.npoints * arrays.sim_len
    times, work, status = [], None, None
    for it in range(warmup + steps):
        work = arrays.copy()          # the reference mutates its inputs in place
        t0 = time.perf_counter()
        status, _ = pyoracle.run_batch(work, settings, params, nthreads=threads, fast=fast, backend=backend)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    total = sum(times)
    return {"value": n * len(times) / total, "seconds": total, "points": arrays.npoints, "sim_len": arrays.sim_len,
            "ms_per_step": 1e3 * total / len(times)}, work, status


def reference_backend():
    """("ref", "reference") when oracle/_ref (the gfortran build of the unmodified reference) exists, else
    ("port", "port") with the reason."""
    from oracle import pyoracle
    try:
        pyoracle.load_ref()
        return "ref", "reference", "oracle/_ref/libroadsurf_ref.so (gfortran build of the unmodified reference)"
    except pyoracle.ReferenceUnavailable as e:
        return "port", "port", ("C++ restatement of the Fortran path built with the reference's -Ofast flag set; "
                                f"the gfortran binary cannot be built here ({e})")


def flops_per_point_step(arrays, settings, params, npts=8):
    """Exact arithmetic-operation count of the reference algorithm on this workload (counting
    scalar in the oracle): each add/mul/div/sqrt/exp/log/trig/pow = 1 flop."""
    from oracle import pyoracle
    tot, steps = {}, 0
    for p in range(min(npts, arrays.npoints)):
        c, s = pyoracle.count_ops(arrays.copy(), settings, params, p)
        steps += s
        for k, v in c.items():
            tot[k] = tot.get(k, 0) + v
    per = {k: v / steps for k, v in tot.items()}
    flops = sum(per[k] for k in ("add", "mul", "div", "sqrt", "exp", "log", "trig", "pow"))
    return flops, {k: round(v, 2) for k, v in per.items()}


def run_reference(args):
    """The reference's CPU implementation of the path on the box's host cores (rank 0 only), on the first
    10240 points of the workload the GPU arm runs (drawn by the same generator call; the GPU, when there
    is one, is used for the data generation only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    cores = os.cpu_count() or 1
    npts = args.cpu_sample_points
    world = max(1, args.gpus)
    if torch.cuda.is_available():
        torch.cuda.set_device(0)
        wl = Workload(args, 0, world, torch.device("cuda", 0), data_only=True)
        arrays, settings, params = wl.cpu_case(npts)
        source = "the first %d points of the GPU arm's rank-0 workload (same generator call, same seed)" % arrays.npoints
        del wl
        torch.cuda.empty_cache()
    else:
        from roadsurf_b200 import synth
        w = WORKLOADS[args.workload]
        hours = args.hours or w["hours"]
        arrays, settings, params, _ = synth.make_case(npts, hours, 20191206, analysis_hours=w["analysis"],
                                                      use_coupling=int(w["coupling"]), use_relaxation=int(w["coupling"]),
                                                      obs_bias=False)
        source = "%d points of the same shape from the numpy generator (no GPU in this process)" % npts
    backend, kind, note = reference_backend()
    r, _, _ = cpu_arm(arrays, settings, params, args.steps, args.warmup, cores, fast=True, backend=backend)
    sample = f"{r['points']} points x {r['sim_len']} steps per step: {source}"
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": workload_config(args, world),
            "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": cores, "kind": kind, "sample": sample, "note": note},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def kernel_traffic_per_point_step():
    """DRAM traffic of the step kernel per point-step from the committed ncu capture (profiles/*.json)."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r02_kernel_traffic.json")))
        return float(d["dram_bytes_per_point_step"]), d.get("source", "profiles/r02_kernel_traffic.json")
    except Exception:
        return None, None


DUMP_LIMIT_BYTES = 64_000_000
DUMP_SEED = 20191206


def dump_outputs(directory, out, status, npoints, state=None, limit=DUMP_LIMIT_BYTES):
    """Writes out [O_NVAR, n_out, >= npoints], status [>= npoints] and, when given, the end-of-run state
    [planes, >= npoints] of a fixed, seeded sample of the points (all of them when they fit `limit` bytes) as
    directory/<output name>.npy [points, n_out], status.npy, state.npy [points, planes] and point_index.npy
    [points], all float64 (status words and indices are exact there)."""
    import numpy as np
    import torch
    from roadsurf_b200 import lib
    n_out = out.shape[1]
    planes = 0 if state is None else state.shape[0]
    headers = 128 * (len(lib.O_NAMES) + 3)
    n = min(npoints, (limit - headers) // ((len(lib.O_NAMES) * n_out + planes + 2) * 8))
    if n < npoints:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(npoints, n, replace=False))
    else:
        idx = np.arange(npoints)
    sel = torch.from_numpy(idx).to(out.device)
    o = out[:len(lib.O_NAMES)].index_select(2, sel).cpu().numpy()
    arrays = {name: np.ascontiguousarray(o[v].T) for v, name in enumerate(lib.O_NAMES)}
    arrays["status"] = status.index_select(0, sel.to(status.device)).cpu().numpy().astype(np.float64)
    if state is not None:
        arrays["state"] = np.ascontiguousarray(state.index_select(1, sel.to(state.device)).cpu().numpy().T)
    arrays["point_index"] = idx.astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def run_inproc(args):
    """One process, N GPUs through the product's own `ngpus` argument; compared with the 1-GPU result."""
    import torch
    from roadsurf_b200 import build as rs_build, lib
    rs_build.build_library()
    lib.load()
    n = max(1, args.gpus)
    torch.cuda.set_device(0)
    one = Workload(args, 0, 1, torch.device("cuda", 0))          # one shard's data ...
    P, total = one.P, one.P * n
    hb = one.host_buffers()
    rep = lambda t: t.repeat(*([1] * (t.dim() - 1)), n).contiguous().pin_memory()   # ... tiled N times along the points
    forcing, local, hor = rep(hb["forcing"]), rep(hb["local"]), rep(hb["horizons"])
    out = torch.empty((lib.O_NVAR, one.db.n_out, total), dtype=torch.float64).pin_memory()
    status = torch.empty(total, dtype=torch.int32).pin_memory()

    def call(ngpus, o, st, sl=slice(None), statics=None):
        lib.run_host_soa(one.settings, one.params, forcing[:, :, sl].contiguous() if sl != slice(None) else forcing, hb["tf"],
                         local[:, sl].contiguous() if sl != slice(None) else local, o, record_step=hb["rs"],
                         horizons=(hor[:, sl].contiguous() if sl != slice(None) else hor) if statics is None else None,
                         status=st, out_stride=120, ngpus=ngpus, coupling_window_end=one.window_end, statics=statics)
    ref_out = torch.empty((lib.O_NVAR, one.db.n_out, P), dtype=torch.float64)
    ref_status = torch.empty(P, dtype=torch.int32)
    call(1, ref_out, ref_status, slice(0, P))
    handle = lib.prepare_statics(local, hor, ngpus=n)
    for _ in range(max(1, args.warmup)):
        call(n, out, status, statics=handle)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        call(n, out, status, statics=handle)
    dt = time.perf_counter() - t0
    st = lib.last_batch_stats()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out, status, total)
    same = all(bool(torch.equal(out[:, :, k * P:(k + 1) * P], ref_out)) and bool(torch.equal(status[k * P:(k + 1) * P], ref_status))
               for k in range(n))
    lib.release_statics(handle)
    v = total * one.sim_len * args.steps / dt
    line = {"impl": "ours-inproc", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": n, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, n, {"api": f"one process, roadsurf_run_host_soa(..., ngpus={n}) over pinned host "
                                                       "buffers; points [g*P/G,(g+1)*P/G) per GPU, one host thread per GPU"}),
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": int(st["h2d_bytes"]), "d2h_bytes_per_step": int(st["d2h_bytes"])},
            "shards_bit_identical_to_one_gpu_run": same, "gpu_launches": int(st["kernel_launches"]) * args.steps}
    print(json.dumps(line), flush=True)


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return
    if args.inproc:
        run_inproc(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from roadsurf_b200 import build as rs_build
    from roadsurf_b200 import lib, sharding

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        rs_build.build_library()
    sharding.barrier(dev)
    lib.load()
    launches0 = lib.last_launch()["launches_total"]

    wl = Workload(args, rank, world, dev)
    db, P, sim_len = wl.db, wl.P, wl.sim_len
    stream = torch.cuda.current_stream()

    for _ in range(max(args.warmup, 0)):
        wl.step(stream)
    torch.cuda.synchronize()
    sharding.barrier(dev)
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.25)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    launches_before = lib.last_launch()["launches_total"] if args.warmup > 0 else launches0
    db.counters.zero_()
    e0.record(stream)
    for _ in range(args.steps):
        wl.step(stream)
    e1.record(stream)
    torch.cuda.synchronize()
    sharding.barrier(dev)
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop()
    kernel_ms = ms_total / args.steps
    ms_max = sharding.reduce_over_ranks(ms_total, "max", dev)
    total_points = sharding.reduce_over_ranks(P, "sum", dev)
    value = total_points * sim_len * args.steps / (ms_max * 1e-3)
    cnt = db.counters.cpu().numpy()
    failed_points = int(cnt[lib.CNT_FAILED_POINTS]) // max(1, args.steps)
    executed_over_nominal = float(cnt[lib.CNT_EXECUTED_STEPS]) / (float(P) * sim_len * args.steps)
    bl_per_step = float(cnt[lib.CNT_BL_ITERATIONS]) / max(1.0, float(cnt[lib.CNT_EXECUTED_STEPS]))
    launch = lib.last_launch()
    gpu_launches = launch["launches_total"] - launches_before
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, db.out, db.status, P, state=db.state)

    # ---- end to end through the C ABI with host buffers ------------------------------------------
    e2e = None
    if not args.no_e2e:
        h = wl.host_buffers()
        statics = lib.prepare_statics(h["local"], h["horizons"], ngpus=1)

        def one():
            lib.run_host_soa(wl.settings, wl.params, h["forcing"], h["tf"], h["local"], h["out"], record_step=h["rs"],
                             status=h["status"], out_stride=120, ngpus=1, coupling_window_end=wl.window_end,
                             statics=statics)
        one()                                              # warm-up: sizes the device work space
        torch.cuda.synchronize()
        sharding.barrier(dev)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            one()
        torch.cuda.synchronize()
        t_e2e = time.perf_counter() - t0
        sharding.barrier(dev)
        st = lib.last_batch_stats()
        t_max = sharding.reduce_over_ranks(t_e2e, "max", dev)
        same = bool(torch.equal(h["out"].to(dev), db.out[:, :, :P]))
        e2e = {"value": total_points * sim_len * args.steps / t_max, "unit": UNIT,
               "h2d_bytes_per_step": int(st["h2d_bytes"]), "d2h_bytes_per_step": int(st["d2h_bytes"]),
               "ms_per_step": 1e3 * t_max / args.steps,
               "api": "roadsurf_run_host_soa (pinned host buffers; horizon table resident via roadsurf_prepare_statics: "
                      "%d bytes uploaded once, outside the timed region)" % (360 * 8 * P),
               "breakdown_ms": {"h2d": st["h2d_ms"], "kernel": st["kernel_ms"], "d2h": st["d2h_ms"], "chunks": st["groups"]},
               "outputs_equal_device_run": same}
        gpu_launches += st["kernel_launches"] * args.steps
        lib.release_statics(statics)
        del h

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- the binding roofline (fp64) and the HBM one ----------------------------------------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    alg_bytes = (db.forcing[:, :, :P].numel() + db.out[:, :, :P].numel() + db.local[:, :P].numel() +
                 db.horizons[:, :P].numel()) * 8 + P * 4
    hbm_achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
    fp64_peak = lib.measure_fp64_tflops(40000)
    nsample = min(args.cpu_sample_points, P)
    arrays, s_settings, s_params = wl.cpu_case(nsample)
    flops, per = flops_per_point_step(arrays, s_settings, s_params)
    fp64_achieved = flops * P * sim_len / (kernel_ms * 1e-3) / 1e12
    traffic_pps, traffic_src = kernel_traffic_per_point_step()
    traffic = traffic_pps * P * sim_len if (traffic_pps and args.workload == "c4") else None
    roofline = {"bound": "fp64", "achieved": fp64_achieved, "peak": fp64_peak, "unit": "TFLOP/s",
                "frac": fp64_achieved / fp64_peak,
                "peak_source": "DFMA micro-benchmark run live by this script (FMA = 2 flop); MEASURED_PEAKS.json has no fp64 figure",
                "algorithmic_flops_per_point_step": flops, "ops_per_point_step": per,
                "traffic": traffic, "traffic_source": traffic_src,
                "pipe_utilisation": "ncu: fp64 pipe 66.5 % busy, issue slots 66.5 % (profiles/r02_c_cold_outline_ncu_summary.txt)",
                "note": "algorithmic flops count div/sqrt/exp/log/trig as 1 each; in issued fp64 instructions they cost "
                        "~10-40, so the pipe utilisation (ncu) is the fairer reading of how full the machine is"}
    roofline_hbm = {"bound": "hbm", "achieved": hbm_achieved, "peak": hbm_peak, "unit": "GB/s",
                    "frac": hbm_achieved / hbm_peak, "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": "MEASURED_PEAKS.json (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                    "algorithmic_bytes_per_point_step": alg_bytes / (P * sim_len),
                    "note": "coarse-forcing mode moves ~2 B per point-step: HBM is not the binding ceiling of this kernel"}

    # ---- CPU baseline + parity of the benchmarked workload itself ---------------------------------
    cpu_baseline, parity_sample = None, None
    if not args.no_cpu_baseline and world == 1:
        cores = os.cpu_count() or 1
        backend, kind, note = reference_backend()
        r, _, _ = cpu_arm(arrays, s_settings, s_params, 1, 0, cores, fast=True, backend=backend)
        sub = arrays.copy()
        r1, _, _ = cpu_arm(_first(sub, 512), s_settings, s_params, 1, 0, 1, fast=True, backend=backend)
        cpu_baseline = {"value": r["value"], "unit": UNIT, "cores": cores, "kind": kind, "one_core_value": r1["value"],
                        "sample": f"first {r['points']} points of the GPU workload x {r['sim_len']} steps, "
                                  f"{r['seconds']:.1f} s wall on {cores} threads", "note": note}
        # the parity oracle (strict build) on the same points against what the GPU produced in the timed run
        _, work, st_cpu = cpu_arm(arrays, s_settings, s_params, 1, 0, cores, fast=False)
        o = db.out[:, :, :nsample].cpu().numpy()
        names = lib.O_NAMES
        identical = all(np.array_equal(np.ascontiguousarray(o[v].T), work.out[name][:, ::120], equal_nan=True)
                        for v, name in enumerate(names))
        st_gpu = db.status[:nsample].cpu().numpy()
        parity_sample = {"points": int(nsample), "steps_compared": int(o.shape[1]), "bit_identical": bool(identical),
                         "status_words_equal": bool(np.array_equal(st_gpu, st_cpu)),
                         "oracle": "oracle/ strict build (parity unpinned: never compared with a gfortran build)"}

    # ---- the full named configuration on ONE GPU (c4: 10^7 points fit) ----------------------------
    full_config = None
    if (args.workload == "c4" and args.scaling == "weak" and world == 1 and not args.no_full_config
            and not args.points_per_gpu and not args.hours):
        del wl, db
        torch.cuda.empty_cache()
        full_config = run_full_c4(args, dev)

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, world),
            "launch": {"kernel_regs": launch["regs_per_thread"], "grid": launch["grid"], "block": launch["block"],
                       "bl_iterations_per_step": bl_per_step, "failed_points": failed_points,
                       "executed_over_nominal_steps": executed_over_nominal},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(gpu_launches),
            "roofline": roofline, "roofline_hbm": roofline_hbm, "cpu_baseline": cpu_baseline,
            "parity_sample": parity_sample, "full_config": full_config}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def _first(arrays, n):
    """The first n points of a PointArrays (views copied)."""
    from roadsurf_b200 import abi
    import ctypes as C
    n = min(n, arrays.npoints)
    sub = abi.PointArrays(n, arrays.sim_len)
    for name in [f[2:] for f in abi.INPUT_DOUBLE_FIELDS] + ["PrecPhase", "local_horizons", "Depth"]:
        getattr(sub, name)[...] = getattr(arrays, name)[:n]
    sub.time[...] = arrays.time
    C.memmove(sub.local, arrays.local, C.sizeof(abi.LocalParameters) * n)
    return sub


def run_full_c4(args, dev):
    """BASELINE config 4 in full on one B200: 10^7 points x 2881 steps, one launch (65 GB resident)."""
    import torch
    from roadsurf_b200 import abi, lib, synth_torch
    P, hours = WORKLOADS["c4"]["total"], WORKLOADS["c4"]["hours"]
    sim_len = 1 + hours * 120
    lib.set_model(abi.default_settings(sim_len), abi.default_parameters(30.0))
    db = lib.DeviceBatch(P, sim_len, n_records=hours + 2, coarse=True, horizons=True, out_stride=120)
    synth_torch.fill_device_batch_chunked(db, seed=20191206)
    st = torch.cuda.current_stream()
    db.build_order(st)
    db.run(st)                                              # warm-up pass
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    db.build_order(st)
    db.run(st)
    e1.record(st)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    cnt = db.counters.cpu().numpy()
    return {"workload": "c4 in full on one GPU: 10^7 points x 2881 steps, single launch", "points": P, "ms_per_step": ms,
            "value": P * sim_len / (ms * 1e-3), "unit": UNIT, "steps": 1, "warmup": 1,
            "hbm_resident_gb": round(torch.cuda.max_memory_allocated() / 1e9, 1),
            "failed_points": int(cnt[lib.CNT_FAILED_POINTS]) // 2, "grid": lib.last_launch()["grid"]}


if __name__ == "__main__":
    main()
