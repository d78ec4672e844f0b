"""Example-1-style file driver (roadsurf_b200/example1.py): config + weather JSON + sky-view files
in the reference's schema -> forecast JSON.  CPU tests use the oracle as the model; the GPU test
runs the same files through the CUDA library."""
import json
import os

import numpy as np
import pytest

from roadsurf_b200 import example1
from record_refs import interpolate_like_json_source


def _oracle_runner(oracle):
    def runner(arrays, settings, params):
        status, _ = oracle.run_batch(arrays, settings, params, nthreads=4)
        return status
    return runner


def test_config_comments_times_and_parameters(tmp_path):
    path = example1.write_synthetic_inputs(str(tmp_path), nstations=3, analysis=6, forecast=4)
    cfg = example1.load_json(path)
    assert cfg["time"]["analysis"] == 6 and cfg["input"][1]["source"] == "observations"
    cfg["parameters"]["Emiss"] = 0.9
    cfg["model"]["NLayers"] = 12
    times, settings, params, out_step = example1.parse_config(cfg)
    assert settings.SimLen == 1 + (6 + 4) * 120 and settings.NLayers == 12 and out_step == 60
    assert times.forecast - times.start == 6 * 3600 and params.Emiss == 0.9 and params.MinPrecmm == 0.05 * 30 / 3600


def test_interpolation_general_time_grids():
    rawtime = [0, 3600, 5400, 9000, 12600]
    raw = np.array([1.0, 2.0, -9999.9, 4.0, 8.0])
    for start, n in ((0, 400), (-900, 300), (1800, 350)):
        simtime = [start + 30 * i for i in range(n)]
        got = example1.interpolate(rawtime, raw, simtime)
        want = interpolate_like_json_source(raw, rawtime, simtime)
        assert np.array_equal(got, want), start
    ph = example1.interpolate(rawtime, np.array([1, 2, 3, -9999, 1.0]), [0, 30, 3600, 3630, 5400, 5430], next_record=True)
    assert list(ph) == [1, 2, 2, 3, 3, -9999]


def test_file_pipeline_with_cpu_model(tmp_path, oracle):
    path = example1.write_synthetic_inputs(str(tmp_path), nstations=4, seed=3, analysis=6, forecast=6)
    forecast, arrays, status = example1.run(path, runner=_oracle_runner(oracle))
    assert len(forecast) == 4 and os.path.exists(os.path.join(str(tmp_path), "output.json"))
    st0 = forecast[0]
    assert set(st0) == {"statId", "lat", "lon", "time", "RoadTemperature", "Water", "Ice", "Snow", "Deposit"}
    assert st0["time"][0] == "2019-12-01T18:00" and st0["time"][-1] == "2019-12-02T06:00" and len(st0["time"]) == 13
    assert all(-60 < v < 60 for v in st0["RoadTemperature"])
    # read_input derivations.  The reference's interpolation loop stops at the last raw record
    # (JsonSource.cpp:84: rawPos+1 < rawLen), so the observation AT the forecast start is not used:
    # 720 observed steps, coupling to the road-temperature value at index 719
    for q in range(4):
        lp = arrays.local[q]
        assert lp.InitLenI == 720 and lp.couplingIndexI == 719 and lp.couplingTsurf > -100
        assert (arrays.TSurfObs[q, 360:] < -9000).all() and arrays.TSurfObs[q, 359] > -100 and (status[q] & 8)
    # observations overlay the forecast during the analysis (DataHandler.cpp:75-82)
    fc = json.load(open(os.path.join(str(tmp_path), "forecast.json")))[0]
    ob = json.load(open(os.path.join(str(tmp_path), "observations.json")))[0]
    assert arrays.tair[0, 0] == ob["Temperature 2m"][0] and arrays.tair[0, 0] != fc["Temperature 2m"][0]
    assert arrays.tair[0, 840] == pytest.approx(fc["Temperature 2m"][7])        # 7 h after start: forecast only
    assert abs(arrays.local[0].sky_view - float(open(os.path.join(str(tmp_path), "skyview.txt")).readline().split()[4])) < 1e-12
    assert np.allclose(arrays.local_horizons[1], [float(v) for v in open(os.path.join(str(tmp_path), "horizons.txt")).readlines()[1].split()[4:]])


def test_station_with_missing_forecast_is_screened_out(tmp_path, oracle):
    path = example1.write_synthetic_inputs(str(tmp_path), nstations=3, seed=4, analysis=6, forecast=3)
    fpath = os.path.join(str(tmp_path), "forecast.json")
    fc = json.load(open(fpath))
    fc[1]["RadiationLW"][4] = -9999.9        # a hole in a required variable
    json.dump(fc, open(fpath, "w"))
    forecast, arrays, status = example1.run(path, runner=_oracle_runner(oracle), write=False)
    assert status[1] == 256 and (arrays.out["TsurfOut"][1] == -9999.0).all()
    assert status[0] != 256 and arrays.out["TsurfOut"][0, -1] != -9999.0


@pytest.mark.gpu
def test_file_pipeline_on_the_gpu_matches_the_cpu_model(tmp_path, rslib, oracle):
    from parity import S_TOL, T_TOL, compare
    path = example1.write_synthetic_inputs(str(tmp_path), nstations=40, seed=6, analysis=6, forecast=8)
    f_gpu, a_gpu, s_gpu = example1.run(path, write=False)
    f_cpu, a_cpu, s_cpu = example1.run(path, runner=_oracle_runner(oracle), write=False)
    assert np.array_equal(s_gpu, s_cpu)
    r = compare(a_gpu.out, a_cpu.out)
    assert r["max_dT_matching"] <= T_TOL and r["max_dS_matching"] <= S_TOL and r["mismatch_fraction"] <= 0.15, r
    assert [s["statId"] for s in f_gpu] == [s["statId"] for s in f_cpu]


def _build_cpp_example(tmp_path, name="batch_main"):
    import os, subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    from roadsurf_b200 import build
    build.build_library()
    exe = str(tmp_path / name)
    libdir = os.path.join(root, "roadsurf_b200")
    subprocess.run(["g++", "-std=c++17", "-O2", "-pthread", "-Wall", "-Werror", "-I", os.path.join(root, "include"),
                    os.path.join(root, "examples", name + ".cpp"), "-o", exe, "-L", libdir, "-lroadsurf_b200",
                    "-Wl,-rpath," + libdir], check=True, capture_output=True, text=True)
    return exe


def test_cpp_example_main_builds_against_the_c_abi_and_reports_a_missing_gpu(tmp_path):
    """examples/batch_main.cpp (a C++ main shaped like the reference's example1 over the C ABI)
    compiles with -Wall -Werror against include/roadsurf_b200.h, links the library, derives the
    per-point parameters on the host and -- without a GPU -- says so and exits 0."""
    import subprocess
    import torch
    exe = _build_cpp_example(tmp_path)
    r = subprocess.run([exe, "16"], capture_output=True, text=True, timeout=300)
    assert "coupling window ends at index 360" in r.stdout, r.stdout + r.stderr
    if not torch.cuda.is_available():
        assert r.returncode == 0 and "no CUDA device visible" in r.stdout


@pytest.mark.gpu
def test_cpp_example_main_runs_a_coupled_batch(tmp_path):
    """The same program on a GPU: all points coupled, surface temperature steered to the last
    observation at the end of the coupling window (exit code 0)."""
    import subprocess
    exe = _build_cpp_example(tmp_path)
    r = subprocess.run([exe, "200"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "coupled points 200, failed 0" in r.stdout, r.stdout


def test_cpp_stepwise_main_builds_and_reports_a_missing_gpu(tmp_path):
    """examples/step_main.cpp: a main that keeps its own time loop over the step-granular entry points (what the
    Fortran module RoadSurf forwards to) compiles with -Wall -Werror and, without a GPU, says so."""
    import subprocess
    import torch
    exe = _build_cpp_example(tmp_path, "step_main")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert "1 point x 481 steps" in r.stdout, r.stdout + r.stderr
    if not torch.cuda.is_available():
        assert r.returncode == 0 and "no CUDA device visible" in r.stdout


@pytest.mark.gpu
def test_cpp_stepwise_main_equals_runsimulation(tmp_path):
    """The stepwise main on a GPU, one launch per step and with a run-ahead chunk: every output value equals
    runsimulation's (exit code 0)."""
    import subprocess
    exe = _build_cpp_example(tmp_path, "step_main")
    for chunk in ("1", "60"):
        r = subprocess.run([exe, chunk], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
        assert "values differing from runsimulation: 0" in r.stdout, r.stdout


@pytest.mark.gpu
def test_cpp_thread_pool_of_runsimulation_calls_is_batched(tmp_path):
    """The reference's main shape (roadrunner.cpp:454-496): a pool of 16 threads, one runsimulation call per point.
    The calls are combined into batches of about the pool size, and every series equals the one-batch run."""
    import re, subprocess
    exe = _build_cpp_example(tmp_path)
    r = subprocess.run([exe, "200", "16"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    m = re.search(r"in (\d+) launches-batches for (\d+) calls; series differing: (\d+)", r.stdout)
    assert m, r.stdout
    batches, calls, differing = map(int, m.groups())
    assert calls == 200 and differing == 0
    assert batches <= 40, r.stdout          # 200 / 16 = 12.5 ideal; one call per launch would be 200
