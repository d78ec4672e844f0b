"""The drop-in boundary: struct layouts and exported symbols (no GPU needed, no compute calls)."""
import ctypes as C
import os
import re
import subprocess
import tempfile

from roadsurf_b200 import abi, lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "roadsurf_b200.h")

PROBE = r"""
#include <stdio.h>
#include <stddef.h>
#include "roadsurf_b200.h"
#define S(t) printf("sizeof " #t " %zu\n", sizeof(t))
#define O(t, f) printf("offsetof " #t "." #f " %zu\n", offsetof(t, f))
int main(void) {
  S(InputPointers); S(OutputPointers); S(InputSettings); S(InputParameters); S(LocalParameters);
  O(InputPointers, c_tair); O(InputPointers, c_PrecPhase); O(InputPointers, c_local_horizons);
  O(InputPointers, c_Depth); O(InputPointers, c_year); O(InputPointers, c_second);
  O(OutputPointers, c_TsurfOut); O(OutputPointers, c_Ice2Out);
  O(InputSettings, use_coupling); O(InputSettings, use_relaxation); O(InputSettings, force_tsurf);
  O(InputSettings, DTSecs); O(InputSettings, tsurfOutputDepth); O(InputSettings, NLayers);
  O(InputSettings, coupling_minutes); O(InputSettings, couplingEffectReduction); O(InputSettings, outputStep);
  O(InputParameters, Grav); O(InputParameters, freezing_limit_normal); O(InputParameters, MinIcemms);
  O(LocalParameters, couplingIndexI); O(LocalParameters, couplingTsurf); O(LocalParameters, lat);
  O(LocalParameters, sky_view); O(LocalParameters, InitLenI);
  S(RsDeviceBatch); S(RsBatchStats); S(RsLaunchInfo);
  O(RsDeviceBatch, forcing); O(RsDeviceBatch, out_stride); O(RsDeviceBatch, scratch); O(RsDeviceBatch, counters);
  O(RsDeviceBatch, solar); O(RsDeviceBatch, step_begin); O(RsDeviceBatch, out_slot0);
  return 0;
}
"""


def _probe():
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "probe.c")
        exe = os.path.join(d, "probe")
        with open(src, "w") as f:
            f.write(PROBE)
        subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), src, "-o", exe], check=True)
        out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    res = {}
    for line in out.splitlines():
        kind, name, val = line.split()
        res[(kind, name)] = int(val)
    return res


def test_reference_struct_layouts_match_the_survey_table():
    """SURVEY.md section 8b: 160 / 56 / 56 / 552 / 72 bytes, force_tsurf at offset 12."""
    p = _probe()
    assert p[("sizeof", "InputPointers")] == 160
    assert p[("sizeof", "OutputPointers")] == 56
    assert p[("sizeof", "InputSettings")] == 56
    assert p[("sizeof", "InputParameters")] == 552
    assert p[("sizeof", "LocalParameters")] == 72
    assert p[("offsetof", "InputPointers.c_tair")] == 8
    assert p[("offsetof", "InputPointers.c_second")] == 152
    assert p[("offsetof", "OutputPointers.c_Ice2Out")] == 48
    expected = {"use_coupling": 4, "use_relaxation": 8, "force_tsurf": 12, "DTSecs": 16, "tsurfOutputDepth": 24,
                "NLayers": 32, "coupling_minutes": 36, "couplingEffectReduction": 40, "outputStep": 48}
    for k, v in expected.items():
        assert p[("offsetof", "InputSettings." + k)] == v
    expected = {"couplingIndexI": 24, "couplingTsurf": 32, "lat": 40, "sky_view": 56, "InitLenI": 64}
    for k, v in expected.items():
        assert p[("offsetof", "LocalParameters." + k)] == v
    assert p[("offsetof", "InputParameters.Grav")] == 6 * 8
    assert p[("offsetof", "InputParameters.MinIcemms")] == 68 * 8


def test_ctypes_mirrors_match_the_c_header():
    p = _probe()
    for t in (abi.InputPointers, abi.OutputPointers, abi.InputSettings, abi.InputParameters, abi.LocalParameters,
              lib.RsDeviceBatch, lib.RsBatchStats, lib.RsLaunchInfo):
        assert C.sizeof(t) == p[("sizeof", t.__name__)], t.__name__
    for (kind, name), val in p.items():
        if kind != "offsetof":
            continue
        tname, field = name.split(".")
        t = getattr(abi, tname, None) or getattr(lib, tname)
        assert getattr(t, field).offset == val, name


def test_parameter_order_follows_the_fortran_type():
    """src/InputParameters.f90.inc:6-89 order, spot-checked at the block boundaries."""
    n = abi.PARAMETER_NAMES
    assert n[0] == "NightOn" and n[5] == "TrFfricDay" and n[6] == "Grav" and n[16] == "PorEvaF"
    assert n[17] == "ZRefW" and n[40] == "Silt2" and n[41] == "freezing_limit_normal"
    assert n[46] == "T4Melt_normal" and n[50] == "WetSnowMeltR" and n[56] == "MaxExtmms"
    assert n[57] == "MissValI" and n[59] == "Snow2IceFac" and n[60] == "MinPrecmm" and n[68] == "MinIcemms"


def test_default_parameters_follow_the_example():
    """examples/example1/src/InputParameters.h:18-110 and InputParameters.cpp:11-22."""
    p = abi.default_parameters(30.0)
    assert p.NightOn == 19.0 and p.NightOff == 4.0 and p.VK_Const == 0.4 and p.WatDens == 999.87
    assert p.freezing_limit_normal == -0.25 and p.frost_melting_limit_normal == 1.25
    assert p.MinPrecmm == 0.05 * 30.0 / 3600.0 and p.MinSnowmms == 0.1 * 30.0 / 3600.0
    assert p.MaxWatmms == 2.0 and p.WWetLim == 0.9 and p.WWearLim == 0.1 and p.Snow2IceFac == 0.5


def _declared_functions():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = re.sub(r"^\s*#.*$", "", text, flags=re.M)  # preprocessor lines (function-like macros)
    names = re.findall(r"\b([A-Za-z_][A-Za-z0-9_]*)\s*\([^;{}]*\)\s*;", text)
    return sorted(set(n for n in names if n.startswith("roadsurf_") or n == "runsimulation"))


def test_library_loads_and_exports_every_declared_symbol():
    declared = _declared_functions()
    assert "runsimulation" in declared and "roadsurf_run_batch" in declared and len(declared) >= 12
    handle = lib.load()
    for name in declared:
        assert hasattr(handle, name), f"{name} declared in include/roadsurf_b200.h but not exported"
    assert set(declared) == set(lib.EXPORTS)
    # no compute here: only calls that are valid without a GPU
    assert handle.roadsurf_version().decode().startswith("roadsurf_b200")
    assert handle.roadsurf_device_count() >= 0


def test_product_package_never_touches_the_oracle():
    """The oracle is test infrastructure: nothing under roadsurf_b200/ may import or link it."""
    pkg = os.path.join(ROOT, "roadsurf_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", ".f90")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "oracle" not in text.lower(), os.path.join(dirpath, f)


def test_batch_entry_fails_loudly_without_a_gpu():
    """No CPU fallback: without a device the batched call returns RS_ERR_NO_DEVICE."""
    handle = lib.load()
    if handle.roadsurf_device_count() > 0:
        return
    import pytest
    from roadsurf_b200 import synth
    arrays, settings, params, _ = synth.make_case(2, 1, seed=1)
    with pytest.raises(lib.RoadSurfError, match="no CUDA device"):
        lib.run_batch(arrays, settings, params)


def test_new_entry_points_fail_loudly_without_a_gpu_and_validate_arguments():
    """Sessions and prepared statics have no CPU path either; argument errors are reported before any device
    work (these run on the CPU box)."""
    import ctypes as C
    import numpy as np
    import pytest
    from roadsurf_b200 import synth
    handle = lib.load()
    arrays, settings, params, rec = synth.make_case(2, 1, seed=1)
    # example2's rule is a device-entry feature: the host-SoA entry says so instead of misreading the records
    forcing = np.zeros((rec.nrec, 11, 2))
    local = np.zeros((lib.L_NLOCAL, 2))
    out = np.zeros((lib.O_NVAR, arrays.sim_len, 2))
    hb = lib.RsHostBatch(npoints=2, sim_len=arrays.sim_len, forcing_mode=2, n_records=rec.nrec, nvar=11, out_stride=1,
                         forcing=forcing.ctypes.data, record_step=rec.record_step.ctypes.data,
                         time_fields=arrays.time.ctypes.data, local=local.ctypes.data, out=out.ctypes.data)
    assert handle.roadsurf_run_host_soa(C.byref(hb), C.byref(settings), C.byref(params), 1) == -4   # RS_ERR_UNSUPPORTED
    assert b"forcing_mode 0 or 1" in handle.roadsurf_last_error()
    if handle.roadsurf_device_count() > 0:
        return
    with pytest.raises(lib.RoadSurfError, match="no CUDA device"):
        lib.Session(arrays, settings, params)
    with pytest.raises(lib.RoadSurfError, match="no CUDA device"):
        lib.prepare_statics(local, None, ngpus=1)
    # a stale / foreign handle is rejected, not dereferenced blindly
    assert handle.roadsurf_session_done(None) < 0


def test_every_run_time_option_is_documented_in_the_header():
    """roadsurf_set_option: every name the library accepts is described in include/roadsurf_b200.h, and an
    unknown name is rejected (host only)."""
    import os
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = open(os.path.join(root, "roadsurf_b200", "csrc", "rs_host.cu")).read()
    body = src[src.index("int roadsurf_set_option("):]
    body = body[:body.index("\n}\n")]
    names = re.findall(r'strcmp\(name, "([a-z_0-9]+)"\)', body)
    assert len(names) >= 6, names
    header = open(os.path.join(root, "include", "roadsurf_b200.h")).read()
    for n in names:
        assert '"%s"' % n in header, n
    from roadsurf_b200 import lib
    import pytest
    with pytest.raises(Exception):
        lib.set_option("no_such_option", 1)


def test_record_grids_are_checked_before_any_device_work():
    """forcing_mode 1 needs record_step strictly increasing with record_step[0] <= 0: the kernel and the host
    derivation extrapolate the first interval back to step 0 where example1's JsonSource leaves those steps
    missing, and two equal steps divide by a zero span.  Every entry that holds record_step in host memory
    rejects another grid with RS_ERR_BAD_ARGUMENT before it looks for a device (these run on the CPU box)."""
    import ctypes as C
    import numpy as np
    import pytest
    from roadsurf_b200 import synth
    arrays, settings, params, rec = synth.make_case(3, 2, seed=1)
    nrec, sim_len = rec.nrec, arrays.sim_len
    forcing = np.zeros((nrec, 11, 3))
    local = np.zeros((lib.L_NLOCAL, 3))
    out = np.zeros((lib.O_NVAR, sim_len, 3))
    good = rec.record_step.astype(np.int32)
    bad_grids = {
        "after step 0": good + 1,
        "repeated step": np.where(np.arange(nrec) == 2, good[1], good).astype(np.int32),
        "decreasing": good[::-1].copy(),
        "two records, equal": np.array([0, 0], dtype=np.int32),
    }
    handle = lib.load()
    for name, rs in bad_grids.items():
        n = len(rs)
        f = np.ascontiguousarray(forcing[:n])
        hb = lib.RsHostBatch(npoints=3, sim_len=sim_len, forcing_mode=1, n_records=n, nvar=11, out_stride=1,
                             forcing=f.ctypes.data, record_step=rs.ctypes.data, time_fields=arrays.time.ctypes.data,
                             local=local.ctypes.data, out=out.ctypes.data)
        assert handle.roadsurf_run_host_soa(C.byref(hb), C.byref(settings), C.byref(params), 1) == -2, name
        assert b"record_step" in handle.roadsurf_last_error(), name
        with pytest.raises(lib.RoadSurfError, match="record_step"):
            lib.read_input_derive_records(f, rs, settings, 0, local)
        if n > 2:
            members = np.zeros((n - 2, 11, 3 * 2))
            with pytest.raises(lib.RoadSurfError, match="record_step"):
                lib.run_ensemble_host_soa(settings, params, f, rs, arrays.time, local, members, 2, 122, lib.stats_spec())
    # the grid the entries are built for passes the check (the derivation is pure host code)
    assert lib.read_input_derive_records(np.ascontiguousarray(forcing), good, settings, 0, local) == 0
    for first in (0, -1, -500):
        lib.read_input_derive_records(np.ascontiguousarray(forcing), (good + first).astype(np.int32), settings, 0, local)
