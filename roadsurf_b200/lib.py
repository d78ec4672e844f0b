"""ctypes binding of libroadsurf_b200.so (the C ABI declared in include/roadsurf_b200.h).

The library is the product; this module only loads it and marshals arguments.  There is no Python
or CPU implementation of the model behind these calls: if the shared library is missing, or no
CUDA device is visible, the calls raise.
"""
import ctypes as C
import os

import numpy as np

from . import abi

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, os.environ.get("ROADSURF_B200_LIBNAME", "libroadsurf_b200.so"))

# enums of include/roadsurf_b200.h
ST_FAILED, ST_BAD_INPUT, ST_ABNORMAL_TSURF, ST_COUPLING_USED, ST_COUPLING_FAILED = 1, 2, 4, 8, 16
ST_BL_NOT_CONVERGED, ST_SOLAR_GEOMETRY, ST_BAD_WINDOW, ST_NOT_RUN = 32, 64, 128, 256
ST_BAD_FORK = 512
F_NVAR, F_NVAR_DEPTH = 11, 12
F_NAMES = ("tair", "tdew", "VZ", "Rhz", "prec", "SW", "LW", "SW_dir", "LW_net", "TSurfObs", "PrecPhase",
           "Depth")
(L_TAIR_RELAX, L_VZ_RELAX, L_RH_RELAX, L_COUPLING_TSURF, L_LAT, L_LON, L_SKY_VIEW, L_COUPLING_INDEX,
 L_INIT_LEN, L_ACTIVE, L_NLOCAL) = range(11)
O_NAMES = ("TsurfOut", "SnowOut", "WaterOut", "IceOut", "DepositOut", "Ice2Out")
O_NVAR = 6
O_NAMES_EXT = ("Tair", "Tdew", "DewPointDeficit")   # examples/example2/src/QueryDataTools.cpp:325-341
O_NVAR_EXT = 9
CNT_EXECUTED_STEPS, CNT_BL_ITERATIONS, CNT_COUPLING_PASSES, CNT_FAILED_POINTS, CNT_N = 0, 1, 2, 3, 8

EXPORTS = ("runsimulation", "roadsurf_last_error", "roadsurf_device_count", "roadsurf_run_batch",
           "roadsurf_run_host_soa", "roadsurf_read_input_derive", "roadsurf_read_input_derive_records",
           "roadsurf_last_batch_stats", "roadsurf_set_model", "roadsurf_run_device",
           "roadsurf_transpose_to_soa", "roadsurf_transpose_from_soa", "roadsurf_fill",
           "roadsurf_measure_fp64_tflops", "roadsurf_selftest_arith", "roadsurf_selftest_libm", "roadsurf_runsimulation_counters", "roadsurf_order_points", "roadsurf_default_parameters",
           "roadsurf_default_settings", "roadsurf_set_option", "roadsurf_release_workspace",
           "roadsurf_last_launch", "roadsurf_prepare_statics", "roadsurf_release_statics",
           "roadsurf_session_open", "roadsurf_step", "roadsurf_session_fetch", "roadsurf_session_set_chunk",
           "roadsurf_session_done", "roadsurf_session_close", "roadsurf_expand_records",
           "roadsurf_sun_position", "roadsurf_eval_primitive",
           "roadsurf_version",
           "roadsurf_run_ensemble_device", "roadsurf_ensemble_stats", "roadsurf_run_ensemble_host_soa",
           "roadsurf_ensemble_area_events", "roadsurf_run_ensemble_host_soa_areas",
           "roadsurf_ensemble_onset", "roadsurf_run_ensemble_host_soa_onset",
           "roadsurf_ensemble_extremes", "roadsurf_run_ensemble_host_soa_extremes")
(PRIM_EXP, PRIM_EXP_SMEM, PRIM_LOG, PRIM_LOG_SMEM, PRIM_EXP_FLAT, PRIM_EXP_FLAT_SMEM, PRIM_PSIH_UNSTABLE,
 PRIM_PSIH_UNSTABLE_SMEM, PRIM_FRCP, PRIM_FDIV, PRIM_DIV_CONST, PRIM_N) = range(12)
ENS_MAX_MEMBERS, ENS_MAX_QUANTILES, ENS_MAX_THRESHOLDS = 128, 8, 8
ENS_MAX_EVENTS, ENS_MAX_CONDITIONS = 8, 4
ENS_NVALID, ENS_MEAN, ENS_STD, ENS_MIN, ENS_MAX, ENS_NFIXED = range(6)
ENS_LT, ENS_LE, ENS_GT, ENS_GE = range(4)
ENS_OPS = {"<": ENS_LT, "<=": ENS_LE, ">": ENS_GT, ">=": ENS_GE}
ENS_MAX_EXTREMES = 8
ENS_WMIN, ENS_WMAX = 0, 1
ENS_KINDS = {"min": ENS_WMIN, "max": ENS_WMAX}


def state_nplanes(nlayers):
    return nlayers + 2 + 19


def scratch_nplanes(nlayers):
    return 2 * nlayers + 17


class RsBatchStats(C.Structure):
    _fields_ = [("pack_ms", C.c_double), ("h2d_ms", C.c_double), ("kernel_ms", C.c_double),
                ("d2h_ms", C.c_double), ("unpack_ms", C.c_double), ("h2d_bytes", C.c_int64),
                ("d2h_bytes", C.c_int64), ("executed_steps", C.c_int64), ("kernel_launches", C.c_int),
                ("groups", C.c_int), ("wall_ms", C.c_double), ("setup_ms", C.c_double)]


class RsLaunchInfo(C.Structure):
    _fields_ = [("grid", C.c_int), ("block", C.c_int), ("smem_bytes", C.c_int),
                ("regs_per_thread", C.c_int), ("nlayers", C.c_int), ("forcing_mode", C.c_int),
                ("launches_total", C.c_int)]


class RsDeviceBatch(C.Structure):
    _fields_ = [("npoints", C.c_int), ("ld", C.c_int), ("sim_len", C.c_int), ("forcing_mode", C.c_int),
                ("n_records", C.c_int), ("nvar", C.c_int),
                ("forcing", C.c_void_p), ("record_step", C.c_void_p), ("time_fields", C.c_void_p),
                ("local", C.c_void_p), ("horizons", C.c_void_p), ("out", C.c_void_p),
                ("out_stride", C.c_int), ("n_out", C.c_int), ("status", C.c_void_p),
                ("state", C.c_void_p), ("scratch", C.c_void_p), ("counters", C.c_void_p),
                ("solar", C.c_void_p), ("step_begin", C.c_int), ("step_end", C.c_int),
                ("forcing_step0", C.c_int), ("out_slot0", C.c_int), ("out_start", C.c_int),
                ("out_nvar", C.c_int), ("order", C.c_void_p), ("expand_workspace", C.c_void_p),
                ("expand_steps", C.c_int), ("coupling_window_end", C.c_int)]


class RsHostBatch(C.Structure):
    _fields_ = [("npoints", C.c_int), ("sim_len", C.c_int), ("forcing_mode", C.c_int), ("n_records", C.c_int),
                ("nvar", C.c_int), ("out_stride", C.c_int),
                ("forcing", C.c_void_p), ("record_step", C.c_void_p), ("time_fields", C.c_void_p),
                ("local", C.c_void_p), ("horizons", C.c_void_p), ("out", C.c_void_p), ("status", C.c_void_p),
                ("coupling_window_end", C.c_int), ("statics", C.c_void_p)]


class RsEnsembleThreshold(C.Structure):
    _fields_ = [("plane", C.c_int), ("op", C.c_int), ("value", C.c_double)]


class RsEnsembleEvent(C.Structure):
    _fields_ = [("n_conditions", C.c_int), ("window", C.c_int), ("conditions", RsEnsembleThreshold * 4)]


class RsEnsembleStatsSpec(C.Structure):
    _fields_ = [("n_quantiles", C.c_int), ("n_thresholds", C.c_int), ("quantiles", C.c_double * 8),
                ("thresholds", RsEnsembleThreshold * 8), ("n_events", C.c_int), ("events", RsEnsembleEvent * 8)]

    @property
    def n_prob(self):
        """Planes of the probability tensor: the thresholds, then the events."""
        return self.n_thresholds + self.n_events


class RsEnsembleBatch(C.Structure):
    _fields_ = [("shared", RsDeviceBatch), ("members", C.c_int), ("fork_step", C.c_int), ("ld_members", C.c_int),
                ("member_forcing", C.c_void_p), ("member_relax", C.c_void_p), ("member_local", C.c_void_p),
                ("member_horizons", C.c_void_p), ("member_state", C.c_void_p), ("member_scratch", C.c_void_p),
                ("member_status", C.c_void_p), ("member_out", C.c_void_p), ("n_out_members", C.c_int),
                ("member_order", C.c_void_p), ("spec", RsEnsembleStatsSpec), ("stats", C.c_void_p),
                ("prob", C.c_void_p)]


class RsEnsembleAreas(C.Structure):
    _fields_ = [("n_areas", C.c_int), ("offsets", C.c_void_p), ("stations", C.c_void_p)]


def ensemble_areas(station_lists):
    """RsEnsembleAreas from a list of areas, each a list of station indices (a route, a district, ...).  The struct
    keeps the int32 arrays it points to alive (attributes `offsets_array`, `stations_array`)."""
    lists = [np.asarray(a, dtype=np.int32).ravel() for a in station_lists]
    offsets = np.zeros(len(lists) + 1, dtype=np.int32)
    offsets[1:] = np.cumsum([len(a) for a in lists])
    stations = np.ascontiguousarray(np.concatenate(lists) if lists else np.zeros(0, dtype=np.int32))
    areas = RsEnsembleAreas(n_areas=len(lists), offsets=offsets.ctypes.data, stations=stations.ctypes.data)
    areas.offsets_array, areas.stations_array = offsets, stations
    return areas


class RsEnsembleExtreme(C.Structure):
    _fields_ = [("plane", C.c_int), ("kind", C.c_int), ("window", C.c_int)]


class RsEnsembleExtremes(C.Structure):
    _fields_ = [("n_extremes", C.c_int), ("extremes", RsEnsembleExtreme * ENS_MAX_EXTREMES)]


def ensemble_extremes(extremes):
    """RsEnsembleExtremes from [(plane, kind, window), ...], kind "min" or "max" (or an ENS_W* code): the minimum or
    maximum of the plane over the window of output slots starting at each slot."""
    extremes = list(extremes)
    if not 1 <= len(extremes) <= ENS_MAX_EXTREMES:
        raise ValueError("1 to 8 extremes")
    ext = RsEnsembleExtremes(n_extremes=len(extremes))
    for x, (plane, kind, window) in enumerate(extremes):
        code = ENS_KINDS.get(kind, kind)
        if code not in (ENS_WMIN, ENS_WMAX) or isinstance(code, bool):
            raise ValueError(f"unknown extreme kind {kind!r}: 'min', 'max', ENS_WMIN or ENS_WMAX")
        ext.extremes[x] = RsEnsembleExtreme(int(plane), code, int(window))
    return ext


def stats_spec(quantiles=(), thresholds=(), events=()):
    """RsEnsembleStatsSpec from quantiles [q, ...], thresholds [(plane, op, value), ...], op one of
    "<", "<=", ">", ">=" (or an ENS_* code), and events [(conditions, window), ...] whose conditions are
    [(plane, op, value), ...] in the threshold form, combined with AND.  Event j is probability plane
    n_thresholds + j."""
    quantiles, thresholds, events = list(quantiles), list(thresholds), list(events)
    if len(quantiles) > ENS_MAX_QUANTILES or len(thresholds) > ENS_MAX_THRESHOLDS:
        raise ValueError("at most 8 quantiles and 8 thresholds")
    if len(events) > ENS_MAX_EVENTS or any(not 1 <= len(conds) <= ENS_MAX_CONDITIONS for conds, _ in events):
        raise ValueError("at most 8 events of 1 to 4 conditions")
    sp = RsEnsembleStatsSpec(n_quantiles=len(quantiles), n_thresholds=len(thresholds), n_events=len(events))
    for j, q in enumerate(quantiles):
        sp.quantiles[j] = float(q)
    for j, (plane, op, value) in enumerate(thresholds):
        sp.thresholds[j] = RsEnsembleThreshold(int(plane), ENS_OPS.get(op, op), float(value))
    for j, (conds, window) in enumerate(events):
        sp.events[j].n_conditions, sp.events[j].window = len(conds), int(window)
        for c, (plane, op, value) in enumerate(conds):
            sp.events[j].conditions[c] = RsEnsembleThreshold(int(plane), ENS_OPS.get(op, op), float(value))
    return sp


class RoadSurfError(RuntimeError):
    pass


_lib = None


def load():
    """Load libroadsurf_b200.so; raises if it has not been built (see roadsurf_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RoadSurfError(f"{LIB_PATH} is missing: run `python -m roadsurf_b200.build` "
                            "(there is no fallback implementation)")
    lib = C.CDLL(LIB_PATH)
    P = C.POINTER
    OP, IP, IS, IPa, LP = (abi.OutputPointers, abi.InputPointers, abi.InputSettings, abi.InputParameters,
                           abi.LocalParameters)
    lib.runsimulation.argtypes = [P(OP), P(IP), P(IS), P(IPa), P(LP)]
    lib.runsimulation.restype = None
    lib.roadsurf_last_error.restype = C.c_char_p
    lib.roadsurf_version.restype = C.c_char_p
    lib.roadsurf_device_count.restype = C.c_int
    lib.roadsurf_run_batch.argtypes = [C.c_int, P(P(OP)), P(P(IP)), P(IS), P(IPa), P(P(LP)), C.c_int,
                                       P(C.c_int)]
    lib.roadsurf_run_batch.restype = C.c_int
    lib.roadsurf_run_host_soa.argtypes = [P(RsHostBatch), P(IS), P(IPa), C.c_int]
    lib.roadsurf_run_host_soa.restype = C.c_int
    lib.roadsurf_read_input_derive.argtypes = [C.c_int, P(P(IP)), P(IS), C.c_int, P(C.c_int), P(P(LP)), P(C.c_int)]
    lib.roadsurf_read_input_derive.restype = C.c_int
    lib.roadsurf_read_input_derive_records.argtypes = [P(RsHostBatch), P(IS), C.c_int, P(C.c_int), C.c_void_p,
                                                       P(C.c_int)]
    lib.roadsurf_read_input_derive_records.restype = C.c_int
    lib.roadsurf_last_batch_stats.argtypes = [P(RsBatchStats)]
    lib.roadsurf_set_model.argtypes = [P(IS), P(IPa)]
    lib.roadsurf_set_model.restype = C.c_int
    lib.roadsurf_run_device.argtypes = [P(RsDeviceBatch), C.c_void_p]
    lib.roadsurf_run_device.restype = C.c_int
    lib.roadsurf_transpose_to_soa.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                              C.c_void_p]
    lib.roadsurf_transpose_to_soa.restype = C.c_int
    lib.roadsurf_transpose_from_soa.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int64,
                                                C.c_void_p]
    lib.roadsurf_transpose_from_soa.restype = C.c_int
    lib.roadsurf_fill.argtypes = [C.c_void_p, C.c_int64, C.c_double, C.c_void_p]
    lib.roadsurf_fill.restype = C.c_int
    lib.roadsurf_eval_primitive.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    lib.roadsurf_eval_primitive.restype = C.c_int
    lib.roadsurf_measure_fp64_tflops.argtypes = [C.c_int]
    lib.roadsurf_measure_fp64_tflops.restype = C.c_double
    lib.roadsurf_set_option.argtypes = [C.c_char_p, C.c_int]
    lib.roadsurf_set_option.restype = C.c_int
    lib.roadsurf_selftest_arith.argtypes = [C.c_longlong, C.c_ulonglong, P(C.c_longlong)]
    lib.roadsurf_selftest_arith.restype = C.c_longlong
    lib.roadsurf_selftest_libm.argtypes = [C.c_longlong, C.c_ulonglong, P(C.c_longlong)]
    lib.roadsurf_selftest_libm.restype = C.c_longlong
    lib.roadsurf_runsimulation_counters.argtypes = [P(C.c_longlong), P(C.c_longlong)]
    lib.roadsurf_runsimulation_counters.restype = None
    lib.roadsurf_order_points.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.roadsurf_order_points.restype = C.c_int
    lib.roadsurf_default_parameters.argtypes = [P(IPa), C.c_double]
    lib.roadsurf_default_parameters.restype = None
    lib.roadsurf_default_settings.argtypes = [P(IS), C.c_int, C.c_double]
    lib.roadsurf_default_settings.restype = None
    lib.roadsurf_last_launch.argtypes = [P(RsLaunchInfo)]
    lib.roadsurf_run_ensemble_device.argtypes = [P(RsEnsembleBatch), C.c_void_p]
    lib.roadsurf_run_ensemble_device.restype = C.c_int
    lib.roadsurf_ensemble_stats.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                            P(RsEnsembleStatsSpec), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    lib.roadsurf_ensemble_stats.restype = C.c_int
    lib.roadsurf_run_ensemble_host_soa.argtypes = [P(RsHostBatch), C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                                   P(RsEnsembleStatsSpec), C.c_void_p, C.c_void_p, C.c_void_p,
                                                   C.c_void_p, P(IS), P(IPa)]
    lib.roadsurf_run_ensemble_host_soa.restype = C.c_int
    lib.roadsurf_ensemble_area_events.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                                  P(RsEnsembleStatsSpec), P(RsEnsembleAreas), C.c_void_p, C.c_void_p]
    lib.roadsurf_ensemble_area_events.restype = C.c_int
    lib.roadsurf_run_ensemble_host_soa_areas.argtypes = [P(RsHostBatch), C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                                         P(RsEnsembleStatsSpec), C.c_void_p, C.c_void_p, C.c_void_p,
                                                         C.c_void_p, P(RsEnsembleAreas), C.c_void_p, P(IS), P(IPa)]
    lib.roadsurf_run_ensemble_host_soa_areas.restype = C.c_int
    lib.roadsurf_ensemble_onset.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                            P(RsEnsembleStatsSpec), C.c_void_p, C.c_int, P(RsEnsembleAreas),
                                            C.c_void_p, C.c_void_p]
    lib.roadsurf_ensemble_onset.restype = C.c_int
    lib.roadsurf_run_ensemble_host_soa_onset.argtypes = [P(RsHostBatch), C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                                         P(RsEnsembleStatsSpec), C.c_void_p, C.c_void_p, C.c_void_p,
                                                         C.c_void_p, P(RsEnsembleAreas), C.c_void_p, C.c_void_p,
                                                         C.c_void_p, P(IS), P(IPa)]
    lib.roadsurf_run_ensemble_host_soa_onset.restype = C.c_int
    lib.roadsurf_ensemble_extremes.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                               P(RsEnsembleStatsSpec), P(RsEnsembleExtremes), C.c_void_p, C.c_int,
                                               P(RsEnsembleAreas), C.c_void_p, C.c_void_p]
    lib.roadsurf_ensemble_extremes.restype = C.c_int
    lib.roadsurf_run_ensemble_host_soa_extremes.argtypes = [P(RsHostBatch), C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                                            P(RsEnsembleStatsSpec), C.c_void_p, C.c_void_p,
                                                            C.c_void_p, C.c_void_p, P(RsEnsembleAreas), C.c_void_p,
                                                            C.c_void_p, C.c_void_p, P(RsEnsembleExtremes),
                                                            C.c_void_p, C.c_void_p, P(IS), P(IPa)]
    lib.roadsurf_run_ensemble_host_soa_extremes.restype = C.c_int
    _lib = lib
    return lib


def _check(rc):
    if rc != 0:
        raise RoadSurfError(f"roadsurf_b200 error {rc}: {load().roadsurf_last_error().decode()}")


def last_batch_stats():
    st = RsBatchStats()
    load().roadsurf_last_batch_stats(C.byref(st))
    return {n: getattr(st, n) for n, _ in RsBatchStats._fields_}


def last_launch():
    li = RsLaunchInfo()
    load().roadsurf_last_launch(C.byref(li))
    return {n: getattr(li, n) for n, _ in RsLaunchInfo._fields_}


class PreparedBatch:
    """The ctypes argument arrays of roadsurf_run_batch for a PointArrays (built once: constructing
    tens of thousands of ctypes structs in Python takes longer than the GPU run)."""

    def __init__(self, arrays):
        self.arrays = arrays
        self.ins = arrays.input_pointers()
        self.outs = arrays.output_pointers()
        self.in_ptrs = abi.pointer_arrays(self.ins, abi.InputPointers)
        self.out_ptrs = abi.pointer_arrays(self.outs, abi.OutputPointers)
        self.loc_ptrs = abi.pointer_arrays(arrays.local, abi.LocalParameters)
        self.status = np.zeros(arrays.npoints, dtype=np.int32)

    def run(self, settings, params, ngpus=1):
        _check(load().roadsurf_run_batch(self.arrays.npoints, self.out_ptrs, self.in_ptrs, C.byref(settings),
                                         C.byref(params), self.loc_ptrs, int(ngpus),
                                         self.status.ctypes.data_as(abi.c_int_p)))
        return self.status


def run_batch(arrays, settings, params, ngpus=1):
    """roadsurf_run_batch over a host-layout PointArrays: fills arrays.out, returns status[npoints]."""
    return PreparedBatch(arrays).run(settings, params, ngpus)


def prepare_statics(local, horizons, ngpus=1):
    """roadsurf_prepare_statics: upload the horizon table of a grid once; returns the handle to pass as
    `statics=` to run_host_soa (release with release_statics)."""
    def ptr(x):
        if x is None:
            return None
        return x.data_ptr() if hasattr(x, "data_ptr") else x.ctypes.data
    npoints = local.shape[1]
    hb = RsHostBatch(npoints=npoints, local=ptr(local), horizons=ptr(horizons))
    handle = C.c_void_p(None)
    lib = load()
    lib.roadsurf_prepare_statics.argtypes = [C.POINTER(RsHostBatch), C.c_int, C.POINTER(C.c_void_p)]
    _check(lib.roadsurf_prepare_statics(C.byref(hb), int(ngpus), C.byref(handle)))
    return handle


def release_statics(handle):
    lib = load()
    lib.roadsurf_release_statics.argtypes = [C.c_void_p]
    lib.roadsurf_release_statics.restype = None
    lib.roadsurf_release_statics(handle)


def run_host_soa(settings, params, forcing, time_fields, local, out, record_step=None, horizons=None,
                 status=None, out_stride=1, ngpus=1, coupling_window_end=0, statics=None):
    """roadsurf_run_host_soa on host tensors/arrays (torch CPU tensors -- ideally pinned -- or numpy):
    forcing [n_records, nvar, npoints] f64, time_fields [6, sim_len] i32, local [L_NLOCAL, npoints],
    out [6, n_out, npoints] (written), record_step [n_records] i32 for coarse forcing."""
    def ptr(x):
        if x is None:
            return None
        return x.data_ptr() if hasattr(x, "data_ptr") else x.ctypes.data
    n_records, nvar, npoints = forcing.shape
    sim_len = time_fields.shape[1]
    n_out = (sim_len + out_stride - 1) // out_stride
    assert tuple(out.shape) == (O_NVAR, n_out, npoints) and tuple(local.shape) == (L_NLOCAL, npoints)
    hb = RsHostBatch(npoints=npoints, sim_len=sim_len, forcing_mode=0 if record_step is None else 1,
                     n_records=n_records, nvar=nvar, out_stride=out_stride, forcing=ptr(forcing),
                     record_step=ptr(record_step), time_fields=ptr(time_fields), local=ptr(local),
                     horizons=ptr(horizons), out=ptr(out), status=ptr(status),
                     coupling_window_end=int(coupling_window_end), statics=statics)
    _check(load().roadsurf_run_host_soa(C.byref(hb), C.byref(settings), C.byref(params), int(ngpus)))


class Session:
    """Step-granular run of a PointArrays on the device (roadsurf_session_open / roadsurf_step /
    roadsurf_session_fetch): what the Fortran subroutine API of module RoadSurf forwards to."""

    def __init__(self, arrays, settings, params, chunk=1):
        lib = load()
        P = C.POINTER
        lib.roadsurf_session_open.argtypes = [C.c_int, P(P(abi.OutputPointers)), P(P(abi.InputPointers)),
                                              P(abi.InputSettings), P(abi.InputParameters),
                                              P(P(abi.LocalParameters)), P(C.c_void_p)]
        lib.roadsurf_step.argtypes = [C.c_void_p, C.c_int]
        lib.roadsurf_session_fetch.argtypes = [C.c_void_p, C.c_int, P(C.c_int)]
        lib.roadsurf_session_set_chunk.argtypes = [C.c_void_p, C.c_int]
        lib.roadsurf_session_done.argtypes = [C.c_void_p]
        lib.roadsurf_session_close.argtypes = [C.c_void_p]
        lib.roadsurf_session_close.restype = None
        self._keep = (arrays.input_pointers(), arrays.output_pointers(), arrays)
        ins, outs, _ = self._keep
        self._ptrs = (abi.pointer_arrays(outs, abi.OutputPointers), abi.pointer_arrays(ins, abi.InputPointers),
                      abi.pointer_arrays(arrays.local, abi.LocalParameters))
        self.handle = C.c_void_p(None)
        self.npoints = arrays.npoints
        _check(lib.roadsurf_session_open(arrays.npoints, self._ptrs[0], self._ptrs[1], C.byref(settings),
                                         C.byref(params), self._ptrs[2], C.byref(self.handle)))
        if chunk > 1:
            _check(lib.roadsurf_session_set_chunk(self.handle, int(chunk)))

    def step(self, i):
        _check(load().roadsurf_step(self.handle, int(i)))

    def fetch(self, i):
        status = np.zeros(self.npoints, dtype=np.int32)
        _check(load().roadsurf_session_fetch(self.handle, int(i), status.ctypes.data_as(abi.c_int_p)))
        return status

    @property
    def done(self):
        return load().roadsurf_session_done(self.handle)

    def close(self):
        if self.handle:
            load().roadsurf_session_close(self.handle)
            self.handle = C.c_void_p(None)


def runsimulation(arrays, settings, params, point=0):
    """The reference's single-point entry, through the exact reference signature."""
    lib = load()
    ins = arrays.input_pointers()
    outs = arrays.output_pointers()
    lib.runsimulation(C.byref(outs[point]), C.byref(ins[point]), C.byref(settings), C.byref(params),
                      C.byref(arrays.local[point]))


class DeviceBatch:
    """Device-resident structure-of-arrays batch (RsDeviceBatch) backed by torch CUDA tensors.

    torch is used for device memory and streams only.  Layouts (point index fastest, `ld` padded to
    a multiple of 32): forcing [n_records, nvar, ld], local [L_NLOCAL, ld], horizons [360, ld],
    out [6, n_out, ld], status [ld]."""

    def __init__(self, npoints, sim_len, nlayers=15, n_records=None, nvar=F_NVAR, out_stride=1,
                 coarse=False, horizons=False, coupling=False, state=False, device="cuda",
                 out_start=0, extended_outputs=False, rule=1, expand_steps=0):
        import torch
        self.torch = torch
        self.npoints, self.sim_len, self.nlayers = int(npoints), int(sim_len), int(nlayers)
        self.ld = (self.npoints + 31) // 32 * 32
        self.coarse = bool(coarse)
        self.rule = int(rule)           # coarse records: 1 = example1's interpolation (in the step kernel), 2 = example2's
        self.expand_steps = int(expand_steps) if expand_steps else self.sim_len
        self.n_records = int(n_records) if coarse else self.sim_len
        self.nvar = int(nvar)
        self.out_stride = int(out_stride)
        self.out_start = int(out_start)
        self.out_nvar = O_NVAR_EXT if extended_outputs else O_NVAR
        self.coupling_window_end = 0    # set by load_local when all coupled points share one window
        self.order = None               # optional slot permutation (build_order)
        self.n_out = (self.sim_len - self.out_start + self.out_stride - 1) // self.out_stride
        f64 = dict(dtype=torch.float64, device=device)
        self.forcing = torch.zeros((self.n_records, self.nvar, self.ld), **f64)
        self.record_step = torch.zeros(self.n_records, dtype=torch.int32, device=device) if coarse else None
        self.time_fields = torch.zeros((6, self.sim_len), dtype=torch.int32, device=device)
        self.local = torch.zeros((L_NLOCAL, self.ld), **f64)
        self.local[L_SKY_VIEW].fill_(1.0)
        self.local[L_ACTIVE, :self.npoints] = 1.0
        self.local[L_COUPLING_TSURF].fill_(-9999.0)
        self.local[L_COUPLING_INDEX].fill_(-9999.0)
        self.local[L_TAIR_RELAX:L_RH_RELAX + 1].fill_(-9999.0)
        self.horizons = torch.zeros((360, self.ld), **f64) if horizons else None
        self.out = torch.empty((self.out_nvar, self.n_out, self.ld), **f64)
        self.status = torch.zeros(self.ld, dtype=torch.int32, device=device)
        self.state = torch.zeros((state_nplanes(nlayers), self.ld), **f64) if state else None
        self.scratch = torch.zeros((scratch_nplanes(nlayers), self.ld), **f64) if coupling else None
        self.counters = torch.zeros(CNT_N, dtype=torch.int64, device=device)
        self.solar = torch.zeros((self.sim_len, 4), **f64)
        self.expand_workspace = (torch.zeros((self.expand_steps, self.nvar, self.ld), **f64)
                                 if (coarse and self.rule == 2) else None)

    def descriptor(self, step_begin=0, step_end=0, forcing=None, forcing_step0=0, out=None, out_slot0=0):
        def ptr(t):
            return None if t is None else t.data_ptr()
        forcing = self.forcing if forcing is None else forcing
        out = self.out if out is None else out
        n_records = forcing.shape[0]
        return RsDeviceBatch(step_begin=step_begin, step_end=step_end, forcing_step0=forcing_step0,
                             out_slot0=out_slot0, npoints=self.npoints, ld=self.ld, sim_len=self.sim_len,
                             forcing_mode=(2 if self.rule == 2 else 1) if self.coarse else 0, n_records=n_records,
                             expand_workspace=ptr(self.expand_workspace), expand_steps=self.expand_steps,
                             nvar=self.nvar, forcing=ptr(forcing), record_step=ptr(self.record_step),
                             time_fields=ptr(self.time_fields), local=ptr(self.local),
                             horizons=ptr(self.horizons), out=ptr(out), out_stride=self.out_stride,
                             n_out=out.shape[1], status=ptr(self.status), state=ptr(self.state),
                             scratch=ptr(self.scratch), counters=ptr(self.counters), solar=ptr(self.solar),
                             out_start=self.out_start, out_nvar=self.out_nvar, order=ptr(self.order),
                             coupling_window_end=self.coupling_window_end if (step_begin, step_end) == (0, 0) else 0)

    def build_order(self, stream=None):
        """roadsurf_order_points: gather the points with sky-view radiation at one end of the launch
        (thread t then runs point order[t]); call after the statics are loaded."""
        st = stream if stream is not None else self.torch.cuda.current_stream()
        if self.order is None:
            self.order = self.torch.empty(self.ld, dtype=self.torch.int32, device=self.local.device)
        _check(load().roadsurf_order_points(C.c_void_p(self.local.data_ptr()), self.ld, self.npoints,
                                            C.c_void_p(self.order.data_ptr()), C.c_void_p(st.cuda_stream)))

    def run(self, stream=None, **chunk):
        """Asynchronous launch on `stream` (a torch.cuda.Stream; default: the current stream).
        Keyword arguments select a time chunk: step_begin, step_end, forcing (tensor holding only the
        chunk's records), forcing_step0, out (tensor holding only the chunk's slots), out_slot0."""
        st = stream if stream is not None else self.torch.cuda.current_stream()
        desc = self.descriptor(**chunk)
        _check(load().roadsurf_run_device(C.byref(desc), C.c_void_p(st.cuda_stream)))

    def expand(self, rule, step_begin, step_end, stream=None):
        """roadsurf_expand_records: the records interpolated to the steps [step_begin, step_end] as a new
        device tensor [steps, nvar, ld] (rule 1 = example1, 2 = example2)."""
        st = stream if stream is not None else self.torch.cuda.current_stream()
        dst = self.torch.empty((step_end - step_begin + 1, self.nvar, self.ld), dtype=self.torch.float64,
                               device=self.forcing.device)
        lib = load()
        lib.roadsurf_expand_records.argtypes = [C.POINTER(RsDeviceBatch), C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        desc = self.descriptor()
        _check(lib.roadsurf_expand_records(C.byref(desc), int(rule), int(step_begin), int(step_end),
                                           C.c_void_p(dst.data_ptr()), C.c_void_p(st.cuda_stream)))
        return dst

    # ---- helpers to fill the batch from host-layout data (tests, small cases) -----------------
    def load_point_arrays(self, arrays):
        """Full-resolution forcing + statics from a host-layout PointArrays (numpy side transpose;
        only used by tests and smoke, the batched C entry point has its own device pack path)."""
        torch = self.torch
        assert not self.coarse and arrays.sim_len == self.sim_len and arrays.npoints == self.npoints
        host = np.zeros((self.sim_len, self.nvar, self.ld))
        for v in range(self.nvar):
            src = getattr(arrays, F_NAMES[v])
            host[:, v, :self.npoints] = src.T
        self.forcing.copy_(torch.from_numpy(host))
        self.time_fields.copy_(torch.from_numpy(arrays.time))
        self.load_local(arrays.local, arrays.local_horizons)

    def load_local(self, local, horizons=None):
        torch = self.torch
        n = self.npoints
        L = np.zeros((L_NLOCAL, self.ld))
        L[L_SKY_VIEW] = 1.0
        L[L_COUPLING_TSURF] = L[L_COUPLING_INDEX] = -9999.0
        for p in range(n):
            lp = local[p]
            L[:, p] = (lp.tair_relax, lp.VZ_relax, lp.RH_relax, lp.couplingTsurf, lp.lat, lp.lon,
                       lp.sky_view, lp.couplingIndexI, lp.InitLenI, 1.0)
        self.local.copy_(torch.from_numpy(L))
        # one common coupling window (the usual case: one analysis time for the whole batch) lets the
        # library compact lanes between coupling iterations
        coupled = (L[L_COUPLING_TSURF, :n] >= -100) & (L[L_COUPLING_INDEX, :n] >= 1)
        ends = np.unique(L[L_COUPLING_INDEX, :n][coupled])
        self.coupling_window_end = int(ends[0]) if (ends.size == 1 and self.state is not None) else 0
        if self.horizons is not None and horizons is not None:
            H = np.zeros((360, self.ld))
            H[:, :n] = np.asarray(horizons).T
            self.horizons.copy_(torch.from_numpy(H))

    def load_records(self, rec):
        """Coarse forcing records (synth.Records) + statics."""
        torch = self.torch
        assert self.coarse and rec.nrec == self.n_records
        host = np.zeros((self.n_records, self.nvar, self.ld))
        names = ("tair", "tdew", "VZ", "Rhz", "prec", "SW", "LW", "SW_dir", "LW_net", "TSurfObs", "PrecPhase")
        for v, name in enumerate(names):
            host[:, v, :self.npoints] = getattr(rec, name).T
        if self.nvar > F_NVAR:
            host[:, F_NVAR, :] = -9999.9
        self.forcing.copy_(torch.from_numpy(host))
        self.record_step.copy_(torch.from_numpy(rec.record_step.astype(np.int32)))

    def outputs(self):
        """dict name -> numpy [npoints, n_out]."""
        o = self.out.cpu().numpy()
        names = O_NAMES + (O_NAMES_EXT if self.out_nvar == O_NVAR_EXT else ())
        return {name: np.ascontiguousarray(o[v, :, :self.npoints].T) for v, name in enumerate(names)}


def set_model(settings, params):
    _check(load().roadsurf_set_model(C.byref(settings), C.byref(params)))


def measure_fp64_tflops(iterations=20000):
    v = load().roadsurf_measure_fp64_tflops(int(iterations))
    if v < 0:
        raise RoadSurfError(load().roadsurf_last_error().decode())
    return v


def selftest_arith(n=200_000_000, seed=12345):
    """(pairs tested, [rcp, div, div_const] mismatch counts) of the arithmetic self-test."""
    bad = (C.c_longlong * 3)()
    tested = load().roadsurf_selftest_arith(int(n), int(seed), bad)
    if tested < 0:
        raise RoadSurfError(load().roadsurf_last_error().decode())
    return int(tested), [int(b) for b in bad]


def runsimulation_counters():
    """(calls served, batches they were combined into) of runsimulation since the library was loaded."""
    a, b = C.c_longlong(0), C.c_longlong(0)
    load().roadsurf_runsimulation_counters(C.byref(a), C.byref(b))
    return a.value, b.value


def selftest_libm(n=2_000_000, seed=7):
    """Host-only: [exp, log] mismatch counts of the library's libm-exact exp/log against this process's libm."""
    bad = (C.c_longlong * 2)()
    load().roadsurf_selftest_libm(int(n), int(seed), bad)
    return [int(b) for b in bad]


def sun_position(time_fields, lat, lon):
    """roadsurf_sun_position on torch CUDA tensors: time_fields [6, n] int32, lat / lon [npoints] f64 ->
    (elevation, azimuth) [n, npoints]."""
    import torch
    n, npts = time_fields.shape[1], lat.shape[0]
    elev = torch.empty((n, npts), dtype=torch.float64, device=lat.device)
    azim = torch.empty_like(elev)
    lib = load()
    lib.roadsurf_sun_position.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                          C.c_void_p]
    _check(lib.roadsurf_sun_position(time_fields.data_ptr(), n, lat.data_ptr(), lon.data_ptr(), npts, elev.data_ptr(),
                                     azim.data_ptr(), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return elev, azim


def eval_primitive(fn, a, b=None):
    """roadsurf_eval_primitive: one of the step kernel's math primitives (PRIM_*) elementwise on float64 torch
    CUDA tensors a (and b for PRIM_FRCP / _FDIV / _DIV_CONST, same shape).  Returns the result tensor
    (synchronised)."""
    import torch
    a = a.contiguous()
    if b is not None:
        b = b.contiguous()
        assert b.shape == a.shape and b.dtype == torch.float64
    assert a.dtype == torch.float64 and a.is_cuda
    out = torch.empty_like(a)
    _check(load().roadsurf_eval_primitive(int(fn), a.data_ptr(), None if b is None else b.data_ptr(), out.data_ptr(),
                                          a.numel(), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    return out


def set_option(name, value):
    _check(load().roadsurf_set_option(name.encode(), int(value)))


def read_input_derive(arrays, settings, forecast_step, latest_obs_index=None):
    """roadsurf_read_input_derive over a PointArrays (host only; fills arrays.local, blanks TSurfObs over
    the coupling window).  Returns ok[npoints]."""
    ins = arrays.input_pointers()
    in_ptrs = abi.pointer_arrays(ins, abi.InputPointers)
    loc_ptrs = abi.pointer_arrays(arrays.local, abi.LocalParameters)
    ok = np.zeros(arrays.npoints, dtype=np.int32)
    lat = None
    if latest_obs_index is not None:
        lat = np.ascontiguousarray(latest_obs_index, dtype=np.int32)
    _check(load().roadsurf_read_input_derive(arrays.npoints, in_ptrs, C.byref(settings), int(forecast_step),
                                             None if lat is None else lat.ctypes.data_as(abi.c_int_p), loc_ptrs,
                                             ok.ctypes.data_as(abi.c_int_p)))
    return ok


def read_input_derive_records(forcing, record_step, settings, forecast_step, local, latest_obs_index=None):
    """roadsurf_read_input_derive_records: forcing [n_records, nvar, npoints] f64 and record_step
    [n_records] i32 on the host (numpy or CPU tensors); fills the derived planes of local
    [L_NLOCAL, npoints] in place.  Returns the common coupling window end (0 if none / not common)."""
    def ptr(x):
        return x.data_ptr() if hasattr(x, "data_ptr") else x.ctypes.data
    n_records, nvar, npoints = forcing.shape
    assert tuple(local.shape) == (L_NLOCAL, npoints)
    hb = RsHostBatch(npoints=npoints, sim_len=settings.SimLen, forcing_mode=1, n_records=n_records, nvar=nvar,
                     out_stride=1, forcing=ptr(forcing), record_step=ptr(record_step))
    lat = None if latest_obs_index is None else np.ascontiguousarray(latest_obs_index, dtype=np.int32)
    wend = C.c_int(0)
    _check(load().roadsurf_read_input_derive_records(C.byref(hb), C.byref(settings), int(forecast_step),
                                                     None if lat is None else lat.ctypes.data_as(abi.c_int_p),
                                                     C.c_void_p(ptr(local)), C.byref(wend)))
    return wend.value


def release_workspace():
    load().roadsurf_release_workspace()


# ---- ensemble runs (include/roadsurf_b200.h, part 3) ---------------------------------------------------

def _ptr(x):
    if x is None:
        return None
    return x.data_ptr() if hasattr(x, "data_ptr") else x.ctypes.data


def ensemble_stats(member_out, npoints, members, spec, stream=None):
    """roadsurf_ensemble_stats on a torch CUDA tensor member_out [out_nvar, n_out, ld_members] (lane
    p * members + m).  Returns (stats [5 + n_quantiles, out_nvar, n_out, npoints],
    prob [n_thresholds + n_events, n_out, npoints]) as CUDA tensors (synchronised)."""
    import torch
    out_nvar, n_out, ldm = member_out.shape
    ld = max(32, (npoints + 31) // 32 * 32)
    f64 = dict(dtype=torch.float64, device=member_out.device)
    stats = torch.full((ENS_NFIXED + spec.n_quantiles, out_nvar, n_out, ld), 12345.0, **f64)
    prob = torch.full((max(1, spec.n_prob), n_out, ld), 12345.0, **f64)
    st = stream if stream is not None else torch.cuda.current_stream()
    _check(load().roadsurf_ensemble_stats(member_out.data_ptr(), out_nvar, n_out, ldm, int(npoints), int(members),
                                          C.byref(spec), stats.data_ptr(), prob.data_ptr(), ld,
                                          C.c_void_p(st.cuda_stream)))
    torch.cuda.synchronize()
    return stats[..., :npoints], prob[:spec.n_prob, :, :npoints]


def ensemble_area_events(member_out, npoints, members, spec, areas, stream=None):
    """roadsurf_ensemble_area_events on a torch CUDA tensor member_out [out_nvar, n_out, ld_members] (lane
    p * members + m); areas is an RsEnsembleAreas (ensemble_areas).  Returns area_prob
    [n_events, n_out, n_areas] as a CUDA tensor (synchronised)."""
    import torch
    out_nvar, n_out, ldm = member_out.shape
    area_prob = torch.full((spec.n_events, n_out, areas.n_areas), 12345.0, dtype=torch.float64,
                           device=member_out.device)
    st = stream if stream is not None else torch.cuda.current_stream()
    _check(load().roadsurf_ensemble_area_events(member_out.data_ptr(), out_nvar, n_out, ldm, int(npoints),
                                                int(members), C.byref(spec), C.byref(areas), area_prob.data_ptr(),
                                                C.c_void_p(st.cuda_stream)))
    torch.cuda.synchronize()
    return area_prob


def ensemble_onset(member_out, npoints, members, spec, areas=None, onset=True, stream=None):
    """roadsurf_ensemble_onset on a torch CUDA tensor member_out [out_nvar, n_out, ld_members] (lane
    p * members + m); areas is an RsEnsembleAreas (ensemble_areas) or None.  Returns (onset [n_events, n_out, npoints]
    or None when onset=False, area_onset [n_events, n_out, n_areas] or None without areas) as CUDA tensors
    (synchronised)."""
    import torch
    out_nvar, n_out, ldm = member_out.shape
    ld = max(32, (npoints + 31) // 32 * 32)
    f64 = dict(dtype=torch.float64, device=member_out.device)
    on = torch.full((spec.n_events, n_out, ld), 12345.0, **f64) if onset else None
    area_on = torch.full((spec.n_events, n_out, areas.n_areas), 12345.0, **f64) if areas is not None else None
    st = stream if stream is not None else torch.cuda.current_stream()
    _check(load().roadsurf_ensemble_onset(member_out.data_ptr(), out_nvar, n_out, ldm, int(npoints), int(members),
                                          C.byref(spec), None if on is None else on.data_ptr(), ld,
                                          None if areas is None else C.byref(areas),
                                          None if area_on is None else area_on.data_ptr(), C.c_void_p(st.cuda_stream)))
    torch.cuda.synchronize()
    return (None if on is None else on[..., :npoints]), area_on


def ensemble_extremes_device(member_out, npoints, members, spec, ext, areas=None, stream=None):
    """roadsurf_ensemble_extremes on a torch CUDA tensor member_out [out_nvar, n_out, ld_members] (lane
    p * members + m); ext an RsEnsembleExtremes (ensemble_extremes), areas an RsEnsembleAreas (ensemble_areas) or None.
    Returns (ext_stats [5 + n_quantiles, n_extremes, n_out, npoints], area_ext_stats
    [5 + n_quantiles, n_extremes, n_out, n_areas] or None without areas) as CUDA tensors (synchronised)."""
    import torch
    out_nvar, n_out, ldm = member_out.shape
    ld = max(32, (npoints + 31) // 32 * 32)
    f64 = dict(dtype=torch.float64, device=member_out.device)
    rows = (ENS_NFIXED + spec.n_quantiles, ext.n_extremes, n_out)
    xs = torch.full(rows + (ld,), 12345.0, **f64)
    area_xs = torch.full(rows + (areas.n_areas,), 12345.0, **f64) if areas is not None else None
    st = stream if stream is not None else torch.cuda.current_stream()
    _check(load().roadsurf_ensemble_extremes(member_out.data_ptr(), out_nvar, n_out, ldm, int(npoints), int(members),
                                             C.byref(spec), C.byref(ext), xs.data_ptr(), ld,
                                             None if areas is None else C.byref(areas),
                                             None if area_xs is None else area_xs.data_ptr(),
                                             C.c_void_p(st.cuda_stream)))
    torch.cuda.synchronize()
    return xs[..., :npoints], area_xs


def fork_record(record_step, fork_step):
    """r_f: the last record at or before 0-based step fork_step - 1."""
    rs = np.asarray(record_step)
    return int(np.nonzero(rs <= fork_step - 1)[0][-1])


class EnsembleBatch:
    """Device-resident ensemble (RsEnsembleBatch): a shared DeviceBatch of the P stations (it needs
    state=True, and coupling=True when the model couples) plus the member tensors of P * M lanes,
    station-major (lane p * M + m).  Fill `shared` as usual (records / full-resolution forcing, time axis,
    statics), then the members' forcing with load_member_records / load_member_forcing, and run()."""

    def __init__(self, shared, members, fork_step, stats_spec=None, member_relax=False, extra_slots=0):
        import torch
        self.torch = torch
        self.shared = shared
        self.members, self.fork_step = int(members), int(fork_step)
        P, M = shared.npoints, self.members
        self.ld_members = max(32, (P * M + 31) // 32 * 32)
        ldm, dev = self.ld_members, shared.local.device
        f64 = dict(dtype=torch.float64, device=dev)
        if shared.coarse:
            rs = shared.record_step.cpu().numpy()
            self.r_f = fork_record(rs, self.fork_step)
            n_rec_m = shared.n_records - self.r_f
        else:
            self.r_f = None
            n_rec_m = shared.sim_len - self.fork_step + 1
        self.member_forcing = torch.zeros((n_rec_m, shared.nvar, ldm), **f64)
        self.member_relax = torch.full((3, ldm), -9999.0, **f64) if member_relax else None
        self.member_local = torch.zeros((L_NLOCAL, ldm), **f64)
        self.member_horizons = torch.zeros((360, ldm), **f64) if shared.horizons is not None else None
        self.member_state = torch.zeros((state_nplanes(shared.nlayers), ldm), **f64)
        self.member_scratch = (torch.zeros((scratch_nplanes(shared.nlayers), ldm), **f64)
                               if shared.scratch is not None else None)
        self.member_status = torch.zeros(ldm, dtype=torch.int32, device=dev)
        # output slots: the steps before F in shared.out, the steps [F, sim_len] in member_out
        k0 = self.fork_step - 1 - shared.out_start
        self.slot0 = (k0 + shared.out_stride - 1) // shared.out_stride if k0 > 0 else 0
        self.n_slots = max(1, shared.n_out - self.slot0)      # output slots of the steps [F, sim_len]
        self.n_out_members = self.n_slots + int(extra_slots)  # slot dimension of member_out / stats / prob
        self.member_out = torch.empty((shared.out_nvar, self.n_out_members, ldm), **f64)
        self.member_order = None
        self.spec = stats_spec if stats_spec is not None else RsEnsembleStatsSpec()
        ld = shared.ld
        self.stats_t = torch.empty((ENS_NFIXED + self.spec.n_quantiles, shared.out_nvar, self.n_out_members, ld), **f64)
        self.prob_t = torch.empty((max(1, self.spec.n_prob), self.n_out_members, ld), **f64)

    def load_member_records(self, member_recs):
        """Coarse records of every member (synth.Records with the full record axis, one per member, equal
        to the station records up to r_f): records r_f + 1 ... go into the member tensor (slot 0 is
        written by the library)."""
        P, M = self.shared.npoints, self.members
        assert self.shared.coarse and len(member_recs) == M
        names = ("tair", "tdew", "VZ", "Rhz", "prec", "SW", "LW", "SW_dir", "LW_net", "TSurfObs", "PrecPhase")
        host = np.zeros(tuple(self.member_forcing.shape))
        for m, rec in enumerate(member_recs):
            for v, name in enumerate(names):
                host[1:, v, m:P * M:M] = getattr(rec, name)[:, self.r_f + 1:].T
        if self.shared.nvar > F_NVAR:
            host[:, F_NVAR, :] = -9999.9
        self.member_forcing.copy_(self.torch.from_numpy(host))

    def load_member_forcing(self, lane_arrays):
        """Full-resolution member forcing: steps F ... of a PointArrays whose point p * M + m is member m of
        station p (abi.PointArrays with P * M points)."""
        P, M, F = self.shared.npoints, self.members, self.fork_step
        assert not self.shared.coarse and lane_arrays.npoints == P * M
        host = np.zeros(tuple(self.member_forcing.shape))
        for v in range(self.shared.nvar):
            host[:, v, :P * M] = getattr(lane_arrays, F_NAMES[v])[:, F - 1:].T
        self.member_forcing.copy_(self.torch.from_numpy(host))

    def set_member_relax(self, relax):
        """relax [3, P * M]: tair, VZ, RH relaxation targets per member lane."""
        assert self.member_relax is not None
        self.member_relax[:, :relax.shape[1]] = self.torch.as_tensor(np.asarray(relax, dtype=np.float64))

    def build_member_order(self, stream=None):
        """roadsurf_order_points over the member statics (needs a first run for member_local)."""
        st = stream if stream is not None else self.torch.cuda.current_stream()
        self.member_order = self.torch.empty(self.ld_members, dtype=self.torch.int32, device=self.member_local.device)
        _check(load().roadsurf_order_points(C.c_void_p(self.member_local.data_ptr()), self.ld_members,
                                            self.shared.npoints * self.members,
                                            C.c_void_p(self.member_order.data_ptr()), C.c_void_p(st.cuda_stream)))

    def descriptor(self, stats=True):
        s = self.shared
        sd = s.descriptor()
        sd.coupling_window_end = s.coupling_window_end
        return RsEnsembleBatch(shared=sd, members=self.members, fork_step=self.fork_step,
                               ld_members=self.ld_members, member_forcing=_ptr(self.member_forcing),
                               member_relax=_ptr(self.member_relax), member_local=_ptr(self.member_local),
                               member_horizons=_ptr(self.member_horizons), member_state=_ptr(self.member_state),
                               member_scratch=_ptr(self.member_scratch), member_status=_ptr(self.member_status),
                               member_out=_ptr(self.member_out), n_out_members=self.n_out_members,
                               member_order=_ptr(self.member_order), spec=self.spec,
                               stats=_ptr(self.stats_t) if stats else None,
                               prob=_ptr(self.prob_t) if (stats and self.spec.n_prob) else None)

    def run(self, stream=None, stats=True):
        """Asynchronous: prefix, fork, members, statistics on `stream` (default: the current stream)."""
        st = stream if stream is not None else self.torch.cuda.current_stream()
        desc = self.descriptor(stats)
        _check(load().roadsurf_run_ensemble_device(C.byref(desc), C.c_void_p(st.cuda_stream)))

    def member_outputs(self):
        """dict name -> numpy [P, M, n_out_members] of the member slots."""
        P, M = self.shared.npoints, self.members
        o = self.member_out.cpu().numpy()[:, :self.n_slots, :P * M]
        names = O_NAMES + (O_NAMES_EXT if self.shared.out_nvar == O_NVAR_EXT else ())
        return {name: np.ascontiguousarray(o[v].T.reshape(P, M, -1)) for v, name in enumerate(names)}

    def stats(self):
        """(stats [5 + n_quantiles, out_nvar, n_slots, P], prob [n_thresholds + n_events, n_slots, P]) numpy: the slots
        of the steps [F, sim_len]."""
        P, n = self.shared.npoints, self.n_slots
        return (self.stats_t.cpu().numpy()[:, :, :n, :P],
                self.prob_t.cpu().numpy()[:self.spec.n_prob, :n, :P])


def run_ensemble_host_soa(settings, params, forcing, record_step, time_fields, local, member_records, members,
                          fork_step, spec, horizons=None, out_stride=1, coupling_window_end=0, out=None,
                          member_out=False, member_status=False, latest_obs_index=None, areas=None, prob=True,
                          onset=False, area_prob=True, extremes=None, stats=True):
    """roadsurf_run_ensemble_host_soa_extremes on host arrays: forcing [n_records, nvar, P], record_step [n_records],
    local [L_NLOCAL, P], member_records [n_records - r_f - 1, nvar, P * members], latest_obs_index [P] int32 (the
    relaxation rule of read_input_derive_records; None = no observations), areas an RsEnsembleAreas (ensemble_areas)
    or None.  Returns a dict with stats [5 + nq, 6, n_out_m, P], prob [nt + n_events, n_out_m, P] (unless prob=False:
    NULL is passed) and, when asked for, member_out [6, n_out_m, P * M], member_status [P * M] and area_prob
    [n_events, n_out_m, n_areas] (unless area_prob=False: NULL is passed).  With onset=True it also returns
    onset [n_events, n_out_m, P] and, with areas, area_onset [n_events, n_out_m, n_areas].  With extremes (an
    RsEnsembleExtremes, ensemble_extremes) it also returns ext_stats [5 + nq, n_extremes, n_out_m, P] and, with areas,
    area_ext_stats [5 + nq, n_extremes, n_out_m, n_areas].  stats=False passes NULL for stats."""
    n_records, nvar, npoints = forcing.shape
    sim_len = time_fields.shape[1]
    k0 = fork_step - 1
    slot0 = (k0 + out_stride - 1) // out_stride
    n_m = (sim_len + out_stride - 1) // out_stride - slot0
    res = {}
    if stats:
        res["stats"] = np.zeros((ENS_NFIXED + spec.n_quantiles, O_NVAR, n_m, npoints))
    if prob:
        res["prob"] = np.zeros((spec.n_prob, n_m, npoints))
    if member_out:
        res["member_out"] = np.zeros((O_NVAR, n_m, npoints * members))
    if member_status:
        res["member_status"] = np.zeros(npoints * members, dtype=np.int32)
    if areas is not None and area_prob:
        res["area_prob"] = np.zeros((spec.n_events, n_m, areas.n_areas))
    if onset:
        res["onset"] = np.zeros((spec.n_events, n_m, npoints))
        if areas is not None:
            res["area_onset"] = np.zeros((spec.n_events, n_m, areas.n_areas))
    if extremes is not None:
        res["ext_stats"] = np.zeros((ENS_NFIXED + spec.n_quantiles, extremes.n_extremes, n_m, npoints))
        if areas is not None:
            res["area_ext_stats"] = np.zeros((ENS_NFIXED + spec.n_quantiles, extremes.n_extremes, n_m, areas.n_areas))
    hb = RsHostBatch(npoints=npoints, sim_len=sim_len, forcing_mode=1, n_records=n_records, nvar=nvar,
                     out_stride=out_stride, forcing=_ptr(forcing), record_step=_ptr(record_step),
                     time_fields=_ptr(time_fields), local=_ptr(local), horizons=_ptr(horizons), out=_ptr(out),
                     coupling_window_end=int(coupling_window_end))
    lat = None if latest_obs_index is None else np.ascontiguousarray(latest_obs_index, dtype=np.int32)
    _check(load().roadsurf_run_ensemble_host_soa_extremes(
        C.byref(hb), _ptr(member_records), int(members), int(fork_step), _ptr(lat), C.byref(spec),
        _ptr(res.get("stats")), _ptr(res.get("prob")), _ptr(res.get("member_out")), _ptr(res.get("member_status")),
        None if areas is None else C.byref(areas), _ptr(res.get("area_prob")), _ptr(res.get("onset")),
        _ptr(res.get("area_onset")), None if extremes is None else C.byref(extremes), _ptr(res.get("ext_stats")),
        _ptr(res.get("area_ext_stats")), C.byref(settings), C.byref(params)))
    return res
