/*
 * roadsurf_b200.h -- C ABI of the B200-native RoadSurf per-point simulation loop.
 *
 * This header is the drop-in boundary.  Part 1 restates the five Bind(C) interop types of the
 * reference library and its single C entry point `runsimulation`; a C++ (or Fortran
 * ISO_C_BINDING) main program that was linked against the reference keeps compiling and running
 * when linked against libroadsurf_b200.so instead.  Part 2 adds the batched and the
 * device-resident entry points that make a GPU behind that boundary worthwhile.
 *
 * Reference interfaces replaced (paths relative to the fmidev/RoadSurf tree):
 *   InputPointers    src/InputPointers.f90.inc:4-27      examples/example1/src/InputPointers.h:7-30
 *   OutputPointers   src/OutputPointers.f90.inc:4-17     examples/example1/src/OutputPointers.h
 *   InputSettings    src/InputSettings.f90.inc:4-18      examples/example1/src/InputSettings.h:9-27
 *   InputParameters  src/InputParameters.f90.inc:4-91    examples/example1/src/InputParameters.h:11-110
 *   LocalParameters  src/LocalParameters.f90.inc:4-15    examples/example1/src/LocalParameters.h:11-30
 *   runsimulation    examples/example1/src/Simulation.f90:4-6 (BIND(C), lower-case symbol)
 *                    examples/example1/src/roadrunner.cpp:22-29 (C++ declaration)
 *
 * No torch / CUDA types appear in any signature: plain pointers, ints and doubles only.
 */
#ifndef ROADSURF_B200_H
#define ROADSURF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------ */
/* Part 1: the reference ABI                                                                   */
/* ------------------------------------------------------------------------------------------ */

/* src/InputPointers.f90.inc:4-27.  160 bytes on x86-64 SysV.  Every array has inputLen
 * elements except local_horizons, which always has 360 (src/ConnectFortran2Carrays.f90:52).
 * The callee mutates VZ[0], SW_dir[i], and (sky view active) SW[i], SW_dir[i], LW[i] in the
 * reference; see INTEGRATION.md for what this library does instead. */
typedef struct InputPointers
{
  int inputLen;
  double* c_tair;           /* air temperature (C) */
  double* c_tdew;           /* dew point temperature (C) */
  double* c_VZ;             /* wind speed (m/s) */
  double* c_Rhz;            /* relative humidity (%) */
  double* c_prec;           /* precipitation (mm/h) */
  double* c_SW;             /* incoming short wave radiation (W/m2) */
  double* c_LW;             /* incoming long wave radiation (W/m2) */
  double* c_SW_dir;         /* direct short wave radiation (W/m2) */
  double* c_LW_net;         /* net long wave radiation (W/m2) */
  double* c_TSurfObs;       /* observed surface temperature (C) */
  int* c_PrecPhase;         /* precipitation phase code 0..6, -9999 = interpret */
  double* c_local_horizons; /* 360 local horizon angles (deg) */
  double* c_Depth;          /* per-step output depth (m), < 0 = mean of layers 1,2 */
  int* c_year;
  int* c_month;
  int* c_day;
  int* c_hour;
  int* c_minute;
  int* c_second;
} InputPointers;

/* src/OutputPointers.f90.inc:4-17.  56 bytes.  Element i-1 receives step i; -9999.0 marks a
 * step that was not computed (src/Initialization.f90:397-412). */
typedef struct OutputPointers
{
  int outputLen;
  double* c_TsurfOut;
  double* c_SnowOut;
  double* c_WaterOut;
  double* c_IceOut;
  double* c_DepositOut;
  double* c_Ice2Out;
} OutputPointers;

/* src/InputSettings.f90.inc:4-18.  56 bytes.  The Fortran type has force_tsurf at offset 12;
 * the reference's C++ struct has no such member, so a C++ caller leaves those four bytes as
 * padding.  This library reads offset 12 exactly as the Fortran does (true iff == 1). */
typedef struct InputSettings
{
  int SimLen;
  int use_coupling;
  int use_relaxation;
  int force_tsurf;
  double DTSecs;
  double tsurfOutputDepth;
  int NLayers;
  int coupling_minutes;
  double couplingEffectReduction;
  int outputStep;
} InputSettings;

/* src/InputParameters.f90.inc:4-91.  69 doubles, 552 bytes. */
typedef struct InputParameters
{
  double NightOn, NightOff, CalmLimDay, CalmLimNgt, TrfFricNgt, TrFfricDay;
  double Grav, SB_Const, VK_Const, LVap, LFus, WatDens, SnowDens, IceDens, DepDens, WatMHeat,
      PorEvaF;
  double ZRefW, ZRefT, ZeroDisp, ZMom, ZHeat, Emiss, Albedo, Albedo_surroundings, MaxPormms,
      TClimG, DampDpth, Omega, AZ, DampWearF, AlbDry, AlbSnow, vsh1, vsh2, Poro1, Poro2, RhoB1,
      RhoB2, Silt1, Silt2;
  double freezing_limit_normal, snow_melting_limit_normal, ice_melting_limit_normal,
      frost_melting_limit_normal, frost_formation_limit_normal, T4Melt_normal;
  double TLimColdH, TLimColdL, WetSnowFormR, WetSnowMeltR;
  double PLimSnow, PLimRain, MaxSnowmms, MaxDepmms, MaxIcemms, MaxExtmms;
  double MissValI, MissValR;
  double Snow2IceFac;
  double MinPrecmm, MinWatmms, MinSnowmms, MaxWatmms, WDampLim, WWetLim, WWearLim, MinDepmms,
      MinIcemms;
} InputParameters;

/* src/LocalParameters.f90.inc:4-15.  72 bytes.  couplingIndexI and InitLenI are consumed as
 * 1-based step indices (src/InputOutput.f90:29, src/Initialization.f90:452). */
typedef struct LocalParameters
{
  double tair_relax;
  double VZ_relax;
  double RH_relax;
  int couplingIndexI;
  double couplingTsurf;
  double lat;
  double lon;
  double sky_view;
  int InitLenI;
} LocalParameters;

/* The reference entry point, unchanged (examples/example1/src/Simulation.f90:4-6).  Runs ONE
 * point; kept for unchanged main programs.  It round-trips host<->device per call and is
 * therefore a correctness drop-in, not the fast path: use roadsurf_run_batch.  Calls made
 * concurrently from several host threads (the reference's mains use a thread pool,
 * examples/example1/src/roadrunner.cpp:454-496) are combined into batches internally. */
void runsimulation(OutputPointers* outPointers, const InputPointers* inPointers,
                   const InputSettings* inSettings, const InputParameters* inputParam,
                   const LocalParameters* localParam);

/* ------------------------------------------------------------------------------------------ */
/* Part 2: batched and device-resident entry points                                            */
/* ------------------------------------------------------------------------------------------ */

/* Per-point status word (bit set).  The reference only prints to stdout for these events. */
enum
{
  RS_ST_FAILED = 1,           /* simulation_failed (src/InputOutput.f90:66,72,81) */
  RS_ST_BAD_INPUT = 2,        /*   ... because of an input range check */
  RS_ST_ABNORMAL_TSURF = 4,   /*   ... because |TsurfAve| > 100 */
  RS_ST_COUPLING_USED = 8,    /* coupling was active for this point */
  RS_ST_COUPLING_FAILED = 16, /* Coupling_failed at the end (src/Coupling.f90:324-360,400,451) */
  RS_ST_BL_NOT_CONVERGED = 32,/* BLCond iteration hit MaxIter (src/BoundaryLayer.f90:98-101) */
  RS_ST_SOLAR_GEOMETRY = 64,  /* the reference would `stop` (src/SunPosition.f90:144-146,176-178) */
  RS_ST_BAD_WINDOW = 128,     /* device SoA entry: coupling windows differ inside one warp */
  RS_ST_NOT_RUN = 256,        /* point was skipped (bad settings) */
  RS_ST_BAD_FORK = 512        /* ensemble member: its relaxation targets differ from the ones the shared
                                 analysis already used (see roadsurf_run_ensemble_device); with RS_ST_NOT_RUN */
};

/* Return codes. */
enum
{
  RS_OK = 0,
  RS_ERR_NO_DEVICE = -1,
  RS_ERR_BAD_ARGUMENT = -2,
  RS_ERR_CUDA = -3,
  RS_ERR_UNSUPPORTED = -4
};

/* The examples' default model parameters and settings (examples/example1/src/InputParameters.h:18-110
 * with the DTSecs-dependent values of InputParameters.cpp:11-22; InputSettings.h:13-23), for callers
 * that do not read a configuration file.  roadsurf_default_settings zeroes the whole struct first
 * (also the force_tsurf bytes that the C++ examples leave uninitialised). */
void roadsurf_default_parameters(InputParameters* params, double DTSecs);
void roadsurf_default_settings(InputSettings* settings, int SimLen, double DTSecs);

/* Text of the last error on the calling thread ("" if none). */
const char* roadsurf_last_error(void);

/* Number of visible CUDA devices (0 if none); never fails. */
int roadsurf_device_count(void);

/* Batched form of runsimulation over `npoints` independent points with shared settings and
 * parameters (what run_locations_async does point by point,
 * examples/example1/src/roadrunner.cpp:423-501).  Host array-of-pointers in, same arrays out.
 * Points are split into contiguous shards over `ngpus` devices (<= 0: all visible devices).
 * `status` (may be NULL) receives one status word per point.  Returns RS_OK or an error code;
 * never falls back to the CPU. */
int roadsurf_run_batch(int npoints, OutputPointers* const* out, const InputPointers* const* in,
                       const InputSettings* settings, const InputParameters* params,
                       const LocalParameters* const* local, int ngpus, int* status);

/* Host-side preparation of a batch: what the example's read_input derives per point before it calls
 * runsimulation (examples/example1/src/roadrunner.cpp:157-278).  For every point p:
 *   - screens the required inputs (tair, Rhz, prec, SW, LW, VZ: NaN or < -9000 at any step) ->
 *     ok[p] = 0 and the point is left untouched (read_input returns success = false);
 *   - InitLenI = 1 + forecast_step; with use_relaxation == 1 and latest_obs_index[p] > -1
 *     (GetLatestObsIndex, JsonSource.cpp:397-414): InitLenI = that index and the relaxation targets
 *     are the inputs at that (0-based) index, else the targets are -9999.9;
 *   - with use_coupling == 1: the latest valid TSurfObs index i (not NaN, >= -100); if
 *     i >= coupling_minutes*60/DTSecs: couplingTsurf = TSurfObs[i], couplingIndexI = i and
 *     TSurfObs is blanked to -9999.9 over (i - span, i] IN THE CALLER'S ARRAY, as read_input does.
 * example2's read_input (examples/example2/src/roadrunner.cpp:139-264) is the same function with one
 * difference in the relaxation block: from the time of the latest air-temperature observation it sets
 * InitLenI = secs/DTSecs + 1 and takes the targets at the 0-based index InitLenI (:223-231) -- pass
 * latest_obs_index[p] = secs/DTSecs + 1 and the two coincide (tests/test_host_logic.py).
 * latest_obs_index and ok may be NULL.  Pure host code: works without a GPU.  Returns RS_OK. */
int roadsurf_read_input_derive(int npoints, const InputPointers* const* in, const InputSettings* settings,
                               int forecast_step, const int* latest_obs_index, LocalParameters* const* local,
                               int* ok);

/* Statistics of the most recent roadsurf_run_batch on this thread. */
typedef struct RsBatchStats
{
  double pack_ms;        /* host AoS -> pinned SoA */
  double h2d_ms;         /* host -> device copies (event timed) */
  double kernel_ms;      /* step kernel(s) */
  double d2h_ms;         /* device -> host copies */
  double unpack_ms;      /* pinned SoA -> caller's arrays */
  int64_t h2d_bytes;
  int64_t d2h_bytes;
  int64_t executed_steps; /* point-steps actually executed, including coupling re-runs */
  int kernel_launches;
  int groups;            /* (time axis, coupling window) groups the batch was split into */
  double wall_ms;        /* host wall-clock time spent inside the call */
  double setup_ms;       /* of which: grouping, depth scan, device/pinned allocations */
} RsBatchStats;
void roadsurf_last_batch_stats(RsBatchStats* stats);

/* ---- device-resident structure-of-arrays entry ------------------------------------------- */

/* Planes of the forcing tensor, in order.  All fp64; PrecPhase is stored as an exact double. */
enum
{
  RS_F_TAIR = 0,
  RS_F_TDEW,
  RS_F_VZ,
  RS_F_RHZ,
  RS_F_PREC,
  RS_F_SW,
  RS_F_LW,
  RS_F_SWDIR,
  RS_F_LWNET,
  RS_F_TSURFOBS,
  RS_F_PHASE,
  RS_F_NVAR = 11,
  RS_F_DEPTH = 11,      /* optional 12th plane */
  RS_F_NVAR_DEPTH = 12
};

/* Planes of the per-point static tensor. */
enum
{
  RS_L_TAIR_RELAX = 0,
  RS_L_VZ_RELAX,
  RS_L_RH_RELAX,
  RS_L_COUPLING_TSURF,
  RS_L_LAT,
  RS_L_LON,
  RS_L_SKY_VIEW,
  RS_L_COUPLING_INDEX,  /* exact integer stored as double */
  RS_L_INIT_LEN,        /* exact integer stored as double */
  RS_L_ACTIVE,          /* 1.0 = a real point, 0.0 = padding slot (never run) */
  RS_L_NLOCAL = 10
};

/* Output planes. */
enum
{
  RS_O_TSURF = 0,
  RS_O_SNOW,
  RS_O_WATER,
  RS_O_ICE,
  RS_O_DEPOSIT,
  RS_O_ICE2,
  RS_O_NVAR = 6,
  /* Extended set (RsDeviceBatch.out_nvar == RS_O_NVAR_EXT): what example2 stores per output time
   * besides the six model outputs (examples/example2/src/QueryDataTools.cpp:325-341): the air and
   * dew point temperature INPUTS at that step and the dew point deficit Tsurf - Tdew
   * (calc_difference, :285-296: -9999 when either operand is NaN or <= -9000). */
  RS_O_TAIR = 6,
  RS_O_TDEW,
  RS_O_DEWDEFICIT,
  RS_O_NVAR_EXT = 9
};

/* Everything a launch needs, as DEVICE pointers (on the current device).  `ld` is the padded
 * point count: a multiple of 32, >= npoints; all planes have `ld` as their fastest dimension so
 * that a warp touches one contiguous 256-byte segment per plane. */
typedef struct RsDeviceBatch
{
  int npoints;
  int ld;
  int sim_len;          /* SimLen: number of model steps */
  int forcing_mode;     /* 0: one forcing record per model step.  1: coarse records, linear
                           interpolation in time inside the step kernel (example1's rule,
                           JsonSource.cpp:49-176).  2: coarse records interpolated by example2's rule
                           (AsciiSource.cpp:223-281: per variable the nearest valid records, at most
                           180 minutes apart, whole-minute weights) by an expansion pass into
                           `expand_workspace`, chunk by chunk, ahead of the step kernel. */
  int n_records;        /* forcing_mode 0: == sim_len.  1: number of coarse records */
  int nvar;             /* RS_F_NVAR or RS_F_NVAR_DEPTH */
  const double* forcing;      /* [n_records][nvar][ld] */
  const int* record_step;     /* forcing_mode 1 / 2: 0-based model step index of every record,
                                 strictly increasing; forcing_mode 1 also needs record_step[0] <= 0
                                 (example1's rule is implemented for grids that start at or before
                                 step 0).  A precondition here: this is device memory and the
                                 asynchronous entry does not read it back to check it.  The host
                                 entries check their copy (RS_ERR_BAD_ARGUMENT); else NULL */
  const int* time_fields;     /* [6][sim_len]: year, month, day, hour, minute, second */
  const double* local;        /* [RS_L_NLOCAL][ld] */
  const double* horizons;     /* [360][ld] local horizon angles, or NULL (all zero) */
  double* out;                /* [out_nvar][n_out][ld] */
  int out_stride;             /* write step i (1-based) when (i-1-out_start) is a non-negative
                                 multiple of out_stride (get_write_stride,
                                 examples/example2/src/QueryDataTools.cpp:270-284) */
  int n_out;                  /* ceil((sim_len - out_start) / out_stride) */
  int* status;                /* [ld] status words (written) */
  double* state;              /* optional [RS_STATE_NPLANES(NLayers)][ld]: full per-point state, written
                                 at the end of every launch, read when step_begin > 1; or NULL */
  double* scratch;            /* [RS_SCRATCH_NPLANES(NLayers)][ld] work space; required when the
                                 model has use_coupling == 1, else may be NULL */
  unsigned long long* counters; /* optional [RS_CNT_N] device counters (accumulated), or NULL */
  double* solar;              /* [sim_len][4] work space: per-step solar table (time-only part of
                                 src/SunPosition.f90), filled by the library at every launch */
  /* Time chunking (all 0 = one launch for the whole run).  A launch runs the model steps
   * [step_begin, step_end] (1-based, inclusive).  With step_begin > 1 the per-point state is loaded
   * from `state` (as written by the launch that ended at step_begin - 1; `status`, `scratch` and
   * `counters` must be the same buffers), so a run may be split into chunks whose forcing is streamed
   * through HBM; results are bit-identical to a single launch.  A chunk must contain a warp's whole
   * coupling window [start, end + 1] or none of it (else RS_ST_BAD_WINDOW). */
  int step_begin;
  int step_end;
  int forcing_step0;          /* forcing_mode 0: model step of forcing record 0 (0 -> 1) */
  int out_slot0;              /* output slot (step-1-out_start)/out_stride stored at out[:, 0, :] */
  int out_start;              /* 0-based index of the first stored step (0 <= out_start < sim_len) */
  int out_nvar;               /* 0 or RS_O_NVAR: the six model outputs; RS_O_NVAR_EXT: plus the
                                 Tair / Tdew inputs and the dew point deficit */
  const int* order;           /* optional [ld] permutation of the point slots (device memory): thread t
                                 runs point order[t].  Work that only some points need (sky-view
                                 radiation: solar geometry + horizon lookup) costs a warp as soon as
                                 one of its 32 points needs it, so gathering such points pays (7 %
                                 on a grid with 30 % of them scattered); roadsurf_order_points builds
                                 the permutation.  Results do not depend on it.  Recommended with
                                 coarse forcing (per-step loads of a permuted warp are gathers). */
  double* expand_workspace;   /* forcing_mode 2: [expand_steps][nvar][ld] device work space */
  int expand_steps;           /* forcing_mode 2: model steps per expansion chunk (>= 1).  More than one
                                 chunk needs `state`; with coupling a chunk must hold a whole window */
  int coupling_window_end;    /* 0, or the caller's assertion that every coupled point of the batch has
                                 couplingIndexI == this value (points that do not are flagged
                                 RS_ST_BAD_WINDOW).  With `state` and `scratch` present it enables lane
                                 compaction between coupling iterations: the run is split at the
                                 window end and only the points that want another iteration are
                                 re-run, in dense warps (option "coupling_compaction_passes").
                                 Results are bit-identical to the single launch. */
} RsDeviceBatch;

enum
{
  RS_CNT_EXECUTED_STEPS = 0, /* point-steps executed incl. coupling re-runs */
  RS_CNT_BL_ITERATIONS,      /* boundary layer iterations summed over point-steps */
  RS_CNT_COUPLING_PASSES,    /* warp-level passes over a coupling window */
  RS_CNT_FAILED_POINTS,
  RS_CNT_N = 8
};

/* Number of fp64 planes of the per-point state for a given NLayers: Tmp(0:N+1), 10 surface scalars,
 * 3 relaxation latches, 5 radiation-coupling scalars, 1 flag word. */
#define RS_STATE_NPLANES(nlayers) ((nlayers) + 2 + 19)
/* Number of fp64 planes of the coupling work space (window snapshot, bracket scalars, one plane for
 * the compaction index list). */
#define RS_SCRATCH_NPLANES(nlayers) (2 * (nlayers) + 17)

/* Upload settings + parameters for subsequent roadsurf_run_device calls on the current device
 * (derives layer geometry, conductivities and log terms: src/Initialization.f90:181-358,
 * src/BalanceModel.f90:158-186,254-279).  Returns RS_OK or an error. */
/* Ordering: a device holds ONE model (constant memory).  roadsurf_run_device uses the model of the most
 * recent roadsurf_set_model on the current device; the batched host entries upload their own.  A model
 * is only replaced after every kernel queued by roadsurf_run_device under the previous one has finished
 * (roadsurf_set_model and the host entries block for them), and an identical model is not uploaded
 * again.  Threads that share a device through the asynchronous entry must therefore agree on its model:
 * thread A's roadsurf_run_device after thread B's roadsurf_set_model runs B's model. */
int roadsurf_set_model(const InputSettings* settings, const InputParameters* params);

/* Launch the step kernel over a device-resident batch on `stream` (a cudaStream_t passed as
 * void*; NULL = default stream).  Asynchronous.  Returns RS_OK or an error code. */
int roadsurf_run_device(const RsDeviceBatch* batch, void* stream);

/* ---- host structure-of-arrays entry (coarse forcing records + strided output) ---------------- */

/* The same batch as RsDeviceBatch but with HOST pointers and no padding (leading dimension =
 * npoints).  This is the host-buffer form of the coarse-forcing / strided-output interface: the
 * library copies the records to the device(s), interpolates them in time inside the kernel
 * (examples/example1/src/JsonSource.cpp:49-176), and copies the strided outputs
 * (examples/example1/src/roadrunner.cpp:285-327: every outputStep) back.  Pinned host memory is
 * recommended (the copies are asynchronous and chunk-pipelined), pageable memory works. */
typedef struct RsHostBatch
{
  int npoints;
  int sim_len;
  int forcing_mode;           /* 0: one record per model step, 1: coarse records (example1's rule); mode 2 is
                                 offered by the device entry only (RS_ERR_UNSUPPORTED here) */
  int n_records;
  int nvar;                   /* RS_F_NVAR or RS_F_NVAR_DEPTH */
  int out_stride;
  const double* forcing;      /* [n_records][nvar][npoints] */
  const int* record_step;     /* [n_records] (forcing_mode 1): strictly increasing, record_step[0] <= 0;
                                 RS_ERR_BAD_ARGUMENT otherwise, before any device work */
  const int* time_fields;     /* [6][sim_len] */
  const double* local;        /* [RS_L_NLOCAL][npoints] */
  const double* horizons;     /* [360][npoints] or NULL */
  double* out;                /* [RS_O_NVAR][n_out][npoints], n_out = ceil(sim_len / out_stride) */
  int* status;                /* [npoints] or NULL */
  int coupling_window_end;    /* as in RsDeviceBatch: 0, or the couplingIndexI every coupled point has
                                 (enables lane compaction between coupling iterations) */
  void* statics;              /* NULL, or a handle from roadsurf_prepare_statics for this grid of points:
                                 the local horizon table (and the point order derived from the sky-view
                                 factors) is then already on the device(s) and `horizons` is not read */
} RsHostBatch;

/* Runs a host SoA batch on `ngpus` devices (<= 0: all visible; 1: the current device), points
 * split into contiguous shards.  Synchronous.  Statistics via roadsurf_last_batch_stats. */
int roadsurf_run_host_soa(const RsHostBatch* batch, const InputSettings* settings,
                          const InputParameters* params, int ngpus);

/* Repeated forecasts over ONE grid of points: the per-point statics that do not change between
 * forecasts -- the 360-entry local horizon table (2880 of the ~5250 bytes a config-4 point uploads per
 * call) and the point order that gathers the sky-view points -- are uploaded once and kept on the
 * device(s).  `batch` supplies npoints, local (only the sky-view plane is read) and horizons, all with
 * the layout of roadsurf_run_host_soa; `ngpus` must be the value later passed to roadsurf_run_host_soa.
 * The handle goes into RsHostBatch.statics of every later call for the same grid; the per-forecast
 * planes of `local` (relaxation targets, coupling observation / index, InitLenI) are still taken from
 * each call's batch.  Returns RS_OK or an error; release with roadsurf_release_statics. */
int roadsurf_prepare_statics(const RsHostBatch* batch, int ngpus, void** handle);
void roadsurf_release_statics(void* handle);

/* roadsurf_read_input_derive for a batch held as coarse records (forcing_mode 1): what read_input
 * would derive from the time-interpolated arrays (examples/example1/src/roadrunner.cpp:157-278 after
 * JsonSource.cpp:49-176), computed from the records without materialising them.  Reads
 * batch->forcing / record_step / npoints / n_records / nvar / sim_len; writes the planes
 * RS_L_TAIR_RELAX, RS_L_VZ_RELAX, RS_L_RH_RELAX, RS_L_COUPLING_TSURF, RS_L_COUPLING_INDEX,
 * RS_L_INIT_LEN and RS_L_ACTIVE (1 = all required inputs present at every step) of
 * `local` [RS_L_NLOCAL][npoints]; lat / lon / sky view are the caller's.  TSurfObs records are NOT
 * modified: the kernel blanks the coupling window itself.  *window_end (may be NULL) receives the
 * common couplingIndexI of the coupled points, or 0 if they differ or there are none (the value to
 * put into coupling_window_end).  A record grid that is not strictly increasing or starts after step 0
 * is RS_ERR_BAD_ARGUMENT.  Pure host code. */
int roadsurf_read_input_derive_records(const RsHostBatch* batch, const InputSettings* settings, int forecast_step,
                                       const int* latest_obs_index, double* local, int* window_end);

/* ---- step-granular sessions (the Fortran subroutine API of module RoadSurf forwards to these) -------- */

/* The library's Fortran API (src/RoadSurf.f90:9-252) advances ONE point ONE step per call sequence
 * (CheckValues ... SaveOutput, CheckEndCoupling; examples/example1/src/Simulation.f90:58-94).  A session
 * holds the same run on the device: inputs uploaded once, per-point state resident between launches
 * (the resumable state planes), one call per model step.
 *
 * roadsurf_session_open   same arguments as roadsurf_run_batch (npoints >= 1; all points must share one
 *                         time axis and, if coupled, one coupling window).  Pre-fills the caller's output
 *                         arrays with -9999.0 as Initialization does (src/Initialization.f90:397-412).
 * roadsurf_step           advance the session to model step i (1-based, <= SimLen): runs the steps
 *                         (done, i] in one launch of the step kernel -- i = done + 1 is one launch with
 *                         step_begin = step_end = i.  A coupling window is indivisible (its rewinds happen
 *                         inside the kernel): a call that enters the window [start, end] runs through
 *                         step end + 1.  i = SimLen runs the "last value" step (Simulation.f90:100-115).
 *                         With a run-ahead chunk K > 1 (roadsurf_session_set_chunk) a call that has to
 *                         launch anyway runs K steps at once; results are bit-identical either way.
 * roadsurf_session_fetch  copy the outputs of every step <= i not yet delivered into the caller's output
 *                         arrays (element i-1 <- step i), and the status words if status != NULL.
 * roadsurf_session_done   number of steps executed so far.
 * Results equal roadsurf_run_batch's bit for bit.  All return RS_OK or an error code. */
int roadsurf_session_open(int npoints, OutputPointers* const* out, const InputPointers* const* in,
                          const InputSettings* settings, const InputParameters* params,
                          const LocalParameters* const* local, void** session);
int roadsurf_step(void* session, int i);
int roadsurf_session_fetch(void* session, int i, int* status);
int roadsurf_session_set_chunk(void* session, int steps);
int roadsurf_session_done(void* session);
void roadsurf_session_close(void* session);

/* Pack kernels for callers that hold point-major data on the device (device pointers, asynchronous):
 * to_soa:   src[point][n] (row stride `src_ld` elements) -> dst[n][ld];
 * from_soa: src[n][ld] -> dst[point][n] (row stride `dst_ld` elements).
 * Values are copied bit for bit; elements outside [0, npoints) x [0, n) are not touched.  Any npoints and n
 * that fit the int arguments are accepted.  RS_ERR_BAD_ARGUMENT for null pointers, npoints < 0, n < 0,
 * ld < npoints or a point-major row stride < n; npoints == 0 or n == 0 is RS_OK without a launch. */
int roadsurf_transpose_to_soa(const double* src, int64_t src_ld, int npoints, int n, double* dst,
                              int ld, void* stream);
int roadsurf_transpose_from_soa(const double* src, int ld, int npoints, int n, double* dst,
                                int64_t dst_ld, void* stream);

/* Fill n doubles with `value` (used for the -9999.0 output pre-fill).  Asynchronous.  RS_ERR_BAD_ARGUMENT
 * for a null dst or n < 0; n == 0 is RS_OK without a launch. */
int roadsurf_fill(double* dst, int64_t n, double value, void* stream);

/* Measure the fp64 FMA throughput of the current device (TFLOP/s, FMA = 2 flop) with a
 * register-resident DFMA kernel; used as the fp64 roofline denominator by bench.py. */
double roadsurf_measure_fp64_tflops(int iterations);

/* The expansion pass of forcing_mode 2 on its own: coarse records -> one record per model step for the
 * steps [step_begin, step_end] into dst [step_end - step_begin + 1][nvar][ld] (device memory).  `records`
 * supplies forcing, record_step, n_records, nvar, ld, npoints; the time step is the current model's.
 * rule 1: example1's interpolation (what forcing_mode 1 does inside the step kernel); rule 2: example2's.
 * Asynchronous on `stream`. */
int roadsurf_expand_records(const RsDeviceBatch* records, int rule, int step_begin, int step_end, double* dst,
                            void* stream);

/* Diagnostic: the solar position (src/SunPosition.f90:20-194) exactly as the step kernel evaluates it, for
 * every (step, point) pair.  Device pointers: time_fields [6][n_steps] (n_steps <= 65535), lat / lon [npoints]
 * in degrees; elevation / azimuth [n_steps][npoints] in degrees, -9999.9 when the sun is down, NaN where the
 * reference would `stop`.  Asynchronous on `stream`. */
int roadsurf_sun_position(const int* time_fields, int n_steps, const double* lat, const double* lon, int npoints,
                          double* elevation, double* azimuth, void* stream);

/* Math primitives of the step kernel, for roadsurf_eval_primitive. */
enum
{
  RS_PRIM_EXP = 0,                 /* exp: libm's algorithm, device-library exp outside its fast path */
  RS_PRIM_EXP_SMEM = 1,            /*   ... tables read from shared memory (latency body) */
  RS_PRIM_LOG = 2,                 /* log: libm's algorithm, device-library log outside its fast path */
  RS_PRIM_LOG_SMEM = 3,            /*   ... tables read from shared memory */
  RS_PRIM_EXP_FLAT = 4,            /* the branch-free exp of the early saturation pressures, with its fallback */
  RS_PRIM_EXP_FLAT_SMEM = 5,       /*   ... tables read from shared memory */
  RS_PRIM_PSIH_UNSTABLE = 6,       /* -2 log((1 + sqrt(1 - 16 a)) / 2), the unstable stability correction */
  RS_PRIM_PSIH_UNSTABLE_SMEM = 7,  /*   ... tables read from shared memory */
  RS_PRIM_FRCP = 8,                /* 1 / b (the values of a are ignored) */
  RS_PRIM_FDIV = 9,                /* a / b */
  RS_PRIM_DIV_CONST = 10,          /* a / b through the constant-divisor form, reciprocal RN(1 / b) */
  RS_PRIM_N = 11
};

/* Diagnostic: out[k] = fn(a[k]) or fn(a[k], b[k]) for k < n, exactly as the step kernel evaluates the primitive
 * (same code, same build flags).  Device pointers; b is read by RS_PRIM_FRCP, _FDIV and _DIV_CONST only and may be
 * NULL otherwise.  Asynchronous on `stream`.  RS_ERR_BAD_ARGUMENT for an unknown fn, n < 0, a null a / out, or a
 * null b where fn reads it; n == 0 is RS_OK without a launch.  The domains on which the results equal the host's
 * libm and IEEE division bit for bit are listed in DESIGN.md section 4. */
int roadsurf_eval_primitive(int fn, const double* a, const double* b, double* out, int64_t n, void* stream);

/* Builds RsDeviceBatch.order on the device: the slots of points without sky-view radiation first, those
 * with it last, original order kept inside both classes.  `local` is the batch's [RS_L_NLOCAL][ld]
 * statics tensor, `order` receives ld ints.  Asynchronous on `stream`; call once per batch layout. */
int roadsurf_order_points(const double* local, int ld, int npoints, int* order, void* stream);

/* roadsurf_run_batch and roadsurf_run_host_soa keep their device and pinned-host work buffers between
 * calls (allocation costs more than a run).  This releases them; they are re-created on demand.  Must
 * not be called while another thread is inside one of those entry points. */
void roadsurf_release_workspace(void);

/* Run-time options.  "forcing_staging": 1 = in full-resolution mode stage the forcing of every warp
 * through a ring of shared-memory tiles filled by TMA bulk copies a few steps ahead, 0 = direct
 * coalesced read-only loads (default; measured 3-6 % faster on B200, see DESIGN.md).  The default can
 * also be set with the environment variable ROADSURF_B200_FORCING_STAGING=1.  Results are identical.
 * "coupling_compaction_passes" (default 6, 0 = off): with RsDeviceBatch.coupling_window_end set, the
 * number of compacted passes over the coupling window before the points still iterating finish
 * inside the last launch.
 * "write_back_inputs" (default 0): 1 = roadsurf_run_batch and runsimulation also leave the caller's INPUT arrays
 * as the reference leaves them -- VZ[0] clamped to 0.4 (src/Initialization.f90:121-123), SW_dir[i] <= SW[i] for every
 * visited step (src/InputOutput.f90:75-77) and, for sky-view points, SW / SW_dir / LW of every executed step rewritten
 * by ModRadiationBySurroundings (src/ModRadiation.f90:57,65,70).  Neither example reads them after the call, so this is
 * off by default (it costs one more pass over three planes); the header declares the inputs const like the examples do.
 * "latency_body" (default -1): the step kernel exists in two bodies with identical results -- the throughput body,
 * and a latency body for launches so small that every warp is alone on its scheduler (exp / log tables in shared
 * memory, the saturation-pressure exponentials evaluated in the shadow of the boundary-layer divisions, no register
 * cap).  -1 = the latency body for grids of at most one 128-thread block per SM, 0 = never, 1 = for every launch of
 * 128-thread blocks.
 * "spread_small" (default 1): batches of at most four points per SM run one point per warp (lane 0 owns the point,
 * the other lanes follow as ghosts), larger ones up to 16 times that 2 .. 16 points per warp: a warp then executes
 * only its own points' branches (4.0 instead of 5.2 us per model step for one point).  0 = always 32 points per
 * warp; a value > 1 caps the points per warp.  Results are identical.
 * "max_points_per_device_batch": cap on the points roadsurf_run_batch puts into one device batch
 * (0 = bounded by free device memory only); batches beyond it are processed one after another. */
int roadsurf_set_option(const char* name, int value);

/* The kernel evaluates exp and log with the algorithm, operation order and tables of the host's libm
 * (glibc >= 2.28, FMA code path; roadsurf_b200/csrc/rs_libm.h), so that it is bit-identical to a
 * reference linked against that libm.  This host-only check compares the same code compiled for the
 * host with the libm of the running process on `n` random arguments: mismatches[0] (exp) and
 * mismatches[1] (log) must be 0 for the bit-identity to hold on this machine (another libm version or
 * a CPU without FMA may differ in the last bit; results then agree to 1 ulp per call, as with any
 * other libm).  Returns the number of arguments tested per function. */
long long roadsurf_selftest_libm(long long n, unsigned long long seed, long long* mismatches);

/* Since the library was loaded: runsimulation calls served, and the batches they were combined into. */
void roadsurf_runsimulation_counters(long long* calls, long long* batches);

/* Arithmetic self-test on the current device: the kernel's branch-free reciprocal, division and
 * constant-division primitives against the compiler's IEEE division on `n` random operand pairs.
 * mismatches[0..2] receive the number of results that differ (must all be 0); returns the number
 * of pairs tested, or -1 on error. */
long long roadsurf_selftest_arith(long long n, unsigned long long seed, long long* mismatches);

/* Name of the most recently launched step kernel variant and its launch geometry. */
typedef struct RsLaunchInfo
{
  int grid;
  int block;
  int smem_bytes;
  int regs_per_thread;
  int nlayers;
  int forcing_mode;
  int launches_total;   /* kernels launched by this library in this process so far */
} RsLaunchInfo;
void roadsurf_last_launch(RsLaunchInfo* info);

/* Library version string. */
const char* roadsurf_version(void);

/* ------------------------------------------------------------------------------------------ */
/* Part 3: ensemble runs                                                                        */
/* ------------------------------------------------------------------------------------------ */

/* An ensemble over P stations and M members shares the analysis period: the steps [1, F - 1] run once
 * per station, the state is then forked on the device into P * M member lanes, the forecast [F, SimLen]
 * runs per member, and the member outputs are reduced to ensemble statistics on the device.  F
 * (`fork_step`, 1-based) is the first step that reads member forcing.  The results are bit for bit
 * those of P * M independent roadsurf_run_device runs in which lane p * M + m gets station p's forcing
 * before F and member m's from F on: every output slot, status word and end-of-run state plane.
 *
 * Member lanes are station-major: lane = p * M + m, `ld_members` a multiple of 32 >= P * M.
 *
 * Where F may sit:
 *   - coupling: the whole window [start, end + 1] of every coupled station lies before F
 *     (F >= couplingIndexI + 2), and coupled stations share ONE window (members of different stations
 *     share warps; a lane whose window differs from its warp's is flagged RS_ST_BAD_WINDOW);
 *   - forcing_mode 1: F - 1 or F - 2 (0-based steps) is a record time, so that no record feeds both the
 *     shared and the member part with different values.  r_f = the last record at or before step F - 1;
 *     member record tensors start at r_f, and their slot 0 is written by the library from the shared
 *     records (the caller fills records r_f + 1 ...).  F = forecast step + 2 (example1's shape: the
 *     coupling window ends at the forecast-start record) is admissible;
 *   - forcing_mode 0: any F in [2, SimLen]; member forcing is [SimLen - F + 1][nvar][ld_members]
 *     (record 0 = step F);
 *   - forcing_mode 2: RS_ERR_UNSUPPORTED (example2's rule interpolates across up to 180 minutes, which
 *     would reach across F).
 * Relaxation targets are read at the first forecast step, so they are per member (`member_relax`).
 *   - The prefix runs on a library-owned copy of the station targets; where the station's fail the
 *     kernel's range test and a member's pass, the copy takes the first passing member's targets, so that
 *     the latch at InitLenI happens wherever a member will relax.
 *   - After the fork, member lanes whose own targets fail the test get the three latch planes reset to
 *     their initial value (the independent run never latched).
 *   - A station with InitLenI <= F - 2 has applied its targets inside the shared part already: its
 *     members whose targets differ from those get RS_ST_BAD_FORK | RS_ST_NOT_RUN and are not run. */

#define RS_ENS_MAX_MEMBERS 128
#define RS_ENS_MAX_QUANTILES 8
#define RS_ENS_MAX_THRESHOLDS 8
#define RS_ENS_MAX_EVENTS 8
#define RS_ENS_MAX_CONDITIONS 4

/* Planes of the statistics tensor, followed by one plane per requested quantile. */
enum
{
  RS_ENS_NVALID = 0, /* number of valid members (value == value and > -9000), as a double */
  RS_ENS_MEAN,       /* left-to-right sum in member order from +0.0, divided by n */
  RS_ENS_STD,        /* population standard deviation (ddof = 0), two passes in member order */
  RS_ENS_MIN,
  RS_ENS_MAX,
  RS_ENS_NFIXED = 5
};

/* Comparison of an exceedance probability. */
enum
{
  RS_ENS_LT = 0,
  RS_ENS_LE,
  RS_ENS_GT,
  RS_ENS_GE
};

typedef struct RsEnsembleThreshold
{
  int plane;    /* output plane (RS_O_*) */
  int op;       /* RS_ENS_LT / LE / GT / GE */
  double value; /* P(member value op value) = count / n */
} RsEnsembleThreshold;

/* A compound event over a window of output slots: "the conditions all hold at one slot or more of the
 * window".  Let S be the member output slots the statistics cover (the output slots of the steps [F, sim_len];
 * slots from S to n_out_members are neither read nor written).  For station p, member m, slot s < S:
 *   - valid: member m is valid for the event at s when every plane referenced by the conditions holds a valid
 *     value (value == value and > -9000) at every slot of the window W(s) = [s, min(s + window, S) - 1].  The
 *     window is truncated at the last member slot, not padded;
 *   - hit: the conjunction of the conditions holds at one slot or more of W(s), the comparisons those of
 *     RsEnsembleThreshold;
 *   - result: prob[n_thresholds + e][s][p] = (valid members that hit) / (valid members), computed as
 *     (double)count / (double)n like the thresholds; -9999.0 where no member is valid.
 * A one-condition event with window 1 equals the threshold with the same (plane, op, value) bit for bit.
 * Example, "wet road freezing within the next 3 h" at hourly output slots: window 3, conditions
 * {RS_O_TSURF, RS_ENS_LT, 0.0} and {RS_O_WATER, RS_ENS_GT, x}. */
typedef struct RsEnsembleEvent
{
  int n_conditions;                                      /* 1 .. RS_ENS_MAX_CONDITIONS, combined with AND */
  int window;                                            /* >= 1 output slots */
  RsEnsembleThreshold conditions[RS_ENS_MAX_CONDITIONS]; /* plane, op, value: as for thresholds */
} RsEnsembleEvent;

/* What the statistics kernel computes per (station, output slot, plane) besides the fixed planes.
 * Quantile q of the valid values sorted y_0 <= ... <= y_{n-1}: h = (n - 1) q, i = floor(h), t = h - i;
 * y_i if t == 0 or i == n - 1, else y_i + t (y_{i+1} - y_i).  Where n == 0 every value but RS_ENS_NVALID (0.0)
 * is -9999.0, the probabilities too.  The event probabilities follow the thresholds in `prob`: event j is
 * plane n_thresholds + j. */
typedef struct RsEnsembleStatsSpec
{
  int n_quantiles;  /* 0 .. RS_ENS_MAX_QUANTILES */
  int n_thresholds; /* 0 .. RS_ENS_MAX_THRESHOLDS */
  double quantiles[RS_ENS_MAX_QUANTILES];
  RsEnsembleThreshold thresholds[RS_ENS_MAX_THRESHOLDS];
  int n_events;     /* 0 .. RS_ENS_MAX_EVENTS */
  RsEnsembleEvent events[RS_ENS_MAX_EVENTS];
} RsEnsembleStatsSpec;

/* Areas: groups of stations such as a maintenance route or a district, for the probability that an event of
 * spec.events occurs anywhere in the group.  An area is a non-empty set of station indices; areas may overlap, and
 * a station may belong to any number of them.  For area A, event e, member m and member slot s < S (the slots the
 * station events cover):
 *   - valid: member m is valid for A at s when it is valid for e at s (RsEnsembleEvent's station rule) at EVERY
 *     station of A.  A station that did not run (RS_ST_NOT_RUN, all -9999) therefore makes every area that holds it
 *     invalid for that member: leave such stations out of the areas;
 *   - hit: the member is valid for A and hits e at s at one station of A or more (each station within its own window
 *     W(s); different stations may hit at different slots of the window);
 *   - result: area_prob[e][s][a] = (double)hits / (double)valid, -9999.0 where no member is valid.
 * So an area of one station equals that station's event plane of `prob` bit for bit, and neither repeated stations
 * nor their order change an area's result.  The arrays are HOST memory in every entry: the library checks every
 * index and copies the arrays, and the caller may reuse them when the call returns. */
typedef struct RsEnsembleAreas
{
  int n_areas;         /* >= 1 */
  const int* offsets;  /* HOST [n_areas + 1]: offsets[0] == 0, strictly increasing (no empty area) */
  const int* stations; /* HOST [offsets[n_areas]]: area a is stations[offsets[a] .. offsets[a + 1] - 1], each in
                          [0, npoints) */
} RsEnsembleAreas;

/* Event onset: the probability that an event of spec.events has begun by each member slot, per station and per
 * area ("by 03:00, how likely is it that freezing has begun on this route?").  It uses the events' conditions; their
 * window does not enter.  For station p, event e, member m and member slot s < S (the slots the station events cover):
 *   - valid: every plane the conditions name holds a valid value (value == value and > -9000) at every slot of
 *     [0, s];
 *   - hit: valid, and the conjunction of the conditions holds at one slot or more of [0, s];
 *   - result: onset[e][s][p] = (double)hits / (double)valid, -9999.0 where no member is valid;
 *   - areas (RsEnsembleAreas): a member is valid for area A at s when it is valid at every station of A, and hits
 *     when it is also a hit at one station of A or more; area_onset[e][s][a] likewise.
 * This is the event rule and the area rule applied to the growing window [0, s].  So onset[e][s][p] equals, bit for
 * bit, the station event probability at slot 0 of an event with the same conditions and window = s + 1, and
 * area_onset[e][s][a] equals area_prob of that event at slot 0.  An area of one station equals that station's onset
 * plane.  Per (station, event, member) the library keeps two integers: X, the first slot where a named plane is
 * invalid (S if none), and O, the first slot before X where the conditions hold (none if there is none); then valid(s)
 * <=> X > s and hit(s) <=> O <= s, and an area takes per member the minimum X and the minimum O over its stations.
 * Where a station's valid members do not change with s (no invalid value after slot 0), its onset never decreases
 * with s, so the lead time by which a fraction q of the members have seen the event is the first s with
 * onset >= q. */

/* Window extremes: statistics of each member's minimum or maximum of one plane over a window of member slots, per
 * station and per area ("how cold will the road get tonight?": the forecast minimum road-surface temperature over the
 * night, or the maximum ice storage over the next hours).  An extreme is {plane, kind, window}.  For station p,
 * extreme x, member m and member slot s < S (the slots the statistics cover):
 *   - valid: the plane holds a valid value (value == value and > -9000) at every slot of
 *     W(s) = [s, min(s + window, S) - 1], RsEnsembleEvent's window, truncated at the last member slot, not padded;
 *   - value: the minimum (RS_ENS_WMIN) or maximum (RS_ENS_WMAX) of the plane over W(s) in the total order of the
 *     order-preserving map of a double's bits b (as int64) to b >= 0 ? b : b ^ 0x7fffffffffffffff, so that -0.0 lies
 *     below +0.0 and the result does not depend on the order of evaluation;
 *   - result: ext_stats[j][x][s][p] holds the statistics of RsEnsembleStatsSpec (planes RS_ENS_NVALID, MEAN, STD, MIN
 *     and MAX, then spec.n_quantiles quantile planes) over the valid members' values, with the definitions, member
 *     order and operation order of `stats` and its -9999.0 / 0.0 convention where no member is valid.  The layout is
 *     that of `stats` with the extremes in place of the output planes: [RS_ENS_NFIXED + n_quantiles][n_extremes]
 *     [n_out][ld].  The spec's thresholds and events are ignored;
 *   - areas (RsEnsembleAreas): a member is valid for area A at s when it is valid at every station of A, and its value
 *     is the minimum (maximum) over A's stations of the station values in the same order; area_ext_stats[j][x][s][a],
 *     [RS_ENS_NFIXED + n_quantiles][n_extremes][n_out][n_areas].
 * Identities: (1) an extreme with window 1 equals the `stats` planes of its plane bit for bit; (2) an area of one
 * station equals that station's values bit for bit, and neither repeated stations nor their order change an area's
 * result; (3) the fraction of valid members whose window minimum is < v is the event probability of
 * {plane, RS_ENS_LT, v} with the same window (area_prob for areas), and likewise the maximum with RS_ENS_GT. */
#define RS_ENS_MAX_EXTREMES 8

enum
{
  RS_ENS_WMIN = 0,
  RS_ENS_WMAX = 1
};

typedef struct RsEnsembleExtreme
{
  int plane;  /* output plane (RS_O_*) */
  int kind;   /* RS_ENS_WMIN / RS_ENS_WMAX */
  int window; /* >= 1 output slots */
} RsEnsembleExtreme;

typedef struct RsEnsembleExtremes
{
  int n_extremes; /* 1 .. RS_ENS_MAX_EXTREMES */
  RsEnsembleExtreme extremes[RS_ENS_MAX_EXTREMES];
} RsEnsembleExtremes;

/* A device-resident ensemble (DEVICE pointers on the current device). */
typedef struct RsEnsembleBatch
{
  RsDeviceBatch shared;          /* the P stations, as for roadsurf_run_device with the whole run's time axis:
                                    `state` is required, `scratch` too when coupled, `out` holds the output
                                    slots of the steps before F (out_slot0 = 0), forcing is the stations'
                                    forcing up to F - 1 (forcing_mode 1: the full record axis; the values of
                                    records after r_f + 1 are never read).  step_begin, step_end,
                                    forcing_step0, out_slot0 and expand_* must be 0.  `local` is not modified */
  int members;                   /* M, 1 .. RS_ENS_MAX_MEMBERS */
  int fork_step;                 /* F, 1-based, 2 <= F <= sim_len */
  int ld_members;                /* multiple of 32, >= P * M */
  double* member_forcing;        /* mode 1: [n_records - r_f][nvar][ld_members], slot 0 written by the library;
                                    mode 0: [sim_len - F + 1][nvar][ld_members] */
  const double* member_relax;    /* [3][ld_members]: tair, VZ, RH relaxation targets per member, or NULL
                                    (the station's targets for every member) */
  double* member_local;          /* [RS_L_NLOCAL][ld_members]                        (written) */
  double* member_horizons;       /* [360][ld_members] when shared.horizons != NULL    (written) */
  double* member_state;          /* [RS_STATE_NPLANES(NLayers)][ld_members]; also the work space of the
                                    prefix's copy of shared.local, so it needs RS_L_NLOCAL * shared.ld
                                    doubles at least                                  (written) */
  double* member_scratch;        /* [RS_SCRATCH_NPLANES(NLayers)][ld_members] when coupled (written) */
  int* member_status;            /* [ld_members]                                      (written) */
  double* member_out;            /* [out_nvar][n_out_members][ld_members]: slot 0 = the first output slot of
                                    a step >= F                                       (written) */
  int n_out_members;             /* slot dimension of member_out, stats and prob: >= the number of output slots of
                                    the steps [F, sim_len]; the statistics cover those slots, later ones are
                                    neither read nor written */
  const int* member_order;       /* optional [ld_members] thread permutation, as RsDeviceBatch.order */
  RsEnsembleStatsSpec spec;
  double* stats;                 /* [RS_ENS_NFIXED + n_quantiles][out_nvar][n_out_members][shared.ld], or NULL */
  double* prob;                  /* [n_thresholds + n_events][n_out_members][shared.ld], or NULL */
} RsEnsembleBatch;

/* Runs an ensemble asynchronously on `stream`: (1) the prefix [1, F - 1] of the P stations (with lane
 * compaction between coupling iterations when shared.coupling_window_end is set, under the rules of
 * roadsurf_run_device), (2) the fork into the member lanes, (3) the member launch [F, sim_len], a resumed
 * launch of the step kernel, (4) the statistics (when stats or prob is given) and, when prob is given and
 * spec.n_events > 0, the event probabilities.  shared.counters, if
 * given, accumulate both launches.  forcing_mode 1 reads record_step back once (a small synchronous
 * copy on `stream`) to check the record grid (strictly increasing, record_step[0] <= 0) and F against
 * it.  Returns RS_OK or an error code. */
int roadsurf_run_ensemble_device(const RsEnsembleBatch* batch, void* stream);

/* The statistics kernel on its own, over any station-major member tensor member_out
 * [out_nvar][n_out][ld_members] (lane p * members + m): stats [RS_ENS_NFIXED + n_quantiles][out_nvar][n_out][ld],
 * prob [n_thresholds + n_events][n_out][ld] (either may be NULL); the events read the planes they name over the
 * n_out slots.  Device pointers; asynchronous on `stream`. */
int roadsurf_ensemble_stats(const double* member_out, int out_nvar, int n_out, int ld_members, int npoints,
                            int members, const RsEnsembleStatsSpec* spec, double* stats, double* prob, int ld,
                            void* stream);

/* Area event probabilities (RsEnsembleAreas) over a station-major member tensor member_out
 * [out_nvar][n_out][ld_members] (lane p * members + m), as for roadsurf_ensemble_stats: area_prob DEVICE
 * [n_events][n_out][n_areas].  spec->n_events >= 1; quantiles and thresholds are ignored.  The area arrays are
 * host memory, checked and copied by the library (the caller may reuse them when the call returns); asynchronous on
 * `stream` otherwise.  After roadsurf_run_ensemble_device, call it on the same stream with the batch's member_out,
 * n_out = n_out_members (equal to the member slots of the run), ld_members, shared.npoints and members:
 *   roadsurf_run_ensemble_device(&e, stream);
 *   roadsurf_ensemble_area_events(e.member_out, e.shared.out_nvar, e.n_out_members, e.ld_members,
 *                                 e.shared.npoints, e.members, &e.spec, &areas, d_area_prob, stream); */
int roadsurf_ensemble_area_events(const double* member_out, int out_nvar, int n_out, int ld_members, int npoints,
                                  int members, const RsEnsembleStatsSpec* spec, const RsEnsembleAreas* areas,
                                  double* area_prob, void* stream);

/* Event onset (defined after RsEnsembleAreas) over a station-major member tensor member_out
 * [out_nvar][n_out][ld_members] (lane p * members + m), as for roadsurf_ensemble_stats: onset DEVICE [n_events][n_out][ld] or NULL, area_onset
 * DEVICE [n_events][n_out][n_areas] or NULL (then areas must be NULL too); one of the two at least.
 * spec->n_events >= 1; quantiles and thresholds are ignored.  The area arrays are host memory, checked and copied as
 * for roadsurf_ensemble_area_events; asynchronous on `stream` otherwise.  After roadsurf_run_ensemble_device:
 *   roadsurf_run_ensemble_device(&e, stream);
 *   roadsurf_ensemble_onset(e.member_out, e.shared.out_nvar, e.n_out_members, e.ld_members, e.shared.npoints,
 *                           e.members, &e.spec, d_onset, e.shared.ld, &areas, d_area_onset, stream); */
int roadsurf_ensemble_onset(const double* member_out, int out_nvar, int n_out, int ld_members, int npoints, int members,
                            const RsEnsembleStatsSpec* spec, double* onset, int ld, const RsEnsembleAreas* areas,
                            double* area_onset, void* stream);

/* Window extremes (defined after RsEnsembleAreas) over a station-major member tensor member_out
 * [out_nvar][n_out][ld_members] (lane p * members + m), as for roadsurf_ensemble_stats: ext_stats DEVICE
 * [RS_ENS_NFIXED + n_quantiles][n_extremes][n_out][ld] or NULL, area_ext_stats DEVICE
 * [RS_ENS_NFIXED + n_quantiles][n_extremes][n_out][n_areas] or NULL (then areas must be NULL too); one of the two at
 * least.  Only spec->n_quantiles and spec->quantiles are used (the spec is checked whole).  Extreme planes lie in
 * [0, out_nvar).  The area arrays are host memory, checked and copied as for roadsurf_ensemble_area_events; a spec
 * without events is accepted with areas.  Asynchronous on `stream`; it takes a work space with cudaMallocAsync and
 * frees it with cudaFreeAsync on `stream`: n_extremes * n_out * ceil32(npoints * members) * 8 bytes, and with areas
 * n_extremes * n_out * n_areas * members * 8 bytes more plus the area plan (about 20 bytes per area station).
 *   roadsurf_run_ensemble_device(&e, stream);
 *   roadsurf_ensemble_extremes(e.member_out, e.shared.out_nvar, e.n_out_members, e.ld_members, e.shared.npoints,
 *                              e.members, &e.spec, &ext, d_ext_stats, e.shared.ld, &areas, d_area_ext_stats, stream); */
int roadsurf_ensemble_extremes(const double* member_out, int out_nvar, int n_out, int ld_members, int npoints,
                               int members, const RsEnsembleStatsSpec* spec, const RsEnsembleExtremes* ext,
                               double* ext_stats, int ld, const RsEnsembleAreas* areas, double* area_ext_stats,
                               void* stream);

/* Host form on the current device, forcing_mode 1 only.  `shared` is the stations' host SoA batch
 * (as for roadsurf_run_host_soa, with the full record axis); its `out`, if not NULL, receives the
 * station outputs of the steps before F, [RS_O_NVAR][n_out_pre][P] with n_out_pre = ceil((F - 1) /
 * out_stride); `status` is not written.  member_records [n_records - r_f - 1][nvar][P * M] are the
 * members' records r_f + 1 ... (lane p * M + m).  With use_relaxation == 1 the member relaxation targets are
 * derived by the rule of roadsurf_read_input_derive_records from each member's records (the station's up to r_f)
 * and `latest_obs_index` (per station, as passed to that call; NULL = no observation anywhere, targets
 * -9999.9); shared->local is expected to hold what that call derived for the stations.
 * Coupled stations must share one window (RS_ERR_UNSUPPORTED otherwise).  Outputs: stats
 * [RS_ENS_NFIXED + n_quantiles][RS_O_NVAR][n_out_m][P], prob [n_thresholds + n_events][n_out_m][P] and, when not NULL,
 * member_out [RS_O_NVAR][n_out_m][P * M] and member_status [P * M], with n_out_m the output slots of the
 * steps [F, sim_len].  Stations are processed in chunks that fit device memory and the option
 * "max_points_per_device_batch" (counted in member lanes).  Synchronous; roadsurf_last_batch_stats reports
 * the phases (kernel_ms: prefix, fork, members, statistics and events). */
int roadsurf_run_ensemble_host_soa(const RsHostBatch* shared, const double* member_records, int members,
                                   int fork_step, const int* latest_obs_index, const RsEnsembleStatsSpec* spec, double* stats, double* prob,
                                   double* member_out, int* member_status, const InputSettings* settings,
                                   const InputParameters* params);

/* roadsurf_run_ensemble_host_soa plus area event probabilities: area_prob HOST [n_events][n_out_m][n_areas].  The
 * areas are planned once per call and accumulated on the device after each station chunk, so an area may span
 * chunks; one device-to-host copy of area_prob at the end (counted in d2h_bytes; the two area kernels in kernel_ms).
 * prob may be NULL with areas given (no station events are computed then).  areas == NULL and area_prob == NULL is
 * exactly roadsurf_run_ensemble_host_soa; one without the other is RS_ERR_BAD_ARGUMENT.  The area accumulators,
 * 2 * n_areas * n_events * ceil(n_out_m / 64) * members * 8 bytes, stay on the device for the whole call:
 * RS_ERR_CUDA where they do not fit. */
int roadsurf_run_ensemble_host_soa_areas(const RsHostBatch* shared, const double* member_records, int members,
                                         int fork_step, const int* latest_obs_index, const RsEnsembleStatsSpec* spec,
                                         double* stats, double* prob, double* member_out, int* member_status,
                                         const RsEnsembleAreas* areas, double* area_prob,
                                         const InputSettings* settings, const InputParameters* params);

/* roadsurf_run_ensemble_host_soa_areas plus event onset (defined after RsEnsembleAreas): onset HOST
 * [n_events][n_out_m][P] and area_onset HOST [n_events][n_out_m][n_areas], each NULL or not.  The onset planes are copied back after each
 * station chunk, area_onset once at the end (both counted in d2h_bytes; the onset kernels in kernel_ms).  Any of
 * prob, area_prob, onset and area_onset may be NULL; areas go with area_prob or area_onset, and area_prob or
 * area_onset without areas is RS_ERR_BAD_ARGUMENT, as are onset outputs with a spec without events.  With onset and
 * area_onset NULL it is exactly roadsurf_run_ensemble_host_soa_areas.  Device memory for the whole call, beside the
 * area event accumulators: the area onset accumulators, n_areas * n_events * members * 8 bytes, and area_onset,
 * n_events * n_out_m * n_areas * 8 bytes (RS_ERR_CUDA where they do not fit); per station chunk a workspace of
 * n_events * 8 bytes per member lane. */
int roadsurf_run_ensemble_host_soa_onset(const RsHostBatch* shared, const double* member_records, int members,
                                         int fork_step, const int* latest_obs_index, const RsEnsembleStatsSpec* spec,
                                         double* stats, double* prob, double* member_out, int* member_status,
                                         const RsEnsembleAreas* areas, double* area_prob, double* onset,
                                         double* area_onset, const InputSettings* settings, const InputParameters* params);

/* roadsurf_run_ensemble_host_soa_onset plus window extremes (defined after RsEnsembleAreas): ext_stats HOST
 * [RS_ENS_NFIXED + n_quantiles][n_extremes][n_out_m][P] and area_ext_stats HOST
 * [RS_ENS_NFIXED + n_quantiles][n_extremes][n_out_m][n_areas], each NULL or not; ext goes with one of them at least,
 * and either needs ext.  Extreme planes are the RS_O_NVAR model planes.  ext_stats is copied back after each station
 * chunk, area_ext_stats once at the end (both counted in d2h_bytes; the extremes kernels in kernel_ms).  Areas may go
 * with area_ext_stats alone, and then the spec needs no events.  With ext, ext_stats and area_ext_stats NULL it is
 * exactly roadsurf_run_ensemble_host_soa_onset.  Device memory for the whole call, beside the area event and onset
 * buffers: the area extreme accumulators, n_extremes * n_out_m * n_areas * members * 8 bytes, and area_ext_stats
 * (RS_ERR_CUDA where they do not fit); per station chunk a work space of n_extremes * n_out_m * 8 bytes per member
 * lane. */
int roadsurf_run_ensemble_host_soa_extremes(const RsHostBatch* shared, const double* member_records, int members,
                                            int fork_step, const int* latest_obs_index, const RsEnsembleStatsSpec* spec,
                                            double* stats, double* prob, double* member_out, int* member_status,
                                            const RsEnsembleAreas* areas, double* area_prob, double* onset,
                                            double* area_onset, const RsEnsembleExtremes* ext, double* ext_stats,
                                            double* area_ext_stats, const InputSettings* settings,
                                            const InputParameters* params);

#ifdef __cplusplus
}
#endif

#endif /* ROADSURF_B200_H */
