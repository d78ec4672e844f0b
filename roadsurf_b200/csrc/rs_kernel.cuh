// rs_kernel.cuh -- launch arguments shared by the kernels and the host code.
#pragma once

#include "rs_model.h"

// Device scratch planes needed when coupling is in use (fp64 planes of `ld` points):
//   [0, N+1]      Tmp(0:N+1) snapshot at the start of the coupling window  (src/Coupling.f90:172-210)
//   N+2 .. N+7    TsurfAve, SrfWatmms, SrfIce2mms, SrfDepmms, SrfSnowmms, Albedo snapshot
//   N+9 .. 2N+8   TmpNw(1:N) of the pass that just ended (read by the first re-run step only)
//   2N+9 .. 2N+15 RadCoeff, RadCoeffPrevious, TsurfNearestAbove/Below, RadCoefNearestAbove/Below,
//                 Tsurf_end_coup1 (touched once per coupling pass)

struct RsArgs
{
  int npoints, ld, sim_len, n_records, nvar, out_stride, n_out, forcing_mode;
  const double* forcing;
  const int* record_step;
  const int* tf;            // [6][sim_len]
  const double* local;      // [RS_L_NLOCAL][ld]
  const double* horizons;   // [360][ld] or null
  const double* solar;      // [sim_len][4] per-step solar table (rs_launch_solar)
  double* out;              // [6][n_out][ld]
  int* status;
  double* scratch;          // [RS_SCRATCH_NPLANES(N)][ld] or null
  int step_begin, step_end;   // model steps this launch runs (1-based, inclusive)
  int forcing_step0;          // full-resolution mode: model step of forcing record 0
  int out_slot0;              // global output slot stored at out[:, 0, :]
  // Kept at 120 bytes on purpose: with a 136-byte parameter struct nvcc 12.9 stops scalarising it
  // and the 128-thread full-resolution kernel picks up 200+ bytes of local-memory traffic per step.
  // Pointers touched only before / after the time loop live in RsArgsCold.
};

struct RsArgsCold
{
  double* state;                 // [RS_STATE_NPLANES(N)][ld] or null
  unsigned long long* counters;  // [RS_CNT_N] or null
  int out_start;                 // 0-based step index of output slot 0
  int out_nvar;                  // RS_O_NVAR or RS_O_NVAR_EXT
  // Lane compaction between coupling passes (see launch_model in rs_host.cu): thread t handles point
  // index[t] for t < *n_index (threads beyond are ghosts that write nothing); null = thread t is point t.
  const int* index;
  const int* n_index;            // device-side list length, or null: n_fixed entries
  int n_fixed;
  int mode;                      // RS_MODE_* bits
  int window_end;                // RS_MODE_SPLIT: the coupling window end every coupled point must have
  int spread;                    // 0, or the number of points per warp (1, 2, 4, 8, 16; they sit in the first lanes,
                                 // the other lanes are ghosts): small batches are latency-bound, and a warp that
                                 // serves fewer points executes fewer sides of every branch (one point: 4.0 instead
                                 // of 5.2 us per model step); set by rs_launch_run
  int tid0, tid_end;             // this launch covers the thread slots [tid0, tid_end) of the batch (0, 0 = all):
                                 // a large grid is launched as whole waves of 512-thread blocks + a tail of
                                 // 128-thread blocks spread over all SMs (see launch_sized)
};

enum
{
  RS_MODE_SPLIT = 1,     // the launch may begin / end at the end of the coupling window (state carries
                         // the iteration), and rewinds may go before step_begin
  RS_MODE_ONE_PASS = 2   // enter at the restart decision of step window_end + 1, re-run the window
                         // once and stop after step window_end (state written)
};

// Per-point state planes (RsArgsCold.state, RS_STATE_NPLANES(N) of them): Tmp(0:N+1) in planes 0 .. N+1, then,
// as offsets from plane N + 2: Ts, Wat, Snow, Ice, Ice2, Dep, Q2Melt, T4Melt, Evap, Alb (0 .. 9), the relaxation
// latches TairInitEnd, VZInitEnd, RhzInitEnd (RS_SP_LATCH + 0 .. 2), SwCof, LwCof, SWcorr, LWcorr, lastObs, and the
// flag word (RS_SP_FLAGS).
enum
{
  RS_SP_LATCH = 10,
  RS_SP_FLAGS = 18
};
// Flag word: coupling iterations + 1 in bits 0..7, then these bits.
enum
{
  RS_FL_CPL_FAILED = 8,
  RS_FL_START_AGAIN = 9,
  RS_FL_IN_CPL = 10,
  RS_FL_ALIVE = 11,
  RS_FL_FAILED = 12
};

// Host-callable launchers (rs_kernel.cu).  Return a cudaError_t as int.
int rs_upload_model(const RsModel* m);
int rs_launch_solar(const int* tf, int sim_len, double* table, void* stream);
// write-back of the reference's input mutations: stage [3][npc][sim_len] = SW, SW_dir, LW as the reference leaves them
int rs_launch_mutation(const double* forcing, int nvar, int ld, int sim_len, const double* local, const double* horizons,
                       const double* solar, const double* tsurf_out, int* nvis, int q0, int npc, double* stage, void* stream);
int rs_launch_sun_position(const int* tf, int n_steps, const double* lat, const double* lon, int npoints, double* elev,
                           double* azim, void* stream);
// coarse records -> per-step forcing [step_end - step_begin + 1][nvar][ld]; rule 1 = example1, 2 = example2
int rs_launch_expand(const double* rec, const int* record_step, int n_records, int nvar, int ld, int npoints, int rule,
                     double DT, int step_begin, int step_end, double* dst, void* stream);
int rs_launch_partition(const double* flags_plane, int ld, int npoints, int sorted, int* index, int* n_index, void* stream);
// `coupling`: the model has use_coupling set; `depth`: it has a fixed output depth (depth_mode != 0).  Both select
// the kernel variant compiled with exactly the features the run needs.
void rs_set_spread_small(int on);      // one point per warp for batches of at most 4 points per SM (default on)
void rs_set_latency_body(int mode);  // -1 auto (small grids), 0 never, 1 every 128-thread launch
int rs_launch_run(const RsArgs* a, const RsArgsCold* cold, int nlayers, int staged, int coupling, int depth, void* stream,
                  int* grid, int* block, int* regs, int* smem);
int rs_launch_transpose_to_soa(const double* src, long long src_ld, int npoints, int n, double* dst,
                               int ld, void* stream);
int rs_launch_transpose_from_soa(const double* src, int ld, int npoints, int n, double* dst,
                                 long long dst_ld, void* stream);
int rs_launch_fill(double* dst, long long n, double value, void* stream);
int rs_launch_eval_primitive(int fn, const double* a, const double* b, double* out, long long n, void* stream);
int rs_launch_pack_forcing(const double* stage, int npoints_chunk, int p0, int sim_len, int nvar,
                           double* forcing, int ld, void* stream);
int rs_launch_unpack_out(const double* out, int ld, int n_out, int p0, int npoints_chunk,
                         double* stage, void* stream);
double rs_measure_fp64(int iterations);
long long rs_selftest_arith(long long n, unsigned long long seed, long long* bad3);
