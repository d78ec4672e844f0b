// rs_ensemble.cuh -- launchers of the ensemble kernels (rs_ensemble.cu), called by rs_host.cu.
#pragma once

#include "../../include/roadsurf_b200.h"

// The kernel's relaxation range test (rs_kernel.cu, rs_run_kernel: relax_on) on REAL(4)-rounded targets.
__host__ __device__ inline bool rs_relax_targets_valid(double tair, double vz, double rh)
{
  const double T = static_cast<float>(tair), V = static_cast<float>(vz), R = static_cast<float>(rh);
  return !(T < static_cast<double>(-100.0f) || T > static_cast<double>(100.0f) || V < 0.0 ||
           V > static_cast<double>(100.0f) || R < 0.0 || R > 110);
}

struct RsForkArgs
{
  int npoints, ld, members, ldm, nlayers, nvar, fork_step, relax;
  int state_planes, scratch_planes;
  int r_f;                       // forcing_mode 1: record copied into member record slot 0; -1: none
  const double* local;           // [RS_L_NLOCAL][ld]  (the caller's, not the prefix copy)
  const double* horizons;        // [360][ld] or null
  const double* state;           // [state_planes][ld]
  const double* scratch;         // [scratch_planes][ld] or null
  const int* status;             // [ld]
  const double* forcing;         // shared records [n_records][nvar][ld] (mode 1)
  const double* member_relax;    // [3][ldm] or null
  double* m_local;
  double* m_horizons;
  double* m_state;
  double* m_scratch;
  double* m_forcing;
  int* m_status;
};

// The prefix's copy of the station statics [RS_L_NLOCAL][ld] into `work`, with the relaxation targets of the
// first member whose targets pass the range test where the station's do not.
int rs_launch_ens_prefix_local(const double* local, int ld, int npoints, const double* member_relax, int ldm,
                               int members, int relax, double* work, void* stream);
int rs_launch_ens_fork(const RsForkArgs* f, void* stream);
// Statistics of the first n_slots output slots.  member_out is [out_nvar][mo_slots][ldm], stats
// [RS_ENS_NFIXED + nq][out_nvar][st_slots][ld] and prob [nt][st_slots][ld]; slots >= n_slots are not written.
int rs_launch_ens_stats(const double* member_out, int out_nvar, int n_slots, int mo_slots, int ldm, int npoints,
                        int members, const RsEnsembleStatsSpec* spec, double* stats, double* prob, int st_slots, int ld,
                        void* stream);
// Event probabilities of the first n_slots output slots into prob planes [n_thresholds, n_thresholds + n_events)
// of [..][st_slots][ld]; slots >= n_slots are not written.
int rs_launch_ens_events(const double* member_out, int n_slots, int mo_slots, int ldm, int npoints, int members,
                         const RsEnsembleStatsSpec* spec, double* prob, int st_slots, int ld, void* stream);

// Area event probabilities (RsEnsembleAreas).  The accumulators acc_valid / acc_hit are
// [n_areas][n_events][rs_area_tiles(n_slots)][members] slot masks (bit j of tile t = slot t * kRsAreaTile + j),
// set to all ones / all zeros before the first chunk.
constexpr int kRsAreaTile = 64;     // slots per accumulator word
constexpr int kRsAreaBlock = 128;   // threads of an area kernel's block (at most 4 warps of members)
inline int rs_area_tiles(int n_slots) { return (n_slots + kRsAreaTile - 1) / kRsAreaTile; }
// Accumulates the stations [p0, p0 + npoints) of member_out [..][mo_slots][ldm] (station p at lanes
// (p - p0) * members + m).  segments [n_segments][4] = {area, begin, end, 0}: the stations stations[begin .. end - 1]
// (global indices, all in the chunk) of one area.  `segments` is 16-byte aligned.
int rs_launch_ens_area_accumulate(const double* member_out, int n_slots, int mo_slots, int ldm, int members,
                                  const RsEnsembleStatsSpec* spec, const int* stations, int p0, const int* segments,
                                  int n_segments, unsigned long long* acc_valid, unsigned long long* acc_hit, void* stream);
// area_prob [n_events][st_slots][n_areas] from the accumulators; slots >= n_slots are not written.
int rs_launch_ens_area_finalize(const unsigned long long* acc_valid, const unsigned long long* acc_hit, int n_areas,
                                int n_events, int n_slots, int members, double* area_prob, int st_slots, void* stream);

// Event onset (roadsurf_ensemble_onset) of the first n_slots slots of member_out [..][mo_slots][ldm].  Per (station,
// event, member): X, the first slot where a named plane is invalid (n_slots if none), and O, the first slot before X
// where the conditions all hold (n_slots if none).  onset [n_events][st_slots][ld] (slots >= n_slots are not
// written) and ws [n_events][npoints * members] {O, X} int pairs are each written where not null.
int rs_launch_ens_onset(const double* member_out, int n_slots, int mo_slots, int ldm, int npoints, int members,
                        const RsEnsembleStatsSpec* spec, double* onset, int st_slots, int ld, int* ws, void* stream);
// Area onset: the minimum {O, X} over each segment's stations (as for rs_launch_ens_area_accumulate; station p at
// ws lane (p - p0) * members + m) into acc [n_areas][n_events][members] {O, X}, set to INT_MAX-like values (bytes
// 0x7f) before the first chunk; then area_onset [n_events][st_slots][n_areas] from acc.
int rs_launch_ens_area_onset_accumulate(const int* ws, int npoints, int members, int n_events, const int* stations, int p0,
                                        const int* segments, int n_segments, int* acc, void* stream);
int rs_launch_ens_area_onset_finalize(const int* acc, int n_areas, int n_events, int n_slots, int members,
                                      double* area_onset, int st_slots, void* stream);

// Window extremes (roadsurf_ensemble_extremes) of the first n_slots slots of member_out [..][mo_slots][ldm], lanes
// [0, lanes), into ws [n_extremes][n_slots][ldw] (-9999.0 where the window is not valid).  The extremes have been
// checked.  The statistics of ws are rs_launch_ens_stats with out_nvar = n_extremes, mo_slots = n_slots and ldm = ldw.
int rs_launch_ens_window_extremes(const double* member_out, int n_slots, int mo_slots, int ldm, int lanes,
                                  const RsEnsembleExtremes* ext, double* ws, int ldw, void* stream);
// Area window extremes: acc [n_extremes][n_slots][n_areas * members] keys, set to each extreme's identity by
// rs_init_ens_area_extremes before the first chunk; each chunk's segments (as for rs_launch_ens_area_accumulate;
// station p at ws lane (p - p0) * members + m) are combined into it; after the last chunk the finalize turns acc into
// doubles in place, which rs_launch_ens_stats reads with npoints = n_areas, ldm = n_areas * members and ld = n_areas.
int rs_init_ens_area_extremes(double* acc, int n_slots, int n_areas, int members, const RsEnsembleExtremes* ext,
                              void* stream);
int rs_launch_ens_area_extremes_accumulate(const double* ws, int n_slots, int ldw, int members,
                                           const RsEnsembleExtremes* ext, const int* stations, int p0,
                                           const int* segments, int n_segments, int n_areas, double* acc, void* stream);
int rs_launch_ens_area_extremes_finalize(double* acc, int n_slots, int n_areas, int members,
                                         const RsEnsembleExtremes* ext, void* stream);
