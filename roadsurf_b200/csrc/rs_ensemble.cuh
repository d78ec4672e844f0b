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
