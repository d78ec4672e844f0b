// rs_ensemble.cu -- the kernels of an ensemble run (roadsurf_run_ensemble_device): the prefix's copy of the
// station statics, the fork of the station state into the member lanes, the ensemble statistics and the event
// probabilities.
// Member lanes are station-major: lane = p * members + m.
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cstddef>
#include <cstring>

#include "rs_ensemble.cuh"
#include "rs_kernel.cuh"

namespace
{
// the three relaxation target planes are consecutive: plane RS_L_TAIR_RELAX + k, k = tair, VZ, RH
static_assert(RS_L_VZ_RELAX == RS_L_TAIR_RELAX + 1 && RS_L_RH_RELAX == RS_L_TAIR_RELAX + 2, "relaxation planes");

// Relaxation targets the prefix runs on for station p: the station's if they pass the range test, else
// those of its first member whose targets pass, else the station's.
__device__ void prefix_targets(const double* __restrict__ local, int ld, int p, const double* __restrict__ member_relax,
                               int ldm, int members, double t[3])
{
  for (int k = 0; k < 3; ++k) t[k] = local[static_cast<size_t>((RS_L_TAIR_RELAX + k)) * ld + p];
  if (rs_relax_targets_valid(t[0], t[1], t[2]) || member_relax == nullptr) return;
  for (int m = 0; m < members; ++m)
  {
    const size_t l = static_cast<size_t>(p) * members + m;
    const double a = member_relax[l], b = member_relax[ldm + l], c = member_relax[2 * static_cast<size_t>(ldm) + l];
    if (rs_relax_targets_valid(a, b, c))
    {
      t[0] = a;
      t[1] = b;
      t[2] = c;
      return;
    }
  }
}

__global__ void rs_ens_prefix_local_kernel(const double* __restrict__ local, int ld, int npoints,
                                           const double* __restrict__ member_relax, int ldm, int members, int relax,
                                           double* __restrict__ work)
{
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= ld) return;
  for (int k = 0; k < RS_L_NLOCAL; ++k) work[static_cast<size_t>(k) * ld + q] = local[static_cast<size_t>(k) * ld + q];
  if (!relax || q >= npoints) return;
  double t[3];
  prefix_targets(local, ld, q, member_relax, ldm, members, t);
  for (int k = 0; k < 3; ++k) work[static_cast<size_t>((RS_L_TAIR_RELAX + k)) * ld + q] = t[k];
}

__device__ __forceinline__ bool same_f32(double a, double b)
{
  return __float_as_uint(static_cast<float>(a)) == __float_as_uint(static_cast<float>(b));
}

// One thread per member lane: station planes -> member lanes.  Memory bound (reads are broadcasts among the
// members of a station, writes coalesced).
__global__ void rs_ens_fork_kernel(const RsForkArgs f)
{
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= f.ldm) return;
  const size_t ldm = f.ldm, ld = f.ld;
  const bool lane = l < f.npoints * f.members;
  const int p = lane ? l / f.members : 0;
  if (!lane)
  {
    // padding lane: never run (RS_L_ACTIVE = 0), no coupling, no relaxation
    for (int k = 0; k < RS_L_NLOCAL; ++k) f.m_local[k * ldm + l] = 0.0;
    f.m_local[RS_L_SKY_VIEW * ldm + l] = 1.0;
    f.m_local[RS_L_COUPLING_TSURF * ldm + l] = -9999.0;
    f.m_local[RS_L_COUPLING_INDEX * ldm + l] = -9999.0;
    for (int k = 0; k < 3; ++k) f.m_local[(RS_L_TAIR_RELAX + k) * ldm + l] = -9999.0;
    for (int k = 0; k < f.state_planes; ++k) f.m_state[k * ldm + l] = 0.0;
    if (f.m_scratch)
      for (int k = 0; k < f.scratch_planes; ++k) f.m_scratch[k * ldm + l] = 0.0;
    if (f.m_horizons)
      for (int k = 0; k < 360; ++k) f.m_horizons[k * ldm + l] = 0.0;
    if (f.r_f >= 0)
      for (int v = 0; v < f.nvar; ++v) f.m_forcing[v * ldm + l] = 0.0;
    f.m_status[l] = 0;
    return;
  }
  for (int k = 0; k < RS_L_NLOCAL; ++k) f.m_local[k * ldm + l] = __ldg(f.local + k * ld + p);
  double mt[3];
  for (int k = 0; k < 3; ++k)
  {
    mt[k] = f.member_relax ? __ldg(f.member_relax + k * ldm + l) : __ldg(f.local + (RS_L_TAIR_RELAX + k) * ld + p);
    f.m_local[(RS_L_TAIR_RELAX + k) * ldm + l] = mt[k];
  }
  for (int k = 0; k < f.state_planes; ++k) f.m_state[k * ldm + l] = __ldg(f.state + k * ld + p);
  if (f.m_scratch)
    for (int k = 0; k < f.scratch_planes; ++k) f.m_scratch[k * ldm + l] = __ldg(f.scratch + k * ld + p);
  if (f.m_horizons)
    for (int k = 0; k < 360; ++k) f.m_horizons[k * ldm + l] = __ldg(f.horizons + k * ld + p);
  if (f.r_f >= 0)
  {
    const double* rec = f.forcing + static_cast<size_t>(f.r_f) * f.nvar * ld + p;
    for (int v = 0; v < f.nvar; ++v) f.m_forcing[v * ldm + l] = __ldg(rec + v * ld);
  }
  int st = __ldg(f.status + p);
  if (f.relax)
  {
    const bool own = rs_relax_targets_valid(mt[0], mt[1], mt[2]);
    const size_t latch = static_cast<size_t>(f.nlayers) + 2 + RS_SP_LATCH;  // TairInitEnd, VZInitEnd, RhzInitEnd
    if (!own)
      for (int k = 0; k < 3; ++k) f.m_state[(latch + k) * ldm + l] = static_cast<double>(-99.9f);
    const bool real = p < f.npoints && __ldg(f.local + RS_L_ACTIVE * ld + p) != 0.0;
    const int init_len = static_cast<int>(__ldg(f.local + RS_L_INIT_LEN * ld + p));
    if (real && init_len <= f.fork_step - 2)
    {
      // the shared part has applied the prefix copy's targets already
      double ct[3];
      prefix_targets(f.local, f.ld, p, f.member_relax, f.ldm, f.members, ct);
      const bool cv = rs_relax_targets_valid(ct[0], ct[1], ct[2]);
      const bool differs = cv != own || (cv && !(same_f32(ct[0], mt[0]) && same_f32(ct[1], mt[1]) && same_f32(ct[2], mt[2])));
      if (differs)
      {
        st |= RS_ST_BAD_FORK | RS_ST_NOT_RUN;
        // clear the `alive` bit of the flag word: the member launch does not run this lane
        const size_t flag = static_cast<size_t>(f.nlayers) + 2 + RS_SP_FLAGS;
        const int fl = static_cast<int>(f.m_state[flag * ldm + l]);
        f.m_state[flag * ldm + l] = static_cast<double>(fl & ~(1 << RS_FL_ALIVE));
      }
    }
  }
  f.m_status[l] = st;
}

constexpr int kStatsBlock = 64;

// The statistics kernel's part of RsEnsembleStatsSpec (everything before the events): its parameter keeps the
// layout it had before the events were appended to the spec.
struct StatsKernelSpec
{
  int n_quantiles;
  int n_thresholds;
  double quantiles[RS_ENS_MAX_QUANTILES];
  RsEnsembleThreshold thresholds[RS_ENS_MAX_THRESHOLDS];
};
static_assert(offsetof(RsEnsembleStatsSpec, n_events) == sizeof(StatsKernelSpec), "spec prefix");

__device__ __forceinline__ bool valid_value(double x) { return x == x && x > -9000.0; }

// One thread per (station, output slot, plane); the valid member values go to this thread's column of shared
// memory (y[k * kStatsBlock]), in member order, and are sorted there for the quantiles.
__global__ void __launch_bounds__(kStatsBlock) rs_ens_stats_kernel(const double* __restrict__ mout, int out_nvar, int n_slots,
                                                                   int mo_slots, int ldm, int npoints, int members,
                                                                   const StatsKernelSpec spec, double* __restrict__ stats,
                                                                   double* __restrict__ prob, int st_slots, int ld)
{
  extern __shared__ double ens_smem[];
  const long long t = static_cast<long long>(blockIdx.x) * kStatsBlock + threadIdx.x;
  const long long total = static_cast<long long>(npoints) * n_slots * out_nvar;
  if (t >= total) return;
  const int p = static_cast<int>(t % npoints);
  const long long vs = t / npoints;  // v * n_slots + s
  const int s = static_cast<int>(vs % n_slots);
  const int v = static_cast<int>(vs / n_slots);
  double* y = ens_smem + threadIdx.x;
  const double* src = mout + (static_cast<size_t>(v) * mo_slots + s) * ldm + static_cast<size_t>(p) * members;
  int n = 0;
  double sum = 0.0;
  for (int m = 0; m < members; ++m)
  {
    const double x = __ldg(src + m);
    if (!valid_value(x)) continue;
    y[n * kStatsBlock] = x;
    sum = sum + x;
    ++n;
  }
  const double miss = -9999.0;
  const size_t plane = static_cast<size_t>(out_nvar) * st_slots * ld;
  double* o = stats ? stats + (static_cast<size_t>(v) * st_slots + s) * ld + p : nullptr;
  if (n == 0)
  {
    if (o)
    {
      o[0] = 0.0;
      for (int j = 1; j < RS_ENS_NFIXED + spec.n_quantiles; ++j) o[j * plane] = miss;
    }
    if (prob)
      for (int j = 0; j < spec.n_thresholds; ++j)
        if (spec.thresholds[j].plane == v) prob[(static_cast<size_t>(j) * st_slots + s) * ld + p] = miss;
    return;
  }
  const double dn = static_cast<double>(n);
  if (prob)
    for (int j = 0; j < spec.n_thresholds; ++j)
    {
      const RsEnsembleThreshold th = spec.thresholds[j];
      if (th.plane != v) continue;
      int c = 0;
      for (int k = 0; k < n; ++k)
      {
        const double x = y[k * kStatsBlock];
        const bool hit = th.op == RS_ENS_LT ? x < th.value
                         : th.op == RS_ENS_LE ? x <= th.value
                         : th.op == RS_ENS_GT ? x > th.value
                                              : x >= th.value;
        c += hit ? 1 : 0;
      }
      prob[(static_cast<size_t>(j) * st_slots + s) * ld + p] = static_cast<double>(c) / dn;
    }
  if (!o) return;
  const double mean = sum / dn;
  double ss = 0.0, mn = y[0], mx = y[0];
  for (int k = 0; k < n; ++k)
  {
    const double x = y[k * kStatsBlock];
    const double d = x - mean;
    ss = ss + d * d;
    if (x < mn) mn = x;
    if (x > mx) mx = x;
  }
  o[RS_ENS_NVALID * plane] = dn;
  o[RS_ENS_MEAN * plane] = mean;
  o[RS_ENS_STD * plane] = sqrt(ss / dn);
  o[RS_ENS_MIN * plane] = mn;
  o[RS_ENS_MAX * plane] = mx;
  if (spec.n_quantiles == 0) return;
  // insertion sort (n <= RS_ENS_MAX_MEMBERS)
  for (int k = 1; k < n; ++k)
  {
    const double x = y[k * kStatsBlock];
    int j = k - 1;
    while (j >= 0 && y[j * kStatsBlock] > x)
    {
      y[(j + 1) * kStatsBlock] = y[j * kStatsBlock];
      --j;
    }
    y[(j + 1) * kStatsBlock] = x;
  }
  for (int j = 0; j < spec.n_quantiles; ++j)
  {
    const double h = static_cast<double>(n - 1) * spec.quantiles[j];
    const int i = static_cast<int>(floor(h));
    const double tt = h - static_cast<double>(i);
    const double yi = y[i * kStatsBlock];
    o[(RS_ENS_NFIXED + j) * plane] = (tt == 0.0 || i == n - 1) ? yi : yi + tt * (y[(i + 1) * kStatsBlock] - yi);
  }
}

constexpr int kEventsBlock = 64;
// Threads the event launch aims for before it splits the slots into tiles (about one resident wave on the B200).
constexpr long long kEventsTargetThreads = 1LL << 17;

// Event probabilities (RsEnsembleEvent).  A block is 64 stations of one event and one tile of output slots
// [s0, s1); the event index varies fastest over the blocks, so that the events of a station block run side by
// side and share the member values through L2.  Each thread scans the slots backward from the end of the tile's
// last window, min(s1 + window - 1, S), down to s0, and loops over the members at each slot, reading every member
// value of a referenced plane once per event and tile.  Per member it keeps, in its column of shared memory
// (st[m * kEventsBlock]), the first slot >= s with an invalid value (x) and the first with a valid hit (y); the
// window W(s) = [s, wend] is then valid when x > wend and hits when also y <= wend.
__global__ void __launch_bounds__(kEventsBlock) rs_ens_events_kernel(const double* __restrict__ mout, int n_slots, int mo_slots,
                                                                     int ldm, int npoints, int members, int n_events, int tile,
                                                                     const RsEnsembleStatsSpec spec, double* __restrict__ prob,
                                                                     int st_slots, int ld)
{
  extern __shared__ int2 ev_smem[];
  const int station_blocks = (npoints + kEventsBlock - 1) / kEventsBlock;
  const int e = static_cast<int>(blockIdx.x % n_events);
  const int rest = static_cast<int>(blockIdx.x / n_events);
  const int p = (rest % station_blocks) * kEventsBlock + threadIdx.x;
  const int s0 = (rest / station_blocks) * tile;
  if (p >= npoints) return;
  const RsEnsembleEvent& ev = spec.events[e];
  const int nc = ev.n_conditions, w = ev.window;
  const double* src[RS_ENS_MAX_CONDITIONS];
  int op[RS_ENS_MAX_CONDITIONS];
  double val[RS_ENS_MAX_CONDITIONS];
#pragma unroll
  for (int c = 0; c < RS_ENS_MAX_CONDITIONS; ++c)
  {
    const RsEnsembleThreshold th = ev.conditions[c < nc ? c : 0];
    src[c] = mout + static_cast<size_t>(th.plane) * mo_slots * ldm + static_cast<size_t>(p) * members;
    op[c] = th.op;
    val[c] = th.value;
  }
  const int s1 = tile >= n_slots - s0 ? n_slots : s0 + tile;
  const int s_end = w - 1 >= n_slots - s1 ? n_slots : s1 + w - 1;  // the last window of the tile ends at s_end - 1
  int2* st = ev_smem + threadIdx.x;
  for (int m = 0; m < members; ++m) st[m * kEventsBlock] = make_int2(INT_MAX, INT_MAX);
  const size_t out_base = (static_cast<size_t>(spec.n_thresholds) + e) * st_slots;
  for (int s = s_end - 1; s >= s0; --s)
  {
    const size_t off = static_cast<size_t>(s) * ldm;
    const int wend = w - 1 >= n_slots - 1 - s ? n_slots - 1 : s + w - 1;
    int n = 0, count = 0;
#pragma unroll 4
    for (int m = 0; m < members; ++m)
    {
      bool ok = true, hit = true;
#pragma unroll
      for (int c = 0; c < RS_ENS_MAX_CONDITIONS; ++c)
        if (c < nc)
        {
          const double x = __ldg(src[c] + off + m);
          const double v = val[c];
          ok &= valid_value(x);
          hit &= op[c] == RS_ENS_LT ? x < v : op[c] == RS_ENS_LE ? x <= v : op[c] == RS_ENS_GT ? x > v : x >= v;
        }
      int2 t = st[m * kEventsBlock];
      if (!ok)
        t.x = s;
      else if (hit)
        t.y = s;
      st[m * kEventsBlock] = t;
      const bool valid = t.x > wend;
      n += valid ? 1 : 0;
      count += (valid && t.y <= wend) ? 1 : 0;
    }
    if (s < s1)
      prob[(out_base + s) * ld + p] = n == 0 ? -9999.0 : static_cast<double>(count) / static_cast<double>(n);
  }
}
}  // namespace

int rs_launch_ens_prefix_local(const double* local, int ld, int npoints, const double* member_relax, int ldm,
                               int members, int relax, double* work, void* stream)
{
  rs_ens_prefix_local_kernel<<<(ld + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      local, ld, npoints, member_relax, ldm, members, relax, work);
  return static_cast<int>(cudaGetLastError());
}

int rs_launch_ens_fork(const RsForkArgs* f, void* stream)
{
  rs_ens_fork_kernel<<<(f->ldm + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(*f);
  return static_cast<int>(cudaGetLastError());
}

int rs_launch_ens_stats(const double* member_out, int out_nvar, int n_slots, int mo_slots, int ldm, int npoints,
                        int members, const RsEnsembleStatsSpec* spec, double* stats, double* prob, int st_slots, int ld,
                        void* stream)
{
  const long long total = static_cast<long long>(npoints) * n_slots * out_nvar;
  if (total == 0) return 0;
  const int smem = static_cast<int>(sizeof(double)) * kStatsBlock * members;
  cudaError_t e = cudaFuncSetAttribute(rs_ens_stats_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return static_cast<int>(e);
  const long long blocks = (total + kStatsBlock - 1) / kStatsBlock;
  StatsKernelSpec ks;
  std::memcpy(&ks, spec, sizeof ks);
  rs_ens_stats_kernel<<<static_cast<unsigned>(blocks), kStatsBlock, smem, static_cast<cudaStream_t>(stream)>>>(
      member_out, out_nvar, n_slots, mo_slots, ldm, npoints, members, ks, stats, prob, st_slots, ld);
  return static_cast<int>(cudaGetLastError());
}

int rs_launch_ens_events(const double* member_out, int n_slots, int mo_slots, int ldm, int npoints, int members,
                         const RsEnsembleStatsSpec* spec, double* prob, int st_slots, int ld, void* stream)
{
  const int E = spec->n_events;
  if (E == 0 || npoints == 0 || n_slots == 0) return 0;
  // One tile of all slots per thread where P * n_events threads fill the GPU; else tiles of at least 32 slots and
  // four look-aheads (window - 1), so that a tile's look-ahead re-reads at most a quarter of it.
  long long tile = n_slots;
  const long long want_tiles = (kEventsTargetThreads + static_cast<long long>(npoints) * E - 1) / (static_cast<long long>(npoints) * E);
  if (want_tiles > 1)
  {
    long long wmax = 1;
    for (int j = 0; j < E; ++j) wmax = std::max<long long>(wmax, spec->events[j].window);
    tile = std::min<long long>(n_slots, std::max({(n_slots + want_tiles - 1) / want_tiles, 4 * (wmax - 1), 32LL}));
  }
  const long long tiles = (n_slots + tile - 1) / tile;
  const long long blocks = static_cast<long long>(E) * ((npoints + kEventsBlock - 1) / kEventsBlock) * tiles;
  const int smem = static_cast<int>(sizeof(int2)) * kEventsBlock * members;
  cudaError_t e = cudaFuncSetAttribute(rs_ens_events_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return static_cast<int>(e);
  rs_ens_events_kernel<<<static_cast<unsigned>(blocks), kEventsBlock, smem, static_cast<cudaStream_t>(stream)>>>(
      member_out, n_slots, mo_slots, ldm, npoints, members, E, static_cast<int>(tile), *spec, prob, st_slots, ld);
  return static_cast<int>(cudaGetLastError());
}
