// rs_ensemble.cu -- the kernels of an ensemble run (roadsurf_run_ensemble_device): the prefix's copy of the
// station statics, the fork of the station state into the member lanes, the ensemble statistics, the event
// probabilities, the area event probabilities, the event onset and the window extremes.
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

// Area event probabilities (RsEnsembleAreas), step 1: the stations of one chunk into the accumulators.  A work item
// is one (segment, event, tile of kRsAreaTile slots); the event index varies fastest, so that the events of a segment
// run side by side and share its member values through L2.  A block holds blockDim.y items, each of 32 * ceil(M / 32)
// threads, one per member.  Per station of the segment a thread scans the tile and its look-ahead backward once,
// keeping the next invalid slot (nx) and the next hit slot (ny) of its member in registers, and sets bit s - s0 of
// the station's masks where W(s) is valid, and valid with a hit.  The masks are ANDed (valid) and ORed (hit) over
// the segment, then once into the accumulators [area][event][tile][member] with atomicAnd / atomicOr.  AND and OR
// are exact whatever the order, so the result does not depend on chunks, segments, tiles or launch geometry.
__global__ void __launch_bounds__(kRsAreaBlock) rs_ens_area_accumulate_kernel(
    const double* __restrict__ mout, int n_slots, int mo_slots, int ldm, int members, int n_events, int tiles,
    long long n_items, const RsEnsembleStatsSpec spec, const int* __restrict__ stations, int p0,
    const int4* __restrict__ segments, unsigned long long* __restrict__ acc_valid, unsigned long long* __restrict__ acc_hit)
{
  const long long item = static_cast<long long>(blockIdx.x) * blockDim.y + threadIdx.y;
  const int m = threadIdx.x;
  if (item >= n_items || m >= members) return;
  const int e = static_cast<int>(item % n_events);
  const long long rest = item / n_events;
  const int t = static_cast<int>(rest % tiles);
  const int4 seg = __ldg(segments + rest / tiles);  // area, first and end index into `stations`
  const RsEnsembleEvent& ev = spec.events[e];
  const int nc = ev.n_conditions, w = ev.window;
  const double* src[RS_ENS_MAX_CONDITIONS];
  int op[RS_ENS_MAX_CONDITIONS];
  double val[RS_ENS_MAX_CONDITIONS];
#pragma unroll
  for (int c = 0; c < RS_ENS_MAX_CONDITIONS; ++c)
  {
    const RsEnsembleThreshold th = ev.conditions[c < nc ? c : 0];
    src[c] = mout + static_cast<size_t>(th.plane) * mo_slots * ldm + m;
    op[c] = th.op;
    val[c] = th.value;
  }
  const int s0 = t * kRsAreaTile;
  const int s1 = kRsAreaTile >= n_slots - s0 ? n_slots : s0 + kRsAreaTile;
  const int s_end = w - 1 >= n_slots - s1 ? n_slots : s1 + w - 1;  // the last window of the tile ends at s_end - 1
  unsigned long long valid = ~0ULL, hit = 0;
  for (int k = seg.y; k < seg.z; ++k)
  {
    const size_t lane = static_cast<size_t>(__ldg(stations + k) - p0) * members;
    int nx = INT_MAX, ny = INT_MAX;
    unsigned long long vm = 0, hm = 0;
#pragma unroll 4
    for (int s = s_end - 1; s >= s0; --s)
    {
      const size_t off = static_cast<size_t>(s) * ldm + lane;
      bool ok = true, h = true;
#pragma unroll
      for (int c = 0; c < RS_ENS_MAX_CONDITIONS; ++c)
        if (c < nc)
        {
          const double x = __ldg(src[c] + off);
          const double v = val[c];
          ok &= valid_value(x);
          h &= op[c] == RS_ENS_LT ? x < v : op[c] == RS_ENS_LE ? x <= v : op[c] == RS_ENS_GT ? x > v : x >= v;
        }
      if (!ok)
        nx = s;
      else if (h)
        ny = s;
      if (s < s1)
      {
        const int wend = w - 1 >= n_slots - 1 - s ? n_slots - 1 : s + w - 1;
        const unsigned long long bit = 1ULL << (s - s0);
        if (nx > wend)
        {
          vm |= bit;
          if (ny <= wend) hm |= bit;
        }
      }
    }
    valid &= vm;
    hit |= hm;
  }
  const size_t a = ((static_cast<size_t>(seg.x) * n_events + e) * tiles + t) * members + m;
  atomicAnd(acc_valid + a, valid);
  atomicOr(acc_hit + a, hit);
}

// Step 2, once after the last chunk: one block per (area, event, tile), one thread per member.  Per slot of the tile,
// a warp ballot and __popc count the members whose valid bit is set and those whose hit bit is set too; the warps'
// counts are summed in shared memory and one thread per slot writes area_prob[e][s][a].
__global__ void __launch_bounds__(kRsAreaBlock) rs_ens_area_finalize_kernel(
    const unsigned long long* __restrict__ acc_valid, const unsigned long long* __restrict__ acc_hit, int n_areas,
    int n_events, int tiles, int n_slots, int members, double* __restrict__ area_prob, int st_slots)
{
  __shared__ int counts[2][kRsAreaBlock / 32][kRsAreaTile];
  const long long b = blockIdx.x;  // (a * n_events + e) * tiles + t
  const int t = static_cast<int>(b % tiles), e = static_cast<int>((b / tiles) % n_events);
  const int a = static_cast<int>(b / (static_cast<long long>(tiles) * n_events));
  const int m = threadIdx.x, warp = m / 32, warps = blockDim.x / 32;
  unsigned long long v = 0, h = 0;
  if (m < members)
  {
    v = acc_valid[static_cast<size_t>(b) * members + m];
    h = acc_hit[static_cast<size_t>(b) * members + m] & v;
  }
  for (int j = 0; j < kRsAreaTile; ++j)
  {
    const unsigned bv = __ballot_sync(0xffffffffu, (v >> j) & 1ULL), bh = __ballot_sync(0xffffffffu, (h >> j) & 1ULL);
    if ((m & 31) == 0)
    {
      counts[0][warp][j] = __popc(bv);
      counts[1][warp][j] = __popc(bh);
    }
  }
  __syncthreads();
  const int s0 = t * kRsAreaTile;
  for (int j = m; j < kRsAreaTile && s0 + j < n_slots; j += blockDim.x)
  {
    int n = 0, count = 0;
    for (int k = 0; k < warps; ++k)
    {
      n += counts[0][k][j];
      count += counts[1][k][j];
    }
    area_prob[(static_cast<size_t>(e) * st_slots + s0 + j) * n_areas + a] =
        n == 0 ? -9999.0 : static_cast<double>(count) / static_cast<double>(n);
  }
}

// Items of one (member-)thread group per block: as many as fill kRsAreaBlock threads.
inline int area_groups(int members) { return kRsAreaBlock / (32 * ((members + 31) / 32)); }

constexpr int kOnsetStations = 64;  // stations of an onset block
constexpr int kOnsetBlock = 256;

// Event onset (roadsurf_ensemble_onset).  A block is one event and kOnsetStations stations; the event index varies
// fastest over the blocks, so that the events of a station block run side by side and share the member values
// through L2.  Step 1: thread t scans the member lanes t, t + kOnsetBlock, ... of the block's stations forward from
// slot 0 and stops at X, the first slot where a named plane is invalid (n_slots if none), keeping O, the first slot
// before X where the conditions all hold (n_slots if none).  Consecutive threads read consecutive lanes, and each
// member value is read at most once.  {O, X} goes to the workspace ws[e][lane] (areas) and to shared memory
// (os[m * kOnsetStations + station]).  Step 2 (onset planes): a thread per (slot, station), the station varying
// fastest, counts the members with X > s (valid) and with O <= s too (hit) and writes onset[e][s][p], so that the
// writes of a warp are consecutive stations of one plane row.
__global__ void __launch_bounds__(kOnsetBlock) rs_ens_onset_kernel(const double* __restrict__ mout, int n_slots, int mo_slots,
                                                                   int ldm, int npoints, int members, int n_events,
                                                                   const RsEnsembleStatsSpec spec, double* __restrict__ onset,
                                                                   int st_slots, int ld, int2* __restrict__ ws)
{
  extern __shared__ int2 os_smem[];
  const int e = static_cast<int>(blockIdx.x % n_events);
  const int pb = static_cast<int>(blockIdx.x / n_events) * kOnsetStations;
  const int nst = min(kOnsetStations, npoints - pb);
  const RsEnsembleEvent& ev = spec.events[e];
  const int nc = ev.n_conditions;
  const double* src[RS_ENS_MAX_CONDITIONS];
  int op[RS_ENS_MAX_CONDITIONS];
  double val[RS_ENS_MAX_CONDITIONS];
#pragma unroll
  for (int c = 0; c < RS_ENS_MAX_CONDITIONS; ++c)
  {
    const RsEnsembleThreshold th = ev.conditions[c < nc ? c : 0];
    src[c] = mout + static_cast<size_t>(th.plane) * mo_slots * ldm + static_cast<size_t>(pb) * members;
    op[c] = th.op;
    val[c] = th.value;
  }
  const int lanes = nst * members;
  for (int l = threadIdx.x; l < lanes; l += kOnsetBlock)
  {
    int x = n_slots, o = n_slots;
    for (int s = 0; s < n_slots; ++s)
    {
      const size_t off = static_cast<size_t>(s) * ldm + l;
      bool ok = true, hit = true;
#pragma unroll
      for (int c = 0; c < RS_ENS_MAX_CONDITIONS; ++c)
        if (c < nc)
        {
          const double v = __ldg(src[c] + off);
          ok &= valid_value(v);
          hit &= op[c] == RS_ENS_LT ? v < val[c] : op[c] == RS_ENS_LE ? v <= val[c] : op[c] == RS_ENS_GT ? v > val[c] : v >= val[c];
        }
      if (!ok)
      {
        x = s;
        break;
      }
      if (hit && o == n_slots) o = s;
    }
    if (ws) ws[static_cast<size_t>(e) * npoints * members + static_cast<size_t>(pb) * members + l] = make_int2(o, x);
    if (onset) os_smem[(l % members) * kOnsetStations + l / members] = make_int2(o, x);
  }
  if (!onset) return;
  __syncthreads();
  for (int i = threadIdx.x; i < nst * n_slots; i += kOnsetBlock)
  {
    const int q = i % nst, s = i / nst;
    int n = 0, count = 0;
    for (int m = 0; m < members; ++m)
    {
      const int2 t = os_smem[m * kOnsetStations + q];
      const bool valid = t.y > s;
      n += valid ? 1 : 0;
      count += (valid && t.x <= s) ? 1 : 0;
    }
    onset[(static_cast<size_t>(e) * st_slots + s) * ld + pb + q] =
        n == 0 ? -9999.0 : static_cast<double>(count) / static_cast<double>(n);
  }
}

// Area onset, step 1: the stations of one chunk into the accumulators.  A work item is one (segment, event), the
// event varying fastest; a block holds blockDim.y items of 32 * ceil(M / 32) threads, one per member.  A thread takes
// the minimum O and the minimum X of its member over the segment's stations from the workspace, then one atomicMin
// each into acc[area][event][member] = {O, X}.  The minimum is exact whatever the order, so the result does not
// depend on chunks, segments or launch geometry.
__global__ void __launch_bounds__(kRsAreaBlock) rs_ens_area_onset_accumulate_kernel(
    const int2* __restrict__ ws, int lanes, int members, int n_events, long long n_items, const int* __restrict__ stations,
    int p0, const int4* __restrict__ segments, int* __restrict__ acc)
{
  const long long item = static_cast<long long>(blockIdx.x) * blockDim.y + threadIdx.y;
  const int m = threadIdx.x;
  if (item >= n_items || m >= members) return;
  const int e = static_cast<int>(item % n_events);
  const int4 seg = __ldg(segments + item / n_events);  // area, first and end index into `stations`
  const int2* w = ws + static_cast<size_t>(e) * lanes + m;
  int o = INT_MAX, x = INT_MAX;
  for (int k = seg.y; k < seg.z; ++k)
  {
    const int2 t = __ldg(w + static_cast<size_t>(__ldg(stations + k) - p0) * members);
    o = min(o, t.x);
    x = min(x, t.y);
  }
  int* a = acc + 2 * ((static_cast<size_t>(seg.x) * n_events + e) * members + m);
  atomicMin(a, o);
  atomicMin(a + 1, x);
}

// Area onset, step 2, once after the last chunk: one thread per (event, slot, area), the area varying fastest, counts
// the members with X > s (valid) and with O <= s too (hit) and writes area_onset[e][s][a].
__global__ void __launch_bounds__(kRsAreaBlock) rs_ens_area_onset_finalize_kernel(
    const int* __restrict__ acc, int n_areas, int n_events, int n_slots, int members, double* __restrict__ area_onset,
    int st_slots)
{
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(n_areas) * n_slots * n_events) return;
  const int a = static_cast<int>(i % n_areas);
  const int s = static_cast<int>((i / n_areas) % n_slots);
  const int e = static_cast<int>(i / (static_cast<long long>(n_areas) * n_slots));
  const int2* t = reinterpret_cast<const int2*>(acc) + (static_cast<size_t>(a) * n_events + e) * members;
  int n = 0, count = 0;
  for (int m = 0; m < members; ++m)
  {
    const int2 v = __ldg(t + m);
    const bool valid = v.y > s;
    n += valid ? 1 : 0;
    count += (valid && v.x <= s) ? 1 : 0;
  }
  area_onset[(static_cast<size_t>(e) * st_slots + s) * n_areas + a] =
      n == 0 ? -9999.0 : static_cast<double>(count) / static_cast<double>(n);
}

// Window extremes (roadsurf_ensemble_extremes) compare keys: the header's order-preserving int64 map of a double's
// bits with its sign bit flipped, an order-preserving map to uint64, so that -0.0 < +0.0.  An invalid value is the
// absorbing element of the order (0 for the minimum, ~0 for the maximum) and the identity is the other end, so that
// validity falls out of the same combine.  No valid value has either key (both are NaN bit patterns).
__device__ __forceinline__ unsigned long long ext_key(double v, bool lo)
{
  if (!valid_value(v)) return lo ? 0ULL : ~0ULL;
  const unsigned long long b = static_cast<unsigned long long>(__double_as_longlong(v));
  return (b >> 63) ? ~b : b | (1ULL << 63);
}

__device__ __forceinline__ unsigned long long ext_combine(unsigned long long a, unsigned long long b, bool lo)
{
  return lo ? (b < a ? b : a) : (b > a ? b : a);
}

// The double of a key, as raw bits; -9999.0 for the absorbing element.
__device__ __forceinline__ unsigned long long ext_bits(unsigned long long k, bool lo)
{
  if (k == (lo ? 0ULL : ~0ULL)) return static_cast<unsigned long long>(__double_as_longlong(-9999.0));
  return (k >> 63) ? k & ~(1ULL << 63) : ~k;
}

constexpr int kExtBlock = 256;

// Station window extremes: one thread per (extreme, member lane), blockIdx.y the extreme and the lanes fastest, so that
// every warp access is one row of consecutive lanes.  Van Herk / Gil-Werman over blocks of w = min(window, S) slots:
// a backward pass writes each slot's suffix extreme within its block into ws; a forward pass keeps the prefix extreme
// of the current block and, at t = s + w - 1, combines it with the suffix of s (W(s) = s's suffix alone where s starts
// a block) and writes the value of W(s); the windows cut at S combine with the prefix of the last block at the end.
// Each member value is read twice and each ws value written twice and read once, whatever the window.
__global__ void __launch_bounds__(kExtBlock) rs_ens_window_extremes_kernel(const double* __restrict__ mout, int n_slots,
                                                                           int mo_slots, int ldm, int lanes,
                                                                           const RsEnsembleExtremes ext,
                                                                           unsigned long long* __restrict__ ws, int ldw)
{
  const int l = blockIdx.x * kExtBlock + threadIdx.x;
  if (l >= lanes) return;
  const RsEnsembleExtreme xt = ext.extremes[blockIdx.y];
  const bool lo = xt.kind == RS_ENS_WMIN;
  const int S = n_slots, w = min(xt.window, S);
  const double* src = mout + static_cast<size_t>(xt.plane) * mo_slots * ldm + l;
  unsigned long long* out = ws + static_cast<size_t>(blockIdx.y) * S * ldw + l;
  const unsigned long long id = lo ? ~0ULL : 0ULL;
  unsigned long long acc = id;
  for (int t = S - 1; t >= 0; --t)
  {
    if (t % w == w - 1) acc = id;
    acc = ext_combine(acc, ext_key(__ldg(src + static_cast<size_t>(t) * ldm), lo), lo);
    out[static_cast<size_t>(t) * ldw] = acc;
  }
  acc = id;
  for (int t = 0; t < S; ++t)
  {
    if (t % w == 0) acc = id;
    acc = ext_combine(acc, ext_key(__ldg(src + static_cast<size_t>(t) * ldm), lo), lo);
    const int s = t - w + 1;
    if (s < 0) continue;
    unsigned long long* o = out + static_cast<size_t>(s) * ldw;
    *o = ext_bits(s % w == 0 ? *o : ext_combine(*o, acc, lo), lo);
  }
  const int last_block = (S - 1) / w * w;  // first slot of the last block
  for (int s = max(0, S - w + 1); s < S; ++s)
  {
    unsigned long long* o = out + static_cast<size_t>(s) * ldw;
    *o = ext_bits(s < last_block ? ext_combine(*o, acc, lo) : *o, lo);
  }
}

// Area window extremes, step 1: the stations of one chunk into the accumulators.  A work item is one (segment,
// extreme), the extreme varying fastest; a block holds blockDim.y items of 32 * ceil(M / 32) threads, one per member.
// Per slot a thread combines its member's station extremes (ws, station p at lane (p - p0) * members + m) over the
// segment in key space and makes one atomicMin (minimum) or atomicMax (maximum) into acc[x][s][area * members + m].
// Both are exact whatever the order, so the result does not depend on chunks, segments or launch geometry.
__global__ void __launch_bounds__(kRsAreaBlock) rs_ens_area_extremes_accumulate_kernel(
    const double* __restrict__ ws, int n_slots, int ldw, int members, long long n_items, int n_extremes,
    unsigned min_mask, const int* __restrict__ stations, int p0, const int4* __restrict__ segments, int n_areas,
    unsigned long long* __restrict__ acc)
{
  const long long item = static_cast<long long>(blockIdx.x) * blockDim.y + threadIdx.y;
  const int m = threadIdx.x;
  if (item >= n_items || m >= members) return;
  const int x = static_cast<int>(item % n_extremes);
  const int4 seg = __ldg(segments + item / n_extremes);  // area, first and end index into `stations`
  const bool lo = (min_mask >> x) & 1u;
  const double* src = ws + static_cast<size_t>(x) * n_slots * ldw + m;
  const size_t row = static_cast<size_t>(n_areas) * members;
  unsigned long long* dst = acc + static_cast<size_t>(x) * n_slots * row + static_cast<size_t>(seg.x) * members + m;
  for (int s = 0; s < n_slots; ++s)
  {
    unsigned long long v = lo ? ~0ULL : 0ULL;
    for (int k = seg.y; k < seg.z; ++k)
      v = ext_combine(v, ext_key(__ldg(src + static_cast<size_t>(s) * ldw + static_cast<size_t>(__ldg(stations + k) - p0) * members), lo), lo);
    if (lo)
      atomicMin(dst + s * row, v);
    else
      atomicMax(dst + s * row, v);
  }
}

// Area window extremes, step 2, once after the last chunk: the keys of acc [n_extremes][per_extreme] back to doubles
// in place, -9999.0 where a member is not valid for the area.
__global__ void __launch_bounds__(kRsAreaBlock) rs_ens_area_extremes_finalize_kernel(unsigned long long* __restrict__ acc,
                                                                                     long long per_extreme,
                                                                                     int n_extremes, unsigned min_mask)
{
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= per_extreme * n_extremes) return;
  acc[i] = ext_bits(acc[i], (min_mask >> (i / per_extreme)) & 1u);
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

int rs_launch_ens_area_accumulate(const double* member_out, int n_slots, int mo_slots, int ldm, int members,
                                  const RsEnsembleStatsSpec* spec, const int* stations, int p0, const int* segments,
                                  int n_segments, unsigned long long* acc_valid, unsigned long long* acc_hit, void* stream)
{
  const int E = spec->n_events, tiles = rs_area_tiles(n_slots);
  if (E == 0 || n_segments == 0 || n_slots == 0) return 0;
  const int groups = area_groups(members);
  const long long items = static_cast<long long>(n_segments) * E * tiles;
  const dim3 block(32 * ((members + 31) / 32), groups);
  rs_ens_area_accumulate_kernel<<<static_cast<unsigned>((items + groups - 1) / groups), block, 0,
                                  static_cast<cudaStream_t>(stream)>>>(
      member_out, n_slots, mo_slots, ldm, members, E, tiles, items, *spec, stations, p0,
      reinterpret_cast<const int4*>(segments), acc_valid, acc_hit);
  return static_cast<int>(cudaGetLastError());
}

int rs_launch_ens_area_finalize(const unsigned long long* acc_valid, const unsigned long long* acc_hit, int n_areas,
                                int n_events, int n_slots, int members, double* area_prob, int st_slots, void* stream)
{
  const int tiles = rs_area_tiles(n_slots);
  if (n_events == 0 || n_areas == 0 || n_slots == 0) return 0;
  const long long blocks = static_cast<long long>(n_areas) * n_events * tiles;
  rs_ens_area_finalize_kernel<<<static_cast<unsigned>(blocks), 32 * ((members + 31) / 32), 0,
                                static_cast<cudaStream_t>(stream)>>>(acc_valid, acc_hit, n_areas, n_events, tiles,
                                                                     n_slots, members, area_prob, st_slots);
  return static_cast<int>(cudaGetLastError());
}

int rs_launch_ens_onset(const double* member_out, int n_slots, int mo_slots, int ldm, int npoints, int members,
                        const RsEnsembleStatsSpec* spec, double* onset, int st_slots, int ld, int* ws, void* stream)
{
  const int E = spec->n_events;
  if (E == 0 || npoints == 0 || n_slots == 0 || (!onset && !ws)) return 0;
  const long long blocks = static_cast<long long>(E) * ((npoints + kOnsetStations - 1) / kOnsetStations);
  const int smem = onset ? static_cast<int>(sizeof(int2)) * kOnsetStations * members : 0;
  cudaError_t e = cudaFuncSetAttribute(rs_ens_onset_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return static_cast<int>(e);
  rs_ens_onset_kernel<<<static_cast<unsigned>(blocks), kOnsetBlock, smem, static_cast<cudaStream_t>(stream)>>>(
      member_out, n_slots, mo_slots, ldm, npoints, members, E, *spec, onset, st_slots, ld, reinterpret_cast<int2*>(ws));
  return static_cast<int>(cudaGetLastError());
}

int rs_launch_ens_area_onset_accumulate(const int* ws, int npoints, int members, int n_events, const int* stations, int p0,
                                        const int* segments, int n_segments, int* acc, void* stream)
{
  if (n_events == 0 || n_segments == 0) return 0;
  const int groups = area_groups(members);
  const long long items = static_cast<long long>(n_segments) * n_events;
  const dim3 block(32 * ((members + 31) / 32), groups);
  rs_ens_area_onset_accumulate_kernel<<<static_cast<unsigned>((items + groups - 1) / groups), block, 0,
                                        static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const int2*>(ws), npoints * members, members, n_events, items, stations, p0,
      reinterpret_cast<const int4*>(segments), acc);
  return static_cast<int>(cudaGetLastError());
}

int rs_launch_ens_area_onset_finalize(const int* acc, int n_areas, int n_events, int n_slots, int members,
                                      double* area_onset, int st_slots, void* stream)
{
  const long long total = static_cast<long long>(n_areas) * n_slots * n_events;
  if (total == 0) return 0;
  rs_ens_area_onset_finalize_kernel<<<static_cast<unsigned>((total + kRsAreaBlock - 1) / kRsAreaBlock), kRsAreaBlock, 0,
                                      static_cast<cudaStream_t>(stream)>>>(acc, n_areas, n_events, n_slots, members,
                                                                           area_onset, st_slots);
  return static_cast<int>(cudaGetLastError());
}

// Bit x set where extreme x is a minimum.
static unsigned min_mask(const RsEnsembleExtremes* ext)
{
  unsigned m = 0;
  for (int x = 0; x < ext->n_extremes; ++x) m |= (ext->extremes[x].kind == RS_ENS_WMIN ? 1u : 0u) << x;
  return m;
}

int rs_launch_ens_window_extremes(const double* member_out, int n_slots, int mo_slots, int ldm, int lanes,
                                  const RsEnsembleExtremes* ext, double* ws, int ldw, void* stream)
{
  if (n_slots == 0 || lanes == 0) return 0;
  const dim3 grid((lanes + kExtBlock - 1) / kExtBlock, ext->n_extremes);
  rs_ens_window_extremes_kernel<<<grid, kExtBlock, 0, static_cast<cudaStream_t>(stream)>>>(
      member_out, n_slots, mo_slots, ldm, lanes, *ext, reinterpret_cast<unsigned long long*>(ws), ldw);
  return static_cast<int>(cudaGetLastError());
}

int rs_launch_ens_area_extremes_accumulate(const double* ws, int n_slots, int ldw, int members,
                                           const RsEnsembleExtremes* ext, const int* stations, int p0,
                                           const int* segments, int n_segments, int n_areas, double* acc, void* stream)
{
  if (n_segments == 0 || n_slots == 0) return 0;
  const int groups = area_groups(members);
  const long long items = static_cast<long long>(n_segments) * ext->n_extremes;
  const dim3 block(32 * ((members + 31) / 32), groups);
  rs_ens_area_extremes_accumulate_kernel<<<static_cast<unsigned>((items + groups - 1) / groups), block, 0,
                                           static_cast<cudaStream_t>(stream)>>>(
      ws, n_slots, ldw, members, items, ext->n_extremes, min_mask(ext), stations, p0, reinterpret_cast<const int4*>(segments), n_areas,
      reinterpret_cast<unsigned long long*>(acc));
  return static_cast<int>(cudaGetLastError());
}

int rs_launch_ens_area_extremes_finalize(double* acc, int n_slots, int n_areas, int members,
                                         const RsEnsembleExtremes* ext, void* stream)
{
  const long long per_extreme = static_cast<long long>(n_slots) * n_areas * members;
  if (per_extreme == 0) return 0;
  const long long total = per_extreme * ext->n_extremes;
  rs_ens_area_extremes_finalize_kernel<<<static_cast<unsigned>((total + kRsAreaBlock - 1) / kRsAreaBlock), kRsAreaBlock,
                                         0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<unsigned long long*>(acc), per_extreme, ext->n_extremes, min_mask(ext));
  return static_cast<int>(cudaGetLastError());
}

int rs_init_ens_area_extremes(double* acc, int n_slots, int n_areas, int members, const RsEnsembleExtremes* ext,
                              void* stream)
{
  const size_t bytes = sizeof(double) * n_slots * n_areas * members;
  for (int x = 0; x < ext->n_extremes; ++x)
  {
    const cudaError_t e = cudaMemsetAsync(reinterpret_cast<char*>(acc) + x * bytes,
                                          ext->extremes[x].kind == RS_ENS_WMIN ? 0xff : 0, bytes,
                                          static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return static_cast<int>(e);
  }
  return 0;
}
