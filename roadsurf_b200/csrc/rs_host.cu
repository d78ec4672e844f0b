// rs_host.cu -- the C ABI of libroadsurf_b200.so (include/roadsurf_b200.h): model upload, the
// device-resident launch, the batched host entry (pack -> H2D -> kernel -> D2H -> unpack, sharded
// over GPUs) and the reference's single-point `runsimulation`.
//
// There is no CPU implementation of the model in this library: every entry point either runs the
// CUDA kernel or returns an error.
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "rs_ensemble.cuh"
#include "rs_kernel.cuh"
#include "rs_libm.h"

namespace
{
// Slots of the pooled work space (pooled / pooled_pinned below), grouped by entry.  An entry holds its device's
// g_device_mu while it uses its buffers, so the entries of one device never run at the same time: a slot only
// needs to be unique within one entry and its second buffer set.  Device and pinned buffers are separate pools.
enum PoolSlot : int
{
  // run_shard (roadsurf_run_batch, runsimulation): the second buffer set adds RB_SET2 (except RB_TIME_FIELDS, RB_SOLAR)
  RB_FORCING = 200, RB_OUT = 201, RB_LOCAL = 202, RB_HOR = 203, RB_STATUS = 204, RB_SCRATCH = 205, RB_STAGE = 206,
  RB_STAGE2 = 207, RB_COUNTERS = 208, RB_TIME_FIELDS = 209, RB_SOLAR = 210, RB_STATE = 211, RB_NVIS = 212,
  RB_SET2 = 50,
  RB_H_STAGE = 0, RB_H_STAGE2 = 1, RB_H_LOCAL = 2, RB_H_HOR = 3, RB_H_STATUS = 4,  // pinned
  // run_host_soa_shard (roadsurf_run_host_soa): the buffers of stream s add s * HS_STREAM
  HS_FORCING = 0, HS_OUT = 1, HS_LOCAL = 2, HS_HOR = 3, HS_SCRATCH = 4, HS_STATUS = 5, HS_STATE = 6, HS_ORDER = 7,
  HS_STREAM = 10,
  HS_TIME_FIELDS = 100, HS_RECORD_STEP = 101, HS_COUNTERS = 102, HS_SOLAR = 103,
  // roadsurf_run_ensemble_host_soa (EH_M_*: member lanes)
  EH_FORCING = 400, EH_LOCAL = 401, EH_HOR = 402, EH_OUT = 403, EH_STATE = 404, EH_SCRATCH = 405, EH_M_FORCING = 406,
  EH_M_LOCAL = 407, EH_M_HOR = 408, EH_M_STATE = 409, EH_M_SCRATCH = 410, EH_M_OUT = 411, EH_RELAX = 412,
  EH_STATS = 413, EH_PROB = 414, EH_SOLAR = 415, EH_STATUS = 416, EH_M_STATUS = 417, EH_TIME_FIELDS = 418,
  EH_RECORD_STEP = 419, EH_COUNTERS = 420, EH_AREAS = 421, EH_AREA_PROB = 422, EH_ONSET = 423, EH_ONSET_WS = 424,
  EH_ONSET_ACC = 425, EH_AREA_ONSET = 426, EH_EXT_WS = 427, EH_EXT_STATS = 428, EH_EXT_ACC = 429,
  EH_AREA_EXT_STATS = 430,
  EH_H_RELAX = 400,  // pinned
};

thread_local std::string g_err;
thread_local RsBatchStats g_stats;
thread_local RsLaunchInfo g_launch;
// The model of a device lives in one __constant__ symbol (rs_kernel.cu).  Ordering rule: the symbol is
// only ever overwritten (a) with DIFFERENT bytes and (b) after every kernel that was launched through
// roadsurf_run_device since the previous upload has finished (the asynchronous entry records an event
// per stream; the host entries synchronise their own streams before they return and hold
// g_device_mu while they run).  An upload of identical bytes is skipped.
struct DeviceModel
{
  RsModel m;
  bool valid = false;
  std::map<cudaStream_t, cudaEvent_t> last_launch;  // per caller stream: after its latest step kernel
};
std::mutex g_model_mu;
std::map<int, DeviceModel> g_models;  // device -> model currently in its constant memory
std::atomic<int> g_launches_total{0};

// Run-time options (roadsurf_set_option).  forcing_staging: 1 = full-resolution forcing through the
// per-warp TMA ring in shared memory, 0 = direct read-only loads (default: measured faster).
std::atomic<int> g_opt_staging{-1};
std::atomic<int> g_opt_max_slots{0};  // test hook: cap on points per device batch in roadsurf_run_batch (0 = memory bound)
// coupling_compaction_passes: number of compacted passes over the coupling window before the points
// still iterating are left to finish inside the last launch (0 = one launch, warps repeat in place).
std::atomic<int> g_opt_compaction{6};
// write_back_inputs: roadsurf_run_batch / runsimulation also reproduce the reference's in-place mutation of the
// caller's input arrays (VZ[0], SW_dir, and SW / SW_dir / LW of sky-view points).  Off by default.
std::atomic<int> g_opt_write_back{0};
int opt_compaction_passes() { return g_opt_compaction.load(); }
int opt_staging()
{
  int v = g_opt_staging.load();
  if (v < 0)
  {
    const char* e = std::getenv("ROADSURF_B200_FORCING_STAGING");
    v = (e && e[0] == '1') ? 1 : 0;
    g_opt_staging.store(v);
  }
  return v;
}

int fail(int code, const std::string& msg)
{
  g_err = msg;
  return code;
}

#define CU(call)                                                                                    \
  do                                                                                                \
  {                                                                                                 \
    cudaError_t e_ = (call);                                                                        \
    if (e_ != cudaSuccess)                                                                          \
      return fail(RS_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));                 \
  } while (0)

// One model run on `stream`: a single launch of the step kernel, or -- coupling with lane compaction --
// several.  A warp repeats the coupling window until its slowest lane has converged; when every
// coupled point of the batch has the same window end `wend` (> 0) and the state planes are there,
// the run is split at the window end instead: [step_begin, wend] for everyone, then passes over a
// compacted list of the points that want another iteration (state through the SoA planes), then
// [wend + 1, step_end] with the few points still iterating gathered in warps of their own.  Same
// arithmetic per point, bit-identical results; all launches are queued without a host
// synchronisation.  *launches receives the number of kernels queued.
int launch_model(const RsArgs& a, const RsArgsCold& ac, const RsModel& m, int wend, void* stream, RsLaunchInfo* li,
                 int* launches)
{
  const int passes = opt_compaction_passes();
  *launches = 0;
  auto run = [&](const RsArgs& ak, const RsArgsCold& ck, int staged) {
    return static_cast<cudaError_t>(rs_launch_run(&ak, &ck, m.nlayers, staged, m.use_coupling, m.depth_mode != 0,
                                                  stream, &li->grid, &li->block, &li->regs_per_thread,
                                                  &li->smem_bytes));
  };
  if (!(m.use_coupling && wend > 0 && passes > 0 && ac.state && a.scratch && !(opt_staging() && a.forcing_mode == 0) &&
        a.forcing_step0 == 1 && a.step_begin <= 1 && wend + 1 < a.step_end))
  {
    CU(run(a, ac, opt_staging()));
    *launches = 1;
    return RS_OK;
  }
  int* index = reinterpret_cast<int*>(a.scratch + static_cast<size_t>(2 * m.nlayers + 16) * a.ld);
  int* n_index = index + a.ld;
  const double* flags = ac.state + static_cast<size_t>(m.nlayers + 2 + RS_SP_FLAGS) * a.ld;
  RsArgs a1 = a;
  RsArgsCold c1 = ac;
  a1.step_end = wend;
  c1.mode = RS_MODE_SPLIT;
  c1.window_end = wend;
  CU(run(a1, c1, 0));
  RsArgs a2 = a;
  RsArgsCold c2 = c1;
  a2.step_begin = wend + 1;
  a2.step_end = wend;
  c2.mode = RS_MODE_SPLIT | RS_MODE_ONE_PASS;
  c2.index = index;
  c2.n_index = n_index;
  for (int k = 0; k < passes; ++k)
  {
    CU(static_cast<cudaError_t>(rs_launch_partition(flags, a.ld, a.npoints, 0, index, n_index, stream)));
    CU(run(a2, c2, 0));
  }
  CU(static_cast<cudaError_t>(rs_launch_partition(flags, a.ld, a.npoints, 1, index, n_index, stream)));
  RsArgs a3 = a;
  RsArgsCold c3 = c1;
  a3.step_begin = wend + 1;
  c3.index = index;
  c3.n_index = n_index;
  CU(run(a3, c3, 0));
  *launches = 2 * passes + 3;
  return RS_OK;
}

// The batch with its documented defaults filled in: step_begin 0 -> 1, step_end 0 -> sim_len, forcing_step0 0 -> 1,
// and out_nvar RS_O_NVAR unless it is RS_O_NVAR_EXT.
RsDeviceBatch with_defaults(RsDeviceBatch b)
{
  if (b.step_begin <= 0) b.step_begin = 1;
  if (b.step_end <= 0) b.step_end = b.sim_len;
  if (b.forcing_step0 <= 0) b.forcing_step0 = 1;
  if (b.out_nvar != RS_O_NVAR_EXT) b.out_nvar = RS_O_NVAR;
  return b;
}

// A checked batch as step-kernel launches on `stream`: the one place the kernel's arguments are built.  forcing_mode
// 2 runs an expansion pass and a full-resolution model run per chunk of expand_steps; the other modes are one model
// run, with lane compaction when b.coupling_window_end is set.  b.solar must already hold the solar table.
// *launches receives the number of kernels queued.
int launch_batch(const RsDeviceBatch& batch, const RsModel& m, cudaStream_t stream, RsLaunchInfo* li, int* launches)
{
  const RsDeviceBatch b = with_defaults(batch);
  RsArgs a;
  std::memset(&a, 0, sizeof a);
  a.npoints = b.npoints;
  a.ld = b.ld;
  a.sim_len = b.sim_len;
  a.n_records = b.n_records;
  a.nvar = b.nvar;
  a.out_stride = b.out_stride;
  a.n_out = b.n_out;
  a.forcing_mode = b.forcing_mode;
  a.step_begin = b.step_begin;
  a.step_end = b.step_end;
  a.forcing_step0 = b.forcing_step0;
  a.out_slot0 = b.out_slot0;
  a.forcing = b.forcing;
  a.record_step = b.record_step;
  a.tf = b.time_fields;
  a.local = b.local;
  a.horizons = b.horizons;
  a.solar = b.solar;
  a.out = b.out;
  a.status = b.status;
  a.scratch = b.scratch;
  RsArgsCold ac;
  std::memset(&ac, 0, sizeof ac);
  ac.state = b.state;
  ac.counters = b.counters;
  ac.out_start = b.out_start;
  ac.out_nvar = b.out_nvar;
  if (b.order && !(opt_staging() && b.forcing_mode == 0))  // (the staged ring needs consecutive points per warp)
  {
    ac.index = b.order;  // thread t runs point order[t]
    ac.n_fixed = b.ld;
  }
  li->nlayers = m.nlayers;
  li->forcing_mode = b.forcing_mode;
  *launches = 0;
  if (b.forcing_mode != 2) return launch_model(a, ac, m, b.coupling_window_end, stream, li, launches);
  for (int cb = b.step_begin; cb <= b.step_end; cb += b.expand_steps)
  {
    const int ce = std::min(b.step_end, cb + b.expand_steps - 1);
    CU(static_cast<cudaError_t>(rs_launch_expand(b.forcing, b.record_step, b.n_records, b.nvar, b.ld, b.npoints, 2,
                                                 m.DT, cb, ce, b.expand_workspace, stream)));
    RsArgs ak = a;
    ak.forcing_mode = 0;
    ak.forcing = b.expand_workspace;
    ak.n_records = ce - cb + 1;
    ak.forcing_step0 = cb;
    ak.step_begin = cb;
    ak.step_end = ce;
    int n = 0;
    const int rc = launch_model(ak, ac, m, 0, stream, li, &n);
    if (rc != RS_OK) return rc;
    *launches += 1 + n;
  }
  return RS_OK;
}

double now_ms()
{
  using namespace std::chrono;
  return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

// Makes `m` the model of device `dev`, the current device, by the ordering rule above.
int upload_model(int dev, const RsModel& m)
{
  std::lock_guard<std::mutex> lk(g_model_mu);
  DeviceModel& dm = g_models[dev];
  if (dm.valid && std::memcmp(&dm.m, &m, sizeof m) == 0) return RS_OK;
  // kernels of the asynchronous entry may still be reading the old model: wait for them
  for (auto& kv : dm.last_launch) CU(cudaEventSynchronize(kv.second));
  CU(static_cast<cudaError_t>(rs_upload_model(&m)));
  dm.m = m;
  dm.valid = true;
  return RS_OK;
}

int set_model_on_current_device(const InputSettings* settings, const InputParameters* params, RsModel* out)
{
  RsModel m;
  char err[256];
  int rc = rs_build_model(settings, params, &m, err, sizeof err);
  if (rc != RS_OK) return fail(rc, err);
  int dev = 0;
  CU(cudaGetDevice(&dev));
  rc = upload_model(dev, m);
  if (rc == RS_OK && out) *out = m;
  return rc;
}

// The model roadsurf_set_model put on device `dev`.
int current_model(int dev, RsModel* out)
{
  std::lock_guard<std::mutex> lk(g_model_mu);
  auto it = g_models.find(dev);
  if (it == g_models.end() || !it->second.valid)
    return fail(RS_ERR_BAD_ARGUMENT, "roadsurf_set_model was not called on this device");
  *out = it->second.m;
  return RS_OK;
}

// roadsurf_run_device: remember that `stream` has kernels in flight that read the device's model.
int note_async_launch(int dev, cudaStream_t stream)
{
  std::lock_guard<std::mutex> lk(g_model_mu);
  DeviceModel& dm = g_models[dev];
  cudaEvent_t& ev = dm.last_launch[stream];
  if (!ev) CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  CU(cudaEventRecord(ev, stream));
  return RS_OK;
}

// Run fn(k) for k in [0, n) on up to `nthreads` host threads (the caller's thread included).
void parallel_for(int n, int nthreads, const std::function<void(int)>& fn)
{
  if (n <= 0) return;
  nthreads = std::max(1, std::min(nthreads, n));
  if (nthreads == 1)
  {
    for (int k = 0; k < n; ++k) fn(k);
    return;
  }
  std::atomic<int> next(0);
  auto work = [&]() {
    for (;;)
    {
      const int k = next.fetch_add(1);
      if (k >= n) break;
      fn(k);
    }
  };
  std::vector<std::thread> th;
  for (int t = 1; t < nthreads; ++t) th.emplace_back(work);
  work();
  for (auto& t : th) t.join();
}

int host_threads()
{
  const unsigned hc = std::thread::hardware_concurrency();
  return static_cast<int>(std::max(1u, std::min(hc ? hc : 4u, 32u)));
}

// What the kernel will decide about a point's coupling window (src/InputOutput.f90:34-36,
// src/Coupling.f90:510-519): used only to order slots so that every warp has one window.
long long window_key(const RsModel& m, const LocalParameters& lp)
{
  if (!m.use_coupling || lp.couplingTsurf < -100 || lp.couplingIndexI < 1) return -1;
  return lp.couplingIndexI;
}

// ---- the reference's point structs <-> the kernel's planes ------------------------------------------
// A point's time axis in the order of the kernel's time-field planes.
std::array<const int*, 6> time_fields(const InputPointers& ip)
{
  return {ip.c_year, ip.c_month, ip.c_day, ip.c_hour, ip.c_minute, ip.c_second};
}

bool same_time_axis(const InputPointers& a, const InputPointers& b, int sim_len)
{
  const auto fa = time_fields(a), fb = time_fields(b);
  for (int k = 0; k < 6; ++k)
    if (fa[k] != fb[k] && std::memcmp(fa[k], fb[k], sizeof(int) * sim_len)) return false;
  return true;
}

// Whether the kernel applies the sky-view correction to a point (RS_L_SKY_VIEW).
bool sky_view_point(double sky_view) { return sky_view < 1.0 && sky_view > -0.01f; }

// Forcing plane v (RS_F_*) of a point, steps 0 .. n-1, to dst[t * stride]; the precipitation phase is an int
// array in the reference and a double plane in the kernel.
void forcing_row(const InputPointers& ip, int v, int n, double* dst, size_t stride)
{
  const double* src[RS_F_NVAR_DEPTH] = {ip.c_tair, ip.c_tdew, ip.c_VZ,     ip.c_Rhz,      ip.c_prec, ip.c_SW,
                                        ip.c_LW,   ip.c_SW_dir, ip.c_LW_net, ip.c_TSurfObs, nullptr,   ip.c_Depth};
  if (v == RS_F_PHASE)
    for (int t = 0; t < n; ++t) dst[t * stride] = static_cast<double>(ip.c_PrecPhase[t]);
  else if (stride == 1)
    std::memcpy(dst, src[v], sizeof(double) * n);
  else
    for (int t = 0; t < n; ++t) dst[t * stride] = src[v][t];
}

// A point's output arrays in the order of the kernel's output planes (RS_O_*).
std::array<double*, RS_O_NVAR> output_planes(const OutputPointers& op)
{
  return {op.c_TsurfOut, op.c_SnowOut, op.c_WaterOut, op.c_IceOut, op.c_DepositOut, op.c_Ice2Out};
}

// A point's values of the statics planes RS_L_* to dst[k * stride]; lp == nullptr gives those of a padding slot.
void local_row(const LocalParameters* lp, double* dst, size_t stride)
{
  double row[RS_L_NLOCAL] = {};
  row[RS_L_SKY_VIEW] = 1.0;
  if (lp)
  {
    row[RS_L_TAIR_RELAX] = lp->tair_relax;
    row[RS_L_VZ_RELAX] = lp->VZ_relax;
    row[RS_L_RH_RELAX] = lp->RH_relax;
    row[RS_L_COUPLING_TSURF] = lp->couplingTsurf;
    row[RS_L_LAT] = lp->lat;
    row[RS_L_LON] = lp->lon;
    row[RS_L_SKY_VIEW] = lp->sky_view;
    row[RS_L_COUPLING_INDEX] = lp->couplingIndexI;
    row[RS_L_INIT_LEN] = lp->InitLenI;
    row[RS_L_ACTIVE] = 1.0;
  }
  for (int k = 0; k < RS_L_NLOCAL; ++k) dst[k * stride] = row[k];
}

// The coupling window end shared by the active coupled points of SoA statics [RS_L_NLOCAL][np]: 0 when no
// point is coupled, -1 when their windows differ.
int common_window_end(const double* local, size_t np)
{
  int w = 0;
  for (size_t p = 0; p < np; ++p)
  {
    const double ts = local[RS_L_COUPLING_TSURF * np + p], ix = local[RS_L_COUPLING_INDEX * np + p];
    if (local[RS_L_ACTIVE * np + p] == 0.0 || ts < -100 || ix < 1) continue;
    if (w == 0)
      w = static_cast<int>(ix);
    else if (w != static_cast<int>(ix))
      return -1;
  }
  return w;
}

// Output slots of the steps [first, last] (1-based) as [slot_begin, slot_end); empty when none.
void slot_range(int first, int last, int out_start, int out_stride, int* s0, int* s1)
{
  *s0 = *s1 = 0;
  if (last - 1 < out_start || last < first) return;
  const int k0 = first - 1 - out_start;
  *s0 = k0 > 0 ? (k0 + out_stride - 1) / out_stride : 0;
  *s1 = (last - 1 - out_start) / out_stride + 1;
  if (*s1 < *s0) *s1 = *s0;
}

// Adds the device time between the events ev[0..3] (input copies, kernels, output copies) to s.
void add_stage_times(RsBatchStats& s, const cudaEvent_t ev[4])
{
  float ms = 0.f;
  cudaEventElapsedTime(&ms, ev[0], ev[1]);
  s.h2d_ms += ms;
  cudaEventElapsedTime(&ms, ev[1], ev[2]);
  s.kernel_ms += ms;
  cudaEventElapsedTime(&ms, ev[2], ev[3]);
  s.d2h_ms += ms;
}

// Points [first, first + count) of a batch, run on `device`.
struct ShardRange
{
  int first = 0, count = 0, device = 0;
};

// The split of npoints over the GPUs: ngpus <= 0 or above the device count means every device, and there are
// never more shards than points.  A single shard runs on the caller's device, *current.
int split_shards(int npoints, int ngpus, int* current, std::vector<ShardRange>* shards)
{
  const int ndev = roadsurf_device_count();
  if (ndev < 1) return fail(RS_ERR_NO_DEVICE, "no CUDA device visible (this library has no CPU path)");
  if (ngpus <= 0 || ngpus > ndev) ngpus = ndev;
  if (ngpus > npoints) ngpus = npoints;
  *current = 0;
  cudaGetDevice(current);
  shards->resize(ngpus);
  for (int g = 0; g < ngpus; ++g)
  {
    ShardRange& s = (*shards)[g];
    s.first = static_cast<int>(static_cast<long long>(npoints) * g / ngpus);
    s.count = static_cast<int>(static_cast<long long>(npoints) * (g + 1) / ngpus) - s.first;
    s.device = (ngpus == 1) ? *current : g;
  }
  return RS_OK;
}

struct Shard : ShardRange
{
  int rc = RS_OK;
  std::string err;
  RsBatchStats stats{};
  RsLaunchInfo launch{};
};

// Grow-only device and pinned-host work space, one buffer per (device, slot), reused across calls so
// that a steady-state call does no cudaMalloc / cudaMallocHost (both cost tens to hundreds of ms at
// these sizes).
struct PoolEntry
{
  void* p = nullptr;
  size_t cap = 0;
};
std::mutex g_pool_mu;
std::map<std::pair<int, int>, PoolEntry> g_pool, g_pinned_pool;

// The pooled buffers of a device are used by one call at a time: concurrent callers (the reference
// calls runsimulation from N host threads) are serialised per device, as the GPU would do anyway.
std::mutex g_device_mu[64];

// The buffer of (device, slot), grown to `count` elements of T (and at least 8 bytes); in pinned host memory
// when `pinned`.  Use pooled / pooled_pinned.
template <class T>
cudaError_t pool_get(bool pinned, int device, int slot, size_t count, T** out)
{
  size_t bytes = sizeof(T) * count;
  if (bytes == 0) bytes = 8;
  std::lock_guard<std::mutex> lk(g_pool_mu);
  PoolEntry& e = (pinned ? g_pinned_pool : g_pool)[{device, slot}];
  if (e.cap < bytes)
  {
    if (e.p) pinned ? cudaFreeHost(e.p) : cudaFree(e.p);
    e.p = nullptr;
    e.cap = 0;
    cudaError_t rc = pinned ? cudaMallocHost(&e.p, bytes) : cudaMalloc(&e.p, bytes);
    if (rc != cudaSuccess) return rc;
    e.cap = bytes;
  }
  *out = static_cast<T*>(e.p);
  return cudaSuccess;
}
template <class T>
cudaError_t pooled(int device, int slot, size_t count, T** out)
{
  return pool_get(false, device, slot, count, out);
}
template <class T>
cudaError_t pooled_pinned(int device, int slot, size_t count, T** out)
{
  return pool_get(true, device, slot, count, out);
}

// Run points [first, first+count) of the batch on `device`.
int run_shard(Shard& sh, OutputPointers* const* out, const InputPointers* const* in,
              const InputSettings* settings, const InputParameters* params,
              const LocalParameters* const* local, int* status)
{
  std::lock_guard<std::mutex> device_lock(g_device_mu[sh.device & 63]);
  const double setup0 = now_ms();
  CU(cudaSetDevice(sh.device));
  RsModel model;
  {
    const int rc = set_model_on_current_device(settings, params, &model);
    if (rc != RS_OK) return rc;
  }
  const int sim_len = settings->SimLen;
  const int nl = model.nlayers;
  cudaStream_t stream;
  CU(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  struct StreamGuard
  {
    cudaStream_t s;
    ~StreamGuard() { cudaStreamDestroy(s); }
  } sguard{stream};

  // ---- group points by time axis; inside a group order slots by coupling window ----------------
  struct Group
  {
    const InputPointers* rep;
    std::vector<int> points;
  };
  std::vector<Group> groups;
  for (int q = 0; q < sh.count; ++q)
  {
    const int p = sh.first + q;
    const InputPointers* ip = in[p];
    if (ip->inputLen < sim_len || out[p]->outputLen < sim_len)
      return fail(RS_ERR_BAD_ARGUMENT, "inputLen/outputLen shorter than SimLen");
    bool placed = false;
    for (auto& g : groups)
    {
      if (same_time_axis(*g.rep, *ip, sim_len))
      {
        g.points.push_back(p);
        placed = true;
        break;
      }
    }
    if (!placed) groups.push_back(Group{ip, {p}});
  }

  size_t free_b = 0, total_b = 0;
  CU(cudaMemGetInfo(&free_b, &total_b));

  for (auto& g : groups)
  {
    // slots: windows sorted, each window padded to a warp boundary; uncoupled points fill the gaps
    std::map<long long, std::vector<int>> by_window;
    for (int p : g.points) by_window[window_key(model, *local[p])].push_back(p);
    // inside a window, points with sky-view radiation go last: the solar geometry and the horizon
    // lookup are skipped by warps without such a point (7 % on a grid with 30 % of them scattered)
    for (auto& kv : by_window)
      std::stable_partition(kv.second.begin(), kv.second.end(),
                            [&](int p) { return !sky_view_point(local[p]->sky_view); });
    std::vector<int> slots;  // point index or -1 (padding)
    std::vector<int> loose;
    if (by_window.count(-1)) loose = by_window[-1];
    size_t loose_pos = 0;
    for (auto& kv : by_window)
    {
      if (kv.first == -1) continue;
      for (int p : kv.second) slots.push_back(p);
      while (slots.size() % 32 != 0)
      {
        if (loose_pos < loose.size())
          slots.push_back(loose[loose_pos++]);
        else
          slots.push_back(-1);
      }
    }
    while (loose_pos < loose.size()) slots.push_back(loose[loose_pos++]);
    while (slots.size() % 32 != 0) slots.push_back(-1);
    ++sh.stats.groups;
    // one coupling window in the whole group (the usual case: one analysis time): lane compaction
    // between coupling iterations (launch_model); needs the per-point state planes
    int wend = 0;
    {
      int nwin = 0;
      for (auto& kv : by_window)
        if (kv.first != -1)
        {
          ++nwin;
          wend = static_cast<int>(kv.first);
        }
      if (nwin != 1 || opt_compaction_passes() < 1) wend = 0;
    }

    std::atomic<bool> any_depth_a(false), any_sky_a(false);
    parallel_for(static_cast<int>(g.points.size()), host_threads(), [&](int k) {
      const int p = g.points[k];
      if (sky_view_point(local[p]->sky_view)) any_sky_a = true;
      if (!any_depth_a.load(std::memory_order_relaxed))  // depth(1), depth(SimLen) are read even with tsurfOutputDepth
      {
        const double* d = in[p]->c_Depth;
        for (int t = 0; t < sim_len; ++t)
          if (d[t] >= 0.0)
          {
            any_depth_a = true;
            break;
          }
      }
    });
    const bool any_depth = any_depth_a, any_sky = any_sky_a;
    const int nvar = any_depth ? RS_F_NVAR_DEPTH : RS_F_NVAR;

    // ---- device batches that fit the memory budget -------------------------------------------
    const size_t per_slot = sizeof(double) * (static_cast<size_t>(sim_len) * (nvar + RS_O_NVAR) + RS_L_NLOCAL +
                                              (any_sky ? 360 : 0) + RS_SCRATCH_NPLANES(nl) +
                                              (wend > 0 ? RS_STATE_NPLANES(nl) : 0)) + sizeof(int);
    // Two buffer sets are in flight (see the pipeline below), and a large group is cut into at least
    // four batches so that copying batch b back overlaps packing and uploading batch b+1.
    const size_t budget = static_cast<size_t>(free_b * 0.80);
    size_t max_slots = budget / 2 / per_slot / 32 * 32;
    if (max_slots < 32) return fail(RS_ERR_CUDA, "not enough device memory for one warp of points");
    {
      const size_t n = slots.size();
      const size_t parts = n >= 4 * 8192 ? 4 : (n >= 2 * 4096 ? 2 : 1);
      max_slots = std::min(max_slots, (n / parts + 31) / 32 * 32);
    }
    if (const int cap = g_opt_max_slots.load()) max_slots = std::min<size_t>(max_slots, (cap + 31) / 32 * 32);
    // staging chunk: <= 192 MiB of pinned memory per direction
    const size_t stage_budget = 192ull << 20;
    int chunk = static_cast<int>(std::max<size_t>(32, stage_budget / (sizeof(double) * sim_len * nvar) / 32 * 32));

    int* d_tf = nullptr;
    CU(pooled(sh.device, RB_TIME_FIELDS, 6 * static_cast<size_t>(sim_len), &d_tf));
    {
      const auto src = time_fields(*g.rep);
      for (int k = 0; k < 6; ++k)
        CU(cudaMemcpyAsync(d_tf + static_cast<size_t>(k) * sim_len, src[k], sizeof(int) * sim_len,
                           cudaMemcpyHostToDevice, stream));
      sh.stats.h2d_bytes += sizeof(int) * 6 * sim_len;
    }
    double* d_solar = nullptr;
    CU(pooled(sh.device, RB_SOLAR, 4 * static_cast<size_t>(sim_len), &d_solar));
    CU(static_cast<cudaError_t>(rs_launch_solar(d_tf, sim_len, d_solar, stream)));
    ++sh.stats.kernel_launches;

    // ---- software pipeline over the device batches: while a helper thread copies batch b back and
    // scatters it into the caller's arrays (its kernels may still be running), the calling thread packs
    // and uploads batch b+1 into the other buffer set.  Each set has its own stream.
    struct Ctx
    {
      double *d_forcing = nullptr, *d_out = nullptr, *d_local = nullptr, *d_hor = nullptr, *d_scratch = nullptr,
             *d_state = nullptr, *d_stage[2] = {}, *h_stage[2] = {}, *h_local = nullptr, *h_hor = nullptr;
      int *d_status = nullptr, *h_status = nullptr;
      unsigned long long* d_counters = nullptr;
      cudaStream_t st = nullptr;
      cudaEvent_t ev_free[2] = {nullptr, nullptr};  // staging buffer reuse
      cudaEvent_t ev[4] = {};                       // input stage begins, ends; kernels end; output stage ends
      size_t s0 = 0;
      int ld = 0, chunk = 0;
      RsBatchStats out_stats{};   // what the helper thread measured
      int rc = RS_OK;
      std::string err;
      std::thread drain;
    };
    Ctx ctx[2];
    struct CtxGuard  // no thread may outlive its buffers; streams and events are per group
    {
      Ctx* c;
      ~CtxGuard()
      {
        for (int k = 0; k < 2; ++k)
        {
          if (c[k].drain.joinable()) c[k].drain.join();
          for (cudaEvent_t e : c[k].ev_free)
            if (e) cudaEventDestroy(e);
          for (cudaEvent_t e : c[k].ev)
            if (e) cudaEventDestroy(e);
          if (c[k].st) cudaStreamDestroy(c[k].st);
        }
      }
    } ctx_guard{ctx};
    const int nthreads = host_threads();
    const size_t max_ld = std::min(max_slots, slots.size());
    const size_t nbatches = (slots.size() + max_slots - 1) / max_slots;
    const int dv = sh.device;
    for (int k = 0; k < (nbatches > 1 ? 2 : 1); ++k)
    {
      Ctx& c = ctx[k];
      const int o = RB_SET2 * k;
      CU(cudaStreamCreateWithFlags(&c.st, cudaStreamNonBlocking));
      for (cudaEvent_t& e : c.ev_free) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      for (cudaEvent_t& e : c.ev) CU(cudaEventCreate(&e));
      c.chunk = static_cast<int>(std::min<size_t>(chunk, max_ld));
      CU(pooled(dv, RB_FORCING + o, static_cast<size_t>(sim_len) * nvar * max_ld, &c.d_forcing));
      CU(pooled(dv, RB_OUT + o, static_cast<size_t>(RS_O_NVAR) * sim_len * max_ld, &c.d_out));
      CU(pooled(dv, RB_LOCAL + o, RS_L_NLOCAL * max_ld, &c.d_local));
      if (any_sky) CU(pooled(dv, RB_HOR + o, 360 * max_ld, &c.d_hor));
      CU(pooled(dv, RB_STATUS + o, max_ld, &c.d_status));
      if (model.use_coupling) CU(pooled(dv, RB_SCRATCH + o, RS_SCRATCH_NPLANES(nl) * max_ld, &c.d_scratch));
      if (wend > 0) CU(pooled(dv, RB_STATE + o, RS_STATE_NPLANES(nl) * max_ld, &c.d_state));
      const size_t stage_n = static_cast<size_t>(c.chunk) * sim_len * std::max(nvar, static_cast<int>(RS_O_NVAR));
      CU(pooled(dv, RB_STAGE + o, stage_n, &c.d_stage[0]));
      CU(pooled(dv, RB_STAGE2 + o, stage_n, &c.d_stage[1]));
      CU(pooled(dv, RB_COUNTERS + o, RS_CNT_N, &c.d_counters));
      CU(pooled_pinned(dv, RB_H_STAGE + o, stage_n, &c.h_stage[0]));
      CU(pooled_pinned(dv, RB_H_STAGE2 + o, stage_n, &c.h_stage[1]));
      CU(pooled_pinned(dv, RB_H_LOCAL + o, RS_L_NLOCAL * max_ld, &c.h_local));
      if (any_sky) CU(pooled_pinned(dv, RB_H_HOR + o, 360 * max_ld, &c.h_hor));
      CU(pooled_pinned(dv, RB_H_STATUS + o, max_ld, &c.h_status));
    }
    // the time axis and the solar table were queued on `stream`: every batch stream reads them
    CU(cudaStreamSynchronize(stream));
    if (sh.stats.setup_ms == 0.0) sh.stats.setup_ms = now_ms() - setup0 - sh.stats.pack_ms;  // everything so far but packing

    // ---- input stage (calling thread): statics, then the forcing: caller's per-point arrays -> pinned
    // [var][point][time] -> device -> SoA.  Rows are packed by all host threads into one of two pinned
    // buffers while the previous buffer is in flight (H2D copy + device-side transpose).
    auto stage_in = [&](Ctx& c) -> int {
      const int ld = c.ld;
      const size_t s0 = c.s0;
      cudaStream_t st = c.st;
      CU(cudaMemsetAsync(c.d_counters, 0, sizeof(unsigned long long) * RS_CNT_N, st));
      double t0 = now_ms();
      {
        for (int q = 0; q < ld; ++q)
        {
          const int p = slots[s0 + q];
          local_row(p >= 0 ? local[p] : nullptr, c.h_local + q, ld);
        }
        if (any_sky)
        {
          double* H = c.h_hor;
          for (int q = 0; q < ld; ++q)
          {
            const int p = slots[s0 + q];
            const double* src = (p >= 0) ? in[p]->c_local_horizons : nullptr;
            for (int k = 0; k < 360; ++k) H[static_cast<size_t>(k) * ld + q] = src ? src[k] : 0.0;
          }
        }
      }
      sh.stats.pack_ms += now_ms() - t0;
      CU(cudaEventRecord(c.ev[0], st));
      CU(cudaMemcpyAsync(c.d_local, c.h_local, sizeof(double) * RS_L_NLOCAL * ld, cudaMemcpyHostToDevice, st));
      sh.stats.h2d_bytes += sizeof(double) * RS_L_NLOCAL * ld;
      if (any_sky)
      {
        CU(cudaMemcpyAsync(c.d_hor, c.h_hor, sizeof(double) * 360 * ld, cudaMemcpyHostToDevice, st));
        sh.stats.h2d_bytes += sizeof(double) * 360 * ld;
      }
      int cidx = 0;
      for (int q0 = 0; q0 < ld; q0 += c.chunk, ++cidx)
      {
        const int npc = std::min(c.chunk, ld - q0);
        const int bsel = cidx & 1;
        if (cidx >= 2) CU(cudaEventSynchronize(c.ev_free[bsel]));
        t0 = now_ms();
        double* S = c.h_stage[bsel];
        const size_t plane = static_cast<size_t>(npc) * sim_len;
        parallel_for(npc, nthreads, [&](int q) {
          const int p = slots[s0 + q0 + q];
          const size_t row = static_cast<size_t>(q) * sim_len;
          if (p < 0)
          {
            for (int v = 0; v < nvar; ++v) std::memset(S + v * plane + row, 0, sizeof(double) * sim_len);
            return;
          }
          for (int v = 0; v < nvar; ++v) forcing_row(*in[p], v, sim_len, S + v * plane + row, 1);
        });
        sh.stats.pack_ms += now_ms() - t0;
        const size_t bytes = sizeof(double) * plane * nvar;
        CU(cudaMemcpyAsync(c.d_stage[bsel], S, bytes, cudaMemcpyHostToDevice, st));
        CU(static_cast<cudaError_t>(
            rs_launch_pack_forcing(c.d_stage[bsel], npc, q0, sim_len, nvar, c.d_forcing, ld, st)));
        CU(cudaEventRecord(c.ev_free[bsel], st));
        ++sh.stats.kernel_launches;
        sh.stats.h2d_bytes += bytes;
      }
      CU(cudaEventRecord(c.ev[1], st));

      // ---- the step kernel(s), queued behind the input stage
      RsDeviceBatch db{};
      db.npoints = ld;
      db.ld = ld;
      db.sim_len = sim_len;
      db.n_records = sim_len;
      db.nvar = nvar;
      db.forcing = c.d_forcing;
      db.time_fields = d_tf;
      db.local = c.d_local;
      db.horizons = any_sky ? c.d_hor : nullptr;
      db.out = c.d_out;
      db.out_stride = 1;
      db.n_out = sim_len;
      db.status = c.d_status;
      db.state = wend > 0 ? c.d_state : nullptr;
      db.scratch = model.use_coupling ? c.d_scratch : nullptr;
      db.counters = c.d_counters;
      db.solar = d_solar;
      db.coupling_window_end = wend;
      {
        int n = 0;
        const int rc = launch_batch(db, model, st, &sh.launch, &n);
        if (rc != RS_OK) return rc;
        sh.stats.kernel_launches += n;
      }
      CU(cudaEventRecord(c.ev[2], st));
      return RS_OK;
    };

    // ---- output stage (helper thread): SoA -> [var][point][time] -> pinned -> caller's arrays, double
    // buffered: chunk c-1 is scattered into the caller's arrays while chunk c is copied back
    auto stage_out = [&](Ctx& c) -> int {
      CU(cudaSetDevice(dv));
      const int ld = c.ld;
      const size_t s0 = c.s0;
      cudaStream_t st = c.st;
      RsBatchStats& os = c.out_stats;
      auto scatter = [&](int q0, int npc, const double* S) {
        const size_t plane = static_cast<size_t>(npc) * sim_len;
        parallel_for(npc, nthreads, [&](int q) {
          const int p = slots[s0 + q0 + q];
          if (p < 0) return;
          const auto dst = output_planes(*out[p]);
          for (int v = 0; v < RS_O_NVAR; ++v)
            std::memcpy(dst[v], S + v * plane + static_cast<size_t>(q) * sim_len, sizeof(double) * sim_len);
        });
      };
      int cidx = 0, prev_q0 = -1, prev_npc = 0;
      for (int q0 = 0; q0 < ld; q0 += c.chunk, ++cidx)
      {
        const int npc = std::min(c.chunk, ld - q0);
        const int bsel = cidx & 1;
        const size_t bytes = sizeof(double) * static_cast<size_t>(npc) * sim_len * RS_O_NVAR;
        CU(static_cast<cudaError_t>(rs_launch_unpack_out(c.d_out, ld, sim_len, q0, npc, c.d_stage[bsel], st)));
        ++os.kernel_launches;
        CU(cudaMemcpyAsync(c.h_stage[bsel], c.d_stage[bsel], bytes, cudaMemcpyDeviceToHost, st));
        CU(cudaEventRecord(c.ev_free[bsel], st));
        os.d2h_bytes += bytes;
        if (prev_q0 >= 0)
        {
          // buffer of the previous chunk: its copy was enqueued before this one
          CU(cudaEventSynchronize(c.ev_free[bsel ^ 1]));
          const double t0 = now_ms();
          scatter(prev_q0, prev_npc, c.h_stage[bsel ^ 1]);
          os.unpack_ms += now_ms() - t0;
        }
        prev_q0 = q0;
        prev_npc = npc;
      }
      CU(cudaEventRecord(c.ev[3], st));
      if (prev_q0 >= 0)
      {
        CU(cudaEventSynchronize(c.ev_free[(cidx - 1) & 1]));
        const double t0 = now_ms();
        scatter(prev_q0, prev_npc, c.h_stage[(cidx - 1) & 1]);
        os.unpack_ms += now_ms() - t0;
      }
      if (g_opt_write_back.load())
      {
        // the reference's caller-visible input mutations (see rs_mutation_kernel), chunk by chunk through the
        // first staging buffer; VZ(1) is clamped on the host (src/Initialization.f90:121-123)
        int* d_nvis = nullptr;
        CU(pooled(dv, RB_NVIS + (&c == &ctx[1] ? RB_SET2 : 0), ld, &d_nvis));
        for (int q0 = 0; q0 < ld; q0 += c.chunk)
        {
          const int npc = std::min(c.chunk, ld - q0);
          const size_t plane = static_cast<size_t>(npc) * sim_len;
          CU(static_cast<cudaError_t>(rs_launch_mutation(c.d_forcing, nvar, ld, sim_len, c.d_local,
                                                         any_sky ? c.d_hor : nullptr, d_solar,
                                                         c.d_out, d_nvis, q0, npc, c.d_stage[0], st)));
          os.kernel_launches += q0 == 0 ? 2 : 1;
          CU(cudaMemcpyAsync(c.h_stage[0], c.d_stage[0], sizeof(double) * 3 * plane, cudaMemcpyDeviceToHost, st));
          CU(cudaStreamSynchronize(st));
          os.d2h_bytes += sizeof(double) * 3 * plane;
          const double* S = c.h_stage[0];
          parallel_for(npc, nthreads, [&](int q) {
            const int p = slots[s0 + q0 + q];
            if (p < 0) return;
            const InputPointers* ip = in[p];
            double* dst[3] = {ip->c_SW, ip->c_SW_dir, ip->c_LW};
            for (int v = 0; v < 3; ++v)
              std::memcpy(dst[v], S + v * plane + static_cast<size_t>(q) * sim_len, sizeof(double) * sim_len);
            if (ip->c_VZ[0] < 0.4f) ip->c_VZ[0] = 0.4f;
          });
        }
      }
      CU(cudaMemcpyAsync(c.h_status, c.d_status, sizeof(int) * ld, cudaMemcpyDeviceToHost, st));
      unsigned long long cnt[RS_CNT_N];
      CU(cudaMemcpyAsync(cnt, c.d_counters, sizeof cnt, cudaMemcpyDeviceToHost, st));
      CU(cudaStreamSynchronize(st));
      add_stage_times(os, c.ev);  // h2d: device-side time of the input stage (copies + transposes, overlapped with packing)
      os.d2h_bytes += sizeof(int) * ld;
      os.executed_steps += static_cast<int64_t>(cnt[RS_CNT_EXECUTED_STEPS]);
      if (status)
        for (int q = 0; q < ld; ++q)
        {
          const int p = slots[s0 + q];
          if (p >= 0) status[p] = c.h_status[q];
        }
      return RS_OK;
    };
    // joins the helper thread of a buffer set and folds its measurements into the shard's
    auto finish = [&](Ctx& c) -> int {
      if (!c.drain.joinable()) return RS_OK;
      c.drain.join();
      sh.stats.h2d_ms += c.out_stats.h2d_ms;
      sh.stats.kernel_ms += c.out_stats.kernel_ms;
      sh.stats.d2h_ms += c.out_stats.d2h_ms;
      sh.stats.unpack_ms += c.out_stats.unpack_ms;
      sh.stats.d2h_bytes += c.out_stats.d2h_bytes;
      sh.stats.executed_steps += c.out_stats.executed_steps;
      sh.stats.kernel_launches += c.out_stats.kernel_launches;
      c.out_stats = RsBatchStats{};
      if (c.rc != RS_OK) return fail(c.rc, c.err);
      return RS_OK;
    };

    // The helper threads reference this frame's lambdas and locals: whatever happens in the loop, they are
    // joined (and, after an error, the batch streams drained: pooled buffers may still be in use by queued
    // kernels and copies) before anything here goes out of scope.
    const int loop_rc = [&]() -> int {
      size_t b = 0;
      for (size_t s0 = 0; s0 < slots.size(); s0 += max_slots, ++b)
      {
        Ctx& c = ctx[b & 1];
        {
          const int rc = finish(c);  // the batch that used this buffer set two rounds ago
          if (rc != RS_OK) return rc;
        }
        c.s0 = s0;
        c.ld = static_cast<int>(std::min(max_slots, slots.size() - s0));
        {
          const int rc = stage_in(c);
          if (rc != RS_OK) return rc;
        }
        c.rc = RS_OK;
        c.drain = std::thread([&stage_out, &c]() {
          c.rc = stage_out(c);
          if (c.rc != RS_OK) c.err = g_err;
        });
      }
      for (int k = 0; k < 2; ++k)
      {
        const int rc = finish(ctx[k]);
        if (rc != RS_OK) return rc;
      }
      return RS_OK;
    }();
    if (loop_rc != RS_OK)
    {
      const std::string err = g_err;
      for (int k = 0; k < 2; ++k)
      {
        if (ctx[k].drain.joinable()) ctx[k].drain.join();
        if (ctx[k].st) cudaStreamSynchronize(ctx[k].st);
      }
      return fail(loop_rc, err);
    }
  }
  return RS_OK;
}
// Column chunks of a host-SoA shard: a multiple of 32 points, about 1/8 of the shard but at least 64 Ki points.
int host_soa_chunk(int count)
{
  int chunk = ((count + 7) / 8 + 31) / 32 * 32;
  if (chunk < 65536) chunk = std::min((count + 31) / 32 * 32, 65536);
  return chunk;
}

// roadsurf_prepare_statics: per device shard and per chunk of roadsurf_run_host_soa's pipeline, the local
// horizon table [360][ld] and the sky-view point order [ld], resident on the device.
struct StaticsChunk
{
  double* hor = nullptr;  // [360][ld] or null (no horizons given)
  int* order = nullptr;   // [ld]
  int ld = 0;
};
struct StaticsShard : ShardRange
{
  int chunk = 0;
  std::vector<StaticsChunk> chunks;
};
struct RsStatics
{
  unsigned magic = 0x52535354u;  // "RSST"
  int npoints = 0, ngpus = 0;
  bool has_horizons = false;
  std::vector<StaticsShard> shards;
};

// Streams and events of the host-SoA pipeline, created once per device and reused by every call (the
// calls of one device are serialised by g_device_mu).
struct SoaStreams
{
  cudaStream_t st[2] = {nullptr, nullptr};
  cudaEvent_t ev[2][4] = {};
};
std::mutex g_soa_mu;
std::map<int, SoaStreams> g_soa_streams;
int soa_streams(int device, SoaStreams** out)
{
  std::lock_guard<std::mutex> lk(g_soa_mu);
  SoaStreams& s = g_soa_streams[device];
  if (!s.st[0])
    for (int k = 0; k < 2; ++k)
    {
      CU(cudaStreamCreateWithFlags(&s.st[k], cudaStreamNonBlocking));
      for (int e = 0; e < 4; ++e) CU(cudaEventCreate(&s.ev[k][e]));
    }
  *out = &s;
  return RS_OK;
}

// Points [first, first+count) of a host SoA batch on `device`, pipelined in column chunks over two
// streams: H2D(chunk c+1) overlaps kernel(chunk c) overlaps D2H(chunk c-1).
int run_host_soa_shard(Shard& sh, const RsHostBatch* b, const InputSettings* settings,
                       const InputParameters* params)
{
  std::lock_guard<std::mutex> device_lock(g_device_mu[sh.device & 63]);
  CU(cudaSetDevice(sh.device));
  RsModel model;
  {
    const int rc = set_model_on_current_device(settings, params, &model);
    if (rc != RS_OK) return rc;
  }
  const int nl = model.nlayers;
  const int n_out = (b->sim_len + b->out_stride - 1) / b->out_stride;
  const size_t np_all = static_cast<size_t>(b->npoints);
  constexpr int NSTREAM = 2;
  const int chunk = host_soa_chunk(sh.count);
  const int nchunks = (sh.count + chunk - 1) / chunk;
  const size_t frows = static_cast<size_t>(b->n_records) * b->nvar;
  const size_t orows = static_cast<size_t>(RS_O_NVAR) * n_out;
  // statics resident on the device (roadsurf_prepare_statics)?
  const StaticsShard* resident = nullptr;
  if (b->statics)
  {
    const RsStatics* h = static_cast<const RsStatics*>(b->statics);
    if (h->magic != 0x52535354u || h->npoints != b->npoints)
      return fail(RS_ERR_BAD_ARGUMENT, "statics handle does not belong to a grid of this many points");
    for (const StaticsShard& s : h->shards)
      if (s.device == sh.device && s.first == sh.first && s.count == sh.count && s.chunk == chunk) resident = &s;
    if (!resident || static_cast<int>(resident->chunks.size()) != nchunks)
      return fail(RS_ERR_BAD_ARGUMENT, "statics handle was prepared for another ngpus / device set");
  }
  const bool hor = resident ? resident->chunks[0].hor != nullptr : b->horizons != nullptr;

  SoaStreams* ss = nullptr;
  {
    const int rc = soa_streams(sh.device, &ss);
    if (rc != RS_OK) return rc;
  }
  cudaStream_t* streams = ss->st;
  cudaEvent_t(*ev)[4] = ss->ev;

  // per-stream device buffers
  const int wend = (model.use_coupling && opt_compaction_passes() > 0) ? b->coupling_window_end : 0;
  double *d_forcing[NSTREAM], *d_out[NSTREAM], *d_local[NSTREAM], *d_hor[NSTREAM] = {}, *d_scratch[NSTREAM] = {},
         *d_state[NSTREAM] = {};
  int *d_status[NSTREAM], *d_order[NSTREAM] = {};
  const size_t cols = chunk;
  for (int s = 0; s < NSTREAM; ++s)
  {
    const int o = HS_STREAM * s;
    CU(pooled(sh.device, HS_FORCING + o, frows * cols, &d_forcing[s]));
    CU(pooled(sh.device, HS_OUT + o, orows * cols, &d_out[s]));
    CU(pooled(sh.device, HS_LOCAL + o, RS_L_NLOCAL * cols, &d_local[s]));
    if (hor && !resident) CU(pooled(sh.device, HS_HOR + o, 360 * cols, &d_hor[s]));
    if (model.use_coupling) CU(pooled(sh.device, HS_SCRATCH + o, RS_SCRATCH_NPLANES(nl) * cols, &d_scratch[s]));
    CU(pooled(sh.device, HS_STATUS + o, cols, &d_status[s]));
    if (wend > 0) CU(pooled(sh.device, HS_STATE + o, RS_STATE_NPLANES(nl) * cols, &d_state[s]));
    if (hor && !resident && b->forcing_mode == 1)  // sky-view points gathered at one end of the chunk (see roadsurf_order_points)
      CU(pooled(sh.device, HS_ORDER + o, cols, &d_order[s]));
  }
  int *d_tf = nullptr, *d_rs = nullptr;
  unsigned long long* d_counters = nullptr;
  double* d_solar = nullptr;
  CU(pooled(sh.device, HS_TIME_FIELDS, 6 * static_cast<size_t>(b->sim_len), &d_tf));
  CU(pooled(sh.device, HS_RECORD_STEP, std::max(1, b->n_records), &d_rs));
  CU(pooled(sh.device, HS_COUNTERS, RS_CNT_N, &d_counters));
  CU(pooled(sh.device, HS_SOLAR, 4 * static_cast<size_t>(b->sim_len), &d_solar));
  CU(cudaMemcpyAsync(d_tf, b->time_fields, sizeof(int) * 6 * b->sim_len, cudaMemcpyHostToDevice, streams[0]));
  if (b->forcing_mode == 1)
    CU(cudaMemcpyAsync(d_rs, b->record_step, sizeof(int) * b->n_records, cudaMemcpyHostToDevice, streams[0]));
  CU(cudaMemsetAsync(d_counters, 0, sizeof(unsigned long long) * RS_CNT_N, streams[0]));
  CU(static_cast<cudaError_t>(rs_launch_solar(d_tf, b->sim_len, d_solar, streams[0])));
  ++sh.stats.kernel_launches;
  CU(cudaStreamSynchronize(streams[0]));
  sh.stats.h2d_bytes += sizeof(int) * (6 * b->sim_len + b->n_records);

  for (int c = 0; c < nchunks; ++c)
  {
    const int s = c % NSTREAM;
    cudaStream_t st = streams[s];
    const int q0 = c * chunk;
    const int npc = std::min(chunk, sh.count - q0);
    const int ld = (npc + 31) / 32 * 32;
    const size_t col0 = static_cast<size_t>(sh.first) + q0;
    if (c >= NSTREAM)
    {
      // buffers of this stream are free once its previous chunk's D2H has finished
      CU(cudaStreamSynchronize(st));
      add_stage_times(sh.stats, ev[s]);
    }
    const size_t wbytes = sizeof(double) * npc;
    CU(cudaEventRecord(ev[s][0], st));
    CU(cudaMemcpy2DAsync(d_forcing[s], sizeof(double) * ld, b->forcing + col0, sizeof(double) * np_all, wbytes,
                         frows, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpy2DAsync(d_local[s], sizeof(double) * ld, b->local + col0, sizeof(double) * np_all, wbytes,
                         RS_L_NLOCAL, cudaMemcpyHostToDevice, st));
    if (hor && !resident)
      CU(cudaMemcpy2DAsync(d_hor[s], sizeof(double) * ld, b->horizons + col0, sizeof(double) * np_all, wbytes, 360,
                           cudaMemcpyHostToDevice, st));
    sh.stats.h2d_bytes += wbytes * (frows + RS_L_NLOCAL + ((hor && !resident) ? 360 : 0));
    CU(cudaEventRecord(ev[s][1], st));
    RsDeviceBatch db{};
    db.npoints = npc;
    db.ld = ld;
    db.sim_len = b->sim_len;
    db.forcing_mode = b->forcing_mode;
    db.n_records = b->n_records;
    db.nvar = b->nvar;
    db.forcing = d_forcing[s];
    db.record_step = d_rs;
    db.time_fields = d_tf;
    db.local = d_local[s];
    db.horizons = resident ? resident->chunks[c].hor : d_hor[s];
    db.out = d_out[s];
    db.out_stride = b->out_stride;
    db.n_out = n_out;
    db.status = d_status[s];
    db.state = d_state[s];
    db.scratch = d_scratch[s];
    db.counters = d_counters;
    db.solar = d_solar;
    db.coupling_window_end = wend;
    if (resident && b->forcing_mode == 1 && resident->chunks[c].order)
      db.order = resident->chunks[c].order;  // built once by roadsurf_prepare_statics
    else if (d_order[s])
    {
      CU(static_cast<cudaError_t>(rs_launch_partition(d_local[s] + static_cast<size_t>(RS_L_SKY_VIEW) * ld, ld, npc, 2,
                                                      d_order[s], nullptr, st)));
      ++sh.stats.kernel_launches;
      db.order = d_order[s];
    }
    {
      int n = 0;
      const int rc = launch_batch(db, model, st, &sh.launch, &n);
      if (rc != RS_OK) return rc;
      sh.stats.kernel_launches += n;
    }
    CU(cudaEventRecord(ev[s][2], st));
    CU(cudaMemcpy2DAsync(b->out + col0, sizeof(double) * np_all, d_out[s], sizeof(double) * ld, wbytes, orows,
                         cudaMemcpyDeviceToHost, st));
    if (b->status)
      CU(cudaMemcpyAsync(b->status + col0, d_status[s], sizeof(int) * npc, cudaMemcpyDeviceToHost, st));
    sh.stats.d2h_bytes += wbytes * orows + (b->status ? sizeof(int) * npc : 0);
    CU(cudaEventRecord(ev[s][3], st));
  }
  for (int s = 0; s < NSTREAM && s < nchunks; ++s)
  {
    CU(cudaStreamSynchronize(streams[s]));
    add_stage_times(sh.stats, ev[s]);
  }
  unsigned long long cnt[RS_CNT_N];
  CU(cudaMemcpy(cnt, d_counters, sizeof cnt, cudaMemcpyDeviceToHost));
  sh.stats.executed_steps += static_cast<int64_t>(cnt[RS_CNT_EXECUTED_STEPS]);
  sh.stats.groups = nchunks;
  return RS_OK;
}

int run_sharded(int npoints, int ngpus, const std::function<int(Shard&)>& fn)
{
  const double wall0 = now_ms();
  int current = 0;
  std::vector<ShardRange> ranges;
  {
    const int rc = split_shards(npoints, ngpus, &current, &ranges);
    if (rc != RS_OK) return rc;
  }
  ngpus = static_cast<int>(ranges.size());
  std::vector<Shard> shards(ngpus);
  for (int g = 0; g < ngpus; ++g) static_cast<ShardRange&>(shards[g]) = ranges[g];
  auto work = [&](int g) {
    Shard& sh = shards[g];
    sh.rc = fn(sh);
    if (sh.rc != RS_OK) sh.err = g_err;
  };
  if (ngpus == 1)
    work(0);
  else
  {
    std::vector<std::thread> th;
    for (int g = 0; g < ngpus; ++g) th.emplace_back(work, g);
    for (auto& t : th) t.join();
    cudaSetDevice(current);
  }
  for (auto& sh : shards)
  {
    g_stats.pack_ms = std::max(g_stats.pack_ms, sh.stats.pack_ms);
    g_stats.h2d_ms = std::max(g_stats.h2d_ms, sh.stats.h2d_ms);
    g_stats.kernel_ms = std::max(g_stats.kernel_ms, sh.stats.kernel_ms);
    g_stats.d2h_ms = std::max(g_stats.d2h_ms, sh.stats.d2h_ms);
    g_stats.unpack_ms = std::max(g_stats.unpack_ms, sh.stats.unpack_ms);
    g_stats.h2d_bytes += sh.stats.h2d_bytes;
    g_stats.d2h_bytes += sh.stats.d2h_bytes;
    g_stats.executed_steps += sh.stats.executed_steps;
    g_stats.kernel_launches += sh.stats.kernel_launches;
    g_stats.groups += sh.stats.groups;
    g_stats.setup_ms = std::max(g_stats.setup_ms, sh.stats.setup_ms);
    g_launches_total += sh.stats.kernel_launches;
    if (sh.launch.grid) g_launch = sh.launch;
  }
  g_stats.wall_ms = now_ms() - wall0;
  for (auto& sh : shards)
    if (sh.rc != RS_OK) return fail(sh.rc, sh.err);
  return RS_OK;
}
// The record grid example1's rule is implemented for (forcing_mode 1): record_step strictly increasing, the
// first record at or before step 0.  The kernel and record_value_at extrapolate the first interval back to
// step 0 where JsonSource leaves the steps before its first record missing, and equal record steps divide
// by a zero span.  Host entries call this before any device work; roadsurf_run_device, whose record_step
// is device memory, keeps it as a precondition.
int check_record_grid(const int* rs, int nrec)
{
  if (rs[0] > 0) return fail(RS_ERR_BAD_ARGUMENT, "record_step[0] must be <= 0 (the first record at or before step 0)");
  for (int k = 1; k < nrec; ++k)
    if (rs[k] <= rs[k - 1]) return fail(RS_ERR_BAD_ARGUMENT, "record_step must be strictly increasing");
  return RS_OK;
}

// The value JsonSource's interpolation gives at vector index t (the kernel's fetch_coarse rule) from coarse
// records at record_step rs[0 .. nrec): rec(k) is record k's value of the variable.  Used by
// roadsurf_read_input_derive_records and, on each member's records, by roadsurf_run_ensemble_host_soa.
template <class Rec>
double record_value_at(const int* rs, int nrec, double DT, int t, const Rec& rec)
{
  int k = 0;
  while (k + 2 < nrec && rs[k + 1] <= t) ++k;
  if (t >= rs[nrec - 1]) return -9999.9;  // at / after the last record: never filled (JsonSource.cpp:85)
  const double va = rec(k), vb = rec(k + 1);
  if (t == rs[k]) return (va > -100.0) ? va : -9999.9;
  if (!(va > -100.0 && vb > -100.0)) return -9999.9;
  const double spn = static_cast<double>(rs[k + 1] - rs[k]) * DT, dt_a = static_cast<double>(t - rs[k]) * DT;
  return va + (dt_a * (vb - va)) / spn;
}
}  // namespace

extern "C" {

int roadsurf_run_host_soa(const RsHostBatch* b, const InputSettings* settings, const InputParameters* params,
                          int ngpus)
{
  g_err.clear();
  std::memset(&g_stats, 0, sizeof g_stats);
  if (!b || !settings || !params) return fail(RS_ERR_BAD_ARGUMENT, "null argument");
  if (b->npoints < 0 || b->sim_len < 1 || b->out_stride < 1) return fail(RS_ERR_BAD_ARGUMENT, "bad sizes");
  if (b->sim_len != settings->SimLen) return fail(RS_ERR_BAD_ARGUMENT, "batch sim_len != settings SimLen");
  if (b->nvar != RS_F_NVAR && b->nvar != RS_F_NVAR_DEPTH) return fail(RS_ERR_BAD_ARGUMENT, "nvar must be 11 or 12");
  if (b->forcing_mode != 0 && b->forcing_mode != 1)
    return fail(RS_ERR_UNSUPPORTED, "roadsurf_run_host_soa takes forcing_mode 0 or 1 (example2's rule, mode 2, is offered by "
                                    "the device entry: roadsurf_run_device / roadsurf_expand_records)");
  if (b->forcing_mode == 0 ? b->n_records != b->sim_len : (b->n_records < 2 || !b->record_step))
    return fail(RS_ERR_BAD_ARGUMENT, "bad n_records / record_step for the forcing mode");
  if (b->forcing_mode == 1)
  {
    const int rc = check_record_grid(b->record_step, b->n_records);
    if (rc != RS_OK) return rc;
  }
  if (b->npoints > 0 && (!b->forcing || !b->time_fields || !b->local || !b->out))
    return fail(RS_ERR_BAD_ARGUMENT, "null host pointer in batch");
  if (b->npoints == 0) return roadsurf_device_count() < 1 ? fail(RS_ERR_NO_DEVICE, "no CUDA device visible") : RS_OK;
  return run_sharded(b->npoints, ngpus, [&](Shard& sh) { return run_host_soa_shard(sh, b, settings, params); });
}

int roadsurf_prepare_statics(const RsHostBatch* b, int ngpus, void** handle)
{
  g_err.clear();
  if (!b || !handle || b->npoints < 1 || !b->local) return fail(RS_ERR_BAD_ARGUMENT, "bad arguments");
  int current = 0;
  std::vector<ShardRange> ranges;
  int rc = split_shards(b->npoints, ngpus, &current, &ranges);
  if (rc != RS_OK) return rc;
  RsStatics* h = new RsStatics;
  h->npoints = b->npoints;
  h->ngpus = static_cast<int>(ranges.size());
  h->has_horizons = b->horizons != nullptr;
  const size_t np_all = static_cast<size_t>(b->npoints);
  for (size_t g = 0; g < ranges.size() && rc == RS_OK; ++g)
  {
    StaticsShard s;
    static_cast<ShardRange&>(s) = ranges[g];
    s.chunk = host_soa_chunk(s.count);
    auto body = [&]() -> int {
      CU(cudaSetDevice(s.device));
      for (int q0 = 0; q0 < s.count; q0 += s.chunk)
      {
        StaticsChunk ch;
        const int npc = std::min(s.chunk, s.count - q0);
        ch.ld = (npc + 31) / 32 * 32;
        const size_t col0 = static_cast<size_t>(s.first) + q0;
        double* d_sky = nullptr;
        CU(cudaMalloc(&d_sky, sizeof(double) * ch.ld));
        CU(cudaMemset(d_sky, 0, sizeof(double) * ch.ld));
        CU(cudaMemcpy(d_sky, b->local + static_cast<size_t>(RS_L_SKY_VIEW) * np_all + col0, sizeof(double) * npc,
                      cudaMemcpyHostToDevice));
        CU(cudaMalloc(&ch.order, sizeof(int) * ch.ld));
        CU(static_cast<cudaError_t>(rs_launch_partition(d_sky, ch.ld, npc, 2, ch.order, nullptr, nullptr)));
        ++g_launches_total;
        if (b->horizons)
        {
          CU(cudaMalloc(&ch.hor, sizeof(double) * 360 * ch.ld));
          CU(cudaMemset(ch.hor, 0, sizeof(double) * 360 * ch.ld));
          CU(cudaMemcpy2D(ch.hor, sizeof(double) * ch.ld, b->horizons + col0, sizeof(double) * np_all,
                          sizeof(double) * npc, 360, cudaMemcpyHostToDevice));
        }
        CU(cudaDeviceSynchronize());
        cudaFree(d_sky);
        s.chunks.push_back(ch);
      }
      return RS_OK;
    };
    rc = body();
    h->shards.push_back(s);
  }
  cudaSetDevice(current);
  if (rc != RS_OK)
  {
    const std::string err = g_err;
    roadsurf_release_statics(h);
    return fail(rc, err);
  }
  *handle = h;
  return RS_OK;
}

void roadsurf_release_statics(void* handle)
{
  RsStatics* h = static_cast<RsStatics*>(handle);
  if (!h || h->magic != 0x52535354u) return;
  int current = 0;
  cudaGetDevice(&current);
  for (StaticsShard& s : h->shards)
  {
    cudaSetDevice(s.device);
    for (StaticsChunk& ch : s.chunks)
    {
      if (ch.hor) cudaFree(ch.hor);
      if (ch.order) cudaFree(ch.order);
    }
  }
  cudaSetDevice(current);
  h->magic = 0;
  delete h;
}

// ---- step-granular sessions -------------------------------------------------------------------------
namespace
{
struct RsSession
{
  unsigned magic = 0x52535345u;  // "RSSE"
  int device = 0;
  RsModel model;
  RsDeviceBatch batch{};  // device buffers this session owns; roadsurf_step sets step_begin / step_end
  cudaStream_t stream = nullptr;
  std::vector<OutputPointers> outs;
  int done = 0, fetched = 0, chunk = 1;
  int wstart = 0, wend = 0;  // common coupling window of the coupled points (0 = none)
};
RsSession* session_of(void* p)
{
  RsSession* s = static_cast<RsSession*>(p);
  return (s && s->magic == 0x52535345u) ? s : nullptr;
}
}  // namespace

int roadsurf_session_open(int npoints, OutputPointers* const* out, const InputPointers* const* in,
                          const InputSettings* settings, const InputParameters* params,
                          const LocalParameters* const* local, void** session)
{
  g_err.clear();
  if (npoints < 1 || !out || !in || !settings || !params || !local || !session)
    return fail(RS_ERR_BAD_ARGUMENT, "null argument");
  if (roadsurf_device_count() < 1) return fail(RS_ERR_NO_DEVICE, "no CUDA device visible (this library has no CPU path)");
  std::unique_ptr<RsSession, void (*)(void*)> guard(new RsSession, roadsurf_session_close);
  RsSession* s = guard.get();
  CU(cudaGetDevice(&s->device));
  {
    std::lock_guard<std::mutex> device_lock(g_device_mu[s->device & 63]);
    const int rc = set_model_on_current_device(settings, params, &s->model);
    if (rc != RS_OK) return rc;
  }
  const int sim_len = settings->SimLen, nl = s->model.nlayers;
  RsDeviceBatch& b = s->batch;
  b.npoints = npoints;
  b.ld = (npoints + 31) / 32 * 32;
  b.sim_len = sim_len;
  b.n_records = sim_len;
  b.out_stride = 1;
  b.n_out = sim_len;
  const size_t ld = b.ld;
  bool any_depth = false, any_sky = false;
  for (int p = 0; p < npoints; ++p)
  {
    const InputPointers* ip = in[p];
    if (ip->inputLen < sim_len || out[p]->outputLen < sim_len)
      return fail(RS_ERR_BAD_ARGUMENT, "inputLen/outputLen shorter than SimLen");
    if (p > 0 && !same_time_axis(*in[0], *ip, sim_len))
      return fail(RS_ERR_UNSUPPORTED, "the points of a session must share one time axis");
    const LocalParameters& lp = *local[p];
    if (sky_view_point(lp.sky_view)) any_sky = true;
    for (int t = 0; t < sim_len && !any_depth; ++t) any_depth = ip->c_Depth[t] >= 0.0;
    const long long w = window_key(s->model, lp);
    if (w > 0)
    {
      const int cend = static_cast<int>(w);
      const int cstart = (static_cast<double>(cend) <= s->model.coupling_span_real) ? 1 : cend - s->model.coupling_span;
      if (s->wend && (s->wend != cend || s->wstart != cstart))
        return fail(RS_ERR_UNSUPPORTED, "the coupled points of a session must share one coupling window");
      s->wend = cend;
      s->wstart = cstart;
    }
  }
  const int nvar = b.nvar = any_depth ? RS_F_NVAR_DEPTH : RS_F_NVAR;
  // ---- pack on the host: forcing [t][var][ld], statics, horizons; pre-fill the caller's outputs
  std::vector<double> hf(static_cast<size_t>(sim_len) * nvar * ld, 0.0), hl(RS_L_NLOCAL * ld, 0.0);
  std::vector<double> hh(any_sky ? 360 * ld : 0, 0.0);
  s->outs.resize(npoints);
  for (size_t q = 0; q < ld; ++q) local_row(q < static_cast<size_t>(npoints) ? local[q] : nullptr, &hl[q], ld);
  for (int p = 0; p < npoints; ++p)
  {
    const InputPointers* ip = in[p];
    for (int v = 0; v < nvar; ++v) forcing_row(*ip, v, sim_len, &hf[static_cast<size_t>(v) * ld + p], nvar * ld);
    if (any_sky)
      for (int k = 0; k < 360; ++k) hh[static_cast<size_t>(k) * ld + p] = ip->c_local_horizons ? ip->c_local_horizons[k] : 0.0;
    s->outs[p] = *out[p];
    for (double* o : output_planes(*out[p])) std::fill(o, o + sim_len, -9999.0);
  }
  CU(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
  // (the batch declares the inputs const: the session fills the buffers it owns through const_cast)
  CU(cudaMalloc(&b.forcing, sizeof(double) * hf.size()));
  CU(cudaMalloc(&b.local, sizeof(double) * hl.size()));
  if (any_sky) CU(cudaMalloc(&b.horizons, sizeof(double) * hh.size()));
  CU(cudaMalloc(&b.out, sizeof(double) * RS_O_NVAR * sim_len * ld));
  CU(cudaMalloc(&b.state, sizeof(double) * RS_STATE_NPLANES(nl) * ld));
  CU(cudaMalloc(&b.scratch, sizeof(double) * RS_SCRATCH_NPLANES(nl) * ld));
  CU(cudaMalloc(&b.solar, sizeof(double) * 4 * sim_len));
  CU(cudaMalloc(&b.time_fields, sizeof(int) * 6 * sim_len));
  CU(cudaMalloc(&b.status, sizeof(int) * ld));
  CU(cudaMalloc(&b.counters, sizeof(unsigned long long) * RS_CNT_N));
  CU(cudaMemcpyAsync(const_cast<double*>(b.forcing), hf.data(), sizeof(double) * hf.size(), cudaMemcpyHostToDevice,
                     s->stream));
  CU(cudaMemcpyAsync(const_cast<double*>(b.local), hl.data(), sizeof(double) * hl.size(), cudaMemcpyHostToDevice,
                     s->stream));
  if (any_sky)
    CU(cudaMemcpyAsync(const_cast<double*>(b.horizons), hh.data(), sizeof(double) * hh.size(), cudaMemcpyHostToDevice,
                       s->stream));
  const auto tf = time_fields(*in[0]);
  for (int k = 0; k < 6; ++k)
    CU(cudaMemcpyAsync(const_cast<int*>(b.time_fields) + static_cast<size_t>(k) * sim_len, tf[k], sizeof(int) * sim_len,
                       cudaMemcpyHostToDevice, s->stream));
  CU(cudaMemsetAsync(b.status, 0, sizeof(int) * ld, s->stream));
  CU(cudaMemsetAsync(b.counters, 0, sizeof(unsigned long long) * RS_CNT_N, s->stream));
  CU(static_cast<cudaError_t>(rs_launch_fill(b.out, static_cast<long long>(RS_O_NVAR) * sim_len * ld, -9999.0, s->stream)));
  CU(static_cast<cudaError_t>(rs_launch_solar(b.time_fields, sim_len, b.solar, s->stream)));
  g_launches_total += 2;
  CU(cudaStreamSynchronize(s->stream));  // the host staging vectors die with this frame
  *session = guard.release();
  return RS_OK;
}

int roadsurf_session_set_chunk(void* session, int steps)
{
  RsSession* s = session_of(session);
  if (!s) return fail(RS_ERR_BAD_ARGUMENT, "not a session");
  s->chunk = steps > 1 ? steps : 1;
  return RS_OK;
}

int roadsurf_session_done(void* session)
{
  RsSession* s = session_of(session);
  return s ? s->done : RS_ERR_BAD_ARGUMENT;
}

int roadsurf_step(void* session, int i)
{
  RsSession* s = session_of(session);
  if (!s) return fail(RS_ERR_BAD_ARGUMENT, "not a session");
  const int sim_len = s->batch.sim_len;
  if (i < 1 || i > sim_len) return fail(RS_ERR_BAD_ARGUMENT, "step outside [1, SimLen]");
  if (i <= s->done) return RS_OK;
  int current = 0;
  CU(cudaGetDevice(&current));
  if (current != s->device) CU(cudaSetDevice(s->device));
  const int begin = s->done + 1;
  int target = std::min(sim_len, std::max(i, s->done + s->chunk));
  // a coupling window [start, end + 1] is indivisible: its rewinds happen inside the kernel
  if (s->wend > 0 && begin <= s->wend + 1 && target >= s->wstart) target = std::max(target, std::min(s->wend + 1, sim_len));
  {
    std::lock_guard<std::mutex> device_lock(g_device_mu[s->device & 63]);
    // (another caller may have replaced the device's model since the session was opened)
    {
      const int rc = upload_model(s->device, s->model);
      if (rc != RS_OK) return rc;
    }
    s->batch.step_begin = begin;
    s->batch.step_end = target;
    RsLaunchInfo li;
    std::memset(&li, 0, sizeof li);
    int n = 0;
    const int rc = launch_batch(s->batch, s->model, s->stream, &li, &n);
    if (rc != RS_OK) return rc;
    g_launches_total += n;
    li.launches_total = g_launches_total;
    g_launch = li;
    CU(cudaStreamSynchronize(s->stream));
  }
  s->done = target;
  if (current != s->device) cudaSetDevice(current);
  return RS_OK;
}

int roadsurf_session_fetch(void* session, int i, int* status)
{
  RsSession* s = session_of(session);
  if (!s) return fail(RS_ERR_BAD_ARGUMENT, "not a session");
  if (i > s->done) return fail(RS_ERR_BAD_ARGUMENT, "step not executed yet: call roadsurf_step first");
  int current = 0;
  CU(cudaGetDevice(&current));
  if (current != s->device) CU(cudaSetDevice(s->device));
  // deliver every executed step not yet delivered; the steps of a coupling window were overwritten by the
  // kernel's re-runs before they became visible here
  const RsDeviceBatch& b = s->batch;
  const int t0 = s->fetched, n = s->done - s->fetched;
  if (n > 0)
  {
    std::vector<double> h(static_cast<size_t>(RS_O_NVAR) * n * b.ld);
    for (int v = 0; v < RS_O_NVAR; ++v)
      CU(cudaMemcpy(h.data() + static_cast<size_t>(v) * n * b.ld,
                    b.out + (static_cast<size_t>(v) * b.sim_len + t0) * b.ld, sizeof(double) * n * b.ld,
                    cudaMemcpyDeviceToHost));
    for (int p = 0; p < b.npoints; ++p)
    {
      const auto dst = output_planes(s->outs[p]);
      for (int v = 0; v < RS_O_NVAR; ++v)
        for (int t = 0; t < n; ++t) dst[v][t0 + t] = h[(static_cast<size_t>(v) * n + t) * b.ld + p];
    }
    s->fetched = s->done;
  }
  if (status) CU(cudaMemcpy(status, b.status, sizeof(int) * b.npoints, cudaMemcpyDeviceToHost));
  if (current != s->device) cudaSetDevice(current);
  return RS_OK;
}

void roadsurf_session_close(void* session)
{
  RsSession* s = session_of(session);
  if (!s) return;
  int current = 0;
  cudaGetDevice(&current);
  cudaSetDevice(s->device);
  const RsDeviceBatch& b = s->batch;
  for (const void* p : {static_cast<const void*>(b.forcing), static_cast<const void*>(b.local),
                        static_cast<const void*>(b.horizons), static_cast<const void*>(b.out),
                        static_cast<const void*>(b.state), static_cast<const void*>(b.scratch),
                        static_cast<const void*>(b.solar), static_cast<const void*>(b.time_fields),
                        static_cast<const void*>(b.status), static_cast<const void*>(b.counters)})
    if (p) cudaFree(const_cast<void*>(p));
  if (s->stream) cudaStreamDestroy(s->stream);
  cudaSetDevice(current);
  s->magic = 0;
  delete s;
}

const char* roadsurf_last_error(void) { return g_err.c_str(); }

const char* roadsurf_version(void) { return "roadsurf_b200 0.4 (RoadSurf 1.6.1 per-point loop, sm_100a)"; }

int roadsurf_device_count(void)
{
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess)
  {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int roadsurf_set_model(const InputSettings* settings, const InputParameters* params)
{
  if (!settings || !params) return fail(RS_ERR_BAD_ARGUMENT, "null settings/params");
  if (roadsurf_device_count() < 1) return fail(RS_ERR_NO_DEVICE, "no CUDA device visible");
  return set_model_on_current_device(settings, params, nullptr);
}

int roadsurf_run_device(const RsDeviceBatch* b, void* stream)
{
  if (!b) return fail(RS_ERR_BAD_ARGUMENT, "null batch");
  int dev = 0;
  CU(cudaGetDevice(&dev));
  RsModel m;
  {
    const int rc = current_model(dev, &m);
    if (rc != RS_OK) return rc;
  }
  if (b->ld < 32|| b->ld % 32 != 0 || b->npoints < 0 || b->npoints > b->ld)
    return fail(RS_ERR_BAD_ARGUMENT, "ld must be a positive multiple of 32 and >= npoints");
  const RsDeviceBatch d = with_defaults(*b);
  const int step_begin = d.step_begin, step_end = d.step_end, forcing_step0 = d.forcing_step0;
  if (b->sim_len < 1 || b->out_stride < 1 || b->n_out < 1)
    return fail(RS_ERR_BAD_ARGUMENT, "bad sim_len / out_stride / n_out");
  if (step_begin > step_end || step_end > b->sim_len || forcing_step0 > step_begin || b->out_slot0 < 0)
    return fail(RS_ERR_BAD_ARGUMENT, "bad step_begin / step_end / forcing_step0 / out_slot0");
  if (b->out_start < 0 || b->out_start >= b->sim_len) return fail(RS_ERR_BAD_ARGUMENT, "out_start outside [0, sim_len)");
  if (b->out_nvar != 0 && b->out_nvar != RS_O_NVAR && b->out_nvar != RS_O_NVAR_EXT)
    return fail(RS_ERR_BAD_ARGUMENT, "out_nvar must be 0, RS_O_NVAR or RS_O_NVAR_EXT");
  {
    int s0, s1;
    slot_range(step_begin, step_end, b->out_start, b->out_stride, &s0, &s1);
    if (s1 > s0 && (s0 < b->out_slot0 || s1 - b->out_slot0 > b->n_out))
      return fail(RS_ERR_BAD_ARGUMENT, "out tensor does not cover the output slots of [step_begin, step_end]");
  }
  if (step_begin > 1 && !b->state) return fail(RS_ERR_BAD_ARGUMENT, "step_begin > 1 needs batch->state from the previous chunk");
  if (b->nvar != RS_F_NVAR && b->nvar != RS_F_NVAR_DEPTH) return fail(RS_ERR_BAD_ARGUMENT, "nvar must be 11 or 12");
  if (!b->forcing || !b->time_fields || !b->local || !b->out || !b->status || !b->solar)
    return fail(RS_ERR_BAD_ARGUMENT, "null device pointer in batch");
  if (b->forcing_mode == 0)
  {
    if (b->n_records < step_end - forcing_step0 + 1)
      return fail(RS_ERR_BAD_ARGUMENT, "forcing_mode 0 needs n_records >= step_end - forcing_step0 + 1");
  }
  else if (b->forcing_mode == 1 || b->forcing_mode == 2)
  {
    if (b->n_records < 2 || !b->record_step) return fail(RS_ERR_BAD_ARGUMENT, "coarse forcing needs >= 2 records");
    if (b->forcing_mode == 2)
    {
      if (!b->expand_workspace || b->expand_steps < 1)
        return fail(RS_ERR_BAD_ARGUMENT, "forcing_mode 2 needs expand_workspace and expand_steps >= 1");
      if (b->expand_steps < step_end - step_begin + 1 && !b->state)
        return fail(RS_ERR_BAD_ARGUMENT, "forcing_mode 2 in several chunks needs batch->state");
    }
  }
  else
    return fail(RS_ERR_BAD_ARGUMENT, "forcing_mode must be 0, 1 or 2");
  if (m.use_coupling && !b->scratch) return fail(RS_ERR_BAD_ARGUMENT, "coupling needs batch->scratch");
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  CU(static_cast<cudaError_t>(rs_launch_solar(b->time_fields, b->sim_len, b->solar, st)));
  RsLaunchInfo li;
  std::memset(&li, 0, sizeof li);
  int n = 0;
  {
    const int rc = launch_batch(d, m, st, &li, &n);
    if (rc != RS_OK) return rc;
  }
  {
    const int rc = note_async_launch(dev, st);
    if (rc != RS_OK) return rc;
  }
  li.launches_total = g_launches_total += 1 + n;  // the solar table and the model run
  g_launch = li;
  return RS_OK;
}

int roadsurf_expand_records(const RsDeviceBatch* b, int rule, int step_begin, int step_end, double* dst, void* stream)
{
  if (!b || !dst || !b->forcing || !b->record_step || b->n_records < 2 || (rule != 1 && rule != 2) || step_begin < 1 ||
      step_end < step_begin || b->ld < 32 || b->ld % 32 != 0)
    return fail(RS_ERR_BAD_ARGUMENT, "bad arguments");
  int dev = 0;
  CU(cudaGetDevice(&dev));
  RsModel m;
  {
    const int rc = current_model(dev, &m);
    if (rc != RS_OK) return rc;
  }
  CU(static_cast<cudaError_t>(rs_launch_expand(b->forcing, b->record_step, b->n_records, b->nvar, b->ld, b->npoints, rule, m.DT,
                                                step_begin, step_end, dst, stream)));
  ++g_launches_total;
  return RS_OK;
}

int roadsurf_sun_position(const int* time_fields, int n_steps, const double* lat, const double* lon, int npoints,
                          double* elevation, double* azimuth, void* stream)
{
  if (!time_fields || !lat || !lon || !elevation || !azimuth || n_steps < 1 || npoints < 1 || n_steps > 65535)
    return fail(RS_ERR_BAD_ARGUMENT, "bad arguments (n_steps <= 65535 per call)");
  CU(static_cast<cudaError_t>(rs_launch_sun_position(time_fields, n_steps, lat, lon, npoints, elevation, azimuth, stream)));
  ++g_launches_total;
  return RS_OK;
}

int roadsurf_order_points(const double* local, int ld, int npoints, int* order, void* stream)
{
  if (!local || !order || ld < 32 || ld % 32 != 0 || npoints < 0 || npoints > ld)
    return fail(RS_ERR_BAD_ARGUMENT, "bad arguments");
  CU(static_cast<cudaError_t>(
      rs_launch_partition(local + static_cast<size_t>(RS_L_SKY_VIEW) * ld, ld, npoints, 2, order, nullptr, stream)));
  ++g_launches_total;
  return RS_OK;
}

int roadsurf_transpose_to_soa(const double* src, int64_t src_ld, int npoints, int n, double* dst, int ld,
                              void* stream)
{
  if (!src || !dst || npoints < 0 || n < 0 || ld < npoints || src_ld < n)
    return fail(RS_ERR_BAD_ARGUMENT, "bad arguments (ld >= npoints >= 0, src_ld >= n >= 0)");
  if (npoints == 0 || n == 0) return RS_OK;
  CU(static_cast<cudaError_t>(rs_launch_transpose_to_soa(src, src_ld, npoints, n, dst, ld, stream)));
  ++g_launches_total;
  return RS_OK;
}

int roadsurf_transpose_from_soa(const double* src, int ld, int npoints, int n, double* dst, int64_t dst_ld,
                                void* stream)
{
  if (!src || !dst || npoints < 0 || n < 0 || ld < npoints || dst_ld < n)
    return fail(RS_ERR_BAD_ARGUMENT, "bad arguments (ld >= npoints >= 0, dst_ld >= n >= 0)");
  if (npoints == 0 || n == 0) return RS_OK;
  CU(static_cast<cudaError_t>(rs_launch_transpose_from_soa(src, ld, npoints, n, dst, dst_ld, stream)));
  ++g_launches_total;
  return RS_OK;
}

int roadsurf_eval_primitive(int fn, const double* a, const double* b, double* out, int64_t n, void* stream)
{
  const bool binary = fn == RS_PRIM_FRCP || fn == RS_PRIM_FDIV || fn == RS_PRIM_DIV_CONST;
  if (fn < 0 || fn >= RS_PRIM_N || n < 0 || !a || !out || (binary && !b))
    return fail(RS_ERR_BAD_ARGUMENT, "bad arguments (fn one of RS_PRIM_*, n >= 0, b where fn reads it)");
  if (n == 0) return RS_OK;
  CU(static_cast<cudaError_t>(rs_launch_eval_primitive(fn, a, b, out, n, stream)));
  ++g_launches_total;
  return RS_OK;
}

int roadsurf_fill(double* dst, int64_t n, double value, void* stream)
{
  if (!dst || n < 0) return fail(RS_ERR_BAD_ARGUMENT, "bad arguments (dst, n >= 0)");
  if (n == 0) return RS_OK;
  CU(static_cast<cudaError_t>(rs_launch_fill(dst, n, value, stream)));
  ++g_launches_total;
  return RS_OK;
}

double roadsurf_measure_fp64_tflops(int iterations)
{
  if (roadsurf_device_count() < 1)
  {
    fail(RS_ERR_NO_DEVICE, "no CUDA device visible");
    return -1.0;
  }
  return rs_measure_fp64(iterations > 0 ? iterations : 20000);
}

void roadsurf_release_workspace(void)
{
  // frees the pooled device and pinned buffers of every device (they are re-created on demand)
  std::lock_guard<std::mutex> lk(g_pool_mu);
  int current = 0;
  cudaGetDevice(&current);
  for (auto& kv : g_pool)
    if (kv.second.p)
    {
      cudaSetDevice(kv.first.first);
      cudaFree(kv.second.p);
    }
  g_pool.clear();
  for (auto& kv : g_pinned_pool)
    if (kv.second.p) cudaFreeHost(kv.second.p);
  g_pinned_pool.clear();
  cudaSetDevice(current);
}

int roadsurf_set_option(const char* name, int value)
{
  if (name && std::strcmp(name, "forcing_staging") == 0)
  {
    g_opt_staging = value ? 1 : 0;
    return RS_OK;
  }
  if (name && std::strcmp(name, "coupling_compaction_passes") == 0)
  {
    g_opt_compaction = value > 0 ? (value > 30 ? 30 : value) : 0;
    return RS_OK;
  }
  if (name && std::strcmp(name, "spread_small") == 0)
  {
    rs_set_spread_small(value);
    return RS_OK;
  }
  if (name && std::strcmp(name, "latency_body") == 0)
  {
    rs_set_latency_body(value);
    return RS_OK;
  }
  if (name && std::strcmp(name, "write_back_inputs") == 0)
  {
    g_opt_write_back = value ? 1 : 0;
    return RS_OK;
  }
  if (name && std::strcmp(name, "max_points_per_device_batch") == 0)
  {
    g_opt_max_slots = value > 0 ? value : 0;
    return RS_OK;
  }
  return fail(RS_ERR_BAD_ARGUMENT, "unknown option");
}

long long roadsurf_selftest_libm(long long n, unsigned long long seed, long long* mismatches)
{
  unsigned long long s = seed * 0x9E3779B97F4A7C15ull + 0x632BE59BD9B4E019ull;
  auto next = [&]() {
    s ^= s << 13;
    s ^= s >> 7;
    s ^= s << 17;
    return s;
  };
  auto same = [](double a, double b) { return !std::memcmp(&a, &b, sizeof a); };
  long long bad_e = 0, bad_l = 0;
  for (long long k = 0; k < n; ++k)
  {
    const double u = static_cast<double>(next() >> 11) * 0x1p-53;
    double x, y;
    switch (k & 3)
    {
      case 0: x = (u - 0.5) * 20; y = 1.0 + u * 0.2; break;               // Magnus exponents; weakly unstable
      case 1: x = (u - 0.5) * 1000; y = std::ldexp(1.0 + u, static_cast<int>(next() % 600) - 300); break;
      case 2: x = (u - 0.5) * 1e-3; y = 0.9 + u * 0.2; break;             // around exp(0), log(1)
      default: x = -u * 6; y = 1.0 + u * 40; break;                       // decays; strongly unstable
    }
    bool ok;
    const double e = rslibm::exp_fast(x, ok);
    if (ok && !same(e, std::exp(x))) ++bad_e;
    const double l = rslibm::log_fast(y, ok);
    if (ok && !same(l, std::log(y))) ++bad_l;
  }
  if (mismatches)
  {
    mismatches[0] = bad_e;
    mismatches[1] = bad_l;
  }
  return n;
}

long long roadsurf_selftest_arith(long long n, unsigned long long seed, long long* mismatches)
{
  if (roadsurf_device_count() < 1)
  {
    fail(RS_ERR_NO_DEVICE, "no CUDA device visible");
    return -1;
  }
  return rs_selftest_arith(n, seed, mismatches);
}

void roadsurf_last_launch(RsLaunchInfo* info)
{
  if (info)
  {
    *info = g_launch;
    info->launches_total = g_launches_total;
  }
}

int roadsurf_read_input_derive(int npoints, const InputPointers* const* in, const InputSettings* settings,
                               int forecast_step, const int* latest_obs_index, LocalParameters* const* local,
                               int* ok)
{
  if (npoints < 0 || !settings || (npoints > 0 && (!in || !local))) return fail(RS_ERR_BAD_ARGUMENT, "null argument");
  const int sim_len = settings->SimLen;
  const int span = static_cast<int>(settings->coupling_minutes * 60 / settings->DTSecs);
  auto missing = [](double x) { return std::isnan(x) || x < -9000; };  // roadrunner.cpp:40-43
  parallel_for(npoints, host_threads(), [&](int p) {
    const InputPointers* ip = in[p];
    LocalParameters* lp = local[p];
    const int n = std::min(sim_len, ip->inputLen);
    bool good = true;
    for (int t = 0; t < n && good; ++t)
      good = !(missing(ip->c_tair[t]) || missing(ip->c_Rhz[t]) || missing(ip->c_prec[t]) || missing(ip->c_SW[t]) ||
               missing(ip->c_LW[t]) || missing(ip->c_VZ[t]));
    if (ok) ok[p] = good ? 1 : 0;
    if (!good) return;
    lp->InitLenI = 1 + forecast_step;
    if (settings->use_relaxation == 1)
    {
      lp->tair_relax = lp->VZ_relax = lp->RH_relax = -9999.9;
      const int last = latest_obs_index ? latest_obs_index[p] : -9999;
      if (last > -1 && last < n)
      {
        lp->InitLenI = last;
        lp->tair_relax = ip->c_tair[last];
        lp->VZ_relax = ip->c_VZ[last];
        lp->RH_relax = ip->c_Rhz[last];
      }
    }
    if (settings->use_coupling == 1)
    {
      lp->couplingTsurf = -9999.9;
      lp->couplingIndexI = -9999;
      double* obs = ip->c_TSurfObs;
      int i = n - 1;
      while (i >= 0 && (missing(obs[i]) || obs[i] < -100)) --i;
      if (i >= span)
      {
        lp->couplingTsurf = obs[i];
        lp->couplingIndexI = i;
        for (int j = i; j > i - span; --j) obs[j] = -9999.9;
      }
    }
  });
  return RS_OK;
}

int roadsurf_read_input_derive_records(const RsHostBatch* b, const InputSettings* settings, int forecast_step,
                                       const int* latest_obs_index, double* local, int* window_end)
{
  if (!b || !settings || !local || !b->forcing || !b->record_step || b->forcing_mode != 1 || b->n_records < 2 ||
      b->npoints < 0 || (b->nvar != RS_F_NVAR && b->nvar != RS_F_NVAR_DEPTH))
    return fail(RS_ERR_BAD_ARGUMENT, "needs a coarse-record host batch");
  {
    const int rc = check_record_grid(b->record_step, b->n_records);
    if (rc != RS_OK) return rc;
  }
  const int sim_len = settings->SimLen, nrec = b->n_records;
  const size_t np = static_cast<size_t>(b->npoints), nvar = static_cast<size_t>(b->nvar);
  const double DT = settings->DTSecs;
  const int span = static_cast<int>(settings->coupling_minutes * 60 / DT);
  const int* rs = b->record_step;
  auto rec = [&](int k, int v, size_t p) { return b->forcing[(static_cast<size_t>(k) * nvar + v) * np + p]; };
  // the value JsonSource's interpolation gives at vector index t (the kernel's fetch_coarse rule)
  auto value_at = [&](int v, size_t p, int t) {
    return record_value_at(rs, nrec, DT, t, [&](int k) { return rec(k, v, p); });
  };
  // vector indices [lo, hi] served by bracket k (the first one reaches back to index 0); false if empty.
  // Indices at or after the last record are served by nobody: the reference's interpolation stops at its
  // last raw record (JsonSource.cpp:85), those steps stay missing and read_input rejects the point.
  auto bracket_range = [&](int k, int& lo, int& hi) {
    lo = (k == 0) ? 0 : std::max(rs[k], 0);
    hi = std::min(rs[k + 1] - 1, sim_len - 1);
    return lo <= hi;
  };
  const bool records_cover_run = rs[nrec - 1] > sim_len - 1;
  parallel_for(b->npoints, host_threads(), [&](int pi) {
    const size_t p = static_cast<size_t>(pi);
    double* L = local + p;
    // ---- screening.  Bracket k serves the vector indices [lo, hi]; an index above rs[k] needs both
    // records valid, the index rs[k] itself only record k
    bool good = records_cover_run;
    const int req[6] = {RS_F_TAIR, RS_F_RHZ, RS_F_PREC, RS_F_SW, RS_F_LW, RS_F_VZ};
    for (int k = 0; k + 1 < nrec && good; ++k)
    {
      int lo, hi;
      if (!bracket_range(k, lo, hi)) continue;
      const bool at_a = lo <= rs[k] && rs[k] <= hi, above = hi >= std::max(rs[k] + 1, lo);
      for (int r = 0; r < 6 && good; ++r)
      {
        const bool va = rec(k, req[r], p) > -100.0, vb = rec(k + 1, req[r], p) > -100.0;
        if ((at_a && !va) || (above && !(va && vb))) good = false;
      }
    }
    L[RS_L_ACTIVE * np] = good ? 1.0 : 0.0;
    if (!good) return;
    L[RS_L_INIT_LEN * np] = 1 + forecast_step;
    if (settings->use_relaxation == 1)
    {
      L[RS_L_TAIR_RELAX * np] = L[RS_L_VZ_RELAX * np] = L[RS_L_RH_RELAX * np] = -9999.9;
      const int last = latest_obs_index ? latest_obs_index[pi] : -9999;
      if (last > -1 && last < sim_len)
      {
        L[RS_L_INIT_LEN * np] = last;
        L[RS_L_TAIR_RELAX * np] = value_at(RS_F_TAIR, p, last);
        L[RS_L_VZ_RELAX * np] = value_at(RS_F_VZ, p, last);
        L[RS_L_RH_RELAX * np] = value_at(RS_F_RHZ, p, last);
      }
    }
    if (settings->use_coupling == 1)
    {
      L[RS_L_COUPLING_TSURF * np] = -9999.9;
      L[RS_L_COUPLING_INDEX * np] = -9999;
      // latest vector index with a valid interpolated observation
      int i = -1;
      for (int k = nrec - 2; k >= 0 && i < 0; --k)
      {
        int lo, hi;
        if (!bracket_range(k, lo, hi)) continue;
        const bool va = rec(k, RS_F_TSURFOBS, p) > -100.0, vb = rec(k + 1, RS_F_TSURFOBS, p) > -100.0;  // NaN fails
        if (va && vb && hi >= std::max(rs[k] + 1, lo))
          i = hi;
        else if (va && lo <= rs[k] && rs[k] <= hi)
          i = rs[k];
      }
      const double obs = (i >= 0) ? value_at(RS_F_TSURFOBS, p, i) : -9999.9;
      if (i >= span)
      {
        L[RS_L_COUPLING_TSURF * np] = obs;
        L[RS_L_COUPLING_INDEX * np] = i;
      }
    }
  });
  if (window_end)
  {
    const int w = settings->use_coupling == 1 ? common_window_end(local, np) : 0;
    *window_end = w < 0 ? 0 : w;  // windows that differ: no common window
  }
  return RS_OK;
}

void roadsurf_last_batch_stats(RsBatchStats* stats)
{
  if (stats) *stats = g_stats;
}

int roadsurf_run_batch(int npoints, OutputPointers* const* out, const InputPointers* const* in,
                       const InputSettings* settings, const InputParameters* params,
                       const LocalParameters* const* local, int ngpus, int* status)
{
  g_err.clear();
  std::memset(&g_stats, 0, sizeof g_stats);
  if (npoints < 0 || !settings || !params || (npoints > 0 && (!out || !in || !local)))
    return fail(RS_ERR_BAD_ARGUMENT, "null argument");
  if (roadsurf_device_count() < 1)
    return fail(RS_ERR_NO_DEVICE, "no CUDA device visible (this library has no CPU path)");
  if (npoints == 0) return RS_OK;
  return run_sharded(npoints, ngpus,
                     [&](Shard& sh) { return run_shard(sh, out, in, settings, params, local, status); });
}

}  // extern "C" (entry points above)

// The reference's mains call runsimulation from a pool of host threads, one point per call
// (examples/example1/src/roadrunner.cpp:454-496).  One point per launch would leave the GPU at its
// single-warp latency (~8 us per model step), so concurrent callers are combined: the first caller
// becomes the leader and runs everything that is queued as ONE batch, the others sleep until their
// point is done; while a batch is on the device the next one accumulates.  A lone caller pays only a
// mutex.  Calls with different settings / parameters go into different batches.
namespace
{
struct PendingCall
{
  OutputPointers* out;
  const InputPointers* in;
  const InputSettings* settings;
  const InputParameters* params;
  const LocalParameters* local;
  int rc = RS_OK;
  bool done = false;
  std::string err;
};
std::mutex g_call_mu;
std::condition_variable g_call_cv;
std::vector<PendingCall*> g_call_queue;
bool g_call_leader = false;
size_t g_call_last_n = 0;     // calls in the last batch (0 = no batch yet); guarded by g_call_mu
double g_call_last_ms = 0.0;  // wall time of the last batch
std::atomic<long long> g_calls_total{0}, g_call_batches_total{0};

void mark_not_computed(OutputPointers* outPointers, const InputSettings* inSettings)
{
  // The reference signature has no error channel: leave the outputs at -9999.0, which is how the
  // reference marks "not computed" (src/Initialization.f90:397-412).
  if (!outPointers || !inSettings) return;
  for (double* o : output_planes(*outPointers))
    if (o)
      for (int t = 0; t < inSettings->SimLen && t < outPointers->outputLen; ++t) o[t] = -9999.0;
}
}  // namespace

extern "C" void roadsurf_runsimulation_counters(long long* calls, long long* batches)
{
  if (calls) *calls = g_calls_total.load();
  if (batches) *batches = g_call_batches_total.load();
}

extern "C" void runsimulation(OutputPointers* outPointers, const InputPointers* inPointers,
                              const InputSettings* inSettings, const InputParameters* inputParam,
                              const LocalParameters* localParam)
{
  if (!outPointers || !inPointers || !inSettings || !inputParam || !localParam)
  {
    std::fprintf(stderr, "roadsurf_b200 runsimulation failed: null argument\n");
    mark_not_computed(outPointers, inSettings);
    return;
  }
  // arguments that would fail a whole batch are rejected here, for this caller only
  if (inPointers->inputLen < inSettings->SimLen || outPointers->outputLen < inSettings->SimLen)
  {
    std::fprintf(stderr, "roadsurf_b200 runsimulation failed: inputLen/outputLen shorter than SimLen\n");
    mark_not_computed(outPointers, inSettings);
    return;
  }
  PendingCall me;
  me.out = outPointers;
  me.in = inPointers;
  me.settings = inSettings;
  me.params = inputParam;
  me.local = localParam;
  std::unique_lock<std::mutex> lk(g_call_mu);
  g_call_queue.push_back(&me);
  while (!me.done)
  {
    if (g_call_leader)
    {
      // a leader is at work: it will run this call, or hand the leadership over when its own is done
      g_call_cv.wait(lk, [&] { return me.done || !g_call_leader; });
      continue;
    }
    // become the leader for ONE batch: everything queued with the same settings and parameters as this call
    g_call_leader = true;
    // Callers of a thread pool come back together after a batch, staggered by whatever each does between two
    // calls (reading the next point, writing the last one out).  A batch costs about the same whatever its
    // size, so the leader waits for the pool to queue up again: until as many calls wait as the last batch
    // held, bounded by a fifth of the last batch's run time (1..20 ms).  With no history (first batch) or a
    // lone caller (last batch of 1) the bound is: at least 1 ms resp. no wait at all, and stop once the queue
    // has not grown for 1 ms.
    {
      using clock = std::chrono::steady_clock;
      const size_t expected = g_call_last_n;
      if (expected != 1)
      {
        const double budget_ms = std::min(20.0, std::max(1.0, 0.2 * g_call_last_ms));
        const auto t0 = clock::now();
        auto last_growth = t0;
        size_t seen = g_call_queue.size();
        while (g_call_queue.size() < expected || expected == 0)
        {
          g_call_cv.wait_for(lk, std::chrono::microseconds(250), [] { return false; });
          const auto now = clock::now();
          if (g_call_queue.size() != seen)
          {
            seen = g_call_queue.size();
            last_growth = now;
          }
          const double waited = std::chrono::duration<double, std::milli>(now - t0).count();
          const double idle = std::chrono::duration<double, std::milli>(now - last_growth).count();
          if (waited >= budget_ms) break;
          if (expected == 0 && waited >= 1.0 && idle >= 1.0) break;
        }
      }
    }
    std::vector<PendingCall*> batch, rest;
    for (PendingCall* c : g_call_queue)
    {
      const bool same = !std::memcmp(c->settings, me.settings, sizeof(InputSettings)) &&
                        !std::memcmp(c->params, me.params, sizeof(InputParameters));
      (same ? batch : rest).push_back(c);
    }
    g_call_queue.swap(rest);
    lk.unlock();
    const int n = static_cast<int>(batch.size());
    g_calls_total += n;
    ++g_call_batches_total;
    std::vector<OutputPointers*> outs(n);
    std::vector<const InputPointers*> ins(n);
    std::vector<const LocalParameters*> locs(n);
    for (int k = 0; k < n; ++k)
    {
      outs[k] = batch[k]->out;
      ins[k] = batch[k]->in;
      locs[k] = batch[k]->local;
    }
    const auto run_t0 = std::chrono::steady_clock::now();
    const int rc = roadsurf_run_batch(n, outs.data(), ins.data(), me.settings, me.params, locs.data(), 1, nullptr);
    const std::string err = (rc != RS_OK) ? std::string(roadsurf_last_error()) : std::string();
    lk.lock();
    g_call_last_n = static_cast<size_t>(n);
    g_call_last_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - run_t0).count();
    for (PendingCall* c : batch)
    {
      c->rc = rc;
      c->err = err;
      c->done = true;
    }
    // this caller's own call is in `batch`, hence done: the leadership goes to whoever still waits
    g_call_leader = false;
    g_call_cv.notify_all();
  }
  lk.unlock();
  if (me.rc != RS_OK)
  {
    std::fprintf(stderr, "roadsurf_b200 runsimulation failed: %s\n", me.err.c_str());
    g_err = me.err;
    mark_not_computed(outPointers, inSettings);
  }
}


// ---- ensemble runs (include/roadsurf_b200.h, part 3) -------------------------------------------------
namespace
{
int check_stats_spec(const RsEnsembleStatsSpec& s, int out_nvar)
{
  if (s.n_quantiles < 0 || s.n_quantiles > RS_ENS_MAX_QUANTILES || s.n_thresholds < 0 ||
      s.n_thresholds > RS_ENS_MAX_THRESHOLDS)
    return fail(RS_ERR_BAD_ARGUMENT, "at most 8 quantiles and 8 thresholds");
  for (int j = 0; j < s.n_quantiles; ++j)
    if (!(s.quantiles[j] >= 0.0 && s.quantiles[j] <= 1.0)) return fail(RS_ERR_BAD_ARGUMENT, "quantiles lie in [0, 1]");
  for (int j = 0; j < s.n_thresholds; ++j)
    if (s.thresholds[j].plane < 0 || s.thresholds[j].plane >= out_nvar || s.thresholds[j].op < RS_ENS_LT ||
        s.thresholds[j].op > RS_ENS_GE)
      return fail(RS_ERR_BAD_ARGUMENT, "threshold plane outside the output planes or unknown comparison");
  if (s.n_events < 0 || s.n_events > RS_ENS_MAX_EVENTS) return fail(RS_ERR_BAD_ARGUMENT, "at most 8 events");
  for (int j = 0; j < s.n_events; ++j)
  {
    const RsEnsembleEvent& ev = s.events[j];
    if (ev.n_conditions < 1 || ev.n_conditions > RS_ENS_MAX_CONDITIONS)
      return fail(RS_ERR_BAD_ARGUMENT, "an event has 1 to 4 conditions");
    if (ev.window < 1) return fail(RS_ERR_BAD_ARGUMENT, "an event window is at least 1 output slot");
    for (int c = 0; c < ev.n_conditions; ++c)
      if (ev.conditions[c].plane < 0 || ev.conditions[c].plane >= out_nvar || ev.conditions[c].op < RS_ENS_LT ||
          ev.conditions[c].op > RS_ENS_GE)
        return fail(RS_ERR_BAD_ARGUMENT, "event condition plane outside the output planes or unknown comparison");
  }
  return RS_OK;
}

// The statistics kernel (when stats, or prob with thresholds, is given), then the events kernel (when prob is given
// and the spec has events), on `stream`.  The spec has been checked.
int launch_stats_and_events(const double* member_out, int out_nvar, int n_slots, int mo_slots, int ldm, int npoints,
                            int members, const RsEnsembleStatsSpec* spec, double* stats, double* prob, int st_slots, int ld,
                            void* stream)
{
  if (stats || (prob && spec->n_thresholds > 0))
  {
    CU(static_cast<cudaError_t>(rs_launch_ens_stats(member_out, out_nvar, n_slots, mo_slots, ldm, npoints, members, spec,
                                                    stats, prob, st_slots, ld, stream)));
    ++g_launches_total;
  }
  if (prob && spec->n_events > 0)
  {
    CU(static_cast<cudaError_t>(
        rs_launch_ens_events(member_out, n_slots, mo_slots, ldm, npoints, members, spec, prob, st_slots, ld, stream)));
    ++g_launches_total;
  }
  return RS_OK;
}

// ---- area event probabilities (RsEnsembleAreas) ----
// Every index the area kernels use comes from here: the arrays are checked against npoints on the host.
// `events`: an area event or onset output is asked for, so the spec needs events.
int check_areas(const RsEnsembleAreas* areas, int npoints, const RsEnsembleStatsSpec& spec, bool events = true)
{
  if (!areas || !areas->offsets || !areas->stations) return fail(RS_ERR_BAD_ARGUMENT, "null area pointer (areas, offsets or stations)");
  if (areas->n_areas < 1) return fail(RS_ERR_BAD_ARGUMENT, "n_areas must be at least 1");
  if (events && spec.n_events == 0) return fail(RS_ERR_BAD_ARGUMENT, "area probabilities need at least one event in the spec");
  const int* o = areas->offsets;
  if (o[0] != 0) return fail(RS_ERR_BAD_ARGUMENT, "area offsets[0] must be 0");
  for (int a = 0; a < areas->n_areas; ++a)
    if (o[a + 1] <= o[a]) return fail(RS_ERR_BAD_ARGUMENT, "area offsets must be strictly increasing (no empty area)");
  for (int k = 0; k < o[areas->n_areas]; ++k)
    if (areas->stations[k] < 0 || areas->stations[k] >= npoints)
      return fail(RS_ERR_BAD_ARGUMENT, "area station index outside [0, npoints)");
  return RS_OK;
}

// The library's copy of a checked area set: each area's stations sorted, without repeats, and the segments that the
// accumulate kernel takes, {area, begin, end, 0}: a run of stations of one area, all in one station chunk.
struct AreaPlan
{
  int n_areas = 0;
  std::vector<int> stations;  // area after area
  std::vector<int> first;     // [n_areas + 1]: area a is stations[first[a] .. first[a + 1] - 1]
  std::vector<int> segments;  // [n][4], every chunk's in chunk order
};

AreaPlan plan_areas(const RsEnsembleAreas& a)
{
  AreaPlan pl;
  pl.n_areas = a.n_areas;
  pl.first.push_back(0);
  for (int k = 0; k < a.n_areas; ++k)
  {
    const size_t b = pl.stations.size();
    pl.stations.insert(pl.stations.end(), a.stations + a.offsets[k], a.stations + a.offsets[k + 1]);
    std::sort(pl.stations.begin() + b, pl.stations.end());
    pl.stations.erase(std::unique(pl.stations.begin() + b, pl.stations.end()), pl.stations.end());
    pl.first.push_back(static_cast<int>(pl.stations.size()));
  }
  return pl;
}

// Stations per segment: enough segments that the accumulate kernel has about 2^15 work items (one warp each) per
// chunk, so that a small ensemble spreads over the GPU, and no more, so that a large one makes few atomics and
// reads a segment's member values in one pass; between 1 and 64.  `per_station`: the work items of one station.
int segment_length(const AreaPlan& pl, long long per_station, long long chunks)
{
  const long long items = static_cast<long long>(pl.stations.size()) * per_station;
  return static_cast<int>(std::min<long long>(64, std::max<long long>(1, items / (chunks << 15))));
}

int area_segment_length(const AreaPlan& pl, int n_events, int n_slots, long long chunks)
{
  return segment_length(pl, static_cast<long long>(n_events) * rs_area_tiles(n_slots), chunks);
}

// Appends the segments of the stations [p0, p0 + n), at most `len` stations each, and returns their count.
int plan_segments(AreaPlan& pl, long long p0, long long n, int len)
{
  const size_t n0 = pl.segments.size();
  for (int a = 0; a < pl.n_areas; ++a)
  {
    const auto b = pl.stations.begin();
    const int lo = static_cast<int>(std::lower_bound(b + pl.first[a], b + pl.first[a + 1], p0) - b);
    const int hi = static_cast<int>(std::lower_bound(b + pl.first[a], b + pl.first[a + 1], p0 + n) - b);
    for (int k = lo; k < hi; k += len) pl.segments.insert(pl.segments.end(), {a, k, std::min(k + len, hi), 0});
  }
  return static_cast<int>((pl.segments.size() - n0) / 4);
}

// Device copy of a plan and its accumulators in one buffer of area_bytes(): the accumulators
// [n_areas][n_events][tiles][members] (valid, then hit), the segments, the stations.  `max_segments` bounds the
// plan's segments where the buffer is sized before they are planned (a segment holds one station at least).
struct AreaDevice
{
  size_t words = 0;  // accumulator words of each kind
  unsigned long long *valid = nullptr, *hit = nullptr;
  int *segments = nullptr, *stations = nullptr;
};

size_t area_bytes(const AreaPlan& pl, int n_events, int n_slots, int members, size_t max_segments)
{
  const size_t words = static_cast<size_t>(pl.n_areas) * n_events * rs_area_tiles(n_slots) * members;
  return 2 * sizeof(unsigned long long) * words + sizeof(int) * (4 * max_segments + pl.stations.size());
}

// Places the buffer's parts, uploads the plan and resets the accumulators (all valid, no hit) on `st`; returns the
// bytes copied to the device in *h2d.
int area_upload(const AreaPlan& pl, int n_events, int n_slots, int members, void* base, cudaStream_t st, AreaDevice* d,
                size_t* h2d)
{
  d->words = static_cast<size_t>(pl.n_areas) * n_events * rs_area_tiles(n_slots) * members;
  d->valid = static_cast<unsigned long long*>(base);
  d->hit = d->valid + d->words;
  d->segments = reinterpret_cast<int*>(d->hit + d->words);  // 16-byte aligned: 2 * words * 8 bytes from base
  d->stations = d->segments + pl.segments.size();
  CU(cudaMemsetAsync(d->valid, 0xff, sizeof(unsigned long long) * d->words, st));
  CU(cudaMemsetAsync(d->hit, 0, sizeof(unsigned long long) * d->words, st));
  CU(cudaMemcpyAsync(d->segments, pl.segments.data(), sizeof(int) * pl.segments.size(), cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d->stations, pl.stations.data(), sizeof(int) * pl.stations.size(), cudaMemcpyHostToDevice, st));
  *h2d = sizeof(int) * (pl.segments.size() + pl.stations.size());
  return RS_OK;
}

int area_accumulate(const AreaDevice& d, const double* member_out, int n_slots, int mo_slots, int ldm, int members,
                    const RsEnsembleStatsSpec* spec, int p0, int first_segment, int n_segments, cudaStream_t st)
{
  if (n_segments == 0 || n_slots == 0) return RS_OK;
  CU(static_cast<cudaError_t>(rs_launch_ens_area_accumulate(member_out, n_slots, mo_slots, ldm, members, spec, d.stations,
                                                            p0, d.segments + 4 * static_cast<size_t>(first_segment),
                                                            n_segments, d.valid, d.hit, st)));
  ++g_launches_total;
  return RS_OK;
}

int area_finalize(const AreaDevice& d, int n_areas, int n_events, int n_slots, int members, double* area_prob, int st_slots,
                  cudaStream_t st)
{
  if (n_slots == 0) return RS_OK;
  CU(static_cast<cudaError_t>(
      rs_launch_ens_area_finalize(d.valid, d.hit, n_areas, n_events, n_slots, members, area_prob, st_slots, st)));
  ++g_launches_total;
  return RS_OK;
}

// ---- event onset (roadsurf_ensemble_onset) ----
// Which outputs may go together, before any device work.  `device`: roadsurf_ensemble_onset, which has no area_prob
// and needs one output at least.  Areas may go with area_ext_stats alone (host entry with window extremes).
int check_onset_outputs(const RsEnsembleStatsSpec& spec, const double* onset, const RsEnsembleAreas* areas,
                        const double* area_prob, const double* area_onset, bool device,
                        const double* area_ext_stats = nullptr)
{
  if (device && !onset && !area_onset) return fail(RS_ERR_BAD_ARGUMENT, "onset and area_onset are both NULL");
  if ((onset || area_onset) && spec.n_events == 0)
    return fail(RS_ERR_BAD_ARGUMENT, "event onset needs at least one event in the spec");
  if (!areas && (area_prob || area_onset))
    return fail(RS_ERR_BAD_ARGUMENT, "null area pointer: area_prob and area_onset need areas");
  if (areas && !area_prob && !area_onset && !area_ext_stats)
    return fail(RS_ERR_BAD_ARGUMENT, device ? "null area pointer: areas need area_onset"
                                            : "null area pointer: areas need area_prob or area_onset");
  return RS_OK;
}

// Area onset accumulators [n_areas][n_events][members] {O, X}, in ints.
size_t onset_acc_ints(int n_areas, int n_events, int members)
{
  return 2 * static_cast<size_t>(n_areas) * n_events * members;
}

int onset_launch(const double* member_out, int n_slots, int mo_slots, int ldm, int npoints, int members,
                 const RsEnsembleStatsSpec* spec, double* onset, int st_slots, int ld, int* ws, cudaStream_t st)
{
  if (n_slots == 0 || npoints == 0 || (!onset && !ws)) return RS_OK;
  CU(static_cast<cudaError_t>(
      rs_launch_ens_onset(member_out, n_slots, mo_slots, ldm, npoints, members, spec, onset, st_slots, ld, ws, st)));
  ++g_launches_total;
  return RS_OK;
}

int onset_area_accumulate(const AreaDevice& d, const int* ws, int npoints, int members, int n_events, int p0,
                          int first_segment, int n_segments, int* acc, cudaStream_t st)
{
  if (n_segments == 0) return RS_OK;
  CU(static_cast<cudaError_t>(rs_launch_ens_area_onset_accumulate(
      ws, npoints, members, n_events, d.stations, p0, d.segments + 4 * static_cast<size_t>(first_segment), n_segments,
      acc, st)));
  ++g_launches_total;
  return RS_OK;
}

int onset_area_finalize(const int* acc, int n_areas, int n_events, int n_slots, int members, double* area_onset,
                        int st_slots, cudaStream_t st)
{
  if (n_slots == 0) return RS_OK;
  CU(static_cast<cudaError_t>(
      rs_launch_ens_area_onset_finalize(acc, n_areas, n_events, n_slots, members, area_onset, st_slots, st)));
  ++g_launches_total;
  return RS_OK;
}

// ---- window extremes (roadsurf_ensemble_extremes) ----
// Which outputs may go together and the extremes themselves, before any device work.  `device`:
// roadsurf_ensemble_extremes, where areas go with area_ext_stats (the host entry's areas may serve other outputs).
int check_extremes(const RsEnsembleExtremes* ext, const double* ext_stats, const RsEnsembleAreas* areas,
                   const double* area_ext_stats, int out_nvar, bool device)
{
  if (!ext && (device || ext_stats || area_ext_stats))
    return fail(RS_ERR_BAD_ARGUMENT, "null extremes pointer: ext_stats and area_ext_stats need ext");
  if (!ext) return RS_OK;
  if (!ext_stats && !area_ext_stats) return fail(RS_ERR_BAD_ARGUMENT, "ext_stats and area_ext_stats are both NULL");
  if (area_ext_stats && !areas) return fail(RS_ERR_BAD_ARGUMENT, "null area pointer: area_ext_stats needs areas");
  if (device && areas && !area_ext_stats) return fail(RS_ERR_BAD_ARGUMENT, "null area pointer: areas need area_ext_stats");
  if (ext->n_extremes < 1 || ext->n_extremes > RS_ENS_MAX_EXTREMES)
    return fail(RS_ERR_BAD_ARGUMENT, "an extremes set has 1 to 8 extremes");
  for (int x = 0; x < ext->n_extremes; ++x)
  {
    const RsEnsembleExtreme& e = ext->extremes[x];
    if (e.kind != RS_ENS_WMIN && e.kind != RS_ENS_WMAX)
      return fail(RS_ERR_BAD_ARGUMENT, "unknown extreme kind (RS_ENS_WMIN or RS_ENS_WMAX)");
    if (e.window < 1) return fail(RS_ERR_BAD_ARGUMENT, "an extreme window is at least 1 output slot");
    if (e.plane < 0 || e.plane >= out_nvar) return fail(RS_ERR_BAD_ARGUMENT, "extreme plane outside the output planes");
  }
  return RS_OK;
}

// The statistics spec of window extremes: the quantiles of `spec`, no thresholds and no events.
RsEnsembleStatsSpec extremes_spec(const RsEnsembleStatsSpec& spec)
{
  RsEnsembleStatsSpec s;
  std::memset(&s, 0, sizeof s);
  s.n_quantiles = spec.n_quantiles;
  std::memcpy(s.quantiles, spec.quantiles, sizeof s.quantiles);
  return s;
}

// The window kernel over the lanes of `npoints` stations into ws [n_extremes][n_slots][ldw], then, with ext_stats,
// the statistics kernel on ws into ext_stats [..][n_extremes][st_slots][ld].
int extremes_launch(const double* member_out, int n_slots, int mo_slots, int ldm, int npoints, int members,
                    const RsEnsembleStatsSpec& xspec, const RsEnsembleExtremes* ext, double* ws, int ldw,
                    double* ext_stats, int st_slots, int ld, cudaStream_t st)
{
  if (n_slots == 0 || npoints == 0) return RS_OK;
  CU(static_cast<cudaError_t>(
      rs_launch_ens_window_extremes(member_out, n_slots, mo_slots, ldm, npoints * members, ext, ws, ldw, st)));
  ++g_launches_total;
  if (!ext_stats) return RS_OK;
  CU(static_cast<cudaError_t>(rs_launch_ens_stats(ws, ext->n_extremes, n_slots, n_slots, ldw, npoints, members, &xspec,
                                                  ext_stats, nullptr, st_slots, ld, st)));
  ++g_launches_total;
  return RS_OK;
}

int extremes_area_accumulate(const AreaDevice& d, const double* ws, int n_slots, int ldw, int members,
                             const RsEnsembleExtremes* ext, int p0, int first_segment, int n_segments, int n_areas,
                             double* acc, cudaStream_t st)
{
  if (n_segments == 0 || n_slots == 0) return RS_OK;
  CU(static_cast<cudaError_t>(rs_launch_ens_area_extremes_accumulate(
      ws, n_slots, ldw, members, ext, d.stations, p0, d.segments + 4 * static_cast<size_t>(first_segment), n_segments,
      n_areas, acc, st)));
  ++g_launches_total;
  return RS_OK;
}

// The finalize kernel, then the statistics kernel on the accumulators into area_ext_stats [..][n_extremes][st_slots]
// [n_areas].
int extremes_area_finalize(double* acc, int n_slots, int n_areas, int members, const RsEnsembleStatsSpec& xspec,
                           const RsEnsembleExtremes* ext, double* area_ext_stats, int st_slots, cudaStream_t st)
{
  if (n_slots == 0) return RS_OK;
  CU(static_cast<cudaError_t>(rs_launch_ens_area_extremes_finalize(acc, n_slots, n_areas, members, ext, st)));
  CU(static_cast<cudaError_t>(rs_launch_ens_stats(acc, ext->n_extremes, n_slots, n_slots, n_areas * members, n_areas,
                                                  members, &xspec, area_ext_stats, nullptr, st_slots, n_areas, st)));
  g_launches_total += 2;
  return RS_OK;
}

// Where the fork may sit (pure host checks).  record_step: host copy (forcing_mode 1) or null.
int check_fork(int forcing_mode, int sim_len, int fork_step, int members, const int* record_step, int n_records, int* r_f)
{
  if (members < 1 || members > RS_ENS_MAX_MEMBERS)
    return fail(RS_ERR_BAD_ARGUMENT, "members must lie in [1, RS_ENS_MAX_MEMBERS = 128]");
  if (forcing_mode == 2)
    return fail(RS_ERR_UNSUPPORTED, "ensembles take forcing_mode 0 or 1 (example2's rule interpolates across the fork)");
  if (forcing_mode != 0 && forcing_mode != 1) return fail(RS_ERR_BAD_ARGUMENT, "forcing_mode must be 0 or 1");
  if (fork_step < 2 || fork_step > sim_len) return fail(RS_ERR_BAD_ARGUMENT, "fork_step must lie in [2, sim_len]");
  *r_f = -1;
  if (forcing_mode == 1)
  {
    bool at_record = false;
    for (int k = 0; k < n_records; ++k)
    {
      if (record_step[k] == fork_step - 1 || record_step[k] == fork_step - 2) at_record = true;
      if (record_step[k] <= fork_step - 1) *r_f = k;
    }
    if (!at_record)
      return fail(RS_ERR_BAD_ARGUMENT, "coarse records: step F - 1 or F - 2 (0-based) must be a record time");
    if (*r_f < 0 || n_records - *r_f < 2)
      return fail(RS_ERR_BAD_ARGUMENT, "coarse records: the members need a record after the fork");
  }
  return RS_OK;
}
}  // namespace

extern "C" {

int roadsurf_ensemble_stats(const double* member_out, int out_nvar, int n_out, int ld_members, int npoints, int members,
                            const RsEnsembleStatsSpec* spec, double* stats, double* prob, int ld, void* stream)
{
  if (!member_out || !spec || members < 1 || members > RS_ENS_MAX_MEMBERS || npoints < 0 || n_out < 0 ||
      (out_nvar != RS_O_NVAR && out_nvar != RS_O_NVAR_EXT) || ld < npoints || ld_members < npoints * members)
    return fail(RS_ERR_BAD_ARGUMENT, "bad arguments");
  {
    const int rc = check_stats_spec(*spec, out_nvar);
    if (rc != RS_OK) return rc;
  }
  return launch_stats_and_events(member_out, out_nvar, n_out, n_out, ld_members, npoints, members, spec, stats, prob, n_out,
                                 ld, stream);
}

int roadsurf_ensemble_area_events(const double* member_out, int out_nvar, int n_out, int ld_members, int npoints,
                                  int members, const RsEnsembleStatsSpec* spec, const RsEnsembleAreas* areas,
                                  double* area_prob, void* stream)
{
  if (!member_out || !spec || !area_prob || members < 1 || members > RS_ENS_MAX_MEMBERS || npoints < 0 || n_out < 0 ||
      (out_nvar != RS_O_NVAR && out_nvar != RS_O_NVAR_EXT) || static_cast<long long>(ld_members) < static_cast<long long>(npoints) * members)
    return fail(RS_ERR_BAD_ARGUMENT, "bad arguments");
  {
    int rc = check_stats_spec(*spec, out_nvar);
    if (rc == RS_OK) rc = check_areas(areas, npoints, *spec);
    if (rc != RS_OK) return rc;
  }
  if (n_out == 0) return RS_OK;
  AreaPlan pl = plan_areas(*areas);
  const int n_segments = plan_segments(pl, 0, npoints, area_segment_length(pl, spec->n_events, n_out, 1));
  const size_t bytes = area_bytes(pl, spec->n_events, n_out, members, n_segments);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  void* buf = nullptr;
  CU(cudaMallocAsync(&buf, bytes, st));
  AreaDevice d;
  size_t h2d = 0;
  int rc = area_upload(pl, spec->n_events, n_out, members, buf, st, &d, &h2d);
  if (rc == RS_OK) rc = area_accumulate(d, member_out, n_out, n_out, ld_members, members, spec, 0, 0, n_segments, st);
  if (rc == RS_OK) rc = area_finalize(d, pl.n_areas, spec->n_events, n_out, members, area_prob, n_out, st);
  const cudaError_t e = cudaFreeAsync(buf, st);
  if (rc == RS_OK && e != cudaSuccess) return fail(RS_ERR_CUDA, std::string("cudaFreeAsync: ") + cudaGetErrorString(e));
  return rc;
}

int roadsurf_ensemble_onset(const double* member_out, int out_nvar, int n_out, int ld_members, int npoints, int members,
                            const RsEnsembleStatsSpec* spec, double* onset, int ld, const RsEnsembleAreas* areas,
                            double* area_onset, void* stream)
{
  if (!member_out || !spec || members < 1 || members > RS_ENS_MAX_MEMBERS || npoints < 0 || n_out < 0 ||
      (out_nvar != RS_O_NVAR && out_nvar != RS_O_NVAR_EXT) || (onset && ld < npoints) ||
      static_cast<long long>(ld_members) < static_cast<long long>(npoints) * members)
    return fail(RS_ERR_BAD_ARGUMENT, "bad arguments");
  {
    int rc = check_stats_spec(*spec, out_nvar);
    if (rc == RS_OK) rc = check_onset_outputs(*spec, onset, areas, nullptr, area_onset, true);
    if (rc == RS_OK && areas) rc = check_areas(areas, npoints, *spec);
    if (rc != RS_OK) return rc;
  }
  if (n_out == 0) return RS_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int E = spec->n_events;
  if (!areas) return onset_launch(member_out, n_out, n_out, ld_members, npoints, members, spec, onset, n_out, ld, nullptr, st);
  // one buffer: the plan (segments, stations; no area event accumulators), the accumulators, the workspace
  AreaPlan pl = plan_areas(*areas);
  const int n_segments = plan_segments(pl, 0, npoints, area_segment_length(pl, E, n_out, 1));
  const size_t plan_bytes = (area_bytes(pl, 0, n_out, members, n_segments) + 15) / 16 * 16;
  const size_t acc_ints = onset_acc_ints(pl.n_areas, E, members);
  const size_t ws_ints = 2 * static_cast<size_t>(E) * npoints * members;
  void* buf = nullptr;
  CU(cudaMallocAsync(&buf, plan_bytes + sizeof(int) * (acc_ints + ws_ints), st));
  int* acc = reinterpret_cast<int*>(static_cast<char*>(buf) + plan_bytes);
  int* ws = acc + acc_ints;
  AreaDevice d;
  size_t h2d = 0;
  int rc = area_upload(pl, 0, n_out, members, buf, st, &d, &h2d);
  if (rc == RS_OK && cudaMemsetAsync(acc, 0x7f, sizeof(int) * acc_ints, st) != cudaSuccess)
    rc = fail(RS_ERR_CUDA, "cudaMemsetAsync of the area onset accumulators");
  if (rc == RS_OK) rc = onset_launch(member_out, n_out, n_out, ld_members, npoints, members, spec, onset, n_out, ld, ws, st);
  if (rc == RS_OK) rc = onset_area_accumulate(d, ws, npoints, members, E, 0, 0, n_segments, acc, st);
  if (rc == RS_OK) rc = onset_area_finalize(acc, pl.n_areas, E, n_out, members, area_onset, n_out, st);
  const cudaError_t e = cudaFreeAsync(buf, st);
  if (rc == RS_OK && e != cudaSuccess) return fail(RS_ERR_CUDA, std::string("cudaFreeAsync: ") + cudaGetErrorString(e));
  return rc;
}

int roadsurf_ensemble_extremes(const double* member_out, int out_nvar, int n_out, int ld_members, int npoints,
                               int members, const RsEnsembleStatsSpec* spec, const RsEnsembleExtremes* ext,
                               double* ext_stats, int ld, const RsEnsembleAreas* areas, double* area_ext_stats,
                               void* stream)
{
  if (!member_out || !spec || members < 1 || members > RS_ENS_MAX_MEMBERS || npoints < 0 || n_out < 0 ||
      (out_nvar != RS_O_NVAR && out_nvar != RS_O_NVAR_EXT) || (ext_stats && ld < npoints) ||
      static_cast<long long>(ld_members) < static_cast<long long>(npoints) * members)
    return fail(RS_ERR_BAD_ARGUMENT, "bad arguments");
  {
    int rc = check_stats_spec(*spec, out_nvar);
    if (rc == RS_OK) rc = check_extremes(ext, ext_stats, areas, area_ext_stats, out_nvar, true);
    if (rc == RS_OK && areas) rc = check_areas(areas, npoints, *spec, false);
    if (rc != RS_OK) return rc;
  }
  if (n_out == 0 || npoints == 0) return RS_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const RsEnsembleStatsSpec xspec = extremes_spec(*spec);
  const int X = ext->n_extremes, ldw = (npoints * members + 31) / 32 * 32;
  // one buffer: the area plan (segments, stations; no area event accumulators), the area accumulators, the work space
  AreaPlan pl;
  int n_segments = 0;
  size_t plan_bytes = 0, acc_n = 0;
  if (areas)
  {
    pl = plan_areas(*areas);
    n_segments = plan_segments(pl, 0, npoints, segment_length(pl, X, 1));
    plan_bytes = (area_bytes(pl, 0, n_out, members, n_segments) + 15) / 16 * 16;
    acc_n = static_cast<size_t>(X) * n_out * pl.n_areas * members;
  }
  const size_t ws_n = static_cast<size_t>(X) * n_out * ldw;
  void* buf = nullptr;
  CU(cudaMallocAsync(&buf, plan_bytes + sizeof(double) * (acc_n + ws_n), st));
  double* acc = reinterpret_cast<double*>(static_cast<char*>(buf) + plan_bytes);
  double* ws = acc + acc_n;
  AreaDevice d;
  int rc = RS_OK;
  if (areas)
  {
    size_t h2d = 0;
    rc = area_upload(pl, 0, n_out, members, buf, st, &d, &h2d);
    if (rc == RS_OK && rs_init_ens_area_extremes(acc, n_out, pl.n_areas, members, ext, st) != 0)
      rc = fail(RS_ERR_CUDA, "cudaMemsetAsync of the area extreme accumulators");
  }
  if (rc == RS_OK)
    rc = extremes_launch(member_out, n_out, n_out, ld_members, npoints, members, xspec, ext, ws, ldw, ext_stats, n_out, ld,
                         st);
  if (rc == RS_OK && areas)
    rc = extremes_area_accumulate(d, ws, n_out, ldw, members, ext, 0, 0, n_segments, pl.n_areas, acc, st);
  if (rc == RS_OK && areas)
    rc = extremes_area_finalize(acc, n_out, pl.n_areas, members, xspec, ext, area_ext_stats, n_out, st);
  const cudaError_t e = cudaFreeAsync(buf, st);
  if (rc == RS_OK && e != cudaSuccess) return fail(RS_ERR_CUDA, std::string("cudaFreeAsync: ") + cudaGetErrorString(e));
  return rc;
}

}  // extern "C"

namespace
{
// roadsurf_run_ensemble_device; `host_record_step` (may be null) is a host copy of shared.record_step, which
// spares the read-back that checks F against the record grid.
int run_ensemble(const RsEnsembleBatch* e, void* stream, const int* host_record_step)
{
  if (!e) return fail(RS_ERR_BAD_ARGUMENT, "null batch");
  const RsDeviceBatch& s = e->shared;
  const int P = s.npoints, M = e->members, F = e->fork_step;
  int r_f = -1;
  {
    // record_step is device memory: checked below, once the pure checks have passed
    const int rc = check_fork(s.forcing_mode == 1 ? 0 : s.forcing_mode, s.sim_len, F, M, nullptr, 0, &r_f);
    if (rc != RS_OK) return rc;
  }
  if (s.step_begin != 0 || s.step_end != 0 || s.forcing_step0 != 0 || s.out_slot0 != 0 || s.expand_workspace)
    return fail(RS_ERR_BAD_ARGUMENT, "shared: step_begin, step_end, forcing_step0, out_slot0 and expand_* must be 0");
  if (P < 0 || s.ld < 32 || s.ld % 32 != 0 || P > s.ld || e->ld_members < 32 || e->ld_members % 32 != 0 ||
      static_cast<long long>(P) * M > e->ld_members)
    return fail(RS_ERR_BAD_ARGUMENT, "ld and ld_members must be multiples of 32, >= npoints and >= npoints * members");
  if (!s.state || !e->member_forcing || !e->member_local || !e->member_state || !e->member_status || !e->member_out ||
      (s.horizons && !e->member_horizons))
    return fail(RS_ERR_BAD_ARGUMENT, "null device pointer in the ensemble batch (shared.state is required)");
  const int out_nvar = s.out_nvar == RS_O_NVAR_EXT ? RS_O_NVAR_EXT : RS_O_NVAR;
  {
    const int rc = check_stats_spec(e->spec, out_nvar);
    if (rc != RS_OK) return rc;
  }
  if (s.out_stride < 1 || s.out_start < 0 || s.out_start >= s.sim_len)
    return fail(RS_ERR_BAD_ARGUMENT, "bad out_stride / out_start");
  int m0, m1;
  slot_range(F, s.sim_len, s.out_start, s.out_stride, &m0, &m1);
  if (e->n_out_members < m1 - m0 || e->n_out_members < 1)
    return fail(RS_ERR_BAD_ARGUMENT, "n_out_members is smaller than the output slots of the steps [F, sim_len]");
  int dev = 0;
  CU(cudaGetDevice(&dev));
  RsModel m;
  {
    const int rc = current_model(dev, &m);
    if (rc != RS_OK) return rc;
  }
  const int nl = m.nlayers;
  if (m.use_coupling && (!s.scratch || !e->member_scratch))
    return fail(RS_ERR_BAD_ARGUMENT, "coupling needs shared.scratch and member_scratch");
  if (static_cast<long long>(RS_STATE_NPLANES(nl)) * e->ld_members < static_cast<long long>(RS_L_NLOCAL) * s.ld)
    return fail(RS_ERR_BAD_ARGUMENT, "member_state is too small to hold the prefix's copy of shared.local");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (s.forcing_mode == 1)
  {
    if (s.n_records < 2 || !s.record_step) return fail(RS_ERR_BAD_ARGUMENT, "coarse forcing needs >= 2 records");
    std::vector<int> rs;
    if (!host_record_step)
    {
      rs.resize(s.n_records);
      CU(cudaMemcpyAsync(rs.data(), s.record_step, sizeof(int) * s.n_records, cudaMemcpyDeviceToHost, st));
      CU(cudaStreamSynchronize(st));
      host_record_step = rs.data();
    }
    int rc = check_record_grid(host_record_step, s.n_records);
    if (rc == RS_OK) rc = check_fork(1, s.sim_len, F, M, host_record_step, s.n_records, &r_f);
    if (rc != RS_OK) return rc;
  }
  const bool relax = m.use_relaxation != 0;

  // (1) the shared part [1, F - 1] on a copy of the statics (member_state is free until the fork)
  double* prefix_local = e->member_state;
  CU(static_cast<cudaError_t>(rs_launch_ens_prefix_local(s.local, s.ld, P, e->member_relax, e->ld_members, M, relax ? 1 : 0,
                                                         prefix_local, stream)));
  ++g_launches_total;
  RsDeviceBatch pre = s;
  pre.local = prefix_local;
  pre.step_begin = 1;
  pre.step_end = F - 1;
  {
    const int rc = roadsurf_run_device(&pre, stream);
    if (rc != RS_OK) return rc;
  }
  // (2) the fork
  RsForkArgs f;
  std::memset(&f, 0, sizeof f);
  f.npoints = P;
  f.ld = s.ld;
  f.members = M;
  f.ldm = e->ld_members;
  f.nlayers = nl;
  f.nvar = s.nvar;
  f.fork_step = F;
  f.relax = relax ? 1 : 0;
  f.state_planes = RS_STATE_NPLANES(nl);
  f.scratch_planes = RS_SCRATCH_NPLANES(nl);
  f.r_f = s.forcing_mode == 1 ? r_f : -1;
  f.local = s.local;
  f.horizons = s.horizons;
  f.state = s.state;
  f.scratch = m.use_coupling ? s.scratch : nullptr;
  f.status = s.status;
  f.forcing = s.forcing;
  f.member_relax = e->member_relax;
  f.m_local = e->member_local;
  f.m_horizons = s.horizons ? e->member_horizons : nullptr;
  f.m_state = e->member_state;
  f.m_scratch = m.use_coupling ? e->member_scratch : nullptr;
  f.m_forcing = e->member_forcing;
  f.m_status = e->member_status;
  CU(static_cast<cudaError_t>(rs_launch_ens_fork(&f, stream)));
  ++g_launches_total;
  // (3) the members [F, sim_len]: a resumed launch
  RsDeviceBatch mb = s;
  mb.npoints = P * M;
  mb.ld = e->ld_members;
  mb.forcing = e->member_forcing;
  if (s.forcing_mode == 1)
  {
    mb.record_step = s.record_step + r_f;
    mb.n_records = s.n_records - r_f;
  }
  else
  {
    mb.n_records = s.sim_len - F + 1;
    mb.forcing_step0 = F;
  }
  mb.local = e->member_local;
  mb.horizons = s.horizons ? e->member_horizons : nullptr;
  mb.out = e->member_out;
  mb.n_out = e->n_out_members;
  mb.out_slot0 = m0;
  mb.status = e->member_status;
  mb.state = e->member_state;
  mb.scratch = m.use_coupling ? e->member_scratch : nullptr;
  mb.step_begin = F;
  mb.step_end = s.sim_len;
  mb.order = e->member_order;
  mb.coupling_window_end = 0;  // the window lies in the shared part
  {
    const int rc = roadsurf_run_device(&mb, stream);
    if (rc != RS_OK) return rc;
  }
  // (4) the statistics and events over the member slots [m0, m1) of member_out [out_nvar][n_out_members][ld_members];
  // slots beyond are not read
  return launch_stats_and_events(e->member_out, out_nvar, m1 - m0, e->n_out_members, e->ld_members, P, M, &e->spec,
                                 e->stats, e->prob, e->n_out_members, s.ld, stream);
}
}  // namespace

extern "C" {

int roadsurf_run_ensemble_device(const RsEnsembleBatch* e, void* stream) { return run_ensemble(e, stream, nullptr); }

int roadsurf_run_ensemble_host_soa(const RsHostBatch* b, const double* member_records, int members, int fork_step,
                                   const int* latest_obs_index, const RsEnsembleStatsSpec* spec, double* stats, double* prob, double* member_out,
                                   int* member_status, const InputSettings* settings, const InputParameters* params)
{
  return roadsurf_run_ensemble_host_soa_areas(b, member_records, members, fork_step, latest_obs_index, spec, stats, prob,
                                              member_out, member_status, nullptr, nullptr, settings, params);
}

int roadsurf_run_ensemble_host_soa_areas(const RsHostBatch* b, const double* member_records, int members, int fork_step,
                                         const int* latest_obs_index, const RsEnsembleStatsSpec* spec, double* stats,
                                         double* prob, double* member_out, int* member_status, const RsEnsembleAreas* areas,
                                         double* area_prob, const InputSettings* settings, const InputParameters* params)
{
  return roadsurf_run_ensemble_host_soa_onset(b, member_records, members, fork_step, latest_obs_index, spec, stats, prob,
                                              member_out, member_status, areas, area_prob, nullptr, nullptr, settings,
                                              params);
}

int roadsurf_run_ensemble_host_soa_onset(const RsHostBatch* b, const double* member_records, int members, int fork_step,
                                         const int* latest_obs_index, const RsEnsembleStatsSpec* spec, double* stats,
                                         double* prob, double* member_out, int* member_status, const RsEnsembleAreas* areas,
                                         double* area_prob, double* onset, double* area_onset,
                                         const InputSettings* settings, const InputParameters* params)
{
  return roadsurf_run_ensemble_host_soa_extremes(b, member_records, members, fork_step, latest_obs_index, spec, stats,
                                                 prob, member_out, member_status, areas, area_prob, onset, area_onset,
                                                 nullptr, nullptr, nullptr, settings, params);
}

int roadsurf_run_ensemble_host_soa_extremes(const RsHostBatch* b, const double* member_records, int members,
                                            int fork_step, const int* latest_obs_index, const RsEnsembleStatsSpec* spec,
                                            double* stats, double* prob, double* member_out, int* member_status,
                                            const RsEnsembleAreas* areas, double* area_prob, double* onset,
                                            double* area_onset, const RsEnsembleExtremes* ext, double* ext_stats,
                                            double* area_ext_stats, const InputSettings* settings,
                                            const InputParameters* params)
{
  g_err.clear();
  std::memset(&g_stats, 0, sizeof g_stats);
  const double wall0 = now_ms();
  if (!b || !settings || !params || !spec) return fail(RS_ERR_BAD_ARGUMENT, "null argument");
  if (b->forcing_mode == 2)
    return fail(RS_ERR_UNSUPPORTED, "ensembles take forcing_mode 0 or 1 (example2's rule interpolates across the fork)");
  if (b->forcing_mode != 1)
    return fail(RS_ERR_UNSUPPORTED, "roadsurf_run_ensemble_host_soa takes coarse records (forcing_mode 1) only");
  if (b->npoints < 0 || b->sim_len < 1 || b->out_stride < 1 || b->sim_len != settings->SimLen)
    return fail(RS_ERR_BAD_ARGUMENT, "bad sizes (sim_len must equal settings->SimLen)");
  if (b->nvar != RS_F_NVAR && b->nvar != RS_F_NVAR_DEPTH) return fail(RS_ERR_BAD_ARGUMENT, "nvar must be 11 or 12");
  if (b->n_records < 2 || !b->record_step || !b->forcing || !b->time_fields || !b->local)
    return fail(RS_ERR_BAD_ARGUMENT, "null host pointer in the shared batch");
  const int P = b->npoints, M = members, F = fork_step, nvar = b->nvar, nrec = b->n_records;
  int r_f = -1;
  {
    int rc = check_record_grid(b->record_step, nrec);
    if (rc == RS_OK) rc = check_fork(1, b->sim_len, F, M, b->record_step, nrec, &r_f);
    if (rc != RS_OK) return rc;
  }
  {
    const int rc = check_stats_spec(*spec, RS_O_NVAR);
    if (rc != RS_OK) return rc;
  }
  {
    int rc = check_onset_outputs(*spec, onset, areas, area_prob, area_onset, false, area_ext_stats);
    if (rc == RS_OK) rc = check_extremes(ext, ext_stats, areas, area_ext_stats, RS_O_NVAR, false);
    if (rc == RS_OK && areas) rc = check_areas(areas, P, *spec, area_prob || area_onset);
    if (rc != RS_OK) return rc;
  }
  if (P > 0 && !member_records) return fail(RS_ERR_BAD_ARGUMENT, "null member_records");
  const size_t np = static_cast<size_t>(P), npm = np * M;
  // one coupling window, and before the fork
  if (settings->use_coupling == 1)
  {
    const int w = common_window_end(b->local, np);
    if (w < 0) return fail(RS_ERR_UNSUPPORTED, "ensembles need one coupling window for all coupled stations");
    if (w > 0 && F < w + 2)
      return fail(RS_ERR_BAD_ARGUMENT, "the coupling window [start, end + 1] must lie before the fork (F >= couplingIndexI + 2)");
  }
  if (P == 0) return roadsurf_device_count() < 1 ? fail(RS_ERR_NO_DEVICE, "no CUDA device visible") : RS_OK;
  if (roadsurf_device_count() < 1) return fail(RS_ERR_NO_DEVICE, "no CUDA device visible (this library has no CPU path)");

  int dev = 0;
  CU(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> device_lock(g_device_mu[dev & 63]);

  // member relaxation targets: roadsurf_read_input_derive_records' rule on each member's records (records up to r_f
  // are the station's), written straight into a pooled pinned buffer [3][P * M]
  const int nrec_m = nrec - r_f - 1;  // records r_f + 1 ... supplied per member
  double* relax_h = nullptr;
  const bool relax = settings->use_relaxation == 1;
  const double setup0 = now_ms();
  if (relax)
  {
    CU(pooled_pinned(dev, EH_H_RELAX, 3 * npm, &relax_h));
    const int* rs = b->record_step;
    const double DT = settings->DTSecs;
    parallel_for(P, host_threads(), [&](int pi) {
      const size_t p = pi;
      const int vars[3] = {RS_F_TAIR, RS_F_VZ, RS_F_RHZ};
      const int last = latest_obs_index ? latest_obs_index[pi] : -9999;
      for (int mm = 0; mm < M; ++mm)
      {
        const size_t l = p * M + mm;
        for (int j = 0; j < 3; ++j)
        {
          double val = -9999.9;
          if (last > -1 && last < b->sim_len)
            val = record_value_at(rs, nrec, DT, last, [&](int k) {
              return k <= r_f ? b->forcing[(static_cast<size_t>(k) * nvar + vars[j]) * np + p]
                              : member_records[(static_cast<size_t>(k - r_f - 1) * nvar + vars[j]) * npm + l];
            });
          relax_h[j * npm + l] = val;
        }
      }
    });
  }
  RsModel model;
  {
    const int rc = set_model_on_current_device(settings, params, &model);
    if (rc != RS_OK) return rc;
  }
  const int nl = model.nlayers;
  const bool cpl = model.use_coupling != 0;
  const bool hor = b->horizons != nullptr;
  const int sim_len = b->sim_len;
  int pre0, pre1, m0, m1;
  slot_range(1, F - 1, 0, b->out_stride, &pre0, &pre1);
  slot_range(F, sim_len, 0, b->out_stride, &m0, &m1);
  const int n_pre = std::max(1, pre1 - pre0), n_m = m1 - m0;
  const int nq = spec->n_quantiles, np_planes = spec->n_thresholds + spec->n_events;  // prob: thresholds, then events
  const size_t frows = static_cast<size_t>(nrec) * nvar, frows_m = static_cast<size_t>(nrec_m + 1) * nvar;
  const size_t NS = RS_STATE_NPLANES(nl), SC = RS_SCRATCH_NPLANES(nl);
  const size_t srows = static_cast<size_t>(RS_ENS_NFIXED + nq) * RS_O_NVAR * n_m, prows = static_cast<size_t>(np_planes) * n_m;
  const int E = spec->n_events;
  const size_t orows = onset ? static_cast<size_t>(E) * n_m : 0;  // onset planes of a station
  // window extremes: the work space [X][n_m] of every member lane and the ext_stats rows of a station
  const int X = ext ? ext->n_extremes : 0;
  const size_t xws = static_cast<size_t>(X) * n_m, xrows = ext_stats ? static_cast<size_t>(RS_ENS_NFIXED + nq) * xws : 0;
  // area onset: the workspace {O, X} of every member lane, E * 8 bytes
  const size_t per_station =
      sizeof(double) * (frows + RS_L_NLOCAL + (hor ? 360 : 0) + RS_O_NVAR * n_pre + NS + (cpl ? SC : 0) + 1 + srows + prows +
                        orows + xrows) +
      sizeof(double) * M * (frows_m + RS_L_NLOCAL + (hor ? 360 : 0) + NS + (cpl ? SC : 0) + 1 + 3 + RS_O_NVAR * n_m +
                            (area_onset ? E : 0) + xws);
  size_t free_b = 0, total_b = 0;
  CU(cudaMemGetInfo(&free_b, &total_b));
  // areas: the plan and the accumulators stay on the device for the whole call, beside area_prob and area_onset (the
  // area event accumulators only where area_prob is asked for)
  AreaPlan area_plan;
  const int E_prob = area_prob ? E : 0;
  size_t area_fixed = 0;
  if (areas)
  {
    area_plan = plan_areas(*areas);
    area_fixed = area_bytes(area_plan, E_prob, n_m, M, area_plan.stations.size()) +
                 sizeof(double) * E * n_m * areas->n_areas * ((area_prob ? 1 : 0) + (area_onset ? 1 : 0)) +
                 (area_onset ? sizeof(int) * onset_acc_ints(areas->n_areas, E, M) : 0);
    if (static_cast<double>(area_fixed) >= free_b * 0.8)
      return fail(RS_ERR_CUDA, "not enough device memory for the area accumulators (area_prob: 2 * n_areas * n_events * "
                               "ceil(n_out_m / 64) * members * 8 bytes; area_onset: n_areas * n_events * members * 8 "
                               "bytes) and the area outputs");
  }
  // area window extremes: their own segments, the accumulators [X][n_m][n_areas * M] and area_ext_stats
  const size_t area_xacc_n = area_ext_stats ? xws * areas->n_areas * M : 0;
  const size_t area_xstats_n = area_ext_stats ? static_cast<size_t>(RS_ENS_NFIXED + nq) * xws * areas->n_areas : 0;
  if (area_ext_stats)
  {
    area_fixed += sizeof(int) * 4 * area_plan.stations.size() + sizeof(double) * (area_xacc_n + area_xstats_n);
    if (static_cast<double>(area_fixed) >= free_b * 0.8)
      return fail(RS_ERR_CUDA, "not enough device memory for the area extreme accumulators (n_extremes * n_out_m * "
                               "n_areas * members * 8 bytes) and area_ext_stats");
  }
  long long pc = static_cast<long long>((free_b * 0.8 - static_cast<double>(area_fixed)) / per_station) - 64;
  if (const int cap = g_opt_max_slots.load()) pc = std::min<long long>(pc, std::max(1, cap / M));
  pc = std::min<long long>(pc, P);
  if (pc < 1) return fail(RS_ERR_CUDA, "not enough device memory for one station's members");
  const int ldc = static_cast<int>((pc + 31) / 32 * 32), ldmc = static_cast<int>((pc * M + 31) / 32 * 32);
  // [chunks + 1]: the segments of chunk c are [chunk_segments[c], chunk_segments[c + 1]), those of the area extremes
  // [ext_segments[c], ext_segments[c + 1]), after the area events' in the same plan
  std::vector<int> chunk_segments, ext_segments;
  auto plan_chunks = [&](int len, std::vector<int>& first) {
    first.push_back(static_cast<int>(area_plan.segments.size() / 4));
    for (long long p0 = 0; p0 < P; p0 += pc)
      first.push_back(first.back() + plan_segments(area_plan, p0, std::min<long long>(pc, P - p0), len));
  };
  const long long chunks = (P + pc - 1) / pc;
  if (area_prob || area_onset) plan_chunks(area_segment_length(area_plan, E, n_m, chunks), chunk_segments);
  if (area_ext_stats) plan_chunks(segment_length(area_plan, X, chunks), ext_segments);

  SoaStreams* ss = nullptr;
  {
    const int rc = soa_streams(dev, &ss);
    if (rc != RS_OK) return rc;
  }
  cudaStream_t st = ss->st[0];
  cudaEvent_t* ev = ss->ev[0];
  double *d_forcing, *d_local, *d_hor = nullptr, *d_out, *d_state, *d_scratch = nullptr, *d_mf, *d_ml, *d_mh = nullptr,
         *d_ms, *d_msc = nullptr, *d_mo, *d_relax = nullptr, *d_stats = nullptr, *d_prob = nullptr, *d_solar;
  int *d_status, *d_mstatus, *d_tf, *d_rs;
  unsigned long long* d_counters;
  const size_t lc = ldc, lm = ldmc;
  CU(pooled(dev, EH_FORCING, frows * lc, &d_forcing));
  CU(pooled(dev, EH_LOCAL, RS_L_NLOCAL * lc, &d_local));
  if (hor) CU(pooled(dev, EH_HOR, 360 * lc, &d_hor));
  CU(pooled(dev, EH_OUT, RS_O_NVAR * n_pre * lc, &d_out));
  CU(pooled(dev, EH_STATE, NS * lc, &d_state));
  if (cpl) CU(pooled(dev, EH_SCRATCH, SC * lc, &d_scratch));
  CU(pooled(dev, EH_M_FORCING, frows_m * lm, &d_mf));
  CU(pooled(dev, EH_M_LOCAL, RS_L_NLOCAL * lm, &d_ml));
  if (hor) CU(pooled(dev, EH_M_HOR, 360 * lm, &d_mh));
  CU(pooled(dev, EH_M_STATE, NS * lm, &d_ms));
  if (cpl) CU(pooled(dev, EH_M_SCRATCH, SC * lm, &d_msc));
  CU(pooled(dev, EH_M_OUT, RS_O_NVAR * n_m * lm, &d_mo));
  if (relax) CU(pooled(dev, EH_RELAX, 3 * lm, &d_relax));
  CU(pooled(dev, EH_STATS, srows * lc, &d_stats));
  if (np_planes) CU(pooled(dev, EH_PROB, prows * lc, &d_prob));
  CU(pooled(dev, EH_SOLAR, 4 * static_cast<size_t>(sim_len), &d_solar));
  CU(pooled(dev, EH_STATUS, lc, &d_status));
  CU(pooled(dev, EH_M_STATUS, lm, &d_mstatus));
  CU(pooled(dev, EH_TIME_FIELDS, 6 * static_cast<size_t>(sim_len), &d_tf));
  CU(pooled(dev, EH_RECORD_STEP, nrec, &d_rs));
  CU(pooled(dev, EH_COUNTERS, RS_CNT_N, &d_counters));
  const size_t D = sizeof(double);
  CU(cudaMemcpyAsync(d_tf, b->time_fields, sizeof(int) * 6 * sim_len, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d_rs, b->record_step, sizeof(int) * nrec, cudaMemcpyHostToDevice, st));
  CU(cudaMemsetAsync(d_counters, 0, sizeof(unsigned long long) * RS_CNT_N, st));
  g_stats.h2d_bytes += sizeof(int) * (6 * sim_len + nrec);
  AreaDevice d_areas;
  double* d_area_prob = nullptr;
  const size_t area_prob_n = areas ? static_cast<size_t>(E) * n_m * areas->n_areas : 0;
  if (areas)
  {
    unsigned long long* buf;
    CU(pooled(dev, EH_AREAS, (area_bytes(area_plan, E_prob, n_m, M, area_plan.segments.size() / 4) + 7) / 8, &buf));
    if (area_prob) CU(pooled(dev, EH_AREA_PROB, std::max<size_t>(1, area_prob_n), &d_area_prob));
    size_t h2d = 0;
    const int rc = area_upload(area_plan, E_prob, n_m, M, buf, st, &d_areas, &h2d);
    if (rc != RS_OK) return rc;
    g_stats.h2d_bytes += h2d;
  }
  double *d_onset = nullptr, *d_area_onset = nullptr;
  int *d_ws = nullptr, *d_onset_acc = nullptr;
  if (onset) CU(pooled(dev, EH_ONSET, std::max<size_t>(1, orows * lc), &d_onset));
  if (area_onset)
  {
    const size_t acc_ints = onset_acc_ints(areas->n_areas, E, M);
    CU(pooled(dev, EH_ONSET_WS, 2 * static_cast<size_t>(E) * lm, &d_ws));
    CU(pooled(dev, EH_ONSET_ACC, acc_ints, &d_onset_acc));
    CU(pooled(dev, EH_AREA_ONSET, std::max<size_t>(1, area_prob_n), &d_area_onset));
    CU(cudaMemsetAsync(d_onset_acc, 0x7f, sizeof(int) * acc_ints, st));
  }
  double *d_xws = nullptr, *d_xstats = nullptr, *d_xacc = nullptr, *d_area_xstats = nullptr;
  const RsEnsembleStatsSpec xspec = extremes_spec(*spec);
  if (ext) CU(pooled(dev, EH_EXT_WS, std::max<size_t>(1, xws * lm), &d_xws));
  if (ext_stats) CU(pooled(dev, EH_EXT_STATS, std::max<size_t>(1, xrows * lc), &d_xstats));
  if (area_ext_stats)
  {
    CU(pooled(dev, EH_EXT_ACC, std::max<size_t>(1, area_xacc_n), &d_xacc));
    CU(pooled(dev, EH_AREA_EXT_STATS, std::max<size_t>(1, area_xstats_n), &d_area_xstats));
    CU(static_cast<cudaError_t>(rs_init_ens_area_extremes(d_xacc, n_m, areas->n_areas, M, ext, st)));
  }
  g_stats.setup_ms = now_ms() - setup0;
  const int launches0 = g_launches_total.load();

  for (long long p0 = 0; p0 < P; p0 += pc)
  {
    const int n = static_cast<int>(std::min<long long>(pc, P - p0));
    const size_t nm = static_cast<size_t>(n) * M, col = static_cast<size_t>(p0), colm = col * M;
    const int ld = (n + 31) / 32 * 32, ldm = static_cast<int>((nm + 31) / 32 * 32);
    CU(cudaEventRecord(ev[0], st));
    CU(cudaMemcpy2DAsync(d_forcing, D * ld, b->forcing + col, D * np, D * n, frows, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpy2DAsync(d_local, D * ld, b->local + col, D * np, D * n, RS_L_NLOCAL, cudaMemcpyHostToDevice, st));
    if (hor) CU(cudaMemcpy2DAsync(d_hor, D * ld, b->horizons + col, D * np, D * n, 360, cudaMemcpyHostToDevice, st));
    if (nrec_m > 0)
      CU(cudaMemcpy2DAsync(d_mf + static_cast<size_t>(nvar) * ldm, D * ldm, member_records + colm, D * npm, D * nm,
                           static_cast<size_t>(nrec_m) * nvar, cudaMemcpyHostToDevice, st));
    if (relax) CU(cudaMemcpy2DAsync(d_relax, D * ldm, relax_h + colm, D * npm, D * nm, 3, cudaMemcpyHostToDevice, st));
    g_stats.h2d_bytes += D * (n * (frows + RS_L_NLOCAL + (hor ? 360 : 0)) + nm * (static_cast<size_t>(nrec_m) * nvar + (relax ? 3 : 0)));
    CU(cudaEventRecord(ev[1], st));
    RsEnsembleBatch e;
    std::memset(&e, 0, sizeof e);
    RsDeviceBatch& s = e.shared;
    s.npoints = n;
    s.ld = ld;
    s.sim_len = sim_len;
    s.forcing_mode = 1;
    s.n_records = nrec;
    s.nvar = nvar;
    s.forcing = d_forcing;
    s.record_step = d_rs;
    s.time_fields = d_tf;
    s.local = d_local;
    s.horizons = hor ? d_hor : nullptr;
    s.out = d_out;
    s.out_stride = b->out_stride;
    s.n_out = n_pre;
    s.status = d_status;
    s.state = d_state;
    s.scratch = d_scratch;
    s.counters = d_counters;
    s.solar = d_solar;
    s.out_nvar = RS_O_NVAR;
    s.coupling_window_end = (cpl && opt_compaction_passes() > 0) ? b->coupling_window_end : 0;
    e.members = M;
    e.fork_step = F;
    e.ld_members = ldm;
    e.member_forcing = d_mf;
    e.member_relax = relax ? d_relax : nullptr;
    e.member_local = d_ml;
    e.member_horizons = d_mh;
    e.member_state = d_ms;
    e.member_scratch = d_msc;
    e.member_status = d_mstatus;
    e.member_out = d_mo;
    e.n_out_members = std::max(1, n_m);
    e.spec = *spec;
    e.stats = stats ? d_stats : nullptr;
    e.prob = (prob && np_planes) ? d_prob : nullptr;
    {
      const int rc = run_ensemble(&e, st, b->record_step);
      if (rc != RS_OK) return rc;
    }
    const long long chunk = p0 / pc;
    const bool last = p0 + pc >= P;
    if (area_prob)
    {
      int rc = area_accumulate(d_areas, d_mo, n_m, e.n_out_members, ldm, M, spec, static_cast<int>(p0),
                               chunk_segments[chunk], chunk_segments[chunk + 1] - chunk_segments[chunk], st);
      if (rc == RS_OK && last) rc = area_finalize(d_areas, areas->n_areas, E, n_m, M, d_area_prob, n_m, st);
      if (rc != RS_OK) return rc;
    }
    {
      int rc = onset_launch(d_mo, n_m, e.n_out_members, ldm, n, M, spec, d_onset, n_m, ld, d_ws, st);
      if (rc == RS_OK && area_onset)
        rc = onset_area_accumulate(d_areas, d_ws, n, M, E, static_cast<int>(p0), chunk_segments[chunk],
                                   chunk_segments[chunk + 1] - chunk_segments[chunk], d_onset_acc, st);
      if (rc == RS_OK && area_onset && last)
        rc = onset_area_finalize(d_onset_acc, areas->n_areas, E, n_m, M, d_area_onset, n_m, st);
      if (rc != RS_OK) return rc;
    }
    if (ext)
    {
      int rc = extremes_launch(d_mo, n_m, e.n_out_members, ldm, n, M, xspec, ext, d_xws, ldm, d_xstats, n_m, ld, st);
      if (rc == RS_OK && area_ext_stats)
        rc = extremes_area_accumulate(d_areas, d_xws, n_m, ldm, M, ext, static_cast<int>(p0), ext_segments[chunk],
                                      ext_segments[chunk + 1] - ext_segments[chunk], areas->n_areas, d_xacc, st);
      if (rc == RS_OK && area_ext_stats && last)
        rc = extremes_area_finalize(d_xacc, n_m, areas->n_areas, M, xspec, ext, d_area_xstats, n_m, st);
      if (rc != RS_OK) return rc;
    }
    CU(cudaEventRecord(ev[2], st));
    if (b->out && pre1 > pre0)
      CU(cudaMemcpy2DAsync(b->out + col, D * np, d_out, D * ld, D * n, static_cast<size_t>(RS_O_NVAR) * (pre1 - pre0),
                           cudaMemcpyDeviceToHost, st));
    if (stats && n_m > 0)
      CU(cudaMemcpy2DAsync(stats + col, D * np, d_stats, D * ld, D * n, srows, cudaMemcpyDeviceToHost, st));
    if (prob && np_planes && n_m > 0) CU(cudaMemcpy2DAsync(prob + col, D * np, d_prob, D * ld, D * n, prows, cudaMemcpyDeviceToHost, st));
    if (member_out && n_m > 0)
      CU(cudaMemcpy2DAsync(member_out + colm, D * npm, d_mo, D * ldm, D * nm, static_cast<size_t>(RS_O_NVAR) * n_m,
                           cudaMemcpyDeviceToHost, st));
    if (member_status)
      CU(cudaMemcpyAsync(member_status + colm, d_mstatus, sizeof(int) * nm, cudaMemcpyDeviceToHost, st));
    g_stats.d2h_bytes += D * (n * ((b->out ? RS_O_NVAR * (pre1 - pre0) : 0) + (stats ? srows : 0) + (prob ? prows : 0)) +
                              (member_out ? nm * RS_O_NVAR * n_m : 0)) + (member_status ? sizeof(int) * nm : 0);
    if (onset && n_m > 0)
    {
      CU(cudaMemcpy2DAsync(onset + col, D * np, d_onset, D * ld, D * n, orows, cudaMemcpyDeviceToHost, st));
      g_stats.d2h_bytes += D * n * orows;
    }
    if (area_prob && last && area_prob_n > 0)
    {
      CU(cudaMemcpyAsync(area_prob, d_area_prob, D * area_prob_n, cudaMemcpyDeviceToHost, st));
      g_stats.d2h_bytes += D * area_prob_n;
    }
    if (area_onset && last && area_prob_n > 0)
    {
      CU(cudaMemcpyAsync(area_onset, d_area_onset, D * area_prob_n, cudaMemcpyDeviceToHost, st));
      g_stats.d2h_bytes += D * area_prob_n;
    }
    if (ext_stats && n_m > 0)
    {
      CU(cudaMemcpy2DAsync(ext_stats + col, D * np, d_xstats, D * ld, D * n, xrows, cudaMemcpyDeviceToHost, st));
      g_stats.d2h_bytes += D * n * xrows;
    }
    if (area_ext_stats && last && area_xstats_n > 0)
    {
      CU(cudaMemcpyAsync(area_ext_stats, d_area_xstats, D * area_xstats_n, cudaMemcpyDeviceToHost, st));
      g_stats.d2h_bytes += D * area_xstats_n;
    }
    CU(cudaEventRecord(ev[3], st));
    CU(cudaStreamSynchronize(st));
    add_stage_times(g_stats, ev);
    ++g_stats.groups;
  }
  unsigned long long cnt[RS_CNT_N];
  CU(cudaMemcpy(cnt, d_counters, sizeof cnt, cudaMemcpyDeviceToHost));
  g_stats.executed_steps = static_cast<int64_t>(cnt[RS_CNT_EXECUTED_STEPS]);
  g_stats.kernel_launches = g_launches_total.load() - launches0;
  g_stats.wall_ms = now_ms() - wall0;
  return RS_OK;
}

}  // extern "C" (ensemble entry points)
