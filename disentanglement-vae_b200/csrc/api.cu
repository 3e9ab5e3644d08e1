// Error / bookkeeping entry points of the C ABI (see include/dvae_b200.h).
#include <stdarg.h>
#include <stdlib.h>

#include <atomic>

#include <mutex>
#include <vector>

#include "common.cuh"
#include "tc_gemm16.cuh"

namespace dvae {
static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
bool force_simt_gemm() {
  const char* e = getenv("DVAE_GEMM_IMPL");
  return e && e[0] == 's';
}

// ---- fork / join side streams ---------------------------------------------------------------------
int join_side_streams(cudaStream_t main);
void set_defer_joins(bool on);
namespace {
struct SideStreams {
  cudaStream_t s[3];
  cudaStream_t sig = nullptr;                   // carries the gradient-exchange kernels forked by dvae_fork_after
  cudaEvent_t fork_ev, join_ev[3], mark_ev, chain_ev, sig_ev[5], sig_join;
  bool ok = false;
  bool pending[3] = {false, false, false};     // detached work (deferred joins)
  bool sig_pending = false;
};
thread_local bool g_defer_joins = false;
SideStreams* side_streams() {
  static thread_local SideStreams* per_dev[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  if (!per_dev[dev]) {
    SideStreams* ss = new SideStreams();
    ss->ok = cudaEventCreateWithFlags(&ss->fork_ev, cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&ss->mark_ev, cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&ss->chain_ev, cudaEventDisableTiming) == cudaSuccess;
    // side streams 0 / 1 carry the weight-gradient GEMMs that run beside the next layer's recurrence: lowest priority, so
    // that CTAs of the caller's (critical-path) stream are placed first whenever SMs free up (DVAE_SIDE_PRIO=0: default priority)
    int least = 0, greatest = 0;
    const char* pe = getenv("DVAE_SIDE_PRIO");
    const bool low = !(pe && pe[0] == '0') && cudaDeviceGetStreamPriorityRange(&least, &greatest) == cudaSuccess;
    for (int i = 0; i < 3 && ss->ok; ++i)
      ss->ok = cudaStreamCreateWithPriority(&ss->s[i], cudaStreamNonBlocking, (low && i < 2) ? least : 0) == cudaSuccess &&
               cudaEventCreateWithFlags(&ss->join_ev[i], cudaEventDisableTiming) == cudaSuccess;
    ss->ok = ss->ok && cudaStreamCreateWithFlags(&ss->sig, cudaStreamNonBlocking) == cudaSuccess &&
             cudaEventCreateWithFlags(&ss->sig_join, cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; i < 5 && ss->ok; ++i) ss->ok = cudaEventCreateWithFlags(&ss->sig_ev[i], cudaEventDisableTiming) == cudaSuccess;
    per_dev[dev] = ss;
  }
  return per_dev[dev]->ok ? per_dev[dev] : nullptr;
}
bool fork_enabled() {
  const char* e = getenv("DVAE_FORK");
  return !(e && e[0] == '0');
}
}  // namespace

Fork::Fork(cudaStream_t main) : main_(main), ok_(false) {
  if (!fork_enabled()) return;
  SideStreams* ss = side_streams();
  if (!ss) return;
  ok_ = cudaEventRecord(ss->fork_ev, main_) == cudaSuccess;
}
cudaStream_t Fork::side(int i) {
  if (!ok_) return main_;
  SideStreams* ss = side_streams();
  if (!used_[i]) {
    if (cudaStreamWaitEvent(ss->s[i], ss->fork_ev, 0) != cudaSuccess) return main_;
    used_[i] = true;
  }
  return ss->s[i];
}
int Fork::join() {
  if (!ok_) return DVAE_OK;
  SideStreams* ss = side_streams();
  for (int i = 0; i < 3; ++i)
    if (used_[i]) {
      DVAE_CUDA(cudaEventRecord(ss->join_ev[i], ss->s[i]));
      DVAE_CUDA(cudaStreamWaitEvent(main_, ss->join_ev[i], 0));
      used_[i] = false;
      ss->pending[i] = false;      // stream order: everything detached earlier on this side stream is covered too
    }
  return DVAE_OK;
}
int Fork::mark(int i) {
  if (!ok_ || !used_[i]) return DVAE_OK;
  DVAE_CUDA(cudaEventRecord(side_streams()->mark_ev, side_streams()->s[i]));
  marked_ = true;
  return DVAE_OK;
}
int Fork::wait_mark() {
  if (!ok_ || !marked_) return DVAE_OK;
  DVAE_CUDA(cudaStreamWaitEvent(main_, side_streams()->mark_ev, 0));
  marked_ = false;
  return DVAE_OK;
}
int Fork::chain(int from, int to) {
  if (!ok_ || !used_[from]) return DVAE_OK;
  cudaStream_t dst = side(to);
  if (dst == main_) return DVAE_OK;
  DVAE_CUDA(cudaEventRecord(side_streams()->chain_ev, side_streams()->s[from]));
  DVAE_CUDA(cudaStreamWaitEvent(dst, side_streams()->chain_ev, 0));
  return DVAE_OK;
}
int Fork::join_or_defer() {
  if (!ok_ || !g_defer_joins) return join();
  SideStreams* ss = side_streams();
  for (int i = 0; i < 3; ++i)
    if (used_[i]) {
      ss->pending[i] = true;
      used_[i] = false;
    }
  return DVAE_OK;
}
int join_side_streams(cudaStream_t main) {
  SideStreams* ss = side_streams();
  if (!ss) return DVAE_OK;
  for (int i = 0; i < 3; ++i)
    if (ss->pending[i]) {
      DVAE_CUDA(cudaEventRecord(ss->join_ev[i], ss->s[i]));
      DVAE_CUDA(cudaStreamWaitEvent(main, ss->join_ev[i], 0));
      ss->pending[i] = false;
    }
  if (ss->sig_pending) {
    DVAE_CUDA(cudaEventRecord(ss->sig_join, ss->sig));
    DVAE_CUDA(cudaStreamWaitEvent(main, ss->sig_join, 0));
    ss->sig_pending = false;
  }
  return DVAE_OK;
}

// ---- scheduling of the gradient exchange inside a captured data-parallel step ---------------------------------------
// The step counter lives in device memory and is advanced by the graph's first node, so the exchange kernels derive a
// fresh barrier epoch on every replay without anything being reset.
namespace {
__global__ void counter_increment_kernel(uint32_t* counter) { *counter += 1; }
}  // namespace

// The library's signal stream, made to wait for everything enqueued so far on `main` (and the detached side-stream work
// and `extra`); work put on it afterwards runs beside `main` and is joined by join_side_streams().
int fork_after(bool include_sides, cudaStream_t extra, cudaStream_t main, cudaStream_t* out) {
  SideStreams* ss = side_streams();
  if (!ss) { *out = main; return DVAE_OK; }
  DVAE_CUDA(cudaEventRecord(ss->sig_ev[3], main));
  DVAE_CUDA(cudaStreamWaitEvent(ss->sig, ss->sig_ev[3], 0));
  if (include_sides)
    for (int i = 0; i < 3; ++i)
      if (ss->pending[i]) {
        DVAE_CUDA(cudaEventRecord(ss->sig_ev[i], ss->s[i]));
        DVAE_CUDA(cudaStreamWaitEvent(ss->sig, ss->sig_ev[i], 0));
      }
  if (extra) {
    DVAE_CUDA(cudaEventRecord(ss->sig_ev[4], extra));
    DVAE_CUDA(cudaStreamWaitEvent(ss->sig, ss->sig_ev[4], 0));
  }
  ss->sig_pending = true;
  *out = ss->sig;
  return DVAE_OK;
}

void set_defer_joins(bool on) { g_defer_joins = on; }
bool defer_joins_enabled() { return g_defer_joins; }
}  // namespace dvae

// ---- weight-plane registry -------------------------------------------------------------------------
// A caller that knows when its weights change (the training engine: once per optimizer step) registers them with
// pre-allocated plane buffers, refreshes all planes with ONE launch, and enables the registry around its own launches.
// While enabled, every tensor-core GEMM whose B operand lies inside a registered weight fetches it as pre-split fp16
// (hi, lo) tiles by bulk copy instead of converting the fp32 matrix again in every CTA.  Disabled (the default), the
// registry is never consulted, so stale entries cannot affect other callers.
namespace dvae {
namespace tc16 {
namespace {
std::mutex g_plane_mu;
std::vector<PlaneTable::Entry> g_plane_reg;
bool g_planes_enabled = false;
}  // namespace

bool find_weight_planes(const float* B, int64_t ldb, int trans_b, int N, int K, PlaneHit* hit) {
  if (!g_planes_enabled) return false;
  std::lock_guard<std::mutex> lk(g_plane_mu);
  for (const PlaneTable::Entry& e : g_plane_reg) {
    if (B < e.w || B >= e.w + (int64_t)e.R * e.C || ldb != e.C) continue;
    const int64_t off = B - e.w;
    const int r0 = (int)(off / e.C), c0 = (int)(off % e.C);
    if (!trans_b) {          // B = W[r0 : r0 + N, c0 : c0 + K]: planes of W (rows = N axis, K along the columns)
      if (!e.planes || r0 % 128 || c0 % 32 || r0 + N > e.R || c0 + K > e.C) return false;
      hit->planes = e.planes; hit->tile0 = r0 / 128; hit->kb0 = c0 / 32; hit->kbtot = (e.C + 31) / 32;
    } else {                 // B stored [K, N] = W[r0 : r0 + K, c0 : c0 + N]: planes of W^T (rows = columns of W, K along W's rows)
      if (!e.planes_t || c0 % 128 || r0 % 32 || r0 + K > e.R || c0 + N > e.C) return false;
      hit->planes = e.planes_t; hit->tile0 = c0 / 128; hit->kb0 = r0 / 32; hit->kbtot = (e.R + 31) / 32;
    }
    return true;
  }
  return false;
}
}  // namespace tc16
}  // namespace dvae

extern "C" int64_t dvae_weight_planes_floats(int R, int C, int transposed) {
  return transposed ? dvae::tc16::plane_floats(C, R) : dvae::tc16::plane_floats(R, C);
}
extern "C" int dvae_weight_planes_register(const float* w, int R, int C, void* planes, void* planes_t) {
  using namespace dvae::tc16;
  DVAE_REQUIRE(w && R > 0 && C > 0 && (planes || planes_t), "dvae_weight_planes_register: bad argument");
  DVAE_REQUIRE(((reinterpret_cast<uintptr_t>(planes) | reinterpret_cast<uintptr_t>(planes_t)) & 15) == 0,
               "dvae_weight_planes_register: plane buffers must be 16-byte aligned");
  std::lock_guard<std::mutex> lk(g_plane_mu);
  for (PlaneTable::Entry& e : g_plane_reg)
    if (e.w == w) { e.R = R; e.C = C; e.planes = planes; e.planes_t = planes_t; return DVAE_OK; }
  DVAE_REQUIRE((int)g_plane_reg.size() < kMaxPlaneEntries, "dvae_weight_planes_register: more than %d weights", kMaxPlaneEntries);
  g_plane_reg.push_back(PlaneTable::Entry{w, R, C, planes, planes_t});
  return DVAE_OK;
}
extern "C" int dvae_weight_planes_clear(void) {
  using namespace dvae::tc16;
  std::lock_guard<std::mutex> lk(g_plane_mu);
  g_plane_reg.clear();
  g_planes_enabled = false;
  return DVAE_OK;
}
extern "C" int dvae_weight_planes_enable(int on) {
  dvae::tc16::g_planes_enabled = on != 0;
  return DVAE_OK;
}
extern "C" int dvae_weight_planes_refresh_ex(int first, int count, void* stream) {
  using namespace dvae::tc16;
  PlaneTable tab;
  {
    std::lock_guard<std::mutex> lk(g_plane_mu);
    const int n = (int)g_plane_reg.size();
    DVAE_REQUIRE(first >= 0 && count >= 0 && first + count <= n, "dvae_weight_planes_refresh_ex: entries [%d, %d) of %d", first, first + count, n);
    tab.n = count;
    for (int i = 0; i < count; ++i) tab.e[i] = g_plane_reg[first + i];
  }
  return weight_planes_launch(tab, (cudaStream_t)stream);
}
extern "C" int dvae_weight_planes_refresh(void* stream) {
  int n;
  {
    std::lock_guard<std::mutex> lk(dvae::tc16::g_plane_mu);
    n = (int)dvae::tc16::g_plane_reg.size();
  }
  return dvae_weight_planes_refresh_ex(0, n, stream);
}

extern "C" int dvae_defer_joins(int on) {
  dvae::set_defer_joins(on != 0);
  return DVAE_OK;
}
extern "C" int dvae_join_side_streams(void* stream) {
  dvae::set_defer_joins(false);
  return dvae::join_side_streams((cudaStream_t)stream);
}
extern "C" int dvae_fork_after(int include_sides, void* extra_stream, void* stream, void** forked_stream_out) {
  DVAE_REQUIRE(forked_stream_out, "dvae_fork_after: null pointer");
  cudaStream_t out = nullptr;
  const int rc = dvae::fork_after(include_sides != 0, (cudaStream_t)extra_stream, (cudaStream_t)stream, &out);
  *forked_stream_out = (void*)out;
  return rc;
}
extern "C" int dvae_counter_increment(uint32_t* counter, void* stream) {
  DVAE_REQUIRE(counter, "dvae_counter_increment: null pointer");
  dvae::counter_increment_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(counter);
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}
extern "C" const char* dvae_last_error_string(void) { return dvae::g_err; }
extern "C" int dvae_version(void) { return 100; }
extern "C" int64_t dvae_launch_count(void) { return dvae::g_launches.load(); }
