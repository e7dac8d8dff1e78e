// harmony_b200.cu — host side of libharmony_b200.so: the C ABI of include/harmony_b200.h on top of the
// kernels in kernels.cuh.  One hb_handle == one instance of the reference's `harmony` class
// (/root/reference/src/harmony.h:20-70).  sm_100a only; there is no CPU path.
#include "../../include/harmony_b200.h"

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>

#include <atomic>
#include <chrono>
#include <condition_variable>
#include <mutex>
#include <thread>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <deque>
#include <map>
#include <numeric>
#include <string>
#include <tuple>
#include <unordered_map>
#include <vector>

#include "kernels.cuh"
#include "update_kernel.cuh"
#include "update_kernel4.cuh"
#include "update_kernel5.cuh"
#include "assign_tc3.cuh"
#include "logits_tc.cuh"
#include "apply_tc3.cuh"
#include "stats_tc3.cuh"
#include "setup_device.cuh"

namespace {

using namespace hb;

// ---- NCCL through dlopen (the process usually already holds torch's libnccl.so.2) ---------------
struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  bool ok = false;
} g_nccl;

bool load_nccl(std::string* why) {
  if (g_nccl.ok) return true;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* nm : names) {
    g_nccl.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
    if (g_nccl.lib) break;
  }
  if (!g_nccl.lib) {
    if (why) *why = "cannot dlopen libnccl.so.2";
    return false;
  }
#define L(sym) *(void**)(&g_nccl.sym) = dlsym(g_nccl.lib, "nccl" #sym)
  L(GetUniqueId);
  L(CommInitRank);
  L(AllReduce);
  L(AllGather);
  L(CommDestroy);
  L(GetErrorString);
#undef L
  g_nccl.ok = g_nccl.GetUniqueId && g_nccl.CommInitRank && g_nccl.AllReduce && g_nccl.AllGather && g_nccl.CommDestroy;
  if (!g_nccl.ok && why) *why = "libnccl lacks required symbols";
  return g_nccl.ok;
}

// one NCCL communicator per (device, rank, world) is kept for the life of the process and shared by every
// handle that asks for it with a NULL id (communicator set-up costs ~1 s; models come and go)
struct CommKey {
  int device, rank, world;
  bool operator<(const CommKey& o) const {
    return std::tie(device, rank, world) < std::tie(o.device, o.rank, o.world);
  }
};
std::map<CommKey, ncclComm_t> g_comms;

struct Region {
  double ms = 0;
  int64_t launches = 0;
};

// ---- host worker pool: widens float -> double into caller memory with several threads ---------------------
// A device -> host copy into pageable memory runs at the speed of one driver thread that also takes the page
// faults of a freshly allocated destination.  The download path (hb_get_field) instead DMA's
// floats into pinned staging and lets this pool widen + scatter them while the next chunk is in flight.
class WidenPool {
 public:
  explicit WidenPool(int nthreads) {
    for (int i = 1; i < nthreads; ++i) workers_.emplace_back([this] { run(); });
  }
  ~WidenPool() {
    {
      std::lock_guard<std::mutex> lk(m_);
      stop_ = true;
      ++gen_;
    }
    cv_job_.notify_all();
    for (auto& t : workers_) t.join();
  }
  int threads() const { return (int)workers_.size() + 1; }
  // dst[i] = (double) src[i], i < n; the caller takes part
  void widen(double* dst, const float* src, size_t n) {
    {
      std::lock_guard<std::mutex> lk(m_);
      dst_ = dst;
      src_ = src;
      n_ = n;
      next_.store(0);
      pending_ = (int)workers_.size();
      ++gen_;
    }
    cv_job_.notify_all();
    work();
    std::unique_lock<std::mutex> lk(m_);
    cv_done_.wait(lk, [this] { return pending_ == 0; });
  }

 private:
  static constexpr size_t kSlice = (size_t)1 << 18;  // elements per grab (2 MiB of doubles)
  void work() {
    for (;;) {
      const size_t i0 = next_.fetch_add(kSlice);
      if (i0 >= n_) break;
      const size_t i1 = std::min(n_, i0 + kSlice);
      for (size_t i = i0; i < i1; ++i) dst_[i] = (double)src_[i];
    }
  }
  void run() {
    uint64_t seen = 0;
    for (;;) {
      {
        std::unique_lock<std::mutex> lk(m_);
        cv_job_.wait(lk, [&] { return gen_ != seen; });
        seen = gen_;
        if (stop_) return;
      }
      work();
      {
        std::lock_guard<std::mutex> lk(m_);
        if (--pending_ == 0) cv_done_.notify_all();
      }
    }
  }
  std::vector<std::thread> workers_;
  std::mutex m_;
  std::condition_variable cv_job_, cv_done_;
  double* dst_ = nullptr;
  const float* src_ = nullptr;
  size_t n_ = 0;
  std::atomic<size_t> next_{0};
  int pending_ = 0;
  uint64_t gen_ = 0;
  bool stop_ = false;
};
WidenPool* widen_pool(int want = 0) {
  static std::mutex mk;
  static WidenPool* pool = nullptr;
  std::lock_guard<std::mutex> lk(mk);
  if (!pool) {
    int n = want;
    if (n <= 0) {
      const char* e = getenv("HB_HOST_THREADS");
      n = e ? atoi(e) : (int)std::min(16u, std::max(1u, std::thread::hardware_concurrency()));
    }
    pool = new WidenPool(std::max(1, n));  // lives until the process exits
  }
  return pool;
}

// Host-side phase timer for the one-off calls (HB_TRACE_HOST=1): every mark() drains the stream and prints the
// wall-clock time since the previous mark to stderr.  Off: a single branch per mark.
struct HostLap {
  cudaStream_t stream;
  const char* call;
  bool on;
  std::chrono::steady_clock::time_point t;
  HostLap(cudaStream_t s, const char* c) : stream(s), call(c), on(getenv("HB_TRACE_HOST") != nullptr) {
    if (on) t = std::chrono::steady_clock::now();
  }
  void mark(const char* what) {
    if (!on) return;
    cudaStreamSynchronize(stream);
    const auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[hb] %s: %-28s %9.3f ms\n", call, what, std::chrono::duration<double, std::milli>(now - t).count());
    t = now;
  }
};

// utils.cpp:102-108
int my_ceil(float num) {
  int inum = (int)num;
  if (num == (float)inum) return inum;
  return inum + 1;
}

// exchange area of the persistent update kernel for sharded cells (see setup_peer_exchange)
struct XchArea {
  int device = 0, world = 0, rank = 0;
  size_t slots = 0, XH = 0, remT_floats = 0;
  float* base = nullptr;     // [inbox: slots * world * XH floats | flags: slots * world words | remT: remT_floats]
  void* peer[U4_MAXWORLD] = {};
  unsigned epoch = 0;
  bool leased = false;
};

// Device buffers come from the device's default memory pool (stream-ordered allocator), whose release threshold
// hb_create raises to "keep everything": a model created after another one was dropped reuses the cached memory
// instead of paying cudaMalloc's OS mapping again (measured: 44 ms of a 100 ms end-to-end run at 1M cells).
// Frees keep cudaFree's contract: nothing of the device may still be using the memory.
template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  ~DevBuf() { release(); }
  void release() {
    if (p) {
      cudaDeviceSynchronize();
      if (cudaFreeAsync(p, 0) != cudaSuccess) {
        cudaGetLastError();
        cudaFree(p);
      }
    }
    p = nullptr;
    n = 0;
  }
  cudaError_t alloc(size_t count) {
    release();
    if (count == 0) count = 1;
    cudaError_t e = cudaMallocAsync((void**)&p, count * sizeof(T), 0);
    if (e == cudaSuccess) e = cudaStreamSynchronize(0);  // ordered on the (idle) default stream: usable from any stream now
    if (e != cudaSuccess) {  // no pool support / pool exhausted: plain allocation
      cudaGetLastError();
      e = cudaMalloc((void**)&p, count * sizeof(T));
    }
    if (e == cudaSuccess) n = count;
    return e;
  }
};
void keep_pool_memory(int device) {
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
    uint64_t keep = ~0ull;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
  }
  cudaGetLastError();
}

}  // namespace

struct hb_handle {
  int device = 0;
  int num_sms = 148;
  cudaStream_t stream = nullptr;
  std::string err;
  std::deque<std::string> warnings;

  // problem
  int64_t N_global = 0, cell_offset = 0, n = 0;
  bool shard_set = false;
  int d = 0, K = 0, B = 0, C = 0, J = 0;
  int KS = 0, DS = 0;  // row strides (multiples of 4 floats) of U/R/O/E and of Zo/Zc
  std::vector<int> B_vec, cov_of;
  float block_size = 0, epsilon_kmeans = 0, epsilon_harmony = 0, alpha = 0, cutoff = 0;
  unsigned max_iter_kmeans = 0, window_size = 3;
  bool lambda_estimation = false, ran_setup = false, ran_init = false;
  int verbose = 0;
  uint64_t seed = 0x5eedULL, round_counter = 0;
  int nb = 0;
  uint32_t cpb = 0;
  int half_bits = 1;
  int (*abort_cb)(void*) = nullptr;
  void* abort_user = nullptr;

  // device state
  DevBuf<float> Zo, Zc, U, R, Y, sigma, theta, Pr_b, N_b, lambda, O, E, P, Oacc, acc, S, V, Wfull, scratch, trace_d;
  DevBuf<float> ring, acc2, Psave, OEend, tmpT;  // persistent update kernel state
  DevBuf<double> obj2;
  DevBuf<unsigned> bar;
  DevBuf<unsigned long long> scan_state;  // chained scan of the plan's histograms: [plan_batch][1 + tiles]
  DevBuf<long long> dbg;  // optional step-phase timestamps (HB_TRACE_STEPS=<cta>)
  int dbg_cta = -1;
  int plan_rounds = 0;   // rounds each plan buffer set holds (two sets: current call / prebuilt next call)
  int plan_set = 0;      // set used by the running cluster_cpp call
  bool next_ready = false;  // the other set holds a prebuilt native plan for the next call ...
  int next_T = 0;           // ... covering this many rounds
  cudaStream_t plan_stream = nullptr;
  cudaEvent_t plan_done = nullptr;
  bool use_v2 = true;
  bool sigma_uniform = false;
  float sigma0 = 0.f;
  bool R_user_set = false;  // R was written through hb_set_field since the last assignment step
  int coop_grid = 0;
  DevBuf<double> obj_acc, stage;
  DevBuf<int> sort_perm, inv_sort, tuple_levels, cov_of_d, tile_cell0, tile_len, tile_tuple, chunk_start,
      tuple_chunk0, blk_of, order, prev_at, H, seg_start, tile_base, iscratch, skipped, err_flag;
  DevBuf<int64_t> perms_d;
  DevBuf<int4> ranges;  // [T][nb][coop_grid] tuple-aligned CTA ranges (when 2 J <= grid)
  bool aligned_ranges = false;
  DevBuf<int> tc_cell0, tc_len, tc_tuple;  // 128-cell tiles of the tensor-core kernels
  int tc_ntiles = 0;
  bool use_tc_assign = false, use_tc_apply = false, use_tc_stats = false;
  bool use_tc_logits = false;  // cold start of shapes outside the fused assignment kernel: logits_tc.cuh
  int kernel_set = 0;            // HB_KERNEL_SET test hook (bits HB_KS_*), read by hb_setup
  bool legacy_centroid = false;  // HB_LEGACY_CENTROID_STEP: centroid update at the top of every clustering round
  DevBuf<float> Rkeep, OEkeep;   // R / O,E saved around the distance-only assignment of that step
  DevBuf<double> objkeep;
  bool use_v4 = false;   // single-pass persistent update kernel (update_kernel4.cuh): the default
  int u5_ring_rows = 0;  // rows of a warp's private ring (update_kernel5.cuh); 0: that kernel cannot run this row width
  int plan_batch = 1;    // rounds sorted per launch (size of the histogram scratch)
  int plan_nsub = 1;     // third sort key of the plan: block in the next round (nb values) or off (1)
  bool use_xch = false;  // sharded cells: block steps exchanged through peer memory (one cooperative launch per call)
  Upd4Xch xch{};
  XchArea* xarea = nullptr;  // leased exchange area (process-wide pool, see setup_peer_exchange)
  int assign_ns = 2;     // operand stages of the tensor-core assignment kernel
  bool zc_pending_norm = false;  // Zc holds the un-normalised corrected embedding although cluster_cpp has run
  DevBuf<int> pt_p0, pt_len, pt_tuple, pt_blk, pt_count, pt_base;  // [2 sets] 128-row tiles of round 0 in plan order
  size_t pt_cap = 0;
  DevBuf<float> remT;    // [2][nb][J][KS] next round's removal sums per (block, tuple)
  DevBuf<float> remS;    // [nb][J][KS] sharded cells: the ranks' remT of one round, summed
  DevBuf<int> next_at, chunk_q0, chunk_nq;
  DevBuf<int> lvl_ptr, lvl_tup;  // CSR level -> tuples (+ one trailing word: B_vec[0])
  int ntiles = 0, nchunks = 0;  // nchunks includes the trailing empty chunk
  int trace_cap = 0;
  std::vector<int> tuple_levels_h;  // [J][C]
  std::vector<int64_t> kmeans_cells;  // global cells chosen by the native initialize_centroids (test hook)

  // traces (harmony.h:55-56); values are produced on the device and pulled lazily
  int obj_count = 0;                      // objective evaluations so far (device slots)
  std::vector<float> obj_vals;            // 4 per slot, host mirror (first obj_synced slots valid)
  int obj_synced = 0;
  std::vector<int> harmony_slots;         // objective_harmony[i] = objective_kmeans[harmony_slots[i]]
  std::vector<int> kmeans_rounds;

  // multi-GPU
  ncclComm_t comm = nullptr;
  int rank = 0, world = 1;

  // instrumentation
  int64_t launches = 0;
  bool timing = false;
  std::map<std::string, Region> regions;
  cudaEvent_t ev0 = nullptr;  // orders the side-stream plan build after the main stream
  cudaEvent_t io_ev = nullptr;  // orders device-memory inputs / outputs against the caller's stream
};

namespace {

int fail(hb_handle* h, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  h->err = buf;
  return code;
}

#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess) return fail(h, 10, "CUDA error %s at %s:%d", cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)
#define CKN(call)                                                                                  \
  do {                                                                                             \
    ncclResult_t r__ = (call);                                                                     \
    if (r__ != ncclSuccess)                                                                        \
      return fail(h, 11, "NCCL error %s at %s:%d", g_nccl.GetErrorString ? g_nccl.GetErrorString(r__) : "?", __FILE__, __LINE__); \
  } while (0)
#define CKL()                                                                                      \
  do {                                                                                             \
    h->launches++;                                                                                 \
    cudaError_t e__ = cudaGetLastError();                                                          \
    if (e__ != cudaSuccess) return fail(h, 10, "kernel launch failed: %s at %s:%d", cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)
#define TRY(expr)            \
  do {                       \
    int st__ = (expr);       \
    if (st__ != 0) return st__; \
  } while (0)

struct RegionScope {
  hb_handle* h;
  const char* name;
  int64_t l0;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  RegionScope(hb_handle* h_, const char* n) : h(h_), name(n), l0(h_->launches) {
    if (h->timing) {
      cudaEventCreate(&e0);
      cudaEventCreate(&e1);
      cudaEventRecord(e0, h->stream);
    }
  }
  ~RegionScope() {
    Region& r = h->regions[name];
    r.launches += h->launches - l0;
    if (e0) {
      cudaEventRecord(e1, h->stream);
      cudaEventSynchronize(e1);
      float ms = 0;
      cudaEventElapsedTime(&ms, e0, e1);
      r.ms += ms;
      cudaEventDestroy(e0);
      cudaEventDestroy(e1);
    }
  }
};

int grid_for(int64_t work_items, int threads, int cap) {
  int64_t g = (work_items + threads - 1) / threads;
  if (g < 1) g = 1;
  if (g > cap) g = cap;
  return (int)g;
}

int allreduce_f(hb_handle* h, float* p, size_t count) {
  if (h->world <= 1) return 0;
  CKN(g_nccl.AllReduce(p, p, count, ncclFloat, ncclSum, h->comm, h->stream));
  return 0;
}
int allreduce_d(hb_handle* h, double* p, size_t count) {
  if (h->world <= 1) return 0;
  CKN(g_nccl.AllReduce(p, p, count, ncclDouble, ncclSum, h->comm, h->stream));
  return 0;
}

int kq_for(int K) {
  int q = (K + 31) / 32;
  int kq = 1;
  while (kq < q) kq <<= 1;
  return kq;
}

template <typename F>
int dispatch_kq(hb_handle* h, int K, F&& f) {
  switch (kq_for(K)) {
    case 1: return f(std::integral_constant<int, 1>());
    case 2: return f(std::integral_constant<int, 2>());
    case 4: return f(std::integral_constant<int, 4>());
    case 8: return f(std::integral_constant<int, 8>());
    case 16: return f(std::integral_constant<int, 16>());
    case 32: return f(std::integral_constant<int, 32>());
  }
  return fail(h, 2, "K = %d is not supported (K <= 1024)", K);
}

// U[i][k] = (2 / sigma_k) (z_i . y_k / |z_i| - 1) for all clusters on the tensor cores, 64 clusters per launch
// (logits_tc.cuh); `sigma`: device array of K values
int launch_logits(hb_handle* h, const float* sigma, bool normalise) {
  LogitsArgs t{};
  t.Zc = h->Zc.p;
  t.Y = h->Y.p;
  t.sigma = sigma;
  t.U = h->U.p;
  t.n = h->n;
  t.d = h->d;
  t.K = h->K;
  t.DS = h->DS;
  t.KS = h->KS;
  t.KD = (h->d + 7) & ~7;
  t.normalise = normalise ? 1 : 0;
  const size_t smem_lg = logits_smem_bytes(t.KD);
  CK(cudaFuncSetAttribute(k_logits_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_lg));
  const int grid_lg = (int)std::max<int64_t>(1, std::min<int64_t>((h->n + LG_TM - 1) / LG_TM, h->num_sms));
  for (t.n_off = 0; t.n_off < h->K; t.n_off += LG_NP) {
    k_logits_tc<<<grid_lg, LG_THREADS, smem_lg, h->stream>>>(t);
    CKL();
  }
  return 0;
}

// ---- K1 launcher: assignment from centroids (init + cold start) -------------------------------
// plan_mode: tiles follow round 0 of the current plan set (tensor-core kernel only); want_obj: objective sums (init)
int run_assign(hb_handle* h, bool normalise, bool plan_mode = false, bool want_obj = true) {
  RegionScope rs(h, "assign");
  const int K = h->K, d = h->d, B = h->B, KS = h->KS;
  const int KP = (K + 63) & ~63, DP4 = (d + 3) & ~3;
  CK(cudaMemsetAsync(h->Oacc.p, 0, sizeof(float) * ((size_t)B * KS + KS), h->stream));
  AssignArgs a;
  a.Zc = h->Zc.p;
  a.Y = h->Y.p;
  a.sigma = h->sigma.p;
  a.U = h->U.p;
  a.R = h->R.p;
  a.tile_cell0 = h->tile_cell0.p;
  a.tile_len = h->tile_len.p;
  a.tile_tuple = h->tile_tuple.p;
  a.tuple_levels = h->tuple_levels.p;
  a.O_acc = h->Oacc.p;
  a.rs_acc = h->Oacc.p + (size_t)B * KS;
  a.obj_acc = h->obj_acc.p;
  a.ntiles = h->ntiles;
  a.d = d;
  a.K = K;
  a.C = h->C;
  a.KP = KP;
  a.DS = h->DS;
  a.KS = KS;
  a.normalise = normalise ? 1 : 0;
  if (h->use_tc_assign) {
    Assign3Args t{};
    t.Zc = a.Zc;
    t.Y = a.Y;
    t.sigma = a.sigma;
    t.U = a.U;
    t.tuple_levels = a.tuple_levels;
    t.obj_acc = a.obj_acc;
    t.d = d;
    t.K = K;
    t.C = h->C;
    t.B = B;
    t.DS = h->DS;
    t.KS = KS;
    t.KD = (d + 7) & ~7;
    t.NP = (K + 15) & ~15;
    t.SS = assign3_stage_stride(KS);
    t.ns = h->assign_ns;
    t.normalise = a.normalise;
    t.want_obj = want_obj ? 1 : 0;
    int grid_tc;
    if (plan_mode) {
      // rows in the order of round 0 of the coming cluster_cpp call: a tile's column sums are a share of its block's
      // removal sums and go to the update kernel's accumulator slots; R is not stored
      const size_t R0 = (size_t)h->plan_set * h->plan_rounds;
      const size_t cap = h->pt_cap;
      t.R = nullptr;
      t.row_index = h->order.p + R0 * h->n;
      t.tile_p0 = h->pt_p0.p + (size_t)h->plan_set * cap;
      t.tile_len = h->pt_len.p + (size_t)h->plan_set * cap;
      t.tile_tuple = h->pt_tuple.p + (size_t)h->plan_set * cap;
      t.tile_blk = h->pt_blk.p + (size_t)h->plan_set * cap;
      t.ntiles_ptr = h->pt_count.p + h->plan_set;
      t.ntiles = 0;
      t.acc = h->acc2.p;
      t.Zc_out = nullptr;
      grid_tc = h->num_sms;
    } else {
      t.R = a.R;
      t.row_index = nullptr;
      t.tile_p0 = h->tc_cell0.p;
      t.tile_len = h->tc_len.p;
      t.tile_tuple = h->tc_tuple.p;
      t.tile_blk = nullptr;
      t.ntiles_ptr = nullptr;
      t.ntiles = h->tc_ntiles;
      t.O_acc = a.O_acc;
      t.rs_acc = a.rs_acc;
      t.Zc_out = normalise ? h->Zc.p : nullptr;  // the compatibility paths read the normalised embedding back
      grid_tc = std::max(1, std::min(h->tc_ntiles, h->num_sms));
    }
    const size_t smem_tc = assign3_smem_bytes(t.ns, t.KD, t.NP, KS);
    t.dbg = nullptr;
    static int as_calls = 0;
    const bool tracing = getenv("HB_TRACE_ASSIGN") != nullptr && plan_mode && (++as_calls == 4);
    if (tracing) {
      if (h->dbg.n < 32 * 16) CK(h->dbg.alloc(32 * 16));
      CK(cudaMemsetAsync(h->dbg.p, 0, sizeof(long long) * 32 * 16, h->stream));
      t.dbg = h->dbg.p;
    }
    if (want_obj) {
      CK(cudaFuncSetAttribute(k_assign_tc3<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_tc));
      k_assign_tc3<true><<<grid_tc, A3_THREADS, smem_tc, h->stream>>>(t);
    } else {
      CK(cudaFuncSetAttribute(k_assign_tc3<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_tc));
      k_assign_tc3<false><<<grid_tc, A3_THREADS, smem_tc, h->stream>>>(t);
    }
    CKL();
    if (tracing) {
      std::vector<long long> st(32 * 16);
      CK(cudaMemcpyAsync(st.data(), h->dbg.p, sizeof(long long) * st.size(), cudaMemcpyDeviceToHost, h->stream));
      CK(cudaStreamSynchronize(h->stream));
      if (FILE* f = fopen("gpurun_out/assign_trace.txt", "w")) {
        for (int i = 0; i < 32; ++i) {
          fprintf(f, "%d", i);
          for (int k = 0; k < 16; ++k) fprintf(f, " %lld", st[(size_t)i * 16 + k] ? st[(size_t)i * 16 + k] - st[0] : -1);
          fprintf(f, "\n");
        }
        fclose(f);
      }
    }
    h->R_user_set = false;
    if (plan_mode) {
      // O, E of the assignment = the sums of the blocks' removal terms (harmony.cpp:226-227)
      const size_t XH = (size_t)B * KS + KS;
      // sharded cells: the rem halves of slots 1 .. nb in ONE all-reduce (their add halves are still zero here)
      if (h->world > 1) TRY(allreduce_f(h, h->acc2.p + 2 * XH, 2 * XH * (size_t)h->nb));
      k_assign_finalize_plan<<<(B * KS + 255) / 256, 256, 0, h->stream>>>(h->acc2.p, h->nb, h->Pr_b.p, h->O.p, h->E.p, B, K, KS);
      CKL();
      h->zc_pending_norm = normalise;  // the normalised embedding (harmony.cpp:220) is materialised on demand
      return 0;
    }
    TRY(allreduce_f(h, h->Oacc.p, (size_t)B * KS + KS));
    k_assign_finalize<<<(B * KS + 255) / 256, 256, 0, h->stream>>>(h->Oacc.p, h->Oacc.p + (size_t)B * KS, h->Pr_b.p,
                                                                    h->O.p, h->E.p, B, K, KS);
    CKL();
    return 0;
  }
  if (plan_mode && h->use_tc_logits) {
    // shapes the fused kernel cannot hold (d > 64 or K > 128): logits per 64-cluster range on the tensor cores, then
    // one gather pass over U in the order of round 0 for the softmax + the blocks' removal sums (harmony.cpp:312-313)
    TRY(launch_logits(h, h->sigma.p, normalise));
    const size_t R0 = (size_t)h->plan_set * h->plan_rounds;
    const int nv = upd4_nv(KS);
    const size_t smem_sm = sizeof(float) * 8 * 128 * (size_t)nv;
    if (nv == 1)
      k_softmax_block_sums<1><<<dim3(h->coop_grid, h->nb), 256, smem_sm, h->stream>>>(
          h->U.p, h->order.p + R0 * h->n, h->ranges.p + R0 * h->nb * h->coop_grid, h->tuple_levels.p, h->acc2.p, h->coop_grid, K, KS,
          h->C, B);
    else
      k_softmax_block_sums<2><<<dim3(h->coop_grid, h->nb), 256, smem_sm, h->stream>>>(
          h->U.p, h->order.p + R0 * h->n, h->ranges.p + R0 * h->nb * h->coop_grid, h->tuple_levels.p, h->acc2.p, h->coop_grid, K, KS,
          h->C, B);
    CKL();
    h->R_user_set = false;
    const size_t XH = (size_t)B * KS + KS;
    if (h->world > 1) TRY(allreduce_f(h, h->acc2.p + 2 * XH, 2 * XH * (size_t)h->nb));
    k_assign_finalize_plan<<<(B * KS + 255) / 256, 256, 0, h->stream>>>(h->acc2.p, h->nb, h->Pr_b.p, h->O.p, h->E.p, B, K, KS);
    CKL();
    h->zc_pending_norm = normalise;
    return 0;
  }
  if (plan_mode) return fail(h, 3, "internal: plan-order assignment without the tensor-core kernel");
  size_t smem = sizeof(float) * ((size_t)DP4 * KP + (size_t)TM * DP4 + (size_t)TM * (KP + 4) + KP + (size_t)NWARP * KP);
  if (smem > 227 * 1024) return fail(h, 2, "K*d too large for the assignment kernel (needs %zu B shared memory)", smem);
  int st = dispatch_kq(h, K, [&](auto kq) -> int {
    constexpr int KQ = decltype(kq)::value;
    CK(cudaFuncSetAttribute(k_assign<KQ>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 1;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_assign<KQ>, ASSIGN_THREADS, smem));
    if (occ < 1) occ = 1;
    int grid = std::min(h->ntiles, h->num_sms * occ);
    if (grid < 1) grid = 1;
    k_assign<KQ><<<grid, ASSIGN_THREADS, smem, h->stream>>>(a);
    CKL();
    return 0;
  });
  TRY(st);
  h->R_user_set = false;
  TRY(allreduce_f(h, h->Oacc.p, (size_t)B * KS + KS));
  k_assign_finalize<<<(B * KS + 255) / 256, 256, 0, h->stream>>>(h->Oacc.p, h->Oacc.p + (size_t)B * KS, h->Pr_b.p,
                                                                  h->O.p, h->E.p, B, K, KS);
  CKL();
  return 0;
}

int ensure_trace_cap(hb_handle* h, int slots) {
  if (slots <= h->trace_cap) return 0;
  int ncap = std::max(1024, h->trace_cap * 2);
  while (ncap < slots) ncap *= 2;
  float* np = nullptr;
  CK(cudaMalloc((void**)&np, sizeof(float) * 4 * (size_t)ncap));
  if (h->trace_d.p && h->obj_count > 0)
    CK(cudaMemcpyAsync(np, h->trace_d.p, sizeof(float) * 4 * (size_t)h->obj_count, cudaMemcpyDeviceToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  if (h->trace_d.p) cudaFree(h->trace_d.p);
  h->trace_d.p = np;
  h->trace_d.n = 4 * (size_t)ncap;
  h->trace_cap = ncap;
  return 0;
}

// obj holds this rank's per-cell sums; fold in the K x B cross term of tables (O, E) and append to the trace
int push_objective_from(hb_handle* h, const float* O, const float* E, double* obj) {
  TRY(ensure_trace_cap(h, h->obj_count + 1));
  TRY(allreduce_d(h, obj, 2));
  k_objective_finalize<<<1, 256, 0, h->stream>>>(O, E, h->theta.p, h->sigma.p, obj, h->trace_d.p, h->obj_count, h->B,
                                                  h->K, h->KS, (double)h->N_global, 1.0);
  CKL();
  h->obj_count++;
  return 0;
}
int push_objective(hb_handle* h) { return push_objective_from(h, h->O.p, h->E.p, h->obj_acc.p); }

int sync_traces(hb_handle* h) {
  if (h->obj_synced == h->obj_count) return 0;
  h->obj_vals.resize(4 * (size_t)h->obj_count);
  CK(cudaMemcpyAsync(h->obj_vals.data() + 4 * (size_t)h->obj_synced, h->trace_d.p + 4 * (size_t)h->obj_synced,
                     sizeof(float) * 4 * (size_t)(h->obj_count - h->obj_synced), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  h->obj_synced = h->obj_count;
  return 0;
}

// harmony.cpp:173-205
int check_convergence_host(hb_handle* h, int type, int* out) {
  TRY(sync_traces(h));
  float obj_new, obj_old;
  auto ok = [&](int slot) { return h->obj_vals[4 * (size_t)slot]; };
  switch (type) {
    case 0: {
      if (h->obj_count < (int)h->window_size + 1) return fail(h, 3, "check_convergence(0): not enough objective values");
      obj_old = 0;
      obj_new = 0;
      for (unsigned i = 0; i < h->window_size; i++) {
        obj_old += ok(h->obj_count - 2 - (int)i);
        obj_new += ok(h->obj_count - 1 - (int)i);
      }
      *out = (std::abs(obj_old - obj_new) / std::abs(obj_old) < h->epsilon_kmeans) ? 1 : 0;
      return 0;
    }
    case 1: {
      if (h->harmony_slots.size() < 2) return fail(h, 3, "check_convergence(1): not enough objective values");
      obj_old = ok(h->harmony_slots[h->harmony_slots.size() - 2]);
      obj_new = ok(h->harmony_slots[h->harmony_slots.size() - 1]);
      *out = ((obj_old - obj_new) / std::abs(obj_old) < h->epsilon_harmony) ? 1 : 0;
      return 0;
    }
  }
  *out = 1;
  return 0;
}

// ---- update-order plan (buffers hold plan_rounds rounds, two sets) ----------------------------------
// Phase A: the block of every local cell in round t (harmony.cpp:272-291: position in the shuffled order / cells
// per block).  Phase B: the round's rows sorted by (block, tuple, block in the next round) + the derived tables.
// rounds [t, t + nt) of a buffer set in one launch (blockIdx.y = round)
int plan_blocks(hb_handle* h, int t, int nt, const int64_t* perm_d /* device, nt x N_global, or null */, int set, cudaStream_t st) {
  RegionScope rs(h, "plan");
  const int64_t n = h->n;
  const size_t R0 = (size_t)set * h->plan_rounds;  // first round slot of this buffer set
  int* blk_of = h->blk_of.p + (R0 + t) * n;
  if (perm_d) {
    CK(cudaMemsetAsync(blk_of, 0xff, sizeof(int) * (size_t)n * nt, st));
    k_plan_block_injected<<<dim3(grid_for(h->N_global, 256, h->num_sms * 8), nt), 256, 0, st>>>(
        perm_d, h->N_global, h->cell_offset, n, h->inv_sort.p, h->cpb, h->nb, blk_of, h->err_flag.p);
    CKL();
  } else {
    k_plan_block_native<<<dim3(grid_for(n, 256, h->num_sms * 8), nt), 256, 0, st>>>(
        h->N_global, h->cell_offset, n, h->sort_perm.p, h->cpb, h->nb, h->half_bits, h->seed, h->round_counter, blk_of);
    CKL();
  }
  h->round_counter += (uint64_t)nt;
  return 0;
}
// counting sort of rounds [t, t + nt) (nt <= plan_batch: the histogram scratch holds that many rounds); round
// t + nt - 1 has a next round iff last_has_next
int plan_sort(hb_handle* h, int t, int nt, bool last_has_next, int set, cudaStream_t st, bool tiles = false) {
  RegionScope rs(h, "plan");
  const int nb = h->nb, J = h->J, nc = h->nchunks, nsub = h->plan_nsub;
  const int64_t n = h->n;
  const int S = nb * J;
  const size_t R0 = (size_t)set * h->plan_rounds;
  const int* blk_of = h->blk_of.p + (R0 + t) * n;
  int* order = h->order.p + (R0 + t) * n;
  int* seg_start = h->seg_start.p + (R0 + t) * (S + 1);
  int* tile_base = h->tile_base.p + (R0 + t) * (S + 1);
  const size_t per_warp = sizeof(int) * (size_t)nb * nsub;
  const int wpb = (int)std::max<size_t>(1, std::min<size_t>(8, (48 * 1024) / per_warp));  // warps per block
  const size_t sm = per_warp * wpb;
  const int with_next = last_has_next ? nt : nt - 1;
  k_plan_hist<<<dim3((nc + wpb - 1) / wpb, nt), wpb * 32, sm, st>>>(blk_of, nullptr, h->chunk_start.p, h->chunk_q0.p,
                                                                   h->chunk_nq.p, nc, nb, nsub, h->H.p, h->err_flag.p, n,
                                                                   with_next);
  CKL();
  {  // offsets of the counting sort: chained multi-CTA scan of the nt histograms (a single CTA per round took ~145 us)
    const int64_t hn = (int64_t)nb * nsub * nc;
    const int tiles = (int)((hn + SCAN_TILE - 1) / SCAN_TILE);
    CK(cudaMemsetAsync(h->scan_state.p, 0, sizeof(unsigned long long) * (size_t)nt * (tiles + 1), st));
    k_scan_chained<<<dim3(tiles, nt), 1024, 0, st>>>(h->H.p, hn, h->scan_state.p, tiles);
    CKL();
  }
  k_plan_scatter<<<dim3((nc + wpb - 1) / wpb, nt), wpb * 32, sm, st>>>(
      blk_of, nullptr, h->chunk_start.p, h->chunk_q0.p, h->chunk_nq.p, nc, nb, nsub, h->H.p, order, nullptr,
      (h->use_v2 && !h->use_v4) ? h->prev_at.p + (R0 + t) * n : nullptr, h->use_v4 ? h->next_at.p + (R0 + t) * n : nullptr, n,
      with_next, t > 0 ? 1 : 0);
  CKL();
  k_plan_segments<<<dim3(grid_for(S + 1, 256, 64), nt), 256, 0, st>>>(h->H.p, h->tuple_chunk0.p, nc, nb, nsub, J, (int)n,
                                                                       seg_start, tile_base);
  CKL();
  if (h->use_v2 && h->aligned_ranges) {
    k_plan_ranges<<<dim3(nb, nt), 256, 0, st>>>(seg_start, nb, J, h->coop_grid,
                                                                            h->ranges.p + (R0 + t) * nb * h->coop_grid);
    CKL();
  }
  if (tiles) {  // tile offsets of the first-generation update kernels (single round)
    k_plan_tilecount<<<grid_for(S + 1, 256, 64), 256, 0, st>>>(seg_start, S, tile_base);
    CKL();
    k_scan_exclusive<<<1, 1024, 0, st>>>(tile_base, (int64_t)S + 1, nullptr);
    CKL();
  }
  return 0;
}
// all T rounds of a cluster_cpp call (orders: device, T x N_global, or null for the native keyed orders)
int build_plans(hb_handle* h, int T, const int64_t* orders_d, int set, cudaStream_t st) {
  if (T > 0) TRY(plan_blocks(h, 0, T, orders_d, set, st));
  for (int t = 0; t < T; t += h->plan_batch) {
    const int nt = std::min(h->plan_batch, T - t);
    TRY(plan_sort(h, t, nt, t + nt < T, set, st));
  }
  if (T > 0 && h->use_tc_assign && h->use_v4) {
    // 128-row tiles of round 0, one (block, tuple) segment at a time: the assignment step of the call runs in this order
    RegionScope rs(h, "plan");
    const int S = h->nb * h->J;
    const int* seg_start = h->seg_start.p + (size_t)set * h->plan_rounds * (S + 1);
    k_plan_tilecount128<<<grid_for(S + 1, 256, 64), 256, 0, st>>>(seg_start, S, h->pt_base.p);
    CKL();
    k_scan_exclusive<<<1, 1024, 0, st>>>(h->pt_base.p, (int64_t)S + 1, h->pt_count.p + set);
    CKL();
    k_plan_tilefill128<<<grid_for(S, 128, 64), 128, 0, st>>>(seg_start, h->pt_base.p, S, h->J, h->pt_p0.p + (size_t)set * h->pt_cap,
                                                          h->pt_len.p + (size_t)set * h->pt_cap,
                                                          h->pt_tuple.p + (size_t)set * h->pt_cap,
                                                          h->pt_blk.p + (size_t)set * h->pt_cap);
    CKL();
  }
  return 0;
}
// one round into slot 0 of set 0 (per-round paths: first-generation kernels, legacy centroid step)
int build_plan_single(hb_handle* h, const int64_t* perm_d, cudaStream_t st) {
  TRY(plan_blocks(h, 0, 1, perm_d, 0, st));
  return plan_sort(h, 0, 1, false, 0, st, true);
}

// ---- v1: one update_R sweep (harmony.cpp:269-342), three launches per block step ------------------
int run_update_R_v1(hb_handle* h, int t) {
  RegionScope rs(h, "update_R");
  const int K = h->K, B = h->B, nb = h->nb, KS = h->KS;
  const int KP = (K + 63) & ~63;
  const size_t slot = 2 * ((size_t)B * KS + KS);  // [add_O | add_rs | rem_O | rem_rs]
  const int S = nb * h->J;
  CK(cudaMemsetAsync(h->acc.p, 0, sizeof(float) * 2 * slot, h->stream));
  StepArgs a;
  a.U = h->U.p;
  a.R = h->R.p;
  a.order = h->order.p + (size_t)t * h->n;  // v1 always plans into set 0
  a.seg_start = h->seg_start.p + (size_t)t * (S + 1);
  a.tile_base = h->tile_base.p + (size_t)t * (S + 1);
  a.tuple_levels = h->tuple_levels.p;
  a.sigma = h->sigma.p;
  a.P = h->P.p;
  a.obj_acc = h->obj_acc.p;
  a.J = h->J;
  a.K = K;
  a.C = h->C;
  a.KP = KP;
  a.KS = KS;
  const int tiles_bound = (int)std::min<int64_t>((h->n / std::max(1, nb)) / TM + h->J + 8, (int64_t)h->num_sms * 8);
  const int grid = std::max(1, tiles_bound);
  const size_t sm_col = sizeof(float) * (size_t)NWARP * KP;
  const size_t sm_upd = sizeof(float) * ((size_t)NWARP * KP + 3 * (size_t)KP);
  return dispatch_kq(h, K, [&](auto kq) -> int {
    constexpr int KQ = decltype(kq)::value;
    for (int j = 0; j <= nb; ++j) {
      float* sl = h->acc.p + (size_t)(j & 1) * slot;  // slot j = [add_{j-1} | rem_j]
      float* add_O = sl;
      float* add_rs = sl + (size_t)B * KS;
      float* rem_O = sl + (size_t)B * KS + KS;
      float* rem_rs = rem_O + (size_t)B * KS;
      if (j < nb) {
        a.blk = j;
        a.acc_O = rem_O;
        a.acc_rs = rem_rs;
        RegionScope r1(h, "k_block_colsum");
        k_block_colsum<KQ><<<grid, ROW_THREADS, sm_col, h->stream>>>(a);
        CKL();
      }
      TRY(allreduce_f(h, sl, slot));
      {
        RegionScope r2(h, "k_step_prepare");
        k_step_prepare<<<(B * KS + 255) / 256, 256, 0, h->stream>>>(h->O.p, h->E.p, add_O, add_rs, rem_O, rem_rs,
                                                                     h->Pr_b.p, h->theta.p, (j < nb) ? h->P.p : nullptr, B, K, KS);
        CKL();
      }
      CK(cudaMemsetAsync(sl, 0, sizeof(float) * slot, h->stream));
      if (j < nb) {
        float* nx = h->acc.p + (size_t)((j + 1) & 1) * slot;  // add_j goes to slot j+1
        a.acc_O = nx;
        a.acc_rs = nx + (size_t)B * KS;
        RegionScope r3(h, "k_block_update");
        k_block_update<KQ><<<grid, ROW_THREADS, sm_upd, h->stream>>>(a);
        CKL();
      }
    }
    return 0;
  });
}

// ---- peer-memory exchange area of the persistent update kernel (sharded cells, one node) ----------------
// Areas live for the life of the process, like the communicators: another rank may still be writing into an
// area when its owner drops the handle, and unmapping needs a collective that a destructor cannot afford.  A
// handle leases an area; areas are created collectively, so area i here is paired with area i of every rank.
constexpr int XCH_MAX_AREAS = 16;
std::vector<XchArea*> g_xch_areas;

void release_peer_exchange(hb_handle* h) {
  if (h->xarea) {
    h->xarea->epoch = h->xch.epoch;  // the next lessee continues the epoch sequence
    h->xarea->leased = false;
    h->xarea = nullptr;
  }
  h->use_xch = false;
}
// layout of an area (floats): inbox [slots][world][XH] of 8-byte (value, epoch) words | remT [2][nb][J][KS]
uint2* xch_inbox(const XchArea* a, void* base) { return reinterpret_cast<uint2*>(base); }
float* xch_remT(const XchArea* a, void* base) { return reinterpret_cast<float*>(base) + 2 * a->slots * a->world * a->XH; }
// Collective over the handle's communicator.  Leases an area all ranks have free, or creates a new one:
// allocates this rank's part, exchanges the IPC handles and maps the other ranks' parts.  If any rank cannot
// map a peer the exchange stays off on all ranks (the update then runs one launch + all-reduce per block step).
int setup_peer_exchange(hb_handle* h, int Tplan) {
  const int W = h->world;
  const size_t BK = (size_t)h->B * h->KS, XH = BK + h->KS;
  const size_t slots = (size_t)Tplan * h->nb + 2;
  const size_t remT_floats = 2 * (size_t)h->nb * h->J * h->KS;
  release_peer_exchange(h);
  // 1. agree on a reusable area: free here AND on every other rank, same shape
  int64_t freev[XCH_MAX_AREAS + 2];
  for (int i = 0; i < XCH_MAX_AREAS; ++i) {
    const XchArea* a = i < (int)g_xch_areas.size() ? g_xch_areas[i] : nullptr;
    freev[i] = (a && !a->leased && a->device == h->device && a->world == W && a->rank == h->rank && a->slots == slots &&
                a->XH == XH && a->remT_floats == remT_floats) ? 1 : 0;
  }
  freev[XCH_MAX_AREAS] = (int64_t)g_xch_areas.size();       // min over ranks = smallest pool ...
  freev[XCH_MAX_AREAS + 1] = -(int64_t)g_xch_areas.size();  // ... and -(largest pool): they must agree
  DevBuf<int64_t> dv;
  CK(dv.alloc(XCH_MAX_AREAS + 2));
  CK(cudaMemcpyAsync(dv.p, freev, sizeof(freev), cudaMemcpyHostToDevice, h->stream));
  CKN(g_nccl.AllReduce(dv.p, dv.p, XCH_MAX_AREAS + 2, ncclInt64, ncclMin, h->comm, h->stream));
  CK(cudaMemcpyAsync(freev, dv.p, sizeof(freev), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  XchArea* area = nullptr;
  for (int i = 0; i < XCH_MAX_AREAS && !area; ++i)
    if (freev[i] == 1) area = g_xch_areas[i];
  if (!area) {
    // every rank sees the same reduced values, so every rank takes the same branch here
    if (freev[XCH_MAX_AREAS] != -freev[XCH_MAX_AREAS + 1] || freev[XCH_MAX_AREAS] >= XCH_MAX_AREAS) return 0;  // out of step / pool full
    // 2. create a new area (collective)
    XchArea tmp;
    tmp.slots = slots;
    tmp.world = W;
    tmp.XH = XH;
    const size_t total = (size_t)(xch_remT(&tmp, nullptr) - (float*)nullptr) + remT_floats;
    float* base = nullptr;
    CK(cudaMalloc((void**)&base, sizeof(float) * total));
    CK(cudaMemsetAsync(base, 0, sizeof(float) * total, h->stream));
    cudaIpcMemHandle_t mine;
    CK(cudaIpcGetMemHandle(&mine, base));
    DevBuf<char> ds, dr;
    CK(ds.alloc(sizeof(mine)));
    CK(dr.alloc(sizeof(mine) * W));
    CK(cudaMemcpyAsync(ds.p, &mine, sizeof(mine), cudaMemcpyHostToDevice, h->stream));
    CKN(g_nccl.AllGather(ds.p, dr.p, sizeof(mine), ncclChar, h->comm, h->stream));
    std::vector<cudaIpcMemHandle_t> all(W);
    CK(cudaMemcpyAsync(all.data(), dr.p, sizeof(mine) * W, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    area = new XchArea();
    area->device = h->device;
    area->world = W;
    area->rank = h->rank;
    area->slots = slots;
    area->XH = XH;
    area->remT_floats = remT_floats;
    area->base = base;
    int64_t ok = 1;
    for (int r = 0; r < W; ++r) {
      if (r == h->rank) continue;
      if (cudaIpcOpenMemHandle(&area->peer[r], all[r], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
        cudaGetLastError();
        area->peer[r] = nullptr;
        ok = 0;
      }
    }
    CK(cudaMemcpyAsync(dv.p, &ok, sizeof(ok), cudaMemcpyHostToDevice, h->stream));
    CKN(g_nccl.AllReduce(dv.p, dv.p, 1, ncclInt64, ncclMin, h->comm, h->stream));
    CK(cudaMemcpyAsync(&ok, dv.p, sizeof(ok), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    area->leased = !ok;            // an unusable area keeps its index (the ranks stay in step) but is never leased
    g_xch_areas.push_back(area);
    if (!ok) {
      h->warnings.push_back("peer-memory exchange unavailable (CUDA IPC mapping failed); using per-step all-reduce");
      return 0;
    }
  }
  area->leased = true;
  h->xarea = area;
  Upd4Xch& x = h->xch;
  x.world = W;
  x.rank = h->rank;
  x.epoch = area->epoch;
  x.XH = (int)XH;
  for (int r = 0; r < W; ++r) {
    void* b = (r == h->rank) ? (void*)area->base : area->peer[r];
    x.peer_inbox[r] = xch_inbox(area, b);
    x.peer_remT[r] = xch_remT(area, b);
  }
  x.inbox = x.peer_inbox[h->rank];
  h->use_xch = true;
  return 0;
}
float* remT_ptr(hb_handle* h) { return h->use_xch ? h->xch.peer_remT[h->rank] : h->remT.p; }

// ---- persistent update kernels over rounds [t0, t1) of this cluster_cpp call ---------------------------
int nv_for(int KS) {
  int nv = 1;
  while (4 * UPD_LPR * nv < KS) nv <<= 1;
  return nv;
}
template <typename F>
int dispatch_nv(hb_handle* h, int KS, F&& f) {
  switch (nv_for(KS)) {
    case 1: return f(std::integral_constant<int, 1>());
    case 2: return f(std::integral_constant<int, 2>());
    case 4: return f(std::integral_constant<int, 4>());
  }
  return fail(h, 2, "K = %d is not supported by the persistent update kernel", h->K);
}
size_t upd_smem_bytes(const hb_handle* h) {
  const size_t tabn = (size_t)std::max(2, h->nb) * h->KS;
  const int nv = nv_for(h->KS);
  const size_t rowbuf = (size_t)UPD_GWARPS * (upd_depth_upd(nv) + upd_depth_look(nv)) * UPD_RPW * h->KS;
  return sizeof(float) * ((size_t)h->KS + 2 * (tabn + (size_t)UPD_GWARPS * h->KS + 2 * (size_t)UPD_STAGE + (size_t)((h->J + 8) & ~3)) + rowbuf);
}
UpdArgs make_upd_args(hb_handle* h, int T) {
  UpdArgs a;
  a.U = h->U.p;
  a.R = h->R.p;
  const size_t R0 = (size_t)h->plan_set * h->plan_rounds;
  a.order = h->order.p + R0 * h->n;
  a.seg_start = h->seg_start.p + R0 * ((size_t)h->nb * h->J + 1);
  a.prev_at = h->prev_at.p + R0 * h->n;
  a.ranges = h->aligned_ranges ? h->ranges.p + R0 * h->nb * h->coop_grid : nullptr;
  a.tuple_levels = h->tuple_levels.p;
  a.sigma = h->sigma.p;
  a.theta = h->theta.p;
  a.Pr_b = h->Pr_b.p;
  a.ring = h->ring.p;
  a.acc = h->acc2.p;
  a.Psave = h->Psave.p;
  a.OEend = h->OEend.p;
  a.obj = h->obj2.p;
  a.bar = h->bar.p;
  a.n = h->n;
  a.K = h->K;
  a.KS = h->KS;
  a.C = h->C;
  a.J = h->J;
  a.B = h->B;
  a.nb = h->nb;
  a.T = T;
  a.first_round_from_R = h->R_user_set ? 1 : 0;
  a.sigma_uniform = h->sigma_uniform ? 1 : 0;
  a.sigma0 = h->sigma0;
  a.dbg = (h->dbg_cta >= 0) ? h->dbg.p : nullptr;
  a.dbg_cta = h->dbg_cta;
  return a;
}
Upd4Args make_upd4_args(hb_handle* h, int T) {
  Upd4Args a;
  a.U = h->U.p;
  a.R = h->R.p;
  const size_t R0 = (size_t)h->plan_set * h->plan_rounds;
  a.order = h->order.p + R0 * h->n;
  a.next_at = h->next_at.p + R0 * h->n;
  a.ranges = h->ranges.p + R0 * h->nb * h->coop_grid;
  a.tuple_levels = h->tuple_levels.p;
  a.lvl_ptr = h->lvl_ptr.p;
  a.lvl_tup = h->lvl_tup.p;
  a.lvl_first1 = h->lvl_ptr.p + h->B + 1;
  a.sigma = h->sigma.p;
  a.theta = h->theta.p;
  a.Pr_b = h->Pr_b.p;
  a.ring = h->ring.p;
  a.acc = h->acc2.p;
  a.remT = remT_ptr(h);
  a.remS = h->remS.p;
  a.OEend = h->OEend.p;
  a.obj = h->obj2.p;
  a.bar = h->bar.p;
  a.n = h->n;
  a.K = h->K;
  a.KS = h->KS;
  a.C = h->C;
  a.J = h->J;
  a.B = h->B;
  a.nb = h->nb;
  a.T = T;
  a.s_begin = a.s_end = 0;
  a.write_from = std::min(T - 1, (int)h->window_size + 1);  // rounds after which cluster_cpp may stop (:250-256)
  a.has_next_from = T - 1;
  a.sigma_uniform = h->sigma_uniform ? 1 : 0;
  a.sigma0 = h->sigma0;
  a.ring_rows = h->u5_ring_rows;
  a.dbg_flags = 0;
  a.coop = 1;
  a.dbg = (h->dbg_cta >= 0) ? h->dbg.p : nullptr;
  a.dbg_cta = h->dbg_cta;
  return a;
}
// zero the per-step accumulators of a cluster_cpp call ...
int upd_begin_zero(hb_handle* h, int T) {
  const size_t BK = (size_t)h->B * h->KS, SL = 2 * (BK + h->KS);
  CK(cudaMemsetAsync(h->acc2.p, 0, sizeof(float) * SL * ((size_t)T * h->nb + 2), h->stream));
  CK(cudaMemsetAsync(h->obj2.p, 0, sizeof(double) * 2 * (size_t)T, h->stream));
  CK(cudaMemsetAsync(h->bar.p, 0, sizeof(unsigned) * 2 * ((size_t)T * h->nb + 2), h->stream));
  if (h->use_v4) CK(cudaMemsetAsync(remT_ptr(h), 0, sizeof(float) * 2 * (size_t)h->nb * h->J * h->KS, h->stream));
  if (h->use_xch) h->xch.epoch++;  // flags of earlier calls no longer match
  return 0;
}
// ... and seed ring[1] (= "O_{-1}") with the tables the call starts from
int upd_begin_seed(hb_handle* h) {
  const size_t BK = (size_t)h->B * h->KS;
  CK(cudaMemcpyAsync(h->ring.p + 2 * BK, h->O.p, sizeof(float) * BK, cudaMemcpyDeviceToDevice, h->stream));
  CK(cudaMemcpyAsync(h->ring.p + 3 * BK, h->E.p, sizeof(float) * BK, cudaMemcpyDeviceToDevice, h->stream));
  return 0;
}
int upd_launch(hb_handle* h, UpdArgs a, bool cooperative) {
  const size_t smem = upd_smem_bytes(h);
  return dispatch_nv(h, h->KS, [&](auto nvc) -> int {
    constexpr int NV = decltype(nvc)::value;
    CK(cudaFuncSetAttribute(k_update_steps<NV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    a.use_barrier = cooperative ? 1 : 0;
    if (cooperative) {
      void* args[] = {&a};
      CK(cudaLaunchCooperativeKernel((void*)k_update_steps<NV>, dim3(h->coop_grid), dim3(UPD_THREADS), args, smem, h->stream));
    } else {
      k_update_steps<NV><<<h->coop_grid, UPD_THREADS, smem, h->stream>>>(a);
    }
    CKL();
    return 0;
  });
}
template <int NV, bool SIGU>
int upd5_launch_nv(hb_handle* h, Upd4Args& a, bool cooperative) {
  const size_t smem = upd5_smem_bytes(NV, a.ring_rows, a.KS);
  CK(cudaFuncSetAttribute(k_update_steps5<NV, SIGU>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  a.coop = cooperative ? 1 : 0;
  Upd4Launch lp;
  lp.a = a;
  if (h->use_xch) lp.x = h->xch;
  if (cooperative) {
    void* args[] = {&lp};
    CK(cudaLaunchCooperativeKernel((void*)k_update_steps5<NV, SIGU>, dim3(h->coop_grid), dim3(U5_THREADS), args, smem,
                                   h->stream));
  } else {
    k_update_steps5<NV, SIGU><<<h->coop_grid, U5_THREADS, smem, h->stream>>>(lp);
  }
  CKL();
  return 0;
}
int upd4_launch(hb_handle* h, Upd4Args a, bool cooperative) {
  const bool su = h->sigma_uniform;  // the default: scalar sigma (objective terms simplify)
  switch (upd4_nv(h->KS)) {
    case 1: return su ? upd5_launch_nv<1, true>(h, a, cooperative) : upd5_launch_nv<1, false>(h, a, cooperative);
    case 2: return su ? upd5_launch_nv<2, true>(h, a, cooperative) : upd5_launch_nv<2, false>(h, a, cooperative);
  }
  return fail(h, 2, "K = %d is not supported by the persistent update kernel", h->K);
}
void dump_step_trace(hb_handle* h, int ns, int per_step) {
  std::vector<long long> st((size_t)(ns + 1) * per_step);
  if (cudaMemcpyAsync(st.data(), h->dbg.p, sizeof(long long) * st.size(), cudaMemcpyDeviceToHost, h->stream) != cudaSuccess) return;
  cudaStreamSynchronize(h->stream);
  static int dumped = 0;
  if (dumped++ != 3) return;
  FILE* f = fopen("gpurun_out/step_trace.txt", "w");
  if (!f) return;
  for (int s = 0; s <= ns; ++s) {
    fprintf(f, "%d", s);
    for (int k = 0; k < per_step; ++k) fprintf(f, " %lld", st[(size_t)s * per_step + k]);
    fprintf(f, "\n");
  }
  fclose(f);
}
// compute_objective() of every round in [t0, t1) (harmony.cpp:248) from the kernels' per-round sums and tables
int push_round_objectives(hb_handle* h, int t0, int t1) {
  const size_t BK = (size_t)h->B * h->KS;
  for (int t = t0; t < t1; ++t) {
    const float* O = (t == t1 - 1) ? h->O.p : h->OEend.p + (size_t)t * 2 * BK;
    const float* E = (t == t1 - 1) ? h->E.p : h->OEend.p + (size_t)t * 2 * BK + BK;
    TRY(push_objective_from(h, O, E, h->obj2.p + 2 * (size_t)t));
  }
  return 0;
}
// single-pass kernel (update_kernel4.cuh), rounds [t0, t1)
int run_update_v4(hb_handle* h, int T, int t0, int t1, bool rem_ready) {
  RegionScope rs(h, "update_R");
  const int nb = h->nb;
  const size_t BK = (size_t)h->B * h->KS, XH = BK + h->KS, SL = 2 * XH;
  Upd4Args a = make_upd4_args(h, T);
  if (t0 == 0 && !rem_ready) {
    // removal sums of round 0 from the R in memory (assignment step / user), harmony.cpp:312-313
    RegionScope r0(h, "k_rem_sums");
    k_rem_sums<<<dim3(h->coop_grid, nb), 256, sizeof(float) * 8 * (size_t)h->KS, h->stream>>>(
        h->R.p, a.order, a.ranges, a.tuple_levels, a.acc, 0, h->coop_grid, h->K, h->KS, h->C, h->B);
    CKL();
    if (h->world > 1) TRY(allreduce_f(h, h->acc2.p + SL, SL * (size_t)nb));  // rem halves of slots 1 .. nb (add halves: zero)
  }
  if (h->world <= 1 || h->use_xch) {
    a.s_begin = t0 * nb;
    a.s_end = t1 * nb;
    RegionScope r3(h, "k_update_steps");
    TRY(upd4_launch(h, a, true));
  } else {
    // sharded cells without peer memory: one launch per block step, the step's add half all-reduced in between; the next round's
    // removal sums (remT) are all-reduced and folded once per round
    RegionScope r3(h, "k_update_steps");
    for (int t = t0; t < t1; ++t) {
      if (t > 0) {
        TRY(allreduce_f(h, h->remT.p + (size_t)(t & 1) * nb * h->J * h->KS, (size_t)nb * h->J * h->KS));
        k_fold_round<<<grid_for((int64_t)nb * h->K, 256, h->num_sms), 256, 0, h->stream>>>(a, t);
        CKL();
      }
      for (int s = t * nb; s < (t + 1) * nb; ++s) {
        if (s > t0 * nb) TRY(allreduce_f(h, h->acc2.p + (size_t)(s + 1) * SL, XH));  // add_{s-1}
        a.s_begin = s;
        a.s_end = s + 1;
        TRY(upd4_launch(h, a, false));
      }
    }
    TRY(allreduce_f(h, h->acc2.p + (size_t)(t1 * nb + 1) * SL, XH));  // add_{S-1}
  }
  if (h->dbg_cta >= 0 && h->rank == 0) dump_step_trace(h, (t1 - t0) * nb, 8);
  {
    RegionScope r4(h, "k_update_finalize");
    k_update_finalize4<<<grid_for(BK, 256, 64), 256, 0, h->stream>>>(a, h->use_xch ? h->xch : Upd4Xch{}, t1 * nb, h->O.p, h->E.p);
    CKL();
  }
  return push_round_objectives(h, t0, t1);
}
// first persistent generation (update_kernel.cuh): look-ahead + update warp groups; serves plans whose CTA
// ranges are not tuple-aligned.  rounds [t0, t1): t0 == 0 runs the prologue look-ahead.  write_mask: rounds that store R.
int run_update_v2(hb_handle* h, int T, int t0, int t1, unsigned write_mask) {
  RegionScope rs(h, "update_R");
  const int nb = h->nb;
  const size_t BK = (size_t)h->B * h->KS, SL = 2 * (BK + h->KS);
  UpdArgs a = make_upd_args(h, T);
  a.write_R_mask = write_mask;
  if (h->world <= 1) {
    a.s_begin = t0 * nb;
    a.s_end = t1 * nb;
    a.prologue = (t0 == 0) ? 1 : 0;
    RegionScope r3(h, "k_update_steps");
    TRY(upd_launch(h, a, true));
  } else {
    // sharded cells: one launch per step, the step's slot [add_{s-1} | rem_s] all-reduced in between
    RegionScope r3(h, "k_update_steps");
    if (t0 == 0) {
      a.s_begin = a.s_end = 0;
      a.prologue = 1;
      TRY(upd_launch(h, a, false));
    }
    a.prologue = 0;
    for (int s = t0 * nb; s < t1 * nb; ++s) {
      TRY(allreduce_f(h, h->acc2.p + (size_t)(s + 1) * SL, SL));
      a.s_begin = s;
      a.s_end = s + 1;
      TRY(upd_launch(h, a, false));
    }
    TRY(allreduce_f(h, h->acc2.p + (size_t)(t1 * nb + 1) * SL, SL));  // slot(S): add_{S-1} (+ look-ahead rem_S)
  }
  if (h->dbg_cta >= 0 && h->world <= 1) dump_step_trace(h, (t1 - t0) * nb, 16);
  // tables at the end of round t1-1 -> O, E (the chain itself continues from the ring)
  {
    RegionScope r4(h, "k_update_finalize");
    k_update_finalize<<<grid_for(BK, 256, 64), 256, 0, h->stream>>>(a, t1 * nb, h->O.p, h->E.p);
    CKL();
  }
  return push_round_objectives(h, t0, t1);
}


// S[q][k][:] += R_q^T [Z_q | 1] on the tensor cores (stats_tc3.cuh): one launch per 128 clusters x 64 columns of [Z | 1]
// (K = 100, d = 50: one launch).  The caller zeroes S.
int run_stats_tc(hb_handle* h, const float* Zsrc) {
  const int K = h->K, D1 = h->d + 1;
  StatsTcArgs t;
  t.R = h->R.p;
  t.Zo = Zsrc;
  t.tile_cell0 = h->tile_cell0.p;
  t.tile_len = h->tile_len.p;
  t.tile_tuple = h->tile_tuple.p;
  t.S = h->S.p;
  t.ntiles = h->ntiles;
  t.d = h->d;
  t.K = K;
  t.KS = h->KS;
  t.DS = h->DS;
  t.tiles_per_cta = std::max(1, (h->ntiles + h->num_sms - 1) / h->num_sms);
  const int grid_tc = (h->ntiles + t.tiles_per_cta - 1) / t.tiles_per_cta;
  const size_t smem_tc = stats_tc_smem_bytes(h->KS, h->DS);
  CK(cudaFuncSetAttribute(k_stats_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_tc));
  for (t.k_off = 0; t.k_off < K; t.k_off += 128)
    for (t.c_off = 0; t.c_off < D1; t.c_off += 64) {
      k_stats_tc<<<grid_tc, ST_THREADS, smem_tc, h->stream>>>(t);
      CKL();
    }
  return 0;
}

// ---- moe_correct_ridge_cpp (harmony.cpp:345-638) -------------------------------------------------
int run_correct(hb_handle* h) {
  const int K = h->K, d = h->d, B = h->B, J = h->J, C = h->C;
  const int D1 = d + 1;
  {
    RegionScope rs(h, "ridge_stats");
    CK(cudaMemsetAsync(h->S.p, 0, sizeof(float) * (size_t)J * K * D1, h->stream));
    if (h->use_tc_stats) {
      TRY(run_stats_tc(h, h->Zo.p));
    } else {
    StatsArgs a;
      a.R = h->R.p;
      a.Zo = h->Zo.p;
      a.tile_cell0 = h->tile_cell0.p;
      a.tile_len = h->tile_len.p;
      a.tile_tuple = h->tile_tuple.p;
      a.S = h->S.p;
      a.ntiles = h->ntiles;
      a.d = d;
      a.K = K;
      a.KS = (K <= 128) ? K : 128;
      a.ldR = h->KS;
      a.ldZ = h->DS;
      const int KSP = (a.KS + 7) & ~7, DP = (D1 + 3) & ~3;
      dim3 block(DP / 4, KSP / 8);
      if (block.x * block.y > 1024) return fail(h, 2, "d = %d is too large for the statistics kernel", d);
      a.tiles_per_cta = std::max(1, (h->ntiles + h->num_sms * 4 - 1) / (h->num_sms * 4));
      dim3 grid((h->ntiles + a.tiles_per_cta - 1) / a.tiles_per_cta, (K + a.KS - 1) / a.KS);
      size_t smem = sizeof(float) * (size_t)TM * (KSP + DP);
      CK(cudaFuncSetAttribute(k_ridge_stats, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      k_ridge_stats<<<grid, block, smem, h->stream>>>(a);
      CKL();
    }
    TRY(allreduce_f(h, h->S.p, (size_t)J * K * D1));
  }
  {
    RegionScope rs(h, "ridge_solve");
    SolveArgs a;
    a.S = h->S.p;
    a.O = h->O.p;
    a.E = h->E.p;
    a.N_b = h->N_b.p;
    a.lambda = h->lambda_estimation ? nullptr : h->lambda.p;
    a.tuple_levels = h->tuple_levels.p;
    a.cov_of = h->cov_of_d.p;
    a.Y = h->Y.p;
    a.V = h->V.p;
    a.Wfull = h->Wfull.p;
    a.skipped = h->skipped.p;
    a.scratch = h->scratch.p;
    a.iscratch = h->iscratch.p;
    a.err_flag = h->err_flag.p;
    a.J = J;
    a.K = K;
    a.B = B;
    a.C = C;
    a.d = d;
    a.KS = h->KS;
    a.alpha = h->alpha;
    a.cutoff = h->cutoff;
    k_ridge_solve<<<K, 256, sizeof(int) * (size_t)(B + C), h->stream>>>(a);
    CKL();
  }
  if (h->use_tc_apply) {
    RegionScope rs(h, "ridge_apply");
    ApplyTcArgs a;
    a.R = h->R.p;
    a.Zo = h->Zo.p;
    a.V = h->V.p;
    a.Zc = h->Zc.p;
    a.tile_cell0 = h->tile_cell0.p;
    a.tile_len = h->tile_len.p;
    a.tile_tuple = h->tile_tuple.p;
    a.ntiles = h->ntiles;
    a.d = d;
    a.K = K;
    a.KS = h->KS;
    a.DS = h->DS;
    a.tiles_per_cta = std::max(1, (h->ntiles + h->num_sms - 1) / h->num_sms);
    a.dbg = nullptr;
    static int ap_calls = 0;
    const bool tracing = getenv("HB_TRACE_APPLY") != nullptr && (++ap_calls == 4);
    if (tracing) {
      if (h->dbg.n < 64 * 12) CK(h->dbg.alloc(64 * 12));
      CK(cudaMemsetAsync(h->dbg.p, 0, sizeof(long long) * 64 * 12, h->stream));
      a.dbg = h->dbg.p;
    }
    const int grid = (h->ntiles + a.tiles_per_cta - 1) / a.tiles_per_cta;
    {
      // cluster ranges of at most AP_MAXK clusters (shared memory), equal sizes, multiples of 8: the first launch
      // subtracts its share from Zo, the following ones from the partial result in Zc
      const int npass = (K + AP_MAXK - 1) / AP_MAXK;
      const int Kpass = (((K + npass - 1) / npass) + 7) & ~7;
      for (int k_off = 0; k_off < K; k_off += Kpass) {
        a.k_off = k_off;
        a.Kp = std::min(Kpass, K - k_off);
        a.KD = (a.Kp + 7) & ~7;
        a.minuend = (k_off == 0) ? h->Zo.p : h->Zc.p;
        const size_t smem = apply_tc_smem_bytes(a.KD, d);
        CK(cudaFuncSetAttribute(k_apply_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_apply_tc<<<grid, AP_THREADS, smem, h->stream>>>(a);
        CKL();
        a.dbg = nullptr;
      }
    }
    if (tracing) {
      std::vector<long long> st(32 * 16);
      CK(cudaMemcpyAsync(st.data(), h->dbg.p, sizeof(long long) * st.size(), cudaMemcpyDeviceToHost, h->stream));
      CK(cudaStreamSynchronize(h->stream));
      if (FILE* f = fopen("gpurun_out/apply_trace.txt", "w")) {
        for (int i = 0; i < 32; ++i) {
          fprintf(f, "%d", i);
          for (int k = 0; k < 16; ++k) fprintf(f, " %lld", st[(size_t)i * 16 + k] ? st[(size_t)i * 16 + k] - st[0] : -1);
          fprintf(f, "\n");
        }
        fclose(f);
      }
    }
    return 0;
  }
  {
    RegionScope rs(h, "ridge_apply");
    ApplyArgs a;
    a.R = h->R.p;
    a.Zo = h->Zo.p;
    a.V = h->V.p;
    a.Zc = h->Zc.p;
    a.tile_cell0 = h->tile_cell0.p;
    a.tile_len = h->tile_len.p;
    a.tile_tuple = h->tile_tuple.p;
    a.ntiles = h->ntiles;
    a.d = d;
    a.K = K;
    a.ldR = h->KS;
    a.ldZ = h->DS;
    const int DP = (d + 3) & ~3, KP4 = (K + 3) & ~3;
    dim3 block(DP / 4, TM / 4);
    if (block.x * block.y > 1024) return fail(h, 2, "d = %d is too large for the apply kernel", d);
    size_t smem = sizeof(float) * ((size_t)KP4 * DP + (size_t)TM * KP4);
    if (smem > 227 * 1024) return fail(h, 2, "K*d too large for the apply kernel (needs %zu B shared memory)", smem);
    CK(cudaFuncSetAttribute(k_ridge_apply, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    a.tiles_per_cta = std::max(1, (h->ntiles + h->num_sms * 4 - 1) / (h->num_sms * 4));
    int grid = (h->ntiles + a.tiles_per_cta - 1) / a.tiles_per_cta;
    k_ridge_apply<<<grid, block, smem, h->stream>>>(a);
    CKL();
  }
  return 0;
}

int check_err_flag(hb_handle* h) {
  int flag = 0;
  CK(cudaMemcpyAsync(&flag, h->err_flag.p, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  if (flag) {
    int z = 0;
    cudaMemcpyAsync(h->err_flag.p, &z, sizeof(int), cudaMemcpyHostToDevice, h->stream);
    if (flag == 1) return fail(h, 4, "update order holds an index outside [0, N)");
    if (flag == 2) return fail(h, 5, "inv(): matrix is singular");
    if (flag == 3) return fail(h, 4, "update order is not a permutation of the cells");
    return fail(h, 6, "device error flag %d", flag);
  }
  return 0;
}

// rows of a per-cell field (device row stride ld), un-sorted and widened to double.  Rows are gathered on the device
// as floats (half the PCIe bytes), DMA'd into two pinned staging buffers and widened into the caller's array by the
// host pool while the next chunk is in flight: a device -> host copy of doubles into a freshly allocated pageable
// array runs at the speed of ONE driver thread that also takes the array's page faults (measured: 88 ms for
// 1M x 50 against ~20 ms this way).  The pinned buffers live for the life of the process and are allocated with the
// first handle (hb_create), not inside the first download.
float* g_pinned[2] = {nullptr, nullptr};
constexpr size_t kPinnedFloats = (size_t)8 << 20;  // 32 MiB per buffer
bool ensure_pinned_staging() {
  static std::mutex mk;
  std::lock_guard<std::mutex> lk(mk);
  if (g_pinned[0]) return true;
  for (int i = 0; i < 2; ++i)
    if (cudaHostAlloc((void**)&g_pinned[i], sizeof(float) * kPinnedFloats, cudaHostAllocDefault) != cudaSuccess) {
      cudaGetLastError();
      if (i == 1) cudaFreeHost(g_pinned[0]);
      g_pinned[0] = g_pinned[1] = nullptr;
      return false;  // no pinned memory: the plain path serves
    }
  return true;
}
int download_rows_mt(hb_handle* h, const float* src, int cols, int ld, double* out, bool* done) {
  float** pinned = g_pinned;
  const size_t kFloats = kPinnedFloats;
  *done = false;
  if (!ensure_pinned_staging()) return 0;
  WidenPool* pool = widen_pool();
  const int64_t n = h->n;
  float* dev = reinterpret_cast<float*>(h->stage.p);  // two halves of the device staging buffer
  const size_t dev_half = std::min(kFloats, h->stage.n);  // stage.n doubles = 2 * stage.n floats
  const int64_t rows_per = std::max<int64_t>(1, (int64_t)(dev_half / (size_t)cols));
  const int64_t nchunks = (n + rows_per - 1) / rows_per;
  cudaEvent_t ev[2];
  CK(cudaEventCreateWithFlags(&ev[0], cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&ev[1], cudaEventDisableTiming));
  auto enqueue = [&](int64_t i) -> int {
    const int64_t r0 = i * rows_per, rows = std::min(rows_per, n - r0);
    float* d = dev + (size_t)(i & 1) * dev_half;
    k_download_rows<<<grid_for(rows * cols, 256, h->num_sms * 8), 256, 0, h->stream>>>(src, d, (int64_t)cols, h->inv_sort.p,
                                                                                       r0, rows, cols, ld);
    CKL();
    CK(cudaMemcpyAsync(pinned[i & 1], d, sizeof(float) * (size_t)rows * cols, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaEventRecord(ev[i & 1], h->stream));
    return 0;
  };
  int rc = nchunks > 0 ? enqueue(0) : 0;
  for (int64_t i = 0; i < nchunks && rc == 0; ++i) {
    if (i + 1 < nchunks) rc = enqueue(i + 1);  // its buffers were released by widen(i - 1)
    if (rc) break;
    if (cudaEventSynchronize(ev[i & 1]) != cudaSuccess) {
      rc = fail(h, 10, "CUDA error while downloading rows");
      break;
    }
    const int64_t r0 = i * rows_per, rows = std::min(rows_per, n - r0);
    pool->widen(out + r0 * cols, pinned[i & 1], (size_t)rows * cols);
  }
  cudaStreamSynchronize(h->stream);
  cudaEventDestroy(ev[0]);
  cudaEventDestroy(ev[1]);
  *done = (rc == 0);
  return rc;
}
int download_rows(hb_handle* h, const float* src, int cols, int ld, double* out) {
  {
    bool done = false;
    TRY(download_rows_mt(h, src, cols, ld, out, &done));
    if (done) return 0;
  }
  const int64_t n = h->n;
  const int64_t rows_per = std::max<int64_t>(1, (int64_t)(h->stage.n / (size_t)cols));
  for (int64_t r0 = 0; r0 < n; r0 += rows_per) {
    int64_t rows = std::min(rows_per, n - r0);
    k_download_rows<<<grid_for(rows * cols, 256, h->num_sms * 8), 256, 0, h->stream>>>(src, h->stage.p, (int64_t)cols,
                                                                                        h->inv_sort.p, r0, rows, cols, ld);
    CKL();
    CK(cudaMemcpyAsync(out + r0 * cols, h->stage.p, sizeof(double) * (size_t)rows * cols, cudaMemcpyDeviceToHost,
                       h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  return 0;
}
int upload_rows(hb_handle* h, const double* in, int cols, int ld, float* dst) {
  const int64_t n = h->n;
  const int64_t rows_per = std::max<int64_t>(1, (int64_t)(h->stage.n / (size_t)cols));
  for (int64_t r0 = 0; r0 < n; r0 += rows_per) {
    int64_t rows = std::min(rows_per, n - r0);
    CK(cudaMemcpyAsync(h->stage.p, in + r0 * cols, sizeof(double) * (size_t)rows * cols, cudaMemcpyHostToDevice,
                       h->stream));
    k_upload_rows<<<grid_for(rows * cols, 256, h->num_sms * 8), 256, 0, h->stream>>>(h->stage.p, (int64_t)cols, (int64_t)1,
                                                                                      dst, h->inv_sort.p, r0, rows, cols, ld);
    CKL();
    CK(cudaStreamSynchronize(h->stream));
  }
  return 0;
}
// K x B tables are stored [B][KS]; the boundary wants them dense
int download_table(hb_handle* h, const float* src, double* out) {
  k_compact<<<(h->B * h->K + 255) / 256, 256, 0, h->stream>>>(src, h->tmpT.p, h->B, h->K, h->KS);
  CKL();
  std::vector<float> tmp((size_t)h->B * h->K);
  CK(cudaMemcpyAsync(tmp.data(), h->tmpT.p, sizeof(float) * tmp.size(), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  for (size_t i = 0; i < tmp.size(); ++i) out[i] = (double)tmp[i];
  return 0;
}
int upload_table(hb_handle* h, const double* in, float* dst) {
  std::vector<float> tmp((size_t)h->B * h->K);
  for (size_t i = 0; i < tmp.size(); ++i) tmp[i] = (float)in[i];
  CK(cudaMemcpyAsync(h->tmpT.p, tmp.data(), sizeof(float) * tmp.size(), cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemsetAsync(dst, 0, sizeof(float) * (size_t)h->B * h->KS, h->stream));
  k_expand<<<(h->B * h->K + 255) / 256, 256, 0, h->stream>>>(h->tmpT.p, dst, h->B, h->K, h->KS);
  CKL();
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}
int download_small(hb_handle* h, const float* src, size_t count, double* out) {
  std::vector<float> tmp(count);
  CK(cudaMemcpyAsync(tmp.data(), src, sizeof(float) * count, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  for (size_t i = 0; i < count; ++i) out[i] = (double)tmp[i];
  return 0;
}
int upload_small(hb_handle* h, const double* in, size_t count, float* dst) {
  std::vector<float> tmp(count);
  for (size_t i = 0; i < count; ++i) tmp[i] = (float)in[i];
  CK(cudaMemcpyAsync(dst, tmp.data(), sizeof(float) * count, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

// ---- pieces of hb_setup / hb_setup_device, in the order they run ------------------------------------
// (a) arguments and scalars (harmony.cpp:29-91)
int setup_scalars(hb_handle* h, const void* Z, int d, int64_t N, const void* phi_i, const int32_t* B_vec, int C,
                  const double* sigma, const double* theta, const double* lambda, double alpha, int max_iter_kmeans,
                  double epsilon_kmeans, double epsilon_harmony, int K, double block_size,
                  double batch_proportion_cutoff, int verbose) {
  if (h->ran_setup) return fail(h, 3, "setup was already run on this object");
  if (!Z || !phi_i || !B_vec || !sigma || !theta) return fail(h, 2, "null argument");
  if (d < 1 || N < 1 || C < 1 || K < 1) return fail(h, 2, "bad dimensions");
  if (K > 1024) return fail(h, 2, "K = %d is not supported (K <= 1024)", K);
  if (N > 2000000000LL) return fail(h, 2, "more than 2e9 cells per GPU are not supported");
  CK(cudaSetDevice(h->device));
  h->n = N;
  if (!h->shard_set) {
    if (h->world > 1) return fail(h, 3, "hb_set_shard is required when world_size > 1");
    h->N_global = N;
    h->cell_offset = 0;
  }
  const int64_t NG = h->N_global;
  h->d = d;
  h->C = C;
  h->K = K;
  h->KS = (K + 3) & ~3;
  h->DS = (d + 3) & ~3;
  h->B_vec.assign(B_vec, B_vec + C);
  h->B = std::accumulate(h->B_vec.begin(), h->B_vec.end(), 0);
  const int B = h->B;
  h->cov_of.resize(B);
  {
    int b = 0;
    for (int c = 0; c < C; ++c)
      for (int l = 0; l < B_vec[c]; ++l) h->cov_of[b++] = c;
  }
  // harmony.cpp:83-91
  if (NG < 6) return fail(h, 1, "Refusing to run with less than 6 cells");
  if (NG < 40) {
    h->warnings.push_back("Too few cells. Setting block_size to 0.2");
    h->block_size = 0.2f;
  } else {
    h->block_size = (float)block_size;
  }
  h->epsilon_kmeans = (float)epsilon_kmeans;
  h->epsilon_harmony = (float)epsilon_harmony;
  h->alpha = (float)alpha;
  h->cutoff = (float)batch_proportion_cutoff;
  h->max_iter_kmeans = (unsigned)max_iter_kmeans;
  h->verbose = verbose;
  h->lambda_estimation = (lambda == nullptr) || (lambda[0] == -1);  // harmony.cpp:75
  // update_R block geometry, harmony.cpp:280-281 (float arithmetic on the GLOBAL cell count)
  h->nb = my_ceil(1.0f / h->block_size);
  h->cpb = (uint32_t)((float)NG * h->block_size);
  if (h->cpb == 0) return fail(h, 2, "block_size * N < 1");
  {
    int bits = 1;
    while ((1ull << bits) < (uint64_t)NG) bits++;
    h->half_bits = (bits + 1) / 2;
  }
  return 0;
}

constexpr uint64_t kSmallKeySpace = 1ull << 22;  // the usual case: a direct table beats sorting N keys

// Radices of the joint covariate key (the last covariate varies fastest) and the size of the key space.
int tuple_radix(hb_handle* h, std::vector<uint64_t>& radix, uint64_t* key_space) {
  const int C = h->C;
  long double prod = 1;
  for (int c = 0; c < C; ++c) prod *= (long double)h->B_vec[c];
  if (prod > 9e18L) return fail(h, 2, "covariate level product overflows 64 bits");
  radix.assign(C, 0);
  uint64_t r = 1;
  for (int c = C - 1; c >= 0; --c) {
    radix[c] = r;
    r *= (uint64_t)h->B_vec[c];
  }
  *key_space = r;
  return 0;
}

// h->J and h->tuple_levels_h from the ascending unique keys
int set_tuples(hb_handle* h, const std::vector<uint64_t>& uniq, const std::vector<uint64_t>& radix) {
  if (uniq.size() > 1000000) return fail(h, 2, "more than 1e6 distinct covariate tuples are not supported");
  const int J = (int)uniq.size(), C = h->C;
  h->J = J;
  h->tuple_levels_h.resize((size_t)J * C);
  std::vector<int> base(C, 0);
  for (int c = 1; c < C; ++c) base[c] = base[c - 1] + h->B_vec[c - 1];
  for (int q = 0; q < J; ++q) {
    uint64_t kk = uniq[q];
    for (int c = 0; c < C; ++c) {
      h->tuple_levels_h[(size_t)q * C + c] = base[c] + (int)(kk / radix[c]);
      kk %= radix[c];
    }
  }
  return 0;
}

// (b) on the host: joint covariate tuples, level counts (summed over ranks) and the stable sort of the cells by tuple.
// Sets h->J / h->tuple_levels_h, fills the device sort_perm / inv_sort and returns the first position of every tuple
// (tstart, J + 1 values).
int tuple_dict_host(hb_handle* h, const int32_t* phi_i, std::vector<int64_t>& lvl_count, std::vector<int64_t>& tstart) {
  const int64_t N = h->n;
  const int C = h->C, B = h->B;
  const int* B_vec = h->B_vec.data();
  lvl_count.assign(B, 0);
  std::vector<uint64_t> key(N);
  std::vector<uint64_t> radix;
  uint64_t key_space = 1;
  TRY(tuple_radix(h, radix, &key_space));
  {
    std::vector<int> base(C, 0);
    for (int c = 1; c < C; ++c) base[c] = base[c - 1] + B_vec[c - 1];
    for (int64_t i = 0; i < N; ++i) {
      uint64_t kk = 0;
      for (int c = 0; c < C; ++c) {
        int b = phi_i[i * C + c];
        if (b < base[c] || b >= base[c] + B_vec[c]) return fail(h, 2, "phi row index %d of cell %lld is not a level of covariate %d", b, (long long)i, c);
        lvl_count[b]++;
        kk += (uint64_t)(b - base[c]) * radix[c];
      }
      key[i] = kk;
    }
  }
  std::vector<uint64_t> uniq;
  const bool small_space = key_space <= kSmallKeySpace;
  if (small_space) {
    std::vector<uint8_t> seen((size_t)key_space, 0);
    for (int64_t i = 0; i < N; ++i) seen[key[i]] = 1;
    for (uint64_t k2 = 0; k2 < key_space; ++k2)
      if (seen[k2]) uniq.push_back(k2);
  } else {
    uniq = key;
    std::sort(uniq.begin(), uniq.end());
    uniq.erase(std::unique(uniq.begin(), uniq.end()), uniq.end());
  }
  if (h->world > 1) {
    // global tuple dictionary = union over ranks; level counts summed over ranks
    long long cnt = (long long)uniq.size(), maxcnt = 0;
    DevBuf<long long> dcnt;
    CK(dcnt.alloc(1));
    CK(cudaMemcpyAsync(dcnt.p, &cnt, sizeof(cnt), cudaMemcpyHostToDevice, h->stream));
    CKN(g_nccl.AllReduce(dcnt.p, dcnt.p, 1, ncclInt64, ncclMax, h->comm, h->stream));
    CK(cudaMemcpyAsync(&maxcnt, dcnt.p, sizeof(cnt), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    std::vector<uint64_t> sendbuf((size_t)maxcnt, ~0ull), recvbuf((size_t)maxcnt * h->world);
    std::copy(uniq.begin(), uniq.end(), sendbuf.begin());
    DevBuf<uint64_t> ds, dr;
    CK(ds.alloc((size_t)maxcnt));
    CK(dr.alloc((size_t)maxcnt * h->world));
    CK(cudaMemcpyAsync(ds.p, sendbuf.data(), sizeof(uint64_t) * (size_t)maxcnt, cudaMemcpyHostToDevice, h->stream));
    CKN(g_nccl.AllGather(ds.p, dr.p, (size_t)maxcnt, ncclUint64, h->comm, h->stream));
    CK(cudaMemcpyAsync(recvbuf.data(), dr.p, sizeof(uint64_t) * recvbuf.size(), cudaMemcpyDeviceToHost, h->stream));
    DevBuf<long long> dl;
    CK(dl.alloc(B));
    std::vector<long long> lc(lvl_count.begin(), lvl_count.end());
    CK(cudaMemcpyAsync(dl.p, lc.data(), sizeof(long long) * B, cudaMemcpyHostToDevice, h->stream));
    CKN(g_nccl.AllReduce(dl.p, dl.p, B, ncclInt64, ncclSum, h->comm, h->stream));
    CK(cudaMemcpyAsync(lc.data(), dl.p, sizeof(long long) * B, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (int b = 0; b < B; ++b) lvl_count[b] = lc[b];
    uniq.assign(recvbuf.begin(), recvbuf.end());
    std::sort(uniq.begin(), uniq.end());
    uniq.erase(std::unique(uniq.begin(), uniq.end()), uniq.end());
    if (!uniq.empty() && uniq.back() == ~0ull) uniq.pop_back();
  }
  TRY(set_tuples(h, uniq, radix));
  const int J = h->J;
  std::vector<int> tuple_of(N);
  tstart.assign(J + 1, 0);
  {
    std::vector<int> lut;
    if (small_space) {
      lut.assign((size_t)key_space, -1);
      for (int q = 0; q < J; ++q) lut[uniq[q]] = q;
    }
    for (int64_t i = 0; i < N; ++i) {
      int q = small_space ? lut[key[i]] : (int)(std::lower_bound(uniq.begin(), uniq.end(), key[i]) - uniq.begin());
      tuple_of[i] = q;
      tstart[q + 1]++;
    }
  }
  for (int q = 0; q < J; ++q) tstart[q + 1] += tstart[q];
  std::vector<int> sort_perm(N), inv_sort(N);
  {
    std::vector<int64_t> cur(tstart.begin(), tstart.end() - 1);
    for (int64_t i = 0; i < N; ++i) {
      int64_t s = cur[tuple_of[i]]++;
      sort_perm[s] = (int)i;
      inv_sort[i] = (int)s;
    }
  }
  CK(h->sort_perm.alloc(N));
  CK(h->inv_sort.alloc(N));
  CK(cudaMemcpyAsync(h->sort_perm.p, sort_perm.data(), sizeof(int) * N, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(h->inv_sort.p, inv_sort.data(), sizeof(int) * N, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

// (b) on the device: phi_i is device memory of the handle's device, ordered on h->stream.  Same results as
// tuple_dict_host (setup_device.cuh); the only host traffic is J + 1 tuple starts and the J unique keys.  A key space
// above kSmallKeySpace, or more tuples than the counting sort's per-warp shared-memory counters hold, downloads phi_i
// and runs tuple_dict_host: one implementation serves those rare shapes.
int tuple_dict_device(hb_handle* h, const int32_t* phi_i, std::vector<int64_t>& lvl_count, std::vector<int64_t>& tstart) {
  const int64_t N = h->n;
  const int C = h->C, B = h->B;
  std::vector<uint64_t> radix;
  uint64_t key_space = 1;
  TRY(tuple_radix(h, radix, &key_space));
  auto on_host = [&]() -> int {
    std::vector<int32_t> phi((size_t)N * C);
    CK(cudaMemcpyAsync(phi.data(), phi_i, sizeof(int32_t) * phi.size(), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return tuple_dict_host(h, phi.data(), lvl_count, tstart);
  };
  if (key_space > kSmallKeySpace) return on_host();
  const int KSP = (int)key_space;
  std::vector<int> lv_h(3 * (size_t)C);
  for (int c = 0, base = 0; c < C; base += h->B_vec[c], ++c) {
    lv_h[3 * c] = base;
    lv_h[3 * c + 1] = h->B_vec[c];
    lv_h[3 * c + 2] = (int)radix[c];
  }
  // ids: presence of every key, then (exclusive scan) its tuple id; int rather than a byte per key because the scan
  // kernels work on ints.  The trailing word becomes J.
  DevBuf<int> lv, key, ids;
  DevBuf<unsigned long long> bad;
  CK(lv.alloc(lv_h.size()));
  CK(key.alloc(N));
  CK(ids.alloc((size_t)KSP + 1));
  CK(bad.alloc(1));
  CK(cudaMemcpyAsync(lv.p, lv_h.data(), sizeof(int) * lv_h.size(), cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemsetAsync(ids.p, 0, sizeof(int) * ((size_t)KSP + 1), h->stream));
  CK(cudaMemsetAsync(bad.p, 0xff, sizeof(unsigned long long), h->stream));
  k_dict_keys<<<grid_for(N, 256, h->num_sms * 8), 256, 0, h->stream>>>(phi_i, N, C, lv.p, key.p, ids.p, bad.p);
  CKL();
  unsigned long long first_bad = 0;
  CK(cudaMemcpyAsync(&first_bad, bad.p, sizeof(first_bad), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  if (first_bad != ~0ull) {  // the host path's report of the same cell
    int b = 0;
    CK(cudaMemcpy(&b, phi_i + first_bad, sizeof(int), cudaMemcpyDeviceToHost));
    return fail(h, 2, "phi row index %d of cell %lld is not a level of covariate %d", b, (long long)(first_bad / C),
                (int)(first_bad % C));
  }
  // global tuple dictionary = union over ranks
  if (h->world > 1) CKN(g_nccl.AllReduce(ids.p, ids.p, (size_t)KSP, ncclInt32, ncclMax, h->comm, h->stream));
  DevBuf<unsigned long long> scan_state;
  auto scan = [&](int* data, int64_t n) -> int {
    const int tiles = (int)((n + SCAN_TILE - 1) / SCAN_TILE);
    CK(scan_state.alloc((size_t)tiles + 1));
    CK(cudaMemsetAsync(scan_state.p, 0, sizeof(unsigned long long) * ((size_t)tiles + 1), h->stream));
    k_scan_chained<<<dim3(tiles, 1), 1024, 0, h->stream>>>(data, n, scan_state.p, tiles);
    CKL();
    return 0;
  };
  TRY(scan(ids.p, (int64_t)KSP + 1));
  int J = 0;
  CK(cudaMemcpyAsync(&J, ids.p + KSP, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  // stable counting sort by tuple id: one warp per chunk of consecutive cells, J counters per warp in shared memory
  const size_t per_warp = sizeof(int) * (size_t)J, smem_max = (size_t)227 * 1024 - 256;
  if (J > 1000000 || per_warp > smem_max) return on_host();
  const int wpb = (int)std::max<size_t>(1, std::min<size_t>(8, (48 * 1024) / per_warp));
  const size_t sm = per_warp * wpb;
  if (sm > 48 * 1024) {
    CK(cudaFuncSetAttribute(k_plan_hist, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    CK(cudaFuncSetAttribute(k_plan_scatter, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  }
  int CH = 1024;  // histogram of at most 2^24 counters (64 MB)
  while (CH < N && ((N + CH - 1) / CH) * (int64_t)J > (1 << 24)) CH <<= 1;
  const int nc = (int)((N + CH - 1) / CH);
  DevBuf<int> uniq_d, cstart, cq0, cnq, H, tst, flag;
  CK(uniq_d.alloc(J));
  CK(cstart.alloc((size_t)nc + 1));
  CK(cq0.alloc(nc));
  CK(cnq.alloc(nc));
  CK(H.alloc((size_t)J * nc));
  CK(tst.alloc((size_t)J + 1));
  CK(flag.alloc(1));
  CK(h->sort_perm.alloc(N));
  CK(h->inv_sort.alloc(N));
  k_dict_tuples<<<grid_for(std::max<int64_t>(KSP, N), 256, h->num_sms * 8), 256, 0, h->stream>>>(ids.p, KSP, uniq_d.p,
                                                                                                 key.p, N);
  CKL();
  k_dict_chunks<<<grid_for((int64_t)nc + 1, 256, 64), 256, 0, h->stream>>>(nc, CH, N, cstart.p, cq0.p, cnq.p);
  CKL();
  k_plan_hist<<<(nc + wpb - 1) / wpb, wpb * 32, sm, h->stream>>>(key.p, nullptr, cstart.p, cq0.p, cnq.p, nc, J, 1, H.p,
                                                                  flag.p, N, 0);
  CKL();
  TRY(scan(H.p, (int64_t)J * nc));
  k_plan_scatter<<<(nc + wpb - 1) / wpb, wpb * 32, sm, h->stream>>>(key.p, nullptr, cstart.p, cq0.p, cnq.p, nc, J, 1, H.p,
                                                                     h->sort_perm.p, nullptr, nullptr, nullptr, N, 0, 0);
  CKL();
  k_dict_finish<<<grid_for(std::max<int64_t>(N, (int64_t)J + 1), 256, h->num_sms * 8), 256, 0, h->stream>>>(
      h->sort_perm.p, h->inv_sort.p, N, H.p, nc, J, tst.p);
  CKL();
  std::vector<int> uniq_h(J), tst_h((size_t)J + 1);
  CK(cudaMemcpyAsync(uniq_h.data(), uniq_d.p, sizeof(int) * (size_t)J, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(tst_h.data(), tst.p, sizeof(int) * ((size_t)J + 1), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  TRY(set_tuples(h, std::vector<uint64_t>(uniq_h.begin(), uniq_h.end()), radix));
  tstart.assign(tst_h.begin(), tst_h.end());
  // level counts: every level's tuples' cell counts, summed (integers, so the same numbers the host loop counts)
  lvl_count.assign(B, 0);
  for (int q = 0; q < J; ++q)
    for (int c = 0; c < C; ++c) lvl_count[h->tuple_levels_h[(size_t)q * C + c]] += tstart[q + 1] - tstart[q];
  if (h->world > 1) {
    DevBuf<long long> dl;
    CK(dl.alloc(B));
    std::vector<long long> lc(lvl_count.begin(), lvl_count.end());
    CK(cudaMemcpyAsync(dl.p, lc.data(), sizeof(long long) * B, cudaMemcpyHostToDevice, h->stream));
    CKN(g_nccl.AllReduce(dl.p, dl.p, B, ncclInt64, ncclSum, h->comm, h->stream));
    CK(cudaMemcpyAsync(lc.data(), dl.p, sizeof(long long) * B, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    lvl_count.assign(lc.begin(), lc.end());
  }
  return 0;
}

// (c) everything that follows from the tuple dictionary: tile and chunk tables, allocations, small uploads and the
// CSR level -> tuple table
int setup_tables(hb_handle* h, HostLap& lap, const std::vector<int64_t>& tstart, const std::vector<int64_t>& lvl_count,
                 const double* sigma, const double* theta, const double* lambda) {
  const int64_t N = h->n, NG = h->N_global;
  const int J = h->J, B = h->B, C = h->C, K = h->K, d = h->d;
  // static tiles (<= TM cells of one tuple) and plan chunks (<= CHUNK cells of one tuple)
  int CHUNK = 1024;  // plan chunks: ~2000 per shard at most (the plan's scan is nb^2 x #chunks long)
  while (CHUNK < 16384 && N / CHUNK > 2048) CHUNK <<= 1;
  std::vector<int> t_cell0, t_len, t_tuple, c_start, t_chunk0(J, 0), c_q0, c_nq;
  for (int q = 0; q < J; ++q) {
    for (int64_t s = tstart[q]; s < tstart[q + 1]; s += TM) {
      t_cell0.push_back((int)s);
      t_len.push_back((int)std::min<int64_t>(TM, tstart[q + 1] - s));
      t_tuple.push_back(q);
    }
    t_chunk0[q] = (int)c_start.size();
    for (int64_t s = tstart[q]; s < tstart[q + 1]; s += CHUNK) c_start.push_back((int)s);
    const int nq = (int)c_start.size() - t_chunk0[q];
    for (int i = 0; i < nq; ++i) {
      c_q0.push_back(t_chunk0[q]);
      c_nq.push_back(nq);
    }
  }
  std::vector<int> tc0, tcl, tct;  // 128-cell tiles for the tensor-core kernels
  for (int q = 0; q < J; ++q)
    for (int64_t s2 = tstart[q]; s2 < tstart[q + 1]; s2 += TC_TM) {
      tc0.push_back((int)s2);
      tcl.push_back((int)std::min<int64_t>(TC_TM, tstart[q + 1] - s2));
      tct.push_back(q);
    }
  h->tc_ntiles = (int)tc0.size();
  c_q0.push_back((int)c_start.size());  // the trailing empty chunk is a group of its own
  c_nq.push_back(1);
  c_start.push_back((int)N);  // start of the trailing empty chunk
  c_start.push_back((int)N);  // and its end
  h->ntiles = (int)t_cell0.size();
  h->nchunks = (int)c_start.size() - 1;
  // tuples without local cells point at the first later chunk (their segments are empty)
  for (int q = J - 1; q >= 0; --q)
    if (tstart[q + 1] == tstart[q]) t_chunk0[q] = (q + 1 < J) ? t_chunk0[q + 1] : h->nchunks - 1;

  // ---- device allocations
  const int KS = h->KS, DS = h->DS;
  const size_t nK = (size_t)N * KS, nd = (size_t)N * DS, BK = (size_t)B * KS;
  const int Tplan = std::max(1, (int)h->max_iter_kmeans);
  // update_R kernels: the single-pass persistent kernel when every CTA's slice of a block can lie inside one
  // covariate tuple (2 J <= #SMs) and its ring fits shared memory; else the first persistent generation (K <= 256,
  // <= 8192 tuples, checked against the shared-memory limit); else one launch triple per block step.
  const size_t smem_limit = (size_t)227 * 1024 - 256;
  const bool force_v1 = (h->kernel_set & HB_KS_UPDATE_PER_STEP) != 0, force_v2 = (h->kernel_set & HB_KS_UPDATE_TWO_PASS) != 0;
  h->coop_grid = h->num_sms;  // one persistent CTA per SM
  h->aligned_ranges = (2 * J <= h->coop_grid);
  h->u5_ring_rows = upd5_ring_rows(KS, smem_limit);
  h->use_v4 = !force_v1 && !force_v2 && h->aligned_ranges && h->u5_ring_rows > 0 && (uint64_t)N * (uint64_t)KS < (1ull << 32);
  h->use_v2 = h->use_v4 || (!force_v1 && (KS <= 256) && (J <= 8192) && upd_smem_bytes(h) <= smem_limit);
  h->plan_nsub = (h->use_v4 && h->nb <= 64) ? h->nb : 1;
  h->plan_rounds = Tplan;
  CK(h->Zo.alloc(nd));
  CK(h->Zc.alloc(nd));
  CK(h->U.alloc(nK));
  CK(h->R.alloc(nK));
  CK(h->Y.alloc((size_t)K * d));
  CK(h->sigma.alloc(K));
  CK(h->theta.alloc(B));
  CK(h->Pr_b.alloc(B));
  CK(h->N_b.alloc(B));
  CK(h->lambda.alloc(B + 1));
  CK(h->O.alloc(BK));
  CK(h->E.alloc(BK));
  CK(h->P.alloc(BK));
  CK(h->tmpT.alloc((size_t)B * K));
  CK(h->Oacc.alloc(BK + KS));
  CK(h->acc.alloc(4 * (BK + KS)));
  CK(h->S.alloc((size_t)J * K * (d + 1)));
  CK(h->V.alloc((size_t)J * K * d));
  CK(h->Wfull.alloc((size_t)K * (B + 1) * d));
  CK(h->scratch.alloc((size_t)K * (2 * (size_t)(B + 1) * (B + 1) + (size_t)(B + 1) * d)));
  CK(h->iscratch.alloc((size_t)K * (2 * (size_t)B + J)));
  CK(h->skipped.alloc(K));
  CK(h->err_flag.alloc(1));
  CK(h->obj_acc.alloc(2));
  CK(h->stage.alloc((size_t)8 << 20));  // 64 MiB of doubles
  CK(h->tuple_levels.alloc((size_t)J * C));
  CK(h->cov_of_d.alloc(B));
  CK(h->tile_cell0.alloc(h->ntiles));
  CK(h->tile_len.alloc(h->ntiles));
  CK(h->tile_tuple.alloc(h->ntiles));
  CK(h->tc_cell0.alloc(h->tc_ntiles));
  CK(h->tc_len.alloc(h->tc_ntiles));
  CK(h->tc_tuple.alloc(h->tc_ntiles));
  h->use_tc_apply = (d <= 128) && !(h->kernel_set & HB_KS_FFMA_CONTRACTIONS);   // cluster ranges of <= AP_MAXK per launch
  h->use_tc_stats = !(h->kernel_set & HB_KS_FFMA_CONTRACTIONS);                  // 128 clusters x 64 columns per launch
  h->assign_ns = assign3_smem_bytes(2, (d + 7) & ~7, (K + 15) & ~15, KS) <= smem_limit ? 2 : 1;
  h->use_tc_assign = (d <= 64) && (K <= 128) && assign3_smem_bytes(h->assign_ns, (d + 7) & ~7, (K + 15) & ~15, KS) <= smem_limit &&
                     !(h->kernel_set & HB_KS_FFMA_CONTRACTIONS);
  h->use_tc_logits = !h->use_tc_assign && (d <= 128) && logits_smem_bytes((d + 7) & ~7) <= smem_limit &&
                     !(h->kernel_set & HB_KS_FFMA_CONTRACTIONS);
  h->pt_cap = (size_t)N / TC_TM + (size_t)h->nb * J + 2;
  if (h->use_tc_assign && h->use_v4) {
    CK(h->pt_p0.alloc(2 * h->pt_cap));
    CK(h->pt_len.alloc(2 * h->pt_cap));
    CK(h->pt_tuple.alloc(2 * h->pt_cap));
    CK(h->pt_blk.alloc(2 * h->pt_cap));
    CK(h->pt_count.alloc(2));
    CK(h->pt_base.alloc((size_t)h->nb * J + 2));
  }
  CK(h->chunk_start.alloc(h->nchunks + 1));
  CK(h->tuple_chunk0.alloc(J));
  CK(h->blk_of.alloc(2 * (size_t)Tplan * N));
  CK(h->order.alloc(2 * (size_t)Tplan * N));
  if (h->use_v4)
    CK(h->next_at.alloc(2 * (size_t)Tplan * N));
  else
    CK(h->prev_at.alloc(2 * (size_t)Tplan * N));
  {  // histogram scratch of the plan's counting sort: as many rounds per launch as fit 64 MB (at most 8)
    const size_t per_round = (size_t)h->nb * h->plan_nsub * h->nchunks;
    h->plan_batch = (int)std::max<size_t>(1, std::min<size_t>({(size_t)8, (size_t)Tplan, ((size_t)16 << 20) / std::max<size_t>(1, per_round)}));
    CK(h->H.alloc(per_round * h->plan_batch));
    CK(h->scan_state.alloc((size_t)h->plan_batch * ((per_round + SCAN_TILE - 1) / SCAN_TILE + 1)));
  }
  CK(h->chunk_q0.alloc(h->nchunks));
  CK(h->chunk_nq.alloc(h->nchunks));
  CK(h->seg_start.alloc(2 * (size_t)Tplan * ((size_t)h->nb * J + 1)));
  CK(h->tile_base.alloc(2 * (size_t)Tplan * ((size_t)h->nb * J + 1)));
  if (h->use_v2) {
    CK(h->ring.alloc(4 * BK));
    CK(h->acc2.alloc(2 * (BK + KS) * ((size_t)Tplan * h->nb + 2)));
    CK(h->Psave.alloc(h->use_v4 ? 1 : 2 * (size_t)h->nb * BK));
    if (h->use_v4) CK(h->remT.alloc(2 * (size_t)h->nb * J * KS));
    if (h->use_v4 && h->world > 1) CK(h->remS.alloc((size_t)h->nb * J * KS));
    CK(h->OEend.alloc((size_t)Tplan * 2 * BK));
    CK(h->obj2.alloc(2 * (size_t)Tplan));
    CK(h->bar.alloc(2 * ((size_t)Tplan * h->nb + 2)));
    if (h->aligned_ranges) CK(h->ranges.alloc(2 * (size_t)Tplan * h->nb * h->coop_grid));
    release_peer_exchange(h);
    if (h->use_v4 && h->world > 1 && h->world <= U4_MAXWORLD && !(h->kernel_set & HB_KS_NO_PEER_EXCHANGE))
      TRY(setup_peer_exchange(h, Tplan));
    if (const char* e = getenv("HB_TRACE_STEPS")) {
      h->dbg_cta = atoi(e);
      CK(h->dbg.alloc((size_t)(32 * h->nb + 2) * 16));
      CK(cudaMemsetAsync(h->dbg.p, 0, sizeof(long long) * (size_t)(32 * h->nb + 2) * 16, h->stream));
    }
    CK(cudaMemsetAsync(h->Psave.p, 0, sizeof(float) * h->Psave.n, h->stream));
    CK(cudaMemsetAsync(h->ring.p, 0, sizeof(float) * 4 * BK, h->stream));
  }
  lap.mark("device allocations");
  CK(cudaMemsetAsync(h->err_flag.p, 0, sizeof(int), h->stream));
  CK(cudaMemsetAsync(h->obj_acc.p, 0, 2 * sizeof(double), h->stream));
  CK(cudaMemsetAsync(h->O.p, 0, sizeof(float) * BK, h->stream));
  CK(cudaMemsetAsync(h->E.p, 0, sizeof(float) * BK, h->stream));
  CK(cudaMemsetAsync(h->Wfull.p, 0, sizeof(float) * (size_t)K * (B + 1) * d, h->stream));
  CK(cudaMemsetAsync(h->skipped.p, 0, sizeof(int) * K, h->stream));
  CK(cudaMemsetAsync(h->R.p, 0, sizeof(float) * nK, h->stream));
  CK(cudaMemsetAsync(h->Zo.p, 0, sizeof(float) * nd, h->stream));
  CK(cudaMemsetAsync(h->Zc.p, 0, sizeof(float) * nd, h->stream));
  k_fill_f<<<grid_for((int64_t)nK, 256, h->num_sms * 8), 256, 0, h->stream>>>(h->U.p, (int64_t)nK, U_PAD);
  CKL();
  CK(cudaMemsetAsync(h->Y.p, 0, sizeof(float) * (size_t)K * d, h->stream));
#define UP(buf, vec) CK(cudaMemcpyAsync(h->buf.p, (vec).data(), sizeof((vec)[0]) * (vec).size(), cudaMemcpyHostToDevice, h->stream))
  UP(tuple_levels, h->tuple_levels_h);
  // CSR level -> tuples containing it, ascending tuple order; trailing word: the number of levels of covariate 0
  std::vector<int> lvl_ptr_h(B + 2, 0), lvl_tup_h((size_t)J * C);
  {
    for (size_t i = 0; i < h->tuple_levels_h.size(); ++i) lvl_ptr_h[h->tuple_levels_h[i] + 1]++;
    for (int b = 0; b < B; ++b) lvl_ptr_h[b + 1] += lvl_ptr_h[b];
    std::vector<int> fill(lvl_ptr_h.begin(), lvl_ptr_h.begin() + B);
    for (int q = 0; q < J; ++q)
      for (int c = 0; c < C; ++c) lvl_tup_h[fill[h->tuple_levels_h[(size_t)q * C + c]]++] = q;
    lvl_ptr_h[B + 1] = h->B_vec[0];
    CK(h->lvl_ptr.alloc(B + 2));
    CK(h->lvl_tup.alloc(std::max<size_t>(1, lvl_tup_h.size())));
    UP(lvl_ptr, lvl_ptr_h);
    UP(lvl_tup, lvl_tup_h);
  }
  UP(cov_of_d, h->cov_of);
  UP(tile_cell0, t_cell0);
  UP(tile_len, t_len);
  UP(tile_tuple, t_tuple);
  UP(tc_cell0, tc0);
  UP(tc_len, tcl);
  UP(tc_tuple, tct);
  UP(chunk_start, c_start);
  UP(chunk_q0, c_q0);
  UP(chunk_nq, c_nq);
  UP(tuple_chunk0, t_chunk0);
  {
    std::vector<float> f(K);
    for (int k = 0; k < K; ++k) f[k] = (float)sigma[k];
    h->sigma0 = f[0];
    h->sigma_uniform = true;
    for (int k = 1; k < K; ++k) h->sigma_uniform = h->sigma_uniform && (f[k] == f[0]);
    UP(sigma, f);
    f.resize(B);
    for (int b = 0; b < B; ++b) f[b] = (float)theta[b];
    UP(theta, f);
    std::vector<float> nbv(B), prb(B);
    for (int b = 0; b < B; ++b) {
      nbv[b] = (float)lvl_count[b];
      prb[b] = (float)lvl_count[b] / (float)NG;  // harmony.cpp:67
    }
    UP(N_b, nbv);
    UP(Pr_b, prb);
    std::vector<float> lam(B + 1, 0.f);
    if (!h->lambda_estimation)
      for (int b = 0; b <= B; ++b) lam[b] = (float)lambda[b];
    UP(lambda, lam);
    CK(cudaStreamSynchronize(h->stream));
  }
#undef UP
  lap.mark("memsets + small uploads");
  return 0;
}

// The pointer is device (or managed) memory of the handle's device.
int check_device_ptr(hb_handle* h, const void* p, const char* what) {
  cudaPointerAttributes a;
  if (!p) return fail(h, 2, "null argument");
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return fail(h, 2, "%s is not CUDA device memory", what);
  }
  if (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) return fail(h, 2, "%s is not CUDA device memory", what);
  if (a.device != h->device) return fail(h, 2, "%s is on CUDA device %d, the handle on device %d", what, a.device, h->device);
  return 0;
}

}  // namespace

// =================================================================================================
extern "C" {

int hb_version(void) { return 100; }

int hb_create(hb_handle** out, int device) {
  if (!out) return 1;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return 10;  // no CUDA device: there is no CPU path
  hb_handle* h = new hb_handle();
  if (device < 0) cudaGetDevice(&device);
  h->device = device;
  if (cudaSetDevice(device) != cudaSuccess) {
    delete h;
    return 10;
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) h->num_sms = prop.multiProcessorCount;
  cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
  cudaStreamCreateWithFlags(&h->plan_stream, cudaStreamNonBlocking);
  cudaEventCreateWithFlags(&h->plan_done, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&h->ev0, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&h->io_ev, cudaEventDisableTiming);
  ensure_pinned_staging();  // process-wide; the first handle pays for it, not the first download
  keep_pool_memory(device);
  widen_pool();
  *out = h;
  return 0;
}

void hb_destroy(hb_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->plan_stream) cudaStreamSynchronize(h->plan_stream);
  if (h->stream) cudaStreamSynchronize(h->stream);
  if (h->plan_done) cudaEventDestroy(h->plan_done);
  if (h->plan_stream) cudaStreamDestroy(h->plan_stream);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->io_ev) cudaEventDestroy(h->io_ev);
  release_peer_exchange(h);
  cudaStream_t s = h->stream;
  delete h;  // frees device buffers
  if (s) cudaStreamDestroy(s);
}

const char* hb_last_error(const hb_handle* h) { return h ? h->err.c_str() : "null handle"; }

int hb_pop_warning(hb_handle* h, char* buf, size_t cap) {
  if (!h || h->warnings.empty()) return 0;
  if (buf && cap) {
    strncpy(buf, h->warnings.front().c_str(), cap - 1);
    buf[cap - 1] = 0;
  }
  h->warnings.pop_front();
  return 1;
}

int hb_comm_unique_id(char id[HB_COMM_ID_BYTES]) {
  static_assert(sizeof(ncclUniqueId) <= HB_COMM_ID_BYTES, "id size");
  std::string why;
  if (!load_nccl(&why)) return 11;
  ncclUniqueId uid;
  if (g_nccl.GetUniqueId(&uid) != ncclSuccess) return 11;
  memset(id, 0, HB_COMM_ID_BYTES);
  memcpy(id, &uid, sizeof(uid));
  return 0;
}

int hb_comm_init(hb_handle* h, int rank, int world_size, const char id[HB_COMM_ID_BYTES]) {
  if (!h) return 1;
  if (h->ran_setup) return fail(h, 3, "hb_comm_init must precede hb_setup");
  if (world_size < 1 || rank < 0 || rank >= world_size) return fail(h, 2, "bad rank/world_size");
  h->rank = rank;
  h->world = world_size;
  if (world_size == 1) return 0;
  std::string why;
  if (!load_nccl(&why)) return fail(h, 11, "%s", why.c_str());
  CK(cudaSetDevice(h->device));
  const CommKey key{h->device, rank, world_size};
  if (!id) {  // reuse the process-wide communicator created by an earlier handle
    auto it = g_comms.find(key);
    if (it == g_comms.end()) return fail(h, 3, "hb_comm_init(NULL id): no communicator has been created yet for this rank/world");
    h->comm = it->second;
    return 0;
  }
  ncclUniqueId uid;
  memcpy(&uid, id, sizeof(uid));
  CKN(g_nccl.CommInitRank(&h->comm, world_size, uid, rank));
  g_comms[key] = h->comm;  // kept until process exit
  return 0;
}

int hb_set_shard(hb_handle* h, int64_t N_global, int64_t cell_offset) {
  if (!h) return 1;
  if (h->ran_setup) return fail(h, 3, "hb_set_shard must precede hb_setup");
  h->N_global = N_global;
  h->cell_offset = cell_offset;
  h->shard_set = true;
  return 0;
}

int hb_set_seed(hb_handle* h, uint64_t seed) {
  if (!h) return 1;
  if (h->plan_stream) cudaStreamSynchronize(h->plan_stream);
  h->next_ready = false;
  h->seed = seed;
  h->round_counter = 0;
  return 0;
}

int hb_set_abort_callback(hb_handle* h, int (*cb)(void*), void* user) {
  if (!h) return 1;
  h->abort_cb = cb;
  h->abort_user = user;
  return 0;
}

int hb_setup(hb_handle* h, const double* Z, int d, int64_t N, const int32_t* phi_i, const int32_t* B_vec, int C,
             const double* sigma, const double* theta, const double* lambda, double alpha, int max_iter_kmeans,
             double epsilon_kmeans, double epsilon_harmony, int K, double block_size,
             double batch_proportion_cutoff, int verbose) {
  TRY(setup_scalars(h, Z, d, N, phi_i, B_vec, C, sigma, theta, lambda, alpha, max_iter_kmeans, epsilon_kmeans,
                    epsilon_harmony, K, block_size, batch_proportion_cutoff, verbose));
  HostLap lap(h->stream, "hb_setup");
  std::vector<int64_t> lvl_count, tstart;
  TRY(tuple_dict_host(h, phi_i, lvl_count, tstart));
  lap.mark("tuple dictionary / sort (host)");
  TRY(setup_tables(h, lap, tstart, lvl_count, sigma, theta, lambda));
  // Z: double -> float, into tuple-sorted order (harmony.cpp:41); Z_corr = normalise(Z_orig) (:42)
  TRY(upload_rows(h, Z, d, h->DS, h->Zo.p));
  k_normalise_rows<<<grid_for(N * 32, 256, h->num_sms * 8), 256, 0, h->stream>>>(h->Zo.p, h->Zc.p, N, d, h->DS);
  CKL();
  CK(cudaStreamSynchronize(h->stream));
  lap.mark("Z upload + normalise");
  h->ran_setup = true;
  return 0;
}

int hb_setup_device(hb_handle* h, const void* Z, int z_dtype, int64_t z_cell_stride, int64_t z_pc_stride, int d,
                    int64_t N, const int32_t* phi_i, const int32_t* B_vec, int C, const double* sigma,
                    const double* theta, const double* lambda, double alpha, int max_iter_kmeans,
                    double epsilon_kmeans, double epsilon_harmony, int K, double block_size,
                    double batch_proportion_cutoff, int verbose, void* stream) {
  TRY(setup_scalars(h, Z, d, N, phi_i, B_vec, C, sigma, theta, lambda, alpha, max_iter_kmeans, epsilon_kmeans,
                    epsilon_harmony, K, block_size, batch_proportion_cutoff, verbose));
  if (z_dtype != HB_F32 && z_dtype != HB_F64) return fail(h, 2, "Z dtype %d is not supported (HB_F32 or HB_F64)", z_dtype);
  if (z_cell_stride < 0 || z_pc_stride < 0) return fail(h, 2, "negative Z strides are not supported");
  TRY(check_device_ptr(h, Z, "Z"));
  TRY(check_device_ptr(h, phi_i, "phi_i"));
  HostLap lap(h->stream, "hb_setup_device");
  // Z and phi_i are ready on the caller's stream: this handle's stream waits for it
  CK(cudaEventRecord(h->io_ev, (cudaStream_t)stream));
  CK(cudaStreamWaitEvent(h->stream, h->io_ev, 0));
  std::vector<int64_t> lvl_count, tstart;
  TRY(tuple_dict_device(h, phi_i, lvl_count, tstart));
  lap.mark("tuple dictionary / sort (device)");
  TRY(setup_tables(h, lap, tstart, lvl_count, sigma, theta, lambda));
  // the host path's conversion and scatter, read straight from the caller's layout
  const int grid = grid_for(N * d, 256, h->num_sms * 8);
  if (z_dtype == HB_F32)
    k_upload_rows<<<grid, 256, 0, h->stream>>>(static_cast<const float*>(Z), z_cell_stride, z_pc_stride, h->Zo.p,
                                               h->inv_sort.p, 0, N, d, h->DS);
  else
    k_upload_rows<<<grid, 256, 0, h->stream>>>(static_cast<const double*>(Z), z_cell_stride, z_pc_stride, h->Zo.p,
                                               h->inv_sort.p, 0, N, d, h->DS);
  CKL();
  k_normalise_rows<<<grid_for(N * 32, 256, h->num_sms * 8), 256, 0, h->stream>>>(h->Zo.p, h->Zc.p, N, d, h->DS);
  CKL();
  CK(cudaStreamSynchronize(h->stream));  // the inputs are consumed: the caller may free them
  lap.mark("Z ingest + normalise");
  h->ran_setup = true;
  return 0;
}

int hb_init_cluster(hb_handle* h, const double* Y0) {
  if (!h) return 1;
  if (!h->ran_setup) return fail(h, 3, "setup has not been run");
  CK(cudaSetDevice(h->device));
  HostLap lap(h->stream, "hb_init_cluster");
  if (Y0) {
    // Y = normalise(kmeans_centers(..)) (harmony.cpp:133-136), centroids injected by the caller
    TRY(upload_small(h, Y0, (size_t)h->K * h->d, h->Y.p));
  } else {
    // native kmeans_centers (utils.cpp:10-64) on the cosine-normalised cells, sharded like everything else:
    // initialize_centroids' rule (K start cells, then per centroid the winner of an exponential race weighted by the
    // distance from its start cell, already-taken cells skipped) with keyed-hash uniforms, then 10 Lloyd iterations
    // (10 x arma::kmeans(.., keep_existing, 1): Euclidean assignment, means of the members).
    const int K = h->K, d = h->d;
    const size_t Kd = (size_t)K * d;
    if (h->N_global >= (1ll << 32)) return fail(h, 2, "native k-means initialisation supports < 2^32 cells; pass Y0");
    DevBuf<float> ysum;
    CK(ysum.alloc(Kd + K));
    const uint64_t seed = hb_mix64(h->seed ^ 0x6b6d65616e73ull);
    DevBuf<int64_t> cells_d;
    DevBuf<unsigned long long> best_d;
    CK(cells_d.alloc(K));
    CK(best_d.alloc(K));
    std::vector<int64_t> cells(K);
    auto gather = [&](int only) -> int {  // Y rows <- cells (all, or one centroid), summed over the ranks that own them
      CK(cudaMemcpyAsync(cells_d.p, cells.data(), sizeof(int64_t) * K, cudaMemcpyHostToDevice, h->stream));
      float* dst = (only >= 0) ? h->Y.p + (size_t)only * d : h->Y.p;
      const size_t cnt = (only >= 0) ? (size_t)d : Kd;
      CK(cudaMemsetAsync(dst, 0, sizeof(float) * cnt, h->stream));
      k_kmeans_gather<<<K, 64, 0, h->stream>>>(h->Zc.p, h->inv_sort.p, h->Y.p, cells_d.p, K, d, h->DS, h->cell_offset, h->n, only);
      CKL();
      return allreduce_f(h, dst, cnt);
    };
    // (1) start cells: floor(u (N - 1))  (utils.cpp:12-16)
    for (int k = 0; k < K; ++k)
      cells[k] = (int64_t)std::floor((double)kmeans_uniform(seed, (uint64_t)K, (uint64_t)k) * (double)(h->N_global - 1));
    TRY(gather(-1));
    // (2) the races of all centroids in one pass over the cells (a centroid's race only looks at its own start cell)
    // both steps run from tensor-core logits U = 2 (z . y - 1) (k_logits_tc, sigma = 1) when that kernel takes the
    // shape; else from the FFMA kernels (thread per cell)
    const bool tc_init = (d <= 128) && logits_smem_bytes((d + 7) & ~7) <= (size_t)227 * 1024 - 256 && h->KS <= 256 &&
                         !(h->kernel_set & HB_KS_FFMA_CONTRACTIONS);
    DevBuf<float> ones, yy;
    if (tc_init) {
      CK(ones.alloc(K));
      CK(yy.alloc(K));
      k_fill_f<<<1, 256, 0, h->stream>>>(ones.p, (int64_t)K, 1.0f);
      CKL();
    }
    const size_t smem_pp = sizeof(float) * Kd;
    if (!tc_init) {
      if (smem_pp > 200 * 1024) return fail(h, 2, "K*d too large for the native k-means initialisation; pass Y0");
      CK(cudaFuncSetAttribute(k_kmeans_race, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_pp));
    }
    std::vector<unsigned long long> best(K);
    bool logits_of_start = false;  // U holds the logits of the start cells
    auto race = [&](int i0, int i1, const std::vector<int64_t>& taken) -> int {
      DevBuf<int64_t> taken_d;
      if (!taken.empty()) {
        CK(taken_d.alloc(taken.size()));
        CK(cudaMemcpyAsync(taken_d.p, taken.data(), sizeof(int64_t) * taken.size(), cudaMemcpyHostToDevice, h->stream));
      }
      CK(cudaMemsetAsync(best_d.p + i0, 0xff, sizeof(unsigned long long) * (i1 - i0), h->stream));
      if (tc_init) {
        if (!logits_of_start) {
          TRY(launch_logits(h, ones.p, false));
          logits_of_start = true;
        }
        const int grid_r = grid_for(h->n * 32, 256, h->num_sms * 8);
        if (upd4_nv(h->KS) == 1)
          k_kmeans_race_u<1><<<grid_r, 256, 0, h->stream>>>(h->U.p, h->sort_perm.p, best_d.p, taken.empty() ? nullptr : taken_d.p,
                                                          (int)taken.size(), h->n, K, h->KS, h->cell_offset, seed, i0, i1);
        else
          k_kmeans_race_u<2><<<grid_r, 256, 0, h->stream>>>(h->U.p, h->sort_perm.p, best_d.p, taken.empty() ? nullptr : taken_d.p,
                                                          (int)taken.size(), h->n, K, h->KS, h->cell_offset, seed, i0, i1);
        CKL();
      } else {
        k_kmeans_race<<<grid_for(h->n, 128, h->num_sms * 4), 128, sizeof(float) * (size_t)(i1 - i0) * d, h->stream>>>(
            h->Zc.p, h->sort_perm.p, h->Y.p, best_d.p, taken.empty() ? nullptr : taken_d.p, (int)taken.size(), h->n, K, d, h->DS,
            h->cell_offset, seed, i0, i1);
        CKL();
      }
      if (h->world > 1) CKN(g_nccl.AllReduce(best_d.p + i0, best_d.p + i0, (size_t)(i1 - i0), ncclUint64, ncclMin, h->comm, h->stream));
      CK(cudaMemcpyAsync(best.data() + i0, best_d.p + i0, sizeof(unsigned long long) * (i1 - i0), cudaMemcpyDeviceToHost, h->stream));
      CK(cudaStreamSynchronize(h->stream));
      return 0;
    };
    TRY(race(0, K, {}));
    // (3) accept in centroid order; a winner that is already taken re-runs that centroid's race without the taken cells
    // (utils.cpp:38-45); the race of centroid i reads its START cell, so Y is only rewritten afterwards
    std::vector<int64_t> taken;
    for (int i = 0; i < K; ++i) {
      int64_t w = (int64_t)(best[i] & 0xffffffffull);
      if (best[i] == ~0ull) return fail(h, 3, "native k-means initialisation: no free cell for centroid %d", i);
      if (std::find(taken.begin(), taken.end(), w) != taken.end()) {
        TRY(race(i, i + 1, taken));
        if (best[i] == ~0ull) return fail(h, 3, "native k-means initialisation: no free cell for centroid %d", i);
        w = (int64_t)(best[i] & 0xffffffffull);
      }
      taken.push_back(w);
      cells[i] = w;
    }
    h->kmeans_cells = cells;
    TRY(gather(-1));
    const size_t smem = sizeof(float) * Kd;
    if (!tc_init) CK(cudaFuncSetAttribute(k_kmeans_assign, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    for (int iter = 0; iter < 10; ++iter) {
      if (tc_init) {
        // Lloyd iteration on the tensor cores: logits -> one-hot rows of R -> members' sums and counts (K3) -> means
        TRY(launch_logits(h, ones.p, false));
        k_kmeans_norms<<<(K + 127) / 128, 128, 0, h->stream>>>(h->Y.p, yy.p, K, d);
        CKL();
        const int grid_p = grid_for(h->n * 32, 256, h->num_sms * 8);
        if (upd4_nv(h->KS) == 1)
          k_kmeans_pick<1><<<grid_p, 256, 0, h->stream>>>(h->U.p, yy.p, h->R.p, h->n, K, h->KS);
        else
          k_kmeans_pick<2><<<grid_p, 256, 0, h->stream>>>(h->U.p, yy.p, h->R.p, h->n, K, h->KS);
        CKL();
        CK(cudaMemsetAsync(h->S.p, 0, sizeof(float) * (size_t)h->J * K * (d + 1), h->stream));
        TRY(run_stats_tc(h, h->Zc.p));
        TRY(allreduce_f(h, h->S.p, (size_t)h->J * K * (d + 1)));
        k_kmeans_means_from_stats<<<(int)((Kd + 255) / 256), 256, 0, h->stream>>>(h->S.p, h->Y.p, h->J, K, d);
        CKL();
        continue;
      }
      CK(cudaMemsetAsync(ysum.p, 0, sizeof(float) * (Kd + K), h->stream));
      k_kmeans_assign<<<grid_for(h->n, 128, h->num_sms * 4), 128, smem, h->stream>>>(h->Zc.p, h->Y.p, ysum.p, ysum.p + Kd,
                                                                                       h->n, K, d, h->DS);
      CKL();
      TRY(allreduce_f(h, ysum.p, Kd + K));
      k_kmeans_update<<<(int)((Kd + 255) / 256), 256, 0, h->stream>>>(h->Y.p, ysum.p, ysum.p + Kd, K, d);
      CKL();
    }
    CK(cudaStreamSynchronize(h->stream));
  }
  // Y = arma::normalise(Y, 2, 0)  (harmony.cpp:136)
  lap.mark("centroids (Y0 / native k-means)");
  k_normalise_rows<<<grid_for((int64_t)h->K * 32, 256, 64), 256, 0, h->stream>>>(h->Y.p, h->Y.p, h->K, h->d, h->d);
  CKL();
  CK(cudaMemsetAsync(h->obj_acc.p, 0, 2 * sizeof(double), h->stream));
  TRY(run_assign(h, false, false, true));
  TRY(push_objective(h));                       // compute_objective() (:152)
  lap.mark("assignment + objective");
  h->harmony_slots.push_back(h->obj_count - 1);  // objective_harmony.push_back (:153)
  h->ran_init = true;
  return 0;
}

// STEP 1 of harmony::cluster_cpp as it ran before 2.0.4 (harmony.cpp:235-238):
//   Y = arma::normalise(Z_corr * R.t(), 2, 0);   dist_mat = 2 * (1 - Y.t() * Z_corr);
// built from the kernels of the ridge statistics (R^T [Z_corr | 1] per tuple) and of the assignment.  The
// assignment kernels also rewrite R, O, E and the objective sums, which this step must leave alone: they are
// saved and restored around the call (compatibility path, not a fast one).
int legacy_centroid_step(hb_handle* h) {
  const int K = h->K, d = h->d, B = h->B, J = h->J, KS = h->KS;
  const int D1 = d + 1;
  const size_t nK = (size_t)h->n * KS, BK = (size_t)B * KS;
  CK(cudaMemsetAsync(h->S.p, 0, sizeof(float) * (size_t)J * K * D1, h->stream));
  if (h->use_tc_stats) {
    TRY(run_stats_tc(h, h->Zc.p));  // the statistics of the corrected, normalised embedding
  } else {
    StatsArgs a;
    a.R = h->R.p;
    a.Zo = h->Zc.p;
    a.tile_cell0 = h->tile_cell0.p;
    a.tile_len = h->tile_len.p;
    a.tile_tuple = h->tile_tuple.p;
    a.S = h->S.p;
    a.ntiles = h->ntiles;
    a.d = d;
    a.K = K;
    a.KS = (K <= 128) ? K : 128;
    a.ldR = KS;
    a.ldZ = h->DS;
    const int KSP = (a.KS + 7) & ~7, DP = (D1 + 3) & ~3;
    dim3 block(DP / 4, KSP / 8);
    if (block.x * block.y > 1024) return fail(h, 2, "d = %d is too large for the statistics kernel", d);
    a.tiles_per_cta = std::max(1, (h->ntiles + h->num_sms * 4 - 1) / (h->num_sms * 4));
    dim3 grid((h->ntiles + a.tiles_per_cta - 1) / a.tiles_per_cta, (K + a.KS - 1) / a.KS);
    size_t smem = sizeof(float) * (size_t)TM * (KSP + DP);
    CK(cudaFuncSetAttribute(k_ridge_stats, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_ridge_stats<<<grid, block, smem, h->stream>>>(a);
    CKL();
  }
  TRY(allreduce_f(h, h->S.p, (size_t)J * K * D1));
  k_centroids_from_stats<<<K, 64, sizeof(float) * (size_t)d, h->stream>>>(h->S.p, h->Y.p, J, K, d);
  CKL();
  // distances to the new centroids -> U; everything else the assignment writes is put back
  if (h->Rkeep.n < nK) CK(h->Rkeep.alloc(nK));
  if (h->OEkeep.n < 2 * BK) CK(h->OEkeep.alloc(2 * BK));
  if (h->objkeep.n < 2) CK(h->objkeep.alloc(2));
  CK(cudaMemcpyAsync(h->Rkeep.p, h->R.p, sizeof(float) * nK, cudaMemcpyDeviceToDevice, h->stream));
  CK(cudaMemcpyAsync(h->OEkeep.p, h->O.p, sizeof(float) * BK, cudaMemcpyDeviceToDevice, h->stream));
  CK(cudaMemcpyAsync(h->OEkeep.p + BK, h->E.p, sizeof(float) * BK, cudaMemcpyDeviceToDevice, h->stream));
  CK(cudaMemcpyAsync(h->objkeep.p, h->obj_acc.p, 2 * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  TRY(run_assign(h, false));
  CK(cudaMemcpyAsync(h->R.p, h->Rkeep.p, sizeof(float) * nK, cudaMemcpyDeviceToDevice, h->stream));
  CK(cudaMemcpyAsync(h->O.p, h->OEkeep.p, sizeof(float) * BK, cudaMemcpyDeviceToDevice, h->stream));
  CK(cudaMemcpyAsync(h->E.p, h->OEkeep.p + BK, sizeof(float) * BK, cudaMemcpyDeviceToDevice, h->stream));
  CK(cudaMemcpyAsync(h->obj_acc.p, h->objkeep.p, 2 * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  return 0;
}

int ensure_plan_rounds(hb_handle* h, int T) {
  if (T <= h->plan_rounds) return 0;
  if (h->plan_stream) CK(cudaStreamSynchronize(h->plan_stream));
  CK(cudaStreamSynchronize(h->stream));
  h->next_ready = false;
  h->plan_set = 0;
  const size_t BK = (size_t)h->B * h->KS;
  const size_t S1 = (size_t)h->nb * h->J + 1;
  CK(h->blk_of.alloc(2 * (size_t)T * h->n));
  CK(h->order.alloc(2 * (size_t)T * h->n));
  if (h->use_v4)
    CK(h->next_at.alloc(2 * (size_t)T * h->n));
  else
    CK(h->prev_at.alloc(2 * (size_t)T * h->n));
  CK(h->seg_start.alloc(2 * (size_t)T * S1));
  CK(h->tile_base.alloc(2 * (size_t)T * S1));
  if (h->use_v2) {
    CK(h->acc2.alloc(2 * (BK + h->KS) * ((size_t)T * h->nb + 2)));
    CK(h->OEend.alloc((size_t)T * 2 * BK));
    CK(h->obj2.alloc(2 * (size_t)T));
    CK(h->bar.alloc(2 * ((size_t)T * h->nb + 2)));
    if (h->aligned_ranges) CK(h->ranges.alloc(2 * (size_t)T * h->nb * h->coop_grid));
    if (h->use_xch) TRY(setup_peer_exchange(h, T));  // collective: every rank grows its plan in the same call
  }
  h->plan_rounds = T;
  return 0;
}

int hb_cluster(hb_handle* h, const int64_t* update_orders) {
  if (!h) return 1;
  if (!h->ran_init) return fail(h, 3, "init_cluster_cpp has not been run");
  CK(cudaSetDevice(h->device));
  const unsigned T = h->max_iter_kmeans;
  const bool cold = h->harmony_slots.size() != 1;  // harmony.cpp:214-228 cold start
  TRY(ensure_plan_rounds(h, (int)std::max(1u, T)));
  // the first persistent generation keeps its R-store rounds in a 32-bit mask: longer calls run the per-round path
  const bool persistent = h->use_v2 && !h->legacy_centroid && (h->use_v4 || T <= 31);
  // The single-pass update kernel takes round 0's removal sums from the assignment step itself when that step
  // runs in plan order (tensor-core kernel); every other combination runs the assignment in natural order first.
  const bool plan_assign = cold && persistent && h->use_v4 && (h->use_tc_assign || h->use_tc_logits) && T > 0;
  if (cold && !plan_assign) {
    TRY(run_assign(h, true, false, false));  // the cold start does not evaluate the objective
    CK(cudaMemsetAsync(h->obj_acc.p, 0, 2 * sizeof(double), h->stream));
  }
  if (update_orders && T > 0) {
    size_t cnt = (size_t)T * (size_t)h->N_global;
    if (h->perms_d.n < cnt) CK(h->perms_d.alloc(cnt));
    CK(cudaMemcpyAsync(h->perms_d.p, update_orders, sizeof(int64_t) * cnt, cudaMemcpyHostToDevice, h->stream));
  }
  if (h->abort_cb && h->abort_cb(h->abort_user)) return -1;  // Progress::check_abort (:233)
  unsigned iter = 0;
  if (h->legacy_centroid) {
    // compatibility path: centroid step + one first-generation update_R per round
    if (h->next_ready) {  // a plan prebuilt by an earlier call on the side stream is not used here
      CK(cudaStreamWaitEvent(h->stream, h->plan_done, 0));
      h->round_counter -= (uint64_t)h->next_T;
      h->next_ready = false;
    }
    for (iter = 0; iter < T; iter++) {
      if (iter > 0 && h->abort_cb && h->abort_cb(h->abort_user)) return -1;
      TRY(legacy_centroid_step(h));  // :235-238
      TRY(build_plan_single(h, update_orders ? h->perms_d.p + (size_t)iter * (size_t)h->N_global : nullptr, h->stream));
      TRY(run_update_R_v1(h, 0));  // :241
      TRY(push_objective(h));      // :248
      if (iter > h->window_size) {  // :250-256
        int conv = 0;
        TRY(check_convergence_host(h, 0, &conv));
        if (conv) {
          iter++;
          break;
        }
      }
    }
  } else if (persistent) {
    // all T update orders are drawn up front (they do not depend on the data), then the rounds run in
    // chunks: [0, window_size + 2) in one launch, afterwards one round per launch (convergence checks)
    // The native orders of a call depend only on (seed, round counter), so the plan of the NEXT call is
    // prebuilt on a side stream while this call's correction / the next assignment run (two buffer sets).
    if (h->next_ready) {
      CK(cudaStreamWaitEvent(h->stream, h->plan_done, 0));  // also serialises the use of the scan scratch
      if (!update_orders && h->next_T >= (int)T) {
        h->plan_set ^= 1;  // adopt the prebuilt plan
      } else {
        h->round_counter -= (uint64_t)h->next_T;  // discard it: its rounds were never run
        TRY(build_plans(h, (int)T, update_orders ? h->perms_d.p : nullptr, h->plan_set, h->stream));
      }
      h->next_ready = false;
    } else {
      TRY(build_plans(h, (int)T, update_orders ? h->perms_d.p : nullptr, h->plan_set, h->stream));
    }
    if (T > 0) TRY(upd_begin_zero(h, (int)T));
    if (plan_assign) {
      TRY(run_assign(h, true, true, false));
      CK(cudaMemsetAsync(h->obj_acc.p, 0, 2 * sizeof(double), h->stream));
    }
    if (T > 0) TRY(upd_begin_seed(h));
    unsigned t0 = 0;
    while (t0 < T) {
      unsigned t1 = (t0 == 0) ? std::min(T, h->window_size + 2) : t0 + 1;
      unsigned mask = 0;
      for (unsigned t = t0; t < t1; ++t)
        if (t < 32 && (t == T - 1 || t > h->window_size)) mask |= 1u << t;  // rounds after which cluster_cpp may stop
      if (t0 > 0 && h->abort_cb && h->abort_cb(h->abort_user)) return -1;
      if (h->use_v4)
        TRY(run_update_v4(h, (int)T, (int)t0, (int)t1, plan_assign));
      else
        TRY(run_update_v2(h, (int)T, (int)t0, (int)t1, mask));
      iter = t1;
      if (t1 - 1 > h->window_size) {  // :250-256
        int conv = 0;
        TRY(check_convergence_host(h, 0, &conv));
        if (conv) break;
      }
      t0 = t1;
    }
  } else {
    if (h->next_ready) {  // a plan prebuilt by an earlier call on the side stream is not used here
      CK(cudaStreamWaitEvent(h->stream, h->plan_done, 0));
      h->round_counter -= (uint64_t)h->next_T;
      h->next_ready = false;
    }
    for (iter = 0; iter < T; iter++) {
      if (iter > 0 && h->abort_cb && h->abort_cb(h->abort_user)) return -1;
      TRY(build_plan_single(h, update_orders ? h->perms_d.p + (size_t)iter * (size_t)h->N_global : nullptr, h->stream));
      TRY(run_update_R_v1(h, 0));  // :241
      TRY(push_objective(h));      // :248
      if (iter > h->window_size) {  // :250-256
        int conv = 0;
        TRY(check_convergence_host(h, 0, &conv));
        if (conv) {
          iter++;
          break;
        }
      }
    }
  }
  if (persistent && !update_orders && T > 0 && !h->timing && !(h->kernel_set & HB_KS_NO_PLAN_OVERLAP)) {
    // prebuild the next call's plan into the other buffer set on the side stream; it starts once this
    // call's own (main-stream) plan build and update kernel are done with the shared scan scratch
    CK(cudaEventRecord(h->ev0, h->stream));
    CK(cudaStreamWaitEvent(h->plan_stream, h->ev0, 0));
    TRY(build_plans(h, (int)T, nullptr, h->plan_set ^ 1, h->plan_stream));
    CK(cudaEventRecord(h->plan_done, h->plan_stream));
    h->next_ready = true;
    h->next_T = (int)T;
  }
  if (T > 0) h->R_user_set = false;
  if (update_orders) TRY(check_err_flag(h));
  h->kmeans_rounds.push_back((int)iter);         // :259
  h->harmony_slots.push_back(h->obj_count - 1);  // :260
  return 0;
}

int hb_moe_correct_ridge(hb_handle* h) {
  if (!h) return 1;
  if (!h->ran_init) return fail(h, 3, "init_cluster_cpp has not been run");
  CK(cudaSetDevice(h->device));
  TRY(run_correct(h));
  h->zc_pending_norm = false;  // Z_corr was rebuilt from Z_orig
  if (h->C > 1) TRY(check_err_flag(h));
  return 0;
}

int hb_check_convergence(hb_handle* h, int type) {
  if (!h) return -1;
  int out = 1;
  int st = check_convergence_host(h, type, &out);
  if (st != 0) return -st;
  return out;
}

int hb_compute_objective(hb_handle* h) {
  if (!h) return 1;
  if (!h->ran_init) return fail(h, 3, "init_cluster_cpp has not been run");
  CK(cudaSetDevice(h->device));
  CK(cudaMemsetAsync(h->obj_acc.p, 0, 2 * sizeof(double), h->stream));
  k_objective_cells<<<grid_for(h->n * 32, ROW_THREADS, h->num_sms * 8), ROW_THREADS, 0, h->stream>>>(
      h->R.p, h->U.p, h->sigma.p, h->n, h->K, h->KS, h->obj_acc.p);
  CKL();
  return push_objective(h);
}

int64_t hb_field_size(const hb_handle* h, int field) {
  if (!h || !h->ran_setup) return 0;
  switch (field) {
    case HB_Z_CORR:
    case HB_Z_ORIG: return (int64_t)h->n * h->d;
    case HB_R: return (int64_t)h->n * h->K;
    case HB_Y: return (int64_t)h->K * h->d;
    case HB_O:
    case HB_E: return (int64_t)h->K * h->B;
    case HB_W: return (int64_t)(h->B + 1) * h->d;
    case HB_PR_B:
    case HB_THETA: return h->B;
    case HB_SIGMA: return h->K;
    case HB_LAMBDA: return (int64_t)h->K * (h->B + 1);
    case HB_LAMBDA_VEC: return h->B + 1;
  }
  return 0;
}

int hb_get_field(hb_handle* h, int field, double* out) {
  if (!h) return 1;
  if (!h->ran_setup) return fail(h, 3, "setup has not been run");
  if (!out) return fail(h, 2, "null output");
  CK(cudaSetDevice(h->device));
  const int K = h->K, B = h->B, d = h->d;
  switch (field) {
    case HB_Z_CORR: {
      HostLap lap(h->stream, "hb_get_field");
      if (h->zc_pending_norm) {  // cluster_cpp leaves Z_corr cosine-normalised (harmony.cpp:220); done on first demand
        k_normalise_rows<<<grid_for((int64_t)h->n * 32, 256, h->num_sms * 8), 256, 0, h->stream>>>(h->Zc.p, h->Zc.p, h->n, d, h->DS);
        CKL();
        h->zc_pending_norm = false;
      }
      const int rc = download_rows(h, h->Zc.p, d, h->DS, out);
      lap.mark("Z_corr download");
      return rc;
    }
    case HB_Z_ORIG: return download_rows(h, h->Zo.p, d, h->DS, out);
    case HB_R: return download_rows(h, h->R.p, K, h->KS, out);
    case HB_Y: return download_small(h, h->Y.p, (size_t)K * d, out);
    case HB_O: return download_table(h, h->O.p, out);
    case HB_E: return download_table(h, h->E.p, out);
    case HB_PR_B: return download_small(h, h->Pr_b.p, B, out);
    case HB_THETA: return download_small(h, h->theta.p, B, out);
    case HB_SIGMA: return download_small(h, h->sigma.p, K, out);
    case HB_LAMBDA_VEC: return download_small(h, h->lambda.p, B + 1, out);
    case HB_LAMBDA: {  // getLambda, harmony.cpp:657-669: K x (B+1) column-major
      std::vector<double> E((size_t)K * B), lam(B + 1);
      TRY(download_table(h, h->E.p, E.data()));
      TRY(download_small(h, h->lambda.p, B + 1, lam.data()));
      for (int k = 0; k < K; ++k) {
        out[k] = h->lambda_estimation ? 0.0 : lam[0];
        for (int b = 0; b < B; ++b)
          out[(size_t)(b + 1) * K + k] =
              h->lambda_estimation ? (double)((float)E[(size_t)b * K + k] * h->alpha) : lam[b + 1];
      }
      return 0;
    }
    case HB_W: {  // (B+1) x d column-major; betas of the last cluster that was corrected
      std::vector<int> sk(K);
      CK(cudaMemcpyAsync(sk.data(), h->skipped.p, sizeof(int) * K, cudaMemcpyDeviceToHost, h->stream));
      CK(cudaStreamSynchronize(h->stream));
      int last = -1;
      for (int k = 0; k < K; ++k)
        if (!sk[k]) last = k;
      std::vector<double> w((size_t)(B + 1) * d, 0.0);
      if (last >= 0) TRY(download_small(h, h->Wfull.p + (size_t)last * (B + 1) * d, (size_t)(B + 1) * d, w.data()));
      for (int b = 0; b <= B; ++b)
        for (int c = 0; c < d; ++c) out[(size_t)c * (B + 1) + b] = w[(size_t)b * d + c];
      return 0;
    }
  }
  return fail(h, 2, "unknown field %d", field);
}

int hb_get_field_device(hb_handle* h, int field, void* out, int dtype, int64_t ld, void* stream) {
  if (!h) return 1;
  if (!h->ran_setup) return fail(h, 3, "setup has not been run");
  if (dtype != HB_F32 && dtype != HB_F64) return fail(h, 2, "output dtype %d is not supported (HB_F32 or HB_F64)", dtype);
  const float* src = nullptr;
  int cols = 0, sld = 0;
  switch (field) {
    case HB_Z_CORR: src = h->Zc.p, cols = h->d, sld = h->DS; break;
    case HB_Z_ORIG: src = h->Zo.p, cols = h->d, sld = h->DS; break;
    case HB_R: src = h->R.p, cols = h->K, sld = h->KS; break;
    default: return fail(h, 2, "field %d is not a per-cell field", field);
  }
  if (ld < cols) return fail(h, 2, "row stride %lld is shorter than a row (%d values)", (long long)ld, cols);
  TRY(check_device_ptr(h, out, "out"));
  CK(cudaSetDevice(h->device));
  CK(cudaEventRecord(h->io_ev, (cudaStream_t)stream));  // the caller's earlier use of `out` ...
  CK(cudaStreamWaitEvent(h->stream, h->io_ev, 0));      // ... precedes the write
  if (field == HB_Z_CORR && h->zc_pending_norm) {  // as hb_get_field
    k_normalise_rows<<<grid_for((int64_t)h->n * 32, 256, h->num_sms * 8), 256, 0, h->stream>>>(h->Zc.p, h->Zc.p, h->n, h->d, h->DS);
    CKL();
    h->zc_pending_norm = false;
  }
  const int grid = grid_for(h->n * cols, 256, h->num_sms * 8);
  if (dtype == HB_F32)
    k_download_rows<<<grid, 256, 0, h->stream>>>(src, static_cast<float*>(out), ld, h->inv_sort.p, 0, h->n, cols, sld);
  else
    k_download_rows<<<grid, 256, 0, h->stream>>>(src, static_cast<double*>(out), ld, h->inv_sort.p, 0, h->n, cols, sld);
  CKL();
  CK(cudaEventRecord(h->io_ev, h->stream));  // the caller's stream reads `out` after the write
  CK(cudaStreamWaitEvent((cudaStream_t)stream, h->io_ev, 0));
  return 0;
}

int hb_debug_sort_perm(const hb_handle* h, int32_t* out) {
  if (!h || !out || !h->ran_setup) return 1;
  if (cudaSetDevice(h->device) != cudaSuccess || cudaStreamSynchronize(h->stream) != cudaSuccess ||
      cudaMemcpy(out, h->sort_perm.p, sizeof(int32_t) * (size_t)h->n, cudaMemcpyDeviceToHost) != cudaSuccess)
    return 10;
  return 0;
}

int hb_set_field(hb_handle* h, int field, const double* in) {
  if (!h) return 1;
  if (!h->ran_setup) return fail(h, 3, "setup has not been run");
  if (!in) return fail(h, 2, "null input");
  CK(cudaSetDevice(h->device));
  const int K = h->K, B = h->B, d = h->d;
  switch (field) {
    case HB_Z_CORR:
      h->zc_pending_norm = false;
      return upload_rows(h, in, d, h->DS, h->Zc.p);
    case HB_R:
      h->R_user_set = true;
      return upload_rows(h, in, K, h->KS, h->R.p);
    case HB_Y: return upload_small(h, in, (size_t)K * d, h->Y.p);
    case HB_O: return upload_table(h, in, h->O.p);
    case HB_E: return upload_table(h, in, h->E.p);
    case HB_THETA: return upload_small(h, in, B, h->theta.p);
    case HB_SIGMA:
      h->sigma0 = (float)in[0];
      h->sigma_uniform = true;
      for (int k = 1; k < K; ++k) h->sigma_uniform = h->sigma_uniform && ((float)in[k] == (float)in[0]);
      return upload_small(h, in, K, h->sigma.p);
    case HB_LAMBDA_VEC:
      h->lambda_estimation = false;
      return upload_small(h, in, B + 1, h->lambda.p);
  }
  return fail(h, 2, "field %d is not writable", field);
}

int hb_get_scalar(const hb_handle* h, int which, double* out) {
  if (!h || !out) return 1;
  switch (which) {
    case HB_N: *out = (double)h->N_global; return 0;
    case HB_N_LOCAL: *out = (double)h->n; return 0;
    case HB_B: *out = h->B; return 0;
    case HB_K: *out = h->K; return 0;
    case HB_D: *out = h->d; return 0;
    case HB_C: *out = h->C; return 0;
    case HB_ALPHA: *out = h->alpha; return 0;
    case HB_MAX_ITER_KMEANS: *out = h->max_iter_kmeans; return 0;
    case HB_BLOCK_SIZE: *out = h->block_size; return 0;
    case HB_EPSILON_KMEANS: *out = h->epsilon_kmeans; return 0;
    case HB_EPSILON_HARMONY: *out = h->epsilon_harmony; return 0;
    case HB_LAMBDA_ESTIMATION: *out = h->lambda_estimation ? 1 : 0; return 0;
    case HB_WINDOW_SIZE: *out = h->window_size; return 0;
    case HB_LEGACY_CENTROID_STEP: *out = h->legacy_centroid ? 1 : 0; return 0;
    case HB_KERNEL_SET: *out = h->kernel_set; return 0;
    case HB_DEVICE: *out = h->device; return 0;
  }
  return 2;
}

int hb_set_scalar(hb_handle* h, int which, double value) {
  if (!h) return 1;
  switch (which) {
    case HB_ALPHA: h->alpha = (float)value; return 0;
    case HB_MAX_ITER_KMEANS:
      if (value < 0) return fail(h, 2, "max_iter_kmeans must be >= 0");
      h->max_iter_kmeans = (unsigned)value;
      return 0;
    case HB_EPSILON_KMEANS: h->epsilon_kmeans = (float)value; return 0;
    case HB_EPSILON_HARMONY: h->epsilon_harmony = (float)value; return 0;
    case HB_LEGACY_CENTROID_STEP: h->legacy_centroid = value != 0.0; return 0;
    case HB_KERNEL_SET: h->kernel_set = (int)value; return 0;  // takes effect at the next hb_setup
  }
  return fail(h, 2, "scalar %d is not writable", which);
}

int hb_get_B_vec(const hb_handle* h, int32_t* out) {
  if (!h || !out) return 1;
  for (int c = 0; c < h->C; ++c) out[c] = h->B_vec[c];
  return 0;
}

int64_t hb_trace(const hb_handle* hc, int trace, double* out, int64_t cap) {
  hb_handle* h = const_cast<hb_handle*>(hc);
  if (!h) return -1;
  if (trace == HB_KMEANS_ROUNDS) {
    if (out)
      for (int64_t i = 0; i < (int64_t)h->kmeans_rounds.size() && i < cap; ++i) out[i] = h->kmeans_rounds[i];
    return (int64_t)h->kmeans_rounds.size();
  }
  if (sync_traces(h) != 0) return -1;
  if (trace >= HB_OBJECTIVE_KMEANS && trace <= HB_OBJECTIVE_KMEANS_CROSS) {
    if (out)
      for (int64_t i = 0; i < h->obj_count && i < cap; ++i) out[i] = h->obj_vals[4 * (size_t)i + trace];
    return h->obj_count;
  }
  if (trace == HB_OBJECTIVE_HARMONY) {
    if (out)
      for (int64_t i = 0; i < (int64_t)h->harmony_slots.size() && i < cap; ++i)
        out[i] = h->obj_vals[4 * (size_t)h->harmony_slots[i]];
    return (int64_t)h->harmony_slots.size();
  }
  return -1;
}

int64_t hb_kernel_launches(const hb_handle* h) { return h ? h->launches : 0; }
void* hb_stream(const hb_handle* h) { return h ? (void*)h->stream : nullptr; }

int hb_synchronize(hb_handle* h) {
  if (!h) return 1;
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

int hb_region_time(hb_handle* h, const char* region, double* ms, int64_t* launches) {
  if (!h || !region) return 1;
  auto it = h->regions.find(region);
  if (it == h->regions.end()) return 2;
  if (ms) *ms = it->second.ms;
  if (launches) *launches = it->second.launches;
  return 0;
}

// Host evaluation of the keyed cell-order permutation used for the native update orders (test hook; the
// same __host__ __device__ code runs in k_plan_block_native / k_kmeans_seed).
uint64_t hb_debug_permute(uint64_t i, uint64_t n, uint64_t key, int inverse) {
  if (n == 0 || i >= n) return ~0ull;
  int bits = 1;
  while ((1ull << bits) < n) bits++;
  const int half_bits = (bits + 1) / 2;
  return inverse ? hb_permute_inv(i, n, half_bits, key) : hb_permute(i, n, half_bits, key);
}

// Host worker pool (test hook, host only): out[i] = (double) in[i] with `threads` threads (first call fixes the
// pool size for the process).  Returns the number of threads of the pool.
int hb_debug_widen(double* out, const float* in, int64_t n, int threads) {
  WidenPool* p = widen_pool(threads);
  if (n > 0) p->widen(out, in, (size_t)n);
  return p->threads();
}

// Ring geometry of the persistent update kernel for rows of KS floats (test hook, host only):
// out = {float4 per lane, groups per warp ring, rows per group, shared-memory bytes, warps}; 0 if the kernel cannot run the shape.
int hb_debug_update_geometry(int KS, int nb, int64_t out[9]) {
  (void)nb;
  if (KS <= 0 || (KS & 3)) return 0;
  const int D = upd5_ring_rows(KS, (size_t)227 * 1024 - 256);
  if (D <= 0) return 0;
  const int nv = upd4_nv(KS), ru = upd5_ru(nv);
  const int64_t v[9] = {nv, D / ru, ru, (int64_t)upd5_smem_bytes(nv, D, KS), U5_NW, 0, 0, 0, 0};
  for (int i = 0; i < 9; ++i) out[i] = v[i];
  return 1;
}

// Test hooks of the native kmeans_centers: the uniform of (centroid i, global cell g) under the handle's seed, and
// the cells initialize_centroids chose (K values; 0 if the native initialisation has not run).
double hb_debug_kmeans_uniform(const hb_handle* h, uint64_t i, uint64_t g) {
  return (double)kmeans_uniform(hb_mix64(h->seed ^ 0x6b6d65616e73ull), i, g);
}
int hb_debug_kmeans_cells(const hb_handle* h, int64_t* out) {
  if (!h || h->kmeans_cells.empty()) return 0;
  for (size_t i = 0; i < h->kmeans_cells.size(); ++i) out[i] = h->kmeans_cells[i];
  return (int)h->kmeans_cells.size();
}

int hb_enable_timing(hb_handle* h, int on) {
  if (!h) return 1;
  h->timing = on != 0;
  return 0;
}

}  // extern "C"
