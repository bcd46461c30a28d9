// C-ABI layer: the sxt_* drop-in entry points and the b200_* device-resident extension
// (include/blitzar_b200.h). Host side is plain C++ over CUDA streams (compute + copy stream per device,
// an auxiliary stream for the two halves of a batch-affine level); all arithmetic runs in the kernels
// of msm.cuh / batch_affine.cuh / lanefield.cuh. There is no CPU fallback: without a usable GPU sxt_init
// aborts, exactly as the reference's gpu backend does (cbindings/backend.cc:50-64).
//
// Also here: the copy / compute pipeline of host-pointer calls (commit_on), the parallel staging of
// pageable memory (HostStager), fixed-base handles with their device-built tables (shard_new), and
// the in-process multi-GPU layer (BLITZAR_B200_DEVICES: worker thread per device; by column, by
// generator range, sharded handles — commit_host / fixed_host / handle_new).
//
// Replaces: cbindings/{backend,pedersen,fixed_pedersen,get_generators,get_one_commit}.cc, the
// gpu_backend methods they dispatch to (sxt/cbindings/backend/gpu_backend.cc:150-334), the multi-device
// split of sxt/multiexp/pippenger2/multiexponentiation.h:100-135,248-287 and the handle accessor of
// sxt/multiexp/pippenger2/in_memory_partition_table_accessor{,_utility}.h.
#include <algorithm>
#include <cctype>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <memory>
#include <string>
#include <vector>

#include "engine_api.cuh"

using namespace b200;

namespace {

struct State {
  bool initialized = false;
  int device = -1;
  cudaStream_t stream = nullptr;       // every kernel of the engine
  cudaStream_t copy_stream = nullptr;  // host-to-device staging of the C-ABI calls
  cudaStream_t tail_stream = nullptr;  // cascade + bucket merge of upload piece k, under piece k+1
  cudaEvent_t range_events[16] = {};
  cudaEvent_t alloc_event = nullptr;
  void* builtin = nullptr;  // g(0..num_builtin) device-resident, ed25519 generator layout,
                            // followed by windows 1.. of their fixed-base table
  uint64_t num_builtin = 0;
  unsigned builtin_window_bits = 0, builtin_windows = 0;
  MsmOptions opt;
};
State g_state;  // the primary device: every entry point runs here
EngineCtx ctx_of(const State& st) {
  EngineCtx c{st.stream, g_state.opt, st.builtin, st.num_builtin};
  c.builtin_window_bits = st.builtin_window_bits;
  c.builtin_windows = st.builtin_windows;
  static const bool tail_on = [] {
    const char* env = std::getenv("BLITZAR_B200_TAIL_STREAM");
    return env != nullptr && std::atoi(env) != 0;  // off by default (measured: no gain, see DESIGN §8)
  }();
  if (tail_on)
    c.tail = st.tail_stream;
  if (const char* env = std::getenv("BLITZAR_B200_GROUP_ENTRIES"))  // test hook: force column groups
    c.opt.max_group_entries = std::strtoull(env, nullptr, 10);
  if (const char* env = std::getenv("BLITZAR_B200_UNIFORM_ADD"))
    c.opt.uniform_add = (u32)std::atoi(env);
  if (const char* env = std::getenv("BLITZAR_B200_LANE_TAIL"))
    c.opt.lane_tail = (u32)std::atoi(env);
  if (const char* env = std::getenv("BLITZAR_B200_SCATTER_WM"))
    c.opt.scatter_window_major = (u32)std::atoi(env);
  if (const char* env = std::getenv("BLITZAR_B200_PAIR_LEVELS"))  // batch-affine levels (-1 = auto)
    c.opt.pair_levels = std::atoi(env);
  if (const char* env = std::getenv("BLITZAR_B200_PAIR_BATCH"))
    c.opt.pair_batch = (u32)std::atoi(env);
  if (const char* env = std::getenv("BLITZAR_B200_TABLE_POLICY"))  // 1 = always use tables, 2 = never
    c.opt.table_policy = (u32)std::atoi(env);
  return c;
}
EngineCtx ctx() { return ctx_of(g_state); }
std::mutex g_mutex;  // calls are serialised on the one library stream

void init_device_state(State& st) {
  B200_CUDA(cudaSetDevice(st.device));
  B200_CUDA(cudaStreamCreateWithFlags(&st.stream, cudaStreamNonBlocking));
  B200_CUDA(cudaStreamCreateWithFlags(&st.copy_stream, cudaStreamNonBlocking));
  int prio_low = 0, prio_high = 0;  // the tail's small kernels must not queue behind a bulk kernel's blocks
  B200_CUDA(cudaDeviceGetStreamPriorityRange(&prio_low, &prio_high));
  B200_CUDA(cudaStreamCreateWithPriority(&st.tail_stream, cudaStreamNonBlocking, prio_high));
  for (auto& e : st.range_events)
    B200_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  B200_CUDA(cudaEventCreateWithFlags(&st.alloc_event, cudaEventDisableTiming));
  cudaMemPool_t pool;
  B200_CUDA(cudaDeviceGetDefaultMemPool(&pool, st.device));
  uint64_t threshold = UINT64_MAX;  // keep freed blocks cached in the pool between calls
  B200_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold));
}

void ensure_device() {
  if (g_state.stream)
    return;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    die("no supported GPUs found (this library has no CPU fallback)", __FILE__, __LINE__);
  if (g_state.device < 0) {
    const char* env = std::getenv("BLITZAR_B200_DEVICE");
    if (env)
      g_state.device = std::atoi(env);
    else
      B200_CUDA(cudaGetDevice(&g_state.device));
  }
  init_device_state(g_state);
}

// Window width of a fixed-base table over n generators of a curve on the current device: at most
// 40 % of the free HBM (180 GB per B200: n = 2^24 bn254 generators take 14 GB at c = 20), overridable
// with BLITZAR_B200_TABLE_WINDOW (0 disables tables).
unsigned choose_table_window(uint64_t n, size_t gen_bytes) {
  if (const char* env = std::getenv("BLITZAR_B200_TABLE_WINDOW")) {
    const int c = std::atoi(env);
    if (c <= 0)
      return 0;
    const unsigned cc = (unsigned)std::min(22, std::max(8, c));
    return (uint64_t)(256 / cc + 1) * n < (1ull << 31) ? cc : 0;
  }
  size_t free_b = 0, total_b = 0;
  B200_CUDA(cudaMemGetInfo(&free_b, &total_b));
  return table_window_bits(n, gen_bytes, 0.4 * (double)free_b);
}

// device array of `windows` x n generators; window 0 = g(0 .. n) built in, the rest their table
void make_builtin_table(State& st, uint64_t np) {
  const CurveVTable& V = kVTableEd25519;
  const unsigned c = choose_table_window(np, V.gen_bytes);
  const unsigned windows = c ? 256 / c + 1 : 1;
  B200_CUDA(cudaMalloc(&st.builtin, (size_t)np * windows * V.gen_bytes));
  EngineCtx cx = ctx_of(st);
  launch_builtin_generators(cx, st.builtin, 0, np);
  V.build_table(cx, st.builtin, np, c, windows);
  stream_sync(st.stream);
  st.num_builtin = np;
  st.builtin_window_bits = c;
  st.builtin_windows = windows;
}

void require_init(const char* fn) {
  if (!g_state.initialized) {
    std::fprintf(stderr, "blitzar_b200: backend uninitialized in `%s`\n", fn);
    std::abort();
  }
  B200_CUDA(cudaSetDevice(g_state.device));
}

const CurveVTable& vt(unsigned curve_id) {
  switch (curve_id) {
  case SXT_CURVE_RISTRETTO255:
    return kVTableEd25519;
  case SXT_CURVE_BLS_381:
    return kVTableBls12381;
  case SXT_CURVE_BN_254:
    return kVTableBn254;
  case SXT_CURVE_GRUMPKIN:
    return kVTableGrumpkin;
  default:
    die("unsupported curve id", __FILE__, __LINE__);
  }
}


// Host-to-device upload of PAGEABLE caller memory. A plain cudaMemcpyAsync from pageable memory is
// staged by the driver on one thread (~8-10 GB/s measured: 192 MiB took ~20 ms of a 23 ms call).
// Here a small persistent thread pool copies 8 MiB chunks into a ring of pinned buffers in parallel
// while the previous chunk is in flight on the copy stream. Pinned caller memory (as bench.py
// passes) goes straight to cudaMemcpyAsync.
class HostStager {
public:
  static HostStager& get() {
    static thread_local HostStager s;  // one staging ring + pool per host thread (= per device)
    return s;
  }
  void copy(void* dst_dev, const void* src_host, size_t bytes, cudaStream_t sc) {
    if (bytes == 0)
      return;
    cudaPointerAttributes attr;
    bool pinned = cudaPointerGetAttributes(&attr, src_host) == cudaSuccess &&
                  (attr.type == cudaMemoryTypeHost || attr.type == cudaMemoryTypeManaged);
    cudaGetLastError();  // unregistered host memory may set a sticky-free error on old drivers
    static const bool enabled = [] {
      const char* env = std::getenv("BLITZAR_B200_STAGER");
      return env == nullptr || std::atoi(env) != 0;  // on by default; BLITZAR_B200_STAGER=0 disables
    }();
    if (!enabled || pinned || bytes < (1u << 20)) {
      B200_CUDA(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, sc));
      return;
    }
    init();
    const unsigned char* src = static_cast<const unsigned char*>(src_host);
    unsigned char* dst = static_cast<unsigned char*>(dst_dev);
    for (size_t off = 0; off < bytes; off += kChunk) {
      const size_t len = std::min(kChunk, bytes - off);
      const int slot = next_++ % kSlots;
      B200_CUDA(cudaEventSynchronize(done_[slot]));
      parallel_memcpy(staging_[slot], src + off, len);
      B200_CUDA(cudaMemcpyAsync(dst + off, staging_[slot], len, cudaMemcpyHostToDevice, sc));
      B200_CUDA(cudaEventRecord(done_[slot], sc));
    }
  }

private:
  static constexpr size_t kChunk = 8u << 20;
  static constexpr int kSlots = 4;
  // threads copying one chunk into the pinned ring (the caller's included); a B200 host has on the
  // order of 100 cores and one core moves ~10 GB/s, PCIe 5 x16 wants ~55 GB/s
  const int kWorkers = [] {
    const char* env = std::getenv("BLITZAR_B200_STAGER_THREADS");
    const int v = env ? std::atoi(env) : 4;  // measured on the B200 host: 2: 16.0, 4: 8.0, 8: 12.4, 16: 9.2 ms (n = 2^20)
    return std::max(1, std::min(32, v));
  }();
  unsigned char* staging_[kSlots] = {};
  cudaEvent_t done_[kSlots] = {};
  unsigned next_ = 0;
  bool ready_ = false;
  // worker pool: one job = one slice of a chunk
  std::vector<std::thread> workers_;
  std::mutex m_;
  std::condition_variable cv_work_, cv_done_;
  struct Job {
    void* d;
    const void* s;
    size_t n;
  };
  std::vector<Job> jobs_;
  int pending_ = 0;
  bool stop_ = false;

  void init() {
    if (ready_)
      return;
    for (int i = 0; i < kSlots; ++i) {
      B200_CUDA(cudaHostAlloc((void**)&staging_[i], kChunk, cudaHostAllocDefault));
      B200_CUDA(cudaEventCreateWithFlags(&done_[i], cudaEventDisableTiming));
    }
    for (int w = 0; w < kWorkers - 1; ++w)
      workers_.emplace_back([this] { worker(); });
    ready_ = true;
  }
  void worker() {
    for (;;) {
      Job j;
      {
        std::unique_lock<std::mutex> lk(m_);
        cv_work_.wait(lk, [this] { return stop_ || !jobs_.empty(); });
        if (stop_ && jobs_.empty())
          return;
        j = jobs_.back();
        jobs_.pop_back();
      }
      std::memcpy(j.d, j.s, j.n);
      {
        std::lock_guard<std::mutex> lk(m_);
        if (--pending_ == 0)
          cv_done_.notify_all();
      }
    }
  }
  void parallel_memcpy(void* d, const void* s, size_t n) {
    const size_t slice = (n + kWorkers - 1) / kWorkers;
    size_t own = std::min(slice, n);
    {
      std::lock_guard<std::mutex> lk(m_);
      for (size_t off = own; off < n; off += slice) {
        jobs_.push_back(Job{(char*)d + off, (const char*)s + off, std::min(slice, n - off)});
        ++pending_;
      }
    }
    cv_work_.notify_all();
    std::memcpy(d, s, own);  // the calling thread copies the first slice itself
    std::unique_lock<std::mutex> lk(m_);
    cv_done_.wait(lk, [this] { return pending_ == 0; });
  }
  ~HostStager() {
    {
      std::lock_guard<std::mutex> lk(m_);
      stop_ = true;
    }
    cv_work_.notify_all();
    for (auto& t : workers_)
      t.join();
    for (int i = 0; i < kSlots; ++i) {  // errors ignored: the context may already be gone at exit
      if (staging_[i])
        cudaFreeHost(staging_[i]);
      if (done_[i])
        cudaEventDestroy(done_[i]);
    }
  }
};

// validates like cbindings/pedersen.cc:44-68 and returns the longest column
uint64_t longest_column(const sxt_sequence_descriptor* d, uint32_t num) {
  B200_REQUIRE(d != nullptr, "descriptors == nullptr");
  uint64_t longest = 0;
  for (uint32_t i = 0; i < num; ++i) {
    B200_REQUIRE(d[i].n == 0 || d[i].data != nullptr, "descriptor.n > 0 with data == nullptr");
    B200_REQUIRE(d[i].element_nbytes != 0 && d[i].element_nbytes <= 32,
                 "descriptor.element_nbytes must be in 1..32");
    longest = longest < d[i].n ? d[i].n : longest;
  }
  return longest;
}

// Host-pointer commitments. The generator range is split into pieces; the copy stream uploads piece
// after piece (scalars rows + generators) while the compute stream sorts and accumulates the
// previous one into the shared bucket array, so most of the PCIe time hides behind the kernels.
struct RangeWaitState {
  uint64_t n;
  uint32_t num_ranges;
  int skew;
  const State* st;
  uint32_t uploaded;                     // pieces [0, uploaded) are already on the copy stream
  std::function<void(uint32_t)> upload;  // enqueue (and, for pageable sources, stage) piece r
};
void wait_for_range(void* user, uint64_t begin, uint64_t end) {
  auto* w = static_cast<RangeWaitState*>(user);
  // wait for every upload piece that intersects [begin, end) (column groups ask for all of them).
  // Pieces are put on the copy stream only now, one piece ahead of the compute being enqueued: a
  // pageable source is staged by THIS thread (HostStager), and staging everything before the first
  // kernel launch would serialise upload and compute.
  for (uint32_t r = 0; r < w->num_ranges; ++r) {
    const uint64_t rb = range_begin(w->n, r, w->num_ranges, w->skew);
    const uint64_t re = range_begin(w->n, r + 1, w->num_ranges, w->skew);
    if (rb < end && begin < re) {
      while (w->uploaded <= std::min(r + 1, w->num_ranges - 1))
        w->upload(w->uploaded++);
      B200_CUDA(cudaStreamWaitEvent(w->st->stream, w->st->range_events[r], 0));
    }
  }
}

// the commitments of `num` columns on one device (the calling thread's current device is st.device)
// Results: `commitments` (host, canonical) or, when out_partials_dev is given instead, the internal
// accumulator points in device memory (multi-GPU callers combine them).
void commit_on(const State& st, unsigned curve_id, void* commitments, uint32_t num,
               const sxt_sequence_descriptor* d, const void* generators,
               uint64_t offset_generators, void* out_partials_dev = nullptr) {
  const CurveVTable& V = vt(curve_id);
  StageRange nvtx("commit (host buffers)");
  cudaStream_t s = st.stream, sc = st.copy_stream;
  uint64_t n = longest_column(d, num);
  size_t total_scalar_bytes = 0;
  for (uint32_t i = 0; i < num; ++i)
    total_scalar_bytes += (size_t)d[i].n * d[i].element_nbytes + 32;
  DevBuf<unsigned char> raw_gens(generators ? n * V.abi_gen_bytes : 1, s);
  DevBuf<unsigned char> scal(total_scalar_bytes, s);
  DevBuf<unsigned char> out((size_t)num * V.abi_commit_bytes, s);
  std::vector<sxt_sequence_descriptor> dd(d, d + num);
  std::vector<size_t> col_off(num);
  size_t off = 0;
  for (uint32_t i = 0; i < num; ++i) {
    col_off[i] = off;
    dd[i].data = scal.p + off;
    off += ((size_t)d[i].n * d[i].element_nbytes + 31) & ~(size_t)31;
  }
  // Upload in pieces so that sorting / accumulating piece r overlaps the PCIe copy of piece r+1
  // (later pieces accumulate into a scratch bucket array and are merged, MergeBucketsBody). Measured
  // on B200 through this call, pinned inputs, ristretto (tests/e2e_ranges.py), ms for 1/2/4/8 pieces:
  //   1 column : n=2^18 2.60/2.51/3.10/3.96  2^20 6.80/5.87/5.51/6.88  2^22 23.7/20.1/17.8/16.8
  //   4 columns: n=2^19 8.31/7.61/8.21/9.82  2^20 15.2/13.3/13.4/15.2  2^22 54.6/45.0/42.1/42.6
  // every piece costs ~0.3 ms of fixed sort / cascade work, hence pieces of >= 2^18 terms.
  uint32_t num_ranges = (uint32_t)std::min<uint64_t>(n >> 18, num == 1 ? 8 : 4);
  if (num == 1 && n >= (1ull << 18))
    num_ranges = std::max(num_ranges, 2u);
  // the Weierstrass curves pay a fixed cost per piece and batch-affine level (inversion trees, scratch
  // bucket merge): pieces of >= 2^21 terms. bls12-381 n = 2^22 from pinned memory, 1 / 2 / 3 / 4 / 8
  // pieces: 42.4 / 41.4 / 46.1 / 46.3 / 52.0 ms (tests/e2e_c3_ranges.py)
  if (curve_id != SXT_CURVE_RISTRETTO255)
    num_ranges = (uint32_t)std::min<uint64_t>(n >> 21, 4);
  num_ranges = std::max(num_ranges, 1u);
  if (const char* env = std::getenv("BLITZAR_B200_RANGES"))
    num_ranges = (uint32_t)std::max(1, std::min(16, std::atoi(env)));
  // piece schedule: equal pieces. Shrinking pieces (less work after the last byte of an upload-bound
  // call) and growing pieces (earlier first kernel of a compute-bound call) were measured and lose:
  // C2 e2e 5.22 -> 5.62 ms, C3 39.3 -> 39.7 ms (BLITZAR_B200_RANGE_SKEW = 1 / -1 selects them)
  int skew = 0;
  if (const char* env = std::getenv("BLITZAR_B200_RANGE_SKEW"))
    skew = std::atoi(env);
  // the destination buffers are stream-ordered allocations of the compute stream
  B200_CUDA(cudaEventRecord(st.alloc_event, s));
  B200_CUDA(cudaStreamWaitEvent(sc, st.alloc_event, 0));
  // BLITZAR_B200_TRACE=1: device timeline of one call (upload pieces vs compute) on stderr
  static const bool trace = std::getenv("BLITZAR_B200_TRACE") != nullptr;
  std::vector<cudaEvent_t> tev;
  auto mark = [&](cudaStream_t on) {
    if (!trace)
      return;
    cudaEvent_t e;
    B200_CUDA(cudaEventCreate(&e));
    B200_CUDA(cudaEventRecord(e, on));
    tev.push_back(e);
  };
  mark(sc);
  auto upload = [&](uint32_t r) {
    const uint64_t b = range_begin(n, r, num_ranges, skew), e = range_begin(n, r + 1, num_ranges, skew);
    for (uint32_t i = 0; i < num; ++i) {
      const uint64_t lo = std::min<uint64_t>(b, d[i].n), hi = std::min<uint64_t>(e, d[i].n);
      HostStager::get().copy(scal.p + col_off[i] + lo * d[i].element_nbytes,
                             d[i].data + lo * d[i].element_nbytes,
                             (hi - lo) * d[i].element_nbytes, sc);
    }
    if (generators)
      HostStager::get().copy(raw_gens.p + b * V.abi_gen_bytes,
                             static_cast<const unsigned char*>(generators) + b * V.abi_gen_bytes,
                             (e - b) * V.abi_gen_bytes, sc);
    B200_CUDA(cudaEventRecord(st.range_events[r], sc));
    mark(sc);
  };
  B200_LOG(2, "commit: curve %u, %u columns, n = %llu, device %d, %u upload pieces, generators %s",
           curve_id, num, (unsigned long long)n, st.device, num_ranges,
           generators ? "from the caller" : "built in");
  RangeWaitState w{n, num_ranges, skew, &st, 0, upload};
  EngineCtx cx = ctx_of(st);
  cx.opt.range_skew = skew;
  V.commit_device(cx, out_partials_dev ? nullptr : out.p, out_partials_dev, num, dd.data(),
                  generators ? raw_gens.p : nullptr, offset_generators, num_ranges, &wait_for_range,
                  &w);
  mark(s);
  if (!out_partials_dev)
    copy_d2h(commitments, out.p, (size_t)num * V.abi_commit_bytes, s);
  stream_sync(s);
  if (trace) {
    std::fprintf(stderr, "blitzar_b200 trace: n=%llu cols=%u pieces=%u:", (unsigned long long)n, num,
                 num_ranges);
    for (size_t i = 1; i < tev.size(); ++i) {
      float ms = 0;
      B200_CUDA(cudaEventElapsedTime(&ms, tev[0], tev[i]));
      std::fprintf(stderr, " %s%.3f", i + 1 == tev.size() ? "compute_done=" : "upload=", ms);
    }
    std::fprintf(stderr, " ms\n");
    for (auto e : tev)
      cudaEventDestroy(e);
  }
}

// ---- optional in-process multi-GPU (BLITZAR_B200_DEVICES=k): independent columns are split over k
// devices, one persistent host thread per extra device, no inter-GPU traffic (SURVEY §8e "by column";
// the reference does the same with one host thread and round-robin cudaSetDevice,
// sxt/execution/device/for_each.cc:57-126). Off by default: under one-process-per-GPU launchers
// every rank already owns its device.
class Worker {
public:
  State st;
  explicit Worker(int device) {
    st.device = device;
    th_ = std::thread([this] { run(); });
  }
  void submit(std::function<void()> f) {
    {
      std::lock_guard<std::mutex> lk(m_);
      task_ = std::move(f);
      busy_ = true;
    }
    cv_.notify_all();
  }
  void wait() {
    std::unique_lock<std::mutex> lk(m_);
    cv_.wait(lk, [this] { return !busy_; });
  }
  ~Worker() {
    {
      std::lock_guard<std::mutex> lk(m_);
      stop_ = true;
    }
    cv_.notify_all();
    if (th_.joinable())
      th_.join();
  }

private:
  std::thread th_;
  std::mutex m_;
  std::condition_variable cv_;
  std::function<void()> task_;
  bool busy_ = false, stop_ = false;
  void run() {
    B200_CUDA(cudaSetDevice(st.device));
    for (;;) {
      std::function<void()> f;
      {
        std::unique_lock<std::mutex> lk(m_);
        cv_.wait(lk, [this] { return stop_ || task_; });
        if (stop_ && !task_)
          return;
        f = std::move(task_);
        task_ = nullptr;
      }
      f();
      {
        std::lock_guard<std::mutex> lk(m_);
        busy_ = false;
      }
      cv_.notify_all();
    }
  }
};
std::vector<std::unique_ptr<Worker>> g_workers;

// Partial points of the k generator-range shards, gathered on the primary device (k x count points,
// shard-major) and summed there. Direct device-to-device copies (NVLink when peer access exists;
// cudaMemcpyPeerAsync stages through the host otherwise) — the only inter-GPU traffic of a call:
// count x point_bytes per device (SURVEY §8e; the reference stages the same partials through the
// host, sxt/multiexp/pippenger2/multiexponentiation.h:105-137).
struct Gather {
  void* buf = nullptr;
  size_t capacity = 0;
  void* ensure(size_t bytes) {
    if (bytes > capacity) {
      if (buf) {
        B200_CUDA(cudaStreamSynchronize(g_state.stream));
        B200_CUDA(cudaFree(buf));
      }
      capacity = std::max<size_t>(bytes, 1u << 16);
      B200_CUDA(cudaMalloc(&buf, capacity));
    }
    return buf;
  }
};
Gather g_gather;

// number of devices a generator range of n terms is split over
size_t range_parts(uint64_t n) {
  static const uint64_t min_terms = [] {
    const char* env = std::getenv("BLITZAR_B200_MIN_SHARD_TERMS");  // test hook
    return env ? std::strtoull(env, nullptr, 10) : (1ull << 15);
  }();
  return (size_t)std::max<uint64_t>(1, std::min<uint64_t>(g_workers.size() + 1, n / std::max<uint64_t>(min_terms, 1)));
}
State& state_of(size_t part) { return part == 0 ? g_state : g_workers[part - 1]->st; }
// runs f(part) for part = 0 .. parts-1: part 0 on the calling thread, the others on their device's
// worker thread; returns when all are done
template <class F> void on_devices(size_t parts, F f) {
  for (size_t p = 1; p < parts; ++p)
    g_workers[p - 1]->submit([=] { f(p); });
  f(0);
  for (size_t p = 1; p < parts; ++p)
    g_workers[p - 1]->wait();
  B200_CUDA(cudaSetDevice(g_state.device));
}
// this shard's `count` partial points -> slot `part` of the primary device's gather buffer
void send_partials(const State& st, size_t part, const void* partials_dev, size_t bytes,
                   void* gather_base) {
  unsigned char* dst = static_cast<unsigned char*>(gather_base) + part * bytes;
  if (part == 0)
    B200_CUDA(cudaMemcpyAsync(dst, partials_dev, bytes, cudaMemcpyDeviceToDevice, st.stream));
  else
    B200_CUDA(cudaMemcpyPeerAsync(dst, g_state.device, partials_dev, st.device, bytes, st.stream));
  B200_CUDA(cudaStreamSynchronize(st.stream));
}

void commit_host(unsigned curve_id, void* commitments, uint32_t num,
                 const sxt_sequence_descriptor* d, const void* generators,
                 uint64_t offset_generators, const char* fn, void* out_partials_dev = nullptr) {
  if (num == 0)
    return;
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init(fn);
  B200_REQUIRE(commitments != nullptr || out_partials_dev != nullptr, "commitments == nullptr");
  const uint64_t n = longest_column(d, num);  // validates the descriptors before any thread starts
  if (curve_id != SXT_CURVE_RISTRETTO255)
    B200_REQUIRE(generators != nullptr, "generators == nullptr");
  const CurveVTable& V = vt(curve_id);
  const size_t stride = V.abi_commit_bytes;
  const size_t devices = g_workers.size() + 1;
  if (devices <= 1 || out_partials_dev) {
    commit_on(g_state, curve_id, commitments, num, d, generators, offset_generators,
              out_partials_dev);
    return;
  }
  if (num >= devices) {
    // ---- by column: contiguous column chunks balanced by scalar bytes, no exchange at all ---------
    const size_t parts = devices;
    std::vector<uint64_t> prefix(num + 1, 0);
    for (uint32_t i = 0; i < num; ++i)
      prefix[i + 1] = prefix[i] + d[i].n * d[i].element_nbytes + 1;
    std::vector<uint32_t> cut(parts + 1, num);
    cut[0] = 0;
    for (size_t p = 1; p < parts; ++p) {
      uint32_t c = cut[p - 1] + 1;
      while (c < num - (parts - p) && prefix[c] * parts < prefix[num] * p)
        ++c;
      cut[p] = c;
    }
    on_devices(parts, [&, curve_id, commitments, d, generators, offset_generators](size_t p) {
      commit_on(state_of(p), curve_id, static_cast<unsigned char*>(commitments) + cut[p] * stride,
                cut[p + 1] - cut[p], d + cut[p], generators, offset_generators);
    });
    return;
  }
  // ---- by generator range (fewer columns than devices): device p computes the partial MSM of every
  // column over rows [n p / k, n (p+1) / k); one partial point per column and device is gathered on
  // the primary device and summed there (the MSM is linear)
  const size_t parts = range_parts(n);
  if (parts <= 1) {
    commit_on(g_state, curve_id, commitments, num, d, generators, offset_generators);
    return;
  }
  const size_t pbytes = (size_t)num * V.point_bytes;
  void* gather = g_gather.ensure(parts * pbytes);
  on_devices(parts, [&, curve_id, num, d, generators, offset_generators, n, parts, pbytes,
                     gather](size_t p) {
    State& st = state_of(p);
    const uint64_t lo = n * p / parts, hi = n * (p + 1) / parts;
    std::vector<sxt_sequence_descriptor> dd(d, d + num);
    for (auto& c : dd) {
      const uint64_t b = std::min<uint64_t>(lo, c.n), e = std::min<uint64_t>(hi, c.n);
      c.data = c.data ? c.data + b * c.element_nbytes : nullptr;
      c.n = e - b;
    }
    const unsigned char* g = static_cast<const unsigned char*>(generators);
    DevBuf<unsigned char> part(pbytes, st.stream);
    commit_on(st, curve_id, nullptr, num, dd.data(), g ? g + lo * V.abi_gen_bytes : nullptr,
              offset_generators + lo, part.p);
    send_partials(st, p, part.p, pbytes, gather);
  });
  cudaStream_t s = g_state.stream;
  DevBuf<unsigned char> sum(pbytes, s);
  DevBuf<unsigned char> out((size_t)num * stride, s);
  V.sum_parts(ctx(), gather, (uint32_t)parts, num, sum.p);
  V.store(ctx(), sum.p, out.p, num, true);
  copy_d2h(commitments, out.p, (size_t)num * stride, s);
  stream_sync(s);
}

// sxt_multiexp_handle: one shard per device (BLITZAR_B200_DEVICES=k splits the generator range at
// construction; SURVEY §8e "fixed-base handle: shard generators at sxt_multiexp_handle_new time")
struct HandleSet {
  unsigned curve_id = 0, n = 0;
  std::vector<Handle*> shards;
  std::vector<unsigned> first;  // first generator of every shard
};

// One shard on st's device (the calling thread's current device). generators: n projective ABI
// structs (host memory, or device_resident: already in HBM), or — compact_window != 0 — the table
// image of a reference partition-table file (host memory). Builds the fixed-base table 2^(c w) G_i
// on the device (replaces the reference's CPU-serial make_in_memory_partition_table_accessor,
// in_memory_partition_table_accessor_utility.h:41-79).
Handle* shard_new(const State& st, unsigned curve_id, const void* generators, unsigned n,
                  bool device_resident, unsigned compact_window, size_t compact_bytes) {
  const CurveVTable& V = vt(curve_id);
  cudaStream_t s = st.stream;
  Handle* h = new Handle{curve_id, n, nullptr};
  h->window_bits = choose_table_window(n, V.gen_bytes);
  h->windows = h->window_bits ? 256 / h->window_bits + 1 : 1;
  B200_CUDA(cudaMalloc(&h->gens, (size_t)(n ? n : 1) * h->windows * V.gen_bytes));
  if (n) {
    B200_REQUIRE(generators != nullptr, "generators == nullptr");
    const EngineCtx cx = ctx_of(st);
    if (compact_window) {
      DevBuf<unsigned char> raw(compact_bytes, s);
      HostStager::get().copy(raw.p, generators, compact_bytes, s);
      V.ingest_compact_table(cx, raw.p, compact_window, h->gens, n);
    } else if (device_resident) {
      V.ingest_projective(cx, generators, h->gens, n);
    } else {
      DevBuf<unsigned char> raw((size_t)n * V.abi_proj_bytes, s);
      HostStager::get().copy(raw.p, generators, (size_t)n * V.abi_proj_bytes, s);
      V.ingest_projective(cx, raw.p, h->gens, n);
    }
    V.build_table(cx, h->gens, n, h->window_bits, h->windows);
    stream_sync(s);
  }
  return h;
}

HandleSet* handle_new(unsigned curve_id, const void* generators, unsigned n,
                      bool device_resident = false, unsigned compact_window = 0,
                      size_t compact_bytes = 0) {
  const CurveVTable& V = vt(curve_id);
  HandleSet* hs = new HandleSet;
  hs->curve_id = curve_id;
  hs->n = n;
  size_t parts = device_resident ? 1 : range_parts(n);
  const unsigned align = compact_window ? compact_window : 1;  // shards start on a table group
  hs->shards.assign(parts, nullptr);
  hs->first.assign(parts + 1, n);
  for (size_t p = 0; p < parts; ++p)
    hs->first[p] = (unsigned)(((uint64_t)n * p / parts) / align * align);
  on_devices(parts, [&, curve_id, generators, device_resident, compact_window](size_t p) {
    const unsigned lo = hs->first[p], cnt = hs->first[p + 1] - lo;
    const unsigned char* g = static_cast<const unsigned char*>(generators);
    size_t off = 0, cbytes = 0;
    if (compact_window) {
      const size_t group_bytes = (size_t)V.abi_compact_bytes << compact_window;
      off = (size_t)(lo / compact_window) * group_bytes;
      cbytes = (size_t)((cnt + compact_window - 1) / compact_window) * group_bytes;
    } else {
      off = (size_t)lo * V.abi_proj_bytes;
    }
    hs->shards[p] = shard_new(state_of(p), curve_id, g ? g + off : nullptr, cnt, device_resident,
                              compact_window, cbytes);
  });
  (void)compact_bytes;
  return hs;
}

struct FixedCall {
  int mode;
  unsigned element_num_bytes;
  const unsigned* bit_table;
  const unsigned* lengths;
  unsigned num_outputs, rows;
  uint64_t row_bytes;
};

// rows [lo, lo + h->n) of a fixed-base call on st's device: canonical projective results to `res`
// (host) or partial points to out_partials_dev
void fixed_on(const State& st, void* res, const Handle* h, const FixedCall& c, unsigned lo,
              const uint8_t* scalars, void* out_partials_dev) {
  cudaStream_t s = st.stream;
  const CurveVTable& V = vt(h->curve_id);
  const unsigned hi = std::min<uint64_t>((uint64_t)lo + h->n, c.rows);
  const unsigned rows = hi > lo ? hi - lo : 0;
  std::vector<unsigned> lens;
  if (c.mode == 2) {
    lens.resize(c.num_outputs);
    for (unsigned j = 0; j < c.num_outputs; ++j)
      lens[j] = c.lengths[j] > lo ? std::min(c.lengths[j] - lo, rows) : 0u;
  }
  const size_t bytes = (size_t)c.row_bytes * rows;
  DevBuf<unsigned char> scal(bytes + 64, s);
  DevBuf<unsigned char> out((size_t)c.num_outputs * V.abi_proj_bytes, s);
  HostStager::get().copy(scal.p, scalars + (size_t)c.row_bytes * lo, bytes, s);
  V.fixed_device(ctx_of(st), out_partials_dev ? nullptr : out.p, out_partials_dev, h, c.mode,
                 c.element_num_bytes, c.bit_table, c.mode == 2 ? lens.data() : nullptr,
                 c.num_outputs, rows, scal.p);
  if (!out_partials_dev)
    copy_d2h(res, out.p, (size_t)c.num_outputs * V.abi_proj_bytes, s);
  stream_sync(s);
}

void fixed_host(void* res, const HandleSet* hs, int mode, unsigned element_num_bytes,
                const unsigned* bit_table, const unsigned* lengths, unsigned num_outputs,
                unsigned n, const uint8_t* scalars, void* out_partials_dev = nullptr) {
  if (num_outputs == 0)
    return;
  FixedCall c{mode, element_num_bytes, bit_table, lengths, num_outputs, n, 0};
  uint64_t row_bits = 0;
  for (unsigned j = 0; j < num_outputs; ++j) {
    row_bits += mode == 0 ? 8ull * element_num_bytes : bit_table[j];
    if (mode == 2) {
      B200_REQUIRE(j == 0 || lengths[j] >= lengths[j - 1],
                   "output lengths must be sorted in ascending order");
      c.rows = j == 0 ? lengths[j] : (lengths[j] > c.rows ? lengths[j] : c.rows);
    }
  }
  c.row_bytes = (row_bits + 7) / 8;
  B200_REQUIRE(c.rows <= hs->n, "more scalars than generators in the handle");
  B200_REQUIRE(c.row_bytes * c.rows == 0 || scalars != nullptr, "scalars == nullptr");
  const size_t parts = hs->shards.size();
  if (parts == 1) {
    fixed_on(g_state, res, hs->shards[0], c, 0, scalars, out_partials_dev);
    return;
  }
  const CurveVTable& V = vt(hs->curve_id);
  const size_t pbytes = (size_t)num_outputs * V.point_bytes;
  void* gather = g_gather.ensure(parts * pbytes);
  on_devices(parts, [&, hs, scalars, pbytes, gather](size_t p) {
    State& st = state_of(p);
    DevBuf<unsigned char> part(pbytes, st.stream);
    fixed_on(st, nullptr, hs->shards[p], c, hs->first[p], scalars, part.p);
    send_partials(st, p, part.p, pbytes, gather);
  });
  cudaStream_t s = g_state.stream;
  if (out_partials_dev) {
    V.sum_parts(ctx(), gather, (uint32_t)parts, num_outputs, out_partials_dev);
    stream_sync(s);
    return;
  }
  DevBuf<unsigned char> sum(pbytes, s);
  DevBuf<unsigned char> out((size_t)num_outputs * V.abi_proj_bytes, s);
  V.sum_parts(ctx(), gather, (uint32_t)parts, num_outputs, sum.p);
  V.store(ctx(), sum.p, out.p, num_outputs, false);
  copy_d2h(res, out.p, (size_t)num_outputs * V.abi_proj_bytes, s);
  stream_sync(s);
}

const uint32_t kHandleMagic = 0x44483242u;  // "B2HD"

}  // namespace

// =====================================================================================================
// Part 1: sxt_*
// =====================================================================================================
extern "C" {

int sxt_init(const struct sxt_config* config) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (config == nullptr)
    die("config input to `sxt_init` is null", __FILE__, __LINE__);
  if (g_state.initialized)
    die("trying to reinitialize the backend in `sxt_init`", __FILE__, __LINE__);
  int backend = config->backend;
  if (const char* env = std::getenv("BLITZAR_BACKEND")) {
    std::string v(env);
    for (auto& ch : v)
      ch = (char)std::tolower(ch);
    if (v == "cpu")
      backend = SXT_CPU_BACKEND;
    else if (v == "gpu")
      backend = SXT_GPU_BACKEND;
    else
      die("invalid BLITZAR_BACKEND value", __FILE__, __LINE__);
  }
  if (backend == SXT_CPU_BACKEND) {
    std::fprintf(stderr, "blitzar_b200: this library provides only the gpu backend "
                         "(SXT_GPU_BACKEND); link the reference libblitzar for the cpu backend\n");
    return 2;
  }
  if (backend != SXT_GPU_BACKEND)
    return 1;
  ensure_device();
  g_state.initialized = true;
  uint64_t np = config->num_precomputed_generators;
  if (np)
    make_builtin_table(g_state, np);
  if (const char* env = std::getenv("BLITZAR_B200_DEVICES")) {
    int want = std::atoi(env), count = 0;
    B200_CUDA(cudaGetDeviceCount(&count));
    want = std::min(want, count);
    for (int k = 1; k < want; ++k) {
      auto w = std::make_unique<Worker>((g_state.device + k) % count);
      Worker* wp = w.get();
      wp->submit([wp, np] {
        init_device_state(wp->st);
        if (np)
          make_builtin_table(wp->st, np);
        wp->st.initialized = true;
      });
      wp->wait();
      g_workers.push_back(std::move(w));
    }
    B200_CUDA(cudaSetDevice(g_state.device));
  }
  return 0;
}

void sxt_curve25519_compute_pedersen_commitments(struct sxt_ristretto255_compressed* commitments,
                                                 uint32_t num_sequences,
                                                 const struct sxt_sequence_descriptor* descriptors,
                                                 uint64_t offset_generators) {
  commit_host(SXT_CURVE_RISTRETTO255, commitments, num_sequences, descriptors, nullptr,
              offset_generators, "sxt_curve25519_compute_pedersen_commitments");
}
void sxt_curve25519_compute_pedersen_commitments_with_generators(
    struct sxt_ristretto255_compressed* commitments, uint32_t num_sequences,
    const struct sxt_sequence_descriptor* descriptors, const struct sxt_ristretto255* generators) {
  // generators == nullptr falls back to the built-in generators at offset 0, as the reference does
  // (cbindings/pedersen.cc:90-96)
  commit_host(SXT_CURVE_RISTRETTO255, commitments, num_sequences, descriptors, generators, 0,
              "sxt_curve25519_compute_pedersen_commitments_with_generators");
}
void sxt_bls12_381_g1_compute_pedersen_commitments_with_generators(
    struct sxt_bls12_381_g1_compressed* commitments, uint32_t num_sequences,
    const struct sxt_sequence_descriptor* descriptors, const struct sxt_bls12_381_g1* generators) {
  commit_host(SXT_CURVE_BLS_381, commitments, num_sequences, descriptors, generators, 0,
              "sxt_bls12_381_g1_compute_pedersen_commitments_with_generators");
}
void sxt_bn254_g1_uncompressed_compute_pedersen_commitments_with_generators(
    struct sxt_bn254_g1* commitments, uint32_t num_sequences,
    const struct sxt_sequence_descriptor* descriptors, const struct sxt_bn254_g1* generators) {
  commit_host(SXT_CURVE_BN_254, commitments, num_sequences, descriptors, generators, 0,
              "sxt_bn254_g1_uncompressed_compute_pedersen_commitments_with_generators");
}
void sxt_grumpkin_uncompressed_compute_pedersen_commitments_with_generators(
    struct sxt_grumpkin* commitments, uint32_t num_sequences,
    const struct sxt_sequence_descriptor* descriptors, const struct sxt_grumpkin* generators) {
  commit_host(SXT_CURVE_GRUMPKIN, commitments, num_sequences, descriptors, generators, 0,
              "sxt_grumpkin_uncompressed_compute_pedersen_commitments_with_generators");
}

int sxt_ristretto255_get_generators(struct sxt_ristretto255* generators, uint64_t num_generators,
                                    uint64_t offset_generators) {
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("sxt_ristretto255_get_generators");
  if (num_generators == 0)
    return 0;
  if (generators == nullptr)
    return 1;
  const CurveVTable& V = kVTableEd25519;
  cudaStream_t s = g_state.stream;
  // generated straight into the ABI layout: the exact (X : Y : Z : T) of the derivation
  // (sqcgn::compute_base_element), not a round trip through the cached generator form
  DevBuf<unsigned char> out(num_generators * V.abi_proj_bytes, s);
  V.synth_generators(ctx(), out.p, num_generators, offset_generators, true);
  copy_d2h(generators, out.p, num_generators * V.abi_proj_bytes, s);
  stream_sync(s);
  return 0;
}

int sxt_curve25519_get_one_commit(struct sxt_ristretto255* one_commit, uint64_t n) {
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("sxt_curve25519_get_one_commit");
  B200_REQUIRE(one_commit != nullptr, "one_commit == nullptr");
  B200_REQUIRE(n < (1ull << 31), "n too large");
  const CurveVTable& V = kVTableEd25519;
  cudaStream_t s = g_state.stream;
  // sum of the first n built-in generators = MSM with all-one 1-byte scalars
  DevBuf<unsigned char> ones(n + 32, s);
  B200_CUDA(cudaMemsetAsync(ones.p, 1, n + 32, s));
  sxt_sequence_descriptor d{1, n, ones.p, 0};
  DevBuf<unsigned char> pt(V.point_bytes, s);
  DevBuf<unsigned char> out(V.abi_proj_bytes, s);
  V.commit_device(ctx(), nullptr, pt.p, 1, &d, nullptr, 0, 1, nullptr, nullptr);
  V.store(ctx(), pt.p, out.p, 1, false);
  copy_d2h(one_commit, out.p, V.abi_proj_bytes, s);
  stream_sync(s);
  return 0;
}

// blitzar_api.h:566 — checks as cbindings/inner_product_proof.cc:34-58
void sxt_curve25519_prove_inner_product(struct sxt_ristretto255_compressed* l_vector,
                                        struct sxt_ristretto255_compressed* r_vector,
                                        struct sxt_curve25519_scalar* ap_value,
                                        struct sxt_transcript* transcript, uint64_t n,
                                        uint64_t generators_offset,
                                        const struct sxt_curve25519_scalar* a_vector,
                                        const struct sxt_curve25519_scalar* b_vector) {
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("sxt_curve25519_prove_inner_product");
  B200_REQUIRE(transcript != nullptr, "transcript must not be null");
  B200_REQUIRE(ap_value != nullptr, "ap_value must not be null");
  B200_REQUIRE(b_vector != nullptr && a_vector != nullptr, "a_vector / b_vector must not be null");
  B200_REQUIRE(n > 0, "a_vector and b_vector lengths must be greater than zero");
  B200_REQUIRE(n == 1 || (l_vector != nullptr && r_vector != nullptr),
               "l_vector and r_vector must not be null when n > 1");
  B200_REQUIRE(n < (1ull << 30), "n too large");
  ipa_prove(ctx(), reinterpret_cast<uint8_t*>(l_vector), reinterpret_cast<uint8_t*>(r_vector),
            ap_value->bytes, transcript->bytes, n, generators_offset,
            reinterpret_cast<const uint8_t*>(a_vector), reinterpret_cast<const uint8_t*>(b_vector));
}
// blitzar_api.h:611 — 1 if the proof verifies, 0 otherwise
int sxt_curve25519_verify_inner_product(struct sxt_transcript* transcript, uint64_t n,
                                        uint64_t generators_offset,
                                        const struct sxt_curve25519_scalar* b_vector,
                                        const struct sxt_curve25519_scalar* product,
                                        const struct sxt_ristretto255* a_commit,
                                        const struct sxt_ristretto255_compressed* l_vector,
                                        const struct sxt_ristretto255_compressed* r_vector,
                                        const struct sxt_curve25519_scalar* ap_value) {
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("sxt_curve25519_verify_inner_product");
  B200_REQUIRE(transcript != nullptr, "transcript must not be null");
  B200_REQUIRE(ap_value != nullptr && product != nullptr && a_commit != nullptr &&
                   b_vector != nullptr,
               "ap_value / product / a_commit / b_vector must not be null");
  B200_REQUIRE(n > 0, "b_vector length must be greater than zero");
  B200_REQUIRE(n == 1 || (l_vector != nullptr && r_vector != nullptr),
               "l_vector and r_vector must not be null when n > 1");
  B200_REQUIRE(n < (1ull << 30), "n too large");
  return ipa_verify(ctx(), transcript->bytes, n, generators_offset,
                    reinterpret_cast<const uint8_t*>(b_vector), product->bytes,
                    reinterpret_cast<const uint8_t*>(a_commit),
                    reinterpret_cast<const uint8_t*>(l_vector),
                    reinterpret_cast<const uint8_t*>(r_vector), ap_value->bytes);
}
// blitzar_api.h:766 — as cpu_backend.cc:73-112 / gpu_backend.cc:106-145; the callback runs with the
// library mutex held
void sxt_prove_sumcheck(void* polynomials, void* evaluation_point, unsigned field_id,
                        const struct sumcheck_descriptor* descriptor, void* transcript_callback,
                        void* transcript_context) {
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("sxt_prove_sumcheck");
  sumcheck_prove(ctx(), polynomials, evaluation_point, field_id, descriptor, transcript_callback,
                 transcript_context, false);
}

struct sxt_multiexp_handle* sxt_multiexp_handle_new(unsigned curve_id, const void* generators,
                                                    unsigned n) {
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("sxt_multiexp_handle_new");
  return reinterpret_cast<sxt_multiexp_handle*>(handle_new(curve_id, generators, n));
}

void sxt_multiexp_handle_free(struct sxt_multiexp_handle* handle) {
  if (!handle)
    return;
  std::lock_guard<std::mutex> lock(g_mutex);
  HandleSet* hs = reinterpret_cast<HandleSet*>(handle);
  on_devices(hs->shards.size(), [hs](size_t p) {
    B200_CUDA(cudaStreamSynchronize(state_of(p).stream));
    B200_CUDA(cudaFree(hs->shards[p]->gens));
    delete hs->shards[p];
  });
  delete hs;
}

// File format written (versioned): u32 magic "B2HD", u32 version = 1, u32 curve_id, u32 n, then n
// projective ABI structs — the generators; the fixed-base table is rebuilt on load (a fraction of a
// second on the device, against the file being 13-26x larger with it). sxt_multiexp_handle_new_from_
// file also reads the reference's [u32 window_width][partition table] files (see there).
void sxt_multiexp_handle_write_to_file(const struct sxt_multiexp_handle* handle,
                                       const char* filename) {
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("sxt_multiexp_handle_write_to_file");
  const HandleSet* h = reinterpret_cast<const HandleSet*>(handle);
  B200_REQUIRE(h && filename, "null handle or filename");
  const CurveVTable& V = vt(h->curve_id);
  size_t bytes = (size_t)h->n * V.abi_proj_bytes;
  std::vector<unsigned char> host(bytes);
  on_devices(h->shards.size(), [&, h](size_t p) {
    const State& st = state_of(p);
    const Handle* sh = h->shards[p];
    const size_t sb = (size_t)sh->n * V.abi_proj_bytes;
    DevBuf<unsigned char> out(sb + 16, st.stream);
    V.gens_to_projective(ctx_of(st), sh->gens, out.p, sh->n);
    copy_d2h(host.data() + (size_t)h->first[p] * V.abi_proj_bytes, out.p, sb, st.stream);
    stream_sync(st.stream);
  });
  FILE* f = std::fopen(filename, "wb");
  B200_REQUIRE(f != nullptr, "cannot open handle file for writing");
  uint32_t hdr[4] = {kHandleMagic, 1u, h->curve_id, h->n};
  B200_REQUIRE(std::fwrite(hdr, sizeof(hdr), 1, f) == 1, "short write");
  B200_REQUIRE(bytes == 0 || std::fwrite(host.data(), bytes, 1, f) == 1, "short write");
  std::fclose(f);
}

struct sxt_multiexp_handle* sxt_multiexp_handle_new_from_file(unsigned curve_id,
                                                              const char* filename) {
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("sxt_multiexp_handle_new_from_file");
  B200_REQUIRE(filename != nullptr, "null filename");
  FILE* f = std::fopen(filename, "rb");
  B200_REQUIRE(f != nullptr, "cannot open handle file");
  uint32_t hdr[4] = {0, 0, 0, 0};
  B200_REQUIRE(std::fread(hdr, sizeof(uint32_t), 1, f) == 1, "short handle file");
  if (hdr[0] != kHandleMagic) {
    // The reference's own format (in_memory_partition_table_accessor.h:42-59,98-105):
    // [u32 window_width][table of compact elements], 2^w subset sums per group of w generators.
    // Entry (1 << j) of group g is generator g*w + j, so the generators are recovered exactly and
    // this library's table is rebuilt from them on the device (groups padded with the identity stay
    // identities, as in the reference).
    const unsigned w = hdr[0];
    const size_t esz = vt(curve_id).abi_compact_bytes;
    B200_REQUIRE(w >= 1 && w <= 24, "not a handle file (bad window width)");
    std::fseek(f, 0, SEEK_END);
    const size_t bytes = (size_t)std::ftell(f) - sizeof(uint32_t);
    std::fseek(f, sizeof(uint32_t), SEEK_SET);
    B200_REQUIRE(bytes % (esz << w) == 0, "partition table size does not match the curve");
    const size_t groups = bytes / (esz << w);
    B200_REQUIRE(groups * w < (1ull << 31), "partition table too large");
    std::vector<unsigned char> host(bytes);
    B200_REQUIRE(bytes == 0 || std::fread(host.data(), bytes, 1, f) == 1, "short handle file");
    std::fclose(f);
    return reinterpret_cast<sxt_multiexp_handle*>(
        handle_new(curve_id, host.data(), (unsigned)(groups * w), false, w, bytes));
  }
  B200_REQUIRE(std::fread(hdr + 1, 3 * sizeof(uint32_t), 1, f) == 1, "short handle file");
  B200_REQUIRE(hdr[1] == 1u, "unsupported blitzar_b200 handle file version");
  B200_REQUIRE(hdr[2] == curve_id, "handle file is for another curve");
  size_t bytes = (size_t)hdr[3] * vt(curve_id).abi_proj_bytes;
  std::vector<unsigned char> host(bytes);
  B200_REQUIRE(bytes == 0 || std::fread(host.data(), bytes, 1, f) == 1, "short handle file");
  std::fclose(f);
  return reinterpret_cast<sxt_multiexp_handle*>(handle_new(curve_id, host.data(), hdr[3]));
}

void sxt_fixed_multiexponentiation(void* res, const struct sxt_multiexp_handle* handle,
                                   unsigned element_num_bytes, unsigned num_outputs, unsigned n,
                                   const uint8_t* scalars) {
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("sxt_fixed_multiexponentiation");
  const HandleSet* h = reinterpret_cast<const HandleSet*>(handle);
  B200_REQUIRE(h != nullptr, "null handle");
  fixed_host(res, h, 0, element_num_bytes, nullptr, nullptr, num_outputs, n, scalars);
}
void sxt_fixed_packed_multiexponentiation(void* res, const struct sxt_multiexp_handle* handle,
                                          const unsigned* output_bit_table, unsigned num_outputs,
                                          unsigned n, const uint8_t* scalars) {
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("sxt_fixed_packed_multiexponentiation");
  const HandleSet* h = reinterpret_cast<const HandleSet*>(handle);
  B200_REQUIRE(h != nullptr, "null handle");
  fixed_host(res, h, 1, 0, output_bit_table, nullptr, num_outputs, n, scalars);
}
void sxt_fixed_vlen_multiexponentiation(void* res, const struct sxt_multiexp_handle* handle,
                                        const unsigned* output_bit_table,
                                        const unsigned* output_lengths, unsigned num_outputs,
                                        const uint8_t* scalars) {
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("sxt_fixed_vlen_multiexponentiation");
  const HandleSet* h = reinterpret_cast<const HandleSet*>(handle);
  B200_REQUIRE(h != nullptr, "null handle");
  fixed_host(res, h, 2, 0, output_bit_table, output_lengths, num_outputs, 0, scalars);
}

// =====================================================================================================
// Part 2: b200_*
// =====================================================================================================
void b200_set_device(int device) {
  std::lock_guard<std::mutex> lock(g_mutex);
  B200_REQUIRE(g_state.stream == nullptr, "b200_set_device must precede sxt_init");
  g_state.device = device;
}
unsigned long long b200_launch_count(void) { return LaunchCounter::value(); }
unsigned b200_point_bytes(unsigned curve_id) { return vt(curve_id).point_bytes; }
void* b200_malloc(uint64_t bytes) {
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("b200_malloc");
  void* p = nullptr;
  B200_CUDA(cudaMalloc(&p, bytes ? bytes : 16));
  return p;
}
void b200_free(void* p) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (p) {
    B200_CUDA(cudaSetDevice(g_state.device));
    B200_CUDA(cudaStreamSynchronize(g_state.stream));
    B200_CUDA(cudaFree(p));
  }
}
void b200_memcpy_h2d(void* d, const void* h, uint64_t bytes) {
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("b200_memcpy_h2d");
  copy_h2d(d, h, bytes, g_state.stream);
  stream_sync(g_state.stream);
}
void b200_memcpy_d2h(void* h, const void* d, uint64_t bytes) {
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("b200_memcpy_d2h");
  copy_d2h(h, d, bytes, g_state.stream);
  stream_sync(g_state.stream);
}
void* b200_stream(void) {
  require_init("b200_stream");
  return (void*)g_state.stream;
}
void b200_synchronize(void) {
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("b200_synchronize");
  stream_sync(g_state.stream);
}
void* b200_event_create(void) {
  require_init("b200_event_create");
  cudaEvent_t e;
  B200_CUDA(cudaEventCreate(&e));
  return (void*)e;
}
void b200_event_record(void* e) {
  std::lock_guard<std::mutex> lock(g_mutex);
  B200_CUDA(cudaEventRecord((cudaEvent_t)e, g_state.stream));
}
float b200_event_elapsed_ms(void* a, void* b) {
  float ms = 0;
  B200_CUDA(cudaEventSynchronize((cudaEvent_t)b));
  B200_CUDA(cudaEventElapsedTime(&ms, (cudaEvent_t)a, (cudaEvent_t)b));
  return ms;
}
void b200_event_destroy(void* e) { B200_CUDA(cudaEventDestroy((cudaEvent_t)e)); }

void b200_commit_device(unsigned curve_id, void* out_commitments, void* out_partials,
                        uint32_t num_sequences, const struct sxt_sequence_descriptor* descriptors,
                        const void* generators, uint64_t offset_generators) {
  if (num_sequences == 0)
    return;
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("b200_commit_device");
  vt(curve_id).commit_device(ctx(), out_commitments, out_partials, num_sequences, descriptors,
                             generators, offset_generators, 1, nullptr, nullptr);
}
void b200_commit_host_partials(unsigned curve_id, void* out_partials,
                               uint32_t num_sequences,
                               const struct sxt_sequence_descriptor* descriptors,
                               const void* generators, uint64_t offset_generators) {
  if (num_sequences == 0)
    return;
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("b200_commit_host_partials");
  B200_REQUIRE(out_partials != nullptr, "out_partials == nullptr");
  commit_on(g_state, curve_id, nullptr, num_sequences, descriptors, generators, offset_generators,
            out_partials);
}
void b200_fixed_msm_host_partials(void* out_partials, const struct sxt_multiexp_handle* handle,
                                  int mode, unsigned element_num_bytes,
                                  const unsigned* output_bit_table, const unsigned* output_lengths,
                                  unsigned num_outputs, unsigned n, const uint8_t* scalars) {
  if (num_outputs == 0)
    return;
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("b200_fixed_msm_host_partials");
  const HandleSet* h = reinterpret_cast<const HandleSet*>(handle);
  B200_REQUIRE(h != nullptr && out_partials != nullptr, "null handle or out_partials");
  fixed_host(nullptr, h, mode, element_num_bytes, output_bit_table, output_lengths, num_outputs, n,
             scalars, out_partials);
}
struct sxt_multiexp_handle* b200_multiexp_handle_new_device(unsigned curve_id,
                                                            const void* generators_dev,
                                                            unsigned n) {
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("b200_multiexp_handle_new_device");
  return reinterpret_cast<sxt_multiexp_handle*>(handle_new(curve_id, generators_dev, n, true));
}
void b200_combine_partials_device(unsigned curve_id, void* out_commitments, const void* partials,
                                  uint32_t num_parts, uint32_t count) {
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("b200_combine_partials_device");
  const CurveVTable& V = vt(curve_id);
  DevBuf<unsigned char> sum((size_t)count * V.point_bytes, g_state.stream);
  V.sum_parts(ctx(), partials, num_parts, count, sum.p);
  V.store(ctx(), sum.p, out_commitments, count, true);
}
void b200_combine_partials_projective_device(unsigned curve_id, void* out_res,
                                             const void* partials, uint32_t num_parts,
                                             uint32_t count) {
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("b200_combine_partials_projective_device");
  const CurveVTable& V = vt(curve_id);
  DevBuf<unsigned char> sum((size_t)count * V.point_bytes, g_state.stream);
  V.sum_parts(ctx(), partials, num_parts, count, sum.p);
  V.store(ctx(), sum.p, out_res, count, false);
}
void b200_fixed_msm_device(void* out_res, void* out_partials,
                           const struct sxt_multiexp_handle* handle, int mode,
                           unsigned element_num_bytes, const unsigned* output_bit_table,
                           const unsigned* output_lengths, unsigned num_outputs, unsigned n,
                           const uint8_t* scalars) {
  if (num_outputs == 0)
    return;
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("b200_fixed_msm_device");
  const HandleSet* hs = reinterpret_cast<const HandleSet*>(handle);
  B200_REQUIRE(hs != nullptr, "null handle");
  B200_REQUIRE(hs->shards.size() == 1, "device-resident fixed MSM needs a single-device handle");
  const Handle* h = hs->shards[0];
  unsigned rows = n;
  if (mode == 2) {
    rows = 0;
    for (unsigned j = 0; j < num_outputs; ++j)
      rows = output_lengths[j] > rows ? output_lengths[j] : rows;
  }
  vt(h->curve_id).fixed_device(ctx(), out_res, out_partials, h, mode, element_num_bytes,
                               output_bit_table, output_lengths, num_outputs, rows, scalars);
}
void b200_synthetic_generators_device(unsigned curve_id, void* out_generators, uint64_t n,
                                      uint64_t first, int projective) {
  if (n == 0)
    return;
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("b200_synthetic_generators_device");
  B200_REQUIRE(out_generators != nullptr, "out_generators == nullptr");
  vt(curve_id).synth_generators(ctx(), out_generators, n, first, projective != 0);
}
void b200_prove_sumcheck_device(void* polynomials, void* evaluation_point, unsigned field_id,
                                const struct sumcheck_descriptor* descriptor,
                                void* transcript_callback, void* transcript_context) {
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("b200_prove_sumcheck_device");
  sumcheck_prove(ctx(), polynomials, evaluation_point, field_id, descriptor, transcript_callback,
                 transcript_context, true);
}
unsigned b200_selftest_lane_arithmetic(unsigned warps, unsigned seed) {
  std::lock_guard<std::mutex> lock(g_mutex);
  require_init("b200_selftest_lane_arithmetic");
  return selftest_lane_arithmetic(ctx(), warps, seed);
}
void b200_set_reduce_groups(unsigned g1, unsigned gn) {
  std::lock_guard<std::mutex> lock(g_mutex);
  auto pow2 = [](unsigned v, unsigned dflt) {
    if (v < 2)
      return dflt;
    unsigned p = 2;
    while (p * 2 <= v)
      p *= 2;
    return p;
  };
  g_state.opt.reduce_g1 = pow2(g1, 16u);
  g_state.opt.reduce_gn = pow2(gn, 4u);
}
void b200_profile_accumulate(int enable) {
  std::lock_guard<std::mutex> lock(g_mutex);
  KernelTimer::get().enabled = enable != 0;
}
void b200_profile_read(float* total_ms, unsigned* launches) {
  std::lock_guard<std::mutex> lock(g_mutex);
  KernelTimer::get().read(total_ms, launches);
}
void b200_set_tuning(unsigned window_bits, unsigned chunk1, unsigned chunkn) {
  std::lock_guard<std::mutex> lock(g_mutex);
  g_state.opt.window_bits = window_bits;
  g_state.opt.chunk1 = chunk1;
  g_state.opt.chunkn = chunkn ? chunkn : 8;
}

}  // extern "C"
