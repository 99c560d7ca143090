// C ABI of casapose_b200 (include/casapose_b200.h): host-side orchestration of the kernels.
// Build:  nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -shared -Xcompiler -fPIC
#include <dlfcn.h>
#include <immintrin.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <chrono>
#include <condition_variable>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

#include "common.cuh"
#include "compaction.cuh"
#include "ls_vote.cuh"
#include "pnp.cuh"
#include "pose_metric.cuh"
#include "predicate.cuh"
#include "ransac.cuh"
#include "selftest.cuh"

using namespace casa;

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define CUDA_TRY(expr)                                                                        \
  do {                                                                                        \
    cudaError_t e__ = (expr);                                                                 \
    if (e__ != cudaSuccess)                                                                   \
      return fail(CASA_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

// ------------------------------------------------------------------------------------------------ host mask packer
// casa_ransac_vote_host: the float one-hot mask carries 4 bits of information per 32 bytes.  A small pool of host
// threads turns it into one u32 membership word per pixel (the same word k_mask_bits builds on the device) while
// the GPU works on the previous image range, so 1/8 of the mask's bytes (1/oc in general) cross PCIe.
namespace {
class MaskPacker {
 public:
  explicit MaskPacker(int n) : n_(n) {
    for (int i = 0; i < n_; ++i) workers_.emplace_back([this, i] { run(i); });
  }
  ~MaskPacker() {
    {
      std::lock_guard<std::mutex> g(m_);
      quit_ = true;
    }
    cv_.notify_all();
    for (std::thread& t : workers_) t.join();
  }
  // packs `mask` ([npx][oc] floats) into `bits`; part k = pixels [bounds[2k], bounds[2k+1]), parts in order.
  // The workers take kChunkPx-pixel chunks of the current part from a shared counter, and a part is done when its
  // last chunk is — not when every worker has reported — so a worker the host has descheduled (the caller's driver
  // threads, the Python thread and the CUDA runtime share the cores) holds up one chunk, not the part.
  void start(const float* mask, uint32_t* bits, int oc, const std::vector<size_t>& bounds) {
    std::shared_ptr<Job> j = std::make_shared<Job>();
    j->mask = mask;
    j->bits = bits;
    j->oc = oc;
    j->bounds = bounds;
    const size_t parts = bounds.size() / 2;
    j->nchunks.resize(parts);
    j->next.reset(new std::atomic<size_t>[parts ? parts : 1]);
    j->done.reset(new std::atomic<size_t>[parts ? parts : 1]);
    for (size_t k = 0; k < parts; ++k) {
      j->nchunks[k] = (bounds[2 * k + 1] - bounds[2 * k] + kChunkPx - 1) / kChunkPx;
      j->next[k].store(0);
      j->done[k].store(0);
    }
    std::lock_guard<std::mutex> g(m_);
    job_ = j;
    ++epoch_;
    cv_.notify_all();
  }
  void wait_part(size_t k) {
    std::unique_lock<std::mutex> g(m_);
    cv_done_.wait(g, [&] { return job_->done[k].load() >= job_->nchunks[k]; });
  }
  int not_binary() const { return job_ ? job_->not_binary.load() : 0; }

 private:
  static constexpr size_t kChunkPx = 8192;  // 256 KB of an 8-channel mask per chunk
  struct Job {  // one start(): a straggler of the previous call keeps its own (exhausted) job
    const float* mask = nullptr;
    uint32_t* bits = nullptr;
    int oc = 0;
    std::vector<size_t> bounds, nchunks;
    std::unique_ptr<std::atomic<size_t>[]> next, done;
    std::atomic<int> not_binary{0};
  };
  void run(int) {
    long long seen = 0;
    for (;;) {
      std::shared_ptr<Job> j;
      {
        std::unique_lock<std::mutex> g(m_);
        cv_.wait(g, [&] { return quit_ || epoch_ != seen; });
        if (quit_) return;
        seen = epoch_;
        j = job_;
      }
      for (size_t k = 0; k < j->nchunks.size(); ++k) {  // parts in order, chunks of a part from the shared counter
        const size_t lo0 = j->bounds[2 * k], hi0 = j->bounds[2 * k + 1];
        for (;;) {
          const size_t c = j->next[k].fetch_add(1);
          if (c >= j->nchunks[k]) break;
          const size_t lo = lo0 + c * kChunkPx, hi = lo + kChunkPx < hi0 ? lo + kChunkPx : hi0;
          if (pack(j->mask, j->bits, j->oc, lo, hi)) j->not_binary.store(1);
          if (j->done[k].fetch_add(1) + 1 == j->nchunks[k]) {
            std::lock_guard<std::mutex> g(m_);
            cv_done_.notify_all();
          }
        }
      }
    }
  }
  // bit c of bits[p] = (mask[p][c] != 0) — NaN counts as set, -0 does not, like tf.not_equal (:304); returns whether a
  // set element differs from 1.0 (CASA_STATUS_MASK_NOT_BINARY)
  __attribute__((target("avx2"))) static bool pack8_avx2(const float* mask, uint32_t* bits, size_t lo, size_t hi) {
    // one 256-bit row per pixel: (v << 1) != 0 per lane -> 8-bit membership word; set lanes must hold 1.0f.  Eight rows
    // per trip: their OR decides with one test whether all eight are background (87 % of the rows of an LM-O frame),
    // which then cost eight loads and one 32-byte store (experimental/pack_bench.cpp: +45 % over the row-by-row loop).
    const __m256i zero = _mm256_setzero_si256(), one = _mm256_set1_epi32(0x3F800000);
    unsigned bad = 0;
    size_t p = lo;
    for (; p + 8 <= hi; p += 8) {
      const __m256i* r = reinterpret_cast<const __m256i*>(mask + 8 * p);
      __m256i v[8];
      for (int k = 0; k < 8; ++k) v[k] = _mm256_loadu_si256(r + k);
      const __m256i any = _mm256_or_si256(_mm256_or_si256(_mm256_or_si256(v[0], v[1]), _mm256_or_si256(v[2], v[3])),
                                          _mm256_or_si256(_mm256_or_si256(v[4], v[5]), _mm256_or_si256(v[6], v[7])));
      if (_mm256_testz_si256(any, any)) {  // +0 everywhere (-0 and NaN have bits set and take the path below)
        _mm256_storeu_si256(reinterpret_cast<__m256i*>(bits + p), zero);
        continue;
      }
      for (int k = 0; k < 8; ++k) {
        const unsigned z = (unsigned)_mm256_movemask_ps(_mm256_castsi256_ps(_mm256_cmpeq_epi32(_mm256_slli_epi32(v[k], 1), zero)));
        const unsigned e1 = (unsigned)_mm256_movemask_ps(_mm256_castsi256_ps(_mm256_cmpeq_epi32(v[k], one)));
        const unsigned m = ~z & 0xFFu;
        bad |= m & ~e1;
        bits[p + k] = m;
      }
    }
    for (; p < hi; ++p) {
      const __m256i v = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(mask + 8 * p));
      const unsigned z = (unsigned)_mm256_movemask_ps(_mm256_castsi256_ps(_mm256_cmpeq_epi32(_mm256_slli_epi32(v, 1), zero)));
      const unsigned e1 = (unsigned)_mm256_movemask_ps(_mm256_castsi256_ps(_mm256_cmpeq_epi32(v, one)));
      const unsigned m = ~z & 0xFFu;
      bad |= m & ~e1;
      bits[p] = m;
    }
    return bad != 0;
  }
  static bool pack(const float* mask, uint32_t* bits, int oc, size_t lo, size_t hi) {
    bool bad = false;
    const uint32_t* w = reinterpret_cast<const uint32_t*>(mask);
    if (oc == 8 && __builtin_cpu_supports("avx2")) return pack8_avx2(mask, bits, lo, hi);
    if (oc == 8) {  // 32 bytes per pixel, all-zero rows (background) leave after four 64-bit tests
      const uint64_t* q = reinterpret_cast<const uint64_t*>(mask);
      for (size_t p = lo; p < hi; ++p) {
        const uint64_t a = q[4 * p], b = q[4 * p + 1], c = q[4 * p + 2], e = q[4 * p + 3];
        uint32_t m = 0;
        if ((a | b | c | e) != 0) {
          for (int k = 0; k < 8; ++k) {
            const uint32_t v = w[8 * p + k];
            if ((v << 1) != 0u) {
              m |= 1u << k;
              bad |= v != 0x3F800000u;
            }
          }
        }
        bits[p] = m;
      }
      return bad;
    }
    for (size_t p = lo; p < hi; ++p) {
      uint32_t m = 0;
      for (int k = 0; k < oc; ++k) {
        const uint32_t v = w[p * oc + k];
        if ((v << 1) != 0u) {
          m |= 1u << k;
          bad |= v != 0x3F800000u;
        }
      }
      bits[p] = m;
    }
    return bad;
  }

  int n_;
  std::vector<std::thread> workers_;
  std::mutex m_;
  std::condition_variable cv_, cv_done_;
  bool quit_ = false;
  long long epoch_ = 0;
  std::shared_ptr<Job> job_;
};
}  // namespace

// Read-back slot of one call: the loop state, the statistics and the events of a call live in their own slot of a ring,
// so that asynchronous callers can queue calls back to back and collect them later (casa_sync / casa_get_timing).
struct CallSlot {
  int* ctrl = nullptr;                   // CTRL_WORDS ints, page-locked
  unsigned long long* stats = nullptr;   // 4 words, page-locked
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_round = nullptr;
  int timed = 0;
  int64_t base_launches = 0, round_launches = 0;
};
constexpr int kCallSlots = 256;
constexpr int kMaxLanes = 4;

struct casa_handle {
  int device = 0;
  int sm_count = 148;
  void* ws_mem = nullptr;
  size_t ws_bytes = 0;
  void* io_mem = nullptr;  // device staging of the host-buffer entry points
  size_t io_bytes = 0;
  void* metric_mem = nullptr;  // scratch of casa_pose_errors
  size_t metric_bytes = 0;
  int* pinned = nullptr;   // CTRL_WORDS ints, page-locked
  cudaStream_t own_stream = nullptr, copy_stream = nullptr;
  cudaEvent_t part_ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_round = nullptr;
  uint32_t last_status = 0;
  int64_t last_launches = 0;
  int timing = 0;
  double score_ms = 0.0;
  int64_t score_launches = 0;
  uint64_t stats[4] = {0, 0, 0, 0};
  int64_t rounds_total = 0, launches_total = 0;
  unsigned long long* pinned_stats = nullptr;  // 4 words, page-locked
  int score_occ = 0, score_occ_narrow = 0;  // resident k_score blocks per SM (8 / 4 hypotheses per lane)
  int fused_occ = 0;              // resident k_ls_fused blocks per SM (persistent grid of the LS forward call)
  int classify_static_smem[2] = {-1, -1};  // static shared memory of k_ls_classify<9> / <0> (queried once)
  int use_graph = 1;
  // keypoint all-gather (NCCL, resolved with dlopen: the library itself does not link against it)
  void* comm = nullptr;           // ncclComm_t
  int comm_owned = 0, comm_rank = 0, comm_world = 1;
  cudaStream_t gather_stream = nullptr;
  cudaEvent_t gather_after[8] = {}, gather_done[8] = {};
  void* deferred_list = nullptr;  // std::vector<DeferredDelete>*: consumed DLPack capsules whose deleters are pending
  MaskPacker* packer = nullptr;   // host threads of casa_ransac_vote_host
  uint32_t* bits_host = nullptr;  // page-locked staging of the packed membership words
  size_t bits_host_bytes = 0;
  CallSlot slots[kCallSlots];
  char* slot_mem = nullptr;       // page-locked backing store of the slots' read-back buffers
  int64_t slot_head = 0, slot_tail = 0;  // calls issued / calls collected (pending = head - tail)
  cudaStream_t last_stream = nullptr;
  const void* clean_ctrl = nullptr;  // address of the ctrl / stats words the previous vote's graph left zeroed (layouts move them)
  int async_mode = 0;             // 1: casa_ransac_vote returns without waiting for the loop state (casa_sync collects errors)
                                  // n = 2..4: as 1, and consecutive votes rotate over n lanes (below)
  // Lanes (casa_set_async(h, n)): n sub-handles with their own workspace and stream.  Vote i runs on lane i % n behind
  // an event recorded on the caller's stream, so the compaction / hypothesis kernels and the refinements of n votes
  // overlap (they are latency-bound; the k_score launches run back to back, each filling the GPU on its own).  Outputs
  // are ordered on a caller's stream by casa_join(), on the host by casa_sync().
  casa_handle* lane[kMaxLanes] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t lane_fork[kMaxLanes] = {nullptr, nullptr, nullptr, nullptr}, lane_done[kMaxLanes] = {nullptr, nullptr, nullptr, nullptr};
  int lane_pending[kMaxLanes] = {0, 0, 0, 0};
  int lane_next = 0, lane_last = -1;
  int is_lane = 0;
  uint32_t* sticky = nullptr;     // device word: OR of the status words of every call since the last casa_sync
  uint32_t* pinned_sticky = nullptr;
  std::vector<struct casa_graph*> graphs;
  // Pipelined host entry (casa_ransac_vote_host_async): kHostDepth driver threads, each with a sub-handle of its own
  // (workspaces, lanes, staging buffers), run casa_ransac_vote_host for consecutive tickets; they share this handle's
  // packer threads behind `pack_gate`, so the host packs call i+1 while the GPU finishes call i.
  struct HostDriver* driver[4] = {nullptr, nullptr, nullptr, nullptr};
  int host_depth = 0;             // drivers in use (fixed at the first asynchronous call)
  int64_t host_ticket = 0;        // tickets issued
  int host_first_rc = 0;          // first error of a call whose ticket was never waited for
  char host_first_err[512] = "";
  casa_handle* host_parent = nullptr;  // set in a driver's sub-handle: owner of the shared packer
  cudaEvent_t ev_block = nullptr;      // driver sub-handles: blocking-sync event (a waiting driver thread sleeps instead of
                                       // spinning on a core the packer threads need)
  std::mutex pack_gate;           // one call at a time uses the packer threads
};

struct casa_graph {
  uint64_t key = 0;
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  std::vector<cudaGraphNode_t> knodes;  // kernel nodes in list order (top level and WHILE body alike)
  cudaGraphConditionalHandle cond = 0;  // condition of the graph's WHILE node (0: the list has no loop)
  cudaGraphNode_t ev0_node = nullptr, ev1_node = nullptr, evr_node = nullptr, ctrl_node = nullptr, stats_node = nullptr;
  std::vector<std::vector<char>> last_args;  // argument bytes each kernel node currently holds: unchanged nodes are not patched
  const void* last_slot = nullptr;           // read-back slot the event / copy nodes currently point at
};

// ------------------------------------------------------------------------------------------------ NCCL (dlopen)
// Only the final [b, oc, vn, 2] keypoints of every rank are exchanged (SURVEY.md 8e).  NCCL is resolved at run time
// so that the library loads on machines without it; in a process that already carries an NCCL (PyTorch's,
// TensorFlow's) dlopen returns that copy.
namespace {
struct NcclId128 {  // ncclUniqueId: 128 opaque bytes, passed by value
  char b[128];
};
struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, NcclId128, int) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
NcclApi g_nccl;

int nccl_load() {
  if (g_nccl.lib) return CASA_OK;
  const char* names[] = {getenv("CASA_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};  // an NCCL outside the loader's path
  void* lib = nullptr;
  for (const char* n : names)
    if (n && !lib) lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
  if (!lib) return fail(CASA_ERR_INVALID, "NCCL not found (dlopen libnccl.so.2: %s); set CASA_NCCL_LIB", dlerror());
  g_nccl.GetUniqueId = (decltype(g_nccl.GetUniqueId))dlsym(lib, "ncclGetUniqueId");
  g_nccl.CommInitRank = (decltype(g_nccl.CommInitRank))dlsym(lib, "ncclCommInitRank");
  g_nccl.CommDestroy = (decltype(g_nccl.CommDestroy))dlsym(lib, "ncclCommDestroy");
  g_nccl.AllGather = (decltype(g_nccl.AllGather))dlsym(lib, "ncclAllGather");
  g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))dlsym(lib, "ncclGetErrorString");
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.CommDestroy || !g_nccl.AllGather)
    return fail(CASA_ERR_INVALID, "NCCL library lacks a required symbol");
  g_nccl.lib = lib;
  return CASA_OK;
}

#define NCCL_TRY(expr)                                                                                     \
  do {                                                                                                     \
    const int r__ = (expr);                                                                                \
    if (r__ != 0)                                                                                          \
      return fail(CASA_ERR_CUDA, "%s failed: %s", #expr, g_nccl.GetErrorString ? g_nccl.GetErrorString(r__) : "NCCL error"); \
  } while (0)
}  // namespace

struct casa_handle;
static void comm_release(casa_handle* h);
static void run_deferred(casa_handle* h, bool wait);
namespace {
struct DeferredDelete;
}
static std::vector<DeferredDelete>& deferred(casa_handle* h);

extern "C" int casa_version(void) { return CASA_VERSION; }
extern "C" const char* casa_last_error(void) { return g_err; }

extern "C" int casa_create(int device, casa_handle** out) {
  if (!out) return fail(CASA_ERR_INVALID, "casa_create: out is NULL");
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) return fail(CASA_ERR_NODEVICE, "casa_create: no CUDA device");
  if (device < 0) CUDA_TRY(cudaGetDevice(&device));
  if (device >= n) return fail(CASA_ERR_INVALID, "casa_create: device %d out of range (%d devices)", device, n);
  CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail(CASA_ERR_NODEVICE, "casa_create: device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
  casa_handle* h = new casa_handle();
  h->device = device;
  h->sm_count = prop.multiProcessorCount;
  CUDA_TRY(cudaHostAlloc((void**)&h->pinned, CTRL_WORDS * sizeof(int), cudaHostAllocDefault));
  CUDA_TRY(cudaHostAlloc((void**)&h->pinned_stats, 4 * sizeof(unsigned long long), cudaHostAllocDefault));
  CUDA_TRY(cudaHostAlloc((void**)&h->pinned_sticky, sizeof(uint32_t), cudaHostAllocDefault));
  CUDA_TRY(cudaMalloc((void**)&h->sticky, sizeof(uint32_t)));
  CUDA_TRY(cudaMemset(h->sticky, 0, sizeof(uint32_t)));
  CUDA_TRY(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
  CUDA_TRY(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
  for (int i = 0; i < 8; ++i) CUDA_TRY(cudaEventCreateWithFlags(&h->part_ev[i], cudaEventDisableTiming));
  CUDA_TRY(cudaEventCreate(&h->ev0));
  CUDA_TRY(cudaEventCreate(&h->ev1));
  CUDA_TRY(cudaEventCreateWithFlags(&h->ev_round, cudaEventDisableTiming));
  CUDA_TRY(cudaHostAlloc((void**)&h->slot_mem, (size_t)kCallSlots * 64, cudaHostAllocDefault));
  for (int i = 0; i < kCallSlots; ++i) {
    CallSlot& c = h->slots[i];
    c.ctrl = (int*)(h->slot_mem + (size_t)i * 64);
    c.stats = (unsigned long long*)(h->slot_mem + (size_t)i * 64 + 32);
    CUDA_TRY(cudaEventCreate(&c.ev0));
    CUDA_TRY(cudaEventCreate(&c.ev1));
    CUDA_TRY(cudaEventCreateWithFlags(&c.ev_round, cudaEventDisableTiming));
  }
  // direct launches stay selectable: LS debug calls need run_direct anyway, and it is the form a debugger can step
  if (getenv("CASA_NO_GRAPH")) h->use_graph = 0;
  *out = h;
  return CASA_OK;
}

static void host_drivers_destroy(casa_handle* h);
static int host_drain(casa_handle* h);

extern "C" int casa_destroy(casa_handle* h) {
  if (!h) return CASA_OK;
  cudaSetDevice(h->device);
  host_drivers_destroy(h);  // pipelined host calls: wait for them, stop the driver threads
  for (casa_graph* g : h->graphs) {
    if (g->exec) cudaGraphExecDestroy(g->exec);
    if (g->graph) cudaGraphDestroy(g->graph);
    delete g;
  }
  for (int i = 0; i < kMaxLanes; ++i) {
    if (h->lane[i]) casa_destroy(h->lane[i]);
    if (h->lane_fork[i]) cudaEventDestroy(h->lane_fork[i]);
    if (h->lane_done[i]) cudaEventDestroy(h->lane_done[i]);
  }
  cudaSetDevice(h->device);
  delete h->packer;
  if (h->bits_host) cudaFreeHost(h->bits_host);
  if (h->deferred_list) {
    run_deferred(h, true);
    delete &deferred(h);
  }
  comm_release(h);
  if (h->gather_stream) cudaStreamDestroy(h->gather_stream);
  for (int i = 0; i < 8; ++i) {
    if (h->gather_after[i]) cudaEventDestroy(h->gather_after[i]);
    if (h->gather_done[i]) cudaEventDestroy(h->gather_done[i]);
  }
  if (h->ws_mem) cudaFree(h->ws_mem);
  if (h->io_mem) cudaFree(h->io_mem);
  if (h->metric_mem) cudaFree(h->metric_mem);
  if (h->pinned) cudaFreeHost(h->pinned);
  if (h->pinned_stats) cudaFreeHost(h->pinned_stats);
  if (h->pinned_sticky) cudaFreeHost(h->pinned_sticky);
  if (h->sticky) cudaFree(h->sticky);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  for (int i = 0; i < 8; ++i)
    if (h->part_ev[i]) cudaEventDestroy(h->part_ev[i]);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->ev_round) cudaEventDestroy(h->ev_round);
  if (h->ev_block) cudaEventDestroy(h->ev_block);
  for (int i = 0; i < kCallSlots; ++i) {
    if (h->slots[i].ev0) cudaEventDestroy(h->slots[i].ev0);
    if (h->slots[i].ev1) cudaEventDestroy(h->slots[i].ev1);
    if (h->slots[i].ev_round) cudaEventDestroy(h->slots[i].ev_round);
  }
  if (h->slot_mem) cudaFreeHost(h->slot_mem);
  delete h;
  return CASA_OK;
}

// ------------------------------------------------------------------------------------------------ workspace

namespace {

struct Layout {
  Dims d;
  size_t off_bits, off_tile_cnt, off_pix, off_vdir, off_job_tn0, off_job_tn, off_job_off, off_job_flags,
      off_job_rounds, off_job_done, off_job_selthr, off_win_ratio, off_win_pts, off_hyp_true, off_hyp_filt, off_exact_list,
      off_n_exact, off_counts, off_item_start, off_rtile_start, off_rtile_job, off_rtile_rec, off_ctrl, off_partial, off_stats, total;
};

size_t bump(size_t& cur, size_t bytes) {
  const size_t o = cur;
  cur += (bytes + 255) & ~size_t(255);
  return o;
}


int make_layout(const casa_ransac_params* p, Layout& L, int ls_tile = kRefineTile) {
  if (!p) return fail(CASA_ERR_INVALID, "params is NULL");
  if (p->b < 1 || p->h < 1 || p->w < 1 || p->h > 65535 || p->w > 65535)
    return fail(CASA_ERR_INVALID, "bad shape b=%d h=%d w=%d", p->b, p->h, p->w);
  if (p->oc < 1 || p->oc > 32) return fail(CASA_ERR_INVALID, "oc=%d outside 1..32", p->oc);
  if (p->vn < 1 || p->vn > 16) return fail(CASA_ERR_INVALID, "vn=%d outside 1..16", p->vn);
  if (p->round_hyp_num < 1 || p->round_hyp_num > 4096) return fail(CASA_ERR_INVALID, "round_hyp_num=%d outside 1..4096", p->round_hyp_num);
  if (p->max_iter < 1 || p->max_iter > 64) return fail(CASA_ERR_INVALID, "max_iter=%d outside 1..64", p->max_iter);
  if ((long long)p->b * p->oc > 65535) return fail(CASA_ERR_INVALID, "b*oc=%lld exceeds 65535 jobs per call", (long long)p->b * p->oc);
  if ((long long)p->h * p->w > (1ll << 30)) return fail(CASA_ERR_INVALID, "image too large");
  if ((long long)p->h * p->w / kChunk + 1 >= (1 << 24)) return fail(CASA_ERR_INVALID, "image too large for the work-item encoding");
  if ((long long)p->round_hyp_num * p->max_iter >= (1 << 24)) return fail(CASA_ERR_INVALID, "hn*max_iter must stay below 2^24");
  Dims& d = L.d;
  d.b = p->b; d.h = p->h; d.w = p->w; d.oc = p->oc; d.vn = p->vn; d.hn = p->round_hyp_num; d.max_iter = p->max_iter;
  d.hw = p->h * p->w;
  d.J = p->b * p->oc;
  d.nct = (d.hw + kCountTile - 1) / kCountTile;
  d.cap = p->pix_capacity > 0 ? p->pix_capacity : d.hw;
  const long long rtiles = (long long)d.b * ((long long)d.cap / ls_tile + d.oc + 1);  // ls_tile <= kVoteTile: covers the voting path too
  if (rtiles > (1ll << 30) || (long long)d.b * ((long long)d.cap / kChunk + d.oc + 1) * d.vn > (1ll << 30))
    return fail(CASA_ERR_INVALID, "too many work items");
  d.max_rtiles = (int)rtiles;
  d.rtile = kVoteTile;
  d.image_offset = p->image_offset;
  d.seed_lo = (uint32_t)(p->seed & 0xFFFFFFFFull);
  d.seed_hi = (uint32_t)(p->seed >> 32);
  d.min_num = p->min_num; d.max_num = p->max_num; d.confidence = p->confidence;
  d.force_exact = p->force_exact;
  d.vpc = p->vertex_per_class ? d.oc : 1;
  size_t cur = 0;
  const size_t J = d.J, jv = J * d.vn, jvh = jv * d.hn;
  L.off_bits = bump(cur, (size_t)d.b * d.hw * 4);
  L.off_tile_cnt = bump(cur, J * d.nct * 4);
  L.off_pix = bump(cur, (size_t)d.b * d.cap * 4);
  L.off_vdir = bump(cur, (size_t)d.b * d.cap * d.vn * 8);
  L.off_job_tn0 = bump(cur, J * 4);
  L.off_job_tn = bump(cur, J * 4);
  L.off_job_off = bump(cur, J * 4);
  L.off_job_flags = bump(cur, J * 4);
  L.off_job_rounds = bump(cur, J * 4);
  L.off_job_done = bump(cur, J * 4);
  L.off_job_selthr = bump(cur, J * 4);
  L.off_win_ratio = bump(cur, jv * 4);
  L.off_win_pts = bump(cur, jv * 8);
  L.off_hyp_true = bump(cur, jvh * 8);
  L.off_hyp_filt = bump(cur, jvh * 8);
  L.off_exact_list = bump(cur, jvh * 4);
  L.off_n_exact = bump(cur, jv * 4);
  L.off_counts = bump(cur, jvh * 4);
  L.off_item_start = bump(cur, (J + 1) * 4);
  L.off_rtile_start = bump(cur, (J + 1) * 4);
  L.off_rtile_job = bump(cur, (size_t)d.max_rtiles * 4);
  L.off_rtile_rec = bump(cur, (size_t)d.max_rtiles * 16);
  L.off_ctrl = bump(cur, CTRL_WORDS * 4);
  L.off_stats = bump(cur, 4 * 8);  // directly behind ctrl: one memset node clears both (run_graph: STEP_CLEAR)
  L.off_partial = bump(cur, (size_t)(d.max_rtiles > d.J ? d.max_rtiles : d.J) * d.vn * 5 * 8);
  L.total = cur;
  return CASA_OK;
}

WS make_ws(const Layout& L, void* base, bool stats) {
  char* b = (char*)base;
  WS w;
  w.bits = (uint32_t*)(b + L.off_bits);
  w.tile_cnt = (int*)(b + L.off_tile_cnt);
  w.pix = (uint32_t*)(b + L.off_pix);
  w.vdir = (float2*)(b + L.off_vdir);
  w.job_tn0 = (int*)(b + L.off_job_tn0);
  w.job_tn = (int*)(b + L.off_job_tn);
  w.job_off = (int*)(b + L.off_job_off);
  w.job_flags = (int*)(b + L.off_job_flags);
  w.job_rounds = (int*)(b + L.off_job_rounds);
  w.job_done = (int*)(b + L.off_job_done);
  w.job_selthr = (float*)(b + L.off_job_selthr);
  w.win_ratio = (float*)(b + L.off_win_ratio);
  w.win_pts = (float2*)(b + L.off_win_pts);
  w.hyp_true = (float2*)(b + L.off_hyp_true);
  w.hyp_filt = (float2*)(b + L.off_hyp_filt);
  w.exact_list = (int*)(b + L.off_exact_list);
  w.n_exact = (int*)(b + L.off_n_exact);
  w.counts = (int*)(b + L.off_counts);
  w.item_start = (int*)(b + L.off_item_start);
  w.rtile_start = (int*)(b + L.off_rtile_start);
  w.rtile_job = (int*)(b + L.off_rtile_job);
  w.rtile_rec = (int4*)(b + L.off_rtile_rec);
  w.ctrl = (int*)(b + L.off_ctrl);
  w.partial = (double*)(b + L.off_partial);
  w.stats = stats ? (unsigned long long*)(b + L.off_stats) : nullptr;
  return w;
}

int ensure(void** mem, size_t* have, size_t need) {
  if (*have >= need) return CASA_OK;
  if (*mem) {
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaFree(*mem));
    *mem = nullptr;
    *have = 0;
  }
  CUDA_TRY(cudaMalloc(mem, need));
  *have = need;
  return CASA_OK;
}

}  // namespace

extern "C" size_t casa_ransac_workspace_bytes(const casa_ransac_params* p) {
  Layout L;
  if (make_layout(p, L) != CASA_OK) return 0;
  return L.total;
}

// ------------------------------------------------------------------------------------------------ ransac vote

// ---- launch lists: the kernel sequence of a round is described once and either launched directly or replayed
// ---- as a CUDA graph whose kernel-node parameters are patched per call (CUDA graphs instead of launch gaps).
namespace {

enum StepKind { STEP_KERNEL, STEP_EV0, STEP_EV1, STEP_READBACK, STEP_CLEAR, STEP_WHILE_BEGIN, STEP_WHILE_END };

struct Step {
  StepKind kind = STEP_KERNEL;
  const void* func = nullptr;
  dim3 grid, block;
  size_t smem = 0;
  alignas(16) char buf[704];
  size_t off[8];
  size_t used = 0;
  int n = 0;
  int cond_arg = -1;  // index of the argument that receives the graph's WHILE condition handle (k_update)
  // graph topology: 0 = main chain; 1 = opens a side branch off the main chain's last node; 2 = continues the side
  // branch.  join: this main-chain step also waits for the side branch (which ends there).
  // Two side branches can be open at a time (slot 0 and slot 1).
  int side = 0;
  int slot = 0;
  bool join = false, join1 = false;
  Step& on_side(int v, int sl = 0) {
    side = v;
    slot = sl;
    return *this;
  }
  Step& joins(int sl = 0) {
    (sl ? join1 : join) = true;
    return *this;
  }
  template <class T>
  Step& arg(const T& v) {
    used = (used + alignof(T) - 1) & ~(alignof(T) - 1);
    memcpy(buf + used, &v, sizeof(T));
    off[n++] = used;
    used += sizeof(T);
    return *this;
  }
  Step& cond() {  // placeholder for the condition handle, filled in by run_graph / run_direct
    cond_arg = n;
    return arg((unsigned long long)0);
  }
  void set_cond(unsigned long long v) {
    if (cond_arg >= 0) memcpy(buf + off[cond_arg], &v, sizeof(v));
  }
  void ptrs(void** out) {
    for (int i = 0; i < n; ++i) out[i] = buf + off[i];
  }
};

Step kstep(const void* func, dim3 grid, dim3 block, size_t smem = 0) {
  Step s;
  s.func = func;
  s.grid = grid;
  s.block = block;
  s.smem = smem;
  return s;
}

Step special(StepKind k, int side = 0) {
  Step s;
  s.kind = k;
  s.side = side;
  return s;
}

uint64_t fnv(uint64_t hsh, const void* p, size_t n) {
  const unsigned char* b = (const unsigned char*)p;
  for (size_t i = 0; i < n; ++i) hsh = (hsh ^ b[i]) * 1099511628211ull;
  return hsh;
}

}  // namespace

static int launch_step(Step& s, cudaStream_t st) {
  void* args[8];
  s.ptrs(args);
  CUDA_TRY(cudaLaunchKernel(s.func, s.grid, s.block, args, s.smem, st));
  return CASA_OK;
}

// Direct launches (CASA_NO_GRAPH=1; debugging and the sanitizer runs): the WHILE section is driven from the host,
// one 32-byte read-back per round — the reference's data-dependent `while` (:318) as the first version ran it.
static int run_direct(casa_handle* h, std::vector<Step>& steps, const WS& ws, cudaStream_t st, CallSlot* slot = nullptr) {
  for (size_t i = 0; i < steps.size(); ++i) {
    Step& s = steps[i];
    switch (s.kind) {
      case STEP_KERNEL: {
        int rc = launch_step(s, st);
        if (rc) return rc;
        break;
      }
      case STEP_CLEAR:
        CUDA_TRY(cudaMemsetAsync(ws.ctrl, 0, CTRL_WORDS * sizeof(int), st));
        CUDA_TRY(cudaMemsetAsync(ws.stats, 0, 4 * sizeof(unsigned long long), st));
        break;
      case STEP_EV0: CUDA_TRY(cudaEventRecord(slot->ev0, st)); break;
      case STEP_EV1: CUDA_TRY(cudaEventRecord(slot->ev1, st)); break;
      case STEP_READBACK:
        CUDA_TRY(cudaMemcpyAsync(slot->ctrl, ws.ctrl, CTRL_WORDS * sizeof(int), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync(slot->stats, ws.stats, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaEventRecord(slot->ev_round, st));
        break;
      case STEP_WHILE_BEGIN: {
        size_t end = i + 1;
        while (end < steps.size() && steps[end].kind != STEP_WHILE_END) ++end;
        for (;;) {
          CUDA_TRY(cudaMemcpyAsync(h->pinned, ws.ctrl, CTRL_WORDS * sizeof(int), cudaMemcpyDeviceToHost, st));
          CUDA_TRY(cudaStreamSynchronize(st));
          if (h->pinned[CTRL_NACTIVE] == 0) break;
          for (size_t k = i + 1; k < end; ++k) {
            int rc = launch_step(steps[k], st);
            if (rc) return rc;
          }
        }
        i = end;
        break;
      }
      case STEP_WHILE_END: break;
    }
  }
  return CASA_OK;
}

// The whole call as ONE CUDA graph: kernel nodes, the clear / read-back nodes, and a conditional WHILE node whose
// body (the RANSAC rounds after the first) repeats on the device until k_update sets the condition to 0.  Graphs are
// cached per launch shape; per call only the kernel-node parameters are patched (cudaGraphExecKernelNodeSetParams
// also reaches the nodes of the WHILE body).
static int run_graph(casa_handle* h, std::vector<Step>& steps, const WS& ws, cudaStream_t st, CallSlot* slot = nullptr) {
  uint64_t key = 1469598103934665603ull;
  for (const Step& s : steps) {
    key = fnv(key, &s.kind, sizeof(s.kind));
    key = fnv(key, &s.func, sizeof(s.func));
    key = fnv(key, &s.grid, sizeof(s.grid));
    key = fnv(key, &s.block, sizeof(s.block));
    key = fnv(key, &s.smem, sizeof(s.smem));
  }
  key = fnv(key, &ws.ctrl, sizeof(ws.ctrl));  // the clear / read-back nodes carry workspace addresses
  casa_graph* g = nullptr;
  for (casa_graph* c : h->graphs)
    if (c->key == key) g = c;
  auto kparams = [](Step& s, void** args, cudaKernelNodeParams& kp) {
    s.ptrs(args);
    memset(&kp, 0, sizeof(kp));
    kp.func = (void*)s.func;
    kp.gridDim = s.grid;
    kp.blockDim = s.block;
    kp.sharedMemBytes = (unsigned)s.smem;
    kp.kernelParams = args;
  };
  if (!g) {
    g = new casa_graph();
    g->key = key;
    CUDA_TRY(cudaGraphCreate(&g->graph, 0));
    bool has_loop = false;
    for (const Step& s : steps) has_loop |= s.kind == STEP_WHILE_BEGIN;
    if (has_loop) CUDA_TRY(cudaGraphConditionalHandleCreate(&g->cond, g->graph, 0, cudaGraphCondAssignDefault));
    cudaGraph_t cur = g->graph;
    cudaGraphNode_t prev = nullptr, side_prev[2] = {nullptr, nullptr}, loop_node = nullptr;
    for (Step& s : steps) {
      cudaGraphNode_t node = nullptr;
      cudaGraphNode_t deps[3];
      size_t nd = 0;
      if (s.side == 2) {
        if (side_prev[s.slot]) deps[nd++] = side_prev[s.slot];
      } else {
        if (prev) deps[nd++] = prev;
        if (s.side == 0 && s.join && side_prev[0]) deps[nd++] = side_prev[0];
        if (s.side == 0 && s.join1 && side_prev[1]) deps[nd++] = side_prev[1];
      }
      cudaGraphNode_t* dep = nd ? deps : nullptr;
      switch (s.kind) {
        case STEP_KERNEL: {
          s.set_cond((unsigned long long)g->cond);
          void* args[8];
          cudaKernelNodeParams kp;
          kparams(s, args, kp);
          CUDA_TRY(cudaGraphAddKernelNode(&node, cur, dep, nd, &kp));
          g->knodes.push_back(node);
          g->last_args.emplace_back(s.buf, s.buf + s.used);
          break;
        }
        case STEP_EV0:
        case STEP_EV1:
          CUDA_TRY(cudaGraphAddEventRecordNode(&node, cur, dep, nd, s.kind == STEP_EV0 ? slot->ev0 : slot->ev1));
          (s.kind == STEP_EV0 ? g->ev0_node : g->ev1_node) = node;
          break;
        case STEP_CLEAR: {  // ctrl and stats are adjacent in the workspace: one memset node
          cudaMemsetParams mp;
          memset(&mp, 0, sizeof(mp));
          mp.dst = ws.ctrl;
          mp.elementSize = 4;
          mp.width = ((char*)ws.stats - (char*)ws.ctrl) / 4 + 8;
          mp.height = 1;
          mp.value = 0;
          CUDA_TRY(cudaGraphAddMemsetNode(&node, cur, dep, nd, &mp));
          break;
        }
        case STEP_READBACK: {
          CUDA_TRY(cudaGraphAddMemcpyNode1D(&node, cur, dep, nd, slot->ctrl, ws.ctrl, CTRL_WORDS * sizeof(int), cudaMemcpyDeviceToHost));
          g->ctrl_node = node;
          cudaGraphNode_t p2 = node;
          CUDA_TRY(cudaGraphAddMemcpyNode1D(&node, cur, &p2, 1, slot->stats, ws.stats, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
          g->stats_node = p2 = node;
          CUDA_TRY(cudaGraphAddEventRecordNode(&node, cur, &p2, 1, slot->ev_round));
          g->evr_node = node;
          break;
        }
        case STEP_WHILE_BEGIN: {
          cudaGraphNodeParams cp = {};
          cp.type = cudaGraphNodeTypeConditional;
          cp.conditional.handle = g->cond;
          cp.conditional.type = cudaGraphCondTypeWhile;
          cp.conditional.size = 1;
          CUDA_TRY(cudaGraphAddNode(&loop_node, cur, dep, nd, &cp));
          cur = cp.conditional.phGraph_out[0];
          prev = nullptr;
          side_prev[0] = side_prev[1] = nullptr;
          continue;
        }
        case STEP_WHILE_END:
          cur = g->graph;
          prev = loop_node;
          side_prev[0] = side_prev[1] = nullptr;
          continue;
      }
      if (s.side == 0) {
        prev = node;
        if (s.join) side_prev[0] = nullptr;
        if (s.join1) side_prev[1] = nullptr;
      } else {
        side_prev[s.slot] = node;
      }
    }
    CUDA_TRY(cudaGraphInstantiate(&g->exec, g->graph, 0));
    g->last_slot = slot;
    if (h->graphs.size() >= 16) {  // tiny cache: drop the oldest shape
      casa_graph* old = h->graphs.front();
      cudaGraphExecDestroy(old->exec);
      cudaGraphDestroy(old->graph);
      delete old;
      h->graphs.erase(h->graphs.begin());
    }
    h->graphs.push_back(g);
  } else {
    size_t k = 0;
    for (Step& s : steps) {
      if (s.kind != STEP_KERNEL) continue;
      s.set_cond((unsigned long long)g->cond);
      std::vector<char>& held = g->last_args[k];
      if (held.size() == s.used && memcmp(held.data(), s.buf, s.used) == 0) {  // same arguments as the node holds
        ++k;
        continue;
      }
      held.assign(s.buf, s.buf + s.used);
      void* args[8];
      cudaKernelNodeParams kp;
      kparams(s, args, kp);
      CUDA_TRY(cudaGraphExecKernelNodeSetParams(g->exec, g->knodes[k++], &kp));
    }
    if (slot && g->last_slot != (const void*)slot) {  // this call's read-back slot
      g->last_slot = slot;
      if (g->ev0_node) CUDA_TRY(cudaGraphExecEventRecordNodeSetEvent(g->exec, g->ev0_node, slot->ev0));
      if (g->ev1_node) CUDA_TRY(cudaGraphExecEventRecordNodeSetEvent(g->exec, g->ev1_node, slot->ev1));
      if (g->evr_node) CUDA_TRY(cudaGraphExecEventRecordNodeSetEvent(g->exec, g->evr_node, slot->ev_round));
      if (g->ctrl_node)
        CUDA_TRY(cudaGraphExecMemcpyNodeSetParams1D(g->exec, g->ctrl_node, slot->ctrl, ws.ctrl, CTRL_WORDS * sizeof(int), cudaMemcpyDeviceToHost));
      if (g->stats_node)
        CUDA_TRY(cudaGraphExecMemcpyNodeSetParams1D(g->exec, g->stats_node, slot->stats, ws.stats, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    }
  }
  CUDA_TRY(cudaGraphLaunch(g->exec, st));
  return CASA_OK;
}

// Collects every call that has been issued but not looked at yet: waits for its loop state (not for its refinement /
// solve), accumulates its statistics and timing into the handle and returns the first error any of them raised.
// A synchronous call collects itself; asynchronous calls are collected by casa_sync / casa_get_timing / when the
// ring of read-back slots is full.
static void reset_totals(casa_handle* h) {
  h->score_ms = 0.0;
  h->score_launches = 0;
  h->rounds_total = 0;
  h->launches_total = 0;
  for (int k = 0; k < 4; ++k) h->stats[k] = 0;
}

struct Collected {  // the calls one collect() took in (lanes included)
  int64_t slots = 0;
  int64_t launches = 0;
  uint32_t status = 0;  // OR of their status words
};

static int collect(casa_handle* h, Collected* got = nullptr) {
  Collected mine;
  if (!got) got = &mine;
  int first_rc = CASA_OK;
  for (int i = 0; i < kMaxLanes; ++i) {  // lanes: their calls are this handle's calls
    casa_handle* s = h->lane[i];
    if (!s) continue;
    Collected lc;
    const int rc = collect(s, &lc);
    if (first_rc == CASA_OK) first_rc = rc;
    h->score_ms += s->score_ms;
    h->score_launches += s->score_launches;
    h->rounds_total += s->rounds_total;
    h->launches_total += s->launches_total;
    for (int k = 0; k < 4; ++k) h->stats[k] += s->stats[k];
    if (lc.slots && i == h->lane_last) {  // the last vote; a pass that finds nothing new keeps what the handle reports
      h->last_status = s->last_status;
      h->last_launches = s->last_launches;
    }
    got->slots += lc.slots;
    got->launches += lc.launches;
    got->status |= lc.status;
    reset_totals(s);
  }
  while (h->slot_tail < h->slot_head) {
    CallSlot& c = h->slots[h->slot_tail % kCallSlots];
    CUDA_TRY(cudaEventSynchronize(c.ev_round));
    ++h->slot_tail;
    const int rounds = c.ctrl[CTRL_ROUND];
    h->score_launches += c.timed ? 1 : 0;
    h->rounds_total += rounds;
    h->last_launches = c.base_launches + (int64_t)(rounds > 1 ? rounds - 1 : 0) * c.round_launches;
    h->launches_total += h->last_launches;
    ++got->slots;
    got->launches += h->last_launches;
    if (c.timed) {
      float ms = 0.f;
      CUDA_TRY(cudaEventElapsedTime(&ms, c.ev0, c.ev1));
      h->score_ms += ms;  // k_score of round 0 (later rounds run inside the WHILE body, which cannot hold event nodes)
    }
    for (int k = 0; k < 4; ++k) h->stats[k] += c.stats[k];
    h->last_status = (uint32_t)c.ctrl[CTRL_STATUS];
    got->status |= h->last_status;
    if (first_rc == CASA_OK) {
      if (h->last_status & CASA_STATUS_PIX_OVERFLOW)
        first_rc = fail(CASA_ERR_WORKSPACE, "pixel lists exceed pix_capacity (mask is not one-hot?); retry with a larger pix_capacity");
      else if (h->last_status & CASA_STATUS_IDX_RANGE)
        first_rc = fail(CASA_ERR_INPUT, "caller-supplied idxs outside [0, tn)");
    }
  }
  return first_rc;
}

// Lanes (casa_set_async(h, n >= 2), the image ranges of casa_ransac_vote_host): the next call runs on sub-handle
// `lane_next` of `n`, on that lane's own stream, behind an event recorded on the caller's stream now (the lane sees
// what the caller queued so far).
static int lane_begin(casa_handle* h, int n, void* stream, casa_handle** sub_out, int* k_out) {
  CUDA_TRY(cudaSetDevice(h->device));
  const int k = h->lane_next % n;
  if (!h->lane[k]) {
    int rcl = casa_create(h->device, &h->lane[k]);
    if (rcl) return rcl;
    h->lane[k]->is_lane = 1;
    h->lane[k]->async_mode = 1;
    CUDA_TRY(cudaEventCreateWithFlags(&h->lane_fork[k], cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&h->lane_done[k], cudaEventDisableTiming));
  }
  casa_handle* sub = h->lane[k];
  sub->timing = h->timing;
  CUDA_TRY(cudaEventRecord(h->lane_fork[k], (cudaStream_t)stream));
  CUDA_TRY(cudaStreamWaitEvent(sub->own_stream, h->lane_fork[k], 0));
  *sub_out = sub;
  *k_out = k;
  return CASA_OK;
}

static int lane_end(casa_handle* h, int k, void* stream) {
  CUDA_TRY(cudaEventRecord(h->lane_done[k], h->lane[k]->own_stream));
  h->lane_pending[k] = 1;
  h->lane_last = k;
  h->lane_next = k + 1;
  h->last_stream = (cudaStream_t)stream;
  return CASA_OK;
}

// How a vote's mask arrives.
enum class MaskForm {
  kOneHot,     // float [b,h,w,oc] one-hot mask (casa_ransac_vote)
  kSeg,        // float [b,h,w,1+oc] segmentation scores, arg-max on the device (casa_ransac_vote_seg)
  kPackedBits  // u32 [b,h,w] membership words packed on the host (casa_ransac_vote_host)
};

// The inputs and outputs of one vote.
struct VoteInput {
  const void* mask = nullptr;
  MaskForm form = MaskForm::kOneHot;
  const float* vertex = nullptr;
  bool vertex_mapped = false;  // the field is mapped host memory: k_gather_dirs reads it over PCIe, not k_place
  int not_binary = 0;          // kPackedBits: the host packer saw a mask value other than 0 / 1
  const int32_t* idxs = nullptr;
  const float* selection = nullptr;
  float* out = nullptr;
};

// Builds the launch list of one vote and launches it on `st` with `h`'s workspace, into the next read-back slot of
// `h` (collect() reads the slot back).  Waits for the host only when that ring of slots is full.
static int vote_enqueue(casa_handle* h, const casa_ransac_params* p, const VoteInput& in, const casa_ransac_debug* debug,
                        cudaStream_t st) {
  Layout L;
  int rc = make_layout(p, L);
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  if (h->ws_bytes < L.total) h->clean_ctrl = nullptr;
  rc = ensure(&h->ws_mem, &h->ws_bytes, L.total);
  if (rc) return rc;
  if (h->slot_head - h->slot_tail >= kCallSlots) {  // the ring of read-back slots is full: collect the queued calls
    rc = collect(h);
    if (rc) return rc;
  }
  CallSlot* slot = &h->slots[h->slot_head % kCallSlots];
  h->last_stream = st;
  casa_ransac_debug dbg;
  memset(&dbg, 0, sizeof(dbg));
  if (debug) dbg = *debug;
  const Dims& d = L.d;
  WS ws = make_ws(L, h->ws_mem, true);
  const FilterConsts fc = filter_consts(p->inlier_thresh, p->force_exact);

  // debug copy of the pixel lists takes the whole [b][cap] buffer: define the unused tail (debug calls only)
  if (dbg.pix) CUDA_TRY(cudaMemsetAsync(ws.pix, 0, (size_t)d.b * d.cap * 4, st));
  ScoreArgs sa;
  sa.ws = ws;
  sa.d = d;
  sa.fc = fc;
  sa.one = 1u;
  if (h->score_occ == 0) {
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&h->score_occ, k_score<kHypPerLaneWide>, kScoreThreads, 0));
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&h->score_occ_narrow, k_score<kHypPerLaneNarrow>, kScoreThreads, 0));
    if (h->score_occ < 1 || h->score_occ_narrow < 1) return fail(CASA_ERR_INVALID, "scoring kernel does not fit");
    // The kernel is compiled for two resident blocks per SM (113 registers: ransac.cuh).  With the four-block build of
    // the first half of round 2 (64 registers) votes on lanes ran three blocks per SM and left the fourth slot to
    // the neighbouring votes' short kernels (1-2 % per step: profiles/r02_lanes_overlap.txt).
    const int cap = h->is_lane ? 3 : h->score_occ;
    if (cap < h->score_occ) h->score_occ = cap;
    if (cap < h->score_occ_narrow) h->score_occ_narrow = cap;
  }
  const bool narrow = score_hpl(d.hn) == kHypPerLaneNarrow;
  const void* score_fn = narrow ? (const void*)k_score<kHypPerLaneNarrow> : (const void*)k_score<kHypPerLaneWide>;
  const int score_occ = narrow ? h->score_occ_narrow : h->score_occ;
  const int refine_gx = d.max_rtiles < h->sm_count * 4 ? d.max_rtiles : h->sm_count * 4;
  const int gather_gx = (d.cap + 255) / 256 < 24 ? (d.cap + 255) / 256 : 24;
  const int vec4 = ((((size_t)d.hw * d.oc) & 3) == 0) && ((((uintptr_t)in.mask) & 15) == 0);
  const int plan_threads = d.J > 256 ? 1024 : 256;

  // The launch list of the whole call.  Round 0 is spelled out (it carries the timing events, which a WHILE body
  // may not hold); rounds >= 1 are the body of a device-driven WHILE (k_update publishes the round index and the
  // condition), entered only when some job has not met the stop test (:344-347).  Refinement and solve run once,
  // after the loop; the 32-byte loop state and the statistics are read back in front of them, so a synchronous
  // caller learns the status while the GPU is still busy.
  std::vector<Step> steps;
  steps.reserve(32);
  int64_t base_launches = 0, round_launches = 0;
  // ctrl / stats are clean when the previous call on this workspace was a vote (its graph clears them at its end);
  // after anything else (first call, re-allocation, the LS layer) they are cleared in front of the graph.
  if (h->clean_ctrl != (const void*)ws.ctrl) {
    CUDA_TRY(cudaMemsetAsync(ws.ctrl, 0, CTRL_WORDS * sizeof(int), st));
    CUDA_TRY(cudaMemsetAsync(ws.stats, 0, 4 * sizeof(unsigned long long), st));
  }
  if (in.form == MaskForm::kPackedBits)  // bit 30 of the flag: not binary
    steps.push_back(kstep((const void*)k_bits_in, dim3(d.nct, d.b), 256).arg((const uint32_t*)in.mask).arg(ws).arg(d).arg(in.not_binary));
  else if (in.form == MaskForm::kSeg)
    steps.push_back(kstep((const void*)k_seg_bits, dim3(d.nct, d.b), 256).arg((const float*)in.mask).arg(ws).arg(d));
  else
    steps.push_back(kstep((const void*)k_mask_bits, dim3(d.nct, d.b), 256).arg((const float*)in.mask).arg(ws).arg(d).arg(vec4));
  // k_place gathers the directions while it scatters the pixels, unless the field lives in mapped host memory (the
  // host entry point: k_gather_dirs reads full lines over PCIe) or is not 8-byte aligned; jobs above max_num are
  // gathered after the cap filter
  const int fuse_gather = (!in.vertex_mapped && (((uintptr_t)in.vertex) & 7) == 0) ? 1 : 0;
  const bool may_cap = (float)d.hw > p->max_num;
  steps.push_back(kstep(d.vn == 9 ? (const void*)k_place<9> : (const void*)k_place<0>, dim3((d.nct + kPlaceSub - 1) / kPlaceSub, d.b), 256).arg(in.vertex).arg(ws).arg(d).arg(fuse_gather));
  if (may_cap) steps.push_back(kstep((const void*)k_cap_filter, d.J, 1024).arg(ws).arg(d).arg(in.selection));
  // round 0's plan (work items, refinement tiles) only needs the job table: it runs beside the direction gather and
  // k_hypgen (side branch in slot 1, joined by k_score)
  steps.push_back(kstep((const void*)k_plan, 1, plan_threads).arg(ws).arg(d).arg((int)0).on_side(1, 1));
  if (!fuse_gather || may_cap)
    steps.push_back(kstep(d.vn == 9 ? (const void*)k_gather_dirs<18> : (const void*)k_gather_dirs<0>, dim3(gather_gx, d.J), 256)
                        .arg(in.vertex).arg(ws).arg(d).arg(fuse_gather));
  for (int part = 0; part < 2; ++part) {  // part 0: round 0; part 1: the WHILE body (rnd = -1: read ctrl[CTRL_ROUND])
    const int rnd = part == 0 ? 0 : -1;
    if (part == 1) {
      if (d.max_iter < 2) break;
      steps.push_back(special(STEP_WHILE_BEGIN));
      steps.push_back(kstep((const void*)k_plan, 1, plan_threads).arg(ws).arg(d).arg(rnd));
    }
    const size_t n0 = steps.size();
    Step hg = kstep((const void*)k_hypgen, dim3((d.hn * d.vn + 255) / 256, d.J), 256).arg(ws).arg(d).arg(fc).arg(in.idxs).arg(rnd).arg(dbg.hyps);
    steps.push_back(hg);
    // the timing events hang off the chain as leaves: ev0 fires when k_hypgen is done, ev1 when k_score is done
    if (part == 0 && h->timing) steps.push_back(special(STEP_EV0, 1));
    {
      Step sc = kstep(score_fn, h->sm_count * score_occ, kScoreThreads).arg(sa);
      if (part == 0) sc.joins(1);
      steps.push_back(sc);
    }
    if (part == 0 && h->timing) steps.push_back(special(STEP_EV1, 1));
    steps.push_back(kstep((const void*)k_update, d.J, 32 * d.vn).arg(ws).arg(d).arg(rnd).arg(dbg).cond().arg(h->sticky));
    if (part == 1) {
      for (size_t k = n0 - 1; k < steps.size(); ++k) round_launches += steps[k].kind == STEP_KERNEL;
      steps.push_back(special(STEP_WHILE_END));
    }
  }
  // the read-back of the loop state (and the clearing of ctrl / stats for the next call) is a side branch: refinement
  // and solve do not wait for the copy engine
  steps.push_back(special(STEP_READBACK, 1));
  steps.push_back(special(STEP_CLEAR, 2));
  steps.push_back(kstep((const void*)k_refine_solve, dim3(refine_gx, d.vn), kRefineThreads).arg(ws).arg(d).arg(fc).arg(in.out).arg(dbg));
  for (const Step& s2 : steps) base_launches += s2.kind == STEP_KERNEL;
  base_launches -= round_launches;  // the body's kernels are counted per executed round below
  slot->timed = h->timing;
  slot->base_launches = base_launches;
  slot->round_launches = round_launches;
  rc = h->use_graph ? run_graph(h, steps, ws, st, slot) : run_direct(h, steps, ws, st, slot);
  if (rc) return rc;
  ++h->slot_head;
  h->clean_ctrl = ws.ctrl;
  CUDA_TRY(cudaGetLastError());
  if (dbg.pix) CUDA_TRY(cudaMemcpyAsync(dbg.pix, ws.pix, (size_t)d.b * d.cap * 4, cudaMemcpyDeviceToDevice, st));
  return CASA_OK;
}

// A vote of the device entry points: on the next lane when the handle rotates over lanes (casa_set_async(h, n >= 2))
// and no debug outputs are asked for, otherwise on `stream`, collected at once when the handle is synchronous.
// *ran_on: the stream the vote's work went to.
static int ransac_vote_route(casa_handle* h, const casa_ransac_params* p, const VoteInput& in,
                             const casa_ransac_debug* debug, void* stream, cudaStream_t* ran_on) {
  const cudaStream_t st = (cudaStream_t)stream;
  *ran_on = st;
  if (!h) return fail(CASA_ERR_INVALID, "handle is NULL");
  if (!in.mask || !in.vertex || !in.out) return fail(CASA_ERR_INVALID, "mask / vertex / out_points must not be NULL");
  if (h->async_mode >= 2 && !debug) {
    casa_handle* sub = nullptr;
    int k = 0;
    int rc = lane_begin(h, h->async_mode, stream, &sub, &k);
    if (rc) return rc;
    *ran_on = sub->own_stream;
    rc = vote_enqueue(sub, p, in, nullptr, sub->own_stream);
    const int rce = lane_end(h, k, stream);
    return rc ? rc : rce;
  }
  if (!h->async_mode) reset_totals(h);  // synchronous calls report per-call statistics
  int rc = vote_enqueue(h, p, in, debug, st);
  if (rc) return rc;
  const bool want_stats = debug && debug->stats;
  if (h->async_mode && !want_stats) return CASA_OK;  // status, statistics and timing are collected by casa_sync()
  rc = collect(h);
  // debug copy of the statistics: from the call's read-back slot (the workspace words are cleared by the graph)
  if (want_stats)
    CUDA_TRY(cudaMemcpyAsync(debug->stats, h->slots[(h->slot_head - 1) % kCallSlots].stats, 4 * 8, cudaMemcpyHostToDevice, st));
  return rc;
}

extern "C" int casa_ransac_vote(casa_handle* h, const casa_ransac_params* p, const float* mask, const float* vertex,
                                const int32_t* idxs, const float* selection, float* out_points,
                                const casa_ransac_debug* debug, void* stream) {
  const VoteInput in{mask, MaskForm::kOneHot, vertex, /*vertex_mapped=*/false, /*not_binary=*/0, idxs, selection, out_points};
  cudaStream_t ran_on;
  return ransac_vote_route(h, p, in, debug, stream, &ran_on);
}

extern "C" int casa_ransac_vote_seg(casa_handle* h, const casa_ransac_params* p, const float* seg, const float* vertex,
                                    const int32_t* idxs, const float* selection, float* out_points,
                                    const casa_ransac_debug* debug, void* stream) {
  const VoteInput in{seg, MaskForm::kSeg, vertex, /*vertex_mapped=*/false, /*not_binary=*/0, idxs, selection, out_points};
  cudaStream_t ran_on;
  return ransac_vote_route(h, p, in, debug, stream, &ran_on);
}

// ------------------------------------------------------------------------------------------------ DLPack shim
// The reference hands tensors to foreign code through tf.numpy_function (ransac_voting.py:513, bpnp_layers.py:322);
// the drop-in's seam is DLPack: any framework's tensor arrives as a DLManagedTensor* (the pointer inside the
// "dltensor" PyCapsule), is validated HERE — device, dtype, shape, strides — and consumed exactly once.
namespace {
// DLPack ABI (dlpack.h, v0.x layout; public standard, restated so that the library has no header dependency)
struct DLDevice {
  int32_t device_type;  // 2 = kDLCUDA, 13 = kDLCUDAManaged
  int32_t device_id;
};
struct DLDataType {
  uint8_t code;  // 2 = kDLFloat
  uint8_t bits;
  uint16_t lanes;
};
struct DLTensor {
  void* data;
  DLDevice device;
  int32_t ndim;
  DLDataType dtype;
  int64_t* shape;
  int64_t* strides;  // NULL = compact row-major
  uint64_t byte_offset;
};
struct DLManagedTensor {
  DLTensor dl_tensor;
  void* manager_ctx;
  void (*deleter)(DLManagedTensor*);
};

int check_dl(const DLManagedTensor* m, const char* name, int device, int ndim_a, int ndim_b) {
  if (!m) return fail(CASA_ERR_INVALID, "%s: DLManagedTensor is NULL", name);
  const DLTensor& t = m->dl_tensor;
  if (t.device.device_type != 2 && t.device.device_type != 13)
    return fail(CASA_ERR_INVALID, "%s: DLPack device type %d is not CUDA", name, t.device.device_type);
  if (t.device.device_id != device) return fail(CASA_ERR_INVALID, "%s lives on CUDA device %d, the handle on %d", name, t.device.device_id, device);
  if (t.dtype.code != 2 || t.dtype.bits != 32 || t.dtype.lanes != 1)
    return fail(CASA_ERR_INVALID, "%s must be float32 (DLPack dtype code %d, %d bits, %d lanes)", name, t.dtype.code, t.dtype.bits, t.dtype.lanes);
  if (t.ndim != ndim_a && t.ndim != ndim_b) return fail(CASA_ERR_INVALID, "%s has %d dimensions", name, t.ndim);
  if (!t.data || !t.shape) return fail(CASA_ERR_INVALID, "%s: NULL data / shape", name);
  if (t.strides) {  // must be compact row-major (NHWC like the reference's tensors): no silent copies
    int64_t expect = 1;
    for (int i = t.ndim - 1; i >= 0; --i) {
      if (t.shape[i] != 1 && t.strides[i] != expect) return fail(CASA_ERR_INVALID, "%s is not C-contiguous (stride %lld of dimension %d)", name, (long long)t.strides[i], i);
      expect *= t.shape[i];
    }
  }
  return CASA_OK;
}

const float* dl_data(const DLManagedTensor* m) { return (const float*)((const char*)m->dl_tensor.data + m->dl_tensor.byte_offset); }

struct DeferredDelete {
  DLManagedTensor* m;
  cudaEvent_t done;
};
}  // namespace

// deleters of consumed capsules run once the GPU work that reads them has finished (polled at later API calls)
static std::vector<DeferredDelete>& deferred(casa_handle* h) {
  if (!h->deferred_list) h->deferred_list = new std::vector<DeferredDelete>();
  return *(std::vector<DeferredDelete>*)h->deferred_list;
}
static void run_deferred(casa_handle* h, bool wait) {
  std::vector<DeferredDelete>& v = deferred(h);
  for (size_t i = 0; i < v.size();) {
    if (wait) cudaEventSynchronize(v[i].done);
    if (wait || cudaEventQuery(v[i].done) == cudaSuccess) {
      if (v[i].m->deleter) v[i].m->deleter(v[i].m);
      bool shared = false;
      for (size_t k = 0; k < v.size(); ++k) shared |= k != i && v[k].done == v[i].done;
      if (!shared) cudaEventDestroy(v[i].done);
      v.erase(v.begin() + i);
    } else {
      ++i;
    }
  }
}

extern "C" int casa_ransac_vote_dlpack(casa_handle* h, const casa_ransac_params* p, void* mask_dlm, void* vertex_dlm, void* out_dlm,
                                       int mask_is_seg, void* stream) {
  if (!h || !p) return fail(CASA_ERR_INVALID, "handle / params is NULL");
  run_deferred(h, false);
  DLManagedTensor* m = (DLManagedTensor*)mask_dlm;
  DLManagedTensor* v = (DLManagedTensor*)vertex_dlm;
  DLManagedTensor* o = (DLManagedTensor*)out_dlm;
  auto reject = [&](int code) {  // the capsules are consumed in every case: a rejected call releases them at once
    if (m && m->deleter) m->deleter(m);
    if (v && v->deleter) v->deleter(v);
    if (o && o->deleter) o->deleter(o);
    return code;
  };
  int rc = check_dl(m, mask_is_seg ? "seg" : "mask", h->device, 4, 4);
  if (!rc) rc = check_dl(v, "vertex", h->device, 5, 6);
  if (!rc) rc = check_dl(o, "out", h->device, 4, 4);
  if (rc) return reject(rc);
  casa_ransac_params q = *p;  // shapes come from the tensors themselves
  const int64_t* ms = m->dl_tensor.shape;
  const int64_t* vs = v->dl_tensor.shape;
  const int64_t* os = o->dl_tensor.shape;
  q.b = (int32_t)ms[0];
  q.h = (int32_t)ms[1];
  q.w = (int32_t)ms[2];
  q.oc = (int32_t)ms[3] - (mask_is_seg ? 1 : 0);
  q.vertex_per_class = v->dl_tensor.ndim == 6;
  q.vn = (int32_t)vs[v->dl_tensor.ndim - 2];
  if (vs[0] != ms[0] || vs[1] != ms[1] || vs[2] != ms[2] || vs[v->dl_tensor.ndim - 1] != 2 || (q.vertex_per_class && vs[3] != q.oc))
    return reject(fail(CASA_ERR_INVALID, "vertex must be [b,h,w,vn,2] or [b,h,w,oc,vn,2] matching the mask"));
  if (os[0] != q.b || os[1] != q.oc || os[2] != q.vn || os[3] != 2) return reject(fail(CASA_ERR_INVALID, "out must be [b,oc,vn,2]"));
  const VoteInput in{dl_data(m), mask_is_seg ? MaskForm::kSeg : MaskForm::kOneHot, dl_data(v), false, 0, nullptr, nullptr,
                     (float*)dl_data(o)};
  cudaStream_t ran_on;
  rc = ransac_vote_route(h, &q, in, nullptr, stream, &ran_on);
  // the capsules are consumed either way: their deleters run once the work queued so far where the vote ran has finished
  cudaEvent_t done = nullptr;
  if (cudaEventCreateWithFlags(&done, cudaEventDisableTiming) == cudaSuccess && cudaEventRecord(done, ran_on) == cudaSuccess) {
    deferred(h).push_back({m, done});
    deferred(h).push_back({v, done});
    deferred(h).push_back({o, done});
  } else {
    cudaStreamSynchronize(ran_on);
    if (m->deleter) m->deleter(m);
    if (v->deleter) v->deleter(v);
    if (o->deleter) o->deleter(o);
  }
  return rc;
}

// true if `p` is page-locked host memory the device can read directly (UVA: same pointer)
static bool host_pointer_is_mapped(const void* p, const void** dev_ptr) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  if (at.type != cudaMemoryTypeHost || at.devicePointer == nullptr) return false;
  *dev_ptr = at.devicePointer;
  return true;
}

// CASA_HOST_TRACE=1: host-side time stamps of the phases of casa_ransac_vote_host on stderr (microseconds); it only
// prints, so it stays for looking at the overlap of packing, copies and votes in a deployment
static double host_now_us() {
  return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
static bool host_trace_on() {
  static const bool on = getenv("CASA_HOST_TRACE") != nullptr;
  return on;
}
#define HOST_TRACE(h, what, k) \
  do {                         \
    if (host_trace_on()) fprintf(stderr, "[host %p] %12.1f %s %d\n", (void*)(h), host_now_us(), what, (int)(k)); \
  } while (0)

// Waits for `st`.  The driver threads of the pipelined host entry sleep on a blocking-sync event: a spinning
// cudaStreamSynchronize would take a core from the packer threads for the two milliseconds of a call's GPU tail.
static int host_wait_stream(casa_handle* h, cudaStream_t st) {
  if (h->host_parent) {
    if (!h->ev_block) CUDA_TRY(cudaEventCreateWithFlags(&h->ev_block, cudaEventBlockingSync | cudaEventDisableTiming));
    CUDA_TRY(cudaEventRecord(h->ev_block, st));
    CUDA_TRY(cudaEventSynchronize(h->ev_block));
    return CASA_OK;
  }
  CUDA_TRY(cudaStreamSynchronize(st));
  return CASA_OK;
}

extern "C" int casa_ransac_vote_host(casa_handle* h, const casa_ransac_params* p, const float* mask_host,
                                     const float* vertex_host, float* out_points_host) {
  if (!h || !p) return fail(CASA_ERR_INVALID, "handle / params is NULL");
  if (!mask_host || !vertex_host || !out_points_host) return fail(CASA_ERR_INVALID, "host buffers must not be NULL");
  Layout L;
  int rc = make_layout(p, L);
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  const size_t hw = (size_t)p->h * p->w;
  const size_t vfields = p->vertex_per_class ? (size_t)p->oc : 1;
  const size_t mask_n = (size_t)p->b * hw * p->oc * 4, vert_n = (size_t)p->b * hw * vfields * p->vn * 2 * 4;
  const size_t out_b = (size_t)p->b * p->oc * p->vn * 2 * 4;
  cudaStream_t st = h->own_stream;
  // Pinned (page-locked) host buffers: the mask is DMA-copied in up to 4 image ranges on a copy stream while the
  // previous range is being voted on, and the vector field is never copied — k_gather_dirs reads only the masked
  // pixels' rows straight from the mapped host buffer.  About 200 MB instead of 511 MB cross PCIe for a 16-frame
  // batch, and the voting hides behind the mask transfer.  Pageable buffers are staged in one piece.
  const void *dm = nullptr, *dv = nullptr;
  const bool vertex_mapped = host_pointer_is_mapped(vertex_host, &dv);
  const bool mask_mapped = host_pointer_is_mapped(mask_host, &dm);
  // host-side packing of the mask (any host memory: the CPU reads it) needs the vector field to be readable in place
  // host threads a rank may use for packing: one process per GPU (torchrun exports LOCAL_WORLD_SIZE) shares the node's
  // cores with the other ranks; with fewer than 4 threads the DMA alone is faster (8 ranks on a 32-core host:
  // profiles/r02_scale_n8*.json), so packing is switched off there
  int pack_threads = (int)std::thread::hardware_concurrency() - 1;
  {
    const char* lws = getenv("LOCAL_WORLD_SIZE");
    if (lws && atoi(lws) > 1) pack_threads = ((int)std::thread::hardware_concurrency() - atoi(lws)) / atoi(lws);
    // CASA_HOST_THREADS: a deployment knob for hosts whose cores are shared with more than the node's ranks
    if (getenv("CASA_HOST_THREADS")) pack_threads = atoi(getenv("CASA_HOST_THREADS"));
    pack_threads = pack_threads > 12 ? 12 : pack_threads;  // 15 of 16 cores lose to oversubscription (profiles/r02_e2e.txt)
  }
  // CASA_NO_HOST_PACK=1: every range crosses PCIe as raw floats (bench.py reads it to count the bytes a step moves)
  const bool pack = vertex_mapped && !getenv("CASA_NO_HOST_PACK") && p->oc <= 32 && (pack_threads >= 4 || !mask_mapped);
  const bool zero_copy = vertex_mapped && (pack || mask_mapped);
  const size_t bits_n = (size_t)p->b * hw * sizeof(uint32_t);
  const size_t bits_b = pack ? (bits_n + 255) & ~size_t(255) : 0;
  const size_t mask_b = ((mask_n + 255) & ~size_t(255)) + bits_b;  // raw float ranges, then the packed words
  const size_t vert_b = zero_copy ? 0 : (vert_n + 255) & ~size_t(255);
  rc = ensure(&h->io_mem, &h->io_bytes, mask_b + vert_b + out_b);
  if (rc) return rc;
  float* dmask = (float*)h->io_mem;
  float* dout = (float*)((char*)h->io_mem + mask_b + vert_b);
  // The votes of the image ranges run on lanes (own workspace and stream each): the direction gather of one range
  // (mapped reads over PCIe) and the short kernels of another overlap the scoring of a third, instead of four votes
  // one behind the other on one stream.  A single range runs on the handle's own stream.
  const int parts = !zero_copy ? 1 : (p->b >= 8 ? 4 : (p->b >= 2 ? 2 : 1));
  if (parts >= 2)
    for (int i = 0; i < kMaxLanes; ++i)  // lanes a caller left busy
      if (h->lane[i] && h->lane_pending[i]) {
        CUDA_TRY(cudaStreamSynchronize(h->lane[i]->own_stream));
        h->lane_pending[i] = 0;
      }
  rc = collect(h);  // the calls before this one: what is collected below is this call's alone
  if (rc) return rc;
  reset_totals(h);
  if (!zero_copy) {
    float* dvert = (float*)((char*)h->io_mem + mask_b);
    CUDA_TRY(cudaMemcpyAsync(dmask, mask_host, mask_n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(dvert, vertex_host, vert_n, cudaMemcpyHostToDevice, st));
    rc = vote_enqueue(h, p, VoteInput{dmask, MaskForm::kOneHot, dvert, false, 0, nullptr, nullptr, dout}, nullptr, st);
    if (rc) return rc;
  } else {
    const size_t mask_img = hw * p->oc, vert_img = hw * vfields * p->vn * 2, out_img = (size_t)p->oc * p->vn * 2;
    int start[kMaxLanes + 1];
    for (int k = 0; k <= parts; ++k) start[k] = (int)((long long)p->b * k / parts);
    // The one-hot mask is 32 bytes per pixel for 4 bits of information.  Two engines move it in parallel: the copy
    // engine DMA-copies the raw floats of the even image ranges over PCIe, host threads (MaskPacker) turn the odd
    // ranges into u32 membership words — 1/oc of the bytes — while the GPU votes on the ranges before them.
    // (Packing everything on the host is no faster than the DMA on a 16-core host: profiles/r02_e2e.txt.)
    uint32_t* dbits = (uint32_t*)((char*)h->io_mem + mask_b - bits_b);
    bool packed[kMaxLanes] = {false, false, false, false};
    int pack_index[kMaxLanes] = {0, 0, 0, 0};
    // pipelined calls (casa_ransac_vote_host_async) share the parent handle's packer threads: the gate is held from the
    // start of this call's packing until its last range is packed, then the next call's packing starts while this
    // call's last ranges are still being voted on
    casa_handle* po = h->host_parent ? h->host_parent : h;
    std::unique_lock<std::mutex> gate;
    int last_packed = -1;
    if (pack) {
      HOST_TRACE(h, "enter", 0);
      if (h->host_parent || h->host_depth) gate = std::unique_lock<std::mutex>(po->pack_gate);
      HOST_TRACE(h, "gate", 0);
      if (!po->packer) {
        po->packer = new MaskPacker(pack_threads < 1 ? 1 : pack_threads);
      }
      if (h->bits_host_bytes < bits_n) {
        if (h->bits_host) CUDA_TRY(cudaFreeHost(h->bits_host));
        h->bits_host = nullptr;
        h->bits_host_bytes = 0;
        CUDA_TRY(cudaHostAlloc((void**)&h->bits_host, bits_n, cudaHostAllocDefault));
        h->bits_host_bytes = bits_n;
      }
      // With 6 or more host threads the packer (111 GB/s on the 16-core host of the pool, experimental/pack_bench.cpp)
      // outruns the DMA of the raw floats: every range is packed and only 4 bytes per pixel cross PCIe (e2e 3.08 ms
      // against 3.76 ms per 16 frames with half of the ranges packed: profiles/r02_e2e.txt).  With 4 or 5 threads the
      // odd ranges are packed beside the DMA of the even ones.  A pageable mask cannot be DMA-copied in place.
      const bool all = pack_threads >= 6 || !mask_mapped;
      std::vector<size_t> bounds;
      for (int k = 0; k < parts; ++k) {
        packed[k] = all || (k & 1);
        if (packed[k]) {
          last_packed = k;
          pack_index[k] = (int)bounds.size() / 2;
          bounds.push_back((size_t)start[k] * hw);
          bounds.push_back((size_t)start[k + 1] * hw);
        }
      }
      po->packer->start(mask_host, h->bits_host, p->oc, bounds);
    }
    for (int k = 0; k < parts; ++k) {  // the raw ranges are queued up front on the copy stream
      if (packed[k]) continue;
      const size_t o = (size_t)start[k] * mask_img, n = (size_t)(start[k + 1] - start[k]) * mask_img;
      CUDA_TRY(cudaMemcpyAsync(dmask + o, mask_host + o, n * 4, cudaMemcpyHostToDevice, h->copy_stream));
      CUDA_TRY(cudaEventRecord(h->part_ev[k], h->copy_stream));
    }
    for (int k = 0; k < parts; ++k) {
      casa_ransac_params pp = *p;
      pp.b = start[k + 1] - start[k];
      pp.image_offset = p->image_offset + start[k];
      VoteInput in;
      in.vertex = (const float*)dv + (size_t)start[k] * vert_img;
      in.vertex_mapped = true;
      in.out = dout + (size_t)start[k] * out_img;
      if (packed[k]) {
        po->packer->wait_part((size_t)pack_index[k]);
        HOST_TRACE(h, "packed", k);
        in.mask = dbits + (size_t)start[k] * hw;
        in.form = MaskForm::kPackedBits;
        in.not_binary = po->packer->not_binary();
        if (k == last_packed && gate.owns_lock()) gate.unlock();  // the packer threads are free for the next call
        const size_t o = (size_t)start[k] * hw, n = (size_t)pp.b * hw;
        CUDA_TRY(cudaMemcpyAsync(dbits + o, h->bits_host + o, n * sizeof(uint32_t), cudaMemcpyHostToDevice, h->copy_stream));
        CUDA_TRY(cudaEventRecord(h->part_ev[k], h->copy_stream));
      } else {
        in.mask = dmask + (size_t)start[k] * mask_img;
      }
      CUDA_TRY(cudaStreamWaitEvent(st, h->part_ev[k], 0));
      if (parts >= 2) {
        casa_handle* sub = nullptr;
        int lane = 0;
        rc = lane_begin(h, parts, (void*)st, &sub, &lane);
        if (!rc) {
          rc = vote_enqueue(sub, &pp, in, nullptr, sub->own_stream);
          const int rce = lane_end(h, lane, (void*)st);
          if (!rc) rc = rce;
        }
      } else {
        rc = vote_enqueue(h, &pp, in, nullptr, st);
      }
      HOST_TRACE(h, "issued", k);
      if (rc) {
        if (pack)
          for (int j = k + 1; j < parts; ++j)
            if (packed[j]) po->packer->wait_part((size_t)pack_index[j]);  // the workers still read the caller's buffer
        return rc;
      }
    }
    if (parts >= 2) {
      rc = casa_join(h, (void*)st);  // the result copy below waits for every lane
      if (rc) return rc;
    }
  }
  CUDA_TRY(cudaMemcpyAsync(out_points_host, dout, out_b, cudaMemcpyDeviceToHost, st));
  rc = host_wait_stream(h, st);
  if (rc) return rc;
  HOST_TRACE(h, "done", 0);
  if (parts >= 2)
    for (int i = 0; i < kMaxLanes; ++i) h->lane_pending[i] = 0;
  // loop states, statistics and the first error of this call's votes; the status is the OR over its image ranges
  Collected got;
  rc = collect(h, &got);
  h->last_status = got.status;
  h->last_launches = got.launches;
  return rc;
}

extern "C" int casa_selftest_pack(const float* mask, uint32_t* bits, int64_t npx, int oc, int threads, int parts) {
  if (!mask || !bits) return fail(CASA_ERR_INVALID, "casa_selftest_pack: NULL buffer");
  if (npx < 0 || oc < 1 || oc > 32 || threads < 1 || threads > 64 || parts < 1 || parts > 8)
    return fail(CASA_ERR_INVALID, "casa_selftest_pack: npx=%lld oc=%d threads=%d parts=%d", (long long)npx, oc, threads, parts);
  MaskPacker packer(threads);
  std::vector<size_t> bounds;
  for (int k = 0; k < parts; ++k) {
    bounds.push_back((size_t)(npx * k / parts));
    bounds.push_back((size_t)(npx * (k + 1) / parts));
  }
  packer.start(mask, bits, oc, bounds);
  for (int k = 0; k < parts; ++k) packer.wait_part((size_t)k);
  return packer.not_binary();
}

// ------------------------------------------------------------------------------------------------ pipelined host entry
// casa_ransac_vote_host is synchronous like the reference's call: it returns with the keypoints on the host, and its
// phases run one behind the other — the host threads pack the mask (about 60 % of the call), then the GPU finishes the
// last image ranges while the host threads idle.  A caller that streams batches (an evaluation loop over a data set)
// can keep kHostDepth calls in flight instead: casa_ransac_vote_host_async hands the call to a driver thread with a
// sub-handle of its own and returns a ticket, casa_host_wait(ticket) returns that call's error code once its keypoints
// are in out_points_host.  The drivers share the packer threads (one call packs at a time, in ticket order for two
// drivers), so call i+1 is packed while the GPU votes on the last ranges of call i.
struct HostJob {
  casa_ransac_params p;
  const float* mask = nullptr;
  const float* vertex = nullptr;
  float* out = nullptr;
  int64_t ticket = -1;
  int rc = 0;
  uint32_t status = 0;
  int64_t launches = 0;
  char err[512] = "";
};

struct HostDriver {
  casa_handle* sub = nullptr;
  std::thread th;
  std::mutex m;
  std::condition_variable cv;
  int state = 0;  // 0 idle, 1 queued / running, 2 done and not yet collected
  bool quit = false;
  HostJob job;
};

static void host_driver_run(HostDriver* d) {
  for (;;) {
    std::unique_lock<std::mutex> g(d->m);
    d->cv.wait(g, [&] { return d->quit || d->state == 1; });
    if (d->quit) return;
    const HostJob j = d->job;
    g.unlock();
    const int rc = casa_ransac_vote_host(d->sub, &j.p, j.mask, j.vertex, j.out);
    g.lock();
    d->job.rc = rc;
    d->job.status = d->sub->last_status;
    d->job.launches = d->sub->last_launches;
    if (rc) snprintf(d->job.err, sizeof(d->job.err), "%s", g_err);  // this thread's last error
    d->state = 2;
    d->cv.notify_all();
  }
}

// keeps the first error of a finished call nobody waited for (reported by the next casa_host_wait / casa_sync)
static void host_fold(casa_handle* h, HostDriver* d) {
  if (d->state != 2) return;
  if (d->job.rc && !h->host_first_rc) {
    h->host_first_rc = d->job.rc;
    snprintf(h->host_first_err, sizeof(h->host_first_err), "%s", d->job.err);
  }
  h->last_status = d->job.status;
  h->last_launches = d->job.launches;
  d->state = 0;
}

static void host_drivers_destroy(casa_handle* h) {
  for (int i = 0; i < 4; ++i) {
    HostDriver* d = h->driver[i];
    if (!d) continue;
    {
      std::unique_lock<std::mutex> g(d->m);
      d->cv.wait(g, [&] { return d->state != 1; });
      d->quit = true;
    }
    d->cv.notify_all();
    if (d->th.joinable()) d->th.join();
    if (d->sub) casa_destroy(d->sub);
    delete d;
    h->driver[i] = nullptr;
  }
}

// waits for every call in flight; returns the first error among the calls that were not waited for by ticket
static int host_drain(casa_handle* h) {
  for (int i = 0; i < 4; ++i) {
    HostDriver* d = h->driver[i];
    if (!d) continue;
    std::unique_lock<std::mutex> g(d->m);
    d->cv.wait(g, [&] { return d->state != 1; });
    host_fold(h, d);
  }
  if (h->host_first_rc) {
    const int rc = h->host_first_rc;
    h->host_first_rc = 0;
    return fail(rc, "%s", h->host_first_err);
  }
  return CASA_OK;
}

extern "C" int casa_ransac_vote_host_async(casa_handle* h, const casa_ransac_params* p, const float* mask_host,
                                           const float* vertex_host, float* out_points_host, int64_t* ticket) {
  if (!h || !p || !ticket) return fail(CASA_ERR_INVALID, "handle / params / ticket is NULL");
  if (!mask_host || !vertex_host || !out_points_host) return fail(CASA_ERR_INVALID, "host buffers must not be NULL");
  if (h->host_parent || h->is_lane) return fail(CASA_ERR_INVALID, "casa_ransac_vote_host_async: not on a sub-handle");
  {
    Layout L;  // shape errors are the caller's at once, not the driver thread's later
    const int rcl = make_layout(p, L);
    if (rcl) return rcl;
  }
  if (!h->host_depth) {
    int depth = 2;
    if (getenv("CASA_HOST_DEPTH")) depth = atoi(getenv("CASA_HOST_DEPTH"));  // documented in casapose_b200.h
    h->host_depth = depth < 1 ? 1 : (depth > 4 ? 4 : depth);
  }
  const int k = (int)(h->host_ticket % h->host_depth);
  if (!h->driver[k]) {
    casa_handle* sub = nullptr;
    const int rcc = casa_create(h->device, &sub);
    if (rcc) return rcc;
    sub->host_parent = h;
    HostDriver* d = new HostDriver();
    d->sub = sub;
    d->th = std::thread(host_driver_run, d);
    h->driver[k] = d;
  }
  HostDriver* d = h->driver[k];
  {
    std::unique_lock<std::mutex> g(d->m);
    d->cv.wait(g, [&] { return d->state != 1; });  // the call `depth` tickets ago still runs
    host_fold(h, d);
    d->job = HostJob();
    d->job.p = *p;
    d->job.mask = mask_host;
    d->job.vertex = vertex_host;
    d->job.out = out_points_host;
    d->job.ticket = h->host_ticket;
    d->state = 1;
  }
  d->cv.notify_all();
  *ticket = h->host_ticket++;
  return CASA_OK;
}

extern "C" int casa_host_wait(casa_handle* h, int64_t ticket) {
  if (!h) return fail(CASA_ERR_INVALID, "NULL argument");
  if (ticket < 0 || ticket >= h->host_ticket || !h->host_depth) return fail(CASA_ERR_INVALID, "casa_host_wait: unknown ticket %lld", (long long)ticket);
  HostDriver* d = h->driver[ticket % h->host_depth];
  std::unique_lock<std::mutex> g(d->m);
  if (d->job.ticket == ticket && d->state != 0) {
    d->cv.wait(g, [&] { return d->state == 2; });
    const int rc = d->job.rc;
    h->last_status = d->job.status;
    h->last_launches = d->job.launches;
    d->state = 0;
    if (rc) return fail(rc, "%s", d->job.err);
    return CASA_OK;
  }
  g.unlock();
  // collected before (waited twice, or overtaken by a later call on its driver): report a kept error once
  if (h->host_first_rc) {
    const int rc = h->host_first_rc;
    h->host_first_rc = 0;
    return fail(rc, "%s", h->host_first_err);
  }
  return CASA_OK;
}

// ------------------------------------------------------------------------------------------------ LS layer

namespace {
struct LsGrad {
  const float* grad_points = nullptr;  // [b,oc,vn,2]
  float* grad_direct = nullptr;        // [b,h,w,2*vn]
  float* grad_conf = nullptr;          // [b,h,w,vn]
};
int ls_vote_impl(casa_handle* h, const casa_ls_params* p, const float* seg, const float* direct, const float* conf,
                 float* out_points, const casa_ls_debug* debug, void* stream, const LsGrad* grad, int pix_capacity = 0);
}  // namespace

extern "C" int casa_ls_vote(casa_handle* h, const casa_ls_params* p, const float* seg, const float* direct,
                            const float* conf, float* out_points, const casa_ls_debug* debug, void* stream) {
  if (!h || !p) return fail(CASA_ERR_INVALID, "handle / params is NULL");
  if (!seg || !direct || !conf || !out_points) return fail(CASA_ERR_INVALID, "seg / direct / conf / out_points must not be NULL");
  if (h->async_mode >= 2 && !debug && !p->check_finite && !h->is_lane) {  // lanes, as for the votes (check_finite waits for the host)
    casa_handle* sub = nullptr;
    int k = 0;
    int rcl = lane_begin(h, h->async_mode, stream, &sub, &k);
    if (rcl) return rcl;
    rcl = ls_vote_impl(sub, p, seg, direct, conf, out_points, nullptr, (void*)sub->own_stream, nullptr);
    const int rce = lane_end(h, k, stream);
    h->last_launches = sub->last_launches;
    return rcl ? rcl : rce;
  }
  return ls_vote_impl(h, p, seg, direct, conf, out_points, debug, stream, nullptr);
}

extern "C" int casa_ls_vote_backward(casa_handle* h, const casa_ls_params* p, const float* seg, const float* direct,
                                     const float* conf, const float* grad_points, float* out_points, float* grad_direct,
                                     float* grad_conf, void* stream) {
  if (!h || !p) return fail(CASA_ERR_INVALID, "handle / params is NULL");
  if (!seg || !direct || !conf || !grad_points || !grad_direct || !grad_conf)
    return fail(CASA_ERR_INVALID, "casa_ls_vote_backward: only out_points may be NULL");
  LsGrad g;
  g.grad_points = grad_points;
  g.grad_direct = grad_direct;
  g.grad_conf = grad_conf;
  return ls_vote_impl(h, p, seg, direct, conf, out_points, nullptr, stream, &g);
}

namespace {
int ls_vote_impl(casa_handle* h, const casa_ls_params* p, const float* seg, const float* direct, const float* conf,
                 float* out_points, const casa_ls_debug* debug, void* stream, const LsGrad* grad, int pix_capacity) {
  if (p->num_classes < 2 || p->num_classes > 33) return fail(CASA_ERR_INVALID, "num_classes=%d outside 2..33", p->num_classes);
  casa_ransac_params rp;
  memset(&rp, 0, sizeof(rp));
  rp.b = p->b; rp.h = p->h; rp.w = p->w; rp.oc = p->num_classes - 1; rp.vn = p->vn;
  rp.round_hyp_num = 1; rp.max_iter = 1;
  rp.min_num = 0.f; rp.max_num = 3.0e38f; rp.inlier_thresh = 0.99f; rp.confidence = 0.99f;
  // A pixel is listed for every class whose softmax(1e6 seg) value is non-zero, so near-tied logits (flat regions, a
  // zero-initialised seg head) can list a pixel several times: the per-image list then needs more than h*w slots.
  // The first attempt uses h*w (or the caller's pix_capacity); an overflow is retried below with the measured need.
  rp.pix_capacity = pix_capacity > 0 ? pix_capacity : p->pix_capacity;
  // The forward call reduces 512-entry tiles in one fused pass and finds the components over horizontal runs
  // (k_cc_runs); gradient and debug calls keep the pixel-level union-find, whose forest the backward pass and the
  // debug outputs read.
  const bool runs_cc = !grad && !debug;
  const int ls_tile = grad ? kRefineTile : kFusedTile;
  Layout L;
  int rc = make_layout(&rp, L, ls_tile);
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  L.d.rtile = ls_tile;
  const Dims& d = L.d;
  const size_t npx = (size_t)d.b * d.hw;
  const size_t nle = (size_t)d.b * d.cap;  // list entries
  size_t cur = L.total;
  const size_t off_cls9 = bump(cur, npx), off_parent = bump(cur, npx * 4), off_count = bump(cur, npx * 4),
               off_roots = bump(cur, npx * 4), off_nroots = bump(cur, (size_t)d.b * 4), off_sel = bump(cur, (size_t)d.J * 4),
               off_wt = bump(cur, nle * 4), off_cconf = bump(cur, nle * d.vn * 4),
               off_adj = bump(cur, (size_t)d.J * d.vn * 6 * 4), off_tmp_out = bump(cur, (size_t)d.J * d.vn * 2 * 4),
               off_ridx = bump(cur, nle * 4), off_keep = bump(cur, nle), off_run_pk = bump(cur, nle * 4),
               off_run_x1 = bump(cur, nle * 4), off_run_parent = bump(cur, nle * 4), off_run_cnt = bump(cur, nle * 4);
  rc = ensure(&h->ws_mem, &h->ws_bytes, cur);
  if (rc) return rc;
  h->clean_ctrl = nullptr;  // the LS layer leaves its own loop state in ctrl / stats
  cudaStream_t st = (cudaStream_t)stream;
  WS ws = make_ws(L, h->ws_mem, true);
  char* base = (char*)h->ws_mem;
  LsWS lw;
  lw.cls9 = (unsigned char*)(base + off_cls9);
  lw.parent = (int*)(base + off_parent);
  lw.count = (int*)(base + off_count);
  lw.roots = (int*)(base + off_roots);
  lw.nroots = (int*)(base + off_nroots);
  lw.sel = (int*)(base + off_sel);
  lw.wt = (float*)(base + off_wt);
  lw.cconf = (float*)(base + off_cconf);
  lw.ridx = (int*)(base + off_ridx);
  lw.keep = (unsigned char*)(base + off_keep);
  lw.run_pk = (uint32_t*)(base + off_run_pk);
  lw.run_x1 = (int*)(base + off_run_x1);
  lw.run_parent = (int*)(base + off_run_parent);
  lw.run_cnt = (int*)(base + off_run_cnt);
  LsDims ld;
  ld.b = d.b; ld.h = d.h; ld.w = d.w; ld.nc = p->num_classes; ld.oc = d.oc; ld.vn = d.vn; ld.hw = d.hw;
  ld.sigmoid_weights = p->sigmoid_weights ? 1 : 0;
  ld.filter = p->filter_estimates ? 1 : 0;
  ld.bins = p->second_largest ? 3 : 2;
  ld.which = p->second_largest ? 2 : 1;
  ld.min_component = p->min_component > 0 ? p->min_component : 50;
  casa_ls_debug dbg;
  memset(&dbg, 0, sizeof(dbg));
  if (debug) dbg = *debug;
  int64_t launches = 0;

  // the launch list: replayed as a CUDA graph (kernel parameters patched per call) unless debug outputs are asked for
  std::vector<Step> steps;
  steps.reserve(16);
  steps.push_back(special(STEP_CLEAR));  // ctrl / stats: one memset node in front of the kernels
  {
    const size_t sm = (size_t)kCountTile * ld.nc * 4;
    const void* classify = ld.nc == 9 ? (const void*)k_ls_classify<9> : (const void*)k_ls_classify<0>;
    // Without the opt-in, static plus dynamic shared memory of a block may not exceed 48 KB: the kernel's own counters
    // (scnt) count too, so nc = 12 (exactly 48 KB of staged logits) needs the attribute as well.
    int& static_sm = h->classify_static_smem[ld.nc == 9 ? 0 : 1];
    if (static_sm < 0) {
      cudaFuncAttributes fa;
      CUDA_TRY(cudaFuncGetAttributes(&fa, classify));
      static_sm = (int)fa.sharedSizeBytes;
    }
    if (sm + (size_t)static_sm > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(classify, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    steps.push_back(kstep(classify, dim3(d.nct, d.b), 256, sm).arg(seg).arg(ws).arg(d).arg(lw).arg(ld).arg((int)(runs_cc ? 1 : 0)));
  }
  steps.push_back(kstep((const void*)k_place<0>, dim3((d.nct + kPlaceSub - 1) / kPlaceSub, d.b), 256).arg((const float*)nullptr).arg(ws).arg(d).arg((int)0));
  // topology: the work-item / tile plan only needs the job table and runs beside the component chain (side branch)
  steps.push_back(kstep((const void*)k_plan, 1, d.J > 256 ? 1024 : 256).arg(ws).arg(d).arg((int)0).on_side(1));
  const int gx = (d.cap + 255) / 256 < 24 ? (d.cap + 255) / 256 : 24;
  if (ld.filter && runs_cc) {
    steps.push_back(kstep((const void*)k_cc_runs, d.J, kCcThreads).arg(ws).arg(d).arg(lw).arg(ld));
  } else if (ld.filter) {
    steps.push_back(kstep((const void*)k_cc_init, dim3(gx, d.J), 256).arg(ws).arg(d).arg(lw).arg(ld));
    steps.push_back(kstep((const void*)k_cc_merge, dim3(gx, d.J), 256).arg(ws).arg(d).arg(lw).arg(ld));
    steps.push_back(kstep((const void*)k_cc_flatten, dim3(gx, d.J), 256).arg(ws).arg(d).arg(lw).arg(ld));
    steps.push_back(kstep((const void*)k_cc_select, d.J, 256).arg(lw).arg(ld));
  }
  const int grid_x = d.max_rtiles < h->sm_count * 4 ? d.max_rtiles : h->sm_count * 4;
  if (grad) {
    // the backward pass reads the gathered directions / weights / confidences: the three-kernel form fills them
    steps.push_back(kstep(d.vn == 9 ? (const void*)k_gather_dirs<18> : (const void*)k_gather_dirs<0>, dim3(gx, d.J), 256)
                        .arg(direct).arg(ws).arg(d).arg((int)0).joins());
    steps.push_back(kstep((const void*)k_ls_weights, dim3(gx, d.J), 256).arg(ws).arg(d).arg(lw).arg(ld).arg(seg).arg(conf));
    steps.push_back(kstep((const void*)k_ls_reduce, dim3(grid_x, d.vn), 256).arg(ws).arg(d).arg(lw).arg(ld));
  } else {
    if (h->fused_occ == 0) {
      CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&h->fused_occ, k_ls_fused<true>, 32 * d.vn, 0));
      if (h->fused_occ < 1) h->fused_occ = 1;
    }
    const int fused_gx = d.max_rtiles < h->sm_count * h->fused_occ ? d.max_rtiles : h->sm_count * h->fused_occ;
    // float2 loads of a pixel's (dy, dx) need an 8-byte aligned `direct`; callers may pass any 4-byte aligned buffer
    const void* fused = (((uintptr_t)direct) & 7) == 0 ? (const void*)k_ls_fused<true> : (const void*)k_ls_fused<false>;
    steps.push_back(kstep(fused, fused_gx, 32 * d.vn).arg(ws).arg(d).arg(lw).arg(ld).arg(seg).arg(direct).arg(conf)
                        .arg((int)(runs_cc ? 1 : 0)).joins());
  }
  if (!out_points) out_points = (float*)(base + off_tmp_out);
  steps.push_back(kstep((const void*)k_ls_solve, d.J, 32).arg(ws).arg(d).arg(ld).arg(out_points).arg(dbg.sums).arg(h->sticky));
  if (grad) {
    float* adj = (float*)(base + off_adj);
    CUDA_TRY(cudaMemsetAsync(grad->grad_direct, 0, npx * 2 * d.vn * sizeof(float), st));
    CUDA_TRY(cudaMemsetAsync(grad->grad_conf, 0, npx * d.vn * sizeof(float), st));
    steps.push_back(kstep((const void*)k_ls_adjoint, d.J, 32).arg(ws).arg(d).arg(ld).arg(grad->grad_points).arg(adj));
    const void* bwd = (((uintptr_t)grad->grad_direct) & 7) == 0 ? (const void*)k_ls_backward<true> : (const void*)k_ls_backward<false>;
    steps.push_back(kstep(bwd, grid_x, 256).arg(ws).arg(d).arg(lw).arg(ld).arg(adj).arg(grad->grad_direct).arg(grad->grad_conf));
  }
  for (const Step& s2 : steps) launches += s2.kind == STEP_KERNEL;
  rc = (h->use_graph && !debug) ? run_graph(h, steps, ws, st) : run_direct(h, steps, ws, st);
  if (rc) return rc;
  CUDA_TRY(cudaGetLastError());
  if (dbg.labels) CUDA_TRY(cudaMemcpyAsync(dbg.labels, lw.cls9, npx, cudaMemcpyDeviceToDevice, st));
  if (dbg.parent && ld.filter) CUDA_TRY(cudaMemcpyAsync(dbg.parent, lw.parent, npx * 4, cudaMemcpyDeviceToDevice, st));
  if (dbg.selected && ld.filter) CUDA_TRY(cudaMemcpyAsync(dbg.selected, lw.sel, (size_t)d.J * 4, cudaMemcpyDeviceToDevice, st));
  if (dbg.tn) CUDA_TRY(cudaMemcpyAsync(dbg.tn, ws.job_tn, (size_t)d.J * 4, cudaMemcpyDeviceToDevice, st));
  h->last_launches = launches;
  h->last_stream = st;
  if (p->check_finite || grad) {  // the backward pass always checks for a list overflow (it would zero gradients silently)
    CUDA_TRY(cudaMemcpyAsync(h->pinned, ws.ctrl, CTRL_WORDS * sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    h->last_status = (uint32_t)h->pinned[CTRL_STATUS];
    if (h->last_status & CASA_STATUS_PIX_OVERFLOW) {
      // measured need: the largest per-image sum of the class counts (the reference has no such limit: it evaluates
      // every class on the dense field, voting_layers_2d.py:107-114)
      std::vector<int> tn0(d.J);
      CUDA_TRY(cudaMemcpy(tn0.data(), ws.job_tn0, (size_t)d.J * sizeof(int), cudaMemcpyDeviceToHost));
      long long need = 0;
      for (int i = 0; i < d.b; ++i) {
        long long sum = 0;
        for (int c = 0; c < d.oc; ++c) sum += tn0[(size_t)i * d.oc + c];
        need = sum > need ? sum : need;
      }
      need = (need + 1023) / 1024 * 1024;
      CUDA_TRY(cudaMemset(h->sticky, 0, sizeof(uint32_t)));  // the retried call reports for itself
      if (need <= d.cap || need > (1ll << 30))
        return fail(CASA_ERR_WORKSPACE, "CoordLSVotingWeighted: pixel lists overflow (need %lld slots per image)", need);
      return ls_vote_impl(h, p, seg, direct, conf, out_points == (float*)(base + off_tmp_out) ? nullptr : out_points, debug, stream, grad, (int)need);
    }
    if (p->check_finite && (h->last_status & CASA_STATUS_LS_NONFINITE))
      return fail(CASA_ERR_INPUT, "CoordLSVotingWeighted: non-finite R / q / p (the reference asserts here, voting_layers_2d.py:109-121)");
  }
  return CASA_OK;
}
}  // namespace

// ------------------------------------------------------------------------------------------------ PnP

extern "C" int casa_pnp(casa_handle* h, int32_t n, int32_t vn, const float* points2d, const float* points3d,
                        const float* camera, const float* offsets, float* poses, void* stream) {
  if (!h) return fail(CASA_ERR_INVALID, "handle is NULL");
  if (!points2d || !points3d || !camera || !poses) return fail(CASA_ERR_INVALID, "points2d / points3d / camera / poses must not be NULL");
  if (n < 0 || vn < 6 || vn > 16) return fail(CASA_ERR_INVALID, "n=%d, vn=%d: need n >= 0 and 6 <= vn <= 16", n, vn);
  if (n == 0) return CASA_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  PnpParams pp;
  pp.n = n;
  pp.vn = vn;
  pp.reproj_px = 12.0f;
  k_pnp<<<(n + 3) / 4, 128, 0, (cudaStream_t)stream>>>(pp, points2d, points3d, camera, offsets, poses);
  CUDA_TRY(cudaGetLastError());
  h->last_launches = 1;
  return CASA_OK;
}

extern "C" int casa_pnp_backward(casa_handle* h, int32_t n, int32_t vn, const float* points3d, const float* camera,
                                 const float* poses, int32_t pose_form, const float* grad_poses, float* grad_points2d,
                                 void* stream) {
  if (!h) return fail(CASA_ERR_INVALID, "handle is NULL");
  if (!points3d || !camera || !poses || !grad_poses || !grad_points2d)
    return fail(CASA_ERR_INVALID, "points3d / camera / poses / grad_poses / grad_points2d must not be NULL");
  if (n < 0 || vn < 6 || vn > 16) return fail(CASA_ERR_INVALID, "n=%d, vn=%d: need n >= 0 and 6 <= vn <= 16", n, vn);
  if (pose_form != 6 && pose_form != 12) return fail(CASA_ERR_INVALID, "pose_form=%d: need 6 (rvec, tvec) or 12 ([R|t])", pose_form);
  if (n == 0) return CASA_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  k_pnp_backward<<<(n + 3) / 4, 128, 0, (cudaStream_t)stream>>>(n, vn, pose_form, points3d, camera, poses, grad_poses,
                                                                grad_points2d);
  CUDA_TRY(cudaGetLastError());
  h->last_launches = 1;
  return CASA_OK;
}

extern "C" int casa_pose_errors(casa_handle* h, int32_t n, int32_t m, int32_t maxp, const float* poses, const float* poses_gt,
                                const float* camera, const float* model_points, const int32_t* model_counts,
                                const int32_t* obj_model, const float* diameters, const int32_t* valid,
                                float allowed_error_2d, float* out_rows, void* stream) {
  if (!h) return fail(CASA_ERR_INVALID, "handle is NULL");
  if (!poses || !poses_gt || !camera || !model_points || !model_counts || !diameters || !valid || !out_rows)
    return fail(CASA_ERR_INVALID, "casa_pose_errors: only obj_model may be NULL");
  if (n < 0 || m < 1 || maxp < 1) return fail(CASA_ERR_INVALID, "n=%d, m=%d, maxp=%d: need n >= 0, m >= 1, maxp >= 1", n, m, maxp);
  if (n == 0) return CASA_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  PoseErrParams pp;
  pp.n = n;
  pp.m = m;
  pp.maxp = maxp;
  pp.allowed_2d = allowed_error_2d;
  const bool may_sym = maxp >= 3417;  // ADD-S only for the 7862 / 3417 vertex meshes (ransac_voting.py:618)
  const int tiles = (maxp + kMetricThreads - 1) / kMetricThreads;
  auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
  const size_t base_b = up((size_t)n * 2 * sizeof(float)), state_b = up((size_t)n * sizeof(int));
  const size_t part_b = may_sym ? up((size_t)n * tiles * sizeof(double)) : 0;
  const size_t cloud_b = may_sym ? up((size_t)n * maxp * sizeof(float4)) : 0;
  int rc = ensure(&h->metric_mem, &h->metric_bytes, base_b + state_b + part_b + 2 * cloud_b);
  if (rc != CASA_OK) return rc;
  char* b = (char*)h->metric_mem;
  float* base = (float*)b;
  int* state = (int*)(b + base_b);
  double* partial = (double*)(b + base_b + state_b);
  float4* cloud_gt = may_sym ? (float4*)(b + base_b + state_b + part_b) : nullptr;
  float4* cloud_est = may_sym ? (float4*)(b + base_b + state_b + part_b + cloud_b) : nullptr;
  k_pose_project<<<n, kMetricThreads, 0, st>>>(pp, poses, poses_gt, camera, model_points, model_counts, obj_model, valid,
                                               cloud_gt, cloud_est, base, state, out_rows);
  int launches = 1;
  if (may_sym) {
    k_adds_min<<<dim3(tiles, min(n, kAddsGridY)), kMetricThreads, 0, st>>>(pp, tiles, model_counts, obj_model, state, cloud_gt,
                                                                          cloud_est, partial);
    ++launches;
  }
  k_pose_finalize<<<(n + 127) / 128, 128, 0, st>>>(pp, tiles, model_counts, obj_model, state, base, partial, diameters, out_rows);
  ++launches;
  CUDA_TRY(cudaGetLastError());
  h->last_launches = launches;
  return CASA_OK;
}

extern "C" int casa_set_async(casa_handle* h, int enable) {
  if (!h) return fail(CASA_ERR_INVALID, "NULL argument");
  if (enable < 0 || enable > kMaxLanes)
    return fail(CASA_ERR_INVALID, "casa_set_async: mode %d (0 synchronous, 1 asynchronous, 2..%d asynchronous on that many lanes)", enable, kMaxLanes);
  if (h->async_mode >= 2 && enable != h->async_mode) {  // leaving a lane mode: everything the lanes hold has run when this returns
    CUDA_TRY(cudaSetDevice(h->device));
    for (int i = 0; i < kMaxLanes; ++i)
      if (h->lane[i] && h->lane_pending[i]) {
        CUDA_TRY(cudaStreamSynchronize(h->lane[i]->own_stream));
        h->lane_pending[i] = 0;
      }
  }
  if (h->async_mode == 0 && enable != 0) {  // an asynchronous session starts clean: synchronous calls reported their own status
    CUDA_TRY(cudaSetDevice(h->device));
    if (h->last_stream) CUDA_TRY(cudaStreamSynchronize(h->last_stream));
    CUDA_TRY(cudaMemset(h->sticky, 0, sizeof(uint32_t)));
  }
  h->async_mode = enable;
  return CASA_OK;
}

// Orders the outputs of every vote issued in the two-lane mode on `stream` (the caller's stream does not wait for the
// lanes by itself); a no-op in the other modes, where a vote runs on the caller's stream.
extern "C" int casa_join(casa_handle* h, void* stream) {
  if (!h) return fail(CASA_ERR_INVALID, "NULL argument");
  CUDA_TRY(cudaSetDevice(h->device));
  for (int i = 0; i < kMaxLanes; ++i)
    if (h->lane[i] && h->lane_pending[i]) CUDA_TRY(cudaStreamWaitEvent((cudaStream_t)stream, h->lane_done[i], 0));
  return CASA_OK;
}

extern "C" int casa_sync(casa_handle* h) {
  if (!h) return fail(CASA_ERR_INVALID, "NULL argument");
  CUDA_TRY(cudaSetDevice(h->device));
  const int rch = host_drain(h);  // pipelined host calls in flight (casa_ransac_vote_host_async)
  if (rch) return rch;
  int rc = collect(h);
  CUDA_TRY(cudaStreamSynchronize(h->last_stream));
  if (h->deferred_list) run_deferred(h, true);
  CUDA_TRY(cudaMemcpy(h->pinned_sticky, h->sticky, sizeof(uint32_t), cudaMemcpyDeviceToHost));
  uint32_t st = *h->pinned_sticky;
  if (st) CUDA_TRY(cudaMemset(h->sticky, 0, sizeof(uint32_t)));
  for (int i = 0; i < kMaxLanes; ++i) {  // lanes: wait for their streams, fold their sticky status words in
    casa_handle* s = h->lane[i];
    if (!s) continue;
    CUDA_TRY(cudaStreamSynchronize(s->own_stream));
    h->lane_pending[i] = 0;
    CUDA_TRY(cudaMemcpy(s->pinned_sticky, s->sticky, sizeof(uint32_t), cudaMemcpyDeviceToHost));
    if (*s->pinned_sticky) CUDA_TRY(cudaMemset(s->sticky, 0, sizeof(uint32_t)));
    st |= *s->pinned_sticky;
  }
  if (rc) return rc;
  if (st & CASA_STATUS_PIX_OVERFLOW)
    return fail(CASA_ERR_WORKSPACE, "a call since the last casa_sync overflowed its pixel lists (mask not one-hot?); retry with a larger pix_capacity");
  if (st & CASA_STATUS_IDX_RANGE) return fail(CASA_ERR_INPUT, "a call since the last casa_sync had caller-supplied idxs outside [0, tn)");
  if (st & CASA_STATUS_LS_NONFINITE) return fail(CASA_ERR_INPUT, "a CoordLSVotingWeighted call since the last casa_sync produced non-finite R / q / p");
  return CASA_OK;
}

extern "C" int casa_last_status(casa_handle* h, uint32_t* status) {
  if (!h || !status) return fail(CASA_ERR_INVALID, "NULL argument");
  const int rc = collect(h);
  if (rc != CASA_OK && rc != CASA_ERR_WORKSPACE && rc != CASA_ERR_INPUT) return rc;
  *status = h->last_status;
  return CASA_OK;
}

extern "C" int casa_set_timing(casa_handle* h, int enable) {
  if (!h) return fail(CASA_ERR_INVALID, "NULL argument");
  h->timing = enable ? 1 : 0;
  return CASA_OK;
}

extern "C" int casa_get_timing(casa_handle* h, double* score_ms, int64_t* score_launches, uint64_t* stats4) {
  if (!h) return fail(CASA_ERR_INVALID, "NULL argument");
  collect(h);
  if (score_ms) *score_ms = h->score_ms;
  if (score_launches) *score_launches = h->score_launches;
  if (stats4)
    for (int k = 0; k < 4; ++k) stats4[k] = h->stats[k];
  if (h->async_mode) reset_totals(h);  // asynchronous callers get the totals since their previous query
  return CASA_OK;
}

extern "C" int casa_last_launches(casa_handle* h, int64_t* launches) {
  if (!h || !launches) return fail(CASA_ERR_INVALID, "NULL argument");
  collect(h);
  *launches = h->async_mode ? h->launches_total : h->last_launches;
  return CASA_OK;
}

// ------------------------------------------------------------------------------------------------ keypoint gather

static void comm_release(casa_handle* h) {
  if (h->comm && h->comm_owned && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
  h->comm = nullptr;
  h->comm_owned = 0;
}

extern "C" int casa_nccl_unique_id(void* id128) {
  if (!id128) return fail(CASA_ERR_INVALID, "NULL argument");
  int rc = nccl_load();
  if (rc) return rc;
  NCCL_TRY(g_nccl.GetUniqueId(id128));
  return CASA_OK;
}

extern "C" int casa_comm_init(casa_handle* h, const void* id128, int rank, int world) {
  if (!h || !id128) return fail(CASA_ERR_INVALID, "NULL argument");
  if (world < 1 || rank < 0 || rank >= world) return fail(CASA_ERR_INVALID, "rank %d of %d", rank, world);
  int rc = nccl_load();
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  comm_release(h);
  NcclId128 id;
  memcpy(&id, id128, sizeof(id));
  NCCL_TRY(g_nccl.CommInitRank(&h->comm, world, id, rank));
  h->comm_owned = 1;
  h->comm_rank = rank;
  h->comm_world = world;
  return CASA_OK;
}

extern "C" int casa_comm_attach(casa_handle* h, void* nccl_comm, int rank, int world) {
  if (!h || !nccl_comm) return fail(CASA_ERR_INVALID, "NULL argument");
  int rc = nccl_load();
  if (rc) return rc;
  comm_release(h);
  h->comm = nccl_comm;
  h->comm_rank = rank;
  h->comm_world = world;
  return CASA_OK;
}

extern "C" int casa_comm_destroy(casa_handle* h) {
  if (!h) return fail(CASA_ERR_INVALID, "NULL argument");
  if (h->gather_stream) CUDA_TRY(cudaStreamSynchronize(h->gather_stream));
  comm_release(h);
  return CASA_OK;
}

extern "C" int casa_allgather_points(casa_handle* h, void* nccl_comm, const float* local, float* gathered,
                                     int64_t floats_per_rank, void* stream) {
  if (!h || !local || !gathered) return fail(CASA_ERR_INVALID, "NULL argument");
  if (floats_per_rank < 0) return fail(CASA_ERR_INVALID, "floats_per_rank=%lld", (long long)floats_per_rank);
  void* comm = nccl_comm ? nccl_comm : h->comm;
  if (!comm) return fail(CASA_ERR_INVALID, "no communicator: call casa_comm_init / casa_comm_attach or pass an ncclComm_t");
  int rc = nccl_load();
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  NCCL_TRY(g_nccl.AllGather(local, gathered, (size_t)floats_per_rank, /* ncclFloat32 */ 7, comm, (cudaStream_t)stream));
  return CASA_OK;
}

extern "C" int casa_allgather_points_overlapped(casa_handle* h, const float* local, float* gathered, int64_t floats_per_rank,
                                                void* after_stream, int slot) {
  if (!h || !local || !gathered) return fail(CASA_ERR_INVALID, "NULL argument");
  if (slot < 0 || slot >= 8) return fail(CASA_ERR_INVALID, "slot %d outside 0..7", slot);
  if (!h->comm) return fail(CASA_ERR_INVALID, "no communicator: call casa_comm_init / casa_comm_attach first");
  CUDA_TRY(cudaSetDevice(h->device));
  if (!h->gather_stream) {
    CUDA_TRY(cudaStreamCreateWithFlags(&h->gather_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 8; ++i) {
      CUDA_TRY(cudaEventCreateWithFlags(&h->gather_after[i], cudaEventDisableTiming));
      CUDA_TRY(cudaEventCreateWithFlags(&h->gather_done[i], cudaEventDisableTiming));
    }
  }
  // the gather stream waits only for what is queued on `after_stream` right now (the vote that produced `local`), so the
  // exchange of step i overlaps the voting of step i + 1 and no compute stream ever waits for a peer
  if (h->async_mode >= 2 && h->lane_last >= 0) after_stream = (void*)h->lane[h->lane_last]->own_stream;  // the vote ran there
  CUDA_TRY(cudaEventRecord(h->gather_after[slot], (cudaStream_t)after_stream));
  CUDA_TRY(cudaStreamWaitEvent(h->gather_stream, h->gather_after[slot], 0));
  NCCL_TRY(g_nccl.AllGather(local, gathered, (size_t)floats_per_rank, 7, h->comm, h->gather_stream));
  CUDA_TRY(cudaEventRecord(h->gather_done[slot], h->gather_stream));
  return CASA_OK;
}

extern "C" int casa_gather_wait(casa_handle* h, int slot, void* stream) {
  if (!h) return fail(CASA_ERR_INVALID, "NULL argument");
  if (slot < 0 || slot >= 8 || !h->gather_done[slot]) return fail(CASA_ERR_INVALID, "slot %d has no gather in flight", slot);
  CUDA_TRY(cudaSetDevice(h->device));
  if (stream == (void*)-1)
    CUDA_TRY(cudaEventSynchronize(h->gather_done[slot]));                       // host wait
  else
    CUDA_TRY(cudaStreamWaitEvent((cudaStream_t)stream, h->gather_done[slot], 0));  // `stream` waits, the host does not
  return CASA_OK;
}

// ------------------------------------------------------------------------------------------------ self tests

extern "C" int casa_selftest_filter(casa_handle* h, uint64_t n, uint64_t seed, float inlier_thresh, float spread,
                                    uint64_t* out4_host) {
  if (!h || !out4_host) return fail(CASA_ERR_INVALID, "NULL argument");
  CUDA_TRY(cudaSetDevice(h->device));
  const FilterConsts fc = filter_consts(inlier_thresh, 0);
  if (!fc.fast_ok) return fail(CASA_ERR_INVALID, "inlier_thresh=%g is outside the filtered range", inlier_thresh);
  unsigned long long* dout = nullptr;
  CUDA_TRY(cudaMalloc(&dout, 4 * 8));
  CUDA_TRY(cudaMemset(dout, 0, 4 * 8));
  k_selftest_filter<<<h->sm_count * 8, 256>>>(n, (uint32_t)seed, (uint32_t)(seed >> 32), fc, acos((double)inlier_thresh), spread, dout);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpy(out4_host, dout, 4 * 8, cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaFree(dout));
  return CASA_OK;
}

extern "C" int casa_measure_fp32_peak(casa_handle* h, int variant, double* tflops, double* ms_out) {
  if (!h || !tflops) return fail(CASA_ERR_INVALID, "NULL argument");
  if (variant != 0) return fail(CASA_ERR_INVALID, "casa_measure_fp32_peak: only variant 0 (FFMA issue rate) is part of the library");
  CUDA_TRY(cudaSetDevice(h->device));
  float* dout = nullptr;
  CUDA_TRY(cudaMalloc(&dout, 4));
  const int iters = 8192, blocks = h->sm_count * 8;
  float best = 1e30f;
  for (int rep = 0; rep < 5; ++rep) {
    CUDA_TRY(cudaEventRecord(h->ev0, 0));
    k_fma_peak<<<blocks, 256>>>(dout, iters, 1e-9f);
    CUDA_TRY(cudaEventRecord(h->ev1, 0));
    CUDA_TRY(cudaEventSynchronize(h->ev1));
    float ms = 0;
    CUDA_TRY(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    if (rep > 0 && ms < best) best = ms;
  }
  CUDA_TRY(cudaFree(dout));
  *tflops = (double)blocks * 256.0 * iters * 32.0 / (best * 1e-3) / 1e12;  // 16 FMA = 32 FLOP per thread-iteration
  if (ms_out) *ms_out = best;
  return CASA_OK;
}
