// C ABI of the B200 join engine (include/gcre_b200.h): host-side orchestration of the CUDA kernels.
// Stands in for JoinExec / PathSet of the reference (src/join_base.cpp, src/gcre_paths.h); no CPU compute path.
#include "../../include/gcre_b200.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <map>
#include <mutex>
#include <set>
#include <unordered_map>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>

#include "common.cuh"
#include "setup_kernels.cuh"
#include "join_dense.cuh"
#include "join_sparse.cuh"
#include "join_sparse_sc.cuh"
#include "value_table.cuh"
#include "decorated.cuh"
#include "perm_gen.cuh"

using namespace gcre;

// ------------------------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------------------------
static thread_local std::string g_last_error;

static int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

#define CK(call)                                                                                         \
  do {                                                                                                   \
    cudaError_t e__ = (call);                                                                            \
    if (e__ != cudaSuccess)                                                                              \
      return fail(e__ == cudaErrorMemoryAllocation ? GCRE_ERR_NOMEM : GCRE_ERR_CUDA, "%s: %s (%s:%d)", #call, \
                  cudaGetErrorString(e__), __FILE__, __LINE__);                                          \
  } while (0)

#define CKS(call)            \
  do {                       \
    int s__ = (call);        \
    if (s__ != GCRE_OK) return s__; \
  } while (0)

// GCRE_TRACE=1: host-side phase timings of every join on stderr (development aid)
struct PhaseTrace {
  bool on;
  std::chrono::steady_clock::time_point t;
  std::string line;
  PhaseTrace() : on(std::getenv("GCRE_TRACE") != nullptr), t(std::chrono::steady_clock::now()) {}
  void mark(const char* name) {
    if (!on) return;
    const auto now = std::chrono::steady_clock::now();
    char buf[64];
    snprintf(buf, sizeof buf, " %s=%.3f", name, std::chrono::duration<double, std::milli>(now - t).count());
    line += buf;
    t = now;
  }
  void done(const char* what) {  // tagged with the calling thread and the wall clock, so interleaved execs can be told apart
    if (!on) return;
    const double at = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
    fprintf(stderr, "[gcre trace] t=%.3f thr=%04zx %s:%s\n", std::fmod(at, 1e6), std::hash<std::thread::id>()(std::this_thread::get_id()) & 0xffff, what,
            line.c_str());
  }
};

static std::atomic<unsigned long long> g_launches{0};
#define LAUNCHED() (g_launches.fetch_add(1, std::memory_order_relaxed))

static inline unsigned grid_for(long long items, int block) { return (unsigned)((items + block - 1) / block); }

// ------------------------------------------------------------------------------------------------------------------
// objects
// ------------------------------------------------------------------------------------------------------------------
struct gcre_exec;

// Process-wide, per-device cache of device blocks keyed by capacity.  Every device allocation of the engine goes through
// it: the level schedule (and every new JoinExec of an R session) allocates and frees the same sizes over and over, and
// going to the driver each time costs milliseconds - with the stream-ordered pool it was measured to stall for 100s of ms
// when the pool had to grow or remap.  A block remembers the stream it was last used on and an event recorded when it was
// freed; a different stream that reuses it first waits on that event (same scheme as PyTorch's caching allocator).
struct CachedBlock {
  void* p;
  size_t cap;
  cudaStream_t stream;
  cudaEvent_t ev;
};

struct BlockCache {
  std::multimap<size_t, CachedBlock> free_blocks;   // capacity -> block
  std::unordered_map<void*, CachedBlock> live;      // blocks currently handed out
  static size_t round_up(size_t b) { return (std::max<size_t>(b, 1) + 511) & ~(size_t)511; }
  cudaError_t alloc(void** out, size_t bytes, cudaStream_t stream) {
    const size_t want = round_up(bytes);
    auto it = free_blocks.lower_bound(want);
    if (it != free_blocks.end() && it->first <= want + want / 8) {  // at most 12.5 % slack
      CachedBlock b = it->second;
      free_blocks.erase(it);
      if (b.stream != stream && b.ev) {
        cudaError_t e = cudaStreamWaitEvent(stream, b.ev, 0);
        if (e != cudaSuccess) return e;
      }
      b.stream = stream;
      live[b.p] = b;
      *out = b.p;
      return cudaSuccess;
    }
    CachedBlock b{nullptr, want, stream, nullptr};
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e == cudaErrorMemoryAllocation && !free_blocks.empty()) {
      cudaGetLastError();
      release_all();
      e = cudaMalloc(&b.p, want);
    }
    if (e != cudaSuccess) return e;
    e = cudaEventCreateWithFlags(&b.ev, cudaEventDisableTiming);
    if (e != cudaSuccess) {
      cudaFree(b.p);
      return e;
    }
    live[b.p] = b;
    *out = b.p;
    return cudaSuccess;
  }
  void free(void* p, cudaStream_t stream) {
    if (!p) return;
    auto it = live.find(p);
    if (it == live.end()) {  // not ours (should not happen): hand it back to the driver
      cudaFree(p);
      return;
    }
    CachedBlock b = it->second;
    live.erase(it);
    b.stream = stream;
    cudaEventRecord(b.ev, stream);
    free_blocks.emplace(b.cap, b);
  }
  // give idle blocks back to the driver, largest first, until at most `limit` bytes stay cached
  void trim(size_t limit) {
    size_t idle = 0;
    for (auto& kv : free_blocks) idle += kv.second.cap;
    while (idle > limit && !free_blocks.empty()) {
      auto it = std::prev(free_blocks.end());
      if (it->second.ev) cudaEventSynchronize(it->second.ev);
      cudaFree(it->second.p);
      cudaEventDestroy(it->second.ev);
      idle -= it->second.cap;
      free_blocks.erase(it);
    }
  }
  void release_all() {
    for (auto& kv : free_blocks) {
      cudaFree(kv.second.p);
      cudaEventDestroy(kv.second.ev);
    }
    free_blocks.clear();
  }
};

static std::mutex g_cache_mu;
static std::map<int, BlockCache> g_cache;  // per device

static size_t cache_limit_bytes() {
  if (const char* e = std::getenv("GCRE_CACHE_MAX_MB")) return (size_t)std::strtoull(e, nullptr, 10) << 20;
  size_t free_b = 0, total_b = 0;
  if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) {
    cudaGetLastError();
    return (size_t)64 << 30;
  }
  return total_b / 2;
}

static cudaError_t dev_alloc(const gcre_exec* ex, void** out, size_t bytes);
static void dev_free(const gcre_exec* ex, void* p);
static void reap_staged(gcre_exec* ex, bool all);
static void free_uidset_buffers(struct gcre_uidset* us);

struct DevBuf {  // grow-only device scratch owned by one exec
  const gcre_exec* owner = nullptr;
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes) {
    if (bytes <= cap) return GCRE_OK;
    dev_free(owner, p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 4 + 256;
    CK(dev_alloc(owner, &p, want));
    cap = want;
    return GCRE_OK;
  }
  void release() {
    dev_free(owner, p);
    p = nullptr;
    cap = 0;
  }
};

namespace gcre_host {
void pack_i32_rows(const int32_t* data, size_t rows, int cols, uint64_t* out, size_t out_stride, int threads);  // host_pack.cpp
}

// Process-wide pools of the small driver objects an exec needs.  Creating and freeing them per exec (page-locked host
// words: ~1 ms for cudaMallocHost, ~0.4 ms for cudaFreeHost; streams, events) was most of the 3-5 ms a vignette-sized run
// took end to end (tools/vignette_breakdown.py); an R session makes one JoinExec per GWASPA() call.
struct HostPools {
  std::mutex mu;
  std::vector<unsigned*> pinned;                              // 16-word page-locked blocks (any device)
  std::map<int, std::vector<cudaStream_t>> streams;           // per device, non-blocking
  std::map<int, std::vector<cudaEvent_t>> timing_events, plain_events;
};
static HostPools g_pools;

// page-locked staging buffers for host-packed uploads (cudaHostAlloc of tens of MB costs milliseconds: allocate once, reuse)
struct PinnedBlock {
  void* p;
  size_t cap;
};
static std::vector<PinnedBlock> g_pinned_big;  // guarded by g_pools.mu

static cudaError_t pinned_big_acquire(size_t bytes, PinnedBlock* out) {
  {
    std::lock_guard<std::mutex> lock(g_pools.mu);
    size_t best = g_pinned_big.size();
    for (size_t i = 0; i < g_pinned_big.size(); i++)
      if (g_pinned_big[i].cap >= bytes && (best == g_pinned_big.size() || g_pinned_big[i].cap < g_pinned_big[best].cap)) best = i;
    if (best != g_pinned_big.size()) {
      *out = g_pinned_big[best];
      g_pinned_big.erase(g_pinned_big.begin() + best);
      return cudaSuccess;
    }
  }
  out->cap = bytes + bytes / 8 + 4096;
  return cudaHostAlloc(&out->p, out->cap, cudaHostAllocDefault);
}
static void pinned_big_release(const PinnedBlock& b) {
  if (!b.p) return;
  std::lock_guard<std::mutex> lock(g_pools.mu);
  g_pinned_big.push_back(b);
}

static cudaError_t pool_pinned(unsigned** out) {
  {
    std::lock_guard<std::mutex> lock(g_pools.mu);
    if (!g_pools.pinned.empty()) {
      *out = g_pools.pinned.back();
      g_pools.pinned.pop_back();
      return cudaSuccess;
    }
  }
  return cudaMallocHost(out, 16 * sizeof(unsigned));
}
static void unpool_pinned(unsigned* p) {
  if (!p) return;
  std::lock_guard<std::mutex> lock(g_pools.mu);
  g_pools.pinned.push_back(p);
}
static cudaError_t pool_stream(int device, cudaStream_t* out) {
  {
    std::lock_guard<std::mutex> lock(g_pools.mu);
    auto& v = g_pools.streams[device];
    if (!v.empty()) {
      *out = v.back();
      v.pop_back();
      return cudaSuccess;
    }
  }
  return cudaStreamCreateWithFlags(out, cudaStreamNonBlocking);
}
static void unpool_stream(int device, cudaStream_t st) {  // the caller has drained it
  if (!st) return;
  std::lock_guard<std::mutex> lock(g_pools.mu);
  g_pools.streams[device].push_back(st);
}
static cudaError_t pool_event(int device, bool timing, cudaEvent_t* out) {
  {
    std::lock_guard<std::mutex> lock(g_pools.mu);
    auto& v = (timing ? g_pools.timing_events : g_pools.plain_events)[device];
    if (!v.empty()) {
      *out = v.back();
      v.pop_back();
      return cudaSuccess;
    }
  }
  return timing ? cudaEventCreate(out) : cudaEventCreateWithFlags(out, cudaEventDisableTiming);
}
static void unpool_event(int device, bool timing, cudaEvent_t ev) {
  if (!ev) return;
  std::lock_guard<std::mutex> lock(g_pools.mu);
  (timing ? g_pools.timing_events : g_pools.plain_events)[device].push_back(ev);
}

struct gcre_pathset;
struct gcre_uidset;

constexpr unsigned kSpecCand = 8192;  // candidates copied to the host speculatively with the scalars (192 KB; the joins of the bench append 2,000 - 6,000)

struct gcre_exec {
  int M = 1, n_cases = 0, n_ctrls = 0, n = 0, W64 = 0, Wp = 0, iters = 0, Ip = 0, Iw = 0, device = 0, sm_count = 0;
  // fixed by the shape (and a test hook each) at creation: carrier lists built at one width are read at the same width
  bool wide = false;      // u32 carrier indices in the sparse views and kernels
  bool split_ok = false;  // the split-carrier kernels (join_sparse_sc.cuh) are the sparse form of this exec
  cudaStream_t own_stream = nullptr, stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaEvent_t ev_piece = nullptr;                                  // upload throttling (copy_pieces)
  cudaEvent_t ev_half[2] = {nullptr, nullptr};                     // staging halves of upload_staged's streamed path
  // host -> device uploads run on their own stream so that they never queue behind (or wait for) kernels
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_copy = nullptr, ev_order = nullptr;
  struct Staged {
    void* p;
    cudaEvent_t consumed;
  };
  std::vector<Staged> staged;  // staging blocks whose unpack kernel may still be pending
  // permutation masks
  uint64_t* d_masks = nullptr;  // canonical perm-major [iters][W64]
  uint64_t* d_pm = nullptr;     // word-major [Wp][Ip]
  uint32_t* d_pt = nullptr;     // patient-major [n][Iw], built on first use by a sparse kernel
  bool pt_valid = false;
  // the same matrix with rows of exactly 4 / 8 / 16 words for the split-carrier kernels (<= 512 permutations): at 128-byte rows
  // of which 16 bytes are used the matrix takes eight times the cache it needs (1.28 MB instead of 160 KB at 10,000 patients)
  uint32_t* d_pt_sc = nullptr;
  bool pt_sc_valid = false;
  unsigned long long mask_gen = 1;  // bumped whenever the permutation masks change: per-path-set pre-count tables depend on them
  // strata of the seeded mask generator (gcre_exec_set_permutation_strata); n_strata == 0: one stratum, no arrays
  int n_strata = 0;
  int32_t* d_strata_idx = nullptr;     // [64 * W64] dense stratum of each patient (0 past n)
  uint32_t* d_strata_m = nullptr;      // [64 * W64] m_i | last-of-its-stratum-in-its-word << 31 (0 past n)
  uint64_t* d_strata_peer = nullptr;   // [64 * W64] earlier same-stratum patients of the word, ballot order (perm_gen.cuh)
  int32_t* d_strata_k = nullptr;       // [n_strata] true case count per stratum
  // value table
  double* d_vt = nullptr;
  int vt_rows = 0, vt_cols = 0;
  double* d_diagD = nullptr;
  float* d_diagF = nullptr;
  double* d_diagDM = nullptr;
  float* d_diagFM = nullptr;
  long long diag_cap = -1;
  // outputs / scratch
  int* d_perm_max = nullptr;
  unsigned long long* d_topk = nullptr;  // [0] self-tightening candidate threshold, [1..64] its hash-bucket maxima (JoinParams::slots)
  unsigned* d_scalars = nullptr;  // [0] candidate count, [1] max_total, [2..3] 64-bit work counter of the sparse kernel,
                                  // [4..5] 64-bit count of pairs that took the exact path of the thresholded look-ups (diagnostic)
  DevBuf cand, scratch, scan_tmp;
  DevBuf ident;             // [ident_rows] entries k << 1: the row map of a pre-counted join whose partners are their own rows
  uint32_t ident_rows = 0;
  unsigned* h_scalars = nullptr;  // pinned
  // page-locked landing area of a join's results: [kSpecCand candidates][Ip permutation maxima].  They are copied behind every
  // launch together with the scalars, so a join waits for the device once instead of three times.
  PinnedBlock h_res{nullptr, 0};
  bool h_perm_fresh = false;      // h_res holds the maxima of the last launch of the last join
  // path sets and join indices created from this exec: gcre_exec_destroy frees their device memory and orphans them (ex =
  // nullptr), so destroying the exec first is legal and a later gcre_pathset_destroy only deletes the host object
  mutable std::mutex child_mu;
  mutable std::set<gcre_pathset*> pathsets;
  mutable std::set<gcre_uidset*> uidsets;
};

// Where the rows of a path set came from: what the tail form of the pre-counted sparse kernel (join_sparse.cuh) needs to know
// that a level-4 partner's first gene is its upstream row's last gene.  Entries name rows of a base set (base row << 1 |
// halves swapped, setup_kernels.cuh).  They hold while neither this set nor the base set has been written since: every write
// drops them (rows_written) and bumps the set's version, which names the base's content.
struct Provenance {
  const gcre_pathset* base = nullptr;
  unsigned long long base_uid = 0, base_ver = 0;  // the base set's identity and version when the entries were made
  uint32_t* sel = nullptr;     // gcre_pathset_select: row k is base row sel[k] >> 1 (entries, halves as they are)
  uint32_t* tail = nullptr;    // KEEP join result: per row, its partner's base row (the path's last gene)
  uint32_t* head = nullptr;    // ... and its upstream row's entry when every upstream row was exactly one base row (else null)
  unsigned long long lo = 0, hi = 0;  // rows [lo, hi) carry entries (a sharded join writes only its rows)
  bool single = false;         // every row IS its tail: the upstream rows were all zero (level 1a)
};

struct gcre_pathset {
  const gcre_exec* ex = nullptr;
  uint32_t size = 0;
  uint64_t* d_rows = nullptr;
  unsigned long long uid = 0;  // process-wide unique: a provenance entry cannot mistake a new set at a reused address for its base
  unsigned long long ver = 0;  // bumped by every write of the rows
  bool known_zero = false;     // every row is zero (created and never written)
  Provenance prov;
  long long max_half_pop = 0;  // max carriers in any half-row; -1 = unknown (recomputed on demand)
  bool zero_pending = false;   // rows are logically zero but the memset has not been issued yet (skipped altogether when
                               // the set's first use is as the fully overwritten result of a join)
  SparseView view;             // carrier lists, built on first use by a sparse join
};

// UidRelSet (src/gcre.h:49-90) resident on the device: the flattened join index plus what the pre-checks need.
struct gcre_uidset {
  gcre_exec* ex = nullptr;
  int path_length = 0;
  uint32_t n_uids = 0, n_signs = 0;
  unsigned long long total = 0, n_units_total = 0, max_loc_end = 0, max_res_end = 0;
  bool res_is_prefix = true;   // every path_idx equals the running sum of counts: a full join overwrites rows [0, total)
  DevBuf count, loc, prefix, res, units, unit_idx, signs;
  // Equal upstream rows grouped for the score-only joins over this index (group_upstream_rows), for one version of one upstream
  // set and one row range: rebuilt when any of them changes, reused by the joins of every permutation batch in between
  struct Grouping {
    bool built = false, collide = false;  // collide: built under the test hook that leaves the fingerprints out of the keys
    unsigned long long set_uid = 0, set_ver = 0;
    uint32_t ub = 0, ue = 0;
    unsigned long long n_units = 0;  // the representatives' work units (unit_list)
    uint32_t dedup_rows = 0;         // rows that are members of another row's group
    bool pays = false;               // enough duplicates to pay for the indirection (GROUP_MAX_UNIT_SHARE)
    DevBuf mem_rng, members, unit_list;  // per row the range of its members in `members`; the representatives' units
    mutable std::vector<uint32_t> h_members;  // host copy of `members`, read back when a candidate first needs it (expand_members)
    mutable bool h_members_valid = false;
  };
  mutable Grouping grp;
};

static int materialize_zero(gcre_pathset* ps) {
  if (!ps->zero_pending) return GCRE_OK;
  ps->zero_pending = false;
  const size_t bytes = (size_t)ps->size * ps->ex->Wp * ps->ex->M * 8;
  if (bytes) CK(cudaMemsetAsync(ps->d_rows, 0, bytes, ps->ex->stream));
  return GCRE_OK;
}

static void drop_prov(gcre_pathset* ps) {
  dev_free(ps->ex, ps->prov.sel);
  dev_free(ps->ex, ps->prov.tail);
  dev_free(ps->ex, ps->prov.head);
  ps->prov = Provenance();
}

// the rows of `ps` are (about to be) rewritten: whatever is known of their origin no longer holds
static void rows_written(gcre_pathset* ps) {
  ps->ver++;
  ps->known_zero = false;
  drop_prov(ps);
}

static std::atomic<unsigned long long> g_pathset_uid{0};

// Only the 1,024-permutation kernel has the tail form: at <= 512 permutations (split-carrier kernels) nothing is recorded
static bool provenance_useful(const gcre_exec* ex) { return !ex->split_ok; }

static void drop_view(gcre_pathset* ps) {
  dev_free(ps->ex, ps->view.off);
  dev_free(ps->ex, ps->view.len);
  dev_free(ps->ex, ps->view.ncase);
  dev_free(ps->ex, ps->view.car);
  dev_free(ps->ex, ps->view.pcnt);
  dev_free(ps->ex, ps->view.fp);
  ps->view = SparseView();
}

static int use_device(const gcre_exec* ex) {
  CK(cudaSetDevice(ex->device));
  return GCRE_OK;
}

static cudaError_t dev_alloc(const gcre_exec* ex, void** out, size_t bytes) {
  std::lock_guard<std::mutex> lock(g_cache_mu);
  return g_cache[ex->device].alloc(out, bytes, ex->stream);
}

static void dev_free(const gcre_exec* ex, void* p) {
  if (!p) return;
  std::lock_guard<std::mutex> lock(g_cache_mu);
  g_cache[ex->device].free(p, ex->stream);
}

// a block whose first use is on `stream` (the cache orders it after the block's previous life on any other stream)
static cudaError_t dev_alloc_on(const gcre_exec* ex, void** out, size_t bytes, cudaStream_t stream) {
  std::lock_guard<std::mutex> lock(g_cache_mu);
  return g_cache[ex->device].alloc(out, bytes, stream);
}

// Staging blocks of upload_staged go back to the cache once their unpack kernel has run (or, with `all`, now: the cache
// records the hand-back on ex->stream, behind that kernel).
static void reap_staged(gcre_exec* ex, bool all) {
  size_t kept = 0;
  for (auto& st : ex->staged) {
    if (all || cudaEventQuery(st.consumed) == cudaSuccess) {
      dev_free(ex, st.p);
      cudaEventDestroy(st.consumed);
    } else {
      ex->staged[kept++] = st;
    }
  }
  ex->staged.resize(kept);
  cudaGetLastError();  // cudaErrorNotReady from the queries is not an error
}

// Return every cached (currently unused) device block to the driver.
extern "C" int gcre_release_cached_memory(void) {
  std::lock_guard<std::mutex> lock(g_cache_mu);
  for (auto& kv : g_cache) {
    cudaSetDevice(kv.first);
    cudaDeviceSynchronize();
    kv.second.release_all();
  }
  std::lock_guard<std::mutex> lock2(g_pools.mu);
  for (auto& b : g_pinned_big) cudaFreeHost(b.p);
  g_pinned_big.clear();
  return GCRE_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// misc
// ------------------------------------------------------------------------------------------------------------------
extern "C" const char* gcre_last_error(void) { return g_last_error.c_str(); }
extern "C" const char* gcre_version(void) { return "gcre-b200 0.1 (sm_100a)"; }

extern "C" int gcre_kernel_launch_count(uint64_t* count) {
  if (!count) return fail(GCRE_ERR_ARG, "null argument");
  *count = g_launches.load();
  return GCRE_OK;
}

extern "C" int gcre_device_count(int* count) {
  if (!count) return fail(GCRE_ERR_ARG, "null argument");
  CK(cudaGetDeviceCount(count));
  return GCRE_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// exec
// ------------------------------------------------------------------------------------------------------------------
extern "C" int gcre_exec_create(int method, int num_cases, int num_ctrls, int iters, int device, gcre_exec** out) {
  if (!out) return fail(GCRE_ERR_ARG, "null argument");
  *out = nullptr;
  // src/join_base.cpp:47: check_true(num_cases > 0 && num_ctrls > 0 && iters >= 0)
  if (!(num_cases > 0 && num_ctrls > 0 && iters >= 0)) return fail(GCRE_ERR_ASSERT, "assertion");
  int ndev = 0;
  CK(cudaGetDeviceCount(&ndev));
  if (ndev <= 0) return fail(GCRE_ERR_CUDA, "no CUDA device (this engine has no CPU path)");
  if (device < 0 || device >= ndev) return fail(GCRE_ERR_ARG, "device %d out of range (have %d)", device, ndev);
  gcre_exec* ex = new (std::nothrow) gcre_exec();
  if (!ex) return fail(GCRE_ERR_NOMEM, "host allocation failed");
  ex->M = (method == 1) ? 1 : 2;  // JoinExec::to_method: anything but "method1" is method 2 (src/gcre.h:125-133)
  ex->n_cases = num_cases;
  ex->n_ctrls = num_ctrls;
  ex->n = num_cases + num_ctrls;
  ex->W64 = (ex->n + 63) / 64;
  ex->Wp = (ex->W64 + 1) & ~1;
  ex->iters = iters;
  ex->Ip = ((std::max(iters, 1) + dense::TI - 1) / dense::TI) * dense::TI;
  ex->Iw = ((ex->Ip / 32 + 31) / 32) * 32;  // words per patient row of the patient-major masks: whole 1,024-perm blocks
  // u32 carrier indices when n (which is also the sentinel index) does not fit u16; GCRE_TEST_WIDE_CARRIERS=1 (test hook)
  // forces the u32 path on small cohorts
  ex->wide = ex->n > 65535 || std::getenv("GCRE_TEST_WIDE_CARRIERS") != nullptr;
  // few permutations; GCRE_TEST_NO_SPLIT=1 (test hook) keeps the one-word-per-lane kernel
  ex->split_ok = ex->Ip <= sparse_sc::MAX_PERMS && ex->Iw == 32 && std::getenv("GCRE_TEST_NO_SPLIT") == nullptr;
  ex->device = device;
  int rc = [&]() -> int {
    CK(cudaSetDevice(device));
    CK(cudaDeviceGetAttribute(&ex->sm_count, cudaDevAttrMultiProcessorCount, device));
    CK(pool_stream(device, &ex->own_stream));
    ex->stream = ex->own_stream;
    CK(pool_event(device, true, &ex->ev0));
    CK(pool_event(device, true, &ex->ev1));
    CK(pool_event(device, false, &ex->ev_piece));
    for (auto& e : ex->ev_half) CK(pool_event(device, false, &e));
    CK(pool_stream(device, &ex->copy_stream));
    CK(pool_event(device, false, &ex->ev_copy));
    CK(pool_event(device, false, &ex->ev_order));
    for (DevBuf* b : {&ex->cand, &ex->scratch, &ex->scan_tmp, &ex->ident}) b->owner = ex;
    CK(dev_alloc(ex, (void**)&ex->d_masks, std::max<size_t>((size_t)iters * ex->W64, 1) * 8));
    CK(dev_alloc(ex, (void**)&ex->d_pm, (size_t)ex->Wp * ex->Ip * 8));
    CK(cudaMemsetAsync(ex->d_masks, 0, std::max<size_t>((size_t)iters * ex->W64, 1) * 8, ex->stream));
    CK(cudaMemsetAsync(ex->d_pm, 0, (size_t)ex->Wp * ex->Ip * 8, ex->stream));
    CK(dev_alloc(ex, (void**)&ex->d_perm_max, (size_t)ex->Ip * 4));
    CK(cudaMemsetAsync(ex->d_perm_max, 0, (size_t)ex->Ip * 4, ex->stream));
    CK(dev_alloc(ex, (void**)&ex->d_topk, 65 * sizeof(unsigned long long)));
    CK(dev_alloc(ex, (void**)&ex->d_scalars, 16 * sizeof(unsigned)));
    CK(cudaMemsetAsync(ex->d_scalars, 0, 16 * sizeof(unsigned), ex->stream));
    CK(pool_pinned(&ex->h_scalars));
    return GCRE_OK;  // no host sync: everything later is ordered on ex->stream (gcre_exec_set_stream carries the order over)
  }();
  if (rc != GCRE_OK) {
    gcre_exec_destroy(ex);
    return rc;
  }
  *out = ex;
  return GCRE_OK;
}

extern "C" int gcre_exec_destroy(gcre_exec* ex) {
  if (!ex) return GCRE_OK;
  cudaSetDevice(ex->device);
  if (ex->own_stream) cudaStreamSynchronize(ex->own_stream);
  if (ex->copy_stream) cudaStreamSynchronize(ex->copy_stream);
  reap_staged(ex, true);
  {
    // children outlive the exec as empty shells: their device memory goes back to the cache now
    std::lock_guard<std::mutex> lock(ex->child_mu);
    for (gcre_pathset* ps : ex->pathsets) {
      dev_free(ex, ps->d_rows);
      ps->d_rows = nullptr;
      drop_view(ps);
      drop_prov(ps);
      ps->ex = nullptr;
    }
    for (gcre_uidset* us : ex->uidsets) {
      free_uidset_buffers(us);
      us->ex = nullptr;
    }
    ex->pathsets.clear();
    ex->uidsets.clear();
  }
  for (void* p : {(void*)ex->d_masks, (void*)ex->d_pm, (void*)ex->d_pt, (void*)ex->d_pt_sc, (void*)ex->d_vt, (void*)ex->d_diagD, (void*)ex->d_diagF,
                  (void*)ex->d_diagDM, (void*)ex->d_diagFM, (void*)ex->d_perm_max, (void*)ex->d_scalars, (void*)ex->d_topk, (void*)ex->d_strata_idx,
                  (void*)ex->d_strata_m, (void*)ex->d_strata_peer, (void*)ex->d_strata_k})
    dev_free(ex, p);
  ex->cand.release();
  ex->scan_tmp.release();
  ex->scratch.release();
  ex->ident.release();
  // streams (drained above), events and the page-locked words go back to the process-wide pools
  unpool_pinned(ex->h_scalars);
  pinned_big_release(ex->h_res);
  unpool_event(ex->device, true, ex->ev0);
  unpool_event(ex->device, true, ex->ev1);
  unpool_event(ex->device, false, ex->ev_piece);
  for (auto e : ex->ev_half) unpool_event(ex->device, false, e);
  unpool_event(ex->device, false, ex->ev_copy);
  unpool_event(ex->device, false, ex->ev_order);
  unpool_stream(ex->device, ex->copy_stream);
  unpool_stream(ex->device, ex->own_stream);
  {
    // keep the cache from starving other allocators of the process (torch, NCCL): above GCRE_CACHE_MAX_MB of idle blocks
    // (default: half of the device memory) the largest ones go back to the driver
    std::lock_guard<std::mutex> lock(g_cache_mu);
    g_cache[ex->device].trim(cache_limit_bytes());
  }
  delete ex;
  return GCRE_OK;
}

extern "C" int gcre_exec_get_info(const gcre_exec* ex, gcre_exec_info* out) {
  if (!ex || !out) return fail(GCRE_ERR_ARG, "null argument");
  out->method = ex->M;
  out->num_cases = ex->n_cases;
  out->num_ctrls = ex->n_ctrls;
  out->width_ul = ex->Wp;
  out->iterations = ex->Ip;
  out->iters_requested = ex->iters;
  out->device = ex->device;
  out->sm_count = ex->sm_count;
  return GCRE_OK;
}

extern "C" int gcre_exec_set_stream(gcre_exec* ex, void* cuda_stream) {
  if (!ex) return fail(GCRE_ERR_ARG, "null argument");
  CKS(use_device(ex));
  cudaStream_t next = cuda_stream ? (cudaStream_t)cuda_stream : ex->own_stream;
  if (next != ex->stream) {  // work already queued on the old stream stays ahead of work on the new one (no host sync)
    CK(cudaEventRecord(ex->ev_order, ex->stream));
    CK(cudaStreamWaitEvent(next, ex->ev_order, 0));
  }
  ex->stream = next;
  return GCRE_OK;
}

// Host -> device upload of `n_units` records of `unit_bytes` each, unpacked on the device by
// consume(d_piece, first_unit, units) (a kernel launch on ex->stream).
//
// Up to kWholeBytes the records land in one staging block, copied on the exec's copy stream in 16 MB transfers, and the
// unpack kernel follows on ex->stream behind an event; the host waits for the copies only.  Nothing here waits for a kernel,
// so an upload proceeds at PCIe rate while another exec of the process has the SMs full with a join (a join kernel's
// persistent CTAs hold every register of an SM until the kernel ends; an unpack kernel between two copies would wait for
// that).  Larger inputs stream through
// the two halves of ex->scratch on ex->stream, copy k+1 overlapping kernel k.  Either way the caller's host buffer is free
// on return.
constexpr size_t kCopyBytes = (size_t)16 << 20;
constexpr size_t kWholeBytes = (size_t)2 << 30;
constexpr size_t kStreamedPiece = (size_t)256 << 20;

// One host -> device copy as 16 MB transfers, each issued only when the previous one has finished.  Measured on this box
// (tools/copy_contention.py): a stream with copies queued back to back keeps the copy engine to itself - a 1 MB copy on
// another stream waited 23 ms, the whole 1.2 GB upload, whether that was queued as one transfer or as 8 MB pieces two deep,
// and a high-priority stream changed nothing; with one piece in flight the other stream waits one piece (0.33 ms at 16 MB)
// and the upload still runs at 52 of 55 GB/s.  That matters when a second exec of the process is joining meanwhile.
static int copy_pieces(gcre_exec* ex, void* dst, const void* src, size_t bytes, cudaStream_t stream) {
  for (size_t b0 = 0; b0 < bytes; b0 += kCopyBytes) {
    if (b0) CK(cudaEventSynchronize(ex->ev_piece));
    CK(cudaMemcpyAsync(static_cast<char*>(dst) + b0, static_cast<const char*>(src) + b0, std::min(kCopyBytes, bytes - b0), cudaMemcpyHostToDevice, stream));
    CK(cudaEventRecord(ex->ev_piece, stream));
  }
  return GCRE_OK;
}

template <class Consume>
static int upload_staged(gcre_exec* ex, const void* src, size_t unit_bytes, size_t n_units, Consume&& consume) {
  if (n_units == 0 || unit_bytes == 0) return GCRE_OK;
  const size_t total = unit_bytes * n_units;
  const char* force_streamed = std::getenv("GCRE_TEST_STREAMED_UPLOAD");  // test hook: piece size in bytes for the > 2 GB path
  if (total <= kWholeBytes && !(force_streamed && *force_streamed)) {
    reap_staged(ex, false);
    gcre_exec::Staged st{nullptr, nullptr};
    CK(dev_alloc_on(ex, &st.p, total, ex->copy_stream));
    int rc = [&]() -> int {
      CKS(copy_pieces(ex, st.p, src, total, ex->copy_stream));
      CK(cudaEventRecord(ex->ev_copy, ex->copy_stream));
      CK(cudaStreamWaitEvent(ex->stream, ex->ev_copy, 0));
      CKS(consume(static_cast<const void*>(st.p), (size_t)0, n_units));
      CK(cudaEventCreateWithFlags(&st.consumed, cudaEventDisableTiming));
      CK(cudaEventRecord(st.consumed, ex->stream));
      return GCRE_OK;
    }();
    if (rc != GCRE_OK || !st.consumed) {
      cudaStreamSynchronize(ex->copy_stream);
      cudaStreamSynchronize(ex->stream);
      dev_free(ex, st.p);
      if (st.consumed) cudaEventDestroy(st.consumed);
      return rc != GCRE_OK ? rc : fail(GCRE_ERR_CUDA, "event creation failed");
    }
    ex->staged.push_back(st);
    CK(cudaEventSynchronize(ex->ev_copy));
    return GCRE_OK;
  }
  const size_t piece = (force_streamed && *force_streamed) ? std::max<size_t>(1, std::strtoull(force_streamed, nullptr, 10)) : kStreamedPiece;
  const size_t per = std::max<size_t>(1, piece / unit_bytes);
  const size_t half = (per * unit_bytes + 255) & ~(size_t)255;
  CKS(ex->scratch.ensure(2 * half));
  size_t k = 0;
  for (size_t u0 = 0; u0 < n_units; u0 += per, k++) {
    const size_t nu = std::min(per, n_units - u0);
    char* d_piece = static_cast<char*>(ex->scratch.p) + (k & 1) * half;
    if (k >= 2) CK(cudaEventSynchronize(ex->ev_half[k & 1]));  // the kernel that read this half two pieces ago is done
    CKS(copy_pieces(ex, d_piece, static_cast<const char*>(src) + u0 * unit_bytes, nu * unit_bytes, ex->stream));
    CKS(consume(static_cast<const void*>(d_piece), u0, nu));
    CK(cudaEventRecord(ex->ev_half[k & 1], ex->stream));
  }
  CK(cudaStreamSynchronize(ex->stream));
  return GCRE_OK;
}

extern "C" int gcre_exec_set_value_table(gcre_exec* ex, const double* table, int rows, int cols) {
  if (!ex || (!table && rows > 0 && cols > 0)) return fail(GCRE_ERR_ARG, "null argument");
  if (rows < 0 || cols < 0) return fail(GCRE_ERR_ARG, "negative table size");
  CKS(use_device(ex));
  dev_free(ex, ex->d_vt);  // stream-ordered: the cache guards the block with an event on ex->stream
  ex->d_vt = nullptr;
  // the reference keeps at most the top-left (n+1)x(n+1) block (src/join_base.cpp:74-78); larger inputs are legal
  ex->vt_rows = rows;
  ex->vt_cols = cols;
  const size_t bytes = std::max<size_t>((size_t)rows * cols, 1) * 8;
  CK(dev_alloc_on(ex, (void**)&ex->d_vt, bytes, ex->copy_stream));
  CKS(copy_pieces(ex, ex->d_vt, table, (size_t)rows * cols * 8, ex->copy_stream));
  CK(cudaEventRecord(ex->ev_copy, ex->copy_stream));
  CK(cudaStreamWaitEvent(ex->stream, ex->ev_copy, 0));
  CK(cudaEventSynchronize(ex->ev_copy));  // the caller's table is free again; readers on ex->stream are ordered behind the copy
  ex->diag_cap = -1;  // anti-diagonal tables are rebuilt on the next join
  return GCRE_OK;
}

// log(k!) for k = 0..n with this library's std::lgamma - the table both value-table generators (device and the numpy
// restatement) start from, so that they make identical "probability <= own" decisions at exact ties.
extern "C" int gcre_log_factorial_table(int n, double* out) {
  if (!out || n < 0) return fail(GCRE_ERR_ARG, "bad argument");
  for (int k = 0; k <= n; k++) out[k] = std::lgamma((double)k + 1.0);
  return GCRE_OK;
}

// getValuesTable (R/Utils.R:137-159) on the device: fills this exec's value table for its own (num_cases, num_ctrls).
extern "C" int gcre_exec_generate_value_table(gcre_exec* ex) {
  if (!ex) return fail(GCRE_ERR_ARG, "null argument");
  CKS(use_device(ex));
  CK(cudaStreamSynchronize(ex->stream));
  const int nc = ex->n_cases, nt = ex->n_ctrls, n = ex->n;
  const size_t entries = (size_t)(nc + 1) * (nt + 1);
  dev_free(ex, ex->d_vt);
  ex->d_vt = nullptr;
  CK(dev_alloc(ex, (void**)&ex->d_vt, entries * 8));
  ex->vt_rows = nc + 1;
  ex->vt_cols = nt + 1;
  ex->diag_cap = -1;
  // log-factorials on the host (synth.make_value_table fetches the same table through gcre_log_factorial_table)
  std::vector<double> lf((size_t)n + 1);
  gcre_log_factorial_table(n, lf.data());
  const int m_max = std::min(nc, nt) + 1;
  const int blocks = std::min(n + 1, ex->sm_count * 8);
  double* d_lf = nullptr;
  double* d_scratch = nullptr;
  unsigned long long* d_key = nullptr;
  int rc = [&]() -> int {
    CK(dev_alloc(ex, (void**)&d_lf, ((size_t)n + 1) * 8));
    CK(dev_alloc(ex, (void**)&d_scratch, (size_t)blocks * 3 * m_max * 8));
    CK(dev_alloc(ex, (void**)&d_key, 8));
    CK(cudaMemcpyAsync(d_lf, lf.data(), ((size_t)n + 1) * 8, cudaMemcpyHostToDevice, ex->stream));
    CK(cudaMemsetAsync(d_key, 0, 8, ex->stream));
    // entries no diagonal reaches do not exist in an (nc+1) x (nt+1) table: every (x, y) has total x + y <= n
    value_table_kernel<<<blocks, VT_THREADS, 0, ex->stream>>>(d_lf, nc, nt, ex->d_vt, d_scratch, m_max, d_key);
    CK(cudaGetLastError());
      LAUNCHED();
    value_table_fixup_kernel<<<ex->sm_count * 8, 256, 0, ex->stream>>>(ex->d_vt, entries, d_key);
    CK(cudaGetLastError());
      LAUNCHED();
    CK(cudaStreamSynchronize(ex->stream));
    return GCRE_OK;
  }();
  dev_free(ex, d_lf);
  dev_free(ex, d_scratch);
  dev_free(ex, d_key);
  return rc;
}

// Copy the exec's value table (as supplied or generated) to the host: rows x cols doubles, row-major.
extern "C" int gcre_exec_get_value_table(const gcre_exec* ex, double* out, int rows, int cols) {
  if (!ex || !out) return fail(GCRE_ERR_ARG, "null argument");
  if (rows != ex->vt_rows || cols != ex->vt_cols || !ex->d_vt) return fail(GCRE_ERR_ASSERT, "assertion");
  CKS(use_device(ex));
  CK(cudaMemcpyAsync(out, ex->d_vt, (size_t)rows * cols * 8, cudaMemcpyDeviceToHost, ex->stream));
  CK(cudaStreamSynchronize(ex->stream));
  return GCRE_OK;
}

// Scratch budget of the decorated p-value calls: splits run in chunks whose scratch fits it (one larger split runs alone).
// GCRE_TEST_DECORATED_SCRATCH (test hook, bytes; read per call) shrinks it so that a short list spans several chunks.
static size_t decorated_scratch_budget() {
  if (const char* e = std::getenv("GCRE_TEST_DECORATED_SCRATCH")) return std::max<size_t>(1, std::strtoull(e, nullptr, 10));
  return (size_t)256 << 20;
}

// decorated_exact_kernel over ni packed splits (d_rows [ni][4][W64]); d_scr: ni * 2 * (n + 1) doubles
static int launch_decorated_exact(gcre_exec* ex, const uint64_t* d_rows, uint32_t ni, double* d_scr, DecoratedOut* d_out) {
  if (ex->M == 1)
    decorated_exact_kernel<1><<<ni, DEC_THREADS, 0, ex->stream>>>(d_rows, ni, ex->W64, ex->n_cases, ex->n_ctrls, ex->d_vt, ex->vt_rows, ex->vt_cols, d_scr, d_out);
  else
    decorated_exact_kernel<2><<<ni, DEC_THREADS, 0, ex->stream>>>(d_rows, ni, ex->W64, ex->n_cases, ex->n_ctrls, ex->d_vt, ex->vt_rows, ex->vt_cols, d_scr, d_out);
  CK(cudaGetLastError());
  LAUNCHED();
  return GCRE_OK;
}

// computeDecoratedPvalue (R/DecoratedPvalue.R:198-304) in its exact limit for n_items splits; see decorated.cuh.
extern "C" int gcre_exec_decorated_exact(gcre_exec* ex, const uint64_t* rows, uint32_t n_items, gcre_decorated* out) {
  static_assert(sizeof(gcre_decorated) == sizeof(DecoratedOut), "gcre_decorated layout");
  if (!ex || ((!rows || !out) && n_items)) return fail(GCRE_ERR_ARG, "null argument");
  CKS(use_device(ex));
  if (!ex->d_vt) return fail(GCRE_ERR_ASSERT, "assertion");  // no value table set
  if (!n_items) return GCRE_OK;
  const size_t per_item = 2 * ((size_t)ex->n + 1) * 8;                                  // scratch: two probability vectors
  const uint32_t chunk = (uint32_t)std::max<size_t>(1, std::min<size_t>(n_items, decorated_scratch_budget() / per_item));
  void *d_rows = nullptr, *d_scr = nullptr, *d_out = nullptr;
  int rc = [&]() -> int {
    CK(dev_alloc(ex, &d_rows, (size_t)chunk * 4 * ex->W64 * 8));
    CK(dev_alloc(ex, &d_scr, (size_t)chunk * per_item));
    CK(dev_alloc(ex, &d_out, (size_t)chunk * sizeof(DecoratedOut)));
    for (uint32_t i0 = 0; i0 < n_items; i0 += chunk) {
      const uint32_t ni = std::min(chunk, n_items - i0);
      CK(cudaMemcpyAsync(d_rows, rows + (size_t)i0 * 4 * ex->W64, (size_t)ni * 4 * ex->W64 * 8, cudaMemcpyHostToDevice, ex->stream));
      CKS(launch_decorated_exact(ex, (const uint64_t*)d_rows, ni, (double*)d_scr, (DecoratedOut*)d_out));
      CK(cudaMemcpyAsync(out + i0, d_out, (size_t)ni * sizeof(DecoratedOut), cudaMemcpyDeviceToHost, ex->stream));
      CK(cudaStreamSynchronize(ex->stream));
    }
    return GCRE_OK;
  }();
  dev_free(ex, d_rows);
  dev_free(ex, d_scr);
  dev_free(ex, d_out);
  return rc;
}

// Decorated p-values of whole paths given as gene rows of a path set; see gcre_b200.h and decorated.cuh.
extern "C" int gcre_exec_decorated_paths(gcre_exec* ex, const gcre_pathset* genes, const int32_t* gene_idx, const int32_t* signs,
                                         const int32_t* lengths, uint32_t n_paths, int stratified, gcre_decorated* out) {
  if (!ex || !genes) return fail(GCRE_ERR_ARG, "null argument");
  if (n_paths && (!gene_idx || !lengths || !out || (ex->M == 2 && !signs))) return fail(GCRE_ERR_ARG, "null argument");
  if (genes->ex != ex) return fail(GCRE_ERR_ARG, "the gene rows belong to another exec");
  if (stratified != 0 && stratified != 1) return fail(GCRE_ERR_ARG, "stratified must be 0 or 1");
  if (!n_paths) return GCRE_OK;
  CKS(use_device(ex));
  if (!ex->d_vt) return fail(GCRE_ERR_ASSERT, "assertion");  // no value table set
  // splits in the order of decorated_pvalues_for_path: forward j = 1 .. L-1 (genes 0 .. j-1, then gene j), backward j = L-1 .. 1
  // (genes L-1 .. j, then gene j-1); slot[i] = path * 8 + split
  std::vector<DecSplit> splits;
  std::vector<uint32_t> slot;
  splits.reserve((size_t)n_paths * 4);
  for (uint32_t p = 0; p < n_paths; p++) {
    const int L = lengths[p];
    if (L < 1 || L > 5) return fail(GCRE_ERR_RANGE, "path %u: length %d is outside 1..5", p, L);
    const int32_t* g = gene_idx + (size_t)p * 5;
    int neg = 0;
    for (int j = 0; j < L; j++) {
      if (g[j] < 0 || (uint32_t)g[j] >= genes->size) return fail(GCRE_ERR_RANGE, "path %u: gene index %d is outside the gene rows", p, g[j]);
      if (ex->M == 2) {
        const int sg = signs[(size_t)p * 5 + j];
        if (sg != 1 && sg != -1) return fail(GCRE_ERR_ARG, "path %u: sign %d is not +1 / -1", p, sg);
        if (sg == -1) neg |= 1 << j;
      }
    }
    uint32_t k = 0;
    for (int j = 1; j < L; j++, k++) {
      DecSplit s{};
      for (int i = 0; i <= j; i++) s.gene[i] = g[i];
      s.n_sub = j;
      s.neg = neg & ((1 << (j + 1)) - 1);
      splits.push_back(s);
      slot.push_back(p * 8 + k);
    }
    for (int j = L - 1; j >= 1; j--, k++) {
      DecSplit s{};
      for (int i = L - 1; i >= j - 1; i--) {  // genes L-1 .. j, then gene j-1
        const int at = L - 1 - i;
        s.gene[at] = g[i];
        s.neg |= ((neg >> i) & 1) << at;
      }
      s.n_sub = L - j;
      splits.push_back(s);
      slot.push_back(p * 8 + k);
    }
  }
  CKS(materialize_zero(const_cast<gcre_pathset*>(genes)));
  std::memset(out, 0, (size_t)n_paths * 8 * sizeof(gcre_decorated));
  const uint32_t n_items = (uint32_t)splits.size();
  if (!n_items) return GCRE_OK;
  const uint64_t* d_genes = genes->d_rows;
  const size_t stride = (size_t)ex->Wp * ex->M;  // row_words: gene rows are read in place
  std::vector<DecoratedOut> res(n_items);
  void *d_splits = nullptr, *d_a = nullptr, *d_b = nullptr, *d_out = nullptr, *d_tot = nullptr, *d_sizes = nullptr, *d_off = nullptr;
  int rc = [&]() -> int {
    CK(dev_alloc(ex, &d_splits, (size_t)n_items * sizeof(DecSplit)));
    CK(cudaMemcpyAsync(d_splits, splits.data(), (size_t)n_items * sizeof(DecSplit), cudaMemcpyHostToDevice, ex->stream));
    const DecSplit* sp = (const DecSplit*)d_splits;
    if (!stratified) {  // form the packed splits on the device, then the kernel of gcre_exec_decorated_exact unchanged
      const size_t per_item = 4 * (size_t)ex->W64 * 8 + 2 * ((size_t)ex->n + 1) * 8;
      const uint32_t chunk = (uint32_t)std::max<size_t>(1, std::min<size_t>(n_items, decorated_scratch_budget() / per_item));
      CK(dev_alloc(ex, &d_a, (size_t)chunk * 4 * ex->W64 * 8));
      CK(dev_alloc(ex, &d_b, (size_t)chunk * 2 * ((size_t)ex->n + 1) * 8));
      CK(dev_alloc(ex, &d_out, (size_t)chunk * sizeof(DecoratedOut)));
      for (uint32_t i0 = 0; i0 < n_items; i0 += chunk) {
        const uint32_t ni = std::min(chunk, n_items - i0);
        decorated_form_kernel<<<ni, DEC_THREADS, 0, ex->stream>>>(d_genes, stride, sp + i0, ni, ex->W64, (uint64_t*)d_a);
        CK(cudaGetLastError());
        LAUNCHED();
        CKS(launch_decorated_exact(ex, (const uint64_t*)d_a, ni, (double*)d_b, (DecoratedOut*)d_out));
        CK(cudaMemcpyAsync(res.data() + i0, d_out, (size_t)ni * sizeof(DecoratedOut), cudaMemcpyDeviceToHost, ex->stream));
      }
      CK(cudaStreamSynchronize(ex->stream));
      return GCRE_OK;
    }
    // stratified: one stratum when none is set; the per-patient dense indices of gcre_exec_set_permutation_strata otherwise
    const int S = ex->n_strata > 1 ? ex->n_strata : 1;
    const int32_t* d_strata = ex->n_strata > 1 ? ex->d_strata_idx : nullptr;
    CK(dev_alloc(ex, &d_tot, (size_t)S * 2 * 4));
    if (d_strata) {
      CK(cudaMemsetAsync(d_tot, 0, (size_t)S * 2 * 4, ex->stream));
      strata_totals_kernel<<<grid_for(ex->n, 256), 256, 0, ex->stream>>>(d_strata, ex->n, ex->n_cases, (int*)d_tot);
      CK(cudaGetLastError());
      LAUNCHED();
    } else {
      const int one[2] = {ex->n_cases, ex->n_ctrls};
      CK(cudaMemcpyAsync(d_tot, one, sizeof(one), cudaMemcpyHostToDevice, ex->stream));
    }
    std::vector<int4> sizes(n_items);
    CK(dev_alloc(ex, &d_sizes, (size_t)n_items * sizeof(int4)));
    decorated_strata_count_kernel<<<n_items, DEC_THREADS, (size_t)4 * S * 4, ex->stream>>>(d_genes, stride, sp, n_items, ex->W64, ex->n_cases, ex->n, d_strata, S,
                                                                                          (const int*)d_tot, (int4*)d_sizes);
    CK(cudaGetLastError());
    LAUNCHED();
    CK(cudaMemcpyAsync(sizes.data(), d_sizes, (size_t)n_items * sizeof(int4), cudaMemcpyDeviceToHost, ex->stream));
    CK(cudaStreamSynchronize(ex->stream));
    for (uint32_t i = 0; i < n_items; i++)
      if (sizes[i].w >= 0)  // R's sample() stops here ("cannot take a sample larger than the population")
        return fail(GCRE_ERR_RANGE, "path %u split %u: stratum %d has fewer free patients than carriers to redraw", slot[i] / 8, slot[i] % 8, sizes[i].w);
    // chunks whose joint-distribution scratch fits the budget; off[i] = split i's scratch offset (doubles) inside its chunk
    std::vector<unsigned long long> off(n_items);
    std::vector<uint32_t> cuts{0};
    const size_t budget = decorated_scratch_budget();
    size_t used = 0, most = 0;
    for (uint32_t i = 0; i < n_items; i++) {
      const size_t need = dec_joint_scratch(sizes[i].x, sizes[i].y);
      if (i > cuts.back() && (used + need) * 8 > budget) {
        cuts.push_back(i);
        used = 0;
      }
      off[i] = used;
      used += need;
      most = std::max(most, used);
    }
    cuts.push_back(n_items);
    CK(dev_alloc(ex, &d_off, (size_t)n_items * 8));
    CK(cudaMemcpyAsync(d_off, off.data(), (size_t)n_items * 8, cudaMemcpyHostToDevice, ex->stream));
    CK(dev_alloc(ex, &d_b, most * 8));
    CK(dev_alloc(ex, &d_out, (size_t)n_items * sizeof(DecoratedOut)));
    const size_t smem = (size_t)5 * S * 4;
    for (size_t c = 0; c + 1 < cuts.size(); c++) {
      const uint32_t i0 = cuts[c], ni = cuts[c + 1] - cuts[c];
      if (ex->M == 1)
        decorated_strata_joint_kernel<1><<<ni, DEC_THREADS, smem, ex->stream>>>(d_genes, stride, sp + i0, ni, ex->W64, ex->n_cases, ex->n_ctrls, d_strata, S,
                                                                                (const int*)d_tot, ex->d_vt, ex->vt_rows, ex->vt_cols,
                                                                                (const unsigned long long*)d_off + i0, (double*)d_b, (DecoratedOut*)d_out + i0);
      else
        decorated_strata_joint_kernel<2><<<ni, DEC_THREADS, smem, ex->stream>>>(d_genes, stride, sp + i0, ni, ex->W64, ex->n_cases, ex->n_ctrls, d_strata, S,
                                                                                (const int*)d_tot, ex->d_vt, ex->vt_rows, ex->vt_cols,
                                                                                (const unsigned long long*)d_off + i0, (double*)d_b, (DecoratedOut*)d_out + i0);
      CK(cudaGetLastError());
      LAUNCHED();
    }
    CK(cudaMemcpyAsync(res.data(), d_out, (size_t)n_items * sizeof(DecoratedOut), cudaMemcpyDeviceToHost, ex->stream));
    CK(cudaStreamSynchronize(ex->stream));
    return GCRE_OK;
  }();
  for (void* p : {d_splits, d_a, d_b, d_out, d_tot, d_sizes, d_off}) dev_free(ex, p);
  if (rc != GCRE_OK) return rc;
  for (uint32_t i = 0; i < n_items; i++) std::memcpy(&out[slot[i]], &res[i], sizeof(gcre_decorated));
  return GCRE_OK;
}

static int rebuild_mask_layouts(gcre_exec* ex) {
  CK(cudaMemsetAsync(ex->d_pm, 0, (size_t)ex->Wp * ex->Ip * 8, ex->stream));
  if (ex->iters > 0) {
    dim3 blk(32, 8), grd((ex->iters + 31) / 32, (ex->W64 + 31) / 32);
    masks_to_word_major_kernel<<<grd, blk, 0, ex->stream>>>(ex->d_masks, ex->iters, ex->W64, ex->d_pm, ex->Wp, ex->Ip);
    CK(cudaGetLastError());
      LAUNCHED();
  }
  ex->pt_valid = ex->pt_sc_valid = false;
  ex->mask_gen++;
  return GCRE_OK;
}

// the patient-major masks of the split-carrier kernels (d_pt_sc) or of the others (d_pt)
static int ensure_patient_major(gcre_exec* ex, bool split) {
  bool& valid = split ? ex->pt_sc_valid : ex->pt_valid;
  if (valid) return GCRE_OK;
  uint32_t*& pt = split ? ex->d_pt_sc : ex->d_pt;
  const int iw = split ? sparse_sc_words(ex->Ip) : ex->Iw;
  // n + 1 rows: row n is all zero and is what the sentinel entries that pad the carrier lists point at
  if (!pt) CK(dev_alloc(ex, (void**)&pt, (size_t)(ex->n + 1) * iw * 4));
  CK(cudaMemsetAsync(pt + (size_t)ex->n * iw, 0, (size_t)iw * 4, ex->stream));
  const long long warps = (long long)iw * ((ex->n + 31) / 32);
  masks_to_patient_major_kernel<<<grid_for(warps * 32, 256), 256, 0, ex->stream>>>(ex->d_masks, ex->iters, ex->W64, ex->n, pt, iw);
  CK(cudaGetLastError());
  LAUNCHED();
  valid = true;
  return GCRE_OK;
}

extern "C" int gcre_exec_set_permuted_cases_i32(gcre_exec* ex, const int32_t* perm, int rows, int cols) {
  if (!ex || (!perm && rows > 0)) return fail(GCRE_ERR_ARG, "null argument");
  if (rows < 0 || cols < 0) return fail(GCRE_ERR_ARG, "negative size");
  CKS(use_device(ex));
  const int have = std::min(rows, ex->iters);
  // src/join_base.cpp:101: check_equal(num_cases + num_ctrls, data[r].size())
  if (have > 0 && cols != ex->n) return fail(GCRE_ERR_ASSERT, "assertion");
  // src/join_base.cpp:116-123 would divide by zero with no rows and iters > 0 (SURVEY App. D8): reject instead
  if (ex->iters > 0 && rows == 0) return fail(GCRE_ERR_ASSERT, "assertion");
  CK(cudaMemsetAsync(ex->d_masks, 0, std::max<size_t>((size_t)ex->iters * ex->W64, 1) * 8, ex->stream));
  CKS(upload_staged(ex, perm, (size_t)cols * 4, (size_t)std::max(have, 0), [&](const void* d_piece, size_t r0, size_t nr) {
    const long long warps = (long long)nr * ex->W64;
    pack_perm_i32_kernel<<<grid_for(warps * 32, 256), 256, 0, ex->stream>>>((const int32_t*)d_piece, (int)nr, cols, ex->n_cases, ex->W64, ex->d_masks,
                                                                           (int)r0);
    CK(cudaGetLastError());
    LAUNCHED();
    return (int)GCRE_OK;
  }));
  if (have < ex->iters) {
    cycle_perm_rows_kernel<<<grid_for((long long)(ex->iters - have) * ex->W64, 256), 256, 0, ex->stream>>>(ex->d_masks, have, ex->iters, ex->W64);
    CK(cudaGetLastError());
      LAUNCHED();
  }
  CKS(rebuild_mask_layouts(ex));
  return GCRE_OK;  // `perm` has been read (upload_staged waits for its copies); the kernels stay queued on ex->stream
}

extern "C" int gcre_exec_set_permuted_masks_u64(gcre_exec* ex, const uint64_t* masks, int n_perms) {
  if (!ex || (!masks && n_perms > 0)) return fail(GCRE_ERR_ARG, "null argument");
  CKS(use_device(ex));
  if (ex->iters > 0 && n_perms <= 0) return fail(GCRE_ERR_ASSERT, "assertion");
  const int have = std::min(n_perms, ex->iters);
  CK(cudaMemsetAsync(ex->d_masks, 0, std::max<size_t>((size_t)ex->iters * ex->W64, 1) * 8, ex->stream));
  if (have > 0) CKS(copy_pieces(ex, ex->d_masks, masks, (size_t)have * ex->W64 * 8, ex->stream));
  if (have < ex->iters) {
    cycle_perm_rows_kernel<<<grid_for((long long)(ex->iters - have) * ex->W64, 256), 256, 0, ex->stream>>>(ex->d_masks, have, ex->iters, ex->W64);
    CK(cudaGetLastError());
      LAUNCHED();
  }
  CKS(rebuild_mask_layouts(ex));
  CK(cudaStreamSynchronize(ex->stream));
  return GCRE_OK;
}

// The same from a buffer in this exec's device memory (permutation batches that stay resident; multi-GPU fan-out).  Ordered on
// the exec's stream; no host wait.
extern "C" int gcre_exec_set_permuted_masks_device(gcre_exec* ex, const uint64_t* d_masks, int n_perms) {
  if (!ex || (!d_masks && n_perms > 0)) return fail(GCRE_ERR_ARG, "null argument");
  CKS(use_device(ex));
  if (ex->iters > 0 && n_perms <= 0) return fail(GCRE_ERR_ASSERT, "assertion");
  const int have = std::min(n_perms, ex->iters);
  CK(cudaMemsetAsync(ex->d_masks, 0, std::max<size_t>((size_t)ex->iters * ex->W64, 1) * 8, ex->stream));
  if (have > 0) CK(cudaMemcpyAsync(ex->d_masks, d_masks, (size_t)have * ex->W64 * 8, cudaMemcpyDeviceToDevice, ex->stream));
  if (have < ex->iters) {
    cycle_perm_rows_kernel<<<grid_for((long long)(ex->iters - have) * ex->W64, 256), 256, 0, ex->stream>>>(ex->d_masks, have, ex->iters, ex->W64);
    CK(cudaGetLastError());
    LAUNCHED();
  }
  CKS(rebuild_mask_layouts(ex));
  return GCRE_OK;
}

static void free_strata(gcre_exec* ex) {
  for (void* p : {(void*)ex->d_strata_idx, (void*)ex->d_strata_m, (void*)ex->d_strata_peer, (void*)ex->d_strata_k}) dev_free(ex, p);
  ex->d_strata_idx = ex->d_strata_k = nullptr;
  ex->d_strata_m = nullptr;
  ex->d_strata_peer = nullptr;
  ex->n_strata = 0;
}

// Strata of the seeded generator: per-patient arrays of perm_gen.cuh, built on the host once per setting (O(n)).
extern "C" int gcre_exec_set_permutation_strata(gcre_exec* ex, const int32_t* labels, int n) {
  if (!ex) return fail(GCRE_ERR_ARG, "null argument");
  if (!labels && n == 0) {
    CKS(use_device(ex));
    free_strata(ex);
    return GCRE_OK;
  }
  if (n != ex->n) return fail(GCRE_ERR_ASSERT, "assertion");
  if (!labels) return fail(GCRE_ERR_ARG, "null argument");
  // dense stratum index in order of first appearance: only the partition matters
  std::unordered_map<int32_t, int> dense;
  std::vector<int> g((size_t)n);
  for (int i = 0; i < n; i++) {
    g[i] = dense.emplace(labels[i], (int)dense.size()).first->second;
    if ((int)dense.size() > PG_MAX_STRATA) return fail(GCRE_ERR_RANGE, "more than %d strata", PG_MAX_STRATA);
  }
  CKS(use_device(ex));
  free_strata(ex);
  const int S = (int)dense.size();
  if (S <= 1) return GCRE_OK;  // one stratum: the arrays would say what the unstratified kernel assumes
  const size_t np = (size_t)ex->W64 * 64;
  std::vector<int32_t> idx(np, 0), k_init((size_t)S, 0);
  std::vector<uint32_t> m(np, 0), after((size_t)S, 0);
  std::vector<uint64_t> peer(np, 0), seen((size_t)S, 0);
  std::vector<int> stamp((size_t)S, -1);
  for (int i = n - 1; i >= 0; i--) m[i] = ++after[g[i]];
  for (int i = 0; i < ex->n_cases; i++) k_init[g[i]]++;
  for (int w = 0; w < ex->W64; w++) {
    const int a = w * 64, b = std::min(n, a + 64);
    for (int i = a; i < b; i++) {
      const int p = i - a;
      idx[i] = g[i];
      peer[i] = seen[g[i]];
      seen[g[i]] |= 1ull << ((p & 1) * 32 + (p >> 1));  // ballot order: lane p/2, half p%2
    }
    for (int i = b - 1; i >= a; i--) {
      if (stamp[g[i]] != w) m[i] |= 1u << 31;  // last of its stratum in this word
      stamp[g[i]] = w;
      seen[g[i]] = 0;
    }
  }
  CK(dev_alloc(ex, (void**)&ex->d_strata_idx, np * 4));
  CK(dev_alloc(ex, (void**)&ex->d_strata_m, np * 4));
  CK(dev_alloc(ex, (void**)&ex->d_strata_peer, np * 8));
  CK(dev_alloc(ex, (void**)&ex->d_strata_k, (size_t)S * 4));
  CK(cudaMemcpyAsync(ex->d_strata_idx, idx.data(), np * 4, cudaMemcpyHostToDevice, ex->stream));
  CK(cudaMemcpyAsync(ex->d_strata_m, m.data(), np * 4, cudaMemcpyHostToDevice, ex->stream));
  CK(cudaMemcpyAsync(ex->d_strata_peer, peer.data(), np * 8, cudaMemcpyHostToDevice, ex->stream));
  CK(cudaMemcpyAsync(ex->d_strata_k, k_init.data(), (size_t)S * 4, cudaMemcpyHostToDevice, ex->stream));
  CK(cudaStreamSynchronize(ex->stream));  // the host vectors go out of scope
  ex->n_strata = S;  // only now: a failure above leaves one stratum
  return GCRE_OK;
}

extern "C" int gcre_exec_generate_permuted_masks(gcre_exec* ex, uint64_t seed, uint64_t first_perm) {
  if (!ex) return fail(GCRE_ERR_ARG, "null argument");
  if (ex->iters == 0) return GCRE_OK;
  CKS(use_device(ex));
  const unsigned grid = grid_for(ex->iters, PG_WARPS);
  if (ex->n_strata > 1)
    perm_gen_kernel<true><<<grid, PG_WARPS * 32, (size_t)PG_WARPS * ex->n_strata * 4, ex->stream>>>(
        ex->d_masks, ex->iters, ex->W64, ex->n, ex->n_cases, seed, first_perm, (const int2*)ex->d_strata_idx, (const uint2*)ex->d_strata_m,
        (const ulonglong2*)ex->d_strata_peer, ex->d_strata_k, ex->n_strata);
  else
    perm_gen_kernel<false><<<grid, PG_WARPS * 32, 0, ex->stream>>>(ex->d_masks, ex->iters, ex->W64, ex->n, ex->n_cases, seed, first_perm, nullptr,
                                                                   nullptr, nullptr, nullptr, 0);
  CK(cudaGetLastError());
  LAUNCHED();
  CKS(rebuild_mask_layouts(ex));  // bumps mask_gen: count tables built against the previous masks are not reused
  return GCRE_OK;
}

extern "C" int gcre_exec_get_permuted_masks(const gcre_exec* ex, uint64_t* out, int n_perms) {
  if (!ex || (!out && n_perms > 0)) return fail(GCRE_ERR_ARG, "null argument");
  if (n_perms < 0 || n_perms > ex->iters) return fail(GCRE_ERR_RANGE, "assertion");
  if (n_perms == 0) return GCRE_OK;
  CKS(use_device(ex));
  CK(cudaMemcpyAsync(out, ex->d_masks, (size_t)n_perms * ex->W64 * 8, cudaMemcpyDeviceToHost, ex->stream));
  CK(cudaStreamSynchronize(ex->stream));
  return GCRE_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// path sets
// ------------------------------------------------------------------------------------------------------------------
static inline size_t row_words(const gcre_exec* ex) { return (size_t)ex->Wp * ex->M; }

// clear bits at patient indices >= n in rows [row0, row0 + rows) (packed inputs / raw row writes may carry them)
static int mask_tail(const gcre_exec* ex, gcre_pathset* ps, uint32_t row0, uint32_t rows);

extern "C" int gcre_pathset_create(const gcre_exec* ex, uint32_t size, gcre_pathset** out) {
  if (!ex || !out) return fail(GCRE_ERR_ARG, "null argument");
  *out = nullptr;
  CKS(use_device(ex));
  gcre_pathset* ps = new (std::nothrow) gcre_pathset();
  if (!ps) return fail(GCRE_ERR_NOMEM, "host allocation failed");
  ps->ex = ex;
  ps->size = size;
  ps->uid = ++g_pathset_uid;
  ps->known_zero = true;
  const size_t bytes = (size_t)size * row_words(ex) * 8;
  if (bytes) {
    cudaError_t e = dev_alloc(ex, (void**)&ps->d_rows, bytes);
    if (e != cudaSuccess) {
      delete ps;
      return fail(GCRE_ERR_NOMEM, "device allocation of %zu bytes for a path set failed: %s", bytes, cudaGetErrorString(e));
    }
    ps->zero_pending = true;
  }
  {
    std::lock_guard<std::mutex> lock(ex->child_mu);
    ex->pathsets.insert(ps);
  }
  *out = ps;
  return GCRE_OK;
}

extern "C" int gcre_pathset_destroy(gcre_pathset* ps) {
  if (!ps) return GCRE_OK;
  if (ps->ex) {  // (an orphan's device memory went back to the cache when its exec was destroyed)
    cudaSetDevice(ps->ex->device);
    {
      std::lock_guard<std::mutex> lock(ps->ex->child_mu);
      ps->ex->pathsets.erase(ps);
    }
    dev_free(ps->ex, ps->d_rows);  // back to the block cache, no driver call
    drop_view(ps);
    drop_prov(ps);
  }
  delete ps;
  return GCRE_OK;
}

#define LIVE(obj)                                                                                  \
  do {                                                                                             \
    if (!(obj)->ex) return fail(GCRE_ERR_ARG, "the JoinExec this object belongs to was destroyed"); \
  } while (0)

static int mask_tail(const gcre_exec* ex, gcre_pathset* ps, uint32_t row0, uint32_t rows) {
  if (!rows || ((ex->n & 63) == 0 && ex->Wp == ex->W64)) return GCRE_OK;
  const long long halves = (long long)rows * ex->M;
  mask_tail_kernel<<<grid_for(halves, 256), 256, 0, ex->stream>>>(ps->d_rows + (size_t)row0 * row_words(ex), halves, ex->Wp, ex->W64, ex->n);
  CK(cudaGetLastError());
  LAUNCHED();
  return GCRE_OK;
}

extern "C" int gcre_pathset_size(const gcre_pathset* ps, uint32_t* size) {
  if (!ps || !size) return fail(GCRE_ERR_ARG, "null argument");
  *size = ps->size;
  return GCRE_OK;
}

static int pathset_max_half_pop(gcre_pathset* ps, long long* out) {
  gcre_exec* ex = const_cast<gcre_exec*>(ps->ex);
  if (ps->max_half_pop < 0) {
    CK(cudaMemsetAsync(ex->d_scalars + 1, 0, sizeof(unsigned), ex->stream));
    if (ps->size) {
      const long long warps = (long long)ps->size * ex->M;
      (ex->M == 1 ? row_maxpop_kernel<1> : row_maxpop_kernel<2>)<<<grid_for(warps * 32, 256), 256, 0, ex->stream>>>(ps->d_rows, ps->size, ex->Wp,
                                                                                                                  ex->d_scalars + 1);
      CK(cudaGetLastError());
      LAUNCHED();
    }
    CK(cudaMemcpyAsync(ex->h_scalars + 1, ex->d_scalars + 1, sizeof(unsigned), cudaMemcpyDeviceToHost, ex->stream));
    CK(cudaStreamSynchronize(ex->stream));
    ps->max_half_pop = ex->h_scalars[1];
  }
  *out = ps->max_half_pop;
  return GCRE_OK;
}

extern "C" int gcre_pathset_load_i32(gcre_pathset* ps, const int32_t* data, uint32_t rows, int cols) {
  if (!ps || (!data && rows > 0)) return fail(GCRE_ERR_ARG, "null argument");
  LIVE(ps);
  gcre_exec* ex = const_cast<gcre_exec*>(ps->ex);
  CKS(use_device(ex));
  // src/gcre_paths.h:60: check_true(size == data.size())
  if (rows != ps->size) return fail(GCRE_ERR_ASSERT, "assertion");
  // src/gcre_paths.h:63: check_index(data[r].size(), width_ul * 64); a column count equal to n is always accepted (the
  // reference throws when n is a multiple of its SIMD width: SURVEY App. D1)
  // Columns beyond the n = num_cases + num_ctrls patients are rejected (the reference would accept up to its SIMD-padded
  // width and count such bits as controls of the true score only - there is no patient they could belong to).
  if (rows > 0 && (cols < 0 || cols > ex->n)) return fail(GCRE_ERR_RANGE, "assertion");
  if (rows == 0) return GCRE_OK;
  rows_written(ps);
  ps->zero_pending = false;
  CK(cudaMemsetAsync(ps->d_rows, 0, (size_t)ps->size * row_words(ex) * 8, ex->stream));
  // Where to pack.  The int matrix is 32x its bits: above a few tens of MB, and with enough host threads to stream it faster
  // than the PCIe link would carry it (measured on the bench box, 600 MB matrix: 16 threads 112 GB/s, 8 threads 86 GB/s,
  // link 52 GB/s), pack on the host and upload the bits; otherwise upload the ints and pack on the device.
  // GCRE_HOST_PACK_THREADS sets the thread count (0 = never; default min(16, hardware threads)); one process per GPU on a
  // shared host should divide the cores between the ranks (bench.py does).  GCRE_TEST_HOST_PACK=1 (test hook) forces the
  // host path on small inputs.
  int pack_threads = (int)std::min(16u, std::max(1u, std::thread::hardware_concurrency()));
  if (const char* e = std::getenv("GCRE_HOST_PACK_THREADS")) pack_threads = std::atoi(e);
  const char* force_host = std::getenv("GCRE_TEST_HOST_PACK");
  bool host_pack = (force_host && *force_host == '1' && pack_threads >= 1) ||
                         (pack_threads >= 8 && (size_t)rows * cols * 4 >= ((size_t)32 << 20));
  const size_t w_in = ((size_t)cols + 63) / 64;  // words per row that carry data (<= W64)
  PinnedBlock stage{nullptr, 0};
  if (host_pack && pinned_big_acquire(std::max<size_t>((size_t)rows * w_in * 8, 8), &stage) != cudaSuccess) {
    cudaGetLastError();  // no page-locked memory to be had: pack on the device instead
    host_pack = false;
  }
  if (host_pack) {
    gcre_host::pack_i32_rows(data, rows, cols, static_cast<uint64_t*>(stage.p), w_in, pack_threads);
    int rc = GCRE_OK;
    if (w_in) {
      rc = upload_staged(ex, stage.p, w_in * 8, rows, [&](const void* d_piece, size_t r0, size_t nr) {
        place_rows_kernel<<<grid_for((long long)nr * (long long)w_in, 256), 256, 0, ex->stream>>>((const uint64_t*)d_piece, (uint32_t)nr, (int)w_in, (int)w_in,
                                                                                               ps->d_rows + r0 * row_words(ex), (int)row_words(ex));
        CK(cudaGetLastError());
        LAUNCHED();
        return (int)GCRE_OK;
      });
    }
    pinned_big_release(stage);  // upload_staged has waited for its copies
    CKS(rc);
  } else {
    CKS(upload_staged(ex, data, (size_t)cols * 4, rows, [&](const void* d_piece, size_t r0, size_t nr) {
      const long long warps = (long long)nr * ex->W64;
      pack_rows_i32_kernel<<<grid_for(warps * 32, 256), 256, 0, ex->stream>>>((const int32_t*)d_piece, (uint32_t)nr, cols,
                                                                             ps->d_rows + r0 * row_words(ex), (int)row_words(ex), ex->W64);
      CK(cudaGetLastError());
      LAUNCHED();
      return (int)GCRE_OK;
    }));
  }
  ps->max_half_pop = -1;
  drop_view(ps);
  return GCRE_OK;
}

// Device-side inputs (multi-GPU fan-out: one rank uploads, NCCL broadcasts over NVLink, every rank adopts the buffer).
// Ordered on the exec's stream; the caller's buffer must stay valid until that stream has passed the copy (any later join
// of this exec synchronises it).
extern "C" int gcre_pathset_load_bits_device(gcre_pathset* ps, const uint64_t* d_bits, uint32_t rows, int words_per_row) {
  if (!ps || (!d_bits && rows > 0)) return fail(GCRE_ERR_ARG, "null argument");
  LIVE(ps);
  gcre_exec* ex = const_cast<gcre_exec*>(ps->ex);
  CKS(use_device(ex));
  if (rows != ps->size) return fail(GCRE_ERR_ASSERT, "assertion");
  if (rows > 0 && (words_per_row < 0 || words_per_row > ex->W64)) return fail(GCRE_ERR_RANGE, "assertion");
  if (rows == 0) return GCRE_OK;
  rows_written(ps);
  ps->zero_pending = false;
  CK(cudaMemsetAsync(ps->d_rows, 0, (size_t)ps->size * row_words(ex) * 8, ex->stream));
  if (words_per_row > 0) {
    place_rows_kernel<<<grid_for((long long)rows * words_per_row, 256), 256, 0, ex->stream>>>(d_bits, rows, words_per_row, words_per_row, ps->d_rows,
                                                                                             (int)row_words(ex));
    CK(cudaGetLastError());
    LAUNCHED();
    if (words_per_row == ex->W64) CKS(mask_tail(ex, ps, 0, rows));
  }
  ps->max_half_pop = -1;
  drop_view(ps);
  return GCRE_OK;
}

extern "C" int gcre_exec_set_value_table_device(gcre_exec* ex, const double* d_table, int rows, int cols) {
  if (!ex || (!d_table && rows > 0 && cols > 0)) return fail(GCRE_ERR_ARG, "null argument");
  if (rows < 0 || cols < 0) return fail(GCRE_ERR_ARG, "negative table size");
  CKS(use_device(ex));
  dev_free(ex, ex->d_vt);
  ex->d_vt = nullptr;
  ex->vt_rows = rows;
  ex->vt_cols = cols;
  const size_t bytes = std::max<size_t>((size_t)rows * cols, 1) * 8;
  CK(dev_alloc(ex, (void**)&ex->d_vt, bytes));
  if ((size_t)rows * cols != 0) CK(cudaMemcpyAsync(ex->d_vt, d_table, (size_t)rows * cols * 8, cudaMemcpyDeviceToDevice, ex->stream));
  ex->diag_cap = -1;
  return GCRE_OK;
}

extern "C" int gcre_host_pack_i32(const int32_t* data, uint32_t rows, int cols, uint64_t* bits, int threads) {
  if ((!data || !bits) && rows > 0 && cols > 0) return fail(GCRE_ERR_ARG, "null argument");
  if (cols < 0) return fail(GCRE_ERR_ARG, "negative size");
  if (threads <= 0) threads = (int)std::min(16u, std::max(1u, std::thread::hardware_concurrency()));
  if (rows && cols) gcre_host::pack_i32_rows(data, rows, cols, bits, ((size_t)cols + 63) / 64, threads);
  return GCRE_OK;
}

extern "C" int gcre_pathset_load_bits(gcre_pathset* ps, const uint64_t* bits, uint32_t rows, int words_per_row) {
  if (!ps || (!bits && rows > 0)) return fail(GCRE_ERR_ARG, "null argument");
  LIVE(ps);
  gcre_exec* ex = const_cast<gcre_exec*>(ps->ex);
  CKS(use_device(ex));
  if (rows != ps->size) return fail(GCRE_ERR_ASSERT, "assertion");
  if (rows > 0 && (words_per_row < 0 || words_per_row > ex->W64)) return fail(GCRE_ERR_RANGE, "assertion");
  if (rows == 0) return GCRE_OK;
  rows_written(ps);
  ps->zero_pending = false;
  CK(cudaMemsetAsync(ps->d_rows, 0, (size_t)ps->size * row_words(ex) * 8, ex->stream));
  const size_t bytes = (size_t)rows * words_per_row * 8;
  if (bytes) {
    CKS(ex->scratch.ensure(bytes));
    CK(cudaMemcpyAsync(ex->scratch.p, bits, bytes, cudaMemcpyHostToDevice, ex->stream));
    place_rows_kernel<<<grid_for((long long)rows * words_per_row, 256), 256, 0, ex->stream>>>((const uint64_t*)ex->scratch.p, rows, words_per_row,
                                                                                             words_per_row, ps->d_rows, (int)row_words(ex));
    CK(cudaGetLastError());
      LAUNCHED();
    if (words_per_row == ex->W64) CKS(mask_tail(ex, ps, 0, rows));
    CK(cudaStreamSynchronize(ex->stream));
  }
  ps->max_half_pop = -1;
  drop_view(ps);
  return GCRE_OK;
}

extern "C" int gcre_pathset_select(const gcre_pathset* ps, const int32_t* indices, uint32_t n, gcre_pathset** out) {
  if (!ps || !out || (!indices && n > 0)) return fail(GCRE_ERR_ARG, "null argument");
  LIVE(ps);
  *out = nullptr;
  gcre_exec* ex = const_cast<gcre_exec*>(ps->ex);
  CKS(use_device(ex));
  // src/gcre_paths.h:85: check_index(indices[k], size)
  for (uint32_t k = 0; k < n; k++)
    if (indices[k] < 0 || (uint32_t)indices[k] >= ps->size) return fail(GCRE_ERR_RANGE, "assertion");
  CKS(materialize_zero(const_cast<gcre_pathset*>(ps)));
  gcre_pathset* res = nullptr;
  CKS(gcre_pathset_create(ex, n, &res));
  if (n) {
    res->zero_pending = false;  // every row is written by the gather below
    res->known_zero = false;
    int rc = [&]() -> int {
      CKS(ex->scratch.ensure((size_t)n * 4));
      CK(cudaMemcpyAsync(ex->scratch.p, indices, (size_t)n * 4, cudaMemcpyHostToDevice, ex->stream));
      const int row_vec = (int)(row_words(ex) / 2);
      select_rows_kernel<<<grid_for((long long)n * row_vec, 256), 256, 0, ex->stream>>>((const ulonglong2*)ps->d_rows, (const int32_t*)ex->scratch.p, n,
                                                                                       row_vec, (ulonglong2*)res->d_rows);
      CK(cudaGetLastError());
      LAUNCHED();
      // the selection remembers its rows' origin (a KEEP join with it as partner scores its rows through the base set's, and
      // records which base row each result row adds)
      if (ps->size <= 0x7fffffffu && provenance_useful(ex)) {
        CK(dev_alloc(ex, (void**)&res->prov.sel, (size_t)n * 4));
        selection_entries_kernel<<<grid_for((long long)n, 256), 256, 0, ex->stream>>>((const int32_t*)ex->scratch.p, n, res->prov.sel);
        CK(cudaGetLastError());
        LAUNCHED();
        res->prov.base = ps;
        res->prov.base_uid = ps->uid;
        res->prov.base_ver = ps->ver;
      }
      // no host wait: the copy above has read `indices` when it returns unless they are page-locked - then wait for it
      cudaPointerAttributes attr;
      if (cudaPointerGetAttributes(&attr, indices) != cudaSuccess || attr.type != cudaMemoryTypeUnregistered) {
        cudaGetLastError();
        CK(cudaStreamSynchronize(ex->stream));
      }
      return GCRE_OK;
    }();
    if (rc != GCRE_OK) {
      gcre_pathset_destroy(res);
      return rc;
    }
  }
  // an upper bound is all a join needs: the source's maximum, computed once and reused by every selection from it
  long long src_max = 0;
  if (n && pathset_max_half_pop(const_cast<gcre_pathset*>(ps), &src_max) != GCRE_OK) {
    gcre_pathset_destroy(res);
    return GCRE_ERR_CUDA;
  }
  res->max_half_pop = n ? src_max : 0;
  *out = res;
  return GCRE_OK;
}

extern "C" int gcre_pathset_set_row(gcre_pathset* ps, uint32_t idx, const uint64_t* words) {
  if (!ps || !words) return fail(GCRE_ERR_ARG, "null argument");
  LIVE(ps);
  gcre_exec* ex = const_cast<gcre_exec*>(ps->ex);
  CKS(use_device(ex));
  if (idx >= ps->size) return fail(GCRE_ERR_RANGE, "assertion");  // src/gcre_paths.h:50
  CKS(materialize_zero(ps));
  rows_written(ps);
  for (int h = 0; h < ex->M; h++)
    CK(cudaMemcpyAsync(ps->d_rows + (size_t)idx * row_words(ex) + (size_t)h * ex->Wp, words + (size_t)h * ex->W64, (size_t)ex->W64 * 8,
                       cudaMemcpyHostToDevice, ex->stream));
  CKS(mask_tail(ex, ps, idx, 1));
  CK(cudaStreamSynchronize(ex->stream));
  ps->max_half_pop = -1;
  drop_view(ps);
  return GCRE_OK;
}

extern "C" int gcre_pathset_get_row(const gcre_pathset* ps, uint32_t idx, uint64_t* words) {
  if (!ps || !words) return fail(GCRE_ERR_ARG, "null argument");
  LIVE(ps);
  const gcre_exec* ex = ps->ex;
  CKS(use_device(ex));
  if (idx >= ps->size) return fail(GCRE_ERR_RANGE, "assertion");  // src/gcre_paths.h:45
  CKS(materialize_zero(const_cast<gcre_pathset*>(ps)));
  for (int h = 0; h < ex->M; h++)
    CK(cudaMemcpyAsync(words + (size_t)h * ex->W64, ps->d_rows + (size_t)idx * row_words(ex) + (size_t)h * ex->Wp, (size_t)ex->W64 * 8,
                       cudaMemcpyDeviceToHost, ex->stream));
  CK(cudaStreamSynchronize(ex->stream));
  return GCRE_OK;
}

extern "C" int gcre_pathset_download(const gcre_pathset* ps, uint64_t* out) {
  if (!ps || (!out && ps->size)) return fail(GCRE_ERR_ARG, "null argument");
  LIVE(ps);
  gcre_exec* ex = const_cast<gcre_exec*>(ps->ex);
  CKS(use_device(ex));
  if (!ps->size) return GCRE_OK;
  CKS(materialize_zero(const_cast<gcre_pathset*>(ps)));
  const size_t words = (size_t)ps->size * ex->W64 * ex->M;
  CKS(ex->scratch.ensure(words * 8));
  if (ex->M == 1)
    unpad_rows_kernel<1><<<grid_for((long long)words, 256), 256, 0, ex->stream>>>(ps->d_rows, ps->size, ex->Wp, ex->W64, (uint64_t*)ex->scratch.p);
  else
    unpad_rows_kernel<2><<<grid_for((long long)words, 256), 256, 0, ex->stream>>>(ps->d_rows, ps->size, ex->Wp, ex->W64, (uint64_t*)ex->scratch.p);
  CK(cudaGetLastError());
      LAUNCHED();
  CK(cudaMemcpyAsync(out, ex->scratch.p, words * 8, cudaMemcpyDeviceToHost, ex->stream));
  CK(cudaStreamSynchronize(ex->stream));
  return GCRE_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// read-backs of a path set's sparse view (tests and diagnostics only; nothing calls them on the join path)
// ------------------------------------------------------------------------------------------------------------------
extern "C" int gcre_pathset_debug_view_info(const gcre_pathset* ps, int64_t* out) {
  if (!ps || !out) return fail(GCRE_ERR_ARG, "null argument");
  LIVE(ps);
  const gcre_exec* ex = ps->ex;
  CKS(use_device(ex));
  const SparseView& v = ps->view;
  uint64_t entries = 0;
  if (v.valid) {
    CK(cudaMemcpyAsync(&entries, v.off + (size_t)ps->size * ex->M, 8, cudaMemcpyDeviceToHost, ex->stream));
    CK(cudaStreamSynchronize(ex->stream));
  }
  const bool table = v.pcnt != nullptr;
  const int64_t info[8] = {v.valid, (int64_t)entries, v.stats_valid, table, table ? v.pcnt_layout : 0, table && v.pcnt_gen == ex->mask_gen,
                           table ? (int64_t)v.emit_lo : 0, table ? (int64_t)v.emit_hi : 0};
  memcpy(out, info, sizeof info);
  return GCRE_OK;
}

extern "C" int gcre_pathset_debug_counts(const gcre_pathset* ps, uint16_t* counts, uint32_t* len, uint32_t* ncase) {
  if (!ps) return fail(GCRE_ERR_ARG, "null argument");
  LIVE(ps);
  const gcre_exec* ex = ps->ex;
  CKS(use_device(ex));
  const SparseView& v = ps->view;
  if (!v.pcnt) return fail(GCRE_ERR_ASSERT, "the path set holds no count table");
  const size_t lo = (size_t)v.emit_lo, items = ((size_t)v.emit_hi - lo) * ex->M;
  if (items && !counts) return fail(GCRE_ERR_ARG, "null argument");
  const size_t entry_words = (v.pcnt_layout == 0 ? (size_t)(ex->Iw / 32) * 2048 : sparse_sc_table_bytes(ex->Ip)) / 4;
  std::vector<uint32_t> raw(items * entry_words);
  if (items) CK(cudaMemcpyAsync(raw.data(), v.pcnt + lo * ex->M * entry_words, raw.size() * 4, cudaMemcpyDeviceToHost, ex->stream));
  if (items && len && v.len) CK(cudaMemcpyAsync(len, v.len + lo * ex->M, items * 4, cudaMemcpyDeviceToHost, ex->stream));
  if (items && ncase && v.ncase) CK(cudaMemcpyAsync(ncase, v.ncase + lo * ex->M, items * 4, cudaMemcpyDeviceToHost, ex->stream));
  CK(cudaStreamSynchronize(ex->stream));
  for (size_t i = 0; i < items; i++) {
    const uint32_t* entry = raw.data() + i * entry_words;
    uint16_t* dst = counts + i * ex->iters;
    for (int r = 0; r < ex->iters; r++)
      dst[r] = (uint16_t)(v.pcnt_layout == 0 ? c16_table_count(entry, r) : sc_table_count(entry, v.pcnt_layout, r));
  }
  return GCRE_OK;
}

extern "C" int gcre_pathset_debug_lists(const gcre_pathset* ps, uint64_t* off, uint32_t* len, uint32_t* ncase, uint32_t* car) {
  if (!ps || !off || !len || !ncase) return fail(GCRE_ERR_ARG, "null argument");
  LIVE(ps);
  const gcre_exec* ex = ps->ex;
  CKS(use_device(ex));
  const SparseView& v = ps->view;
  if (!v.valid) return fail(GCRE_ERR_ASSERT, "the path set's carrier lists are not built");
  const size_t items = (size_t)ps->size * ex->M;
  CK(cudaMemcpyAsync(off, v.off, (items + 1) * 8, cudaMemcpyDeviceToHost, ex->stream));
  if (items) {
    CK(cudaMemcpyAsync(len, v.len, items * 4, cudaMemcpyDeviceToHost, ex->stream));
    CK(cudaMemcpyAsync(ncase, v.ncase, items * 4, cudaMemcpyDeviceToHost, ex->stream));
  }
  CK(cudaStreamSynchronize(ex->stream));
  const size_t total = (size_t)off[items];
  if (total && !car) return fail(GCRE_ERR_ARG, "null argument");
  if (total && ex->wide) {
    CK(cudaMemcpyAsync(car, v.car, total * 4, cudaMemcpyDeviceToHost, ex->stream));
    CK(cudaStreamSynchronize(ex->stream));
  } else if (total) {
    std::vector<uint16_t> narrow(total);
    CK(cudaMemcpyAsync(narrow.data(), v.car, total * 2, cudaMemcpyDeviceToHost, ex->stream));
    CK(cudaStreamSynchronize(ex->stream));
    for (size_t k = 0; k < total; k++) car[k] = narrow[k];
  }
  return GCRE_OK;
}

extern "C" int gcre_pathset_debug_bounds(const gcre_pathset* ps, int64_t* out) {
  if (!ps || !out) return fail(GCRE_ERR_ARG, "null argument");
  LIVE(ps);
  out[0] = ps->max_half_pop;  // as recorded, not recomputed
  out[1] = ps->view.valid ? (int64_t)ps->view.total : 0;
  return GCRE_OK;
}

extern "C" int gcre_exec_debug_diag_cap(const gcre_exec* ex, int64_t* out) {
  if (!ex || !out) return fail(GCRE_ERR_ARG, "null argument");
  *out = ex->diag_cap;
  return GCRE_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// value-table re-layout
// ------------------------------------------------------------------------------------------------------------------
static int ensure_diag(gcre_exec* ex, long long t_needed) {
  if (t_needed <= ex->diag_cap) return GCRE_OK;
  if (!ex->d_vt) {
    // no table set: the reference's value_table would be empty and indexing it is undefined; treat as all -1.0
    CK(dev_alloc(ex, (void**)&ex->d_vt, 8));
    ex->vt_rows = ex->vt_cols = 0;
  }
  long long cap = std::min<long long>(ex->n, std::max<long long>(t_needed + t_needed / 4 + 64, 1024));
  cap = std::max(cap, t_needed);
  CK(cudaStreamSynchronize(ex->stream));
  dev_free(ex, ex->d_diagD);
  dev_free(ex, ex->d_diagF);
  dev_free(ex, ex->d_diagDM);
  dev_free(ex, ex->d_diagFM);
  ex->d_diagD = nullptr;
  ex->d_diagF = nullptr;
  ex->d_diagDM = nullptr;
  ex->d_diagFM = nullptr;
  ex->diag_cap = -1;
  const size_t entries = (size_t)(cap + 1) * (size_t)(cap + 2) / 2;
  {
    // (cap+1)(cap+2)/2 entries of 12 (method 1) or 20 (method 2) bytes: 26-43 GB at 65,535 carriers per half-row
    cudaError_t e = dev_alloc(ex, (void**)&ex->d_diagD, entries * 8);
    if (e == cudaSuccess) e = (ex->M == 1) ? dev_alloc(ex, (void**)&ex->d_diagF, entries * 4) : dev_alloc(ex, (void**)&ex->d_diagDM, entries * 8);
    if (e == cudaSuccess && ex->M != 1) e = dev_alloc(ex, (void**)&ex->d_diagFM, entries * 4);
    if (e != cudaSuccess) {
      cudaGetLastError();
      dev_free(ex, ex->d_diagD);
      ex->d_diagD = nullptr;
      return fail(GCRE_ERR_NOMEM, "anti-diagonal value tables for joined rows of up to %lld carriers need %zu bytes of device memory (%s); "
                  "the limit is set by the densest operand rows", t_needed, entries * (ex->M == 1 ? 12 : 20), cudaGetErrorString(e));
    }
  }
  build_diag_kernel<<<(unsigned)(cap + 1), 128, 0, ex->stream>>>(ex->d_vt, ex->vt_rows, ex->vt_cols, (unsigned)cap, ex->d_diagD, ex->d_diagF, ex->d_diagDM,
                                                                 ex->d_diagFM);
  CK(cudaGetLastError());
      LAUNCHED();
  ex->diag_cap = cap;
  return GCRE_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// top-K bookkeeping (host): K largest scores, ties broken by smaller (src, trg)
// ------------------------------------------------------------------------------------------------------------------
static inline bool better(const gcre_score& a, const gcre_score& b) {
  if (a.score != b.score) return a.score > b.score;
  if (a.src != b.src) return (uint32_t)a.src < (uint32_t)b.src;
  return (uint32_t)a.trg < (uint32_t)b.trg;
}

static void trim_topk(std::vector<gcre_score>& held, int top_k) {
  if ((int)held.size() > top_k) {
    std::nth_element(held.begin(), held.begin() + top_k, held.end(), better);
    held.resize(top_k);
  }
}

// src/join_base.cpp:138-154: ascending order, leading -inf sentinel when fewer than top_k real entries
static int emit_topk(std::vector<gcre_score>& held, int top_k, gcre_score* out_scores, int* n_scores) {
  trim_topk(held, top_k);
  std::sort(held.begin(), held.end(), better);
  int n = 0;
  if ((int)held.size() < top_k) {
    gcre_score s;
    s.score = -std::numeric_limits<double>::infinity();
    s.src = -1;
    s.trg = -1;
    s.cases = 0;
    s.ctrls = 0;
    out_scores[n++] = s;
  }
  for (int k = (int)held.size() - 1; k >= 0; k--) out_scores[n++] = held[k];
  *n_scores = n;
  return GCRE_OK;
}

extern "C" int gcre_merge_topk(const gcre_score* lists, const int* list_sizes, int n_lists, int top_k, gcre_score* out_scores, int* n_scores) {
  if (!lists || !list_sizes || !out_scores || !n_scores) return fail(GCRE_ERR_ARG, "null argument");
  if (top_k < 1) top_k = 1;
  std::vector<gcre_score> held;
  size_t off = 0;
  for (int l = 0; l < n_lists; l++) {
    for (int k = 0; k < list_sizes[l]; k++)
      if (lists[off + k].src >= 0) held.push_back(lists[off + k]);
    off += list_sizes[l];
  }
  return emit_topk(held, top_k, out_scores, n_scores);
}

// ------------------------------------------------------------------------------------------------------------------
// carrier-list views for the sparse kernels
// ------------------------------------------------------------------------------------------------------------------
constexpr unsigned long long kViewBoundEntries = 16ull << 20;  // carrier lists up to this many entries (32 / 64 MB) are allocated by their bound
static int ensure_view(gcre_exec* ex, gcre_pathset* ps, bool view_exact) {
  if (ps->view.valid) return GCRE_OK;
  CKS(materialize_zero(ps));
  {  // (re)build lists and stats; counts emitted with the rows stay - the rows have not changed
    uint32_t* pcnt = ps->view.pcnt;
    unsigned long long* fp = ps->view.fp;
    const unsigned long long gen = ps->view.pcnt_gen, elo = ps->view.emit_lo, ehi = ps->view.emit_hi;
    const int layout = ps->view.pcnt_layout;
    ps->view.pcnt = nullptr;
    ps->view.fp = nullptr;
    drop_view(ps);
    ps->view.pcnt = pcnt;
    ps->view.fp = fp;
    ps->view.pcnt_gen = gen;
    ps->view.pcnt_layout = layout;
    ps->view.emit_lo = elo;
    ps->view.emit_hi = ehi;
  }
  const long long items = (long long)ps->size * ex->M;
  CK(dev_alloc(ex, (void**)&ps->view.off, (size_t)(items + 1) * 8));
  CK(dev_alloc(ex, (void**)&ps->view.len, std::max<size_t>(items, 1) * 4));
  CK(dev_alloc(ex, (void**)&ps->view.ncase, std::max<size_t>(items, 1) * 4));
  CK(cudaMemsetAsync(ps->view.off, 0, (size_t)(items + 1) * 8, ex->stream));
  unsigned long long total = 0;
  if (items > 0) {
    // true counts + padded counts -> exclusive offsets (cub scan over items + 1 entries, the last input is 0).  Offsets are
    // 64-bit: the carriers of a large kept set do not fit 32 bits (a 32-bit scan wrapped silently).
    CKS(ex->scratch.ensure((size_t)(items + 1) * 8));
    unsigned long long* padded = (unsigned long long*)ex->scratch.p;
    CK(cudaMemsetAsync(padded, 0, (size_t)(items + 1) * 8, ex->stream));
    half_popcount_kernel<<<grid_for(items * 32, 256), 256, 0, ex->stream>>>(ps->d_rows, items, ex->Wp, ps->view.len, padded);
    CK(cudaGetLastError());
    LAUNCHED();
    size_t tmp_bytes = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, padded, ps->view.off, (long long)(items + 1), ex->stream));
    CKS(ex->scan_tmp.ensure(tmp_bytes));
    CK(cub::DeviceScan::ExclusiveSum(ex->scan_tmp.p, tmp_bytes, padded, ps->view.off, (long long)(items + 1), ex->stream));
    LAUNCHED();
    // How many entries to allocate.  join_impl has the set's largest half-row by now (an upper bound is enough): when rows x
    // that bound is small the lists are allocated by the bound and the host does not wait for the scan's total
    // (one device round trip per view, ~10 views per level schedule).
    const unsigned long long bound = ps->max_half_pop >= 0 ? (unsigned long long)items * (((unsigned long long)ps->max_half_pop + 7ull) & ~7ull) : ~0ull;
    if (bound <= kViewBoundEntries && !view_exact) {
      total = bound;
    } else {
      CK(cudaMemcpyAsync(&total, ps->view.off + items, 8, cudaMemcpyDeviceToHost, ex->stream));
      CK(cudaStreamSynchronize(ex->stream));
    }
  }
  ps->view.total = (size_t)total;
  {
    const size_t car_bytes = std::max<size_t>((size_t)total, 8) * (ex->wide ? 4 : 2);
    cudaError_t e = dev_alloc(ex, (void**)&ps->view.car, car_bytes);
    if (e != cudaSuccess) {
      cudaGetLastError();
      drop_view(ps);
      return fail(GCRE_ERR_NOMEM, "carrier lists of a %u-row path set need %zu bytes of device memory: %s", ps->size, car_bytes, cudaGetErrorString(e));
    }
  }
  if (items > 0) {
    if (ex->wide)
      build_lists_kernel<uint32_t><<<grid_for(items * 32, 256), 256, 0, ex->stream>>>(ps->d_rows, items, ex->Wp, ex->n_cases, ex->n, ps->view.off,
                                                                                     (uint32_t*)ps->view.car, ps->view.ncase);
    else
      build_lists_kernel<uint16_t><<<grid_for(items * 32, 256), 256, 0, ex->stream>>>(ps->d_rows, items, ex->Wp, ex->n_cases, ex->n, ps->view.off,
                                                                                     (uint16_t*)ps->view.car, ps->view.ncase);
    CK(cudaGetLastError());
    LAUNCHED();
  }
  ps->view.valid = ps->view.stats_valid = true;
  return GCRE_OK;
}

// per-permutation counts of every (row, half) of a path set under the exec's current masks (join_sparse.cuh, PC kernels)
// (a table a KEEP join emitted serves when it is current and holds every row: a row-sharded join emits its rows only)
static int ensure_precount(gcre_exec* ex, gcre_pathset* ps) {
  if (ps->view.pcnt && ps->view.pcnt_gen == ex->mask_gen && ps->view.pcnt_layout == 0 && ps->view.emit_lo == 0 && ps->view.emit_hi >= ps->size)
    return GCRE_OK;
  dev_free(ex, ps->view.pcnt);
  ps->view.pcnt = nullptr;
  ps->view.pcnt_layout = 0;
  dev_free(ex, ps->view.fp);  // emitted over the rows the table covered; the new table covers every row
  ps->view.fp = nullptr;
  const long long items = (long long)ps->size * ex->M;
  const int nb = ex->Iw / 32;
  CK(dev_alloc(ex, (void**)&ps->view.pcnt, std::max<size_t>((size_t)items * nb, 1) * 2048));
  if (items > 0) {
    const unsigned grid = grid_for(items * nb * 32, 128);
    if (ex->wide)
      build_precount_kernel<uint32_t><<<grid, 128, 0, ex->stream>>>(ps->view.off, (const uint32_t*)ps->view.car, items, nb, ex->d_pt, ex->Iw, ps->view.pcnt);
    else
      build_precount_kernel<uint16_t><<<grid, 128, 0, ex->stream>>>(ps->view.off, (const uint16_t*)ps->view.car, items, nb, ex->d_pt, ex->Iw, ps->view.pcnt);
    CK(cudaGetLastError());
    LAUNCHED();
  }
  ps->view.pcnt_gen = ex->mask_gen;
  ps->view.emit_lo = 0;
  ps->view.emit_hi = ps->size;
  return GCRE_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// provenance (tail form of the pre-counted sparse kernel, join_sparse.cuh)
// ------------------------------------------------------------------------------------------------------------------
// the base set `p` names is alive and unchanged since the entries were made
static bool base_current(const gcre_exec* ex, const Provenance& p) {
  if (!p.base) return false;
  std::lock_guard<std::mutex> lock(ex->child_mu);
  return ex->pathsets.count(const_cast<gcre_pathset*>(p.base)) && p.base->uid == p.base_uid && p.base->ver == p.base_ver;
}

static bool same_base(const Provenance& a, const Provenance& b) {
  return a.base == b.base && a.base_uid == b.base_uid && a.base_ver == b.base_ver;
}

// A KEEP join has written result rows [pair_lo, pair_hi): record their tails (and heads) when the partner set is a selection
// of a live base set.  Called after rows_written(paths_res).
static int record_provenance(gcre_exec* ex, const gcre_uidset* us, const gcre_pathset* paths0, const gcre_pathset* paths1, gcre_pathset* paths_res,
                             uint32_t ub, uint32_t ue, unsigned long long pair_lo, unsigned long long pair_hi, unsigned long long unit_lo,
                             unsigned long long unit_hi) {
  const Provenance& sel = paths1->prov;
  if (!provenance_useful(ex) || !us->res_is_prefix || pair_hi <= pair_lo || paths_res == paths0 || paths_res == paths1 || !sel.sel || !base_current(ex, sel)) return GCRE_OK;
  const Provenance& up = paths0->prov;
  const bool single = paths0->known_zero;
  const bool heads = !single && up.tail && up.single && same_base(up, sel) && ub >= up.lo && ue <= up.hi;
  Provenance& p = paths_res->prov;
  CK(dev_alloc(ex, (void**)&p.tail, (size_t)paths_res->size * 4));
  if (heads) CK(dev_alloc(ex, (void**)&p.head, (size_t)paths_res->size * 4));
  (ex->M == 1 ? record_rows_kernel<1> : record_rows_kernel<2>)<<<grid_for((long long)(unit_hi - unit_lo), 256), 256, 0, ex->stream>>>(
      unit_lo, unit_hi, (const uint32_t*)us->unit_idx.p, (const unsigned long long*)us->units.p, sparse::PB, (const int32_t*)us->count.p,
      (const uint32_t*)us->loc.p, (const unsigned long long*)us->res.p, (const int32_t*)us->signs.p, us->path_length, sel.sel, up.tail, p.tail, p.head);
  CK(cudaGetLastError());
  LAUNCHED();
  p.base = sel.base;
  p.base_uid = sel.base_uid;
  p.base_ver = sel.base_ver;
  p.lo = pair_lo;
  p.hi = pair_hi;
  p.single = single;
  return GCRE_OK;
}

// The base set whose gene rows a score-only join over upstream rows [ub, ue) may be scored against (tail form), or null:
// both operands carry entries over the same live base set, and every pair's partner head, oriented by the pair, is its
// upstream row's tail (one pass over the work units [unit_lo, unit_hi) of those rows, one flag read back).
static int tail_form_base(gcre_exec* ex, const gcre_uidset* us, const gcre_pathset* paths0, const gcre_pathset* paths1, uint32_t ub, uint32_t ue,
                          unsigned long long unit_lo, unsigned long long unit_hi, const gcre_pathset** out) {
  *out = nullptr;
  const Provenance &up = paths0->prov, &pt = paths1->prov;
  if (!up.tail || !pt.tail || !pt.head || !same_base(up, pt) || !base_current(ex, up) || ub < up.lo || ue > up.hi || ue <= ub) return GCRE_OK;
  unsigned* d_bad = ex->d_scalars + 12;
  CK(cudaMemsetAsync(d_bad, 0, sizeof(unsigned), ex->stream));
  (ex->M == 1 ? tail_eligible_kernel<1> : tail_eligible_kernel<2>)<<<grid_for((long long)(unit_hi - unit_lo), 256), 256, 0, ex->stream>>>(
      unit_lo, unit_hi, (const uint32_t*)us->unit_idx.p, (const unsigned long long*)us->units.p, sparse::PB, (const int32_t*)us->count.p,
      (const uint32_t*)us->loc.p, (const int32_t*)us->signs.p, us->path_length, up.tail, pt.head, pt.lo, pt.hi, d_bad);
  CK(cudaGetLastError());
  LAUNCHED();
  CK(cudaMemcpyAsync(ex->h_scalars + 12, d_bad, sizeof(unsigned), cudaMemcpyDeviceToHost, ex->stream));
  CK(cudaStreamSynchronize(ex->stream));
  if (ex->h_scalars[12] == 0) *out = up.base;
  return GCRE_OK;
}

// The row map of a pre-counted join whose partner set of `rows` rows is scored through itself: entries k << 1 (precount_mode
// refuses sets of 2^31 rows or more)
static int identity_map(gcre_exec* ex, uint32_t rows, const uint32_t** out) {
  if (rows > ex->ident_rows) {
    CKS(ex->ident.ensure((size_t)rows * 4));
    selection_entries_kernel<<<grid_for((long long)rows, 256), 256, 0, ex->stream>>>(nullptr, rows, (uint32_t*)ex->ident.p);
    CK(cudaGetLastError());
    LAUNCHED();
    ex->ident_rows = rows;
  }
  *out = (const uint32_t*)ex->ident.p;
  return GCRE_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// join
// ------------------------------------------------------------------------------------------------------------------
static int launch_join_dense(gcre_exec* ex, const JoinParams& jp, bool keep, int* launches) {
  const unsigned long long n_pairs = jp.pair_end - jp.pair_begin;
  if (n_pairs == 0) return GCRE_OK;
  const unsigned long long tiles = (n_pairs + dense::TP - 1) / dense::TP;
  const unsigned long long blocks = tiles * jp.n_perm_tiles;
  if (blocks > 0x7fffffffull) return fail(GCRE_ERR_ARG, "join chunk too large");
  const unsigned g = (unsigned)blocks;
  if (ex->M == 1) {
    if (keep) join_dense_kernel<1, true><<<g, dense::THREADS, 0, ex->stream>>>(jp);
    else join_dense_kernel<1, false><<<g, dense::THREADS, 0, ex->stream>>>(jp);
  } else {
    if (keep) join_dense_kernel<2, true><<<g, dense::THREADS, 0, ex->stream>>>(jp);
    else join_dense_kernel<2, false><<<g, dense::THREADS, 0, ex->stream>>>(jp);
  }
  CK(cudaGetLastError());
      LAUNCHED();
  (*launches)++;
  return GCRE_OK;
}

// Build the device-resident join index.  The host only copies the uid_ref array; splitting it into the arrays the kernels
// read, the two prefix sums, the unit table and the pre-check bounds are computed on the device (the host loop this
// replaces took 14 ms for the 1.35 M upstream rows of the level-4 join - as long as the join itself).
static int build_uidset(gcre_exec* ex, int path_length, const gcre_uid_ref* uids, uint32_t n_uids, const int32_t* signs, uint32_t n_signs,
                        gcre_uidset* us) {
  static_assert(sizeof(UidRefPOD) == sizeof(gcre_uid_ref), "uid_ref layout");
  us->ex = ex;
  for (DevBuf* b : {&us->count, &us->loc, &us->prefix, &us->res, &us->units, &us->unit_idx, &us->signs, &us->grp.mem_rng, &us->grp.members,
                    &us->grp.unit_list})
    b->owner = ex;
  us->path_length = path_length;
  us->n_uids = n_uids;
  us->n_signs = n_signs;
  const size_t n1 = (size_t)n_uids + 1;
  CKS(us->count.ensure(std::max<size_t>(n_uids, 1) * 4));
  CKS(us->loc.ensure(std::max<size_t>(n_uids, 1) * 4));
  CKS(us->res.ensure(std::max<size_t>(n_uids, 1) * 8));
  CKS(us->prefix.ensure(n1 * 8));
  CKS(us->units.ensure(n1 * 8));
  CKS(us->signs.ensure(std::max<size_t>(n_signs, 1) * 4));
  if (n_signs) CK(cudaMemcpyAsync(us->signs.p, signs, (size_t)n_signs * 4, cudaMemcpyHostToDevice, ex->stream));
  CKS(ex->scratch.ensure(std::max<size_t>(n_uids, 1) * sizeof(gcre_uid_ref) + sizeof(UidStats)));
  UidRefPOD* d_aos = (UidRefPOD*)ex->scratch.p;
  UidStats* d_stats = (UidStats*)((char*)ex->scratch.p + std::max<size_t>(n_uids, 1) * sizeof(gcre_uid_ref));
  if (n_uids) CK(cudaMemcpyAsync(d_aos, uids, (size_t)n_uids * sizeof(gcre_uid_ref), cudaMemcpyHostToDevice, ex->stream));
  CK(cudaMemsetAsync(d_stats, 0, sizeof(UidStats), ex->stream));
  split_uids_kernel<<<grid_for((long long)n1, 256), 256, 0, ex->stream>>>(d_aos, n_uids, sparse::PB, (int32_t*)us->count.p, (uint32_t*)us->loc.p,
                                                                         (unsigned long long*)us->res.p, (unsigned long long*)us->prefix.p,
                                                                         (unsigned long long*)us->units.p, d_stats);
  CK(cudaGetLastError());
      LAUNCHED();
  // exclusive prefix sums in place over n + 1 entries: prefix[u] = first pair of row u, units[u] = first work unit of row u
  size_t tmp_bytes = 0;
  unsigned long long* d_prefix = (unsigned long long*)us->prefix.p;
  unsigned long long* d_units = (unsigned long long*)us->units.p;
  CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_prefix, d_prefix, (int)n1, ex->stream));
  CKS(ex->scan_tmp.ensure(tmp_bytes));
  CK(cub::DeviceScan::ExclusiveSum(ex->scan_tmp.p, tmp_bytes, d_prefix, d_prefix, (int)n1, ex->stream));
  CK(cub::DeviceScan::ExclusiveSum(ex->scan_tmp.p, tmp_bytes, d_units, d_units, (int)n1, ex->stream));
      LAUNCHED();
      LAUNCHED();
  unsigned long long tails[2] = {0, 0};
  CK(cudaMemcpyAsync(&tails[0], d_prefix + n_uids, 8, cudaMemcpyDeviceToHost, ex->stream));
  CK(cudaMemcpyAsync(&tails[1], d_units + n_uids, 8, cudaMemcpyDeviceToHost, ex->stream));
  CK(cudaStreamSynchronize(ex->stream));
  us->total = tails[0];
  us->n_units_total = tails[1];
  if (us->n_units_total > 0xfffffff0ull) return fail(GCRE_ERR_ARG, "join too large: more than 2^32 work units");
  CKS(us->unit_idx.ensure(std::max<size_t>((size_t)us->n_units_total, 1) * 4));
  if (n_uids) {
    finish_uids_kernel<<<grid_for((long long)n_uids, 256), 256, 0, ex->stream>>>(n_uids, (const int32_t*)us->count.p, (const unsigned long long*)us->res.p,
                                                                                d_prefix, d_units, (uint32_t*)us->unit_idx.p, d_stats);
    CK(cudaGetLastError());
      LAUNCHED();
  }
  UidStats h_stats;
  CK(cudaMemcpyAsync(&h_stats, d_stats, sizeof h_stats, cudaMemcpyDeviceToHost, ex->stream));
  CK(cudaStreamSynchronize(ex->stream));  // also: the caller's uid array and the scratch staging are free again
  us->max_loc_end = h_stats.max_loc_end;
  us->max_res_end = h_stats.max_res_end;
  us->res_is_prefix = h_stats.res_not_prefix == 0;
  return GCRE_OK;
}

// first pair / first work unit of upstream row u (u == n_uids gives the totals)
static int uidset_bounds(const gcre_uidset* us, uint32_t u, unsigned long long* pair, unsigned long long* unit) {
  if (u == 0) {
    *pair = 0;
    *unit = 0;
    return GCRE_OK;
  }
  if (u >= us->n_uids) {
    *pair = us->total;
    *unit = us->n_units_total;
    return GCRE_OK;
  }
  CK(cudaMemcpyAsync(pair, (const unsigned long long*)us->prefix.p + u, 8, cudaMemcpyDeviceToHost, us->ex->stream));
  CK(cudaMemcpyAsync(unit, (const unsigned long long*)us->units.p + u, 8, cudaMemcpyDeviceToHost, us->ex->stream));
  CK(cudaStreamSynchronize(us->ex->stream));
  return GCRE_OK;
}

static void free_uidset_buffers(gcre_uidset* us) {
  us->count.release();
  us->loc.release();
  us->prefix.release();
  us->res.release();
  us->units.release();
  us->unit_idx.release();
  us->signs.release();
  us->grp.mem_rng.release();
  us->grp.members.release();
  us->grp.unit_list.release();
  us->grp.built = false;
}

extern "C" int gcre_uidset_create(gcre_exec* ex, int path_length, const gcre_uid_ref* uids, uint32_t n_uids, const int32_t* signs,
                                  uint32_t n_signs, gcre_uidset** out) {
  if (!ex || !out || (!uids && n_uids) || (!signs && n_signs)) return fail(GCRE_ERR_ARG, "null argument");
  *out = nullptr;
  CKS(use_device(ex));
  gcre_uidset* us = new (std::nothrow) gcre_uidset();
  if (!us) return fail(GCRE_ERR_NOMEM, "host allocation failed");
  const int rc = build_uidset(ex, path_length, uids, n_uids, signs, n_signs, us);
  if (rc != GCRE_OK) {
    free_uidset_buffers(us);
    delete us;
    return rc;
  }
  {
    std::lock_guard<std::mutex> lock(ex->child_mu);
    ex->uidsets.insert(us);
  }
  *out = us;
  return GCRE_OK;
}

extern "C" int gcre_uidset_destroy(gcre_uidset* us) {
  if (!us) return GCRE_OK;
  if (us->ex) {
    cudaSetDevice(us->ex->device);
    cudaStreamSynchronize(us->ex->stream);
    {
      std::lock_guard<std::mutex> lock(us->ex->child_mu);
      us->ex->uidsets.erase(us);
    }
    free_uidset_buffers(us);
  }
  delete us;
  return GCRE_OK;
}

static int env_01(const char* name) {  // '0' / '1' -> 0 / 1, anything else -1
  const char* e = std::getenv(name);
  return e && (*e == '0' || *e == '1') ? *e - '0' : -1;
}

static size_t env_mb(const char* name, size_t otherwise) {  // megabytes, in bytes
  const char* e = std::getenv(name);
  return e ? (size_t)std::strtoull(e, nullptr, 10) << 20 : otherwise;
}

static int env_precount() {  // GCRE_PRECOUNT (GCRE_TEST_PRECOUNT in the tests) = 0 / 1 / s
  const char* f = std::getenv("GCRE_TEST_PRECOUNT");
  if (!f) f = std::getenv("GCRE_PRECOUNT");
  if (f && (*f == '0' || *f == '1')) return *f == '1' ? PRECOUNT_YES : PRECOUNT_NO;
  return f && *f == 's' ? PRECOUNT_SAMPLE : -1;
}

// Tuning knobs and test hooks of one join, read from the environment when the join starts (not once per process: tests change
// them between joins).  -1: not set.
struct JoinKnobs {
  int thr = env_01("GCRE_THR");            // 0 / 1: thresholded look-ups off / on for every join
  int precount = env_precount();           // PRECOUNT_NO / _YES / _SAMPLE for every join the budget allows (precount_mode)
  int tail = env_01("GCRE_TEST_TAIL");     // 0 / 1: the tail form never / on joins of any size
  int dedup = env_01("GCRE_TEST_DEDUP");   // 0 / 1: grouping of equal upstream rows never / on joins of any size, however few duplicates
  bool dedup_collide = env_01("GCRE_TEST_DEDUP_COLLIDE") == 1;  // grouping keys without the fingerprints: every row of a partner
                                                                // range collides and only the word compare tells
  int sc_pts = env_01("GCRE_SC_PTS");      // 0 / 1: the shared-memory form of the split-carrier kernels off / on where it fits
  bool no_emit = env_01("GCRE_TEST_EMIT") == 0;  // kept rows do not take their counts along
  // every launch-plan size shrunk, so the prefix / budget-overflow / redo paths of run_launch_plan run on tiny joins
  bool small_plan = std::getenv("GCRE_TEST_SMALL_PLAN") != nullptr;
  bool view_exact = std::getenv("GCRE_TEST_VIEW_EXACT") != nullptr;  // carrier lists allocated by their exact total (ensure_view)
  size_t precount_budget = env_mb("GCRE_PRECOUNT_MAX_MB", (size_t)24 << 30);  // device bytes a table of per-permutation counts may take
};

// One join: its operands and the upstream rows [ub, ue) it covers, with their pairs and sparse work units
struct JoinCall {
  gcre_exec* ex;
  const gcre_uidset* us;
  const gcre_pathset *paths0, *paths1;
  gcre_pathset* paths_res;
  bool keep;
  int top_k;
  uint32_t ub, ue;
  unsigned long long pair_lo, pair_hi, unit_lo, unit_hi;
  JoinKnobs knobs;
};

// How a join runs.  choose_join_form decides it; what follows reads it and decides nothing again.
struct JoinForm {
  int kernel = GCRE_KERNEL_DENSE;
  bool split = false;                        // the split-carrier kernels (join_sparse_sc.cuh)
  bool precount = false;                     // pre-counted partners: the partner set itself, or the base set of a selection partner
  const gcre_pathset* pc_set = nullptr;      // PC kernels of join_sparse.cuh: partners are scored through this set's carrier lists
                                             // and pre-counted table (with `precount` as above, else the base set of the tail form)
  const uint32_t* map1 = nullptr;            // ... through these rows of it: per partner row, pc_set row << 1 | halves swapped
  bool emit = false;                         // kept rows take their counts along
  bool base_emitted = false;                 // the upstream rows carry counts and totals from the join that made them
  bool thr = false;                          // thresholded look-ups
  int layout = 0;                            // count-table layout: 0, or the split-carrier kernels' words per lane group
  size_t entry_bytes = 0;                    // bytes of one (row, half) entry of a count table in that layout
  const gcre_uidset::Grouping* grp = nullptr;  // representatives of equal upstream rows only (group_upstream_rows)
};

// the kernel parameters that name a join's operands and its index: the pairs, whatever the form
static JoinParams pair_params(const gcre_exec* ex, const gcre_uidset* us, const gcre_pathset* paths0, const gcre_pathset* paths1) {
  JoinParams q;
  memset(&q, 0, sizeof q);
  q.p0 = paths0->d_rows;
  q.p1 = paths1->d_rows;
  q.Wp = ex->Wp;
  q.count = (const int32_t*)us->count.p;
  q.location = (const uint32_t*)us->loc.p;
  q.prefix = (const unsigned long long*)us->prefix.p;
  q.res_idx = (const unsigned long long*)us->res.p;
  q.n_uids = us->n_uids;
  q.signs = (const int32_t*)us->signs.p;
  q.path_length = us->path_length;
  return q;
}

// Carriers the partner rows share with (sums[0]) and add to (sums[1]) their upstream rows, over n_samples pairs spread evenly
// over [pair_lo, pair_hi): one launch and one read-back (~40 us)
static int sample_overlap(gcre_exec* ex, const gcre_uidset* us, const gcre_pathset* paths0, const gcre_pathset* paths1, unsigned long long pair_lo,
                          unsigned long long pair_hi, int n_samples, unsigned long long sums[2]) {
  const JoinParams q = pair_params(ex, us, paths0, paths1);
  unsigned long long* d_sums = reinterpret_cast<unsigned long long*>(ex->d_scalars + 8);
  CK(cudaMemsetAsync(d_sums, 0, 2 * sizeof(unsigned long long), ex->stream));
  (ex->M == 1 ? sample_overlap_kernel<1> : sample_overlap_kernel<2>)<<<grid_for((long long)n_samples * 32, 256), 256, 0, ex->stream>>>(q, pair_lo, pair_hi,
                                                                                                                                      n_samples, d_sums);
  CK(cudaGetLastError());
  LAUNCHED();
  CK(cudaMemcpyAsync(ex->h_scalars + 8, d_sums, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ex->stream));
  CK(cudaStreamSynchronize(ex->stream));
  memcpy(sums, ex->h_scalars + 8, 2 * sizeof(unsigned long long));
  return GCRE_OK;
}

// Grouping of equal upstream rows (setup_kernels.cuh: group_*).  A score-only join scores one representative of rows with equal
// bits and equal index entries, and its candidates are taken in for the other rows too (expand_members).  Measured on B200 at
// 1,000 W with the level-4 join of BASELINE config 3 (1.35 M upstream rows, 12 M pairs; profiles/r7_*): the set-up costs 0.95 /
// 1.05 ms per join (methods 1 / 2; the word compare of the members 0.70 / 0.79 of it, the sort 0.17), the fingerprints 0.38 ms of
// the level-3 join that emits them; 827 K / 766 K rows are members, and the join kernel falls from 5.9 / 11.3 to
// 2.6 / 5.7 ms.  GROUP_MIN_PAIRS: smaller joins do not group (below ~1 M pairs the whole join takes about what the set-up
// takes).  GROUP_MAX_UNIT_SHARE: the grouping is used when the representatives keep at most this share of the units - the
// kernel time saved, (1 - share) x 5.9 ms for method 1, then still pays for the ~1 ms set-up (break-even ~0.83; method 2 ~0.91).
constexpr unsigned long long GROUP_MIN_PAIRS = 1ull << 20;
constexpr double GROUP_MAX_UNIT_SHARE = 0.8;

struct MaxU32 {
  __device__ __forceinline__ uint32_t operator()(uint32_t a, uint32_t b) const { return a > b ? a : b; }
};

// The grouping of upstream rows [ub, ue) of the join, built or found current on the join index.  One read-back.
static int group_upstream_rows(const JoinCall& c, const gcre_uidset::Grouping** out) {
  gcre_exec* ex = c.ex;
  const gcre_uidset* us = c.us;
  gcre_uidset::Grouping& g = us->grp;
  const gcre_pathset* p0 = c.paths0;
  const bool collide = c.knobs.dedup_collide;
  *out = nullptr;
  if (!(g.built && g.set_uid == p0->uid && g.set_ver == p0->ver && g.ub == c.ub && g.ue == c.ue && g.collide == collide)) {
    g.built = false;
    const uint32_t n = c.ue - c.ub;
    const unsigned long long n_units = c.unit_hi - c.unit_lo;
    const int32_t* signs = ex->M == 2 && us->path_length >= 3 ? (const int32_t*)us->signs.p : nullptr;  // need_flip reads signs[idx]
    unsigned long long *keys = nullptr, *keys_s = nullptr;
    uint32_t *rows = nullptr, *rows_s = nullptr, *head = nullptr, *member = nullptr, *slot = nullptr, *unit_ids = nullptr;
    unsigned long long* d_out = nullptr;  // [0] representatives' units, [1] members
    uint8_t *is_rep = nullptr, *flags = nullptr;
    int rc = [&]() -> int {
      CK(dev_alloc(ex, (void**)&keys, (size_t)n * 8));
      CK(dev_alloc(ex, (void**)&keys_s, (size_t)n * 8));
      CK(dev_alloc(ex, (void**)&rows, (size_t)n * 4));
      CK(dev_alloc(ex, (void**)&rows_s, (size_t)n * 4));
      CK(dev_alloc(ex, (void**)&head, (size_t)n * 4));
      CK(dev_alloc(ex, (void**)&member, ((size_t)n + 1) * 4));
      CK(dev_alloc(ex, (void**)&slot, ((size_t)n + 1) * 4));
      CK(dev_alloc(ex, (void**)&is_rep, std::max<size_t>(us->n_uids, 1)));
      CK(dev_alloc(ex, (void**)&unit_ids, std::max<size_t>(n_units, 1) * 4));
      CK(dev_alloc(ex, (void**)&flags, std::max<size_t>(n_units, 1)));
      CK(dev_alloc(ex, (void**)&d_out, 2 * sizeof(unsigned long long)));
      CK(cudaMemsetAsync(d_out, 0, 2 * sizeof(unsigned long long), ex->stream));
      CKS(g.mem_rng.ensure(std::max<size_t>(us->n_uids, 1) * sizeof(uint2)));
      CKS(g.members.ensure(std::max<size_t>(n, 1) * 4));
      CKS(g.unit_list.ensure(std::max<size_t>(n_units, 1) * 4));
      size_t b_sort = 0, b_max = 0, b_sum = 0, b_sel = 0;
      CK(cub::DeviceRadixSort::SortPairs(nullptr, b_sort, keys, keys_s, rows, rows_s, (int)n, 0, 64, ex->stream));
      CK(cub::DeviceScan::InclusiveScan(nullptr, b_max, head, head, MaxU32(), (int)n, ex->stream));
      CK(cub::DeviceScan::ExclusiveSum(nullptr, b_sum, member, slot, (int)n + 1, ex->stream));
      CK(cub::DeviceSelect::Flagged(nullptr, b_sel, unit_ids, flags, (uint32_t*)g.unit_list.p, d_out, (long long)n_units, ex->stream));
      const size_t tmp_bytes = std::max(std::max(b_sort, b_max), std::max(b_sum, b_sel));
      CKS(ex->scan_tmp.ensure(tmp_bytes));
      void* tmp = ex->scan_tmp.p;
      size_t tb = tmp_bytes;
      group_keys_kernel<<<grid_for(n, 256), 256, 0, ex->stream>>>(c.ub, n, collide ? nullptr : p0->view.fp, (const int32_t*)us->count.p,
                                                                  (const uint32_t*)us->loc.p, signs, keys, rows);
      CK(cudaGetLastError());
      LAUNCHED();
      CK(cub::DeviceRadixSort::SortPairs(tmp, tb, keys, keys_s, rows, rows_s, (int)n, 0, 64, ex->stream));
      LAUNCHED();
      group_heads_kernel<<<grid_for(n, 256), 256, 0, ex->stream>>>(n, keys_s, head);
      CK(cudaGetLastError());
      LAUNCHED();
      tb = tmp_bytes;
      CK(cub::DeviceScan::InclusiveScan(tmp, tb, head, head, MaxU32(), (int)n, ex->stream));
      LAUNCHED();
      group_verify_kernel<<<grid_for((long long)n * 32, 256), 256, 0, ex->stream>>>(n, rows_s, head, p0->d_rows, (int)row_words(ex),
                                                                                   (const int32_t*)us->count.p, (const uint32_t*)us->loc.p, signs, member);
      CK(cudaGetLastError());
      LAUNCHED();
      CK(cudaMemsetAsync(member + n, 0, 4, ex->stream));
      tb = tmp_bytes;
      CK(cub::DeviceScan::ExclusiveSum(tmp, tb, member, slot, (int)n + 1, ex->stream));
      LAUNCHED();
      CK(cudaMemsetAsync(g.mem_rng.p, 0, (size_t)us->n_uids * sizeof(uint2), ex->stream));
      group_finish_kernel<<<grid_for(n, 256), 256, 0, ex->stream>>>(n, rows_s, head, member, slot, (uint32_t*)g.members.p, (uint2*)g.mem_rng.p, is_rep);
      CK(cudaGetLastError());
      LAUNCHED();
      group_unit_flags_kernel<<<grid_for((long long)n_units, 256), 256, 0, ex->stream>>>(c.unit_lo, n_units, (const uint32_t*)us->unit_idx.p, is_rep,
                                                                                        unit_ids, flags);
      CK(cudaGetLastError());
      LAUNCHED();
      tb = tmp_bytes;
      CK(cub::DeviceSelect::Flagged(tmp, tb, unit_ids, flags, (uint32_t*)g.unit_list.p, d_out, (long long)n_units, ex->stream));
      LAUNCHED();
      CK(cudaMemcpyAsync(d_out + 1, slot + n, 4, cudaMemcpyDeviceToDevice, ex->stream));
      CK(cudaMemcpyAsync(ex->h_scalars + 8, d_out, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ex->stream));
      CK(cudaStreamSynchronize(ex->stream));
      unsigned long long h[2];
      memcpy(h, ex->h_scalars + 8, sizeof h);
      g.n_units = h[0];
      g.dedup_rows = (uint32_t)h[1];
      g.pays = (double)g.n_units <= GROUP_MAX_UNIT_SHARE * (double)n_units;
      g.set_uid = p0->uid;
      g.set_ver = p0->ver;
      g.ub = c.ub;
      g.ue = c.ue;
      g.collide = collide;
      g.h_members_valid = false;
      g.built = true;
      return GCRE_OK;
    }();
    for (void* p : {(void*)keys, (void*)keys_s, (void*)rows, (void*)rows_s, (void*)head, (void*)member, (void*)slot, (void*)is_rep, (void*)unit_ids,
                    (void*)flags, (void*)d_out})
      dev_free(ex, p);
    CKS(rc);
  }
  if (g.pays || c.knobs.dedup == 1) *out = &g;
  return GCRE_OK;
}

// The kernel form of a join, in this order: the requested family or AUTO's (cost model, and an overlap sample when the bound
// does not decide); the fallback to dense where the sparse kernel cannot run; for the sparse kernel the tail form (one device
// pass), pre-counted partners, split carriers, emitted counts, and the overlap sample that settles pre-counting.  The only
// device work of the decision is here.  t_needed: carriers a joined half-row may have; mp1: the partner's densest half-row.
static int choose_join_form(const JoinCall& c, int requested, long long t_needed, long long mp1, JoinForm* f) {
  gcre_exec* ex = c.ex;
  const unsigned long long pairs = c.pair_hi - c.pair_lo;
  const int npb = ex->Iw / 32;
  f->kernel = requested == GCRE_KERNEL_SPARSE ? GCRE_KERNEL_SPARSE : GCRE_KERNEL_DENSE;
  if (requested != GCRE_KERNEL_DENSE && requested != GCRE_KERNEL_SPARSE && sparse_supported(ex->n, t_needed, ex->Iw)) {  // AUTO
    const double dense_ns = dense_pair_ns(ex->W64, ex->Ip, ex->M);
    if (sparse_pair_ns(npb, ex->M, (double)mp1 * ex->M) <= dense_ns) {
      f->kernel = GCRE_KERNEL_SPARSE;  // wins even if every partner added its densest half-row in full
    } else if (sparse_pair_ns(npb, ex->M, 0.0) < dense_ns && pairs > 0) {
      // it depends on the rows: carriers a partner adds to its upstream row, averaged over 2,048 pairs spread over the join
      const int n_samples = (int)std::min<unsigned long long>(2048, pairs);
      unsigned long long sums[2];
      CKS(sample_overlap(ex, c.us, c.paths0, c.paths1, c.pair_lo, c.pair_hi, n_samples, sums));
      if (sparse_pair_ns(npb, ex->M, (double)sums[1] / n_samples) <= dense_ns) f->kernel = GCRE_KERNEL_SPARSE;
    }
  }
  // an explicit request for the sparse kernel is honoured whenever its index widths allow
  if (f->kernel == GCRE_KERNEL_SPARSE && !sparse_supported(ex->n, t_needed, ex->Iw)) f->kernel = GCRE_KERNEL_DENSE;
  if (f->kernel != GCRE_KERNEL_SPARSE) return GCRE_OK;
  const size_t budget = c.knobs.precount_budget;
  // Tail form (join_sparse.cuh): large score-only joins on the 1,024-permutation kernel whose every pair adds one gene of a
  // base set to its upstream row, when the base set's count table fits the budget.  GCRE_TEST_TAIL=1 / 0 (test hook) takes
  // it on joins of any size / never.
  if (!c.keep && !ex->split_ok && pairs > 0) {
    const bool want = c.knobs.tail >= 0 ? c.knobs.tail == 1 : pairs >= (1ull << 20);
    if (want) CKS(tail_form_base(ex, c.us, c.paths0, c.paths1, c.ub, c.ue, c.unit_lo, c.unit_hi, &f->pc_set));
    if (f->pc_set && (size_t)f->pc_set->size * ex->M * npb * 2048 > budget) f->pc_set = nullptr;
    if (f->pc_set) f->map1 = c.paths1->prov.tail;
  }
  // A KEEP join whose partner set is a live selection of a base set (level 3: data1's gene rows) may score its partners through
  // the base set's rows and pre-counted table (join_sparse.cuh): a selected row is its base row, so no eligibility pass
  const Provenance& sel = c.paths1->prov;
  const gcre_pathset* sel_base = c.keep && !ex->split_ok && sel.sel && base_current(ex, sel) ? sel.base : nullptr;
  int pc_mode = f->pc_set ? PRECOUNT_NO
                : sel_base   ? precount_mode(pairs, sel_base->size, ex->M, npb, budget, c.knobs.precount, true)
                             : precount_mode(pairs, c.paths1->size, ex->M, npb, budget, c.knobs.precount, false);
  if (ex->split_ok && pc_mode == PRECOUNT_SAMPLE) pc_mode = PRECOUNT_NO;  // the split-carrier kernel is the better form there
  // <= 512 permutations: the split-carrier kernels (join_sparse_sc.cuh) run - unless pre-counted partners are forced
  // (GCRE_PRECOUNT=1) - and emit / consume count tables in their own, smaller layout
  f->split = ex->split_ok && pc_mode != PRECOUNT_YES;
  f->layout = f->split ? sparse_sc_words(ex->Ip) : 0;
  f->entry_bytes = f->split ? sparse_sc_table_bytes(ex->Ip) : (size_t)npb * 2048;
  f->thr = !f->split && sparse_thr(ex->M, pairs, c.knobs.thr);
  // upstream operand: rows that came out of a KEEP join carry their counts and totals - no carrier lists needed
  const SparseView& v0 = c.paths0->view;
  f->base_emitted = v0.pcnt && v0.pcnt_gen == ex->mask_gen && v0.pcnt_layout == f->layout && v0.stats_valid && c.paths0 != c.paths_res &&
                    c.ub >= v0.emit_lo && c.ue <= v0.emit_hi;
  // kept rows take their counts along (join_sparse.cuh, join_sparse_sc.cuh) when result rows are the running sums of the
  // counts (res_is_prefix: rows [pair_lo, pair_hi) are exactly the ones this call writes)
  f->emit = (f->split || !ex->split_ok) && c.keep && pairs > 0 && c.us->res_is_prefix && c.paths_res != c.paths0 && c.paths_res != c.paths1 &&
            !c.knobs.no_emit && (size_t)c.paths_res->size * ex->M * f->entry_bytes <= budget;
  // unforced, an emitting join pre-counts only through a selection's base set (a table of the partner set itself would be built
  // for this one join)
  if (f->emit && !f->split && !sel_base && c.knobs.precount < 0) pc_mode = PRECOUNT_NO;
  if (pc_mode == PRECOUNT_SAMPLE) {
    // how much of a partner row is already in its upstream row
    unsigned long long sums[2];
    CKS(sample_overlap(ex, c.us, c.paths0, c.paths1, c.pair_lo, c.pair_hi, 2048, sums));
    pc_mode = (sums[0] * 10 < sums[1] * 6) ? PRECOUNT_YES : PRECOUNT_NO;
  }
  f->precount = pc_mode == PRECOUNT_YES;
  if (f->precount) {
    f->pc_set = sel_base ? sel_base : c.paths1;
    if (sel_base) f->map1 = sel.sel;
    else CKS(identity_map(ex, c.paths1->size, &f->map1));
  }
  // score-only joins whose upstream rows carry fingerprints score each group of equal rows once; GCRE_TEST_DEDUP=1 / 0 (test
  // hook) groups on joins of any size / never
  if (!c.keep && pairs > 0 && v0.fp && c.ub >= v0.emit_lo && c.ue <= v0.emit_hi && c.ue > c.ub) {
    const bool want = c.knobs.dedup >= 0 ? c.knobs.dedup == 1 : pairs >= GROUP_MIN_PAIRS;
    if (want) CKS(group_upstream_rows(c, &f->grp));
  }
  return GCRE_OK;
}

// What the form reads: patient-major masks, carrier lists of the upstream rows and of the partner (the tail base in tail form),
// count tables, the result's emitted tables; then the kernel parameters
static int prepare_join_operands(const JoinCall& c, const JoinForm& f, JoinParams* jp, SparseParams* sp) {
  gcre_exec* ex = c.ex;
  memset(sp, 0, sizeof *sp);
  if (f.kernel == GCRE_KERNEL_SPARSE) {
    CKS(ensure_patient_major(ex, f.split));
    gcre_pathset* p0 = const_cast<gcre_pathset*>(c.paths0);
    gcre_pathset* p1 = const_cast<gcre_pathset*>(f.pc_set ? f.pc_set : c.paths1);
    if (!f.base_emitted) CKS(ensure_view(ex, p0, c.knobs.view_exact));
    CKS(ensure_view(ex, p1, c.knobs.view_exact));
    if (f.pc_set) CKS(ensure_precount(ex, p1));
    sp->off0 = p0->view.off; sp->len0 = p0->view.len; sp->car0 = p0->view.car; sp->ncase0 = p0->view.ncase;
    sp->pcnt0 = f.base_emitted ? p0->view.pcnt : nullptr;
    sp->off1 = p1->view.off; sp->len1 = p1->view.len; sp->car1 = p1->view.car; sp->ncase1 = p1->view.ncase;
    sp->pcnt1 = f.pc_set ? p1->view.pcnt : nullptr;
    sp->map1 = f.map1;
    sp->n = ex->n;
    sp->unit_prefix = (const unsigned long long*)c.us->units.p;
    sp->unit_idx = (const uint32_t*)c.us->unit_idx.p;
    sp->work_counter = (unsigned long long*)(ex->d_scalars + 2);
    sp->n_perm_blocks = ex->Iw / 32;
    sp->exact_pairs = reinterpret_cast<unsigned long long*>(ex->d_scalars + 4);
    gcre_pathset* res = c.paths_res;
    if (c.keep && res != c.paths0 && res != c.paths1) drop_view(res);  // its rows are about to be rewritten
    if (f.emit) {
      const size_t items = (size_t)res->size * ex->M;
      CK(dev_alloc(ex, (void**)&res->view.pcnt, items * f.entry_bytes));
      res->view.pcnt_layout = f.layout;
      CK(dev_alloc(ex, (void**)&res->view.len, items * 4));
      CK(dev_alloc(ex, (void**)&res->view.ncase, items * 4));
      CK(dev_alloc(ex, (void**)&res->view.fp, std::max<size_t>(res->size, 1) * 8));
      sp->fp_res = res->view.fp;
      sp->pcnt_res = res->view.pcnt;
      sp->len_res = res->view.len;
      sp->ncase_res = res->view.ncase;
    }
  }
  CK(cudaMemsetAsync(ex->d_perm_max, 0, (size_t)ex->Ip * 4, ex->stream));
  CK(cudaMemsetAsync(ex->d_scalars, 0, 2 * sizeof(unsigned), ex->stream));
  *jp = pair_params(ex, c.us, c.paths0, c.paths1);
  jp->pres = c.keep ? c.paths_res->d_rows : nullptr;
  jp->n_cases = ex->n_cases;
  jp->pm = ex->d_pm;
  jp->pt = f.split ? ex->d_pt_sc : ex->d_pt;
  jp->Ip = ex->Ip;
  jp->Iw = f.split ? sparse_sc_words(ex->Ip) : ex->Iw;
  jp->n_perm_tiles = ex->Ip / dense::TI;
  jp->diagD = ex->d_diagD;
  jp->diagF = ex->d_diagF;
  jp->diagDM = ex->d_diagDM;
  jp->diagFM = ex->d_diagFM;
  jp->perm_max = ex->d_perm_max;
  jp->cand_count = ex->d_scalars;
  jp->max_total = ex->d_scalars + 1;
  if (f.kernel == GCRE_KERNEL_SPARSE && c.top_k <= 64) {
    CK(cudaMemsetAsync(ex->d_topk, 0, 65 * sizeof(unsigned long long), ex->stream));
    jp->dyn_thr = ex->d_topk;
    jp->slots = ex->d_topk + 1;
    jp->n_slots = c.top_k;
  }
  if (f.grp) {
    sp->unit_list = (const uint32_t*)f.grp->unit_list.p;
  }
  return GCRE_OK;
}

struct LaunchStats {  // of one join's launch plan (gcre_join_opts)
  double kernel_ms = 0.0;
  int launches = 0;
  unsigned long long exact_pairs = 0;
  bool shared_masks = false;
};

// Grouped upstream rows: the candidates `cand` of representatives, taken in by the host, are also candidates of the member rows
// of their rows - the same pair but for the row, so the same score and counts.  Of a group only the first top_k - 1 members can
// be among the K best with a given partner (ties go to the smaller row), so no more are taken in.  One small gather of the
// candidates' member ranges on the device; the members themselves are read back once per grouping, when first needed.
static int expand_members(gcre_exec* ex, const gcre_uidset::Grouping& g, const std::vector<Cand>& cand, int top_k, std::vector<gcre_score>* held) {
  const unsigned n = (unsigned)cand.size();
  if (n == 0 || g.dedup_rows == 0 || top_k < 2) return GCRE_OK;
  CKS(ex->scratch.ensure((size_t)n * (sizeof(uint32_t) + sizeof(uint2)) + 8));
  uint32_t* d_rows = (uint32_t*)ex->scratch.p;
  uint2* d_rng = (uint2*)(d_rows + n + (n & 1));
  std::vector<uint32_t> rows(n);
  for (unsigned k = 0; k < n; k++) rows[k] = cand[k].idx;
  std::vector<uint2> rng(n);
  CK(cudaMemcpyAsync(d_rows, rows.data(), (size_t)n * 4, cudaMemcpyHostToDevice, ex->stream));
  group_ranges_kernel<<<grid_for(n, 256), 256, 0, ex->stream>>>(n, d_rows, (const uint2*)g.mem_rng.p, d_rng);
  CK(cudaGetLastError());
  LAUNCHED();
  CK(cudaMemcpyAsync(rng.data(), d_rng, (size_t)n * sizeof(uint2), cudaMemcpyDeviceToHost, ex->stream));
  CK(cudaStreamSynchronize(ex->stream));
  for (unsigned k = 0; k < n; k++) {
    if (rng[k].y <= rng[k].x) continue;
    if (!g.h_members_valid) {
      g.h_members.resize(g.dedup_rows);
      CK(cudaMemcpyAsync(g.h_members.data(), g.members.p, (size_t)g.dedup_rows * 4, cudaMemcpyDeviceToHost, ex->stream));
      CK(cudaStreamSynchronize(ex->stream));
      g.h_members_valid = true;
    }
    const uint32_t e = std::min<uint32_t>(rng[k].y, rng[k].x + (uint32_t)(top_k - 1));
    for (uint32_t m = rng[k].x; m < e; m++) {
      gcre_score sc;
      sc.score = key_score(cand[k].key);
      sc.src = (int32_t)g.h_members[m];
      sc.trg = (int32_t)cand[k].loc;
      sc.cases = cand[k].cases;
      sc.ctrls = cand[k].ctrls;
      held->push_back(sc);
    }
  }
  return GCRE_OK;
}

// The join's launches; their candidates are merged on the host into the top-K `held`.
static int run_launch_plan(const JoinCall& c, const JoinForm& f, JoinParams jp, SparseParams sp, PhaseTrace& tr, std::vector<gcre_score>* held,
                           LaunchStats* st) {
  gcre_exec* ex = c.ex;
  // dense kernel: chunks are ranges of flattened pairs; sparse kernel: ranges of units (<= PB pairs each)
  const bool sparse_k = f.kernel == GCRE_KERNEL_SPARSE;
  const unsigned long long per_item = sparse_k ? sparse::PB : 1;
  // (grouped upstream rows: items index the representatives' units, in ascending order)
  const unsigned long long item_lo = f.grp ? 0 : sparse_k ? c.unit_lo : c.pair_lo, item_hi = f.grp ? f.grp->n_units : sparse_k ? c.unit_hi : c.pair_hi;
  // Launch plan.  Top-K candidates are appended by the kernels only when their score beats the K-th best known so far,
  // and a launch must be able to hold every candidate it may produce:
  //   * small joins (<= 64K pairs): one launch with room for every pair;
  //   * large joins, sparse kernel, top_k <= 64: ONE launch with the fixed candidate budget - the kernel raises its own
  //     threshold as candidates arrive (JoinParams::slots; measured: ~300 candidates out of 12 M pairs);
  //   * other large joins: a short prefix (threshold unknown: every pair is a candidate) establishes the K-th score, then
  //     ONE launch covers the rest with a fixed candidate budget.  Pairs are visited in ascending (src, trg) order
  //     across launches, so later pairs only displace on a strictly greater score.  If the budget overflows (scores that
  //     keep rising), that launch's candidates are dropped and the range is redone in safe chunks (cap = chunk size);
  //     permutation maxima are max-merged, so re-scoring a pair is harmless.
  // With grouped upstream rows the kernels append the representatives' candidates only; each is then also a candidate of the
  // first top_k - 1 members of its row (expand_members).  The K-th score no longer rules out a tie in later launches (a member
  // taken in early has a larger row than a representative of a later launch), so ties with it stay candidates.
  struct Seg { unsigned long long b, e; bool safe; };
  std::vector<Seg> plan;
  const bool tiny_plan = c.knobs.small_plan;
  const unsigned long long small_items = std::max<unsigned long long>(1, (tiny_plan ? 128ull : (64ull << 10)) / per_item);
  const unsigned long long prefix_items = std::max<unsigned long long>(1, (tiny_plan ? 64ull : (16ull << 10)) / per_item);
  const unsigned budget = tiny_plan ? 16u : (1u << 20);
  const unsigned long long redo_first = std::max<unsigned long long>(1, (tiny_plan ? 128ull : (256ull << 10)) / per_item);
  const unsigned long long redo_max = std::max<unsigned long long>(1, (tiny_plan ? 512ull : (4ull << 20)) / per_item);
  if (item_hi - item_lo <= small_items) {
    if (item_hi > item_lo) plan.push_back({item_lo, item_hi, true});
  } else if (jp.n_slots > 0) {
    // the kernel tightens its own threshold (JoinParams::slots): no prefix launch needed, a few hundred candidates in all
    plan.push_back({item_lo, item_hi, false});
  } else {
    plan.push_back({item_lo, item_lo + prefix_items, true});
    plan.push_back({item_lo + prefix_items, item_hi, false});
  }
  ex->h_perm_fresh = false;
  std::vector<Cand> h_cand;
  unsigned long long thr_key = score_key(-std::numeric_limits<double>::infinity());
  for (size_t si = 0; si < plan.size(); si++) {
    const Seg seg = plan[si];
    const unsigned long long p = seg.b, pe = seg.e;
    const unsigned cap = seg.safe ? (unsigned)((pe - p) * per_item) : budget;
    CKS(ex->cand.ensure((size_t)cap * sizeof(Cand)));
    jp.cand = (Cand*)ex->cand.p;
    jp.cand_cap = cap;
    jp.thr_key = thr_key;
    CK(cudaMemsetAsync(ex->d_scalars, 0, sizeof(unsigned), ex->stream));
    CK(cudaEventRecord(ex->ev0, ex->stream));
    if (sparse_k) {
      sp.unit_begin = p;
      sp.n_units = pe - p;
      CK(cudaMemsetAsync(ex->d_scalars + 2, 0, 6 * sizeof(unsigned), ex->stream));
      if (f.split) CK(launch_join_sparse_sc(ex->stream, jp, sp, ex->M, c.keep, ex->sm_count, ex->wide, c.knobs.sc_pts, &st->shared_masks));
      else CK(launch_join_sparse(ex->stream, jp, sp, ex->M, c.keep, ex->sm_count, f.pc_set != nullptr, f.thr, ex->wide));
      LAUNCHED();
      st->launches++;
    } else {
      jp.pair_begin = p;
      jp.pair_end = pe;
      CKS(launch_join_dense(ex, jp, c.keep, &st->launches));
    }
    CK(cudaEventRecord(ex->ev1, ex->stream));
    CK(cudaMemcpyAsync(ex->h_scalars, ex->d_scalars, 6 * sizeof(unsigned), cudaMemcpyDeviceToHost, ex->stream));
    if (!ex->h_res.p) CK(pinned_big_acquire((size_t)kSpecCand * sizeof(Cand) + (size_t)ex->Ip * 4, &ex->h_res));
    Cand* h_spec = static_cast<Cand*>(ex->h_res.p);
    const unsigned n_spec = std::min(cap, kSpecCand);
    CK(cudaMemcpyAsync(h_spec, ex->cand.p, (size_t)n_spec * sizeof(Cand), cudaMemcpyDeviceToHost, ex->stream));
    CK(cudaMemcpyAsync(h_spec + kSpecCand, ex->d_perm_max, (size_t)ex->Ip * 4, cudaMemcpyDeviceToHost, ex->stream));
    CK(cudaStreamSynchronize(ex->stream));
    ex->h_perm_fresh = true;
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, ex->ev0, ex->ev1));
    st->kernel_ms += ms;
    st->exact_pairs += (unsigned long long)ex->h_scalars[4] | ((unsigned long long)ex->h_scalars[5] << 32);
    if (ex->h_scalars[0] > cap) {
      // budget overflow: redo this range in safe chunks (growing x8 up to 4M pairs)
      unsigned long long chunk = redo_first;
      std::vector<Seg> redo;
      for (unsigned long long q = p; q < pe;) {
        const unsigned long long qe = std::min(pe, q + chunk);
        redo.push_back({q, qe, true});
        q = qe;
        chunk = std::min(chunk * 8, redo_max);
      }
      plan.insert(plan.begin() + si + 1, redo.begin(), redo.end());
      continue;
    }
    const unsigned n_cand = ex->h_scalars[0];
    if (tr.on) {
      char buf[96];
      snprintf(buf, sizeof buf, " [launch %llu..%llu cand=%u %.3fms]", p, pe, n_cand, ms);
      tr.line += buf;
      tr.mark("run");
    }
    if (n_cand) {
      h_cand.resize(n_cand);
      if (n_cand <= n_spec) {
        memcpy(h_cand.data(), h_spec, (size_t)n_cand * sizeof(Cand));  // already here
      } else {
        CK(cudaMemcpyAsync(h_cand.data(), ex->cand.p, (size_t)n_cand * sizeof(Cand), cudaMemcpyDeviceToHost, ex->stream));
        CK(cudaStreamSynchronize(ex->stream));
      }
      for (unsigned k = 0; k < n_cand; k++) {
        gcre_score sc;
        sc.score = key_score(h_cand[k].key);
        sc.src = (int32_t)h_cand[k].idx;
        sc.trg = (int32_t)h_cand[k].loc;
        sc.cases = h_cand[k].cases;
        sc.ctrls = h_cand[k].ctrls;
        held->push_back(sc);
      }
      if (f.grp) CKS(expand_members(ex, *f.grp, h_cand, c.top_k, held));
      trim_topk(*held, c.top_k);
      if ((int)held->size() == c.top_k) {
        double kth = (*held)[0].score;
        for (const auto& sc : *held) kth = std::min(kth, sc.score);
        // later launches hold larger (src, trg) only, so a tie with the K-th score can no longer win a place (with grouped rows
        // it can: ties stay candidates)
        thr_key = score_key(kth) - (f.grp ? 1 : 0);
      }
    }
    tr.mark("cands");
  }
  return GCRE_OK;
}

static int join_impl(gcre_exec* ex, const gcre_uidset* us, const gcre_pathset* paths0, const gcre_pathset* paths1, gcre_pathset* paths_res,
                     int top_k, gcre_score* out_scores, int* n_scores, double* out_perm, gcre_join_opts* opts, PhaseTrace& tr) {
  if (!out_perm && ex->iters > 0 && !(opts && opts->skip_host_perm)) return fail(GCRE_ERR_ARG, "null argument");
  if (paths0->ex != ex || paths1->ex != ex || (paths_res && paths_res->ex != ex)) return fail(GCRE_ERR_ARG, "path set belongs to another exec");
  if (top_k < 1) top_k = 1;
  const bool keep = paths_res && paths_res->size != 0;
  const uint32_t n_uids = us->n_uids, n_signs = us->n_signs;
  const int path_length = us->path_length;
  const unsigned long long total = us->total;

  // ---- pre-checks, src/join_base.cpp:196-200 ----
  if (n_uids != paths0->size) return fail(GCRE_ERR_ASSERT, "assertion");
  if (paths_res && !(paths_res->size == 0 || paths_res->size == total)) return fail(GCRE_ERR_ASSERT, "assertion");
  if (us->max_loc_end > paths1->size) return fail(GCRE_ERR_RANGE, "assertion");
  if (keep && us->max_res_end > paths_res->size) return fail(GCRE_ERR_RANGE, "assertion");
  if (ex->M == 2 && total > 0) {
    // need_flip indexes signs by upstream row and/or partner row (src/gcre.h:71-81); the reference reads unchecked
    const unsigned long long need = path_length > 3 ? n_uids : (path_length < 3 ? us->max_loc_end : std::max<unsigned long long>(n_uids, us->max_loc_end));
    if (n_signs < need) return fail(GCRE_ERR_RANGE, "assertion");
  }

  uint32_t ub = 0, ue = n_uids;
  if (opts && opts->uid_end != 0) {
    ub = std::min(opts->uid_begin, n_uids);
    ue = std::min(std::max(opts->uid_end, ub), n_uids);
  }
  unsigned long long pair_lo = 0, pair_hi = 0, unit_lo = 0, unit_hi = 0;
  CKS(uidset_bounds(us, ub, &pair_lo, &unit_lo));
  CKS(uidset_bounds(us, ue, &pair_hi, &unit_hi));

  reap_staged(ex, true);  // upload staging blocks go back to the cache, stream-ordered behind their unpack kernels
  CKS(materialize_zero(const_cast<gcre_pathset*>(paths0)));
  CKS(materialize_zero(const_cast<gcre_pathset*>(paths1)));
  if (keep) {
    rows_written(paths_res);  // (provenance of the new rows is recorded once they are written)
    // result rows that are the running sums of the counts: the join overwrites every word of rows [pair_lo, pair_hi); only the
    // rest of a fresh set needs its zeros (nothing for a full join)
    if (us->res_is_prefix) {
      if (paths_res->zero_pending) {
        const size_t rb = row_words(ex) * 8;
        if (pair_lo > 0) CK(cudaMemsetAsync(paths_res->d_rows, 0, (size_t)pair_lo * rb, ex->stream));
        if (pair_hi < total) CK(cudaMemsetAsync(paths_res->d_rows + (size_t)pair_hi * row_words(ex), 0, (size_t)(total - pair_hi) * rb, ex->stream));
        paths_res->zero_pending = false;
      }
    } else {
      CKS(materialize_zero(paths_res));
    }
  }

  tr.mark("checks");
  // ---- value-table coverage: a joined half-row has at most maxpop0 + maxpop1 carriers ----
  long long mp0 = 0, mp1 = 0;
  CKS(pathset_max_half_pop(const_cast<gcre_pathset*>(paths0), &mp0));
  CKS(pathset_max_half_pop(const_cast<gcre_pathset*>(paths1), &mp1));
  const long long t_needed = std::min<long long>(ex->n, mp0 + mp1);
  tr.mark("maxpop");
  CKS(ensure_diag(ex, t_needed));
  tr.mark("diag");

  const JoinCall c{ex, us, paths0, paths1, paths_res, keep, top_k, ub, ue, pair_lo, pair_hi, unit_lo, unit_hi, JoinKnobs()};
  JoinForm form;
  CKS(choose_join_form(c, opts ? opts->kernel : GCRE_KERNEL_AUTO, t_needed, mp1, &form));
  JoinParams jp;
  SparseParams sp;
  CKS(prepare_join_operands(c, form, &jp, &sp));
  tr.mark("views");
  std::vector<gcre_score> held;
  LaunchStats st;
  CKS(run_launch_plan(c, form, jp, sp, tr, &held, &st));
  tr.mark("launches");
  if (keep) {
    // The kernel's maximum covers the rows it wrote.  A join that wrote every row (a full one with prefix result rows) sets the
    // bound from them; after any other join the rows it did not write keep theirs, so an unknown bound (-1: the set was
    // loaded or set since its last join) stays unknown and a known one (0 for a fresh set) grows to cover the new rows.
    const long long prev = paths_res->max_half_pop;
    const bool every_row = us->res_is_prefix && pair_lo == 0 && pair_hi == total;
    paths_res->max_half_pop = (every_row || prev >= 0) ? std::max<long long>(prev, (long long)ex->h_scalars[1]) : -1;
    if (form.emit) {  // emitted with the rows
      paths_res->view.pcnt_gen = ex->mask_gen;
      paths_res->view.stats_valid = true;
      paths_res->view.emit_lo = pair_lo;
      paths_res->view.emit_hi = pair_hi;
    } else {
      drop_view(paths_res);
    }
    CKS(record_provenance(ex, us, paths0, paths1, paths_res, ub, ue, pair_lo, pair_hi, unit_lo, unit_hi));
  }

  CKS(emit_topk(held, top_k, out_scores, n_scores));
  if (out_perm && !(opts && opts->skip_host_perm)) {
    if (ex->h_perm_fresh && st.launches > 0) {  // the maxima came back with the last launch's scalars
      const float* hp = reinterpret_cast<const float*>(static_cast<Cand*>(ex->h_res.p) + kSpecCand);
      for (int r = 0; r < ex->iters; r++) out_perm[r] = (double)hp[r];  // src/join_base.cpp:145-146
    } else {
      CKS(gcre_exec_read_perm_max(ex, out_perm));
    }
  }
  tr.mark("results");
  tr.done(keep ? "join(keep)" : "join");
  if (opts) {
    opts->pairs_scored = pair_hi - pair_lo;
    opts->kernel_ms = st.kernel_ms;
    opts->kernel_used = form.kernel;
    opts->launches = st.launches;
    opts->precounted = form.precount;
    opts->tail_form = form.pc_set != nullptr && !form.precount;
    opts->dedup_rows = form.grp ? form.grp->dedup_rows : 0;
    opts->split_carrier = form.split;
    opts->shared_masks = st.shared_masks;
    opts->thresholded = form.thr && st.launches > 0 ? 1 : 0;
    opts->exact_pairs = st.exact_pairs;
  }
  return GCRE_OK;
}

extern "C" int gcre_join(gcre_exec* ex, int path_length, const gcre_uid_ref* uids, uint32_t n_uids, const int32_t* signs, uint32_t n_signs,
                         const gcre_pathset* paths0, const gcre_pathset* paths1, gcre_pathset* paths_res, int top_k, gcre_score* out_scores,
                         int* n_scores, double* out_perm, gcre_join_opts* opts) {
  if (!ex || !paths0 || !paths1 || !out_scores || !n_scores || (!uids && n_uids) || (!signs && n_signs))
    return fail(GCRE_ERR_ARG, "null argument");
  if (paths0->ex != ex || paths1->ex != ex || (paths_res && paths_res->ex != ex)) return fail(GCRE_ERR_ARG, "path set belongs to another exec");
  CKS(use_device(ex));
  PhaseTrace tr;
  // src/join_base.cpp:196: check_equal(uids.size(), paths0.size) - before any work on the index
  if (n_uids != paths0->size) return fail(GCRE_ERR_ASSERT, "assertion");
  gcre_uidset us;
  int rc = build_uidset(ex, path_length, uids, n_uids, signs, n_signs, &us);
  tr.mark("index");
  if (rc == GCRE_OK) rc = join_impl(ex, &us, paths0, paths1, paths_res, top_k, out_scores, n_scores, out_perm, opts, tr);
  if (rc == GCRE_OK) cudaStreamSynchronize(ex->stream);
  free_uidset_buffers(&us);
  return rc;
}

extern "C" int gcre_join_uidset(gcre_exec* ex, const gcre_uidset* uidset, const gcre_pathset* paths0, const gcre_pathset* paths1,
                                gcre_pathset* paths_res, int top_k, gcre_score* out_scores, int* n_scores, double* out_perm,
                                gcre_join_opts* opts) {
  if (!ex || !uidset || !paths0 || !paths1 || !out_scores || !n_scores) return fail(GCRE_ERR_ARG, "null argument");
  if (uidset->ex != ex) return fail(GCRE_ERR_ARG, "join index belongs to another exec");
  CKS(use_device(ex));
  PhaseTrace tr;
  return join_impl(ex, uidset, paths0, paths1, paths_res, top_k, out_scores, n_scores, out_perm, opts, tr);
}

extern "C" int gcre_exec_device_perm_max(const gcre_exec* ex, void** device_ptr, int* n_floats) {
  if (!ex || !device_ptr || !n_floats) return fail(GCRE_ERR_ARG, "null argument");
  *device_ptr = ex->d_perm_max;
  *n_floats = ex->Ip;
  return GCRE_OK;
}

extern "C" int gcre_exec_export_perm_max(const gcre_exec* ex, void* device_dst, int count) {
  if (!ex || !device_dst) return fail(GCRE_ERR_ARG, "null argument");
  if (count < 0 || count > ex->Ip) return fail(GCRE_ERR_RANGE, "assertion");
  CKS(use_device(ex));
  CK(cudaMemcpyAsync(device_dst, ex->d_perm_max, (size_t)count * 4, cudaMemcpyDeviceToDevice, ex->stream));
  return GCRE_OK;
}

extern "C" int gcre_exec_import_perm_max(gcre_exec* ex, const void* device_src, int count) {
  if (!ex || !device_src) return fail(GCRE_ERR_ARG, "null argument");
  if (count < 0 || count > ex->Ip) return fail(GCRE_ERR_RANGE, "assertion");
  CKS(use_device(ex));
  CK(cudaMemcpyAsync(ex->d_perm_max, device_src, (size_t)count * 4, cudaMemcpyDeviceToDevice, ex->stream));
  ex->h_perm_fresh = false;
  return GCRE_OK;
}

extern "C" int gcre_exec_read_perm_max(const gcre_exec* ex, double* out_perm) {
  if (!ex || (!out_perm && ex->iters)) return fail(GCRE_ERR_ARG, "null argument");
  CKS(use_device(ex));
  if (!ex->iters) return GCRE_OK;
  std::vector<float> h(ex->iters);
  CK(cudaMemcpyAsync(h.data(), ex->d_perm_max, (size_t)ex->iters * 4, cudaMemcpyDeviceToHost, ex->stream));
  CK(cudaStreamSynchronize(ex->stream));
  for (int r = 0; r < ex->iters; r++) out_perm[r] = (double)h[r];  // src/join_base.cpp:145-146
  return GCRE_OK;
}
