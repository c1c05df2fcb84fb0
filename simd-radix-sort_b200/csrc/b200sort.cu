// b200sort.cu -- host side of libb200sort.so: the C ABI of include/b200sort.h, workspace management,
// host-array staging and the launch sequence of a sort.
//
// Replaces (paths under /root/reference): the public sort<> overloads and radixRecursion,
// src/radix_sort.hpp:270-337.  There is deliberately no CPU code path in this file: if CUDA is not
// usable every entry point fails.
#include "../../include/b200sort.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdlib>
#include <utility>
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

#include <cuda_runtime.h>

#include "kernels.cuh"
#include "sweep_select.cuh"
#include "hybrid.cuh"
#include "segmented.cuh"
#include "topk.cuh"
#include "unique.cuh"

namespace b200sort {

// ------------------------------------------------------------------------------------------------
// errors, options, counters
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_last_error;
static thread_local b200sort_stats g_last_stats = {-1};  // what the last successful sort on this thread did (num < 0: none yet)
static std::atomic<uint64_t> g_launches{0};

constexpr int MGPU_MAX_CHUNKS = 8;  // multi-GPU overlapped exchange: at most this many chunks (mgpu.cuh)

// b200sort_stats::algo (include/b200sort.h), and the values of option "algo", which picks one of the first two
enum Algo { ALGO_AUTO = 0, ALGO_LSD = 1, ALGO_HYBRID = 2, ALGO_SEGMENTED = 3, ALGO_TOPK = 4, ALGO_UNIQUE = 5 };

// The tuning options of b200sort_set_option; the member initialisers are the defaults.  The process-wide values
// are read once when a sort call starts (options()) and that snapshot is passed down.
struct Options {
  int64_t algo = ALGO_AUTO, tile_cfg = -1;  // algo: auto, LSD or hybrid; tile_cfg: -1 auto, else the index of a tile geometry
  int64_t wide_tiles = 1;     // 4-byte keys, all chunks <= 4 bytes: 8192-key tiles
  int64_t nstage = 0;         // 0 auto, 1 single staging buffer, 2 double-buffered columns
  int64_t max_chunk = 16;     // largest chunk a stream is moved in (ablation: 8 = AoS records as 8-byte columns)
  int64_t tma_keys = 1;       // key tiles arrive by one TMA bulk copy per tile (cp.async.bulk + mbarrier)
  int64_t prefetch_cols = 1;  // the tile's part of the payload columns is prefetched into L2 when the tile starts
  int64_t bytewise = 1;       // lean kernels when the host knows the plan (no range reduction / shift)
  int64_t first_atomic = 1;   // first executed pass of a large sort: unstable atomicAdd ranking
  int64_t allow_skip = 1, allow_reduce = 1, allow_lshift = 1, spin_ns = 0, hist_match = 0, margin_bits = 2, probe_guess = 1;
  // the last pass orders tile-local segments + junction fix instead of the full finish; the junction kernel compares
  // fingerprints left by the last pass
  int64_t fix_in_pass = 1, junction_table = 1;
  int64_t probe_sample = 16;  // large sorts: every this-many-th tile feeds the sampled histograms
  int64_t host_plan_min_log2 = 24;  // hybrid sorts of at least 2^this records read the plan back
  int64_t host_pipeline = 1;  // host SoA arrays: sort keys + index while the payloads upload
  int64_t profile = 0;        // CUDA events around every launch of the sort (b200sort_last_profile)
  int64_t mgpu_landing = 1;  // multi-GPU: receive into a third set of arrays (saves the final copy)
  int64_t mgpu_p2p = 1;      // multi-GPU: scatter straight into peer memory (0: NCCL send/recv)
  int64_t mgpu_refine = 1;   // multi-GPU: refine heavy splitter bins / split heavy key values (0: fail with ENOMEM)
  int64_t mgpu_wide = 1;     // multi-GPU: 16-byte peer stores of element pairs
  // multi-GPU: chunked exchange overlapped with the receivers' first pass (measured: no gain, see DESIGN.md), in
  // mgpu_chunks chunks when a rank holds at least 2^mgpu_chunk_min_log2 records
  int64_t mgpu_overlap = 0, mgpu_chunks = 4, mgpu_chunk_min_log2 = 24;
  int64_t mgpu_cons_smem_kb = 0;   // overlapped first pass: shared memory requested per CTA (bounds its CTAs per SM; 0 = what it needs)
  int64_t mgpu_persist_x2 = 0;     // overlapped exchange: CTAs per SM of the looping partition kernel, times two
};
static const struct { const char *name; int64_t Options::*member; } kOptionNames[] = {
    {"algo", &Options::algo}, {"tile_cfg", &Options::tile_cfg}, {"wide_tiles", &Options::wide_tiles}, {"nstage", &Options::nstage},
    {"max_chunk", &Options::max_chunk}, {"tma_keys", &Options::tma_keys}, {"prefetch_cols", &Options::prefetch_cols},
    {"bytewise", &Options::bytewise}, {"first_atomic", &Options::first_atomic}, {"allow_skip", &Options::allow_skip},
    {"allow_reduce", &Options::allow_reduce}, {"allow_lshift", &Options::allow_lshift}, {"spin_ns", &Options::spin_ns},
    {"hist_match", &Options::hist_match}, {"margin_bits", &Options::margin_bits}, {"probe_guess", &Options::probe_guess},
    {"fix_in_pass", &Options::fix_in_pass}, {"junction_table", &Options::junction_table}, {"probe_sample", &Options::probe_sample},
    {"host_plan_min_log2", &Options::host_plan_min_log2}, {"host_pipeline", &Options::host_pipeline}, {"profile", &Options::profile},
    {"mgpu_landing", &Options::mgpu_landing}, {"mgpu_p2p", &Options::mgpu_p2p}, {"mgpu_refine", &Options::mgpu_refine},
    {"mgpu_wide", &Options::mgpu_wide}, {"mgpu_overlap", &Options::mgpu_overlap}, {"mgpu_chunks", &Options::mgpu_chunks},
    {"mgpu_chunk_min_log2", &Options::mgpu_chunk_min_log2}, {"mgpu_cons_smem_kb", &Options::mgpu_cons_smem_kb},
    {"mgpu_persist_x2", &Options::mgpu_persist_x2}};
static std::mutex g_opt_mu;
static Options g_opt;  // (under g_opt_mu) the values b200sort_set_option set

// the options a sort call runs with: the values set when it starts, brought into their valid ranges
static Options options() {
  Options o;
  { std::lock_guard<std::mutex> lk(g_opt_mu); o = g_opt; }
  o.host_plan_min_log2 = std::clamp<int64_t>(o.host_plan_min_log2, 0, 62);
  o.probe_sample = std::max<int64_t>(o.probe_sample, 1);
  o.mgpu_chunks = std::clamp<int64_t>(o.mgpu_chunks, 1, MGPU_MAX_CHUNKS);
  o.mgpu_chunk_min_log2 = std::clamp<int64_t>(o.mgpu_chunk_min_log2, 12, 40);
  o.mgpu_cons_smem_kb = std::max<int64_t>(o.mgpu_cons_smem_kb, 0);
  return o;
}

// What one host thread keeps for one device, created on first use: events and streams belong to the device they
// were created on, and two host threads sorting on one device (with their own workspaces) must not share them.
struct ThreadDeviceState {
  cudaEvent_t plan_event = nullptr;          // the plan read-back of large sorts
  std::vector<cudaEvent_t> prof_pool;        // free events of option "profile"
  cudaStream_t in = nullptr, comp = nullptr, out = nullptr;  // the pipelined host path: upload, sort, download
};
static thread_local std::map<int, ThreadDeviceState> t_dev;

// optional per-kernel timing (option "profile"): CUDA events around every launch of the last sort
enum ProfKind { PK_NONE = -1, PK_HIST = 0, PK_SCAN = 1, PK_SWEEP = 2, PK_COPYBACK = 3, PK_SEGFIX = 4, PK_OTHER = 5, PK_SEGMENT = 6, PK_SELECT = 7, PK_UNIQUE = 8 };
struct ProfEntry { int kind; cudaEvent_t e0, e1; int dev; };
static thread_local bool g_prof_on = false;  // the sort running on this thread has option "profile" set
static thread_local std::vector<ProfEntry> g_prof;

static void prof_reset() {
  for (auto &p : g_prof) { t_dev[p.dev].prof_pool.push_back(p.e0); t_dev[p.dev].prof_pool.push_back(p.e1); }
  g_prof.clear();
}
// a public call starts over and times its launches if option "profile" is set; the calls it makes inside (the
// fall-back, the sorts a segmented sort, top-k or unique runs) add to its entries
static void start_profile(const Options &o) {
  g_prof_on = o.profile != 0;
  prof_reset();
}
static cudaEvent_t prof_event(int dev) {
  auto &pool = t_dev[dev].prof_pool;
  if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
  cudaEvent_t e; cudaEventCreate(&e); return e;
}
struct ProfScope {  // (kind PK_NONE: records nothing)
  bool on; ProfEntry pe; cudaStream_t st;
  ProfScope(int kind, cudaStream_t s) : on(kind != PK_NONE && g_prof_on), st(s), kind_(kind) {
    if (on) { pe.dev = 0; cudaGetDevice(&pe.dev); pe.kind = kind; pe.e0 = prof_event(pe.dev); pe.e1 = prof_event(pe.dev); cudaEventRecord(pe.e0, st); }
  }
  ~ProfScope() {
    if (on) { cudaEventRecord(pe.e1, st); g_prof.push_back(pe); }
    static const bool dbg = getenv("B200SORT_DEBUG_SYNC") != nullptr;  // development: wait for every kernel, say which one
    if (dbg && kind_ != PK_NONE) {
      static const char *names[] = {"hist", "scan", "sweep", "copyback", "segfix", "other", "segment", "select", "unique"};
      fprintf(stderr, "[b200sort] %s launched ...", names[kind_ < 9 ? kind_ : 5]);
      const cudaError_t e = cudaStreamSynchronize(st);
      fprintf(stderr, " done (%s)\n", cudaGetErrorString(e));
    }
  }
  int kind_ = 5;
};

// Every kernel of the library is launched here: on stream st, counted (b200sort_launch_count), and timed for
// b200sort_last_profile under profile kind `kind` (PK_NONE: not timed).  Returns the launch's error.
template <typename... P, typename... A>
static cudaError_t launch(int kind, void (*k)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, A &&...args) {
  {
    ProfScope ps(kind, st);
    k<<<grid, block, smem, st>>>(std::forward<A>(args)...);
  }
  g_launches++;
  return cudaGetLastError();
}

// f(std::integral_constant<int, KB>{}) for the key width kb (1, 2, 4 or 8 bytes): one instantiation per width
template <typename F>
static auto with_kb(int kb, F &&f) {
  switch (kb) {
    case 1: return f(std::integral_constant<int, 1>{});
    case 2: return f(std::integral_constant<int, 2>{});
    case 4: return f(std::integral_constant<int, 4>{});
    default: return f(std::integral_constant<int, 8>{});
  }
}

static int fail(int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

#define CUDA_TRY(expr)                                                                              \
  do {                                                                                              \
    cudaError_t _e = (expr);                                                                        \
    if (_e != cudaSuccess)                                                                          \
      return fail(B200SORT_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

static int key_bytes_of(int kt) {
  switch (kt) {
    case B200SORT_U8: case B200SORT_I8: return 1;
    case B200SORT_U16: case B200SORT_I16: return 2;
    case B200SORT_U32: case B200SORT_I32: case B200SORT_F32: return 4;
    case B200SORT_U64: case B200SORT_I64: case B200SORT_F64: return 8;
    default: return 0;
  }
}

KeyOrder make_key_order(int key_type, bool ascending) {
  const int kb = key_bytes_of(key_type);
  const uint64_t mask = kb == 8 ? ~0ull : ((1ull << (8 * kb)) - 1);
  const uint64_t sign = 1ull << (8 * kb - 1);
  const bool is_signed = key_type == B200SORT_I8 || key_type == B200SORT_I16 || key_type == B200SORT_I32 ||
                         key_type == B200SORT_I64;
  const bool is_float = key_type == B200SORT_F32 || key_type == B200SORT_F64;
  KeyOrder ko{0, 0, 0, 0, 0};
  if (is_signed || is_float) ko.xor_const = sign;
  if (is_float) ko.neg_xor = mask ^ sign;
  if (!ascending) ko.xor_const ^= mask;
  return ko;
}

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// arrays of these sizes placed back to back at 256-byte boundaries: their offsets; *total: the bytes they span
static std::vector<size_t> back_to_back(const std::vector<size_t> &bytes, size_t *total) {
  std::vector<size_t> offs(bytes.size());
  size_t off = 0;
  for (size_t i = 0; i < bytes.size(); i++) {
    offs[i] = off;
    off = align_up(off + bytes[i], 256);
  }
  *total = off;
  return offs;
}

// ------------------------------------------------------------------------------------------------
// tile geometries of the scatter kernel
// ------------------------------------------------------------------------------------------------
static size_t sweep_smem_bytes(const TileCfg &c, uint32_t stage_bytes, int nstage = 1, bool fix = false, bool lut = false) {
  const size_t tile = (size_t)c.threads * c.ipt;
  return (size_t)nstage * tile * stage_bytes + (size_t)(c.threads / 32) * RADIX * 4 + RADIX * 8 + RADIX * 4 + 32 * 4 + tile * 3 +
         (fix ? tile : 0) +       // FIX: per-slot displacement
         (lut ? RADIX * 8 : 0);   // LUT: peer byte offsets
}

inline SweepFn sweep_fn(int kb, int cfg, const SweepSel &s) {
  switch (kb * 2 + cfg) {
    case 2: return sweep_fn_inst<1, 0>(s);
    case 3: return sweep_fn_inst<1, 1>(s);
    case 4: return sweep_fn_inst<2, 0>(s);
    case 5: return sweep_fn_inst<2, 1>(s);
    case 8: return sweep_fn_inst<4, 0>(s);
    case 9: return sweep_fn_inst<4, 1>(s);
    case 10: return sweep_fn_inst<4, 2>(s);
    case 16: return sweep_fn_inst<8, 0>(s);
    default: return sweep_fn_inst<8, 1>(s);
  }
}

// first_pass_unordered: the caller knows that this launch is the first executed pass of the sort and that its
// digit's histogram is not skewed -- the unstable ranking may be used
// smem_floor: request at least this much dynamic shared memory (bounds how many CTAs of this launch an SM holds:
// the overlapped first pass of the multi-GPU sort must leave room for the partition kernel's CTAs)
static cudaError_t launch_sweep(const Options &o, int kb, int cfg, const SweepArgs &a, int64_t n_tiles, size_t smem_optin, cudaStream_t st,
                                bool first_pass_unordered = false, size_t smem_floor = 0, int64_t grid_cap = 0) {
  bool any = false;  // a stream with 1- or 2-byte chunks in the move loop needs the ANYCHUNK instantiation
  int n_cols = 0;
  const bool soa = a.ss.streams[0].chunk_bytes * a.ss.streams[0].chunks_per_elem == (uint32_t)kb;
  for (int s = soa ? 1 : 0; s < a.ss.n_streams; s++) {
    any = any || a.ss.streams[s].chunk_bytes < 4;
    n_cols += (int)a.ss.streams[s].chunks_per_elem;
  }
  n_cols += soa ? 1 : 0;
  const TileCfg tc = kTileCfgs[cfg];
  const bool lut = a.part.key != nullptr;
  const bool fix = !lut && a.fix_cut != 0;  // (the caller only sets fix_cut where the FIX instantiation exists)
  int rank = RANK_BALLOT;
  // digits are whole bytes of the raw key when the host knows that the plan has no range reduction and no shift
  const bool bytewise = !lut && a.plan_in_args != 0 && a.arg_sub == 0 && a.arg_lshift == 0 && o.bytewise != 0;
  if (first_pass_unordered && a.plan_in_args != 0 && !lut && !fix && o.first_atomic != 0) rank = RANK_ATOMIC;
  // double-buffer the columns when there is more than one and minb CTAs still fit on an SM
  int nstage = (int)o.nstage;
  if (nstage != 1 && nstage != 2)
    nstage = (n_cols >= 2 && (sweep_smem_bytes(tc, a.stage_bytes, 2) + 1024) * tc.minb <= smem_optin + 1024) ? 2 : 1;
  if (nstage == 2 && sweep_smem_bytes(tc, a.stage_bytes, 2) > smem_optin) nstage = 1;
  if (lut || fix) nstage = 1;
  SweepSel sel{nstage, any || lut, lut, fix, rank, bytewise};
  SweepArgs a2 = a;
  // TMA bulk load of the key tile: SoA keys whose arrays (both sides of the ping-pong) are 16-byte aligned
  a2.tma_keys = (o.tma_keys != 0 && soa && (((uintptr_t)a.ss.streams[0].buf[0] | (uintptr_t)a.ss.streams[0].buf[1]) & 15) == 0 &&
                 ((size_t)tc.threads * tc.ipt * kb) % 16 == 0) ? 1u : 0u;
  SweepFn k = sweep_fn(kb, cfg, sel);
  const size_t smem = std::min(std::max(sweep_smem_bytes(tc, a.stage_bytes, nstage, fix, lut), smem_floor), smem_optin);
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  // one shared-memory carve-out for every instantiation: kernels that want different L1 / shared-memory splits
  // cannot be resident on an SM together (the overlapped exchange runs two of them side by side)
  // (only for the kernels of the overlapped exchange: a maximal carve-out leaves the other sorts 28 KB of L1,
  //  which costs them 4 % -- 38.2 vs 36.8 ms at 1e9 records).  Set on every launch: the setting outlives the sort.
  e = cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, (smem_floor != 0 || grid_cap != 0 || o.mgpu_overlap != 0)
                           ? (int)cudaSharedmemCarveoutMaxShared : (int)cudaSharedmemCarveoutDefault);
  if (e != cudaSuccess) return e;
  // L2 prefetch of the tile's part of the first column after the keys (16-byte aligned on both sides)
  a2.prefetch_cols = 0;
  {
    const int s2 = a2.tma_keys ? 1 : 0;
    if (o.prefetch_cols != 0 && s2 < a.ss.n_streams) {
      const Stream &st2 = a.ss.streams[s2];
      const size_t bytes = (size_t)tc.threads * tc.ipt * st2.chunk_bytes * st2.chunks_per_elem;
      if ((((uintptr_t)st2.buf[0] | (uintptr_t)st2.buf[1] | bytes) & 15) == 0) {
        a2.prefetch_cols = 1; a2.prefetch_bytes = (uint32_t)bytes;
        a2.prefetch_ptr[0] = st2.buf[0]; a2.prefetch_ptr[1] = st2.buf[1];
      }
    }
  }
  // (grid_cap: the partition pass of the overlapped exchange runs with fewer, looping CTAs)
  return launch(PK_SWEEP, k, (unsigned)(grid_cap > 0 ? std::min<int64_t>(n_tiles, grid_cap) : n_tiles), tc.threads, smem, st, a2);
}

constexpr int HIST_THREADS = 256;  // key-only sweeps: 256 threads x NLD x 16 B per tile, 4 CTAs per SM
constexpr int hist_nld(int kb) { return kb == 1 ? 2 : (kb >= 4 ? 8 : 4); }  // at most 32 keys per thread; 128 bytes in flight per thread for 8-byte keys

template <int KB, int NLD>
static cudaError_t launch_hist_t(const HistArgs &a, int grid, bool use_match, int probe, cudaStream_t st) {
  auto *k = probe == 2 ? minmax_kernel<KB, HIST_THREADS, NLD>
            : probe    ? (use_match ? probe_kernel<KB, HIST_THREADS, NLD, true> : probe_kernel<KB, HIST_THREADS, NLD, false>)
                       : (use_match ? hist_kernel<KB, HIST_THREADS, NLD, true> : hist_kernel<KB, HIST_THREADS, NLD, false>);
  return launch(PK_HIST, k, grid, HIST_THREADS, 0, st, a);
}

// keys per tile of the key-only sweeps over this key array
static int64_t hist_tile_keys(int kb, const void *keys, uint32_t stride) {
  // (8-byte keys in a dense, 16-byte aligned array: eight 16-byte vectors in flight per thread -- probe 1.66 ->
  //  1.33 ms at 1e9 keys; records with the key inside are read one key per load, where more per thread is slower)
  const bool dense = stride == (uint32_t)kb && (((uintptr_t)keys) & 15) == 0;
  const int nld = (kb == 8 && !dense) ? 4 : hist_nld(kb);  // (4-byte keys: 8 vectors = 32 keys per thread either way)
  return (int64_t)HIST_THREADS * nld * (16 / kb);
}

static cudaError_t launch_hist(const Options &o, int kb, const HistArgs &a, int sm_count, int probe, cudaStream_t st) {
  const int64_t tile_keys = hist_tile_keys(kb, a.keys, a.stride);
  const int64_t tiles = (a.n + tile_keys - 1) / tile_keys;
  const int grid = (int)std::min<int64_t>(tiles, (int64_t)sm_count * 8);
  const bool m = o.hist_match != 0;
  return with_kb(kb, [&](auto K) {
    constexpr int KB = decltype(K)::value;
    if constexpr (KB == 8)
      if (tile_keys == (int64_t)HIST_THREADS * 4 * 2) return launch_hist_t<8, 4>(a, grid, m, probe, st);
    return launch_hist_t<KB, hist_nld(KB)>(a, grid, m, probe, st);
  });
}

// ------------------------------------------------------------------------------------------------
// per-device state: device properties, the library-owned caches and their guard
// ------------------------------------------------------------------------------------------------
struct DevInfo { int sm_count = 0; size_t smem_optin = 0; bool ok = false; };
struct CacheEntry { void *ptr = nullptr; size_t bytes = 0; uint64_t gen = 0; };  // gen: bumped by every (re)allocation

// What the library keeps for one device, process-wide.  The caches (the sort's workspace, the staging of host
// arrays) are one allocation each, and the sorts that use them are serialised, so that two host threads, or two
// streams, never have kernels in flight on the same scratch memory.  Callers who want concurrent sorts of device
// arrays pass their own workspace.  Rule: a device's cache entries are read and written only while its guard
// (`mu`, taken by CacheGuard) is held.
struct DeviceState {
  DevInfo info;                    // filled once, on first use (under g_mu)
  std::recursive_mutex mu;         // held from acquiring a cache until the sort's work is queued
  cudaEvent_t last_use = nullptr;  // recorded when the guard is released; the next user's stream waits for it
  CacheEntry workspace, stage;
};
static std::mutex g_mu;                    // guards the map and every record's `info`; never held while waiting for `mu`
static std::map<int, DeviceState> g_devs;  // (std::map nodes are stable: a reference to a record stays valid)

static DeviceState &device_state(int dev) {
  std::lock_guard<std::mutex> lk(g_mu);
  return g_devs[dev];
}

// holds a device's DeviceState::mu from acquire() until it is destroyed, which records `last_use` on the stream
struct CacheGuard {
  DeviceState *state = nullptr;
  cudaStream_t stream = nullptr;
  DeviceState &acquire(int dev, cudaStream_t s) {
    state = &device_state(dev);
    stream = s;
    state->mu.lock();
    if (state->last_use == nullptr) cudaEventCreateWithFlags(&state->last_use, cudaEventDisableTiming);
    else cudaStreamWaitEvent(stream, state->last_use, 0);
    return *state;
  }
  ~CacheGuard() {
    if (!state) return;
    cudaEventRecord(state->last_use, stream);
    state->mu.unlock();
  }
};

static int dev_info(int dev, DevInfo *out) {
  std::lock_guard<std::mutex> lk(g_mu);
  DevInfo &d = g_devs[dev].info;
  if (!d.ok) {
    int v = 0;
    CUDA_TRY(cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev));
    d.sm_count = v;
    CUDA_TRY(cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    d.smem_optin = (size_t)v;
    d.ok = true;
  }
  *out = d;
  return 0;
}

// the buffer of cache entry `c` of the current device (its guard held), grown to at least `bytes`; `what` names it
static int cached_buffer(CacheEntry &c, size_t bytes, const char *what, void **out) {
  if (c.bytes < bytes) {
    if (c.ptr) {
      CUDA_TRY(cudaDeviceSynchronize());
      CUDA_TRY(cudaFree(c.ptr));
      c.ptr = nullptr;
      c.bytes = 0;
    }
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) {
      cudaGetLastError();
      return fail(B200SORT_ENOMEM, "cudaMalloc of %zu %s bytes failed: %s", bytes, what, cudaGetErrorString(e));
    }
    c.ptr = p;
    c.bytes = bytes;
    c.gen++;
  }
  *out = c.ptr;
  return 0;
}

// ------------------------------------------------------------------------------------------------
// job description
// ------------------------------------------------------------------------------------------------
struct StreamDesc { void *ptr; uint32_t elem_bytes; };

struct Layout {
  size_t shadow_off[MAX_STREAMS];
  size_t land_off[MAX_STREAMS];
  size_t ctrl_off, ctrl_bytes;       // zeroed at the start of every sort
  size_t ghist_off, ghist2_off, probe_off, tilectr_off, plan_off, binbase_off, lookback_off, hyb_off, jtable_off, flags_off;
  size_t total;
  int64_t n_tiles;
};

static int pick_tile_cfg(const Options &o, int kb, uint32_t stage_bytes, size_t smem_optin, int64_t n) {
  int cfg = (int)o.tile_cfg;
  const bool automatic = cfg < 0 || cfg >= kNumTileCfgs;
  // (wide tiles only where there are plenty of them: 10^6 records are 123 wide tiles for 148 SMs -- 0.18 vs 0.13 ms)
  if (automatic) cfg = (kb == 4 && stage_bytes <= 4 && n >= ((int64_t)1 << 24) && o.wide_tiles != 0) ? kWideTileCfg : kDefaultTileCfg;
  if (cfg == kWideTileCfg && (kb != 4 || stage_bytes > 4)) cfg = kDefaultTileCfg;  // (only instantiated for that shape)
  // fall back to the smaller tile if the staging buffer would not fit
  if (sweep_smem_bytes(kTileCfgs[cfg], stage_bytes) > smem_optin) cfg = 1;
  return cfg;
}

static void make_layout(const std::vector<StreamDesc> &streams, int64_t n, int tile, Layout *L, bool landing = false) {
  size_t off = 0;
  for (size_t s = 0; s < streams.size(); s++) {
    L->shadow_off[s] = off;
    off = align_up(off + (size_t)n * streams[s].elem_bytes, 256);
  }
  L->n_tiles = (n + tile - 1) / tile;
  // hybrid path tiles may be smaller than the sweep tiles; size the look-back for the smallest tile used
  L->ctrl_off = off;
  L->ghist_off = off;               off += (size_t)8 * RADIX * 8;   // sampled histograms (probe)
  L->ghist2_off = off;              off += (size_t)8 * RADIX * 8;   // exact histograms, one digit position at a time
  L->probe_off = off;               off += 64;
  L->tilectr_off = off;             off += MAX_PASSES * 4;
  L->plan_off = off;                off = align_up(off + sizeof(Plan), 256);
  L->hyb_off = off;                 off = align_up(off + sizeof(HybridCtrl), 256);
  L->lookback_off = off;            off += (size_t)L->n_tiles * RADIX * 8;
  L->ctrl_bytes = off - L->ctrl_off;
  L->binbase_off = off;             off += (size_t)MAX_PASSES * RADIX * 8;
  L->jtable_off = off;              off += (size_t)L->n_tiles * RADIX * 8;   // FIX pass -> junction_fix_kernel
  off = align_up(off, 256);
  L->flags_off = off;               off += 4096;  // multi-GPU: arrival flags written by the peers (never zeroed: epochs)
  // multi-GPU: a third copy of every stream, where the peers deliver this rank's records (see mgpu.cuh)
  for (size_t s = 0; s < streams.size(); s++) {
    L->land_off[s] = off;
    if (landing) off = align_up(off + (size_t)n * streams[s].elem_bytes, 256);
  }
  L->total = align_up(off, 256);
}

// the streams of a call of this shape, without addresses: SoA keys of kb bytes and n_payloads payloads of the given
// sizes, or (record_bytes != 0) records
static std::vector<StreamDesc> streams_of_shape(int kb, int n_payloads, const uint32_t *sizes, uint32_t record_bytes) {
  if (record_bytes) return {{nullptr, record_bytes}};
  std::vector<StreamDesc> streams = {{nullptr, (uint32_t)kb}};
  for (int p = 0; p < n_payloads; p++) streams.push_back({nullptr, sizes[p]});
  return streams;
}

// the workspace a sort_device of these streams needs, whatever tile geometry it picks
static size_t sort_workspace_bytes(const std::vector<StreamDesc> &streams, int64_t n) {
  Layout L;
  // the smallest tile any geometry uses bounds the look-back size from above
  make_layout(streams, std::max<int64_t>(n, 1), HYB_MIN_TILE, &L);
  return L.total;
}

// What the work on device arrays of the current device (DevSort, sort_segmented_device, topk_device, unique_device)
// starts with: open() finds the device and its properties; workspace() takes the caller's workspace, or the library's
// cached one through `guard`, which is held until the work is queued.
struct DevSetup {
  uint64_t launches_before = g_launches.load();  // the launch counter when the function started
  int dev = 0;
  DevInfo di;
  CacheGuard guard;
  unsigned char *ws = nullptr;

  int open() {
    CUDA_TRY(cudaGetDevice(&dev));
    return dev_info(dev, &di);
  }
  // ws: `bytes` of workspace, from `caller_ws` (NULL for none) of `caller_bytes` or from the cache
  int workspace(cudaStream_t stream, void *caller_ws, size_t caller_bytes, size_t bytes) {
    if (caller_ws == nullptr) {
      void *p = nullptr;
      if (int rc = cached_buffer(guard.acquire(dev, stream).workspace, bytes, "workspace", &p)) return rc;
      ws = (unsigned char *)p;
      return 0;
    }
    if (caller_bytes < bytes) return fail(B200SORT_ENOMEM, "workspace of %zu bytes given, %zu needed", caller_bytes, bytes);
    if (((uintptr_t)caller_ws % 256) != 0) return fail(B200SORT_EINVAL, "workspace must be 256-byte aligned");
    ws = (unsigned char *)caller_ws;
    return 0;
  }
  // the stats fields every call reports: what it worked on, and the kernels launched since the function started
  b200sort_stats stats(int64_t n, const std::vector<StreamDesc> &streams, int kb, int algo) const {
    b200sort_stats s{};
    s.num = n;
    for (const StreamDesc &d : streams) s.record_bytes += d.elem_bytes;
    s.key_bytes = (uint32_t)kb;
    s.algo = (uint32_t)algo;
    s.kernel_launches = (uint32_t)(g_launches.load() - launches_before);
    return s;
  }
};

// The arrays as the streams the scatter kernel moves: each one in chunks of the largest power of two <= max_chunk
// (and <= 16) dividing both its address and its element size; the key stream (keys or records) in chunks no narrower
// than the key, whatever max_chunk says.  Returns the staging buffer's element size: the largest chunk, at least the key.
static uint32_t make_stream_set(const std::vector<StreamDesc> &streams, int kb, uint32_t max_chunk, StreamSet *ss) {
  uint32_t stage_bytes = (uint32_t)kb;
  *ss = StreamSet{};
  ss->n_streams = (int)streams.size();
  for (size_t s = 0; s < streams.size(); s++) {
    uint32_t c = 16;
    while (c > 1 && ((streams[s].elem_bytes % c) != 0 || ((uintptr_t)streams[s].ptr % c) != 0)) c >>= 1;
    if (c > max_chunk) c = std::max(max_chunk, s == 0 ? (uint32_t)kb : 1u);
    ss->streams[s].chunk_bytes = c;
    ss->streams[s].chunks_per_elem = streams[s].elem_bytes / c;
    ss->streams[s].buf[0] = (unsigned char *)streams[s].ptr;
    stage_bytes = std::max(stage_bytes, c);
  }
  return stage_bytes;
}

// Sort arrays that are all in device memory.  streams[0] carries the key at offset 0.
struct DevSortOpts {
  int start_sel = 0;         // 1: the input lies in the workspace's shadow arrays, the result still goes to the caller's
  int64_t layout_n = 0;      // lay the workspace out for this many records (>= n)
  int hint_lead_bits = 0;    // leading bits the caller expects all keys to agree on (steers the probe's guess)
  bool layout_landing = false;  // the layout has landing arrays (make_layout(..., landing))
  bool landing_input = false;   // the input lies in the landing arrays: the first executed pass reads it from
                                // there (landing -> shadow -> caller -> ...), so that an even number of passes
                                // ends in the caller's arrays without a copy
  // Multi-GPU sort with the exchange overlapped (mgpu.cuh): the plan is fixed by the caller (forced_plan), the
  // control block has been cleared by the caller, and the FIRST executed pass has already been run by the
  // caller (landing arrays -> shadow arrays, its successor's digit counted into the exact histograms).
  bool forced = false;
  uint32_t forced_lshift = 0, forced_cut = 0;
  // Partial-sort mode (B200SORT_CMP_NONE with a threshold >= CMP_NONE_MIN_THRESH): the segments below the plan's
  // cut need not be ordered as long as none has more than this many keys (0 = full sort)
  int64_t cmp_none_thresh = 0;
};
constexpr int64_t CMP_NONE_MIN_THRESH = 8;  // below it nearly every sort would need the finish anyway: full sort

// The plan of the overlapped multi-GPU exchange's local sort: the hybrid sweep of digit positions cut .. kb-1 of
// the key shifted left by lshift, in LSD order, without range reduction; the first of them is run by the caller.
static Plan forced_plan(int kb, uint32_t cut, uint32_t lshift) {
  Plan p{};
  uint32_t sel = 0, prev = 0;
  bool any_prev = false;
  for (int d = 0; d < kb; d++) {
    p.skip[d] = (uint32_t)d < cut ? 1u : 0u;
    p.src_sel[d] = sel;
    if (!p.skip[d]) {
      sel ^= 1u;
      p.n_exec++;
      if (!any_prev) p.first_exec_p1 = (uint32_t)d + 1; else p.next_exec_p1[prev] = (uint32_t)d + 1;
      prev = (uint32_t)d;
      any_prev = true;
    }
  }
  p.final_sel = sel;
  p.cut_digit = cut;
  p.lshift = lshift;
  p.hist_done = 1;
  return p;
}

// One sort of device arrays, phase by phase: one histogram sweep over all digit positions, the bucket-offset scan
// (+ pass plan), one scatter pass per digit position, the segment finish, the copy-back.
struct DevSort : DevSetup {
  const Options &o;
  const int key_type;
  const bool ascending;
  const int64_t n;
  const std::vector<StreamDesc> &streams;
  const cudaStream_t stream;
  void *const caller_workspace;
  const size_t workspace_bytes;
  const DevSortOpts &xo;
  const int kb = key_bytes_of(key_type);
  // set-up
  int cfg = 0, tile = 0, algo = ALGO_AUTO;
  bool hybrid = false;
  StreamSet ss{};
  uint32_t stage_bytes = 0;
  Layout L;
  Plan *plan = nullptr;  // (device)
  HybridCtrl *ctrl = nullptr;
  KeyOrder ko{};
  // plan
  Plan hplan{};
  bool have_plan = false;    // the host knows the plan (hplan): launches only what executes
  bool landing = false;      // the first executed pass reads the landing arrays (ss_in)
  StreamSet ss_in{};         // what the key sweeps and the first executed pass read
  uint32_t hist_sweeps = 1;  // probe (+ exact min/max) (+ exact histogram of the first pass)
  // passes, finish
  bool partial = false;      // partial-sort mode: no ordering of the final segments, only a check of their lengths
  int last_pass = -1;        // the last pass orders the tile-local final segments (junction fix follows)
  bool fix_flow = false;     // the finish is gated on the device by ctrl->flags[1]
  bool finish_ran = false;

  // set-up: streams, tile geometry, workspace layout, workspace (and the cache guard if it is the library's)
  int setup() {
    if (int rc = open()) return rc;
    stage_bytes = make_stream_set(streams, kb, (uint32_t)o.max_chunk, &ss);
    if (streams[0].elem_bytes != (uint32_t)kb && ((uintptr_t)streams[0].ptr % kb) != 0)
      return fail(B200SORT_EINVAL, "record array is not aligned to its key type");
    if (((uintptr_t)streams[0].ptr % kb) != 0) return fail(B200SORT_EINVAL, "key array is not aligned to its key type");

    cfg = pick_tile_cfg(o, kb, stage_bytes, di.smem_optin, n);
    const TileCfg tc = kTileCfgs[cfg];
    tile = tc.threads * tc.ipt;
    const size_t smem = sweep_smem_bytes(tc, stage_bytes);
    if (smem > di.smem_optin) return fail(B200SORT_ECUDA, "device offers %zu B of shared memory, %zu needed", di.smem_optin, smem);

    make_layout(streams, std::max(n, xo.layout_n), std::min(tile, HYB_MIN_TILE), &L, xo.layout_landing);
    if (int rc = workspace(stream, caller_workspace, workspace_bytes, L.total)) return rc;
    for (size_t s = 0; s < streams.size(); s++) ss.streams[s].buf[1] = ws + L.shadow_off[s];
    plan = (Plan *)(ws + L.plan_off);
    ctrl = (HybridCtrl *)(ws + L.hyb_off);
    if (!xo.forced) CUDA_TRY(cudaMemsetAsync(ws + L.ctrl_off, 0, L.ctrl_bytes, stream));

    ko = make_key_order(key_type, ascending);
    algo = xo.forced ? ALGO_HYBRID : (int)o.algo;
    if (algo == ALGO_AUTO) algo = (kb == 8 && n >= HYB_MIN_N) ? ALGO_HYBRID : ALGO_LSD;
    if (algo == ALGO_HYBRID && kb != 8) algo = ALGO_LSD;
    hybrid = algo == ALGO_HYBRID;
    return 0;
  }

  // input in the landing arrays, delivered into the caller's arrays by a copy
  int deliver_landing() {
    for (size_t s = 0; s < streams.size(); s++)
      CUDA_TRY(cudaMemcpyAsync(streams[s].ptr, ws + L.land_off[s], (size_t)n * streams[s].elem_bytes, cudaMemcpyDeviceToDevice, stream));
    return 0;
  }

  int read_plan(cudaEvent_t ev) {
    CUDA_TRY(cudaMemcpyAsync(&hplan, plan, sizeof hplan, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaEventRecord(ev, stream));
    CUDA_TRY(cudaEventSynchronize(ev));
    return 0;
  }

  // plan: the probe (sampled histograms + the exact histogram of the guessed first digit) and the scan that makes
  // the plan.  Large sorts read the plan back (small D2H, one host wait) and launch only what executes: the exact
  // min/max sweep and a second planning step if asked for, the histogram kernel unless the probe's guess was
  // right, the passes that are not skipped.  Smaller sorts launch everything; what is not needed returns at once.
  int make_plan() {
    uint64_t *ghist = (uint64_t *)(ws + L.ghist_off), *ghist_exact = (uint64_t *)(ws + L.ghist2_off);
    const bool big = xo.forced || n >= (int64_t)1 << o.host_plan_min_log2;
    // Input in the landing arrays (multi-GPU): only the large hybrid flow knows on the host which pass runs
    // first; everything else simply starts with a copy into the caller's arrays.
    landing = xo.landing_input;
    if (landing && !big) {
      if (int rc = deliver_landing()) return rc;
      landing = false;
    }
    ss_in = ss;
    if (landing)
      for (size_t s = 0; s < streams.size(); s++) ss_in.streams[s].buf[0] = ws + L.land_off[s];
    HistArgs ha{};
    ha.keys = ss_in.streams[0].buf[xo.start_sel];
    ha.stride = streams[0].elem_bytes;
    ha.n = n; ha.ko = ko; ha.digit_mask = (1u << kb) - 1; ha.ghist = ghist; ha.probe = (ProbeOut *)(ws + L.probe_off);
    // entropies from one key per thread of every 16th tile (option probe_sample) once there are plenty of tiles
    const bool sparse = (n / hist_tile_keys(kb, ha.keys, ha.stride)) >= 8192;
    ha.sample = sparse ? (uint32_t)o.probe_sample : 1;
    ha.sample_one = sparse ? 1 : 0;
    // Large sorts leave the exact key range to a sweep of its own that only runs when the sampled range says
    // range reduction may pay; the others get it from the probe.
    ha.with_minmax = big ? 0 : 1;
    // The digit position the first pass will sweep if the keys are (close to) uniformly distributed: the
    // probe counts it exactly, and if the plan comes out that way hist_kernel is not needed.
    // (digit-by-digit path: the least significant digit, guess = 0, is the first pass unless it is constant)
    uint32_t guess = 0;
    if (hybrid) {
      // hint_lead_bits: leading bits the caller expects all keys to agree on (a shard of the multi-GPU sort)
      const double need = std::log2((double)n) + (double)o.margin_bits;
      const int cut = 8 - xo.hint_lead_bits / 8 - (int)std::ceil(need / 8.0);
      if (cut >= 2) {
        guess = (uint32_t)cut;
        ha.guess_lshift = o.allow_lshift != 0 ? (uint32_t)(xo.hint_lead_bits & 7) : 0u;
      }
    }
    ha.guess_p1 = o.probe_guess != 0 ? guess + 1 : 0;
    ha.ghist_exact = ghist_exact;
    if (xo.forced) {  // the caller's plan (its probe, scan and first pass ran overlapped with the exchange)
      hist_sweeps = 0;
      hplan = forced_plan(kb, xo.forced_cut, xo.forced_lshift);
      CUDA_TRY(cudaMemcpyAsync(plan, &hplan, sizeof hplan, cudaMemcpyHostToDevice, stream));
      have_plan = true;
      return 0;
    }
    CUDA_TRY(launch_hist(o, kb, ha, di.sm_count, /*probe=*/1, stream));

    ScanArgs sa{};
    sa.ghist = ghist; sa.probe = ha.probe; sa.plan = plan; sa.n = n; sa.n_passes = kb;
    sa.allow_skip = (int)o.allow_skip;
    sa.hybrid = hybrid ? 1 : 0;
    sa.allow_reduce = (int)o.allow_reduce;
    sa.margin_bits = (float)o.margin_bits;
    sa.have_minmax = (int)ha.with_minmax;
    sa.allow_lshift = (int)o.allow_lshift;
    sa.start_sel = (uint32_t)xo.start_sel;
    sa.guess_p1 = ha.guess_p1; sa.guess_lshift = ha.guess_lshift; sa.ghist_exact = ghist_exact;
    CUDA_TRY(launch(PK_SCAN, scan_kernel, 1, RADIX, 0, stream, sa));

    HistArgs hb = ha;  // exact histogram of the first executed pass only; every pass counts its successor's digit
    hb.ghist = ghist_exact; hb.plan = plan; hb.probe = nullptr;
    if (big) {
      cudaEvent_t &ev = t_dev[dev].plan_event;
      if (ev == nullptr && cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) {
        ev = nullptr;
        return fail(B200SORT_ECUDA, "cudaEventCreate failed on device %d", dev);
      }
      if (int rc = read_plan(ev)) return rc;
      if (hplan.want_minmax) {
        CUDA_TRY(launch_hist(o, kb, ha, di.sm_count, /*minmax=*/2, stream));
        hist_sweeps++;
        sa.have_minmax = 1;
        CUDA_TRY(launch(PK_SCAN, scan_kernel, 1, RADIX, 0, stream, sa));
        if (int rc = read_plan(ev)) return rc;
      }
      have_plan = true;
      if (hplan.hist_done) return 0;
    }
    CUDA_TRY(launch_hist(o, kb, hb, di.sm_count, /*probe=*/0, stream));
    hist_sweeps++;
    return 0;
  }

  // passes: one scatter pass per digit position (skipped ones return at once, or are not launched if the host
  // knows the plan).  With the plan on the host, an 8-byte-key SoA sort lets the LAST pass order the final
  // segments each tile holds and repairs the tile-straddling ones with junction_fix_kernel (see finish).
  int run_passes() {
    const bool soa = streams[0].elem_bytes == (uint32_t)kb;
    partial = have_plan && hplan.cut_digit != 0 && xo.cmp_none_thresh >= CMP_NONE_MIN_THRESH;
    const bool use_fix = !partial && have_plan && hplan.cut_digit != 0 && (soa || ss.streams[0].chunk_bytes >= (uint32_t)kb) &&
                         cfg == kDefaultTileCfg && o.fix_in_pass != 0;
    if (landing && hplan.n_exec == 0)  // nothing will move the records: deliver them
      if (int rc = deliver_landing()) return rc;
    bool first_exec = true;
    for (int p = 0; p < kb; p++) {
      if (have_plan && hplan.skip[p]) continue;
      const bool was_first = first_exec;
      first_exec = false;
      if (xo.forced && was_first) continue;  // run by the caller, overlapped with the exchange
      SweepArgs wa{};
      wa.ss = (landing && was_first) ? ss_in : ss; wa.n = n;
      wa.ko = ko; wa.pass = p; wa.shift = p * RADIX_BITS;
      wa.bin_base = nullptr; wa.ghist = (uint64_t *)(ws + L.ghist2_off);
      wa.lookback = (uint64_t *)(ws + L.lookback_off); wa.tile_counter = (uint32_t *)(ws + L.tilectr_off); wa.plan = plan;
      wa.tag = (uint32_t)(p + 1); wa.stage_bytes = stage_bytes; wa.spin_ns = (uint32_t)o.spin_ns;
      if (have_plan) {
        wa.plan_in_args = 1; wa.arg_sel = hplan.src_sel[p]; wa.arg_next_p1 = hplan.next_exec_p1[p];
        wa.arg_next_skewed = hplan.next_exec_p1[p] ? hplan.skewed[hplan.next_exec_p1[p] - 1] : 0; wa.arg_sub = hplan.sub; wa.arg_lshift = hplan.lshift;
        if (use_fix && hplan.next_exec_p1[p] == 0) { wa.fix_cut = hplan.cut_digit; wa.fix_flag = &ctrl->flags[1]; wa.jtable = (uint64_t *)(ws + L.jtable_off); last_pass = p; }
      }
      // the first executed pass may rank its keys in any order (nothing has been established yet)
      const bool unordered = have_plan && was_first && hplan.skewed[p] == 0;
      CUDA_TRY(launch_sweep(o, kb, cfg, wa, (n + tile - 1) / tile, di.smem_optin, stream, unordered));
    }
    return 0;
  }

  // the full segment finish (gate: it only runs if *gate != 0), which delivers into the caller's arrays
  cudaError_t launch_segfix(const uint32_t *gate) {
    SegfixArgs fa{};
    fa.ss = ss; fa.n = n; fa.ko = ko; fa.plan = plan; fa.ctrl = ctrl; fa.gate = gate;
    if (have_plan) { fa.plan_in_args = 1; fa.arg_cut = hplan.cut_digit; fa.arg_sel = hplan.final_sel; fa.arg_sub = hplan.sub; fa.arg_lshift = hplan.lshift; }
    bool any = false;
    for (int s = 0; s < ss.n_streams; s++) any = any || ss.streams[s].chunk_bytes < 4;
    const unsigned grid = (unsigned)std::min<int64_t>((n + SF_FT - 1) / SF_FT, (int64_t)di.sm_count * 16);
    return launch(PK_SEGFIX, any ? segfix_kernel<8, true> : segfix_kernel<8, false>, grid, SF_THREADS, 0, stream, fa);
  }

  // the result out of the shadow arrays if it ended there (force: whatever the plan says; skip_if: not if *skip_if)
  cudaError_t launch_copyback(bool force, const uint32_t *skip_if) {
    CopyBackArgs ca{};
    ca.ss = ss; ca.n = n; ca.plan = plan; ca.force = force ? 1 : 0; ca.skip_if = skip_if;
    return launch(PK_COPYBACK, copyback_kernel, di.sm_count * 8, 256, 0, stream, ca);
  }

  // finish: the final segments ordered, or checked in partial-sort mode, and the result in the caller's arrays
  int finish() {
    const uint32_t *flag = &ctrl->flags[1];
    if (last_pass >= 0) {
      const int64_t n_tiles = (n + tile - 1) / tile;
      JunctionArgs ja{};
      ja.ss = ss; ja.n = n; ja.ko = ko; ja.ko.sub = hplan.sub; ja.ko.lshift = hplan.lshift; ja.lookback = (uint64_t *)(ws + L.lookback_off);
      ja.n_tiles = n_tiles; ja.tag = (uint32_t)(last_pass + 1); ja.cut = hplan.cut_digit; ja.sel = hplan.final_sel; ja.flag = &ctrl->flags[1];
      ja.jtable = o.junction_table != 0 ? (const uint64_t *)(ws + L.jtable_off) : nullptr;
      CUDA_TRY(launch(PK_SEGFIX, junction_fix_kernel<8>, (unsigned)((n_tiles * RADIX + 255) / 256), 256, 0, stream, ja));
    } else if (partial) {
      PartialCheckArgs pa{};
      pa.ss = ss; pa.n = n; pa.ko = ko; pa.ko.sub = hplan.sub; pa.ko.lshift = hplan.lshift; pa.cut = hplan.cut_digit; pa.sel = hplan.final_sel;
      pa.thresh = xo.cmp_none_thresh; pa.flag = &ctrl->flags[1];
      CUDA_TRY(launch(PK_SEGFIX, partial_check_kernel<8>, di.sm_count * 8, 256, 0, stream, pa));
    } else {
      if (hybrid && !(have_plan && hplan.cut_digit == 0)) {
        CUDA_TRY(launch_segfix(nullptr));
        finish_ran = true;
      }
      CUDA_TRY(launch_copyback(false, nullptr));
      return 0;
    }
    // Both possible continuations are launched; which one does anything is decided on the device by the flag the
    // last pass / the junction kernel / the partial check raise when they meet a run that is too long for them:
    // the full segment finish repairs everything (and delivers the result into the caller's arrays), else the
    // result is copied out of the shadow if it ended there.  No host round trip in between.
    CUDA_TRY(launch_segfix(flag));
    if (hplan.final_sel == 1) CUDA_TRY(launch_copyback(true, flag));
    fix_flow = true;
    return 0;
  }

  // statistics of what ran.  The hybrid path reads its plan (made on the device) and its flags back: its one
  // host synchronisation.  *fall_back: a long bucket with distinct keys is left for the digit-by-digit path.
  int statistics(b200sort_stats *stt, bool *fall_back) {
    HybridCtrl hctrl{};
    if (hybrid) {
      if (!have_plan) CUDA_TRY(cudaMemcpyAsync(&hplan, plan, sizeof hplan, cudaMemcpyDeviceToHost, stream));
      CUDA_TRY(cudaMemcpyAsync(&hctrl, ctrl, sizeof hctrl, cudaMemcpyDeviceToHost, stream));
      CUDA_TRY(cudaStreamSynchronize(stream));
      if (fix_flow) finish_ran = hctrl.flags[1] != 0;
    }
    *stt = stats(n, streams, kb, algo);
    stt->hist_sweeps = hist_sweeps;
    stt->passes_planned = (have_plan || hybrid) ? hplan.n_exec : (uint32_t)kb;  // (otherwise every pass is launched)
    if (hybrid) {
      // (the flow that plans on the device launches the finish whatever the plan is; without a cut it returns at once)
      stt->segfix_passes = (finish_ran && hplan.cut_digit != 0) ? 1 : 0;
      stt->cut_digit = hplan.cut_digit;
      memcpy(&stt->segfix_moved, &hctrl.flags[2], 8);
    }
    stt->algorithmic_bytes = (uint64_t)hist_sweeps * (uint64_t)n * kb + (uint64_t)(stt->passes_planned + stt->segfix_passes) * 2ull * (uint64_t)n * stt->record_bytes;
    *fall_back = hybrid && hctrl.flags[0] != 0;
    return 0;
  }

  // fall-back: finish with the plain digit-by-digit path (the array is a permutation of the input, already ordered
  // by its top digits)
  int fall_back(b200sort_stats *stt) {
    Options lsd = o; lsd.algo = ALGO_LSD;  // (whatever option "algo" says)
    DevSortOpts fo;
    fo.layout_n = xo.layout_n; fo.layout_landing = xo.layout_landing;
    b200sort_stats s2;
    if (int rc = DevSort{{}, lsd, key_type, ascending, n, streams, stream, caller_workspace, workspace_bytes, fo}.run(&s2)) return rc;
    stt->fell_back = 1;
    stt->passes_planned += s2.passes_planned;
    stt->hist_sweeps += s2.hist_sweeps;
    stt->algorithmic_bytes += s2.algorithmic_bytes;
    stt->kernel_launches += s2.kernel_launches;
    return 0;
  }

  // the sort, phase by phase; *stats: what ran (written when the sort succeeds)
  int run(b200sort_stats *stats) {
    if (int rc = setup()) return rc;
    if (int rc = make_plan()) return rc;
    if (int rc = run_passes()) return rc;
    if (int rc = finish()) return rc;
    b200sort_stats stt;
    bool fell_back = false;
    if (int rc = statistics(&stt, &fell_back)) return rc;
    if (fell_back)
      if (int rc = fall_back(&stt)) return rc;
    *stats = stt;
    return B200SORT_OK;
  }
};

static int sort_device(const Options &o, int key_type, bool ascending, int64_t n, const std::vector<StreamDesc> &streams,
                       cudaStream_t stream, void *workspace, size_t workspace_bytes, const DevSortOpts &xo, b200sort_stats *stats) {
  return DevSort{{}, o, key_type, ascending, n, streams, stream, workspace, workspace_bytes, xo}.run(stats);
}

// ------------------------------------------------------------------------------------------------
// host/device dispatch
// ------------------------------------------------------------------------------------------------
enum Side { SIDE_HOST = 0, SIDE_DEVICE = 1 };

// makes `dev` the current device for the duration of a call (device arrays are sorted on the device that owns
// them, whatever the caller's current device is)
struct DeviceScope {
  int prev = -1;
  bool switched = false;
  int enter(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess || (prev != dev && cudaSetDevice(dev) != cudaSuccess)) {
      cudaGetLastError();
      return fail(B200SORT_ECUDA, "cannot make device %d current", dev);
    }
    switched = prev != dev;
    return 0;
  }
  ~DeviceScope() { if (switched) cudaSetDevice(prev); }
};

static int side_of(const void *p, Side *out, int *dev_out) {
  cudaPointerAttributes at{};
  cudaError_t e = cudaPointerGetAttributes(&at, p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(B200SORT_ECUDA, "cudaPointerGetAttributes failed: %s (no usable CUDA device? there is no CPU fallback)",
                cudaGetErrorString(e));
  }
  *out = (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged) ? SIDE_DEVICE : SIDE_HOST;
  *dev_out = at.device;
  return 0;
}

// Where the arrays of one call live, each pointer asked once: all in host memory, or all on one device (*dev).
// offsets (NULL for none): a segmented sort's, which must live where the arrays do.  device_only (NULL for none): the
// name of a call that takes device arrays only, for the error that refuses host arrays.  Fails without a device.
static int place_arrays(const std::vector<StreamDesc> &arrays, const int64_t *offsets, const char *device_only, Side *side, int *dev) {
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(B200SORT_ECUDA, "no CUDA device available (%s); libb200sort has no CPU fallback",
                e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
  }
  std::vector<Side> sd(arrays.size() + (offsets != nullptr ? 1 : 0));  // (the offsets last)
  std::vector<int> dv(sd.size());
  for (size_t i = 0; i < sd.size(); i++)
    if (int rc = side_of(i < arrays.size() ? arrays[i].ptr : offsets, &sd[i], &dv[i])) return rc;
  if (device_only != nullptr && std::count(sd.begin(), sd.end(), SIDE_HOST) != 0)
    return fail(B200SORT_EUNSUPPORTED, "%s takes device arrays only; an array is in host memory", device_only);
  *side = sd[0];
  *dev = dv[0];
  for (size_t i = 1; i < arrays.size(); i++) {
    if (sd[i] != *side) return fail(B200SORT_EINVAL, "arrays must be all in host memory or all in device memory");
    if (sd[i] == SIDE_DEVICE && dv[i] != *dev) return fail(B200SORT_EINVAL, "device arrays live on different devices (%d and %d)", *dev, dv[i]);
  }
  if (offsets != nullptr && (sd.back() != *side || (*side == SIDE_DEVICE && dv.back() != *dev)))
    return fail(B200SORT_EINVAL, "offsets must live where the arrays do (host memory, or the arrays' device)");
  return 0;
}

// What every public single-GPU call does once its arguments have passed their checks: it takes the options snapshot,
// places its arrays (place_arrays), runs on their device (host arrays: on the current one) and starts its profile.
// done(rc) makes `stats` the call's statistics (b200sort_last_stats) when the call succeeded.
struct CallScope {
  const Options o = options();
  Side side = SIDE_HOST;
  int dev = 0;
  b200sort_stats stats{};
  DeviceScope device;

  int enter(const std::vector<StreamDesc> &arrays, const int64_t *offsets, const char *device_only) {
    if (int rc = place_arrays(arrays, offsets, device_only, &side, &dev)) return rc;
    if (side == SIDE_DEVICE) {
      if (int rc = device.enter(dev)) return rc;
    } else {
      CUDA_TRY(cudaGetDevice(&dev));
    }
    start_profile(o);
    return 0;
  }
  int done(int rc) {
    if (rc == B200SORT_OK) g_last_stats = stats;
    return rc;
  }
};

// ------------------------------------------------------------------------------------------------
// Host arrays, SoA with payloads: pipelined staging (SURVEY 8f rank 2).  PCIe is the bottleneck of a sort
// called with host arrays (16 GB each way for 1e9 u64+u64 records, 0.3 s per direction, against a 44 ms
// sort), and the two directions are independent.  So only the KEYS are waited for: they are sorted together
// with a 32-bit index while the payload arrays are still on their way in, the sorted keys start their way
// out as soon as the sort is done (full duplex with the payload upload), and every payload array is
// permuted by the index when it has arrived and follows the keys out.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) iota_kernel(uint32_t *idx, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) idx[i] = (uint32_t)i;
}

template <typename T>
__global__ void __launch_bounds__(256) gather_kernel(const uint32_t *__restrict__ idx, const T *__restrict__ in, T *__restrict__ out,
                                                     int64_t n, uint32_t cpe) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const size_t src = (size_t)idx[i] * cpe, dst = (size_t)i * cpe;
    for (uint32_t c = 0; c < cpe; c++) out[dst + c] = in[src + c];
  }
}

static bool host_is_pinned(const void *p) {
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return at.type == cudaMemoryTypeHost;
}

// `stage`: the staging cache entry of the current device `dev`, whose guard the caller holds
static int sort_host_pipelined(const Options &o, int dev, CacheEntry &stage, int key_type, bool ascending, int64_t n,
                               const std::vector<StreamDesc> &streams, cudaStream_t caller, b200sort_stats *stats) {
  const int kb = key_bytes_of(key_type);
  DevInfo di;
  if (int rc = dev_info(dev, &di)) return rc;
  ThreadDeviceState &t = t_dev[dev];
  if (t.in == nullptr) {
    CUDA_TRY(cudaStreamCreateWithFlags(&t.in, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&t.comp, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&t.out, cudaStreamNonBlocking));
  }
  const cudaStream_t st_in = t.in, st_comp = t.comp, st_out = t.out;
  const size_t np = streams.size() - 1;
  // device staging: keys | index | payload s in | payload s out
  std::vector<size_t> bytes = {(size_t)n * kb, (size_t)n * 4};
  for (size_t s = 0; s < np; s++) bytes.insert(bytes.end(), 2, (size_t)n * streams[s + 1].elem_bytes);
  size_t total = 0;
  const std::vector<size_t> offs = back_to_back(bytes, &total);
  const size_t off_keys = offs[0], off_idx = offs[1];
  auto off_in = [&](size_t s) { return offs[2 + 2 * s]; };
  auto off_out = [&](size_t s) { return offs[3 + 2 * s]; };
  void *dbuf_v = nullptr;
  if (int rc = cached_buffer(stage, total, "staging", &dbuf_v)) return rc;
  unsigned char *dbuf = (unsigned char *)dbuf_v;

  std::vector<cudaEvent_t> ev;
  auto new_event = [&]() -> cudaEvent_t {
    cudaEvent_t e = nullptr;
    cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    ev.push_back(e);
    return e;
  };
  int rc = B200SORT_OK;
  auto run = [&]() -> int {
    // everything is ordered after what the caller already queued on its stream
    cudaEvent_t e_begin = new_event();
    CUDA_TRY(cudaEventRecord(e_begin, caller));
    CUDA_TRY(cudaStreamWaitEvent(st_in, e_begin, 0));
    CUDA_TRY(cudaStreamWaitEvent(st_comp, e_begin, 0));
    CUDA_TRY(cudaStreamWaitEvent(st_out, e_begin, 0));

    cudaEvent_t e_keys = new_event();
    CUDA_TRY(cudaMemcpyAsync(dbuf + off_keys, streams[0].ptr, (size_t)n * kb, cudaMemcpyHostToDevice, st_in));
    CUDA_TRY(cudaEventRecord(e_keys, st_in));
    std::vector<cudaEvent_t> e_pay(np);
    auto upload_payloads = [&]() -> int {
      for (size_t s = 0; s < np; s++) {
        CUDA_TRY(cudaMemcpyAsync(dbuf + off_in(s), streams[s + 1].ptr, (size_t)n * streams[s + 1].elem_bytes, cudaMemcpyHostToDevice, st_in));
        e_pay[s] = new_event();
        CUDA_TRY(cudaEventRecord(e_pay[s], st_in));
      }
      return 0;
    };
    // pinned host arrays: the uploads are asynchronous, queue them all before the sort (whose plan read-back
    // blocks this thread); pageable arrays: an upload blocks this thread, so launch the sort first
    bool pinned = true;
    for (size_t s = 0; s < streams.size(); s++) pinned = pinned && host_is_pinned(streams[s].ptr);
    if (pinned)
      if (int r = upload_payloads()) return r;

    CUDA_TRY(cudaStreamWaitEvent(st_comp, e_keys, 0));
    CUDA_TRY(launch(PK_NONE, iota_kernel, di.sm_count * 8, 256, 0, st_comp, (uint32_t *)(dbuf + off_idx), n));
    std::vector<StreamDesc> ds = {{dbuf + off_keys, (uint32_t)kb}, {dbuf + off_idx, 4u}};
    if (int r = sort_device(o, key_type, ascending, n, ds, st_comp, nullptr, 0, DevSortOpts(), stats)) return r;
    cudaEvent_t e_sorted = new_event();
    CUDA_TRY(cudaEventRecord(e_sorted, st_comp));
    if (!pinned)
      if (int r = upload_payloads()) return r;

    CUDA_TRY(cudaStreamWaitEvent(st_out, e_sorted, 0));
    CUDA_TRY(cudaMemcpyAsync(streams[0].ptr, dbuf + off_keys, (size_t)n * kb, cudaMemcpyDeviceToHost, st_out));
    for (size_t s = 0; s < np; s++) {
      const uint32_t eb = streams[s + 1].elem_bytes;
      uint32_t ck = 16;
      while (ck > 1 && (eb % ck) != 0) ck >>= 1;
      const uint32_t cpe = eb / ck;
      CUDA_TRY(cudaStreamWaitEvent(st_comp, e_pay[s], 0));
      const uint32_t *idx = (const uint32_t *)(dbuf + off_idx);
      const unsigned grid = (unsigned)std::min<int64_t>((n + 255) / 256, (int64_t)di.sm_count * 16);
      auto gather = [&](auto *t) {  // (t: the type of one chunk)
        using T = std::remove_pointer_t<decltype(t)>;
        return launch(PK_NONE, gather_kernel<T>, grid, 256, 0, st_comp, idx, (const T *)(dbuf + off_in(s)), (T *)(dbuf + off_out(s)), n, cpe);
      };
      CUDA_TRY(ck == 16 ? gather((uint4 *)nullptr) : ck == 8 ? gather((uint64_t *)nullptr) : ck == 4 ? gather((uint32_t *)nullptr)
               : ck == 2 ? gather((uint16_t *)nullptr) : gather((uint8_t *)nullptr));
      cudaEvent_t e_g = new_event();
      CUDA_TRY(cudaEventRecord(e_g, st_comp));
      CUDA_TRY(cudaStreamWaitEvent(st_out, e_g, 0));
      CUDA_TRY(cudaMemcpyAsync(streams[s + 1].ptr, dbuf + off_out(s), (size_t)n * eb, cudaMemcpyDeviceToHost, st_out));
    }
    return 0;
  };
  rc = run();
  // host arrays: the call returns when the data is back
  cudaError_t e1 = cudaStreamSynchronize(st_in), e2 = cudaStreamSynchronize(st_comp), e3 = cudaStreamSynchronize(st_out);
  for (cudaEvent_t e : ev) cudaEventDestroy(e);
  if (rc == 0 && (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess))
    rc = fail(B200SORT_ECUDA, "pipelined host sort failed on the device: %s",
              cudaGetErrorString(e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3)));
  return rc;
}

// Host arrays sorted whole on the current device `dev`: the arrays, and `upload_bytes` at `upload` (NULL for none)
// that the sort only reads, copied up into the device's staging buffer; sort(the arrays' device streams, the device
// copy of `upload`); the arrays copied back unless it failed.  Returns when they are back.
template <typename SortFn>
static int sort_staged(int dev, int64_t n, const std::vector<StreamDesc> &streams, const void *upload, size_t upload_bytes,
                       cudaStream_t stream, SortFn &&sort) {
  std::vector<size_t> bytes;
  for (const StreamDesc &s : streams) bytes.push_back((size_t)n * s.elem_bytes);
  if (upload != nullptr) bytes.push_back(upload_bytes);
  size_t total = 0;
  const std::vector<size_t> offs = back_to_back(bytes, &total);
  CacheGuard guard;  // the staging buffer is the library's, like the workspace; the call is synchronous anyway
  void *dbuf_v = nullptr;
  if (int rc = cached_buffer(guard.acquire(dev, stream).stage, total, "staging", &dbuf_v)) return rc;
  unsigned char *dbuf = (unsigned char *)dbuf_v;
  std::vector<StreamDesc> dstreams(streams.size());
  for (size_t s = 0; s < streams.size(); s++) dstreams[s] = {dbuf + offs[s], streams[s].elem_bytes};
  int rc = B200SORT_OK;
  cudaError_t e = cudaSuccess;
  for (size_t i = 0; i < bytes.size() && rc == 0; i++) {
    e = cudaMemcpyAsync(dbuf + offs[i], i < streams.size() ? streams[i].ptr : upload, bytes[i], cudaMemcpyHostToDevice, stream);
    if (e != cudaSuccess) rc = fail(B200SORT_ECUDA, "H2D copy failed: %s", cudaGetErrorString(e));
  }
  if (rc == 0) rc = sort(dstreams, upload != nullptr ? dbuf + offs.back() : nullptr);
  for (size_t s = 0; s < streams.size() && rc == 0; s++) {
    e = cudaMemcpyAsync(streams[s].ptr, dstreams[s].ptr, bytes[s], cudaMemcpyDeviceToHost, stream);
    if (e != cudaSuccess) rc = fail(B200SORT_ECUDA, "D2H copy failed: %s", cudaGetErrorString(e));
  }
  e = cudaStreamSynchronize(stream);
  if (e != cudaSuccess && rc == 0) rc = fail(B200SORT_ECUDA, "sort failed on the device: %s", cudaGetErrorString(e));
  return rc;
}

static int sort_any(int key_type, bool ascending, int64_t n, const std::vector<StreamDesc> &streams, void *stream_v,
                    void *workspace, size_t workspace_bytes, const DevSortOpts &base) {
  cudaStream_t stream = (cudaStream_t)stream_v;
  if (n <= 1) return B200SORT_OK;  // src/radix_sort.hpp:276: nothing to do for 0 or 1 element
  CallScope call;  // device arrays: sorted on the device that owns them (include/b200sort.h)
  if (int rc = call.enter(streams, nullptr, nullptr)) return rc;
  const Options &o = call.o;
  auto sort = [&](const std::vector<StreamDesc> &dstreams, const void *) {
    return sort_device(o, key_type, ascending, n, dstreams, stream, workspace, workspace_bytes, base, &call.stats);
  };
  if (call.side == SIDE_DEVICE) return call.done(sort(streams, nullptr));

  // ---- host arrays: staged on the current device, through its cached staging buffer ----------------
  // SoA with payloads, big enough to care: pipelined staging
  if (o.host_pipeline != 0 && base.cmp_none_thresh == 0 && workspace == nullptr && streams.size() >= 2 &&
      streams[0].elem_bytes == (uint32_t)key_bytes_of(key_type) && n >= ((int64_t)1 << 20) && n < ((int64_t)1 << 32)) {
    CacheGuard guard;
    CacheEntry &stage = guard.acquire(call.dev, stream).stage;
    size_t need = 0;
    for (size_t s = 0; s < streams.size(); s++) need += (size_t)n * streams[s].elem_bytes * (s ? 2 : 1);
    need += (size_t)n * 4 + 2 * ((size_t)n * (key_bytes_of(key_type) + 4));  // index + the sort's own workspace
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && need < free_b / 10 * 9 + stage.bytes)
      return call.done(sort_host_pipelined(o, call.dev, stage, key_type, ascending, n, streams, stream, &call.stats));
    cudaGetLastError();
  }
  // everything else: the whole arrays up, the sort, the whole arrays down
  return call.done(sort_staged(call.dev, n, streams, nullptr, 0, stream, sort));
}

static int check_soa(void *keys, int key_type, int64_t num, int n_payloads, void *const *payloads,
                     const uint32_t *payload_elem_bytes, std::vector<StreamDesc> *out) {
  const int kb = key_bytes_of(key_type);
  if (kb == 0) return fail(B200SORT_EINVAL, "unknown key type %d", key_type);
  if (num < 0) return fail(B200SORT_EINVAL, "negative element count");
  if (n_payloads < 0 || n_payloads > MAX_STREAMS - 1)
    return fail(B200SORT_ESHAPE, "%d payload streams (0..%d supported)", n_payloads, MAX_STREAMS - 1);
  if (num > 1 && keys == nullptr) return fail(B200SORT_EINVAL, "keys is NULL");
  out->push_back({keys, (uint32_t)kb});
  for (int p = 0; p < n_payloads; p++) {
    const uint32_t eb = payload_elem_bytes ? payload_elem_bytes[p] : 0;
    if (eb < 1 || eb > 64) return fail(B200SORT_ESHAPE, "payload %d has element size %u (1..64 supported)", p, eb);
    if (num > 1 && (payloads == nullptr || payloads[p] == nullptr)) return fail(B200SORT_EINVAL, "payload %d is NULL", p);
    out->push_back({payloads ? payloads[p] : nullptr, eb});
  }
  return 0;
}

static int check_aos(void *records, int key_type, uint32_t record_bytes, int64_t num, std::vector<StreamDesc> *out) {
  const int kb = key_bytes_of(key_type);
  if (kb == 0) return fail(B200SORT_EINVAL, "unknown key type %d", key_type);
  if (num < 0) return fail(B200SORT_EINVAL, "negative element count");
  if (record_bytes < (uint32_t)kb || record_bytes > 64 || (record_bytes & (record_bytes - 1)) != 0)
    return fail(B200SORT_ERECORD, "record size %u is not a power of two in [%d, 64]", record_bytes, kb);
  if (num > 1 && records == nullptr) return fail(B200SORT_EINVAL, "records is NULL");
  out->push_back({records, record_bytes});
  return 0;
}

// EINVAL unless no output overlaps an input and no two outputs overlap each other (NULL and empty ranges overlap
// nothing); the calls whose outputs are not written in place check this before any device work
struct ByteRange { const void *ptr; size_t bytes; };
static int check_disjoint(const std::vector<ByteRange> &in, const std::vector<ByteRange> &out) {
  auto overlap = [](const ByteRange &a, const ByteRange &b) {
    const uintptr_t x = (uintptr_t)a.ptr, y = (uintptr_t)b.ptr;
    return a.ptr && b.ptr && a.bytes != 0 && b.bytes != 0 && x < y + b.bytes && y < x + a.bytes;
  };
  for (size_t i = 0; i < out.size(); i++) {
    for (const ByteRange &r : in)
      if (overlap(r, out[i])) return fail(B200SORT_EINVAL, "an output overlaps the input");
    for (size_t j = 0; j < i; j++)
      if (overlap(out[j], out[i])) return fail(B200SORT_EINVAL, "two outputs overlap");
  }
  return 0;
}

// the options of the _ex calls' comparison sorter.  CmpSorterInsertionSort: the full sort whatever the threshold.
// CmpSorterNoSort: buckets of at most cmp_sort_threshold elements may stay unordered (src/radix_sort.hpp:279,
// src/cmp_sorters.hpp:66-78).
static int cmp_sorter_opts(int64_t cmp_sort_threshold, int cmp_sorter, DevSortOpts *out) {
  if (cmp_sorter != B200SORT_CMP_INSERTION && cmp_sorter != B200SORT_CMP_NONE)
    return fail(B200SORT_EINVAL, "unknown cmp_sorter %d", cmp_sorter);
  if (cmp_sorter == B200SORT_CMP_NONE && cmp_sort_threshold >= CMP_NONE_MIN_THRESH) out->cmp_none_thresh = cmp_sort_threshold;
  return 0;
}

}  // namespace b200sort

using namespace b200sort;

extern "C" {

int b200sort_sort_soa_ex(void *keys, int key_type, int64_t num, int ascending, int n_payloads, void *const *payloads,
                         const uint32_t *payload_elem_bytes, int64_t cmp_sort_threshold, int cmp_sorter, void *stream,
                         void *workspace, size_t workspace_bytes) {
  DevSortOpts base;
  if (int rc = cmp_sorter_opts(cmp_sort_threshold, cmp_sorter, &base)) return rc;
  std::vector<StreamDesc> streams;
  if (int rc = check_soa(keys, key_type, num, n_payloads, payloads, payload_elem_bytes, &streams)) return rc;
  return sort_any(key_type, ascending != 0, num, streams, stream, workspace, workspace_bytes, base);
}

int b200sort_sort_aos_ex(void *records, int key_type, uint32_t record_bytes, int64_t num, int ascending,
                         int64_t cmp_sort_threshold, int cmp_sorter, void *stream, void *workspace,
                         size_t workspace_bytes) {
  DevSortOpts base;
  if (int rc = cmp_sorter_opts(cmp_sort_threshold, cmp_sorter, &base)) return rc;
  std::vector<StreamDesc> streams;
  if (int rc = check_aos(records, key_type, record_bytes, num, &streams)) return rc;
  return sort_any(key_type, ascending != 0, num, streams, stream, workspace, workspace_bytes, base);
}

int b200sort_sort_soa(void *keys, int key_type, int64_t num, int ascending, int n_payloads, void *const *payloads,
                      const uint32_t *payload_elem_bytes, void *stream, void *workspace, size_t workspace_bytes) {
  return b200sort_sort_soa_ex(keys, key_type, num, ascending, n_payloads, payloads, payload_elem_bytes, 16,
                              B200SORT_CMP_INSERTION, stream, workspace, workspace_bytes);
}

int b200sort_sort_aos(void *records, int key_type, uint32_t record_bytes, int64_t num, int ascending, void *stream,
                      void *workspace, size_t workspace_bytes) {
  return b200sort_sort_aos_ex(records, key_type, record_bytes, num, ascending, 16, B200SORT_CMP_INSERTION, stream,
                              workspace, workspace_bytes);
}

size_t b200sort_workspace_bytes(int key_type, int64_t num, int n_payloads, const uint32_t *payload_elem_bytes,
                                uint32_t record_bytes) {
  const int kb = key_bytes_of(key_type);
  if (kb == 0 || num < 0) return 0;
  return sort_workspace_bytes(streams_of_shape(kb, n_payloads, payload_elem_bytes, record_bytes), num);
}

const char *b200sort_last_error(void) { return g_last_error.c_str(); }
int b200sort_version(void) { return B200SORT_VERSION; }
uint64_t b200sort_launch_count(void) { return g_launches.load(); }

static int64_t Options::*find_opt(const char *name) {
  for (const auto &e : kOptionNames) if (name && !strcmp(name, e.name)) return e.member;
  return nullptr;
}
int b200sort_set_option(const char *name, int64_t value) {
  int64_t Options::*m = find_opt(name);
  if (!m) return fail(B200SORT_EINVAL, "unknown option '%s'", name ? name : "(null)");
  if (m == &Options::max_chunk && (value < 1 || value > 16 || (value & (value - 1)) != 0))
    return fail(B200SORT_EINVAL, "max_chunk must be a power of two in [1, 16], not %lld", (long long)value);
  std::lock_guard<std::mutex> lk(g_opt_mu);
  g_opt.*m = value;
  return 0;
}
int64_t b200sort_get_option(const char *name) {
  int64_t Options::*m = find_opt(name);
  std::lock_guard<std::mutex> lk(g_opt_mu);
  return m ? g_opt.*m : INT64_MIN;
}

int b200sort_last_stats(b200sort_stats *out) {
  if (!out || g_last_stats.num < 0) return B200SORT_EINVAL;
  *out = g_last_stats;
  return 0;
}

int b200sort_last_profile(int *kinds, float *ms, int capacity) {
  int n = 0;
  for (auto &p : g_prof) {
    if (n >= capacity) break;
    if (cudaEventSynchronize(p.e1) != cudaSuccess) return fail(B200SORT_ECUDA, "profile event failed");
    float t = 0;
    cudaEventElapsedTime(&t, p.e0, p.e1);
    kinds[n] = p.kind;
    ms[n] = t;
    n++;
  }
  return n;
}

void b200sort_release_cache(void) {
  std::vector<std::pair<int, DeviceState *>> devs;
  {
    std::lock_guard<std::mutex> lk(g_mu);
    for (auto &kv : g_devs) devs.push_back({kv.first, &kv.second});
  }
  for (auto [dev, ds] : devs) {
    std::lock_guard<std::recursive_mutex> guard(ds->mu);  // (a sort being launched on the caches finishes that first)
    for (CacheEntry *c : {&ds->workspace, &ds->stage}) {
      if (!c->ptr) continue;
      DeviceScope scope;  // (each buffer is freed on its own device)
      if (scope.enter(dev) == 0) { cudaDeviceSynchronize(); cudaFree(c->ptr); }
      c->ptr = nullptr;
      c->bytes = 0;  // (gen survives: a later allocation is a new one for the multi-GPU handle check)
    }
  }
}

}  // extern "C"

#include "mgpu.cuh"
#include "segmented_host.cuh"
#include "topk_host.cuh"
#include "unique_host.cuh"
