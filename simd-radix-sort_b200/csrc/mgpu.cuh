// mgpu.cuh -- multi-GPU sort: MSB range partition over the GPUs of one box (SURVEY.md 8e).
// Included at the end of b200sort.cu (it uses that file's internals).
//
//   1. every rank histograms the top 16 bits of a sample of its order-mapped keys (top_hist_kernel)
//   2. ncclAllReduce(sum) of the histograms -> identical splitters on every rank (b200sort_mgpu_splitters)
//   3. exact number of records per destination (dest_count_kernel); ncclAllGather of these rows together
//      with every rank's workspace IPC handle -> receive offsets, peer mappings
//   4. partition + exchange in ONE kernel: a scatter pass of onesweep_kernel in LUT mode whose bucket d is
//      the receive region of GPU d -- the records leave the staging tile as coalesced stores straight
//      into peer memory over NVLink (cudaIpc mapping of the peer's workspace); a 1-element all-reduce is
//      the barrier after it.  Fallback when the workspaces cannot be mapped (or option mgpu_p2p = 0): the
//      same pass into local memory, then grouped ncclSend/ncclRecv per peer.
//   5. local sort of the received range, which starts in the workspace's shadow arrays (sort_device)
// The reference has nothing here (single thread); NCCL is loaded lazily with dlopen so that the
// single-GPU library has no NCCL dependency.
#pragma once
#include <dlfcn.h>
#include <nccl.h>

namespace b200sort {

struct NcclApi {
  ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char *(*GetErrorString)(ncclResult_t) = nullptr;
  bool ok = false;
  std::string why;
};

static NcclApi &nccl_api() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) { api.why = std::string("dlopen(libnccl.so.2) failed: ") + dlerror(); return; }
#define SYM(field, name)                                                   \
    api.field = reinterpret_cast<decltype(api.field)>(dlsym(h, name));     \
    if (!api.field) { api.why = std::string("missing symbol ") + name; return; }
    SYM(GetUniqueId, "ncclGetUniqueId") SYM(CommInitRank, "ncclCommInitRank") SYM(CommDestroy, "ncclCommDestroy")
    SYM(AllReduce, "ncclAllReduce") SYM(AllGather, "ncclAllGather") SYM(Send, "ncclSend") SYM(Recv, "ncclRecv")
    SYM(GroupStart, "ncclGroupStart") SYM(GroupEnd, "ncclGroupEnd") SYM(GetErrorString, "ncclGetErrorString")
#undef SYM
    api.ok = true;
  });
  return api;
}

#define NCCL_TRY(expr)                                                                                   \
  do {                                                                                                   \
    ncclResult_t _r = (expr);                                                                            \
    if (_r != ncclSuccess)                                                                               \
      return fail(B200SORT_ENCCL, "%s failed: %s", #expr, nccl_api().GetErrorString(_r));                 \
  } while (0)

constexpr int MGPU_MAX_BITS = 16;

// counts of the top `bits` bits of the ordered key; warp-aggregated global atomics
struct TopHistArgs {
  const unsigned char *keys;
  uint32_t stride;
  int64_t n;
  KeyOrder ko;
  int shift;            // bin = range_bin(ordered key, lo, shift, nb)
  unsigned long long *hist;  // [nb], zeroed
  int64_t sample;       // every sample-th row of 32 keys is counted
  unsigned long long lo;
  uint32_t nb;
  unsigned long long *range;  // range_kernel: [0] = min ordered key, [1] = min of the complements (= ~max)
};

template <int KB>
__global__ void __launch_bounds__(256) top_hist_kernel(TopHistArgs a) {
  // every sample-th row of 32 consecutive keys (splitters only need proportions; the exact numbers of
  // records per destination are counted afterwards by dest_count_kernel)
  const int lane = threadIdx.x & 31;
  const int64_t n_rows = (a.n + 31) / 32;
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x / 32);
  for (int64_t w = (int64_t)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5); w * a.sample < n_rows; w += n_warps) {
    const int64_t i = w * a.sample * 32 + lane;
    const bool valid = i < a.n;
    const unsigned vmask = __ballot_sync(0xffffffffu, valid);
    if (valid) {
      const uint32_t bin = range_bin((unsigned long long)to_ordered<KB, false>(load_key<KB>(a.keys, i, a.stride), a.ko), a.lo, a.shift, a.nb);
      const unsigned peers = __match_any_sync(vmask, bin);
      if ((peers & lanemask_lt()) == 0) atomicAdd(&a.hist[bin], (unsigned long long)__popc(peers));
    }
  }
}

// smallest and largest ordered key of the same sample: the histogram bins cover that range, not the whole key
// space (keys of a narrow range -- small integers, N(0,1) doubles -- would otherwise share one or two bins)
template <int KB>
__global__ void __launch_bounds__(256) range_kernel(TopHistArgs a) {
  const int lane = threadIdx.x & 31;
  const int64_t n_rows = (a.n + 31) / 32;
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x / 32);
  unsigned long long mn = ~0ull, nmx = ~0ull;
  for (int64_t w = (int64_t)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5); w * a.sample < n_rows; w += n_warps) {
    const int64_t i = w * a.sample * 32 + lane;
    if (i < a.n) {
      const unsigned long long u = (unsigned long long)to_ordered<KB, false>(load_key<KB>(a.keys, i, a.stride), a.ko);
      mn = u < mn ? u : mn;
      nmx = ~u < nmx ? ~u : nmx;
    }
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) {
    const unsigned long long m2 = __shfl_xor_sync(0xffffffffu, mn, s), n2 = __shfl_xor_sync(0xffffffffu, nmx, s);
    mn = m2 < mn ? m2 : mn;
    nmx = n2 < nmx ? n2 : nmx;
  }
  if (lane == 0) {
    atomicMin(&a.range[0], mn);
    atomicMin(&a.range[1], nmx);
  }
}

static cudaError_t launch_top_hist(int kb, const TopHistArgs &a, int sm_count, cudaStream_t st, bool range_only = false) {
  const int64_t rows = ((a.n + 31) / 32 + a.sample - 1) / a.sample;
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((rows + 7) / 8, (int64_t)sm_count * 16));
  return with_kb(kb, [&](auto K) {
    constexpr int KB = decltype(K)::value;
    return launch(PK_HIST, range_only ? range_kernel<KB> : top_hist_kernel<KB>, grid, 256, 0, st, a);
  });
}

// ---- refinement of heavy histogram bins (SURVEY 8e(3)) -------------------------------------------------------
// Histograms of up to MGPU_MAX_REFINE sub-ranges of the key space at once, on the same sample of rows as
// top_hist_kernel: range j covers [lo[j], lo[j] + (nb[j] << shift[j])), bin = (u - lo[j]) >> shift[j].
constexpr int MGPU_MAX_REFINE = 8;
struct RefineArgs {
  const unsigned char *keys;
  uint32_t stride;
  int64_t n;
  KeyOrder ko;
  int64_t sample;
  int n_ranges;
  unsigned long long lo[MGPU_MAX_REFINE];
  int shift[MGPU_MAX_REFINE];
  uint32_t nb[MGPU_MAX_REFINE];
  unsigned long long *hist;  // [n_ranges][2^16], zeroed
};

template <int KB>
__global__ void __launch_bounds__(256) refine_hist_kernel(RefineArgs a) {
  const int lane = threadIdx.x & 31;
  const int64_t n_rows = (a.n + 31) / 32;
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x / 32);
  for (int64_t w = (int64_t)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5); w * a.sample < n_rows; w += n_warps) {
    const int64_t i = w * a.sample * 32 + lane;
    if (i >= a.n) continue;
    const unsigned long long u = (unsigned long long)to_ordered<KB, false>(load_key<KB>(a.keys, i, a.stride), a.ko);
    for (int j = 0; j < a.n_ranges; j++) {
      if (u < a.lo[j]) continue;
      const unsigned long long b = (u - a.lo[j]) >> a.shift[j];
      if (b < a.nb[j]) atomicAdd(&a.hist[((size_t)j << MGPU_MAX_BITS) + b], 1ull);
    }
  }
}

// ---- heavy key values: exact counts ---------------------------------------------------------------------
// For every tie value v[j] (a splitter sits on it): the exact number of local keys below it and the number of
// local keys EQUAL to it in each of MGPU_TIE_BLOCKS position blocks of the local array.  Full pass over the keys;
// only launched when a heavy single value exists.
constexpr int MGPU_TIE_BLOCKS = 1024;
struct TieCountArgs {
  const unsigned char *keys;
  uint32_t stride;
  int64_t n;
  KeyOrder ko;
  int n_ties;
  unsigned long long v[MGPU_MAX_REFINE];
  int blk_shift;
  unsigned long long *less;  // [n_ties], zeroed
  uint32_t *eq;              // [n_ties][MGPU_TIE_BLOCKS], zeroed
};

template <int KB>
__global__ void __launch_bounds__(256) tie_count_kernel(TieCountArgs a) {
  const int lane = threadIdx.x & 31;
  unsigned long long less[MGPU_MAX_REFINE];
#pragma unroll
  for (int j = 0; j < MGPU_MAX_REFINE; j++) less[j] = 0;
  const int64_t n_rows = (a.n + 31) / 32;
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x / 32);
  for (int64_t w = (int64_t)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5); w < n_rows; w += n_warps) {
    const int64_t i = w * 32 + lane;
    const bool valid = i < a.n;
    const unsigned long long u = valid ? (unsigned long long)to_ordered<KB, false>(load_key<KB>(a.keys, i, a.stride), a.ko) : 0ull;
#pragma unroll
    for (int j = 0; j < MGPU_MAX_REFINE; j++) {
      if (j >= a.n_ties) break;
      less[j] += (valid && u < a.v[j]) ? 1ull : 0ull;
      // a row of 32 consecutive keys lies in one position block (blk_shift >= 5): one atomic per row and value
      const unsigned m = __ballot_sync(0xffffffffu, valid && u == a.v[j]);
      if (m != 0 && lane == 0) atomicAdd(&a.eq[j * MGPU_TIE_BLOCKS + (int)((w * 32) >> a.blk_shift)], (uint32_t)__popc(m));
    }
  }
#pragma unroll
  for (int j = 0; j < MGPU_MAX_REFINE; j++) {
    if (j >= a.n_ties) break;
    unsigned long long x = less[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if (lane == 0 && x) atomicAdd(&a.less[j], x);
  }
}

// ---- exact number of records this rank sends to every destination (destination = part_dest) ---------------
// With `digit_hist` set (overlapped exchange): additionally, per destination, the exact histogram of the digit
// the destination's local sort sweeps first -- what its probe kernel would otherwise have to count after the
// exchange -- for the tiles [tile_lo, tile_hi) of one chunk.
struct DestCountArgs {
  const unsigned char *keys;
  uint32_t stride;
  int64_t n;
  KeyOrder ko;
  PartArgs part;
  unsigned long long *counts;  // [RADIX], zeroed
  int world;
  int64_t tile_lo, tile_hi;    // KeyTile tiles of this launch (whole array: 0, n_tiles)
  uint32_t *digit_hist;        // [world][RADIX] or nullptr
  uint32_t digit_lshift[8];    // per destination: digit = ((u << lshift) >> shift) & 255
  uint32_t digit_shift[8];
  // fast form of the destination (8-byte keys, no ties, splitters with zero low words -- bin boundaries of
  // full-width keys): destination = number of r with (high word of u) > hi_m1[r]
  uint32_t hi_only;
  uint32_t hi_m1[8];           // 0xffffffff: never
};

template <int KB, int NLD>
__global__ void __launch_bounds__(HIST_THREADS, 1024 / HIST_THREADS) dest_count_kernel(DestCountArgs a) {
  using KT = KeyTile<KB, HIST_THREADS, NLD>;
  __shared__ uint32_t sh[RADIX];
  __shared__ uint32_t sdh[8 * RADIX];
  for (int i = threadIdx.x; i < RADIX; i += HIST_THREADS) sh[i] = 0;
  const bool dh = a.digit_hist != nullptr;  // (world <= 8 then)
  if (dh)
    for (int i = threadIdx.x; i < 8 * RADIX; i += HIST_THREADS) sdh[i] = 0;
  __syncthreads();
  const bool dense = a.stride == KB && (((uintptr_t)a.keys) & 15) == 0;
  uint32_t cnt[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // world <= 8: lane-private counters
  uint32_t n_ge[7] = {0, 0, 0, 0, 0, 0, 0}, n_all = 0;
  for (int64_t tile = a.tile_lo + blockIdx.x; tile < a.tile_hi; tile += gridDim.x) {
    KT kt;
    kt.template load<false>(a.keys, a.stride, a.n, tile, a.ko);
    const int64_t base = tile * KT::TILE;
    const bool full = kt.valid == (KT::PER_THREAD >= 32 ? 0xffffffffu : ((1u << KT::PER_THREAD) - 1));
    if (KB == 8 && !dh && a.hi_only && full) {
      // lane-private cumulative counters: n_ge[r] = keys at or above splitter r (one 32-bit compare each); the
      // records per destination are their differences
#pragma unroll
      for (int i = 0; i < KT::PER_THREAD; i++) {
        const uint32_t h = (uint32_t)((unsigned long long)kt.u[i] >> 32);
#pragma unroll
        for (int r = 0; r < 7; r++) n_ge[r] += h > a.hi_m1[r] ? 1u : 0u;
      }
      n_all += KT::PER_THREAD;
      continue;
    }
    if (KB == 8 && dh && a.hi_only && full) {
      // the overlapped exchange's common case: seven 32-bit compares for the destination, one shift pair for the
      // digit, one shared-memory atomic (the records per destination are the sums of its histogram)
#pragma unroll
      for (int i = 0; i < KT::PER_THREAD; i++) {
        const unsigned long long u = (unsigned long long)kt.u[i];
        const uint32_t h = (uint32_t)(u >> 32);
        uint32_t d = 0;
#pragma unroll
        for (int r = 0; r < 7; r++) d += h > a.hi_m1[r] ? 1u : 0u;
        atomicAdd(&sdh[d * RADIX + ((uint32_t)((u << a.digit_lshift[d]) >> a.digit_shift[d]) & (RADIX - 1))], 1u);
      }
      continue;
    }
    const bool vec = dense && base + KT::TILE <= a.n;  // KeyTile's vector layout: thread t holds keys (j*THREADS+t)*VEC+e
#pragma unroll
    for (int i = 0; i < KT::PER_THREAD; i++) {
      const bool v = (kt.valid >> i) & 1;
      const int64_t idx = vec ? base + ((int64_t)(i / KT::VEC) * HIST_THREADS + threadIdx.x) * KT::VEC + (i % KT::VEC)
                              : base + (int64_t)i * HIST_THREADS + threadIdx.x;
      const unsigned long long u = (unsigned long long)kt.u[i];
      const uint32_t d = v ? part_dest(u, idx, a.part) : 0u;
      if (a.world <= 8) {
        if (!(dh && a.hi_only)) {  // (hi_only: the records per destination are taken from the histogram sums)
#pragma unroll
          for (int r = 0; r < 8; r++) cnt[r] += (v && d == (uint32_t)r) ? 1u : 0u;
        }
        if (dh && v) atomicAdd(&sdh[d * RADIX + ((uint32_t)((u << a.digit_lshift[d]) >> a.digit_shift[d]) & (RADIX - 1))], 1u);
      } else {
        const unsigned vmask = __ballot_sync(0xffffffffu, v);
        if (v) hist_add<true>(sh, d, vmask);
      }
    }
  }
  if (a.world <= 8) {
#pragma unroll
    for (int r = 0; r < 8; r++) {
      uint32_t c = cnt[r] + (r == 0 ? n_all : n_ge[r - 1]) - (r < 7 ? n_ge[r] : 0u);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
      if ((threadIdx.x & 31) == 0 && c) atomicAdd(&sh[r], c);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < RADIX; i += HIST_THREADS) {
    const uint32_t c = sh[i];
    if (c) atomicAdd(&a.counts[i], (unsigned long long)c);
  }
  if (dh)
    for (int i = threadIdx.x; i < a.world * RADIX; i += HIST_THREADS) {
      const uint32_t c = sdh[i];
      if (c) {
        atomicAdd(&a.digit_hist[i], c);
        if (a.hi_only) atomicAdd(&a.counts[i / RADIX], (unsigned long long)c);  // (the fast path keeps no separate counters)
      }
    }
}

// The fast forms of dest_count_kernel as a kernel of their own (8-byte keys, splitters with zero low words, no
// ties, full tiles only -- the caller sends the last, partial tile through the general kernel): the general
// kernel's three code paths cost it registers and a third of its speed.
template <int NLD>
__global__ void __launch_bounds__(HIST_THREADS, 1024 / HIST_THREADS) dest_count_fast_kernel(DestCountArgs a) {
  using KT = KeyTile<8, HIST_THREADS, NLD>;
  __shared__ uint32_t sdh[8 * RADIX];
  const bool dh = a.digit_hist != nullptr;
  if (dh)
    for (int i = threadIdx.x; i < 8 * RADIX; i += HIST_THREADS) sdh[i] = 0;
  __syncthreads();
  uint32_t n_ge[7] = {0, 0, 0, 0, 0, 0, 0}, n_all = 0;
  for (int64_t tile = a.tile_lo + blockIdx.x; tile < a.tile_hi; tile += gridDim.x) {
    KT kt;
    kt.template load<false>(a.keys, a.stride, a.n, tile, a.ko);  // (full tiles: every key valid)
    if (dh) {
#pragma unroll
      for (int i = 0; i < KT::PER_THREAD; i++) {
        const unsigned long long u = (unsigned long long)kt.u[i];
        const uint32_t h = (uint32_t)(u >> 32);
        uint32_t d = 0;
#pragma unroll
        for (int r = 0; r < 7; r++) d += h > a.hi_m1[r] ? 1u : 0u;
        atomicAdd(&sdh[d * RADIX + ((uint32_t)((u << a.digit_lshift[d]) >> a.digit_shift[d]) & (RADIX - 1))], 1u);
      }
    } else {
#pragma unroll
      for (int i = 0; i < KT::PER_THREAD; i++) {
        const uint32_t h = (uint32_t)((unsigned long long)kt.u[i] >> 32);
#pragma unroll
        for (int r = 0; r < 7; r++) n_ge[r] += h > a.hi_m1[r] ? 1u : 0u;
      }
      n_all += KT::PER_THREAD;
    }
  }
  if (dh) {
    __syncthreads();
    for (int i = threadIdx.x; i < a.world * RADIX; i += HIST_THREADS) {
      const uint32_t c = sdh[i];
      if (c) {
        atomicAdd(&a.digit_hist[i], c);
        atomicAdd(&a.counts[i / RADIX], (unsigned long long)c);
      }
    }
  } else {
#pragma unroll
    for (int r = 0; r < 8; r++) {
      uint32_t c = (r == 0 ? n_all : n_ge[r - 1]) - (r < 7 ? n_ge[r] : 0u);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
      if ((threadIdx.x & 31) == 0 && r < a.world && c) atomicAdd(&a.counts[r], (unsigned long long)c);
    }
  }
}

static cudaError_t launch_dest_count(int kb, const DestCountArgs &a0, int sm_count, cudaStream_t st) {
  DestCountArgs a = a0;
  const int64_t tile_keys = (int64_t)HIST_THREADS * hist_nld(kb) * (16 / kb);
  const int64_t n_tiles = (a.n + tile_keys - 1) / tile_keys;
  if (a.tile_hi <= 0 || a.tile_hi > n_tiles) a.tile_hi = n_tiles;
  ProfScope ps(PK_HIST, st);  // (one profile entry for the one or two kernels)
  const bool dense = a.stride == (uint32_t)kb && (((uintptr_t)a.keys) & 15) == 0;
  if (kb == 8 && a.hi_only && a.world <= 8 && dense) {
    // full tiles through the lean kernel, a partial last tile (if it belongs to this launch) through the general one
    const int64_t full_hi = std::min<int64_t>(a.tile_hi, a.n / tile_keys);
    if (full_hi > a.tile_lo) {
      DestCountArgs f = a;
      f.tile_hi = full_hi;
      const int gridf = (int)std::max<int64_t>(1, std::min<int64_t>(full_hi - a.tile_lo, (int64_t)sm_count * 4));
      const cudaError_t e = launch(PK_NONE, dest_count_fast_kernel<hist_nld(8)>, gridf, HIST_THREADS, 0, st, f);
      if (e != cudaSuccess) return e;
    }
    if (full_hi >= a.tile_hi) return cudaSuccess;
    a.tile_lo = std::max(a.tile_lo, full_hi);
  }
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(a.tile_hi - a.tile_lo, (int64_t)sm_count * 8));
  return with_kb(kb, [&](auto K) {
    constexpr int KB = decltype(K)::value;
    return launch(PK_NONE, dest_count_kernel<KB, hist_nld(KB)>, grid, HIST_THREADS, 0, st, a);
  });
}

// From the smallest / largest sampled ordered key to the binning of the splitter histogram:
// bin(u) = clamp((u - lo) >> shift, 0, 2^bits - 1)  (range_bin(), kernels.cuh).
static void choose_range_bins(unsigned long long lo_key, unsigned long long hi_key, int key_bytes, int bits,
                              unsigned long long *out_lo, int *out_shift) {
  unsigned long long lo = lo_key, hi = hi_key;
  if (lo > hi) lo = hi = 0;  // no keys anywhere
  const unsigned long long span = hi - lo;
  const int span_bits = span ? 64 - __builtin_clzll(span) : 0;
  int shift = std::max(0, span_bits - bits);
  // full-width keys: keep the bins aligned with the key's own leading bits (the local sorts then see shards
  // with constant leading bits and can shift them out)
  if (span_bits > 8 * key_bytes - 2) { lo = 0; shift = 8 * key_bytes - bits; }
  *out_lo = lo;
  *out_shift = shift;
}

// Splitters on bin boundaries.  Rank r ideally ends where the running count reaches r/world of the total; any
// boundary whose prefix is within 1/64 of a rank's share of that target is acceptable (capacities leave
// 1/8), and among those the one with the most trailing zero bits wins: the keys of a shard then agree on as
// many leading bits as possible (for uniform keys and a power-of-two world: exactly log2(world) bits),
// which is what lets the local sort shift them out (Plan::lshift).  Identical on every rank because the
// input is the reduced histogram.
static void compute_splitters(const uint64_t *hist, int bits, int world, uint32_t *bounds) {
  const uint32_t nb = 1u << bits;
  std::vector<uint64_t> prefix((size_t)nb + 1);
  prefix[0] = 0;
  for (uint32_t b = 0; b < nb; b++) prefix[b + 1] = prefix[b] + hist[b];
  const uint64_t total = prefix[nb];
  const uint64_t tol = total / (uint64_t)world / 64;
  bounds[0] = 0;
  for (int r = 1; r < world; r++) {
    const uint64_t target = (uint64_t)(((unsigned __int128)total * (unsigned)r) / (unsigned)world);
    // first boundary whose prefix reaches the target, then the closer of it and the one before
    uint32_t b = (uint32_t)(std::lower_bound(prefix.begin(), prefix.end(), target) - prefix.begin());
    if (b > nb) b = nb;
    if (b > 0 && target - prefix[b - 1] < prefix[b] - target) b--;
    if (b < bounds[r - 1]) b = bounds[r - 1];
    // most aligned acceptable boundary around it
    uint32_t best = b;
    int best_tz = b ? __builtin_ctz(b) : 32;
    for (int dir = -1; dir <= 1; dir += 2) {
      for (int64_t c = (int64_t)b + dir; c >= (int64_t)bounds[r - 1] && c <= (int64_t)nb; c += dir) {
        const uint64_t pc = prefix[(size_t)c];
        const uint64_t dist = pc > target ? pc - target : target - pc;
        if (dist > tol) break;
        const int tz = c ? __builtin_ctz((uint32_t)c) : 32;
        if (tz > best_tz) { best = (uint32_t)c; best_tz = tz; }
      }
    }
    bounds[r] = best;
  }
  bounds[world] = nb;
}

// ---- heavy bins: refinement of the splitters down to single key values (SURVEY 8e(3)) -----------------------
// `hist_fn(ctx, n_ranges, lo, shift, nb, out)` must fill out[j][0 .. nb[j]) with the GLOBAL (all ranks) counts of
// the (sampled) keys u in range j: bin = (u - lo[j]) >> shift[j], u in [lo[j], lo[j] + (nb[j] << shift[j])).
// Every call costs one sampled sweep + one all-reduce, so it is only made while a splitter still sits in a bin
// heavier than the tolerance.  The ranges nest: level 0 is the whole key space by its top 16 bits, a heavy bin is
// split by its next 16 bits, and so on until the bin is a single key value -- then the splitter is a TIE
// (out_tie[r] = 1): the equal keys are divided by position (tie_thresholds below).

static int refine_splitters(int world, int key_bits, uint64_t total, b200sort_hist_fn hist_fn, void *ctx,
                            uint64_t *out_key, uint32_t *out_tie, uint64_t *out_below) {
  struct Cur { uint64_t lo; int wb; uint64_t below; bool done; };
  const int ns = world - 1;
  std::vector<Cur> cur(ns, Cur{0, key_bits, 0, false});
  const uint64_t tol = std::max<uint64_t>(total / (uint64_t)world / 64, 1);
  std::vector<uint64_t> hist((size_t)MGPU_MAX_REFINE << MGPU_MAX_BITS);
  for (int level = 0; level < 8; level++) {
    // distinct ranges still to refine (at most world - 1; processed MGPU_MAX_REFINE at a time)
    std::vector<int> todo;
    for (int r = 0; r < ns; r++)
      if (!cur[r].done) todo.push_back(r);
    if (todo.empty()) break;
    size_t pos = 0;
    while (pos < todo.size()) {
      uint64_t lo[MGPU_MAX_REFINE];
      int shift[MGPU_MAX_REFINE], wbq[MGPU_MAX_REFINE];
      uint32_t nb[MGPU_MAX_REFINE];
      std::vector<std::vector<int>> members;
      int nr = 0;
      while (pos < todo.size()) {
        const Cur &c = cur[todo[pos]];
        int j = -1;
        for (int q = 0; q < nr; q++)
          if (lo[q] == c.lo && wbq[q] == c.wb) j = q;  // same range already queued
        if (j < 0) {
          if (nr == MGPU_MAX_REFINE) break;
          j = nr++;
          lo[j] = c.lo;
          wbq[j] = c.wb;
          shift[j] = std::max(c.wb - MGPU_MAX_BITS, 0);
          nb[j] = 1u << (c.wb - shift[j]);
          members.emplace_back();
        }
        members[j].push_back(todo[pos]);
        pos++;
      }
      if (int rc = hist_fn(ctx, nr, lo, shift, nb, hist.data())) return rc;
      for (int j = 0; j < nr; j++) {
        const uint64_t *h = hist.data() + ((size_t)j << MGPU_MAX_BITS);
        for (int r : members[j]) {
          Cur &c = cur[r];
          const uint64_t target = (uint64_t)(((unsigned __int128)total * (unsigned)(r + 1)) / (unsigned)world);
          // first bin whose inclusive prefix exceeds the target
          uint64_t run = c.below;
          uint32_t b = 0;
          for (; b + 1 < nb[j]; b++) {
            if (run + h[b] > target) break;
            run += h[b];
          }
          const uint64_t w = h[b];
          const uint64_t bin_lo = lo[j] + ((uint64_t)b << shift[j]);
          if (w <= tol) {
            // light bin: the boundary is the closer bin edge (an edge past the end of the key space is not one)
            const uint64_t d_lo = target - run, d_hi = run + w - target;
            const uint64_t bin_hi = bin_lo + ((uint64_t)1 << shift[j]);
            const bool hi_ok = bin_hi > bin_lo;  // no wrap-around
            if (hi_ok && d_hi < d_lo) { out_key[r] = bin_hi; out_below[r] = run + w; }
            else { out_key[r] = bin_lo; out_below[r] = run; }
            out_tie[r] = 0;
            c.done = true;
          } else if (shift[j] == 0) {
            out_key[r] = bin_lo;  // a single key value heavier than the tolerance
            out_below[r] = run;
            out_tie[r] = 1;
            c.done = true;
          } else {
            c.lo = bin_lo;
            c.wb = shift[j];
            c.below = run;
          }
        }
      }
    }
  }
  for (int r = 0; r < ns; r++)
    if (!cur[r].done) return fail(B200SORT_EINVAL, "splitter refinement did not converge");
  // splitters are monotonic by construction up to sampling noise at equal targets; enforce it
  for (int r = 1; r < ns; r++)
    if (out_key[r] < out_key[r - 1]) { out_key[r] = out_key[r - 1]; out_tie[r] = out_tie[r - 1]; }
  return 0;
}

// Division of the keys equal to a tie value among the ranks whose splitters sit on it.  In the global order the
// equal keys are taken as ordered by (source rank, position block); `eq[s][b]` is the exact number of them in
// block b of source s, `less_total` the exact number of keys below the value (all ranks), targets[i] the global
// position (number of records that must lie left of splitter i).  For every target the boundary is put at the
// block edge nearest to it; out_blk[i] is the threshold for rank `rank`: its equal keys in blocks >= out_blk[i]
// go right of splitter i (0: all of them, 0xffffffff: none).
static void tie_thresholds(int world, int rank, int n_blocks, uint64_t less_total, const uint32_t *eq /*[world][n_blocks]*/,
                           int n_targets, const uint64_t *targets, uint32_t *out_blk) {
  for (int i = 0; i < n_targets; i++) {
    const uint64_t want = targets[i] > less_total ? targets[i] - less_total : 0;  // equal keys that stay left
    uint64_t run = 0;
    int bs = world, bb = 0;  // boundary = (source, block): default "after everything"
    bool found = false;
    for (int s2 = 0; s2 < world && !found; s2++) {
      for (int b = 0; b < n_blocks; b++) {
        const uint64_t c = eq[(size_t)s2 * n_blocks + b];
        if (run + c > want) {
          // the boundary falls into this block: before or after it, whichever is closer
          if (want - run <= run + c - want) { bs = s2; bb = b; }
          else if (b + 1 < n_blocks) { bs = s2; bb = b + 1; }
          else { bs = s2 + 1; bb = 0; }
          found = true;
          break;
        }
        run += c;
      }
    }
    if (rank < bs) out_blk[i] = 0xffffffffu;
    else if (rank > bs) out_blk[i] = 0u;
    else out_blk[i] = (uint32_t)bb;
  }
}

}  // namespace b200sort

// what every rank tells the others before the exchange (all-gathered in one go)
struct MgpuBlob {
  cudaIpcMemHandle_t handle;        // its workspace allocation
  unsigned long long ws_bytes;      // size of that allocation's layout (equal layouts <=> equal shadow offsets)
  long long capacity;
  unsigned long long p2p;           // 1: this rank is willing to use the peer-memory path
  unsigned long long counts[b200sort::RADIX];  // records it sends to every destination
  // overlapped exchange: records per (chunk, destination) and, per (chunk, destination), the exact histogram of
  // the digit the destination's local sort sweeps first
  unsigned long long chunk_counts[MGPU_MAX_CHUNKS][8];
  uint32_t chunk_hist[MGPU_MAX_CHUNKS][8][b200sort::RADIX];
};

struct b200sort_comm {
  ncclComm_t comm = nullptr;
  int world = 0, rank = 0, dev = 0;
  unsigned long long *d_hist = nullptr;   // [MGPU_MAX_REFINE][2^16] local, then reduced in place
  unsigned long long *d_counts = nullptr; // scratch words for small all-reduces
  unsigned long long *d_split_key = nullptr;  // [RADIX] splitters (PartArgs)
  uint32_t *d_split_blk = nullptr;            // [RADIX]
  uint64_t *d_bin_base = nullptr;         // [MGPU_MAX_CHUNKS][RADIX]
  uint64_t *d_cons_base = nullptr;        // [MGPU_MAX_CHUNKS * 8][RADIX] bucket offsets of the overlapped first-pass launches
  uint32_t *d_cons_ctr = nullptr;         // [MGPU_MAX_CHUNKS * 8] their tile tickets
  int64_t *d_peer_delta = nullptr;        // [RADIX]
  unsigned long long *d_tie_less = nullptr;  // [MGPU_MAX_REFINE], then [world][MGPU_MAX_REFINE] gathered
  uint32_t *d_tie_eq = nullptr;              // [MGPU_MAX_REFINE][MGPU_TIE_BLOCKS], then gathered [world][...]
  MgpuBlob *d_blob = nullptr;             // [world]
  b200sort::Plan *d_plan = nullptr;
  // peer workspaces mapped into this process (cudaIpcOpenMemHandle), keyed by the handle they were opened from
  std::vector<cudaIpcMemHandle_t> peer_handle;
  std::vector<void *> peer_base;
  bool p2p_failed = false;                // mapping failed once: stay on the NCCL path
  cudaIpcMemHandle_t my_handle{};         // handle of this rank's workspace ...
  void *my_handle_of = nullptr;           // ... taken for this allocation
  uint64_t my_handle_gen = 0;
  bool last_p2p = false, last_overlap = false;
  uint32_t seq = 0;                       // sorts done on this communicator (epoch of the arrival flags)
  cudaStream_t side = nullptr;            // high-priority stream of the overlapped first pass
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
};

// B200SORT_MGPU_TRACE=1: per-phase device times of every multi-GPU sort on stderr (adds a stream sync at the end),
// and for the overlapped exchange a timeline of its two streams: when each chunk's partition kernel, arrival and
// first-pass kernels finished, relative to the first timeline mark (the fork)
struct MgpuTrace {
  using Marks = std::vector<std::pair<std::string, cudaEvent_t>>;
  bool on = false;
  cudaStream_t st = nullptr;
  Marks phases, timeline;
  explicit MgpuTrace(cudaStream_t s) : st(s) {
    const char *e = getenv("B200SORT_MGPU_TRACE");
    on = e && *e == '1';
    mark("start");
  }
  void record(Marks &m, const std::string &name, cudaStream_t s) {
    if (!on) return;
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, s);
    m.emplace_back(name, e);
  }
  // end of a phase on the sort's stream
  void mark(const char *name) {
    static const bool dbg = getenv("B200SORT_MGPU_DEBUG") != nullptr;  // host-side progress lines (locating a hang)
    if (dbg) {
      fprintf(stderr, "[b200sort mgpu] reached %s ...", name);
      const cudaError_t e = cudaStreamSynchronize(st);
      fprintf(stderr, " device done (%s)\n", cudaGetErrorString(e));
    }
    record(phases, name, st);
  }
  // a point of the overlapped exchange's timeline, on stream s
  void mark(const std::string &name, cudaStream_t s) { record(timeline, name, s); }
  void report(int rank) {
    if (!on) return;
    cudaStreamSynchronize(st);
    const std::string head = "[b200sort mgpu rank " + std::to_string(rank) + "]";
    auto line = [](const Marks &m, bool from_first, const char *fmt) {
      std::string out;
      for (size_t i = 1; i < m.size(); i++) {
        float ms = 0;
        cudaEventElapsedTime(&ms, m[from_first ? 0 : i - 1].second, m[i].second);
        char buf[96];
        snprintf(buf, sizeof buf, fmt, m[i].first.c_str(), ms);
        out += buf;
      }
      return out;
    };
    if (!timeline.empty()) fprintf(stderr, "%s timeline (ms after the fork):%s\n", head.c_str(), line(timeline, true, " %s=%.2f").c_str());
    float tot = 0;
    cudaEventElapsedTime(&tot, phases.front().second, phases.back().second);
    fprintf(stderr, "%s%s total=%.3f ms\n", head.c_str(), line(phases, false, " %s=%.3f").c_str(), tot);
    for (Marks *m : {&phases, &timeline}) {
      for (auto &e : *m) cudaEventDestroy(e.second);
      m->clear();
    }
  }
};

namespace b200sort {

// ---- arrival flags of the overlapped exchange -------------------------------------------------------------
// After a rank's partition kernel for chunk c has finished, one thread tells every destination so: a system-
// scope fence (the kernel boundary ordered the chunk's peer stores before this thread) and a store of the
// sort's epoch value into the destination's flag word (source, chunk).  The destination's side stream waits for
// all sources' flags of a chunk with a one-warp kernel before it launches the first-pass kernels over what
// arrived.  Nothing on the sending side ever waits for a receiver, so the spinning warp cannot deadlock anything.
struct SignalArgs {
  uint32_t *peer_flags[8];  // flag arrays of all ranks (mapped), [8 sources][MGPU_MAX_CHUNKS]
  int world, me, chunk;
  uint32_t value;
};
static __global__ void mgpu_signal_kernel(SignalArgs a) {
  const int d = threadIdx.x;
  if (d >= a.world) return;
  __threadfence_system();
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(a.peer_flags[d] + a.me * MGPU_MAX_CHUNKS + a.chunk), "r"(a.value) : "memory");
}
static __global__ void mgpu_wait_kernel(const uint32_t *flags, int world, int chunk, uint32_t value) {
  const int s = threadIdx.x;
  if (s < world) {
    uint32_t v;
    do {
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + s * MGPU_MAX_CHUNKS + chunk) : "memory");
      if ((int32_t)(v - value) < 0) __nanosleep(200);
    } while ((int32_t)(v - value) < 0);
  }
  __syncwarp();
  __threadfence_system();
}

}  // namespace b200sort

extern "C" {

int b200sort_mgpu_unique_id(void *out) {
  using namespace b200sort;
  NcclApi &api = nccl_api();
  if (!api.ok) return fail(B200SORT_ENCCL, "NCCL unavailable: %s", api.why.c_str());
  if (!out) return fail(B200SORT_EINVAL, "out is NULL");
  static_assert(sizeof(ncclUniqueId) == B200SORT_UNIQUE_ID_BYTES, "ncclUniqueId size");
  ncclUniqueId id;
  NCCL_TRY(api.GetUniqueId(&id));
  memcpy(out, &id, sizeof id);
  return 0;
}

int b200sort_mgpu_comm_create(b200sort_comm **out, int world_size, int rank, const void *id_bytes) {
  using namespace b200sort;
  NcclApi &api = nccl_api();
  if (!api.ok) return fail(B200SORT_ENCCL, "NCCL unavailable: %s", api.why.c_str());
  if (!out || !id_bytes || world_size < 1 || world_size > RADIX || rank < 0 || rank >= world_size)
    return fail(B200SORT_EINVAL, "bad communicator arguments");
  ncclUniqueId id;
  memcpy(&id, id_bytes, sizeof id);
  // (a failing step returns; the communicator is then destroyed with whatever the steps before it created)
  std::unique_ptr<b200sort_comm, decltype(&b200sort_mgpu_comm_destroy)> c(new b200sort_comm(), b200sort_mgpu_comm_destroy);
  c->world = world_size;
  c->rank = rank;
  c->peer_handle.resize(world_size);
  c->peer_base.assign(world_size, nullptr);
  for (auto &h : c->peer_handle) memset(&h, 0, sizeof h);
  CUDA_TRY(cudaGetDevice(&c->dev));
  NCCL_TRY(api.CommInitRank(&c->comm, world_size, id, rank));
  CUDA_TRY(cudaMalloc(&c->d_hist, (sizeof(unsigned long long) * MGPU_MAX_REFINE) << MGPU_MAX_BITS));
  CUDA_TRY(cudaMalloc(&c->d_counts, sizeof(unsigned long long) * 64));
  CUDA_TRY(cudaMalloc(&c->d_split_key, sizeof(unsigned long long) * RADIX));
  CUDA_TRY(cudaMalloc(&c->d_split_blk, sizeof(uint32_t) * RADIX));
  CUDA_TRY(cudaMalloc(&c->d_bin_base, sizeof(uint64_t) * RADIX * MGPU_MAX_CHUNKS));
  CUDA_TRY(cudaMalloc(&c->d_cons_base, sizeof(uint64_t) * RADIX * MGPU_MAX_CHUNKS * 8));
  CUDA_TRY(cudaMalloc(&c->d_cons_ctr, sizeof(uint32_t) * (MGPU_MAX_CHUNKS * 8 + MGPU_MAX_CHUNKS)));  // (+ the chunks' delivery counters)
  CUDA_TRY(cudaMalloc(&c->d_plan, sizeof(Plan)));
  CUDA_TRY(cudaMalloc(&c->d_peer_delta, sizeof(int64_t) * RADIX));
  CUDA_TRY(cudaMalloc(&c->d_tie_less, sizeof(unsigned long long) * MGPU_MAX_REFINE * (size_t)(world_size + 1)));
  CUDA_TRY(cudaMalloc(&c->d_tie_eq, sizeof(uint32_t) * MGPU_MAX_REFINE * MGPU_TIE_BLOCKS * (size_t)(world_size + 1)));
  CUDA_TRY(cudaMalloc(&c->d_blob, sizeof(MgpuBlob) * (size_t)(world_size + 1)));
  int lo_prio = 0, hi_prio = 0;
  CUDA_TRY(cudaDeviceGetStreamPriorityRange(&lo_prio, &hi_prio));
  CUDA_TRY(cudaStreamCreateWithPriority(&c->side, cudaStreamNonBlocking, hi_prio));
  CUDA_TRY(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
  CUDA_TRY(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
  *out = c.release();
  return 0;
}

int b200sort_mgpu_comm_destroy(b200sort_comm *c) {
  using namespace b200sort;
  if (!c) return 0;
  if (c->comm) nccl_api().CommDestroy(c->comm);
  for (int p = 0; p < c->world; p++)
    if (p != c->rank && c->peer_base[p]) cudaIpcCloseMemHandle(c->peer_base[p]);
  cudaFree(c->d_hist); cudaFree(c->d_counts); cudaFree(c->d_split_key); cudaFree(c->d_split_blk); cudaFree(c->d_bin_base);
  cudaFree(c->d_cons_base); cudaFree(c->d_cons_ctr); cudaFree(c->d_plan); cudaFree(c->d_peer_delta); cudaFree(c->d_tie_less);
  cudaFree(c->d_tie_eq); cudaFree(c->d_blob);
  if (c->side) cudaStreamDestroy(c->side);
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  if (c->ev_join) cudaEventDestroy(c->ev_join);
  delete c;
  return 0;
}

int b200sort_mgpu_used_p2p(const b200sort_comm *c) { return c && c->last_p2p ? 1 : 0; }
int b200sort_mgpu_used_overlap(const b200sort_comm *c) { return c && c->last_overlap ? 1 : 0; }

int b200sort_mgpu_range_bins(uint64_t lo_key, uint64_t hi_key, int key_bytes, int bits, uint64_t *out_lo, int *out_shift) {
  using namespace b200sort;
  if (!out_lo || !out_shift || bits < 1 || bits > MGPU_MAX_BITS || (key_bytes != 1 && key_bytes != 2 && key_bytes != 4 && key_bytes != 8))
    return fail(B200SORT_EINVAL, "bad range arguments");
  unsigned long long lo = 0;
  choose_range_bins(lo_key, hi_key, key_bytes, std::min(bits, 8 * key_bytes), &lo, out_shift);
  *out_lo = lo;
  return 0;
}

int b200sort_mgpu_splitters(const uint64_t *global_hist, int bits, int world_size, uint32_t *out_bounds) {
  using namespace b200sort;
  if (!global_hist || !out_bounds || bits < 1 || bits > MGPU_MAX_BITS || world_size < 1 || world_size > RADIX)
    return fail(B200SORT_EINVAL, "bad splitter arguments");
  compute_splitters(global_hist, bits, world_size, out_bounds);
  return 0;
}

int b200sort_mgpu_refine_splitters(int world_size, int key_bytes, uint64_t total, b200sort_hist_fn hist_fn, void *ctx,
                                   uint64_t *out_keys, uint32_t *out_is_tie) {
  using namespace b200sort;
  if (!hist_fn || !out_keys || !out_is_tie || world_size < 1 || world_size > RADIX ||
      (key_bytes != 1 && key_bytes != 2 && key_bytes != 4 && key_bytes != 8))
    return fail(B200SORT_EINVAL, "bad refinement arguments");
  std::vector<uint64_t> below((size_t)std::max(world_size - 1, 1));
  return refine_splitters(world_size, 8 * key_bytes, total, hist_fn, ctx, out_keys, out_is_tie, below.data());
}

int b200sort_mgpu_tie_thresholds(int world_size, int rank, int n_blocks, uint64_t less_total, const uint32_t *eq, int n_targets,
                                 const uint64_t *targets, uint32_t *out_blk) {
  using namespace b200sort;
  if (!eq || !targets || !out_blk || world_size < 1 || rank < 0 || rank >= world_size || n_blocks < 1 || n_targets < 0)
    return fail(B200SORT_EINVAL, "bad tie arguments");
  tie_thresholds(world_size, rank, n_blocks, less_total, eq, n_targets, targets, out_blk);
  return 0;
}

int b200sort_mgpu_plan(const uint64_t *local_hist, int bits, int world_size, const uint32_t *bounds,
                       uint64_t *out_send_counts) {
  using namespace b200sort;
  if (!local_hist || !bounds || !out_send_counts || bits < 1 || bits > MGPU_MAX_BITS || world_size < 1)
    return fail(B200SORT_EINVAL, "bad plan arguments");
  for (int r = 0; r < world_size; r++) {
    uint64_t s = 0;
    for (uint32_t b = bounds[r]; b < bounds[r + 1]; b++) s += local_hist[b];
    out_send_counts[r] = s;
  }
  return 0;
}

}  // extern "C"

namespace b200sort {

struct RefineCtx {
  b200sort_comm *c;
  NcclApi *api;
  RefineArgs ra;
  int kb, sm_count;
  cudaStream_t stream;
};

// hist_fn of refine_splitters on the device: sampled sweep + all-reduce + read-back
static int mgpu_refine_hist(void *ctx_v, int n_ranges, const uint64_t *lo, const int *shift, const uint32_t *nb, uint64_t *out) {
  RefineCtx *x = (RefineCtx *)ctx_v;
  RefineArgs ra = x->ra;
  ra.n_ranges = n_ranges;
  for (int j = 0; j < n_ranges; j++) { ra.lo[j] = lo[j]; ra.shift[j] = shift[j]; ra.nb[j] = nb[j]; }
  ra.hist = x->c->d_hist;
  const size_t words = (size_t)n_ranges << MGPU_MAX_BITS;
  CUDA_TRY(cudaMemsetAsync(x->c->d_hist, 0, words * 8, x->stream));
  if (ra.n > 0) {
    const int64_t rows = ((ra.n + 31) / 32 + ra.sample - 1) / ra.sample;
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((rows + 7) / 8, (int64_t)x->sm_count * 16));
    CUDA_TRY(with_kb(x->kb, [&](auto K) { return launch(PK_NONE, refine_hist_kernel<decltype(K)::value>, grid, 256, 0, x->stream, ra); }));
  }
  NCCL_TRY(x->api->AllReduce(x->c->d_hist, x->c->d_hist, words, ncclUint64, ncclSum, x->c->comm, x->stream));
  CUDA_TRY(cudaMemcpyAsync(out, x->c->d_hist, words * 8, cudaMemcpyDeviceToHost, x->stream));
  CUDA_TRY(cudaStreamSynchronize(x->stream));
  return 0;
}

// The distributed sort of b200sort_mgpu_sort_soa / b200sort_mgpu_sort_aos, phase by phase (mgpu_sort); streams[0]
// carries the key at offset 0.
struct MgpuSort {
  const Options &o;
  b200sort_comm *const c;
  NcclApi &api;
  const int key_type;
  const std::vector<StreamDesc> &streams;
  const int64_t num_local, capacity;
  const bool ascending;
  const cudaStream_t stream;
  b200sort_stats *const stats;  // of the local sort
  const int kb = key_bytes_of(key_type);
  const int world = c->world;
  const int bits = std::min(MGPU_MAX_BITS, 8 * kb);
  const uint32_t nb = 1u << bits;
  const unsigned char *const keys = (const unsigned char *)streams[0].ptr;
  const uint32_t kstride = streams[0].elem_bytes;
  const int64_t n_ws = std::max<int64_t>(capacity, 1);
  const int64_t sample = std::max<int64_t>(1, num_local >> 24);  // about 2^24 sampled keys at most
  const KeyOrder ko = make_key_order(key_type, ascending);
  MgpuTrace trace{stream};
  // set-up
  DevInfo di;
  StreamSet ss{};
  uint32_t stage_bytes = 0;
  int cfg = 0, tile = 0;
  bool landing = false;
  Layout L;
  unsigned char *ws = nullptr;
  CacheGuard cache_guard;  // (recursive: the local sort takes it again)
  // splitters
  std::vector<uint64_t> global_hist;  // reduced histogram of the sampled keys in 2^bits bins: bin(u) = (u - lo) >> shift
  uint64_t sampled_total = 0;
  unsigned long long lo = 0;
  int shift = 0;
  std::vector<uint32_t> bounds;       // rank r: bins [bounds[r], bounds[r+1])
  bool heavy = false, has_tie = false;
  std::vector<unsigned long long> split_key;
  std::vector<uint32_t> split_blk, split_tie;
  int blk_shift = 5;
  PartArgs part{};
  // overlap decision
  bool overlap = false;
  int n_chunks = 1;
  uint32_t d_lshift[8] = {0}, d_cut[8] = {0};  // per destination: the first digit its local sort sweeps
  std::vector<int> lead;                        // per rank: leading key bits all keys of its shard agree on
  std::vector<int64_t> ct;                      // chunk ch = sweep tiles [ct[ch], ct[ch+1]) of the local input
  // blob exchange, peer mapping
  std::vector<MgpuBlob> blobs;
  MgpuBlob *my_slot = nullptr;  // (device) my contribution, behind the gathered array
  bool my_handle_changed = false, p2p = false;
  std::vector<int64_t> recv_off, send_off;
  int64_t recv_total = 0;

  uint64_t m(int src, int dst) const { return blobs[src].counts[dst]; }  // records rank src sends to rank dst

  // set-up: streams, tile geometry, workspace layout, cache guard
  int setup() {
    if (int rc = dev_info(c->dev, &di)) return rc;
    // workspace, laid out for `capacity` records on every rank (so that equal capacities give equal layouts
    // and the local sort finds what the peers wrote where it expects its shadow arrays)
    g_prof_on = o.profile != 0;
    stage_bytes = make_stream_set(streams, kb, 16, &ss);
    cfg = pick_tile_cfg(o, kb, stage_bytes, di.smem_optin, num_local);
    tile = kTileCfgs[cfg].threads * kTileCfgs[cfg].ipt;
    // Large 8-byte-key sorts receive into a third set of arrays (landing): the local sort then runs
    // landing -> shadow -> caller -> shadow -> caller and an even number of passes ends in the caller's arrays
    // without a copy.  The choice depends on nothing but the arguments all ranks share.
    landing = kb == 8 && n_ws >= ((int64_t)1 << o.host_plan_min_log2) && o.mgpu_landing != 0 && o.mgpu_p2p != 0;
    make_layout(streams, n_ws, std::min(tile, HYB_MIN_TILE), &L, landing);
    cache_guard.acquire(c->dev, stream);
    return 0;
  }

  // splitters: key range of a sample of all ranks' keys (min / max all-reduced), then the histogram of that range
  // in 2^bits bins on the same sample, all-reduced; splitters on its bin boundaries, refined where a bin is too
  // heavy (down to single key values: ties).  The same on every rank.  Also takes the workspace.
  int splitters() {
    // A rank whose cached workspace is too small is going to free and re-allocate it.  Its peers may still have
    // the old allocation mapped (cudaIpcOpenMemHandle): they have to let go of it first.  The flag travels with
    // the first all-reduce.
    const bool will_realloc = cache_guard.state->workspace.bytes < L.total;
    unsigned long long range_h[3] = {~0ull, ~0ull, will_realloc ? 0ull : 1ull};
    CUDA_TRY(cudaMemcpyAsync(c->d_counts, range_h, sizeof range_h, cudaMemcpyHostToDevice, stream));
    TopHistArgs ha{keys, kstride, num_local, ko, 0, c->d_hist, sample, 0ull, nb, c->d_counts};
    if (num_local > 0) CUDA_TRY(launch_top_hist(kb, ha, di.sm_count, stream, /*range_only=*/true));
    NCCL_TRY(api.AllReduce(c->d_counts, c->d_counts, 3, ncclUint64, ncclMin, c->comm, stream));
    CUDA_TRY(cudaMemcpyAsync(range_h, c->d_counts, sizeof range_h, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaMemsetAsync(c->d_hist, 0, sizeof(unsigned long long) * nb, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    if (range_h[2] == 0) {
      // somebody re-allocates: every rank drops all its mappings, and nobody frees anything before all have
      for (int r = 0; r < world; r++) {
        if (r != c->rank && c->peer_base[r]) cudaIpcCloseMemHandle(c->peer_base[r]);
        c->peer_base[r] = nullptr;
      }
      NCCL_TRY(api.AllReduce(c->d_counts + 4, c->d_counts + 4, 1, ncclUint64, ncclSum, c->comm, stream));
      CUDA_TRY(cudaStreamSynchronize(stream));
    }
    void *ws_v = nullptr;
    if (int rc = cached_buffer(cache_guard.state->workspace, L.total, "workspace", &ws_v)) return rc;
    ws = (unsigned char *)ws_v;
    for (size_t s = 0; s < streams.size(); s++) ss.streams[s].buf[1] = ws + L.shadow_off[s];
    choose_range_bins(range_h[0], ~range_h[1], kb, bits, &lo, &shift);
    ha.lo = lo; ha.shift = shift;
    if (num_local > 0) CUDA_TRY(launch_top_hist(kb, ha, di.sm_count, stream));
    global_hist.assign(nb, 0);
    NCCL_TRY(api.AllReduce(c->d_hist, c->d_hist, nb, ncclUint64, ncclSum, c->comm, stream));
    CUDA_TRY(cudaMemcpyAsync(global_hist.data(), c->d_hist, sizeof(uint64_t) * nb, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    trace.mark("hist+allreduce");

    // Ordinary case: splitters on bin boundaries of that histogram.  A rank that would get more than its share
    // + 1/16 means a bin too heavy to be kept whole (skewed keys, few distinct values, SURVEY 8e(3)): the
    // splitters are then refined, 16 key bits per level, down to single key values if need be, and the keys
    // EQUAL to such a value are divided by source rank and position.
    bounds.assign(world + 1, 0);
    compute_splitters(global_hist.data(), bits, world, bounds.data());
    std::vector<uint64_t> prefix((size_t)nb + 1, 0);
    for (uint32_t b = 0; b < nb; b++) prefix[b + 1] = prefix[b] + global_hist[b];
    sampled_total = prefix[nb];
    const uint64_t share = sampled_total / (uint64_t)world;
    for (int r = 0; r < world; r++) heavy = heavy || prefix[bounds[r + 1]] - prefix[bounds[r]] > share + share / 16 + 64;
    const int ns = world - 1;
    split_key.assign(std::max(ns, 1), 0ull);
    split_blk.assign(std::max(ns, 1), 0u);
    split_tie.assign(std::max(ns, 1), 0u);
    while (((int64_t)MGPU_TIE_BLOCKS << blk_shift) < std::max<int64_t>(capacity, 1)) blk_shift++;  // capacity: the same on all ranks
    if (!heavy || o.mgpu_refine == 0) {
      heavy = false;
      for (int r = 0; r < ns; r++) {
        const uint32_t b = bounds[r + 1];
        split_key[r] = b == 0 ? 0ull : (b >= nb ? ~0ull : lo + ((unsigned long long)b << shift));
      }
    } else {
      RefineCtx rx{c, &api, RefineArgs{}, kb, di.sm_count, stream};
      rx.ra.keys = keys; rx.ra.stride = kstride; rx.ra.n = num_local; rx.ra.ko = ko; rx.ra.sample = sample;
      std::vector<uint64_t> rk(std::max(ns, 1)), below(std::max(ns, 1));
      if (int rc = refine_splitters(world, 8 * kb, sampled_total, mgpu_refine_hist, &rx, rk.data(), split_tie.data(), below.data())) return rc;
      for (int r = 0; r < ns; r++) { split_key[r] = rk[r]; has_tie = has_tie || split_tie[r] != 0; }
      trace.mark("refine");
      if (has_tie)
        if (int rc = tie_blocks()) return rc;
    }
    CUDA_TRY(cudaMemcpyAsync(c->d_split_key, split_key.data(), sizeof(unsigned long long) * std::max(ns, 1), cudaMemcpyHostToDevice, stream));
    CUDA_TRY(cudaMemcpyAsync(c->d_split_blk, split_blk.data(), sizeof(uint32_t) * std::max(ns, 1), cudaMemcpyHostToDevice, stream));
    part = PartArgs{c->d_split_key, c->d_split_blk, ns, blk_shift, has_tie ? 1 : 0, 0u, {}};
    part.hi_only = (kb == 8 && !has_tie && world <= 8) ? 1u : 0u;
    for (int r = 0; r < 7; r++) {
      part.hi_m1[r] = 0xffffffffu;
      if (r < ns) {
        const unsigned long long kv = split_key[r];
        if ((uint32_t)kv != 0 || (kv >> 32) == 0) part.hi_only = 0;  // (a splitter at 0 or with low bits: general form)
        else part.hi_m1[r] = (uint32_t)(kv >> 32) - 1u;
      }
    }
    return 0;
  }

  // ties: exact counts around the (distinct) tie values -- keys below, equal keys per position block -- all-gathered,
  // and from them this rank's position-block threshold of every splitter that sits on a tie
  int tie_blocks() {
    const int ns = world - 1;
    std::vector<unsigned long long> tv;
    for (int r = 0; r < ns; r++)
      if (split_tie[r] && (tv.empty() || tv.back() != split_key[r])) tv.push_back(split_key[r]);
    std::vector<uint32_t> blk_all(std::max(ns, 1), 0u);
    for (size_t t0 = 0; t0 < tv.size(); t0 += MGPU_MAX_REFINE) {
      const int nt = (int)std::min<size_t>(MGPU_MAX_REFINE, tv.size() - t0);
      unsigned long long *my_less = c->d_tie_less + (size_t)world * MGPU_MAX_REFINE;          // my slot, then gathered at 0
      uint32_t *my_eq = c->d_tie_eq + (size_t)world * MGPU_MAX_REFINE * MGPU_TIE_BLOCKS;
      CUDA_TRY(cudaMemsetAsync(my_less, 0, sizeof(unsigned long long) * MGPU_MAX_REFINE, stream));
      CUDA_TRY(cudaMemsetAsync(my_eq, 0, sizeof(uint32_t) * MGPU_MAX_REFINE * MGPU_TIE_BLOCKS, stream));
      TieCountArgs ta{keys, kstride, num_local, ko, nt, {}, blk_shift, my_less, my_eq};
      for (int j = 0; j < nt; j++) ta.v[j] = tv[t0 + j];
      if (num_local > 0) {
        const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((num_local + 255) / 256, (int64_t)di.sm_count * 16));
        CUDA_TRY(with_kb(kb, [&](auto K) { return launch(PK_NONE, tie_count_kernel<decltype(K)::value>, grid, 256, 0, stream, ta); }));
      }
      NCCL_TRY(api.AllGather(my_less, c->d_tie_less, MGPU_MAX_REFINE, ncclUint64, c->comm, stream));
      NCCL_TRY(api.AllGather(my_eq, c->d_tie_eq, (size_t)MGPU_MAX_REFINE * MGPU_TIE_BLOCKS, ncclUint32, c->comm, stream));
      std::vector<unsigned long long> less_h((size_t)world * MGPU_MAX_REFINE);
      std::vector<uint32_t> eq_h((size_t)world * MGPU_MAX_REFINE * MGPU_TIE_BLOCKS);
      unsigned long long tot_h[2] = {(unsigned long long)num_local, 0};
      CUDA_TRY(cudaMemcpyAsync(c->d_counts + 8, tot_h, 8, cudaMemcpyHostToDevice, stream));
      NCCL_TRY(api.AllReduce(c->d_counts + 8, c->d_counts + 8, 1, ncclUint64, ncclSum, c->comm, stream));
      CUDA_TRY(cudaMemcpyAsync(tot_h, c->d_counts + 8, 8, cudaMemcpyDeviceToHost, stream));
      CUDA_TRY(cudaMemcpyAsync(less_h.data(), c->d_tie_less, less_h.size() * 8, cudaMemcpyDeviceToHost, stream));
      CUDA_TRY(cudaMemcpyAsync(eq_h.data(), c->d_tie_eq, eq_h.size() * 4, cudaMemcpyDeviceToHost, stream));
      CUDA_TRY(cudaStreamSynchronize(stream));
      const uint64_t n_total = tot_h[0];
      for (int j = 0; j < nt; j++) {
        uint64_t less_total = 0;
        std::vector<uint32_t> eq((size_t)world * MGPU_TIE_BLOCKS);
        for (int s2 = 0; s2 < world; s2++) {
          less_total += less_h[(size_t)s2 * MGPU_MAX_REFINE + j];
          memcpy(&eq[(size_t)s2 * MGPU_TIE_BLOCKS], &eq_h[((size_t)s2 * MGPU_MAX_REFINE + j) * MGPU_TIE_BLOCKS], sizeof(uint32_t) * MGPU_TIE_BLOCKS);
        }
        std::vector<uint64_t> targets;
        std::vector<int> which;
        for (int r = 0; r < ns; r++)
          if (split_tie[r] && split_key[r] == tv[t0 + j]) {
            targets.push_back((uint64_t)(((unsigned __int128)n_total * (unsigned)(r + 1)) / (unsigned)world));
            which.push_back(r);
          }
        std::vector<uint32_t> out(targets.size());
        tie_thresholds(world, c->rank, MGPU_TIE_BLOCKS, less_total, eq.data(), (int)targets.size(), targets.data(), out.data());
        for (size_t q = 0; q < which.size(); q++) blk_all[which[q]] = out[q];
      }
    }
    for (int r = 0; r < ns; r++) split_blk[r] = split_tie[r] ? blk_all[r] : 0u;
    // (key, block) pairs must ascend: an ordinary splitter on the same key value as a tie keeps the tie's threshold
    for (int r = 1; r < ns; r++)
      if (split_key[r] == split_key[r - 1] && split_blk[r] < split_blk[r - 1]) split_blk[r] = split_blk[r - 1];
    trace.mark("ties");
    return 0;
  }

  // Overlapped exchange (the headline shape): full-width 8-byte keys, close to uniform, one box, peer memory.
  // Then every destination's local plan is known in advance (hybrid: the four -- or five -- digit positions
  // below its shard's common leading bits), the senders count the first of those digits per destination while
  // they count the records, and the destination runs its first pass chunk by chunk while later chunks are
  // still on the NVLink.
  void decide_overlap() {
    // leading key bits each rank's range [bounds[r], bounds[r+1]) of top-`bits` values has in common (bins aligned
    // with the key's own leading bits only)
    const bool aligned = !heavy && kb == 8 && lo == 0 && shift == 8 * kb - bits;
    lead.assign(world, 0);
    for (int r = 0; r < world; r++)
      if (aligned && bounds[r + 1] > bounds[r]) {
        const uint32_t x = bounds[r] ^ (bounds[r + 1] - 1);
        lead[r] = x ? __builtin_clz(x) - (32 - bits) : bits;
      }
    const int64_t chunk_min = (int64_t)1 << o.mgpu_chunk_min_log2;
    n_chunks = (int)o.mgpu_chunks;
    overlap = landing && aligned && world <= 8 && (world >= 2 || o.mgpu_overlap == 2) && o.mgpu_overlap != 0 &&
              o.mgpu_p2p != 0 && !c->p2p_failed && cfg == kDefaultTileCfg && streams[0].elem_bytes == (uint32_t)kb;
    if (overlap) {
      // flat enough?  (by the top 8 bits of the sampled histogram inside every shard)
      std::vector<uint64_t> g256(256, 0);
      for (uint32_t b = 0; b < nb; b++) g256[b >> (bits - 8)] += global_hist[b];
      uint64_t mx = 0, mn = ~0ull;
      for (int g = 0; g < 256; g++) { mx = std::max(mx, g256[g]); mn = std::min(mn, g256[g]); }
      overlap = mn > 0 && mx <= mn + mn / 4;
      for (int r = 0; r < world && overlap; r++) {
        if (bounds[r + 1] <= bounds[r]) { overlap = false; break; }
        const double est_n = (double)sampled_total * (double)sample / (double)world;
        const int swept = (int)std::ceil((std::log2(std::max(est_n, 2.0)) + (double)o.margin_bits) / 8.0);
        const int cut = 8 - lead[r] / 8 - swept;
        if (cut < 2 || o.allow_lshift == 0) { overlap = false; break; }
        d_lshift[r] = (uint32_t)(lead[r] & 7);
        d_cut[r] = (uint32_t)cut;
      }
      // (all ranks took the same decision: it depends on the reduced histogram and shared arguments only; the
      //  records per rank must be large enough for chunks to make sense, which is also a shared quantity here)
      overlap = overlap && capacity >= chunk_min;
      while (n_chunks > 1 && capacity / n_chunks < chunk_min / 2) n_chunks--;
    }
    const int64_t n_tiles_local = (num_local + tile - 1) / tile;
    ct.assign(n_chunks + 1, 0);
    for (int ch = 0; ch <= n_chunks; ch++) ct[ch] = overlap ? (n_tiles_local * ch) / n_chunks : (ch == 0 ? 0 : n_tiles_local);
  }

  // blob exchange: my blob = {workspace handle, layout size, capacity, exact send counts (+ first-digit
  // histograms)}, all-gathered; the send and receive offsets from them
  int exchange_blobs() {
    auto mine = std::make_unique<MgpuBlob>();
    const bool want_p2p = o.mgpu_p2p != 0 && !c->p2p_failed;
    if (want_p2p) {
      const uint64_t gen = cache_guard.state->workspace.gen;
      if (c->my_handle_of != ws || c->my_handle_gen != gen) {  // (a slow driver call: once per workspace allocation)
        cudaError_t e = cudaIpcGetMemHandle(&c->my_handle, ws);
        if (e != cudaSuccess) { cudaGetLastError(); c->p2p_failed = true; }
        else { c->my_handle_of = ws; c->my_handle_gen = gen; my_handle_changed = true; }
      }
      mine->handle = c->my_handle;
    }
    // arrival flags of the overlapped exchange: cleared by their owner before the all-gather below, i.e. before
    // any peer can write this sort's flags (the previous sort's are dead: its waits are stream-ordered before this)
    CUDA_TRY(cudaMemsetAsync(ws + L.flags_off, 0, 4096, stream));
    mine->ws_bytes = L.total;
    mine->capacity = capacity;
    mine->p2p = (want_p2p && !c->p2p_failed) ? 1 : 0;
    my_slot = c->d_blob + world;
    CUDA_TRY(cudaMemcpyAsync(my_slot, mine.get(), sizeof(MgpuBlob), cudaMemcpyHostToDevice, stream));  // counts zeroed with it
    trace.mark("host_prep");
    if (num_local > 0) {
      DestCountArgs da{};
      da.keys = keys; da.stride = kstride; da.n = num_local; da.ko = ko; da.part = part; da.world = world;
      da.hi_only = part.hi_only;
      for (int r = 0; r < 8; r++) da.hi_m1[r] = r < 7 ? part.hi_m1[r] : 0xffffffffu;
      if (!overlap) {
        da.counts = my_slot->counts; da.tile_lo = 0; da.tile_hi = 0;
        CUDA_TRY(launch_dest_count(kb, da, di.sm_count, stream));
      } else {
        const int64_t ktile_keys = (int64_t)HIST_THREADS * hist_nld(kb) * (16 / kb);
        for (int r = 0; r < world; r++) { da.digit_lshift[r] = d_lshift[r]; da.digit_shift[r] = d_cut[r] * RADIX_BITS; }
        for (int ch = 0; ch < n_chunks; ch++) {
          // (sweep tiles are a multiple of the counting kernel's tiles: 4096 vs 2048 keys)
          da.counts = my_slot->chunk_counts[ch];  // [8] used, the kernel's [RADIX] view stays inside the blob
          da.digit_hist = &my_slot->chunk_hist[ch][0][0];
          da.tile_lo = ct[ch] * tile / ktile_keys;
          da.tile_hi = std::min<int64_t>(ct[ch + 1] * tile / ktile_keys, (num_local + ktile_keys - 1) / ktile_keys);
          if (da.tile_hi > da.tile_lo) CUDA_TRY(launch_dest_count(kb, da, di.sm_count, stream));
        }
      }
    }
    trace.mark("count");
    NCCL_TRY(api.AllGather(my_slot, c->d_blob, sizeof(MgpuBlob), ncclUint8, c->comm, stream));
    blobs.resize(world);
    CUDA_TRY(cudaMemcpyAsync(blobs.data(), c->d_blob, sizeof(MgpuBlob) * world, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    trace.mark("allgather");
    if (overlap)  // totals per destination from the chunks
      for (int s2 = 0; s2 < world; s2++)
        for (int r = 0; r < world; r++) {
          uint64_t t = 0;
          for (int ch = 0; ch < n_chunks; ch++) t += blobs[s2].chunk_counts[ch][r];
          blobs[s2].counts[r] = t;
        }
    recv_off.assign(world, 0);
    send_off.assign(world, 0);
    for (int s = 0; s < world; s++) { recv_off[s] = recv_total; recv_total += (int64_t)m(s, c->rank); }
    for (int r = 1; r < world; r++) send_off[r] = send_off[r - 1] + (int64_t)m(c->rank, r - 1);
    // every rank can evaluate every rank's receive total, so all ranks fail together
    for (int r = 0; r < world; r++) {
      int64_t t = 0;
      for (int s = 0; s < world; s++) t += (int64_t)m(s, r);
      if (t > blobs[r].capacity)
        return fail(B200SORT_ENOMEM, "rank %d would receive %lld records, its capacity is %lld", r, (long long)t, (long long)blobs[r].capacity);
    }
    return 0;
  }

  // peer mapping: the peer-memory path if everybody is willing and has an equal layout; maps the workspaces that
  // changed since the last sort
  int map_peers() {
    p2p = true;
    for (int r = 0; r < world; r++) p2p = p2p && blobs[r].p2p == 1 && blobs[r].ws_bytes == L.total && blobs[r].capacity == capacity;
    if (p2p) {
      bool ok = true;
      bool changed = false;
      for (int r = 0; r < world; r++) {
        if (r == c->rank) { c->peer_base[r] = ws; continue; }
        if (c->peer_base[r] && memcmp(&c->peer_handle[r], &blobs[r].handle, sizeof(cudaIpcMemHandle_t)) == 0) continue;
        changed = true;
        if (c->peer_base[r]) { cudaIpcCloseMemHandle(c->peer_base[r]); c->peer_base[r] = nullptr; }
        void *pp = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&pp, blobs[r].handle, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) { cudaGetLastError(); ok = false; continue; }
        c->peer_base[r] = pp;
        c->peer_handle[r] = blobs[r].handle;
      }
      // agreement: one failed mapping anywhere sends everybody to the NCCL path for good.  Every rank sees every
      // handle, so all ranks know alike whether any mapping had to be (re)opened -- a rank's own new handle is new
      // for all the others at once -- and the all-reduce is only paid then.
      if (changed || my_handle_changed) {
        unsigned long long flag = ok ? 0ull : 1ull;
        CUDA_TRY(cudaMemcpyAsync(c->d_counts, &flag, sizeof flag, cudaMemcpyHostToDevice, stream));
        NCCL_TRY(api.AllReduce(c->d_counts, c->d_counts, 1, ncclUint64, ncclSum, c->comm, stream));
        CUDA_TRY(cudaMemcpyAsync(&flag, c->d_counts, sizeof flag, cudaMemcpyDeviceToHost, stream));
        CUDA_TRY(cudaStreamSynchronize(stream));
        if (flag != 0) { c->p2p_failed = true; p2p = false; }
      }
    }
    trace.mark("map");
    c->last_p2p = p2p;
    overlap = overlap && p2p;  // (p2p is an agreed value)
    c->last_overlap = overlap;
    return 0;
  }

  // what the partition pass(es) need on the device: cleared control block, peer offsets, a one-pass plan, and the
  // bucket offsets -- one table per chunk: where my records (of chunk ch) go inside rank r's receive range (peer
  // path), or inside my own shadow arrays (NCCL path); buckets past the world take none
  int prepare_partition() {
    CUDA_TRY(cudaMemsetAsync(ws + L.ctrl_off, 0, L.ctrl_bytes, stream));
    int64_t peer_delta[RADIX] = {0};
    for (int r = 0; r < world; r++) peer_delta[r] = p2p ? (int64_t)((intptr_t)c->peer_base[r] - (intptr_t)ws) : 0;
    CUDA_TRY(cudaMemcpyAsync(c->d_peer_delta, peer_delta, sizeof peer_delta, cudaMemcpyHostToDevice, stream));
    Plan plan{};
    plan.final_sel = 1; plan.n_exec = 1;
    CUDA_TRY(cudaMemcpyAsync(c->d_plan, &plan, sizeof plan, cudaMemcpyHostToDevice, stream));
    const int n_tables = overlap ? n_chunks : 1;
    std::vector<uint64_t> bb((size_t)n_tables * RADIX, (uint64_t)num_local);
    for (int r = 0; r < world; r++) {
      int64_t o = p2p ? 0 : send_off[r];
      for (int s2 = 0; p2p && s2 < c->rank; s2++) o += (int64_t)m(s2, r);
      for (int ch = 0; ch < n_tables; ch++) {
        bb[(size_t)ch * RADIX + r] = (uint64_t)o;
        if (overlap) o += (int64_t)blobs[c->rank].chunk_counts[ch][r];
      }
    }
    CUDA_TRY(cudaMemcpyAsync(c->d_bin_base, bb.data(), bb.size() * 8, cudaMemcpyHostToDevice, stream));
    return 0;
  }

  // the partition pass over my tiles from t_first on (records < n_end): bucket d = what goes to rank d
  SweepArgs partition_args(int pass, int64_t t_first, int64_t n_end) {
    SweepArgs wa{};
    wa.ss = ss; wa.n = n_end; wa.ko = ko; wa.pass = pass; wa.shift = 0;
    if (p2p && landing)
      for (size_t s2 = 0; s2 < streams.size(); s2++) wa.ss.streams[s2].buf[1] = ws + L.land_off[s2];
    wa.bin_base = c->d_bin_base + (size_t)pass * RADIX; wa.lookback = (uint64_t *)(ws + L.lookback_off);
    // (look-back tags 16.. : the local sort's passes, tags 1..8, reuse the same table later)
    wa.tile_counter = (uint32_t *)(ws + L.tilectr_off); wa.plan = c->d_plan; wa.tag = 16u + (uint32_t)pass; wa.stage_bytes = stage_bytes;
    wa.part = part; wa.lut_world = world; wa.tile_first = (uint32_t)t_first; wa.peer_wide = o.mgpu_wide != 0 ? 1u : 0u;
    wa.peer_delta = p2p ? c->d_peer_delta : nullptr;
    return wa;
  }

  // plain exchange: one partition pass.  Peer path: caller arrays -> shadow (or landing) arrays OF RANK d, at the
  // offset where this rank's records belong.  NCCL path: caller arrays -> own shadow arrays, then send/recv.
  // Then the local sort of what arrived.
  int plain_exchange() {
    if (num_local > 0) {
      SweepArgs wa = partition_args(0, 0, num_local);
      CUDA_TRY(launch_sweep(o, kb, cfg, wa, ct[n_chunks], di.smem_optin, stream));
    }
    trace.mark(p2p ? "partition+exchange" : "partition");
    DevSortOpts so;
    so.layout_n = n_ws;
    so.layout_landing = landing;
    if (p2p) {
      // barrier: nobody reads its shadow arrays before every rank's scatter kernel has finished (the
      // all-reduce is ordered after the local kernel on each rank's stream and completes when all joined)
      NCCL_TRY(api.AllReduce(c->d_counts, c->d_counts, 1, ncclUint64, ncclSum, c->comm, stream));
      trace.mark("barrier");
      // local sort, input in the shadow (or landing) arrays, result in the caller's arrays
      so.start_sel = landing ? 0 : 1;
      so.hint_lead_bits = lead[c->rank];
      so.landing_input = landing;
      if (recv_total > 0)
        if (int rc = sort_device(o, key_type, ascending, recv_total, streams, stream, nullptr, 0, so, stats)) return rc;
    } else {
      // all-to-all-v, shadow -> caller arrays
      NCCL_TRY(api.GroupStart());
      for (size_t s = 0; s < streams.size(); s++) {
        const size_t eb = streams[s].elem_bytes;
        for (int p = 0; p < world; p++) {
          const size_t sb = (size_t)m(c->rank, p) * eb, rb = (size_t)m(p, c->rank) * eb;
          if (sb) NCCL_TRY(api.Send(ss.streams[s].buf[1] + (size_t)send_off[p] * eb, sb, ncclUint8, p, c->comm, stream));
          if (rb) NCCL_TRY(api.Recv(ss.streams[s].buf[0] + (size_t)recv_off[p] * eb, rb, ncclUint8, p, c->comm, stream));
        }
      }
      NCCL_TRY(api.GroupEnd());
      trace.mark("exchange");
      if (recv_total > 1)
        if (int rc = sort_device(o, key_type, ascending, recv_total, streams, stream, nullptr, 0, so, stats)) return rc;
    }
    trace.mark("local_sort");
    return 0;
  }

  // ---- overlapped exchange --------------------------------------------------------------------------------
  // main stream : partition kernel of chunk 0, signal, chunk 1, signal, ...
  // side stream : wait for all sources' chunk 0, first-pass kernels over the eight regions of it, wait chunk 1, ...
  // then the main stream joins and runs the remaining passes of the local sort.
  int overlapped_exchange() {
    const uint32_t my_cut = d_cut[c->rank], my_lshift = d_lshift[c->rank];
    const int n_launch = n_chunks * world;
    {
      // bucket offsets of my first pass: launch (ch, s2) sweeps what source s2 sent me in chunk ch; its keys of digit d
      // go behind those of all earlier launches (any order is fine for a first pass)
      std::vector<uint64_t> cb((size_t)n_launch * RADIX, 0);
      uint64_t tot[RADIX] = {0};
      for (int ch = 0; ch < n_chunks; ch++)
        for (int s2 = 0; s2 < world; s2++)
          for (int d = 0; d < RADIX; d++) tot[d] += blobs[s2].chunk_hist[ch][c->rank][d];
      uint64_t run[RADIX];
      uint64_t acc = 0;
      for (int d = 0; d < RADIX; d++) { run[d] = acc; acc += tot[d]; }
      if ((int64_t)acc != recv_total) return fail(B200SORT_ECUDA, "internal: first-digit histograms (%llu) disagree with the record counts (%lld)", (unsigned long long)acc, (long long)recv_total);
      for (int ch = 0; ch < n_chunks; ch++)
        for (int s2 = 0; s2 < world; s2++) {
          const int Lx = ch * world + s2;
          for (int d = 0; d < RADIX; d++) { cb[(size_t)Lx * RADIX + d] = run[d]; run[d] += blobs[s2].chunk_hist[ch][c->rank][d]; }
        }
      CUDA_TRY(cudaMemcpyAsync(c->d_cons_base, cb.data(), cb.size() * 8, cudaMemcpyHostToDevice, stream));
      CUDA_TRY(cudaMemsetAsync(c->d_cons_ctr, 0, sizeof(uint32_t) * (MGPU_MAX_CHUNKS * 8 + MGPU_MAX_CHUNKS), stream));
      // the first pass's look-back table: the junction table's memory (unused until the last pass)
      CUDA_TRY(cudaMemsetAsync(ws + L.jtable_off, 0, (size_t)L.n_tiles * RADIX * 8, stream));
    }
    CUDA_TRY(cudaEventRecord(c->ev_fork, stream));
    CUDA_TRY(cudaStreamWaitEvent(c->side, c->ev_fork, 0));
    trace.mark("fork", stream);
    SignalArgs sg{};
    sg.world = world; sg.me = c->rank;
    for (int r = 0; r < world; r++) sg.peer_flags[r] = (uint32_t *)((unsigned char *)c->peer_base[r] + L.flags_off);
    const uint32_t epoch = c->seq * 16u;
    // ONE partition kernel for all chunks, launched with about one and a half CTAs per SM that loop over the tile
    // tickets (so that the first-pass kernels of the side stream find room on every SM the whole time); the CTA
    // that delivers the last tile of a chunk writes the chunk's arrival flag into every destination's flag array.
    // (A chunk without tiles is signalled from here.)
    for (int ch = 0; ch < n_chunks; ch++)
      if (ct[ch + 1] == ct[ch]) {
        sg.chunk = ch; sg.value = epoch + (uint32_t)ch + 1u;
        CUDA_TRY(launch(PK_NONE, mgpu_signal_kernel, 1, 32, 0, stream, sg));
      }
    const int64_t persist_x2 = o.mgpu_persist_x2;
    if (persist_x2 <= 0) {
      // variant: one ordinary partition kernel per chunk (one CTA per tile), each followed by a one-warp kernel
      // that writes the chunk's flags (the first-pass kernels of the high-priority side stream then alternate with
      // the chunks' partition kernels rather than run beside them)
      for (int ch = 0; ch < n_chunks; ch++) {
        if (ct[ch + 1] == ct[ch]) continue;  // (signalled above)
        SweepArgs wa = partition_args(ch, ct[ch], std::min<int64_t>(num_local, ct[ch + 1] * tile));
        CUDA_TRY(launch_sweep(o, kb, cfg, wa, ct[ch + 1] - ct[ch], di.smem_optin, stream));
        sg.chunk = ch; sg.value = epoch + (uint32_t)ch + 1u;
        CUDA_TRY(launch(PK_NONE, mgpu_signal_kernel, 1, 32, 0, stream, sg));
      }
    } else if (ct[n_chunks] > 0) {
      SweepArgs wa = partition_args(0, 0, num_local);
      wa.sig_n = (uint32_t)n_chunks;
      for (int ch = 0; ch <= n_chunks; ch++) wa.sig_ct[ch] = (uint32_t)ct[ch];
      wa.sig_done = c->d_cons_ctr + MGPU_MAX_CHUNKS * 8;
      for (int r = 0; r < world; r++) wa.sig_flags[r] = sg.peer_flags[r];
      wa.sig_me = (uint32_t)c->rank; wa.sig_value = epoch + 1u;
      const int64_t cap = std::max<int64_t>(1, (int64_t)di.sm_count * persist_x2 / 2);
      CUDA_TRY(launch_sweep(o, kb, cfg, wa, ct[n_chunks], di.smem_optin, stream, false, 0, cap));
    }
    trace.mark("sent_all", stream);
    int64_t tiles_before = 0;
    for (int ch = 0; ch < n_chunks; ch++) {
      // receiver side of the same chunk
      CUDA_TRY(launch(PK_NONE, mgpu_wait_kernel, 1, 32, 0, c->side, (const uint32_t *)(ws + L.flags_off), world, ch, epoch + (uint32_t)ch + 1u));
      trace.mark("arrived" + std::to_string(ch), c->side);
      for (int s2 = 0; s2 < world; s2++) {
        const int64_t cnt = (int64_t)blobs[s2].chunk_counts[ch][c->rank];
        const int64_t tiles_here = (cnt + tile - 1) / tile;
        if (cnt > 0) {
          int64_t lo_rec = recv_off[s2];
          for (int c2 = 0; c2 < ch; c2++) lo_rec += (int64_t)blobs[s2].chunk_counts[c2][c->rank];
          SweepArgs wa{};
          wa.ss = ss;
          for (size_t q = 0; q < streams.size(); q++) {  // landing sub-range in, shadow arrays out
            wa.ss.streams[q].buf[0] = ws + L.land_off[q] + (size_t)lo_rec * streams[q].elem_bytes;
            wa.ss.streams[q].buf[1] = ws + L.shadow_off[q];
          }
          wa.n = cnt; wa.ko = ko; wa.pass = ch * world + s2; wa.shift = (int)my_cut * RADIX_BITS;
          wa.bin_base = c->d_cons_base + (size_t)(ch * world + s2) * RADIX;
          wa.ghist = (uint64_t *)(ws + L.ghist2_off);
          wa.lookback = (uint64_t *)(ws + L.jtable_off) + (size_t)tiles_before * RADIX;
          wa.tile_counter = c->d_cons_ctr; wa.plan = c->d_plan; wa.tag = my_cut + 1; wa.stage_bytes = stage_bytes;
          wa.plan_in_args = 1; wa.arg_sel = 0; wa.arg_next_p1 = my_cut + 2; wa.arg_next_skewed = 0; wa.arg_sub = 0; wa.arg_lshift = my_lshift;
          // (high-priority stream: without a bound on its CTAs per SM the first pass would take every slot that frees
          //  up and starve the partition kernel -- measured: the two then simply alternate)
          CUDA_TRY(launch_sweep(o, kb, cfg, wa, tiles_here, di.smem_optin, c->side, /*first_pass_unordered=*/true,
                                (size_t)o.mgpu_cons_smem_kb << 10));
        }
        tiles_before += tiles_here;
      }
      trace.mark("swept" + std::to_string(ch), c->side);
    }
    CUDA_TRY(cudaEventRecord(c->ev_join, c->side));
    CUDA_TRY(cudaStreamWaitEvent(stream, c->ev_join, 0));
    trace.mark("exchange+first_pass");
    if (recv_total > 0) {
      DevSortOpts so;
      so.layout_n = n_ws;
      so.layout_landing = landing;
      so.landing_input = true;
      so.forced = true;
      so.forced_cut = my_cut;
      so.forced_lshift = my_lshift;
      if (int rc = sort_device(o, key_type, ascending, recv_total, streams, stream, nullptr, 0, so, stats)) return rc;
    }
    trace.mark("local_sort_rest");
    return 0;
  }
};

static int mgpu_sort(const Options &o, b200sort_comm *c, int key_type, const std::vector<StreamDesc> &streams, int64_t num_local,
                     int64_t capacity, bool ascending, int64_t *out_num_local, cudaStream_t stream, b200sort_stats *stats) {
  DeviceScope dev_scope;  // the communicator's device, whatever the caller's current device is
  if (int rc = dev_scope.enter(c->dev)) return rc;
  MgpuSort s{o, c, nccl_api(), key_type, streams, num_local, capacity, ascending, stream, stats};
  c->seq++;
  c->last_overlap = false;
  if (int rc = s.setup()) return rc;
  if (int rc = s.splitters()) return rc;
  s.decide_overlap();
  if (int rc = s.exchange_blobs()) return rc;
  if (int rc = s.map_peers()) return rc;
  *out_num_local = s.recv_total;
  if (int rc = s.prepare_partition()) return rc;
  if (int rc = s.overlap ? s.overlapped_exchange() : s.plain_exchange()) return rc;
  s.trace.report(c->rank);
  return 0;
}

// what both multi-GPU entry points check before anything else
static int mgpu_check(const b200sort_comm *c, int64_t num_local, int64_t capacity, const int64_t *out_num_local) {
  NcclApi &api = nccl_api();
  if (!api.ok) return fail(B200SORT_ENCCL, "NCCL unavailable: %s", api.why.c_str());
  if (!c || !out_num_local) return fail(B200SORT_EINVAL, "comm/out_num_local is NULL");
  if (capacity < num_local) return fail(B200SORT_EINVAL, "capacity smaller than num_local");
  return 0;
}

}  // namespace b200sort

extern "C" {

int b200sort_mgpu_sort_soa(b200sort_comm *c, void *keys, int key_type, int64_t num_local, int64_t capacity,
                           int ascending, int n_payloads, void *const *payloads, const uint32_t *payload_elem_bytes,
                           int64_t *out_num_local, void *stream_v) {
  using namespace b200sort;
  std::vector<StreamDesc> streams;
  if (int rc = mgpu_check(c, num_local, capacity, out_num_local)) return rc;
  if (int rc = check_soa(keys, key_type, num_local, n_payloads, payloads, payload_elem_bytes, &streams)) return rc;
  if (!keys) return fail(B200SORT_EINVAL, "keys is NULL");
  return mgpu_sort(options(), c, key_type, streams, num_local, capacity, ascending != 0, out_num_local, (cudaStream_t)stream_v, &g_last_stats);
}

int b200sort_mgpu_sort_aos(b200sort_comm *c, void *records, int key_type, uint32_t record_bytes, int64_t num_local,
                           int64_t capacity, int ascending, int64_t *out_num_local, void *stream_v) {
  using namespace b200sort;
  std::vector<StreamDesc> streams;
  if (int rc = mgpu_check(c, num_local, capacity, out_num_local)) return rc;
  if (int rc = check_aos(records, key_type, record_bytes, num_local, &streams)) return rc;
  if (!records) return fail(B200SORT_EINVAL, "records is NULL");
  return mgpu_sort(options(), c, key_type, streams, num_local, capacity, ascending != 0, out_num_local, (cudaStream_t)stream_v, &g_last_stats);
}

}  // extern "C"
