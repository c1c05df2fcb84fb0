// segmented.cuh -- segmented sort: many independent segments of one array sorted in one call
// (b200sort_sort_segmented_soa / _aos).  Included at the end of b200sort.cu (it uses that file's internals).
//
//   1. seg_classify_kernel reads the offsets once: it validates them, puts every segment of >= 2 records into a
//      bin by length (a list of segment ids per bin) and records the longest length.  The host reads the bin
//      counts back (one wait) and launches only what has work.
//   2. segments of 2..32 records: seg_tiny_kernel, one warp per segment, rank by counting, in-register move;
//   3. segments of 33..CAP records: seg_medium_kernel, one persistent CTA per segment at a time (atomic ticket
//      per bin), one CTA size per power-of-two bin: an LSD radix sort of (ordered key, 16-bit index) pairs in
//      shared memory over the digits that vary inside the segment, then every column staged and written back
//      permuted (every byte read once and written once);
//   4. segments longer than CAP: keys of <= 4 bytes -- one whole-range sort_device of a u64 composite key
//      (segment index, ordered key); 8-byte keys -- one sort_device per long segment (the composite would not
//      fit in 64 bits).
// seg_medium_kernel (dynamic shared memory) is instantiated in segmented_inst.cu: a kernel with an extern
// __shared__ array gives every other kernel of its module a 1 KB shared-memory reservation.  The host side is
// segmented_host.cuh.
#pragma once
#include "kernels.cuh"

namespace b200sort {

constexpr int SEG_NBINS = 10;              // bin 0: 2..32 records; bin b >= 1: (2^(b+4), 2^(b+5)] records
constexpr int SEG_CAP_LOG2_NARROW = 14;    // CAP = 16384 for keys of <= 4 bytes ...
constexpr int SEG_CAP_LOG2_WIDE = 13;      // ... and 8192 for 8-byte keys (the shared-memory budget, seg_smem_bytes)
constexpr int SEG_TINY_THREADS = 256;
constexpr int SEG_CLASSIFY_THREADS = 256;

__host__ __device__ constexpr int seg_cap_log2(int kb) { return kb == 8 ? SEG_CAP_LOG2_WIDE : SEG_CAP_LOG2_NARROW; }
// threads of the CTA that sorts the segments of the bin whose bound is 2^log_cap records (8 records per thread,
// at least one warp, at most 1024 threads)
__host__ __device__ constexpr int seg_threads(int log_cap) { return log_cap <= 8 ? 32 : (log_cap >= 13 ? 1024 : (1 << log_cap) / 8); }

// written by seg_classify_kernel (zeroed by the host), read back by the host after it
struct SegCtrl {
  uint32_t count[SEG_NBINS];    // segments in each bin's list
  uint32_t ticket[SEG_NBINS];   // next list entry a medium CTA takes
  uint32_t bad;                 // != 0: the offsets are invalid
  uint32_t n_large;             // segments longer than CAP (listed in `large` as (start, length) pairs)
  unsigned long long max_len;   // longest segment (capped at 2^32 - 1)
  long long first, last;        // offsets[0], offsets[n_segments]
};

struct SegClassifyArgs {
  const int64_t *offsets;
  int64_t n_segments, num;
  uint32_t cap;                 // longest segment the tiny and medium kernels sort
  SegCtrl *ctrl;
  uint32_t *list[SEG_NBINS];    // segment ids, one list per bin
  uint32_t list_cap[SEG_NBINS]; // entries each list has room for (enough for valid offsets)
  int64_t *large;               // [n_large][2]
  uint32_t large_cap;
};

// bin of a segment of len (>= 2) records: 0 for <= 32, else b with 2^(b+4) < len <= 2^(b+5)
__device__ __forceinline__ int seg_bin(int64_t len) {
  const int lg = 64 - __clzll((unsigned long long)(len - 1));  // ceil(log2(len))
  return lg <= 5 ? 0 : lg - 5;
}

static __global__ void __launch_bounds__(SEG_CLASSIFY_THREADS) seg_classify_kernel(const __grid_constant__ SegClassifyArgs a) {
  const int lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  // (uniform trip count per warp: the warp-wide votes below need every lane)
  for (int64_t base = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31); base < a.n_segments; base += stride) {
    const int64_t i = base + lane;
    int64_t len = 0;
    bool bad = false;
    if (i < a.n_segments) {
      const int64_t s = a.offsets[i], e = a.offsets[i + 1];
      bad = s < 0 || e < s || e > a.num;
      if (i == 0) a.ctrl->first = s;
      if (i == a.n_segments - 1) a.ctrl->last = e;
      len = bad ? 0 : e - s;
    }
    if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(&a.ctrl->bad, 1u);
    const uint32_t len32 = len > 0xffffffffll ? 0xffffffffu : (uint32_t)len;
    const uint32_t wmax = __reduce_max_sync(0xffffffffu, len32);
    if (lane == 0 && wmax >= 2) atomicMax(&a.ctrl->max_len, (unsigned long long)wmax);
    int bin = -1;  // -1: nothing to do, SEG_NBINS: longer than CAP
    if (len >= 2) bin = len > (int64_t)a.cap ? SEG_NBINS : seg_bin(len);
    // Segments of valid offsets are disjoint and lie inside [0, num), which bounds every list.  Invalid offsets
    // (that decrease somewhere) can make more segments valid on their own than a list holds: no write past the
    // list, and the flag is raised anyway.
    bool overflow = false;
    if (bin == SEG_NBINS) {
      const uint32_t slot = atomicAdd(&a.ctrl->n_large, 1u);
      if (slot < a.large_cap) {
        a.large[2 * (size_t)slot] = a.offsets[i];
        a.large[2 * (size_t)slot + 1] = len;
      } else {
        overflow = true;
      }
    }
    // one atomic per (warp, bin)
    const unsigned peers = __match_any_sync(0xffffffffu, bin);
    const int leader = __ffs(peers) - 1;
    uint32_t slot0 = 0;
    if (lane == leader && bin >= 0 && bin < SEG_NBINS) slot0 = atomicAdd(&a.ctrl->count[bin], (uint32_t)__popc(peers));
    slot0 = __shfl_sync(0xffffffffu, slot0, leader);
    if (bin >= 0 && bin < SEG_NBINS) {
      const uint32_t slot = slot0 + __popc(peers & lanemask_lt());
      if (slot < a.list_cap[bin]) a.list[bin][slot] = (uint32_t)i;
      else overflow = true;
    }
    if (overflow) atomicOr(&a.ctrl->bad, 1u);
  }
}

// ------------------------------------------------------------------------------------------------
// the sorts of short segments
// ------------------------------------------------------------------------------------------------
struct SegSortArgs {
  StreamSet ss;                 // the caller's arrays (buf[0]); streams[0] carries the key at byte offset 0
  KeyOrder ko;
  const int64_t *offsets;
  const uint32_t *list;         // segment ids of this bin
  uint32_t count;               // entries in `list`
  uint32_t *ticket;             // medium: next entry to take
};

template <typename T>
__device__ __forceinline__ void seg_warp_move(unsigned char *buf, int64_t start, int len, uint32_t cpe, uint32_t c, int dest, int lane) {
  T *col = reinterpret_cast<T *>(buf) + (size_t)start * cpe + c;
  T v;
  if (lane < len) v = col[(size_t)lane * cpe];
  __syncwarp();
  if (lane < len) col[(size_t)dest * cpe] = v;
  __syncwarp();
}

// One warp per segment of 2..32 records: every lane holds one ordered key, its destination is the number of keys
// that sort before it (ties by position), and every column moves through registers, in place.
template <int KB>
__global__ void __launch_bounds__(SEG_TINY_THREADS) seg_tiny_kernel(const __grid_constant__ SegSortArgs a) {
  using O = typename OrdOf<KB>::type;
  const int lane = threadIdx.x & 31;
  const Stream &ks = a.ss.streams[0];
  const uint32_t key_stride = ks.chunk_bytes * ks.chunks_per_elem;
  for (int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < a.count; w += ((int64_t)gridDim.x * blockDim.x) >> 5) {
    const uint32_t seg = a.list[w];
    const int64_t start = a.offsets[seg];
    const int len = (int)(a.offsets[seg + 1] - start);
    const O mine = lane < len ? to_ordered<KB, false>(load_key<KB>(ks.buf[0], start + lane, key_stride), a.ko) : (O)0;
    int dest = 0;
    for (int q = 0; q < len; q++) {
      const O o = __shfl_sync(0xffffffffu, mine, q);
      dest += (o < mine || (o == mine && q < lane)) ? 1 : 0;
    }
    if (!__any_sync(0xffffffffu, lane < len && dest != lane)) continue;  // already in order
    for (int s = 0; s < a.ss.n_streams; s++) {
      const Stream &st = a.ss.streams[s];
      for (uint32_t c = 0; c < st.chunks_per_elem; c++) {
        switch (st.chunk_bytes) {
          case 1: seg_warp_move<uint8_t>(st.buf[0], start, len, st.chunks_per_elem, c, dest, lane); break;
          case 2: seg_warp_move<uint16_t>(st.buf[0], start, len, st.chunks_per_elem, c, dest, lane); break;
          case 4: seg_warp_move<uint32_t>(st.buf[0], start, len, st.chunks_per_elem, c, dest, lane); break;
          case 8: seg_warp_move<uint64_t>(st.buf[0], start, len, st.chunks_per_elem, c, dest, lane); break;
          default: seg_warp_move<uint4>(st.buf[0], start, len, st.chunks_per_elem, c, dest, lane); break;
        }
      }
    }
  }
}

// bytes of dynamic shared memory of seg_medium_kernel: two (ordered key, u16 index) buffers, the per-warp digit
// counters (u16) and the digit bases
template <int KB>
constexpr size_t seg_smem_bytes(int log_cap) {
  return (size_t)2 * (sizeof(typename OrdOf<KB>::type) + 2) * ((size_t)1 << log_cap) + (size_t)(seg_threads(log_cap) / 32) * RADIX * 2 + RADIX * 4;
}
static_assert(seg_smem_bytes<4>(SEG_CAP_LOG2_NARROW) <= 227 * 1024 && seg_smem_bytes<8>(SEG_CAP_LOG2_WIDE) <= 227 * 1024,
              "CAP exceeds the shared memory of one CTA");

// one column of the segment: read whole into the stage (the key buffers, free after the sort), then written
// back in sorted order -- safe in place
template <typename T, int THREADS>
__device__ __forceinline__ void seg_block_move(unsigned char *buf, int64_t start, int len, uint32_t cpe, uint32_t c, const uint16_t *perm,
                                               void *stage_raw) {
  T *col = reinterpret_cast<T *>(buf) + (size_t)start * cpe + c;
  T *stage = reinterpret_cast<T *>(stage_raw);
  for (int i = threadIdx.x; i < len; i += THREADS) stage[i] = col[(size_t)i * cpe];
  __syncthreads();
  for (int r = threadIdx.x; r < len; r += THREADS) col[(size_t)r * cpe] = stage[perm[r]];
  __syncthreads();
}

// One CTA per segment of up to 2^LOG_CAP records (persistent: CTAs take the bin's segments by ticket).  Warp w
// ranks positions [w * 32 * IPT, (w + 1) * 32 * IPT) in position order, which keeps every pass stable.
template <int KB, int LOG_CAP>
__global__ void __launch_bounds__(seg_threads(LOG_CAP)) seg_medium_kernel(const __grid_constant__ SegSortArgs a) {
  using O = typename OrdOf<KB>::type;
  constexpr int CAP = 1 << LOG_CAP, THREADS = seg_threads(LOG_CAP), IPT = CAP / THREADS, NW = THREADS / 32;
  extern __shared__ __align__(16) unsigned char seg_smem[];
  O *const s_key = reinterpret_cast<O *>(seg_smem);                         // [2][CAP]
  uint16_t *const s_idx = reinterpret_cast<uint16_t *>(s_key + 2 * CAP);      // [2][CAP]
  uint16_t *const s_cnt = s_idx + 2 * CAP;                                  // [NW][RADIX]
  uint32_t *s_dbase = reinterpret_cast<uint32_t *>(s_cnt + NW * RADIX);  // [RADIX]
  __shared__ uint32_t s_ticket;
  __shared__ O s_or[NW], s_and[NW];  // per warp

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const Stream &ks = a.ss.streams[0];
  const uint32_t key_stride = ks.chunk_bytes * ks.chunks_per_elem;
  for (;;) {
    if (threadIdx.x == 0) s_ticket = atomicAdd(a.ticket, 1u);
    __syncthreads();
    const uint32_t t = s_ticket;
    if (t >= a.count) return;
    const uint32_t seg = a.list[t];
    const int64_t start = a.offsets[seg];
    const int len = (int)(a.offsets[seg + 1] - start);

    // load: ordered keys + local index; OR / AND over the segment tell which digits vary
    O kor = 0, kand = ~(O)0;
    for (int i = threadIdx.x; i < len; i += THREADS) {
      const O k = to_ordered<KB, false>(load_key<KB>(ks.buf[0], start + i, key_stride), a.ko);
      s_key[i] = k;
      s_idx[i] = (uint16_t)i;
      kor |= k;
      kand &= k;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      kor |= __shfl_xor_sync(0xffffffffu, kor, o);
      kand &= __shfl_xor_sync(0xffffffffu, kand, o);
    }
    if (lane == 0) {
      s_or[warp] = kor;
      s_and[warp] = kand;
    }
    __syncthreads();
    kor = 0;
    kand = ~(O)0;
    for (int w = 0; w < NW; w++) {
      kor |= s_or[w];
      kand &= s_and[w];
    }
    const O vary = kor ^ kand;

    int sel = 0;  // the (key, index) buffer that holds the current order
    for (int d = 0; d < KB; d++) {
      const int shift = d * RADIX_BITS;
      if (((vary >> shift) & (RADIX - 1)) == 0) continue;  // constant digit: the pass would not move anything
      uint16_t *cnt = s_cnt + warp * RADIX;
      for (int b = lane; b < RADIX; b += 32) cnt[b] = 0;
      __syncwarp();
      // warp-local stable ranking, item j of lane l = position warp * 32 * IPT + 32 j + l
      int off[IPT];
#pragma unroll
      for (int j = 0; j < IPT; j++) {
        const int p = warp * 32 * IPT + j * 32 + lane;
        const uint32_t dg = p < len ? (uint32_t)(s_key[sel * CAP + p] >> shift) & (RADIX - 1) : (uint32_t)RADIX;  // RADIX: no record
        const unsigned peers = digit_peers<true>(dg);
        const int rank = __popc(peers & lanemask_lt());
        const int base = dg < RADIX ? cnt[dg] : 0;
        __syncwarp();
        if (rank == 0 && dg < RADIX) cnt[dg] = (uint16_t)(base + __popc(peers));
        __syncwarp();
        off[j] = base + rank;
      }
      __syncthreads();
      // bases: digit-major, warp-minor exclusive prefix
      for (int b = threadIdx.x; b < RADIX; b += THREADS) {
        uint32_t run = 0;
        for (int w = 0; w < NW; w++) {
          const uint32_t c = s_cnt[w * RADIX + b];
          s_cnt[w * RADIX + b] = (uint16_t)run;
          run += c;
        }
        s_dbase[b] = run;
      }
      __syncthreads();
      if (warp == 0) {
        uint32_t v[RADIX / 32], sum = 0;
#pragma unroll
        for (int e = 0; e < RADIX / 32; e++) { v[e] = s_dbase[lane * (RADIX / 32) + e]; sum += v[e]; }
        uint32_t incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
          if (lane >= o) incl += y;
        }
        uint32_t run = incl - sum;
#pragma unroll
        for (int e = 0; e < RADIX / 32; e++) { s_dbase[lane * (RADIX / 32) + e] = run; run += v[e]; }
      }
      __syncthreads();
#pragma unroll
      for (int j = 0; j < IPT; j++) {
        const int p = warp * 32 * IPT + j * 32 + lane;
        if (p < len) {
          const O k = s_key[sel * CAP + p];
          const uint32_t dg = (uint32_t)(k >> shift) & (RADIX - 1);
          const int dst = (int)s_dbase[dg] + s_cnt[warp * RADIX + dg] + off[j];
          s_key[(sel ^ 1) * CAP + dst] = k;
          s_idx[(sel ^ 1) * CAP + dst] = s_idx[sel * CAP + p];
        }
      }
      __syncthreads();
      sel ^= 1;
    }

    const uint16_t *perm = s_idx + sel * CAP;
    bool moved = false;
    for (int r = threadIdx.x; r < len; r += THREADS) moved = moved || perm[r] != r;
    if (__syncthreads_or(moved)) {
      void *stage = seg_smem;  // both key buffers: room for CAP 8-byte chunks
      for (int s = 0; s < a.ss.n_streams; s++) {
        const Stream &st = a.ss.streams[s];
        const uint32_t cpe = st.chunks_per_elem;
        for (uint32_t c = 0; c < cpe; c++) {
          switch (st.chunk_bytes) {
            case 1: seg_block_move<uint8_t, THREADS>(st.buf[0], start, len, cpe, c, perm, stage); break;
            case 2: seg_block_move<uint16_t, THREADS>(st.buf[0], start, len, cpe, c, perm, stage); break;
            case 4: seg_block_move<uint32_t, THREADS>(st.buf[0], start, len, cpe, c, perm, stage); break;
            case 8: seg_block_move<uint64_t, THREADS>(st.buf[0], start, len, cpe, c, perm, stage); break;
            default:  // 16-byte chunks as two 8-byte halves (the stage holds CAP 8-byte values)
              seg_block_move<uint64_t, THREADS>(st.buf[0], start, len, cpe * 2, c * 2, perm, stage);
              seg_block_move<uint64_t, THREADS>(st.buf[0], start, len, cpe * 2, c * 2 + 1, perm, stage);
              break;
          }
        }
      }
    }
    __syncthreads();  // s_ticket, s_or, s_and and the buffers are reused by the next segment
  }
}

// ------------------------------------------------------------------------------------------------
// keys of <= 4 bytes with a segment longer than CAP: one sort of u64 composite keys over the whole range
// ------------------------------------------------------------------------------------------------
// the inverse of to_ordered<KB, false>: raw key bits from ordered ones (sub = 0, lshift = 0).  With t = u ^
// xor_const, t = k ^ (sign(k) ? neg_xor : 0), and neg_xor leaves the sign bit alone, so sign(t) = sign(k).
template <int KB>
__device__ __forceinline__ typename UIntOf<KB>::type from_ordered(typename OrdOf<KB>::type u, const KeyOrder &ko) {
  using O = typename OrdOf<KB>::type;
  const O t = u ^ (O)ko.xor_const;
  const O neg = (O)0 - ((t >> (8 * KB - 1)) & 1);
  return (typename UIntOf<KB>::type)(t ^ (neg & (O)ko.neg_xor));
}

struct SegCompositeArgs {
  unsigned char *keys;          // the caller's key (or record) array
  uint32_t key_stride;
  const int64_t *offsets;
  int64_t n_segments;
  int64_t first, span;          // records [first, first + span) = [offsets[0], offsets[n_segments])
  KeyOrder ko;
  unsigned long long *comp;     // [span] (segment index << 8 KB) | ordered key
};

template <int KB>  // (KB <= 4)
__global__ void __launch_bounds__(256) seg_pack_kernel(const __grid_constant__ SegCompositeArgs a) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.span; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = a.first + i;
    int64_t lo = 0, hi = a.n_segments - 1;  // the last segment that starts at or before r
    while (lo < hi) {
      const int64_t mid = (lo + hi + 1) >> 1;
      if (a.offsets[mid] <= r) lo = mid; else hi = mid - 1;
    }
    a.comp[i] = ((unsigned long long)lo << (8 * KB)) | (unsigned long long)to_ordered<KB, false>(load_key<KB>(a.keys, r, a.key_stride), a.ko);
  }
}

// SoA: the caller's keys back from the sorted composite keys
template <int KB>
__global__ void __launch_bounds__(256) seg_unpack_kernel(const __grid_constant__ SegCompositeArgs a) {
  using K = typename UIntOf<KB>::type;
  using O = typename OrdOf<KB>::type;
  constexpr unsigned long long LOW = (1ull << (8 * KB)) - 1;
  K *keys = reinterpret_cast<K *>(a.keys) + a.first;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.span; i += (int64_t)gridDim.x * blockDim.x)
    keys[i] = from_ordered<KB>((O)(a.comp[i] & LOW), a.ko);
}

// seg_medium_kernel<KB, LOG_CAP> for the bins LOG_CAP = 6 .. seg_cap_log2(KB) (segmented_inst.cu)
struct SegMediumKernel { void (*fn)(SegSortArgs); int threads; size_t smem; };
SegMediumKernel seg_medium_kernel_of(int kb, int log_cap);

}  // namespace b200sort
