// topk.cuh -- top-k selection: the k smallest or largest records of every row by radix select
// (b200sort_topk_soa / _aos).  Included at the end of b200sort.cu (it uses that file's internals); the host side is
// topk_host.cuh.
//
// The keys are order-mapped with make_key_order(key_type, !largest), so the k largest are the k smallest ordered
// keys and one code path serves both directions.  Digits are 8 bits of the ordered key, most significant first.
//
//   pass 0      counts digit 0 of every record of the row;
//   decision d  (one CTA per row) scans the histogram of digit d and picks the bucket where the k-th record falls.
//               The top d + 1 digits of the threshold key, T, are then known; k_left drops by the records below
//               the bucket.  It also lists the next pass's work items (row, chunk) for the persistent CTAs;
//   pass p >= 1 takes every candidate of pass p - 1 (top p - 1 digits equal those of T): top p digits below T:
//               selected, emitted to the row's next output slot; equal: still a candidate -- kept, as (ordered key,
//               position), in a candidate buffer for pass p + 1, and digit p counted.
// A row is finished by the pass after the decision that finds its bucket must be taken whole, or that decides
// the last digit: that pass emits the records below T and the first k_left of those equal to T (an atomic ticket),
// and later passes skip the row.
//
// The decision is a kernel of its own rather than the last CTA of a row to finish: it needs no cross-CTA
// arrival protocol, it runs after every histogram contribution of every row by stream order, and it is the point
// where the next pass's work list is made.  For the same reason one histogram per row suffices: the decision reads
// and clears it before the next pass starts.
//
// Candidate buffers: two per row (pass p writes buffer p & 1, pass p + 1 reads it), each of
// TOPK_CAP(row_len) = ceil(row_len / 16) entries.  Pass p writes its candidates only if they fit, which the decision
// before it knows (the count of the chosen bucket); otherwise pass p + 1 re-reads the row and filters on T.  Uniform
// keys cost two reads of the keys (pass 0 and pass 1) and a read of ~N/256 candidates; adversarial keys (all
// equal, a constant top byte) at most key-width + 1 reads of the keys.
#pragma once
#include "kernels.cuh"
#include "segmented.cuh"  // (from_ordered)

namespace b200sort {

constexpr int TOPK_THREADS = 256;
constexpr int TOPK_CHUNK = 8192;      // records (or candidate entries) of one work item
constexpr int TOPK_CAP_DIV = 16;      // candidate buffer entries per row: ceil(row_len / 16)
constexpr int TOPK_PASS_CTAS_PER_SM = 3;  // (the register budget of the pass kernel without spills)
enum TopkMode : uint32_t { TOPK_ACTIVE = 0, TOPK_LAST = 1, TOPK_DONE = 2 };

__host__ __device__ constexpr int64_t topk_cap(int64_t row_len) { return (row_len + TOPK_CAP_DIV - 1) / TOPK_CAP_DIV; }

// per-row state, zeroed by the host, k_left set by topk_init_kernel; written by the decisions, read by the passes
struct TopkRow {
  unsigned long long T;         // decided top digits of the ordered threshold key
  unsigned long long k_left;    // records still to select
  unsigned long long cand;      // records whose top digits equal T: what the running pass keeps as candidates
  unsigned long long src_n;     // candidate-buffer entries the running pass reads (in_buf)
  unsigned long long out_ctr;   // next output slot
  unsigned long long tie_ctr;   // records equal to T seen by the finishing pass
  unsigned long long wr_ctr;    // entries the running pass has written to its candidate buffer
  unsigned long long item_base; // first work item of the running pass (its items are item_base ...)
  uint32_t mode;                // TopkMode of the running pass
  uint32_t in_buf;              // the running pass reads the candidate buffer (else the row)
  uint32_t write_buf;           // the running pass writes its candidates to the candidate buffer
  uint32_t pad_;
};

struct TopkCtrl {
  unsigned long long items[MAX_PASSES];  // work items of pass p (p >= 1), counted up by the decision before it
};
static_assert(sizeof(TopkRow) == 80 && sizeof(TopkCtrl) == 8 * MAX_PASSES, "mirrored by tests/topk_model.py");

struct TopkArgs {
  const unsigned char *keys;   // the input's keys (SoA keys, or AoS records with the key at offset 0)
  uint32_t stride;             // bytes between consecutive keys
  uint32_t n_rows;
  int64_t row_len, k, cap;     // cap: candidate-buffer entries per row
  int64_t chunks_per_row;      // work items of one row in pass 0
  KeyOrder ko;
  TopkRow *rows;
  unsigned long long *hist;    // [n_rows][RADIX]
  TopkCtrl *ctrl;
  uint32_t *item_row;          // row of every work item of the running pass
  void *cand_key[2];           // [n_rows][cap] ordered keys ...
  unsigned long long *cand_pos[2];  // ... and their positions in the row
  void *out_keys;              // [n_rows][k] raw keys of the selected records, in no particular order
  int64_t *out_index;          // [n_rows][k] their positions
  int64_t *offsets;            // [n_rows + 1] r * k (the segments of the ordering step)
  int pass;
};

__global__ void __launch_bounds__(256) topk_init_kernel(TopkArgs a) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r <= (int64_t)a.n_rows; r += (int64_t)gridDim.x * blockDim.x) {
    a.offsets[r] = r * a.k;
    if (r < a.n_rows) a.rows[r].k_left = (unsigned long long)a.k;
  }
}

// Pass a.pass over the work items of this pass: persistent CTAs, grid-stride over the items.  The shared-memory
// histogram collects one row's counts and is added to the row's global histogram when the CTA moves to another row.
// It has one counter per (digit, lane): bins[d * 32 + lane] lies in bank `lane`, so the lanes of a warp never
// contend, however few digits the keys have (the top byte of normally distributed floats takes about four values).
template <int KB>
__global__ void __launch_bounds__(TOPK_THREADS, TOPK_PASS_CTAS_PER_SM) topk_pass_kernel(const __grid_constant__ TopkArgs a) {
  using O = typename OrdOf<KB>::type;
  using K = typename UIntOf<KB>::type;
  constexpr int VEC = 16 / KB;                                     // keys per 16-byte vector
  // vectors in flight per thread: 8 for 4-byte keys, 4 for 8-byte keys, 16 keys' worth for 1- and 2-byte keys (more
  // spill registers at 3 CTAs per SM)
  constexpr int NLD_MAX = KB == 8 ? 4 : (KB == 4 ? 8 : 16 / VEC);
  constexpr int NLD = (TOPK_CHUNK / VEC / TOPK_THREADS) < NLD_MAX ? (TOPK_CHUNK / VEC / TOPK_THREADS) : NLD_MAX;
  __shared__ uint32_t bins[RADIX * 32];
  __shared__ unsigned long long s_warp[TOPK_THREADS / 32], s_base[2];  // (reserve)
  const int p = a.pass;
  const unsigned long long n_items = p == 0 ? (unsigned long long)a.n_rows * (unsigned long long)a.chunks_per_row : a.ctrl->items[p];
  const uint32_t lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < RADIX * 32; i += TOPK_THREADS) bins[i] = 0;
  __syncthreads();
  int64_t cur = -1;  // row whose counts `bins` holds
  uint32_t since = 0;  // items counted into `bins` since the last flush (flushed before a counter could wrap)
  auto flush = [&]() {
    __syncthreads();
    for (int d = threadIdx.x; d < RADIX; d += TOPK_THREADS) {
      uint32_t c = 0;
      for (int l = 0; l < 32; l++) {  // (lanes in rotated order: the threads of a warp read 32 different banks)
        uint32_t &b = bins[d * 32 + ((l + d) & 31)];
        c += b;
        b = 0;
      }
      if (c) atomicAdd(&a.hist[(size_t)cur * RADIX + d], (unsigned long long)c);
    }
    __syncthreads();
  };
  for (unsigned long long item = blockIdx.x; item < n_items; item += gridDim.x) {
    int64_t row, chunk;
    if (p == 0) { row = (int64_t)(item / a.chunks_per_row); chunk = (int64_t)(item % a.chunks_per_row); }
    else { row = a.item_row[item]; chunk = (int64_t)(item - a.rows[row].item_base); }
    if (row != cur || since == (1u << 31) / TOPK_CHUNK) {
      if (cur >= 0) flush();
      cur = row;
      since = 0;
    }
    since++;
    TopkRow &rs = a.rows[row];
    const uint32_t mode = p == 0 ? TOPK_ACTIVE : rs.mode;
    const bool in_buf = p > 0 && rs.in_buf != 0;
    const bool write_buf = p > 0 && rs.write_buf != 0;
    const O T = (O)rs.T;
    const unsigned long long k_left = rs.k_left;
    const int64_t len = in_buf ? (int64_t)rs.src_n : a.row_len;
    const int64_t start = chunk * TOPK_CHUNK, end = start + TOPK_CHUNK < len ? start + TOPK_CHUNK : len;
    O *const ckey = (O *)a.cand_key[p & 1] + (size_t)row * a.cap;
    unsigned long long *const cpos = a.cand_pos[p & 1] + (size_t)row * a.cap;
    K *const okey = (K *)a.out_keys + (size_t)row * a.k;
    int64_t *const oidx = a.out_index + (size_t)row * a.k;
    const int hi_shift = 8 * (KB - (p > 0 ? p : 1));  // (p == 0: unused)
    const int dg_shift = 8 * (KB - 1 - (p < KB ? p : KB - 1));

    // the kind of one record in pass p >= 1: 1 selected (below T), 2 kept as a candidate (finishing pass: equal to T),
    // 0 neither.  count: digit p of the candidates goes into the histogram (pass 0: every record's digit 0)
    auto kind = [&](O o, bool valid, bool count) -> uint32_t {
      if (!valid) return 0;
      if (p == 0) {
        if (count) atomicAdd(&bins[(((uint32_t)(o >> dg_shift) & (RADIX - 1)) << 5) + lane], 1u);
        return 0;
      }
      const O H = o >> hi_shift;
      if ((H >> 8) != (T >> 8)) return 0;
      if (H < T) return 1;
      if (H != T) return 0;
      if (mode == TOPK_LAST) return 2;
      if (count) atomicAdd(&bins[(((uint32_t)(o >> dg_shift) & (RADIX - 1)) << 5) + lane], 1u);
      return write_buf ? 2u : 0u;
    };
    // The first slots of this thread's n1 records of kind 1 (*b1) and n2 of kind 2 (*b2), from one atomic per CTA and
    // counter (a whole row's candidates share one counter: per-warp atomics on it serialise).  Every thread calls it.
    auto reserve = [&](uint32_t n1, uint32_t n2, unsigned long long *b1, unsigned long long *b2) {
      const unsigned long long mine = ((unsigned long long)n1 << 32) | n2;
      unsigned long long x = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xffffffffu, x, o);
        if ((int)lane >= o) x += t;
      }
      if (lane == 31) s_warp[threadIdx.x >> 5] = x;
      __syncthreads();
      unsigned long long before = 0, total = 0;
#pragma unroll
      for (int w = 0; w < TOPK_THREADS / 32; w++) {
        const unsigned long long t = s_warp[w];
        before += w < (int)(threadIdx.x >> 5) ? t : 0ull;
        total += t;
      }
      if (threadIdx.x == 0) {
        const unsigned long long t1 = total >> 32, t2 = total & 0xffffffffull;
        s_base[0] = t1 ? atomicAdd(&rs.out_ctr, t1) : 0ull;
        s_base[1] = t2 ? atomicAdd(mode == TOPK_LAST ? &rs.tie_ctr : &rs.wr_ctr, t2) : 0ull;
      }
      __syncthreads();
      const unsigned long long excl = before + x - mine;
      *b1 = s_base[0] + (excl >> 32);
      *b2 = s_base[1] + (excl & 0xffffffffull);
    };
    // a record of kind kd to its place: kind 1 to the next output slot; kind 2 to the candidate buffer, or in the
    // finishing pass, if its ticket is below k_left, to the output slots after those of every record below T
    auto put = [&](O o, unsigned long long pos, uint32_t kd, unsigned long long *b1, unsigned long long *b2) {
      if (kd == 1) {
        const unsigned long long s1 = (*b1)++;
        okey[s1] = from_ordered<KB>(o, a.ko);
        oidx[s1] = (int64_t)pos;
      } else if (kd == 2) {
        const unsigned long long t = (*b2)++;
        if (mode != TOPK_LAST) {
          ckey[t] = o;
          cpos[t] = pos;
        } else if (t < k_left) {
          const unsigned long long s2 = (unsigned long long)a.k - k_left + t;
          okey[s2] = from_ordered<KB>(o, a.ko);
          oidx[s2] = (int64_t)pos;
        }
      }
    };
    // one record per thread (candidate buffer, or rows that are not 16-byte aligned); every thread calls it
    auto one = [&](O o, unsigned long long pos, bool valid) {
      const uint32_t kd = kind(o, valid, true);
      if (p == 0) return;
      unsigned long long b1, b2;
      reserve(kd == 1 ? 1u : 0u, kd == 2 ? 1u : 0u, &b1, &b2);
      put(o, pos, kd, &b1, &b2);
    };

    if (in_buf) {
      const O *bk = (const O *)a.cand_key[(p - 1) & 1] + (size_t)row * a.cap;
      const unsigned long long *bp = a.cand_pos[(p - 1) & 1] + (size_t)row * a.cap;
      for (int64_t base = start; base < end; base += TOPK_THREADS) {
        const int64_t i = base + threadIdx.x;
        const bool v = i < end;
        one(v ? bk[i] : (O)0, v ? bp[i] : 0ull, v);
      }
    } else {
      const unsigned char *rk = a.keys + (size_t)row * (size_t)a.row_len * a.stride;
      const bool dense = a.stride == (uint32_t)KB && (((uintptr_t)rk) & 15) == 0;
      if (dense && end - start == TOPK_CHUNK) {
        // (whole chunks of a 16-byte aligned row: NLD vectors in flight per thread, one reservation per round)
        const uint4 *v = reinterpret_cast<const uint4 *>(rk + (size_t)start * KB);
        for (int g = 0; g < TOPK_CHUNK / VEC; g += NLD * TOPK_THREADS) {
          uint4 q[NLD];
#pragma unroll
          for (int j = 0; j < NLD; j++) q[j] = v[g + j * TOPK_THREADS + threadIdx.x];
          uint32_t n1 = 0, n2 = 0;
#pragma unroll
          for (int j = 0; j < NLD; j++) {
            K kk[VEC];
            memcpy(kk, &q[j], 16);
#pragma unroll
            for (int e = 0; e < VEC; e++) {
              const uint32_t kd = kind(to_ordered<KB, false>(kk[e], a.ko), true, true);
              n1 += kd == 1;
              n2 += kd == 2;
            }
          }
          if (p == 0) continue;
          unsigned long long b1, b2;
          reserve(n1, n2, &b1, &b2);
          if (n1 + n2 == 0) continue;
#pragma unroll
          for (int j = 0; j < NLD; j++) {
            K kk[VEC];
            memcpy(kk, &q[j], 16);
            const int64_t i0 = start + (int64_t)(g + j * TOPK_THREADS + threadIdx.x) * VEC;
#pragma unroll
            for (int e = 0; e < VEC; e++) {
              const O o = to_ordered<KB, false>(kk[e], a.ko);
              put(o, (unsigned long long)(i0 + e), kind(o, true, false), &b1, &b2);
            }
          }
        }
      } else {
        for (int64_t base = start; base < end; base += TOPK_THREADS) {
          const int64_t i = base + threadIdx.x;
          const bool v = i < end;
          one(v ? to_ordered<KB, false>(load_key<KB>(rk, i, a.stride), a.ko) : (O)0, (unsigned long long)i, v);
        }
      }
    }
  }
  if (cur >= 0) flush();
}

// Decision after pass d (a.pass): one CTA per row (grid-stride over the rows).  Picks the bucket of digit d where the
// k-th record falls, updates the row's state for pass d + 1 and lists that pass's work items.
template <int KB>
__global__ void __launch_bounds__(RADIX) topk_decide_kernel(const __grid_constant__ TopkArgs a) {
  __shared__ unsigned long long warp_sum[RADIX / 32];
  __shared__ unsigned long long s_below, s_cnt;
  __shared__ uint32_t s_b;
  __shared__ unsigned long long s_base, s_chunks;
  const int d = a.pass;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t row = blockIdx.x; row < (int64_t)a.n_rows; row += gridDim.x) {
    TopkRow &rs = a.rows[row];
    const uint32_t mode = rs.mode;
    if (mode == TOPK_DONE) continue;
    if (mode == TOPK_LAST) {  // finished by pass d
      __syncthreads();
      if (threadIdx.x == 0) rs.mode = TOPK_DONE;
      continue;
    }
    // inclusive scan of the 256 counters
    unsigned long long *h = a.hist + (size_t)row * RADIX;
    const unsigned long long c = h[threadIdx.x];
    unsigned long long incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) warp_sum[warp] = incl;
    __syncthreads();
    for (int w = 0; w < warp; w++) incl += warp_sum[w];
    const unsigned long long excl = incl - c;
    const unsigned long long k_left = rs.k_left;
    if (excl < k_left && k_left <= incl) { s_b = threadIdx.x; s_below = excl; s_cnt = c; }
    h[threadIdx.x] = 0;  // (for the next pass)
    __syncthreads();
    if (threadIdx.x == 0) {
      const bool in_buf = rs.write_buf != 0;  // pass d wrote its candidates to the buffer pass d + 1 reads
      const unsigned long long src_n = rs.cand, kl = k_left - s_below, cand = s_cnt;
      const uint32_t next_mode = (cand == kl || d == KB - 1) ? TOPK_LAST : TOPK_ACTIVE;
      rs.T = d == 0 ? (unsigned long long)s_b : ((rs.T << 8) | s_b);
      rs.k_left = kl;
      rs.cand = cand;
      rs.src_n = src_n;
      rs.in_buf = in_buf ? 1u : 0u;
      rs.write_buf = (next_mode == TOPK_ACTIVE && (int64_t)cand <= a.cap) ? 1u : 0u;
      rs.mode = next_mode;
      rs.wr_ctr = 0;
      rs.tie_ctr = 0;
      const int64_t len = in_buf ? (int64_t)src_n : a.row_len;
      const unsigned long long chunks = (unsigned long long)((len + TOPK_CHUNK - 1) / TOPK_CHUNK);
      const unsigned long long base = atomicAdd(&a.ctrl->items[d + 1], chunks);
      rs.item_base = base;
      s_base = base;
      s_chunks = chunks;
    }
    __syncthreads();
    for (unsigned long long i = threadIdx.x; i < s_chunks; i += RADIX) a.item_row[s_base + i] = (uint32_t)row;
    __syncthreads();
  }
}

// The payload streams (or AoS records) of the selected records, in their final order: out[r k + j] = in[r row_len +
// index[r k + j]].  Each stream moves in chunks of its own width (TopkGatherSet).
struct TopkGatherStream {
  const unsigned char *in;
  unsigned char *out;
  uint32_t chunk_bytes, chunks_per_elem;
};
struct TopkGatherSet {
  int n_streams;
  int64_t row_len, k, total;  // total = n_rows * k
  const int64_t *index;
  TopkGatherStream s[MAX_STREAMS];
};

template <typename T>
__device__ __forceinline__ void topk_gather_stream(const TopkGatherSet &g, const TopkGatherStream &s) {
  const int64_t cpe = s.chunks_per_elem, n = g.total * cpe;
  const T *in = (const T *)s.in;
  T *out = (T *)s.out;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = t / cpe, c = t - i * cpe;
    const int64_t r = i / g.k;
    out[t] = in[(r * g.row_len + g.index[i]) * cpe + c];
  }
}

__global__ void __launch_bounds__(256) topk_gather_kernel(const __grid_constant__ TopkGatherSet g) {
  for (int s = 0; s < g.n_streams; s++) {
    switch (g.s[s].chunk_bytes) {
      case 16: topk_gather_stream<uint4>(g, g.s[s]); break;
      case 8: topk_gather_stream<uint64_t>(g, g.s[s]); break;
      case 4: topk_gather_stream<uint32_t>(g, g.s[s]); break;
      case 2: topk_gather_stream<uint16_t>(g, g.s[s]); break;
      default: topk_gather_stream<uint8_t>(g, g.s[s]); break;
    }
  }
}

}  // namespace b200sort
