// unique.cuh -- the run compaction of unique (b200sort_unique): the distinct keys of an array, their counts and the
// inverse map.  Included by b200sort.cu; the host side is unique_host.cuh.
//
// The keys arrive sorted (a copy in the workspace, sorted together with its positions by sort_device) or, in
// consecutive mode, as the caller's array in input order.  Either way every run of equal adjacent keys is one entry,
// and one pass finds them:
//
//   unique_scan_kernel    one tile of UNQ_TILE keys per CTA, taken by ticket.  Every key is compared with its
//                         predecessor (bit patterns): a difference, or position 0, makes it the head of a run.  The
//                         heads are counted with warp ballots, then across the CTA's warps, then across tiles by a
//                         decoupled look-back on ONE status word per tile (the LB_FLAG_* encoding of kernels.cuh,
//                         tag 0: the words are zeroed per call).  That gives every key its run id.  Heads write
//                         out_keys[run] and start[run] = position; every key writes its inverse, out_inverse[position]
//                         = run (consecutive mode) or out_inverse[index[position]] = run (after the sort: a scatter).
//                         The last tile writes U and start[U] = num.
//   unique_counts_kernel  counts[j] = start[j + 1] - start[j] for j < U, U read on the device.  Keeping this apart
//                         spares the scan kernel any cross-tile "where does the previous run start" protocol.
//
// Static shared memory only: a kernel with dynamic shared memory would add a reservation to every kernel of the module.
#pragma once
#include "kernels.cuh"

namespace b200sort {

constexpr int UNQ_THREADS = 256;
constexpr int UNQ_ITEMS = 16;                          // keys per thread
constexpr int UNQ_TILE = UNQ_THREADS * UNQ_ITEMS;      // keys per tile (one ticket): 4096
constexpr int UNQ_WARP_KEYS = 32 * UNQ_ITEMS;          // keys per warp, contiguous

struct UniqueArgs {
  const unsigned char *keys;  // the sorted copy, or the caller's keys (consecutive mode)
  const void *index;          // after the sort: the input position of every sorted key (u32 or u64); else nullptr
  int64_t num;
  int64_t n_tiles;
  uint32_t vec;               // keys are 16-byte aligned: full tiles are read in 16-byte vectors
  void *out_keys;             // [U] the first key of every run
  int64_t *out_inverse;       // [num] run of every key, or nullptr
  int64_t *start;             // [U + 1] position of every run's first key, then num; nullptr without counts
  int64_t *out_num_unique;    // U
  uint32_t *ticket;           // tile tickets (zeroed per call)
  uint64_t *status;           // [n_tiles] look-back status words (zeroed per call)
};

// IDX: 0 -- the inverse of key i is written at i (consecutive mode, or no inverse); 4 / 8 -- at index[i], of that
// many bytes (after the sort)
template <int KB, int IDX>
__global__ void __launch_bounds__(UNQ_THREADS) unique_scan_kernel(const __grid_constant__ UniqueArgs a) {
  using K = typename UIntOf<KB>::type;
  using S = typename std::conditional<KB == 8, unsigned long long, uint32_t>::type;  // what a shuffle moves
  constexpr int VEC = 16 / KB;           // keys per 16-byte vector
  constexpr int NV = UNQ_ITEMS / VEC;    // rounds: in round r lane l holds keys (r * 32 + l) * VEC .. + VEC - 1 of its warp
  constexpr unsigned FULL = 0xffffffffu;
  static_assert(UNQ_ITEMS % VEC == 0 && VEC <= 32, "a thread's keys are whole vectors");
  __shared__ uint32_t s_tile;
  __shared__ uint32_t s_warp[UNQ_THREADS / 32];
  __shared__ unsigned long long s_base;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_tile = atomicAdd(a.ticket, 1u);
  __syncthreads();
  const int64_t tile = s_tile;
  const int64_t wbase = tile * UNQ_TILE + (int64_t)warp * UNQ_WARP_KEYS;  // this warp's first key
  auto pos_of = [&](int r, int j) { return wbase + (int64_t)(r * 32 + lane) * VEC + j; };

  // ---- load: 16-byte vectors when the whole tile exists and the array allows it, else key by key
  K k[NV][VEC];
  if (a.vec && (tile + 1) * UNQ_TILE <= a.num) {
#pragma unroll
    for (int r = 0; r < NV; r++) {
      union { uint4 v; K e[VEC]; } u;
      u.v = *reinterpret_cast<const uint4 *>(a.keys + (size_t)pos_of(r, 0) * KB);
#pragma unroll
      for (int j = 0; j < VEC; j++) k[r][j] = u.e[j];
    }
  } else {
#pragma unroll
    for (int r = 0; r < NV; r++)
#pragma unroll
      for (int j = 0; j < VEC; j++) {
        const int64_t p = pos_of(r, j);
        k[r][j] = p < a.num ? load_key<KB>(a.keys, p, KB) : (K)0;
      }
  }

  // ---- heads: bit j of head[r] is set when key (r, j) exists and differs from its predecessor (or is key 0).
  //      off[r]: heads of this warp before round r's keys of this lane.
  uint32_t head[NV], off[NV];
  uint32_t wcount = 0;  // heads of this warp so far
  K before = 0;         // the key just before the warp's first one
  if (lane == 0 && wbase > 0 && wbase < a.num) before = load_key<KB>(a.keys, wbase - 1, KB);
#pragma unroll
  for (int r = 0; r < NV; r++) {
    S prev = __shfl_up_sync(FULL, (S)k[r][VEC - 1], 1);
    const S last_of_prev_round = __shfl_sync(FULL, (S)k[r > 0 ? r - 1 : 0][VEC - 1], 31);
    if (lane == 0) prev = r == 0 ? (S)before : last_of_prev_round;
    uint32_t h = 0;
#pragma unroll
    for (int j = 0; j < VEC; j++) {
      const int64_t p = pos_of(r, j);
      const K pred = j == 0 ? (K)prev : k[r][j - 1];
      if (p < a.num && (p == 0 || k[r][j] != pred)) h |= 1u << j;
    }
    head[r] = h;
    uint32_t before_me = 0, total = 0;
#pragma unroll
    for (int j = 0; j < VEC; j++) {
      const unsigned b = __ballot_sync(FULL, (h >> j) & 1u);
      before_me += __popc(b & lanemask_lt());
      total += __popc(b);
    }
    off[r] = wcount + before_me;
    wcount += total;
  }
  if (lane == 0) s_warp[warp] = wcount;
  __syncthreads();

  // ---- this tile's heads, and those of all tiles before it (look-back by warp 0, 32 predecessors per round trip)
  uint32_t wexcl = 0, agg = 0;
#pragma unroll
  for (int w = 0; w < UNQ_THREADS / 32; w++) {
    wexcl += w < warp ? s_warp[w] : 0u;
    agg += s_warp[w];
  }
  if (warp == 0) {
    unsigned long long excl = 0;
    if (tile == 0) {
      if (lane == 0) st_relaxed_u64(&a.status[0], LB_FLAG_PREFIX | agg);
    } else {
      if (lane == 0) st_relaxed_u64(&a.status[tile], LB_FLAG_AGG | agg);
      int64_t t = tile - 1;  // lane l looks at tile t - l
      for (;;) {
        const int64_t q = t - lane;
        uint64_t w;
        do {
          w = q >= 0 ? ld_relaxed_u64(&a.status[q]) : LB_FLAG_PREFIX;
        } while (__any_sync(FULL, (w & LB_FLAG_MASK) == 0));
        const unsigned pre = __ballot_sync(FULL, (w & LB_FLAG_MASK) == LB_FLAG_PREFIX);
        const int stop = pre ? __ffs(pre) - 1 : 31;  // lanes 0 .. stop contribute (the nearest prefix ends the walk)
        unsigned long long v = lane <= stop ? (w & LB_VALUE_MASK) : 0ull;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(FULL, v, d);
        excl += v;
        if (pre) break;
        t -= 32;
      }
      if (lane == 0) st_relaxed_u64(&a.status[tile], LB_FLAG_PREFIX | (excl + agg));
    }
    if (lane == 0) {
      s_base = excl;
      if (tile == a.n_tiles - 1) {
        *a.out_num_unique = (int64_t)(excl + agg);
        if (a.start) a.start[excl + agg] = a.num;
      }
    }
  }
  __syncthreads();

  // ---- outputs: run id of key (r, j) = heads up to and including it, minus one
  const int64_t base = (int64_t)s_base + wexcl;
  K *out_keys = reinterpret_cast<K *>(a.out_keys);
#pragma unroll
  for (int r = 0; r < NV; r++) {
    const bool vec_out = IDX == 0 && a.out_inverse && VEC % 2 == 0 && ((uintptr_t)a.out_inverse & 15) == 0 && pos_of(r, VEC - 1) < a.num;
    int64_t run[VEC];
#pragma unroll
    for (int j = 0; j < VEC; j++) {
      const int64_t p = pos_of(r, j);
      run[j] = base + off[r] + __popc(head[r] & ((2u << j) - 1u)) - 1;
      if ((head[r] >> j) & 1u) {
        out_keys[run[j]] = k[r][j];
        if (a.start) a.start[run[j]] = p;
      }
      if (a.out_inverse && !vec_out && p < a.num) {
        if constexpr (IDX == 0) a.out_inverse[p] = run[j];
        else if constexpr (IDX == 4) a.out_inverse[static_cast<const uint32_t *>(a.index)[p]] = run[j];
        else a.out_inverse[static_cast<const unsigned long long *>(a.index)[p]] = run[j];
      }
    }
    if constexpr (VEC % 2 == 0) {
      if (vec_out)  // (16-byte stores of consecutive positions: pos_of(r, 0) is a multiple of VEC, so even)
#pragma unroll
        for (int j = 0; j < VEC; j += 2)
          *reinterpret_cast<longlong2 *>(a.out_inverse + pos_of(r, j)) = make_longlong2(run[j], run[j + 1]);
    }
  }
}

__global__ void __launch_bounds__(256) unique_counts_kernel(const int64_t *__restrict__ start, const int64_t *__restrict__ n_unique,
                                                            int64_t *__restrict__ counts) {
  const int64_t u = *n_unique;
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < u; j += (int64_t)gridDim.x * blockDim.x)
    counts[j] = start[j + 1] - start[j];
}

// the positions 0 .. n - 1 as u64 (iota_kernel writes u32, which covers n <= 2^32)
__global__ void __launch_bounds__(256) unique_iota64_kernel(unsigned long long *idx, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    idx[i] = (unsigned long long)i;
}

}  // namespace b200sort
