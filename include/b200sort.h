/*
 * b200sort.h -- C ABI of libb200sort.so, the B200 (sm_100a) key + payload sort that replaces the hot
 * path of jonicho/simd-radix-sort.
 *
 * The reference has no FFI layer: its boundary is the C++20 function-template signature
 *     simd_sort::radix_sort::sort<Up>(num, keys, payloads...)            (radixSort.hpp:1780-1783)
 *     simd_sort::radix_sort::sort<Up>(num, DataElement<K, Ps...>*)       (radixSort.hpp:1770-1778)
 * include/b200sort/radixSort.hpp re-declares exactly those templates and forwards every
 * instantiation, type-erased, to the entry points below.  Anything else (ctypes, cgo, JNI ...) binds
 * the same symbols; INTEGRATION.md shows the stubs.
 *
 * Conventions
 *  - plain pointers and sizes only; no C++/torch types.
 *  - every array may live in HOST memory (sorted through a staged copy on the current CUDA device) or
 *    in DEVICE memory (sorted in place on the device that owns it: the fast path).  All arrays of
 *    one call must be on the same side.  The exceptions are the top-k selection and unique, which take device arrays
 *    only (B200SORT_EUNSUPPORTED otherwise): staging a whole row over PCIe to return k records of it is the wrong tool,
 *    and unique returns results whose size only the device knows.
 *  - the sort is in place from the caller's point of view (reference: radix_sort.hpp:297-337): the
 *    result overwrites keys/payloads/records.  Scratch (one shadow copy of every stream + per-tile
 *    status words) comes from `workspace` or, when that is NULL, from a per-device cache owned by
 *    the library.  Sorts that use that cache (and all host-memory calls, which stage through a cached
 *    buffer) are serialised per device by the library; give concurrent sorts of device arrays their own
 *    workspaces.  Both cached buffers are kept until b200sort_release_cache().
 *  - return value: 0 on success, a negative B200SORT_E* code otherwise; b200sort_last_error() gives
 *    a thread-local human-readable message.  There is NO CPU fallback: without a usable CUDA device
 *    every sort call fails with B200SORT_ECUDA.
 *  - `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream).  Host-memory calls
 *    return after the data is back.  Device-memory calls are ordered on that stream; whether the call
 *    itself waits for the device depends on the size:
 *      * fewer than 2^24 records, keys of <= 4 bytes (or 8-byte keys below 2^22 records): asynchronous;
 *      * 8-byte keys from 2^22 records (MSB hybrid plan): returns when the sort is complete (one wait at
 *        the end: the device-made plan may ask the host for the digit-by-digit fall-back);
 *      * any sort of >= 2^24 records: additionally waits once, early, for the 200-byte pass plan made
 *        on the device, so that only the passes that execute are launched.
 *      * a segmented sort: one wait for the segment classification, two with 8-byte keys and a segment
 *        longer than 8192 records, plus the waits above of the whole-array sorts it runs for long segments.
 *      * a top-k: the selection waits for nothing; its ordering step is a segmented sort of n_rows segments of
 *        k records and adds that sort's waits (one; more with 8-byte keys and k > 8192; none when k = 1).
 *      * a unique: consecutive mode waits for nothing; sorted mode adds the waits of the whole-array sort of num
 *        records it runs.
 *    These calls therefore cannot be captured into a CUDA graph; everything between the two waits
 *    (all passes, the junction kernel, the flag-gated segment finish / copy-back) is queued without one.
 *  - device arrays are sorted on the device that owns them, whatever the caller's current device is;
 *    all arrays of one call must live on the same device.
 */
#ifndef B200SORT_H_
#define B200SORT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200SORT_VERSION 100

/* key types: the ten arithmetic key types of the reference's test matrix (src/test.cpp:155-169) */
enum {
  B200SORT_U8 = 0, B200SORT_I8 = 1, B200SORT_U16 = 2, B200SORT_I16 = 3, B200SORT_U32 = 4,
  B200SORT_I32 = 5, B200SORT_U64 = 6, B200SORT_I64 = 7, B200SORT_F32 = 8, B200SORT_F64 = 9
};

enum {
  B200SORT_OK = 0,
  B200SORT_EINVAL = -1,     /* bad key type, negative num, NULL array, mixed host/device arrays */
  B200SORT_ESHAPE = -2,     /* payload element size not in 1..64, > 63 payload streams */
  B200SORT_ERECORD = -3,    /* AoS record size not a power of two in [sizeof(key), 64]
                               (the reference static_asserts this, radix_sort.hpp:318-319) */
  B200SORT_ENOMEM = -4,     /* workspace too small / device allocation failed */
  B200SORT_ECUDA = -5,      /* CUDA runtime error or no device; see b200sort_last_error() */
  B200SORT_ENCCL = -6,      /* NCCL error or libnccl not loadable (multi-GPU entry points only) */
  B200SORT_EUNSUPPORTED = -7
};

/* cmp_sorter values for the *_ex entry points (reference: template parameter CmpSorter) */
enum {
  B200SORT_CMP_INSERTION = 0, /* CmpSorterInsertionSort, src/cmp_sorters.hpp:18-37: full sort */
  B200SORT_CMP_NONE = 1       /* CmpSorterNoSort, src/cmp_sorters.hpp:66-78: buckets of at most
                                 `cmp_sort_threshold` elements are left in arbitrary internal order */
};

/* Replaces simd_sort::radix_sort::sort<Up>(num, keys, payloads...)  (radixSort.hpp:1780-1783,
 * src/radix_sort.hpp:334-337).  payload_elem_bytes[i] in 1..64; n_payloads in 0..63. */
int b200sort_sort_soa(void *keys, int key_type, int64_t num, int ascending, int n_payloads,
                      void *const *payloads, const uint32_t *payload_elem_bytes, void *stream,
                      void *workspace, size_t workspace_bytes);

/* Replaces simd_sort::radix_sort::sort<Up>(num, DataElement<K, Ps...>*)  (radixSort.hpp:1770-1778,
 * src/radix_sort.hpp:314-332).  Records of `record_bytes` bytes, key of `key_type` at byte offset 0. */
int b200sort_sort_aos(void *records, int key_type, uint32_t record_bytes, int64_t num, int ascending,
                      void *stream, void *workspace, size_t workspace_bytes);

/* Replaces the advanced overloads sort<Up, BitSorter, CmpSorter>(cmpSortThreshold, num, ...)
 * (src/radix_sort.hpp:297-332).  With B200SORT_CMP_INSERTION the result is the full sort whatever the
 * threshold (as in the reference).  With B200SORT_CMP_NONE the result satisfies the reference's
 * partial-sort contract: the array is a permutation of the input in which every maximal group of
 * elements sharing the key bits above the point where the reference would stop recursing is
 * contiguous and groups appear in key order.  (Thresholds below 8 give the full sort: nearly every input would
 * need the finish anyway.  From 8 on, the digit sweeps run, a key-only sweep checks that no group longer than the
 * threshold is out of order -- only then does the segment finish run.) */
int b200sort_sort_soa_ex(void *keys, int key_type, int64_t num, int ascending, int n_payloads,
                         void *const *payloads, const uint32_t *payload_elem_bytes,
                         int64_t cmp_sort_threshold, int cmp_sorter, void *stream, void *workspace,
                         size_t workspace_bytes);
int b200sort_sort_aos_ex(void *records, int key_type, uint32_t record_bytes, int64_t num, int ascending,
                         int64_t cmp_sort_threshold, int cmp_sorter, void *stream, void *workspace,
                         size_t workspace_bytes);

/* Bytes of device scratch a call with these shapes needs (record_bytes = 0 for the SoA form, in
 * which case n_payloads/payload_elem_bytes describe the streams; for the AoS form they are ignored). */
size_t b200sort_workspace_bytes(int key_type, int64_t num, int n_payloads,
                                const uint32_t *payload_elem_bytes, uint32_t record_bytes);

/* ---- segmented sort: many independent segments of one array in one call ---------------------------
 * (An extension: the reference has no counterpart.)
 *  - Segments: segment i is records [offsets[i], offsets[i+1]).  `offsets` holds n_segments + 1 values,
 *    non-decreasing, with 0 <= offsets[0] and offsets[n_segments] <= num.
 *  - Result: each segment is sorted on its own, with the order and payload contract of b200sort_sort_soa /
 *    _aos (the total order on bit patterns; not stable).  Records outside [offsets[0], offsets[n_segments])
 *    are not touched.  n_segments == 0 and empty segments are no-ops; with num <= 1 nothing moves, but the offsets
 *    are still checked.  There is no partial-sort mode.
 *  - Memory side: `offsets` lives where the arrays do (host memory, or the arrays' device).  Host arrays are
 *    staged whole through the device's staging cache, and the call returns when the data is back.
 *  - Errors: offsets that decrease, are negative or pass num: B200SORT_EINVAL, and no record has moved.
 *    n_segments outside [0, 2^31 - 1] or offsets NULL: B200SORT_EINVAL.  Key type, payload shapes and record
 *    size are checked as in b200sort_sort_soa / _aos.
 *  - Workspace: NULL (the library's per-device cache) or a 256-byte aligned buffer of at least
 *    b200sort_segmented_workspace_bytes(...) bytes.
 *  - Host waits: a device-array call reads a few bytes of segment classification back (one wait; two when keys
 *    of 8 bytes have segments longer than CAP = 8192 records), plus the waits of the whole-array sorts below.
 *  - Segments of up to CAP records (16384 for keys of <= 4 bytes, 8192 for 8-byte keys) are sorted in shared
 *    memory.  With a longer segment, keys of <= 4 bytes are sorted as ONE whole-array sort of u64 (segment
 *    index, key) pairs over [offsets[0], offsets[n_segments]); 8-byte keys cost one whole-array sort per long
 *    segment (b200sort_sort_soa's sequence and host waits each).
 *  - b200sort_last_stats afterwards: algo = 3, num, record_bytes, key_bytes and kernel_launches of the whole call;
 *    every other field 0. */
int b200sort_sort_segmented_soa(void *keys, int key_type, int64_t num, int64_t n_segments, const int64_t *offsets,
                                int ascending, int n_payloads, void *const *payloads,
                                const uint32_t *payload_elem_bytes, void *stream, void *workspace, size_t workspace_bytes);
int b200sort_sort_segmented_aos(void *records, int key_type, uint32_t record_bytes, int64_t num, int64_t n_segments,
                                const int64_t *offsets, int ascending, void *stream, void *workspace, size_t workspace_bytes);
/* Bytes of device scratch a segmented call with these shapes needs, whatever the segment lengths (record_bytes = 0
 * for the SoA form). */
size_t b200sort_segmented_workspace_bytes(int key_type, int64_t num, int64_t n_segments, int n_payloads,
                                          const uint32_t *payload_elem_bytes, uint32_t record_bytes);

/* ---- top-k selection: the k smallest or largest records of every row -------------------------------------------
 * (An extension: the reference has no counterpart.)
 *  - Input: n_rows contiguous rows of row_len records (a whole array is n_rows = 1).  Payload streams have one
 *    element per record, as in b200sort_sort_soa; AoS records follow the rules of b200sort_sort_aos.  The inputs are
 *    only read.
 *  - Result: row r of every output holds k records.  out_keys[r k + j] equals, byte for byte, the j-th key of row r
 *    after b200sort_sort_soa(row r, ascending = !largest): largest = 1 gives the k largest in descending order (like
 *    torch.topk(sorted=True)), largest = 0 the k smallest in ascending order, in the total order on bit patterns
 *    (-NaN < -inf < ... < -0.0 < +0.0 < ... < +inf < +NaN).  out_index[r k + j] (int64, required) is the record's
 *    position inside its row; the indices of a row are distinct, keys[r row_len + out_index[r k + j]] equals
 *    out_keys[r k + j], and every output payload element (or AoS record) is the input's element at that position.
 *    When equal keys straddle the k-th place, which of them are chosen is unspecified.
 *  - Errors, checked before any device work: B200SORT_EINVAL for a negative n_rows, row_len or k, k > row_len,
 *    n_rows > 2^31 - 1, an n_rows * row_len that overflows, a NULL input, output or out_index when k > 0, a key
 *    array, key output or record array not aligned to the key type, out_index not 8-byte aligned, and an output
 *    whose address range overlaps an input's or another output's.  Payload shapes (up to 63 streams) and record
 *    sizes are checked as for the sort (B200SORT_ESHAPE / B200SORT_ERECORD).  k == 0 or n_rows == 0 is a no-op that
 *    returns 0.
 *  - Memory side: device arrays only, all on one device (the call runs on it); an array in host memory gives
 *    B200SORT_EUNSUPPORTED.
 *  - Workspace: NULL (the library's per-device cache) or a 256-byte aligned buffer of at least
 *    b200sort_topk_workspace_bytes(...) bytes, which covers any key distribution.  All work is ordered on `stream`;
 *    host waits: see the conventions above.
 *  - Method: radix select on 8-bit digits of the order-mapped key, most significant first: key-width + 1 passes of
 *    one fused kernel (select below the threshold's bucket, keep the candidates equal to it, count their next
 *    digit), each followed but the last by a decision kernel.  Each row has two candidate buffers of
 *    ceil(row_len / 16) entries; candidates that do not fit are found again by re-reading the row.  Uniform keys cost
 *    about two reads of the keys, adversarial ones (all equal, a constant top byte) at most key-width + 1.  The k
 *    winners of every row are then ordered by the segmented sort, and one gather moves the payloads / records.
 *  - b200sort_last_stats afterwards: algo = 4, num = n_rows * row_len, record_bytes, key_bytes and kernel_launches;
 *    every other field 0.  No tuning option applies. */
int b200sort_topk_soa(const void *keys, int key_type, int64_t n_rows, int64_t row_len, int64_t k, int largest,
                      int n_payloads, const void *const *payloads, const uint32_t *payload_elem_bytes,
                      void *out_keys, int64_t *out_index, void *const *out_payloads,
                      void *stream, void *workspace, size_t workspace_bytes);
int b200sort_topk_aos(const void *records, int key_type, uint32_t record_bytes, int64_t n_rows, int64_t row_len,
                      int64_t k, int largest, void *out_records, int64_t *out_index,
                      void *stream, void *workspace, size_t workspace_bytes);
/* Bytes of device scratch a top-k call with these shapes needs (record_bytes = 0 for the SoA form); 0 for an unknown
 * key type or invalid counts. */
size_t b200sort_topk_workspace_bytes(int key_type, int64_t n_rows, int64_t row_len, int64_t k, int n_payloads,
                                     const uint32_t *payload_elem_bytes, uint32_t record_bytes);

/* ---- unique: the distinct keys of an array, with their counts and inverse map --------------------------------------
 * (An extension: the reference has no counterpart.)
 *  - Equality is bit-pattern equality, consistent with the library's total order: +0.0 and -0.0 are two values, NaNs
 *    with the same bits are one value, NaNs with different payloads are different values.  (torch.unique merges
 *    +-0.0 and keeps every NaN apart.)
 *  - consecutive = 0, like torch.unique(sorted=True): out_keys[0, U) holds the distinct keys in ascending total order
 *    (-NaN < -inf < ... < -0.0 < +0.0 < ... < +inf < +NaN).
 *    consecutive = 1, like torch.unique_consecutive: every maximal run of equal adjacent keys, in input order, gives
 *    one entry, and no sort runs.
 *  - out_counts[j] (int64, optional: NULL for none) is the number of input keys equal to entry j, or the length of
 *    run j.  out_inverse[i] (int64, optional) is the j whose entry equals keys[i], or the run that contains i.
 *  - *out_num_unique = U (int64, required) is written on `stream` into device memory.  Every output has room for num
 *    entries; entries >= U are not written.  The input is only read.
 *  - Errors, checked before any device work: B200SORT_EINVAL for an unknown key type, a negative num, a NULL keys,
 *    out_keys or out_num_unique when num > 0, keys or out_keys not aligned to the key type, an int64 output not
 *    8-byte aligned, and an output whose address range overlaps the input or another output.  With num == 0 only
 *    *out_num_unique = 0 is written (nothing at all when out_num_unique is NULL).
 *  - Memory side: device arrays only, all on one device (the call runs on it); an array in host memory gives
 *    B200SORT_EUNSUPPORTED.
 *  - Workspace: NULL (the library's per-device cache) or a 256-byte aligned buffer of at least
 *    b200sort_unique_workspace_bytes(key_type, num, consecutive, with_inverse = out_inverse != NULL) bytes, which
 *    depends on the shape only.  Host waits: consecutive = 1 waits for nothing; consecutive = 0 adds exactly the waits
 *    of the whole-array sort it runs (see the conventions above).
 *  - Method: consecutive = 0 copies the keys into the workspace (with their positions, u32 up to 2^32 records and u64
 *    above, when the inverse is wanted) and sorts the copy with the whole-array sort.  Then one pass over the keys
 *    compares each with its predecessor, numbers the runs (warp ballots, a block scan and a decoupled look-back over
 *    tiles of 4096 keys) and writes the entries, the run starts and the inverse (a scatter through the positions after
 *    the sort); a second small kernel turns the run starts into counts.
 *  - b200sort_last_stats afterwards: algo = 5, num, record_bytes = key_bytes, kernel_launches (the sort's included);
 *    every other field 0. */
int b200sort_unique(const void *keys, int key_type, int64_t num, int consecutive,
                    void *out_keys, int64_t *out_counts, int64_t *out_inverse, int64_t *out_num_unique,
                    void *stream, void *workspace, size_t workspace_bytes);
/* Bytes of device scratch a unique call with this shape needs; 0 for an unknown key type or a negative num. */
size_t b200sort_unique_workspace_bytes(int key_type, int64_t num, int consecutive, int with_inverse);

/* Thread-local message of the last failing call on this thread ("" if none). */
const char *b200sort_last_error(void);

int b200sort_version(void);

/* Number of kernels this library has launched in this process so far (monotonic; used by bench.py
 * for its gpu_launches field). */
uint64_t b200sort_launch_count(void);

/* Tuning/ablation knobs: process-wide defaults, read once when a call starts.  Known names: "algo" (0 auto, 1 LSD one-sweep passes,
 * 2 hybrid MSB), "tile_cfg" (index of the scatter tile geometry), "first_atomic", "tma_keys", "bytewise",
 * "hist_match", "allow_skip", "profile", "mgpu_overlap", "mgpu_chunks", "mgpu_refine" (INTEGRATION.md lists them
 * all).  Returns 0, or B200SORT_EINVAL for an unknown name or a value "max_chunk" does not take. */
int b200sort_set_option(const char *name, int64_t value);
int64_t b200sort_get_option(const char *name);

/* What the last successful device-side sort on this thread did (for roofline accounting). */
typedef struct b200sort_stats {
  int64_t num;
  uint32_t record_bytes;      /* sum of all stream element sizes */
  uint32_t key_bytes;
  uint32_t algo;              /* 1 LSD, 2 hybrid, 3 segmented sort, 4 top-k, 5 unique (3 to 5: only num, record_bytes,
                                 key_bytes and kernel_launches are set) */
  uint32_t passes_planned;    /* scatter passes executed (hybrid) / launched (LSD; constant digits return at once) */
  uint32_t hist_sweeps;       /* key-only sweeps launched */
  uint32_t kernel_launches;   /* kernels launched by this call */
  uint32_t segfix_passes;     /* hybrid: 1 when the in-shared-memory segment finish ran */
  uint32_t cut_digit;         /* hybrid: digit positions below this were left to the segment finish */
  uint32_t fell_back;         /* hybrid: 1 when a long bucket with distinct keys forced the digit-by-digit path */
  uint64_t algorithmic_bytes; /* H*N*K + P*2*N*R with the executed pass counts (SURVEY.md 8d) */
  uint64_t segfix_moved;      /* hybrid: records the segment finish had to move */
} b200sort_stats;
int b200sort_last_stats(b200sort_stats *out);

/* Per-kernel device times of the last sort on this thread, recorded with CUDA events on the sort's
 * stream when option "profile" is 1.  kinds[i]: 0 histogram, 1 scan, 2 scatter pass, 3 copy-back,
 * 4 segment finish, 5 other, 6 segmented-sort kernels of short segments, 7 top-k selection and gather,
 * 8 unique (index, run compaction, counts; the sort it runs keeps its own kinds).  A single-GPU call lists one entry
 * per kernel its kernel_launches counts, those of the sorts it runs inside and of a fall-back included.  Returns the
 * number of entries written (<= capacity) or a negative code. */
int b200sort_last_profile(int *kinds, float *ms, int capacity);

/* Releases the per-device workspace and host-staging buffers held by the library.  A sort another thread
 * is launching on them is queued first; the call then waits for each device to be idle. */
void b200sort_release_cache(void);

/* ---- multi-GPU: one process per GPU, NCCL over NVLink (SURVEY.md 8e) -------------------------
 * The communicator is created by the library from an ncclUniqueId that rank 0 obtains with
 * b200sort_mgpu_unique_id() and distributes by any means (torch.distributed, MPI, a file). */
typedef struct b200sort_comm b200sort_comm;
#define B200SORT_UNIQUE_ID_BYTES 128
int b200sort_mgpu_unique_id(void *out_id_128_bytes);
int b200sort_mgpu_comm_create(b200sort_comm **out, int world_size, int rank, const void *id_128_bytes);
int b200sort_mgpu_comm_destroy(b200sort_comm *comm);
/* 1 if the last b200sort_mgpu_sort_soa on this communicator scattered its records straight into the peers'
 * memory (cudaIpc-mapped workspaces over NVLink), 0 if it exchanged them with ncclSend/ncclRecv. */
int b200sort_mgpu_used_p2p(const b200sort_comm *comm);
/* Note: while a communicator is alive its peers may have this process's cached workspace mapped.  The library
 * makes them let go before b200sort_mgpu_sort_soa re-allocates it; do not call b200sort_release_cache(), or a
 * larger single-GPU sort with workspace == NULL, between multi-GPU sorts without destroying the communicator. */

/* Host-side splitter selection used by the multi-GPU sort (exported so that it can be tested without
 * a GPU): given the globally reduced histogram of the top `bits` bits of the order-mapped keys
 * (2^bits counters), writes world_size+1 bin boundaries b[0]=0 <= ... <= b[world]=2^bits such that
 * rank r owns bins [b[r], b[r+1]) and the loads are even to within bin granularity plus 1/64 of a share,
 * which a boundary may give up to land on an aligned bin index (shards then share leading key bits). */
int b200sort_mgpu_splitters(const uint64_t *global_hist, int bits, int world_size, uint32_t *out_bounds);
/* The binning of that histogram: from the smallest / largest order-mapped key of the ranks' samples to
 * bin(u) = clamp((u - lo) >> shift, 0, 2^bits - 1).  Keys of a narrow range get bins as fine as single values;
 * full-width keys keep bin = their top `bits` bits.  Exported for the same reason. */
int b200sort_mgpu_range_bins(uint64_t lo_key, uint64_t hi_key, int key_bytes, int bits, uint64_t *out_lo, int *out_shift);

/* Host-side exchange plan (also exported for GPU-less tests): number of local records destined to each
 * rank, given this rank's own top-bits histogram and the splitters above. */
int b200sort_mgpu_plan(const uint64_t *local_hist, int bits, int world_size, const uint32_t *bounds,
                       uint64_t *out_send_counts);

/* Distributed SoA sort.  On entry every rank holds `num_local` unsorted records in device memory; on
 * return rank r holds *out_num_local records, sorted, all of them ordered before those of rank r+1.
 * `capacity` is the number of records each of keys/payloads can hold (>= the largest partition; the
 * call fails with B200SORT_ENOMEM, before moving data, if a partition would not fit -- which skewed or
 * duplicate-heavy keys do not cause: heavy key values are split, see below). */
int b200sort_mgpu_sort_soa(b200sort_comm *comm, void *keys, int key_type, int64_t num_local,
                           int64_t capacity, int ascending, int n_payloads, void *const *payloads,
                           const uint32_t *payload_elem_bytes, int64_t *out_num_local, void *stream);

/* The same for combined records (the DataElement<K, Ps...> form, radixSort.hpp:1770-1778): `records` holds
 * `num_local` records of `record_bytes` bytes (a power of two <= 64, key of `key_type` at byte offset 0) and
 * has room for `capacity` of them. */
int b200sort_mgpu_sort_aos(b200sort_comm *comm, void *records, int key_type, uint32_t record_bytes,
                           int64_t num_local, int64_t capacity, int ascending, int64_t *out_num_local,
                           void *stream);

/* 1 if the last multi-GPU sort on this communicator overlapped the exchange with the receivers' first pass
 * (chunked partition kernels + arrival flags; uniform full-width 8-byte keys), 0 otherwise. */
int b200sort_mgpu_used_overlap(const b200sort_comm *comm);

/* Skewed keys (SURVEY 8e(3)): when a histogram bin is heavier than a rank may hold, the splitters are refined
 * 16 key bits per level down to single key values, and the keys EQUAL to such a value are divided among the
 * ranks by source rank and position.  The host-side logic is exported so that it can be tested without a GPU:
 *  - b200sort_mgpu_refine_splitters: `hist_fn(ctx, n_ranges, lo, shift, nb, out)` must fill out[j * 65536 + b]
 *    with the global count of keys u with (u - lo[j]) >> shift[j] == b < nb[j] (ordered-key space); writes the
 *    world_size-1 splitter keys and whether each one sits on a single heavy key value;
 *  - b200sort_mgpu_tie_thresholds: for one heavy value, `eq[s * n_blocks + b]` = number of keys equal to it in
 *    position block b of source rank s, `less_total` = keys below it (all ranks), targets[i] = records that must
 *    lie left of the i-th splitter sitting on it; out_blk[i] = first position block of rank `rank` whose equal
 *    keys go right of that splitter (0: all, 0xffffffff: none). */
typedef int (*b200sort_hist_fn)(void *ctx, int n_ranges, const uint64_t *lo, const int *shift, const uint32_t *nb,
                                uint64_t *out);
int b200sort_mgpu_refine_splitters(int world_size, int key_bytes, uint64_t total, b200sort_hist_fn hist_fn,
                                   void *ctx, uint64_t *out_keys, uint32_t *out_is_tie);
int b200sort_mgpu_tie_thresholds(int world_size, int rank, int n_blocks, uint64_t less_total, const uint32_t *eq,
                                 int n_targets, const uint64_t *targets, uint32_t *out_blk);

#ifdef __cplusplus
}
#endif
#endif /* B200SORT_H_ */
