// segmented_host.cuh -- host side of the segmented sort (b200sort_sort_segmented_soa / _aos; kernels in
// segmented.cuh).  Included at the end of b200sort.cu (it uses that file's internals).
#pragma once

namespace b200sort {

// workspace: control block | bin lists | long-segment list | the region of the long-segment branch
struct SegLayout {
  size_t list_off[SEG_NBINS], large_off, region_off, region_bytes, total;
  uint32_t list_cap[SEG_NBINS], large_cap;  // entries of each list
  size_t comp_off, sort_off;  // (inside the region) composite keys, whole-array sort workspace
};

static SegLayout seg_layout(int kb, int64_t num, int64_t n_segments, const std::vector<StreamDesc> &streams, bool soa) {
  SegLayout s{};
  const int64_t cap = (int64_t)1 << seg_cap_log2(kb);
  size_t off = align_up(sizeof(SegCtrl), 256);
  for (int b = 0; b < SEG_NBINS; b++) {
    // a bin whose segments have more than `lo` records holds at most num / (lo + 1) of them
    const int64_t lo = b == 0 ? 1 : ((int64_t)1 << (b + 4));
    const int64_t entries = (lo < cap) ? std::min(n_segments, num / (lo + 1)) : 0;
    s.list_off[b] = off;
    s.list_cap[b] = (uint32_t)entries;  // (n_segments < 2^31)
    off = align_up(off + (size_t)entries * 4, 256);
  }
  s.large_off = off;
  s.large_cap = (uint32_t)std::min(n_segments, num / (cap + 1));
  off = align_up(off + (size_t)s.large_cap * 16, 256);
  s.region_off = off;
  if (kb <= 4) {
    // composite keys + the sort of (composite, payloads...) or (composite, records)
    std::vector<StreamDesc> cs = {{nullptr, 8u}};
    for (size_t i = soa ? 1 : 0; i < streams.size(); i++) cs.push_back(streams[i]);
    s.comp_off = 0;
    s.sort_off = align_up((size_t)num * 8, 256);
    s.region_bytes = s.sort_off + sort_workspace_bytes(cs, num);
  } else {
    s.comp_off = s.sort_off = 0;  // one sort of the caller's streams at a time, at most num records
    s.region_bytes = sort_workspace_bytes(streams, num);
  }
  s.total = s.region_off + s.region_bytes;
  return s;
}

// the medium kernel of bin b >= 1 (segments of up to 2^(b+5) records): persistent CTAs, as many as fit
static cudaError_t seg_launch_medium(int kb, int b, const SegSortArgs &a, int sm_count, cudaStream_t st) {
  const SegMediumKernel k = seg_medium_kernel_of(kb, b + 5);
  if (k.fn == nullptr) return cudaErrorInvalidValue;
  cudaError_t e = cudaFuncSetAttribute(k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.smem);
  if (e != cudaSuccess) return e;
  int per_sm = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k.fn, k.threads, k.smem);
  if (e != cudaSuccess) return e;
  const unsigned grid = (unsigned)std::min<int64_t>(a.count, (int64_t)sm_count * std::max(per_sm, 1));
  return launch(PK_SEGMENT, k.fn, grid, k.threads, k.smem, st, a);
}

// the sort of the segments of bin b
static cudaError_t seg_launch_bin(int kb, int b, const SegSortArgs &a, int sm_count, cudaStream_t st) {
  if (b > 0) return seg_launch_medium(kb, b, a, sm_count, st);
  const unsigned grid = (unsigned)std::min<int64_t>((a.count + SEG_TINY_THREADS / 32 - 1) / (SEG_TINY_THREADS / 32), (int64_t)sm_count * 8);
  return with_kb(kb, [&](auto K) { return launch(PK_SEGMENT, seg_tiny_kernel<decltype(K)::value>, grid, SEG_TINY_THREADS, 0, st, a); });
}

// The segmented sort of arrays that are all in device memory (the current device), offsets included.
static int sort_segmented_device(const Options &o, int key_type, bool ascending, int64_t num, int64_t n_segments, const int64_t *offsets,
                                 const std::vector<StreamDesc> &streams, bool soa, cudaStream_t stream, void *caller_workspace,
                                 size_t workspace_bytes, b200sort_stats *stats) {
  const int kb = key_bytes_of(key_type);
  const uint64_t launches_before = g_launches.load();
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  DevInfo di;
  if (int rc = dev_info(dev, &di)) return rc;
  if (((uintptr_t)streams[0].ptr % kb) != 0) return fail(B200SORT_EINVAL, "key array is not aligned to its key type");
  const SegLayout sl = seg_layout(kb, num, n_segments, streams, soa);
  CacheGuard cache_guard;
  unsigned char *ws = nullptr;
  if (int rc = acquire_workspace(dev, stream, caller_workspace, workspace_bytes, sl.total, cache_guard, &ws)) return rc;
  start_profile(o, false);

  // classify (one host wait: the bin counts, the validity flag, the longest segment)
  const int cap_log2 = seg_cap_log2(kb);
  SegCtrl *ctrl = (SegCtrl *)ws;
  CUDA_TRY(cudaMemsetAsync(ctrl, 0, sizeof(SegCtrl), stream));
  SegClassifyArgs ca{};
  ca.offsets = offsets; ca.n_segments = n_segments; ca.num = num; ca.cap = 1u << cap_log2; ca.ctrl = ctrl;
  for (int b = 0; b < SEG_NBINS; b++) { ca.list[b] = (uint32_t *)(ws + sl.list_off[b]); ca.list_cap[b] = sl.list_cap[b]; }
  ca.large = (int64_t *)(ws + sl.large_off);
  ca.large_cap = sl.large_cap;
  const unsigned cgrid = (unsigned)std::min<int64_t>((n_segments + SEG_CLASSIFY_THREADS - 1) / SEG_CLASSIFY_THREADS, (int64_t)di.sm_count * 8);
  CUDA_TRY(launch(PK_OTHER, seg_classify_kernel, cgrid, SEG_CLASSIFY_THREADS, 0, stream, ca));
  SegCtrl h{};
  CUDA_TRY(cudaMemcpyAsync(&h, ctrl, sizeof h, cudaMemcpyDeviceToHost, stream));
  CUDA_TRY(cudaStreamSynchronize(stream));
  if (h.bad) return fail(B200SORT_EINVAL, "offsets must be non-decreasing, within [0, num]");

  KeyOrder ko = make_key_order(key_type, ascending);
  std::vector<StreamDesc> sub = streams;
  b200sort_stats inner;
  DevSortOpts whole;
  whole.keep_profile = true;  // (the profile of this call lists the segment kernels too)
  const bool long_segments = h.max_len > ca.cap;  // (then n_large > 0)
  if (long_segments && kb <= 4) {
    // one sort of (segment index, ordered key) over [offsets[0], offsets[n_segments])
    const int64_t first = h.first, span = h.last - h.first;
    SegCompositeArgs pa{};
    pa.keys = (unsigned char *)streams[0].ptr; pa.key_stride = streams[0].elem_bytes; pa.offsets = offsets; pa.n_segments = n_segments;
    pa.first = first; pa.span = span; pa.ko = ko; pa.comp = (unsigned long long *)(ws + sl.region_off + sl.comp_off);
    const unsigned grid = (unsigned)std::min<int64_t>((span + 255) / 256, (int64_t)di.sm_count * 16);
    auto pack = [&](auto K, bool unpack) -> cudaError_t {
      constexpr int KB = decltype(K)::value;
      if constexpr (KB <= 4) return launch(PK_OTHER, unpack ? seg_unpack_kernel<KB> : seg_pack_kernel<KB>, grid, 256, 0, stream, pa);
      return cudaErrorInvalidValue;
    };
    CUDA_TRY(with_kb(kb, [&](auto K) { return pack(K, false); }));
    std::vector<StreamDesc> cs = {{pa.comp, 8u}};
    for (size_t i = soa ? 1 : 0; i < streams.size(); i++) cs.push_back({(unsigned char *)streams[i].ptr + (size_t)first * streams[i].elem_bytes, streams[i].elem_bytes});
    if (int rc = sort_device(o, B200SORT_U64, true, span, cs, stream, ws + sl.region_off + sl.sort_off, sl.region_bytes - sl.sort_off,
                             whole, &inner))
      return rc;
    if (soa) CUDA_TRY(with_kb(kb, [&](auto K) { return pack(K, true); }));
  } else {
    if (long_segments) {
      // 8-byte keys: one sort per long segment (second host wait: their starts and lengths)
      std::vector<int64_t> large(2 * (size_t)h.n_large);
      CUDA_TRY(cudaMemcpyAsync(large.data(), ws + sl.large_off, large.size() * 8, cudaMemcpyDeviceToHost, stream));
      CUDA_TRY(cudaStreamSynchronize(stream));
      for (uint32_t i = 0; i < h.n_large; i++) {
        for (size_t s = 0; s < streams.size(); s++) sub[s].ptr = (unsigned char *)streams[s].ptr + (size_t)large[2 * i] * streams[s].elem_bytes;
        if (int rc = sort_device(o, key_type, ascending, large[2 * i + 1], sub, stream, ws + sl.region_off, sl.region_bytes, whole, &inner))
          return rc;
      }
    }
    SegSortArgs sa{};
    make_stream_set(streams, kb, 16, &sa.ss);
    sa.ko = ko; sa.offsets = offsets;
    for (int b = 0; b < SEG_NBINS; b++) {
      if (h.count[b] == 0) continue;
      sa.list = (const uint32_t *)(ws + sl.list_off[b]); sa.count = h.count[b]; sa.ticket = &ctrl->ticket[b];
      CUDA_TRY(seg_launch_bin(kb, b, sa, di.sm_count, stream));
    }
  }
  *stats = call_stats(num, streams, kb, launches_before);
  stats->algo = 3;
  return B200SORT_OK;
}

// num <= 1: no segment has two records, but invalid offsets are still an error.  The offsets are checked on the
// host (device offsets are copied there first: the arrays may be empty, so there is nothing to sort on the device).
static int check_offsets_only(int64_t num, int64_t n_segments, const int64_t *offsets, cudaStream_t stream) {
  if (int rc = require_device()) return rc;
  Side side;
  int dev = 0;
  if (int rc = side_of(offsets, &side, &dev)) return rc;
  std::vector<int64_t> h;
  const int64_t *v = offsets;
  if (side == SIDE_DEVICE) {
    DeviceScope scope;
    if (int rc = scope.enter(dev)) return rc;
    h.resize((size_t)n_segments + 1);
    CUDA_TRY(cudaMemcpyAsync(h.data(), offsets, h.size() * 8, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    v = h.data();
  }
  for (int64_t i = 0; i < n_segments; i++)
    if (v[i] < 0 || v[i + 1] < v[i] || v[i + 1] > num) return fail(B200SORT_EINVAL, "offsets must be non-decreasing, within [0, num]");
  return B200SORT_OK;
}

// argument checks, then the device path, or the host path (everything staged whole through the staging cache)
static int sort_segmented_any(int key_type, bool ascending, int64_t num, int64_t n_segments, const int64_t *offsets,
                              const std::vector<StreamDesc> &streams, bool soa, void *stream_v, void *workspace, size_t workspace_bytes) {
  if (n_segments < 0 || n_segments > INT32_MAX) return fail(B200SORT_EINVAL, "%lld segments (0..2^31-1 supported)", (long long)n_segments);
  if (offsets == nullptr) return fail(B200SORT_EINVAL, "offsets is NULL");
  if (n_segments == 0) return B200SORT_OK;
  cudaStream_t stream = (cudaStream_t)stream_v;
  if (num <= 1) return check_offsets_only(num, n_segments, offsets, stream);  // (nothing can move)
  const Options o = options();
  Side side;
  int dev = 0;
  if (int rc = arrays_side(streams, offsets, &side, &dev)) return rc;
  if (side == SIDE_DEVICE) {
    DeviceScope scope;
    if (int rc = scope.enter(dev)) return rc;
    return sort_segmented_device(o, key_type, ascending, num, n_segments, offsets, streams, soa, stream, workspace, workspace_bytes,
                                 &g_last_stats);
  }
  // host arrays: the whole arrays and the offsets up, the sort, the arrays down (not when it failed)
  CUDA_TRY(cudaGetDevice(&dev));
  CacheGuard cache_guard;
  return sort_staged(cache_guard.acquire(dev, stream).stage, num, streams, offsets, (size_t)(n_segments + 1) * 8, stream,
                     [&](const std::vector<StreamDesc> &dstreams, const void *doffsets) {
                       return sort_segmented_device(o, key_type, ascending, num, n_segments, (const int64_t *)doffsets, dstreams, soa,
                                                    stream, workspace, workspace_bytes, &g_last_stats);
                     });
}

}  // namespace b200sort

extern "C" {

int b200sort_sort_segmented_soa(void *keys, int key_type, int64_t num, int64_t n_segments, const int64_t *offsets, int ascending,
                                int n_payloads, void *const *payloads, const uint32_t *payload_elem_bytes, void *stream, void *workspace,
                                size_t workspace_bytes) {
  std::vector<StreamDesc> streams;
  if (int rc = check_soa(keys, key_type, num, n_payloads, payloads, payload_elem_bytes, &streams)) return rc;
  return sort_segmented_any(key_type, ascending != 0, num, n_segments, offsets, streams, true, stream, workspace, workspace_bytes);
}

int b200sort_sort_segmented_aos(void *records, int key_type, uint32_t record_bytes, int64_t num, int64_t n_segments,
                                const int64_t *offsets, int ascending, void *stream, void *workspace, size_t workspace_bytes) {
  std::vector<StreamDesc> streams;
  if (int rc = check_aos(records, key_type, record_bytes, num, &streams)) return rc;
  return sort_segmented_any(key_type, ascending != 0, num, n_segments, offsets, streams, false, stream, workspace, workspace_bytes);
}

size_t b200sort_segmented_workspace_bytes(int key_type, int64_t num, int64_t n_segments, int n_payloads, const uint32_t *payload_elem_bytes,
                                          uint32_t record_bytes) {
  const int kb = key_bytes_of(key_type);
  if (kb == 0 || num < 0 || n_segments < 0) return 0;
  return seg_layout(kb, num, n_segments, streams_of_shape(kb, n_payloads, payload_elem_bytes, record_bytes), record_bytes == 0).total;
}

}  // extern "C"
