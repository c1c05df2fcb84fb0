// unique_host.cuh -- host side of unique (b200sort_unique; kernels in unique.cuh).  Included at the end of b200sort.cu
// (it uses that file's internals).
#pragma once

namespace b200sort {

// workspace: tile ticket + look-back status words (zeroed per call) | sorted mode: the key copy | the index | the region
// the sort of those uses as its workspace, and that then holds the run starts (the sort is done with it by then)
struct UniqueLayout {
  size_t ctrl_bytes, keys_off, index_off, region_off, total;
  int64_t n_tiles;
  uint32_t index_bytes;  // 0: no index (consecutive mode, or no inverse wanted)
};

static UniqueLayout unique_layout(int kb, int64_t num, bool consecutive, bool with_inverse) {
  UniqueLayout u{};
  u.n_tiles = (num + UNQ_TILE - 1) / UNQ_TILE;
  u.ctrl_bytes = 256 + (size_t)u.n_tiles * 8;
  u.index_bytes = (consecutive || !with_inverse) ? 0u : (num <= ((int64_t)1 << 32) ? 4u : 8u);
  size_t region = ((size_t)num + 1) * 8;  // the run starts
  std::vector<size_t> bytes = {u.ctrl_bytes, 0, 0};
  if (!consecutive) {
    std::vector<StreamDesc> sorted = {{nullptr, (uint32_t)kb}};
    if (u.index_bytes) sorted.push_back({nullptr, u.index_bytes});
    region = std::max(region, sort_workspace_bytes(sorted, num));
    bytes[1] = (size_t)num * kb;
    bytes[2] = (size_t)num * u.index_bytes;
  }
  bytes.push_back(region);
  const std::vector<size_t> offs = back_to_back(bytes, &u.total);
  u.keys_off = offs[1]; u.index_off = offs[2]; u.region_off = offs[3];
  return u;
}

// unique of device arrays on the current device
static int unique_device(const Options &o, int key_type, int64_t num, bool consecutive, const void *keys, void *out_keys,
                         int64_t *out_counts, int64_t *out_inverse, int64_t *out_num_unique, cudaStream_t stream,
                         void *caller_workspace, size_t workspace_bytes, b200sort_stats *stats) {
  const int kb = key_bytes_of(key_type);
  const std::vector<StreamDesc> in = {{const_cast<void *>(keys), (uint32_t)kb}};
  DevSetup su;
  if (num == 0) {  // U = 0 is all there is to write
    CUDA_TRY(cudaMemsetAsync(out_num_unique, 0, 8, stream));
    *stats = su.stats(0, in, kb, ALGO_UNIQUE);
    return B200SORT_OK;
  }
  if (int rc = su.open()) return rc;
  const UniqueLayout ul = unique_layout(kb, num, consecutive, out_inverse != nullptr);
  if (int rc = su.workspace(stream, caller_workspace, workspace_bytes, ul.total)) return rc;
  CUDA_TRY(cudaMemsetAsync(su.ws, 0, ul.ctrl_bytes, stream));

  UniqueArgs a{};
  a.keys = (const unsigned char *)keys;
  if (!consecutive) {
    // 1. a copy of the keys (and their positions, for the inverse), sorted by the whole-array sort
    unsigned char *copy = su.ws + ul.keys_off, *idx = su.ws + ul.index_off;
    CUDA_TRY(cudaMemcpyAsync(copy, keys, (size_t)num * kb, cudaMemcpyDeviceToDevice, stream));
    std::vector<StreamDesc> sorted = {{copy, (uint32_t)kb}};
    if (ul.index_bytes) {
      const unsigned grid = (unsigned)std::min<int64_t>((num + 255) / 256, (int64_t)su.di.sm_count * 8);
      if (ul.index_bytes == 4) CUDA_TRY(launch(PK_UNIQUE, iota_kernel, grid, 256, 0, stream, (uint32_t *)idx, num));
      else CUDA_TRY(launch(PK_UNIQUE, unique_iota64_kernel, grid, 256, 0, stream, (unsigned long long *)idx, num));
      sorted.push_back({idx, ul.index_bytes});
      a.index = idx;
    }
    if (num > 1) {
      b200sort_stats inner;
      if (int rc = sort_device(o, key_type, true, num, sorted, stream, su.ws + ul.region_off, ul.total - ul.region_off, DevSortOpts(),
                               &inner))
        return rc;
    }
    a.keys = copy;
  }

  // 2. the run compaction; 3. the counts
  a.num = num; a.n_tiles = ul.n_tiles;
  a.vec = ((uintptr_t)a.keys & 15) == 0 ? 1u : 0u;
  a.out_keys = out_keys; a.out_inverse = out_inverse; a.out_num_unique = out_num_unique;
  a.start = out_counts ? (int64_t *)(su.ws + ul.region_off) : nullptr;
  a.ticket = (uint32_t *)su.ws; a.status = (uint64_t *)(su.ws + 256);
  CUDA_TRY(with_kb(kb, [&](auto K) {
    constexpr int KB = decltype(K)::value;
    auto *k = ul.index_bytes == 4 ? unique_scan_kernel<KB, 4> : ul.index_bytes == 8 ? unique_scan_kernel<KB, 8> : unique_scan_kernel<KB, 0>;
    return launch(PK_UNIQUE, k, (unsigned)ul.n_tiles, UNQ_THREADS, 0, stream, a);
  }));
  if (out_counts) {
    const unsigned grid = (unsigned)std::min<int64_t>((num + 255) / 256, (int64_t)su.di.sm_count * 16);
    CUDA_TRY(launch(PK_UNIQUE, unique_counts_kernel, grid, 256, 0, stream, (const int64_t *)a.start, (const int64_t *)out_num_unique,
                    out_counts));
  }
  *stats = su.stats(num, in, kb, ALGO_UNIQUE);
  return B200SORT_OK;
}

// argument checks (all before any device work), then the call on the arrays' device
static int unique_any(int key_type, int64_t num, bool consecutive, const void *keys, void *out_keys, int64_t *out_counts,
                      int64_t *out_inverse, int64_t *out_num_unique, void *stream_v, void *workspace, size_t workspace_bytes) {
  const int kb = key_bytes_of(key_type);
  if (kb == 0) return fail(B200SORT_EINVAL, "unknown key type %d", key_type);
  if (num < 0) return fail(B200SORT_EINVAL, "negative element count");
  if (num > 0) {
    if (keys == nullptr) return fail(B200SORT_EINVAL, "keys is NULL");
    if (out_keys == nullptr) return fail(B200SORT_EINVAL, "out_keys is NULL");
    if (out_num_unique == nullptr) return fail(B200SORT_EINVAL, "out_num_unique is NULL");
  }
  if ((uintptr_t)keys % kb != 0 || (uintptr_t)out_keys % kb != 0) return fail(B200SORT_EINVAL, "keys / out_keys are not aligned to their key type");
  if (((uintptr_t)out_counts | (uintptr_t)out_inverse | (uintptr_t)out_num_unique) % 8 != 0)
    return fail(B200SORT_EINVAL, "out_counts, out_inverse and out_num_unique must be 8-byte aligned");
  const size_t n = (size_t)num;
  if (int rc = check_disjoint({{keys, n * kb}}, {{out_keys, n * kb}, {out_counts, n * 8}, {out_inverse, n * 8}, {out_num_unique, 8}}))
    return rc;
  if (num == 0 && out_num_unique == nullptr) return B200SORT_OK;

  std::vector<StreamDesc> all;
  for (const void *p : {keys, (const void *)out_keys, (const void *)out_counts, (const void *)out_inverse, (const void *)out_num_unique})
    if (p != nullptr) all.push_back({const_cast<void *>(p), 1u});
  CallScope call;
  if (int rc = call.enter(all, nullptr, "unique")) return rc;
  return call.done(unique_device(call.o, key_type, num, consecutive, keys, out_keys, out_counts, out_inverse, out_num_unique,
                                 (cudaStream_t)stream_v, workspace, workspace_bytes, &call.stats));
}

}  // namespace b200sort

extern "C" {

int b200sort_unique(const void *keys, int key_type, int64_t num, int consecutive, void *out_keys, int64_t *out_counts,
                    int64_t *out_inverse, int64_t *out_num_unique, void *stream, void *workspace, size_t workspace_bytes) {
  return unique_any(key_type, num, consecutive != 0, keys, out_keys, out_counts, out_inverse, out_num_unique, stream, workspace,
                    workspace_bytes);
}

size_t b200sort_unique_workspace_bytes(int key_type, int64_t num, int consecutive, int with_inverse) {
  const int kb = key_bytes_of(key_type);
  if (kb == 0 || num < 0) return 0;
  return unique_layout(kb, num, consecutive != 0, with_inverse != 0).total;
}

}  // extern "C"
