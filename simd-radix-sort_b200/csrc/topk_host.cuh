// topk_host.cuh -- host side of the top-k selection (b200sort_topk_soa / _aos; kernels in topk.cuh).  Included at the
// end of b200sort.cu, after segmented_host.cuh (it orders the winners with sort_segmented_device).
#pragma once

namespace b200sort {

// workspace: row states | histograms | control block (zeroed together) | work-item table | candidate buffers |
// selected keys (AoS) | offsets of the ordering step | the segmented sort's workspace
struct TopkLayout {
  size_t zero_bytes, hist_off, ctrl_off, items_off, cand_key_off[2], cand_pos_off[2], keys_off, offsets_off, seg_off, total;
  int64_t cap, chunks_per_row;
};

static TopkLayout topk_layout(int kb, int64_t n_rows, int64_t row_len, int64_t k, bool soa) {
  TopkLayout t{};
  t.cap = topk_cap(row_len);
  t.chunks_per_row = (row_len + TOPK_CHUNK - 1) / TOPK_CHUNK;
  const size_t rows = (size_t)n_rows, ord = kb == 8 ? 8 : 4;
  std::vector<size_t> bytes = {rows * sizeof(TopkRow), rows * RADIX * 8, sizeof(TopkCtrl), rows * (size_t)t.chunks_per_row * 4};
  for (int b = 0; b < 2; b++) bytes.insert(bytes.end(), {rows * (size_t)t.cap * ord, rows * (size_t)t.cap * 8});
  bytes.push_back(soa ? 0 : rows * (size_t)k * kb);
  bytes.push_back((rows + 1) * 8);
  const std::vector<StreamDesc> sorted = {{nullptr, (uint32_t)kb}, {nullptr, 8u}};
  bytes.push_back(seg_layout(kb, n_rows * k, n_rows, sorted, true).total);
  const std::vector<size_t> offs = back_to_back(bytes, &t.total);
  t.hist_off = offs[1]; t.ctrl_off = offs[2]; t.zero_bytes = offs[2] + sizeof(TopkCtrl);
  t.items_off = offs[3];
  t.cand_key_off[0] = offs[4]; t.cand_pos_off[0] = offs[5]; t.cand_key_off[1] = offs[6]; t.cand_pos_off[1] = offs[7];
  t.keys_off = offs[8]; t.offsets_off = offs[9]; t.seg_off = offs[10];
  return t;
}

// The top-k of device arrays on the current device.  in[0]: keys (SoA) or records (AoS), in[1..]: payloads; out[s]:
// the output of in[s].
static int topk_device(const Options &o, int key_type, bool largest, int64_t n_rows, int64_t row_len, int64_t k,
                       const std::vector<StreamDesc> &in, const std::vector<StreamDesc> &out, int64_t *out_index, bool soa,
                       cudaStream_t stream, void *caller_workspace, size_t workspace_bytes, b200sort_stats *stats) {
  const int kb = key_bytes_of(key_type);
  DevSetup su;
  if (int rc = su.open()) return rc;
  const TopkLayout tl = topk_layout(kb, n_rows, row_len, k, soa);
  if (int rc = su.workspace(stream, caller_workspace, workspace_bytes, tl.total)) return rc;

  // 1. the selection: the k winners of every row, unordered, into (keys, out_index)
  CUDA_TRY(cudaMemsetAsync(su.ws, 0, tl.zero_bytes, stream));
  TopkArgs a{};
  a.keys = (const unsigned char *)in[0].ptr; a.stride = in[0].elem_bytes; a.n_rows = (uint32_t)n_rows;
  a.row_len = row_len; a.k = k; a.cap = tl.cap; a.chunks_per_row = tl.chunks_per_row;
  a.ko = make_key_order(key_type, !largest);
  a.rows = (TopkRow *)su.ws; a.hist = (unsigned long long *)(su.ws + tl.hist_off); a.ctrl = (TopkCtrl *)(su.ws + tl.ctrl_off);
  a.item_row = (uint32_t *)(su.ws + tl.items_off);
  for (int b = 0; b < 2; b++) { a.cand_key[b] = su.ws + tl.cand_key_off[b]; a.cand_pos[b] = (unsigned long long *)(su.ws + tl.cand_pos_off[b]); }
  void *sel_keys = soa ? out[0].ptr : (void *)(su.ws + tl.keys_off);
  a.out_keys = sel_keys; a.out_index = out_index; a.offsets = (int64_t *)(su.ws + tl.offsets_off);
  const unsigned init_grid = (unsigned)std::min<int64_t>((n_rows + 256) / 256, (int64_t)su.di.sm_count * 8);
  CUDA_TRY(launch(PK_SELECT, topk_init_kernel, init_grid, 256, 0, stream, a));
  const unsigned pass_grid = (unsigned)std::min<int64_t>(n_rows * tl.chunks_per_row, (int64_t)su.di.sm_count * TOPK_PASS_CTAS_PER_SM);
  const unsigned decide_grid = (unsigned)std::min<int64_t>(n_rows, (int64_t)su.di.sm_count * 8);
  // (key-width + 1 passes and key-width decisions, whatever the keys: rows with nothing left to do exit at once)
  for (int p = 0; p <= kb; p++) {
    a.pass = p;
    CUDA_TRY(with_kb(kb, [&](auto K) { return launch(PK_SELECT, topk_pass_kernel<decltype(K)::value>, pass_grid, TOPK_THREADS, 0, stream, a); }));
    if (p < kb)
      CUDA_TRY(with_kb(kb, [&](auto K) { return launch(PK_SELECT, topk_decide_kernel<decltype(K)::value>, decide_grid, RADIX, 0, stream, a); }));
  }

  // 2. the order: the (key, index) pairs of the n_rows segments of k records sorted by the segmented sort, in the
  //    direction of the output (its waits: see include/b200sort.h).  Segments of one record need no sort.
  if (k > 1) {
    const std::vector<StreamDesc> pairs = {{sel_keys, (uint32_t)kb}, {out_index, 8u}};
    b200sort_stats inner;
    if (int rc = sort_segmented_device(o, key_type, !largest, n_rows * k, n_rows, a.offsets, pairs, true, stream, su.ws + tl.seg_off,
                                       tl.total - tl.seg_off, &inner))
      return rc;
  }

  // 3. the payloads (or the AoS records) of the winners, in that order
  TopkGatherSet g{};
  g.row_len = row_len; g.k = k; g.total = n_rows * k; g.index = out_index;
  for (size_t s = soa ? 1 : 0; s < in.size(); s++) {
    uint32_t c = 16;
    const uint32_t eb = in[s].elem_bytes;
    while (c > 1 && ((eb % c) != 0 || ((uintptr_t)in[s].ptr % c) != 0 || ((uintptr_t)out[s].ptr % c) != 0)) c >>= 1;
    g.s[g.n_streams++] = {(const unsigned char *)in[s].ptr, (unsigned char *)out[s].ptr, c, eb / c};
  }
  if (g.n_streams > 0) {
    const unsigned grid = (unsigned)std::min<int64_t>((g.total + 255) / 256, (int64_t)su.di.sm_count * 16);
    CUDA_TRY(launch(PK_SELECT, topk_gather_kernel, grid, 256, 0, stream, g));
  }
  *stats = su.stats(n_rows * row_len, in, kb, ALGO_TOPK);
  return B200SORT_OK;
}

// argument checks (all before any device work), then the selection on the arrays' device.  in / out as in topk_device,
// shapes checked by check_soa / check_aos.
static int topk_any(int key_type, int64_t n_rows, int64_t row_len, int64_t k, bool largest, const std::vector<StreamDesc> &in,
                    const std::vector<StreamDesc> &out, int64_t *out_index, bool soa, void *stream_v, void *workspace,
                    size_t workspace_bytes) {
  const int kb = key_bytes_of(key_type);
  if (k == 0 || n_rows == 0) return B200SORT_OK;
  for (size_t s = 0; s < in.size(); s++) {
    if (in[s].ptr == nullptr) return fail(B200SORT_EINVAL, s == 0 ? "the input is NULL" : "payload %zu is NULL", s - 1);
    if (out[s].ptr == nullptr) return fail(B200SORT_EINVAL, s == 0 ? "the key / record output is NULL" : "output payload %zu is NULL", s - 1);
  }
  if (out_index == nullptr) return fail(B200SORT_EINVAL, "out_index is NULL");
  if ((uintptr_t)in[0].ptr % kb != 0 || (uintptr_t)out[0].ptr % kb != 0) return fail(B200SORT_EINVAL, "keys / records are not aligned to their key type");
  if ((uintptr_t)out_index % 8 != 0) return fail(B200SORT_EINVAL, "out_index is not 8-byte aligned");
  const size_t num = (size_t)(n_rows * row_len), sel = (size_t)(n_rows * k);
  std::vector<ByteRange> ins, outs = {{out_index, sel * 8}};
  for (const StreamDesc &d : in) ins.push_back({d.ptr, num * d.elem_bytes});
  for (const StreamDesc &d : out) outs.push_back({d.ptr, sel * d.elem_bytes});
  if (int rc = check_disjoint(ins, outs)) return rc;

  std::vector<StreamDesc> all = in;
  all.insert(all.end(), out.begin(), out.end());
  all.push_back({out_index, 8u});
  CallScope call;
  if (int rc = call.enter(all, nullptr, "top-k")) return rc;
  return call.done(topk_device(call.o, key_type, largest, n_rows, row_len, k, in, out, out_index, soa, (cudaStream_t)stream_v, workspace,
                               workspace_bytes, &call.stats));
}

// the checks of the three counts: EINVAL unless 0 <= k <= row_len, 0 <= n_rows < 2^31 and n_rows * row_len fits
static int check_topk_shape(int64_t n_rows, int64_t row_len, int64_t k) {
  if (n_rows < 0 || row_len < 0 || k < 0) return fail(B200SORT_EINVAL, "negative n_rows, row_len or k");
  if (k > row_len) return fail(B200SORT_EINVAL, "k = %lld exceeds row_len = %lld", (long long)k, (long long)row_len);
  if (n_rows > INT32_MAX) return fail(B200SORT_EINVAL, "%lld rows (0..2^31-1 supported)", (long long)n_rows);
  if (row_len > 0 && n_rows > INT64_MAX / row_len) return fail(B200SORT_EINVAL, "n_rows * row_len overflows");
  return 0;
}

}  // namespace b200sort

extern "C" {

int b200sort_topk_soa(const void *keys, int key_type, int64_t n_rows, int64_t row_len, int64_t k, int largest, int n_payloads,
                      const void *const *payloads, const uint32_t *payload_elem_bytes, void *out_keys, int64_t *out_index,
                      void *const *out_payloads, void *stream, void *workspace, size_t workspace_bytes) {
  if (key_bytes_of(key_type) == 0) return fail(B200SORT_EINVAL, "unknown key type %d", key_type);
  if (int rc = check_topk_shape(n_rows, row_len, k)) return rc;
  std::vector<StreamDesc> in, out;
  // (check_soa only reads the payload pointers; the inputs are never written.  NULL arrays: topk_any, when k > 0)
  if (int rc = check_soa(const_cast<void *>(keys), key_type, 0, n_payloads, const_cast<void *const *>(payloads),
                         payload_elem_bytes, &in))
    return rc;
  if (n_payloads > 0 && out_payloads == nullptr && k > 0 && n_rows > 0) return fail(B200SORT_EINVAL, "out_payloads is NULL");
  out.push_back({out_keys, in[0].elem_bytes});
  for (int p = 0; p < n_payloads; p++) out.push_back({out_payloads ? out_payloads[p] : nullptr, in[p + 1].elem_bytes});
  return topk_any(key_type, n_rows, row_len, k, largest != 0, in, out, out_index, true, stream, workspace, workspace_bytes);
}

int b200sort_topk_aos(const void *records, int key_type, uint32_t record_bytes, int64_t n_rows, int64_t row_len, int64_t k, int largest,
                      void *out_records, int64_t *out_index, void *stream, void *workspace, size_t workspace_bytes) {
  if (key_bytes_of(key_type) == 0) return fail(B200SORT_EINVAL, "unknown key type %d", key_type);
  if (int rc = check_topk_shape(n_rows, row_len, k)) return rc;
  std::vector<StreamDesc> in;
  if (int rc = check_aos(const_cast<void *>(records), key_type, record_bytes, 0, &in)) return rc;
  const std::vector<StreamDesc> out = {{out_records, record_bytes}};
  return topk_any(key_type, n_rows, row_len, k, largest != 0, in, out, out_index, false, stream, workspace, workspace_bytes);
}

size_t b200sort_topk_workspace_bytes(int key_type, int64_t n_rows, int64_t row_len, int64_t k, int n_payloads,
                                     const uint32_t *payload_elem_bytes, uint32_t record_bytes) {
  (void)n_payloads; (void)payload_elem_bytes;  // (the payloads move straight from input to output)
  const int kb = key_bytes_of(key_type);
  if (kb == 0 || n_rows < 0 || row_len < 0 || k < 0 || k > row_len || n_rows > INT32_MAX || (row_len > 0 && n_rows > INT64_MAX / row_len))
    return 0;
  return topk_layout(kb, n_rows, row_len, k, record_bytes == 0).total;
}

}  // extern "C"
