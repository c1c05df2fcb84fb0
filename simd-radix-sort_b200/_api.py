"""ctypes binding of include/b200sort.h + the Python mirror of the reference's sort<> overloads."""
from __future__ import annotations

import contextlib
import ctypes
from pathlib import Path

import numpy as np

_PKG = Path(__file__).resolve().parent
_LIB_PATH = _PKG / "libb200sort.so"

# key type codes of include/b200sort.h (same order as the reference's test matrix, src/test.cpp:155-169)
KEY_TYPES = {"uint8": 0, "int8": 1, "uint16": 2, "int16": 3, "uint32": 4, "int32": 5, "uint64": 6, "int64": 7,
             "float32": 8, "float64": 9}


class B200SortError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"b200sort error {code}: {message}")
        self.code = code


class _Stats(ctypes.Structure):
    _fields_ = [("num", ctypes.c_int64), ("record_bytes", ctypes.c_uint32), ("key_bytes", ctypes.c_uint32),
                ("algo", ctypes.c_uint32), ("passes_planned", ctypes.c_uint32), ("hist_sweeps", ctypes.c_uint32),
                ("kernel_launches", ctypes.c_uint32), ("segfix_passes", ctypes.c_uint32), ("cut_digit", ctypes.c_uint32),
                ("fell_back", ctypes.c_uint32), ("algorithmic_bytes", ctypes.c_uint64), ("segfix_moved", ctypes.c_uint64)]


_lib = None

# b200sort_hist_fn (include/b200sort.h): histogram callback of the splitter refinement
HIST_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_int),
                           ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(ctypes.c_uint64))


def lib_path() -> Path:
    return _LIB_PATH


def lib():
    """The loaded C-ABI library.  Fails loudly when it has not been built (no fallback exists)."""
    global _lib
    if _lib is None:
        if not _LIB_PATH.exists():
            raise B200SortError(-5, f"{_LIB_PATH} not built: run `python simd-radix-sort_b200/build.py` "
                                    "(nvcc, sm_100a); there is no CPU fallback")
        L = ctypes.CDLL(str(_LIB_PATH))
        vp, i32, i64, u32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint32
        vpp, u32p, sz = ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_uint32), ctypes.c_size_t
        L.b200sort_sort_soa.argtypes = [vp, i32, i64, i32, i32, vpp, u32p, vp, vp, sz]
        L.b200sort_sort_soa.restype = i32
        L.b200sort_sort_aos.argtypes = [vp, i32, u32, i64, i32, vp, vp, sz]
        L.b200sort_sort_aos.restype = i32
        L.b200sort_sort_soa_ex.argtypes = [vp, i32, i64, i32, i32, vpp, u32p, i64, i32, vp, vp, sz]
        L.b200sort_sort_soa_ex.restype = i32
        L.b200sort_sort_aos_ex.argtypes = [vp, i32, u32, i64, i32, i64, i32, vp, vp, sz]
        L.b200sort_sort_aos_ex.restype = i32
        L.b200sort_workspace_bytes.argtypes = [i32, i64, i32, u32p, u32]
        L.b200sort_workspace_bytes.restype = sz
        L.b200sort_sort_segmented_soa.argtypes = [vp, i32, i64, i64, vp, i32, i32, vpp, u32p, vp, vp, sz]
        L.b200sort_sort_segmented_soa.restype = i32
        L.b200sort_sort_segmented_aos.argtypes = [vp, i32, u32, i64, i64, vp, i32, vp, vp, sz]
        L.b200sort_sort_segmented_aos.restype = i32
        L.b200sort_segmented_workspace_bytes.argtypes = [i32, i64, i64, i32, u32p, u32]
        L.b200sort_segmented_workspace_bytes.restype = sz
        L.b200sort_topk_soa.argtypes = [vp, i32, i64, i64, i64, i32, i32, vpp, u32p, vp, vp, vpp, vp, vp, sz]
        L.b200sort_topk_soa.restype = i32
        L.b200sort_topk_aos.argtypes = [vp, i32, u32, i64, i64, i64, i32, vp, vp, vp, vp, sz]
        L.b200sort_topk_aos.restype = i32
        L.b200sort_topk_workspace_bytes.argtypes = [i32, i64, i64, i64, i32, u32p, u32]
        L.b200sort_topk_workspace_bytes.restype = sz
        L.b200sort_unique.argtypes = [vp, i32, i64, i32, vp, vp, vp, vp, vp, vp, sz]
        L.b200sort_unique.restype = i32
        L.b200sort_unique_workspace_bytes.argtypes = [i32, i64, i32, i32]
        L.b200sort_unique_workspace_bytes.restype = sz
        L.b200sort_last_error.restype = ctypes.c_char_p
        L.b200sort_version.restype = i32
        L.b200sort_launch_count.restype = ctypes.c_uint64
        L.b200sort_set_option.argtypes = [ctypes.c_char_p, i64]
        L.b200sort_set_option.restype = i32
        L.b200sort_get_option.argtypes = [ctypes.c_char_p]
        L.b200sort_get_option.restype = i64
        L.b200sort_last_stats.argtypes = [ctypes.POINTER(_Stats)]
        L.b200sort_last_stats.restype = i32
        L.b200sort_release_cache.restype = None
        L.b200sort_last_profile.argtypes = [ctypes.POINTER(i32), ctypes.POINTER(ctypes.c_float), i32]
        L.b200sort_last_profile.restype = i32
        L.b200sort_mgpu_unique_id.argtypes = [vp]
        L.b200sort_mgpu_unique_id.restype = i32
        L.b200sort_mgpu_comm_create.argtypes = [vpp, i32, i32, vp]
        L.b200sort_mgpu_comm_create.restype = i32
        L.b200sort_mgpu_comm_destroy.argtypes = [vp]
        L.b200sort_mgpu_comm_destroy.restype = i32
        L.b200sort_mgpu_splitters.argtypes = [ctypes.POINTER(ctypes.c_uint64), i32, i32, u32p]
        L.b200sort_mgpu_splitters.restype = i32
        L.b200sort_mgpu_sort_soa.argtypes = [vp, vp, i32, i64, i64, i32, i32, vpp, u32p, ctypes.POINTER(i64), vp]
        L.b200sort_mgpu_sort_soa.restype = i32
        L.b200sort_mgpu_sort_aos.argtypes = [vp, vp, i32, u32, i64, i64, i32, ctypes.POINTER(i64), vp]
        L.b200sort_mgpu_sort_aos.restype = i32
        L.b200sort_mgpu_used_p2p.argtypes = [vp]
        L.b200sort_mgpu_used_p2p.restype = i32
        L.b200sort_mgpu_used_overlap.argtypes = [vp]
        L.b200sort_mgpu_used_overlap.restype = i32
        L.b200sort_mgpu_refine_splitters.argtypes = [i32, i32, ctypes.c_uint64, HIST_FN, vp, ctypes.POINTER(ctypes.c_uint64), u32p]
        L.b200sort_mgpu_refine_splitters.restype = i32
        L.b200sort_mgpu_tie_thresholds.argtypes = [i32, i32, i32, ctypes.c_uint64, u32p, i32, ctypes.POINTER(ctypes.c_uint64), u32p]
        L.b200sort_mgpu_tie_thresholds.restype = i32
        _lib = L
    return _lib


def _check(rc: int):
    if rc != 0:
        raise B200SortError(rc, lib().b200sort_last_error().decode())


def version() -> int:
    return lib().b200sort_version()


def launch_count() -> int:
    return int(lib().b200sort_launch_count())


def set_option(name: str, value: int):
    _check(lib().b200sort_set_option(name.encode(), int(value)))


def get_option(name: str) -> int:
    return int(lib().b200sort_get_option(name.encode()))


@contextlib.contextmanager
def options(**values):
    """Sets options for the body of a `with` block: `with options(algo=2, margin_bits=-2): ...`.

    The values they had before are restored on the way out, also when the body raises.  Options are
    process-wide defaults that a sort reads once when it starts."""
    saved = {}
    try:
        for name, value in values.items():
            before = get_option(name)
            set_option(name, value)
            saved[name] = before
        yield
    finally:
        for name, value in saved.items():
            set_option(name, value)


def last_stats() -> dict:
    s = _Stats()
    _check(lib().b200sort_last_stats(ctypes.byref(s)))
    return {f: getattr(s, f) for f, _ in _Stats._fields_}


PROFILE_KINDS = ["hist", "scan", "sweep", "copyback", "segfix", "other", "segment", "select", "unique"]


def last_profile():
    """[(kernel kind, milliseconds)] of the last sort on this thread (needs set_option("profile", 1))."""
    kinds = (ctypes.c_int * 256)()
    ms = (ctypes.c_float * 256)()
    n = lib().b200sort_last_profile(kinds, ms, 256)
    if n < 0:
        _check(n)
    return [(PROFILE_KINDS[kinds[i]], float(ms[i])) for i in range(n)]


# ---------------------------------------------------------------------------------------------
# array plumbing: torch tensors (cuda or cpu) and numpy arrays are accepted; nothing is copied here
# ---------------------------------------------------------------------------------------------
def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


def _describe(x):
    """-> (address, dtype name, bytes per element, number of elements, is_cuda).

    A 2-D (or higher) array is a stream whose elements are its rows (e.g. a (num, 16) uint8 array is a
    stream of 16-byte payload elements)."""
    if _is_torch(x):
        if not x.is_contiguous():
            raise ValueError("arrays must be contiguous")
        rows = x.shape[0] if x.dim() > 0 else 1
        per_row = (x.numel() // rows if rows else int(np.prod(x.shape[1:]))) if x.dim() > 1 else 1
        return x.data_ptr(), str(x.dtype).replace("torch.", ""), x.element_size() * per_row, rows, x.is_cuda
    a = x
    if not isinstance(a, np.ndarray) or not a.flags.c_contiguous:
        raise ValueError("arrays must be contiguous numpy arrays or torch tensors")
    if not a.flags.writeable:
        raise ValueError("arrays are sorted in place and must be writeable")
    rows = a.shape[0] if a.ndim > 0 else 1
    per_row = int(np.prod(a.shape[1:])) if a.ndim > 1 else 1
    return a.ctypes.data, a.dtype.name, a.dtype.itemsize * per_row, rows, False


def _stream_for(arrays, stream):
    if stream is not None:
        return ctypes.c_void_p(int(stream))
    for x in arrays:
        if _is_torch(x) and x.is_cuda:
            import torch
            return ctypes.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)
    return ctypes.c_void_p(0)


def _device_guard(arrays):
    for x in arrays:
        if _is_torch(x) and x.is_cuda:
            import torch
            return torch.cuda.device(x.device)
    return contextlib.nullcontext()


def _key_code(key_dtype) -> int:
    """The key type code of a dtype (numpy, or anything np.dtype takes) or a dtype name such as "int32"."""
    name = key_dtype if isinstance(key_dtype, str) else np.dtype(key_dtype).name
    if name not in KEY_TYPES:
        raise TypeError(f"unsupported key type {name}; the reference sorts {sorted(KEY_TYPES)}")
    return KEY_TYPES[name]


def _payload_args(payloads, num: int):
    """-> (count, addresses, element sizes) of the payload arrays, as the C calls take them; each has at least num rows"""
    n = len(payloads)
    ptrs = (ctypes.c_void_p * max(n, 1))()
    sizes = (ctypes.c_uint32 * max(n, 1))()
    for i, p in enumerate(payloads):
        addr, _, item, pn, _ = _describe(p)
        if pn < num:
            raise ValueError(f"payload {i} has fewer than {num} rows")
        ptrs[i], sizes[i] = addr, item
    return n, ptrs, sizes


def _call(fn, arrays, stream, workspace, *args):
    """fn(*args, stream, workspace address, workspace bytes) on the device and stream of the arrays (unless `stream` is
    given); raises B200SortError when it fails."""
    ws = (None, 0) if workspace is None else (workspace.data_ptr(), workspace.numel() * workspace.element_size())
    with _device_guard(arrays):
        rc = fn(*args, _stream_for(arrays, stream), *ws)
    _check(rc)


def sort(num, keys, *payloads, up: bool = True, stream=None, cmp_sort_threshold: int | None = None,
         cmp_sorter: int = 0, workspace=None):
    """simd_sort::radix_sort::sort<Up>(num, keys, payloads...)  (radixSort.hpp:1780-1783).

    Sorts `keys[:num]` in place, ascending (`up=True`) or descending, and applies the same
    permutation to every payload array.  With `cmp_sort_threshold` the advanced overload
    sort<Up,BitSorter,CmpSorter>(thresh, num, ...) (src/radix_sort.hpp:297-312) is mirrored.
    """
    kaddr, kname, _, kn, _ = _describe(keys)
    if num < 0 or num > kn:
        raise ValueError("num exceeds the key array")
    pay = _payload_args(payloads, num)
    args = (kaddr, _key_code(kname), num, int(up), *pay)
    if cmp_sort_threshold is None:
        _call(lib().b200sort_sort_soa, (keys,) + payloads, stream, workspace, *args)
    else:
        _call(lib().b200sort_sort_soa_ex, (keys,) + payloads, stream, workspace, *args, cmp_sort_threshold, cmp_sorter)


def sort_combined(num, records, key_dtype, up: bool = True, stream=None, workspace=None):
    """simd_sort::radix_sort::sort<Up>(num, (DataElement<K,Ps...>*)records)  (radixSort.hpp:1770-1778).

    `records` is a contiguous (num, record_bytes) uint8 tensor/array (or any contiguous array whose
    rows are the records); the key of type `key_dtype` sits at byte offset 0 of every record and
    record_bytes must be a power of two (the reference's static_assert, src/radix_sort.hpp:318-319).
    """
    addr, _, record_bytes, rows, _ = _describe(records)
    if rows < num:
        raise ValueError("num exceeds the record array")
    _call(lib().b200sort_sort_aos, (records,), stream, workspace, addr, _key_code(key_dtype), record_bytes, num, int(up))


def workspace_bytes(key_dtype, num: int, payload_itemsizes=(), record_bytes: int = 0) -> int:
    n = len(payload_itemsizes)
    sizes = (ctypes.c_uint32 * max(n, 1))(*payload_itemsizes)
    return int(lib().b200sort_workspace_bytes(_key_code(key_dtype), num, n, sizes, record_bytes))


def _offsets_arg(offsets):
    """-> (address, n_segments) of a contiguous 1-D int64 offsets array (n_segments + 1 values)"""
    addr, name, _, count, _ = _describe(offsets)
    if name != "int64":
        raise TypeError(f"offsets must be int64, not {name}")
    if count < 1:
        raise ValueError("offsets holds n_segments + 1 values, at least one")
    return addr, count - 1


def sort_segmented(offsets, keys, *payloads, up: bool = True, stream=None, workspace=None):
    """Sorts every segment keys[offsets[i]:offsets[i+1]] on its own, in place, and applies each segment's
    permutation to the payload arrays (b200sort_sort_segmented_soa; an extension, the reference has none).

    `offsets` is a 1-D int64 array or tensor of n_segments + 1 non-decreasing values in [0, len(keys)],
    on the same side (and device) as the arrays.  Records outside [offsets[0], offsets[-1]) are not touched."""
    kaddr, kname, _, num, _ = _describe(keys)
    oaddr, n_seg = _offsets_arg(offsets)
    pay = _payload_args(payloads, num)
    _call(lib().b200sort_sort_segmented_soa, (keys,) + payloads, stream, workspace, kaddr, _key_code(kname), num, n_seg, oaddr, int(up),
          *pay)


def sort_segmented_combined(offsets, records, key_dtype, up: bool = True, stream=None, workspace=None):
    """sort_segmented for combined records (b200sort_sort_segmented_aos): `records` as in sort_combined."""
    addr, _, record_bytes, num, _ = _describe(records)
    oaddr, n_seg = _offsets_arg(offsets)
    _call(lib().b200sort_sort_segmented_aos, (records,), stream, workspace, addr, _key_code(key_dtype), record_bytes, num, n_seg, oaddr,
          int(up))


def segmented_workspace_bytes(key_dtype, num: int, n_segments: int, payload_itemsizes=(), record_bytes: int = 0) -> int:
    n = len(payload_itemsizes)
    sizes = (ctypes.c_uint32 * max(n, 1))(*payload_itemsizes)
    return int(lib().b200sort_segmented_workspace_bytes(_key_code(key_dtype), num, n_segments, n, sizes, record_bytes))


def sort_rows(keys, *payloads, up: bool = True, stream=None):
    """Sorts every row of a contiguous (B, L) array or tensor in place, like torch.sort(keys, dim=-1), and
    applies each row's permutation to the payloads, whose first two dimensions are (B, L)."""
    if keys.ndim != 2:
        raise ValueError("keys must be 2-D (B, L)")
    B, L = int(keys.shape[0]), int(keys.shape[1])
    for i, p in enumerate(payloads):
        if p.ndim < 2 or tuple(p.shape[:2]) != (B, L):
            raise ValueError(f"payload {i} does not have the keys' (B, L) shape")

    # 2-D arrays are streams of row-sized elements (_describe): pass flat views, one element per (row, column)
    def flat(x):
        return x.reshape(B * L) if x.ndim == 2 else x.reshape(B * L, -1)

    if _is_torch(keys):
        import torch
        if keys.is_cuda and stream is not None:
            # the offsets are made on the stream the sort runs on, and freed only after it
            with torch.cuda.stream(torch.cuda.ExternalStream(int(stream), device=keys.device)):
                offsets = torch.arange(B + 1, dtype=torch.int64, device=keys.device) * L
                sort_segmented(offsets, flat(keys), *[flat(p) for p in payloads], up=up, stream=stream)
            return
        offsets = torch.arange(B + 1, dtype=torch.int64, device=keys.device) * L
    else:
        offsets = np.arange(B + 1, dtype=np.int64) * L
    sort_segmented(offsets, flat(keys), *[flat(p) for p in payloads], up=up, stream=stream)


def _empty(like, shape, dtype=None):
    """a new array of `shape` where `like` lives (a torch tensor on its device, or a numpy array); `like`'s dtype unless given"""
    if _is_torch(like):
        import torch
        return torch.empty(shape, dtype=like.dtype if dtype is None else dtype, device=like.device)
    return np.empty(shape, dtype=like.dtype if dtype is None else dtype)


def _index_dtype(like):
    if _is_torch(like):
        import torch
        return torch.int64
    return np.int64


def _itemsize(x) -> int:
    return x.element_size() if _is_torch(x) else x.dtype.itemsize


def _on_stream(like, stream, fn):
    """fn() with a given CUDA `stream` current, so that the arrays fn allocates belong to the stream the call runs on"""
    if stream is not None and _is_torch(like) and like.is_cuda:
        import torch
        with torch.cuda.stream(torch.cuda.ExternalStream(int(stream), device=like.device)):
            return fn()
    return fn()


def _topk_shape(lead, k):
    """-> (n_rows, row_len) of keys of shape `lead` (1-D: one row; 2-D: (B, L)); k must be in [0, L]"""
    if len(lead) not in (1, 2):
        raise ValueError("keys must be 1-D (one row) or 2-D (B, L)")
    n_rows, row_len = (1, lead[0]) if len(lead) == 1 else lead
    if not 0 <= k <= row_len:
        raise ValueError(f"k = {k} is not in [0, {row_len}]")
    return n_rows, row_len


def topk(keys, k: int, *payloads, largest: bool = True, stream=None, workspace=None):
    """The k largest (or smallest) keys of a 1-D array, or of every row of a 2-D (B, L) one, like torch.topk(dim=-1):
    -> (values, indices, *payload outputs), new arrays of shape (..., k) (plus each payload's trailing dimensions)
    where the keys are (b200sort_topk_soa).

    values are in descending order for largest=True and ascending otherwise, in the library's total order of bit
    patterns; indices are int64 positions inside the row; every payload's leading dimensions equal the keys' shape,
    and its output holds the elements at the selected positions.  The keys must be on a CUDA device: host arrays
    raise B200SortError with code -7."""
    kaddr, kname, _, _, _ = _describe(keys)
    lead, k = tuple(int(d) for d in keys.shape), int(k)
    n_rows, row_len = _topk_shape(lead, k)
    for i, p in enumerate(payloads):
        if tuple(p.shape[:len(lead)]) != lead:
            raise ValueError(f"payload {i} does not have the keys' leading shape {lead}")
    code = _key_code(kname)
    out_shape = lead[:-1] + (k,)
    sizes = (ctypes.c_uint32 * max(len(payloads), 1))()
    ptrs = (ctypes.c_void_p * max(len(payloads), 1))()
    for i, p in enumerate(payloads):
        ptrs[i] = _describe(p)[0]
        sizes[i] = _itemsize(p) * int(np.prod(p.shape[len(lead):], dtype=np.int64))

    def run():
        values, indices = _empty(keys, out_shape), _empty(keys, out_shape, _index_dtype(keys))
        outs = [_empty(p, out_shape + tuple(p.shape[len(lead):])) for p in payloads]
        out_ptrs = (ctypes.c_void_p * max(len(outs), 1))(*[_describe(o)[0] for o in outs])
        _call(lib().b200sort_topk_soa, (keys,) + payloads, stream, workspace, kaddr, code, n_rows, row_len, k, int(largest),
              len(payloads), ptrs, sizes, _describe(values)[0], _describe(indices)[0], out_ptrs)
        return (values, indices, *outs)

    return _on_stream(keys, stream, run)


def topk_combined(records, key_dtype, k: int, largest: bool = True, stream=None, workspace=None):
    """topk for combined records (b200sort_topk_aos): `records` is (L, R) for one row or (B, L, R) for rows, whose last
    dimension holds the record's bytes (a power of two, key of `key_dtype` at byte offset 0).  -> (records_out,
    indices) of shapes (..., k, R) and (..., k)."""
    addr, _, _, _, _ = _describe(records)
    if records.ndim not in (2, 3):
        raise ValueError("records must be (L, R) or (B, L, R)")
    lead, k = tuple(int(d) for d in records.shape[:-1]), int(k)
    n_rows, row_len = _topk_shape(lead, k)
    record_bytes = _itemsize(records) * int(records.shape[-1])
    code = _key_code(key_dtype)

    def run():
        out = _empty(records, lead[:-1] + (k, int(records.shape[-1])))
        indices = _empty(records, lead[:-1] + (k,), _index_dtype(records))
        _call(lib().b200sort_topk_aos, (records,), stream, workspace, addr, code, record_bytes, n_rows, row_len, k, int(largest),
              _describe(out)[0], _describe(indices)[0])
        return out, indices

    return _on_stream(records, stream, run)


def topk_workspace_bytes(key_dtype, n_rows: int, row_len: int, k: int, payload_itemsizes=(), record_bytes: int = 0) -> int:
    """Bytes of workspace a topk (record_bytes = 0) or topk_combined call of these shapes needs, whatever the keys."""
    n = len(payload_itemsizes)
    sizes = (ctypes.c_uint32 * max(n, 1))(*payload_itemsizes)
    return int(lib().b200sort_topk_workspace_bytes(_key_code(key_dtype), n_rows, row_len, k, n, sizes, record_bytes))


def _unique(x, consecutive: bool, return_inverse: bool, return_counts: bool, stream, workspace):
    flat = x.reshape(-1)
    kaddr, kname, _, num, _ = _describe(flat)
    code = _key_code(kname)

    def run():
        values, n_unique = _empty(flat, (num,)), _empty(flat, (1,), _index_dtype(flat))
        inverse = _empty(flat, tuple(x.shape), _index_dtype(flat)) if return_inverse else None
        counts = _empty(flat, (num,), _index_dtype(flat)) if return_counts else None
        _call(lib().b200sort_unique, (flat,), stream, workspace, kaddr, code, num, int(consecutive), _describe(values)[0],
              None if counts is None else _describe(counts)[0], None if inverse is None else _describe(inverse)[0],
              _describe(n_unique)[0])
        u = int(n_unique[0])  # (the call's one host wait)
        out = (values[:u],) + ((inverse,) if return_inverse else ()) + ((counts[:u],) if return_counts else ())
        return out[0] if len(out) == 1 else out

    return _on_stream(flat, stream, run)


def unique(x, return_inverse: bool = False, return_counts: bool = False, stream=None, workspace=None):
    """The distinct keys of `x` (flattened) in ascending order, like torch.unique(sorted=True) (b200sort_unique): -> values,
    or a tuple (values, inverse, counts) holding the ones asked for, in torch's order.

    Keys are equal when their bit patterns are: +0.0 and -0.0 are two values, and NaNs with the same bits are one (torch
    merges +-0.0 and keeps every NaN apart).  The order is the library's total order of bit patterns.  inverse has x's
    shape and dtype int64 (values[inverse] == x); counts are int64.  values and counts are views of the first U entries of
    arrays sized for x.numel(): they keep that storage alive.  Reading U waits for the device once.  The keys must be on
    a CUDA device: host arrays raise B200SortError with code -7."""
    return _unique(x, False, return_inverse, return_counts, stream, workspace)


def unique_consecutive(x, return_inverse: bool = False, return_counts: bool = False, stream=None, workspace=None):
    """One entry per maximal run of equal adjacent keys of `x` (flattened), in input order, like torch.unique_consecutive
    (b200sort_unique with consecutive = 1; no sort runs).  Returns and conventions as for unique."""
    return _unique(x, True, return_inverse, return_counts, stream, workspace)


def unique_workspace_bytes(key_dtype, num: int, consecutive: bool = False, return_inverse: bool = False) -> int:
    """Bytes of workspace a unique (or unique_consecutive) call on num keys needs, whatever the keys."""
    if num < 0:
        raise ValueError(f"num = {num} is negative")
    return int(lib().b200sort_unique_workspace_bytes(_key_code(key_dtype), num, int(consecutive), int(return_inverse)))
