"""simd-radix-sort_b200: B200 (sm_100a) drop-in for the sort of jonicho/simd-radix-sort.

Host-side mirror of the reference interface (radixSort.hpp:1761-1783):

    sort(num, keys, *payloads, up=True)              <- simd_sort::radix_sort::sort<Up>(num, keys, payloads...)
    sort_combined(num, records, key_dtype, up=True)  <- simd_sort::radix_sort::sort<Up>(num, DataElement<K,Ps...>*)

and, as an extension without a counterpart there, segmented sorts of many independent segments in one call:

    sort_segmented(offsets, keys, *payloads, up=True)
    sort_segmented_combined(offsets, records, key_dtype, up=True)
    sort_rows(keys, *payloads, up=True)              <- every row of a (B, L) array, like torch.sort(dim=-1)

and a top-k selection that returns new arrays (device arrays only):

    topk(keys, k, *payloads, largest=True)           <- the k largest / smallest of a row or of every row, like torch.topk
    topk_combined(records, key_dtype, k, largest=True)

and unique, which also returns new arrays (device arrays only):

    unique(x, return_inverse=False, return_counts=False)              <- like torch.unique(sorted=True)
    unique_consecutive(x, return_inverse=False, return_counts=False)  <- like torch.unique_consecutive

The sorts work IN PLACE, like the reference, and go through the C ABI of include/b200sort.h
(libb200sort.so, hand-written CUDA for sm_100a).  There is no CPU implementation in this package:
if the library is missing or no CUDA device is usable the calls raise.
"""
from ._api import (B200SortError, KEY_TYPES, last_profile, last_stats, launch_count, lib, lib_path, options, set_option, get_option,
                   segmented_workspace_bytes, sort, sort_combined, sort_rows, sort_segmented, sort_segmented_combined, topk, topk_combined,
                   topk_workspace_bytes, unique, unique_consecutive, unique_workspace_bytes, workspace_bytes, version)

__all__ = ["B200SortError", "KEY_TYPES", "last_profile", "last_stats", "launch_count", "lib", "lib_path", "options", "set_option",
           "get_option", "segmented_workspace_bytes", "sort", "sort_combined", "sort_rows", "sort_segmented", "sort_segmented_combined",
           "topk", "topk_combined", "topk_workspace_bytes", "unique", "unique_consecutive", "unique_workspace_bytes", "workspace_bytes",
           "version"]
