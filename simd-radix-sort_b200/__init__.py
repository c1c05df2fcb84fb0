"""simd-radix-sort_b200: B200 (sm_100a) drop-in for the sort of jonicho/simd-radix-sort.

Host-side mirror of the reference interface (radixSort.hpp:1761-1783):

    sort(num, keys, *payloads, up=True)              <- simd_sort::radix_sort::sort<Up>(num, keys, payloads...)
    sort_combined(num, records, key_dtype, up=True)  <- simd_sort::radix_sort::sort<Up>(num, DataElement<K,Ps...>*)

and, as an extension without a counterpart there, segmented sorts of many independent segments in one call:

    sort_segmented(offsets, keys, *payloads, up=True)
    sort_segmented_combined(offsets, records, key_dtype, up=True)
    sort_rows(keys, *payloads, up=True)              <- every row of a (B, L) array, like torch.sort(dim=-1)

Both sort IN PLACE, like the reference, and go through the C ABI of include/b200sort.h
(libb200sort.so, hand-written CUDA for sm_100a).  There is no CPU implementation in this package:
if the library is missing or no CUDA device is usable the calls raise.
"""
from ._api import (B200SortError, KEY_TYPES, last_profile, last_stats, launch_count, lib, lib_path, options, set_option, get_option,
                   segmented_workspace_bytes, sort, sort_combined, sort_rows, sort_segmented, sort_segmented_combined, workspace_bytes,
                   version)

__all__ = ["B200SortError", "KEY_TYPES", "last_profile", "last_stats", "launch_count", "lib", "lib_path", "options", "set_option",
           "get_option", "segmented_workspace_bytes", "sort", "sort_combined", "sort_rows", "sort_segmented", "sort_segmented_combined",
           "workspace_bytes", "version"]
