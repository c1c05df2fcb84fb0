//=============================================================================
// b200sort/radixSort.hpp -- drop-in for the single header of jonicho/simd-radix-sort.
//
// Same names, same signatures, same static_asserts as the reference's
// radixSort.hpp (public surface at radixSort.hpp:1761-1783, record type at
// radixSort.hpp:180-195, SortIndex at radixSort.hpp:88), but every
// instantiation forwards, type-erased, to the C ABI of libb200sort.so
// (include/b200sort.h): the sort itself runs as hand-written CUDA kernels on a
// B200.  Replace
//     #include "radixSort.hpp"
// with
//     #include "b200sort/radixSort.hpp"
// and link -lb200sort.  No AVX-512 flags are needed any more.
//
//   simd_sort::radix_sort::sort(num, keyArray, payloadArrays...);
//   simd_sort::radix_sort::sort(num, (simd_sort::DataElement<K, Ps...> *)combinedArray);
//   simd_sort::radix_sort::sort<false>(...)   // descending
//
// Arrays may be host memory (staged through the GPU) or device memory (sorted
// in place on the device).  Like the reference the functions return void; a
// failing call (no CUDA device, out of memory ...) throws std::runtime_error
// carrying b200sort_last_error() -- there is no CPU fallback to hide it.
//
// Requires C++17 (the reference needs C++20; nothing here does).
//=============================================================================
#pragma once

#include <sys/types.h>

#include <cstddef>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <tuple>
#include <type_traits>

#include "../b200sort.h"

namespace simd_sort {

template <typename>
inline constexpr bool always_false_v = false;

using SortIndex = ssize_t;  // radixSort.hpp:88

template <std::size_t X>
inline constexpr bool is_power_of_two = X > 0 && (X & (X - 1)) == 0;  // radixSort.hpp:155-156

// radixSort.hpp:180-195 -- key first, payloads in a std::tuple, key-only comparison
template <typename K, typename... Ps>
struct DataElement {
  K key;
  std::tuple<Ps...> payloads;
  bool operator<(const DataElement &other) const { return key < other.key; }
  bool operator>(const DataElement &other) const { return key > other.key; }
};

template <typename K>
struct DataElement<K> {
  K key;
  bool operator<(const DataElement &other) const { return key < other.key; }
  bool operator>(const DataElement &other) const { return key > other.key; }
};

// tag types kept so that code naming the reference's policy classes still compiles
struct CmpSorterInsertionSort {
  static std::string name() { return "CmpSorterInsertionSort"; }
  static constexpr int b200sort_code = B200SORT_CMP_INSERTION;
};
struct CmpSorterNoSort {
  static std::string name() { return "CmpSorterNoSort"; }
  static constexpr int b200sort_code = B200SORT_CMP_NONE;
};

namespace radix_sort {

struct BitSorterSIMD {
  static std::string name() { return "BitSorterB200"; }
};
struct BitSorterSequential {
  static std::string name() { return "BitSorterB200"; }
};

namespace internal {

template <typename K>
constexpr int key_type_code() {
  using T = std::remove_cv_t<K>;
  if constexpr (std::is_same_v<T, float>) return B200SORT_F32;
  else if constexpr (std::is_same_v<T, double>) return B200SORT_F64;
  else if constexpr (std::is_integral_v<T> && !std::is_same_v<T, bool>) {
    if constexpr (sizeof(T) == 1) return std::is_signed_v<T> ? B200SORT_I8 : B200SORT_U8;
    else if constexpr (sizeof(T) == 2) return std::is_signed_v<T> ? B200SORT_I16 : B200SORT_U16;
    else if constexpr (sizeof(T) == 4) return std::is_signed_v<T> ? B200SORT_I32 : B200SORT_U32;
    else if constexpr (sizeof(T) == 8) return std::is_signed_v<T> ? B200SORT_I64 : B200SORT_U64;
    else return -1;
  } else return -1;
}

inline void check(int rc) {
  if (rc != B200SORT_OK) throw std::runtime_error(std::string("b200sort: ") + b200sort_last_error());
}

}  // namespace internal

// src/radix_sort.hpp:297-312 / radixSort.hpp:1761-1768
template <bool Up = true, typename BitSorter = BitSorterSIMD, typename CmpSorter = CmpSorterInsertionSort,
          typename K, typename... Ps>
void sort(SortIndex cmpSortThreshold, const SortIndex num, K *const keys, Ps *const... payloads) {
  static_assert(internal::key_type_code<K>() >= 0,
                "key type must be one of (u)int8/16/32/64, float, double");
  static_assert(((std::is_trivially_copyable_v<Ps> && sizeof(Ps) >= 1 && sizeof(Ps) <= 64) && ...),
                "payload types must be trivially copyable and at most 64 bytes");
  static_assert(sizeof...(Ps) <= 63, "at most 63 payload streams");
  void *ptrs[sizeof...(Ps) + 1] = {const_cast<void *>(static_cast<const void *>(payloads))..., nullptr};
  const uint32_t sizes[sizeof...(Ps) + 1] = {static_cast<uint32_t>(sizeof(Ps))..., 0u};
  internal::check(b200sort_sort_soa_ex(const_cast<std::remove_cv_t<K> *>(keys), internal::key_type_code<K>(), num,
                                       Up ? 1 : 0, static_cast<int>(sizeof...(Ps)), ptrs, sizes, cmpSortThreshold,
                                       CmpSorter::b200sort_code, nullptr, nullptr, 0));
}

// src/radix_sort.hpp:314-332 / radixSort.hpp:1770-1778
template <bool Up, typename BitSorter, typename CmpSorter, typename K, typename... Ps>
void sort(SortIndex cmpSortThreshold, const SortIndex num, DataElement<K, Ps...> *const elements) {
  static_assert(is_power_of_two<sizeof(DataElement<K, Ps...>)>,
                "size of DataElement<K, Ps...> must be a power of two");
  static_assert(sizeof(DataElement<K, Ps...>) <= 64, "records of at most 64 bytes are supported");
  static_assert(internal::key_type_code<K>() >= 0,
                "key type must be one of (u)int8/16/32/64, float, double");
  internal::check(b200sort_sort_aos_ex(elements, internal::key_type_code<K>(),
                                       static_cast<uint32_t>(sizeof(DataElement<K, Ps...>)), num, Up ? 1 : 0,
                                       cmpSortThreshold, CmpSorter::b200sort_code, nullptr, nullptr, 0));
}

// src/radix_sort.hpp:334-337 / radixSort.hpp:1780-1783
template <bool Up = true, typename K, typename... Ps>
void sort(const SortIndex num, K *const keys, Ps *const... payloads) {
  sort<Up, BitSorterSIMD, CmpSorterInsertionSort>(16, num, keys, payloads...);
}

// An extension with no counterpart in the reference: sorts every segment [offsets[i], offsets[i+1]) of
// keys[0, num) on its own (b200sort_sort_segmented_soa; `offsets` holds n_segments + 1 values and lives
// where the arrays do).
template <bool Up = true, typename K, typename... Ps>
void sort_segmented(const SortIndex num, const int64_t n_segments, const int64_t *const offsets, K *const keys,
                    Ps *const... payloads) {
  static_assert(internal::key_type_code<K>() >= 0,
                "key type must be one of (u)int8/16/32/64, float, double");
  static_assert(((std::is_trivially_copyable_v<Ps> && sizeof(Ps) >= 1 && sizeof(Ps) <= 64) && ...),
                "payload types must be trivially copyable and at most 64 bytes");
  static_assert(sizeof...(Ps) <= 63, "at most 63 payload streams");
  void *ptrs[sizeof...(Ps) + 1] = {const_cast<void *>(static_cast<const void *>(payloads))..., nullptr};
  const uint32_t sizes[sizeof...(Ps) + 1] = {static_cast<uint32_t>(sizeof(Ps))..., 0u};
  internal::check(b200sort_sort_segmented_soa(const_cast<std::remove_cv_t<K> *>(keys), internal::key_type_code<K>(), num,
                                              n_segments, offsets, Up ? 1 : 0, static_cast<int>(sizeof...(Ps)), ptrs, sizes,
                                              nullptr, nullptr, 0));
}

}  // namespace radix_sort
}  // namespace simd_sort
