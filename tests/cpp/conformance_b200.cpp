// conformance_b200.cpp -- TEST INFRASTRUCTURE: the reference's test matrix run against the GPU path.
//
// The matrix of jonicho/simd-radix-sort's only test (src/test.cpp:76-179): 10 key types x 14 payload shapes x
// separate/combined x ascending/descending x 8 distributions, sizes 1, 10, ... maxNum, every call through
// the C ABI of libb200sort.so (include/b200sort.h) with host arrays and the reference's threshold of 16.
// The generators follow the shape of the reference's Data<> (src/data.hpp:105-170, std::mt19937): Uniform
// over the key's full range (floats in (-1,1)), Gaussian N(0,100) rounded for integers and N(0,1) for
// floats, Zero, ZeroOne, Sorted, ReverseSorted and Almost(Reverse)Sorted (floor(2^log10(n)) random swaps).
// Like the reference, payload bytes are a function of their key; combined records are
// simd_sort::DataElement<K, Ps...>, and shapes whose size is not a power of two are not sorted combined.
//
// The check is stricter than the reference's checkData(): the key sequence must equal std::sort of the input
// byte for byte (multiplicities included), and every payload byte must still belong to its key.
//
// Built by `make -C oracle conformance` (part of __graft_entry__.build()).  Run: conformance_b200 [maxNum=10000]
// [seed=42].  Exit 0 with "All tests passed", 1 when a case failed, 3 when a sort call failed (no GPU: there
// is no CPU fallback).
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <limits>
#include <random>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "b200sort.h"
#include "b200sort/radixSort.hpp"

namespace {

template <typename K>
constexpr int key_code() {
  return simd_sort::radix_sort::internal::key_type_code<K>();
}

template <typename K>
const char *key_name() {
  static const char *names[] = {"uint8", "int8", "uint16", "int16", "uint32", "int32", "uint64", "int64", "float", "double"};
  return names[key_code<K>()];
}

void b200_check(int rc) {
  if (rc != 0) {
    std::printf("b200sort error %d: %s\n", rc, b200sort_last_error());
    std::exit(3);
  }
}

long g_sorts = 0;

// payload shape Ps... of the reference's testAllPayloads (src/test.cpp:100-153)
template <typename... Ps>
struct Shape {
  static std::vector<uint32_t> sizes() { return {static_cast<uint32_t>(sizeof(Ps))...}; }
  template <typename K>
  static constexpr std::size_t record_bytes() { return sizeof(simd_sort::DataElement<K, Ps...>); }
};
template <std::size_t, typename T>
using Same = T;
template <typename T, std::size_t... I>
Shape<Same<I, T>...> repeat(std::index_sequence<I...>);
template <typename T, std::size_t N>
using Rep = decltype(repeat<T>(std::make_index_sequence<N>{}));

enum Dist { Gaussian, Uniform, Zero, ZeroOne, Sorted, ReverseSorted, AlmostSorted, AlmostReverseSorted, NumDists };
const char *dist_name[] = {"Gaussian", "Uniform", "Zero", "ZeroOne", "Sorted", "ReverseSorted", "AlmostSorted",
                           "AlmostReverseSorted"};

template <typename K>
K uniform_key(std::mt19937 &gen) {
  if constexpr (std::is_floating_point_v<K>) {
    return std::uniform_real_distribution<K>(-1, 1)(gen);
  } else if constexpr (std::is_signed_v<K>) {
    return static_cast<K>(std::uniform_int_distribution<int64_t>(std::numeric_limits<K>::min(), std::numeric_limits<K>::max())(gen));
  } else {
    return static_cast<K>(std::uniform_int_distribution<uint64_t>(0, std::numeric_limits<K>::max())(gen));
  }
}

template <typename K>
K gaussian_key(std::mt19937 &gen) {
  if constexpr (std::is_floating_point_v<K>) {
    return std::normal_distribution<K>(0, 1)(gen);
  } else {
    return static_cast<K>(static_cast<int64_t>(std::llround(std::normal_distribution<double>(0, 100)(gen))));
  }
}

template <typename K>
bool less(K a, K b, bool up) {
  return up ? a < b : a > b;
}

template <typename K>
std::vector<K> make_keys(Dist d, std::size_t n, unsigned seed) {
  std::mt19937 gen(seed);
  std::vector<K> k(n);
  for (auto &x : k) {
    switch (d) {
      case Gaussian: x = gaussian_key<K>(gen); break;
      case Zero: x = K(0); break;
      case ZeroOne: x = static_cast<K>(gen() % 2); break;
      case Uniform: x = uniform_key<K>(gen); break;
      default: x = std::is_floating_point_v<K> ? gaussian_key<K>(gen) : uniform_key<K>(gen); break;
    }
  }
  if (d >= Sorted) {
    const bool up = d == Sorted || d == AlmostSorted;
    std::sort(k.begin(), k.end(), [up](K a, K b) { return less(a, b, up); });
    if (d >= AlmostSorted) {
      const auto swaps = static_cast<std::size_t>(std::pow(2.0, std::floor(std::log10(static_cast<double>(n)))));
      std::uniform_int_distribution<std::size_t> pos(0, n - 1);
      for (std::size_t s = 0; s < swaps; s++) std::swap(k[pos(gen)], k[pos(gen)]);
    }
  }
  return k;
}

uint64_t mix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

// `bytes` payload bytes of stream `stream` that belong to a key with bit pattern `key_bits`
void fill_payload(uint8_t *dst, std::size_t bytes, uint64_t key_bits, unsigned stream) {
  for (std::size_t w = 0; w * 8 < bytes; w++) {
    const uint64_t v = mix64(key_bits ^ (uint64_t(stream) << 56) ^ (w * 0xD1B54A32D192ED03ull));
    std::memcpy(dst + 8 * w, &v, std::min<std::size_t>(8, bytes - 8 * w));
  }
}

template <typename K>
uint64_t bits_of(K k) {
  uint64_t b = 0;
  std::memcpy(&b, &k, sizeof(K));
  return b;
}

// one case: sorts `keys` (and key-derived payloads) on the GPU, either as separate streams of `sizes` bytes or
// as combined records of `record_bytes`, and checks the result against std::sort
template <typename K>
bool run_case(const std::vector<K> &keys, bool up, bool combined, const std::vector<uint32_t> &sizes, std::size_t record_bytes,
              const std::string &label) {
  const std::size_t n = keys.size();
  std::vector<K> want(keys);
  std::sort(want.begin(), want.end(), [up](K a, K b) { return less(a, b, up); });
  std::vector<K> got(n);
  std::string err;
  std::vector<uint8_t> expect(64);
  if (!combined) {
    std::vector<K> k(keys);
    std::vector<std::vector<uint8_t>> streams(sizes.size());
    std::vector<void *> ptrs(sizes.size() + 1, nullptr);
    std::vector<uint32_t> elem_bytes(sizes);
    elem_bytes.push_back(0);
    for (std::size_t s = 0; s < sizes.size(); s++) {
      streams[s].resize(n * sizes[s]);
      for (std::size_t i = 0; i < n; i++) fill_payload(&streams[s][i * sizes[s]], sizes[s], bits_of(k[i]), unsigned(s));
      ptrs[s] = streams[s].data();
    }
    g_sorts++;
    b200_check(b200sort_sort_soa_ex(k.data(), key_code<K>(), (int64_t)n, up ? 1 : 0, (int)sizes.size(), ptrs.data(),
                                    elem_bytes.data(), 16, B200SORT_CMP_INSERTION, nullptr, nullptr, 0));
    got = k;
    for (std::size_t s = 0; s < sizes.size() && err.empty(); s++) {
      for (std::size_t i = 0; i < n; i++) {
        fill_payload(expect.data(), sizes[s], bits_of(got[i]), unsigned(s));
        if (std::memcmp(expect.data(), &streams[s][i * sizes[s]], sizes[s]) != 0) {
          err = "payload stream " + std::to_string(s) + " lost its key at index " + std::to_string(i);
          break;
        }
      }
    }
  } else {
    const std::size_t pb = record_bytes - sizeof(K);  // everything after the key, padding included, moves with it
    std::vector<uint8_t> rec(n * record_bytes);
    for (std::size_t i = 0; i < n; i++) {
      std::memcpy(&rec[i * record_bytes], &keys[i], sizeof(K));
      fill_payload(&rec[i * record_bytes + sizeof(K)], pb, bits_of(keys[i]), 0);
    }
    g_sorts++;
    b200_check(b200sort_sort_aos_ex(rec.data(), key_code<K>(), (uint32_t)record_bytes, (int64_t)n, up ? 1 : 0, 16,
                                    B200SORT_CMP_INSERTION, nullptr, nullptr, 0));
    for (std::size_t i = 0; i < n; i++) {
      std::memcpy(&got[i], &rec[i * record_bytes], sizeof(K));
      fill_payload(expect.data(), pb, bits_of(got[i]), 0);
      if (err.empty() && std::memcmp(expect.data(), &rec[i * record_bytes + sizeof(K)], pb) != 0)
        err = "record payload lost its key at index " + std::to_string(i);
    }
  }
  if (n && std::memcmp(got.data(), want.data(), n * sizeof(K)) != 0) {
    std::size_t i = 0;
    while (std::memcmp(&got[i], &want[i], sizeof(K)) == 0) i++;
    err = "key sequence differs from std::sort at index " + std::to_string(i);
  }
  if (!err.empty()) {
    std::cout << label << ": FAILED (" << err << ")" << std::endl;
    return false;
  }
  std::cout << label << ": passed\n";
  return true;
}

template <typename K, typename S>
bool test_shape(std::size_t n, unsigned seed) {
  const std::vector<uint32_t> sizes = S::sizes();
  constexpr std::size_t rb = S::template record_bytes<K>();
  std::string shape = "[";
  for (std::size_t s = 0; s < sizes.size(); s++) shape += (s ? "," : "") + std::to_string(sizes[s]);
  shape += "]";
  bool ok = true;
  for (int d = 0; d < NumDists; d++) {
    const std::vector<K> keys = make_keys<K>(Dist(d), n, seed);
    for (bool combined : {false, true}) {
      if (combined && !simd_sort::is_power_of_two<rb>) continue;  // src/test.cpp:76-98
      for (bool up : {true, false}) {
        const std::string label = std::string("RadixB200 ") + key_name<K>() + " payload bytes " + shape + " " + dist_name[d] +
                                  (combined ? " combined " : " separate ") + (up ? "up" : "down") + " n=" + std::to_string(n);
        ok &= run_case<K>(keys, up, combined, sizes, rb, label);
      }
    }
  }
  return ok;
}

template <typename K>
bool test_payloads(std::size_t n, unsigned seed) {
  bool ok = true;
  ok &= test_shape<K, Shape<>>(n, seed);
  ok &= test_shape<K, Shape<uint8_t>>(n, seed);
  ok &= test_shape<K, Shape<uint16_t>>(n, seed);
  ok &= test_shape<K, Shape<uint32_t>>(n, seed);
  ok &= test_shape<K, Shape<uint64_t>>(n, seed);
  ok &= test_shape<K, Shape<uint64_t, uint8_t>>(n, seed);
  ok &= test_shape<K, Shape<uint64_t, uint64_t>>(n, seed);
  ok &= test_shape<K, Rep<uint64_t, 3>>(n, seed);
  ok &= test_shape<K, Rep<uint64_t, 7>>(n, seed);
  ok &= test_shape<K, Rep<uint8_t, 63>>(n, seed);
  ok &= test_shape<K, Rep<uint8_t, 31>>(n, seed);
  ok &= test_shape<K, Rep<uint8_t, 15>>(n, seed);
  ok &= test_shape<K, Rep<uint8_t, 7>>(n, seed);
  ok &= test_shape<K, Rep<uint8_t, 3>>(n, seed);
  return ok;
}

bool test_all(std::size_t n, unsigned seed) {
  bool ok = true;
  ok &= test_payloads<uint8_t>(n, seed);
  ok &= test_payloads<int8_t>(n, seed);
  ok &= test_payloads<uint16_t>(n, seed);
  ok &= test_payloads<int16_t>(n, seed);
  ok &= test_payloads<uint32_t>(n, seed);
  ok &= test_payloads<int32_t>(n, seed);
  ok &= test_payloads<uint64_t>(n, seed);
  ok &= test_payloads<int64_t>(n, seed);
  ok &= test_payloads<float>(n, seed);
  ok &= test_payloads<double>(n, seed);
  return ok;
}

}  // namespace

int main(int argc, char const *argv[]) {
  const std::size_t maxNum = argc > 1 ? std::stoul(argv[1]) : 10000;
  const unsigned int seed = argc > 2 ? (unsigned)std::stoul(argv[2]) : 42u;
  bool passed = true;
  for (std::size_t num = 1; num <= maxNum; num *= 10) {  // src/test.cpp:185
    std::cout << "Testing " << num << " elements" << std::endl;
    passed &= test_all(num, seed);
  }
  std::cout << "sorts through libb200sort: " << g_sorts << ", kernels launched: " << b200sort_launch_count() << std::endl;
  if (passed) {
    std::cout << "All tests passed" << std::endl;
    return 0;
  }
  std::cout << "Tests failed, see above for details" << std::endl;
  return 1;
}
