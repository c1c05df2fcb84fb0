// segmented_inst.cu -- the instantiations of seg_medium_kernel (segmented.cuh), in a module of their own: its
// dynamic shared memory would otherwise reserve 1 KB of shared memory for every kernel of b200sort.cu.
#include "segmented.cuh"

namespace b200sort {

template <int KB, int LOG_CAP>
static SegMediumKernel medium() {
  return {seg_medium_kernel<KB, LOG_CAP>, seg_threads(LOG_CAP), seg_smem_bytes<KB>(LOG_CAP)};
}

template <int KB>
static SegMediumKernel medium_of(int log_cap) {
  switch (log_cap) {
    case 6: return medium<KB, 6>();
    case 7: return medium<KB, 7>();
    case 8: return medium<KB, 8>();
    case 9: return medium<KB, 9>();
    case 10: return medium<KB, 10>();
    case 11: return medium<KB, 11>();
    case 12: return medium<KB, 12>();
    case 13: return medium<KB, 13>();
    default:
      if constexpr (KB <= 4)
        if (log_cap == 14) return medium<KB, 14>();
      return {nullptr, 0, 0};  // (no bin above CAP)
  }
}

SegMediumKernel seg_medium_kernel_of(int kb, int log_cap) {
  switch (kb) {
    case 1: return medium_of<1>(log_cap);
    case 2: return medium_of<2>(log_cap);
    case 4: return medium_of<4>(log_cap);
    default: return medium_of<8>(log_cap);
  }
}

}  // namespace b200sort
