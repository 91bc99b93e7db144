// dkb_scan_inst.cu - the instantiations of kernel 2 for ONE probe stride (DKB_INST_D = 1, 2,
// 4, 8 or 16), compiled as its own translation unit so that the strides build in parallel.
// Shared-memory filter: 1..4 filter bits; L2 filter with and without the pre-filter (strides
// 2..16): 1..2 bits; each with and without the profiling counters, and in region mode (RG,
// DESIGN.md §2) without them.
#include "dkb_scan.cuh"

#ifndef DKB_INST_D
#error "compile with -DDKB_INST_D=<stride>"
#endif
#define DKB_CAT2(a, b) a##b
#define DKB_CAT(a, b) DKB_CAT2(a, b)

namespace dkb {
typedef void (*scan_fn)(const ScanParams);

// fm: 0 = filter in shared memory, 1 = in L2, 2 = in L2 behind the shared-memory pre-filter,
// 3 / 4 = 1 / 2 with gated lookups (macro path: strides 8 and 16).  Region mode with the
// profiling counters is not built: nullptr.
scan_fn DKB_CAT(pick_scan_d, DKB_INST_D)(int NH, int fm, bool prof, bool rg) {
  constexpr int D = DKB_INST_D;
#define PICK(h, m)                                                                      \
  if (NH == h && fm == m)                                                               \
    return rg ? (prof ? nullptr : (scan_fn)k_scan<D, h, m, false, true>)                \
              : prof ? (scan_fn)k_scan<D, h, m, true, false> : (scan_fn)k_scan<D, h, m, false, false>;
  PICK(2, 0)
#if DKB_INST_D >= 2
  PICK(2, 1) PICK(2, 2)
#endif
#if DKB_INST_D >= 8
  PICK(2, 3) PICK(2, 4)
#endif
  PICK(1, 0) PICK(3, 0) PICK(4, 0)
#if DKB_INST_D >= 2
  PICK(1, 1) PICK(1, 2)
#endif
#if DKB_INST_D >= 8
  PICK(1, 3) PICK(1, 4)
#endif
#undef PICK
  return nullptr;
}
}  // namespace dkb
