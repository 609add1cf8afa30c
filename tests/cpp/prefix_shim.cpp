// Test shim (CPU tests only): the shared-prefix decision of hmk_bulk_filter (hmk_common.h) for one warp of 32 lanes, with
// the warp's min / max reductions done by a loop.  Compiled with plain g++ by tests/test_filter_prefix.py.
#include "../../hammock_b200/csrc/hmk_common.h"

extern "C" {
int32_t shim_warp_prefix(const uint64_t* w, const uint8_t* scored) {
    uint32_t kmin = 0xffffffffu, kmax = 0u;
    for (int l = 0; l < 32; l++) {
        const uint32_t lo = hmk_prefix_lo(w[l], scored[l] != 0), hi = hmk_prefix_hi(w[l], scored[l] != 0);
        kmin = lo < kmin ? lo : kmin;
        kmax = hi > kmax ? hi : kmax;
    }
    return hmk_prefix_shared(kmin, kmax);
}
}
