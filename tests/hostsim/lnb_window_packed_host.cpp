/* lnb_window_packed_host.cpp -- TEST INFRASTRUCTURE: the packed sample-window gather of the CUDA shim (lnb_shim.h:
 * lnb_shim_gather_windows_packed) for the loop-based stand-in of lnb_shim_host.cpp.
 *
 * The very same item body as the product (lnb_window.cuh, LnbItemGatherWindowsPacked), stepped through as a plain loop.
 * Linked into tests/hostsim/liblinne_hostsim.so next to lnb_window_host.cpp; liblinne_b200.so never contains or loads it.
 */
#include "lnb_shim.h"
#include "lnb_window.cuh"

/* the simulator's device context: the same definition as in lnb_shim_host.cpp (one launch counted per item pass) */
struct LnbDevice { LnbDevTables tables; uint64_t launches; };

namespace {
struct PackedWindowLoopExec {
    LnbDevice *dev;
    template <class F> void run(const char *, uint32_t n, const F &f)
    {
        for (uint32_t i = 0; i < n; i++) f(i);
        dev->launches++;
    }
};
}  // namespace

extern "C" int lnb_shim_gather_windows_packed(LnbDevice *dev, const int32_t *scratch, uint32_t sstride, const LnbGatherWin *wins,
                                              uint32_t nw, uint32_t items, uint8_t *dst, uint32_t ch, uint32_t bytes)
{ PackedWindowLoopExec ex{dev}; lnb_gather_windows_packed_pipeline(ex, scratch, sstride, wins, nw, items, dst, ch, bytes); return 0; }
