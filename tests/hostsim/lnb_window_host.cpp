/* lnb_window_host.cpp -- TEST INFRASTRUCTURE: the sample-window entry points of the CUDA shim (lnb_shim.h:
 * lnb_shim_seek_blocks, lnb_shim_gather_windows) for the loop-based stand-in of lnb_shim_host.cpp.
 *
 * The very same item bodies as the product (lnb_window.cuh), stepped through as plain loops.  Linked into
 * tests/hostsim/liblinne_hostsim.so next to lnb_shim_host.cpp; liblinne_b200.so never contains or loads it.
 */
#include "lnb_shim.h"
#include "lnb_window.cuh"

/* the simulator's device context: the same definition as in lnb_shim_host.cpp (one launch counted per item pass) */
struct LnbDevice { LnbDevTables tables; uint64_t launches; };

namespace {
struct WindowLoopExec {
    LnbDevice *dev;
    template <class F> void run(const char *, uint32_t n, const F &f)
    {
        for (uint32_t i = 0; i < n; i++) f(i);
        dev->launches++;
    }
};
}  // namespace

extern "C" {
int lnb_shim_seek_blocks(LnbDevice *dev, const uint8_t *img, const LnbSeekIn *in, uint32_t n, uint32_t ch, uint32_t bits, LnbBlockDesc *out)
{ WindowLoopExec ex{dev}; lnb_seek_pipeline(ex, img, in, n, ch, bits, out); return 0; }
int lnb_shim_gather_windows(LnbDevice *dev, const int32_t *scratch, uint32_t sstride, const LnbGatherWin *wins, uint32_t nw, uint32_t items,
                            int32_t *dst, uint32_t dstride)
{ WindowLoopExec ex{dev}; lnb_gather_windows_pipeline(ex, scratch, sstride, wins, nw, items, dst, dstride); return 0; }
}
