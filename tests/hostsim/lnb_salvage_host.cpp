/* lnb_salvage_host.cpp -- TEST INFRASTRUCTURE: the salvage entry points of the CUDA shim (lnb_shim.h:
 * lnb_shim_resync_scan, lnb_shim_crc_blocks) for the loop-based stand-in of lnb_shim_host.cpp.
 *
 * The scan runs the product's item body (lnb_salvage.cuh); the CRC pass runs the decoder's flat CRC item (lnb_pipeline.cuh),
 * which the simulator's decode uses too.  Linked into tests/hostsim/liblinne_hostsim.so next to lnb_shim_host.cpp;
 * liblinne_b200.so never contains or loads it.
 */
#include <string.h>
#include "lnb_shim.h"
#include "lnb_pipeline.cuh"
#include "lnb_salvage.cuh"

/* the simulator's device context: the same definition as in lnb_shim_host.cpp (one launch counted per item pass) */
struct LnbDevice { LnbDevTables tables; uint64_t launches; };

namespace {
struct SalvageLoopExec {
    LnbDevice *dev;
    template <class F> void run(const char *, uint32_t n, const F &f)
    {
        for (uint32_t i = 0; i < n; i++) f(i);
        dev->launches++;
    }
};
}  // namespace

extern "C" {
int lnb_shim_resync_scan(LnbDevice *dev, const uint8_t *img, uint32_t size, uint32_t ch, uint32_t bits, uint32_t block,
                         LnbBlockDesc *table, uint32_t *count, uint32_t cap)
{ SalvageLoopExec ex{dev}; lnb_resync_scan_pipeline(ex, img, size, ch, bits, block, table, count, cap); return 0; }
int lnb_shim_crc_blocks(LnbDevice *dev, const uint8_t *img, uint32_t size, LnbBlockDesc *table, const uint32_t *count, uint32_t cap)
{
    if (cap == 0) return 0;
    LnbDecodeBatch b;
    memset(&b, 0, sizeof(b));
    b.cfg.check_crc = 1u;
    b.tab = dev->tables;
    b.stream = img;
    b.stream_size = size;
    b.blocks = table;
    b.num_blocks = *count < cap ? *count : cap;
    SalvageLoopExec ex{dev};
    ex.run("salvage_crc", b.num_blocks, LnbItemCrc{b});
    return 0;
}
}
