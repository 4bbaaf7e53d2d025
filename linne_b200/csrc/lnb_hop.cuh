/* lnb_hop.cuh -- the hop over a stream's block size fields, on the device.
 *
 * Reference: the serial loop of libs/linne_decoder/src/linne_decoder.c:708-726 reads sync code, size, type and
 * sample count of one block to find the next.  When the stream image already lives in HBM (device-resident and
 * corpus decodes) the host used to copy the whole image back (38 MB per six-minute file) just to read those 11 bytes
 * per block.  Here one lane per file follows the chain where the image is -- a dependent load per block, served from
 * L2 when an encoder has just written the image -- and fills the block table; only the table (32 bytes per block)
 * and a result record per file travel to the host.  The checks and the loop are those of the host hop
 * (lnb_framing.h).
 */
#pragma once
#include "lnb_common.cuh"
#include "lnb_framing.h"

LNB_HD void lnb_hop_file(const uint8_t *image, const LnbHopFile &f, LnbBlockDesc *table, LnbHopResult &out)
{
    const uint8_t *data = image + f.offset;
    uint32_t channels = 0, sample_limit = 0, bits = 0;             /* no header: nothing to hop, the host looks at it */
    for (uint32_t i = 0; i < 32u; i++) out.header[i] = (i < f.size && i < LNB_HEADER_SIZE) ? data[i] : (uint8_t)0;
    if (f.size >= LNB_HEADER_SIZE && data[0] == 'I' && data[1] == 'B' && data[2] == 'R' && data[3] == 'A') {
        channels = lnb_rd_be(data + 12, 2); sample_limit = lnb_rd_be(data + 14, 4); bits = lnb_rd_be(data + 22, 2);
    }
    lnb_hop_blocks(data, f.size, LNB_HEADER_SIZE, channels, bits, f.room_samples, sample_limit, 0u, table, f.table_cap, f.offset, &out);
}

#if defined(__CUDACC__)
/* one warp per file, lane 0 hops (the chain is serial; files hop side by side) */
__global__ void __launch_bounds__(32) lnb_hop_kernel(const uint8_t *image, const LnbHopFile *files, uint32_t num_files,
                                                     LnbBlockDesc *table, LnbHopResult *results)
{
    const uint32_t i = blockIdx.x;
    if (i >= num_files || threadIdx.x != 0) return;
    const LnbHopFile f = files[i];
    LnbHopResult r;
    lnb_hop_file(image, f, table + f.table_first, r);
    results[i] = r;
}
#endif
