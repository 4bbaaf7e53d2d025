/* lnb_salvage.cuh -- salvage decodes: the resynchronising scan over a damaged stream image and its CRC pass.
 *
 * After damage the hop over the size fields (lnb_framing.h) has lost its place; every block start that is left is
 * found again by testing every byte position of the image as a block start, in parallel.  Flat item kind, launched
 * through the executor like the window kernels, so the simulator runs the same body:
 *
 *   resync_scan    item = aligned group of 16 image positions in [30, data_size): reads the group's 16 + 16 bytes once
 *                  (two 16-byte loads; the image is padded to a multiple of 16 bytes plus 16) and tests each position
 *                  with the sync code, lnb_block_frame, lnb_block_body, 1 <= samples <= the header's block size and
 *                  a size of at most lnb_salvage_max_block_bytes (so the CRC pass reads at most that much per
 *                  candidate, however the image was damaged or crafted).  A survivor is appended to a capped candidate
 *                  table with one atomic add; the counter counts every survivor, so the host can grow the table and
 *                  scan again.
 *
 * The candidates' CRCs are checked by the decoder's CRC arithmetic (lnb_crc_v2_block, one CTA per candidate) in a
 * grid sized by the table's capacity whose CTAs past the counter return at once -- the host learns the count only
 * with the table, behind the call's one synchronisation.  The host walks the verified candidates
 * (csrc/host/linne_decoder_host.c, decode_salvage).
 */
#pragma once
#include "lnb_common.cuh"
#include "lnb_framing.h"

LNB_HD uint32_t lnb_salvage_claim(uint32_t *count)
{
#if defined(__CUDA_ARCH__)
    return atomicAdd(count, 1u);
#else
    return (*count)++;
#endif
}

/* The longest block the scan takes: twice the raw block of B samples plus 4 KiB and the block header.  The library's
 * encoder stages a stream of one block in that much room (stream_room, csrc/host/linne_encoder_host.c), so no block it
 * writes is longer; a compressed block can be longer than raw, since its type comes from an estimate. */
LNB_HD uint32_t lnb_salvage_max_block_bytes(uint32_t block_size, uint32_t channels, uint32_t bits)
{
    const uint64_t n = (uint64_t)LNB_BLOCK_HEADER_SIZE + 2u * ((uint64_t)block_size * channels * ((bits + 7u) / 8u)) + 4096u + 64u;
    return n > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)n;
}

struct LnbItemResyncScan {
    const uint8_t *image;
    uint32_t data_size, channels, bits, block_size, max_bytes;
    LnbBlockDesc *table; uint32_t *count; uint32_t cap;
    LNB_HDM void operator()(uint32_t i) const
    {
        const uint32_t p0 = (LNB_HEADER_SIZE / 16u + i) * 16u;
        uint8_t w[32];                                      /* the block headers of positions p0 .. p0 + 15 lie in here */
#if defined(__CUDA_ARCH__)
        const uint4 a = ((const uint4 *)(image + p0))[0], c = ((const uint4 *)(image + p0))[1];
        const uint32_t words[8] = {a.x, a.y, a.z, a.w, c.x, c.y, c.z, c.w};
#pragma unroll
        for (uint32_t k = 0; k < 32u; k++) w[k] = (uint8_t)(words[k >> 2] >> (8u * (k & 3u)));
#else
        for (uint32_t k = 0; k < 32u; k++) w[k] = image[(size_t)p0 + k];
#endif
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (uint32_t k = 0; k < 16u; k++) {
            const uint32_t p = p0 + k;
            if (p < LNB_HEADER_SIZE || p >= data_size || w[k] != 0xFFu || w[k + 1u] != 0xFFu) continue;
            const uint32_t remain = data_size - p;
            uint32_t size32 = 0;
            if (lnb_block_frame(w + k, remain, &size32) != LNB_HOP_OK || size32 + 6u > max_bytes) continue;
            const uint32_t type = w[k + 8u], ns = lnb_rd_be(w + k + 9u, 2);
            if (lnb_block_body(type, ns, remain, channels, bits) != LNB_HOP_OK || ns == 0u || ns > block_size) continue;
            const uint32_t j = lnb_salvage_claim(count);
            if (j >= cap) continue;
            LnbBlockDesc d;
            d.smp_off = 0; d.nsmp = ns; d.byte_off = p; d.byte_size = size32 + 6u; d.type = type;
            d.na = 0; d.status = 0; d.crc = 0;
            table[j] = d;
        }
    }
};

/* items covering the positions [30, data_size) */
LNB_HD uint32_t lnb_resync_items(uint32_t data_size)
{
    return data_size > LNB_HEADER_SIZE ? (data_size - 1u) / 16u - LNB_HEADER_SIZE / 16u + 1u : 0u;
}

template <class Exec>
void lnb_resync_scan_pipeline(Exec &ex, const uint8_t *image, uint32_t data_size, uint32_t channels, uint32_t bits,
                              uint32_t block_size, LnbBlockDesc *table, uint32_t *count, uint32_t cap)
{
    ex.run("resync_scan", lnb_resync_items(data_size), LnbItemResyncScan{image, data_size, channels, bits, block_size,
                                                                      lnb_salvage_max_block_bytes(block_size, channels, bits),
                                                                      table, count, cap});
}

#if defined(__CUDACC__)
#include "lnb_crc_v2.cuh"
/* the CRC pass over the first min(*count, b.num_blocks) candidates: one CTA per table entry, those past the count return */
__global__ void __launch_bounds__(LNB_CRC_THREADS) lnb_salvage_crc_kernel(LnbDecodeBatch b, const uint32_t *count)
{
    if (blockIdx.x >= *count) return;
    lnb_crc_v2_block(b, blockIdx.x);
}
#endif
