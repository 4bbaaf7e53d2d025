/* lnb_window.cuh -- sample-window decodes: the parallel seek and the window gather.
 *
 * A seek index (one point per block: first sample, byte offset) turns "which blocks hold samples [a, b)" into a binary
 * search on the host.  The blocks the windows need then go through the unchanged decode pipeline as one batch, into
 * compact scratch planes, and the windows are copied out of those planes in one pass.  Two flat item kinds, launched
 * through the executor like the packed-PCM conversions:
 *
 *   seek           item = needed block: reads the 11-byte block header at the indexed offset (never past the indexed
 *                  span) and fills the batch's LnbBlockDesc.  The checks and their order are those of lnb_framing.h,
 *                  plus the two the index adds: the block may not run past the next indexed block, and its sample
 *                  count must be the index's.  The result code (include/linne.h numbering) is left in
 *                  LnbBlockDesc.status; the host clears it before the decode.
 *   window_gather  item = (window, channel, aligned group of four destination samples): coalesced copy from the
 *                  scratch planes to the window's place, 16-byte loads and stores where both sides are aligned.
 */
#pragma once
#include "lnb_common.cuh"
#include "lnb_framing.h"

struct LnbItemSeek {
    const uint8_t *image;           /* the batch's stream image (the caller's device image or the staged blocks) */
    const LnbSeekIn *in;
    LnbBlockDesc *out;
    uint32_t channels, bits;
    LNB_HDM void operator()(uint32_t j) const
    {
        const LnbSeekIn s = in[j];
        uint8_t h[LNB_BLOCK_HEADER_SIZE];
        const uint32_t avail = s.span < (uint32_t)LNB_BLOCK_HEADER_SIZE ? s.span : (uint32_t)LNB_BLOCK_HEADER_SIZE;
        for (uint32_t k = 0; k < (uint32_t)LNB_BLOCK_HEADER_SIZE; k++) h[k] = k < avail ? image[(size_t)s.img_off + k] : (uint8_t)0;
        LnbBlockDesc d;
        d.smp_off = s.smp_off; d.nsmp = s.nsmp; d.byte_off = s.img_off; d.byte_size = 0; d.type = 0xFFu;
        d.na = 0; d.crc = 0;
        uint32_t size32 = 0;
        uint32_t err = lnb_block_frame(h, s.remain, &size32);
        if (err == LNB_HOP_OK) {
            const uint32_t type = h[8], ns = lnb_rd_be(h + 9, 2);
            d.byte_size = size32 + 6u;
            d.type = type;
            if (d.byte_size > s.span || ns != s.nsmp) err = LNB_HOP_INVALID_FORMAT;       /* the index's two checks */
            else err = lnb_block_body(type, ns, s.remain, channels, bits);
            if (err == LNB_HOP_OK && type == LNB_BLOCK_RAW && LNB_BLOCK_HEADER_SIZE + (uint64_t)(bits / 8u) * ns * channels > s.span)
                err = LNB_HOP_INVALID_FORMAT;                                             /* a raw payload past the span */
        }
        if (err != LNB_HOP_OK) d.type = 0xFFu;
        d.status = err;
        out[j] = d;
    }
};

struct LnbItemGatherWindows {
    const int32_t *scratch; int32_t *dst;
    uint32_t scratch_stride, dst_stride;
    const LnbGatherWin *wins; uint32_t num_wins;
    LNB_HDM void operator()(uint32_t i) const
    {
        uint32_t lo = 0, hi = num_wins - 1u;                 /* last window whose items start at or before i */
        while (lo < hi) {
            const uint32_t mid = (lo + hi + 1u) >> 1;
            if (wins[mid].item_first <= i) lo = mid; else hi = mid - 1u;
        }
        const LnbGatherWin w = wins[lo];
        const uint32_t g0 = w.dst >> 2, groups = ((w.dst + w.len + 3u) >> 2) - g0;
        const uint32_t r = i - w.item_first, c = r / groups, d0 = (g0 + r % groups) << 2;
        const uint32_t a = d0 > w.dst ? d0 : w.dst, b = (d0 + 4u < w.dst + w.len) ? d0 + 4u : w.dst + w.len;
        const int32_t *s = scratch + (size_t)c * scratch_stride + w.src + (a - w.dst);   /* the sample for destination a */
        int32_t *o = dst + (size_t)c * dst_stride + a;
#if defined(__CUDA_ARCH__)
        if (b - a == 4u && ((uintptr_t)o & 15u) == 0u) {
            int4 v;
            if (((uintptr_t)s & 15u) == 0u) v = *(const int4 *)s;
            else { v.x = s[0]; v.y = s[1]; v.z = s[2]; v.w = s[3]; }
            *(int4 *)o = v;
            return;
        }
#endif
        for (uint32_t k = 0; k < b - a; k++) o[k] = s[k];
    }
};

template <class Exec>
void lnb_seek_pipeline(Exec &ex, const uint8_t *image, const LnbSeekIn *in, uint32_t n, uint32_t channels, uint32_t bits, LnbBlockDesc *out)
{
    ex.run("seek", n, LnbItemSeek{image, in, out, channels, bits});
}

template <class Exec>
void lnb_gather_windows_pipeline(Exec &ex, const int32_t *scratch, uint32_t scratch_stride, const LnbGatherWin *wins, uint32_t num_wins,
                                 uint32_t num_items, int32_t *dst, uint32_t dst_stride)
{
    if (num_wins == 0u) return;
    ex.run("window_gather", num_items, LnbItemGatherWindows{scratch, dst, scratch_stride, dst_stride, wins, num_wins});
}
