/* lnb_window.cuh -- sample-window decodes: the parallel seek and the window gather.
 *
 * A seek index (one point per block: first sample, byte offset) turns "which blocks hold samples [a, b)" into a binary
 * search on the host.  The blocks the windows need then go through the unchanged decode pipeline as one batch, into
 * compact scratch planes, and the windows are copied out of those planes in one pass.  Flat item kinds, launched
 * through the executor like the packed-PCM conversions:
 *
 *   seek           item = needed block: reads the 11-byte block header at the indexed offset (never past the indexed
 *                  span) and fills the batch's LnbBlockDesc.  The checks and their order are those of lnb_framing.h,
 *                  plus the two the index adds: the block may not run past the next indexed block, and its sample
 *                  count must be the index's.  The result code (include/linne.h numbering) is left in
 *                  LnbBlockDesc.status; the host clears it before the decode.
 *   window_gather  item = (window, channel, aligned group of four destination samples): coalesced copy from the
 *                  scratch planes to the window's place, 16-byte loads and stores where both sides are aligned.
 *   window_gather_packed
 *                  item = (window, aligned group of four destination frames): reads the group's 4 x C samples from
 *                  the scratch planes and writes them as the 4 x C x bytes bytes of a WAV data chunk (lnb_wav_sample)
 *                  to a dense staging buffer, with 32-bit stores, 16-byte ones where the group allows.
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

/* the window that item i belongs to: the last one whose items start at or before i */
LNB_HD uint32_t lnb_window_of_item(const LnbGatherWin *wins, uint32_t num_wins, uint32_t i)
{
    uint32_t lo = 0, hi = num_wins - 1u;
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1u) >> 1;
        if (wins[mid].item_first <= i) lo = mid; else hi = mid - 1u;
    }
    return lo;
}

struct LnbItemGatherWindows {
    const int32_t *scratch; int32_t *dst;
    uint32_t scratch_stride, dst_stride;
    const LnbGatherWin *wins; uint32_t num_wins;
    LNB_HDM void operator()(uint32_t i) const
    {
        const LnbGatherWin w = wins[lnb_window_of_item(wins, num_wins, i)];
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

/* `dst` holds the windows as dense frames of F = channels * bytes bytes, each window starting on a 4-frame boundary
 * (w.dst % 4 == 0), so a group is F 32-bit words and the groups of two windows never share a byte.  A window's last
 * group is written whole; its frames past the window's end carry zero samples and are not read from the planes. */
struct LnbItemGatherWindowsPacked {
    const int32_t *scratch; uint8_t *dst;
    uint32_t scratch_stride, channels, bytes;
    const LnbGatherWin *wins; uint32_t num_wins;
    LNB_HDM void operator()(uint32_t i) const
    {
        const LnbGatherWin w = wins[lnb_window_of_item(wins, num_wins, i)];
        const uint32_t f0 = (i - w.item_first) << 2, n = w.len - f0 < 4u ? w.len - f0 : 4u;   /* n frames in the window */
        const uint32_t F = channels * bytes;
        const int32_t *s = scratch + w.src + f0;
        uint32_t *o = (uint32_t *)(dst + (size_t)(w.dst + f0) * F);
        uint64_t acc = 0;                                    /* bytes not yet stored, the first in the low bits */
        uint32_t nb = 0, nw = 0;                             /* bits in acc, words stored */
#if defined(__CUDA_ARCH__)
        const bool quad = (F & 3u) == 0u && ((uintptr_t)o & 15u) == 0u;   /* F words = whole 16-byte stores */
        uint32_t q0 = 0, q1 = 0, q2 = 0;                     /* the last three words of a pending 16-byte store */
#endif
        for (uint32_t f = 0; f < 4u; f++)
            for (uint32_t c = 0; c < channels; c++) {
                const int32_t v = f < n ? s[(size_t)c * scratch_stride + f] : 0;
                acc |= (uint64_t)lnb_wav_sample(v, bytes) << nb;
                nb += 8u * bytes;
                if (nb < 32u) continue;
                const uint32_t word = (uint32_t)acc;
                acc >>= 32;
                nb -= 32u;
#if defined(__CUDA_ARCH__)
                if (quad) {
                    if ((nw & 3u) == 3u) *(uint4 *)(o + nw - 3u) = make_uint4(q0, q1, q2, word);
                    q0 = q1; q1 = q2; q2 = word;
                    nw++;
                    continue;
                }
#endif
                o[nw++] = word;
            }
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

template <class Exec>
void lnb_gather_windows_packed_pipeline(Exec &ex, const int32_t *scratch, uint32_t scratch_stride, const LnbGatherWin *wins,
                                        uint32_t num_wins, uint32_t num_items, uint8_t *dst, uint32_t channels, uint32_t bytes)
{
    if (num_wins == 0u) return;
    ex.run("window_gather_packed", num_items, LnbItemGatherWindowsPacked{scratch, dst, scratch_stride, channels, bytes, wins, num_wins});
}
