/* lnb_framing.h -- the framing of a stream's blocks: the checks of one block header and the hop over them.
 *
 * One definition for every reader of a stream: the host hop (csrc/host/linne_decoder_host.c), the device hop
 * (lnb_hop.cuh) and the seek of sample-window decodes (lnb_window.cuh).  Compiles as C99 (host code), as CUDA and as
 * C++ (the CPU simulator).
 *
 * Per block the reference checks, in this order (linne_decoder.c:604-653):
 *   sync (INVALID_FORMAT) -> size (INSUFFICIENT_DATA) -> CRC (DETECT_DATA_CORRUPTION)
 *   -> sample count vs buffer (INSUFFICIENT_BUFFER) -> type (INVALID_FORMAT, :651)
 *   -> raw payload size (INSUFFICIENT_DATA, :383)
 * Sync and size stop the hop (`framing_error`); the later ones are recorded as the terminal block's `post_crc_error`,
 * because a CRC mismatch (known only after the decode pass) outranks them.
 */
#ifndef LNB_FRAMING_H
#define LNB_FRAMING_H

#include "lnb_types.h"

#if defined(__CUDACC__)
#define LNB_FRAMING_FN static __host__ __device__ __forceinline__
#else
#define LNB_FRAMING_FN static inline
#endif

/* result codes as in include/linne.h (LINNEApiResult) */
#define LNB_HOP_OK                  0u
#define LNB_HOP_INVALID_FORMAT      2u
#define LNB_HOP_INSUFFICIENT_BUFFER 3u
#define LNB_HOP_INSUFFICIENT_DATA   4u

LNB_FRAMING_FN uint32_t lnb_rd_be(const uint8_t *p, int n) { uint32_t v = 0; int i; for (i = 0; i < n; i++) v = (v << 8) | p[i]; return v; }

/* sync code and size field of the block at p, `remain` bytes of the stream from p on; *size32 is set when they pass */
LNB_FRAMING_FN uint32_t lnb_block_frame(const uint8_t *p, uint32_t remain, uint32_t *size32)
{
    if (remain < 2u) return LNB_HOP_INSUFFICIENT_DATA;
    if (lnb_rd_be(p, 2) != LNB_SYNC_CODE) return LNB_HOP_INVALID_FORMAT;
    if (remain < 6u) return LNB_HOP_INSUFFICIENT_DATA;
    *size32 = lnb_rd_be(p + 2, 4);
    if ((uint64_t)*size32 + 6u > remain) return LNB_HOP_INSUFFICIENT_DATA;
    if (*size32 < 5u) return LNB_HOP_INVALID_FORMAT;               /* cannot hold crc+type+count */
    return LNB_HOP_OK;
}

/* type and raw payload size of a framed block */
LNB_FRAMING_FN uint32_t lnb_block_body(uint32_t type, uint32_t ns, uint32_t remain, uint32_t channels, uint32_t bits)
{
    if (type > LNB_BLOCK_RAW) return LNB_HOP_INVALID_FORMAT;
    if (type == LNB_BLOCK_RAW && remain - LNB_BLOCK_HEADER_SIZE < (bits * ns * channels) / 8u) return LNB_HOP_INSUFFICIENT_DATA;
    return LNB_HOP_OK;
}

/* The hop over the blocks of data[off, data_size) until `sample_limit` samples or `block_limit` blocks (0: no limit),
 * checked against `room` samples of output.  Fills table[] (byte offsets plus `base`) and *out; sets out->overflow and
 * stops when more than `table_cap` entries are needed. */
LNB_FRAMING_FN void lnb_hop_blocks(const uint8_t *data, uint32_t data_size, uint32_t off, uint32_t channels, uint32_t bits,
                                   uint32_t room, uint32_t sample_limit, uint32_t block_limit,
                                   LnbBlockDesc *table, uint32_t table_cap, uint32_t base, LnbHopResult *out)
{
    uint32_t progress = 0, nb = 0;
    out->num_decodable = 0u;
    out->framing_error = out->post_crc_error = LNB_HOP_OK;
    out->overflow = 0u;
    while (progress < sample_limit && off < data_size) {
        const uint8_t *p = data + off;
        const uint32_t remain = data_size - off;
        uint32_t size32 = 0, type, ns, err;
        LnbBlockDesc d;
        if (nb >= table_cap) { out->overflow = 1u; break; }
        if ((err = lnb_block_frame(p, remain, &size32)) != LNB_HOP_OK) { out->framing_error = err; break; }
        type = p[8];
        ns = lnb_rd_be(p + 9, 2);
        d.smp_off = progress; d.nsmp = ns; d.byte_off = base + off; d.byte_size = size32 + 6u; d.type = type;
        d.na = 0; d.status = 0; d.crc = 0;
        table[nb] = d;
        nb++;
        if (ns > room - progress) { out->post_crc_error = LNB_HOP_INSUFFICIENT_BUFFER; break; }
        if ((err = lnb_block_body(type, ns, remain, channels, bits)) != LNB_HOP_OK) { out->post_crc_error = err; break; }
        out->num_decodable = nb;
        progress += ns;
        if (type == LNB_BLOCK_RAW) off += LNB_BLOCK_HEADER_SIZE + (bits / 8u) * ns * channels;
        else if (type == LNB_BLOCK_SILENT) off += LNB_BLOCK_HEADER_SIZE;
        else off += size32 + 6u;                                   /* == 11 + ceil(bits/8) for any stream an encoder wrote */
        if (block_limit && nb >= block_limit) break;
    }
    out->num_blocks = nb;
    out->total_samples = progress;
    out->end_offset = off;
}

#endif
