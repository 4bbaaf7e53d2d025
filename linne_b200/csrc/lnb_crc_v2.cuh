/* lnb_crc_v2.cuh -- cooperative CRC16 check of every block: one CTA per block.
 * Replaces the flat one-thread-per-block CRC (D0); reference linne_decoder.c:617-625 and
 * linne_utility.c:72-89.  256 chunk CRCs (table in shared memory) are combined by multiplication with
 * x^(8*len) modulo the CRC polynomial -- the same arithmetic the packer uses (lnb_pack_v2.cuh). */
#pragma once
#include "lnb_common.cuh"
#include "lnb_pack_v2.cuh"

#define LNB_CRC_THREADS 256

/* the check of block i of the batch by the whole CTA (also the salvage decodes' CRC pass, lnb_salvage.cuh) */
__device__ __forceinline__ void lnb_crc_v2_block(const LnbDecodeBatch &b, uint32_t i)
{
    __shared__ uint16_t tab[256];
    __shared__ uint32_t part[LNB_CRC_THREADS];
    const uint32_t tid = threadIdx.x;
    LnbBlockDesc &gblk = b.blocks[i];
    const LnbBlockDesc blk = gblk;
    tab[tid] = b.tab.crc_table[tid];
    const uint8_t *base = b.stream + blk.byte_off;
    const uint32_t first = 8u, end = blk.byte_size, L = end - first;      /* body = type, count, payload */
    const uint32_t Lc = (L + LNB_CRC_THREADS - 1u) / LNB_CRC_THREADS;
    const int32_t start = (int32_t)end - (int32_t)(Lc * LNB_CRC_THREADS);  /* virtual zeros in front are free */
    int32_t lo = start + (int32_t)(tid * Lc), hi = lo + (int32_t)Lc;
    if (lo < (int32_t)first) lo = (int32_t)first;
    __syncthreads();
    uint32_t crc = 0;
    for (int32_t i = lo; i < hi; i++) crc = (crc >> 8) ^ tab[(crc ^ base[i]) & 0xFFu];
    part[tid] = crc;
    uint32_t pw = lnb_crc_xpow_bytes(Lc);
    for (uint32_t stride = 1; stride < LNB_CRC_THREADS; stride <<= 1) {
        __syncthreads();
        uint32_t v = 0;
        const bool active = (tid % (2u * stride)) == 0u;
        if (active) v = lnb_crc_mulmod(part[tid], pw) ^ part[tid + stride];
        __syncthreads();
        if (active) part[tid] = v;
        pw = lnb_crc_mulmod(pw, pw);
    }
    __syncthreads();
    if (tid == 0) {
        const uint32_t got = part[0];
        gblk.crc = got;
        if (b.cfg.check_crc && got != lnb_get_be(base + 6, 2)) atomicOr(&gblk.status, (uint32_t)LNB_ST_CRC_MISMATCH);   /* the throughput entropy stage may flag the block at the same time */
    }
}

__global__ void __launch_bounds__(LNB_CRC_THREADS) lnb_crc_v2_kernel(LnbDecodeBatch b)
{
    lnb_crc_v2_block(b, blockIdx.x);
}
