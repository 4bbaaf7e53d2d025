/* lnb_common.cuh -- types and small helpers shared by every kernel of the B200 LINNE path.
 *
 * Everything marked LNB_HD compiles both as device code (nvcc, sm_100a) and as plain host C++
 * (g++, used ONLY by tests/hostsim to exercise the very same kernel bodies on a machine without
 * a GPU; the product library never calls the host instantiation -- there is no CPU fallback).
 */
#pragma once

#include <stdint.h>
#include <math.h>
#include <float.h>
#include "lnb_types.h"

#if defined(__CUDACC__)
#define LNB_HD  __host__ __device__ __forceinline__          /* free functions */
#define LNB_HDM __host__ __device__ __forceinline__          /* member functions */
#else
#define LNB_HD  static inline
#define LNB_HDM inline
#endif

/* ---- integer helpers (reference libs/linne_internal/include/linne_utility.h:30-32, :55) ---- */
LNB_HD uint32_t lnb_zz_enc(int32_t s) { return ((uint32_t)s << 1) ^ (uint32_t)(s >> 31); }
LNB_HD int32_t lnb_zz_dec(uint32_t u) { return (int32_t)(u >> 1) ^ -(int32_t)(u & 1u); }

/* A sample as the `bytes` (1..4) bytes of a WAV data chunk, little-endian in the low bytes of the result: 8-bit is
 * unsigned with a bias of 128, 16/24/32-bit two's complement (reference libs/wav/src/wav.c:665-700). */
LNB_HD uint32_t lnb_wav_sample(int32_t v, uint32_t bytes)
{
    return bytes == 1u ? (uint32_t)(v + 128) & 0xFFu : (uint32_t)v & (0xFFFFFFFFu >> (32u - 8u * bytes));
}

LNB_HD uint32_t lnb_clz32(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return (uint32_t)__clz((int)x);
#else
    return x ? (uint32_t)__builtin_clz(x) : 32u;
#endif
}
LNB_HD uint32_t lnb_clz64(uint64_t x)
{
#if defined(__CUDA_ARCH__)
    return (uint32_t)__clzll((long long)x);
#else
    return x ? (uint32_t)__builtin_clzll(x) : 64u;
#endif
}
LNB_HD uint32_t lnb_log2_ceil(uint32_t x) { return 32u - lnb_clz32(x - 1u); }
LNB_HD uint32_t lnb_bswap32(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return __byte_perm(x, 0, 0x0123);
#else
    return __builtin_bswap32(x);
#endif
}
LNB_HD double lnb_round_half_away(double d) { return d >= 0.0 ? floor(d + 0.5) : -floor(-d + 0.5); }

/* Unfused multiply-add: the coefficient path (Levinson, quantiser) keeps the reference's
 * two-rounding arithmetic so that it reproduces the CPU result bit for bit; the O(N*P) signal
 * loops (autocorrelation, residual evaluation) use fused DFMA for throughput (DESIGN.md). */
LNB_HD double lnb_mul_rn(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
LNB_HD double lnb_add_rn(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
LNB_HD double lnb_fma(double a, double b, double c)
{
#if defined(__CUDA_ARCH__)
    return fma(a, b, c);
#else
    return __builtin_fma(a, b, c);
#endif
}

/* big-endian field access on a byte pointer (block framing: reference libs/byte_array/include/byte_array.h) */
LNB_HD uint32_t lnb_get_be(const uint8_t *p, int nbytes)
{
    uint32_t v = 0;
    for (int i = 0; i < nbytes; i++) v = (v << 8) | p[i];
    return v;
}
LNB_HD void lnb_put_be(uint8_t *p, uint32_t v, int nbytes)
{
    for (int i = 0; i < nbytes; i++) p[i] = (uint8_t)(v >> (8 * (nbytes - 1 - i)));
}

/* CRC16-IBM (reflected 0xA001, init 0, no final xor): reference linne_utility.c:72-89 */
LNB_HD uint16_t lnb_crc16_serial(const uint16_t *table, const uint8_t *data, uint32_t size)
{
    uint16_t crc = 0;
    for (uint32_t i = 0; i < size; i++) crc = (uint16_t)((crc >> 8) ^ table[(crc ^ data[i]) & 0xFFu]);
    return crc;
}
