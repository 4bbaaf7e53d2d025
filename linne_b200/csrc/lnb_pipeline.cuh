/* lnb_pipeline.cuh -- the batch pipelines: which work-item functor runs over which index space,
 * in which order.  Templated on an executor so the same sequence is
 *   - launched as CUDA kernels on a stream by the product (lnb_kernels.cu), and
 *   - stepped through as plain loops by tests/hostsim (CPU-only CI; not part of the product).
 *
 * An executor provides:  template<class F> void run(const char *name, uint32_t n_items, const F &f);
 */
#pragma once
#include "lnb_common.cuh"
#include "lnb_decode_core.cuh"
#include "lnb_encode_core.cuh"

#define LNB_ITEMS_PER_SLOT 255u          /* units over all unit-count levels: 1 + 2 + ... + 128 */

/* =============================================================================================
 * Decode
 * ============================================================================================= */

/* D0: CRC16 of every block body (type, sample count, payload) vs the transmitted field.
 * reference linne_decoder.c:617-625 */
struct LnbItemCrc {
    LnbDecodeBatch b;
    LNB_HDM void operator()(uint32_t i) const
    {
        LnbBlockDesc &blk = b.blocks[i];
        const uint8_t *p = b.stream + blk.byte_off;
        const uint16_t crc = lnb_crc16_serial(b.tab.crc_table, p + 8, blk.byte_size - 8u);
        blk.crc = crc;
        if (b.cfg.check_crc && crc != (uint16_t)lnb_get_be(p + 6, 2)) blk.status |= LNB_ST_CRC_MISMATCH;
    }
};

/* D1: side information + entropy decode, one block per item */
struct LnbItemEntropy {
    LnbDecodeBatch b;
    LNB_HDM void operator()(uint32_t i) const
    {
        lnb_decode_block_payload(b.cfg, b.tab, b.stream, b.stream_size, b.blocks[i],
                                 b.params + (size_t)i * b.cfg.num_channels, b.pcm);
    }
};

/* D2: synthesis of one layer; item = (block, channel, unit slot) */
struct LnbItemSynth {
    LnbDecodeBatch b;
    uint32_t layer;
    uint32_t skip_upto;             /* block-channels of at most this many samples were done cooperatively */
    LNB_HDM void operator()(uint32_t i) const
    {
        const uint32_t u = i % LNB_MAX_UNITS, bc = i / LNB_MAX_UNITS;
        const uint32_t blk_i = bc / b.cfg.num_channels, c = bc % b.cfg.num_channels;
        const LnbBlockDesc &blk = b.blocks[blk_i];
        if (blk.type != LNB_BLOCK_COMPRESSED || blk.status || blk.nsmp <= skip_upto) return;
        const LnbChanParams &prm = b.params[bc];
        const uint32_t P = b.cfg.layer_params[layer];
        uint32_t U = 1u << prm.log2_units[layer];
        if (u >= U || U > P) return;
        const uint32_t p = P / U, m = blk.nsmp / U;
        int32_t *x = b.pcm + (size_t)c * b.cfg.pcm_stride + blk.smp_off + (size_t)u * m;
        lnb_synthesize_unit(x, m, prm.coef + layer * LNB_MAX_PARAMS + u * p, p, prm.rshift[layer]);
    }
};

/* D3: de-emphasis; item = (block, channel) */
struct LnbItemDeemph {
    LnbDecodeBatch b;
    uint32_t skip_upto;
    LNB_HDM void operator()(uint32_t bc) const
    {
        const uint32_t blk_i = bc / b.cfg.num_channels, c = bc % b.cfg.num_channels;
        const LnbBlockDesc &blk = b.blocks[blk_i];
        if (blk.type != LNB_BLOCK_COMPRESSED || blk.status || blk.nsmp <= skip_upto) return;
        const LnbChanParams &prm = b.params[bc];
        lnb_deemphasis(b.pcm + (size_t)c * b.cfg.pcm_stride + blk.smp_off, blk.nsmp, prm.preem_prev, prm.preem_coef);
    }
};

/* D4: M/S -> L/R; item = (block, sample); a block may be longer than the header's block size */
LNB_HD uint32_t lnb_ms_span(const LnbDecodeBatch &b) { return b.max_nsmp > b.cfg.block_size ? b.max_nsmp : b.cfg.block_size; }
struct LnbItemMsInverse {
    LnbDecodeBatch b;
    LNB_HDM void operator()(uint32_t i) const
    {
        const uint32_t span = lnb_ms_span(b);
        const uint32_t blk_i = i / span, s = i % span;
        const LnbBlockDesc &blk = b.blocks[blk_i];
        if (blk.type != LNB_BLOCK_COMPRESSED || blk.status || s >= blk.nsmp) return;
        if (b.fused_max_n && blk.nsmp <= b.fused_max_n) return;       /* done inside the fused streaming kernel */
        int32_t *l = b.pcm + blk.smp_off + s;
        lnb_ms_to_lr(l[0], l[b.cfg.pcm_stride]);
    }
};

template <class Exec>
void lnb_decode_pipeline(Exec &ex, const LnbDecodeBatch &b)
{
    const uint32_t B = b.num_blocks, C = b.cfg.num_channels;
    if (B == 0) return;
    if (Exec::cooperative) {
        if (b.fused_max_n && b.tput) {
            /* large batches: the full blocks take the lane-per-block kernels; CRC pass and the per-block pipeline kernel
             * for the rest run beside them */
            ex.tput_decode(b);
        } else {
            ex.crc_cooperative(b);                        /* one CTA per block, chunk CRCs combined in GF(2) */
            if (b.fused_max_n) ex.stream_cooperative(b);  /* one CTA per block: entropy decode feeding synthesis, de-emphasis, M/S */
        }
        if (!b.fused_max_n || b.num_plain_blocks) {       /* raw / silent / long blocks (or the fused kernel switched off) */
            ex.entropy_cooperative(b);                    /* one warp per block: 32 speculative code-word starts per round */
            ex.synth_cooperative(b);                      /* one warp per (block, channel): systolic synthesis + de-emphasis */
            if (b.max_nsmp > ex.synth_max_n()) {    /* longer block-channels: flat kernels (they skip the short ones) */
                for (int l = (int)b.cfg.num_layers - 1; l >= 0; l--)
                    ex.run("synth", B * C * LNB_MAX_UNITS, LnbItemSynth{b, (uint32_t)l, ex.synth_max_n()});
                ex.run("deemph", B * C, LnbItemDeemph{b, ex.synth_max_n()});
            }
        }
    } else {
        ex.run("crc", B, LnbItemCrc{b});
        ex.run("entropy", B, LnbItemEntropy{b});
        for (int l = (int)b.cfg.num_layers - 1; l >= 0; l--)
            ex.run("synth", B * C * LNB_MAX_UNITS, LnbItemSynth{b, (uint32_t)l, 0u});
        ex.run("deemph", B * C, LnbItemDeemph{b, 0u});
    }
    if (b.cfg.ms && C >= 2u && (!b.fused_max_n || b.num_plain_blocks))
        ex.run("ms_inverse", B * lnb_ms_span(b), LnbItemMsInverse{b});
}

/* =============================================================================================
 * Packed PCM <-> int32 planes (SURVEY 8f.2): interleaved little-endian samples as in a WAV data chunk
 * (8-bit unsigned with a bias of 128, 16/24/32-bit signed; reference libs/wav/src/wav.c:388-414, :665-700),
 * right-justified in the planes like tools/linne_codec/linne_codec.c:100-105.  Item = one frame.
 * ============================================================================================= */
struct LnbItemUnpackPcm {
    const uint8_t *packed; int32_t *pcm; uint32_t stride, channels, bytes;
    LNB_HDM void operator()(uint32_t i) const
    {
        const uint8_t *p = packed + (size_t)i * channels * bytes;
        for (uint32_t c = 0; c < channels; c++, p += bytes) {
            int32_t v;
            if (bytes == 1u) v = (int32_t)p[0] - 128;
            else if (bytes == 2u) v = (int16_t)((uint32_t)p[0] | ((uint32_t)p[1] << 8));
            else if (bytes == 3u) v = (int32_t)(((uint32_t)p[0] << 8) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 24)) >> 8;
            else v = (int32_t)((uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24));
            pcm[(size_t)c * stride + i] = v;
        }
    }
};
struct LnbItemPackPcm {
    const int32_t *pcm; uint8_t *packed; uint32_t stride, channels, bytes;
    LNB_HDM void operator()(uint32_t i) const
    {
        uint8_t *p = packed + (size_t)i * channels * bytes;
        for (uint32_t c = 0; c < channels; c++, p += bytes) {
            const uint32_t u = lnb_wav_sample(pcm[(size_t)c * stride + i], bytes);
            for (uint32_t k = 0; k < bytes; k++) p[k] = (uint8_t)(u >> (8u * k));
        }
    }
};
template <class Exec>
void lnb_unpack_pcm_pipeline(Exec &ex, const uint8_t *packed, int32_t *pcm, uint32_t stride, uint32_t frames, uint32_t channels, uint32_t bytes)
{
    ex.run("unpack_pcm", frames, LnbItemUnpackPcm{packed, pcm, stride, channels, bytes});
}
template <class Exec>
void lnb_pack_pcm_pipeline(Exec &ex, const int32_t *pcm, uint8_t *packed, uint32_t stride, uint32_t frames, uint32_t channels, uint32_t bytes)
{
    ex.run("pack_pcm", frames, LnbItemPackPcm{pcm, packed, stride, channels, bytes});
}

/* =============================================================================================
 * Encode
 * ============================================================================================= */


struct LnbItemEstimate {            /* E0: (block, channel) */
    LnbEncodeBatch b;
    LNB_HDM void operator()(uint32_t bc) const
    {
        const uint32_t blk_i = bc / b.cfg.num_channels, c = bc % b.cfg.num_channels;
        const LnbBlockDesc &blk = b.blocks[blk_i];
        if (blk.status & LNB_ENC_FLAG_COOP) return;
        b.est[bc] = lnb_estimate_bits(b.pcm + (size_t)c * b.cfg.pcm_stride + blk.smp_off, blk.nsmp,
                                      b.cfg.bits_per_sample, b.cfg.layer_params[0]);
    }
};

struct LnbItemPrepare {             /* E1: (block) */
    LnbEncodeBatch b;
    LNB_HDM void operator()(uint32_t i) const
    {
        const uint32_t C = b.cfg.num_channels;
        if (b.blocks[i].status & LNB_ENC_FLAG_COOP) return;
        lnb_prepare_block(b.cfg, b.blocks[i], b.est + (size_t)i * C, b.pcm,
                          b.work + (size_t)i * C * b.cfg.work_stride, b.params + (size_t)i * C);
    }
};

struct LnbItemToDouble {            /* (slot, sample): normalised copy of the work signal */
    LnbEncodeBatch b;
    LNB_HDM void operator()(uint32_t i) const
    {
        const uint32_t s = i / b.cfg.work_stride, t = i % b.cfg.work_stride;
        const uint32_t bc = s / b.cfg.num_lambdas, blk_i = bc / b.cfg.num_channels;
        const LnbBlockDesc &blk = b.blocks[blk_i];
        if (blk.type != LNB_BLOCK_COMPRESSED || (blk.status & (LNB_ENC_FLAG_FAST | LNB_ENC_FLAG_GENERIC))) return;
        const double norm = ldexp(1.0, -(int)(b.cfg.bits_per_sample - 1u));
        b.sig_a[(size_t)s * b.cfg.work_stride + t] =
            (t < blk.na) ? (double)b.work[(size_t)bc * b.cfg.work_stride + t] * norm : 0.0;
    }
};

#define LNB_CHUNK 64u                       /* samples per loss / forward work item of the flat path */

LNB_HDM uint32_t lnb_num_chunks(uint32_t na) { return (na + LNB_CHUNK - 1u) / LNB_CHUNK; }

struct LnbItemAcorr {               /* E2a: (slot, level, unit, lag) -- 256 (unit, lag) cells per level */
    LnbEncodeBatch b;
    uint32_t layer;
    const double *sig;
    LNB_HDM void operator()(uint32_t i) const
    {
        const uint32_t s = i / (LNB_MAX_LEVELS * 256u), cell = i % (LNB_MAX_LEVELS * 256u);
        const uint32_t level = cell / 256u, r = cell % 256u;
        const uint32_t bc = s / b.cfg.num_lambdas, blk_i = bc / b.cfg.num_channels;
        const LnbBlockDesc &blk = b.blocks[blk_i];
        if (blk.type != LNB_BLOCK_COMPRESSED || (blk.status & (LNB_ENC_FLAG_FAST | LNB_ENC_FLAG_GENERIC))) return;
        const uint32_t P = b.cfg.layer_params[layer];
        if (!lnb_level_valid(level, P, blk.na)) return;
        const uint32_t U = 1u << level, p = P / U, m = blk.na / U;
        if (r >= U * (p + 1u)) return;
        const uint32_t u = r / (p + 1u), lag = r % (p + 1u);
        b.acorr[(size_t)s * LNB_MAX_LEVELS * 256u + cell] =
            lnb_acorr_lag(sig + (size_t)s * b.cfg.work_stride + (size_t)u * m, m, lag,
                          b.welch[(size_t)blk_i * LNB_MAX_LEVELS + level]);
    }
};

struct LnbItemSolve {               /* E2b: (slot, level, unit) */
    LnbEncodeBatch b;
    uint32_t layer;
    LNB_HDM void operator()(uint32_t i) const
    {
        const uint32_t s = i / LNB_ITEMS_PER_SLOT, id = i % LNB_ITEMS_PER_SLOT + 1u;
        const uint32_t level = 31u - lnb_clz32(id), u = id - (1u << level);
        const uint32_t bc = s / b.cfg.num_lambdas, lam = s % b.cfg.num_lambdas;
        const uint32_t blk_i = bc / b.cfg.num_channels;
        const LnbBlockDesc &blk = b.blocks[blk_i];
        if (blk.type != LNB_BLOCK_COMPRESSED || (blk.status & (LNB_ENC_FLAG_FAST | LNB_ENC_FLAG_GENERIC))) return;
        const uint32_t P = b.cfg.layer_params[layer];
        if (!lnb_level_valid(level, P, blk.na)) return;
        const uint32_t U = 1u << level, p = P / U, m = blk.na / U;
        lnb_solve_unit(b.acorr + ((size_t)s * LNB_MAX_LEVELS + level) * 256u + (size_t)u * (p + 1u), p, m,
                       b.cfg.lambdas[lam],
                       b.cand + ((size_t)s * LNB_MAX_LEVELS + level) * LNB_MAX_PARAMS + (size_t)u * p);
    }
};

struct LnbItemLoss {                /* E2c: (slot, level, chunk) */
    LnbEncodeBatch b;
    uint32_t layer;
    const double *sig;
    uint32_t chunks_per_slot;       /* lnb_num_chunks(work_stride) */
    LNB_HDM void operator()(uint32_t i) const
    {
        const uint32_t per_slot = LNB_MAX_LEVELS * chunks_per_slot;
        const uint32_t s = i / per_slot, level = (i % per_slot) / chunks_per_slot, g = i % chunks_per_slot;
        const uint32_t bc = s / b.cfg.num_lambdas, blk_i = bc / b.cfg.num_channels;
        const LnbBlockDesc &blk = b.blocks[blk_i];
        if (blk.type != LNB_BLOCK_COMPRESSED || (blk.status & (LNB_ENC_FLAG_FAST | LNB_ENC_FLAG_GENERIC))) return;
        const uint32_t P = b.cfg.layer_params[layer];
        if (!lnb_level_valid(level, P, blk.na)) return;
        const uint32_t t0 = g * LNB_CHUNK;
        if (t0 >= blk.na) return;
        const uint32_t t1 = (t0 + LNB_CHUNK < blk.na) ? t0 + LNB_CHUNK : blk.na;
        const uint32_t U = 1u << level, p = P / U, m = blk.na / U;
        b.unit_loss[((size_t)s * LNB_MAX_LEVELS + level) * chunks_per_slot + g] =
            lnb_loss_chunk(sig + (size_t)s * b.cfg.work_stride, t0, t1, m, p,
                           b.cand + ((size_t)s * LNB_MAX_LEVELS + level) * LNB_MAX_PARAMS);
    }
};

struct LnbItemSelect {              /* E3: (slot): first minimum over the unit counts (linne_network.c:337-341) */
    LnbEncodeBatch b;
    uint32_t layer;
    uint32_t chunks_per_slot;
    LNB_HDM void operator()(uint32_t s) const
    {
        const uint32_t bc = s / b.cfg.num_lambdas, blk_i = bc / b.cfg.num_channels;
        const LnbBlockDesc &blk = b.blocks[blk_i];
        if (blk.type != LNB_BLOCK_COMPRESSED || (blk.status & (LNB_ENC_FLAG_FAST | LNB_ENC_FLAG_GENERIC))) return;
        const uint32_t P = b.cfg.layer_params[layer];
        const uint32_t nch = lnb_num_chunks(blk.na);
        double best_loss = (double)FLT_MAX;
        uint32_t best = 0;
        for (uint32_t level = 0; level < LNB_MAX_LEVELS; level++) {
            if (!lnb_level_valid(level, P, blk.na)) continue;
            const double *ul = b.unit_loss + ((size_t)s * LNB_MAX_LEVELS + level) * chunks_per_slot;
            double loss = 0.0;
            for (uint32_t g = 0; g < nch; g++) loss += ul[g];
            loss /= (double)blk.na;
            if (loss < best_loss) { best_loss = loss; best = level; }
        }
        b.chosen_log2u[(size_t)s * LNB_MAX_LAYERS + layer] = (uint8_t)best;
        const double *src = b.cand + ((size_t)s * LNB_MAX_LEVELS + best) * LNB_MAX_PARAMS;
        double *dst = b.chosen_w + ((size_t)s * LNB_MAX_LAYERS + layer) * LNB_MAX_PARAMS;
        for (uint32_t k = 0; k < P; k++) dst[k] = src[k];
    }
};

struct LnbItemForward {             /* E4: (slot, chunk) */
    LnbEncodeBatch b;
    uint32_t layer;
    const double *sig_in;
    double *sig_out;
    uint32_t chunks_per_slot;
    LNB_HDM void operator()(uint32_t i) const
    {
        const uint32_t s = i / chunks_per_slot, g = i % chunks_per_slot;
        const uint32_t bc = s / b.cfg.num_lambdas, blk_i = bc / b.cfg.num_channels;
        const LnbBlockDesc &blk = b.blocks[blk_i];
        if (blk.type != LNB_BLOCK_COMPRESSED || (blk.status & (LNB_ENC_FLAG_FAST | LNB_ENC_FLAG_GENERIC))) return;
        double *fs = b.final_sum + (size_t)s * chunks_per_slot + g;
        const uint32_t t0 = g * LNB_CHUNK;
        if (t0 >= blk.na) { *fs = 0.0; return; }
        const uint32_t t1 = (t0 + LNB_CHUNK < blk.na) ? t0 + LNB_CHUNK : blk.na;
        const uint32_t U = 1u << b.chosen_log2u[(size_t)s * LNB_MAX_LAYERS + layer];
        const uint32_t P = b.cfg.layer_params[layer], p = P / U, m = blk.na / U;
        const size_t ws = b.cfg.work_stride;
        *fs = lnb_forward_chunk(sig_in + (size_t)s * ws, sig_out + (size_t)s * ws, t0, t1, m, p,
                                b.chosen_w + ((size_t)s * LNB_MAX_LAYERS + layer) * LNB_MAX_PARAMS);
    }
};

struct LnbItemFinish {              /* E5: (block, channel): best regulariser, quantise (linne_network.c:618-629) */
    LnbEncodeBatch b;
    uint32_t chunks_per_slot;
    LNB_HDM void operator()(uint32_t bc) const
    {
        const uint32_t blk_i = bc / b.cfg.num_channels;
        const LnbBlockDesc &blk = b.blocks[blk_i];
        if (blk.type != LNB_BLOCK_COMPRESSED) return;
        const uint32_t nch = lnb_num_chunks(blk.na);
        double best_loss = (double)FLT_MAX;
        uint32_t best = 0;
        for (uint32_t lam = 0; lam < b.cfg.num_lambdas; lam++) {
            const size_t s = (size_t)bc * b.cfg.num_lambdas + lam;
            double sum = 0.0;
            for (uint32_t g = 0; g < nch; g++) sum += b.final_sum[s * chunks_per_slot + g];
            const double loss = sum / (double)blk.na;
            if (loss < best_loss) { best_loss = loss; best = lam; }
        }
        const size_t s = (size_t)bc * b.cfg.num_lambdas + best;
        LnbChanParams &prm = b.params[bc];
        for (uint32_t l = 0; l < b.cfg.num_layers; l++) {
            prm.log2_units[l] = b.chosen_log2u[s * LNB_MAX_LAYERS + l];
            lnb_quantize_layer(b.chosen_w + (s * LNB_MAX_LAYERS + l) * LNB_MAX_PARAMS, b.cfg.layer_params[l],
                               prm.coef + l * LNB_MAX_PARAMS, &prm.rshift[l]);
        }
    }
};

struct LnbItemPredict {             /* E6: (block, channel, unit slot), one layer */
    LnbEncodeBatch b;
    uint32_t layer;
    LNB_HDM void operator()(uint32_t i) const
    {
        const uint32_t u = i % LNB_MAX_UNITS, bc = i / LNB_MAX_UNITS;
        const uint32_t blk_i = bc / b.cfg.num_channels;
        const LnbBlockDesc &blk = b.blocks[blk_i];
        if (blk.type != LNB_BLOCK_COMPRESSED || (blk.status & LNB_ENC_FLAG_COOP)) return;
        const LnbChanParams &prm = b.params[bc];
        const uint32_t P = b.cfg.layer_params[layer], U = 1u << prm.log2_units[layer];
        if (u >= U || U > P) return;
        const uint32_t p = P / U, m = blk.nsmp / U;
        lnb_predict_unit_inplace(b.work + (size_t)bc * b.cfg.work_stride + (size_t)u * m, m,
                                 prm.coef + layer * LNB_MAX_PARAMS + u * p, p, prm.rshift[layer]);
    }
};

struct LnbItemPlan {                /* E7: (block, channel) */
    LnbEncodeBatch b;
    LNB_HDM void operator()(uint32_t bc) const
    {
        const uint32_t blk_i = bc / b.cfg.num_channels;
        const LnbBlockDesc &blk = b.blocks[blk_i];
        if (blk.type != LNB_BLOCK_COMPRESSED || (blk.status & LNB_ENC_FLAG_COOP)) return;
        lnb_coder_plan(b.tab.k2_threshold, b.work + (size_t)bc * b.cfg.work_stride, blk.nsmp,
                       b.plan_mean + (size_t)bc * 2u * LNB_MAX_PARTITIONS, b.plans[bc]);
    }
};

struct LnbItemSize {                /* E8a: (block) */
    LnbEncodeBatch b;
    LNB_HDM void operator()(uint32_t i) const
    {
        LnbBlockDesc &blk = b.blocks[i];
        const uint32_t C = b.cfg.num_channels;
        uint32_t payload = 0;
        if (blk.type == LNB_BLOCK_RAW) payload = (b.cfg.bits_per_sample >> 3) * blk.nsmp * C;
        else if (blk.type == LNB_BLOCK_COMPRESSED) {
            uint64_t bits = lnb_side_info_bits(b.cfg, b.tab, b.params + (size_t)i * C);
            for (uint32_t c = 0; c < C; c++) bits += b.plans[(size_t)i * C + c].bits;
            payload = (uint32_t)((bits + 7u) >> 3);
        }
        blk.byte_size = LNB_BLOCK_HEADER_SIZE + payload;
    }
};

struct LnbItemScan {                /* E8b: single item: exclusive scan of the block sizes */
    LnbEncodeBatch b;
    LNB_HDM void operator()(uint32_t) const
    {
        uint32_t off = b.out_base;
        for (uint32_t i = 0; i < b.num_blocks; i++) { b.blocks[i].byte_off = off; off += b.blocks[i].byte_size; }
        *b.total_size = off - b.out_base;
    }
};

struct LnbItemPack {                /* E9: (block) */
    LnbEncodeBatch b;
    uint32_t out_capacity;
    LNB_HDM void operator()(uint32_t i) const
    {
        const LnbBlockDesc &blk = b.blocks[i];
        const uint32_t C = b.cfg.num_channels;
        if ((uint64_t)blk.byte_off + blk.byte_size > out_capacity) return;      /* host reports INSUFFICIENT_BUFFER */
        if (blk.status & LNB_ENC_FLAG_PACKED) return;                           /* done by the cooperative packer */
        lnb_pack_block(b.cfg, b.tab, blk, b.params + (size_t)i * C, b.plans + (size_t)i * C, b.pcm,
                       b.work + (size_t)i * C * b.cfg.work_stride, b.out + blk.byte_off);
    }
};

/* Stages E0..E8: everything up to (and including) the size scan.  Packing is a separate call so the
 * host can check the output capacity (and place the batch) in between. */
template <class Exec>
void lnb_encode_analyze_pipeline(Exec &ex, const LnbEncodeBatch &b)
{
    const uint32_t B = b.num_blocks, C = b.cfg.num_channels;
    if (B == 0) return;
    const uint32_t S = B * C * b.cfg.num_lambdas;
    const uint32_t CH = lnb_num_chunks(b.cfg.work_stride);    /* chunk slots per analysis slot */
    const bool flat = b.num_coop_blocks < B;                /* some blocks are too long for the cooperative kernels */
    if (b.num_coop_blocks) ex.prepare_cooperative(b);
    if (flat) {
        ex.run("estimate", B * C, LnbItemEstimate{b});
        ex.run("prepare", B, LnbItemPrepare{b});
    }
    if (!b.forced_params) {
        if (b.num_fast_blocks) ex.analyze_cooperative(b);        /* one CTA per slot, signal in shared memory */
        if (b.num_slow_blocks) {                                  /* shapes the cooperative kernel does not take */
            ex.run("to_double", S * b.cfg.work_stride, LnbItemToDouble{b});
            double *cur = b.sig_a, *nxt = b.sig_b;
            for (uint32_t l = 0; l < b.cfg.num_layers; l++) {
                ex.run("acorr", S * LNB_MAX_LEVELS * 256u, LnbItemAcorr{b, l, cur});
                ex.run("solve", S * LNB_ITEMS_PER_SLOT, LnbItemSolve{b, l});
                ex.run("loss", S * LNB_MAX_LEVELS * CH, LnbItemLoss{b, l, cur, CH});
                ex.run("select", S, LnbItemSelect{b, l, CH});
                ex.run("forward", S * CH, LnbItemForward{b, l, cur, nxt, CH});
                double *t = cur; cur = nxt; nxt = t;
            }
        }
        if (b.af_iterations || b.enable_learning) ex.refine_cooperative(b, CH);   /* IRLS / SGD final pass (rows a14, a15) */
        ex.run("finish", B * C, LnbItemFinish{b, CH});
    }
    if (b.num_coop_blocks) ex.predict_plan_cooperative(b);
    if (flat) {
        for (uint32_t l = 0; l < b.cfg.num_layers; l++)
            ex.run("predict", B * C * LNB_MAX_UNITS, LnbItemPredict{b, l});
        ex.run("plan", B * C, LnbItemPlan{b});
    }
    ex.run("size", B, LnbItemSize{b});
    if (Exec::cooperative) ex.scan_cooperative(b);           /* one CTA: run sums -> scan -> offsets */
    else ex.run("scan", 1, LnbItemScan{b});
}

template <class Exec>
void lnb_encode_pack_pipeline(Exec &ex, const LnbEncodeBatch &b, uint32_t out_capacity)
{
    if (b.num_blocks == 0) return;
    ex.pack_cooperative(b, out_capacity);                 /* one CTA per block; skips images too large for shared memory */
    ex.run("pack", b.num_blocks, LnbItemPack{b, out_capacity});
}
