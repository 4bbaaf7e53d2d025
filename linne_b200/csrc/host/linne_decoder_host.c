/* linne_decoder_host.c -- LINNEDecoder_* entry points (include/linne_decoder.h) on top of the CUDA shim.
 *
 * Replaces reference libs/linne_decoder/src/linne_decoder.c.  The host side does what is serial and
 * tiny (argument checks, the 30-byte header, hopping over the block size fields to build the block
 * table); everything that touches samples or payload bits runs on the GPU, batched over every block
 * of the call.  Error results and their precedence follow the reference (cited per check).
 */
#define _POSIX_C_SOURCE 200112L
#include "linne_decoder.h"
#include "linne_b200.h"
#include "lnb_host_util.h"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <pthread.h>
#include <time.h>

/* LINNE_B200_TRACE=1: host-side time stamps of a range's phases on stderr (debugging aid) */
static int dec_trace_on(void) { static int on = -1; if (on < 0) { const char *e = getenv("LINNE_B200_TRACE"); on = (e && *e == '1') ? 1 : 0; } return on; }
static double dec_now_ms(void) { struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; }
#define DEC_TRACE(dec, what) do { if (dec_trace_on()) fprintf(stderr, "[trace] range %2u %-16s %.3f\n", (unsigned)(dec)->turn_index, what, dec_now_ms()); } while (0)

#define DEC_FLAG_OWN_WORK   (1u << 0)
#define DEC_FLAG_HEADER_SET (1u << 1)
#define DEC_FLAG_CHECK_CRC  (1u << 2)

struct LINNEDecoder {
    struct LINNEHeader header;
    uint32_t max_num_channels, max_num_layers, max_num_parameters_per_layer;
    uint32_t flags;
    void *work;
    LnbDevice *dev;
    LnbBuf d_stream, d_blocks, d_params, d_pcm, d_packed;
    LnbBuf h_blocks;                       /* pinned LnbBlockDesc[]: the block table of every call */
    LnbBuf h_stream;                       /* pinned copy of a device-resident stream (block hop on the host: fallback only) */
    LnbBuf d_hop_files, d_hop_res, d_hop_table, h_hop;     /* device-side block hop: records, results, table; pinned staging */
    LnbBuf h_pcm;                          /* pinned int32 [C][stage_stride]: PCM staging of DecodeBlock / read-ahead cache */
    LnbBuf h_win, d_win;                   /* window decodes: seek inputs + gather records (pinned staging, device copy) */
    LnbBuf h_win_img, h_win_pcm;           /* window decodes of host buffers: the needed blocks' bytes, the windows' samples (pinned) */
    /* DecodeBlock read-ahead (SURVEY 8f.4): blocks decoded ahead of the caller in one batch and served from here */
    uint32_t readahead;                    /* blocks decoded per batch by DecodeBlock (<= 1: batch of one) */
    uint32_t tput_min_blocks;              /* batches of at least this many blocks take the throughput kernels (0 = never) */
    uint32_t stage_stride;                 /* samples per plane of h_pcm in the last staged call */
    uint32_t ra_count, ra_next;            /* cached blocks / next one to serve */
    uint8_t *ra_image;                     /* the cached blocks' bytes (validated against the caller's on every hit) */
    size_t ra_image_cap;
    struct LnbCachedBlock { uint32_t byte_off, byte_size, smp_off, nsmp; } *ra_blocks;
    uint32_t ra_blocks_cap;
    /* several GPUs behind one handle (SURVEY 8e): DecodeWhole splits the block table into contiguous ranges, one child
     * handle (own device, own host thread) per range */
    uint32_t num_devices;
    struct LINNEDecoder *child[LNB_MAX_DEVICES];
    LnbTurnstile *turn;                    /* a child: the turnstile of the call it works for (else NULL) and its range index */
    uint32_t turn_index;
    int rank_override;                     /* >= 0: the stream priority rank of a child (its place in the pipeline) instead of the preset's */
    struct LINNEDecoderConfig config;
};
#define LNB_MAX_READAHEAD 1024u
#define LNB_READAHEAD_MAX_SAMPLES (1u << 21)  /* per channel and batch: bounds the pinned PCM cache (8 ch: 64 MiB) */
#define LNB_TPUT_MIN_BLOCKS 2560ul

/* reference linne_decoder.c:60-131 */
LINNEApiResult LINNEDecoder_DecodeHeader(const uint8_t *data, uint32_t data_size, struct LINNEHeader *header)
{
    if (data == NULL || header == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (data_size < LINNE_HEADER_SIZE) return LINNE_APIRESULT_INSUFFICIENT_DATA;
    if (data[0] != 'I' || data[1] != 'B' || data[2] != 'R' || data[3] != 'A') return LINNE_APIRESULT_INVALID_FORMAT;
    lnb_header_read(data, header);
    return LINNE_APIRESULT_OK;
}

static int config_ok(const struct LINNEDecoderConfig *c)
{
    return c && c->max_num_channels && c->max_num_layers && c->max_num_parameters_per_layer;
}

/* reference linne_decoder.c:187-216: the work area only has to hold the host handle here */
int32_t LINNEDecoder_CalculateWorkSize(const struct LINNEDecoderConfig *config)
{
    if (!config_ok(config)) return -1;
    return (int32_t)(sizeof(struct LINNEDecoder) + LNB_ALIGNMENT);
}

/* reference linne_decoder.c:219-296 */
struct LINNEDecoder *LINNEDecoder_Create(const struct LINNEDecoderConfig *config, void *work, int32_t work_size)
{
    struct LINNEDecoder *dec;
    int own = 0;
    if (work == NULL && work_size == 0) {
        if ((work_size = LINNEDecoder_CalculateWorkSize(config)) < 0) return NULL;
        work = malloc((size_t)work_size);
        own = 1;
    }
    if (!config_ok(config) || work == NULL || work_size < LINNEDecoder_CalculateWorkSize(config)) {
        if (own) free(work);
        return NULL;
    }
    dec = (struct LINNEDecoder *)LNB_ROUNDUP((uintptr_t)work, LNB_ALIGNMENT);
    memset(dec, 0, sizeof(*dec));
    dec->rank_override = -1;
    dec->work = work;
    dec->max_num_channels = config->max_num_channels;
    dec->max_num_layers = config->max_num_layers;
    dec->max_num_parameters_per_layer = config->max_num_parameters_per_layer;
    dec->config = *config;
    if (own) dec->flags |= DEC_FLAG_OWN_WORK;
    if (config->check_crc == 1) dec->flags |= DEC_FLAG_CHECK_CRC;
    {   /* LINNE_B200_READAHEAD=K: DecodeBlock decodes K blocks per batch (same results, see decode_block_cached) */
        const char *e = getenv("LINNE_B200_READAHEAD");
        const long k = e ? strtol(e, NULL, 10) : 0;
        dec->readahead = (k > 1) ? (uint32_t)(k > (long)LNB_MAX_READAHEAD ? (long)LNB_MAX_READAHEAD : k) : 0u;
    }
    {   /* LINNE_B200_TPUT_MIN_BLOCKS=N moves the switch-over point to the throughput decoder (0 = never) */
        const char *e = getenv("LINNE_B200_TPUT_MIN_BLOCKS");
        dec->tput_min_blocks = e ? (uint32_t)strtoul(e, NULL, 10) : (uint32_t)LNB_TPUT_MIN_BLOCKS;
    }
    if (lnb_shim_open(&dec->dev, -1) != 0) {
        fprintf(stderr, "linne_b200: no usable CUDA device -- the decoder has no CPU fallback\n");
        if (own) free(work);
        return NULL;
    }
    {   /* LINNE_B200_GPUS=N (or "all"): DecodeWhole of this handle shards its blocks over N devices */
        const char *e = getenv("LINNE_B200_GPUS");
        if (e && *e) LINNEB200_DecoderSetDevices(dec, (e[0] == 'a') ? (uint32_t)lnb_shim_device_count() : (uint32_t)strtoul(e, NULL, 10));
    }
    return dec;
}

/* reference linne_decoder.c:299-306 */
void LINNEDecoder_Destroy(struct LINNEDecoder *dec)
{
    uint32_t k;
    if (dec == NULL) return;
    for (k = 0; k < LNB_MAX_DEVICES; k++) if (dec->child[k]) { LINNEDecoder_Destroy(dec->child[k]); dec->child[k] = NULL; }
    if (dec->dev) {
        lnb_buf_release_device(dec->dev, &dec->d_stream);
        lnb_buf_release_device(dec->dev, &dec->d_blocks);
        lnb_buf_release_device(dec->dev, &dec->d_params);
        lnb_buf_release_device(dec->dev, &dec->d_pcm);
        lnb_buf_release_device(dec->dev, &dec->d_packed);
        lnb_buf_release_device(dec->dev, &dec->d_hop_files);
        lnb_buf_release_device(dec->dev, &dec->d_hop_res);
        lnb_buf_release_device(dec->dev, &dec->d_hop_table);
        lnb_buf_release_host(&dec->h_hop);
        lnb_buf_release_host(&dec->h_blocks);
        lnb_buf_release_host(&dec->h_stream);
        lnb_buf_release_host(&dec->h_pcm);
        lnb_buf_release_device(dec->dev, &dec->d_win);
        lnb_buf_release_host(&dec->h_win);
        lnb_buf_release_host(&dec->h_win_img);
        lnb_buf_release_host(&dec->h_win_pcm);
        free(dec->ra_image); dec->ra_image = NULL; dec->ra_image_cap = 0;
        free(dec->ra_blocks); dec->ra_blocks = NULL; dec->ra_blocks_cap = 0;
        dec->ra_count = dec->ra_next = 0;
        lnb_shim_close(dec->dev);
        dec->dev = NULL;
    }
    if (dec->flags & DEC_FLAG_OWN_WORK) free(dec->work);
}

/* reference linne_decoder.c:309-354 */
LINNEApiResult LINNEDecoder_SetHeader(struct LINNEDecoder *dec, const struct LINNEHeader *header)
{
    const LnbPreset *ps;
    int i;
    if (dec == NULL || header == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (!lnb_header_fields_valid(header)) return LINNE_APIRESULT_INVALID_FORMAT;
    if (dec->max_num_channels < header->num_channels) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
    ps = &g_lnb_presets[header->preset];
    if (dec->max_num_layers < (uint32_t)ps->num_layers) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
    for (i = 0; i < ps->num_layers; i++)
        if (dec->max_num_parameters_per_layer < (uint32_t)ps->layer_params[i]) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
    if (header->num_channels > LINNE_MAX_NUM_CHANNELS) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
    dec->header = *header;
    dec->flags |= DEC_FLAG_HEADER_SET;
    dec->ra_count = dec->ra_next = 0;                          /* cached blocks belong to the previous header */
    lnb_shim_set_cost_rank(dec->dev, dec->rank_override >= 0 ? dec->rank_override : (int)header->preset);     /* longer predictors first (scheduling hint) */
    return LINNE_APIRESULT_OK;
}

/* Block table: the hop over the size fields (lnb_framing.h; serial by nature, a few ns per block) of data[off, data_size)
 * into dec->h_blocks from entry `first` on, the entries before it kept (a call over several streams appends them).  The
 * table grows until the hop fits.  Byte offsets are relative to `data`. */
static int hop_host(struct LINNEDecoder *dec, const struct LINNEHeader *h, const uint8_t *data, uint32_t data_size, uint32_t off,
                    uint32_t room, uint32_t sample_limit, uint32_t block_limit, uint32_t first, LnbHopResult *res)
{
    uint32_t want = block_limit ? block_limit : (uint32_t)((uint64_t)(data_size - off) / 64u + 16u);
    if (!block_limit && h->num_samples_per_block && sample_limit / h->num_samples_per_block + 16u < want)
        want = (sample_limit / h->num_samples_per_block + 16u) * 2u;
    for (;;) {
        const size_t cap = dec->h_blocks.cap / sizeof(LnbBlockDesc);
        if (dec->h_blocks.ptr == NULL || cap < (size_t)first + want) {
            LnbBuf grown = { NULL, 0 };
            if (lnb_buf_reserve_host(&grown, ((size_t)first + want) * sizeof(LnbBlockDesc))) return 1;
            if (first) memcpy(grown.ptr, dec->h_blocks.ptr, (size_t)first * sizeof(LnbBlockDesc));
            lnb_buf_release_host(&dec->h_blocks);
            dec->h_blocks = grown;
            continue;
        }
        lnb_hop_blocks(data, data_size, off, h->num_channels, h->bits_per_sample, room, sample_limit, block_limit,
                       (LnbBlockDesc *)dec->h_blocks.ptr + first, (uint32_t)(cap - first), 0u, res);
        if (!res->overflow) return 0;
        want = (uint32_t)(cap - first) * 2u;
    }
}

/* the result of a stream whose blocks all pass their CRC check */
static LINNEApiResult hop_status(const LnbHopResult *r)
{
    return (LINNEApiResult)(r->num_blocks > r->num_decodable ? r->post_crc_error : r->framing_error);
}

/* Reserves the device block table and parameters of `nb` blocks and fills `batch` for them: the handle's stream
 * parameters and CRC setting, the tables, the pointers and the routing.  The routing is the same for every caller:
 * compressed blocks go to the fused streaming kernel (unless LINNE_B200_SPLIT_DECODE=1), what is left is counted for the
 * split kernels, the longest block sizes their shared-memory lines, and batches of at least tput_min_blocks blocks take
 * the throughput kernels (eight lanes per block / one per (block, channel) instead of one CTA per block,
 * lnb_tput_v2.cuh). */
static int setup_batch(struct LINNEDecoder *dec, LnbDecodeBatch *batch, const LnbBlockDesc *blocks, uint32_t nb,
                       const uint8_t *stream, uint32_t stream_size, int32_t *pcm, uint32_t pcm_stride)
{
    const char *split = getenv("LINNE_B200_SPLIT_DECODE");
    const uint32_t min_blocks = dec->tput_min_blocks;
    uint32_t i;
    if (lnb_buf_reserve_device(dec->dev, &dec->d_blocks, (size_t)nb * sizeof(LnbBlockDesc))
        || lnb_buf_reserve_device(dec->dev, &dec->d_params, (size_t)nb * dec->header.num_channels * sizeof(LnbChanParams)))
        return 1;
    lnb_fill_stream_cfg(&batch->cfg, &dec->header);
    batch->cfg.pcm_stride = pcm_stride;
    batch->cfg.work_stride = 0;
    batch->cfg.check_crc = (dec->flags & DEC_FLAG_CHECK_CRC) ? 1u : 0u;
    batch->fused_max_n = (split && *split == '1') ? 0u : lnb_shim_fused_max_n();
    batch->num_plain_blocks = 0;
    batch->max_nsmp = 0;
    for (i = 0; i < nb; i++) {
        if (blocks[i].type != LNB_BLOCK_COMPRESSED || blocks[i].nsmp == 0u || blocks[i].nsmp > batch->fused_max_n)
            batch->num_plain_blocks++;
        if (blocks[i].nsmp > batch->max_nsmp) batch->max_nsmp = blocks[i].nsmp;
    }
    batch->tput = (min_blocks && nb >= min_blocks && batch->fused_max_n
                   && ((uintptr_t)pcm & 15u) == 0u && (pcm_stride & 3u) == 0u
                   && lnb_shim_tput_supported(&batch->cfg)) ? 1u : 0u;
    batch->tab = *lnb_shim_tables(dec->dev);
    batch->stream = stream;
    batch->stream_size = stream_size;
    batch->blocks = (LnbBlockDesc *)dec->d_blocks.ptr;
    batch->num_blocks = nb;
    batch->params = (LnbChanParams *)dec->d_params.ptr;
    batch->pcm = pcm;
    return 0;
}

/* the first block of blocks[from, to) whose CRC failed, or `to` (also when the handle does not check CRCs) */
static uint32_t first_crc_failure(const struct LINNEDecoder *dec, const LnbBlockDesc *blocks, uint32_t from, uint32_t to)
{
    uint32_t i;
    if (dec->flags & DEC_FLAG_CHECK_CRC)
        for (i = from; i < to; i++) if (blocks[i].status & LNB_ST_CRC_MISMATCH) return i;
    return to;
}

/* One range of a stream for decode_range(), shared by DecodeBlock (block_limit >= 1, staged) and DecodeWhole
 * (block_limit = 0): the blocks found from data[start_offset] on (header already set), at most block_limit blocks /
 * sample_limit samples, checked against `room` samples of output.
 * Resident mode (d_stream / d_pcm non-NULL): the stream image and/or the PCM planes (stride pcm_stride) already live on
 * the device, so the corresponding bulk copy is skipped; `data` (host) is still needed for the block hop.
 * Staged mode (`staged`): the PCM comes back into the handle's pinned planes (dec->h_pcm, stride dec->stage_stride)
 * together with the block table, behind ONE synchronisation; the caller hands samples on from there.  Otherwise the
 * samples go to the caller's planes `buffer`. */
typedef struct {
    const uint8_t *data;
    uint32_t data_size, start_offset;
    int32_t **buffer;
    uint32_t room, sample_limit, block_limit;
    int staged;
    const uint8_t *d_stream;
    int32_t *d_pcm;
    uint32_t pcm_stride;
} RangeRequest;

/* What decode_range() found: the hop's result (the block table stays in dec->h_blocks), the first block that failed
 * (hop.num_blocks: none), the bytes the hop walked over and the samples handed back. */
typedef struct {
    LnbHopResult hop;
    uint32_t first_bad, consumed, decoded;
} RangeResult;

static LINNEApiResult decode_range(struct LINNEDecoder *dec, const RangeRequest *rq, RangeResult *out)
{
    const struct LINNEHeader *h = &dec->header;
    const uint32_t C = h->num_channels;
    LnbDecodeBatch batch;
    LnbHopResult scan;
    LnbBlockDesc *blocks;
    uint32_t pcm_stride, first_bad, ok_samples, c, i, used;
    size_t padded;
    LINNEApiResult result;

    memset(out, 0, sizeof(*out));
    if (hop_host(dec, h, rq->data, rq->data_size, rq->start_offset, rq->room, rq->sample_limit, rq->block_limit, 0u, &scan))
        return LINNE_APIRESULT_NG;
    out->hop = scan;
    blocks = (LnbBlockDesc *)dec->h_blocks.ptr;
    if (scan.num_blocks == 0) return (LINNEApiResult)scan.framing_error;    /* OK when there was simply nothing to do */

    /* bytes of the image the blocks of this call span: a streaming caller passes everything that is left of its
     * stream with every DecodeBlock (tools/linne_player/linne_player.c:110-121) -- only this much is uploaded */
    used = scan.end_offset;
    for (i = 0; i < scan.num_blocks; i++) {
        const uint64_t end = (uint64_t)blocks[i].byte_off + blocks[i].byte_size;
        if (end > used) used = (end > rq->data_size) ? rq->data_size : (uint32_t)end;
    }
    if (!rq->block_limit || rq->d_stream) used = rq->data_size;

    /* device buffers */
    padded = LNB_ROUNDUP((size_t)used + 16u, 16u);
    {   /* the terminal block (post-CRC error) may not fit the PCM planes: park it inside the stride */
        uint32_t worst = scan.total_samples;
        if (scan.num_blocks > scan.num_decodable) worst += blocks[scan.num_blocks - 1].nsmp;
        pcm_stride = (uint32_t)LNB_ROUNDUP((size_t)worst + 4u, 4u);
    }
    if (rq->d_pcm) pcm_stride = rq->pcm_stride;
    if ((!rq->d_stream && lnb_buf_reserve_device(dec->dev, &dec->d_stream, padded))
        || (!rq->d_pcm && lnb_buf_reserve_device(dec->dev, &dec->d_pcm, (size_t)pcm_stride * C * sizeof(int32_t)))
        || (rq->staged && lnb_buf_reserve_host(&dec->h_pcm, (size_t)pcm_stride * C * sizeof(int32_t))))
        return LINNE_APIRESULT_NG;

    /* a terminal block with a post-CRC error takes part in the CRC pass only */
    for (i = scan.num_decodable; i < scan.num_blocks; i++) blocks[i].type = 0xFFu;
    if (setup_batch(dec, &batch, blocks, scan.num_blocks, rq->d_stream ? rq->d_stream : (const uint8_t *)dec->d_stream.ptr, used,
                    rq->d_pcm ? rq->d_pcm : (int32_t *)dec->d_pcm.ptr, pcm_stride))
        return LINNE_APIRESULT_NG;

    DEC_TRACE(dec, "hopped");
    if (!rq->d_stream) {
        if (dec->turn) lnb_turnstile_wait(dec->turn, 0, dec->turn_index);
        DEC_TRACE(dec, "upload turn");
        lnb_shim_memset(dec->dev, (uint8_t *)dec->d_stream.ptr + (padded - 16u), 0, 16u);
        lnb_shim_h2d(dec->dev, dec->d_stream.ptr, rq->data, used);
    }
    lnb_shim_h2d(dec->dev, dec->d_blocks.ptr, blocks, (size_t)scan.num_blocks * sizeof(LnbBlockDesc));
    if (dec->turn && !rq->d_stream) {                            /* the next range of this device may upload while this one computes */
        const int bad = lnb_shim_sync(dec->dev);
        lnb_turnstile_pass(dec->turn, 0, dec->turn_index);
        DEC_TRACE(dec, "uploaded");
        if (bad) return LINNE_APIRESULT_NG;
    }
    if (lnb_shim_decode(dec->dev, &batch)) return LINNE_APIRESULT_NG;
    DEC_TRACE(dec, "launched");
    lnb_shim_d2h(dec->dev, blocks, dec->d_blocks.ptr, (size_t)scan.num_blocks * sizeof(LnbBlockDesc));
    if (rq->staged && scan.total_samples) {
        /* pinned planes: the samples travel with the block table, the verdict below decides what is handed on */
        dec->stage_stride = pcm_stride;
        for (c = 0; c < C; c++)
            lnb_shim_d2h(dec->dev, (int32_t *)dec->h_pcm.ptr + (size_t)c * pcm_stride,
                         (int32_t *)dec->d_pcm.ptr + (size_t)c * pcm_stride, (size_t)scan.total_samples * sizeof(int32_t));
    }
    if (lnb_shim_sync(dec->dev)) return LINNE_APIRESULT_NG;
    DEC_TRACE(dec, "kernels done");

    /* first block (stream order) whose CRC failed outranks everything after it */
    first_bad = first_crc_failure(dec, blocks, 0, scan.num_blocks);
    if (first_bad < scan.num_blocks) {
        result = LINNE_APIRESULT_DETECT_DATA_CORRUPTION;
        ok_samples = blocks[first_bad].smp_off;
    } else {
        result = hop_status(&scan);
        ok_samples = scan.total_samples;
        if (scan.num_blocks > scan.num_decodable) first_bad = scan.num_decodable;
    }
    out->first_bad = first_bad;

    /* hand back every sample the reference would have produced before stopping */
    if (!rq->d_pcm && !rq->staged) {
        int bad;
        if (dec->turn) lnb_turnstile_wait(dec->turn, 1, dec->turn_index);
        DEC_TRACE(dec, "download turn");
        for (c = 0; c < C; c++)
            lnb_shim_d2h(dec->dev, rq->buffer[c], (int32_t *)dec->d_pcm.ptr + (size_t)c * pcm_stride,
                         (size_t)ok_samples * sizeof(int32_t));
        bad = lnb_shim_sync(dec->dev);
        if (dec->turn) lnb_turnstile_pass(dec->turn, 1, dec->turn_index);
        DEC_TRACE(dec, "downloaded");
        if (bad) return LINNE_APIRESULT_NG;
    }

    out->consumed = scan.end_offset - rq->start_offset;
    out->decoded = ok_samples;
    return result;
}

/* ---- DecodeBlock: batch of one, or read-ahead (SURVEY 8f.4) ---------------------------------------------
 * A streaming caller (tools/linne_player/linne_player.c:110-121) asks for one block per call and passes all
 * that is left of its stream.  With read-ahead K the first call decodes the next K blocks in ONE batch
 * (K CTAs instead of one: the kernel is latency-bound per block, so K blocks take about as long as one) and
 * keeps their PCM in pinned host memory; the following calls are served from there.  A hit requires the
 * caller's bytes to equal the bytes that were decoded (memcmp of the whole block), so the result is the
 * function of (header, block bytes) it is in the reference, whatever the caller did in between; only
 * blocks that decoded cleanly are kept, every error takes the ordinary batch-of-one path. */
static int serve_cached_block(struct LINNEDecoder *dec, const uint8_t *data, uint32_t data_size,
                              int32_t **buffer, uint32_t buffer_num_samples, uint32_t *decode_size, uint32_t *num_decode_samples)
{
    const struct LnbCachedBlock *b;
    uint32_t c;
    if (dec->ra_next >= dec->ra_count) return 0;
    b = &dec->ra_blocks[dec->ra_next];
    if (data_size < b->byte_size || b->nsmp > buffer_num_samples
        || memcmp(data, dec->ra_image + b->byte_off, b->byte_size) != 0) {
        dec->ra_count = dec->ra_next = 0;
        return 0;
    }
    for (c = 0; c < dec->header.num_channels; c++)
        memcpy(buffer[c], (const int32_t *)dec->h_pcm.ptr + (size_t)c * dec->stage_stride + b->smp_off, (size_t)b->nsmp * sizeof(int32_t));
    *decode_size = b->byte_size;
    *num_decode_samples = b->nsmp;
    dec->ra_next++;
    return 1;
}

static void fill_block_cache(struct LINNEDecoder *dec, const uint8_t *data, uint32_t data_size)
{
    const RangeRequest rq = { .data = data, .data_size = data_size, .room = 0xFFFFFFFFu,
                              .sample_limit = LNB_READAHEAD_MAX_SAMPLES, .block_limit = dec->readahead, .staged = 1 };
    const LnbBlockDesc *blocks;
    RangeResult r;
    uint32_t i, n, span;
    dec->ra_count = dec->ra_next = 0;
    if (decode_range(dec, &rq, &r) == LINNE_APIRESULT_NG) return;
    blocks = (const LnbBlockDesc *)dec->h_blocks.ptr;
    n = (r.first_bad < r.hop.num_decodable) ? r.first_bad : r.hop.num_decodable;
    /* a block whose payload does not end where its size field says is left to the ordinary path */
    for (i = 0; i < n; i++) {
        uint32_t walked = LNB_BLOCK_HEADER_SIZE;
        if (blocks[i].type == LNB_BLOCK_COMPRESSED) walked += blocks[i].na;
        else if (blocks[i].type == LNB_BLOCK_RAW) walked += (dec->header.bits_per_sample / 8u) * blocks[i].nsmp * dec->header.num_channels;
        if (walked != blocks[i].byte_size) { n = i; break; }
    }
    if (n < 2) return;                                         /* nothing gained over a batch of one */
    span = blocks[n - 1].byte_off + blocks[n - 1].byte_size;
    if (span > dec->ra_image_cap) {
        uint8_t *p = (uint8_t *)realloc(dec->ra_image, span);
        if (!p) return;
        dec->ra_image = p; dec->ra_image_cap = span;
    }
    if (n > dec->ra_blocks_cap) {
        struct LnbCachedBlock *p = (struct LnbCachedBlock *)realloc(dec->ra_blocks, (size_t)n * sizeof(*p));
        if (!p) return;
        dec->ra_blocks = p; dec->ra_blocks_cap = n;
    }
    memcpy(dec->ra_image, data, span);
    for (i = 0; i < n; i++) {
        dec->ra_blocks[i].byte_off = blocks[i].byte_off; dec->ra_blocks[i].byte_size = blocks[i].byte_size;
        dec->ra_blocks[i].smp_off = blocks[i].smp_off; dec->ra_blocks[i].nsmp = blocks[i].nsmp;
    }
    dec->ra_count = n;
}

/* reference linne_decoder.c:564-668 */
LINNEApiResult LINNEDecoder_DecodeBlock(struct LINNEDecoder *dec, const uint8_t *data, uint32_t data_size,
        int32_t **buffer, uint32_t buffer_num_channels, uint32_t buffer_num_samples,
        uint32_t *decode_size, uint32_t *num_decode_samples)
{
    const RangeRequest rq = { .data = data, .data_size = data_size, .room = buffer_num_samples, .sample_limit = 0xFFFFFFFFu,
                              .block_limit = 1, .staged = 1 };
    RangeResult r;
    LINNEApiResult ret;
    uint32_t c;
    if (dec == NULL || data == NULL || buffer == NULL || decode_size == NULL || num_decode_samples == NULL)
        return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (!(dec->flags & DEC_FLAG_HEADER_SET)) return LINNE_APIRESULT_PARAMETER_NOT_SET;
    if (buffer_num_channels < dec->header.num_channels) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
    for (c = 0; c < dec->header.num_channels; c++) if (buffer[c] == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (data_size == 0) return LINNE_APIRESULT_INSUFFICIENT_DATA;

    if (dec->readahead > 1u) {
        if (serve_cached_block(dec, data, data_size, buffer, buffer_num_samples, decode_size, num_decode_samples))
            return LINNE_APIRESULT_OK;
        fill_block_cache(dec, data, data_size);
        if (serve_cached_block(dec, data, data_size, buffer, buffer_num_samples, decode_size, num_decode_samples))
            return LINNE_APIRESULT_OK;
        dec->ra_count = dec->ra_next = 0;
    }
    ret = decode_range(dec, &rq, &r);
    for (c = 0; r.decoded && c < dec->header.num_channels; c++)
        memcpy(buffer[c], (const int32_t *)dec->h_pcm.ptr + (size_t)c * dec->stage_stride, (size_t)r.decoded * sizeof(int32_t));
    if (ret == LINNE_APIRESULT_OK) {
        /* the bytes the payload reader walked over (linne_decoder.c:655-661) */
        const LnbBlockDesc *blk = (const LnbBlockDesc *)dec->h_blocks.ptr;
        r.consumed = LNB_BLOCK_HEADER_SIZE + blk[0].na;
    }
    *decode_size = r.consumed;
    *num_decode_samples = r.decoded;
    return ret;
}


/* ---- several GPUs behind one handle -----------------------------------------------------------------------------
 * The hop over the size fields gives the block table; contiguous block ranges go to one child handle each (own device,
 * own host thread): a range is a stream of its own for the child -- it uploads the range's bytes, decodes, and copies
 * its samples to their place in the caller's planes.  Outputs are disjoint, nothing is exchanged.  The call returns
 * the first error in stream order; samples behind a failing block may have been written by later ranges (the reference
 * leaves them untouched). */
void LINNEB200_DecoderSetDevices(struct LINNEDecoder *dec, uint32_t num_devices)
{
    if (dec == NULL) return;
    if (num_devices > LNB_MAX_DEVICES) num_devices = LNB_MAX_DEVICES;
    dec->num_devices = num_devices;
}

struct LnbDecShard {
    struct LINNEDecoder *child;
    const uint8_t *data; uint32_t data_size;
    int32_t *planes[LINNE_MAX_NUM_CHANNELS];   /* int32 planes, or ... */
    uint8_t *packed;                       /* ... interleaved packed PCM for this range */
    uint32_t room, sample_limit, block_limit;
    uint32_t first_sample;                 /* of the range, in the whole stream */
    uint32_t decoded;
    LINNEApiResult result;
    int ordinal;
};

static LINNEApiResult decode_packed_range(struct LINNEDecoder *dec, const uint8_t *data, uint32_t data_size, uint32_t start_offset,
        uint8_t *pcm, uint32_t room_frames, uint32_t sample_limit, uint32_t block_limit, uint32_t *decoded_out);

static void *dec_shard_main(void *arg)
{
    struct LnbDecShard *sh = (struct LnbDecShard *)arg;
    lnb_shim_set_device(sh->ordinal);
    sh->decoded = 0;
    if (sh->packed) sh->result = decode_packed_range(sh->child, sh->data, sh->data_size, 0, sh->packed, sh->room, sh->sample_limit, sh->block_limit, &sh->decoded);
    else {
        const RangeRequest rq = { .data = sh->data, .data_size = sh->data_size, .buffer = sh->planes, .room = sh->room,
                                  .sample_limit = sh->sample_limit, .block_limit = sh->block_limit };
        RangeResult r;
        sh->result = decode_range(sh->child, &rq, &r);
        sh->decoded = r.decoded;
    }
    if (sh->child->turn) {                                       /* whatever happened: nobody waits for this range any more */
        lnb_turnstile_pass(sh->child->turn, 0, sh->child->turn_index);
        lnb_turnstile_pass(sh->child->turn, 1, sh->child->turn_index);
        sh->child->turn = NULL;
    }
    return NULL;
}

/* DecodeWhole over dec->num_devices block ranges; returns 0 when the stream is too short to be worth it (*ret untouched) */
static int decode_whole_sharded(struct LINNEDecoder *dec, const uint8_t *data, uint32_t data_size,
                                int32_t **buffer, uint8_t *packed, uint32_t buffer_num_samples, LINNEApiResult *ret, uint32_t *decoded_total)
{
    const struct LINNEHeader *h = &dec->header;
    const int ndev = lnb_shim_device_count();
    struct LnbDecShard sh[LNB_MAX_DEVICES];
    pthread_t th[LNB_MAX_DEVICES];
    LnbTurnstile turn;
    LnbHopResult scan;
    const LnbBlockDesc *table;
    uint32_t G, k, c, started = 0, ndev_used;
    int home, ordinal[LNB_MAX_DEVICES];
    if (ndev <= 0) return 0;
    /* the handle's own block table: the children decode their ranges with tables of their own */
    if (hop_host(dec, h, data, data_size, LINNE_HEADER_SIZE, buffer_num_samples, h->num_samples, 0u, 0u, &scan)) return 0;
    table = (const LnbBlockDesc *)dec->h_blocks.ptr;
    /* ranges per requested device (pipelining), devices shared round-robin when fewer are visible than asked for */
    G = lnb_plan_ranges(scan.num_decodable, dec->num_devices > 1u ? dec->num_devices : 1u);
    if (G < 2u) return 0;                                        /* a handful of blocks: the handle's own device */
    home = lnb_shim_current_device();
    ndev_used = lnb_place_ranges(dec->num_devices, ndev, lnb_shim_device_ordinal(dec->dev), G, ordinal);
    for (k = 0; k < G; k++) {
        if (!dec->child[k]) {
            lnb_shim_set_device(ordinal[k]);
            dec->child[k] = LINNEDecoder_Create(&dec->config, NULL, 0);
            if (dec->child[k]) dec->child[k]->num_devices = 0;
        }
        if (dec->child[k]) {
            /* the kernels of an earlier range of a device go first wherever SMs free up: its download can start while the
             * later ranges still compute (without this all ranges' kernels end together and the link idles until then) */
            const uint32_t depth = (G + ndev_used - 1u) / ndev_used, place = k / ndev_used;
            dec->child[k]->rank_override = depth > 1u ? (int)(7u - (place * 7u) / (depth - 1u)) : -1;
        }
        if (!dec->child[k] || LINNEDecoder_SetHeader(dec->child[k], h) != LINNE_APIRESULT_OK) { if (home >= 0) lnb_shim_set_device(home); return 0; }
        /* ranges of one call keep each other's kernels company: the throughput kernels pay from ~1000 blocks on then
         * (include/linne_b200.h: LINNEB200_DecoderSetThroughputBlocks) */
        dec->child[k]->tput_min_blocks = (dec->tput_min_blocks > 1024u) ? 1024u : dec->tput_min_blocks;
    }
    if (home >= 0) lnb_shim_set_device(home);
    lnb_turnstile_init(&turn, dec->num_devices > 1u ? ndev_used : 1u);
    for (k = 0; k < G; k++) {
        /* contiguous ranges of the decodable blocks; the last range runs to the end of the data and meets whatever ends
         * the stream (framing error, terminal block) exactly as the single-device path does */
        const uint32_t b0 = (uint32_t)((uint64_t)scan.num_decodable * k / G), b1 = (uint32_t)((uint64_t)scan.num_decodable * (k + 1u) / G);
        const LnbBlockDesc *first = &table[b0];
        const int last = (k + 1u == G);
        const uint32_t end_byte = last ? data_size : table[b1].byte_off;
        memset(&sh[k], 0, sizeof(sh[k]));
        sh[k].child = dec->child[k];
        sh[k].data = data + first->byte_off;
        sh[k].data_size = end_byte - first->byte_off;
        for (c = 0; c < h->num_channels && buffer; c++) sh[k].planes[c] = buffer[c] + first->smp_off;
        if (packed) sh[k].packed = packed + (size_t)first->smp_off * h->num_channels * (h->bits_per_sample / 8u);
        sh[k].first_sample = first->smp_off;
        sh[k].room = buffer_num_samples - first->smp_off;
        sh[k].sample_limit = last ? h->num_samples - first->smp_off : table[b1].smp_off - first->smp_off;
        sh[k].block_limit = last ? 0u : b1 - b0;
        sh[k].ordinal = ordinal[k];
        dec->child[k]->turn = &turn; dec->child[k]->turn_index = k;
        if (pthread_create(&th[k], NULL, dec_shard_main, &sh[k]) != 0) {
            dec->child[k]->turn = NULL;
            lnb_turnstile_pass(&turn, 0, k); lnb_turnstile_pass(&turn, 1, k);
            break;
        }
        started++;
    }
    for (k = 0; k < started; k++) pthread_join(th[k], NULL);
    lnb_turnstile_destroy(&turn);
    if (started < G) { *ret = LINNE_APIRESULT_NG; return 1; }
    *ret = LINNE_APIRESULT_OK;
    if (decoded_total) *decoded_total = 0;
    for (k = 0; k < G; k++) {                                    /* first error in stream order; frames up to there count */
        if (decoded_total) *decoded_total = sh[k].first_sample + sh[k].decoded;
        if (sh[k].result != LINNE_APIRESULT_OK) { *ret = sh[k].result; break; }
    }
    return 1;
}

/* several devices, or a stream long enough to pipeline its transfers against its kernels on one */
static int worth_sharding(const struct LINNEDecoder *dec, uint32_t data_size)
{
    return dec->num_devices > 1u || data_size >= (32u << 20);
}

/* reference linne_decoder.c:671-730 */
LINNEApiResult LINNEDecoder_DecodeWhole(struct LINNEDecoder *dec, const uint8_t *data, uint32_t data_size,
        int32_t **buffer, uint32_t buffer_num_channels, uint32_t buffer_num_samples)
{
    struct LINNEHeader header;
    LINNEApiResult ret;
    RangeResult r;
    uint32_t c;
    if (dec == NULL || data == NULL || buffer == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if ((ret = LINNEDecoder_DecodeHeader(data, data_size, &header)) != LINNE_APIRESULT_OK) return ret;
    if ((ret = LINNEDecoder_SetHeader(dec, &header)) != LINNE_APIRESULT_OK) return ret;
    if (buffer_num_channels < header.num_channels || buffer_num_samples < header.num_samples)
        return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
    for (c = 0; c < header.num_channels; c++) if (buffer[c] == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (worth_sharding(dec, data_size) && decode_whole_sharded(dec, data, data_size, buffer, NULL, buffer_num_samples, &ret, NULL)) return ret;
    {
        const RangeRequest rq = { .data = data, .data_size = data_size, .start_offset = LINNE_HEADER_SIZE, .buffer = buffer,
                                  .room = buffer_num_samples, .sample_limit = header.num_samples };
        return decode_range(dec, &rq, &r);
    }
}

LnbDevice *lnb_decoder_device(const struct LINNEDecoder *dec) { return dec->dev; }

void lnb_decoder_set_tput_min_blocks(struct LINNEDecoder *dec, uint32_t blocks) { dec->tput_min_blocks = blocks; }

void lnb_decoder_set_readahead(struct LINNEDecoder *dec, uint32_t blocks)
{
    dec->readahead = (blocks > LNB_MAX_READAHEAD) ? LNB_MAX_READAHEAD : blocks;
    dec->ra_count = dec->ra_next = 0;
}

/* ---- extension entry point (include/linne_b200.h) ---- */
#include "linne_b200.h"

static LINNEApiResult decode_files(struct LINNEDecoder *dec, const uint8_t *host_image, const uint8_t *d_data, uint32_t data_size,
        struct LINNEB200FileDesc *files, uint32_t num_files, int32_t *d_pcm, uint32_t pcm_stride, uint32_t max_channels);

LINNEApiResult LINNEB200_DecodeWholeResident(struct LINNEDecoder *dec, const uint8_t *data, const uint8_t *d_data,
        uint32_t data_size, int32_t *d_pcm, uint32_t pcm_stride, uint32_t buffer_num_channels, uint32_t buffer_num_samples)
{
    struct LINNEHeader header;
    LINNEApiResult ret;
    RangeResult r;
    if (dec == NULL || d_data == NULL || d_pcm == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (data == NULL) {
        /* no host copy supplied: the hop over the size fields runs on the device (one stream of a corpus batch) */
        struct LINNEB200FileDesc one = { .num_samples = buffer_num_samples, .out_size = data_size };
        if (pcm_stride < buffer_num_samples) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
        return decode_files(dec, NULL, d_data, data_size, &one, 1, d_pcm, pcm_stride, buffer_num_channels);
    }
    if ((ret = LINNEDecoder_DecodeHeader(data, data_size, &header)) != LINNE_APIRESULT_OK) return ret;
    if ((ret = LINNEDecoder_SetHeader(dec, &header)) != LINNE_APIRESULT_OK) return ret;
    if (buffer_num_channels < header.num_channels || buffer_num_samples < header.num_samples
        || pcm_stride < buffer_num_samples) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
    {
        const RangeRequest rq = { .data = data, .data_size = data_size, .start_offset = LINNE_HEADER_SIZE,
                                  .room = buffer_num_samples, .sample_limit = header.num_samples,
                                  .d_stream = d_data, .d_pcm = d_pcm, .pcm_stride = pcm_stride };
        return decode_range(dec, &rq, &r);
    }
}

/* The hop over the streams `files` of the device image d_data, run where the image is (lnb_hop.cuh): what comes back is
 * a result record per stream (with its 30 header bytes) in *hr and the filled table slices, one after the other in
 * dec->h_blocks -- not the image.  A stream of tiny blocks overflows its slice: then the image comes to the host once
 * (dec->h_stream) for hop_host() and *hr is NULL.  Returns nonzero on a device error. */
static int hop_device(struct LINNEDecoder *dec, const uint8_t *d_data, uint32_t data_size,
                      const struct LINNEB200FileDesc *files, uint32_t num_files, const LnbHopResult **hr_out)
{
    LnbHopFile *hf;
    LnbHopResult *hr;
    uint32_t i, total_cap = 0, nb = 0;
    *hr_out = NULL;
    /* table slices: a conforming stream has one block per num_samples_per_block frames; the frames the caller gave
     * room for bound that from above for any block size >= 256 (smaller: the hop reports the overflow) */
    for (i = 0; i < num_files; i++) total_cap += files[i].num_samples / 256u + 64u;
    if (lnb_buf_reserve_host(&dec->h_hop, (size_t)num_files * (sizeof(LnbHopFile) + sizeof(LnbHopResult)))
        || lnb_buf_reserve_device(dec->dev, &dec->d_hop_files, (size_t)num_files * sizeof(LnbHopFile))
        || lnb_buf_reserve_device(dec->dev, &dec->d_hop_res, (size_t)num_files * sizeof(LnbHopResult))
        || lnb_buf_reserve_device(dec->dev, &dec->d_hop_table, (size_t)total_cap * sizeof(LnbBlockDesc))) return 1;
    hf = (LnbHopFile *)dec->h_hop.ptr;
    hr = (LnbHopResult *)(hf + num_files);
    total_cap = 0;
    for (i = 0; i < num_files; i++) {
        hf[i].offset = files[i].out_offset; hf[i].size = files[i].out_size; hf[i].room_samples = files[i].num_samples;
        hf[i].table_first = total_cap; hf[i].table_cap = files[i].num_samples / 256u + 64u;
        total_cap += hf[i].table_cap;
    }
    lnb_shim_h2d(dec->dev, dec->d_hop_files.ptr, hf, (size_t)num_files * sizeof(LnbHopFile));
    if (lnb_shim_hop(dec->dev, d_data, (const LnbHopFile *)dec->d_hop_files.ptr, num_files,
                     (LnbBlockDesc *)dec->d_hop_table.ptr, (LnbHopResult *)dec->d_hop_res.ptr)) return 1;
    lnb_shim_d2h(dec->dev, hr, dec->d_hop_res.ptr, (size_t)num_files * sizeof(LnbHopResult));
    if (lnb_shim_sync(dec->dev)) return 1;
    for (i = 0; i < num_files; i++) {
        if (hr[i].overflow) {
            if (lnb_buf_reserve_host(&dec->h_stream, (size_t)data_size + 16u)) return 1;
            lnb_shim_d2h(dec->dev, dec->h_stream.ptr, d_data, data_size);
            return lnb_shim_sync(dec->dev);
        }
        nb += hr[i].num_blocks;
    }
    /* only the slices that were filled travel */
    if (lnb_buf_reserve_host(&dec->h_blocks, (size_t)nb * sizeof(LnbBlockDesc))) return 1;
    for (i = 0, nb = 0; i < num_files; i++) {
        if (hr[i].num_blocks) lnb_shim_d2h(dec->dev, (LnbBlockDesc *)dec->h_blocks.ptr + nb, (LnbBlockDesc *)dec->d_hop_table.ptr + hf[i].table_first,
                                           (size_t)hr[i].num_blocks * sizeof(LnbBlockDesc));
        nb += hr[i].num_blocks;
    }
    if (lnb_shim_sync(dec->dev)) return 1;
    *hr_out = hr;
    return 0;
}

/* one set of stream parameters per batch */
static int same_stream_params(const struct LINNEHeader *h0, const struct LINNEHeader *h1)
{
    return h1->num_channels == h0->num_channels && h1->bits_per_sample == h0->bits_per_sample && h1->preset == h0->preset
        && h1->num_samples_per_block == h0->num_samples_per_block && h1->ch_process_method == h0->ch_process_method
        && h1->format_version == h0->format_version && h1->codec_version == h0->codec_version;
}

/* Several streams per call (corpus batches, SURVEY 8e): the streams sit one after the other in the device image
 * `d_data` (files[i].out_offset / out_size), all with the same stream parameters; the blocks of all of them go
 * through the kernels as ONE batch and every file's PCM lands at files[i].first_sample of the planes.  Without a host
 * copy of the image (`host_image`) the hop runs on the device. */
static LINNEApiResult decode_files(struct LINNEDecoder *dec, const uint8_t *host_image, const uint8_t *d_data, uint32_t data_size,
        struct LINNEB200FileDesc *files, uint32_t num_files, int32_t *d_pcm, uint32_t pcm_stride, uint32_t max_channels)
{
    struct LINNEHeader h0, h1;
    LnbDecodeBatch batch;
    LnbBlockDesc *blocks;
    const LnbHopResult *hr = NULL;
    const uint8_t *img = host_image;
    LINNEApiResult ret, overall = LINNE_APIRESULT_OK;
    uint32_t i, k, nb = 0, slice = 0;
    uint32_t *first_block;
    if (dec == NULL || d_data == NULL || files == NULL || num_files == 0 || d_pcm == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    for (i = 0; i < num_files; i++) {
        if ((uint64_t)files[i].out_offset + files[i].out_size > data_size
            || (uint64_t)files[i].first_sample + files[i].num_samples > pcm_stride) return LINNE_APIRESULT_INVALID_ARGUMENT;
        files[i].status = (int32_t)LINNE_APIRESULT_OK;
    }
    if (!(first_block = (uint32_t *)malloc(((size_t)num_files + 1u) * sizeof(uint32_t)))) return LINNE_APIRESULT_NG;
    if (!host_image) {
        if (hop_device(dec, d_data, data_size, files, num_files, &hr)) { overall = LINNE_APIRESULT_NG; goto done; }
        if (!hr) img = (const uint8_t *)dec->h_stream.ptr;
    }
    if ((overall = LINNEDecoder_DecodeHeader(hr ? hr[0].header : img + files[0].out_offset, files[0].out_size, &h0)) != LINNE_APIRESULT_OK
        || (overall = LINNEDecoder_SetHeader(dec, &h0)) != LINNE_APIRESULT_OK) goto done;
    if (max_channels && max_channels < h0.num_channels) { overall = LINNE_APIRESULT_INSUFFICIENT_BUFFER; goto done; }

    for (i = 0; i < num_files; i++) {
        LnbHopResult res;
        first_block[i] = nb;
        ret = LINNEDecoder_DecodeHeader(hr ? hr[i].header : img + files[i].out_offset, files[i].out_size, &h1);
        if (ret == LINNE_APIRESULT_OK && !same_stream_params(&h0, &h1)) ret = LINNE_APIRESULT_INVALID_FORMAT;
        if (ret == LINNE_APIRESULT_OK && files[i].num_samples < h1.num_samples) ret = LINNE_APIRESULT_INSUFFICIENT_BUFFER;
        if (hr) {                                   /* the device hop's slices lie back to back: a rejected stream's closes up */
            res = hr[i];
            slice += res.num_blocks;
            if (ret == LINNE_APIRESULT_OK && slice - res.num_blocks != nb)
                memmove((LnbBlockDesc *)dec->h_blocks.ptr + nb, (LnbBlockDesc *)dec->h_blocks.ptr + (slice - res.num_blocks),
                        (size_t)res.num_blocks * sizeof(LnbBlockDesc));
        }
        if (ret != LINNE_APIRESULT_OK) { files[i].status = (int32_t)ret; continue; }
        /* offsets relative to the image; a file's hop cannot run into its neighbour */
        if (!hr && hop_host(dec, &h1, img, files[i].out_offset + files[i].out_size, files[i].out_offset + LINNE_HEADER_SIZE,
                            files[i].num_samples, h1.num_samples, 0u, nb, &res)) { overall = LINNE_APIRESULT_NG; goto done; }
        blocks = (LnbBlockDesc *)dec->h_blocks.ptr + nb;
        for (k = 0; k < res.num_blocks; k++) blocks[k].smp_off += files[i].first_sample;
        for (k = res.num_decodable; k < res.num_blocks; k++) blocks[k].type = 0xFFu;    /* CRC pass only */
        files[i].status = (int32_t)hop_status(&res);
        nb += res.num_blocks;
    }
    first_block[num_files] = nb;

    blocks = (LnbBlockDesc *)dec->h_blocks.ptr;
    if (nb) {
        if (setup_batch(dec, &batch, blocks, nb, d_data, data_size, d_pcm, pcm_stride)) { overall = LINNE_APIRESULT_NG; goto done; }
        lnb_shim_h2d(dec->dev, dec->d_blocks.ptr, blocks, (size_t)nb * sizeof(LnbBlockDesc));
        if (lnb_shim_decode(dec->dev, &batch)) { overall = LINNE_APIRESULT_NG; goto done; }
        lnb_shim_d2h(dec->dev, blocks, dec->d_blocks.ptr, (size_t)nb * sizeof(LnbBlockDesc));
        if (lnb_shim_sync(dec->dev)) { overall = LINNE_APIRESULT_NG; goto done; }
    }
    for (i = 0; i < num_files; i++) {
        if (first_crc_failure(dec, blocks, first_block[i], first_block[i + 1u]) < first_block[i + 1u])
            files[i].status = (int32_t)LINNE_APIRESULT_DETECT_DATA_CORRUPTION;
        if (overall == LINNE_APIRESULT_OK && files[i].status != (int32_t)LINNE_APIRESULT_OK) overall = (LINNEApiResult)files[i].status;
    }
done:
    free(first_block);
    return overall;
}

LINNEApiResult LINNEB200_DecodeFilesResident(struct LINNEDecoder *dec, const uint8_t *d_data, uint32_t data_size,
        struct LINNEB200FileDesc *files, uint32_t num_files, int32_t *d_pcm, uint32_t pcm_stride)
{
    return decode_files(dec, NULL, d_data, data_size, files, num_files, d_pcm, pcm_stride, 0u);
}

/* The same for host buffers: the streams in the host image `data` (files[i].out_offset / out_size), the PCM of the
 * files back to back as packed interleaved samples in `pcm`, files[i].num_samples frames of room each
 * (first_sample is filled in: the frame offset of the file in `pcm`).  One transfer up, one batch, one down. */
LINNEApiResult LINNEB200_DecodeFilesPacked(struct LINNEDecoder *dec, const uint8_t *data, uint32_t data_size,
        struct LINNEB200FileDesc *files, uint32_t num_files, uint8_t *pcm)
{
    struct LINNEHeader h0;
    LINNEApiResult ret;
    uint64_t total = 0;
    uint32_t i, bytes, C;
    size_t stride, padded;
    if (dec == NULL || data == NULL || files == NULL || num_files == 0 || pcm == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (files[0].out_offset > data_size || files[0].out_size > data_size - files[0].out_offset) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if ((ret = LINNEDecoder_DecodeHeader(data + files[0].out_offset, files[0].out_size, &h0)) != LINNE_APIRESULT_OK) return ret;
    bytes = h0.bits_per_sample / 8u; C = h0.num_channels;
    if (bytes == 0 || bytes > 4u || (h0.bits_per_sample % 8u) != 0u || C == 0u) return LINNE_APIRESULT_INVALID_FORMAT;
    for (i = 0; i < num_files; i++) { files[i].first_sample = (uint32_t)total; total += files[i].num_samples; }
    if (total == 0 || total > 0xFFFFFFF0ull) return LINNE_APIRESULT_INVALID_ARGUMENT;
    stride = LNB_ROUNDUP((size_t)total + 4u, 4u);
    padded = LNB_ROUNDUP((size_t)data_size + 16u, 16u);
    if (lnb_buf_reserve_device(dec->dev, &dec->d_stream, padded)
        || lnb_buf_reserve_device(dec->dev, &dec->d_pcm, stride * C * sizeof(int32_t))
        || lnb_buf_reserve_device(dec->dev, &dec->d_packed, (size_t)total * C * bytes + 16u)) return LINNE_APIRESULT_NG;
    lnb_shim_memset(dec->dev, (uint8_t *)dec->d_stream.ptr + (padded - 16u), 0, 16u);
    lnb_shim_h2d(dec->dev, dec->d_stream.ptr, data, data_size);
    ret = decode_files(dec, data, (const uint8_t *)dec->d_stream.ptr, data_size, files, num_files, (int32_t *)dec->d_pcm.ptr, (uint32_t)stride, 0u);
    /* every file that decoded is handed back; a failed file's frames are undefined */
    if (lnb_shim_pack_pcm(dec->dev, (const int32_t *)dec->d_pcm.ptr, (uint8_t *)dec->d_packed.ptr, (uint32_t)stride,
                          (uint32_t)total, C, bytes)) return LINNE_APIRESULT_NG;
    lnb_shim_d2h(dec->dev, pcm, dec->d_packed.ptr, (size_t)total * C * bytes);
    if (lnb_shim_sync(dec->dev)) return LINNE_APIRESULT_NG;
    return ret;
}

/* Packed interleaved PCM out (the bytes of a WAV data chunk), converted from the planes on the device: the blocks found
 * from `start_offset` on (header already set), at most block_limit blocks (0: all) / sample_limit frames. */
static LINNEApiResult decode_packed_range(struct LINNEDecoder *dec, const uint8_t *data, uint32_t data_size, uint32_t start_offset,
        uint8_t *pcm, uint32_t room_frames, uint32_t sample_limit, uint32_t block_limit, uint32_t *decoded_out)
{
    const struct LINNEHeader *h = &dec->header;
    const uint32_t bytes = h->bits_per_sample / 8u;
    const uint32_t frames = sample_limit < room_frames ? sample_limit : room_frames;
    LINNEApiResult ret;
    uint32_t decoded = 0;
    size_t stride = LNB_ROUNDUP((size_t)frames + (size_t)h->num_samples_per_block + 65536u + 4u, 4u);   /* room for a parked terminal block */
    if (lnb_buf_reserve_device(dec->dev, &dec->d_pcm, stride * h->num_channels * sizeof(int32_t))
        || lnb_buf_reserve_device(dec->dev, &dec->d_packed, (size_t)frames * h->num_channels * bytes + 16u))
        return LINNE_APIRESULT_NG;
    {
        const RangeRequest rq = { .data = data, .data_size = data_size, .start_offset = start_offset, .room = room_frames,
                                  .sample_limit = sample_limit, .block_limit = block_limit,
                                  .d_pcm = (int32_t *)dec->d_pcm.ptr, .pcm_stride = (uint32_t)stride };
        RangeResult r;
        ret = decode_range(dec, &rq, &r);
        decoded = r.decoded;
    }
    if (decoded) {          /* every sample the reference would have produced before stopping */
        if (lnb_shim_pack_pcm(dec->dev, (const int32_t *)dec->d_pcm.ptr, (uint8_t *)dec->d_packed.ptr, (uint32_t)stride,
                              decoded, h->num_channels, bytes)) return LINNE_APIRESULT_NG;
        if (dec->turn) {                                         /* kernels done before this range takes its turn on the link */
            if (lnb_shim_sync(dec->dev)) return LINNE_APIRESULT_NG;
            lnb_turnstile_wait(dec->turn, 1, dec->turn_index);
        }
        lnb_shim_d2h(dec->dev, pcm, dec->d_packed.ptr, (size_t)decoded * h->num_channels * bytes);
        {
            const int bad = lnb_shim_sync(dec->dev);
            if (dec->turn) lnb_turnstile_pass(dec->turn, 1, dec->turn_index);
            if (bad) return LINNE_APIRESULT_NG;
        }
    }
    *decoded_out = decoded;
    return ret;
}

LINNEApiResult LINNEB200_DecodeWholePacked(struct LINNEDecoder *dec, const uint8_t *data, uint32_t data_size,
        uint8_t *pcm, uint32_t pcm_capacity_frames, uint32_t *num_frames)
{
    struct LINNEHeader header;
    LINNEApiResult ret;
    uint32_t decoded = 0, bytes;
    if (dec == NULL || data == NULL || pcm == NULL || num_frames == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    *num_frames = 0;
    if ((ret = LINNEDecoder_DecodeHeader(data, data_size, &header)) != LINNE_APIRESULT_OK) return ret;
    if ((ret = LINNEDecoder_SetHeader(dec, &header)) != LINNE_APIRESULT_OK) return ret;
    if (pcm_capacity_frames < header.num_samples) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
    bytes = header.bits_per_sample / 8u;
    if (bytes == 0 || bytes > 4u || (header.bits_per_sample % 8u) != 0u) return LINNE_APIRESULT_INVALID_FORMAT;
    if (worth_sharding(dec, data_size) && decode_whole_sharded(dec, data, data_size, NULL, pcm, header.num_samples, &ret, &decoded)) {
        *num_frames = decoded;
        return ret;
    }
    ret = decode_packed_range(dec, data, data_size, LINNE_HEADER_SIZE, pcm, header.num_samples, header.num_samples, 0, &decoded);
    *num_frames = decoded;
    return ret;
}

/* ---- seek index and sample-window decodes (include/linne_b200.h) ------------------------------------------------------
 * Every block is self-contained, so an excerpt needs only the blocks it overlaps.  BuildIndex hops once over the stream
 * and keeps (first sample, byte offset) per block; DecodeWindows finds each window's blocks by binary search in that index,
 * decodes the union of them as ONE batch into compact scratch planes and copies every window out of those planes. */
LINNEApiResult LINNEB200_DecoderBuildIndex(struct LINNEDecoder *dec, const uint8_t *data, const uint8_t *d_data,
        uint32_t data_size, struct LINNEB200SeekPoint *points, uint32_t capacity, uint32_t *num_points)
{
    struct LINNEHeader h;
    const LnbBlockDesc *table;
    const LnbHopResult *hr = NULL;
    LnbHopResult scan;
    LINNEApiResult ret;
    uint32_t i, n;
    if (dec == NULL || num_points == NULL || (data == NULL && d_data == NULL) || (points == NULL && capacity)) return LINNE_APIRESULT_INVALID_ARGUMENT;
    *num_points = 0;
    if (data == NULL) {
        /* the image is in HBM: its header comes up first (the hop's table is sized from the sample count) */
        uint8_t *hdr;
        if (data_size < LINNE_HEADER_SIZE) return LINNE_APIRESULT_INSUFFICIENT_DATA;
        if (lnb_buf_reserve_host(&dec->h_hop, 64u)) return LINNE_APIRESULT_NG;
        hdr = (uint8_t *)dec->h_hop.ptr;
        lnb_shim_d2h(dec->dev, hdr, d_data, LINNE_HEADER_SIZE);
        if (lnb_shim_sync(dec->dev)) return LINNE_APIRESULT_NG;
        if ((ret = LINNEDecoder_DecodeHeader(hdr, data_size, &h)) != LINNE_APIRESULT_OK) return ret;
    } else if ((ret = LINNEDecoder_DecodeHeader(data, data_size, &h)) != LINNE_APIRESULT_OK) {
        return ret;
    }
    if ((ret = LINNEDecoder_SetHeader(dec, &h)) != LINNE_APIRESULT_OK) return ret;

    if (data == NULL) {
        /* the device hop of one stream, as DecodeWholeResident without a host copy runs it */
        const struct LINNEB200FileDesc one = { .num_samples = h.num_samples, .out_size = data_size };
        if (hop_device(dec, d_data, data_size, &one, 1u, &hr)) return LINNE_APIRESULT_NG;
        if (hr) scan = hr[0];
        else data = (const uint8_t *)dec->h_stream.ptr;
    }
    if (!hr && hop_host(dec, &h, data, data_size, LINNE_HEADER_SIZE, h.num_samples, h.num_samples, 0u, 0u, &scan)) return LINNE_APIRESULT_NG;
    /* the blocks a DecodeWhole would decode; the result is what its hop reports for the stream's framing */
    table = (const LnbBlockDesc *)dec->h_blocks.ptr;
    n = scan.num_decodable;
    for (i = 0; i < n && i < capacity; i++) { points[i].first_sample = table[i].smp_off; points[i].byte_offset = table[i].byte_off; }
    *num_points = n;
    if (n > capacity) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
    return hop_status(&scan);
}

/* index of the block that holds sample s: the last point whose first sample is <= s */
static uint32_t find_block(const struct LINNEB200SeekPoint *points, uint32_t num_points, uint32_t s)
{
    uint32_t lo = 0, hi = num_points - 1u;
    while (lo < hi) {
        const uint32_t mid = lo + (hi - lo + 1u) / 2u;
        if (points[mid].first_sample <= s) lo = mid; else hi = mid - 1u;
    }
    return lo;
}

/* Shared by DecodeWindows (host image `data`, PCM into the caller's planes `buffer`), DecodeWindowsPacked (host image,
 * packed interleaved PCM into `packed`) and DecodeWindowsResident (device image `d_data`, PCM into the device planes
 * `d_pcm`); `out_stride` = samples per output plane, or frames of `packed`.  Host outputs are gathered densely into
 * d_packed (planes [C][dense_stride], or packed frames), come down in one piece and are copied per window. */
static LINNEApiResult decode_windows(struct LINNEDecoder *dec, const uint8_t *data, const uint8_t *d_data, uint32_t data_size,
        const struct LINNEB200SeekPoint *points, uint32_t num_points, struct LINNEB200Window *windows, uint32_t num_windows,
        int32_t **buffer, int32_t *d_pcm, uint8_t *packed, uint32_t out_stride)
{
    const struct LINNEHeader *h = &dec->header;
    const uint32_t C = h->num_channels, N = num_points, bytes = h->bits_per_sample / 8u;
    const int resident = (d_pcm != NULL);
    const size_t frame = packed ? (size_t)C * bytes : (size_t)C * sizeof(int32_t);   /* bytes per frame of the dense gather */
    LnbDecodeBatch batch;
    LnbSeekIn *seek;
    LnbGatherWin *gw;
    LnbBlockDesc *blocks;
    LINNEApiResult overall = LINNE_APIRESULT_OK;
    int32_t *mark;
    uint32_t *cpos, *err, *first_bad, *ok_block, *wk, i, k, j, c, nneed = 0, nok = 0, ngw = 0, run_start = 0, img_bytes = 0, scratch = 0, stride, dense_stride = 0;
    uint64_t items = 0, dense = 0;
    size_t win_bytes;

    /* ---- validation: nothing is written and no status is set when the request is rejected ---- */
    if (num_points == 0 || points[0].first_sample != 0u || points[0].byte_offset != LINNE_HEADER_SIZE) return LINNE_APIRESULT_INVALID_ARGUMENT;
    for (k = 0; k < N; k++) {
        if (points[k].byte_offset >= data_size || points[k].first_sample >= h->num_samples) return LINNE_APIRESULT_INVALID_ARGUMENT;
        if (k && (points[k].first_sample <= points[k - 1].first_sample || points[k].byte_offset <= points[k - 1].byte_offset))
            return LINNE_APIRESULT_INVALID_ARGUMENT;
    }
    for (i = 0; i < num_windows; i++)
        if ((uint64_t)windows[i].first_sample + windows[i].num_samples > h->num_samples
            || (uint64_t)windows[i].out_offset + windows[i].num_samples > out_stride) return LINNE_APIRESULT_INVALID_ARGUMENT;

    /* ---- planning: the blocks every window needs, marked as ranges; needed blocks in stream order, each once ---- */
    if (!(mark = (int32_t *)calloc((size_t)5u * N + 1u + 2u * (size_t)num_windows, sizeof(uint32_t)))) return LINNE_APIRESULT_NG;
    cpos = (uint32_t *)(mark + N + 1u);                 /* scratch sample offset of a needed block */
    err = cpos + N;                                     /* result of every block (OK for the ones nobody needs) */
    first_bad = err + N;                                /* the first failing block at or after a block (N: none) */
    ok_block = first_bad + N;                           /* stream index of each block of the decode batch */
    wk = ok_block + N;                                  /* first and last block of each window */
    for (i = 0; i < num_windows; i++) {
        if (windows[i].num_samples == 0u) continue;
        wk[2u * i] = find_block(points, N, windows[i].first_sample);
        wk[2u * i + 1u] = find_block(points, N, windows[i].first_sample + windows[i].num_samples - 1u);
        mark[wk[2u * i]]++;
        mark[wk[2u * i + 1u] + 1u]--;
    }
    win_bytes = LNB_ROUNDUP((size_t)N * sizeof(LnbSeekIn), 16u);
    if (lnb_buf_reserve_host(&dec->h_win, win_bytes + (size_t)num_windows * sizeof(LnbGatherWin))
        || lnb_buf_reserve_host(&dec->h_blocks, (size_t)N * sizeof(LnbBlockDesc))) { overall = LINNE_APIRESULT_NG; goto done; }
    seek = (LnbSeekIn *)dec->h_win.ptr;
    gw = (LnbGatherWin *)((uint8_t *)dec->h_win.ptr + win_bytes);
    blocks = (LnbBlockDesc *)dec->h_blocks.ptr;
    {
        int32_t depth = 0;
        uint32_t last = 0;
        for (k = 0; k < N; k++) {
            const uint32_t end_byte = (k + 1u < N) ? points[k + 1u].byte_offset : data_size;
            const uint32_t nsmp = ((k + 1u < N) ? points[k + 1u].first_sample : h->num_samples) - points[k].first_sample;
            depth += mark[k];
            if (depth <= 0) continue;
            if (nneed == 0 || last + 1u != k) {
                /* a run of adjacent blocks starts 4-aligned in the scratch planes (the throughput kernels want smp_off % 4 == 0);
                 * inside a run the blocks follow each other, so that every window is one contiguous run of the planes */
                scratch = (uint32_t)LNB_ROUNDUP(scratch, 4u);
                img_bytes = (uint32_t)LNB_ROUNDUP(img_bytes, 16u);
                run_start = points[k].byte_offset;
            }
            cpos[k] = scratch;
            /* host image: the needed blocks' bytes are staged run after run; device image: read where they are */
            seek[nneed].img_off = data ? img_bytes + (points[k].byte_offset - run_start) : points[k].byte_offset;
            seek[nneed].span = end_byte - points[k].byte_offset;
            seek[nneed].remain = data_size - points[k].byte_offset;
            seek[nneed].nsmp = nsmp;
            seek[nneed].smp_off = scratch;
            scratch += nsmp;
            if (data) img_bytes = seek[nneed].img_off + seek[nneed].span;
            last = k;
            nneed++;
        }
    }
    stride = (uint32_t)LNB_ROUNDUP((size_t)scratch + 4u, 4u);
    for (i = 0; i < num_windows; i++) {                  /* gather records (zero-length windows have none) */
        const struct LINNEB200Window *w = &windows[i];
        uint32_t dst;
        if (w->num_samples == 0u) continue;
        dense = LNB_ROUNDUP(dense, 4u);
        dst = resident ? w->out_offset : (uint32_t)dense;
        gw[ngw].src = cpos[wk[2u * i]] + (w->first_sample - points[wk[2u * i]].first_sample);
        gw[ngw].dst = dst;
        gw[ngw].len = w->num_samples;
        gw[ngw].item_first = (uint32_t)items;
        items += (uint64_t)(((dst + w->num_samples + 3u) >> 2) - (dst >> 2)) * (packed ? 1u : C);   /* packed: one item per group */
        dense += w->num_samples;
        ngw++;
    }
    dense_stride = (uint32_t)LNB_ROUNDUP(dense, 4u);
    if (items > 0xFFFFFFFFull || dense > 0xFFFFFFF0ull) { overall = LINNE_APIRESULT_NG; goto done; }   /* more than 2^32 items */

    if (nneed) {
        const uint8_t *image = d_data;
        uint32_t image_size = data_size;
        /* ---- the needed blocks' bytes: a host image uploads only those, adjacent blocks in one piece ---- */
        if (data) {
            const size_t padded = LNB_ROUNDUP((size_t)img_bytes + 16u, 16u);
            uint8_t *stage;
            if (lnb_buf_reserve_host(&dec->h_win_img, padded) || lnb_buf_reserve_device(dec->dev, &dec->d_stream, padded)) { overall = LINNE_APIRESULT_NG; goto done; }
            stage = (uint8_t *)dec->h_win_img.ptr;
            for (j = 0; j < nneed; ) {
                const uint32_t src = data_size - seek[j].remain, dst = seek[j].img_off;
                uint32_t len = seek[j].span;
                for (j++; j < nneed && seek[j].img_off == dst + len && data_size - seek[j].remain == src + len; j++) len += seek[j].span;
                memcpy(stage + dst, data + src, len);
            }
            memset(stage + img_bytes, 0, padded - img_bytes);
            lnb_shim_h2d(dec->dev, dec->d_stream.ptr, stage, padded);
            image = (const uint8_t *)dec->d_stream.ptr;
            image_size = img_bytes;
        }
        /* ---- seek: the block table, built in parallel from the index; back to the host for routing and status ---- */
        if (lnb_buf_reserve_device(dec->dev, &dec->d_win, win_bytes + (size_t)num_windows * sizeof(LnbGatherWin))
            || lnb_buf_reserve_device(dec->dev, &dec->d_blocks, (size_t)nneed * sizeof(LnbBlockDesc))
            || lnb_buf_reserve_device(dec->dev, &dec->d_pcm, (size_t)stride * C * sizeof(int32_t))
            || (!resident && ngw && lnb_buf_reserve_device(dec->dev, &dec->d_packed, (size_t)dense_stride * frame))
            || (!resident && ngw && lnb_buf_reserve_host(&dec->h_win_pcm, (size_t)dense_stride * frame))) { overall = LINNE_APIRESULT_NG; goto done; }
        lnb_shim_h2d(dec->dev, dec->d_win.ptr, dec->h_win.ptr, win_bytes + (size_t)ngw * sizeof(LnbGatherWin));
        if (lnb_shim_seek_blocks(dec->dev, image, (const LnbSeekIn *)dec->d_win.ptr, nneed, C, h->bits_per_sample, (LnbBlockDesc *)dec->d_blocks.ptr))
            { overall = LINNE_APIRESULT_NG; goto done; }
        lnb_shim_d2h(dec->dev, blocks, dec->d_blocks.ptr, (size_t)nneed * sizeof(LnbBlockDesc));
        if (lnb_shim_sync(dec->dev)) { overall = LINNE_APIRESULT_NG; goto done; }
        /* blocks whose framing failed are neither CRC-checked nor decoded: the batch holds the others */
        {
            int32_t depth = 0;
            for (k = 0, j = 0; k < N; k++) {
                depth += mark[k];
                if (depth <= 0) continue;
                err[k] = blocks[j].status;
                if (blocks[j].status == LINNE_APIRESULT_OK) { blocks[nok] = blocks[j]; blocks[nok].status = 0; ok_block[nok++] = k; }
                j++;
            }
        }
        /* ---- decode of the needed blocks into the scratch planes, then the gather of every window ---- */
        if (nok) {
            if (setup_batch(dec, &batch, blocks, nok, image, image_size, (int32_t *)dec->d_pcm.ptr, stride)) { overall = LINNE_APIRESULT_NG; goto done; }
            lnb_shim_h2d(dec->dev, dec->d_blocks.ptr, blocks, (size_t)nok * sizeof(LnbBlockDesc));
            if (lnb_shim_decode(dec->dev, &batch)) { overall = LINNE_APIRESULT_NG; goto done; }
            lnb_shim_d2h(dec->dev, blocks, dec->d_blocks.ptr, (size_t)nok * sizeof(LnbBlockDesc));
            const LnbGatherWin *d_gw = (const LnbGatherWin *)((uint8_t *)dec->d_win.ptr + win_bytes);
            if (packed ? lnb_shim_gather_windows_packed(dec->dev, (const int32_t *)dec->d_pcm.ptr, stride, d_gw, ngw, (uint32_t)items,
                                                        (uint8_t *)dec->d_packed.ptr, C, bytes)
                       : lnb_shim_gather_windows(dec->dev, (const int32_t *)dec->d_pcm.ptr, stride, d_gw, ngw, (uint32_t)items,
                                                 resident ? d_pcm : (int32_t *)dec->d_packed.ptr, resident ? out_stride : dense_stride))
                { overall = LINNE_APIRESULT_NG; goto done; }
            if (packed && ngw)
                lnb_shim_d2h(dec->dev, dec->h_win_pcm.ptr, dec->d_packed.ptr, (size_t)dense * frame);
            else if (!resident && ngw)
                for (c = 0; c < C; c++)
                    lnb_shim_d2h(dec->dev, (int32_t *)dec->h_win_pcm.ptr + (size_t)c * dense_stride,
                                 (const int32_t *)dec->d_packed.ptr + (size_t)c * dense_stride, (size_t)dense * sizeof(int32_t));
            if (lnb_shim_sync(dec->dev)) { overall = LINNE_APIRESULT_NG; goto done; }
            for (j = 0; (j = first_crc_failure(dec, blocks, j, nok)) < nok; j++) err[ok_block[j]] = LINNE_APIRESULT_DETECT_DATA_CORRUPTION;
        }
    }

    /* ---- statuses: the first failing block a window needs, in stream order; host buffers get their samples ---- */
    for (k = N; k-- > 0; ) first_bad[k] = (err[k] != LINNE_APIRESULT_OK) ? k : (k + 1u < N ? first_bad[k + 1u] : N);
    for (i = 0, j = 0; i < num_windows; i++) {
        struct LINNEB200Window *w = &windows[i];
        const uint32_t f = w->num_samples ? first_bad[wk[2u * i]] : N;
        w->status = (int32_t)((w->num_samples && f <= wk[2u * i + 1u]) ? err[f] : LINNE_APIRESULT_OK);
        if (overall == LINNE_APIRESULT_OK && w->status != (int32_t)LINNE_APIRESULT_OK) overall = (LINNEApiResult)w->status;
        if (w->num_samples == 0u) continue;
        if (packed && nok && w->status == (int32_t)LINNE_APIRESULT_OK)
            memcpy(packed + (size_t)w->out_offset * frame, (const uint8_t *)dec->h_win_pcm.ptr + (size_t)gw[j].dst * frame,
                   (size_t)w->num_samples * frame);
        else if (!resident && nok && w->status == (int32_t)LINNE_APIRESULT_OK)
            for (c = 0; c < C; c++)
                memcpy(buffer[c] + w->out_offset, (const int32_t *)dec->h_win_pcm.ptr + (size_t)c * dense_stride + gw[j].dst,
                       (size_t)w->num_samples * sizeof(int32_t));
        j++;
    }
done:
    free(mark);
    return overall;
}

LINNEApiResult LINNEB200_DecodeWindows(struct LINNEDecoder *dec, const uint8_t *data, uint32_t data_size,
        const struct LINNEB200SeekPoint *points, uint32_t num_points, struct LINNEB200Window *windows, uint32_t num_windows,
        int32_t **buffer, uint32_t buffer_num_channels, uint32_t buffer_num_samples)
{
    uint32_t c;
    if (dec == NULL || data == NULL || points == NULL || windows == NULL || buffer == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (!(dec->flags & DEC_FLAG_HEADER_SET)) return LINNE_APIRESULT_PARAMETER_NOT_SET;
    if (buffer_num_channels < dec->header.num_channels) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
    for (c = 0; c < dec->header.num_channels; c++) if (buffer[c] == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    return decode_windows(dec, data, NULL, data_size, points, num_points, windows, num_windows, buffer, NULL, NULL, buffer_num_samples);
}

LINNEApiResult LINNEB200_DecodeWindowsPacked(struct LINNEDecoder *dec, const uint8_t *data, uint32_t data_size,
        const struct LINNEB200SeekPoint *points, uint32_t num_points, struct LINNEB200Window *windows, uint32_t num_windows,
        uint8_t *pcm, uint32_t pcm_capacity_frames)
{
    uint32_t bits;
    if (dec == NULL || data == NULL || points == NULL || windows == NULL || pcm == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (!(dec->flags & DEC_FLAG_HEADER_SET)) return LINNE_APIRESULT_PARAMETER_NOT_SET;
    bits = dec->header.bits_per_sample;
    if (bits != 8u && bits != 16u && bits != 24u && bits != 32u) return LINNE_APIRESULT_INVALID_FORMAT;
    return decode_windows(dec, data, NULL, data_size, points, num_points, windows, num_windows, NULL, NULL, pcm, pcm_capacity_frames);
}

LINNEApiResult LINNEB200_DecodeWindowsResident(struct LINNEDecoder *dec, const uint8_t *d_data, uint32_t data_size,
        const struct LINNEB200SeekPoint *points, uint32_t num_points, struct LINNEB200Window *windows, uint32_t num_windows,
        int32_t *d_pcm, uint32_t pcm_stride)
{
    if (dec == NULL || d_data == NULL || points == NULL || windows == NULL || d_pcm == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (!(dec->flags & DEC_FLAG_HEADER_SET)) return LINNE_APIRESULT_PARAMETER_NOT_SET;
    return decode_windows(dec, NULL, d_data, data_size, points, num_points, windows, num_windows, NULL, d_pcm, NULL, pcm_stride);
}

/* ---- salvage decodes (include/linne_b200.h) -------------------------------------------------------------------------
 * The resynchronising scan finds every position of the image that frames as a block, one CRC pass verifies them, and one
 * serial walk over the verified blocks (sorted by offset) follows the stream's chain, steps over damage and places what it
 * can account for.  The placed blocks go through the unchanged decode pipeline as one batch, at their sample positions in
 * the intact stream. */
static int by_byte_off(const void *a, const void *b)
{
    const uint32_t x = ((const LnbBlockDesc *)a)->byte_off, y = ((const LnbBlockDesc *)b)->byte_off;
    return (x > y) - (x < y);
}

/* the offset DecodeWhole's hop goes to after the verified block *b */
static uint32_t salvage_next(const struct LINNEHeader *h, const LnbBlockDesc *b)
{
    return lnb_block_next(b->byte_off, b->type, b->byte_size - 6u, b->nsmp, h->num_channels, h->bits_per_sample);
}

/* the first of the n verified blocks (sorted) at or after byte o */
static uint32_t salvage_find(const LnbBlockDesc *v, uint32_t n, uint32_t o)
{
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        const uint32_t mid = lo + (hi - lo) / 2u;
        if (v[mid].byte_off < o) lo = mid + 1u; else hi = mid;
    }
    return lo;
}

/* the status of damage that starts at byte pos: the framing error DecodeWhole reports there, or DETECT_DATA_CORRUPTION
 * for bytes that frame as a block (a block that frames but is not verified failed its CRC or a later check) */
static int32_t salvage_status(const uint8_t *data, uint32_t data_size, uint32_t pos)
{
    uint32_t size32 = 0, err;
    if (pos >= data_size) return (int32_t)LINNE_APIRESULT_INSUFFICIENT_DATA;
    err = lnb_block_frame(data + pos, data_size - pos, &size32);
    return err != LNB_HOP_OK ? (int32_t)err : (int32_t)LINNE_APIRESULT_DETECT_DATA_CORRUPTION;
}

/* Damage in place: from pos a chain of blocks leads exactly to the confirmed block v -- damaged ones that still frame as
 * blocks of B samples (a damaged payload), verified ones between them.  Their positions then follow from pos. */
static int salvage_in_place(const struct LINNEHeader *h, const uint8_t *data, uint32_t data_size,
                            const LnbBlockDesc *v, uint32_t nv, uint32_t pos, uint32_t to)
{
    while (pos < to) {
        const uint32_t j = salvage_find(v, nv, pos);
        uint32_t size32 = 0, ns;
        if (j < nv && v[j].byte_off == pos) { pos = salvage_next(h, &v[j]); continue; }
        if (lnb_block_frame(data + pos, data_size - pos, &size32) != LNB_HOP_OK) return 0;
        if ((ns = lnb_rd_be(data + pos + 9, 2)) != h->num_samples_per_block) return 0;
        pos = lnb_block_next(pos, data[pos + 8], size32, ns, h->num_channels, h->bits_per_sample);
    }
    return pos == to;
}

/* a segment of the walk: blocks [first, first + count) of the walk's table, the samples it spans (damage in place
 * included), the offset where its chain ended, and its first sample once placed */
typedef struct { uint32_t first, count, span, end, base, placed; } SalvageSeg;

/* Shared by DecodeSalvage (planes into `buffer`) and DecodeSalvagePacked (packed PCM into `packed`); arguments checked. */
static LINNEApiResult decode_salvage(struct LINNEDecoder *dec, const uint8_t *data, uint32_t data_size, int32_t **buffer,
        uint8_t *packed, struct LINNEB200Damage *damage, uint32_t capacity, uint32_t *num_damage)
{
    const struct LINNEHeader *h = &dec->header;
    const uint32_t C = h->num_channels, N = h->num_samples, B = h->num_samples_per_block, bytes = h->bits_per_sample / 8u;
    const uint32_t nblocks = (uint32_t)(((uint64_t)N + B - 1u) / B), T = N ? N - B * (nblocks - 1u) : 0u;
    const uint32_t start = data_size < LINNE_HEADER_SIZE ? data_size : (uint32_t)LINNE_HEADER_SIZE;
    const size_t padded = LNB_ROUNDUP((size_t)data_size + 16u, 16u), stride = LNB_ROUNDUP((size_t)N + 4u, 4u);
    LINNEApiResult overall = LINNE_APIRESULT_NG;
    LnbDecodeBatch batch;
    LnbBlockDesc *v, *w;
    SalvageSeg *seg = NULL;
    struct LINNEB200Damage *rec = NULL;
    uint32_t *next_conf = NULL, cap = nblocks + nblocks / 8u + 64u, count, nv = 0, nw = 0, nseg = 1, nrec = 0, np = 0, i, k, c;
    uint32_t pos, s, prev_s, prev_byte;

    *num_damage = 0;
    if (N == 0) return LINNE_APIRESULT_OK;
    /* ---- the whole image up; scan and CRC pass; the candidates come back in one piece (grown and run again if they
     * did not fit) ---- */
    if (lnb_buf_reserve_device(dec->dev, &dec->d_stream, padded)
        || lnb_buf_reserve_device(dec->dev, &dec->d_pcm, stride * C * sizeof(int32_t))
        || (packed && lnb_buf_reserve_device(dec->dev, &dec->d_packed, (size_t)N * C * bytes + 16u))) return LINNE_APIRESULT_NG;
    lnb_shim_memset(dec->dev, (uint8_t *)dec->d_stream.ptr + (padded - 16u), 0, 16u);
    lnb_shim_h2d(dec->dev, dec->d_stream.ptr, data, data_size);
    for (;;) {
        const size_t table_bytes = 16u + (size_t)cap * sizeof(LnbBlockDesc);     /* the counter, then the table */
        LnbBlockDesc *d_table;
        if (lnb_buf_reserve_device(dec->dev, &dec->d_hop_table, table_bytes) || lnb_buf_reserve_host(&dec->h_hop, table_bytes))
            return LINNE_APIRESULT_NG;
        d_table = (LnbBlockDesc *)((uint8_t *)dec->d_hop_table.ptr + 16);
        lnb_shim_memset(dec->dev, dec->d_hop_table.ptr, 0, sizeof(uint32_t));
        if (lnb_shim_resync_scan(dec->dev, (const uint8_t *)dec->d_stream.ptr, data_size, C, h->bits_per_sample, B,
                                 d_table, (uint32_t *)dec->d_hop_table.ptr, cap)
            || lnb_shim_crc_blocks(dec->dev, (const uint8_t *)dec->d_stream.ptr, data_size, d_table,
                                   (const uint32_t *)dec->d_hop_table.ptr, cap)) return LINNE_APIRESULT_NG;
        lnb_shim_d2h(dec->dev, dec->h_hop.ptr, dec->d_hop_table.ptr, table_bytes);
        if (lnb_shim_sync(dec->dev)) return LINNE_APIRESULT_NG;
        count = *(const uint32_t *)dec->h_hop.ptr;
        if (count <= cap) break;
        cap = count + count / 8u + 64u;
    }

    /* ---- the verified blocks by offset; which are confirmed; the first confirmed one at or after each ---- */
    v = (LnbBlockDesc *)((uint8_t *)dec->h_hop.ptr + 16);
    for (i = 0; i < count; i++) if (!(v[i].status & LNB_ST_CRC_MISMATCH)) v[nv++] = v[i];
    qsort(v, nv, sizeof(LnbBlockDesc), by_byte_off);
    if (lnb_buf_reserve_host(&dec->h_blocks, ((size_t)nv + 1u) * sizeof(LnbBlockDesc))
        || !(next_conf = (uint32_t *)malloc(((size_t)nv + 1u) * sizeof(uint32_t)))
        || !(seg = (SalvageSeg *)calloc((size_t)nv + 2u, sizeof(SalvageSeg)))
        || !(rec = (struct LINNEB200Damage *)malloc(((size_t)nv + 2u) * sizeof(struct LINNEB200Damage)))) goto done;
    w = (LnbBlockDesc *)dec->h_blocks.ptr;
    next_conf[nv] = nv;
    for (k = nv; k-- > 0; ) {
        const uint32_t succ = salvage_next(h, &v[k]), j = salvage_find(v, nv, succ);
        next_conf[k] = (succ == data_size || (j < nv && v[j].byte_off == succ)) ? k : next_conf[k + 1u];
    }

    /* ---- the walk ---- */
    pos = LINNE_HEADER_SIZE; s = 0;
    seg[0].end = start;
    while (pos < data_size) {
        SalvageSeg *g = &seg[nseg - 1u];
        const uint32_t j = salvage_find(v, nv, pos);
        if (nseg == 1u && s >= N) break;
        if (j < nv && v[j].byte_off == pos) {
            if (nseg == 1u && v[j].nsmp > N - s) break;            /* it would run past the stream's samples */
            w[nw] = v[j];
            w[nw].smp_off = s;
            w[nw].status = 0;
            nw++; g->count++;
            s += v[j].nsmp;
            pos = salvage_next(h, &v[j]);
            g->span = s; g->end = pos;
            continue;
        }
        {
            const uint32_t nc = next_conf[j];
            if (nc < nv && salvage_in_place(h, data, data_size, v, nv, pos, v[nc].byte_off)) {
                uint32_t size32 = 0;                                /* the damaged block: B samples of silence */
                lnb_block_frame(data + pos, data_size - pos, &size32);
                s += B;
                pos = lnb_block_next(pos, data[pos + 8], size32, B, C, h->bits_per_sample);
                g->span = s; g->end = pos;
                continue;
            }
            if (nc == nv) break;                                    /* the damage runs to the end of the image */
            seg[nseg].first = nw;
            seg[nseg].end = pos = v[nc].byte_off;
            nseg++;
            s = 0;
        }
    }

    /* ---- placing: the first segment as walked; the last one from the end; those between only when every framing gap
     * cost exactly one block ---- */
    seg[0].placed = 1;
    if (nseg >= 2u) {
        SalvageSeg *L = &seg[nseg - 1u];
        uint64_t middle = 0;
        for (k = 1; k + 1u < nseg; k++) middle += seg[k].span;
        if (L->count && L->end == data_size && w[L->first + L->count - 1u].nsmp == T && L->span <= N - seg[0].span) {
            L->base = N - L->span;
            L->placed = 1;
            if (nseg > 2u && (uint64_t)L->base - seg[0].span == middle + (uint64_t)B * (nseg - 1u)) {
                uint32_t b = seg[0].span;
                for (k = 1; k + 1u < nseg; k++) { seg[k].base = b + B; seg[k].placed = 1; b = seg[k].base + seg[k].span; }
            }
        }
    }
    for (k = 0; k < nseg; k++) {                                    /* the placed blocks, in stream order, compacted */
        if (!seg[k].placed) continue;
        for (i = seg[k].first; i < seg[k].first + seg[k].count; i++) { w[np] = w[i]; w[np].smp_off += seg[k].base; np++; }
    }

    /* ---- the report: every run of samples no placed block writes ---- */
    prev_s = 0; prev_byte = start;
    for (i = 0; i <= np; i++) {
        const uint32_t at_s = i < np ? w[i].smp_off : N, at_byte = i < np ? w[i].byte_off : data_size;
        if (at_s > prev_s || (i < np && at_byte > prev_byte)) {
            struct LINNEB200Damage *r = &rec[nrec++];
            r->first_sample = prev_s; r->num_samples = at_s - prev_s;
            r->byte_offset = prev_byte; r->byte_size = at_byte - prev_byte;
            r->status = salvage_status(data, data_size, prev_byte);
        }
        if (i < np) { prev_s = w[i].smp_off + w[i].nsmp; prev_byte = salvage_next(h, &w[i]); }
    }

    /* ---- the decode: silence where nothing is placed, the placed blocks as one batch ---- */
    if (nrec) lnb_shim_memset(dec->dev, dec->d_pcm.ptr, 0, stride * C * sizeof(int32_t));
    if (np) {
        if (setup_batch(dec, &batch, w, np, (const uint8_t *)dec->d_stream.ptr, data_size, (int32_t *)dec->d_pcm.ptr, (uint32_t)stride)) goto done;
        lnb_shim_h2d(dec->dev, dec->d_blocks.ptr, w, (size_t)np * sizeof(LnbBlockDesc));
        if (lnb_shim_decode(dec->dev, &batch)) goto done;
    }
    if (packed) {
        if (lnb_shim_pack_pcm(dec->dev, (const int32_t *)dec->d_pcm.ptr, (uint8_t *)dec->d_packed.ptr, (uint32_t)stride, N, C, bytes)) goto done;
        lnb_shim_d2h(dec->dev, packed, dec->d_packed.ptr, (size_t)N * C * bytes);
    } else {
        for (c = 0; c < C; c++) lnb_shim_d2h(dec->dev, buffer[c], (const int32_t *)dec->d_pcm.ptr + (size_t)c * stride, (size_t)N * sizeof(int32_t));
    }
    if (lnb_shim_sync(dec->dev)) goto done;
    for (i = 0; i < nrec && i < capacity; i++) damage[i] = rec[i];
    *num_damage = nrec;
    overall = nrec ? LINNE_APIRESULT_DETECT_DATA_CORRUPTION : LINNE_APIRESULT_OK;
done:
    free(next_conf);
    free(seg);
    free(rec);
    return overall;
}

LINNEApiResult LINNEB200_DecodeSalvage(struct LINNEDecoder *dec, const uint8_t *data, uint32_t data_size,
        int32_t **buffer, uint32_t buffer_num_channels, uint32_t buffer_num_samples,
        struct LINNEB200Damage *damage, uint32_t capacity, uint32_t *num_damage)
{
    uint32_t c;
    if (dec == NULL || data == NULL || buffer == NULL || num_damage == NULL || (damage == NULL && capacity)) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (!(dec->flags & DEC_FLAG_HEADER_SET)) return LINNE_APIRESULT_PARAMETER_NOT_SET;
    if (buffer_num_channels < dec->header.num_channels || buffer_num_samples < dec->header.num_samples) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
    for (c = 0; c < dec->header.num_channels; c++) if (buffer[c] == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    return decode_salvage(dec, data, data_size, buffer, NULL, damage, capacity, num_damage);
}

LINNEApiResult LINNEB200_DecodeSalvagePacked(struct LINNEDecoder *dec, const uint8_t *data, uint32_t data_size,
        uint8_t *pcm, uint32_t pcm_capacity_frames,
        struct LINNEB200Damage *damage, uint32_t capacity, uint32_t *num_damage)
{
    uint32_t bits;
    if (dec == NULL || data == NULL || pcm == NULL || num_damage == NULL || (damage == NULL && capacity)) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (!(dec->flags & DEC_FLAG_HEADER_SET)) return LINNE_APIRESULT_PARAMETER_NOT_SET;
    if (pcm_capacity_frames < dec->header.num_samples) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
    bits = dec->header.bits_per_sample;
    if (bits != 8u && bits != 16u && bits != 24u && bits != 32u) return LINNE_APIRESULT_INVALID_FORMAT;
    return decode_salvage(dec, data, data_size, NULL, pcm, damage, capacity, num_damage);
}
