/* linne_encoder_host.c -- LINNEEncoder_* entry points (include/linne_encoder.h) on top of the CUDA shim.
 *
 * Replaces reference libs/linne_encoder/src/linne_encoder.c.  Host side: argument / parameter
 * validation, the 30-byte header, cutting the stream into blocks, chunking the batch so the
 * analysis scratch fits, and copying the packed chunk back.  All signal processing, analysis,
 * coding and bit packing of every block x channel runs on the GPU.
 */
#define _POSIX_C_SOURCE 200112L
#include "linne_encoder.h"
#include "linne_b200.h"
#include "lnb_host_util.h"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <pthread.h>

/* LINNE_B200_TRACE=1: host-side time stamps of the encode call's phases on stderr (debugging aid) */
static int trace_on(void) { static int on = -1; if (on < 0) { const char *e = getenv("LINNE_B200_TRACE"); on = (e && *e == '1') ? 1 : 0; } return on; }
static double now_ms(void) { struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; }
#define TRACE(enc, what) do { if (trace_on()) fprintf(stderr, "[trace] m%u %-14s %.3f\n", (unsigned)(enc)->header.preset, what, now_ms()); } while (0)

struct LnbFileRange { uint32_t first_sample, num_samples, first_block, num_blocks; };

struct LINNEEncoder {
    struct LINNEHeader header;
    uint32_t max_num_channels, max_num_samples_per_block, max_num_layers, max_num_parameters_per_layer;
    uint8_t set_parameter, enable_learning, num_afmethod_iterations, own_work;
    void *work;
    LnbDevice *dev;
    size_t scratch_budget;                 /* bytes of analysis scratch per chunk */
    LnbBuf d_pcm, d_blocks, d_params, d_est, d_work, d_sig_a, d_sig_b, d_acorr, d_cand, d_unit_loss,
           d_chosen_w, d_chosen_u, d_final_sum, d_welch, d_plans, d_plan_mean, d_out, d_total, d_train, d_refine, d_packed, d_sinwin, d_image;
    LnbBuf h_blocks, h_welch, h_total;
    uint32_t sinwin_n;                     /* block length d_sinwin was tabulated for (0 = none) */
    LnbBuf h_headers;                      /* pinned 32-byte slots for the stream headers of a corpus batch */
    /* several GPUs behind ONE handle (SURVEY 8e, north star): EncodeWhole splits its blocks into contiguous ranges, one
     * child handle (own device, own host thread) per range */
    uint32_t num_devices;                  /* 0/1: this handle's device only */
    struct LINNEEncoder *child[LNB_MAX_DEVICES];
    LnbBuf d_shard;                        /* a child's shard of the stream, on its device */
    struct LINNEEncoderConfig config;      /* to create the children with ... */
    struct LINNEEncodeParameter param;     /* ... and the parameters they encode with (the last ones set) */
};

/* reference linne_encoder.c:53-138 */
LINNEApiResult LINNEEncoder_EncodeHeader(const struct LINNEHeader *header, uint8_t *data, uint32_t data_size)
{
    LINNEApiResult r;
    if (header == NULL || data == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (data_size < LINNE_HEADER_SIZE) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
    if ((r = lnb_header_check_for_encode(header)) != LINNE_APIRESULT_OK) return r;
    lnb_header_write(header, data);
    return LINNE_APIRESULT_OK;
}

static int config_ok(const struct LINNEEncoderConfig *c)
{
    return c && c->max_num_samples_per_block && c->max_num_channels && c->max_num_layers
        && c->max_num_parameters_per_layer && c->max_num_parameters_per_layer <= c->max_num_samples_per_block;
}

/* reference linne_encoder.c:201-265 */
int32_t LINNEEncoder_CalculateWorkSize(const struct LINNEEncoderConfig *config)
{
    if (!config_ok(config)) return -1;
    return (int32_t)(sizeof(struct LINNEEncoder) + LNB_ALIGNMENT);
}

/* reference linne_encoder.c:268-396 */
struct LINNEEncoder *LINNEEncoder_Create(const struct LINNEEncoderConfig *config, void *work, int32_t work_size)
{
    struct LINNEEncoder *enc;
    int own = 0;
    const char *budget;
    if (work == NULL && work_size == 0) {
        if ((work_size = LINNEEncoder_CalculateWorkSize(config)) < 0) return NULL;
        work = malloc((size_t)work_size);
        own = 1;
    }
    if (!config_ok(config) || work == NULL || work_size < LINNEEncoder_CalculateWorkSize(config)) {
        if (own) free(work);
        return NULL;
    }
    enc = (struct LINNEEncoder *)LNB_ROUNDUP((uintptr_t)work, LNB_ALIGNMENT);
    memset(enc, 0, sizeof(*enc));
    enc->work = work;
    enc->own_work = (uint8_t)own;
    enc->max_num_channels = config->max_num_channels;
    enc->max_num_samples_per_block = config->max_num_samples_per_block;
    enc->max_num_layers = config->max_num_layers;
    enc->max_num_parameters_per_layer = config->max_num_parameters_per_layer;
    enc->config = *config;
    enc->scratch_budget = (size_t)8 << 30;
    if ((budget = getenv("LINNE_B200_SCRATCH_MB")) != NULL && atol(budget) > 0) enc->scratch_budget = (size_t)atol(budget) << 20;
    if (lnb_shim_open(&enc->dev, -1) != 0) {
        fprintf(stderr, "linne_b200: no usable CUDA device -- the encoder has no CPU fallback\n");
        if (own) free(work);
        return NULL;
    }
    {   /* LINNE_B200_GPUS=N (or "all"): the whole-stream calls of this handle shard their blocks over N devices */
        const char *e = getenv("LINNE_B200_GPUS");
        if (e && *e) LINNEB200_EncoderSetDevices(enc, (e[0] == 'a') ? (uint32_t)lnb_shim_device_count() : (uint32_t)strtoul(e, NULL, 10));
    }
    return enc;
}

/* reference linne_encoder.c:399-407 */
void LINNEEncoder_Destroy(struct LINNEEncoder *enc)
{
    uint32_t k;
    if (enc == NULL) return;
    for (k = 0; k < LNB_MAX_DEVICES; k++) if (enc->child[k]) { LINNEEncoder_Destroy(enc->child[k]); enc->child[k] = NULL; }
    if (enc->dev) {
        LnbBuf *dbufs[] = { &enc->d_pcm, &enc->d_blocks, &enc->d_params, &enc->d_est, &enc->d_work, &enc->d_sig_a,
                            &enc->d_sig_b, &enc->d_acorr, &enc->d_cand, &enc->d_unit_loss, &enc->d_chosen_w,
                            &enc->d_chosen_u, &enc->d_final_sum, &enc->d_welch, &enc->d_plans, &enc->d_plan_mean,
                            &enc->d_out, &enc->d_total, &enc->d_train, &enc->d_refine, &enc->d_packed, &enc->d_sinwin, &enc->d_image, &enc->d_shard };
        size_t i;
        for (i = 0; i < sizeof(dbufs) / sizeof(dbufs[0]); i++) lnb_buf_release_device(enc->dev, dbufs[i]);
        lnb_buf_release_host(&enc->h_blocks);
        lnb_buf_release_host(&enc->h_welch);
        lnb_buf_release_host(&enc->h_total);
        lnb_buf_release_host(&enc->h_headers);
        lnb_shim_close(enc->dev);
        enc->dev = NULL;
    }
    if (enc->own_work) free(enc->work);
}

/* reference linne_encoder.c:141-198 (validation) and :410-477 */
LINNEApiResult LINNEEncoder_SetEncodeParameter(struct LINNEEncoder *enc, const struct LINNEEncodeParameter *prm)
{
    const LnbPreset *ps;
    int l;
    if (enc == NULL || prm == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (prm->num_channels == 0 || prm->bits_per_sample == 0 || prm->bits_per_sample > LNB_MAX_BITS_PER_SAMPLE
        || prm->sampling_rate == 0 || prm->num_samples_per_block == 0 || prm->preset >= LINNE_NUM_PARAMETER_PRESETS
        || (unsigned)prm->ch_process_method >= (unsigned)LINNE_CH_PROCESS_METHOD_INVALID)
        return LINNE_APIRESULT_INVALID_FORMAT;
    ps = &g_lnb_presets[prm->preset];
    for (l = 0; l < ps->num_layers; l++)
        if (prm->num_samples_per_block <= (uint32_t)ps->layer_params[l]) return LINNE_APIRESULT_INVALID_FORMAT;
    if (enc->max_num_samples_per_block < prm->num_samples_per_block || enc->max_num_channels < prm->num_channels)
        return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
    if (enc->max_num_layers < (uint32_t)ps->num_layers) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
    for (l = 0; l < ps->num_layers; l++)
        if (enc->max_num_parameters_per_layer < (uint32_t)ps->layer_params[l]) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
    if (prm->num_channels > LINNE_MAX_NUM_CHANNELS) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;

    memset(&enc->header, 0, sizeof(enc->header));
    enc->header.format_version = LINNE_FORMAT_VERSION;
    enc->header.codec_version = LINNE_CODEC_VERSION;
    enc->header.num_channels = prm->num_channels;
    enc->header.sampling_rate = prm->sampling_rate;
    enc->header.bits_per_sample = prm->bits_per_sample;
    enc->header.num_samples_per_block = prm->num_samples_per_block;
    enc->header.preset = prm->preset;
    enc->header.ch_process_method = prm->ch_process_method;
    enc->enable_learning = prm->enable_learning;
    enc->num_afmethod_iterations = prm->num_afmethod_iterations;
    enc->set_parameter = 1;
    enc->param = *prm;
    /* scheduling hint: analysis cost grows with layers x regularisers, i.e. with the preset number */
    lnb_shim_set_cost_rank(enc->dev, (int)prm->preset);
    return LINNE_APIRESULT_OK;
}

/* samples the analysis looks at: reference linne_encoder.c:644-655 */
static uint32_t analysis_length(const LnbStreamCfg *cfg, uint32_t n)
{
    uint32_t maxp = 0, na, l;
    for (l = 0; l < cfg->num_layers; l++) if (maxp < cfg->layer_params[l]) maxp = cfg->layer_params[l];
    na = LNB_ROUNDUP(n, 8u);
    if (na < maxp) na = maxp;
    if (na > cfg->block_size) na = cfg->block_size;
    return na;
}

/* blocks of num_samples samples, cut every header.num_samples_per_block samples (the last one may be shorter) */
static uint64_t num_blocks(const struct LINNEHeader *h, uint64_t num_samples)
{
    return (num_samples + h->num_samples_per_block - 1u) / h->num_samples_per_block;
}

/* Room to give the stream of n samples (header and blocks) where it is staged before its size is known: twice its PCM
 * bytes, 16 bytes per block and 4 KiB.  Its all-raw size (reference linne_encoder.c:556-585) is no bound: the block
 * type comes from an estimate (lnb_encode_core.cuh), so a compressed block can come out longer than raw.  A stream
 * that needs more than this room fails with INSUFFICIENT_BUFFER. */
static uint64_t stream_room(const struct LINNEHeader *h, uint64_t n)
{
    const uint64_t pcm_bytes = n * h->num_channels * ((h->bits_per_sample + 7u) / 8u);
    return LINNE_HEADER_SIZE + 2u * (pcm_bytes + 16u * (n / h->num_samples_per_block + 2u)) + 4096u;
}

/* Output of encode_blocks(): the blocks of one stream into a host or a device buffer, or (corpus batch) the streams of
 * several files, header + blocks each, one after the other into a device buffer. */
typedef enum { ENC_OUT_HOST, ENC_OUT_DEVICE, ENC_OUT_FILES } EncOutput;

/* One call of encode_blocks(): PCM in device planes [C][pcm_stride]; one stream of num_samples samples from sample 0
 * on, or the files `ranges` with their result table `files`.  `forced` (optional, host memory, [blocks * C]) supplies
 * unit counts / shifts / coefficients and skips the analysis.  Output goes to out[first_byte, out_size): a whole-stream
 * call has written its header in front. */
typedef struct {
    const int32_t *pcm;
    uint32_t pcm_stride, num_samples;
    const struct LnbFileRange *ranges;
    uint32_t num_ranges;
    struct LINNEB200FileDesc *files;
    const LnbChanParams *forced;
    uint8_t *out;
    uint32_t first_byte, out_size;
    EncOutput mode;
} EncodeRequest;

/* reserves enc->d_pcm for n samples and points rq at it: 4 spare samples per plane, stride a multiple of 4 */
static int reserve_planes(struct LINNEEncoder *enc, uint32_t n, EncodeRequest *rq)
{
    rq->pcm_stride = (uint32_t)LNB_ROUNDUP((size_t)n + 4u, 4u);
    rq->num_samples = n;
    if (lnb_buf_reserve_device(enc->dev, &enc->d_pcm, (size_t)rq->pcm_stride * enc->header.num_channels * sizeof(int32_t))) return 1;
    rq->pcm = (const int32_t *)enc->d_pcm.ptr;
    return 0;
}

/* packed PCM holds whole bytes per sample, at most 4 */
static int packed_bits_ok(const struct LINNEHeader *h)
{
    return h->bits_per_sample % 8u == 0u && h->bits_per_sample >= 8u && h->bits_per_sample <= 32u;
}

/* samples [first, first + n) of the caller's int32 planes into enc->d_pcm, the PCM of rq */
static LINNEApiResult upload_planes(struct LINNEEncoder *enc, const int32_t *const *input, uint32_t first, uint32_t n, EncodeRequest *rq)
{
    uint32_t c;
    for (c = 0; c < enc->header.num_channels; c++) if (input[c] == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (reserve_planes(enc, n, rq)) return LINNE_APIRESULT_NG;
    for (c = 0; c < enc->header.num_channels; c++)
        lnb_shim_h2d(enc->dev, (int32_t *)enc->d_pcm.ptr + (size_t)c * rq->pcm_stride, input[c] + first, (size_t)n * sizeof(int32_t));
    return LINNE_APIRESULT_OK;
}

/* frames [first, first + n) of packed interleaved PCM (WAV data-chunk layout) into enc->d_pcm, converted on the device */
static LINNEApiResult upload_packed(struct LINNEEncoder *enc, const uint8_t *pcm, uint32_t first, uint32_t n, EncodeRequest *rq)
{
    const uint32_t C = enc->header.num_channels, bytes = enc->header.bits_per_sample / 8u;
    const size_t frame = (size_t)C * bytes;
    if (reserve_planes(enc, n, rq) || lnb_buf_reserve_device(enc->dev, &enc->d_packed, (size_t)n * frame + 16u)) return LINNE_APIRESULT_NG;
    lnb_shim_h2d(enc->dev, enc->d_packed.ptr, pcm + (size_t)first * frame, (size_t)n * frame);
    if (lnb_shim_unpack_pcm(enc->dev, (const uint8_t *)enc->d_packed.ptr, (int32_t *)enc->d_pcm.ptr, rq->pcm_stride, n, C, bytes))
        return LINNE_APIRESULT_NG;
    return LINNE_APIRESULT_OK;
}

/* Reserves the analysis scratch of a chunk and points `batch` at it.  Returns the chunk size in blocks (0: no memory).
 * Chunks keep the per-chunk scratch inside the budget.  Blocks of up to lnb_shim_fast_max_na() samples are analysed by
 * the cooperative kernel (signal in shared memory): they need only the integer work signal and the per-slot results.
 * Longer blocks take the flat kernels, which keep two double-precision planes and per-level tables in HBM. */
static uint32_t reserve_scratch(struct LINNEEncoder *enc, LnbEncodeBatch *batch, uint32_t total_blocks, int forced)
{
    const struct LINNEHeader *h = &enc->header;
    const uint32_t C = h->num_channels, NB = h->num_samples_per_block, slots_per_block = C * batch->cfg.num_lambdas;
    const int need_flat = NB > lnb_shim_fast_max_na();
    const int need_sig_a = need_flat || (enc->num_afmethod_iterations && !forced);    /* IRLS scratch: one plane per slot */
    /* IRLS / SGD on blocks too long for the refinement kernel's shared memory: its two signal buffers in HBM (lnb_shim.h) */
    const int refine_global = !forced && (enc->enable_learning || enc->num_afmethod_iterations)
                              && lnb_shim_refine_max_na() && NB > lnb_shim_refine_max_na();
    const size_t ws = batch->cfg.work_stride, chunks = (ws + 63u) / 64u;
    size_t per_block, refine_doubles = 0, S, BC;
    uint32_t chunk_blocks;
    per_block = (size_t)slots_per_block * (LNB_MAX_LAYERS * LNB_MAX_PARAMS * sizeof(double) + chunks * sizeof(double) + 64u)
              + (size_t)C * (ws * sizeof(int32_t) + sizeof(LnbChanParams) + sizeof(LnbCoderPlan)
                             + 2u * LNB_MAX_PARTITIONS * sizeof(double) + 64u)
              + (enc->enable_learning ? (size_t)C * (2u * LNB_MAX_LAYERS + 1u) * ws * sizeof(double) : 0u);
    if (refine_global) {
        size_t na_max = NB;
        int l;
        for (l = 0; l < g_lnb_presets[h->preset].num_layers; l++) {
            const size_t P = (size_t)g_lnb_presets[h->preset].layer_params[l], tri = P * (P + 1u) / 2u;
            if (enc->num_afmethod_iterations && na_max < tri) na_max = tri;
        }
        na_max = (na_max + 7u) & ~(size_t)7u;
        refine_doubles = 2u * (na_max + lnb_shim_refine_hist());
        per_block += (size_t)C * refine_doubles * sizeof(double);
    }
    if (need_sig_a && !need_flat) per_block += (size_t)slots_per_block * ws * sizeof(double);
    if (need_flat)
        per_block += (size_t)slots_per_block * (ws * sizeof(double) * 2u
                                                + LNB_MAX_LEVELS * (256u + LNB_MAX_PARAMS + chunks) * sizeof(double));
    chunk_blocks = (uint32_t)(enc->scratch_budget / per_block);
    if (chunk_blocks < 1u) chunk_blocks = 1u;
    if (chunk_blocks > total_blocks) chunk_blocks = total_blocks;
    while ((uint64_t)chunk_blocks * slots_per_block * ws >= 0x7FFFFFFFull && chunk_blocks > 1u) chunk_blocks /= 2u;
    S = (size_t)chunk_blocks * slots_per_block;
    BC = (size_t)chunk_blocks * C;
    if (lnb_buf_reserve_host(&enc->h_blocks, 2u * (size_t)chunk_blocks * sizeof(LnbBlockDesc))
        || lnb_buf_reserve_host(&enc->h_welch, (size_t)chunk_blocks * LNB_MAX_LEVELS * sizeof(double))
        || lnb_buf_reserve_host(&enc->h_total, 64)
        || lnb_buf_reserve_device(enc->dev, &enc->d_blocks, chunk_blocks * sizeof(LnbBlockDesc))
        || lnb_buf_reserve_device(enc->dev, &enc->d_params, BC * sizeof(LnbChanParams))
        || lnb_buf_reserve_device(enc->dev, &enc->d_est, BC * sizeof(double))
        || lnb_buf_reserve_device(enc->dev, &enc->d_work, BC * ws * sizeof(int32_t))
        || (need_sig_a && lnb_buf_reserve_device(enc->dev, &enc->d_sig_a, S * ws * sizeof(double)))
        || (need_flat
            && (lnb_buf_reserve_device(enc->dev, &enc->d_sig_b, S * ws * sizeof(double))
                || lnb_buf_reserve_device(enc->dev, &enc->d_acorr, S * LNB_MAX_LEVELS * 256u * sizeof(double))
                || lnb_buf_reserve_device(enc->dev, &enc->d_cand, S * LNB_MAX_LEVELS * LNB_MAX_PARAMS * sizeof(double))
                || lnb_buf_reserve_device(enc->dev, &enc->d_unit_loss, S * LNB_MAX_LEVELS * chunks * sizeof(double))))
        || lnb_buf_reserve_device(enc->dev, &enc->d_chosen_w, S * LNB_MAX_LAYERS * LNB_MAX_PARAMS * sizeof(double))
        || lnb_buf_reserve_device(enc->dev, &enc->d_chosen_u, S * LNB_MAX_LAYERS)
        || lnb_buf_reserve_device(enc->dev, &enc->d_final_sum, S * chunks * sizeof(double))
        || lnb_buf_reserve_device(enc->dev, &enc->d_welch, (size_t)chunk_blocks * LNB_MAX_LEVELS * sizeof(double))
        || lnb_buf_reserve_device(enc->dev, &enc->d_plans, BC * sizeof(LnbCoderPlan))
        || lnb_buf_reserve_device(enc->dev, &enc->d_plan_mean, BC * 2u * LNB_MAX_PARTITIONS * sizeof(double))
        || lnb_buf_reserve_device(enc->dev, &enc->d_total, 64)
        || (enc->enable_learning && !forced
            && lnb_buf_reserve_device(enc->dev, &enc->d_train, BC * (2u * LNB_MAX_LAYERS + 1u) * ws * sizeof(double)))
        || (refine_global && lnb_buf_reserve_device(enc->dev, &enc->d_refine, BC * refine_doubles * sizeof(double))))
        return 0;
    batch->blocks = (LnbBlockDesc *)enc->d_blocks.ptr;
    batch->params = (LnbChanParams *)enc->d_params.ptr;
    batch->est = (double *)enc->d_est.ptr;
    batch->work = (int32_t *)enc->d_work.ptr;
    batch->sig_a = (double *)enc->d_sig_a.ptr;
    batch->sig_b = (double *)enc->d_sig_b.ptr;
    batch->acorr = (double *)enc->d_acorr.ptr;
    batch->cand = (double *)enc->d_cand.ptr;
    batch->unit_loss = (double *)enc->d_unit_loss.ptr;
    batch->chosen_w = (double *)enc->d_chosen_w.ptr;
    batch->chosen_log2u = (uint8_t *)enc->d_chosen_u.ptr;
    batch->final_sum = (double *)enc->d_final_sum.ptr;
    batch->welch = (const double *)enc->d_welch.ptr;
    /* sine window of the block-type estimate, tabulated once per block length for the cooperative prepare kernel */
    if (NB >= 2u && NB <= lnb_shim_coop_max_n() && enc->sinwin_n != NB) {
        enc->sinwin_n = 0;
        if (!lnb_buf_reserve_device(enc->dev, &enc->d_sinwin, (size_t)NB * sizeof(double))
            && lnb_shim_fill_sine_window(enc->dev, (double *)enc->d_sinwin.ptr, NB) == 0) enc->sinwin_n = NB;
    }
    batch->sinwin = (enc->sinwin_n == NB) ? (const double *)enc->d_sinwin.ptr : NULL;
    batch->sinwin_n = enc->sinwin_n;
    batch->plans = (LnbCoderPlan *)enc->d_plans.ptr;
    batch->plan_mean = (double *)enc->d_plan_mean.ptr;
    batch->total_size = (uint32_t *)enc->d_total.ptr;
    batch->train_scratch = (double *)enc->d_train.ptr;
    batch->refine_xy = refine_global ? (double *)enc->d_refine.ptr : NULL;
    return chunk_blocks;
}

/* Cuts blocks [first, first + nb) into the handle's pinned tables: block descriptors (h_blocks) and Welch scales
 * (h_welch), and the batch's block counts.  *file: the range of block `first`, advanced as blocks go by. */
static void cut_chunk(struct LINNEEncoder *enc, LnbEncodeBatch *batch, const struct LnbFileRange *ranges,
                      uint32_t first, uint32_t nb, uint32_t *file)
{
    const uint32_t NB = enc->header.num_samples_per_block;
    const uint32_t fast_max_na = lnb_shim_fast_max_na(), coop_max_n = lnb_shim_coop_max_n();
    LnbBlockDesc *hb = (LnbBlockDesc *)enc->h_blocks.ptr;
    double *hw = (double *)enc->h_welch.ptr;
    uint32_t i, lvl, num_fast = 0, num_coop = 0;
    for (i = 0; i < nb; i++) {
        const struct LnbFileRange *fr;
        uint32_t start, n;
        while (first + i >= ranges[*file].first_block + ranges[*file].num_blocks) (*file)++;
        fr = &ranges[*file];
        start = (first + i - fr->first_block) * NB;
        n = (fr->num_samples - start < NB) ? fr->num_samples - start : NB;
        start += fr->first_sample;
        memset(&hb[i], 0, sizeof(hb[i]));
        hb[i].smp_off = start; hb[i].nsmp = n; hb[i].na = analysis_length(&batch->cfg, n);
        if (hb[i].na <= fast_max_na) {                      /* cooperative analysis: fast layout or generic path */
            hb[i].status |= ((hb[i].na % 1024u) == 0u) ? LNB_ENC_FLAG_FAST : LNB_ENC_FLAG_GENERIC;
            num_fast++;
        }
        if (n <= coop_max_n && NB <= coop_max_n) { hb[i].status |= LNB_ENC_FLAG_COOP; num_coop++; }
        for (lvl = 0; lvl < LNB_MAX_LEVELS; lvl++) {
            const uint32_t m = hb[i].na >> lvl;
            hw[(size_t)i * LNB_MAX_LEVELS + lvl] = (m >= 2u) ? lnb_welch_scale(m) : 0.0;
        }
    }
    batch->num_blocks = nb;
    batch->num_coop_blocks = num_coop;
    batch->num_fast_blocks = num_fast;
    batch->num_slow_blocks = nb - num_fast;
}

/* Uploads the chunk cut_chunk() left in the pinned tables, analyses it and packs it speculatively right behind the size
 * scan (no host round trip): into rq->out at out_off, or a staging buffer of twice its raw size.  Should it not fit, the
 * packer skips the blocks that do not, and the chunk is packed once more at its exact size, *chunk_bytes. */
static LINNEApiResult pack_chunk(struct LINNEEncoder *enc, const EncodeRequest *rq, LnbEncodeBatch *batch, uint32_t first,
                                 uint32_t chunk_blocks, uint32_t out_off, uint32_t *chunk_bytes)
{
    const uint32_t nb = batch->num_blocks, C = enc->header.num_channels;
    LnbBlockDesc *hb = (LnbBlockDesc *)enc->h_blocks.ptr;
    size_t spec_cap;
    int attempt;
    if (rq->forced) lnb_shim_h2d(enc->dev, enc->d_params.ptr, rq->forced + (size_t)first * C, (size_t)nb * C * sizeof(LnbChanParams));
    lnb_shim_h2d(enc->dev, enc->d_blocks.ptr, hb, nb * sizeof(LnbBlockDesc));
    lnb_shim_h2d(enc->dev, enc->d_welch.ptr, enc->h_welch.ptr, (size_t)nb * LNB_MAX_LEVELS * sizeof(double));
    for (attempt = 0; attempt < 2; attempt++) {
        TRACE(enc, "enqueue");
        if (attempt == 1)     /* rare: start the chunk over (the packed flags live in the block table) */
            lnb_shim_h2d(enc->dev, enc->d_blocks.ptr, hb, nb * sizeof(LnbBlockDesc));
        if (lnb_shim_encode_analyze(enc->dev, batch)) return LINNE_APIRESULT_NG;
        if (attempt == 0) {
            if (rq->mode == ENC_OUT_DEVICE) {
                spec_cap = (size_t)rq->out_size - out_off;
                batch->out = rq->out + out_off;        /* block offsets from the scan are relative to the chunk */
            } else {
                spec_cap = 2u * (size_t)nb * (LNB_BLOCK_HEADER_SIZE + (size_t)enc->header.num_samples_per_block * C
                                              * ((enc->header.bits_per_sample + 7u) / 8u)) + 4096u;     /* twice the all-raw size */
                if (spec_cap > 0xFFFFFF00u) spec_cap = 0xFFFFFF00u;
                if (lnb_buf_reserve_device(enc->dev, &enc->d_out, spec_cap + 64u)) return LINNE_APIRESULT_NG;
                batch->out = (uint8_t *)enc->d_out.ptr;
            }
            if (lnb_shim_encode_pack(enc->dev, batch, (uint32_t)spec_cap)) return LINNE_APIRESULT_NG;
        }
        lnb_shim_d2h(enc->dev, enc->h_total.ptr, enc->d_total.ptr, sizeof(uint32_t));
        if (rq->mode == ENC_OUT_FILES)      /* byte offsets for place_files(): into the second half of h_blocks */
            lnb_shim_d2h(enc->dev, hb + chunk_blocks, enc->d_blocks.ptr, nb * sizeof(LnbBlockDesc));
        TRACE(enc, "enqueued");
        if (lnb_shim_sync(enc->dev)) return LINNE_APIRESULT_NG;
        TRACE(enc, "sizes known");
        *chunk_bytes = *(uint32_t *)enc->h_total.ptr;
        if (rq->mode != ENC_OUT_FILES && (uint64_t)out_off + *chunk_bytes > rq->out_size) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
        if (attempt == 0 && *chunk_bytes <= spec_cap) break;          /* everything fitted: the chunk is packed */
        if (attempt == 1) {
            if (rq->mode != ENC_OUT_DEVICE) {
                if (lnb_buf_reserve_device(enc->dev, &enc->d_out, (size_t)*chunk_bytes + 64u)) return LINNE_APIRESULT_NG;
                batch->out = (uint8_t *)enc->d_out.ptr;
            }
            if (lnb_shim_encode_pack(enc->dev, batch, *chunk_bytes)) return LINNE_APIRESULT_NG;
        }
    }
    return LINNE_APIRESULT_OK;
}

/* Corpus batch: moves each file's run of blocks of the chunk (contiguous in the staging buffer, byte offsets in `hb`)
 * behind its header in rq->out; a file that has all its blocks gets its header and its entry in rq->files. */
static LINNEApiResult place_files(struct LINNEEncoder *enc, const EncodeRequest *rq, const LnbBlockDesc *hb, uint32_t first,
                                  uint32_t nb, uint32_t *file, uint32_t *file_bytes, uint32_t *out_off)
{
    uint32_t lo = 0;
    while (lo < nb) {
        const struct LnbFileRange *fr = &rq->ranges[*file];
        const uint32_t file_end = fr->first_block + fr->num_blocks;            /* global block index */
        const uint32_t hi = (file_end - first < nb) ? file_end - first : nb;   /* chunk-relative */
        const uint32_t run = hb[hi - 1u].byte_off + hb[hi - 1u].byte_size - hb[lo].byte_off;
        if ((uint64_t)*out_off + LINNE_HEADER_SIZE + *file_bytes + run > rq->out_size) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
        lnb_shim_d2d(enc->dev, rq->out + *out_off + LINNE_HEADER_SIZE + *file_bytes,
                     (const uint8_t *)enc->d_out.ptr + hb[lo].byte_off, run);
        *file_bytes += run;
        lo = hi;
        if (first + hi == file_end) {                                          /* the file is complete */
            uint8_t *hdr = (uint8_t *)enc->h_headers.ptr + 32u * *file;
            struct LINNEHeader h1 = enc->header;
            h1.num_samples = fr->num_samples;
            lnb_header_write(&h1, hdr);
            lnb_shim_h2d(enc->dev, rq->out + *out_off, hdr, LINNE_HEADER_SIZE);
            rq->files[*file].out_offset = *out_off;
            rq->files[*file].out_size = LINNE_HEADER_SIZE + *file_bytes;
            *out_off += LINNE_HEADER_SIZE + *file_bytes;
            *file_bytes = 0;
            (*file)++;
        }
    }
    return LINNE_APIRESULT_OK;
}

/* Encodes the blocks of a request chunk by chunk: blocks are cut every header.num_samples_per_block samples of each
 * stream, every block x channel of a chunk is one batch for the kernels.  *written: the end of the output in rq->out. */
static LINNEApiResult encode_blocks(struct LINNEEncoder *enc, const EncodeRequest *rq, uint32_t *written)
{
    const struct LINNEHeader *h = &enc->header;
    const int files_mode = (rq->mode == ENC_OUT_FILES);
    const struct LnbFileRange whole = { 0u, rq->num_samples, 0u, (uint32_t)num_blocks(h, rq->num_samples) };
    const struct LnbFileRange *ranges = files_mode ? rq->ranges : &whole;
    const struct LnbFileRange *last = &ranges[files_mode ? rq->num_ranges - 1u : 0u];
    const uint32_t total_blocks = last->first_block + last->num_blocks;
    LnbEncodeBatch batch;
    LINNEApiResult ret;
    uint32_t chunk_blocks, first, chunk_bytes, out_off = rq->first_byte;
    uint32_t fcur = 0;                     /* file of the first block of the chunk being cut */
    uint32_t fdone = 0, fbytes = 0;        /* files mode: file being written out, block bytes it has received so far */

    memset(&batch, 0, sizeof(batch));
    lnb_fill_stream_cfg(&batch.cfg, h);
    batch.cfg.pcm_stride = rq->pcm_stride;
    batch.cfg.work_stride = (uint32_t)LNB_ROUNDUP((size_t)h->num_samples_per_block, 4u);
    batch.tab = *lnb_shim_tables(enc->dev);
    batch.pcm = rq->pcm;
    if ((chunk_blocks = reserve_scratch(enc, &batch, total_blocks, rq->forced != NULL)) == 0) return LINNE_APIRESULT_NG;
    batch.af_iterations = rq->forced ? 0u : enc->num_afmethod_iterations;
    batch.enable_learning = rq->forced ? 0u : (enc->enable_learning ? 1u : 0u);
    batch.forced_params = rq->forced ? 1u : 0u;

    for (first = 0; first < total_blocks; first += chunk_blocks) {
        cut_chunk(enc, &batch, ranges, first, (total_blocks - first < chunk_blocks) ? total_blocks - first : chunk_blocks, &fcur);
        if ((ret = pack_chunk(enc, rq, &batch, first, chunk_blocks, out_off, &chunk_bytes)) != LINNE_APIRESULT_OK) return ret;
        if (rq->mode == ENC_OUT_HOST) lnb_shim_d2h(enc->dev, rq->out + out_off, enc->d_out.ptr, chunk_bytes);
        if (files_mode && (ret = place_files(enc, rq, (const LnbBlockDesc *)enc->h_blocks.ptr + chunk_blocks, first,
                                             batch.num_blocks, &fdone, &fbytes, &out_off)) != LINNE_APIRESULT_OK) return ret;
        TRACE(enc, "pack enqueued");
        if (lnb_shim_sync(enc->dev)) return LINNE_APIRESULT_NG;
        TRACE(enc, "chunk done");
        if (!files_mode) out_off += chunk_bytes;
    }
    *written = out_off;
    return LINNE_APIRESULT_OK;
}

/* the header step of the whole-stream calls: enc->header for num_samples into data[0, 30), host or device memory */
static LINNEApiResult write_header(struct LINNEEncoder *enc, uint32_t num_samples, uint8_t *data, uint32_t data_size, int on_device)
{
    uint8_t hdr[LINNE_HEADER_SIZE];
    LINNEApiResult ret;
    enc->header.num_samples = num_samples;
    if ((ret = LINNEEncoder_EncodeHeader(&enc->header, on_device ? hdr : data, data_size)) != LINNE_APIRESULT_OK) return ret;
    if (on_device) lnb_shim_h2d(enc->dev, data, hdr, LINNE_HEADER_SIZE);
    return LINNE_APIRESULT_OK;
}

/* reference linne_encoder.c:774-862 */
LINNEApiResult LINNEEncoder_EncodeBlock(struct LINNEEncoder *enc, const int32_t *const *input, uint32_t num_samples,
        uint8_t *data, uint32_t data_size, uint32_t *output_size)
{
    EncodeRequest rq = { .out = data, .out_size = data_size, .mode = ENC_OUT_HOST };
    LINNEApiResult ret;
    if (enc == NULL || input == NULL || num_samples == 0 || data == NULL || data_size == 0 || output_size == NULL)
        return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (enc->set_parameter != 1) return LINNE_APIRESULT_PARAMETER_NOT_SET;
    if (num_samples > enc->header.num_samples_per_block) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
    if ((ret = upload_planes(enc, input, 0, num_samples, &rq)) != LINNE_APIRESULT_OK) return ret;
    return encode_blocks(enc, &rq, output_size);
}

/* ---- several GPUs behind one handle -----------------------------------------------------------------------------
 * Blocks are independent (SURVEY 8e), so EncodeWhole cuts [0, B) into contiguous block ranges, one per device.  Every
 * range has a child handle bound to its device and a host thread: it uploads its samples, encodes them into a shard on
 * its device and reports the shard's size; an exclusive scan of the sizes on the host gives every shard its place, and
 * each child copies its shard straight into the caller's buffer there.  No collective, no inter-process machinery;
 * the stream is byte-identical with the single-device one.  (With more ranges than devices the ranges share devices
 * round-robin: that is how a one-GPU box exercises this path.) */
void LINNEB200_EncoderSetDevices(struct LINNEEncoder *enc, uint32_t num_devices)
{
    if (enc == NULL) return;
    if (num_devices > LNB_MAX_DEVICES) num_devices = LNB_MAX_DEVICES;
    enc->num_devices = num_devices;
}

struct LnbEncShard {
    struct LINNEEncoder *child;
    const int32_t *const *input;           /* int32 planes, or ... */
    const uint8_t *packed;                 /* ... interleaved packed PCM (WAV data-chunk layout) */
    uint32_t first_sample, num_samples;
    uint32_t size, offset;                 /* shard bytes (blocks only) / where they go in the caller's buffer */
    uint32_t room;                         /* bytes of the caller's buffer behind the header */
    uint8_t *data;
    LINNEApiResult result;
    LnbRendezvous *meet;
    int ordinal;
};

static void *enc_shard_main(void *arg)
{
    struct LnbEncShard *sh = (struct LnbEncShard *)arg;
    struct LINNEEncoder *enc = sh->child;
    /* no more than the caller's whole buffer: a shard larger than that fails the call in any case */
    const uint64_t room = stream_room(&enc->header, sh->num_samples);
    const uint32_t cap = (uint32_t)(room < sh->room ? (room < 0xFFFFFF00u ? room : 0xFFFFFF00u) : sh->room);
    EncodeRequest rq = { .out_size = cap, .mode = ENC_OUT_DEVICE };
    lnb_shim_set_device(sh->ordinal);
    if (lnb_buf_reserve_device(enc->dev, &enc->d_shard, cap)) sh->result = LINNE_APIRESULT_NG;
    else if (sh->packed) sh->result = upload_packed(enc, sh->packed, sh->first_sample, sh->num_samples, &rq);
    else sh->result = upload_planes(enc, sh->input, sh->first_sample, sh->num_samples, &rq);
    rq.out = (uint8_t *)enc->d_shard.ptr;
    if (sh->result == LINNE_APIRESULT_OK) sh->result = encode_blocks(enc, &rq, &sh->size);
    lnb_rendezvous_report_and_wait(sh->meet);   /* every shard's size is known: the caller scans them and says where each goes */
    if (sh->result == LINNE_APIRESULT_OK && sh->data) {
        lnb_shim_d2h(enc->dev, sh->data + sh->offset, enc->d_shard.ptr, sh->size);
        if (lnb_shim_sync(enc->dev)) sh->result = LINNE_APIRESULT_NG;
    }
    return NULL;
}

/* the blocks of EncodeWhole over G block ranges, behind the stream header in data[0, 30) */
static LINNEApiResult encode_whole_sharded(struct LINNEEncoder *enc, uint32_t G, const int32_t *const *input, const uint8_t *packed,
                                           uint32_t num_samples, uint8_t *data, uint32_t data_size, uint32_t *output_size)
{
    const uint32_t NB = enc->header.num_samples_per_block, total_blocks = (uint32_t)num_blocks(&enc->header, num_samples);
    const int ndev = lnb_shim_device_count();
    struct LnbEncShard sh[LNB_MAX_DEVICES];
    pthread_t th[LNB_MAX_DEVICES];
    int ordinal[LNB_MAX_DEVICES];
    LnbRendezvous meet;
    LINNEApiResult ret = LINNE_APIRESULT_OK;
    uint32_t k, started = 0, off = 0;
    int home = -1;
    if (ndev <= 0) return LINNE_APIRESULT_NG;
    home = lnb_shim_current_device();
    lnb_place_ranges(enc->num_devices, ndev, lnb_shim_device_ordinal(enc->dev), G, ordinal);      /* devices in use: not needed */
    for (k = 0; k < G; k++) {
        if (!enc->child[k]) {
            lnb_shim_set_device(ordinal[k]);
            enc->child[k] = LINNEEncoder_Create(&enc->config, NULL, 0);
            if (enc->child[k]) enc->child[k]->num_devices = 0;          /* children never shard again */
        }
        if (!enc->child[k] || LINNEEncoder_SetEncodeParameter(enc->child[k], &enc->param) != LINNE_APIRESULT_OK) { ret = LINNE_APIRESULT_NG; break; }
        enc->child[k]->scratch_budget = enc->scratch_budget;
    }
    if (home >= 0) lnb_shim_set_device(home);
    if (ret != LINNE_APIRESULT_OK) return ret;
    lnb_rendezvous_init(&meet);
    for (k = 0; k < G; k++) {
        /* contiguous block ranges, as even as the block count allows */
        const uint32_t b0 = (uint32_t)((uint64_t)total_blocks * k / G), b1 = (uint32_t)((uint64_t)total_blocks * (k + 1u) / G);
        const uint64_t s0 = (uint64_t)b0 * NB, s1 = (uint64_t)b1 * NB;
        memset(&sh[k], 0, sizeof(sh[k]));
        sh[k].child = enc->child[k]; sh[k].input = input; sh[k].packed = packed;
        sh[k].first_sample = (uint32_t)s0;
        sh[k].num_samples = (uint32_t)((s1 > num_samples ? num_samples : s1) - s0);
        sh[k].data = data + LINNE_HEADER_SIZE; sh[k].room = data_size - LINNE_HEADER_SIZE; sh[k].meet = &meet;
        sh[k].ordinal = ordinal[k];
        if (pthread_create(&th[k], NULL, enc_shard_main, &sh[k]) != 0) { sh[k].result = LINNE_APIRESULT_NG; break; }
        started++;
    }
    lnb_rendezvous_collect(&meet, started);
    for (k = 0; k < started; k++) {                                /* exclusive scan of the shard byte counts */
        if (sh[k].result != LINNE_APIRESULT_OK && ret == LINNE_APIRESULT_OK) ret = sh[k].result;
        sh[k].offset = off;
        off += sh[k].size;
    }
    if (ret == LINNE_APIRESULT_OK && (started < G || off > data_size - LINNE_HEADER_SIZE)) ret = (started < G) ? LINNE_APIRESULT_NG : LINNE_APIRESULT_INSUFFICIENT_BUFFER;
    if (ret != LINNE_APIRESULT_OK) for (k = 0; k < started; k++) sh[k].data = NULL;
    lnb_rendezvous_release(&meet);
    for (k = 0; k < started; k++) {
        pthread_join(th[k], NULL);
        if (sh[k].result != LINNE_APIRESULT_OK && ret == LINNE_APIRESULT_OK) ret = sh[k].result;
    }
    lnb_rendezvous_destroy(&meet);
    if (ret == LINNE_APIRESULT_OK) *output_size = LINNE_HEADER_SIZE + off;
    return ret;
}

/* EncodeWhole and EncodeWholePacked (PCM in `input` planes or `packed`): the header, then the blocks behind it -- over
 * several block ranges when there are several devices, or a stream long enough to pipeline its transfers against its
 * kernels on one */
static LINNEApiResult encode_whole(struct LINNEEncoder *enc, const int32_t *const *input, const uint8_t *packed,
                                   uint32_t num_samples, uint8_t *data, uint32_t data_size, uint32_t *output_size)
{
    EncodeRequest rq = { .out = data, .first_byte = LINNE_HEADER_SIZE, .out_size = data_size, .mode = ENC_OUT_HOST };
    LINNEApiResult ret;
    uint32_t G, c;
    if (enc == NULL || data == NULL || output_size == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (enc->set_parameter != 1) return LINNE_APIRESULT_PARAMETER_NOT_SET;
    if (packed && !packed_bits_ok(&enc->header)) return LINNE_APIRESULT_INVALID_FORMAT;
    if ((ret = write_header(enc, num_samples, data, data_size, 0)) != LINNE_APIRESULT_OK) return ret;
    for (c = 0; input && c < enc->header.num_channels; c++) if (input[c] == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if ((G = lnb_plan_ranges((uint32_t)num_blocks(&enc->header, num_samples), enc->num_devices > 1u ? enc->num_devices : 1u)) > 1u)
        return encode_whole_sharded(enc, G, input, packed, num_samples, data, data_size, output_size);
    if ((ret = input ? upload_planes(enc, input, 0, num_samples, &rq) : upload_packed(enc, packed, 0, num_samples, &rq)) != LINNE_APIRESULT_OK)
        return ret;
    return encode_blocks(enc, &rq, output_size);
}

/* reference linne_encoder.c:865-932 */
LINNEApiResult LINNEEncoder_EncodeWhole(struct LINNEEncoder *enc, const int32_t *const *input, uint32_t num_samples,
        uint8_t *data, uint32_t data_size, uint32_t *output_size)
{
    if (input == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    return encode_whole(enc, input, NULL, num_samples, data, data_size, output_size);
}

LnbDevice *lnb_encoder_device(const struct LINNEEncoder *enc) { return enc->dev; }

/* ---- extension entry points (include/linne_b200.h) ---- */

LINNEApiResult LINNEB200_EncodeWholeWithParams(struct LINNEEncoder *enc, const int32_t *const *input,
        uint32_t num_samples, const struct LINNEB200ChannelParams *params, uint32_t num_param_blocks,
        uint8_t *data, uint32_t data_size, uint32_t *output_size)
{
    LINNEApiResult ret;
    LnbChanParams *forced;
    uint64_t blocks;
    size_t i;
    EncodeRequest rq = { .out = data, .first_byte = LINNE_HEADER_SIZE, .out_size = data_size, .mode = ENC_OUT_HOST };
    uint32_t l, C;
    if (enc == NULL || input == NULL || params == NULL || data == NULL || output_size == NULL)
        return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (enc->set_parameter != 1) return LINNE_APIRESULT_PARAMETER_NOT_SET;
    C = enc->header.num_channels;
    blocks = num_blocks(&enc->header, num_samples);
    if (num_param_blocks < blocks) return LINNE_APIRESULT_INVALID_ARGUMENT;
    /* the stream stores these in 3 and 4 bits: a larger value would be written masked but predicted with unmasked */
    for (i = 0; i < blocks * C; i++)
        for (l = 0; l < (uint32_t)g_lnb_presets[enc->header.preset].num_layers; l++)
            if (params[i].log2_units[l] > 7u || params[i].rshift[l] > 15u) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if ((ret = write_header(enc, num_samples, data, data_size, 0)) != LINNE_APIRESULT_OK) return ret;
    forced = (LnbChanParams *)calloc((size_t)blocks * C, sizeof(LnbChanParams));
    if (!forced) return LINNE_APIRESULT_NG;
    for (i = 0; i < blocks * C; i++)
        for (l = 0; l < LNB_MAX_LAYERS; l++) {
            forced[i].log2_units[l] = params[i].log2_units[l];
            forced[i].rshift[l] = params[i].rshift[l];
            memcpy(forced[i].coef + l * LNB_MAX_PARAMS, params[i].coef[l], LNB_MAX_PARAMS);
        }
    rq.forced = forced;
    if ((ret = upload_planes(enc, input, 0, num_samples, &rq)) == LINNE_APIRESULT_OK) ret = encode_blocks(enc, &rq, output_size);
    free(forced);
    return ret;
}

LINNEApiResult LINNEB200_EncodeWholeResident(struct LINNEEncoder *enc, const int32_t *d_pcm, uint32_t pcm_stride,
        uint32_t num_samples, uint8_t *d_data, uint32_t data_size, uint32_t *output_size)
{
    const EncodeRequest rq = { .pcm = d_pcm, .pcm_stride = pcm_stride, .num_samples = num_samples, .out = d_data,
                               .first_byte = LINNE_HEADER_SIZE, .out_size = data_size, .mode = ENC_OUT_DEVICE };
    LINNEApiResult ret;
    if (enc == NULL || d_pcm == NULL || d_data == NULL || output_size == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (enc->set_parameter != 1) return LINNE_APIRESULT_PARAMETER_NOT_SET;
    if (pcm_stride < num_samples) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if ((ret = write_header(enc, num_samples, d_data, data_size, 1)) != LINNE_APIRESULT_OK) return ret;
    return encode_blocks(enc, &rq, output_size);
}

/* Several files per call (corpus batches, SURVEY 8e: "concatenate files' block lists, keeping per-file boundaries").
 * All files share the encoder's parameters; their PCM sits in one set of device planes [C][pcm_stride], file i at
 * samples [first_sample, first_sample + num_samples).  Every block x channel of every file is one batch for the
 * kernels; the streams are written one after the other into `d_data` (header + blocks each, byte-identical with
 * what EncodeWhole writes for that file) and files[i].out_offset / out_size say where. */
LINNEApiResult LINNEB200_EncodeFilesResident(struct LINNEEncoder *enc, const int32_t *d_pcm, uint32_t pcm_stride,
        struct LINNEB200FileDesc *files, uint32_t num_files, uint8_t *d_data, uint32_t data_size, uint32_t *output_size)
{
    struct LnbFileRange *ranges;
    LINNEApiResult ret;
    uint32_t written = 0, i, blocks = 0;
    if (enc == NULL || d_pcm == NULL || files == NULL || num_files == 0 || d_data == NULL || output_size == NULL)
        return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (enc->set_parameter != 1) return LINNE_APIRESULT_PARAMETER_NOT_SET;
    if (!(ranges = (struct LnbFileRange *)malloc((size_t)num_files * sizeof(*ranges)))) return LINNE_APIRESULT_NG;
    for (i = 0; i < num_files; i++) {
        if (files[i].num_samples == 0 || (uint64_t)files[i].first_sample + files[i].num_samples > pcm_stride) { free(ranges); return LINNE_APIRESULT_INVALID_ARGUMENT; }
        ranges[i].first_sample = files[i].first_sample; ranges[i].num_samples = files[i].num_samples;
        ranges[i].first_block = blocks;
        ranges[i].num_blocks = (uint32_t)num_blocks(&enc->header, files[i].num_samples);
        blocks += ranges[i].num_blocks;
        files[i].out_offset = files[i].out_size = 0;
    }
    if (lnb_buf_reserve_host(&enc->h_headers, (size_t)num_files * 32u)) { free(ranges); return LINNE_APIRESULT_NG; }
    {
        const EncodeRequest rq = { .pcm = d_pcm, .pcm_stride = pcm_stride, .ranges = ranges, .num_ranges = num_files, .files = files,
                                   .out = d_data, .out_size = data_size, .mode = ENC_OUT_FILES };
        ret = encode_blocks(enc, &rq, &written);
    }
    free(ranges);
    if (ret != LINNE_APIRESULT_OK) return ret;
    *output_size = written;
    return LINNE_APIRESULT_OK;
}

/* The same for host buffers (what a corpus tool holds after reading its files): the files' frames back to back as
 * packed interleaved PCM (WAV data-chunk layout) in `pcm`, files[i].num_samples frames each; ONE transfer up, one
 * conversion, one batch for the kernels, one transfer down.  The streams land one after the other in the host
 * buffer `data`; files[i].first_sample (frame offset in `pcm`), out_offset and out_size are filled in. */
LINNEApiResult LINNEB200_EncodeFilesPacked(struct LINNEEncoder *enc, const uint8_t *pcm, struct LINNEB200FileDesc *files,
        uint32_t num_files, uint8_t *data, uint32_t data_size, uint32_t *output_size)
{
    LINNEApiResult ret;
    EncodeRequest planes;                  /* the PCM of the files, as upload_packed() leaves it */
    uint64_t total = 0, bound = 0;
    uint32_t i, written = 0;
    if (enc == NULL || pcm == NULL || files == NULL || num_files == 0 || data == NULL || output_size == NULL)
        return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (enc->set_parameter != 1) return LINNE_APIRESULT_PARAMETER_NOT_SET;
    if (!packed_bits_ok(&enc->header)) return LINNE_APIRESULT_INVALID_FORMAT;
    for (i = 0; i < num_files; i++) {
        if (files[i].num_samples == 0) return LINNE_APIRESULT_INVALID_ARGUMENT;
        files[i].first_sample = (uint32_t)total;
        total += files[i].num_samples;
        bound += stream_room(&enc->header, files[i].num_samples);
    }
    if (total > 0xFFFFFFF0ull) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (bound > data_size) bound = data_size;
    if (lnb_buf_reserve_device(enc->dev, &enc->d_image, (size_t)bound + 64u)) return LINNE_APIRESULT_NG;
    if ((ret = upload_packed(enc, pcm, 0, (uint32_t)total, &planes)) != LINNE_APIRESULT_OK) return ret;
    ret = LINNEB200_EncodeFilesResident(enc, planes.pcm, planes.pcm_stride, files, num_files,
                                        (uint8_t *)enc->d_image.ptr, (uint32_t)bound, &written);
    if (ret != LINNE_APIRESULT_OK) return ret;
    lnb_shim_d2h(enc->dev, data, enc->d_image.ptr, written);
    if (lnb_shim_sync(enc->dev)) return LINNE_APIRESULT_NG;
    *output_size = written;
    return LINNE_APIRESULT_OK;
}

/* Packed interleaved PCM in (the bytes of a WAV data chunk), converted to planes on the device: half (16-bit) or
 * three quarters (24-bit) of the PCIe bytes of the int32-planar call.  SURVEY 8f.2. */
LINNEApiResult LINNEB200_EncodeWholePacked(struct LINNEEncoder *enc, const uint8_t *pcm, uint32_t num_samples,
        uint8_t *data, uint32_t data_size, uint32_t *output_size)
{
    if (pcm == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    return encode_whole(enc, NULL, pcm, num_samples, data, data_size, output_size);
}
