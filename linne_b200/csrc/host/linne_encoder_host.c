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
    const int32_t *cur_pcm;                /* device PCM planes of the call in flight */
    uint32_t cur_pcm_stride;
    /* corpus batches (LINNEB200_EncodeFilesResident): the sample ranges of the files of the call in flight */
    const struct LnbFileRange *ranges;
    uint32_t num_ranges;
    struct LINNEB200FileDesc *file_out;    /* per-file results of that call */
    LnbBuf h_headers;                      /* pinned 32-byte slots for the files' stream headers */
    /* several GPUs behind ONE handle (SURVEY 8e, north star): EncodeWhole splits its blocks into contiguous ranges, one
     * child handle (own device, own host thread) per range */
    uint32_t num_devices;                  /* 0/1: this handle's device only */
    struct LINNEEncoder *child[LNB_MAX_DEVICES];
    LnbBuf d_shard;                        /* a child's shard of the stream, on its device */
    struct LINNEEncoderConfig config;      /* to create the children with */
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

/* Encode the blocks covering samples [first_sample, first_sample + num_samples) of the device PCM
 * planes into data[0..data_size); blocks are cut every header.num_samples_per_block samples. */
/* `data` is a host buffer unless `data_on_device` is set; `forced` (optional, host memory,
 * [total_blocks * C]) supplies unit counts / shifts / coefficients and skips the analysis.
 * data_on_device == 2 (corpus batch, enc->ranges set): the blocks of SEVERAL files go through the kernels as one
 * batch -- blocks are cut per file, packed back to back into the staging buffer, and every file's byte range is then
 * moved behind its own 30-byte header in `data` (device-to-device), files laid out one after the other. */
static LINNEApiResult encode_blocks(struct LINNEEncoder *enc, uint32_t num_samples,
                                    uint8_t *data, uint32_t data_size, int data_on_device,
                                    const LnbChanParams *forced, uint32_t *written)
{
    const struct LINNEHeader *h = &enc->header;
    const uint32_t C = h->num_channels, NB = h->num_samples_per_block;
    const int files_mode = (data_on_device == 2);
    const uint32_t total_blocks = files_mode
        ? enc->ranges[enc->num_ranges - 1u].first_block + enc->ranges[enc->num_ranges - 1u].num_blocks
        : (uint32_t)(((uint64_t)num_samples + NB - 1u) / NB);
    LnbEncodeBatch batch;
    uint32_t lambdas, slots_per_block, chunk_blocks, first, out_off = 0, i, lvl;
    uint32_t fcur = 0;                     /* files mode: file of the first block of the chunk being built */
    uint32_t fdone = 0, fbytes = 0;        /* files mode: file being written out, block bytes it has received so far */
    size_t per_block, refine_doubles = 0;
    int refine_global = 0;

    memset(&batch, 0, sizeof(batch));
    lnb_fill_stream_cfg(&batch.cfg, h);
    batch.cfg.pcm_stride = enc->cur_pcm_stride;
    batch.cfg.work_stride = (uint32_t)LNB_ROUNDUP((size_t)NB, 4u);
    batch.tab = *lnb_shim_tables(enc->dev);
    batch.pcm = enc->cur_pcm;
    lambdas = batch.cfg.num_lambdas;
    slots_per_block = C * lambdas;

    /* Chunk so the per-chunk scratch stays inside the budget.  Blocks of up to lnb_shim_fast_max_na()
     * samples are analysed by the cooperative kernel (signal in shared memory): they need only the
     * integer work signal and the per-slot results.  Longer blocks take the flat kernels, which keep
     * two double-precision planes and per-level tables in HBM. */
    {
        const int need_flat = NB > lnb_shim_fast_max_na();
        const size_t ws = batch.cfg.work_stride, chunks = (ws + 63u) / 64u;
        per_block = (size_t)slots_per_block * (LNB_MAX_LAYERS * LNB_MAX_PARAMS * sizeof(double) + chunks * sizeof(double) + 64u)
                  + (size_t)C * (ws * sizeof(int32_t) + sizeof(LnbChanParams) + sizeof(LnbCoderPlan)
                                 + 2u * LNB_MAX_PARTITIONS * sizeof(double) + 64u)
                  + (enc->enable_learning ? (size_t)C * (2u * LNB_MAX_LAYERS + 1u) * ws * sizeof(double) : 0u);
        const int need_sig_a = need_flat || (enc->num_afmethod_iterations && !forced);    /* IRLS scratch: one plane per slot */
        /* IRLS / SGD on blocks too long for the refinement kernel's shared memory: its two signal buffers in HBM (lnb_shim.h) */
        refine_global = !forced && (enc->enable_learning || enc->num_afmethod_iterations)
                        && lnb_shim_refine_max_na() && NB > lnb_shim_refine_max_na();
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
        {
            const size_t S = (size_t)chunk_blocks * slots_per_block, BC = (size_t)chunk_blocks * C;
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
                return LINNE_APIRESULT_NG;
        }
    }
    batch.blocks = (LnbBlockDesc *)enc->d_blocks.ptr;
    batch.params = (LnbChanParams *)enc->d_params.ptr;
    batch.est = (double *)enc->d_est.ptr;
    batch.work = (int32_t *)enc->d_work.ptr;
    batch.sig_a = (double *)enc->d_sig_a.ptr;
    batch.sig_b = (double *)enc->d_sig_b.ptr;
    batch.acorr = (double *)enc->d_acorr.ptr;
    batch.cand = (double *)enc->d_cand.ptr;
    batch.unit_loss = (double *)enc->d_unit_loss.ptr;
    batch.chosen_w = (double *)enc->d_chosen_w.ptr;
    batch.chosen_log2u = (uint8_t *)enc->d_chosen_u.ptr;
    batch.final_sum = (double *)enc->d_final_sum.ptr;
    batch.welch = (const double *)enc->d_welch.ptr;
    /* sine window of the block-type estimate, tabulated once per block length for the cooperative prepare kernel */
    if (NB >= 2u && NB <= lnb_shim_coop_max_n() && enc->sinwin_n != NB) {
        enc->sinwin_n = 0;
        if (!lnb_buf_reserve_device(enc->dev, &enc->d_sinwin, (size_t)NB * sizeof(double))
            && lnb_shim_fill_sine_window(enc->dev, (double *)enc->d_sinwin.ptr, NB) == 0) enc->sinwin_n = NB;
    }
    batch.sinwin = (enc->sinwin_n == NB) ? (const double *)enc->d_sinwin.ptr : NULL;
    batch.sinwin_n = enc->sinwin_n;
    batch.plans = (LnbCoderPlan *)enc->d_plans.ptr;
    batch.plan_mean = (double *)enc->d_plan_mean.ptr;
    batch.total_size = (uint32_t *)enc->d_total.ptr;
    batch.af_iterations = forced ? 0u : enc->num_afmethod_iterations;
    batch.enable_learning = forced ? 0u : (enc->enable_learning ? 1u : 0u);
    batch.train_scratch = (double *)enc->d_train.ptr;
    batch.refine_xy = refine_global ? (double *)enc->d_refine.ptr : NULL;
    batch.out_base = 0;

    for (first = 0; first < total_blocks; first += chunk_blocks) {
        const uint32_t nb = (total_blocks - first < chunk_blocks) ? total_blocks - first : chunk_blocks;
        LnbBlockDesc *hb = (LnbBlockDesc *)enc->h_blocks.ptr;
        LnbBlockDesc *hres = hb + chunk_blocks;                 /* files mode: second half of h_blocks */
        double *hw = (double *)enc->h_welch.ptr;
        uint32_t chunk_bytes, num_fast = 0, num_coop = 0;
        const uint32_t fast_max_na = lnb_shim_fast_max_na(), coop_max_n = lnb_shim_coop_max_n();
        for (i = 0; i < nb; i++) {
            uint32_t start, n;
            if (files_mode) {
                const struct LnbFileRange *fr;
                while (first + i >= enc->ranges[fcur].first_block + enc->ranges[fcur].num_blocks) fcur++;
                fr = &enc->ranges[fcur];
                start = (first + i - fr->first_block) * NB;
                n = (fr->num_samples - start < NB) ? fr->num_samples - start : NB;
                start += fr->first_sample;
            } else {
                start = (first + i) * NB;
                n = (num_samples - start < NB) ? num_samples - start : NB;
            }
            memset(&hb[i], 0, sizeof(hb[i]));
            hb[i].smp_off = start; hb[i].nsmp = n; hb[i].na = analysis_length(&batch.cfg, n);
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
        batch.num_blocks = nb;
        batch.num_coop_blocks = num_coop;
        batch.num_fast_blocks = num_fast;
        batch.num_slow_blocks = nb - num_fast;
        batch.forced_params = forced ? 1u : 0u;
        if (forced) lnb_shim_h2d(enc->dev, enc->d_params.ptr, forced + (size_t)first * C, (size_t)nb * C * sizeof(LnbChanParams));
        lnb_shim_h2d(enc->dev, enc->d_blocks.ptr, hb, nb * sizeof(LnbBlockDesc));
        lnb_shim_h2d(enc->dev, enc->d_welch.ptr, hw, (size_t)nb * LNB_MAX_LEVELS * sizeof(double));
        {
            /* Pack speculatively right behind the size scan -- no host round trip in between.  The staging buffer is
             * sized for twice the raw bound of the chunk; should a chunk ever exceed that (or the caller's device
             * buffer be too small) the packer skips the blocks that do not fit and the second attempt below packs
             * again once the exact size is known. */
            const size_t raw_bound = (size_t)nb * (LNB_BLOCK_HEADER_SIZE + (size_t)NB * C * ((h->bits_per_sample + 7u) / 8u));
            size_t spec_cap;
            int attempt;
            for (attempt = 0; attempt < 2; attempt++) {
                TRACE(enc, "enqueue");
                if (attempt == 1) {   /* rare: start the chunk over (the packed flags live in the block table) */
                    lnb_shim_h2d(enc->dev, enc->d_blocks.ptr, hb, nb * sizeof(LnbBlockDesc));
                }
                if (lnb_shim_encode_analyze(enc->dev, &batch)) return LINNE_APIRESULT_NG;
                if (attempt == 0) {
                    if (data_on_device == 1) {
                        spec_cap = (size_t)data_size - out_off;
                        batch.out = data + out_off;       /* block offsets from the scan are relative to the chunk */
                    } else {
                        spec_cap = 2u * raw_bound + 4096u;
                        if (spec_cap > 0xFFFFFF00u) spec_cap = 0xFFFFFF00u;
                        if (lnb_buf_reserve_device(enc->dev, &enc->d_out, spec_cap + 64u)) return LINNE_APIRESULT_NG;
                        batch.out = (uint8_t *)enc->d_out.ptr;
                    }
                    if (lnb_shim_encode_pack(enc->dev, &batch, (uint32_t)spec_cap)) return LINNE_APIRESULT_NG;
                }
                lnb_shim_d2h(enc->dev, enc->h_total.ptr, enc->d_total.ptr, sizeof(uint32_t));
                if (files_mode) lnb_shim_d2h(enc->dev, hres, enc->d_blocks.ptr, nb * sizeof(LnbBlockDesc));   /* byte offsets */
                TRACE(enc, "enqueued");
                if (lnb_shim_sync(enc->dev)) return LINNE_APIRESULT_NG;
                TRACE(enc, "sizes known");
                chunk_bytes = *(uint32_t *)enc->h_total.ptr;
                if (!files_mode && (uint64_t)out_off + chunk_bytes > data_size) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
                if (attempt == 0 && chunk_bytes <= spec_cap) break;          /* everything fitted: the chunk is packed */
                if (attempt == 1) {
                    if (data_on_device != 1) {
                        if (lnb_buf_reserve_device(enc->dev, &enc->d_out, (size_t)chunk_bytes + 64u)) return LINNE_APIRESULT_NG;
                        batch.out = (uint8_t *)enc->d_out.ptr;
                    }
                    if (lnb_shim_encode_pack(enc->dev, &batch, chunk_bytes)) return LINNE_APIRESULT_NG;
                }
            }
            if (!data_on_device) lnb_shim_d2h(enc->dev, data + out_off, enc->d_out.ptr, chunk_bytes);
            if (files_mode) {
                /* runs of blocks of one file are contiguous in the staging buffer: move each run behind its file's
                 * header; a file that has all its blocks gets its header and its entry in the result table */
                uint32_t lo = 0;
                const LnbBlockDesc *hb = hres;                                             /* the table as the device left it */
                while (lo < nb) {
                    const struct LnbFileRange *fr = &enc->ranges[fdone];
                    const uint32_t file_end = fr->first_block + fr->num_blocks;            /* global block index */
                    const uint32_t hi = (file_end - first < nb) ? file_end - first : nb;   /* chunk-relative */
                    const uint32_t run = hb[hi - 1u].byte_off + hb[hi - 1u].byte_size - hb[lo].byte_off;
                    if ((uint64_t)out_off + LINNE_HEADER_SIZE + fbytes + run > data_size) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
                    lnb_shim_d2d(enc->dev, data + out_off + LINNE_HEADER_SIZE + fbytes,
                                 (const uint8_t *)enc->d_out.ptr + hb[lo].byte_off, run);
                    fbytes += run;
                    lo = hi;
                    if (first + hi == file_end) {                                          /* the file is complete */
                        uint8_t *hdr = (uint8_t *)enc->h_headers.ptr + 32u * fdone;
                        struct LINNEHeader h1 = *h;
                        h1.num_samples = fr->num_samples;
                        lnb_header_write(&h1, hdr);
                        lnb_shim_h2d(enc->dev, data + out_off, hdr, LINNE_HEADER_SIZE);
                        enc->file_out[fdone].out_offset = out_off;
                        enc->file_out[fdone].out_size = LINNE_HEADER_SIZE + fbytes;
                        out_off += LINNE_HEADER_SIZE + fbytes;
                        fbytes = 0; fdone++;
                    }
                }
            }
            TRACE(enc, "pack enqueued");
            if (lnb_shim_sync(enc->dev)) return LINNE_APIRESULT_NG;
            TRACE(enc, "chunk done");
        }
        if (!files_mode) out_off += chunk_bytes;
    }
    *written = out_off;
    return LINNE_APIRESULT_OK;
}

static LINNEApiResult upload_and_encode(struct LINNEEncoder *enc, const int32_t *const *input, uint32_t num_samples,
                                        uint8_t *data, uint32_t data_size, const LnbChanParams *forced, uint32_t *written)
{
    const uint32_t C = enc->header.num_channels;
    const size_t stride = LNB_ROUNDUP((size_t)num_samples + 4u, 4u);
    uint32_t c;
    if (lnb_buf_reserve_device(enc->dev, &enc->d_pcm, stride * C * sizeof(int32_t))) return LINNE_APIRESULT_NG;
    for (c = 0; c < C; c++) {
        if (input[c] == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
        lnb_shim_h2d(enc->dev, (int32_t *)enc->d_pcm.ptr + c * stride, input[c], (size_t)num_samples * sizeof(int32_t));
    }
    enc->cur_pcm = (const int32_t *)enc->d_pcm.ptr;
    enc->cur_pcm_stride = (uint32_t)stride;
    return encode_blocks(enc, num_samples, data, data_size, 0, forced, written);
}

/* reference linne_encoder.c:774-862 */
LINNEApiResult LINNEEncoder_EncodeBlock(struct LINNEEncoder *enc, const int32_t *const *input, uint32_t num_samples,
        uint8_t *data, uint32_t data_size, uint32_t *output_size)
{
    if (enc == NULL || input == NULL || num_samples == 0 || data == NULL || data_size == 0 || output_size == NULL)
        return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (enc->set_parameter != 1) return LINNE_APIRESULT_PARAMETER_NOT_SET;
    if (num_samples > enc->header.num_samples_per_block) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
    return upload_and_encode(enc, input, num_samples, data, data_size, NULL, output_size);
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
    struct LINNEEncoder *parent, *child;
    const int32_t *const *input;           /* int32 planes, or ... */
    const uint8_t *packed;                 /* ... interleaved packed PCM (WAV data-chunk layout) */
    uint32_t first_sample, num_samples;
    uint32_t size, offset;                 /* shard bytes (blocks only) / where they go in the caller's buffer */
    uint8_t *data;
    LINNEApiResult result;
    LnbRendezvous *meet;
    int ordinal;
};

static void *enc_shard_main(void *arg)
{
    struct LnbEncShard *sh = (struct LnbEncShard *)arg;
    struct LINNEEncoder *enc = sh->child;
    const uint32_t C = enc->header.num_channels;
    const size_t stride = LNB_ROUNDUP((size_t)sh->num_samples + 4u, 4u);
    /* worst case of a shard: every block stored raw (linne_encoder.c:556-585) */
    const size_t NB = enc->header.num_samples_per_block, blocks = (sh->num_samples + NB - 1u) / NB;
    const size_t cap = blocks * (LNB_BLOCK_HEADER_SIZE + NB * C * ((enc->header.bits_per_sample + 7u) / 8u)) + 64u;
    uint32_t c, written = 0;
    sh->result = LINNE_APIRESULT_OK;
    sh->size = 0;
    lnb_shim_set_device(sh->ordinal);
    if (cap > 0xFFFFFF00u || lnb_buf_reserve_device(enc->dev, &enc->d_pcm, stride * C * sizeof(int32_t))
        || lnb_buf_reserve_device(enc->dev, &enc->d_shard, cap)) sh->result = LINNE_APIRESULT_NG;
    if (sh->result == LINNE_APIRESULT_OK && sh->packed) {
        const uint32_t bytes = enc->header.bits_per_sample / 8u;
        const size_t frame = (size_t)C * bytes;
        if (lnb_buf_reserve_device(enc->dev, &enc->d_packed, (size_t)sh->num_samples * frame + 16u)) sh->result = LINNE_APIRESULT_NG;
        else {
            lnb_shim_h2d(enc->dev, enc->d_packed.ptr, sh->packed + (size_t)sh->first_sample * frame, (size_t)sh->num_samples * frame);
            if (lnb_shim_unpack_pcm(enc->dev, (const uint8_t *)enc->d_packed.ptr, (int32_t *)enc->d_pcm.ptr, (uint32_t)stride,
                                    sh->num_samples, C, bytes)) sh->result = LINNE_APIRESULT_NG;
        }
    }
    if (sh->result == LINNE_APIRESULT_OK) {
        for (c = 0; c < C && !sh->packed; c++)
            lnb_shim_h2d(enc->dev, (int32_t *)enc->d_pcm.ptr + c * stride, sh->input[c] + sh->first_sample, (size_t)sh->num_samples * sizeof(int32_t));
        enc->cur_pcm = (const int32_t *)enc->d_pcm.ptr;
        enc->cur_pcm_stride = (uint32_t)stride;
        sh->result = encode_blocks(enc, sh->num_samples, (uint8_t *)enc->d_shard.ptr, (uint32_t)cap, 1, NULL, &written);
        sh->size = written;
    }
    lnb_rendezvous_report_and_wait(sh->meet);   /* every shard's size is known: the caller scans them and says where each goes */
    if (sh->result == LINNE_APIRESULT_OK && sh->data) {
        lnb_shim_d2h(enc->dev, sh->data + sh->offset, enc->d_shard.ptr, sh->size);
        if (lnb_shim_sync(enc->dev)) sh->result = LINNE_APIRESULT_NG;
    }
    return NULL;
}

/* EncodeWhole over enc->num_devices block ranges; `data` starts behind the stream header */
static LINNEApiResult encode_whole_sharded(struct LINNEEncoder *enc, const int32_t *const *input, const uint8_t *packed, uint32_t num_samples,
                                           uint8_t *data, uint32_t data_size, uint32_t *written)
{
    const uint32_t NB = enc->header.num_samples_per_block;
    const uint32_t total_blocks = (uint32_t)(((uint64_t)num_samples + NB - 1u) / NB);
    const uint32_t G = lnb_plan_ranges(total_blocks, enc->num_devices > 1u ? enc->num_devices : 1u);
    const int ndev = lnb_shim_device_count();
    const uint32_t ndev_used = enc->num_devices > 1u ? (enc->num_devices < (uint32_t)(ndev > 0 ? ndev : 1) ? enc->num_devices : (uint32_t)(ndev > 0 ? ndev : 1)) : 1u;
    const int own = lnb_shim_device_ordinal(enc->dev);
    struct LnbEncShard sh[LNB_MAX_DEVICES];
    pthread_t th[LNB_MAX_DEVICES];
    LnbRendezvous meet;
    struct LINNEEncodeParameter prm;
    LINNEApiResult ret = LINNE_APIRESULT_OK;
    uint32_t k, started = 0, off = 0;
    int home = -1;
    if (ndev <= 0) return LINNE_APIRESULT_NG;
    home = lnb_shim_current_device();
    prm.num_channels = enc->header.num_channels; prm.bits_per_sample = enc->header.bits_per_sample;
    prm.sampling_rate = enc->header.sampling_rate; prm.num_samples_per_block = (uint16_t)NB;
    prm.preset = enc->header.preset; prm.ch_process_method = enc->header.ch_process_method;
    prm.enable_learning = enc->enable_learning; prm.num_afmethod_iterations = enc->num_afmethod_iterations;
    for (k = 0; k < G; k++) {
        if (!enc->child[k]) {
            lnb_shim_set_device(enc->num_devices > 1u ? (int)(k % ndev_used) : own);
            enc->child[k] = LINNEEncoder_Create(&enc->config, NULL, 0);
            if (enc->child[k]) enc->child[k]->num_devices = 0;          /* children never shard again */
        }
        if (!enc->child[k] || LINNEEncoder_SetEncodeParameter(enc->child[k], &prm) != LINNE_APIRESULT_OK) { ret = LINNE_APIRESULT_NG; break; }
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
        sh[k].parent = enc; sh[k].child = enc->child[k]; sh[k].input = input; sh[k].packed = packed;
        sh[k].first_sample = (uint32_t)s0;
        sh[k].num_samples = (uint32_t)((s1 > num_samples ? num_samples : s1) - s0);
        sh[k].child->header.num_samples = sh[k].num_samples;
        sh[k].data = data; sh[k].meet = &meet;
        sh[k].ordinal = enc->num_devices > 1u ? (int)(k % ndev_used) : own;
        if (pthread_create(&th[k], NULL, enc_shard_main, &sh[k]) != 0) { sh[k].result = LINNE_APIRESULT_NG; break; }
        started++;
    }
    lnb_rendezvous_collect(&meet, started);
    for (k = 0; k < started; k++) {                                /* exclusive scan of the shard byte counts */
        if (sh[k].result != LINNE_APIRESULT_OK && ret == LINNE_APIRESULT_OK) ret = sh[k].result;
        sh[k].offset = off;
        off += sh[k].size;
    }
    if (ret == LINNE_APIRESULT_OK && (started < G || off > data_size)) ret = (started < G) ? LINNE_APIRESULT_NG : LINNE_APIRESULT_INSUFFICIENT_BUFFER;
    if (ret != LINNE_APIRESULT_OK) for (k = 0; k < started; k++) sh[k].data = NULL;
    lnb_rendezvous_release(&meet);
    for (k = 0; k < started; k++) {
        pthread_join(th[k], NULL);
        if (sh[k].result != LINNE_APIRESULT_OK && ret == LINNE_APIRESULT_OK) ret = sh[k].result;
    }
    lnb_rendezvous_destroy(&meet);
    *written = off;
    return ret;
}

/* reference linne_encoder.c:865-932 */
LINNEApiResult LINNEEncoder_EncodeWhole(struct LINNEEncoder *enc, const int32_t *const *input, uint32_t num_samples,
        uint8_t *data, uint32_t data_size, uint32_t *output_size)
{
    LINNEApiResult ret;
    uint32_t written = 0;
    if (enc == NULL || input == NULL || data == NULL || output_size == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (enc->set_parameter != 1) return LINNE_APIRESULT_PARAMETER_NOT_SET;
    enc->header.num_samples = num_samples;
    if ((ret = LINNEEncoder_EncodeHeader(&enc->header, data, data_size)) != LINNE_APIRESULT_OK) return ret;
    /* several devices, or a stream long enough to pipeline its transfers against its kernels on one */
    if (lnb_plan_ranges((uint32_t)(((uint64_t)num_samples + enc->header.num_samples_per_block - 1u) / enc->header.num_samples_per_block),
                        enc->num_devices > 1u ? enc->num_devices : 1u) > 1u) {
        uint32_t c;
        for (c = 0; c < enc->header.num_channels; c++) if (input[c] == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
        ret = encode_whole_sharded(enc, input, NULL, num_samples, data + LINNE_HEADER_SIZE, data_size - LINNE_HEADER_SIZE, &written);
    } else {
        ret = upload_and_encode(enc, input, num_samples, data + LINNE_HEADER_SIZE, data_size - LINNE_HEADER_SIZE, NULL, &written);
    }
    if (ret != LINNE_APIRESULT_OK) return ret;
    *output_size = LINNE_HEADER_SIZE + written;
    return LINNE_APIRESULT_OK;
}

LnbDevice *lnb_encoder_device(const struct LINNEEncoder *enc) { return enc->dev; }

/* ---- extension entry points (include/linne_b200.h) ---- */
#include "linne_b200.h"

LINNEApiResult LINNEB200_EncodeWholeWithParams(struct LINNEEncoder *enc, const int32_t *const *input,
        uint32_t num_samples, const struct LINNEB200ChannelParams *params, uint32_t num_param_blocks,
        uint8_t *data, uint32_t data_size, uint32_t *output_size)
{
    LINNEApiResult ret;
    LnbChanParams *forced;
    uint32_t written = 0, blocks, i, l, C;
    if (enc == NULL || input == NULL || params == NULL || data == NULL || output_size == NULL)
        return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (enc->set_parameter != 1) return LINNE_APIRESULT_PARAMETER_NOT_SET;
    C = enc->header.num_channels;
    blocks = (num_samples + enc->header.num_samples_per_block - 1u) / enc->header.num_samples_per_block;
    if (num_param_blocks < blocks) return LINNE_APIRESULT_INVALID_ARGUMENT;
    /* the stream stores these in 3 and 4 bits: a larger value would be written masked but predicted with unmasked */
    for (i = 0; i < blocks * C; i++)
        for (l = 0; l < (uint32_t)g_lnb_presets[enc->header.preset].num_layers; l++)
            if (params[i].log2_units[l] > 7u || params[i].rshift[l] > 15u) return LINNE_APIRESULT_INVALID_ARGUMENT;
    enc->header.num_samples = num_samples;
    if ((ret = LINNEEncoder_EncodeHeader(&enc->header, data, data_size)) != LINNE_APIRESULT_OK) return ret;
    forced = (LnbChanParams *)calloc((size_t)blocks * C, sizeof(LnbChanParams));
    if (!forced) return LINNE_APIRESULT_NG;
    for (i = 0; i < blocks * C; i++)
        for (l = 0; l < LNB_MAX_LAYERS; l++) {
            forced[i].log2_units[l] = params[i].log2_units[l];
            forced[i].rshift[l] = params[i].rshift[l];
            memcpy(forced[i].coef + l * LNB_MAX_PARAMS, params[i].coef[l], LNB_MAX_PARAMS);
        }
    ret = upload_and_encode(enc, input, num_samples, data + LINNE_HEADER_SIZE, data_size - LINNE_HEADER_SIZE, forced, &written);
    free(forced);
    if (ret != LINNE_APIRESULT_OK) return ret;
    *output_size = LINNE_HEADER_SIZE + written;
    return LINNE_APIRESULT_OK;
}

LINNEApiResult LINNEB200_EncodeWholeResident(struct LINNEEncoder *enc, const int32_t *d_pcm, uint32_t pcm_stride,
        uint32_t num_samples, uint8_t *d_data, uint32_t data_size, uint32_t *output_size)
{
    uint8_t hdr[LINNE_HEADER_SIZE];
    LINNEApiResult ret;
    uint32_t written = 0;
    if (enc == NULL || d_pcm == NULL || d_data == NULL || output_size == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (enc->set_parameter != 1) return LINNE_APIRESULT_PARAMETER_NOT_SET;
    if (pcm_stride < num_samples) return LINNE_APIRESULT_INVALID_ARGUMENT;
    enc->header.num_samples = num_samples;
    if (data_size < LINNE_HEADER_SIZE) return LINNE_APIRESULT_INSUFFICIENT_BUFFER;
    if ((ret = LINNEEncoder_EncodeHeader(&enc->header, hdr, sizeof(hdr))) != LINNE_APIRESULT_OK) return ret;
    lnb_shim_h2d(enc->dev, d_data, hdr, LINNE_HEADER_SIZE);
    enc->cur_pcm = d_pcm;
    enc->cur_pcm_stride = pcm_stride;
    ret = encode_blocks(enc, num_samples, d_data + LINNE_HEADER_SIZE, data_size - LINNE_HEADER_SIZE, 1, NULL, &written);
    if (ret != LINNE_APIRESULT_OK) return ret;
    *output_size = LINNE_HEADER_SIZE + written;
    return LINNE_APIRESULT_OK;
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
    uint32_t written = 0, i, blocks = 0, NB;
    if (enc == NULL || d_pcm == NULL || files == NULL || num_files == 0 || d_data == NULL || output_size == NULL)
        return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (enc->set_parameter != 1) return LINNE_APIRESULT_PARAMETER_NOT_SET;
    NB = enc->header.num_samples_per_block;
    if (!(ranges = (struct LnbFileRange *)malloc((size_t)num_files * sizeof(*ranges)))) return LINNE_APIRESULT_NG;
    for (i = 0; i < num_files; i++) {
        if (files[i].num_samples == 0 || (uint64_t)files[i].first_sample + files[i].num_samples > pcm_stride) { free(ranges); return LINNE_APIRESULT_INVALID_ARGUMENT; }
        ranges[i].first_sample = files[i].first_sample; ranges[i].num_samples = files[i].num_samples;
        ranges[i].first_block = blocks;
        ranges[i].num_blocks = (uint32_t)(((uint64_t)files[i].num_samples + NB - 1u) / NB);
        blocks += ranges[i].num_blocks;
        files[i].out_offset = files[i].out_size = 0;
    }
    if (lnb_buf_reserve_host(&enc->h_headers, (size_t)num_files * 32u)) { free(ranges); return LINNE_APIRESULT_NG; }
    enc->ranges = ranges; enc->num_ranges = num_files; enc->file_out = files;
    enc->cur_pcm = d_pcm; enc->cur_pcm_stride = pcm_stride;
    enc->header.num_samples = files[0].num_samples;
    ret = encode_blocks(enc, 0, d_data, data_size, 2, NULL, &written);
    enc->ranges = NULL; enc->num_ranges = 0; enc->file_out = NULL;
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
    uint64_t total = 0, bound = 0;
    uint32_t i, C, bytes, written = 0, NB;
    size_t stride, packed_bytes;
    if (enc == NULL || pcm == NULL || files == NULL || num_files == 0 || data == NULL || output_size == NULL)
        return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (enc->set_parameter != 1) return LINNE_APIRESULT_PARAMETER_NOT_SET;
    C = enc->header.num_channels; NB = enc->header.num_samples_per_block;
    bytes = enc->header.bits_per_sample / 8u;
    if (bytes == 0 || bytes > 4u || (enc->header.bits_per_sample % 8u) != 0u) return LINNE_APIRESULT_INVALID_FORMAT;
    for (i = 0; i < num_files; i++) {
        if (files[i].num_samples == 0) return LINNE_APIRESULT_INVALID_ARGUMENT;
        files[i].first_sample = (uint32_t)total;
        total += files[i].num_samples;
        /* no stream is longer than its raw form plus framing (blocks that would be are stored raw) -- with slack */
        bound += LINNE_HEADER_SIZE + 2u * ((uint64_t)files[i].num_samples * C * bytes + 16u * (files[i].num_samples / NB + 2u)) + 4096u;
    }
    if (total > 0xFFFFFFF0ull) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (bound > data_size) bound = data_size;
    stride = LNB_ROUNDUP((size_t)total + 4u, 4u);
    packed_bytes = (size_t)total * C * bytes;
    if (lnb_buf_reserve_device(enc->dev, &enc->d_pcm, stride * C * sizeof(int32_t))
        || lnb_buf_reserve_device(enc->dev, &enc->d_packed, packed_bytes + 16u)
        || lnb_buf_reserve_device(enc->dev, &enc->d_image, (size_t)bound + 64u)) return LINNE_APIRESULT_NG;
    lnb_shim_h2d(enc->dev, enc->d_packed.ptr, pcm, packed_bytes);
    if (lnb_shim_unpack_pcm(enc->dev, (const uint8_t *)enc->d_packed.ptr, (int32_t *)enc->d_pcm.ptr, (uint32_t)stride,
                            (uint32_t)total, C, bytes)) return LINNE_APIRESULT_NG;
    ret = LINNEB200_EncodeFilesResident(enc, (const int32_t *)enc->d_pcm.ptr, (uint32_t)stride, files, num_files,
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
    LINNEApiResult ret;
    uint32_t written = 0, C, bytes;
    size_t stride, packed_bytes;
    if (enc == NULL || pcm == NULL || data == NULL || output_size == NULL) return LINNE_APIRESULT_INVALID_ARGUMENT;
    if (enc->set_parameter != 1) return LINNE_APIRESULT_PARAMETER_NOT_SET;
    C = enc->header.num_channels;
    bytes = enc->header.bits_per_sample / 8u;
    if (bytes == 0 || bytes > 4u || (enc->header.bits_per_sample % 8u) != 0u) return LINNE_APIRESULT_INVALID_FORMAT;
    enc->header.num_samples = num_samples;
    if ((ret = LINNEEncoder_EncodeHeader(&enc->header, data, data_size)) != LINNE_APIRESULT_OK) return ret;
    if (lnb_plan_ranges((uint32_t)(((uint64_t)num_samples + enc->header.num_samples_per_block - 1u) / enc->header.num_samples_per_block),
                        enc->num_devices > 1u ? enc->num_devices : 1u) > 1u) {
        ret = encode_whole_sharded(enc, NULL, pcm, num_samples, data + LINNE_HEADER_SIZE, data_size - LINNE_HEADER_SIZE, &written);
        if (ret != LINNE_APIRESULT_OK) return ret;
        *output_size = LINNE_HEADER_SIZE + written;
        return LINNE_APIRESULT_OK;
    }
    stride = LNB_ROUNDUP((size_t)num_samples + 4u, 4u);
    packed_bytes = (size_t)num_samples * C * bytes;
    if (lnb_buf_reserve_device(enc->dev, &enc->d_pcm, stride * C * sizeof(int32_t))
        || lnb_buf_reserve_device(enc->dev, &enc->d_packed, packed_bytes + 16u)) return LINNE_APIRESULT_NG;
    lnb_shim_h2d(enc->dev, enc->d_packed.ptr, pcm, packed_bytes);
    if (lnb_shim_unpack_pcm(enc->dev, (const uint8_t *)enc->d_packed.ptr, (int32_t *)enc->d_pcm.ptr, (uint32_t)stride,
                            num_samples, C, bytes)) return LINNE_APIRESULT_NG;
    enc->cur_pcm = (const int32_t *)enc->d_pcm.ptr;
    enc->cur_pcm_stride = (uint32_t)stride;
    ret = encode_blocks(enc, num_samples, data + LINNE_HEADER_SIZE, data_size - LINNE_HEADER_SIZE, 0, NULL, &written);
    if (ret != LINNE_APIRESULT_OK) return ret;
    *output_size = LINNE_HEADER_SIZE + written;
    return LINNE_APIRESULT_OK;
}
