/* lnb_host_util.c -- header (de)serialisation and buffer helpers for the host side. */
#include "lnb_host_util.h"
#include <stdlib.h>
#include <string.h>

int lnb_buf_reserve_device(LnbDevice *dev, LnbBuf *buf, size_t bytes)
{
    if (buf->cap >= bytes && buf->ptr) return 0;
    if (buf->ptr) { lnb_shim_free(dev, buf->ptr); buf->ptr = NULL; buf->cap = 0; }
    bytes = LNB_ROUNDUP(bytes + 256, 256);
    buf->ptr = lnb_shim_alloc(dev, bytes);
    if (!buf->ptr) return 1;
    buf->cap = bytes;
    return 0;
}
void lnb_buf_release_device(LnbDevice *dev, LnbBuf *buf)
{
    if (buf->ptr) lnb_shim_free(dev, buf->ptr);
    buf->ptr = NULL; buf->cap = 0;
}
int lnb_buf_reserve_host(LnbBuf *buf, size_t bytes)
{
    if (buf->cap >= bytes && buf->ptr) return 0;
    if (buf->ptr) { lnb_shim_free_pinned(buf->ptr); buf->ptr = NULL; buf->cap = 0; }
    bytes = LNB_ROUNDUP(bytes + 256, 256);
    buf->ptr = lnb_shim_alloc_pinned(bytes);
    if (!buf->ptr) return 1;
    buf->cap = bytes;
    return 0;
}
void lnb_buf_release_host(LnbBuf *buf)
{
    if (buf->ptr) lnb_shim_free_pinned(buf->ptr);
    buf->ptr = NULL; buf->cap = 0;
}

/* Field checks in the order of reference linne_encoder.c:68-102. */
LINNEApiResult lnb_header_check_for_encode(const struct LINNEHeader *h)
{
    if (h->num_channels == 0 || h->num_samples == 0 || h->sampling_rate == 0 || h->bits_per_sample == 0
        || h->num_samples_per_block == 0) return LINNE_APIRESULT_INVALID_FORMAT;
    /* The pre-emphasis state travels in bits_per_sample + 1 bits and the reference's bit reader/writer take at
     * most 32 bits per field (bit_stream.h:317 asserts it, a Release build shifts out of range), so 32-bit PCM
     * never worked there; refuse it instead of writing or reading a field nobody can parse. */
    if (h->bits_per_sample > LNB_MAX_BITS_PER_SAMPLE) return LINNE_APIRESULT_INVALID_FORMAT;
    if (h->preset >= LINNE_NUM_PARAMETER_PRESETS) return LINNE_APIRESULT_INVALID_FORMAT;
    if ((unsigned)h->ch_process_method >= (unsigned)LINNE_CH_PROCESS_METHOD_INVALID) return LINNE_APIRESULT_INVALID_FORMAT;
    if (h->ch_process_method == LINNE_CH_PROCESS_METHOD_MS && h->num_channels == 1) return LINNE_APIRESULT_INVALID_FORMAT;
    return LINNE_APIRESULT_OK;
}

/* reference linne_decoder.c:134-184 */
int lnb_header_fields_valid(const struct LINNEHeader *h)
{
    if (h->format_version != LINNE_FORMAT_VERSION || h->codec_version != LINNE_CODEC_VERSION) return 0;
    return lnb_header_check_for_encode(h) == LINNE_APIRESULT_OK;
}

static void wr_be(uint8_t **p, uint32_t v, int n) { int i; for (i = n - 1; i >= 0; i--) *(*p)++ = (uint8_t)(v >> (8 * i)); }

/* layout: reference linne_encoder.c:107-131 */
void lnb_header_write(const struct LINNEHeader *h, uint8_t *dst)
{
    uint8_t *p = dst;
    *p++ = 'I'; *p++ = 'B'; *p++ = 'R'; *p++ = 'A';
    wr_be(&p, LINNE_FORMAT_VERSION, 4);
    wr_be(&p, LINNE_CODEC_VERSION, 4);
    wr_be(&p, h->num_channels, 2);
    wr_be(&p, h->num_samples, 4);
    wr_be(&p, h->sampling_rate, 4);
    wr_be(&p, h->bits_per_sample, 2);
    wr_be(&p, h->num_samples_per_block, 4);
    wr_be(&p, h->preset, 1);
    wr_be(&p, (uint32_t)h->ch_process_method, 1);
}

/* reference linne_decoder.c:97-123 */
void lnb_header_read(const uint8_t *src, struct LINNEHeader *h)
{
    h->format_version = lnb_rd_be(src + 4, 4);
    h->codec_version = lnb_rd_be(src + 8, 4);
    h->num_channels = (uint16_t)lnb_rd_be(src + 12, 2);
    h->num_samples = lnb_rd_be(src + 14, 4);
    h->sampling_rate = lnb_rd_be(src + 18, 4);
    h->bits_per_sample = (uint16_t)lnb_rd_be(src + 22, 2);
    h->num_samples_per_block = lnb_rd_be(src + 24, 4);
    h->preset = (uint8_t)src[28];
    h->ch_process_method = (LINNEChannelProcessMethod)src[29];
}

void lnb_fill_stream_cfg(LnbStreamCfg *cfg, const struct LINNEHeader *h)
{
    const LnbPreset *ps = &g_lnb_presets[h->preset];
    int i;
    memset(cfg, 0, sizeof(*cfg));
    cfg->num_channels = h->num_channels;
    cfg->bits_per_sample = h->bits_per_sample;
    cfg->block_size = h->num_samples_per_block;
    cfg->num_layers = (uint32_t)ps->num_layers;
    for (i = 0; i < ps->num_layers; i++) cfg->layer_params[i] = (uint32_t)ps->layer_params[i];
    cfg->num_lambdas = (uint32_t)ps->num_lambdas;
    for (i = 0; i < ps->num_lambdas; i++) cfg->lambdas[i] = ps->lambdas[i];
    cfg->ms = (h->ch_process_method == LINNE_CH_PROCESS_METHOD_MS) ? 1u : 0u;
}

void lnb_rendezvous_init(LnbRendezvous *r)
{
    pthread_mutex_init(&r->lock, NULL); pthread_cond_init(&r->cv, NULL); r->reported = 0; r->released = 0;
}
void lnb_rendezvous_destroy(LnbRendezvous *r) { pthread_cond_destroy(&r->cv); pthread_mutex_destroy(&r->lock); }
void lnb_rendezvous_report_and_wait(LnbRendezvous *r)
{
    pthread_mutex_lock(&r->lock);
    r->reported++;
    pthread_cond_broadcast(&r->cv);
    while (!r->released) pthread_cond_wait(&r->cv, &r->lock);
    pthread_mutex_unlock(&r->lock);
}
void lnb_rendezvous_collect(LnbRendezvous *r, uint32_t workers)
{
    pthread_mutex_lock(&r->lock);
    while (r->reported < workers) pthread_cond_wait(&r->cv, &r->lock);
    pthread_mutex_unlock(&r->lock);
}
void lnb_rendezvous_release(LnbRendezvous *r)
{
    pthread_mutex_lock(&r->lock);
    r->released = 1;
    pthread_cond_broadcast(&r->cv);
    pthread_mutex_unlock(&r->lock);
}

void lnb_turnstile_init(LnbTurnstile *t, uint32_t stride)
{
    pthread_mutex_init(&t->lock, NULL); pthread_cond_init(&t->cv, NULL);
    t->stride = stride ? stride : 1u;
    memset(t->passed, 0, sizeof(t->passed));
}
void lnb_turnstile_destroy(LnbTurnstile *t) { pthread_cond_destroy(&t->cv); pthread_mutex_destroy(&t->lock); }
void lnb_turnstile_wait(LnbTurnstile *t, int phase, uint32_t k)
{
    if (k < t->stride || k >= LNB_MAX_DEVICES) return;
    pthread_mutex_lock(&t->lock);
    while (!t->passed[phase][k - t->stride]) pthread_cond_wait(&t->cv, &t->lock);
    pthread_mutex_unlock(&t->lock);
}
void lnb_turnstile_pass(LnbTurnstile *t, int phase, uint32_t k)
{
    if (k >= LNB_MAX_DEVICES) return;
    pthread_mutex_lock(&t->lock);
    t->passed[phase][k] = 1;
    pthread_cond_broadcast(&t->cv);
    pthread_mutex_unlock(&t->lock);
}

uint32_t lnb_plan_ranges(uint32_t blocks, uint32_t devices)
{
    const char *e = getenv("LINNE_B200_PIPELINE");
    uint32_t depth, ranges;
    if (devices < 1u) devices = 1u;
    if (e && *e) {
        depth = (uint32_t)strtoul(e, NULL, 10);
        if (depth < 1u) depth = 1u;
    } else {
        const uint32_t per_device = blocks / devices;
        depth = per_device >= 6144u ? 4u : (per_device >= 3072u ? 2u : 1u);      /* measured on a 1-hour stream: 8 ranges gain nothing over 4 */
    }
    ranges = devices * depth;
    if (ranges > LNB_MAX_DEVICES) ranges = LNB_MAX_DEVICES;
    if (ranges * 2u > blocks) ranges = blocks / 2u;              /* at least two blocks per range */
    return ranges < 1u ? 1u : ranges;
}

uint32_t lnb_place_ranges(uint32_t requested, int visible, int own, uint32_t G, int *ordinal)
{
    const uint32_t used = requested > 1u ? (requested < (uint32_t)visible ? requested : (uint32_t)visible) : 1u;
    uint32_t k;
    for (k = 0; k < G; k++) ordinal[k] = requested > 1u ? (int)(k % used) : own;
    return used;
}
