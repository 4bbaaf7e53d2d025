/* linne_b200 -- batch command-line driver on top of the LINNE C API as served by liblinne_b200.so.
 *
 * SURVEY section 8(f).1: a `linne`-compatible tool (reference tools/linne_codec/linne_codec.c: same
 * -e / -d / -m / -l / -a / -c options, same WAV <-> .lnn mapping, same encoder settings: block 10240,
 * mid/side for >= 2 channels) that
 *   - encodes / decodes a whole FILE per call (LINNEB200_EncodeWholePacked / DecodeWholePacked: the WAV data
 *     chunk goes to the device as it is and is converted there), so every block x channel of a file is one
 *     GPU batch (the reference tool encodes block by block through int32 planes), and
 *   - takes any number of input/output pairs, or a list file, and
 *   - runs them through an asynchronous file pipeline (SURVEY section 8(f).3; the reference tool reads, codes and
 *     writes one file after the other, linne_codec.c:89-105,215-222): `-j N` workers, each with its own handle
 *     (its own CUDA stream) and its own page-locked staging buffers, pull files from a shared queue, so one
 *     worker's disk read / write and its DMA transfers overlap with the kernels of the others.
 * WAV sample conventions follow reference libs/wav/src/wav.c:388-414 and :665-700 (8-bit is unsigned with
 * a bias of 128; 16/24/32-bit little-endian signed); samples are handed to the codec right-justified
 * (linne_codec.c:100-105) and written back the same way (:262-268).
 *
 *   linne_b200 -e [-m 0..7] [-l] [-a N] in.wav out.lnn [in2.wav out2.lnn ...]
 *   linne_b200 -d [-c] [--start FRAME] [--length FRAMES]  in.lnn out.wav [in2.lnn out2.wav ...]
 *   linne_b200 -d -F in.lnn out.wav [...]   (decode through damage)
 *   linne_b200 -e|-d ... -L pairs.txt   (one "input output" pair per line)
 *   -j N  workers (default: min(4, files))      -s  print a timing summary (samples, seconds, MSamples/s)
 *
 * --start / --length cut the same excerpt of every stream of a -d run: frames [FRAME, FRAME + FRAMES), to the end of the
 * stream when --length is not given.  Each file is indexed (LINNEB200_DecoderBuildIndex) and only the blocks the excerpt
 * overlaps are decoded, in one LINNEB200_DecodeWindowsPacked call straight into the WAV staging buffer.  An excerpt that
 * does not lie inside a stream fails that file, and nothing is written for it.
 *
 * -F decodes through damage (LINNEB200_DecodeSalvagePacked): every intact block lands where it belongs in a WAV of the
 * stream's full length, what was lost is silence, and each lost run is reported on stderr as
 * "in.lnn: frames [a, b) lost, bytes [x, y): STATUS".  The stream's own 30-byte header must be readable.  The exit code is
 * 2 when a file was damaged (and none failed), 1 when one failed, 0 otherwise.  -F does not combine with --start / --length.
 */
#define _POSIX_C_SOURCE 200809L
#include <linne_encoder.h>
#include <linne_decoder.h>
#include <linne_b200.h>

#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#define CLI_BLOCK 10240u                       /* linne_codec.c:75 */
#define CLI_MAX_BLOCK (16u * 1024u)            /* linne_codec.c:54 */

/* grow-only page-locked buffer (LINNEB200_HostAlloc): what lands here goes to the device by DMA */
struct Staging { uint8_t *ptr; size_t cap; };

static uint8_t *staging_reserve(struct Staging *s, size_t bytes)
{
    if (s->cap < bytes || !s->ptr) {
        if (s->ptr) LINNEB200_HostFree(s->ptr);
        s->cap = bytes + bytes / 4u + 4096u;
        s->ptr = (uint8_t *)LINNEB200_HostAlloc(s->cap);
        if (!s->ptr) s->cap = 0;
    }
    return s->ptr;
}
static void staging_release(struct Staging *s) { if (s->ptr) LINNEB200_HostFree(s->ptr); s->ptr = NULL; s->cap = 0; }

struct Wav {
    uint32_t channels, rate, bits, frames;
    const uint8_t *data;                       /* interleaved little-endian samples inside the file image */
};

/* one pipeline worker: a handle and its staging buffers, reused for every file the worker takes */
struct Worker {
    struct LINNEEncoder *enc;
    struct LINNEDecoder *dec;
    struct Staging in, out;
    struct LINNEB200SeekPoint *points;         /* seek index of the current stream (excerpts), grow-only */
    uint32_t points_cap;
    struct LINNEB200Damage *damage;            /* salvage records of the current stream (-F), grow-only */
    uint32_t damage_cap;
    int damaged;                               /* files decoded through damage */
    uint64_t samples;                          /* samples (frames x channels) that went through */
    int failures;
};

static uint32_t rd_le(const uint8_t *p, int n) { uint32_t v = 0; int i; for (i = n - 1; i >= 0; i--) v = (v << 8) | p[i]; return v; }
static void wr_le(uint8_t *p, uint32_t v, int n) { int i; for (i = 0; i < n; i++) p[i] = (uint8_t)(v >> (8 * i)); }

static uint8_t *read_file(const char *path, struct Staging *st, size_t *size)
{
    FILE *fp = fopen(path, "rb");
    uint8_t *buf;
    long n;
    if (!fp) return NULL;
    if (fseek(fp, 0, SEEK_END) != 0 || (n = ftell(fp)) < 0 || fseek(fp, 0, SEEK_SET) != 0) { fclose(fp); return NULL; }
    buf = staging_reserve(st, (size_t)n + 16u);
    if (buf && fread(buf, 1, (size_t)n, fp) != (size_t)n) buf = NULL;
    fclose(fp);
    *size = (size_t)n;
    return buf;
}

/* RIFF/WAVE, PCM (format tag 1, or WAVE_FORMAT_EXTENSIBLE carrying PCM), 8/16/24 bits (the format's
 * (bits + 1)-bit pre-emphasis field rules out 32, as in the reference: bit_stream.h:317) */
static int wav_read(const char *path, struct Staging *st, struct Wav *w)
{
    size_t size = 0, off = 12, data_off = 0, data_len = 0;
    uint8_t *f = read_file(path, st, &size);
    uint32_t bytes, have_fmt = 0;
    memset(w, 0, sizeof(*w));
    if (!f || size < 12 || memcmp(f, "RIFF", 4) != 0 || memcmp(f + 8, "WAVE", 4) != 0) return 1;
    while (off + 8 <= size) {
        const uint32_t len = rd_le(f + off + 4, 4);
        const uint8_t *body = f + off + 8;
        if (memcmp(f + off, "fmt ", 4) == 0 && len >= 16 && off + 8 + len <= size) {
            uint32_t tag = rd_le(body, 2);
            if (tag == 0xFFFEu && len >= 26) tag = rd_le(body + 24, 2);
            if (tag != 1u) return 2;
            w->channels = rd_le(body + 2, 2); w->rate = rd_le(body + 4, 4); w->bits = rd_le(body + 14, 2);
            have_fmt = 1;
        } else if (memcmp(f + off, "data", 4) == 0) {
            data_off = off + 8;
            data_len = (off + 8 + len <= size) ? len : size - (off + 8);
            break;
        }
        off += 8 + (size_t)len + (len & 1u);
    }
    bytes = w->bits / 8u;
    if (!have_fmt || !data_off || w->channels == 0 || w->channels > LINNE_MAX_NUM_CHANNELS
        || (w->bits != 8 && w->bits != 16 && w->bits != 24)) return 3;
    w->frames = (uint32_t)(data_len / ((size_t)bytes * w->channels));
    w->data = f + data_off;
    return 0;
}

/* canonical 44-byte header + data chunk; `buf` = 44 bytes of room followed by the samples */
static int wav_write(const char *path, uint8_t *buf, const struct Wav *w)
{
    const uint32_t bytes = w->bits / 8u;
    const size_t data_len = (size_t)w->frames * w->channels * bytes;
    FILE *fp;
    int rc = 0;
    memcpy(buf, "RIFF", 4); wr_le(buf + 4, (uint32_t)(36u + data_len), 4); memcpy(buf + 8, "WAVEfmt ", 8);
    wr_le(buf + 16, 16, 4); wr_le(buf + 20, 1, 2); wr_le(buf + 22, w->channels, 2); wr_le(buf + 24, w->rate, 4);
    wr_le(buf + 28, w->rate * w->channels * bytes, 4); wr_le(buf + 32, w->channels * bytes, 2); wr_le(buf + 34, w->bits, 2);
    memcpy(buf + 36, "data", 4); wr_le(buf + 40, (uint32_t)data_len, 4);
    if (!(fp = fopen(path, "wb"))) return 2;
    if (fwrite(buf, 1, 44u + data_len, fp) != 44u + data_len) rc = 3;
    fclose(fp);
    return rc;
}

struct Options {
    int encode, decode, preset, learning, af, no_crc, jobs, stats;
    int excerpt, has_length;                   /* --start and/or --length given; --length given */
    int salvage;                               /* -F: decode through damage */
    uint32_t start, length;
    const char *list;
};

static pthread_mutex_t g_print = PTHREAD_MUTEX_INITIALIZER;
#define SAY(stream, ...) do { pthread_mutex_lock(&g_print); fprintf(stream, __VA_ARGS__); pthread_mutex_unlock(&g_print); } while (0)

static int encode_one(struct Worker *wk, const struct Options *o, const char *in, const char *out)
{
    struct Wav w;
    struct LINNEEncodeParameter prm;
    uint8_t *buf;
    uint32_t cap, size = 0;
    LINNEApiResult ret;
    FILE *fp;
    int rc;
    if ((rc = wav_read(in, &wk->in, &w)) != 0) { SAY(stderr, "linne_b200: cannot read %s (%d)\n", in, rc); return 1; }
    prm.num_channels = (uint16_t)w.channels;
    prm.bits_per_sample = (uint16_t)w.bits;
    prm.sampling_rate = w.rate;
    prm.num_samples_per_block = (uint16_t)CLI_BLOCK;
    prm.preset = (uint8_t)o->preset;
    prm.ch_process_method = (w.channels >= 2) ? LINNE_CH_PROCESS_METHOD_MS : LINNE_CH_PROCESS_METHOD_NONE;
    prm.enable_learning = (uint8_t)o->learning;
    prm.num_afmethod_iterations = (uint8_t)o->af;
    if ((ret = LINNEEncoder_SetEncodeParameter(wk->enc, &prm)) != LINNE_APIRESULT_OK) {
        SAY(stderr, "linne_b200: %s: cannot set the encode parameters (%d)\n", in, (int)ret);
        return 1;
    }
    /* worst case: every block stored raw, plus block and stream headers */
    cap = LINNE_HEADER_SIZE + w.frames * w.channels * (w.bits / 8u) + 11u * (w.frames / CLI_BLOCK + 2u) + 4096u;
    if (!(buf = staging_reserve(&wk->out, cap))) return 1;
    ret = LINNEB200_EncodeWholePacked(wk->enc, w.data, w.frames, buf, cap, &size);
    if (ret != LINNE_APIRESULT_OK) { SAY(stderr, "linne_b200: %s: encode failed (%d)\n", in, (int)ret); return 1; }
    if (!(fp = fopen(out, "wb")) || fwrite(buf, 1, size, fp) != size) { SAY(stderr, "linne_b200: cannot write %s\n", out); if (fp) fclose(fp); return 1; }
    fclose(fp);
    SAY(stdout, "%s -> %s: %u samples x %u ch, %u bytes\n", in, out, w.frames, w.channels, size);
    wk->samples += (uint64_t)w.frames * w.channels;
    return 0;
}

/* the excerpt of a -d run: index the stream, then decode the frames [o->start, o->start + w->frames) as one window */
static int decode_excerpt(struct Worker *wk, const struct Options *o, const char *in, const uint8_t *buf, uint32_t size,
                          uint8_t *wav, const struct Wav *w)
{
    struct LINNEB200Window win;
    LINNEApiResult ret;
    uint32_t n = 0;
    while ((ret = LINNEB200_DecoderBuildIndex(wk->dec, buf, NULL, size, wk->points, wk->points_cap, &n)) == LINNE_APIRESULT_INSUFFICIENT_BUFFER
           && n > wk->points_cap) {
        struct LINNEB200SeekPoint *p = (struct LINNEB200SeekPoint *)realloc(wk->points, (size_t)n * sizeof(*p));
        if (!p) { SAY(stderr, "linne_b200: %s: out of memory for the seek index\n", in); return 1; }
        wk->points = p;
        wk->points_cap = n;
    }
    if (ret != LINNE_APIRESULT_OK) { SAY(stderr, "linne_b200: %s: cannot index the stream (%d)\n", in, (int)ret); return 1; }
    win.first_sample = o->start; win.num_samples = w->frames; win.out_offset = 0; win.status = (int32_t)LINNE_APIRESULT_OK;
    ret = LINNEB200_DecodeWindowsPacked(wk->dec, buf, size, wk->points, n, &win, 1u, wav + 44, w->frames);
    if (ret != LINNE_APIRESULT_OK || win.status != (int32_t)LINNE_APIRESULT_OK) {
        SAY(stderr, "linne_b200: %s: decode failed (%d)\n", in, ret != LINNE_APIRESULT_OK ? (int)ret : (int)win.status);
        return 1;
    }
    return 0;
}

static const char *result_name(int32_t r)
{
    static const char *names[] = {"OK", "INVALID_ARGUMENT", "INVALID_FORMAT", "INSUFFICIENT_BUFFER", "INSUFFICIENT_DATA",
                                  "PARAMETER_NOT_SET", "DETECT_DATA_CORRUPTION", "NG"};
    return (r >= 0 && r < 8) ? names[r] : "?";
}

/* -F: the whole stream through damage, straight into the WAV staging buffer; one stderr line per lost run */
static int decode_salvage(struct Worker *wk, const char *in, const uint8_t *buf, uint32_t size, uint8_t *wav,
                          const struct LINNEHeader *h)
{
    LINNEApiResult ret;
    uint32_t n = 0, i;
    if ((ret = LINNEDecoder_SetHeader(wk->dec, h)) != LINNE_APIRESULT_OK) { SAY(stderr, "linne_b200: %s: decode failed (%d)\n", in, (int)ret); return 1; }
    if (!wk->damage) {                         /* room for the usual reports: the call runs once */
        if (!(wk->damage = (struct LINNEB200Damage *)malloc(256u * sizeof(*wk->damage)))) { SAY(stderr, "linne_b200: %s: out of memory for the damage report\n", in); return 1; }
        wk->damage_cap = 256u;
    }
    for (;;) {
        ret = LINNEB200_DecodeSalvagePacked(wk->dec, buf, size, wav + 44, h->num_samples, wk->damage, wk->damage_cap, &n);
        if ((ret != LINNE_APIRESULT_OK && ret != LINNE_APIRESULT_DETECT_DATA_CORRUPTION) || n <= wk->damage_cap) break;
        {   /* more lost runs than records: room for all of them, and the call again */
            struct LINNEB200Damage *d = (struct LINNEB200Damage *)realloc(wk->damage, (size_t)n * sizeof(*d));
            if (!d) { SAY(stderr, "linne_b200: %s: out of memory for the damage report\n", in); return 1; }
            wk->damage = d;
            wk->damage_cap = n;
        }
    }
    if (ret != LINNE_APIRESULT_OK && ret != LINNE_APIRESULT_DETECT_DATA_CORRUPTION) { SAY(stderr, "linne_b200: %s: decode failed (%d)\n", in, (int)ret); return 1; }
    pthread_mutex_lock(&g_print);
    for (i = 0; i < n; i++)
        fprintf(stderr, "%s: frames [%u, %u) lost, bytes [%u, %u): %s\n", in, wk->damage[i].first_sample,
                wk->damage[i].first_sample + wk->damage[i].num_samples, wk->damage[i].byte_offset,
                wk->damage[i].byte_offset + wk->damage[i].byte_size, result_name(wk->damage[i].status));
    pthread_mutex_unlock(&g_print);
    if (n) wk->damaged++;
    return 0;
}

static int decode_one(struct Worker *wk, const struct Options *o, const char *in, const char *out)
{
    size_t size = 0;
    uint8_t *buf = read_file(in, &wk->in, &size), *wav;
    struct LINNEHeader h;
    struct Wav w;
    LINNEApiResult ret;
    uint32_t frames = 0;
    if (!buf) { SAY(stderr, "linne_b200: cannot read %s\n", in); return 1; }
    if (size > 0xFFFFFFFFull) { SAY(stderr, "linne_b200: %s: larger than 4 GiB, not a stream this API can take\n", in); return 1; }
    if ((ret = LINNEDecoder_DecodeHeader(buf, (uint32_t)size, &h)) != LINNE_APIRESULT_OK) {
        SAY(stderr, "linne_b200: %s: not a LINNE stream (%d)\n", in, (int)ret); return 1;
    }
    memset(&w, 0, sizeof(w));
    w.channels = h.num_channels; w.rate = h.sampling_rate; w.bits = h.bits_per_sample; w.frames = h.num_samples;
    if (w.channels == 0 || w.channels > LINNE_MAX_NUM_CHANNELS || (w.bits != 8 && w.bits != 16 && w.bits != 24)) return 1;
    if (o->excerpt) {
        if (o->start > h.num_samples || (o->has_length && o->length > h.num_samples - o->start)) {
            SAY(stderr, "linne_b200: %s: excerpt [%u, +%u) outside the stream's %u frames\n", in, o->start,
                o->has_length ? o->length : 0u, h.num_samples);
            return 1;
        }
        w.frames = o->has_length ? o->length : h.num_samples - o->start;
    }
    if (!(wav = staging_reserve(&wk->out, 44u + (size_t)w.frames * w.channels * (w.bits / 8u) + 16u))) return 1;
    if (o->excerpt) {
        if (decode_excerpt(wk, o, in, buf, (uint32_t)size, wav, &w)) return 1;
        frames = w.frames;
    } else if (o->salvage) {
        if (decode_salvage(wk, in, buf, (uint32_t)size, wav, &h)) return 1;
        frames = w.frames;
    } else if ((ret = LINNEB200_DecodeWholePacked(wk->dec, buf, (uint32_t)size, wav + 44, w.frames, &frames)) != LINNE_APIRESULT_OK) {
        SAY(stderr, "linne_b200: %s: decode failed (%d)\n", in, (int)ret);
        return 1;
    }
    /* a stream that ends on a block boundary before num_samples decodes OK with fewer frames (as in the reference,
     * whose tool writes zeros there): the staging buffer is reused between files, so clear what was not written */
    if (frames < w.frames) {
        const size_t fb = (size_t)w.channels * (w.bits / 8u);
        memset(wav + 44 + (size_t)frames * fb, (w.bits == 8) ? 0x80 : 0, (size_t)(w.frames - frames) * fb);
    }
    if (wav_write(out, wav, &w) != 0) { SAY(stderr, "linne_b200: cannot write %s\n", out); return 1; }
    SAY(stdout, "%s -> %s: %u samples x %u ch\n", in, out, w.frames, w.channels);
    wk->samples += (uint64_t)w.frames * w.channels;
    return 0;
}

/* ---- the file pipeline: workers pull (input, output) pairs from one queue ---- */
struct Queue {
    const struct Options *opt;
    const char **files;
    int nfiles, next;
    pthread_mutex_t lock;
};

struct WorkerArg { struct Queue *q; struct Worker wk; pthread_t thread; int started; };

static void *worker_main(void *p)
{
    struct WorkerArg *a = (struct WorkerArg *)p;
    struct Queue *q = a->q;
    for (;;) {
        int i;
        pthread_mutex_lock(&q->lock);
        i = q->next; q->next += 2;
        pthread_mutex_unlock(&q->lock);
        if (i >= q->nfiles) break;
        a->wk.failures += q->opt->encode ? encode_one(&a->wk, q->opt, q->files[i], q->files[i + 1])
                                         : decode_one(&a->wk, q->opt, q->files[i], q->files[i + 1]);
    }
    return NULL;
}

/* a frame count: decimal digits only, below 2^32 */
static int parse_frames(const char *a, uint32_t *v)
{
    unsigned long long x = 0;
    if (!*a) return 1;
    for (; *a; a++) {
        if (*a < '0' || *a > '9') return 1;
        if ((x = x * 10u + (unsigned)(*a - '0')) > 0xFFFFFFFFull) return 1;
    }
    *v = (uint32_t)x;
    return 0;
}

static double now_s(void) { struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec; }

static void usage(const char *argv0)
{
    fprintf(stderr,
        "usage: %s -e [-m 0..7] [-l] [-a N] in.wav out.lnn [in2.wav out2.lnn ...]\n"
        "       %s -d [-c] [--start FRAME] [--length FRAMES] in.lnn out.wav [in2.lnn out2.wav ...]\n"
        "       %s -d -F in.lnn out.wav [...]   decode through damage\n"
        "       -L FILE reads \"input output\" pairs from FILE (one per line)\n"
        "       -j N    pipeline workers (handles) working on different files at the same time (default min(4, files))\n"
        "       -s      print a timing summary\n"
        "  -e encode  -d decode  -m compress mode (default 0)  -l learning  -a auxiliary-function iterations\n"
        "  -c do NOT check CRC16 when decoding\n"
        "  --start FRAME, --length FRAMES  decode only frames [FRAME, FRAME + FRAMES) of every stream (-d only;\n"
        "                                  default start 0, length to the end of the stream)\n"
        "  -F decode every intact block of a damaged stream (-d only): a full-length WAV with silence where blocks\n"
        "     were lost, one stderr line per lost run; exit code 2 when a file was damaged\n", argv0, argv0, argv0);
}

int main(int argc, char **argv)
{
    struct Options o;
    const char *files[4096];
    char *owned[4096];
    int nfiles = 0, nowned = 0, i, failures = 0, damaged = 0, jobs;
    struct Queue q;
    struct WorkerArg *workers;
    uint64_t samples = 0;
    double t0, t1;
    memset(&o, 0, sizeof(o));
    for (i = 1; i < argc; i++) {
        const char *a = argv[i];
        if (!strcmp(a, "-e") || !strcmp(a, "--encode")) o.encode = 1;
        else if (!strcmp(a, "-d") || !strcmp(a, "--decode")) o.decode = 1;
        else if (!strcmp(a, "-l") || !strcmp(a, "--enable-learning")) o.learning = 1;
        else if (!strcmp(a, "-c") || !strcmp(a, "--no-crc-check")) o.no_crc = 1;
        else if ((!strcmp(a, "-m") || !strcmp(a, "--mode")) && i + 1 < argc) o.preset = atoi(argv[++i]);
        else if ((!strcmp(a, "-a") || !strcmp(a, "--auxiliary-function-iteration")) && i + 1 < argc) o.af = atoi(argv[++i]);
        else if (!strcmp(a, "-L") && i + 1 < argc) o.list = argv[++i];
        else if ((!strcmp(a, "-j") || !strcmp(a, "--jobs")) && i + 1 < argc) o.jobs = atoi(argv[++i]);
        else if (!strcmp(a, "-s") || !strcmp(a, "--stats")) o.stats = 1;
        else if (!strcmp(a, "-F") || !strcmp(a, "--salvage")) o.salvage = 1;
        else if (!strcmp(a, "--start") || !strcmp(a, "--length")) {
            const int is_len = (a[2] == 'l');
            if (i + 1 >= argc || parse_frames(argv[++i], is_len ? &o.length : &o.start)) {
                fprintf(stderr, "%s: %s needs a frame count\n", argv[0], a); usage(argv[0]); return 1;
            }
            o.excerpt = 1;
            if (is_len) o.has_length = 1;
        }
        else if (!strcmp(a, "-h") || !strcmp(a, "--help")) { usage(argv[0]); return 0; }
        else if (a[0] == '-' && a[1] != '\0') { fprintf(stderr, "%s: unknown option %s\n", argv[0], a); usage(argv[0]); return 1; }
        else if (nfiles < 4096) files[nfiles++] = a;
    }
    if (o.list) {
        FILE *fp = fopen(o.list, "r");
        char a[2048], b[2048];
        if (!fp) { fprintf(stderr, "%s: cannot open %s\n", argv[0], o.list); return 1; }
        while (fscanf(fp, "%2047s %2047s", a, b) == 2 && nfiles + 2 <= 4096 && nowned + 2 <= 4096) {
            files[nfiles++] = owned[nowned++] = strdup(a);
            files[nfiles++] = owned[nowned++] = strdup(b);
        }
        fclose(fp);
    }
    if (o.encode == o.decode) { fprintf(stderr, "%s: exactly one of -e and -d must be given\n", argv[0]); usage(argv[0]); return 1; }
    if (o.excerpt && o.encode) { fprintf(stderr, "%s: --start and --length apply to -d only\n", argv[0]); usage(argv[0]); return 1; }
    if (o.salvage && (o.encode || o.excerpt)) { fprintf(stderr, "%s: -F applies to -d without --start / --length\n", argv[0]); usage(argv[0]); return 1; }
    if (nfiles < 2 || (nfiles & 1)) { fprintf(stderr, "%s: input and output files must come in pairs\n", argv[0]); return 1; }
    if (o.preset < 0 || o.preset >= LINNE_NUM_PARAMETER_PRESETS || o.af < 0 || o.af >= 255) { fprintf(stderr, "%s: option out of range\n", argv[0]); return 1; }

    if (o.jobs < 0 || o.jobs > 64) { fprintf(stderr, "%s: -j out of range (1..64)\n", argv[0]); return 1; }
    jobs = o.jobs ? o.jobs : (nfiles / 2 < 4 ? nfiles / 2 : 4);

    memset(&q, 0, sizeof(q));
    q.opt = &o; q.files = files; q.nfiles = nfiles;
    pthread_mutex_init(&q.lock, NULL);
    if (!(workers = (struct WorkerArg *)calloc((size_t)jobs, sizeof(*workers)))) return 1;
    for (i = 0; i < jobs; i++) {
        workers[i].q = &q;
        if (o.encode) {
            struct LINNEEncoderConfig cfg;
            cfg.max_num_channels = LINNE_MAX_NUM_CHANNELS; cfg.max_num_samples_per_block = CLI_MAX_BLOCK;
            cfg.max_num_layers = 5; cfg.max_num_parameters_per_layer = 128;          /* linne_codec.c:53-56 */
            workers[i].wk.enc = LINNEEncoder_Create(&cfg, NULL, 0);
        } else {
            struct LINNEDecoderConfig cfg;
            cfg.max_num_channels = LINNE_MAX_NUM_CHANNELS; cfg.max_num_layers = 5;
            cfg.max_num_parameters_per_layer = 128; cfg.check_crc = (uint8_t)(o.no_crc ? 0 : 1);   /* linne_codec.c:205-208 */
            workers[i].wk.dec = LINNEDecoder_Create(&cfg, NULL, 0);
            /* several decoders at work: long files take the throughput kernels, whose calls overlap (linne_b200.h) */
            if (workers[i].wk.dec && jobs > 1) LINNEB200_DecoderSetThroughputBlocks(workers[i].wk.dec, 1024u);
        }
        if (!workers[i].wk.enc && !workers[i].wk.dec) {
            fprintf(stderr, "%s: cannot create the %s\n", argv[0], o.encode ? "encoder" : "decoder");
            return 1;
        }
    }
    t0 = now_s();
    if (jobs == 1) {
        worker_main(&workers[0]);                                   /* no thread for the plain one-file case */
    } else {
        for (i = 0; i < jobs; i++) workers[i].started = (pthread_create(&workers[i].thread, NULL, worker_main, &workers[i]) == 0);
        if (!workers[0].started) worker_main(&workers[0]);
        for (i = 0; i < jobs; i++) if (workers[i].started) pthread_join(workers[i].thread, NULL);
    }
    t1 = now_s();
    for (i = 0; i < jobs; i++) {
        failures += workers[i].wk.failures;
        damaged += workers[i].wk.damaged;
        samples += workers[i].wk.samples;
        if (workers[i].wk.enc) LINNEEncoder_Destroy(workers[i].wk.enc);
        if (workers[i].wk.dec) LINNEDecoder_Destroy(workers[i].wk.dec);
        staging_release(&workers[i].wk.in);
        staging_release(&workers[i].wk.out);
        free(workers[i].wk.points);
        free(workers[i].wk.damage);
    }
    free(workers);
    pthread_mutex_destroy(&q.lock);
    if (o.stats)
        fprintf(stderr, "{\"files\": %d, \"workers\": %d, \"samples\": %llu, \"seconds\": %.6f, \"msamples_per_s\": %.3f}\n",
                nfiles / 2, jobs, (unsigned long long)samples, t1 - t0, (t1 > t0) ? (double)samples / (t1 - t0) / 1e6 : 0.0);
    for (i = 0; i < nowned; i++) free(owned[i]);
    return failures ? 1 : damaged ? 2 : 0;
}
