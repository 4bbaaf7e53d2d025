/* lnb_types.h -- plain-C data types shared by the host code (C), the CUDA shim and the kernels.
 * No CUDA or C++ constructs here: this is what crosses the host <-> shim boundary.
 */
#ifndef LNB_TYPES_H
#define LNB_TYPES_H

#include <stdint.h>
#include <stddef.h>
#include "linne_tables.h"
#include "linne_host_tables.h"

/* ---- stream-level configuration, passed to kernels by value ---- */
typedef struct LnbStreamCfg {
    uint32_t num_channels;
    uint32_t bits_per_sample;
    uint32_t block_size;          /* header.num_samples_per_block */
    uint32_t num_layers;
    uint32_t layer_params[LNB_MAX_LAYERS];
    uint32_t num_lambdas;
    double   lambdas[LNB_MAX_LAMBDAS];
    uint32_t ms;                  /* 1: mid/side on channels 0/1 */
    uint32_t pcm_stride;          /* samples between channel planes of the device PCM buffer */
    uint32_t work_stride;         /* samples between (block,channel) rows of the work buffer */
    uint32_t check_crc;
} LnbStreamCfg;

/* ---- one block of the batch ---- */
typedef struct LnbBlockDesc {
    uint32_t smp_off;             /* first sample (per channel) of the block in the PCM planes */
    uint32_t nsmp;                /* samples per channel */
    uint32_t byte_off;            /* offset of the block's sync code in the stream buffer */
    uint32_t byte_size;           /* bytes of the whole block incl. the 11-byte block header */
    uint32_t type;                /* LNB_BLOCK_* */
    uint32_t na;                  /* encoder: number of samples the analysis looks at; decoder: payload bytes consumed */
    uint32_t status;              /* decoder: LNB_ST_* flags */
    uint32_t crc;                 /* decoder: CRC16 computed over the block body */
} LnbBlockDesc;

/* encoder-side use of LnbBlockDesc.status: the block takes the cooperative (shared-memory) kernels */
#define LNB_ENC_FLAG_FAST 1u
/* encoder-side: the block image has already been written by the cooperative packer */
#define LNB_ENC_FLAG_PACKED 2u
/* encoder-side: block short enough for the cooperative prepare / predict+plan kernels */
#define LNB_ENC_FLAG_COOP 4u
/* encoder-side: analysis length fits the cooperative analysis kernel but not its fast layout (any
 * length up to its maximum, e.g. a tail block): the same launch runs it on the generic path */
#define LNB_ENC_FLAG_GENERIC 8u

enum { LNB_ST_OK = 0, LNB_ST_CRC_MISMATCH = 1, LNB_ST_OVERRUN = 2, LNB_ST_BAD_TYPE = 4 };

/* ---- analysis result / parsed side information of one (block, channel) ---- */
typedef struct LnbChanParams {
    int32_t preem_prev[LNB_NUM_PREEM];
    uint8_t preem_coef[LNB_NUM_PREEM];
    uint8_t log2_units[LNB_MAX_LAYERS];
    uint8_t rshift[LNB_MAX_LAYERS];
    int8_t  coef[LNB_MAX_LAYERS * LNB_MAX_PARAMS];   /* layer l starts at l * LNB_MAX_PARAMS */
} LnbChanParams;

/* ---- residual-coder plan of one (block, channel) ---- */
typedef struct LnbCoderPlan {
    uint32_t porder;
    uint32_t bits;                /* bits of the whole channel payload (10-bit porder field included) */
    uint8_t  k2[LNB_MAX_PARTITIONS];
} LnbCoderPlan;

/* ---- device-resident constant tables ---- */
typedef struct LnbDevTables {
    const uint16_t *huff_lut;     /* [1 << LNB_HUFF_LUT_BITS] (symbol << 4) | length */
    const uint32_t *huff_code;    /* [256] */
    const uint8_t  *huff_len;     /* [256] */
    const double   *k2_threshold; /* [LNB_NUM_K2_THRESHOLDS] */
    const uint16_t *crc_table;    /* [256] */
} LnbDevTables;


/* ---- one decode batch (all pointers are device pointers) ---- */
typedef struct LnbDecodeBatch {
    LnbStreamCfg cfg;
    LnbDevTables tab;
    const uint8_t *stream;          /* whole .lnn file image, padded by >= 16 zero bytes */
    uint32_t stream_size;
    LnbBlockDesc *blocks;
    uint32_t num_blocks;
    LnbChanParams *params;          /* [num_blocks * C] */
    int32_t *pcm;                   /* [C][pcm_stride] */
    uint32_t fused_max_n;           /* > 0: compressed blocks of at most this many samples take the fused streaming kernel */
    uint32_t num_plain_blocks;      /* blocks left to the split kernels (raw, silent, longer than fused_max_n) */
    uint32_t tput;                  /* 1: full compressed blocks take the throughput kernels (lnb_tput_v2.cuh); needs fused_max_n */
    uint32_t max_nsmp;              /* longest block of the batch (samples per channel): sizes the shared-memory lines of the
                                     * per-block kernels -- a block may be longer than the header's block size (the reference
                                     * checks it against the caller's buffer only, linne_decoder.c:632-635) */
} LnbDecodeBatch;

/* ---- the hop over block size fields (lnb_framing.h; on the device lnb_hop.cuh): one record per stream of the image ---- */
typedef struct LnbHopFile {
    uint32_t offset, size;          /* the stream inside the image */
    uint32_t room_samples;          /* frames the destination planes hold for it */
    uint32_t table_first, table_cap;/* its slice of the block table */
} LnbHopFile;
typedef struct LnbHopResult {
    uint8_t  header[32];            /* device hop: the stream's 30 header bytes (for the host's header checks) */
    uint32_t num_blocks, num_decodable, framing_error, post_crc_error, total_samples, end_offset;
    uint32_t overflow;              /* 1: more blocks than table_cap (the host hop grows its table; a device hop falls back to it) */
} LnbHopResult;

/* ---- sample-window decodes (lnb_window.cuh) ----
 * LnbSeekIn: one block a window needs, found through the caller's seek index.  The block header is read at `img_off` of
 * the batch's image; `span` bytes are there (up to the next indexed block), `remain` bytes of the stream follow the
 * block's start (the framing checks of lnb_framing.h use it).  `nsmp` is the index's sample count of the block and
 * `smp_off` its place in the scratch planes. */
typedef struct LnbSeekIn {
    uint32_t img_off, span, remain, nsmp, smp_off;
} LnbSeekIn;
/* LnbGatherWin: one window of a gather: `len` samples per channel from scratch sample `src` to destination sample `dst`;
 * its items (one per aligned group of four destination samples and channel) start at item `item_first`. */
typedef struct LnbGatherWin {
    uint32_t src, dst, len, item_first;
} LnbGatherWin;

/* ---- one encode batch (all pointers are device pointers) ---- */
typedef struct LnbEncodeBatch {
    LnbStreamCfg cfg;
    LnbDevTables tab;
    const int32_t *pcm;             /* [C][pcm_stride] */
    LnbBlockDesc *blocks;
    uint32_t num_blocks;
    LnbChanParams *params;          /* [B*C] */
    double *est;                    /* [B*C] */
    int32_t *work;                  /* [B*C][work_stride] */
    /* analysis scratch; slot s = (block*C + ch)*num_lambdas + lambda */
    double *sig_a, *sig_b;          /* [S][work_stride] ping-pong layer signal */
    double *acorr;                  /* [S][LNB_MAX_LEVELS][256] autocorrelations: U*(p+1) <= 256 cells per level */
    double *cand;                   /* [S][LNB_MAX_LEVELS][LNB_MAX_PARAMS] candidate coefficients */
    double *unit_loss;              /* [S][LNB_MAX_LEVELS][chunks] partial L1 losses, chunks = ceil(work_stride/64) */
    double *chosen_w;               /* [S][LNB_MAX_LAYERS][LNB_MAX_PARAMS] */
    uint8_t *chosen_log2u;          /* [S][LNB_MAX_LAYERS] */
    double *final_sum;              /* [S][chunks] partial |residual| sums of the last layer */
    const double *welch;            /* [B][LNB_MAX_LEVELS] window scale per unit-count level */
    const double *sinwin;           /* [sinwin_n] sine window of the block-type estimate for blocks of sinwin_n samples, or NULL */
    uint32_t sinwin_n;
    LnbCoderPlan *plans;            /* [B*C] */
    double *plan_mean;              /* [B*C][2*LNB_MAX_PARTITIONS] */
    uint8_t *out;                   /* device image of the output stream */
    uint32_t *total_size;           /* device scalar: bytes of all blocks of this batch */
    uint32_t out_base;              /* byte offset of the first block of this batch in `out` */
    uint32_t num_coop_blocks;       /* blocks flagged LNB_ENC_FLAG_COOP */
    uint32_t num_fast_blocks;       /* blocks flagged LNB_ENC_FLAG_FAST (0: skip the cooperative launch) */
    uint32_t num_slow_blocks;       /* compressed-candidate blocks left to the flat kernels */
    uint32_t af_iterations;         /* IRLS iterations of the final pass (0 = off) */
    uint32_t enable_learning;       /* 1: momentum-SGD refinement of the final coefficients */
    double *train_scratch;          /* [B*C][2*layers+1][work_stride], only when enable_learning */
    double *refine_xy;              /* NULL, or the refinement kernel's signal buffers for blocks too long for shared memory */
    uint32_t forced_params;         /* 1: `params` already hold units/shift/coefficients -- skip the analysis stages */
} LnbEncodeBatch;

#endif
