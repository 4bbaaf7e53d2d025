/* lnb_shim.h -- the thin C-ABI shim between the host code (plain C) and the CUDA side.
 *
 * The host code (linne_encoder_host.c / linne_decoder_host.c) sees ONLY these functions: device
 * memory, copies, stream synchronisation and the three batch pipelines.  lnb_shim_cuda.cu
 * implements them with CUDA runtime calls and sm_100a kernels.  (tests/hostsim links the same host
 * code against a loop-based stand-in to exercise host logic and kernel bodies in CPU-only CI; that
 * stand-in is test infrastructure and is never part of liblinne_b200.so.)
 */
#ifndef LNB_SHIM_H
#define LNB_SHIM_H

#include "lnb_types.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct LnbDevice LnbDevice;      /* one CUDA stream + the uploaded constant tables */

/* Returns 0 and a device context, or non-zero when no usable CUDA device exists (callers then fail:
 * there is no CPU fallback).  `device_ordinal` < 0 keeps the current device. */
int  lnb_shim_open(LnbDevice **dev, int device_ordinal);
void lnb_shim_close(LnbDevice *dev);
const LnbDevTables *lnb_shim_tables(const LnbDevice *dev);
/* Launch on an externally owned stream (cudaStream_t as void*) instead of the context's own. */
void lnb_shim_use_stream(LnbDevice *dev, void *cuda_stream);
/* Scheduling hint: `cost_rank` 0 = cheapest work .. 7 = most expensive.  Handles that run side by side on one
 * GPU (a server encoding several streams) finish soonest when the longest job's kernels are placed first, so
 * the context's own stream is re-created with a CUDA stream priority that grows with the rank.  No effect on
 * an externally supplied stream. */
void lnb_shim_set_cost_rank(LnbDevice *dev, int cost_rank);
const char *lnb_shim_backend(void);      /* "cuda-sm_100a" for the product */
/* devices visible to the process / bind the calling host thread to one / the one it is bound to (-1: none) */
int lnb_shim_device_count(void);
int lnb_shim_set_device(int ordinal);
int lnb_shim_current_device(void);
int lnb_shim_device_ordinal(const LnbDevice *dev);    /* the device a context was opened on */
/* Largest analysis length the cooperative (shared-memory) encoder kernels take; 0 = none. */
uint32_t lnb_shim_fast_max_na(void);
/* Longest block (samples per channel) the cooperative prepare / predict+plan kernels take; 0 = none. */
uint32_t lnb_shim_coop_max_n(void);
/* Longest block the fused streaming decoder (entropy decode -> synthesis -> de-emphasis in one kernel) takes; 0 = none. */
uint32_t lnb_shim_fused_max_n(void);
/* 1 when the throughput decoder (one lane per block / per block-channel, for large batches) takes streams of this
 * configuration; 0 = never (the host then leaves LnbDecodeBatch.tput clear). */
int lnb_shim_tput_supported(const LnbStreamCfg *cfg);
/* Longest analysis length the IRLS / SGD refinement kernel keeps in shared memory (0 = those paths are unavailable);
 * longer blocks need LnbEncodeBatch.refine_xy: 2 * (roundup8(max(block, P(P+1)/2)) + lnb_shim_refine_hist()) doubles per
 * (block, channel). */
uint32_t lnb_shim_refine_max_na(void);
uint32_t lnb_shim_refine_hist(void);

void *lnb_shim_alloc(LnbDevice *dev, size_t bytes);
void  lnb_shim_free(LnbDevice *dev, void *ptr);
void *lnb_shim_alloc_pinned(size_t bytes);
void  lnb_shim_free_pinned(void *ptr);
int   lnb_shim_h2d(LnbDevice *dev, void *dst, const void *src, size_t bytes);      /* async on the stream */
int   lnb_shim_d2h(LnbDevice *dev, void *dst, const void *src, size_t bytes);      /* async on the stream */
int   lnb_shim_d2d(LnbDevice *dev, void *dst, const void *src, size_t bytes);      /* async on the stream */
int   lnb_shim_memset(LnbDevice *dev, void *dst, int value, size_t bytes);
int   lnb_shim_sync(LnbDevice *dev);     /* 0 on success; non-zero reports a CUDA error */

/* the batch pipelines (enqueue only; results are valid after lnb_shim_sync) */
int lnb_shim_decode(LnbDevice *dev, const LnbDecodeBatch *batch);
int lnb_shim_encode_analyze(LnbDevice *dev, const LnbEncodeBatch *batch);
int lnb_shim_encode_pack(LnbDevice *dev, const LnbEncodeBatch *batch, uint32_t out_capacity);

/* hop over the block size fields of `num_files` streams of a device image (enqueue only): d_files / d_table / d_results
 * are device buffers; d_table receives byte offsets relative to the image and sample offsets relative to each stream */
int lnb_shim_hop(LnbDevice *dev, const uint8_t *d_image, const LnbHopFile *d_files, uint32_t num_files,
                 LnbBlockDesc *d_table, LnbHopResult *d_results);

/* sample-window decodes (lnb_window.cuh), enqueue only.  seek: one item per block a window needs -- reads the block header
 * at d_in[j].img_off of d_image, checks it against the index and fills d_out[j] (result code in .status).  gather: copies
 * every window of d_wins from the scratch planes [C][scratch_stride] to d_dst [C][dst_stride]; `num_items` is the item
 * count after the last window's item_first (one item per channel and aligned group of four destination samples). */
int lnb_shim_seek_blocks(LnbDevice *dev, const uint8_t *d_image, const LnbSeekIn *d_in, uint32_t n,
                         uint32_t channels, uint32_t bits, LnbBlockDesc *d_out);
int lnb_shim_gather_windows(LnbDevice *dev, const int32_t *d_scratch, uint32_t scratch_stride, const LnbGatherWin *d_wins,
                            uint32_t num_wins, uint32_t num_items, int32_t *d_dst, uint32_t dst_stride);
/* the same windows as packed interleaved PCM (WAV data-chunk layout, `bytes` per sample) into the dense staging buffer
 * d_dst: window w at byte d_wins[w].dst * channels * bytes, every dst a multiple of 4; one item per aligned group of
 * four frames; d_dst has room for every window rounded up to whole groups. */
int lnb_shim_gather_windows_packed(LnbDevice *dev, const int32_t *d_scratch, uint32_t scratch_stride, const LnbGatherWin *d_wins,
                                   uint32_t num_wins, uint32_t num_items, uint8_t *d_dst, uint32_t channels, uint32_t bytes);

/* packed interleaved PCM (WAV data-chunk layout, `bytes` per sample) <-> int32 planes, on the device (enqueue only) */
int lnb_shim_unpack_pcm(LnbDevice *dev, const uint8_t *d_packed, int32_t *d_pcm, uint32_t pcm_stride,
                        uint32_t frames, uint32_t channels, uint32_t bytes);
int lnb_shim_pack_pcm(LnbDevice *dev, const int32_t *d_pcm, uint8_t *d_packed, uint32_t pcm_stride,
                      uint32_t frames, uint32_t channels, uint32_t bytes);

/* dst[j] = sin(pi * j / (n - 1)), j < n: the sine window of the block-type estimate (reference lpc.c:176-212 via
 * :810-865), tabulated once per handle and block length with the very function the prepare kernel would call per
 * sample.  Enqueue only; non-zero when the back end has no use for the table (the host then passes none). */
int lnb_shim_fill_sine_window(LnbDevice *dev, double *dst, uint32_t n);

/* number of kernels launched through this context since it was opened (bench.py's gpu_launches) */
uint64_t lnb_shim_launch_count(const LnbDevice *dev);

/* Per-stage device timing (CUDA events on the launching stream around every kernel).  Off by default.
 * Stats accumulate until reset; `get` returns the number of stages filled in. */
typedef struct LnbStageStat { char name[24]; uint64_t launches; double total_ms; } LnbStageStat;
void lnb_shim_profile_enable(LnbDevice *dev, int on);
void lnb_shim_profile_reset(LnbDevice *dev);
int  lnb_shim_profile_get(LnbDevice *dev, LnbStageStat *out, int max_stages);
/* Launch timeline of the profiled kernels: begin/end in ms since a process-wide reference event, so that
 * the timelines of handles running side by side on their own streams can be merged. */
typedef struct LnbTimelineEntry { char name[24]; float begin_ms, end_ms; } LnbTimelineEntry;
int  lnb_shim_profile_timeline(LnbDevice *dev, LnbTimelineEntry *out, int max_entries);

/* Sustained FP64 FMA throughput of the device in TFLOP/s (2 flops per DFMA), measured with a
 * register-resident microbenchmark: the roofline denominator of the analysis kernels. */
double lnb_shim_measure_fp64_tflops(LnbDevice *dev);

/* ---- raw device memory and cross-process peer mappings (multi-GPU sharding, one process per GPU) ----
 * All act on the calling thread's current CUDA device.  `kind`: 0 device->device (either side may be a
 * peer mapping: the copy then runs over NVLink), 1 host->device, 2 device->host.  Copies are synchronous. */
void *lnb_shim_device_alloc(size_t bytes);
void  lnb_shim_device_free(void *ptr);
int   lnb_shim_ipc_export(const void *ptr, unsigned char handle[64]);     /* 0 on success */
void *lnb_shim_ipc_open(const unsigned char handle[64]);                  /* NULL on failure */
void  lnb_shim_ipc_close(void *peer_ptr);
int   lnb_shim_copy(void *dst, const void *src, size_t bytes, int kind);  /* 0 on success */

#ifdef __cplusplus
}
#endif
#endif
