/* linne_b200.h -- extension entry points of liblinne_b200.so next to the reference API.
 *
 * These do not exist in the reference; they expose what a GPU implementation adds: device-resident and
 * packed-PCM variants of the whole-file calls, corpus batches (several files per call), block read-ahead
 * for streaming callers, page-locked host memory, device buffers and peer mappings for multi-GPU sharding,
 * launch accounting and per-kernel timing for benchmarks.  Plain C ABI: pointers and sizes only.
 */
#ifndef LINNE_B200_H_INCLUDED
#define LINNE_B200_H_INCLUDED

#include <stddef.h>
#include "linne.h"
#include "linne_encoder.h"
#include "linne_decoder.h"

#ifdef __cplusplus
extern "C" {
#endif

/* "cuda-sm_100a" for the product library. */
const char *LINNEB200_Backend(void);

/* 1 if a CUDA device is usable from this process, else 0 (handles cannot be created then). */
int LINNEB200_DeviceAvailable(void);

/* Kernels launched so far on behalf of a handle (for bench.py's gpu_launches accounting). */
uint64_t LINNEB200_EncoderLaunchCount(const struct LINNEEncoder *encoder);
uint64_t LINNEB200_DecoderLaunchCount(const struct LINNEDecoder *decoder);

/* Run a handle's GPU work on an externally owned CUDA stream (cudaStream_t passed as void*), so a
 * caller can bracket the work with its own CUDA events.  API calls stay synchronous. */
void LINNEB200_EncoderUseStream(struct LINNEEncoder *encoder, void *cuda_stream);
void LINNEB200_DecoderUseStream(struct LINNEDecoder *decoder, void *cuda_stream);

/* ---- several GPUs behind one handle (SURVEY 8e) -------------------------------------------------------------
 * LINNEEncoder_EncodeWhole / LINNEDecoder_DecodeWhole of a handle with N > 1 devices cut the stream's blocks into N
 * contiguous ranges, one per device (ranges share devices round-robin when N exceeds the visible devices), each driven
 * by its own host thread inside the call: upload of the range, kernels, and -- after an exclusive scan of the shard
 * byte counts on the host -- the copy of every shard to its place in the caller's buffer.  Results are byte-identical
 * with one device.  Replaces nothing in the reference (it has no threads); the environment variable
 * LINNE_B200_GPUS=N (or "all") sets the default for every handle, so an unmodified caller of the reference API
 * (tools/linne_codec/linne_codec.c built against this library) uses all GPUs of a box.  0 or 1: one device. */
void LINNEB200_EncoderSetDevices(struct LINNEEncoder *encoder, uint32_t num_devices);
void LINNEB200_DecoderSetDevices(struct LINNEDecoder *decoder, uint32_t num_devices);

/* ---- device-resident entry points: bulk data stays in HBM -------------------------------------
 * EncodeWholeResident: `d_pcm` = device int32 planes [C][pcm_stride]; the stream is written to the
 * device buffer `d_data`.  DecodeWholeResident: `d_data` = device copy of the stream padded with
 * >= 16 zero bytes (`data` = the host copy, needed only to hop over the block size fields; pass NULL
 * and the library fetches the image from the device itself);
 * PCM is left in the device planes `d_pcm` [C][pcm_stride].  Same result codes as the host calls. */
LINNEApiResult LINNEB200_EncodeWholeResident(struct LINNEEncoder *encoder,
        const int32_t *d_pcm, uint32_t pcm_stride, uint32_t num_samples,
        uint8_t *d_data, uint32_t data_size, uint32_t *output_size);
LINNEApiResult LINNEB200_DecodeWholeResident(struct LINNEDecoder *decoder,
        const uint8_t *data, const uint8_t *d_data, uint32_t data_size,
        int32_t *d_pcm, uint32_t pcm_stride, uint32_t buffer_num_channels, uint32_t buffer_num_samples);

/* ---- corpus batches: several files per call (SURVEY 8e) -------------------------------------------------
 * Blocks are independent, across files too, so a corpus tool can hand the kernels the blocks of many files at once:
 * fewer, larger launches (the per-file chain of a dozen launches and several synchronisations is what limits many
 * handles on many GPUs) and full waves for every kernel.  All files of a call share the handle's stream parameters.
 * The PCM of the files sits in one set of device planes [C][pcm_stride], file i at samples [first_sample,
 * first_sample + num_samples); the streams sit one after the other in `d_data` (out_offset / out_size: written by
 * the encoder, read by the decoder; the image must be followed by >= 16 readable bytes).  Every stream is
 * byte-identical with what EncodeWhole writes for that file; the decoder returns the first file's error, if any,
 * and leaves every file's own result in `status`. */
struct LINNEB200FileDesc {
    uint32_t first_sample, num_samples;     /* where the file's PCM is (encode: in, decode: in) */
    uint32_t out_offset, out_size;          /* where the file's stream is in d_data (encode: out, decode: in) */
    int32_t  status;                        /* decode: LINNEApiResult of this file */
};
LINNEApiResult LINNEB200_EncodeFilesResident(struct LINNEEncoder *encoder, const int32_t *d_pcm, uint32_t pcm_stride,
        struct LINNEB200FileDesc *files, uint32_t num_files, uint8_t *d_data, uint32_t data_size, uint32_t *output_size);
LINNEApiResult LINNEB200_DecodeFilesResident(struct LINNEDecoder *decoder, const uint8_t *d_data, uint32_t data_size,
        struct LINNEB200FileDesc *files, uint32_t num_files, int32_t *d_pcm, uint32_t pcm_stride);
/* The same with host buffers, as a corpus tool holds them: the files' frames back to back as packed interleaved PCM
 * (WAV data-chunk layout, files[i].num_samples frames each; first_sample is filled in) and the streams one after the
 * other in a host image.  One transfer up, one conversion, one batch for the kernels, one transfer down. */
LINNEApiResult LINNEB200_EncodeFilesPacked(struct LINNEEncoder *encoder, const uint8_t *pcm, struct LINNEB200FileDesc *files,
        uint32_t num_files, uint8_t *data, uint32_t data_size, uint32_t *output_size);
LINNEApiResult LINNEB200_DecodeFilesPacked(struct LINNEDecoder *decoder, const uint8_t *data, uint32_t data_size,
        struct LINNEB200FileDesc *files, uint32_t num_files, uint8_t *pcm);

/* ---- random access: seek index and sample-window decodes -----------------------------------------------
 * Every block is self-contained, so an excerpt of a stream needs only the blocks it overlaps.  A seek index holds one
 * point per block, in stream order: the block's first sample and the byte offset of its sync code, counted from the
 * start of the image (30-byte header included).  The first point is always (0, 30).  A caller may keep the index next to
 * the stream (a sidecar file); the library checks every index it is given and never reads outside the image because of it.
 *
 * BuildIndex hops once over the stream -- the host image `data`, or the device image `d_data` when data == NULL (the hop
 * then runs on the device, as in DecodeWholeResident) -- latches the stream's header on the handle (as SetHeader does)
 * and writes one point per block to `points`.  It returns the result the hop of DecodeWhole gives for the stream's
 * framing; on a stream damaged part-way through, the points of the blocks before the damage are written.  `*num_points`
 * is always the number of blocks found; if it exceeds `capacity`, the first `capacity` points are written and the call
 * returns INSUFFICIENT_BUFFER (call again with that capacity; points may be NULL when capacity is 0). */
struct LINNEB200SeekPoint { uint32_t first_sample, byte_offset; };
LINNEApiResult LINNEB200_DecoderBuildIndex(struct LINNEDecoder *decoder, const uint8_t *data, const uint8_t *d_data,
        uint32_t data_size, struct LINNEB200SeekPoint *points, uint32_t capacity, uint32_t *num_points);

/* DecodeWindows decodes sample windows of the stream whose header is latched on the handle.  Window w receives samples
 * [first_sample, first_sample + num_samples) of every channel, exactly as DecodeWhole writes them, at out_offset of the
 * caller's planes (buffer[c][out_offset ...]; resident: d_pcm[c * pcm_stride + out_offset ...]).  The blocks the
 * windows need go through the kernels as ONE batch and each is decoded once, even when windows overlap; windows may be
 * unsorted, overlapping, repeated or empty.  A host image uploads only the bytes of the needed blocks.  The device image
 * of DecodeWindowsResident must be followed by >= 16 readable bytes.  A handle with several devices decodes windows on
 * its own device; the DecodeBlock read-ahead cache is left as it was.
 *
 * Rejected as a whole (nothing written, no status set): NULL pointers (INVALID_ARGUMENT), no latched header
 * (PARAMETER_NOT_SET), fewer buffer channels than the stream has (INSUFFICIENT_BUFFER), and INVALID_ARGUMENT for a
 * window that ends past the stream's num_samples or whose output range leaves the buffer (buffer_num_samples /
 * pcm_stride), and for an index that does not start at (0, 30), is not strictly increasing in both fields, or has a
 * point at or beyond data_size or num_samples.
 *
 * Stream damage is reported per window: `status` = the result of the first failing block the window needs, in stream
 * order -- INVALID_FORMAT (no sync code at the indexed offset, a bad block type, a block that disagrees with the index
 * in its sample count or runs past the next indexed block), INSUFFICIENT_DATA (a block that runs past the image),
 * DETECT_DATA_CORRUPTION (CRC mismatch, when the handle checks CRCs).  A failed window's samples are undefined, every
 * other window is exact.  The call returns the first non-OK status in window order.
 *
 * A player seeks without these calls: LINNEDecoder_DecodeBlock(decoder, data + points[k].byte_offset,
 * data_size - points[k].byte_offset, ...) decodes block k and the ones after it, one per call. */
struct LINNEB200Window { uint32_t first_sample, num_samples, out_offset; int32_t status; };
LINNEApiResult LINNEB200_DecodeWindows(struct LINNEDecoder *decoder, const uint8_t *data, uint32_t data_size,
        const struct LINNEB200SeekPoint *points, uint32_t num_points, struct LINNEB200Window *windows, uint32_t num_windows,
        int32_t **buffer, uint32_t buffer_num_channels, uint32_t buffer_num_samples);
LINNEApiResult LINNEB200_DecodeWindowsResident(struct LINNEDecoder *decoder, const uint8_t *d_data, uint32_t data_size,
        const struct LINNEB200SeekPoint *points, uint32_t num_points, struct LINNEB200Window *windows, uint32_t num_windows,
        int32_t *d_pcm, uint32_t pcm_stride);

/* DecodeWindowsPacked is DecodeWindows with the output of DecodeWholePacked: window w writes frames [first_sample,
 * first_sample + num_samples) as interleaved little-endian samples (the bytes of a WAV data chunk, see the packed PCM
 * entry points below) at byte out_offset * F of `pcm`, F = num_channels * bits_per_sample / 8.  On success these bytes
 * equal the same frames of DecodeWholePacked's output.  The samples are converted on the device, come down as bits/8
 * bytes per sample in one transfer and are copied with one memcpy per window.
 *
 * Rejected as DecodeWindows is, with the same codes (nothing written, no status set), except that the output range of a
 * window must end at or before pcm_capacity_frames (else INVALID_ARGUMENT), and a header whose bits_per_sample is not 8,
 * 16, 24 or 32 gives INVALID_FORMAT.  Statuses and the result as in DecodeWindows.  The bytes of a failed window, and
 * every byte of `pcm` outside the windows, are left as they were. */
LINNEApiResult LINNEB200_DecodeWindowsPacked(struct LINNEDecoder *decoder, const uint8_t *data, uint32_t data_size,
        const struct LINNEB200SeekPoint *points, uint32_t num_points, struct LINNEB200Window *windows, uint32_t num_windows,
        uint8_t *pcm, uint32_t pcm_capacity_frames);

/* ---- salvage decodes: every intact block of a damaged stream -------------------------------------------------------
 * DecodeSalvage decodes what is left of a damaged stream.  Every block that can be verified and placed is decoded to
 * its place, samples it cannot account for are zero (silence; the biased 128 in 8-bit packed output), and the damage is
 * reported.  The stream's header is the one latched on the handle (SetHeader or BuildIndex), as for DecodeWindows: the
 * image's first 30 bytes are skipped and not parsed, so a caller who knows the parameters recovers a stream whose header
 * is damaged.  CRCs are always checked, whatever the handle's check_crc.  B = num_samples_per_block, N = num_samples and
 * T = N - B * (ceil(N / B) - 1), the length of the tail block, all from the header.
 *
 * A verified block at byte offset o >= 30 passes the framing checks of DecodeWhole with data_size - o bytes left, holds
 * 1 .. B samples, is at most 2 * B * num_channels * ceil(bits_per_sample / 8) + 4171 bytes long (twice a raw block plus
 * 4 KiB: more room than this library's encoder gives a block) and matches its CRC16.  Its successor is the offset DecodeWhole's hop goes to next.  It is confirmed
 * when its successor is another verified block or data_size.  The walk runs from offset 30, sample 0:
 *   - a verified block at the current offset is accepted at the current sample;
 *   - otherwise a damaged region starts there; v is the first confirmed block after it.  When the damaged bytes still
 *     frame as a block of B samples and a chain of such blocks (verified ones between them) leads from there exactly to
 *     v (damaged payloads), the damaged block is lost in place: the walk moves on B samples and to its successor.  Any
 *     other damage (a framing gap) ends the segment of blocks; a new one starts at v, not knowing its sample position.
 *     With no v the region runs to the end of the image.
 *   - the first segment (anchored at sample 0) ends when it reaches N samples; bytes after that are ignored.
 * The last segment is placed when its chain ends exactly at data_size with a block of T samples (it then ends at sample
 * N) and it starts at or after the end of the first.  Segments between two framing gaps are placed only when the last
 * one is and the samples lost between the first and the last are B times the number of framing gaps, i.e. when each
 * gap cost exactly one block (a damaged block header).  Any other segment is not decoded.
 * Every placed block lands where it is in the intact stream and its samples are exactly what DecodeWhole writes for it;
 * a block whose CRC failed never reaches the decode kernels.
 *
 * Two limits.  Blocks do not store their position, so whole blocks removed exactly at block boundaries leave no trace in
 * the bytes and the walk cannot see them, just as DecodeWhole cannot.  And the rule for segments between framing gaps
 * counts only the total: when the gaps cost different numbers of blocks that add up to B samples per gap (one gap of
 * inserted bytes that cost nothing and one that cost two blocks, say), the segments between them are placed at the
 * wrong sample positions, and samples outside the records then differ from the intact stream's.
 *
 * `damage` gets one record per maximal run of output samples that no placed block wrote, in stream order: the sample range,
 * the bytes of the image it covers (undecoded segments included) and the status of its first failing position --
 * INVALID_FORMAT or INSUFFICIENT_DATA when the bytes there do not frame as a block (sync code, size field; as DecodeWhole
 * reports them), DETECT_DATA_CORRUPTION when they do.  Bytes inserted between two blocks give a record with
 * num_samples = 0; a stream that ends on a block boundary before N gives (s, N - s, data_size, 0, INSUFFICIENT_DATA).
 * `*num_damage` is always the number of records; the first `capacity` are written (damage may be NULL when capacity is 0).
 *
 * Returns OK when there are no records -- the output then equals DecodeWhole's / DecodeWholePacked's -- and
 * DETECT_DATA_CORRUPTION when there are: the output is complete (N samples per channel) and the records say what is
 * missing.  Rejected as a whole (nothing written): NULL pointers (INVALID_ARGUMENT), no latched header
 * (PARAMETER_NOT_SET), fewer buffer channels than the stream has or room for fewer than N samples (buffer_num_samples,
 * pcm_capacity_frames: INSUFFICIENT_BUFFER), and for the packed call bits_per_sample other than 8, 16, 24 or 32
 * (INVALID_FORMAT).  The whole image goes to the device; a call is the scan, one CRC pass, one decode batch (and one
 * conversion to packed PCM), whatever the damage.  A handle with several devices salvages on its own device; the
 * DecodeBlock read-ahead cache is left as it was. */
struct LINNEB200Damage { uint32_t first_sample, num_samples, byte_offset, byte_size; int32_t status; };
LINNEApiResult LINNEB200_DecodeSalvage(struct LINNEDecoder *decoder, const uint8_t *data, uint32_t data_size,
        int32_t **buffer, uint32_t buffer_num_channels, uint32_t buffer_num_samples,
        struct LINNEB200Damage *damage, uint32_t capacity, uint32_t *num_damage);
LINNEApiResult LINNEB200_DecodeSalvagePacked(struct LINNEDecoder *decoder, const uint8_t *data, uint32_t data_size,
        uint8_t *pcm, uint32_t pcm_capacity_frames,
        struct LINNEB200Damage *damage, uint32_t capacity, uint32_t *num_damage);

/* ---- packed PCM entry points (SURVEY 8f.2) ------------------------------------------------------------
 * `pcm` = interleaved little-endian samples exactly as in a WAV data chunk (8-bit unsigned with a bias of 128,
 * 16/24/32-bit signed; bits per sample = the encoder's parameter / the stream header).  The conversion to and
 * from the int32 planes runs on the device, so the PCIe bytes per sample are bits/8 instead of 4.
 * `num_samples` and `pcm_capacity_frames` count frames (samples per channel).  Same result codes as
 * EncodeWhole / DecodeWhole; `*num_frames` = frames written (all of them on success). */
LINNEApiResult LINNEB200_EncodeWholePacked(struct LINNEEncoder *encoder, const uint8_t *pcm, uint32_t num_samples,
        uint8_t *data, uint32_t data_size, uint32_t *output_size);
LINNEApiResult LINNEB200_DecodeWholePacked(struct LINNEDecoder *decoder, const uint8_t *data, uint32_t data_size,
        uint8_t *pcm, uint32_t pcm_capacity_frames, uint32_t *num_frames);

/* ---- streaming (SURVEY 8f.4): block-at-a-time callers ------------------------------------------------
 * LINNEDecoder_DecodeBlock decodes `blocks` blocks per GPU batch when the caller's buffer holds that many
 * (a player passes everything that is left of its stream, tools/linne_player/linne_player.c:110-121) and
 * serves the following calls from pinned host memory.  A cached block is handed out only if the bytes the
 * caller passes equal the bytes that were decoded, so results and error codes are those of the batch of one.
 * 0 or 1 switches it off (the default; the environment variable LINNE_B200_READAHEAD sets the default). */
void LINNEB200_DecoderSetReadahead(struct LINNEDecoder *decoder, uint32_t blocks);

/* ---- decoding many streams at once ------------------------------------------------------------------
 * DecodeWhole has two data paths.  The per-block pipeline (one CTA per block) has the shortest latency for one
 * call but fills the GPU's issue slots from ~600 blocks on, so concurrent calls queue behind each other.  The
 * throughput kernels (eight lanes per block, one lane per block-channel) need ~10x fewer instructions per sample
 * but ~5 ms per call whatever its size; calls of several handles overlap almost freely.  A call takes them when it
 * holds at least `min_blocks` full blocks: default 2560 (where they win for a single call); a corpus tool that
 * keeps several handles busy lowers it to ~1024 (what linne_b200_cli -j N and bench.py's corpus leg do);
 * 0 = never.  Results are identical either way.  Environment default: LINNE_B200_TPUT_MIN_BLOCKS. */
void LINNEB200_DecoderSetThroughputBlocks(struct LINNEDecoder *decoder, uint32_t min_blocks);

/* Page-locked host memory for the buffers handed to EncodeWhole / DecodeWhole and their packed variants
 * (SURVEY 8f.3): copies from and to such memory are DMA transfers that overlap with kernels of other
 * handles.  NULL when no device is usable. */
void *LINNEB200_HostAlloc(size_t bytes);
void  LINNEB200_HostFree(void *h_ptr);

/* ---- encode with externally supplied analysis results ------------------------------------------
 * One record per (block, channel), block-major.  Used to show that identical quantised
 * coefficients yield byte-identical residuals and coded bits (north star, parity leg 3).
 * For every layer of the preset, log2_units must be at most 7 and rshift at most 15: the stream
 * stores them in 3 and 4 bits.  A record with a larger value makes the call return
 * INVALID_ARGUMENT before anything is written.  A layer with more units than taps predicts nothing. */
struct LINNEB200ChannelParams {
    uint8_t log2_units[3];
    uint8_t rshift[3];
    int8_t  coef[3][128];
};
LINNEApiResult LINNEB200_EncodeWholeWithParams(struct LINNEEncoder *encoder,
        const int32_t *const *input, uint32_t num_samples,
        const struct LINNEB200ChannelParams *params, uint32_t num_param_blocks,
        uint8_t *data, uint32_t data_size, uint32_t *output_size);

/* ---- device memory and peer mappings: multi-GPU sharding with one process per GPU ---------------
 * A stream is sharded by contiguous block ranges (blocks are independent).  Every rank encodes its
 * range into a local device buffer; after an exclusive scan of the shard byte counts each rank writes
 * its shard straight into the destination buffer of rank 0 through a CUDA IPC peer mapping -- a
 * device-to-device copy over NVLink, no collective.  All calls act on the calling thread's current
 * CUDA device; copies are synchronous; int results are 0 on success. */
void *LINNEB200_DeviceAlloc(size_t bytes);
void  LINNEB200_DeviceFree(void *d_ptr);
int   LINNEB200_IpcExport(const void *d_ptr, uint8_t handle[64]);      /* d_ptr from LINNEB200_DeviceAlloc */
void *LINNEB200_IpcOpen(const uint8_t handle[64]);                     /* peer mapping in this process, NULL on failure */
void  LINNEB200_IpcClose(void *d_peer_ptr);
int   LINNEB200_DeviceCopy(void *d_dst, const void *d_src, size_t bytes);   /* either side may be a peer mapping */
int   LINNEB200_CopyToDevice(void *d_dst, const void *h_src, size_t bytes);
int   LINNEB200_CopyToHost(void *h_dst, const void *d_src, size_t bytes);

/* ---- per-stage device timing (CUDA events around every kernel of a handle) ---------------------- */
struct LINNEB200StageStat { char name[24]; uint64_t launches; double total_ms; };
void LINNEB200_EncoderSetProfiling(struct LINNEEncoder *encoder, int on);
void LINNEB200_DecoderSetProfiling(struct LINNEDecoder *decoder, int on);
void LINNEB200_EncoderResetStageStats(struct LINNEEncoder *encoder);
void LINNEB200_DecoderResetStageStats(struct LINNEDecoder *decoder);
int  LINNEB200_EncoderGetStageStats(struct LINNEEncoder *encoder, struct LINNEB200StageStat *out, int max_stages);
int  LINNEB200_DecoderGetStageStats(struct LINNEDecoder *decoder, struct LINNEB200StageStat *out, int max_stages);

/* Launch timeline of a profiled handle: kernel begin/end in ms since a process-wide origin (recorded when
 * profiling is first switched on), so handles running side by side on their own streams can be merged. */
struct LINNEB200TimelineEntry { char name[24]; float begin_ms, end_ms; };
int  LINNEB200_EncoderGetTimeline(struct LINNEEncoder *encoder, struct LINNEB200TimelineEntry *out, int max_entries);
int  LINNEB200_DecoderGetTimeline(struct LINNEDecoder *decoder, struct LINNEB200TimelineEntry *out, int max_entries);

/* Sustained FP64 FMA throughput (TFLOP/s) of the current device: roofline denominator of the
 * encoder's analysis kernels.  Returns 0 without a device. */
double LINNEB200_MeasureFp64Tflops(void);

#ifdef __cplusplus
}
#endif
#endif
