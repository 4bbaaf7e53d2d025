/* lnb_shim_cuda.cu -- CUDA implementation of lnb_shim.h for sm_100a (B200).
 *
 * Round-1 kernel shape: every pipeline stage is a flat grid of independent work items (one thread
 * per block / block-channel / unit, see lnb_pipeline.cuh).  The grid is sized in whole waves of
 * 148 SMs where the item count allows.
 */
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <sched.h>
#include <string.h>

#include "lnb_shim.h"
#include "lnb_pipeline.cuh"
#include "lnb_analyze_v3.cuh"
#include "lnb_pack_v2.cuh"
#include "lnb_front_v2.cuh"
#include "lnb_synth_v2.cuh"
#include "lnb_crc_v2.cuh"
#include "lnb_entropy_v3.cuh"
#include "lnb_refine_v2.cuh"
#include "lnb_scan_v2.cuh"
#include "lnb_stream_v2.cuh"
#include "lnb_hop.cuh"
#include "lnb_window.cuh"
#include "lnb_salvage.cuh"

#define LNB_MAX_STAGES 32
#define LNB_MAX_PENDING 8192
#define LNB_MAX_TIMELINE 2048

struct LnbDevice {
    cudaStream_t stream;
    int owns_stream;
    int cost_rank;
    int ordinal;
    LnbDevTables tables;
    void *table_mem;
    uint64_t launches;
    cudaError_t last_error;
    /* optional per-stage timing */
    int profiling;
    int num_stages;
    LnbStageStat stages[LNB_MAX_STAGES];
    int num_pending;
    cudaEvent_t ev_begin[LNB_MAX_PENDING], ev_end[LNB_MAX_PENDING];
    int pending_stage[LNB_MAX_PENDING];
    int events_created;
    int num_timeline;
    LnbTimelineEntry timeline[LNB_MAX_TIMELINE];
    cudaEvent_t sync_event;              /* LINNE_B200_SYNC=block: host threads sleep in the driver instead of spinning */
    int blocking_sync;
    int yield_sync;
    /* side stream of the throughput decoder: the per-block pipeline kernel for the few blocks the lane-per-block
     * kernels leave (tail blocks) runs beside them instead of behind them */
    cudaStream_t aux_stream;
    cudaEvent_t ev_fork, ev_join;
    int aux_created;
};

static cudaEvent_t g_ref_event;              /* process-wide time origin of the launch timelines */
static int g_ref_recorded = 0;

/* The CUDA "current device" is per host thread: a handle created on one thread (and device) may be
 * driven from another, so every entry point re-binds the calling thread to the handle's device. */
static inline void bind_device(const LnbDevice *dev)
{
    int cur = -1;
    if (cudaGetDevice(&cur) != cudaSuccess || cur != dev->ordinal) cudaSetDevice(dev->ordinal);
}

static int stage_index(LnbDevice *dev, const char *name)
{
    for (int i = 0; i < dev->num_stages; i++) if (strcmp(dev->stages[i].name, name) == 0) return i;
    if (dev->num_stages >= LNB_MAX_STAGES) return LNB_MAX_STAGES - 1;
    LnbStageStat *s = &dev->stages[dev->num_stages];
    memset(s, 0, sizeof(*s));
    strncpy(s->name, name, sizeof(s->name) - 1);
    return dev->num_stages++;
}

static void drain_profile(LnbDevice *dev)
{
    for (int i = 0; i < dev->num_pending; i++) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, dev->ev_begin[i], dev->ev_end[i]) == cudaSuccess) {
            dev->stages[dev->pending_stage[i]].total_ms += ms;
            dev->stages[dev->pending_stage[i]].launches += 1;
            float t0 = 0.f;
            if (g_ref_recorded && dev->num_timeline < LNB_MAX_TIMELINE
                && cudaEventElapsedTime(&t0, g_ref_event, dev->ev_begin[i]) == cudaSuccess) {
                LnbTimelineEntry *e = &dev->timeline[dev->num_timeline++];
                memcpy(e->name, dev->stages[dev->pending_stage[i]].name, sizeof(e->name));
                e->begin_ms = t0; e->end_ms = t0 + ms;
            }
        }
    }
    dev->num_pending = 0;
}

template <class F>
__global__ void __launch_bounds__(128) lnb_items_kernel(uint32_t n, F f)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) f(i);
}

/* one work item per WARP (lane 0 runs it): for strictly serial items such as the entropy decode of a
 * block, where lanes of one warp would otherwise serialise each other's divergent paths */
template <class F>
__global__ void __launch_bounds__(128) lnb_items_per_warp_kernel(uint32_t n, F f)
{
    const uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (i < n && (threadIdx.x & 31u) == 0u) f(i);
}

/* layer shapes the throughput decoder is instantiated for (the presets of linne_internal.c:16-41) */
static int lnb_tput_shape(const LnbStreamCfg *cfg)
{
    const uint32_t *P = cfg->layer_params;
    if (cfg->num_layers == 2u && P[0] == 2u && P[1] == 32u) return 1;
    if (cfg->num_layers == 3u && P[0] == 4u && P[1] == 64u && P[2] == 8u) return 2;
    if (cfg->num_layers == 3u && P[0] == 4u && P[1] == 128u && P[2] == 16u) return 3;
    return 0;
}

struct CudaExec {
    static constexpr bool cooperative = true;
    LnbDevice *dev;
    template <class F> void run_per_warp(const char *name, uint32_t n, const F &f)
    {
        if (n == 0) return;
        const int slot = begin_stage(name);
        lnb_items_per_warp_kernel<F><<<(n + 3u) / 4u, 128, 0, dev->stream>>>(n, f);
        end_stage(slot);
    }
    void entropy_cooperative(const LnbDecodeBatch &b)
    {
        const int slot = begin_stage("entropy_v3");
        lnb_entropy_v3_kernel<<<(b.num_blocks + LNB_E3_WARPS - 1) / LNB_E3_WARPS, LNB_E3_THREADS, 0, dev->stream>>>(b);
        end_stage(slot);
    }
    /* dynamic shared memory of the per-block decoders: one line of the longest block of the batch */
    static uint32_t line_samples(const LnbDecodeBatch &b, uint32_t cap)
    {
        uint32_t n_max = b.max_nsmp < cap ? b.max_nsmp : cap;
        if (n_max == 0u) n_max = 4u;
        return (n_max + 3u) & ~3u;
    }
    void stream_cooperative(const LnbDecodeBatch &b, cudaStream_t on = nullptr)
    {
        const uint32_t n_max = line_samples(b, LNB_DS_MAX_N);
        const size_t smem = (size_t)n_max * sizeof(int32_t);
        const int slot = begin_stage("stream_v2", on);
        /* the walk on one lane (default) or as a warp (LINNE_B200_WALK=warp; measured slower inside this kernel, kept for
         * A/B runs): lnb_stream_v2.cuh */
        const char *walk_env = getenv("LINNE_B200_WALK");         /* read per call: the tests switch forms inside one process */
        const bool lane_walk = !(walk_env && walk_env[0] == 'w');
        LnbDecodeBatch b2 = b;
#ifdef LNB_DS_TIMING
        if (getenv("LINNE_B200_DBG_WALKONLY")) b2.cfg.check_crc |= 0x100u;
#endif
        if (lane_walk) lnb_stream_v2_kernel<false><<<b.num_blocks, LNB_DS_THREADS, smem, on ? on : dev->stream>>>(b2, n_max);
        else lnb_stream_v2_kernel<true><<<b.num_blocks, LNB_DS_THREADS, smem, on ? on : dev->stream>>>(b2, n_max);
        end_stage(slot, on);
    }
    template <int Q0, int Q1, int Q2> void tput_synth(const LnbDecodeBatch &b)
    {
        const size_t smem = LnbTpLayer<Q0>::smem_bytes + LnbTpLayer<Q1>::smem_bytes + LnbTpLayer<Q2>::smem_bytes + 16u;
        const uint32_t seqs = b.num_blocks * b.cfg.num_channels;
        const int slot = begin_stage("tp_synth");
        lnb_tp_synth_kernel<Q0, Q1, Q2><<<(seqs + 31u) / 32u, 32, smem, dev->stream>>>(b);
        end_stage(slot);
    }
    /* Large batches (b.tput, lnb_tput_v2.cuh).  The entropy stage needs nothing from the CRC pass -- it decodes every
     * full block and the synthesis stage drops those whose CRC failed -- so the CRC pass and the per-block pipeline
     * kernel for what the lane-per-block kernels leave (tail blocks) run beside it on a side stream:
     *     side:  crc_v2 -> stream_v2            main:  tp_entropy -> (join) -> tp_synth                          */
    void tput_decode(const LnbDecodeBatch &b)
    {
        const int shape = lnb_tput_shape(&b.cfg);           /* non-zero: the host asked lnb_shim_tput_supported(cfg) */
        if (!dev->aux_created) {
            int prio = 0;                                       /* the side stream runs at the priority of the handle's own */
            if (cudaStreamGetPriority(dev->stream, &prio) != cudaSuccess) { cudaGetLastError(); prio = 0; }
            cudaStreamCreateWithPriority(&dev->aux_stream, cudaStreamNonBlocking, prio);
            cudaEventCreateWithFlags(&dev->ev_fork, cudaEventDisableTiming);
            cudaEventCreateWithFlags(&dev->ev_join, cudaEventDisableTiming);
            dev->aux_created = 1;
        }
        cudaEventRecord(dev->ev_fork, dev->stream);
        cudaStreamWaitEvent(dev->aux_stream, dev->ev_fork, 0);
        {
            const int slot = begin_stage("crc_v2", dev->aux_stream);
            lnb_crc_v2_kernel<<<b.num_blocks, LNB_CRC_THREADS, 0, dev->aux_stream>>>(b);
            end_stage(slot, dev->aux_stream);
            stream_cooperative(b, dev->aux_stream);
        }
        cudaEventRecord(dev->ev_join, dev->aux_stream);
        const int slot = begin_stage("tp_entropy");
        /* eight lanes per block with fix-up rounds (default); LINNE_B200_TP_ENTROPY=8: rounds that end at the first long code
         * word (round 1), =w: a warp per block, =l / =s: a lane per block, one code word per pass / groups of eight (measured
         * alternatives, profiles/r2_tp_entropy_forms.md) */
        const char *form_env = getenv("LINNE_B200_TP_ENTROPY");  /* read per call: the tests switch forms inside one process */
        const char form = form_env && form_env[0] ? form_env[0] : 'i';
        const uint32_t grid8 = (b.num_blocks + LNB_TG_PER_WARP - 1u) / LNB_TG_PER_WARP;
        if (form == '8') lnb_tp_entropy_kernel<false><<<grid8, 32, 0, dev->stream>>>(b);
        else if (form == 'w') lnb_tp_entropy_w_kernel<<<(b.num_blocks + LNB_TW_WARPS - 1u) / LNB_TW_WARPS, 32u * LNB_TW_WARPS, 0, dev->stream>>>(b);
        else if (form == 'l') lnb_tp_entropy_l_kernel<<<(b.num_blocks + 31u) / 32u, 32, 0, dev->stream>>>(b);
        else if (form == 's') lnb_tp_entropy_s_kernel<<<(b.num_blocks + 31u) / 32u, 32, 0, dev->stream>>>(b);
        else lnb_tp_entropy_kernel<true><<<grid8, 32, 0, dev->stream>>>(b);
        end_stage(slot);
        cudaStreamWaitEvent(dev->stream, dev->ev_join, 0);
        if (shape == 1) tput_synth<32, 2, 0>(b);
        else if (shape == 2) tput_synth<8, 64, 4>(b);
        else tput_synth<16, 128, 4>(b);
    }
    void crc_cooperative(const LnbDecodeBatch &b)
    {
        const int slot = begin_stage("crc_v2");
        lnb_crc_v2_kernel<<<b.num_blocks, LNB_CRC_THREADS, 0, dev->stream>>>(b);
        end_stage(slot);
    }
    uint32_t synth_max_n() const { return LNB_SY_MAX_N; }
    void synth_cooperative(const LnbDecodeBatch &b)
    {
        const uint32_t items = b.num_blocks * b.cfg.num_channels;
        const uint32_t n_max = line_samples(b, LNB_SY_MAX_N);
        const size_t smem = (size_t)LNB_SY_WARPS * n_max * sizeof(int32_t);
        const int slot = begin_stage("synth_v2");
        lnb_synth_v2_kernel<<<(items + LNB_SY_WARPS - 1) / LNB_SY_WARPS, LNB_SY_THREADS, smem, dev->stream>>>(b, n_max);
        end_stage(slot);
    }
    int begin_stage(const char *name, cudaStream_t on = nullptr)
    {
        if (!dev->profiling) return -1;
        if (dev->num_pending >= LNB_MAX_PENDING) {
            cudaStreamSynchronize(dev->stream);
            if (dev->aux_created) cudaStreamSynchronize(dev->aux_stream);
            drain_profile(dev);
        }
        const int slot = dev->num_pending++;
        dev->pending_stage[slot] = stage_index(dev, name);
        cudaEventRecord(dev->ev_begin[slot], on ? on : dev->stream);
        return slot;
    }
    void end_stage(int slot, cudaStream_t on = nullptr)
    {
        if (slot >= 0) cudaEventRecord(dev->ev_end[slot], on ? on : dev->stream);
        dev->launches++;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess && dev->last_error == cudaSuccess) dev->last_error = e;
    }
    void scan_cooperative(const LnbEncodeBatch &b)
    {
        const int slot = begin_stage("scan_v2");
        lnb_scan_v2_kernel<<<1, LNB_SC_THREADS, 0, dev->stream>>>(b);
        end_stage(slot);
    }
    void refine_cooperative(const LnbEncodeBatch &b, uint32_t chunks_per_slot)
    {
        uint32_t na_max = b.cfg.block_size;
        uint32_t max_p = 0;
        for (uint32_t l = 0; l < b.cfg.num_layers; l++) if (b.cfg.layer_params[l] > max_p) max_p = b.cfg.layer_params[l];
        const uint32_t tri = max_p * (max_p + 1u) / 2u;          /* the signal buffers double as the packed Gram matrix */
        if (b.af_iterations && na_max < tri) na_max = tri;
        na_max = (na_max + 7u) & ~7u;
        /* signals in shared memory while they fit; blocks beyond LNB_RF_MAX_NA samples take the global scratch the host sized for them */
        const bool global_xy = b.refine_xy != nullptr;
        const size_t smem = (global_xy ? 0u : (size_t)2 * (na_max + LNB_RF_HIST) * sizeof(double)) + sizeof(LnbRefineSmem);
        const int slot = begin_stage("refine_v2");
        lnb_refine_v2_kernel<<<b.num_blocks * b.cfg.num_channels, LNB_RF_THREADS, smem, dev->stream>>>(
            b, na_max, b.af_iterations, b.enable_learning, b.train_scratch, chunks_per_slot, global_xy ? b.refine_xy : nullptr);
        end_stage(slot);
    }
    void prepare_cooperative(const LnbEncodeBatch &b)
    {
        const int slot = begin_stage("prepare_v2");
        lnb_prepare_v2_kernel<<<b.num_blocks, LNB_FR_THREADS, 0, dev->stream>>>(b);
        end_stage(slot);
    }
    void predict_plan_cooperative(const LnbEncodeBatch &b)
    {
        uint32_t n_max = b.cfg.block_size < LNB_FR_MAX_N ? b.cfg.block_size : LNB_FR_MAX_N;
        n_max = (n_max + 3u) & ~3u;
        const size_t smem = (size_t)2 * n_max * sizeof(int32_t) + sizeof(LnbPlanSmem);
        const int slot = begin_stage("predict_plan_v2");
        lnb_predict_plan_v2_kernel<<<b.num_blocks * b.cfg.num_channels, LNB_FR_THREADS, smem, dev->stream>>>(b, n_max);
        end_stage(slot);
    }
    void pack_cooperative(const LnbEncodeBatch &b, uint32_t out_capacity)
    {
        /* staging buffer: the raw-block size bound of this stream format plus slack, capped by the SM */
        size_t bytes = 64 + LNB_BLOCK_HEADER_SIZE + (size_t)b.cfg.block_size * b.cfg.num_channels * ((b.cfg.bits_per_sample + 7u) / 8u);
        bytes += bytes / 8;
        if (bytes > 220u * 1024u) bytes = 220u * 1024u;
        const uint32_t img_words = (uint32_t)((bytes + 3) / 4);
        const int slot = begin_stage("pack_v2");
        lnb_pack_v2_kernel<<<b.num_blocks, LNB_PK_THREADS, (size_t)img_words * 4, dev->stream>>>(b, out_capacity, img_words);
        end_stage(slot);
    }
    void analyze_cooperative(const LnbEncodeBatch &b)
    {
        const uint32_t S = b.num_blocks * b.cfg.num_channels * b.cfg.num_lambdas;
        uint32_t na_max = b.cfg.block_size < LNB_A3_MAX_NA ? b.cfg.block_size : LNB_A3_MAX_NA;
        na_max = (na_max + 7u) & ~7u;
        const size_t smem = lnb_a3_smem_doubles(na_max) * sizeof(double);
        const int slot = begin_stage("analyze_v3");
        lnb_analyze_v3_kernel<<<S, LNB_A3_THREADS, smem, dev->stream>>>(b, na_max);
        end_stage(slot);
    }
    template <class F> void run(const char *name, uint32_t n, const F &f)
    {
        if (n == 0) return;
        const uint32_t threads = 128;
        const uint32_t grid = (n + threads - 1) / threads;
        int slot = -1;
        if (dev->profiling) {
            if (dev->num_pending >= LNB_MAX_PENDING) { cudaStreamSynchronize(dev->stream); drain_profile(dev); }
            slot = dev->num_pending++;
            dev->pending_stage[slot] = stage_index(dev, name);
            cudaEventRecord(dev->ev_begin[slot], dev->stream);
        }
        lnb_items_kernel<F><<<grid, threads, 0, dev->stream>>>(n, f);
        if (slot >= 0) cudaEventRecord(dev->ev_end[slot], dev->stream);
        dev->launches++;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess && dev->last_error == cudaSuccess) dev->last_error = e;
    }
};

/* Dynamic shared memory above 48 KB is an opt-in per kernel AND per device.  Every kernel that may need it gets the
 * device's maximum once, when the first context of that device is opened (under a lock: handles are opened from
 * many worker threads), and the attribute is never lowered afterwards -- a launcher only passes the size it needs. */
#include <mutex>
static std::mutex g_kernel_cfg_lock;
static unsigned char g_kernel_cfg_done[64];

template <class K> static cudaError_t lnb_optin_smem(K kernel, int optin_bytes)
{
    cudaFuncAttributes at;
    cudaError_t e = cudaFuncGetAttributes(&at, kernel);
    if (e != cudaSuccess) return e;
    const int dyn = optin_bytes - (int)at.sharedSizeBytes;
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn > 0 ? dyn : 0);
}
static int lnb_configure_kernels(int ordinal)
{
    std::lock_guard<std::mutex> guard(g_kernel_cfg_lock);
    if (ordinal >= 0 && ordinal < 64 && g_kernel_cfg_done[ordinal]) return 0;
    int optin = 0;
    if (cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, ordinal) != cudaSuccess) return 1;
    cudaError_t e = cudaSuccess;
    if (e == cudaSuccess) e = lnb_optin_smem(lnb_stream_v2_kernel<true>, optin);
    if (e == cudaSuccess) e = lnb_optin_smem(lnb_stream_v2_kernel<false>, optin);
    if (e == cudaSuccess) e = lnb_optin_smem(lnb_tp_synth_kernel<32, 2, 0>, optin);
    if (e == cudaSuccess) e = lnb_optin_smem(lnb_tp_synth_kernel<8, 64, 4>, optin);
    if (e == cudaSuccess) e = lnb_optin_smem(lnb_tp_synth_kernel<16, 128, 4>, optin);
    if (e == cudaSuccess) e = lnb_optin_smem(lnb_synth_v2_kernel, optin);
    if (e == cudaSuccess) e = lnb_optin_smem(lnb_refine_v2_kernel, optin);
    if (e == cudaSuccess) e = lnb_optin_smem(lnb_predict_plan_v2_kernel, optin);
    if (e == cudaSuccess) e = lnb_optin_smem(lnb_pack_v2_kernel, optin);
    if (e == cudaSuccess) e = lnb_optin_smem(lnb_analyze_v3_kernel, optin);
    if (e != cudaSuccess) {
        fprintf(stderr, "linne_b200: cannot configure kernels on device %d: %s\n", ordinal, cudaGetErrorString(e));
        cudaGetLastError();
        return 1;
    }
    if (ordinal >= 0 && ordinal < 64) g_kernel_cfg_done[ordinal] = 1;
    return 0;
}

extern "C" {

const char *lnb_shim_backend(void) { return "cuda-sm_100a"; }
int lnb_shim_device_count(void) { int n = 0; if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; } return n; }
int lnb_shim_set_device(int ordinal) { if (cudaSetDevice(ordinal) != cudaSuccess) { cudaGetLastError(); return 1; } return 0; }
int lnb_shim_device_ordinal(const LnbDevice *dev) { return dev->ordinal; }
int lnb_shim_current_device(void) { int d = -1; if (cudaGetDevice(&d) != cudaSuccess) { cudaGetLastError(); return -1; } return d; }
uint32_t lnb_shim_fast_max_na(void) { return LNB_A3_MAX_NA; }
uint32_t lnb_shim_coop_max_n(void) { return LNB_FR_MAX_N; }
uint32_t lnb_shim_refine_max_na(void) { return LNB_RF_MAX_NA; }
uint32_t lnb_shim_refine_hist(void) { return LNB_RF_HIST; }
uint32_t lnb_shim_fused_max_n(void) { return LNB_DS_MAX_N; }
int lnb_shim_tput_supported(const LnbStreamCfg *cfg)
{
    return lnb_tput_shape(cfg) != 0 && cfg->block_size <= LNB_DS_MAX_N && (cfg->block_size & 1023u) == 0u
        && cfg->bits_per_sample <= 31u && !(cfg->ms && (cfg->num_channels & 1u));
}

int lnb_shim_open(LnbDevice **out, int device_ordinal)
{
    int count = 0;
    /* Handles, their side streams and the ranges of a pipelined call each own a stream; with the default of eight
     * hardware queues unrelated streams share one and wait for each other's copies and kernels.  Only effective while
     * the process has not created its CUDA context yet (a host that did so first sets the variable itself). */
    {
        static int once = 0;                                     /* the environment is touched by the first open only */
        if (!__atomic_exchange_n(&once, 1, __ATOMIC_ACQ_REL)) setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0);
    }
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) return 1;
    if (device_ordinal >= 0) {
        if (device_ordinal >= count || cudaSetDevice(device_ordinal) != cudaSuccess) return 2;
    }
    LnbDevice *dev = (LnbDevice *)calloc(1, sizeof(LnbDevice));
    if (!dev) return 3;
    cudaGetDevice(&dev->ordinal);
    if (lnb_configure_kernels(dev->ordinal)) { free(dev); return 7; }
    if (cudaStreamCreateWithFlags(&dev->stream, cudaStreamNonBlocking) != cudaSuccess) { free(dev); return 4; }
    dev->owns_stream = 1;
    dev->cost_rank = -1;
    {   /* many handles driven from many host threads (several ranks per box) oversubscribe the cores when every
         * waiting thread spins; LINNE_B200_SYNC=block makes the waits sleep (a little more wake-up latency) */
        const char *mode = getenv("LINNE_B200_SYNC");
        if (mode && mode[0] == 'b' && cudaEventCreateWithFlags(&dev->sync_event, cudaEventBlockingSync | cudaEventDisableTiming) == cudaSuccess)
            dev->blocking_sync = 1;
        /* LINNE_B200_SYNC=yield: poll the stream and give the core away between polls -- no wake-up latency, and waiting
         * threads that outnumber the cores do not starve the ones with work */
        if (mode && mode[0] == 'y') dev->yield_sync = 1;
    }

    const LnbHostTables *ht = lnb_tables_get();
    const size_t sz_lut = sizeof(ht->huff_lut), sz_code = sizeof(ht->huff_code), sz_len = 256,
                 sz_thr = sizeof(ht->k2_threshold), sz_crc = sizeof(ht->crc_table);
    const size_t total = sz_lut + sz_code + sz_thr + sz_crc + sz_len + 64;
    uint8_t *mem = NULL;
    if (cudaMalloc((void **)&mem, total) != cudaSuccess) { cudaStreamDestroy(dev->stream); free(dev); return 5; }
    size_t off = 0;
    /* doubles first (8-byte alignment), then 4-, 2-, 1-byte tables */
    cudaMemcpy(mem + off, ht->k2_threshold, sz_thr, cudaMemcpyHostToDevice); dev->tables.k2_threshold = (const double *)(mem + off); off += sz_thr;
    cudaMemcpy(mem + off, ht->huff_code, sz_code, cudaMemcpyHostToDevice);   dev->tables.huff_code = (const uint32_t *)(mem + off); off += sz_code;
    cudaMemcpy(mem + off, ht->huff_lut, sz_lut, cudaMemcpyHostToDevice);     dev->tables.huff_lut = (const uint16_t *)(mem + off); off += sz_lut;
    cudaMemcpy(mem + off, ht->crc_table, sz_crc, cudaMemcpyHostToDevice);    dev->tables.crc_table = (const uint16_t *)(mem + off); off += sz_crc;
    cudaMemcpy(mem + off, ht->huff_len, sz_len, cudaMemcpyHostToDevice);     dev->tables.huff_len = (const uint8_t *)(mem + off); off += sz_len;
    dev->table_mem = mem;
    if (cudaDeviceSynchronize() != cudaSuccess) { cudaFree(mem); cudaStreamDestroy(dev->stream); free(dev); return 6; }
    *out = dev;
    return 0;
}

void lnb_shim_close(LnbDevice *dev)
{
    bind_device(dev);
    if (!dev) return;
    cudaStreamSynchronize(dev->stream);
    if (dev->events_created)
        for (int i = 0; i < LNB_MAX_PENDING; i++) { cudaEventDestroy(dev->ev_begin[i]); cudaEventDestroy(dev->ev_end[i]); }
    cudaFree(dev->table_mem);
    if (dev->blocking_sync) cudaEventDestroy(dev->sync_event);
    if (dev->aux_created) { cudaStreamDestroy(dev->aux_stream); cudaEventDestroy(dev->ev_fork); cudaEventDestroy(dev->ev_join); }
    if (dev->owns_stream) cudaStreamDestroy(dev->stream);
    free(dev);
}

const LnbDevTables *lnb_shim_tables(const LnbDevice *dev) { return &dev->tables; }

void lnb_shim_use_stream(LnbDevice *dev, void *cuda_stream)
{
    bind_device(dev);
    if (dev->owns_stream) { cudaStreamSynchronize(dev->stream); cudaStreamDestroy(dev->stream); dev->owns_stream = 0; }
    dev->stream = (cudaStream_t)cuda_stream;
}

void lnb_shim_set_cost_rank(LnbDevice *dev, int cost_rank)
{
    bind_device(dev);
    if (!dev->owns_stream || dev->cost_rank == cost_rank) return;
    { const char *e = getenv("LINNE_B200_STREAM_PRIORITY"); if (e && *e == '0') return; }
    int least = 0, greatest = 0;                              /* numerically: greatest priority <= least priority */
    if (cudaDeviceGetStreamPriorityRange(&least, &greatest) != cudaSuccess) { cudaGetLastError(); return; }
    int span = least - greatest;
    if (span <= 0) return;
    if (cost_rank < 0) cost_rank = 0;
    if (cost_rank > 7) cost_rank = 7;
    const int prio = least - (cost_rank * span + 3) / 7;
    cudaStream_t s;
    if (cudaStreamCreateWithPriority(&s, cudaStreamNonBlocking, prio) != cudaSuccess) { cudaGetLastError(); return; }
    cudaStreamSynchronize(dev->stream);
    cudaStreamDestroy(dev->stream);
    dev->stream = s;
    dev->cost_rank = cost_rank;
    if (dev->aux_created) {                                      /* re-created at the new priority when next needed */
        cudaStreamSynchronize(dev->aux_stream);
        cudaStreamDestroy(dev->aux_stream); cudaEventDestroy(dev->ev_fork); cudaEventDestroy(dev->ev_join);
        dev->aux_created = 0;
    }
}

void *lnb_shim_alloc(LnbDevice *dev, size_t bytes)
{
    void *p = NULL;
    bind_device(dev);
    if (bytes == 0) bytes = 16;
    if (cudaMalloc(&p, bytes) != cudaSuccess) { cudaGetLastError(); return NULL; }
    return p;
}
void lnb_shim_free(LnbDevice *dev, void *ptr) { bind_device(dev); if (ptr) cudaFree(ptr); }
void *lnb_shim_alloc_pinned(size_t bytes)
{
    void *p = NULL;
    if (cudaMallocHost(&p, bytes ? bytes : 16) != cudaSuccess) { cudaGetLastError(); return NULL; }
    return p;
}
void lnb_shim_free_pinned(void *ptr) { if (ptr) cudaFreeHost(ptr); }

static int note(LnbDevice *dev, cudaError_t e)
{
    if (e != cudaSuccess && dev->last_error == cudaSuccess) dev->last_error = e;
    return e == cudaSuccess ? 0 : 1;
}
int lnb_shim_h2d(LnbDevice *dev, void *dst, const void *src, size_t bytes)
{
    bind_device(dev);
    return bytes ? note(dev, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, dev->stream)) : 0;
}
int lnb_shim_d2d(LnbDevice *dev, void *dst, const void *src, size_t bytes)
{
    bind_device(dev);
    return bytes ? note(dev, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, dev->stream)) : 0;
}
int lnb_shim_d2h(LnbDevice *dev, void *dst, const void *src, size_t bytes)
{
    bind_device(dev);
    return bytes ? note(dev, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, dev->stream)) : 0;
}
int lnb_shim_memset(LnbDevice *dev, void *dst, int value, size_t bytes)
{
    bind_device(dev);
    return bytes ? note(dev, cudaMemsetAsync(dst, value, bytes, dev->stream)) : 0;
}
int lnb_shim_sync(LnbDevice *dev)
{
    bind_device(dev);
    cudaError_t e;
    if (dev->blocking_sync) {
        e = cudaEventRecord(dev->sync_event, dev->stream);
        if (e == cudaSuccess) e = cudaEventSynchronize(dev->sync_event);
    } else if (dev->yield_sync) {
        while ((e = cudaStreamQuery(dev->stream)) == cudaErrorNotReady) sched_yield();
    } else {
        e = cudaStreamSynchronize(dev->stream);
    }
    if (e == cudaSuccess && dev->profiling) drain_profile(dev);
    if (e == cudaSuccess) e = dev->last_error;
    if (e != cudaSuccess) {
        fprintf(stderr, "linne_b200: CUDA error: %s\n", cudaGetErrorString(e));
        dev->last_error = cudaSuccess;
        cudaGetLastError();
        return 1;
    }
    return 0;
}

int lnb_shim_decode(LnbDevice *dev, const LnbDecodeBatch *batch)
{
    bind_device(dev);
    CudaExec ex{dev};
    lnb_decode_pipeline(ex, *batch);
    return dev->last_error == cudaSuccess ? 0 : 1;
}
int lnb_shim_encode_analyze(LnbDevice *dev, const LnbEncodeBatch *batch)
{
    bind_device(dev);
    CudaExec ex{dev};
    lnb_encode_analyze_pipeline(ex, *batch);
    return dev->last_error == cudaSuccess ? 0 : 1;
}
int lnb_shim_encode_pack(LnbDevice *dev, const LnbEncodeBatch *batch, uint32_t out_capacity)
{
    bind_device(dev);
    CudaExec ex{dev};
    lnb_encode_pack_pipeline(ex, *batch, out_capacity);
    return dev->last_error == cudaSuccess ? 0 : 1;
}

int lnb_shim_hop(LnbDevice *dev, const uint8_t *d_image, const LnbHopFile *d_files, uint32_t num_files,
                 LnbBlockDesc *d_table, LnbHopResult *d_results)
{
    bind_device(dev);
    if (num_files == 0) return 0;
    CudaExec ex{dev};
    const int slot = ex.begin_stage("hop");
    lnb_hop_kernel<<<num_files, 32, 0, dev->stream>>>(d_image, d_files, num_files, d_table, d_results);
    ex.end_stage(slot);
    return dev->last_error == cudaSuccess ? 0 : 1;
}

int lnb_shim_seek_blocks(LnbDevice *dev, const uint8_t *d_image, const LnbSeekIn *d_in, uint32_t n,
                         uint32_t channels, uint32_t bits, LnbBlockDesc *d_out)
{
    bind_device(dev);
    CudaExec ex{dev};
    lnb_seek_pipeline(ex, d_image, d_in, n, channels, bits, d_out);
    return dev->last_error == cudaSuccess ? 0 : 1;
}
int lnb_shim_gather_windows(LnbDevice *dev, const int32_t *d_scratch, uint32_t scratch_stride, const LnbGatherWin *d_wins,
                            uint32_t num_wins, uint32_t num_items, int32_t *d_dst, uint32_t dst_stride)
{
    bind_device(dev);
    CudaExec ex{dev};
    lnb_gather_windows_pipeline(ex, d_scratch, scratch_stride, d_wins, num_wins, num_items, d_dst, dst_stride);
    return dev->last_error == cudaSuccess ? 0 : 1;
}
int lnb_shim_gather_windows_packed(LnbDevice *dev, const int32_t *d_scratch, uint32_t scratch_stride, const LnbGatherWin *d_wins,
                                   uint32_t num_wins, uint32_t num_items, uint8_t *d_dst, uint32_t channels, uint32_t bytes)
{
    bind_device(dev);
    CudaExec ex{dev};
    lnb_gather_windows_packed_pipeline(ex, d_scratch, scratch_stride, d_wins, num_wins, num_items, d_dst, channels, bytes);
    return dev->last_error == cudaSuccess ? 0 : 1;
}

int lnb_shim_resync_scan(LnbDevice *dev, const uint8_t *d_image, uint32_t data_size, uint32_t channels, uint32_t bits,
                         uint32_t block_size, LnbBlockDesc *d_table, uint32_t *d_count, uint32_t cap)
{
    bind_device(dev);
    CudaExec ex{dev};
    lnb_resync_scan_pipeline(ex, d_image, data_size, channels, bits, block_size, d_table, d_count, cap);
    return dev->last_error == cudaSuccess ? 0 : 1;
}
int lnb_shim_crc_blocks(LnbDevice *dev, const uint8_t *d_image, uint32_t data_size, LnbBlockDesc *d_table,
                        const uint32_t *d_count, uint32_t cap)
{
    bind_device(dev);
    if (cap == 0) return 0;
    CudaExec ex{dev};
    LnbDecodeBatch b;
    memset(&b, 0, sizeof(b));
    b.cfg.check_crc = 1u;
    b.tab = dev->tables;
    b.stream = d_image;
    b.stream_size = data_size;
    b.blocks = d_table;
    b.num_blocks = cap;
    const int slot = ex.begin_stage("salvage_crc");
    lnb_salvage_crc_kernel<<<cap, LNB_CRC_THREADS, 0, dev->stream>>>(b, d_count);
    ex.end_stage(slot);
    return dev->last_error == cudaSuccess ? 0 : 1;
}

int lnb_shim_unpack_pcm(LnbDevice *dev, const uint8_t *d_packed, int32_t *d_pcm, uint32_t pcm_stride,
                        uint32_t frames, uint32_t channels, uint32_t bytes)
{
    bind_device(dev);
    CudaExec ex{dev};
    lnb_unpack_pcm_pipeline(ex, d_packed, d_pcm, pcm_stride, frames, channels, bytes);
    return dev->last_error == cudaSuccess ? 0 : 1;
}
int lnb_shim_pack_pcm(LnbDevice *dev, const int32_t *d_pcm, uint8_t *d_packed, uint32_t pcm_stride,
                      uint32_t frames, uint32_t channels, uint32_t bytes)
{
    bind_device(dev);
    CudaExec ex{dev};
    lnb_pack_pcm_pipeline(ex, d_pcm, d_packed, pcm_stride, frames, channels, bytes);
    return dev->last_error == cudaSuccess ? 0 : 1;
}

uint64_t lnb_shim_launch_count(const LnbDevice *dev) { return dev->launches; }

void lnb_shim_profile_enable(LnbDevice *dev, int on)
{
    bind_device(dev);
    if (on && !g_ref_recorded) {
        cudaEventCreate(&g_ref_event);
        cudaEventRecord(g_ref_event, 0);
        cudaEventSynchronize(g_ref_event);
        g_ref_recorded = 1;
    }
    if (on && !dev->events_created) {
        for (int i = 0; i < LNB_MAX_PENDING; i++) { cudaEventCreate(&dev->ev_begin[i]); cudaEventCreate(&dev->ev_end[i]); }
        dev->events_created = 1;
    }
    cudaStreamSynchronize(dev->stream);
    drain_profile(dev);
    dev->profiling = on ? 1 : 0;
}
void lnb_shim_profile_reset(LnbDevice *dev)
{
    bind_device(dev);
    cudaStreamSynchronize(dev->stream);
    drain_profile(dev);
    for (int i = 0; i < dev->num_stages; i++) { dev->stages[i].launches = 0; dev->stages[i].total_ms = 0.0; }
    dev->num_timeline = 0;
}
int lnb_shim_profile_timeline(LnbDevice *dev, LnbTimelineEntry *out, int max_entries)
{
    bind_device(dev);
    cudaStreamSynchronize(dev->stream);
    drain_profile(dev);
    int n = dev->num_timeline < max_entries ? dev->num_timeline : max_entries;
    for (int i = 0; i < n; i++) out[i] = dev->timeline[i];
    return n;
}
int lnb_shim_profile_get(LnbDevice *dev, LnbStageStat *out, int max_stages)
{
    bind_device(dev);
    cudaStreamSynchronize(dev->stream);
    drain_profile(dev);
    int n = dev->num_stages < max_stages ? dev->num_stages : max_stages;
    for (int i = 0; i < n; i++) out[i] = dev->stages[i];
    return n;
}

/* 8 independent DFMA chains per thread, 2048 x 8 DFMA each; grid fills every SM several times over */
__global__ void __launch_bounds__(256) lnb_fp64_peak_kernel(double *sink, double a, double b)
{
    double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
#pragma unroll 16
    for (int i = 0; i < 2048; i++) {
        x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
        x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
    }
    const double s = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
    if (s == 12345.678) sink[0] = s;
}

__global__ void __launch_bounds__(256) lnb_sine_window_kernel(double *dst, uint32_t n)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    const double pi = 3.1415926535897932384626433832795029;
    if (j < n) dst[j] = sin((pi * (double)j) / (double)(n - 1u));       /* the expression of lnb_prepare_v2_kernel */
}

int lnb_shim_fill_sine_window(LnbDevice *dev, double *dst, uint32_t n)
{
    bind_device(dev);
    if (n < 2u) return 1;
    lnb_sine_window_kernel<<<(n + 255u) / 256u, 256, 0, dev->stream>>>(dst, n);
    dev->launches++;
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

double lnb_shim_measure_fp64_tflops(LnbDevice *dev)
{
    bind_device(dev);
    double *sink = NULL;
    cudaEvent_t e0, e1;
    const int grid = 148 * 16, threads = 256, reps = 5;
    float best = 1e30f;
    if (cudaMalloc(&sink, 64) != cudaSuccess) return 0.0;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    lnb_fp64_peak_kernel<<<grid, threads, 0, dev->stream>>>(sink, 0.999999, 1e-9);
    for (int r = 0; r < reps; r++) {
        float ms = 0.f;
        cudaEventRecord(e0, dev->stream);
        lnb_fp64_peak_kernel<<<grid, threads, 0, dev->stream>>>(sink, 0.999999, 1e-9);
        cudaEventRecord(e1, dev->stream);
        cudaEventSynchronize(e1);
        cudaEventElapsedTime(&ms, e0, e1);
        if (ms < best) best = ms;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(sink);
    const double flops = 2.0 * 8.0 * 2048.0 * (double)grid * threads;
    return flops / (best * 1e-3) / 1e12;
}

void *lnb_shim_device_alloc(size_t bytes)
{
    void *p = NULL;
    if (cudaMalloc(&p, bytes ? bytes : 16) != cudaSuccess) { cudaGetLastError(); return NULL; }
    return p;
}
void lnb_shim_device_free(void *ptr) { if (ptr) cudaFree(ptr); }
int lnb_shim_ipc_export(const void *ptr, unsigned char handle[64])
{
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t h;
    if (cudaIpcGetMemHandle(&h, (void *)ptr) != cudaSuccess) { cudaGetLastError(); return 1; }
    memcpy(handle, &h, 64);
    return 0;
}
void *lnb_shim_ipc_open(const unsigned char handle[64])
{
    cudaIpcMemHandle_t h;
    void *p = NULL;
    memcpy(&h, handle, 64);
    if (cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
        fprintf(stderr, "linne_b200: cudaIpcOpenMemHandle: %s\n", cudaGetErrorString(cudaGetLastError()));
        return NULL;
    }
    return p;
}
void lnb_shim_ipc_close(void *peer_ptr) { if (peer_ptr) cudaIpcCloseMemHandle(peer_ptr); }
int lnb_shim_copy(void *dst, const void *src, size_t bytes, int kind)
{
    const cudaMemcpyKind k = kind == 1 ? cudaMemcpyHostToDevice : kind == 2 ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    if (bytes == 0) return 0;
    if (cudaMemcpy(dst, src, bytes, k) != cudaSuccess) {
        fprintf(stderr, "linne_b200: cudaMemcpy: %s\n", cudaGetErrorString(cudaGetLastError()));
        return 1;
    }
    return 0;
}

}  /* extern "C" */
