/* lnb_front_v2.cuh -- cooperative encoder front/back ends around the analysis kernel.
 *
 *   lnb_prepare_v2_kernel        one CTA per block: block-type estimate, copy + M/S + 2x pre-emphasis
 *                                (replaces flat stages E0 + E1; reference rows a3, a5, a6)
 *   lnb_predict_plan_v2_kernel   one CTA per (block, channel): integer predictor cascade in shared
 *                                memory, then the residual coder's partition search
 *                                (replaces flat stages E6 + E7; reference rows a17, a19)
 *
 * Both take blocks of at most LNB_FR_MAX_N samples per channel (flag LNB_ENC_FLAG_COOP); longer
 * blocks keep the flat kernels.
 */
#pragma once
#include "lnb_common.cuh"
#include "lnb_encode_core.cuh"

#define LNB_FR_THREADS 256
#define LNB_FR_MAX_N   10240
#define LNB_FR_T       (LNB_FR_MAX_N / LNB_FR_THREADS)      /* samples per thread (register resident) */

/* deterministic block-wide sum (double); result in every thread */
__device__ __forceinline__ double lnb_fr_sum(double v, double *scratch /* [8] */)
{
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    __syncthreads();
    if ((threadIdx.x & 31u) == 0) scratch[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < LNB_FR_THREADS / 32; w++) s += scratch[w];
    __syncthreads();
    return s;
}

/* the same for N values at once: every value sees exactly the operations (and their order) lnb_fr_sum gives it, behind
 * three barriers instead of 3 N.  scratch: [N * 8] */
template <int N>
__device__ __forceinline__ void lnb_fr_sum_n(double (&v)[N], double *scratch)
{
#pragma unroll
    for (int k = 0; k < N; k++) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], off);
    }
    __syncthreads();
    if ((threadIdx.x & 31u) == 0) {
#pragma unroll
        for (int k = 0; k < N; k++) scratch[k * 8 + (threadIdx.x >> 5)] = v[k];
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < N; k++) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < LNB_FR_THREADS / 32; w++) s += scratch[k * 8 + w];
        v[k] = s;
    }
    __syncthreads();
}

/* ------------------------------------------------------------------------------------------------
 * Prepare: reference linne_encoder.c:480-529 (type decision, via lpc.c:810-865) and :613-641.
 * Thread c owns samples [c*T, c*T+T), T = ceil(n/256) <= 40, held in registers.
 * ------------------------------------------------------------------------------------------------ */
__global__ void __launch_bounds__(LNB_FR_THREADS) lnb_prepare_v2_kernel(LnbEncodeBatch b)
{
    __shared__ double red[9 * 8];
    __shared__ double est_sum;
    __shared__ int32_t edge_first[LNB_FR_THREADS + 1], edge_last[LNB_FR_THREADS + 1];
    __shared__ int32_t bcast[4];

    const uint32_t tid = threadIdx.x;
    LnbBlockDesc &gblk = b.blocks[blockIdx.x];
    const LnbBlockDesc blk = gblk;
    if (!(blk.status & LNB_ENC_FLAG_COOP)) return;
    const uint32_t C = b.cfg.num_channels, n = blk.nsmp;
    const uint32_t T = (n + LNB_FR_THREADS - 1u) / LNB_FR_THREADS;
    const uint32_t i0 = tid * T;
    const uint32_t cnt = (i0 < n) ? ((n - i0 < T) ? n - i0 : T) : 0u;      /* samples this thread owns */

    /* ---- (a) entropy estimate per channel: sine window, order P0 autocorrelation + Levinson ---- */
    {
        const uint32_t p0 = (b.cfg.layer_params[0] > 8u) ? 8u : b.cfg.layer_params[0];
        const double norm = ldexp(1.0, -(int)(b.cfg.bits_per_sample - 1u));
        const double pi = 3.1415926535897932384626433832795029;
        if (tid == 0) est_sum = 0.0;
        bool nonzero = false;
        for (uint32_t c = 0; c < C; c++) {
            const int32_t *x = b.pcm + (size_t)c * b.cfg.pcm_stride + blk.smp_off;
            double r[9], w[LNB_FR_T + 8];
#pragma unroll
            for (int k = 0; k < 9; k++) r[k] = 0.0;
            /* windowed samples of the chunk and the p0 samples after it */
#pragma unroll
            for (int e = 0; e < LNB_FR_T + 8; e++) {
                const uint32_t j = i0 + (uint32_t)e;
                double v = 0.0;
                if ((uint32_t)e < cnt + p0 && j < n && cnt) {
                    const int32_t xi = x[j];
                    if ((uint32_t)e < cnt && xi != 0) nonzero = true;
                    /* the window of full blocks is tabulated (same expression, lnb_sine_window_kernel): FP64 sin per
                     * sample was four fifths of this kernel */
                    const double sw = (b.sinwin && n == b.sinwin_n) ? __ldg(b.sinwin + j) : sin((pi * (double)j) / (double)(n - 1u));
                    v = ((double)xi * norm) * sw;
                }
                w[e] = v;
            }
#pragma unroll
            for (int e = 0; e < LNB_FR_T; e++) {
                if ((uint32_t)e < cnt) {
#pragma unroll
                    for (int k = 0; k < 9; k++) if ((uint32_t)k <= p0) r[k] = fma(w[e], w[e + k], r[k]);
                }
            }
            double rr[9];
#pragma unroll
            for (int k = 0; k < 9; k++) rr[k] = r[k];            /* lags beyond p0 are zero and unused */
            lnb_fr_sum_n<9>(rr, red);                            /* one reduction for all lags: 3 barriers instead of 27 */
            if (tid == 0) {
                double a[12], coef[10], parcor[10];
                for (uint32_t k = 0; k <= p0; k++) parcor[k] = 0.0;
                if (n >= p0) lnb_levinson(rr, p0, a, coef, parcor);
                double est;
                double power = rr[0] * ldexp(1.0, (int)(2u * (b.cfg.bits_per_sample - 1u)));
                if (fabs(power) <= (double)FLT_MIN) est = 0.0;
                else {
                    power = log(power) * 1.4426950408889634 - log((double)n) * 1.4426950408889634;
                    double ratio = 0.0;
                    for (uint32_t k = 1; k < p0; k++) ratio += log(1.0 - parcor[k] * parcor[k]) * 1.4426950408889634;
                    est = 1.9426950408889634 + 0.5 * (power + ratio);
                    if (est <= 0.0) est = 1.0;
                }
                b.est[(size_t)blockIdx.x * C + c] = est;
                est_sum += est;
            }
        }
        const int any = __syncthreads_or(nonzero ? 1 : 0);
        if (tid == 0) {
            double mean = est_sum / (double)C;
            mean /= (double)b.cfg.bits_per_sample;
            uint32_t type = LNB_BLOCK_COMPRESSED;
            if (mean >= (double)LNB_RAW_THRESHOLD) type = LNB_BLOCK_RAW;
            else if (!any) type = LNB_BLOCK_SILENT;
            bcast[0] = (int32_t)type;
            gblk.type = type;
        }
        __syncthreads();
        if ((uint32_t)bcast[0] != LNB_BLOCK_COMPRESSED) return;
    }

    /* ---- (b) integer signal: copy, M/S on channels 0/1, two pre-emphasis passes per channel ---- */
    int32_t side_keep[LNB_FR_T];                    /* channel 1 after M/S, kept while channel 0 is processed */
    for (uint32_t c = 0; c < C; c++) {
        int32_t xs[LNB_FR_T];
        const int32_t *x = b.pcm + (size_t)c * b.cfg.pcm_stride + blk.smp_off;
        if (b.cfg.ms && C >= 2u && c == 0) {
            const int32_t *x1 = x + b.cfg.pcm_stride;
#pragma unroll
            for (int e = 0; e < LNB_FR_T; e++) {
                int32_t l = 0, r = 0;
                if ((uint32_t)e < cnt) { l = x[i0 + e]; r = x1[i0 + e]; }
                r -= l; l += r >> 1;                                  /* linne_utility.c:128-131 */
                xs[e] = l; side_keep[e] = r;
            }
        } else if (b.cfg.ms && C >= 2u && c == 1) {
#pragma unroll
            for (int e = 0; e < LNB_FR_T; e++) xs[e] = side_keep[e];
        } else {
#pragma unroll
            for (int e = 0; e < LNB_FR_T; e++) xs[e] = ((uint32_t)e < cnt) ? x[i0 + e] : 0;
        }
        LnbChanParams &prm = b.params[(size_t)blockIdx.x * C + c];
        for (int f = 0; f < LNB_NUM_PREEM; f++) {
            /* neighbours across chunk edges */
            if (cnt) {
                edge_first[tid] = xs[0];
                int32_t last = xs[0];
#pragma unroll
                for (int e = 0; e < LNB_FR_T; e++) if ((uint32_t)e < cnt) last = xs[e];
                edge_last[tid] = last;
            }
            __syncthreads();
            const int32_t prev0 = edge_first[0];                       /* block's first sample: transmitted state */
            /* coefficient: sums over i = 0 .. n-2 of x_i^2 and x_i x_{i+1} (linne_utility.c:158-193) */
            double c0 = 0.0, c1 = 0.0;
#pragma unroll
            for (int e = 0; e < LNB_FR_T; e++) {
                const uint32_t i = i0 + (uint32_t)e;
                if ((uint32_t)e < cnt && i + 1u < n) {
                    const double cur = (double)xs[e];
                    const double nxt = ((uint32_t)(e + 1) < cnt) ? (double)xs[(e + 1 < LNB_FR_T) ? e + 1 : e]
                                                                : (double)edge_first[tid + 1u];
                    c0 += cur * cur;
                    c1 += cur * nxt;
                }
            }
            {
                double cc[2] = {c0, c1};
                lnb_fr_sum_n<2>(cc, red);
                c0 = cc[0]; c1 = cc[1];
            }
            int32_t coef = 0;
            {
                const double q = c1 / c0;
                if (!(c0 < 1e-6 || q < 0.0)) {
                    coef = (int32_t)lnb_round_half_away(q * 32.0);
                    if (coef >= 16) coef = 15;
                }
            }
            /* filter (linne_utility.c:196-212): y[i] = x[i] - ((x[i-1] * coef) >> 5), x[-1] = x[0] */
            {
                int32_t left = (tid == 0) ? prev0 : edge_last[tid - 1u];
#pragma unroll
                for (int e = 0; e < LNB_FR_T; e++) {
                    if ((uint32_t)e < cnt) {
                        const int32_t cur = xs[e];
                        xs[e] = cur - ((left * coef) >> LNB_PREEM_SHIFT);
                        left = cur;
                    }
                }
            }
            if (tid == 0) { prm.preem_prev[f] = prev0; prm.preem_coef[f] = (uint8_t)coef; }
            __syncthreads();
        }
        int32_t *dst = b.work + ((size_t)blockIdx.x * C + c) * b.cfg.work_stride;
#pragma unroll
        for (int e = 0; e < LNB_FR_T; e++) if ((uint32_t)e < cnt) dst[i0 + e] = xs[e];
        for (uint32_t i = n + tid; i < b.cfg.work_stride; i += LNB_FR_THREADS) dst[i] = 0;
    }
}

/* ------------------------------------------------------------------------------------------------
 * Predict + plan: reference linne_lpc_predict.c:7-38 (cascade order linne_encoder.c:687-696) and
 * linne_coder.c:217-278 (partition search).
 * ------------------------------------------------------------------------------------------------ */
struct LnbPlanSmem {
    double mean[2 * LNB_MAX_PARTITIONS];
    uint8_t k2[2 * LNB_MAX_PARTITIONS];
    int32_t coef[LNB_MAX_PARAMS];
    uint32_t red[(LNB_MAX_PORDER + 1) * (LNB_FR_THREADS / 32)];
    uint32_t bits[LNB_MAX_PORDER + 1];
};

__global__ void __launch_bounds__(LNB_FR_THREADS) lnb_predict_plan_v2_kernel(LnbEncodeBatch b, uint32_t n_max)
{
    extern __shared__ __align__(16) unsigned char lnb_pp_raw[];
    int32_t *bufA = (int32_t *)lnb_pp_raw;
    int32_t *bufB = bufA + n_max;
    LnbPlanSmem &sm = *(LnbPlanSmem *)(bufB + n_max);

    const uint32_t tid = threadIdx.x, bc = blockIdx.x;
    const uint32_t blk_i = bc / b.cfg.num_channels;
    const LnbBlockDesc blk = b.blocks[blk_i];
    if (blk.type != LNB_BLOCK_COMPRESSED || !(blk.status & LNB_ENC_FLAG_COOP)) return;
    const uint32_t n = blk.nsmp;
    const LnbChanParams &prm = b.params[bc];
    int32_t *gwork = b.work + (size_t)bc * b.cfg.work_stride;

    for (uint32_t i = tid; i < n; i += LNB_FR_THREADS) bufA[i] = gwork[i];
    __syncthreads();

    /* ---- integer predictor cascade, out of place between the two buffers ---- */
    int32_t *in = bufA, *out = bufB;
    for (uint32_t l = 0; l < b.cfg.num_layers; l++) {
        const uint32_t P = b.cfg.layer_params[l];
        const uint32_t U = 1u << prm.log2_units[l];
        const uint32_t p = P / U, m = n / U, rshift = prm.rshift[l];
        const uint32_t half = rshift ? (1u << (rshift - 1u)) : 0u;
        for (uint32_t k = tid; k < P; k += LNB_FR_THREADS) sm.coef[k] = (int32_t)prm.coef[l * LNB_MAX_PARAMS + k];
        __syncthreads();
        for (uint32_t t = tid; t < n; t += LNB_FR_THREADS) {
            const uint32_t u = (m > 0u) ? t / m : U;
            const uint32_t pos = t - u * m;
            int32_t v = in[t];
            /* more units than taps: the layer predicts nothing, as in the reference and every decoder */
            if (u < U && U <= P && pos >= p && m > p) {
                const int32_t *h = in + t - p;
                const int32_t *cf = sm.coef + u * p;
                uint32_t acc = half;
                for (uint32_t k = 0; k < p; k++) acc += (uint32_t)cf[k] * (uint32_t)h[k];
                v = (int32_t)((uint32_t)v + (uint32_t)((int32_t)acc >> rshift));
            }
            out[t] = v;
        }
        __syncthreads();
        int32_t *tmp = in; in = out; out = tmp;
    }
    const int32_t *res = in;
    for (uint32_t i = tid; i < n; i += LNB_FR_THREADS) gwork[i] = res[i];

    /* ---- residual coder plan ---- */
    const uint32_t maxp = lnb_max_porder(n);
    const uint32_t fparts = 1u << maxp, flen = n / fparts;
    for (uint32_t part = tid; part < fparts; part += LNB_FR_THREADS) {
        uint64_t s = 0;
        const int32_t *r = res + part * flen;
        for (uint32_t i = 0; i < flen; i++) s += lnb_zz_enc(r[i]);
        sm.mean[(fparts - 1u) + part] = (double)s / (double)flen;
    }
    __syncthreads();
    for (int lvl = (int)maxp - 1; lvl >= 0; lvl--) {
        const uint32_t cnt = 1u << lvl;
        for (uint32_t part = tid; part < cnt; part += LNB_FR_THREADS)
            sm.mean[(cnt - 1u) + part] = __dadd_rn(sm.mean[(2u * cnt - 1u) + 2u * part], sm.mean[(2u * cnt - 1u) + 2u * part + 1u]) / 2.0;
        __syncthreads();
    }
    for (uint32_t idx = tid; idx < 2u * fparts - 1u; idx += LNB_FR_THREADS)
        sm.k2[idx] = (uint8_t)lnb_rice_k2(b.tab.k2_threshold, sm.mean[idx]);
    __syncthreads();

    uint32_t bits[LNB_MAX_PORDER + 1];
#pragma unroll
    for (int j = 0; j <= LNB_MAX_PORDER; j++) bits[j] = 0;
    /* code lengths of every sample under every partition order */
    for (uint32_t i = tid; i < n; i += LNB_FR_THREADS) {
        const uint32_t uv = lnb_zz_enc(res[i]);
        const uint32_t f = i / flen;
#pragma unroll
        for (int j = 0; j <= LNB_MAX_PORDER; j++) {
            if ((uint32_t)j <= maxp) bits[j] += lnb_rice_len(sm.k2[((1u << j) - 1u) + (f >> (maxp - (uint32_t)j))], uv);
        }
    }
    /* parameter bits of every partition of every order */
    for (uint32_t idx = tid; idx < 2u * fparts - 1u; idx += LNB_FR_THREADS) {
        const uint32_t lvl = 31u - lnb_clz32(idx + 1u), part = idx + 1u - (1u << lvl);
        const uint32_t add = (part == 0u) ? 5u
            : lnb_gamma_bits(lnb_zz_enc((int32_t)sm.k2[idx] - (int32_t)sm.k2[idx - 1u]));
#pragma unroll
        for (int j = 0; j <= LNB_MAX_PORDER; j++) if ((uint32_t)j == lvl) bits[j] += add;
    }
    /* block-wide sums (uint32, wrapping like the reference) */
#pragma unroll
    for (int j = 0; j <= LNB_MAX_PORDER; j++) {
        uint32_t v = bits[j];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        if ((tid & 31u) == 0) sm.red[j * (LNB_FR_THREADS / 32) + (tid >> 5)] = v;
    }
    __syncthreads();
    if (tid <= maxp) {
        uint32_t s = 0;
        for (uint32_t w = 0; w < LNB_FR_THREADS / 32; w++) s += sm.red[tid * (LNB_FR_THREADS / 32) + w];
        sm.bits[tid] = s;
    }
    __syncthreads();
    uint32_t best = 0, best_bits = 0xFFFFFFFFu;
    for (uint32_t j = 0; j <= maxp; j++) if (best_bits > sm.bits[j]) { best_bits = sm.bits[j]; best = j; }
    LnbCoderPlan &plan = b.plans[bc];
    if (tid == 0) { plan.porder = best; plan.bits = best_bits + 10u; }
    for (uint32_t part = tid; part < (1u << best); part += LNB_FR_THREADS) plan.k2[part] = sm.k2[((1u << best) - 1u) + part];
}
