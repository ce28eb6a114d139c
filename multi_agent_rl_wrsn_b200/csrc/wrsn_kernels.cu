/*
 * wrsn_kernels.cu — sm_100a kernels and the C ABI (include/wrsn_b200.h) of the batched WRSN simulator.
 *
 * One CTA per environment.  A launch copies the environment's resident record from HBM into shared
 * memory with 16-byte vector loads, runs the engine (wrsn_engine.cuh) there, and writes it back.
 * There is no CPU path: every entry point launches a kernel or returns an error.
 */
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>

#include "wrsn_launch.h"

#define WRSN_MAX_DEVICES 64
#define WRSN_CUDA(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) WRSN_FAIL("%s: %s", #x, cudaGetErrorString(e_)); } while (0)

/* 2^(j/64), j = 0..63, correctly rounded: the table of wrsn_exp_b (wrsn_engine.cuh; reward path only) */
__device__ const double wrsn_exp2_tab[64] = {
    0x1.0000000000000p+0, 0x1.02c9a3e778061p+0, 0x1.059b0d3158574p+0, 0x1.0874518759bc8p+0,
    0x1.0b5586cf9890fp+0, 0x1.0e3ec32d3d1a2p+0, 0x1.11301d0125b51p+0, 0x1.1429aaea92de0p+0,
    0x1.172b83c7d517bp+0, 0x1.1a35beb6fcb75p+0, 0x1.1d4873168b9aap+0, 0x1.2063b88628cd6p+0,
    0x1.2387a6e756238p+0, 0x1.26b4565e27cddp+0, 0x1.29e9df51fdee1p+0, 0x1.2d285a6e4030bp+0,
    0x1.306fe0a31b715p+0, 0x1.33c08b26416ffp+0, 0x1.371a7373aa9cbp+0, 0x1.3a7db34e59ff7p+0,
    0x1.3dea64c123422p+0, 0x1.4160a21f72e2ap+0, 0x1.44e086061892dp+0, 0x1.486a2b5c13cd0p+0,
    0x1.4bfdad5362a27p+0, 0x1.4f9b2769d2ca7p+0, 0x1.5342b569d4f82p+0, 0x1.56f4736b527dap+0,
    0x1.5ab07dd485429p+0, 0x1.5e76f15ad2148p+0, 0x1.6247eb03a5585p+0, 0x1.6623882552225p+0,
    0x1.6a09e667f3bcdp+0, 0x1.6dfb23c651a2fp+0, 0x1.71f75e8ec5f74p+0, 0x1.75feb564267c9p+0,
    0x1.7a11473eb0187p+0, 0x1.7e2f336cf4e62p+0, 0x1.82589994cce13p+0, 0x1.868d99b4492edp+0,
    0x1.8ace5422aa0dbp+0, 0x1.8f1ae99157736p+0, 0x1.93737b0cdc5e5p+0, 0x1.97d829fde4e50p+0,
    0x1.9c49182a3f090p+0, 0x1.a0c667b5de565p+0, 0x1.a5503b23e255dp+0, 0x1.a9e6b5579fdbfp+0,
    0x1.ae89f995ad3adp+0, 0x1.b33a2b84f15fbp+0, 0x1.b7f76f2fb5e47p+0, 0x1.bcc1e904bc1d2p+0,
    0x1.c199bdd85529cp+0, 0x1.c67f12e57d14bp+0, 0x1.cb720dcef9069p+0, 0x1.d072d4a07897cp+0,
    0x1.d5818dcfba487p+0, 0x1.da9e603db3285p+0, 0x1.dfc97337b9b5fp+0, 0x1.e502ee78b3ff6p+0,
    0x1.ea4afa2a490dap+0, 0x1.efa1bee615a27p+0, 0x1.f50765b6e4540p+0, 0x1.fa7c1819e90d8p+0,
};

extern __shared__ uint4 wrsn_smem_u4[];             /* the environment's image (k_env), addressed by 32-bit offsets */

namespace g32 {                                      /* one warp per environment (N <= 128) */
#define WRSN_GFIX 32
#include "wrsn_engine.cuh"
#include "wrsn_env_kernel.cuh"
#undef WRSN_GFIX
}
namespace gany {                                     /* 64 ... 256 threads per environment */
#define WRSN_GFIX 0
#include "wrsn_engine.cuh"
#include "wrsn_env_kernel.cuh"
#undef WRSN_GFIX
}

/* ------------------------------------------------------------------ WRSN.get_state (rl_env/WRSN.py:130-186)
 * The sources and their weights: wrsn_layout.h (obs_source).  The raster is separable, so it is a rank-(number of sources)
 * outer-product sum.  A chunk of sources is expanded into two S-vectors each in shared memory (2 S exponentials per source
 * instead of S^2, always evaluated in fp64) and every thread accumulates a 4 x 10 register tile of output cells over the sources
 * IN SOURCE ORDER.  AccT = double: multiply and add rounded separately, exactly the reference's `map += w*gx*gy`
 * (parity path, float64 out).  AccT = float: the vectors are rounded to fp32 once and accumulated with FFMA (the
 * observation the policy networks consume is float32; error ~1e-6 of the channel maximum). */
#define OBS_THREADS64 256           /* fp64 parity raster: 4 x 10 tiles (OBS_TI x OBS_TJ64, wrsn_layout.h) */
#define OBS_THREADS32 128           /* fp32 raster: 4 x 20 tiles (OBS_TI x OBS_TJ32) */
#define OBS_CH32 32                 /* sources staged per pass (fp32 raster) */
#define OBS_MINB32 4                /* CTAs per SM the fp32 raster is compiled for */

/* the node terms of get_state are static: one table row per node, float (the fp32 raster reads them, the fp64 parity
 * raster evaluates its exponentials itself) */
__global__ void k_obs_tables(const wrsn_dims d, const WrsnLayout L, char *scen) {
    char *row = scen + (size_t)blockIdx.x * L.scen_total;
    const double *par = (const double *)(row + L.soff[WRSN_S_PAR]);
    const double *nx = (const double *)(row + L.soff[WRSN_S_NX]), *ny = (const double *)(row + L.soff[WRSN_S_NY]);
    float *gx = (float *)(row + L.soff[WRSN_S_OBS_GX]), *gy = (float *)(row + L.soff[WRSN_S_OBS_GY]);
    const int n = blockIdx.y, S = d.S, TP = d.obs_pitch;
    const ObsGrid g(par, S);
    const double x0 = g.cx(nx[n]), y0 = g.cy(ny[n]), hx = g.R / g.Wd, hy = g.R / g.Hd;
    const double dnx = -2.0 * (hx * hx), dny = -2.0 * (hy * hy);
    for (int i = threadIdx.x; i < TP; i += blockDim.x) {
        const bool in = i < S && n < (int)par[WRSN_P_NNODES];
        gx[(size_t)n * TP + i] = in ? (float)obs_gauss(g.cell(i), x0, dnx) : 0.f;
        gy[(size_t)n * TP + i] = in ? (float)obs_gauss(g.cell(i), y0, dny) : 0.f;
    }
}

/* tile = OBS_TI rows x TJ columns of output cells per thread.  fp64 parity raster: 4 x 10 on 256 threads; fp32 raster: 4 x 20 on
 * 128 threads (125 tiles of a 100 x 100 map: 80 FFMA per source against one 16-byte and five 16-byte shared-memory loads) */
template <typename AccT, int TJ, int THREADS>
__global__ void __launch_bounds__(THREADS, sizeof(AccT) == 4 ? OBS_MINB32 : 1) k_observe(const KParams P, const int32_t *agent_id, AccT *obs) {
    constexpr int CH = sizeof(AccT) == 4 ? OBS_CH32 : 16;      /* sources staged per pass */
    extern __shared__ uint4 smem_u4[];
    const int S = P.d.S, M = P.d.M, TP = P.d.obs_pitch;
    const int tiles_i = (S + OBS_TI - 1) / OBS_TI, tiles_j = (S + TJ - 1) / TJ;
    AccT *gx = reinterpret_cast<AccT *>(smem_u4);                             /* [CH][TP] */
    AccT *gy = gx + CH * TP;                                                  /* [CH][TP] */
    __shared__ ObsSrc src[CH];
    const int b = blockIdx.x, tid = threadIdx.x;
    const int ag = agent_id[b];
    if (ag < 0) return;
    const WrsnRow rw(P.L, P.state, P.scen, P.scen_id, b);
    const ObsGrid g(rw.par, S);
    const int N = rw.N;
    const int SS = S * S;
    AccT *out = obs + (size_t)b * 4 * SS;
    const int n_tiles = tiles_i * tiles_j;

    for (int tbase = 0; tbase < n_tiles; tbase += THREADS) {
        const int tile = tbase + tid;
        const bool has_tile = tile < n_tiles;
        const int ti = has_tile ? tile / tiles_j : 0, tj = has_tile ? tile - ti * tiles_j : 0;
        const int i0 = ti * OBS_TI, j0 = tj * TJ;
        for (int ch = 0; ch < 4; ch++) {
            AccT acc[OBS_TI][TJ];
#pragma unroll
            for (int r = 0; r < OBS_TI; r++)
#pragma unroll
                for (int q = 0; q < TJ; q++) acc[r][q] = (AccT)0;
            const int total = ch == 0 ? N : (ch == 1 ? 1 : M);
            for (int s0 = 0; s0 < total; s0 += CH) {
                const int nq = total - s0 < CH ? total - s0 : CH;
                __syncthreads();
                /* the sources of this pass, one thread each, in id order; unused ones are skipped — the reference skips them
                   too, and the sum order of the rest is unchanged */
                for (int q = tid; q < nq; q += THREADS) src[q] = obs_source(rw, g, ag, ch, s0 + q);
                __syncthreads();
                /* expand every source into its two S-vectors.  Node sources of the fp32 raster are a scaled copy of the
                   scenario's table (contiguous, independent loads); everything else is one fp64 exponential per entry. */
                for (int q = tid >> 5; q < nq; q += THREADS / 32) {        /* one warp per source row: no index division */
                    const int mode = src[q].mode;
                    if (mode < 0) continue;
                    const int node = src[q].node;
                    if (sizeof(AccT) == 4 && node >= 0) {
                        const float wq = (float)src[q].w;
                        const float *rx = rw.tab_gx + (size_t)node * TP, *ry = rw.tab_gy + (size_t)node * TP;
                        /* TP is a multiple of 4 and every row starts 16-byte aligned: four entries per lane and instruction */
                        const float4 *rx4 = reinterpret_cast<const float4 *>(rx), *ry4 = reinterpret_cast<const float4 *>(ry);
                        float4 *gx4 = reinterpret_cast<float4 *>(gx + q * TP), *gy4 = reinterpret_cast<float4 *>(gy + q * TP);
                        for (int i = tid & 31; i < (TP >> 2); i += 32) {
                            float4 vx = rx4[i];
                            vx.x *= wq; vx.y *= wq; vx.z *= wq; vx.w *= wq;
                            gx4[i] = vx; gy4[i] = ry4[i];
                        }
                    } else {
                        const double x0 = src[q].x0, y0 = src[q].y0;
                        const double dnx = -2.0 * (src[q].hx * src[q].hx), dny = -2.0 * (src[q].hy * src[q].hy);
                        /* fp32 raster: the constant factor of the source (w, or w / moving_time_max for the travel-time
                           channel) is folded into the x-vector, so every channel shares the FFMA loop below */
                        const double fold = mode == 0 ? src[q].w : (sizeof(AccT) == 4 ? src[q].w / g.mtm : 1.0);
                        for (int i = tid & 31; i < TP; i += 32) {
                            const double ex = i < S ? obs_gauss(g.cell(i), x0, dnx) : 0.0;
                            const double ey = i < S ? obs_gauss(g.cell(i), y0, dny) : 0.0;
                            gx[q * TP + i] = (AccT)((mode == 0 || sizeof(AccT) == 4) ? fold * ex : ex);
                            gy[q * TP + i] = (AccT)ey;
                        }
                    }
                }
                __syncthreads();
                if (!has_tile) continue;
                if (ch != 3 || sizeof(AccT) == 4) {
                    for (int q = 0; q < nq; q++) {
                        if (src[q].mode < 0) continue;
                        AccT a[OBS_TI], v[TJ];
                        if (sizeof(AccT) == 4) {     /* i0 is a multiple of 4, j0 of 2: one 16-byte and five 8-byte loads */
                            const float4 a4 = *reinterpret_cast<const float4 *>(gx + q * TP + i0);
                            a[0] = (AccT)a4.x; a[1] = (AccT)a4.y; a[2] = (AccT)a4.z; a[3] = (AccT)a4.w;
                            if (TJ % 4 == 0) {           /* j0 is a multiple of 4 */
                                const float4 *v4 = reinterpret_cast<const float4 *>(gy + q * TP + j0);
#pragma unroll
                                for (int x = 0; x < TJ; x += 4) {
                                    const float4 t4 = v4[x >> 2];
                                    v[x] = (AccT)t4.x; v[x + 1] = (AccT)t4.y; v[x + 2] = (AccT)t4.z; v[x + 3] = (AccT)t4.w;
                                }
                            } else {
                                const float2 *v2 = reinterpret_cast<const float2 *>(gy + q * TP + j0);
#pragma unroll
                                for (int x = 0; x < TJ; x += 2) { const float2 t2 = v2[x >> 1]; v[x] = (AccT)t2.x; v[x + 1] = (AccT)t2.y; }
                            }
                        } else {
#pragma unroll
                            for (int r = 0; r < OBS_TI; r++) a[r] = gx[q * TP + i0 + r];
#pragma unroll
                            for (int x = 0; x < TJ; x++) v[x] = gy[q * TP + j0 + x];
                        }
#pragma unroll
                        for (int r = 0; r < OBS_TI; r++)
#pragma unroll
                            for (int x = 0; x < TJ; x++) {
                                if (sizeof(AccT) == 4) acc[r][x] = fmaf((float)a[r], (float)v[x], (float)acc[r][x]);
                                else acc[r][x] = acc[r][x] + a[r] * v[x];       /* -fmad=false: two roundings, as numpy */
                            }
                    }
                } else {
                    for (int q = 0; q < nq; q++) {
                        if (src[q].mode < 0) continue;
                        const AccT w = (AccT)src[q].w, d = (AccT)g.mtm;
#pragma unroll
                        for (int r = 0; r < OBS_TI; r++)
#pragma unroll
                            for (int x = 0; x < TJ; x++)
                                acc[r][x] = acc[r][x] + gx[q * TP + i0 + r] * gy[q * TP + j0 + x] * w / d;
                    }
                }
            }
            if (has_tile) {
                if (sizeof(AccT) == 4 && TJ % 4 == 0 && (S & 3) == 0 && j0 + TJ <= S) {   /* 16-byte aligned row segments */
#pragma unroll
                    for (int r = 0; r < OBS_TI; r++) {
                        if (i0 + r >= S) continue;
                        float4 *o4 = reinterpret_cast<float4 *>(out + (size_t)ch * SS + (size_t)(i0 + r) * S + j0);
#pragma unroll
                        for (int x = 0; x < TJ; x += 4)
                            o4[x >> 2] = make_float4((float)acc[r][x], (float)acc[r][x + 1], (float)acc[r][x + 2], (float)acc[r][x + 3]);
                    }
                } else if (sizeof(AccT) == 4 && (S & 1) == 0 && j0 + TJ <= S) {  /* even map size: every row segment is 8-byte aligned */
#pragma unroll
                    for (int r = 0; r < OBS_TI; r++) {
                        if (i0 + r >= S) continue;
                        float2 *o2 = reinterpret_cast<float2 *>(out + (size_t)ch * SS + (size_t)(i0 + r) * S + j0);
#pragma unroll
                        for (int x = 0; x < TJ; x += 2) o2[x >> 1] = make_float2((float)acc[r][x], (float)acc[r][x + 1]);
                    }
                } else {
#pragma unroll
                    for (int r = 0; r < OBS_TI; r++)
#pragma unroll
                        for (int x = 0; x < TJ; x++)
                            if (i0 + r < S && j0 + x < S) out[(size_t)ch * SS + (size_t)(i0 + r) * S + j0 + x] = acc[r][x];
                }
            }
        }
    }
}


/* ------------------------------------------------------------------ the float32 raster, windowed
 * Same sum as k_observe<float> (WRSN.get_state, rl_env/WRSN.py:130-186), restructured around two facts: (1) the sources of
 * channels 1, 3 and 4 (nodes, other chargers) are Gaussians of bandwidth charging_range / extent — 2.7 cells on the
 * 1 km fields of the shipped scenarios — so outside a window of OBW cells around its centre a source contributes less
 * than 3e-9 of its peak (the float32 observation is held to 1e-5 of the channel maximum; the float64 parity raster is
 * untouched); (2) the time of the chunked kernel goes to its staging rounds (setup -> barrier -> expand -> barrier, seven
 * times per map), not to its FFMAs.  Here ALL sources of a map are staged once — one warp per source: its scalars, then
 * its window of the scenario's table scaled by its weight (the own-position source of channel 2, half the field wide, is
 * staged full width) — one barrier, then every thread accumulates its 4 x 20 tile over the sources whose window meets the
 * tile, in source order.  Shared memory per source: OBW row entries and OBW column entries between two 16-entry zero
 * margins (a partly covered tile reads zeros instead of branching): 448 bytes at OBW = 40. */
#define OBM 16                       /* zero margin on either side of the column window (a tile is 20 columns wide) */
#define OBW 40                       /* window in cells (multiple of 4): >= 12.2 sigma + 6 */
#define OBW_THREADS 128
struct WinSrc { int sx, sy; };       /* first row / column of the window; sx < -1000: source unused */
__global__ void __launch_bounds__(OBW_THREADS, 4) k_observe_win(const KParams P, const int32_t *agent_id, float *obs) {
    extern __shared__ uint4 smem_u4[];
    const int S = P.d.S, M = P.d.M, TP = P.d.obs_pitch;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const int ag = agent_id[b];
    if (ag < 0) return;
    const WrsnRow rw(P.L, P.state, P.scen, P.scen_id, b);
    const ObsGrid g(rw.par, S);
    const int N = rw.N;                                         /* (P.d.N, the batch's largest, sizes smem) */
    const int NS = N + 2 * M;                                   /* nodes | chargers as channel-3 sources | as channel-4 sources */
    float *gxw = reinterpret_cast<float *>(smem_u4);            /* [NS][OBW] */
    float *gyw = gxw + (size_t)NS * OBW;                        /* [NS][OBM + OBW + OBM] */
    float *own = gyw + (size_t)NS * (OBW + 2 * OBM);            /* [2][TP]: the observer's own position, full width */
    WinSrc *win = reinterpret_cast<WinSrc *>(own + 2 * TP);     /* [NS] */
    /* ---- stage every source: one warp per source */
    for (int q = wrp; q < NS + 1; q += OBW_THREADS / 32) {
        if (q == NS) {                                          /* channel 2: own position */
            const ObsSrc v = obs_source(rw, g, ag, 1, 0);
            const double dnx = -2.0 * (v.hx * v.hx), dny = -2.0 * (v.hy * v.hy);
            for (int i = lane; i < TP; i += 32) {
                own[i] = (float)(i < S ? v.w * obs_gauss(g.cell(i), v.x0, dnx) : 0.0);
                own[TP + i] = (float)(i < S ? obs_gauss(g.cell(i), v.y0, dny) : 0.0);
            }
            continue;
        }
        /* channel 1: alive nodes with traffic; channels 3 / 4: the other chargers at their destinations */
        const ObsSrc v = q < N ? obs_source(rw, g, ag, 0, q) : obs_source(rw, g, ag, q < N + M ? 2 : 3, (q - N) % M);
        const double w = v.mode == 1 ? v.w / g.mtm : v.w;
        int sx = -100000, sy = -100000;
        if (v.mode >= 0) {
            sx = (((int)floor(v.x0 * (double)S) - OBW / 2) >> 2) << 2; sy = (((int)floor(v.y0 * (double)S) - OBW / 2) >> 2) << 2;
            sx = sx < 0 ? 0 : (sx > S - OBW ? S - OBW : sx); sy = sy < 0 ? 0 : (sy > S - OBW ? S - OBW : sy);
            float *gx = gxw + (size_t)q * OBW, *gy = gyw + (size_t)q * (OBW + 2 * OBM);
            if (v.node >= 0) {                                  /* scaled copy of the scenario's table rows */
                const float wq = (float)w;
                const float *rx = rw.tab_gx + (size_t)v.node * TP, *ry = rw.tab_gy + (size_t)v.node * TP;
                for (int i = lane; i < OBW; i += 32) gx[i] = rx[sx + i] * wq;
                for (int i = lane; i < OBW + 2 * OBM; i += 32) {
                    const int k = i - OBM;
                    gy[i] = (k >= 0 && k < OBW) ? ry[sy + k] : 0.f;
                }
            } else {
                const double dnx = -2.0 * (v.hx * v.hx), dny = -2.0 * (v.hy * v.hy);
                for (int i = lane; i < OBW; i += 32) gx[i] = (float)(w * obs_gauss(g.cell(sx + i), v.x0, dnx));
                for (int i = lane; i < OBW + 2 * OBM; i += 32) {
                    const int k = i - OBM;
                    gy[i] = (k >= 0 && k < OBW) ? (float)obs_gauss(g.cell(sy + k), v.y0, dny) : 0.f;
                }
            }
        }
        if (lane == 0) { win[q].sx = sx; win[q].sy = sy; }
    }
    __syncthreads();
    /* ---- accumulate: 4 x 20 tile per thread */
    const int tiles_j = S / OBS_TJ32, n_tiles = (S / OBS_TI) * tiles_j;
    if (tid >= n_tiles) return;
    const int ti = tid / tiles_j, tj = tid - ti * tiles_j, i0 = ti * OBS_TI, j0 = tj * OBS_TJ32;
    const int SS = S * S;
    float *out = obs + (size_t)b * 4 * SS;
    for (int ch = 0; ch < 4; ch++) {
        float acc[OBS_TI][OBS_TJ32];
#pragma unroll
        for (int r = 0; r < OBS_TI; r++)
#pragma unroll
            for (int x = 0; x < OBS_TJ32; x++) acc[r][x] = 0.f;
        if (ch == 1) {
            const float4 a4 = *reinterpret_cast<const float4 *>(own + i0);
            const float a[OBS_TI] = {a4.x, a4.y, a4.z, a4.w};
            const float4 *v4 = reinterpret_cast<const float4 *>(own + TP + j0);
#pragma unroll
            for (int x = 0; x < OBS_TJ32; x += 4) {
                const float4 t4 = v4[x >> 2];
                const float v[4] = {t4.x, t4.y, t4.z, t4.w};
#pragma unroll
                for (int r = 0; r < OBS_TI; r++)
#pragma unroll
                    for (int y = 0; y < 4; y++) acc[r][x + y] = fmaf(a[r], v[y], acc[r][x + y]);
            }
        } else {
            const int q0 = ch == 0 ? 0 : (ch == 2 ? N : N + M), q1 = ch == 0 ? N : q0 + M;
#pragma unroll 1
            for (int q = q0; q < q1; q++) {
                const WinSrc ws = win[q];
                const int ri = i0 - ws.sx, rj = j0 - ws.sy;      /* multiples of 4 */
                if (ri < 0 || ri > OBW - OBS_TI || rj <= -OBS_TJ32 || rj >= OBW) continue;   /* (an unused source has sx = -100000) */
                const float4 a4 = *reinterpret_cast<const float4 *>(gxw + (size_t)q * OBW + ri);
                const float a[OBS_TI] = {a4.x, a4.y, a4.z, a4.w};
                const float4 *v4 = reinterpret_cast<const float4 *>(gyw + (size_t)q * (OBW + 2 * OBM) + OBM + rj);
#pragma unroll
                for (int x = 0; x < OBS_TJ32; x += 4) {
                    const float4 t4 = v4[x >> 2];
                    const float v[4] = {t4.x, t4.y, t4.z, t4.w};
#pragma unroll
                    for (int r = 0; r < OBS_TI; r++)
#pragma unroll
                        for (int y = 0; y < 4; y++) acc[r][x + y] = fmaf(a[r], v[y], acc[r][x + y]);
                }
            }
        }
#pragma unroll
        for (int r = 0; r < OBS_TI; r++) {
            float4 *o4 = reinterpret_cast<float4 *>(out + (size_t)ch * SS + (size_t)(i0 + r) * S + j0);
#pragma unroll
            for (int x = 0; x < OBS_TJ32; x += 4) o4[x >> 2] = make_float4(acc[r][x], acc[r][x + 1], acc[r][x + 2], acc[r][x + 3]);
        }
    }
}

/* ------------------------------------------------------------------ WRSN.density_map_to_action (rl_env/WRSN.py:229-287)
 * and the map normalisation of WRSN.step (:293-296): an S x S density map -> (x-frac, y-frac, charge-time frac).
 * One CTA per environment, ONE streaming pass over the map in HBM (the only traffic that matters: S*S values in, 24
 * bytes out); nothing but a few scalars is staged on chip.
 *   - every thread keeps min / max / sum and the two largest values of its (strided) share of the map in registers;
 *   - np.argmax (first maximum in row-major order) and the order statistics around np.percentile(flat, 99.9) come from
 *     n - floor(0.999 (n - 1)) + 1 rounds (12 for a 100 x 100 map) of block-wide "largest remaining head, smallest
 *     index"; a thread whose two heads are both taken rescans its share (rare: neighbouring cells belong to different
 *     threads).  If the map is not a distribution the reference replaces it by exp(map) / (sum + eps): monotone, so the
 *     ORDER is taken from the raw values, exp() is applied to the handful of selected ones only, and the common divisor
 *     cancels in everything computed here;
 *   - third component = map[argmax] / sum of the values >= that percentile: the selected values — unless values tie
 *     with the percentile beyond the selected ones (uniform or one-hot maps), then a second pass over the map sums them;
 *   - location: the reference maximises  sum_{alive n, d_n <= R} energyCS_n / (E_n - thr) * alpha / (d_n + beta)^2  inside
 *     the +-R box around the argmax cell with scipy's L-BFGS-B from the box centre.  With the magnitudes of this model
 *     L-BFGS-B stops at once (projected gradient <= pgtol = 1e-5: the centre itself is returned, bit for bit) in most
 *     calls, takes one unit step along the gradient and stops on its ftol in most of the others, and otherwise climbs
 *     to the nearest cusp (a node).  Warp 0 runs the same three regimes: scipy's two stopping rules with their default
 *     constants, a unit first step, then spectral (Barzilai-Borwein, the L-BFGS scaling) steps with backtracking.  The
 *     objective is discontinuous and scipy's answer depends on its version (SURVEY 8f-1): parity is tolerance-based
 *     (tests/test_decode.py), exact whenever scipy returns the centre. */
#define DEC_THREADS 256
#define DEC_MAXR 34
#define DEC_MAXC 64
/* LIN = false: dmap[b][S][S] is the map.  LIN = true: the map is a linear combination of the channels of the observation
 * tensor, dmap[b][C][S][S] (float), formed on the fly in float32 with one rounding per multiply and per add, channel by
 * channel — (((w0 o0) + w1 o1) + w2 o2) + ... — which is, bit for bit, what torch computes for the reference's
 * RandomController (controller/random/RandomController.py:12-15: s0 + s1 - 10 s2 + s3; multiplying by 1 and negating are
 * exact): the controller's three elementwise passes over the observations and the map itself never touch HBM. */
struct LinMap { int C; float w[8]; };
/* LINC: 0 = plain map; 4 = four channels, unrolled (weights in registers); -1 = any number of channels (rolled).
 * This kernel produces the statistics of the map — charge-time fraction -> action[b][2], flat index of the argmax cell ->
 * action[b][0] (as a double) — with all 256 threads busy; the location search, a serial climb of ONE warp, runs in
 * k_decode_locate (one warp per environment) so that no warp waits at a barrier for it. */
template <typename MapT, int LINC>
__global__ void __launch_bounds__(DEC_THREADS, 4) k_decode_map(const KParams P, const int32_t *agent_id, const MapT *dmap, double *action,
                                                               const LinMap lin) {
    constexpr bool LIN = LINC != 0;
    __shared__ double cand_v[(DEC_THREADS / 32) * DEC_MAXR];
    __shared__ int cand_i[(DEC_THREADS / 32) * DEC_MAXR];
    __shared__ double red_s[3][DEC_THREADS / 32];
    __shared__ double top_v[DEC_MAXR];
    __shared__ int top_i[DEC_MAXR];
    __shared__ double bc[4];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (agent_id[b] < 0) return;
    const int S = P.d.S, n = S * S;
    const MapT *src0 = dmap + (size_t)b * n * (LIN ? lin.C : 1);
    const float w0 = lin.w[0], w1 = lin.w[1], w2 = lin.w[2], w3 = lin.w[3];
    auto at = [&](int k) -> MapT {
        if (LINC == 0) return src0[k];
        if (LINC == 4) {
            float acc = __fmul_rn(w0, (float)src0[k]);
            acc = __fadd_rn(acc, __fmul_rn(w1, (float)src0[n + k]));
            acc = __fadd_rn(acc, __fmul_rn(w2, (float)src0[2 * n + k]));
            return (MapT)__fadd_rn(acc, __fmul_rn(w3, (float)src0[3 * n + k]));
        }
        float acc = __fmul_rn(lin.w[0], (float)src0[k]);
        for (int ch = 1; ch < lin.C; ch++) acc = __fadd_rn(acc, __fmul_rn(lin.w[ch], (float)src0[(size_t)ch * n + k]));
        return (MapT)acc;
    };
    /* pass 1: min / max / sum and this thread's two heads (value descending, index ascending; k only grows here) */
    MapT mn = (MapT)INFINITY, mx = (MapT)-INFINITY; double sm = 0.0;
    MapT h1v = (MapT)-INFINITY, h2v = (MapT)-INFINITY; int h1i = 0x7fffffff, h2i = 0x7fffffff;
#pragma unroll 4
    for (int k = tid; k < n; k += DEC_THREADS) {
        const MapT v = at(k);
        mn = v < mn ? v : mn; mx = v > mx ? v : mx; sm += (double)v;
        /* an empty head also takes a -inf cell (k ascending: the first one, as np.argmax does for a map that is -inf
           everywhere); NaN cells never become heads */
        if (v > h1v || (h1i == 0x7fffffff && v == h1v)) { h2v = h1v; h2i = h1i; h1v = v; h1i = k; }
        else if (v > h2v || (h2i == 0x7fffffff && v == h2v)) { h2v = v; h2i = k; }
    }
    double dmn = (double)mn, dmx = (double)mx;
    for (int o = 16; o > 0; o >>= 1) {
        dmn = fmin(dmn, __shfl_xor_sync(0xffffffffu, dmn, o)); dmx = fmax(dmx, __shfl_xor_sync(0xffffffffu, dmx, o)); sm += __shfl_xor_sync(0xffffffffu, sm, o);
    }
    if (lane == 0) { red_s[0][wid] = dmn; red_s[1][wid] = dmx; red_s[2][wid] = sm; }
    /* np.percentile(., 99.9), method "linear": virtual index n q + (alpha + q (1 - alpha - beta)) - 1 with alpha = beta = 1 */
    const double qf = 99.9 / 100.0;
    const double vidx = (double)n * qf + (1.0 + qf * (1.0 - 1.0 - 1.0)) - 1.0;
    const int lo_idx = (int)floor(vidx);
    const double tq = vidx - (double)lo_idx;
    int R = n - lo_idx;                              /* the R-th largest value is sorted[lo_idx]; R <= DEC_MAXR - 2: the host
                                                        refuses larger maps (wrsn_abi_host.h: check_decode_size) */
    const int rounds = R + 1 < n ? R + 1 : n;        /* one more: does anything tie with sorted[lo_idx] beyond the selection? */
    /* every warp selects ITS `rounds` largest (shuffles only): the block's `rounds` largest are among those */
    {
        int taken = 0; MapT lastv = (MapT)INFINITY; int lasti = -1;
        for (int r = 0; r < rounds; r++) {
            if (taken == 2) {                        /* both heads gone: the next two of this thread's share after (lastv, lasti) */
                h1v = h2v = (MapT)-INFINITY; h1i = h2i = 0x7fffffff;
                for (int k = tid; k < n; k += DEC_THREADS) {
                    const MapT v = at(k);
                    if (!(v < lastv || (v == lastv && k > lasti))) continue;
                    if (v > h1v || (h1i == 0x7fffffff && v == h1v)) { h2v = h1v; h2i = h1i; h1v = v; h1i = k; }
                    else if (v > h2v || (h2i == 0x7fffffff && v == h2v)) { h2v = v; h2i = k; }
                }
                taken = 0;
            }
            const MapT pv = taken == 0 ? h1v : h2v; const int pi = taken == 0 ? h1i : h2i;
            MapT bv = pv; int bi = pi;
            for (int o = 16; o > 0; o >>= 1) {
                const MapT ov = __shfl_xor_sync(0xffffffffu, bv, o); const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
            }
            if (lane == 0) { cand_v[wid * DEC_MAXR + r] = (double)bv; cand_i[wid * DEC_MAXR + r] = bi; }
            if (pi == bi && bi != 0x7fffffff) { taken++; lastv = pv; lasti = pi; }
        }
    }
    __syncthreads();
    double mn_d = red_s[0][0], mx_d = red_s[1][0]; sm = red_s[2][0];
    for (int w = 1; w < DEC_THREADS / 32; w++) { mn_d = fmin(mn_d, red_s[0][w]); mx_d = fmax(mx_d, red_s[1][w]); sm += red_s[2][w]; }
    /* WRSN.step :294: np.all((a >= 0) & (a <= 1)) and np.isclose(np.sum(a), 1)  (rtol 1e-5, atol 1e-8) */
    const bool is_dist = mn_d >= 0.0 && mx_d <= 1.0 && fabs(sm - 1.0) <= 1e-8 + 1e-5;
    /* warp 0 merges the 8 sorted lists: `rounds` times the largest list head */
    if (wid == 0) {
        int pos = 0;                                 /* lane w < 8 walks list w */
        for (int r = 0; r < rounds; r++) {
            double bv = -INFINITY; int bi = 0x7fffffff;
            if (lane < DEC_THREADS / 32 && pos < rounds) { bv = cand_v[lane * DEC_MAXR + pos]; bi = cand_i[lane * DEC_MAXR + pos]; }
            const int mine = bi;
            for (int o = 4; o > 0; o >>= 1) {
                const double ov = __shfl_xor_sync(0xffffffffu, bv, o); const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
            }
            bv = __shfl_sync(0xffffffffu, bv, 0); bi = __shfl_sync(0xffffffffu, bi, 0);
            if (lane == 0) { top_v[r] = bv; top_i[r] = bi; }
            if (mine == bi && bi != 0x7fffffff) pos++;
        }
    }
    __syncthreads();
    /* the transformed values of the selection (exp only here), threshold, kept mass */
    if (R > rounds) R = rounds;
    const double a_x = top_v[R - 1];
    const double a_q = is_dist ? a_x : exp(a_x);
    const double b_q = R >= 2 ? (is_dist ? top_v[R - 2] : exp(top_v[R - 2])) : a_q;
    double thr_q = a_q + (b_q - a_q) * tq;           /* numpy _lerp */
    if (tq >= 0.5) thr_q = b_q - (b_q - a_q) * (1.0 - tq);
    if (lo_idx + 1 > n - 1) thr_q = a_q;
    const bool ties_beyond = a_q >= thr_q && rounds > R && top_v[R] == a_x;
    double keep = 0.0;
    if (!ties_beyond) {
        if (tid == 0) {
            for (int r = 0; r < R; r++) { const double v = is_dist ? top_v[r] : exp(top_v[r]); if (v >= thr_q) keep += v; }
            bc[0] = (is_dist ? top_v[0] : exp(top_v[0])) / keep;
        }
    } else {                                         /* values equal to the percentile all over the map: sum them in a second pass */
        for (int k = tid; k < n; k += DEC_THREADS) {
            const double x = (double)at(k);
            if (x >= a_x) { const double v = is_dist ? x : exp(x); if (v >= thr_q) keep += v; }
        }
        for (int o = 16; o > 0; o >>= 1) keep += __shfl_xor_sync(0xffffffffu, keep, o);
        if (lane == 0) red_s[0][wid] = keep;
        __syncthreads();
        if (tid == 0) {
            double tot = 0.0;
            for (int w = 0; w < DEC_THREADS / 32; w++) tot += red_s[0][w];
            bc[0] = (is_dist ? top_v[0] : exp(top_v[0])) / tot;
        }
    }
    __syncthreads();
    if (tid == 0) { action[3 * (size_t)b] = (double)top_i[0]; action[3 * (size_t)b + 2] = bc[0]; }
}

/* the location search of WRSN.density_map_to_action (:240-262), one warp per environment: reads the argmax cell left in
 * action[b][0] by k_decode_map, writes action[b][0..1] */
#define LOC_WARPS 4
__global__ void __launch_bounds__(32 * LOC_WARPS) k_decode_locate(const KParams P, const int32_t *agent_id, double *action) {
    __shared__ double s_cn[LOC_WARPS][3][DEC_MAXC];
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    const int b = blockIdx.x * LOC_WARPS + wrp;
    if (b >= P.d.B || agent_id[b] < 0) return;           /* whole warps leave together; only __syncwarp below */
    double *cn_x = s_cn[wrp][0], *cn_y = s_cn[wrp][1], *cn_w = s_cn[wrp][2];
    const int S = P.d.S;
    const int flat0 = (int)action[3 * (size_t)b];
    double out_x, out_y;
    {
        const WrsnRow rw(P.L, P.state, P.scen, P.scen_id, b);
        const double *par = rw.par, *nx = rw.nx, *ny = rw.ny, *energy = rw.energy, *cs = rw.cs;
        const uint8_t *status = rw.status;
        const int N = rw.N;
        const double f0 = par[WRSN_P_F0], f1 = par[WRSN_P_F1], f2 = par[WRSN_P_F2], f3 = par[WRSN_P_F3];
        const double R = par[WRSN_P_MC_R], alpha = par[WRSN_P_MC_ALPHA], beta = par[WRSN_P_MC_BETA], thr = par[WRSN_P_THR];
        const double unit = 1.0 / (double)S;
        const int flat = flat0, m0 = flat / S, m1 = flat - m0 * S;
        const double cx = ((double)m0 + 0.5) * unit, cy = ((double)m1 + 0.5) * unit;
        const double rx = R / (f1 - f0), ry = R / (f3 - f2);
        const double lox = (cx - rx) * (f1 - f0) + f0, loy = (cy - ry) * (f3 - f2) + f2;      /* up_mapping :91-93 */
        const double hix = (cx + rx) * (f1 - f0) + f0, hiy = (cy + ry) * (f3 - f2) + f2;
        double x = (lox + hix) / 2.0, y = (loy + hiy) / 2.0;
        /* only nodes within R of SOME point of the box can ever count: collect them once (id order) with their weights;
           the climb then evaluates the objective from shared memory instead of walking all N nodes in HBM per trial */
        const double reach = R * 2.4143 + 1e-6;      /* R + half diagonal of the +-R box */
        int cnt = 0;
        for (int base = 0; base < N; base += 32) {
            const int i = base + lane;
            bool c = false; double wx = 0.0, wy = 0.0, ww = 0.0;
            if (i < N && status[i] != 0) {
                wx = nx[i]; wy = ny[i];
                const double dx = x - wx, dy = y - wy;
                if (dx * dx + dy * dy <= reach * reach) { c = true; ww = cs[i] / (energy[i] - thr) * alpha; }
            }
            const unsigned m = __ballot_sync(0xffffffffu, c);
            const int slot = cnt + __popc(m & ((1u << lane) - 1u));
            if (c && slot < DEC_MAXC) { cn_x[slot] = wx; cn_y[slot] = wy; cn_w[slot] = ww; }
            cnt += __popc(m);
        }
        __syncwarp();
        const bool listed = cnt <= DEC_MAXC;
        /* value and gradient of the (positive) objective at (px, py): every lane its nodes, shuffle-tree sums */
        auto eval = [&](double px, double py, double &F, double &gx, double &gy) {
            double f = 0.0, ax = 0.0, ay = 0.0;
            if (listed) {
                for (int j = lane; j < cnt; j += 32) {
                    const double dx = px - cn_x[j], dy = py - cn_y[j];
                    const double d = sqrt(dx * dx + dy * dy);
                    if (d <= R) {
                        const double w = cn_w[j], t = d + beta;
                        f += w / (t * t);
                        if (d > 0.0) { const double c = -2.0 * w / (t * t * t) / d; ax += c * dx; ay += c * dy; }
                    }
                }
            } else {
                for (int i = lane; i < N; i += 32) {
                    if (status[i] == 0) continue;
                    const double dx = px - nx[i], dy = py - ny[i];
                    const double d = sqrt(dx * dx + dy * dy);
                    if (d <= R) {
                        const double w = cs[i] / (energy[i] - thr) * alpha, t = d + beta;
                        f += w / (t * t);
                        if (d > 0.0) { const double c = -2.0 * w / (t * t * t) / d; ax += c * dx; ay += c * dy; }
                    }
                }
            }
            for (int o = 16; o > 0; o >>= 1) {
                f += __shfl_xor_sync(0xffffffffu, f, o); ax += __shfl_xor_sync(0xffffffffu, ax, o); ay += __shfl_xor_sync(0xffffffffu, ay, o);
            }
            F = f; gx = ax; gy = ay;
        };
        double F, gx, gy;
        eval(x, y, F, gx, gy);
        double t = 1.0;                              /* L-BFGS-B's first step: the Cauchy point of the unit-Hessian model */
        for (int it = 0; it < 100; it++) {
            double px = gx, py = gy;                 /* projected gradient */
            if ((x <= lox && px < 0.0) || (x >= hix && px > 0.0)) px = 0.0;
            if ((y <= loy && py < 0.0) || (y >= hiy && py > 0.0)) py = 0.0;
            if (fmax(fabs(px), fabs(py)) <= 1e-5) break;                      /* pgtol */
            double tt = t, xn = x, yn = y, Fn = F, gxn = gx, gyn = gy;
            bool ok = false;
            for (int ls = 0; ls < 40; ls++) {
                xn = fmin(fmax(x + tt * px, lox), hix); yn = fmin(fmax(y + tt * py, loy), hiy);
                eval(xn, yn, Fn, gxn, gyn);
                if (Fn > F) { ok = true; break; }
                tt *= 0.5;
            }
            if (!ok) break;
            const double sx = xn - x, sy = yn - y, yx = -(gxn - gx), yy = -(gyn - gy);     /* s, y of the minimised -F */
            const double s_y = sx * yx + sy * yy, y_y = yx * yx + yy * yy;
            const bool done = (Fn - F) <= 2.220446049250313e-09 * fmax(fmax(fabs(F), fabs(Fn)), 1.0);   /* ftol = factr * epsmch */
            x = xn; y = yn; F = Fn; gx = gxn; gy = gyn;
            if (done) break;
            t = (s_y > 0.0 && y_y > 0.0) ? s_y / y_y : tt * 4.0;
        }
        out_x = (x - f0) / (f1 - f0); out_y = (y - f2) / (f3 - f2);                            /* down_mapping :86-88 */
        }
    if (lane == 0) { action[3 * (size_t)b] = out_x; action[3 * (size_t)b + 1] = out_y; }
}

/* Launch order of the step kernel: the hardware hands CTAs to the SMs in index order, and a launch whose last CTAs are long
 * environments ends on a tail of idle SMs (measured: 11 of 16 resident warps active on average).  One CTA sorts the rows by the
 * work their step is expected to take — the time to the earliest next decision among the alive chargers, read from the process
 * slots (a move's remaining time + its charge, a charge's remaining time; MobileCharger.py:80-98, :55-70) or, for the charger
 * that has just been given an action, from that action (WRSN.py:95-98) — capped by the step budget, into five classes, longest
 * first; rows the launch does not touch come last.  Only the ORDER of execution changes, never a result. */
#define ORD_THREADS 1024
#define ORD_MAX_ROWS 16                              /* rows per thread: B <= 16384 */
__global__ void __launch_bounds__(ORD_THREADS) k_step_order(const KParams P, int32_t *order) {
    __shared__ int s_cnt[5], s_off[5];
    const int B = P.d.B, M = P.d.M;
    const double W = P.d.step_budget > 0 ? (double)P.d.step_budget : 100.0;
    if (threadIdx.x < 5) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    int bins[ORD_MAX_ROWS];
#pragma unroll
    for (int q = 0; q < ORD_MAX_ROWS; q++) {
        const int b = threadIdx.x + q * ORD_THREADS;
        bins[q] = -1;
        if (b >= B) continue;
        const int aid = P.agent_in ? P.agent_in[b] : -1;
        const int raid = P.req.agent_id ? P.req.agent_id[b] : 0;
        int bin = 4;
        if (!((P.mask && !P.mask[b]) || (P.mask_mode == 1 && raid < 0 && raid != -4))) {
            const WrsnRow rw(P.L, P.state, P.scen, P.scen_id, b);
            const double *hdr = rw.hdr, *mc = rw.mc, *proc = rw.proc, *par = rw.par;
            const double now = hdr[WRSN_H_NOW];
            const bool fresh = hdr[WRSN_H_INFLIGHT] == 0.0 && aid >= 0 && aid < M && P.action_in;
            double rem = INFINITY;
            for (int a = 0; a < M; a++) {
                const double *m = mc + a * WRSN_MC_LEN;
                if (m[WRSN_MC_STATUS] == 0.0) continue;
                double r = 0.0;
                if (fresh && a == aid) {
                    const double *act = P.action_in + 3 * (size_t)b;
                    const double a0 = fmin(fmax(act[0], 0.0), 1.0), a1 = fmin(fmax(act[1], 0.0), 1.0), a2 = fmin(fmax(act[2], 0.0), 1.0);
                    const double dx = a0 * (par[WRSN_P_F1] - par[WRSN_P_F0]) + par[WRSN_P_F0] - m[WRSN_MC_X];
                    const double dy = a1 * (par[WRSN_P_F3] - par[WRSN_P_F2]) + par[WRSN_P_F2] - m[WRSN_MC_Y];
                    r = sqrt(dx * dx + dy * dy) / par[WRSN_P_MC_V] + par[WRSN_P_CTM] * a2;
                } else {
                    const int s = (int)m[WRSN_MC_SLOT];
                    if (s >= 0 && s < P.d.n_slot) {
                        const double *p = proc + s * WRSN_PR_LEN;
                        const int pc = reinterpret_cast<const int *>(p)[WRSN_PRI_PC];
                        if (pc == g32::PC_MS_FIRE) r = (p[WRSN_PR_T] - now) + p[WRSN_PR_MT] + p[WRSN_PR_PHY2];
                        else if (pc == g32::PC_CS_FIRE) r = (p[WRSN_PR_T] - now) + p[WRSN_PR_CHTMP];
                    }
                }
                rem = fmin(rem, r);
            }
            if (!(rem < INFINITY) || !(rem > 0.0)) rem = 0.0;
            bin = rem >= W ? 0 : (rem >= 0.6 * W ? 1 : (rem >= 0.3 * W ? 2 : 3));
        }
        bins[q] = bin;
        atomicAdd(&s_cnt[bin], 1);
    }
    __syncthreads();
    if (threadIdx.x == 0) { int o = 0; for (int k = 0; k < 5; k++) { s_off[k] = o; o += s_cnt[k]; } }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < ORD_MAX_ROWS; q++)
        if (bins[q] >= 0) order[atomicAdd(&s_off[bins[q]], 1)] = threadIdx.x + q * ORD_THREADS;
}

/* the charging model, dense: one warp per environment (see include/wrsn_b200.h: wrsn_k_charge) */
#define CHG_WARPS 4
__global__ void __launch_bounds__(32 * CHG_WARPS) k_charge(const KParams P, const uint8_t *__restrict__ charging,
                                                           double *__restrict__ node_rate, double *__restrict__ mc_rate) {
    __shared__ double s_mx[CHG_WARPS][WRSN_MAX_MC], s_my[CHG_WARPS][WRSN_MAX_MC], s_sum[CHG_WARPS][WRSN_MAX_MC];
    __shared__ uint8_t s_on[CHG_WARPS][WRSN_MAX_MC];
    const int wrp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * CHG_WARPS + wrp;
    if (b >= P.d.B) return;                                   /* whole warps leave together; only __syncwarp below */
    const int NP = P.d.N, M = P.d.M;                          /* node_rate's row pitch: the batch's largest node count */
    const WrsnRow rw(P.L, P.state, P.scen, P.scen_id, b);
    const int N = rw.N;                                       /* this scenario's nodes; node_rate[b][N..NP) is left untouched */
    const double *nx = rw.nx, *ny = rw.ny, *mc = rw.mc;
    const uint8_t *status = rw.status;
    const double R = rw.par[WRSN_P_MC_R], alpha = rw.par[WRSN_P_MC_ALPHA], beta = rw.par[WRSN_P_MC_BETA];
    for (int m = lane; m < M; m += 32) {                      /* stage the chargers of this environment */
        s_mx[wrp][m] = mc[(size_t)m * WRSN_MC_LEN + WRSN_MC_X];
        s_my[wrp][m] = mc[(size_t)m * WRSN_MC_LEN + WRSN_MC_Y];
        s_on[wrp][m] = charging ? charging[(size_t)b * M + m] : 1;
        s_sum[wrp][m] = 0.0;
    }
    __syncwarp();
    for (int base = 0; base < N; base += 32) {
        const int n = base + lane;
        const bool live = n < N && status[n] != 0;            /* charger_connection returns at once for a dead node */
        const double x = live ? nx[n] : 0.0, y = live ? ny[n] : 0.0;
        double acc = 0.0;                                     /* this node's energyRR: += in charger order */
        for (int m = 0; m < M; m++) {
            if (!s_on[wrp][m]) continue;                      /* warp-uniform */
            double rate = 0.0;
            bool in = false;
            if (live) {
                const double dx = x - s_mx[wrp][m], dy = y - s_my[wrp][m];
                const double dist = sqrt(dx * dx + dy * dy);  /* scipy's euclidean: sqrt(dot(u - v, u - v)) */
                in = dist <= R;
                if (in) { const double t = dist + beta; rate = alpha / (t * t); acc = acc + rate; }
            }
            /* the charger's chargingRate: += over its connected nodes IN NODE ORDER — lane by lane through the ballot */
            unsigned bits = __ballot_sync(0xffffffffu, in);
            if (bits) {
                double sum = s_sum[wrp][m];
                for (unsigned rest = bits; rest; rest &= rest - 1u) {
                    const double r = __shfl_sync(0xffffffffu, rate, __ffs(rest) - 1);
                    sum = sum + r;
                }
                if (lane == 0) s_sum[wrp][m] = sum;
                __syncwarp();
            }
        }
        if (n < N) node_rate[(size_t)b * NP + n] = acc;
    }
    __syncwarp();
    for (int m = lane; m < M; m += 32) mc_rate[(size_t)b * M + m] = s_sum[wrp][m];
}

/* roll_out bookkeeping (IPPO.py:138-155): one thread per environment, see include/wrsn_b200.h */
__global__ void k_record_transitions(int B, int M, wrsn_request req, int64_t t, const int64_t *__restrict__ agent_prev,
                                     int64_t *__restrict__ last, double *__restrict__ resets_seen,
                                     int64_t *__restrict__ agent_next, int64_t *__restrict__ link_next,
                                     uint8_t *__restrict__ new_episode_next, double *__restrict__ reward_next,
                                     double *__restrict__ now_next) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    record_transition(b, M, req, t, agent_prev, last, resets_seen, agent_next, link_next, new_episode_next, reward_next, now_next);
}

#include "wrsn_abi_host.h"
#include "wrsn_abi_aux.h"
static_assert(WRSN_DEC_MAX_RANK == DEC_MAXR - 2, "the host refuses the map sizes whose rank k_decode_map cannot hold");

template <int MODE>
static int launch_env(KParams &P, void *stream) {
    if (prepare_launch(P)) return -1;
    /* the opt-in dynamic shared-memory limit is a per-DEVICE attribute of the function: cache it per template instance, group
       build and device (a second GPU in the same process needs its own opt-in) */
    static int64_t attr_cache[2][WRSN_MAX_DEVICES];
    static bool attr_init = false;
    if (!attr_init) { for (int w_ = 0; w_ < 2; w_++) for (int q = 0; q < WRSN_MAX_DEVICES; q++) attr_cache[w_][q] = 48 * 1024; attr_init = true; }
    int dev = 0;
    WRSN_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= WRSN_MAX_DEVICES) WRSN_FAIL("device ordinal %d not supported", dev);
    static int64_t pad = -1;                         /* TUNING KNOB (WRSN_SMEM_PAD bytes): fewer resident environments per SM */
    if (pad < 0) { const char *e = getenv("WRSN_SMEM_PAD"); pad = e ? atoll(e) : 0; if (pad < 0 || pad > 200 * 1024) pad = 0; }
    const int w = P.d.threads == 32 ? 0 : 1;
    const int64_t smem = P.L.smem_total + pad;
    if (smem > attr_cache[w][dev]) {
        if (w == 0) WRSN_CUDA(cudaFuncSetAttribute(g32::k_env<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        else WRSN_CUDA(cudaFuncSetAttribute(gany::k_env<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_cache[w][dev] = smem;
    }
    if (w == 0) g32::k_env<MODE><<<P.d.B, 32, (size_t)smem, (cudaStream_t)stream>>>(P);
    else gany::k_env<MODE><<<P.d.B, P.d.threads, (size_t)smem, (cudaStream_t)stream>>>(P);
    WRSN_CUDA(cudaGetLastError());
    return 0;
}

/* Measured (4096 environments, RandomController law): one launch of 4096 rows 1.03 -> 1.13 M decisions/s with the order; four
   groups of 1024 rows on four streams 1.20 -> 1.23 M (the other groups' kernels already fill the tail, and the ordering kernel
   costs 23 us per launch).  So: rows are ordered when one launch holds at least 2048 of them.  TUNING KNOB WRSN_STEP_ORDER:
   0 never, 1 always (B > 32). */
static int order_rows(KParams &P, void *stream) {
    static int use_order = -1;
    if (use_order < 0) { const char *e = getenv("WRSN_STEP_ORDER"); use_order = e ? atoi(e) : 2; }
    if (use_order && P.req.order && P.d.B > (use_order == 2 ? 2047 : 32) && P.d.B <= ORD_THREADS * ORD_MAX_ROWS && P.scen && P.scen_id && P.state) {
        if (check_dims(&P.d)) return -1;
        wrsn_make_layout(&P.d, &P.L);
        k_step_order<<<1, ORD_THREADS, 0, (cudaStream_t)stream>>>(P, P.req.order);
        WRSN_CUDA(cudaGetLastError());
        P.order = P.req.order;
    }
    return 0;
}

extern "C" {

int wrsn_device_ok(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) { cudaGetLastError(); snprintf(g_err, sizeof(g_err), "no CUDA device"); return 0; }
    int dev = 0; cudaGetDevice(&dev);
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, dev) != cudaSuccess) return 0;
    if (p.major != 10) { snprintf(g_err, sizeof(g_err), "device is sm_%d%d, this library is built for sm_100a only", p.major, p.minor); return 0; }
    return 1;
}

}  /* extern "C" */

static int launch_obs_tables(KParams &P, void *stream) {
    k_obs_tables<<<dim3(P.d.n_scen, P.d.Npad), 128, 0, (cudaStream_t)stream>>>(P.d, P.L, const_cast<char *>(P.scen));
    WRSN_CUDA(cudaGetLastError());
    return 0;
}

static int launch_observe(KParams &P, const int32_t *agent_id, void *obs, int obs_f64, void *stream) {
    const wrsn_dims *d = &P.d;
    if (obs_f64) {
        size_t smem = sizeof(double) * 2 * 16 * (size_t)d->obs_pitch;
        if (smem > 200 * 1024) WRSN_FAIL("map_size too large");
        if (smem > 48 * 1024) WRSN_CUDA(cudaFuncSetAttribute(k_observe<double, OBS_TJ64, OBS_THREADS64>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        k_observe<double, OBS_TJ64, OBS_THREADS64><<<d->B, OBS_THREADS64, smem, (cudaStream_t)stream>>>(P, agent_id, (double *)obs);
    } else {
        /* the windowed raster: map sizes it is laid out for, sources narrow enough for its window (the host layer says so in
           dims.obs_sigma_cells: the largest charging_range / extent * S over the scenarios; 0 = unknown), shared memory
           (measured: the 40-cell window — 4 CTAs per SM — beats the chunked raster; 56 / 72 cells leave 3 / 2 CTAs per SM and
           lose to it, 0.79 ms against 0.52 ms per 4096 maps at 72: wider sources stay with the chunked kernel) */
        const float sg = d->obs_sigma_cells;
        const size_t wsmem = sizeof(float) * ((size_t)(d->N + 2 * d->M) * (OBW + OBW + 2 * OBM) + 2 * (size_t)d->obs_pitch) + sizeof(WinSrc) * (size_t)(d->N + 2 * d->M);
        if (sg > 0.0f && sg <= 2.9f && d->S % 20 == 0 && d->S >= OBW && (d->S / OBS_TI) * (d->S / OBS_TJ32) <= OBW_THREADS && wsmem <= 100 * 1024) {
            static bool wattr[WRSN_MAX_DEVICES];
            int dev = 0;
            WRSN_CUDA(cudaGetDevice(&dev));
            if (dev < 0 || dev >= WRSN_MAX_DEVICES) WRSN_FAIL("device ordinal %d not supported", dev);
            if (!wattr[dev]) { WRSN_CUDA(cudaFuncSetAttribute(k_observe_win, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024)); wattr[dev] = true; }
            k_observe_win<<<d->B, OBW_THREADS, wsmem, (cudaStream_t)stream>>>(P, agent_id, (float *)obs);
            WRSN_CUDA(cudaGetLastError());
            return 0;
        }
        size_t smem = sizeof(float) * 2 * OBS_CH32 * (size_t)d->obs_pitch;
        if (smem > 200 * 1024) WRSN_FAIL("map_size too large");
        static bool attr[WRSN_MAX_DEVICES];            /* per device, see launch_env */
        int dev = 0;
        WRSN_CUDA(cudaGetDevice(&dev));
        if (dev < 0 || dev >= WRSN_MAX_DEVICES) WRSN_FAIL("device ordinal %d not supported", dev);
        if (!attr[dev]) { WRSN_CUDA(cudaFuncSetAttribute(k_observe<float, OBS_TJ32, OBS_THREADS32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)); attr[dev] = true; }
        k_observe<float, OBS_TJ32, OBS_THREADS32><<<d->B, OBS_THREADS32, smem, (cudaStream_t)stream>>>(P, agent_id, (float *)obs);
    }
    WRSN_CUDA(cudaGetLastError());
    return 0;
}

/* channels = 0: dmap is the map (float64 if dmap_f64); otherwise the float observations, combined with weights[channels] */
static int launch_decode(KParams &P, const int32_t *agent_id, const void *dmap, int dmap_f64, int channels, const float *weights,
                         double *action_out, void *stream) {
    const int B = P.d.B;
    LinMap lin; memset(&lin, 0, sizeof(lin));
    lin.C = channels;
    for (int k = 0; k < channels; k++) lin.w[k] = weights[k];
    if (channels == 0 && dmap_f64) k_decode_map<double, 0><<<B, DEC_THREADS, 0, (cudaStream_t)stream>>>(P, agent_id, (const double *)dmap, action_out, lin);
    else if (channels == 0) k_decode_map<float, 0><<<B, DEC_THREADS, 0, (cudaStream_t)stream>>>(P, agent_id, (const float *)dmap, action_out, lin);
    else if (channels == 4) k_decode_map<float, 4><<<B, DEC_THREADS, 0, (cudaStream_t)stream>>>(P, agent_id, (const float *)dmap, action_out, lin);
    else k_decode_map<float, -1><<<B, DEC_THREADS, 0, (cudaStream_t)stream>>>(P, agent_id, (const float *)dmap, action_out, lin);
    k_decode_locate<<<(B + LOC_WARPS - 1) / LOC_WARPS, 32 * LOC_WARPS, 0, (cudaStream_t)stream>>>(P, agent_id, action_out);
    WRSN_CUDA(cudaGetLastError());
    return 0;
}

static int launch_charge(KParams &P, const uint8_t *charging, double *node_rate, double *mc_rate, void *stream) {
    k_charge<<<(P.d.B + CHG_WARPS - 1) / CHG_WARPS, 32 * CHG_WARPS, 0, (cudaStream_t)stream>>>(P, charging, node_rate, mc_rate);
    WRSN_CUDA(cudaGetLastError());
    return 0;
}
