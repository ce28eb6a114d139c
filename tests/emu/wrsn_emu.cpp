/*
 * wrsn_emu.cpp — TEST INFRASTRUCTURE.  Single-lane host build of the kernel source
 * (multi_agent_rl_wrsn_b200/csrc/wrsn_engine.cuh with WRSN_HOST_EMU): the same event logic, the same per-environment
 * driver (wrsn_env_kernel.cuh: env_run) and the same host side of the ABI (wrsn_abi_host.h) as the sm_100a library,
 * with one "thread" per environment, on host memory.  It exists so the
 * `-m "not gpu"` tests can check the engine's event ordering and arithmetic against the oracle on a box
 * without a GPU.  It is built only by tests/ (tests/emu/Makefile), exports the C ABI of
 * include/wrsn_b200.h, and is never loaded by the product package, which has no CPU path.
 * The entry points' checks are those of the CUDA library (wrsn_abi_host.h).  wrsn_observe is a host restatement of the fp64
 * parity raster over the same sources (wrsn_layout.h: obs_source), and wrsn_k_charge one of k_charge (the raster kernels and
 * the charging kernel themselves are checked on the GPU); the density-map decoder is not emulated: its entry points refuse
 * what the CUDA library refuses, then report that they are not available.
 */
#define WRSN_HOST_EMU 1
#include <stdio.h>
#include <stdlib.h>
#include <algorithm>
#include <vector>

#include "wrsn_launch.h"
static thread_local char *wrsn_smem_host = nullptr;
#define WRSN_GFIX 1
#include "wrsn_engine.cuh"

#include "wrsn_env_kernel.cuh"
#include "wrsn_abi_host.h"
#include "wrsn_abi_aux.h"

/* one "launch": every row of the batch in turn, on one lane, in the image the engine addresses as its shared memory */
template <int MODE>
static int launch_env(KParams &P, void *) {
    if (prepare_launch(P)) return -1;
    std::vector<char> smem((size_t)P.L.smem_total + 64);
    wrsn_smem_host = smem.data();
    for (int b = 0; b < P.d.B; b++) env_run<MODE>(P, b, 0, 1);
    return 0;
}

static int order_rows(KParams &, void *) { return 0; }   /* rows run one after the other: the order changes nothing */

static int launch_obs_tables(KParams &, void *) { return 0; }   /* only the CUDA raster reads them */

/* WRSN.get_state (rl_env/WRSN.py:130-186) as k_observe<double> computes it: the same sources in the same order, the same
 * rounding ((w * gx) * gy added term by term; channel 3 as ((gx * gy) * w) / moving_time_max).  float output = the fp64 map
 * rounded once (the GPU's fp32 rasters accumulate in fp32: equal to ~1e-6 of the channel maximum, not bit for bit). */
static int launch_observe(KParams &P, const int32_t *agent_id, void *obs, int obs_f64, void *) {
    const int S = P.d.S, M = P.d.M;
    const size_t SS = (size_t)S * S;
    std::vector<double> out(SS), gx(S), gy(S);
    for (int b = 0; b < P.d.B; b++) {
        const int ag = agent_id[b];
        if (ag < 0) continue;
        const WrsnRow rw(P.L, P.state, P.scen, P.scen_id, b);
        const ObsGrid g(rw.par, S);
        for (int ch = 0; ch < 4; ch++) {
            std::fill(out.begin(), out.end(), 0.0);
            const int total = ch == 0 ? rw.N : (ch == 1 ? 1 : M);
            for (int s = 0; s < total; s++) {
                const ObsSrc v = obs_source(rw, g, ag, ch, s);
                if (v.mode < 0) continue;
                const double dnx = -2.0 * (v.hx * v.hx), dny = -2.0 * (v.hy * v.hy);
                for (int i = 0; i < S; i++) { gx[i] = obs_gauss(g.cell(i), v.x0, dnx); gy[i] = obs_gauss(g.cell(i), v.y0, dny); }
                for (int i = 0; i < S; i++)
                    for (int j = 0; j < S; j++) {
                        double &o = out[(size_t)i * S + j];
                        if (v.mode == 0) { const double a = v.w * gx[i]; o = o + a * gy[j]; }
                        else o = o + gx[i] * gy[j] * v.w / g.mtm;
                    }
            }
            for (size_t k = 0; k < SS; k++) {
                if (obs_f64) ((double *)obs)[((size_t)b * 4 + ch) * SS + k] = out[k];
                else ((float *)obs)[((size_t)b * 4 + ch) * SS + k] = (float)out[k];
            }
        }
    }
    return 0;
}

static int launch_decode(KParams &, const int32_t *, const void *, int, int channels, const float *, double *, void *) {
    WRSN_FAIL("%s is not available in the host emulation", channels ? "wrsn_decode_linear_controller" : "wrsn_decode_density_map");
}

/* k_charge: the reference's loops, literally, over each row's own nodes; node_rate[b][N..) is left untouched */
static int launch_charge(KParams &P, const uint8_t *charging, double *node_rate, double *mc_rate, void *) {
    const int NP = P.d.N, M = P.d.M;
    for (int b = 0; b < P.d.B; b++) {
        const WrsnRow rw(P.L, P.state, P.scen, P.scen_id, b);
        const double *par = rw.par;
        for (int n = 0; n < rw.N; n++) node_rate[(size_t)b * NP + n] = 0.0;
        for (int m = 0; m < M; m++) {
            double sum = 0.0;
            if (!charging || charging[(size_t)b * M + m])
                for (int n = 0; n < rw.N; n++) {
                    if (rw.status[n] == 0) continue;
                    const double dist = euclid2(rw.nx[n], rw.ny[n], rw.mc[(size_t)m * WRSN_MC_LEN + WRSN_MC_X], rw.mc[(size_t)m * WRSN_MC_LEN + WRSN_MC_Y]);
                    if (!(dist <= par[WRSN_P_MC_R])) continue;
                    const double t = dist + par[WRSN_P_MC_BETA], rate = par[WRSN_P_MC_ALPHA] / (t * t);
                    node_rate[(size_t)b * NP + n] += rate;
                    sum += rate;
                }
            mc_rate[(size_t)b * M + m] = sum;
        }
    }
    return 0;
}

extern "C" {
int wrsn_is_emulation(void) { return 1; }
int wrsn_device_ok(void) { return 0; }
}  /* extern "C" */
