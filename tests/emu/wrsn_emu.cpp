/*
 * wrsn_emu.cpp — TEST INFRASTRUCTURE.  Single-lane host build of the kernel source
 * (multi_agent_rl_wrsn_b200/csrc/wrsn_engine.cuh with WRSN_HOST_EMU): the same event logic, the same per-environment
 * driver (wrsn_env_kernel.cuh: env_run) and the same host side of the ABI (wrsn_abi_host.h) as the sm_100a library,
 * with one "thread" per environment, on host memory.  It exists so the
 * `-m "not gpu"` tests can check the engine's event ordering and arithmetic against the oracle on a box
 * without a GPU.  It is built only by tests/ (tests/emu/Makefile), exports the C ABI of
 * include/wrsn_b200.h, and is never loaded by the product package, which has no CPU path.
 * wrsn_observe is a plain host restatement of the fp64 parity raster (the raster kernels themselves are checked on the GPU);
 * wrsn_decode_density_map is not emulated (it only checks its dims and map size, as the CUDA library does).
 */
#define WRSN_HOST_EMU 1
#include <stdio.h>
#include <stdlib.h>
#include <vector>

#include "wrsn_launch.h"
static thread_local char *wrsn_smem_host = nullptr;
#define WRSN_GFIX 1
#include "wrsn_engine.cuh"

#include "wrsn_env_kernel.cuh"
#include "wrsn_abi_host.h"

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

extern "C" {
int wrsn_is_emulation(void) { return 1; }
int wrsn_device_ok(void) { return 0; }
int wrsn_build_obs_tables(const wrsn_dims *, void *, void *) { return 0; }   /* only the CUDA raster reads them */

/* WRSN.get_state (rl_env/WRSN.py:130-186), host restatement of the fp64 parity raster k_observe<double> (same source order,
 * same rounding: (w * gx) * gy added term by term; channel 4 as ((gx * gy) * w) / moving_time_max).  float output = the fp64
 * map rounded once (the GPU's fp32 raster accumulates in fp32: equal to ~1e-6 of the channel maximum, not bit for bit). */
static void emu_add_source(std::vector<double> &out, int S, double x0, double y0, double hx, double hy, double w, int mode, double mtm) {
    const double unit = 1.0 / (double)S, start = unit / 2.0, delta = (start + unit) - start;
    const double dnx = -2.0 * (hx * hx), dny = -2.0 * (hy * hy);
    std::vector<double> gx(S), gy(S);
    for (int i = 0; i < S; i++) {
        const double cc = start + (double)i * delta, ux = cc - x0, uy = cc - y0;
        const double ax = ux * ux / dnx, ay = uy * uy / dny;
        gx[i] = ax > -745.2 ? exp(ax) : 0.0;
        gy[i] = ay > -745.2 ? exp(ay) : 0.0;
    }
    for (int i = 0; i < S; i++)
        for (int j = 0; j < S; j++) {
            double &o = out[(size_t)i * S + j];
            if (mode == 0) { const double a = w * gx[i]; o = o + a * gy[j]; }
            else o = o + gx[i] * gy[j] * w / mtm;
        }
}
int wrsn_observe(const wrsn_dims *d, const void *scen, const int32_t *scen_id, const void *state, const int32_t *agent_id,
                 void *obs, int obs_f64, void *) {
    if (!d || !scen || !scen_id || !state || !agent_id || !obs) WRSN_FAIL("NULL argument");
    WrsnLayout L; wrsn_make_layout(d, &L);
    const int S = d->S, M = d->M;
    const size_t SS = (size_t)S * S;
    for (int b = 0; b < d->B; b++) {
        const int ag = agent_id[b];
        if (ag < 0) continue;
        const char *row = (const char *)state + (size_t)b * L.total;
        const char *scen_row = (const char *)scen + (size_t)scen_id[b] * L.scen_total;
        const double *par = (const double *)(scen_row + L.soff[WRSN_S_PAR]);
        const double *nx = (const double *)(scen_row + L.soff[WRSN_S_NX]), *ny = (const double *)(scen_row + L.soff[WRSN_S_NY]);
        const double *energy = (const double *)(row + L.off[WRSN_F_ENERGY]), *cs = (const double *)(row + L.off[WRSN_F_CS]);
        const uint8_t *status = (const uint8_t *)(row + L.off[WRSN_F_STATUS]);
        const double *mc = (const double *)(row + L.off[WRSN_F_MC]);
        const double f0 = par[WRSN_P_F0], f1 = par[WRSN_P_F1], f2 = par[WRSN_P_F2], f3 = par[WRSN_P_F3];
        const double Wd = f1 - f0, Hd = f3 - f2, R = par[WRSN_P_MC_R], mtm = par[WRSN_P_MTM];
        const double *me = mc + (size_t)ag * WRSN_MC_LEN;
        for (int ch = 0; ch < 4; ch++) {
            std::vector<double> out(SS, 0.0);
            if (ch == 0) {
                const int Nrow = (int)par[WRSN_P_NNODES];        /* this row's own nodes, as the kernels read them */
                for (int s = 0; s < Nrow; s++) {
                    if (status[s] == 0) continue;
                    const double w = (cs[s] / par[WRSN_P_MC_AB2]) / ((energy[s] - par[WRSN_P_THR]) / par[WRSN_P_CAPMTHR]);
                    if (w == 0.0) continue;
                    emu_add_source(out, S, (nx[s] - f0) / Wd, (ny[s] - f2) / Hd, R / Wd, R / Hd, w, 0, mtm);
                }
            } else if (ch == 1) {
                const double tmp = fmin(Hd, Wd);
                emu_add_source(out, S, (me[WRSN_MC_X] - f0) / Wd, (me[WRSN_MC_Y] - f2) / Hd, 0.5 * tmp / Wd, 0.5 * tmp / Hd,
                               me[WRSN_MC_ENERGY] / par[WRSN_P_MC_CAP], 0, mtm);
            } else {
                for (int s = 0; s < M; s++) {
                    const double *an = mc + (size_t)s * WRSN_MC_LEN;
                    const bool charging = an[WRSN_MC_TYPE] != 0.0;
                    if (s == ag || (ch == 2 ? !charging : charging)) continue;
                    const double x0 = (an[WRSN_MC_CPA0] - f0) / Wd, y0 = (an[WRSN_MC_CPA1] - f2) / Hd;
                    if (ch == 2) emu_add_source(out, S, x0, y0, R / Wd, R / Hd, an[WRSN_MC_CPA2] / par[WRSN_P_CTM], 0, mtm);
                    else {                               /* SURVEY Q5: the observer's destination y */
                        const double dx = an[WRSN_MC_X] - an[WRSN_MC_CPA0], dy = an[WRSN_MC_Y] - me[WRSN_MC_CPA1];
                        emu_add_source(out, S, x0, y0, R / Wd, R / Hd, sqrt(dx * dx + dy * dy) / par[WRSN_P_MC_V], 1, mtm);
                    }
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
/* the decoder is not emulated; its entry points refuse what the CUDA library refuses first, with the same message */
int wrsn_decode_linear_controller(const wrsn_dims *d, const void *, const int32_t *, const void *, const int32_t *, const float *, int, const float *,
                                  double *, void *) {
    if (check_dims(d) || check_decode_size(d)) return -1;
    WRSN_FAIL("wrsn_decode_linear_controller is not available in the host emulation");
}
int wrsn_decode_density_map(const wrsn_dims *d, const void *, const int32_t *, const void *, const int32_t *, const void *, int, double *, void *) {
    if (check_dims(d) || check_decode_size(d)) return -1;
    WRSN_FAIL("wrsn_decode_density_map is not available in the host emulation");
}
int wrsn_k_charge(const wrsn_dims *d, const void *scen, const int32_t *scen_id, const void *state, const uint8_t *charging,
                  double *node_rate, double *mc_rate, void *) {
    if (!d || !scen || !scen_id || !state || !node_rate || !mc_rate) WRSN_FAIL("NULL argument");
    if (d->M <= 0) WRSN_FAIL("no chargers");
    WrsnLayout L; wrsn_make_layout(d, &L);
    for (int b = 0; b < d->B; b++) {                     /* host restatement of k_charge: the reference's loops, literally */
        const char *row = (const char *)state + (size_t)b * L.total;
        const char *scen_row = (const char *)scen + (size_t)scen_id[b] * L.scen_total;
        const double *par = (const double *)(scen_row + L.soff[WRSN_S_PAR]);
        const double *nx = (const double *)(scen_row + L.soff[WRSN_S_NX]), *ny = (const double *)(scen_row + L.soff[WRSN_S_NY]);
        const uint8_t *status = (const uint8_t *)(row + L.off[WRSN_F_STATUS]);
        const double *mc = (const double *)(row + L.off[WRSN_F_MC]);
        for (int n = 0; n < d->N; n++) node_rate[(size_t)b * d->N + n] = 0.0;
        for (int m = 0; m < d->M; m++) {
            double sum = 0.0;
            if (!charging || charging[(size_t)b * d->M + m])
                for (int n = 0; n < d->N; n++) {
                    if (status[n] == 0) continue;
                    const double dist = euclid2(nx[n], ny[n], mc[(size_t)m * WRSN_MC_LEN + WRSN_MC_X], mc[(size_t)m * WRSN_MC_LEN + WRSN_MC_Y]);
                    if (!(dist <= par[WRSN_P_MC_R])) continue;
                    const double t = dist + par[WRSN_P_MC_BETA], rate = par[WRSN_P_MC_ALPHA] / (t * t);
                    node_rate[(size_t)b * d->N + n] += rate;
                    sum += rate;
                }
            mc_rate[(size_t)b * d->M + m] = sum;
        }
    }
    return 0;
}
}  /* extern "C" */
