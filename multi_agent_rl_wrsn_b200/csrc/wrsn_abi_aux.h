/*
 * wrsn_abi_aux.h — the entry points of the C ABI (include/wrsn_b200.h) outside the environment kernel: the observation raster,
 * the density-map decoder, the charging model and the raster's scenario tables.  The CUDA library (wrsn_kernels.cu) and the
 * tests' host emulation (tests/emu/wrsn_emu.cpp) share their argument checks and KParams; included once, after
 * wrsn_abi_host.h, and the including file supplies the work on checked arguments:
 *   launch_obs_tables(P, stream)                                  wrsn_build_obs_tables;
 *   launch_observe(P, agent_id, obs, obs_f64, stream)             wrsn_observe;
 *   launch_decode(P, agent_id, dmap, dmap_f64, channels, weights, action_out, stream)
 *                                                                 both decode entry points (channels = 0: dmap is the map);
 *   launch_charge(P, charging, node_rate, mc_rate, stream)        wrsn_k_charge.
 */
#pragma once
#include "wrsn_abi_host.h"

static int launch_obs_tables(KParams &P, void *stream);
static int launch_observe(KParams &P, const int32_t *agent_id, void *obs, int obs_f64, void *stream);
static int launch_decode(KParams &P, const int32_t *agent_id, const void *dmap, int dmap_f64, int channels, const float *weights,
                         double *action_out, void *stream);
static int launch_charge(KParams &P, const uint8_t *charging, double *node_rate, double *mc_rate, void *stream);

/* once the arguments are checked: the dims and the layout they imply */
static KParams aux_params(const wrsn_dims *d, const void *scen, const int32_t *scen_id, const void *state) {
    KParams P = base_params(d, scen, scen_id, const_cast<void *>(state), nullptr);
    wrsn_make_layout(&P.d, &P.L);
    return P;
}

extern "C" {

int wrsn_build_obs_tables(const wrsn_dims *d, void *scen, void *stream) {
    if (check_dims(d)) return -1;
    if (!scen) WRSN_FAIL("scen is NULL");
    KParams P = aux_params(d, scen, nullptr, nullptr);
    return launch_obs_tables(P, stream);
}

int wrsn_observe(const wrsn_dims *d, const void *scen, const int32_t *scen_id, const void *state,
                 const int32_t *agent_id, void *obs, int obs_f64, void *stream) {
    if (check_dims(d)) return -1;
    if (!agent_id || !obs || !scen || !scen_id || !state) WRSN_FAIL("NULL argument");
    KParams P = aux_params(d, scen, scen_id, state);
    return launch_observe(P, agent_id, obs, obs_f64, stream);
}

int wrsn_decode_density_map(const wrsn_dims *d, const void *scen, const int32_t *scen_id, const void *state,
                            const int32_t *agent_id, const void *dmap, int dmap_f64, double *action_out, void *stream) {
    if (check_dims(d)) return -1;
    if (!agent_id || !dmap || !action_out || !scen || !scen_id || !state) WRSN_FAIL("NULL argument");
    if (check_decode_size(d)) return -1;
    KParams P = aux_params(d, scen, scen_id, state);
    return launch_decode(P, agent_id, dmap, dmap_f64, 0, nullptr, action_out, stream);
}

int wrsn_decode_linear_controller(const wrsn_dims *d, const void *scen, const int32_t *scen_id, const void *state,
                                  const int32_t *agent_id, const float *obs, int channels, const float *weights,
                                  double *action_out, void *stream) {
    if (check_dims(d)) return -1;
    if (!agent_id || !obs || !weights || !action_out || !scen || !scen_id || !state) WRSN_FAIL("NULL argument");
    if (channels < 1 || channels > 8) WRSN_FAIL("1 to 8 channels");
    if (check_decode_size(d)) return -1;
    KParams P = aux_params(d, scen, scen_id, state);
    return launch_decode(P, agent_id, obs, 0, channels, weights, action_out, stream);
}

int wrsn_k_charge(const wrsn_dims *d, const void *scen, const int32_t *scen_id, const void *state, const uint8_t *charging,
                  double *node_rate, double *mc_rate, void *stream) {
    if (check_dims(d)) return -1;
    if (!scen || !scen_id || !state || !node_rate || !mc_rate) WRSN_FAIL("NULL argument");
    if (d->M <= 0) WRSN_FAIL("no chargers");
    KParams P = aux_params(d, scen, scen_id, state);
    return launch_charge(P, charging, node_rate, mc_rate, stream);
}

}  /* extern "C" */
