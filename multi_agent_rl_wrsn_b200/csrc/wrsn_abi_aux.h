/*
 * wrsn_abi_aux.h — the entry points of the C ABI (include/wrsn_b200.h) outside the environment kernel: the observation raster,
 * the density-map decoder, the charging model, the heuristic charging rules and the raster's scenario tables.  The CUDA library (wrsn_kernels.cu) and the
 * tests' host emulation (tests/emu/wrsn_emu.cpp) share their argument checks and KParams; included once, after
 * wrsn_abi_host.h, and the including file supplies the work on checked arguments:
 *   launch_obs_tables(P, stream)                                  wrsn_build_obs_tables;
 *   launch_observe(P, agent_id, obs, obs_f64, stream)             wrsn_observe;
 *   launch_decode(P, agent_id, dmap, dmap_f64, channels, weights, action_out, stream)
 *                                                                 both decode entry points (channels = 0: dmap is the map);
 *   launch_charge(P, charging, node_rate, mc_rate, stream)        wrsn_k_charge;
 *   launch_heuristic(P, agent_id, kind, action, stream)           wrsn_heuristic_action;
 *   launch_candidates(P, agent_id, kind, K, action, node, stream) wrsn_heuristic_candidates (these two in the CUDA library
 *                                                                 only: the host emulation's row-by-row loops are defined below).
 *   launch_roll(P, R, stream)                                     wrsn_rule_rollout: env_run<MODE_RULE_ROLLOUT> with its
 *                                                                 arguments R (the CUDA library's k_env_roll; the host
 *                                                                 emulation's row-by-row loop is defined below as well).
 */
#pragma once
#include "wrsn_abi_host.h"
#if defined(WRSN_HOST_EMU)
#include <vector>
#endif

static int launch_obs_tables(KParams &P, void *stream);
static int launch_observe(KParams &P, const int32_t *agent_id, void *obs, int obs_f64, void *stream);
static int launch_decode(KParams &P, const int32_t *agent_id, const void *dmap, int dmap_f64, int channels, const float *weights,
                         double *action_out, void *stream);
static int launch_charge(KParams &P, const uint8_t *charging, double *node_rate, double *mc_rate, void *stream);
static int launch_heuristic(KParams &P, const int32_t *agent_id, int kind, double *action, void *stream);
static int launch_candidates(KParams &P, const int32_t *agent_id, int kind, int K, double *action, int32_t *node, void *stream);
static int launch_roll(KParams &P, const RollArgs &R, void *stream);

/* once the arguments are checked: the dims and the layout they imply */
#if defined(WRSN_HOST_EMU)
/* the host emulation's wrsn_heuristic_action: k_heuristic's rule (wrsn_layout.h: heur_key, heur_action) row by row and node by
 * node; the minimum of a total order on (key, id) does not depend on the order in which the nodes are seen */
static int launch_heuristic(KParams &P, const int32_t *agent_id, int kind, double *action, void *) {
    for (int b = 0; b < P.d.B; b++) {
        const int a = agent_id[b];
        if (a < 0 || a >= P.d.M) continue;
        const WrsnRow rw(P.L, P.state, P.scen, P.scen_id, b);
        HeurFleet f = HeurFleet();
        f.M = P.d.M;
        for (int j = 0; j < f.M; j++) heur_charger(rw, a, j, &f);
        int pick = -1;
        for (int pass = 0; pass < 2 && pick < 0; pass++) {
            HeurPick p;
            for (int i = 0; i < rw.N; i++) {
                double key[2] = {0.0, 0.0};
                p.add(heur_key(rw, f, kind, i, pass, key), key, i);
            }
            pick = p.choice();
        }
        heur_action(rw, a, pick, action + 3 * (size_t)b);
    }
    return 0;
}

/* the host emulation's wrsn_heuristic_candidates: the K first nodes of the order (wrsn_layout.h: heur_rank, heur_insert), row by
 * row and node by node, pass 1 only when pass 0 has no candidate */
static int launch_candidates(KParams &P, const int32_t *agent_id, int kind, int K, double *action, int32_t *node, void *) {
    for (int b = 0; b < P.d.B; b++) {
        const int a = agent_id[b];
        if (a < 0 || a >= P.d.M) continue;
        const WrsnRow rw(P.L, P.state, P.scen, P.scen_id, b);
        HeurFleet f = HeurFleet();
        f.M = P.d.M;
        for (int j = 0; j < f.M; j++) heur_charger(rw, a, j, &f);
        HeurRank l[WRSN_CAND_MAX];
        int n = 0;
        for (int pass = 0; pass < 2 && n == 0; pass++)
            for (int i = 0; i < rw.N; i++) {
                HeurRank r;
                if (heur_rank(rw, f, kind, i, pass, &r)) heur_insert(l, 1, n, K, r);
            }
        for (int k = 0; k < K; k++)
            heur_slot(rw, a, k < n ? l[k].id : -1, n ? l[0].id : -1, action + 3 * ((size_t)b * K + k), node + (size_t)b * K + k);
    }
    return 0;
}

/* the host emulation's wrsn_rule_rollout: env_run<MODE_RULE_ROLLOUT> row by row on one lane, as its launch_env runs every mode */
static int launch_roll(KParams &P, const RollArgs &R, void *) {
    if (prepare_launch(P)) return -1;
    std::vector<char> smem((size_t)P.L.smem_total + 64);
    wrsn_smem_host = smem.data();
    for (int b = 0; b < P.d.B; b++) env_run<MODE_RULE_ROLLOUT>(P, b, 0, 1, R);
    return 0;
}
#endif

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

int wrsn_heuristic_action(const wrsn_dims *d, const void *scen, const int32_t *scen_id, const void *state,
                          const int32_t *agent_id, int kind, double *action, void *stream) {
    if (check_dims(d)) return -1;
    if (!agent_id || !action || !scen || !scen_id || !state) WRSN_FAIL("NULL argument");
    if (kind < 0 || kind >= WRSN_HEUR_COUNT) WRSN_FAIL("heuristic kind %d: 0 (min_lifetime) or 1 (nearest_urgent)", kind);
    KParams P = aux_params(d, scen, scen_id, state);
    return launch_heuristic(P, agent_id, kind, action, stream);
}

int wrsn_heuristic_candidates(const wrsn_dims *d, const void *scen, const int32_t *scen_id, const void *state,
                              const int32_t *agent_id, int kind, int K, double *action, int32_t *node, void *stream) {
    if (check_dims(d)) return -1;
    if (!agent_id || !action || !node || !scen || !scen_id || !state) WRSN_FAIL("NULL argument");
    if (kind < 0 || kind >= WRSN_HEUR_COUNT) WRSN_FAIL("heuristic kind %d: 0 (min_lifetime) or 1 (nearest_urgent)", kind);
    if (K < 1 || K > WRSN_CAND_MAX) WRSN_FAIL("K = %d candidates: 1 to %d", K, WRSN_CAND_MAX);
    KParams P = aux_params(d, scen, scen_id, state);
    return launch_candidates(P, agent_id, kind, K, action, node, stream);
}

int wrsn_rule_rollout(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state, uint8_t *running, int kind,
                      const double *first_action, int64_t limit, int32_t launch_max, int64_t *decisions, double *returns,
                      wrsn_request *req, void *stream) {
    if (check_dims(d)) return -1;
    if (!scen || !scen_id || !state || !running || !decisions || !returns || !req || !req->agent_id) WRSN_FAIL("NULL argument");
    if (kind < 0 || kind >= WRSN_HEUR_COUNT) WRSN_FAIL("heuristic kind %d: 0 (min_lifetime) or 1 (nearest_urgent)", kind);
    if (limit < 0) WRSN_FAIL("limit = %lld decisions: must not be negative", (long long)limit);
    if (launch_max < 1 || launch_max > WRSN_ROLL_MAX) WRSN_FAIL("launch_max = %d decisions: 1 to %d", (int)launch_max, WRSN_ROLL_MAX);
    KParams P = base_params(d, scen, scen_id, state, nullptr);
    P.req = *req;
    RollArgs R;
    R.running = running; R.decisions = decisions; R.returns = returns; R.first = first_action;
    R.limit = limit; R.kind = kind; R.launch_max = launch_max;
    return launch_roll(P, R, stream);
}

}  /* extern "C" */
