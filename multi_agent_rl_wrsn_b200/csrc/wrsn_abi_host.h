/*
 * wrsn_abi_host.h — the host side of the C ABI (include/wrsn_b200.h) that the CUDA library (wrsn_kernels.cu) and the tests'
 * host emulation (tests/emu/wrsn_emu.cpp) share: errors, dims, layouts and every entry point that only fills KParams and
 * launches the environment kernel.  Included once, after the kernels; the including file supplies
 *   launch_env<MODE>(P, stream)   one launch of env_run<MODE> (wrsn_env_kernel.cuh) over the rows of the batch;
 *   order_rows(P, stream)         before a step: the order in which the launch takes the rows (P.order; NULL = index order);
 * and the CUDA build the kernels k_record_transitions and k_copy_rows.  The entry points of the raster, the decoder and the charging model:
 * wrsn_abi_aux.h.
 */
#pragma once
#include <stdio.h>

#include "wrsn_launch.h"

static thread_local char g_err[512] = "";
#define WRSN_FAIL(...) do { snprintf(g_err, sizeof(g_err), __VA_ARGS__); return -1; } while (0)

template <int MODE> static int launch_env(KParams &P, void *stream);
static int order_rows(KParams &P, void *stream);

static int check_dims(const wrsn_dims *d) {
    if (!d) WRSN_FAIL("dims is NULL");
    if (d->N <= 0 || d->N > 32000 || d->T < 0 || d->T > 65000 || d->M < 0 || d->M > WRSN_MAX_MC || d->B <= 0 || d->S <= 0)
        WRSN_FAIL("bad dims N=%d T=%d M=%d B=%d S=%d", d->N, d->T, d->M, d->B, d->S);
    if (d->Npad < d->N || (d->Npad & 15) || d->state_bytes <= 0) WRSN_FAIL("dims not finalized (call wrsn_dims_finalize)");
    /* the register-resident per-node loops hold at most 4 (one warp) / 9 (several warps) nodes per thread */
    if (d->threads < 32 || d->threads % 32 || d->threads > 256 || (int64_t)d->N > (int64_t)d->threads * (d->threads == 32 ? 4 : 9))
        WRSN_FAIL("threads = %d cannot hold N = %d nodes (at most %d per thread)", d->threads, d->N, d->threads == 32 ? 4 : 9);
    if (d->step_rounds < 0) WRSN_FAIL("step_rounds = %d: 0 (one launch per step) or the number of rounds of a split step", d->step_rounds);
    return 0;
}

/* The density-map decoder (k_decode_map) keeps the WRSN_DEC_MAX_RANK largest values of a map: np.percentile(., 99.9) needs the
 * R-th largest, R = n - floor(0.999 n - 0.999) with n = S * S (the kernel's own expression), so maps up to 176 x 176 (R = 32).
 * A larger map is refused here instead of being ranked wrongly. */
#define WRSN_DEC_MAX_RANK 32
static int wrsn_decode_rank(int S) {
    const int n = S * S;
    const double qf = 99.9 / 100.0;
    const double vidx = (double)n * qf + (1.0 + qf * (1.0 - 1.0 - 1.0)) - 1.0;
    return n - (int)floor(vidx);
}
static int check_decode_size(const wrsn_dims *d) {
    if (d->S > 46340 || wrsn_decode_rank(d->S) > WRSN_DEC_MAX_RANK) {
        int smax = 1;
        while (wrsn_decode_rank(smax + 1) <= WRSN_DEC_MAX_RANK) smax++;
        WRSN_FAIL("map_size = %d: the density-map decoder supports map sizes up to %d (np.percentile(., 99.9) of a larger map "
                  "needs more than the %d largest values it keeps)", d->S, smax, WRSN_DEC_MAX_RANK);
    }
    return 0;
}

/* every launch of the environment kernel: valid dims, the layout they imply, the buffers every mode reads */
static int prepare_launch(KParams &P) {
    if (check_dims(&P.d)) return -1;
    wrsn_make_layout(&P.d, &P.L);
    if (!P.scen || !P.scen_id || !P.state) WRSN_FAIL("scen / scen_id / state must not be NULL");
    return 0;
}

static KParams base_params(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state, const uint8_t *mask) {
    KParams P;
    memset(&P, 0, sizeof(P));
    if (d) P.d = *d;
    P.scen = (const char *)scen; P.scen_id = scen_id; P.state = (char *)state; P.mask = mask;
    return P;
}

/* WRSN.step: one launch of the whole engine, or — wrsn_dims.step_rounds > 0 with a step budget — rounds of two launches, the
 * events kernel and the batch kernel (see include/wrsn_b200.h).  In the later launches a row is selected by its own state
 * (request record -4 + hdr[INFLIGHT]); rows that finished their step stay out. */
static int launch_step(KParams &P, void *stream) {
    if (order_rows(P, stream)) return -1;
    if (!(P.d.step_budget > 0 && P.d.step_rounds > 0)) return launch_env<MODE_STEP>(P, stream);
    if (!P.req.agent_id) WRSN_FAIL("split steps need req->agent_id");
    for (int r = 0; r < P.d.step_rounds; r++) {
        if (launch_env<MODE_STEP>(P, stream)) return -1;
        KParams Q = P;
        Q.agent_in = nullptr; Q.action_in = nullptr;
        if (launch_env<MODE_STEP_BATCH>(Q, stream)) return -1;
        P.resume_only = 1;                           /* later rounds: only rows still in flight (the others hold a fresh request) */
    }
    return 0;
}

extern "C" {

const char *wrsn_last_error(void) { return g_err; }
int wrsn_abi_version(void) { return WRSN_ABI_VERSION; }
int wrsn_field_count(int which) {
    switch (which) {
    case 0: return WRSN_P_LEN; case 1: return WRSN_H_LEN; case 2: return WRSN_MC_LEN; case 3: return WRSN_PR_LEN;
    case 4: return WRSN_F_COUNT; case 5: return WRSN_S_COUNT; default: return -1;
    }
}

int wrsn_dims_finalize(wrsn_dims *d) {
    if (!d) WRSN_FAIL("dims is NULL");
    d->Npad = (d->N + 15) & ~15;
    d->W = (d->N + 31) / 32;
    d->Tw = (d->T + 31) / 32; if (d->Tw < 1) d->Tw = 1;
    d->n_slot = d->M + 3;
    if (d->Emax < 1) d->Emax = 1;
    if (d->TEmax < 1) d->TEmax = 1;
    if (d->threads <= 0) {
        int per = (d->N + 3) / 4;                    /* about four nodes per thread: 100 nodes run on ONE warp (measured on the
                                                        RandomController workload: 1.08 M decisions/s against 0.88 M on two
                                                        warps — no block-wide barriers, no shared-memory reductions, and the
                                                        per-second loops keep four independent chains per lane in flight) */
        int t = 32; while (t < per && t < 128) t *= 2;    /* above 128 nodes: at most four warps, then up to nine nodes per thread
                                                        (measured, RandomController law, 2 CTAs per SM: 1000 nodes 0.079 M decisions/s on
                                                        128 threads against 0.074 M on 256; 500 nodes 0.340 M on 128 against 0.287 M on 64) */
        if (d->N > 9 * t) t = 256;
        d->threads = t;
    }
    if (d->threads % 32 || d->threads > 256) WRSN_FAIL("threads must be a multiple of 32, at most 256");
    if ((int64_t)d->N > (int64_t)d->threads * (d->threads == 32 ? 4 : 9))
        WRSN_FAIL("threads = %d cannot hold N = %d nodes (at most %d per thread)", d->threads, d->N, d->threads == 32 ? 4 : 9);
    d->obs_pitch = wrsn_obs_pitch(d->S);
    WrsnLayout L;
    wrsn_make_layout(d, &L);
    d->state_bytes = (int32_t)L.total; d->state_resident_bytes = (int32_t)L.resident;
    d->scen_bytes = (int32_t)L.scen_total; d->smem_bytes = (int32_t)L.smem_total;
    if (L.smem_total > 227 * 1024) WRSN_FAIL("environment does not fit shared memory (%lld bytes)", (long long)L.smem_total);
    return 0;
}

int wrsn_state_layout(const wrsn_dims *d, int64_t *offsets) {
    if (check_dims(d)) return -1;
    WrsnLayout L; wrsn_make_layout(d, &L);
    for (int k = 0; k < WRSN_F_COUNT; k++) offsets[k] = L.off[k];
    return 0;
}
int wrsn_scen_layout(const wrsn_dims *d, int64_t *offsets) {
    if (check_dims(d)) return -1;
    WrsnLayout L; wrsn_make_layout(d, &L);
    for (int k = 0; k < WRSN_S_COUNT; k++) offsets[k] = L.soff[k];
    return 0;
}

int wrsn_init_network(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state,
                      const uint8_t *env_mask, int with_reward_process, void *stream) {
    KParams P = base_params(d, scen, scen_id, state, env_mask);
    P.with_reward = with_reward_process;
    return launch_env<MODE_INIT>(P, stream);
}

int wrsn_run_until(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state,
                   const uint8_t *env_mask, const double *t_until, void *stream) {
    if (!t_until) WRSN_FAIL("t_until is NULL");
    KParams P = base_params(d, scen, scen_id, state, env_mask);
    P.t_until = t_until;
    return launch_env<MODE_RUN_UNTIL>(P, stream);
}

int wrsn_reset_finish(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state,
                      const uint8_t *env_mask, wrsn_request *req, void *stream) {
    if (!req) WRSN_FAIL("req is NULL");
    KParams P = base_params(d, scen, scen_id, state, env_mask);
    P.req = *req;
    return launch_env<MODE_RESET_FINISH>(P, stream);
}

int wrsn_reset_from_snapshot(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state,
                             const void *snap, const uint8_t *env_mask, wrsn_request *req, void *stream) {
    if (!req || !snap) WRSN_FAIL("req / snap is NULL");
    KParams P = base_params(d, scen, scen_id, state, env_mask);
    P.req = *req; P.snap = (const char *)snap;
    return launch_env<MODE_RESTORE_RESET>(P, stream);
}

int wrsn_step(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state,
              const uint8_t *env_mask, const int32_t *agent_id_in, const double *action_in,
              wrsn_request *req, void *stream) {
    if (!req) WRSN_FAIL("req is NULL");
    if (agent_id_in && !action_in) WRSN_FAIL("action_in is NULL");
    KParams P = base_params(d, scen, scen_id, state, env_mask);
    P.agent_in = agent_id_in; P.action_in = action_in; P.req = *req;
    return launch_step(P, stream);
}

int wrsn_rollout_step(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state, const void *snap,
                      const double *action_in, wrsn_request *req, void *obs, int obs_f64, void *stream) {
    if (!req || !req->agent_id || !snap || !action_in) WRSN_FAIL("req / req->agent_id / snap / action_in is NULL");
    KParams P = base_params(d, scen, scen_id, state, nullptr);
    P.req = *req; P.agent_in = req->agent_id; P.action_in = action_in; P.mask_mode = 1;
    if (launch_step(P, stream)) return -1;
    KParams R = base_params(d, scen, scen_id, state, nullptr);
    R.req = *req; R.snap = (const char *)snap; R.mask_mode = 2;
    if (launch_env<MODE_RESTORE_RESET>(R, stream)) return -1;
    if (obs) return wrsn_observe(d, scen, scen_id, state, req->agent_id, obs, obs_f64, stream);
    return 0;
}

int wrsn_record_transitions(const wrsn_dims *d, const wrsn_request *req, int64_t t, const int64_t *agent_prev,
                            int64_t *last, double *resets_seen, int64_t *agent_next, int64_t *link_next,
                            uint8_t *new_episode_next, double *reward_next, double *now_next, void *stream) {
    if (!d || !req || !req->agent_id || !req->reward || !req->now || !req->stats) WRSN_FAIL("req / its agent_id, reward, now or stats is NULL");
    if (!agent_prev || !last || !resets_seen || !agent_next || !link_next || !new_episode_next || !reward_next || !now_next)
        WRSN_FAIL("a record pointer is NULL");
    if (d->B <= 0 || d->M <= 0) WRSN_FAIL("bad dims");
#if defined(WRSN_HOST_EMU)
    (void)stream;
    for (int b = 0; b < d->B; b++)
        record_transition(b, d->M, *req, t, agent_prev, last, resets_seen, agent_next, link_next, new_episode_next, reward_next, now_next);
#else
    k_record_transitions<<<(d->B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
        d->B, d->M, *req, t, agent_prev, last, resets_seen, agent_next, link_next, new_episode_next, reward_next, now_next);
    WRSN_CUDA(cudaGetLastError());
#endif
    return 0;
}

int wrsn_copy_rows(const wrsn_dims *d, int32_t n,
                   const void *src_state, const wrsn_request *src_req, const int32_t *src_scen_id, const int32_t *src_rows, int32_t src_B,
                   void *dst_state, const wrsn_request *dst_req, int32_t *dst_scen_id, const int32_t *dst_rows, int32_t dst_B,
                   void *stream) {
    if (check_dims(d)) return -1;
    if (n < 0) WRSN_FAIL("n = %d: the number of rows to copy must not be negative", n);
    if (src_B <= 0 || dst_B <= 0) WRSN_FAIL("src_B = %d, dst_B = %d: both must be positive", src_B, dst_B);
    if (!src_state || !dst_state || !src_rows || !dst_rows || !src_scen_id || !dst_scen_id)
        WRSN_FAIL("a state, row list or scen_id is NULL");
    if (!src_req || !dst_req) WRSN_FAIL("src_req / dst_req is NULL");
    for (int side = 0; side < 2; side++) {
        const wrsn_request *q = side ? dst_req : src_req;
        if (!q->agent_id || !q->terminal || !q->reward || !q->now || !q->action || !q->detail || !q->flags)
            WRSN_FAIL("%s: agent_id, terminal, reward, now, action, detail and flags must not be NULL", side ? "dst_req" : "src_req");
    }
    if (n == 0) return 0;
#if defined(WRSN_HOST_EMU)
    (void)stream;
    for (int i = 0; i < n; i++) {
        const int s = src_rows[i], o = dst_rows[i];
        if (s < 0 || s >= src_B || o < 0 || o >= dst_B) continue;
        memcpy((char *)dst_state + (size_t)o * d->state_bytes, (const char *)src_state + (size_t)s * d->state_bytes, (size_t)d->state_bytes);
        copy_row_request(*src_req, src_scen_id, s, *dst_req, dst_scen_id, o);
    }
#else
    k_copy_rows<<<n, COPY_THREADS, 0, (cudaStream_t)stream>>>(d->state_bytes, (const char *)src_state, *src_req, src_scen_id, src_rows, src_B,
                                                              (char *)dst_state, *dst_req, dst_scen_id, dst_rows, dst_B);
    WRSN_CUDA(cudaGetLastError());
#endif
    return 0;
}

int wrsn_fitness(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state,
                 double *fitness, double *fit_min, void *stream) {
    KParams P = base_params(d, scen, scen_id, state, nullptr);
    P.fitness = fitness; P.fit_min = fit_min;
    return launch_env<MODE_FITNESS>(P, stream);
}

int wrsn_k_bfs(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state, void *stream) {
    KParams P = base_params(d, scen, scen_id, state, nullptr);
    return launch_env<MODE_K_BFS>(P, stream);
}
int wrsn_k_drain(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state, void *stream) {
    KParams P = base_params(d, scen, scen_id, state, nullptr);
    return launch_env<MODE_K_DRAIN>(P, stream);
}
int wrsn_k_bookkeep(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state, void *stream) {
    KParams P = base_params(d, scen, scen_id, state, nullptr);
    return launch_env<MODE_K_BOOK>(P, stream);
}
int wrsn_k_reward(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state, void *stream) {
    KParams P = base_params(d, scen, scen_id, state, nullptr);
    return launch_env<MODE_K_REWARD>(P, stream);
}

}  /* extern "C" */
