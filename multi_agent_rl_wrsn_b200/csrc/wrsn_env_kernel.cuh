/* wrsn_env_kernel.cuh — one environment for one launch (env_run) and the one-CTA-per-environment kernel around it; included
 * once per group-size specialisation (see wrsn_engine.cuh), inside the same namespace, and once by the host emulation, whose
 * launcher calls env_run row by row on one lane. */
#ifndef WRSN_GANY_MINB
#define WRSN_GANY_MINB 2                            /* CTAs per SM the multi-warp build is compiled for: 128 registers (a few hundred bytes of spills)
                                                       instead of 238 — 1000 nodes / 10 chargers 0.046 -> 0.074 M decisions/s, 500 / 5 0.269 -> 0.340 M */
#endif
#ifndef WRSN_G32_MINB
#define WRSN_G32_MINB 16                            /* CTAs per SM the one-warp build is compiled for (128 registers; measured: 18 CTAs at 96 registers
                                                       and 0.7 KB of spills is 3 % slower, shared memory allows no more than 18) */
#endif

/* bytes: a multiple of 16 */
WRSN_DI void copy16(char *dst, const char *src, int64_t bytes, int tid, int G) {
#if defined(WRSN_HOST_EMU)
    (void)tid; (void)G;
    memcpy(dst, src, (size_t)bytes);
#else
    const uint4 *s = reinterpret_cast<const uint4 *>(src);
    uint4 *d = reinterpret_cast<uint4 *>(dst);
    const int n = (int)(bytes >> 4);
    for (int i = tid; i < n; i += G) d[i] = s[i];
#endif
}

WRSN_DI void zero16(char *dst, int64_t bytes, int tid, int G) {
#if defined(WRSN_HOST_EMU)
    (void)tid; (void)G;
    memset(dst, 0, (size_t)bytes);
#else
    uint4 *z = reinterpret_cast<uint4 *>(dst);
    for (int i = tid; i < (int)(bytes >> 4); i += G) z[i] = make_uint4(0u, 0u, 0u, 0u);
#endif
}

WRSN_DI void write_request(const wrsn_request &q, int b, const ReqOut &r) {
    if (q.agent_id) q.agent_id[b] = r.agent;
    if (q.terminal) q.terminal[b] = (uint8_t)r.terminal;
    if (q.reward) q.reward[b] = r.reward;
    if (q.now) q.now[b] = r.now;
    if (q.action) for (int k = 0; k < 3; k++) q.action[3 * b + k] = r.act[k];
    if (q.detail) { q.detail[2 * b] = r.detail[0]; q.detail[2 * b + 1] = r.detail[1]; }
    if (q.flags) q.flags[b] = r.flags;
    if (q.sticky && r.flags) q.sticky[b] |= r.flags;
}

/* Row `blk` of the launch (the CTA index; MODE_STEP maps it through P.order) on threads tid = 0 .. G-1: select the row, load its
 * image into shared memory, run the mode's entry point, write the image back and, for the modes that hand out a request, the
 * request record and the running totals. */
template <int MODE>
WRSN_DI void env_run(const KParams &P, int blk, int tid, int G) {
    char *smem = WRSN_SMEM_BASE;
    const int b = (MODE == MODE_STEP && P.order) ? P.order[blk] : blk;
    if (P.mask && !P.mask[b]) return;
    if (P.mask_mode == 1 && P.req.agent_id[b] < 0 && P.req.agent_id[b] != -4) return;     /* (-4: a step in flight continues) */
    if (P.mask_mode == 2 && (P.req.agent_id[b] >= 0 || P.req.agent_id[b] == -4)) return;
    if (P.resume_only && P.req.agent_id[b] != -4) return;
    char *row = P.state + (size_t)b * P.L.total;
    const bool split = P.d.step_budget > 0 && P.d.step_rounds > 0;
    if (MODE == MODE_STEP && split && P.req.agent_id && P.req.agent_id[b] == -4 &&
        reinterpret_cast<const double *>(row + P.L.off[WRSN_F_HDR])[WRSN_H_INFLIGHT] == 2.0) return;   /* waits for the batch kernel */
    if (MODE == MODE_STEP_BATCH && (P.req.agent_id[b] != -4 ||
        reinterpret_cast<const double *>(row + P.L.off[WRSN_F_HDR])[WRSN_H_INFLIGHT] != 2.0)) return;
    const char *scen_row = P.scen + (size_t)P.scen_id[b] * P.L.scen_total;
    Ctx c;
    ctx_bind(c, P.d, P.L, scen_row, row, tid, G);
    if (MODE == MODE_RESTORE_RESET) {
        const char *src = P.snap + (size_t)P.scen_id[b] * P.L.total;
        copy16(row + P.L.resident, src + P.L.resident, P.L.total - P.L.resident, tid, G);
        copy16(smem, src, P.L.resident, tid, G);
    } else if (MODE != MODE_INIT) {
        copy16(smem, row, P.L.resident, tid, G);
    } else {                                         /* alignment gaps between the fields: defined bytes in the record */
        zero16(smem, P.L.resident, tid, G);
    }
    for (int i = tid; i < c.Npad; i += G) c.own[i] = i < c.N ? (uint16_t)(c.tgt_ptr[i + 1] - c.tgt_ptr[i]) : (uint16_t)0;
    gsync(c);

    const double now_before = c.hdr[WRSN_H_NOW];
#if defined(WRSN_PROF) && !defined(WRSN_HOST_EMU)
    const long long prof_start = clock64();
    if (MODE == MODE_STEP) { gsync(c); if (tid == 0) for (int q = WRSN_H_PROF0; q <= WRSN_H_PROF4; q++) c.hdr[q] = 0.0; gsync(c); }
#endif
    ReqOut r;
    r.agent = -3; r.terminal = 0; r.reward = 0; r.now = 0; r.flags = 0;
    r.act[0] = r.act[1] = r.act[2] = 0; r.detail[0] = r.detail[1] = 0;
    switch (MODE) {
    case MODE_INIT: entry_init_network(c, P.with_reward); break;
    case MODE_RUN_UNTIL: entry_run_until(c, P.t_until[b]); break;
    case MODE_RESET_FINISH:
    case MODE_RESTORE_RESET: entry_reset_finish(c, &r); break;
    case MODE_STEP: entry_step(c, P.agent_in ? P.agent_in[b] : -1, P.action_in ? P.action_in + 3 * (size_t)b : nullptr, &r, P.d.step_budget, split ? 1 : 0); break;
    case MODE_STEP_BATCH: entry_batches(c, &r, P.d.step_budget); break;
    case MODE_FITNESS: {
        double mn = do_fitness(c, P.fitness ? P.fitness + (size_t)b * P.d.T : nullptr);
        if (tid == 0 && P.fit_min) P.fit_min[b] = mn;
        break;
    }
    case MODE_K_BFS: do_bfs(c); break;
    case MODE_K_DRAIN: ev_nodes_drain(c); break;
    case MODE_K_BOOK: ev_nodes_book(c); break;
    case MODE_K_REWARD: ev_update_reward(c); break;
    }
    gsync(c);
#if defined(WRSN_PROF) && !defined(WRSN_HOST_EMU)
    if (MODE == MODE_STEP) { if (tid == 0) c.hdr[WRSN_H_PROF0] = (double)(clock64() - prof_start); gsync(c); }
#endif
    if (MODE != MODE_FITNESS) copy16(row, smem, P.L.resident, tid, G);
    if ((MODE == MODE_RESET_FINISH || MODE == MODE_RESTORE_RESET || MODE == MODE_STEP || MODE == MODE_STEP_BATCH) && tid == 0) {
        write_request(P.req, b, r);
        if (P.req.stats) {
            if (r.agent >= 0) P.req.stats[3 * b] += 1.0;
            if (MODE == MODE_STEP || MODE == MODE_STEP_BATCH) P.req.stats[3 * b + 1] += r.now - now_before;
            if (MODE == MODE_RESTORE_RESET || MODE == MODE_RESET_FINISH) P.req.stats[3 * b + 2] += 1.0;
        }
    }
}

#if !defined(WRSN_HOST_EMU)
template <int MODE>
__global__ void __launch_bounds__(WRSN_GFIX ? WRSN_GFIX : 256, WRSN_GFIX ? WRSN_G32_MINB : WRSN_GANY_MINB) k_env(const KParams P) {
    env_run<MODE>(P, (int)blockIdx.x, threadIdx.x, blockDim.x);
}
#endif
