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

/* The rule's node for charger a (wrsn_layout.h: heur_charger, heur_key, HeurPick) over the row's shared-memory image, on every
 * thread of the group: threads stride the nodes, then the group reduces — a shuffle butterfly in the one-warp build, across warps
 * through c.red in the other; one lane runs the plain loop in the host emulation.  Every comparison is the total order on
 * (key, id), so the thread count does not change the choice.  Returns the node (-1: none alive), the same in every thread. */
WRSN_DI int roll_pick(Ctx &c, const WrsnRow &rw, HeurFleet &f, int kind, int a) {
    gsync(c);                                        /* f and c.red: the previous users are done */
    if (c.tid < c.M) heur_charger(rw, a, c.tid, &f);
#if defined(WRSN_HOST_EMU)
    for (int j = 1; j < c.M; j++) heur_charger(rw, a, j, &f);
#endif
    if (c.tid == 0) f.M = c.M;
    gsync(c);
    int pick = -1;
    for (int pass = 0; pass < 2 && pick < 0; pass++) {
        HeurPick p;
        for (int i = c.tid; i < rw.N; i += WRSN_GSZ(c)) {
            double key[2] = {0.0, 0.0};
            p.add(heur_key(rw, f, kind, i, pass, key), key, i);
        }
#if !defined(WRSN_HOST_EMU)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
#pragma unroll
            for (int s = 0; s < 2; s++) {
                const double k = __shfl_xor_sync(0xffffffffu, p.k[s], o);
                const int id = __shfl_xor_sync(0xffffffffu, p.i[s], o);
                p.take(s, k, id);
            }
#if WRSN_GFIX != 32
        double *rk = c.red;                          /* [warp][2] keys, then [warp][2] ids */
        int *ri = reinterpret_cast<int *>(rk + 16);
        if ((c.tid & 31) == 0)
            for (int s = 0; s < 2; s++) { rk[2 * (c.tid >> 5) + s] = p.k[s]; ri[2 * (c.tid >> 5) + s] = p.i[s]; }
        gsync(c);
        for (int w = 0; w < (c.G >> 5); w++)
            for (int s = 0; s < 2; s++) p.take(s, rk[2 * w + s], ri[2 * w + s]);
        gsync(c);
#endif
#endif
        pick = p.choice();
    }
    return pick;
}

/* MODE_RULE_ROLLOUT (include/wrsn_b200.h: wrsn_rule_rollout): row b's requests, one after the other in the loaded image, with
 * controllers.evaluate's accounting (batched.py: episode_ends, episode_step).  All threads run the loop; thread 0 alone writes
 * the row's running totals.  The launch's step budget is shared by its steps. */
WRSN_DI void roll_row(Ctx &c, const KParams &P, const RollArgs &R, const WrsnRow &rw, int b) {
#if defined(WRSN_HOST_EMU)
    HeurFleet f;
#else
    __shared__ HeurFleet f;
#endif
    const int64_t limit = R.limit;
    int agent = P.req.agent_id[b];
    int64_t dec = R.decisions[b];
    const int64_t dec0 = dec;
    double ret = R.returns[b];
    int budget = P.d.step_budget, handed = 0;
    bool stepped = false, running = true;
    ReqOut r;
    for (;;) {
        if (agent == -1 || (agent != -4 && dec >= limit)) { running = false; break; }    /* the episode ends here */
        if ((agent >= 0 && handed >= R.launch_max) || (P.d.step_budget > 0 && budget <= 0)) break;
        double act[3] = {0.0, 0.0, 0.0};
        if (agent >= 0 && agent < c.M) {
            if (R.first && dec == 0) {
                for (int k = 0; k < 3; k++) act[k] = R.first[3 * (size_t)b + k];
            } else {
                const int node = roll_pick(c, rw, f, R.kind, agent);
                heur_action(rw, agent, node, act);
            }
        }
        const double now_before = c.hdr[WRSN_H_NOW];
        gsync(c);
        int work = 0;
        entry_step(c, agent >= 0 ? agent : -1, act, &r, P.d.step_budget > 0 ? budget : 0, 0, &work);
        budget -= work;
        stepped = true;
        if (agent >= 0) { dec++; handed++; }
        if (c.tid == 0) {
            const double x = r.reward;               /* torch.nan_to_num(x, nan=0.0): NaN -> 0, +-inf -> +-DBL_MAX */
            ret += x != x ? 0.0 : (x == (double)INFINITY ? DBL_MAX : (x == -(double)INFINITY ? -DBL_MAX : x));
            if (P.req.stats) {
                if (r.agent >= 0) P.req.stats[3 * b] += 1.0;
                P.req.stats[3 * b + 1] += r.now - now_before;
            }
            if (P.req.sticky && r.flags) P.req.sticky[b] |= r.flags;
            c.bcast[0] = r.agent;
        }
        gsync(c);
        agent = c.bcast[0];
        gsync(c);
        if (agent == -4) break;                      /* in flight: the next launch continues it */
    }
    if (c.tid == 0) {
        if (stepped) write_request(P.req, b, r);
        if (dec != dec0) R.decisions[b] = dec;
        if (stepped) R.returns[b] = ret;
        if (!running) R.running[b] = 0;
    }
}

/* Row `blk` of the launch (the CTA index; MODE_STEP maps it through P.order) on threads tid = 0 .. G-1: select the row, load its
 * image into shared memory, run the mode's entry point, write the image back and, for the modes that hand out a request, the
 * request record and the running totals. */
template <int MODE>
WRSN_DI void env_run(const KParams &P, int blk, int tid, int G, const RollArgs &R = RollArgs()) {
    char *smem = WRSN_SMEM_BASE;
    const int b = (MODE == MODE_STEP && P.order) ? P.order[blk] : blk;
    if (P.mask && !P.mask[b]) return;
    if (P.mask_mode == 1 && P.req.agent_id[b] < 0 && P.req.agent_id[b] != -4) return;     /* (-4: a step in flight continues) */
    if (P.mask_mode == 2 && (P.req.agent_id[b] >= 0 || P.req.agent_id[b] == -4)) return;
    if (P.resume_only && P.req.agent_id[b] != -4) return;
    if (MODE == MODE_RULE_ROLLOUT && !R.running[b]) return;
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
    if constexpr (MODE == MODE_RULE_ROLLOUT) roll_row(c, P, R, WrsnRow(P.L, smem, scen_row), b);   /* writes its own request and totals */
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

/* MODE_RULE_ROLLOUT, with its arguments in a parameter of their own */
__global__ void __launch_bounds__(WRSN_GFIX ? WRSN_GFIX : 256, WRSN_GFIX ? WRSN_G32_MINB : WRSN_GANY_MINB) k_env_roll(const KParams P, const RollArgs R) {
    env_run<MODE_RULE_ROLLOUT>(P, (int)blockIdx.x, threadIdx.x, blockDim.x, R);
}
#endif
