/*
 * wrsn_b200.h — C ABI of the B200-native batched WRSN simulator (libwrsn_b200.so).
 *
 * The reference has no FFI layer: its boundary for this hot path is the Python class
 * rl_env.WRSN.WRSN (reset rl_env/WRSN.py:41, step :289, get_state :130,
 * get_network_fitness :188, get_reward :222, update_reward :100) over
 * physical_env/{network,mc}.  The entry points below are what a ctypes binding of that
 * class binds instead of running SimPy: plain pointers and sizes, device memory owned by
 * the caller (PyTorch is only the allocator), a CUDA stream handle, int return codes
 * (0 = ok) and wrsn_last_error().  INTEGRATION.md shows the reference-side stub.
 *
 * Memory model.  Two caller-allocated device buffers:
 *   scen  [n_scen][scen_bytes]   static graph + constants of every distinct scenario
 *   state [B][state_bytes]       one contiguous record per environment; inside the record the
 *                                node quantities are struct-of-arrays rows of pitch Npad
 * The byte offsets of every field inside a record come from wrsn_state_layout() /
 * wrsn_scen_layout(), so a host can build typed views without knowing a C struct.
 * Records that only the per-environment leader thread touches (event clock, charger
 * records, charger process slots) are rows of doubles indexed by the enums below.
 */
#ifndef WRSN_B200_H
#define WRSN_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WRSN_ABI_VERSION 20
#define WRSN_MAX_MC 16          /* chargers per environment */
#define WRSN_RING 10            /* Node.operate keeps the last 10 per-second consumptions (Node.py:70-77) */

/* ---- per-scenario scalar row  par[WRSN_P_LEN]  (filled by the host loader with the
 *      reference's own Python arithmetic so thresholds / constants are bit-identical) ---- */
enum {
    WRSN_P_CAP = 0, WRSN_P_THR, WRSN_P_ERECV,          /* node capacity, threshold, er*package_size */
    WRSN_P_BSX, WRSN_P_BSY,
    WRSN_P_F0, WRSN_P_F1, WRSN_P_F2, WRSN_P_F3,        /* Network.frame (Network.py:16-26) */
    WRSN_P_MAXTIME, WRSN_P_WARMUP,
    WRSN_P_MTM, WRSN_P_CTM, WRSN_P_AVGNA,              /* moving_time_max, charging_time_max, avg_nodes_agent (WRSN.py:50-52) */
    WRSN_P_MC_CAP, WRSN_P_MC_THR, WRSN_P_MC_V, WRSN_P_MC_PM, WRSN_P_MC_R, WRSN_P_MC_ALPHA, WRSN_P_MC_BETA,
    WRSN_P_MC_EPS, WRSN_P_MC_AB2,                      /* alpha / beta**2 */
    WRSN_P_MC_CAP200, WRSN_P_MC_PMV,                   /* capacity / 200.0 ; pm * velocity */
    WRSN_P_EPSENV,                                     /* WRSN.epsilon = 1e-9 */
    WRSN_P_CAPMTHR,                                    /* capacity - threshold */
    WRSN_P_ESMAX,                                      /* largest per-hop cost in the scenario (slack of the no-death test) */
    WRSN_P_INVN,                                       /* 1 / number of nodes (mean and variance of update_reward's priorities) */
    WRSN_P_NNODES, WRSN_P_NTARGETS,                    /* this scenario's own node and target counts (at most wrsn_dims.N / T) */
    WRSN_P_LEN = 32
};

/* ---- per-environment event clock  hdr[WRSN_H_LEN] ---- */
enum {
    WRSN_H_NOW = 0, WRSN_H_SEQ,
    WRSN_H_NET_ON, WRSN_H_NET_T, WRSN_H_NET_SEQ, WRSN_H_NET_STATE,  /* Network.operate: 1 next=setLevels, 2 next=exit check */
    WRSN_H_UR_ON, WRSN_H_UR_T, WRSN_H_UR_SEQ,                       /* WRSN.update_reward */
    WRSN_H_NODES_T, WRSN_H_NODES_SEQ, WRSN_H_NODES_PHASE,           /* Node.operate block: 1 next=k+0.5 drain, 2 next=k+1.0 bookkeeping */
    WRSN_H_UNTIL_ON, WRSN_H_UNTIL_T, WRSN_H_UNTIL_SEQ,              /* env.run(until=number) */
    WRSN_H_ALIVE, WRSN_H_BFS_DIRTY, WRSN_H_LOG_LEN, WRSN_H_LOG_HEAD, WRSN_H_LOG_UNIFORM, WRSN_H_LOG_LITERAL,
    WRSN_H_FIT_MIN,                                                 /* min(get_network_fitness()) at the last request */
    WRSN_H_ERR, WRSN_H_HANG,
    WRSN_H_NTICKS, WRSN_H_NEVENTS, WRSN_H_NSLOW, WRSN_H_NBFS, WRSN_H_NDECISIONS,
    WRSN_H_CHAIN_N, WRSN_H_CHAIN_DETACH,                            /* AnyOf chain of WRSN.step (:307-311) */
    WRSN_H_NSTALE,                                                  /* routing-tree rebuilds on stale levels (after Network.operate stopped) */
    WRSN_H_NLAZY,                                                   /* charger spans replayed lazily (slot_ff) */
    WRSN_H_NBATCH,                                                  /* simulated seconds advanced by whole-cycle batches (nodes_batch) */
    WRSN_H_OPT_NOBATCH,                                             /* TEST SWITCH: 1 disables the batches (every second runs event by event) and the split
                                                                       death tick in pieces; 2 disables only the latter (plain serial death ticks) */
    WRSN_H_PROF0, WRSN_H_PROF1, WRSN_H_PROF2, WRSN_H_PROF3, WRSN_H_PROF4, /* SM cycles of the last launch (builds with -DWRSN_PROF only):
                                                                       total, serial ticks, batches, BFS + tree, fitness */
    WRSN_H_NSPLIT,                                                  /* death ticks handled in pieces (drain_pieces: closed form around the death packet) */
    WRSN_H_INFLIGHT,                                                /* WRSN.step ran out of its launch budget (wrsn_dims.step_budget) and continues at the next call:
                                                                       1 in the events kernel, 2 in the batch kernel (wrsn_dims.step_rounds) */
    WRSN_H_NRESUME,                                                 /* how often that happened */
    WRSN_H_NOBATCH_ONCE,                                            /* split steps: the batch kernel handed the pending second back to the events kernel */
    WRSN_H_CHAIN_SLOT = 48,                                         /* [WRSN_MAX_MC] process slot watched by member j */
    WRSN_H_COND_TRIG = WRSN_H_CHAIN_SLOT + WRSN_MAX_MC,
    WRSN_H_COND_T = WRSN_H_COND_TRIG + WRSN_MAX_MC,                 /* time of the pending condition event, +inf when none */
    WRSN_H_COND_KEY = WRSN_H_COND_T + WRSN_MAX_MC,                  /* 2^40 + insertion counter */
    WRSN_H_LEN = WRSN_H_COND_KEY + WRSN_MAX_MC                      /* 112 */
};

/* ---- charger record  mc[M][WRSN_MC_LEN]  (MobileCharger.py:6-32 + WRSN per-agent lists) ---- */
enum {
    WRSN_MC_X = 0, WRSN_MC_Y, WRSN_MC_ENERGY, WRSN_MC_STATUS,
    WRSN_MC_CPA0, WRSN_MC_CPA1, WRSN_MC_CPA2,          /* cur_phy_action */
    WRSN_MC_TYPE,                                      /* 0 "moving", 1 "charging" */
    WRSN_MC_RATE, WRSN_MC_CHTIME, WRSN_MC_NCONN,
    WRSN_MC_EXCL, WRSN_MC_PREVFIT,                     /* agents_exclusive_reward, min(agents_prev_fitness) */
    WRSN_MC_ACT0, WRSN_MC_ACT1, WRSN_MC_ACT2,          /* agents_action (clipped) */
    WRSN_MC_SLOT,                                      /* process slot holding agents_process[id] */
    WRSN_MC_LEN = 20
};

/* ---- charger process slot  proc[n_slot][WRSN_PR_LEN]  (one running MobileCharger.operate_step generator tree:
 *      operate_step -> move -> move_step / recharge / charge -> charge_step, flattened to one state machine with one
 *      pending event).  The first four doubles hold eight int32 fields (WRSN_PRI_*); the rest are doubles.
 *      A slot in the middle of a move (or of a charge without an alive connected node) only touches its own charger:
 *      it is marked LAZY, the engine schedules just the instant TINT at which that run of spans ends, and the spans in
 *      between are replayed in one tight loop when they are first needed. ---- */
enum { WRSN_PRI_USED = 0, WRSN_PRI_PROCESSED, WRSN_PRI_CURRENT, WRSN_PRI_AGENT, WRSN_PRI_PC, WRSN_PRI_STAGE, WRSN_PRI_LAZY,
       WRSN_PRI_SPARE };
enum {
    WRSN_PR_T = 4,                                     /* time of the pending event, +inf when none is pending */
    WRSN_PR_KEY,                                       /* priority * 2^40 + insertion counter of the pending event */
    WRSN_PR_PHY0, WRSN_PR_PHY1, WRSN_PR_PHY2,
    WRSN_PR_DESTX, WRSN_PR_DESTY, WRSN_PR_MT, WRSN_PR_VX, WRSN_PR_VY, WRSN_PR_TOTAL, WRSN_PR_SPAN,
    WRSN_PR_SVX, WRSN_PR_SVY, WRSN_PR_CHTMP, WRSN_PR_CHSPAN,
    WRSN_PR_TINT,                                      /* LAZY: time of the span event that ends the run of private spans */
    WRSN_PR_OWED,                                      /* LAZY: insertion counters drawn by the replayed spans, taken at wake-up */
    WRSN_PR_LEN = 22
};

/* ---- fields of one environment record (wrsn_state_layout) ---- */
enum {
    WRSN_F_HDR = 0, WRSN_F_MC, WRSN_F_PROC,            /* double rows, leader-only */
    WRSN_F_ENERGY, WRSN_F_RR, WRSN_F_CS,               /* double[Npad]  Node.energy / energyRR / energyCS */
    WRSN_F_ESEND, WRSN_F_LOGC,                         /* double[Npad]  e_send to the current receiver; log_energy of a no-death tick */
    WRSN_F_NBEF, WRSN_F_NAFT,                          /* uint16[Npad]  packets relayed per tick for lower / higher source ids */
    WRSN_F_LEVEL, WRSN_F_PARENT,                       /* int16[Npad]   Node.level; receiver (-2 base station, -1 none) */
    WRSN_F_STATUS,                                     /* uint8[Npad] */
    WRSN_F_TACT,                                       /* uint32[Tw]    Network.targets_active as a bitmask */
    WRSN_F_CONN,                                       /* uint32[M][W]  MobileCharger.connected_nodes as bitmasks */
    WRSN_F_LOGTICK,                                    /* double[Npad]  literal log_energy of a death tick */
    WRSN_F_RING,                                       /* double[WRSN_RING][Npad]  Node.log */
    WRSN_F_SCRATCH,                                    /* engine scratch: backup of energy / energyCS / status during a death tick */
    WRSN_F_COUNT
};

/* ---- fields of one scenario record (wrsn_scen_layout) ---- */
enum {
    WRSN_S_PAR = 0,                                    /* double[WRSN_P_LEN] */
    WRSN_S_NX, WRSN_S_NY, WRSN_S_BS_ESEND,             /* double[Npad] */
    WRSN_S_NBR_DIST, WRSN_S_NBR_ESEND,                 /* double[Emax]  per CSR entry (Node.probe_neighbors :80, send_package :107-115) */
    WRSN_S_NBR_PTR, WRSN_S_TGT_PTR,                    /* int32[Npad+1] */
    WRSN_S_NBR_IDX,                                    /* int32[Emax]   neighbour ids in id order */
    WRSN_S_TGT_IDX,                                    /* int32[TEmax]  covered target ids in id order (Node.probe_targets :86) */
    WRSN_S_DIRECT,                                     /* uint8[Npad]   d(node, BS) <= com_range (BaseStation.probe_neighbors :20) */
    WRSN_S_OBS_GX, WRSN_S_OBS_GY,                      /* float[Npad][obs_pitch]  exp(-(c_i - x_n)^2 / (2 hX^2)) of every node and map row /
                                                          column: the node terms of get_state never change (wrsn_build_obs_tables) */
    WRSN_S_COUNT
};

typedef struct wrsn_dims {
    int32_t B;        /* environments in this shard */
    int32_t N, T, M;  /* nodes and targets: the largest over the batch's scenarios (each scenario's own counts are its par
                         row's WRSN_P_NNODES / WRSN_P_NTARGETS; its node slots [own N, Npad) are dead padding); chargers
                         (the same for every scenario).  Npad, W, Tw, the layouts, the shared-memory size and `threads`
                         derive from these maxima, so every environment of a batch runs on the same thread count */
    int32_t S;        /* map_size */
    int32_t Emax;     /* neighbour CSR capacity per scenario */
    int32_t TEmax;    /* node->target CSR capacity per scenario */
    int32_t n_scen;   /* distinct scenarios */
    int32_t threads;  /* threads per environment (one CTA per environment), multiple of 32; 0 = choose */
    /* filled by wrsn_dims_finalize */
    int32_t Npad;     /* row pitch of node arrays (multiple of 16) */
    int32_t W;        /* 32-bit words per node bitmask */
    int32_t Tw;       /* 32-bit words per target bitmask */
    int32_t n_slot;   /* charger process slots per environment */
    int32_t state_bytes, state_resident_bytes, scen_bytes, smem_bytes;
    int32_t obs_pitch;  /* row pitch of the observation tables */
    /* set by the caller at any time (not touched by wrsn_dims_finalize) */
    int32_t step_budget;  /* 0: WRSN.step returns when the environment's next request is due, as the reference does.
                             > 0: work units per launch and environment (about one per simulated second in which a charger
                             charges a node, one per other event); a step that needs more returns agent_id = -4 ("in
                             flight") and continues at the next wrsn_step / wrsn_rollout_step call, so that a launch over many
                             environments lasts as long as the budget, not as long as its slowest environment */
    float obs_sigma_cells;  /* set by the caller (0 = unknown): the largest bandwidth of a node / charger source of get_state in map
                               cells over the batch's scenarios, charging_range / min(frame width, height) * S.  Narrow sources
                               (<= 2.9 cells: the shipped 1 km fields give 2.8) let wrsn_observe use its windowed float32 raster. */
    int32_t step_rounds;  /* with step_budget > 0.  0: one launch of the whole engine per wrsn_step / wrsn_rollout_step.
                             R > 0: a step is cut by KIND of work as well — R rounds of two launches, the events kernel (charger
                             events, fitness, deaths, cheap batches: everything but ...) and the batch kernel (... the
                             second-by-second loop of the seconds in which update_reward is active, at most step_budget of them
                             per launch).  Same results; the hot loop runs in launches of its own, where nothing else
                             competes for the instruction caches.  R < 0 is rejected. */
} wrsn_dims;

/* request record written by reset / step, device pointers, one row per environment */
typedef struct wrsn_request {
    int32_t *agent_id;                  /* [B]  -1 = None (terminal), -2 = implicit None (SURVEY Q7), -3 = untouched (masked out),
                                           -4 = the step is still in flight (wrsn_dims.step_budget): call again */
    uint8_t *terminal;                  /* [B] */
    double *reward;                     /* [B] */
    double *now;                        /* [B]  env.now */
    double *action;                     /* [B][3] agents_action[agent_id] */
    double *detail;                     /* [B][2] term_all, term_exclusive of get_reward (WRSN.py:225-226) */
    int32_t *flags;                     /* [B]  bit0 = every charger dead (the reference would never return, Q1), bit1 = engine error */
    double *stats;                      /* [B][3] running totals, never cleared by the library (may be NULL): requests handed out
                                           with a deciding charger; simulated seconds advanced by step; resets (episodes begun) */
    int32_t *sticky;                    /* [B]  OR of every `flags` value ever written for the row, never cleared by the library (may be NULL): a
                                           rollout that resets finished rows inside wrsn_rollout_step checks it once per window, not per step */
    int32_t *order;                     /* [B]  scratch of wrsn_step / wrsn_rollout_step (may be NULL): the order in which the step kernel's CTAs take the
                                           rows — longest predicted step first (time to the earliest charger's next decision, read from the
                                           process slots and the new actions), so that the launch does not end on a late, long environment */
} wrsn_request;

const char *wrsn_last_error(void);
int wrsn_abi_version(void);
int wrsn_field_count(int which);        /* 0 par, 1 hdr, 2 mc, 3 proc, 4 state fields, 5 scenario fields */
int wrsn_dims_finalize(wrsn_dims *d);
int wrsn_state_layout(const wrsn_dims *d, int64_t *offsets /* [WRSN_F_COUNT] */);
int wrsn_scen_layout(const wrsn_dims *d, int64_t *offsets /* [WRSN_S_COUNT] */);
int wrsn_device_ok(void);               /* 1 when a CUDA device of compute capability 10.x is usable */

/* Fill WRSN_S_OBS_GX / WRSN_S_OBS_GY of every scenario record (once, after uploading `scen`; needs par, node_x, node_y). */
int wrsn_build_obs_tables(const wrsn_dims *d, void *scen, void *stream);

/* NetworkIO.makeNetwork + Network.operate start (NetworkIO.py:19-34, Network.py:69-73): node / clock state at
 * t = 0.  with_reward_process != 0 also starts WRSN.update_reward (WRSN.py:43).  env_mask (may be NULL) selects rows. */
int wrsn_init_network(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state,
                      const uint8_t *env_mask, int with_reward_process, void *stream);
/* env.run(until=t) (WRSN.py:53): advance every selected environment to simulated time t_until[b]. */
int wrsn_run_until(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state,
                   const uint8_t *env_mask, const double *t_until, void *stream);
/* remainder of WRSN.reset after the warm-up (:44-83): chargers at the base station, fitness, reset-time
 * charger processes, first request. */
int wrsn_reset_finish(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state,
                      const uint8_t *env_mask, wrsn_request *req, void *stream);
/* reset from a snapshot: state[b] = snap[scen_id[b]] for selected rows (the t = warm_up state is a pure function
 * of the scenario, SURVEY Q8), then wrsn_reset_finish. */
int wrsn_reset_from_snapshot(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state,
                             const void *snap, const uint8_t *env_mask, wrsn_request *req, void *stream);
/* WRSN.step (:289-330): agent_id_in[b] = -1 means "no new action" (agent_id None); env_mask as above. */
int wrsn_step(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state,
              const uint8_t *env_mask, const int32_t *agent_id_in, const double *action_in,
              wrsn_request *req, void *stream);
/* One rollout step of every environment, three launches on `stream`, no host round trip:
 *   1. WRSN.step for the rows whose last request names a deciding charger (req->agent_id[b] >= 0), with that charger
 *      and action_in[b];
 *   2. WRSN.reset (from `snap`) for the rows whose episode has just ended (req->agent_id[b] < 0 after 1.);
 *   3. WRSN.get_state of the deciding charger of every row into obs (skipped when obs == NULL).
 * This is the reference's rollout loop body (controller/ippo/IPPO.py:137-143: reset on terminal, else step) for B
 * environments at once. */
int wrsn_rollout_step(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state, const void *snap,
                      const double *action_in, wrsn_request *req, void *obs, int obs_f64, void *stream);
/* WRSN.get_state (:130-186) for agent agent_id[b] of every environment with agent_id[b] >= 0, written to
 * obs[b][4][S][S] as float (obs_f64 == 0) or double.  Rows with agent_id[b] < 0 are left untouched. */
int wrsn_observe(const wrsn_dims *d, const void *scen, const int32_t *scen_id, const void *state,
                 const int32_t *agent_id, void *obs, int obs_f64, void *stream);
/* WRSN.density_map_to_action (:229-287) with the map normalisation of WRSN.step (:293-296): dmap[b][S][S] (float, or
 * double when dmap_f64 != 0) -> action_out[b][3] = (x-frac, y-frac, charge-time frac) for every row with
 * agent_id[b] >= 0; other rows are left untouched.  The location search replaces scipy's L-BFGS-B (see the kernel's
 * comment for what is reproduced exactly and what within tolerance).  Map sizes 1 to 176: the 99.9th percentile of a
 * larger map needs more order statistics than the decoder keeps, and such a map_size fails with an error (here and in
 * wrsn_decode_linear_controller).  A map that is -inf everywhere decodes to the box of cell 0, as np.argmax gives it. */
int wrsn_decode_density_map(const wrsn_dims *d, const void *scen, const int32_t *scen_id, const void *state,
                            const int32_t *agent_id, const void *dmap, int dmap_f64, double *action_out, void *stream);
/* The same decode for a controller whose density map is a LINEAR COMBINATION of the observation's channels — the reference's
 * RandomController (controller/random/RandomController.py:12-15: state[0] + state[1] - 10 * state[2] + state[3]) with
 * weights = {1, 1, -10, 1}: obs[b][channels][S][S] (float, as wrsn_observe writes it), weights[channels] on the HOST.  The
 * map is formed on the fly in float32, one rounding per multiply and add, channel by channel — the bits torch produces for
 * that expression — so the result equals wrsn_decode_density_map on the materialised map, without the controller's
 * elementwise passes over the observations. */
int wrsn_decode_linear_controller(const wrsn_dims *d, const void *scen, const int32_t *scen_id, const void *state,
                                  const int32_t *agent_id, const float *obs, int channels, const float *weights,
                                  double *action_out, void *stream);
/* The bookkeeping of the trainers' roll_out loop (controller/ippo/IPPO.py:138-155, controller/ppo/PPO.py likewise) for
 * every environment after rollout step t, one thread per environment:
 *   last[b][agent_prev[b]] = t                      log_probs_pre[agent] = log_prob            (:140)
 *   episode ended (req->stats[b][2] != resets_seen[b], then resets_seen[b] = it):  last[b][:] = -1   (:137-138, :143-144)
 *   agent_next[b] = req->agent_id[b]                the request handed out for step t + 1; -1 when the row has none (its step
 *                                                   is still in flight, wrsn_dims.step_budget)
 *   link_next[b]  = last[b][agent_next[b]]          step at which that agent last acted in this episode, -1: none (:145-146)
 *   new_episode_next[b], reward_next[b] (NaN -> 0), now_next[b]
 * `last` is int64 [B][M], the *_next pointers are row t + 1 of the caller's time-major record. */
int wrsn_record_transitions(const wrsn_dims *d, const wrsn_request *req, int64_t t, const int64_t *agent_prev,
                            int64_t *last, double *resets_seen, int64_t *agent_next, int64_t *link_next,
                            uint8_t *new_episode_next, double *reward_next, double *now_next, void *stream);
/* WRSN.get_network_fitness (:188-220): per-target values fitness[B][T] (may be NULL) and their minimum fit_min[B] over the row's own
 * targets; the columns beyond a row's own target count are not written. */
int wrsn_fitness(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state,
                 double *fitness, double *fit_min, void *stream);

/* standalone per-tick kernels (the same device functions the fused step uses; unit parity + ncu evidence) */
int wrsn_k_bfs(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state, void *stream);      /* Network.setLevels + receivers + relay counts */
int wrsn_k_drain(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state, void *stream);    /* Node.operate k+0.5 tick */
int wrsn_k_bookkeep(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state, void *stream); /* Node.operate k+1.0 tick */
int wrsn_k_reward(const wrsn_dims *d, const void *scen, const int32_t *scen_id, void *state, void *stream);   /* WRSN.update_reward tick */
/* The node x charger charging model, dense (Node.charger_connection Node.py:134-139 for the connected_nodes of
 * MobileCharger.charge MobileCharger.py:56-59): for every environment, every charger m with charging[b][m] != 0 (all chargers
 * when charging == NULL) at its position in the state record, and every ALIVE node n with d(n, m) <= charging_range,
 *     rate = alpha / (d + beta) ** 2;   node_rate[b][n] += rate  (chargers in id order);   mc_rate[b][m] += rate  (nodes in id order)
 * i.e. the energyRR every node would carry and the chargingRate every charger would draw if those chargers charged now.
 * One warp per environment, charger positions staged in shared memory, per-charger sums by warp ballot / shuffle IN NODE
 * ORDER (bit-exact with the reference's sequential +=).  The fused step kernel applies the same model incrementally (connect /
 * disconnect events); this entry point is the standalone form for unit parity and profiling.  Does not modify the state. */
int wrsn_k_charge(const wrsn_dims *d, const void *scen, const int32_t *scen_id, const void *state, const uint8_t *charging,
                  double *node_rate /* [B][N]: columns beyond a row's own node count are not written */, double *mc_rate /* [B][M] */,
                  void *stream);

#ifdef __cplusplus
}
#endif
#endif
