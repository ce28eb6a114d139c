/*
 * wrsn_layout.h — byte layout of one environment record / one scenario record / the shared-memory image
 * (shared by the host side of the C ABI, the kernels and the tests' host emulation).
 */
#pragma once
#include <float.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#include "wrsn_b200.h"

#if defined(WRSN_HOST_EMU)
#define WRSN_HD static inline
#define WRSN_HDM inline                             /* (member functions) */
#else
#define WRSN_HD __host__ __device__ static inline
#define WRSN_HDM __host__ __device__ inline
#endif

#define WRSN_SPEC_MAX 16                            /* charged (or otherwise irregular) nodes a whole-cycle batch handles by table */
#define WRSN_PAIR_MAX 32                            /* (charger, node) pairs the incentive sums of a batch handle by list */
#define WRSN_SPEC_LEN 6                             /* D1, D2, H, lo guard, hi guard, node id */

/* ------------------------------------------------------------------ layouts */
struct WrsnLayout {
    int64_t off[WRSN_F_COUNT];
    int64_t resident, total;                        /* bytes mirrored in shared memory / bytes per record */
    int64_t s_own, s_scr0, s_scr1, s_bcast, s_red, s_par, s_spec, s_exptab, s_pairs, smem_total;
    int64_t soff[WRSN_S_COUNT];
    int64_t scen_total;
    int32_t scr_len;                                /* doubles per scratch row */
};

WRSN_HD int64_t wrsn_a16(int64_t x) { return (x + 15) & ~(int64_t)15; }

WRSN_HD void wrsn_make_layout(const wrsn_dims *d, WrsnLayout *L) {
    const int64_t Np = d->Npad;
    int64_t o = 0;
    L->off[WRSN_F_HDR] = o; o += wrsn_a16(8 * WRSN_H_LEN);
    L->off[WRSN_F_MC] = o; o += wrsn_a16(8 * (int64_t)(d->M > 0 ? d->M : 1) * WRSN_MC_LEN);
    L->off[WRSN_F_PROC] = o; o += wrsn_a16(8 * (int64_t)d->n_slot * WRSN_PR_LEN);
    L->off[WRSN_F_ENERGY] = o; o += 8 * Np;
    L->off[WRSN_F_RR] = o; o += 8 * Np;
    L->off[WRSN_F_CS] = o; o += 8 * Np;
    L->off[WRSN_F_ESEND] = o; o += 8 * Np;
    L->off[WRSN_F_LOGC] = o; o += 8 * Np;
    L->off[WRSN_F_NBEF] = o; o += 2 * Np;
    L->off[WRSN_F_NAFT] = o; o += 2 * Np;
    L->off[WRSN_F_LEVEL] = o; o += 2 * Np;
    L->off[WRSN_F_PARENT] = o; o += 2 * Np;
    L->off[WRSN_F_STATUS] = o; o += Np;
    L->off[WRSN_F_TACT] = o; o += wrsn_a16(4 * (int64_t)d->Tw);
    L->off[WRSN_F_CONN] = o; o += wrsn_a16(4 * (int64_t)(d->M > 0 ? d->M : 1) * d->W);
    L->resident = o;
    L->off[WRSN_F_LOGTICK] = o; o += 8 * Np;
    L->off[WRSN_F_RING] = o; o += 8 * Np * WRSN_RING;
    L->off[WRSN_F_SCRATCH] = o; o += wrsn_a16(17 * Np);
    L->total = o;
    /* shared-memory extras behind the resident image */
    int64_t Tp = ((int64_t)d->T + 15) & ~(int64_t)15;
    L->scr_len = (int32_t)(Np > Tp ? Np : Tp);
    int64_t s = L->resident;
    L->s_own = s; s += 2 * Np;
    L->s_scr0 = s; s += 8 * (int64_t)L->scr_len;
    L->s_scr1 = s; s += 8 * (int64_t)L->scr_len;
    L->s_bcast = s; s += 64;
    L->s_red = s; s += 8 * 32;
    L->s_par = s; s += 8 * WRSN_P_LEN;             /* scenario constants: copied next to the state, never re-read from HBM */
    L->s_spec = s; s += 8 * WRSN_SPEC_LEN * WRSN_SPEC_MAX;   /* per-batch table of the charged nodes (wrsn_engine.cuh: reward_cycles) */
    L->s_exptab = s; s += 8 * 64;                  /* 2^(j/64): table of the reward path's exponential */
    L->s_pairs = s; s += 8 * WRSN_PAIR_MAX + 4 * 2 * WRSN_PAIR_MAX + 4 * 2 * WRSN_MAX_MC;   /* (charging charger, connected alive node) pairs of the current batch:
                                                      term double[PAIR_MAX]; {charger, node} int[PAIR_MAX][2]; per charger {first, end} int[MAX_MC][2] */
    L->smem_total = s;
    /* scenario record */
    o = 0;
    L->soff[WRSN_S_PAR] = o; o += wrsn_a16(8 * WRSN_P_LEN);
    L->soff[WRSN_S_NX] = o; o += 8 * Np;
    L->soff[WRSN_S_NY] = o; o += 8 * Np;
    L->soff[WRSN_S_BS_ESEND] = o; o += 8 * Np;
    L->soff[WRSN_S_NBR_DIST] = o; o += wrsn_a16(8 * (int64_t)d->Emax);
    L->soff[WRSN_S_NBR_ESEND] = o; o += wrsn_a16(8 * (int64_t)d->Emax);
    L->soff[WRSN_S_NBR_PTR] = o; o += wrsn_a16(4 * (Np + 1));
    L->soff[WRSN_S_TGT_PTR] = o; o += wrsn_a16(4 * (Np + 1));
    L->soff[WRSN_S_NBR_IDX] = o; o += wrsn_a16(4 * (int64_t)d->Emax);
    L->soff[WRSN_S_TGT_IDX] = o; o += wrsn_a16(4 * (int64_t)d->TEmax);
    L->soff[WRSN_S_DIRECT] = o; o += Np;
    o = wrsn_a16(o);
    L->soff[WRSN_S_OBS_GX] = o; o += 4 * Np * (int64_t)d->obs_pitch;
    L->soff[WRSN_S_OBS_GY] = o; o += 4 * Np * (int64_t)d->obs_pitch;
    L->scen_total = wrsn_a16(o);
}


/* ------------------------------------------------------------------ one row of the batch
 * Where the fields of environment b's record and of its scenario's record are, for everything outside the environment kernel
 * (the raster, the decoder, the charging model, the launch order; their host restatements in the tests' emulation). */
struct WrsnRow {
    const double *par, *nx, *ny;                    /* scenario record */
    const float *tab_gx, *tab_gy;                   /* its observation tables (wrsn_kernels.cu: k_obs_tables) */
    const double *hdr, *mc, *proc, *energy, *cs;    /* environment record */
    const uint8_t *status;
    int N;                                          /* this scenario's nodes (dims.N: the batch's largest) */
    WRSN_HDM WrsnRow(const WrsnLayout &L, const char *state, const char *scen, const int32_t *scen_id, int b)
        : WrsnRow(L, state + (size_t)b * L.total, scen + (size_t)scen_id[b] * L.scen_total) {}
    /* `row`: a record, or its resident image in shared memory (the fields read here are all resident); `srow`: its scenario's record */
    WRSN_HDM WrsnRow(const WrsnLayout &L, const char *row, const char *srow) {
        par = (const double *)(srow + L.soff[WRSN_S_PAR]);
        nx = (const double *)(srow + L.soff[WRSN_S_NX]);
        ny = (const double *)(srow + L.soff[WRSN_S_NY]);
        tab_gx = (const float *)(srow + L.soff[WRSN_S_OBS_GX]);
        tab_gy = (const float *)(srow + L.soff[WRSN_S_OBS_GY]);
        hdr = (const double *)(row + L.off[WRSN_F_HDR]);
        mc = (const double *)(row + L.off[WRSN_F_MC]);
        proc = (const double *)(row + L.off[WRSN_F_PROC]);
        energy = (const double *)(row + L.off[WRSN_F_ENERGY]);
        cs = (const double *)(row + L.off[WRSN_F_CS]);
        status = (const uint8_t *)(row + L.off[WRSN_F_STATUS]);
        N = (int)par[WRSN_P_NNODES];
    }
};

/* ------------------------------------------------------------------ the sources of WRSN.get_state (rl_env/WRSN.py:130-186)
 * 4 x S x S map per environment.  Every source (alive node, charger) contributes w * G(x - x0; hX) * G(y - y0; hY) with
 * G(u; h) = exp(u^2 / (-2 h^2)) on the cell centres np.arange(unit / 2, 1.0, unit) of the frame scaled to [0, 1]. */
struct ObsGrid {
    double f0, f2, Wd, Hd, unit, start, delta, R, mtm;
    WRSN_HDM ObsGrid(const double *par, int S) {
        f0 = par[WRSN_P_F0]; f2 = par[WRSN_P_F2];
        Wd = par[WRSN_P_F1] - f0; Hd = par[WRSN_P_F3] - f2;
        unit = 1.0 / (double)S; start = unit / 2.0; delta = (start + unit) - start;
        R = par[WRSN_P_MC_R]; mtm = par[WRSN_P_MTM];
    }
    WRSN_HDM double cx(double x) const { return (x - f0) / Wd; }
    WRSN_HDM double cy(double y) const { return (y - f2) / Hd; }
    WRSN_HDM double cell(int i) const { return start + (double)i * delta; }
};

/* one entry of a source's 1-D vector: exp(u^2 / dn), dn = -2 h^2, at cell centre c (below -745.2 exp underflows to 0 anyway) */
WRSN_HD double obs_gauss(double c, double x0, double dn) {
    const double u = c - x0, a = u * u / dn;
    return a > -745.2 ? exp(a) : 0.0;
}

/* source s of channel ch as seen by charger ag; mode < 0: unused (a dead node, a node without traffic — energyCS == 0 adds
 * exact zeros —, the observer itself or a charger of the other type in channels 2 and 3).  Mode 1 (channel 3, the travel
 * time) is divided by moving_time_max as well, which every raster folds in at its own place.  node >= 0: the node's row of
 * the scenario's observation tables. */
struct ObsSrc { double x0, y0, hx, hy, w; int mode; int node; };
WRSN_HD ObsSrc obs_source(const WrsnRow &r, const ObsGrid &g, int ag, int ch, int s) {
    ObsSrc v; v.mode = -1; v.node = -1; v.x0 = v.y0 = v.w = 0.0; v.hx = v.hy = 1.0;
    const double *par = r.par, *me = r.mc + (size_t)ag * WRSN_MC_LEN;
    if (ch == 0) {                                  /* alive nodes with traffic */
        if (r.status[s] != 0) {
            v.mode = 0; v.node = s;
            v.x0 = g.cx(r.nx[s]); v.y0 = g.cy(r.ny[s]); v.hx = g.R / g.Wd; v.hy = g.R / g.Hd;
            v.w = (r.cs[s] / par[WRSN_P_MC_AB2]) / ((r.energy[s] - par[WRSN_P_THR]) / par[WRSN_P_CAPMTHR]);
            if (v.w == 0.0) v.mode = -1;
        }
    } else if (ch == 1) {                           /* the observer: bandwidth 0.5 min(W, H) / extent */
        const double tmp = fmin(g.Hd, g.Wd);
        v.mode = 0;
        v.x0 = g.cx(me[WRSN_MC_X]); v.y0 = g.cy(me[WRSN_MC_Y]);
        v.hx = 0.5 * tmp / g.Wd; v.hy = 0.5 * tmp / g.Hd;
        v.w = me[WRSN_MC_ENERGY] / par[WRSN_P_MC_CAP];
    } else {                                        /* the other chargers at their destinations, by type */
        const double *an = r.mc + (size_t)s * WRSN_MC_LEN;
        const bool charging = an[WRSN_MC_TYPE] != 0.0;
        if (s != ag && (ch == 2 ? charging : !charging)) {
            v.x0 = g.cx(an[WRSN_MC_CPA0]); v.y0 = g.cy(an[WRSN_MC_CPA1]); v.hx = g.R / g.Wd; v.hy = g.R / g.Hd;
            if (ch == 2) { v.mode = 0; v.w = an[WRSN_MC_CPA2] / par[WRSN_P_CTM]; }
            else {                                  /* SURVEY Q5: the observer's destination y */
                const double dx = an[WRSN_MC_X] - an[WRSN_MC_CPA0], dy = an[WRSN_MC_Y] - me[WRSN_MC_CPA1];
                v.w = sqrt(dx * dx + dy * dy) / par[WRSN_P_MC_V];
                v.mode = 1;
            }
        }
    }
    return v;
}

/* ------------------------------------------------------------------ observation tables
 * Output tile of a thread of the observation rasters (wrsn_kernels.cu: k_observe, k_observe_win): OBS_TI rows x OBS_TJ64 columns
 * in the fp64 raster, x OBS_TJ32 in the fp32 one.  The node tables of the scenario record are padded to whole tiles. */
#define OBS_TI 4
#define OBS_TJ64 10
#define OBS_TJ32 20

WRSN_HD int32_t wrsn_obs_pitch(int S) {
    const int ti = (S + OBS_TI - 1) / OBS_TI;
    const int tj = (S + OBS_TJ64 - 1) / OBS_TJ64, tk = (S + OBS_TJ32 - 1) / OBS_TJ32;
    const int pk = (tk * OBS_TJ32 + 3) & ~3;
    int pi = ti * OBS_TI, pj = (tj * OBS_TJ64 + 3) & ~3;
    if (pk > pj) pj = pk;
    return pi > pj ? pi : pj;
}

/* ------------------------------------------------------------------ the hand-written charging rules (include/wrsn_b200.h:
 * wrsn_heuristic_action).  k_heuristic, the rule rollout (wrsn_env_kernel.cuh: roll_pick) and the host emulation state the rule
 * only through these functions. */
#define HEUR_NONE 0x7fffffff                        /* id of an empty set's best: sorts after every node */

struct HeurFleet {                                  /* what the rule reads of a row's chargers, once per row */
    double ax, ay;                                  /* the deciding charger's position */
    double dx[WRSN_MAX_MC], dy[WRSN_MAX_MC];        /* every charger's destination (cur_phy_action) */
    uint8_t on[WRSN_MAX_MC];                        /* 1: charger j can claim a node (alive, not the deciding one) */
    int M;
};

WRSN_HD void heur_charger(const WrsnRow &rw, int a, int j, HeurFleet *f) {
    const double *m = rw.mc + (size_t)j * WRSN_MC_LEN;
    f->dx[j] = m[WRSN_MC_CPA0]; f->dy[j] = m[WRSN_MC_CPA1];
    f->on[j] = (j != a && m[WRSN_MC_STATUS] != 0.0) ? 1 : 0;
    if (j == a) { f->ax = m[WRSN_MC_X]; f->ay = m[WRSN_MC_Y]; }
}

/* euclid2's arithmetic (wrsn_engine.cuh): both builds compile without contraction, so products and sum round separately */
WRSN_HD double heur_dist(double ax, double ay, double bx, double by) {
    const double dx = ax - bx, dy = ay - by;
    return sqrt(dx * dx + dy * dy);
}

/* Node i under the rule.  pass 0: claimed nodes are not candidates; pass 1 (when pass 0 has none): every alive node is.
 * Returns 0 when i is not a candidate, 1 when it is, 2 when it is also urgent under WRSN_HEUR_NEAREST_URGENT.
 * key[0]: the lifetime (min_lifetime's key, nearest_urgent's fallback); key[1] (urgent nodes): the distance from charger a. */
WRSN_HD int heur_key(const WrsnRow &rw, const HeurFleet &f, int kind, int i, int pass, double key[2]) {
    if (rw.status[i] != 1) return 0;
    const double *par = rw.par;
    const double x = rw.nx[i], y = rw.ny[i];
    if (pass == 0)
        for (int j = 0; j < f.M; j++)
            if (f.on[j] && heur_dist(x, y, f.dx[j], f.dy[j]) <= par[WRSN_P_MC_R]) return 0;
    const double cs = rw.cs[i];
    key[0] = cs <= 0.0 ? (double)INFINITY : (rw.energy[i] - par[WRSN_P_THR]) / cs;   /* no traffic: never needs a charger */
    if (kind == WRSN_HEUR_NEAREST_URGENT && key[0] < par[WRSN_P_MTM] + par[WRSN_P_CTM]) {
        key[1] = heur_dist(f.ax, f.ay, x, y);
        return 2;
    }
    return 1;
}

/* the smallest (key, id) of the candidates (k[0], i[0]) and of the urgent ones (k[1], i[1]) seen so far */
struct HeurPick {
    double k[2]; int i[2];
    WRSN_HDM HeurPick() { k[0] = k[1] = (double)INFINITY; i[0] = i[1] = HEUR_NONE; }
    WRSN_HDM void take(int s, double key, int id) {
        if (key < k[s] || (key == k[s] && id < i[s])) { k[s] = key; i[s] = id; }
    }
    WRSN_HDM void add(int cls, const double key[2], int id) {
        if (cls) take(0, key[0], id);
        if (cls == 2) take(1, key[1], id);
    }
    WRSN_HDM int choice() const { return i[1] != HEUR_NONE ? i[1] : (i[0] != HEUR_NONE ? i[0] : -1); }
};

/* the action of charger a for node i (i < 0: no alive node, charger a stays where it is) */
WRSN_HD void heur_action(const WrsnRow &rw, int a, int i, double *out) {
    const double *par = rw.par, *m = rw.mc + (size_t)a * WRSN_MC_LEN;
    const double W = par[WRSN_P_F1] - par[WRSN_P_F0], H = par[WRSN_P_F3] - par[WRSN_P_F2];
    const double x = i >= 0 ? rw.nx[i] : m[WRSN_MC_X], y = i >= 0 ? rw.ny[i] : m[WRSN_MC_Y];
    out[0] = W == 0.0 ? 0.0 : (x - par[WRSN_P_F0]) / W;
    out[1] = H == 0.0 ? 0.0 : (y - par[WRSN_P_F2]) / H;
    double c = 0.0;                                 /* time to refill at the peak rate alpha / beta^2, over charging_time_max */
    if (i >= 0) { c = (par[WRSN_P_CAP] - rw.energy[i]) / par[WRSN_P_CAPMTHR]; c = c > 1.0 ? 1.0 : (c > 0.0 ? c : 0.0); }
    out[2] = c;
}

/* The rule's candidate order (include/wrsn_b200.h: wrsn_heuristic_candidates): one total order on (class, key, id), node ids
 * being distinct.  heur_key's urgent nodes come first (class 0, key: the distance from charger a), then the rest (class 1,
 * key: the lifetime), so the order's first node is HeurPick's choice.  k_heuristic_candidates and the host emulation state the
 * order only through these functions. */
struct HeurRank { double key; int cls, id; };

/* node i's place in the order; false when i is not a candidate in this pass */
WRSN_HD bool heur_rank(const WrsnRow &rw, const HeurFleet &f, int kind, int i, int pass, HeurRank *r) {
    double key[2] = {0.0, 0.0};
    const int c = heur_key(rw, f, kind, i, pass, key);
    if (c == 0) return false;
    r->cls = c == 2 ? 0 : 1;
    r->key = key[c - 1];
    r->id = i;
    return true;
}

WRSN_HD bool heur_before(const HeurRank &p, const HeurRank &q) {
    return p.cls < q.cls || (p.cls == q.cls && (p.key < q.key || (p.key == q.key && p.id < q.id)));
}

/* insert r into the ascending list l[0], l[s], ..., l[(n - 1) s] that keeps the cap smallest entries seen (stride s: one lane's
 * column of k_heuristic_candidates' shared list, 1 on the host) */
WRSN_HD void heur_insert(HeurRank *l, int s, int &n, int cap, const HeurRank &r) {
    if (n == cap && !heur_before(r, l[(n - 1) * s])) return;
    int p = n < cap ? n++ : cap - 1;
    for (; p > 0 && heur_before(r, l[(p - 1) * s]); p--) l[p * s] = l[(p - 1) * s];
    l[p * s] = r;
}

/* slot k of row b: the node of rank k (node_k < 0: fewer candidates than slots), with slot 0's action when it has none */
WRSN_HD void heur_slot(const WrsnRow &rw, int a, int node_k, int node_0, double *action, int32_t *node) {
    heur_action(rw, a, node_k >= 0 ? node_k : node_0, action);
    *node = node_k;
}

/* request record of one environment, as the engine's entry points produce it */
struct ReqOut { int agent; int terminal; double reward, now, act[3], detail[2]; int flags; };

/* roll_out bookkeeping of row b (see include/wrsn_b200.h: wrsn_record_transitions) */
WRSN_HD void record_transition(int b, int M, const wrsn_request &req, int64_t t, const int64_t *agent_prev, int64_t *last,
                               double *resets_seen, int64_t *agent_next, int64_t *link_next, uint8_t *new_episode_next,
                               double *reward_next, double *now_next) {
    int64_t *row = last + (size_t)b * M;
    const int64_t ap = agent_prev[b];
    if (ap >= 0 && ap < M) row[ap] = t;
    const double resets = req.stats[(size_t)b * 3 + 2];
    const bool ended = resets != resets_seen[b];
    resets_seen[b] = resets;
    if (ended)
        for (int a = 0; a < M; a++) row[a] = -1;
    int an = req.agent_id[b];                        /* < 0: no request for this row (-4: its step is still in flight) */
    if (an >= M) an = M - 1;
    agent_next[b] = an < 0 ? -1 : an;
    link_next[b] = an < 0 ? -1 : row[an];
    new_episode_next[b] = ended ? 1 : 0;
    const double r = req.reward[b];
    reward_next[b] = (r == r) ? r : 0.0;
    now_next[b] = req.now[b];
}

/* continuation state of row s outside its state record, copied to row d (see include/wrsn_b200.h: wrsn_copy_rows): scen_id and
 * the request row.  `order` is launch scratch of the next step call (k_step_order rewrites it from the state records), so it is
 * not part of a row's state. */
WRSN_HD void copy_row_request(const wrsn_request &src, const int32_t *src_scen_id, int s, const wrsn_request &dst,
                              int32_t *dst_scen_id, int d) {
    dst_scen_id[d] = src_scen_id[s];
    dst.agent_id[d] = src.agent_id[s];
    dst.terminal[d] = src.terminal[s];
    dst.reward[d] = src.reward[s];
    dst.now[d] = src.now[s];
    for (int k = 0; k < 3; k++) dst.action[(size_t)d * 3 + k] = src.action[(size_t)s * 3 + k];
    for (int k = 0; k < 2; k++) dst.detail[(size_t)d * 2 + k] = src.detail[(size_t)s * 2 + k];
    dst.flags[d] = src.flags[s];
    if (src.stats && dst.stats)
        for (int k = 0; k < 3; k++) dst.stats[(size_t)d * 3 + k] = src.stats[(size_t)s * 3 + k];
    if (src.sticky && dst.sticky) dst.sticky[d] = src.sticky[s];
}
