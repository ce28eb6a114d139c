/*
 * wrsn_oracle.c — CPU restatement of the reference WRSN simulator hot path.
 *
 * TEST INFRASTRUCTURE.  This file is the parity ORACLE.  It is linked / loaded only by
 * tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs,
 * and only as the checker or the reported CPU baseline — never by the product package
 * (multi_agent_rl_wrsn_b200/), which has no CPU path at all.
 *
 * Pinning: the reference ships no tests or golden vectors (SURVEY.md §4).  This
 * restatement is pinned against outputs of the reference itself, run unmodified in the
 * build container under oracle/shims (fixtures tests/golden/*.npz, made by
 * oracle/gen_golden.py; checked by tests/test_oracle_golden.py).  The one third-party
 * layer underneath — simpy==4.0.1 (requirements.txt:52), absent from the image — is
 * restated from its published scheduling contract in BOTH oracle/shims/simpy and here;
 * against a real SimPy wheel that layer is "parity unpinned".
 *
 * Structure: a literal discrete-event engine (heap keyed (time, priority, eid), URGENT
 * process starts, NORMAL timeouts / completions / conditions, nested AnyOf chain with
 * check-callback removal) plus one explicit state machine per reference generator:
 *   Network.operate      physical_env/network/Network.py:69-81   (setLevels :37-66, check_targets :84-85)
 *   Node.operate         physical_env/network/Node.py:45-78      (send/receive/find_receiver :92-132, check_status :148-151)
 *   BaseStation.operate  physical_env/network/BaseStation.py:29-31 (probe_neighbors :20-23)
 *   MobileCharger.*      physical_env/mc/MobileCharger.py:34-140
 *   WRSN.update_reward   rl_env/WRSN.py:100-127;  reset :41-83;  step :289-330;
 *   get_state :130-186;  get_network_fitness :188-220;  get_reward :222-227;  translate :95-98
 * Per-packet routing is done packet by packet, hop by hop, exactly as the reference
 * does it (no aggregation), so the floating-point operation order is the reference's.
 *
 * Build: see oracle/Makefile (gcc -O2 -ffp-contract=off; no FMA contraction).
 */
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define URGENT 0
#define NORMAL 1

enum { EV_INIT, EV_TIMEOUT, EV_PROCDONE, EV_COND, EV_UNTIL };
enum { P_NETOP, P_UR, P_NODE, P_BS, P_OPSTEP, P_MOVE, P_MOVESTEP, P_RECHARGE, P_CHARGE, P_CHARGESTEP };
enum { CB_RESUME, CB_CHECK, CB_BUILD, CB_STOP };
enum { OP_PROC, OP_COND };
#define CB_MAX 8

typedef struct { double t; int prio; long long eid; int type; int idx; } Ev;

typedef struct {
    int kind, state, id, in_use, processed, triggered, recyclable;
    int ncb, cb_type[CB_MAX], cb_idx[CB_MAX];
    double d[10];            /* generator locals */
} Proc;

typedef struct {
    int all;                 /* 1 = AllOf, 0 = AnyOf */
    int op_type[2], op_idx[2];
    int count, triggered, processed;
    int ncb, cb_type[CB_MAX], cb_idx[CB_MAX];
} Cond;

typedef struct {
    double x, y, energy, capacity, threshold, alpha, beta, velocity, pm, range, epsilon;
    double charging_rate, cpa[3], charging_time;
    int status, type_charging, nconn, *conn;
} MC;

typedef struct Oracle {
    /* scenario */
    int N, T, M, S;
    double *nx, *ny, *tx, *ty, bsx, bsy;
    double capacity, threshold, com_range, sen_range, prob_gp, package_size, er, et, efs, emp, max_time;
    /* static graph (Node.probe_neighbors/probe_targets, BaseStation.probe_neighbors) */
    int *nbr_ptr, *nbr_idx, *tgt_ptr, *tgt_idx, *direct, ndirect, *direct_list;
    int probed_bs;
    /* node state */
    double *energy, *rr, *cs, *log_energy, *logbuf; int *loglen, *status, *level;
    unsigned char *targets_active; int alive;
    double frame[4], nodes_density;
    /* engine */
    Ev *heap; int hn, hcap; long long eid; double now; int stop;
    Proc *procs; int nprocs, pcap; int *freelist, nfree;
    Cond *conds; int nconds, ccap;
    /* wrsn layer */
    MC *mc; double mcpar[8];
    int netop_proc, ur_proc, netp_cond, *agent_proc;
    double *excl, *prev_fit_min, *agents_action;
    double moving_time_max, charging_time_max, avg_nodes_agent, eps_env, warm_up;
    long long nevents, event_budget; int budget_hit;
    long long n_ticks_drain;
} Oracle;

/* ------------------------------------------------------------------ helpers */
static double euclid(double ax, double ay, double bx, double by) {
    /* scipy.spatial.distance.euclidean -> numpy.linalg.norm -> sqrt(dot(d, d)); verified
       bit-identical to sqrt(dx*dx + dy*dy) for 2-vectors with the installed numpy. */
    double dx = ax - bx, dy = ay - by;
    return sqrt(dx * dx + dy * dy);
}

/* numpy pairwise summation (add.reduce on a contiguous float64 vector) */
static double pairwise_sum(const double *a, int n) {
    if (n < 8) {
        double r = 0.;
        for (int i = 0; i < n; i++) r += a[i];
        return r;
    } else if (n <= 128) {
        double r[8];
        int i;
        for (i = 0; i < 8; i++) r[i] = a[i];
        for (i = 8; i < n - (n % 8); i += 8)
            for (int j = 0; j < 8; j++) r[j] += a[i + j];
        double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
        for (; i < n; i++) res += a[i];
        return res;
    } else {
        int n2 = n / 2;
        n2 -= n2 % 8;
        return pairwise_sum(a, n2) + pairwise_sum(a + n2, n - n2);
    }
}

/* ------------------------------------------------------------------ heap */
static int ev_less(const Ev *a, const Ev *b) {
    if (a->t != b->t) return a->t < b->t;
    if (a->prio != b->prio) return a->prio < b->prio;
    return a->eid < b->eid;
}
static void schedule(Oracle *o, int type, int idx, int prio, double delay) {
    if (o->hn == o->hcap) { o->hcap *= 2; o->heap = realloc(o->heap, sizeof(Ev) * o->hcap); }
    Ev e = { o->now + delay, prio, o->eid++, type, idx };
    int i = o->hn++;
    while (i > 0) {
        int p = (i - 1) / 2;
        if (!ev_less(&e, &o->heap[p])) break;
        o->heap[i] = o->heap[p]; i = p;
    }
    o->heap[i] = e;
}
static Ev heap_pop(Oracle *o) {
    Ev top = o->heap[0];
    Ev last = o->heap[--o->hn];
    int i = 0;
    for (;;) {
        int l = 2 * i + 1, r = l + 1, m = i;
        const Ev *me = &last;
        if (l < o->hn && ev_less(&o->heap[l], me)) { m = l; me = &o->heap[l]; }
        if (r < o->hn && ev_less(&o->heap[r], me)) { m = r; }
        if (m == i) break;
        o->heap[i] = o->heap[m]; i = m;
    }
    if (o->hn > 0) o->heap[i] = last;
    return top;
}

/* ------------------------------------------------------------------ processes / conditions */
static int new_proc(Oracle *o, int kind, int id, int recyclable) {
    int p;
    if (o->nfree > 0) p = o->freelist[--o->nfree];
    else {
        if (o->nprocs == o->pcap) {
            o->pcap *= 2;
            o->procs = realloc(o->procs, sizeof(Proc) * o->pcap);
            o->freelist = realloc(o->freelist, sizeof(int) * o->pcap);
        }
        p = o->nprocs++;
    }
    Proc *P = &o->procs[p];
    memset(P, 0, sizeof(*P));
    P->kind = kind; P->id = id; P->in_use = 1; P->recyclable = recyclable;
    schedule(o, EV_INIT, p, URGENT, 0.0);     /* Initialize event */
    return p;
}
static void proc_add_cb(Oracle *o, int p, int type, int idx) {
    Proc *P = &o->procs[p];
    if (P->ncb >= CB_MAX) { fprintf(stderr, "oracle: proc callback overflow\n"); abort(); }
    P->cb_type[P->ncb] = type; P->cb_idx[P->ncb] = idx; P->ncb++;
}
static void cond_add_cb(Oracle *o, int c, int type, int idx) {
    Cond *C = &o->conds[c];
    if (C->ncb >= CB_MAX) { fprintf(stderr, "oracle: cond callback overflow\n"); abort(); }
    C->cb_type[C->ncb] = type; C->cb_idx[C->ncb] = idx; C->ncb++;
}
static void remove_cb(int *ncb, int *types, int *idxs, int type, int idx) {
    for (int i = 0; i < *ncb; i++)
        if (types[i] == type && idxs[i] == idx) {        /* list.remove: first match */
            for (int j = i; j + 1 < *ncb; j++) { types[j] = types[j + 1]; idxs[j] = idxs[j + 1]; }
            (*ncb)--;
            return;
        }
}
static void cond_check(Oracle *o, int c) {
    Cond *C = &o->conds[c];
    if (C->triggered) return;
    C->count++;
    int ok = C->all ? (C->count == 2) : (C->count > 0);
    if (ok) { C->triggered = 1; schedule(o, EV_COND, c, NORMAL, 0.0); }
}
static int op_processed(Oracle *o, int type, int idx) {
    return type == OP_PROC ? o->procs[idx].processed : o->conds[idx].processed;
}
static int new_cond(Oracle *o, int all, int t0, int i0, int t1, int i1) {
    if (o->nconds == o->ccap) { o->ccap *= 2; o->conds = realloc(o->conds, sizeof(Cond) * o->ccap); }
    int c = o->nconds++;
    Cond *C = &o->conds[c];
    memset(C, 0, sizeof(*C));
    C->all = all; C->op_type[0] = t0; C->op_idx[0] = i0; C->op_type[1] = t1; C->op_idx[1] = i1;
    for (int k = 0; k < 2; k++) {
        if (op_processed(o, C->op_type[k], C->op_idx[k])) cond_check(o, c);
        else if (C->op_type[k] == OP_PROC) proc_add_cb(o, C->op_idx[k], CB_CHECK, c);
        else cond_add_cb(o, C->op_idx[k], CB_CHECK, c);
        C = &o->conds[c];
    }
    cond_add_cb(o, c, CB_BUILD, c);
    return c;
}
static void cond_remove_checks(Oracle *o, int c) {
    Cond *C = &o->conds[c];
    for (int k = 0; k < 2; k++) {
        int ty = C->op_type[k], ix = C->op_idx[k];
        if (ty == OP_PROC) {
            Proc *P = &o->procs[ix];
            if (!P->processed) remove_cb(&P->ncb, P->cb_type, P->cb_idx, CB_CHECK, c);
        } else {
            Cond *D = &o->conds[ix];
            if (!D->processed) remove_cb(&D->ncb, D->cb_type, D->cb_idx, CB_CHECK, c);
            cond_remove_checks(o, ix);
        }
    }
}

static void proc_finish(Oracle *o, int p) {       /* StopIteration -> schedule completion */
    o->procs[p].triggered = 1;
    schedule(o, EV_PROCDONE, p, NORMAL, 0.0);
}
static void wait_timeout(Oracle *o, int p, double delay) {
    if (delay < 0) { fprintf(stderr, "oracle: negative delay %g\n", delay); abort(); }
    schedule(o, EV_TIMEOUT, p, NORMAL, delay);
}
static int spawn_child(Oracle *o, int parent, int kind, int id) {
    int c = new_proc(o, kind, id, 1);
    proc_add_cb(o, c, CB_RESUME, parent);
    return c;
}

/* ------------------------------------------------------------------ network physics */
static void check_status(Oracle *o, int i) {               /* Node.py:148-151 */
    if (o->energy[i] <= o->threshold) { o->status[i] = 0; o->cs[i] = 0.0; }
}
static int find_receiver(Oracle *o, int i) {               /* Node.py:92-100 */
    int best = -1; double bd = 0.0;
    for (int e = o->nbr_ptr[i]; e < o->nbr_ptr[i + 1]; e++) {
        int j = o->nbr_idx[e];
        if (o->level[j] < o->level[i] && o->status[j] == 1) {
            double d = euclid(o->nx[j], o->ny[j], o->nx[i], o->ny[i]);
            if (best < 0 || d < bd) { best = j; bd = d; }   /* np.argmin: first minimum */
        }
    }
    return best;
}
static void send_package(Oracle *o, int i);
static void receive_package(Oracle *o, int i) {            /* Node.py:124-132 */
    double e_receive = o->er * o->package_size;
    if (o->energy[i] - o->threshold < e_receive) o->energy[i] = o->threshold;
    else {
        o->energy[i] -= e_receive;
        send_package(o, i);
        o->log_energy[i] += e_receive;
    }
    check_status(o, i);
}
/* Node.send_package's `d ** 2` / `d ** 4` are libm pow calls in the reference (and in scenario.py's e_send table).  A literal
   pow(d, 2.0) is folded by gcc into d * d, the correctly rounded square, which glibc's pow misses by one ulp for some d (e.g.
   61.71026423045482): the pointer keeps the call a call. */
static double (*volatile libm_pow)(double, double) = pow;
static void send_package(Oracle *o, int i) {               /* Node.py:106-122 */
    double d0 = pow(o->efs / o->emp, 0.5);
    int recv;                                               /* -2 = base station, -1 = none */
    if (euclid(o->nx[i], o->ny[i], o->bsx, o->bsy) > o->com_range) recv = find_receiver(o, i);
    else recv = -2;
    if (recv != -1) {
        double d = recv == -2 ? euclid(o->nx[i], o->ny[i], o->bsx, o->bsy)
                              : euclid(o->nx[i], o->ny[i], o->nx[recv], o->ny[recv]);
        double e_send = ((d <= d0) ? (o->et + o->efs * libm_pow(d, 2.0)) : (o->et + o->emp * libm_pow(d, 4.0))) * o->package_size;
        if (o->energy[i] - o->threshold < e_send) o->energy[i] = o->threshold;
        else {
            o->energy[i] -= e_send;
            if (recv >= 0) receive_package(o, recv);
            o->log_energy[i] += e_send;
        }
    }
    check_status(o, i);
}
static void set_levels(Oracle *o) {                        /* Network.py:37-66 */
    int N = o->N;
    int *f1 = malloc(sizeof(int) * (size_t)(N + 1) * 8), *f2 = malloc(sizeof(int) * (size_t)(N + 1) * 8);
    int n1 = 0, n2 = 0;
    for (int i = 0; i < N; i++) o->level[i] = -1;
    for (int k = 0; k < o->ndirect; k++) {
        int i = o->direct_list[k];
        if (o->status[i] == 1) { o->level[i] = 1; f1[n1++] = i; }
    }
    for (int t = 0; t < o->T; t++) o->targets_active[t] = 0;
    while (n1 > 0) {
        for (int a = 0; a < n1; a++) {
            int i = f1[a];
            for (int e = o->tgt_ptr[i]; e < o->tgt_ptr[i + 1]; e++) o->targets_active[o->tgt_idx[e]] = 1;
            for (int e = o->nbr_ptr[i]; e < o->nbr_ptr[i + 1]; e++) {
                int j = o->nbr_idx[e];
                if (o->status[j] == 1 && o->level[j] == -1) { f2[n2++] = j; o->level[j] = o->level[i] + 1; }
            }
        }
        int *t = f1; f1 = f2; f2 = t; n1 = n2; n2 = 0;
    }
    free(f1); free(f2);
}
static int check_targets(Oracle *o) {                      /* Network.py:84-85 */
    int m = 1;
    for (int t = 0; t < o->T; t++) if (o->targets_active[t] < m) m = o->targets_active[t];
    return o->T > 0 ? m : 1;
}

/* ------------------------------------------------------------------ chargers */
static void mc_check_status(MC *m) {                       /* MobileCharger.py:134-140 */
    if (m->energy <= m->threshold) { m->status = 0; m->energy = m->threshold; }
}
static double charge_rate(Oracle *o, MC *m, int node) {    /* alpha / (d + beta) ** 2 */
    double d = euclid(o->nx[node], o->ny[node], m->x, m->y);
    return m->alpha / pow(d + m->beta, 2.0);
}

static void update_reward(Oracle *o) {                     /* rl_env/WRSN.py:100-127 */
    int N = o->N, any = 0;
    for (int a = 0; a < o->M; a++)
        if (o->mc[a].status != 0 && o->mc[a].type_charging) any = 1;
    if (!any) return;                                      /* the priority vector has no other reader */
    double *p = malloc(sizeof(double) * N), *q = malloc(sizeof(double) * N);
    for (int i = 0; i < N; i++)
        p[i] = o->status[i] != 0 ? o->cs[i] / (o->energy[i] - o->threshold + o->eps_env) : 0.0;
    double mean = pairwise_sum(p, N) / N;
    for (int i = 0; i < N; i++) { double x = p[i] - mean; q[i] = x * x; }
    double sd = sqrt(pairwise_sum(q, N) / N);
    if (sd == 0) sd = o->eps_env;
    for (int i = 0; i < N; i++) p[i] = exp((p[i] - mean) / sd);
    double tot = pairwise_sum(p, N);
    if (tot == 0) tot = o->eps_env;
    for (int i = 0; i < N; i++) p[i] = p[i] / tot;
    for (int a = 0; a < o->M; a++) {
        MC *m = &o->mc[a];
        if (m->status == 0) continue;
        if (!m->type_charging) continue;
        double incentive = 0;
        for (int k = 0; k < m->nconn; k++) {
            int i = m->conn[k];
            if (o->status[i] == 1) {
                double rate = m->alpha / pow(euclid(o->nx[i], o->ny[i], m->x, m->y) + m->beta, 2.0);
                double e_no = fmin(o->energy[i] - o->cs[i], o->threshold);
                double e_with = fmax(o->energy[i] - o->cs[i] + rate, o->capacity);
                incentive += p[i] * (e_with - e_no) / (m->alpha / pow(m->beta, 2.0));
            }
        }
        o->excl[a] += incentive;
    }
    free(p); free(q);
}

/* ------------------------------------------------------------------ generator state machines */
static void resume(Oracle *o, int p) {
    Proc *P = &o->procs[p];
    int N = o->N;
    switch (P->kind) {
    case P_NETOP:                                          /* Network.operate */
        if (P->state == 0) {
            for (int i = 0; i < N; i++) new_proc(o, P_NODE, i, 0);
            new_proc(o, P_BS, 0, 0);
            P = &o->procs[p];
            wait_timeout(o, p, 1.0 / 10.0); P->state = 1;
        } else if (P->state == 1) {
            set_levels(o);
            o->alive = check_targets(o);
            wait_timeout(o, p, 9.0 * 1.0 / 10.0); P->state = 2;
        } else {
            if (o->alive == 0 || o->now >= o->max_time) { proc_finish(o, p); return; }
            wait_timeout(o, p, 1.0 / 10.0); P->state = 1;
        }
        return;
    case P_UR:                                             /* WRSN.update_reward */
        update_reward(o);
        wait_timeout(o, p, 1.0);
        return;
    case P_BS:                                             /* BaseStation.operate */
        if (P->state == 0) { o->probed_bs = 1; P->state = 1; }
        wait_timeout(o, p, 1.0);
        return;
    case P_NODE: {                                         /* Node.operate */
        int i = P->id;
        if (P->state == 0) {
            o->log_energy[i] = 0;
            wait_timeout(o, p, 1 * 0.5); P->state = 1;
        } else if (P->state == 1) {
            if (o->status[i] == 0) { proc_finish(o, p); return; }
            o->energy[i] = fmin(o->energy[i] + o->rr[i] * 1 * 0.5, o->capacity);
            /* random.random() < prob_gp with prob_gp == 1 is always true (checked at create) */
            for (int e = o->tgt_ptr[i]; e < o->tgt_ptr[i + 1]; e++) send_package(o, i);
            wait_timeout(o, p, 1 * 0.5); P->state = 2;
        } else {
            if (o->status[i] == 0) { proc_finish(o, p); return; }
            o->energy[i] = fmin(o->energy[i] + o->rr[i] * 1 * 0.5, o->capacity);
            int L = o->loglen[i];
            double *lb = o->logbuf + (size_t)i * 10;
            if (L < 10) {
                lb[L] = o->log_energy[i]; o->loglen[i] = L + 1;
                o->cs[i] = (o->cs[i] * L + o->log_energy[i]) / (L + 1);
            } else {
                o->cs[i] = (o->cs[i] * L - lb[0] + o->log_energy[i]) / L;
                memmove(lb, lb + 1, sizeof(double) * 9);
                lb[9] = o->log_energy[i];
            }
            o->log_energy[i] = 0;
            wait_timeout(o, p, 1 * 0.5); P->state = 1;
        }
        return;
    }
    case P_OPSTEP: {                                       /* MobileCharger.operate_step; d[0..2] = phy_action */
        MC *m = &o->mc[P->id];
        if (P->state == 0) {
            double dx = P->d[0], dy = P->d[1], ct = P->d[2];
            double used = euclid(dx, dy, m->x, m->y) * m->pm;
            double tmp = 0;
            for (int i = 0; i < N; i++) {
                double dis = euclid(dx, dy, o->nx[i], o->ny[i]);
                if (dis <= m->range && o->status[i] == 1) tmp += m->alpha / pow(dis + m->beta, 2.0);
            }
            used += tmp * ct;
            used += euclid(dx, dy, o->bsx, o->bsy) * m->pm;
            m->cpa[0] = dx; m->cpa[1] = dy; m->cpa[2] = ct;
            m->type_charging = 0;
            if (used > m->energy - m->threshold - m->capacity / 200.0) {
                int c = spawn_child(o, p, P_MOVE, P->id);
                o->procs[c].d[0] = o->bsx; o->procs[c].d[1] = o->bsy;
                o->procs[p].state = 1;
            } else {
                int c = spawn_child(o, p, P_MOVE, P->id);
                o->procs[c].d[0] = dx; o->procs[c].d[1] = dy;
                o->procs[p].state = 3;
            }
        } else if (P->state == 1) {
            spawn_child(o, p, P_RECHARGE, P->id);
            o->procs[p].state = 2;
        } else if (P->state == 2) {
            double dx = P->d[0], dy = P->d[1];
            int c = spawn_child(o, p, P_MOVE, P->id);
            o->procs[c].d[0] = dx; o->procs[c].d[1] = dy;
            o->procs[p].state = 3;
        } else if (P->state == 3) {
            double ct = P->d[2];
            m->type_charging = 1;
            int c = spawn_child(o, p, P_CHARGE, P->id);
            o->procs[c].d[0] = ct;
            o->procs[p].state = 4;
        } else {
            proc_finish(o, p);
        }
        return;
    }
    case P_MOVE: {                                         /* MobileCharger.move; d0,d1 dest; d2 moving_time; d3,d4 vec; d5 total; d6 span */
        MC *m = &o->mc[P->id];
        if (P->state == 0) {
            P->d[2] = euclid(P->d[0], P->d[1], m->x, m->y) / m->velocity;
            P->d[3] = P->d[0] - m->x; P->d[4] = P->d[1] - m->y;
            P->d[5] = P->d[2];
        } else if (P->state == 1) {                        /* back from move_step */
            P->d[2] -= P->d[6];
            mc_check_status(m);
        } else {                                           /* dead wait elapsed */
            proc_finish(o, p); return;
        }
        if (P->d[2] <= 0) { proc_finish(o, p); return; }
        if (m->status == 0) { wait_timeout(o, p, P->d[2]); P->state = 2; return; }
        P->d[2] = euclid(P->d[0], P->d[1], m->x, m->y) / m->velocity;
        double span = fmin(fmin(P->d[2], 1.0), (m->energy - m->threshold) / (m->pm * m->velocity));
        P->d[6] = span;
        double vx = P->d[3] / P->d[5] * span, vy = P->d[4] / P->d[5] * span;
        int c = spawn_child(o, p, P_MOVESTEP, o->procs[p].id);
        o->procs[c].d[0] = vx; o->procs[c].d[1] = vy; o->procs[c].d[2] = span;
        o->procs[p].state = 1;
        return;
    }
    case P_MOVESTEP: {                                     /* MobileCharger.move_step */
        MC *m = &o->mc[P->id];
        if (P->state == 0) { wait_timeout(o, p, P->d[2]); P->state = 1; return; }
        m->x = m->x + P->d[0]; m->y = m->y + P->d[1];
        m->energy -= m->pm * P->d[2] * m->velocity;
        proc_finish(o, p);
        return;
    }
    case P_RECHARGE: {                                     /* MobileCharger.recharge */
        MC *m = &o->mc[P->id];
        if (P->state == 0) {
            if (euclid(m->x, m->y, o->bsx, o->bsy) <= m->epsilon) { m->x = o->bsx; m->y = o->bsy; m->energy = m->capacity; }
            wait_timeout(o, p, 0.0); P->state = 1; return;
        }
        proc_finish(o, p);
        return;
    }
    case P_CHARGE: {                                       /* MobileCharger.charge; d0 = tmp, d1 = span */
        MC *m = &o->mc[P->id];
        if (P->state == 0) {
            m->charging_time = P->d[0];
            m->nconn = 0;
            for (int i = 0; i < N; i++)
                if (euclid(o->nx[i], o->ny[i], m->x, m->y) <= m->range) m->conn[m->nconn++] = i;
        } else if (P->state == 1) {
            P->d[0] -= P->d[1];
            m->charging_time = P->d[0];
            mc_check_status(m);
        } else { proc_finish(o, p); return; }
        if (P->d[0] == 0) { proc_finish(o, p); return; }
        if (m->status == 0) { m->cpa[2] = 0; wait_timeout(o, p, P->d[0]); P->state = 2; return; }
        double span = fmin(P->d[0], 1.0);
        if (m->charging_rate != 0) span = fmin(span, (m->energy - m->threshold) / m->charging_rate);
        P->d[1] = span;
        int c = spawn_child(o, p, P_CHARGESTEP, o->procs[p].id);
        o->procs[c].d[0] = span;
        o->procs[p].state = 1;
        return;
    }
    case P_CHARGESTEP: {                                   /* MobileCharger.charge_step + Node.charger_(dis)connection */
        MC *m = &o->mc[P->id];
        if (P->state == 0) {
            for (int k = 0; k < m->nconn; k++) {
                int i = m->conn[k];
                if (o->status[i] == 0) continue;
                double r = charge_rate(o, m, i);
                o->rr[i] += r; m->charging_rate += r;
            }
            wait_timeout(o, p, P->d[0]); P->state = 1; return;
        }
        double t = P->d[0];
        m->energy = m->energy - m->charging_rate * t;
        m->cpa[2] = fmax(0.0, m->cpa[2] - t);
        for (int k = 0; k < m->nconn; k++) {
            int i = m->conn[k];
            if (o->status[i] == 0) continue;
            double r = charge_rate(o, m, i);
            o->rr[i] -= r; m->charging_rate -= r;
        }
        m->charging_rate = 0;
        proc_finish(o, p);
        return;
    }
    }
}

/* one SimPy Environment.step() */
static void env_step(Oracle *o) {
    Ev e = heap_pop(o);
    o->now = e.t;
    o->nevents++;
    switch (e.type) {
    case EV_UNTIL: o->stop = 1; break;
    case EV_INIT: case EV_TIMEOUT: resume(o, e.idx); break;
    case EV_PROCDONE: {
        Proc *P = &o->procs[e.idx];
        int n = P->ncb, ty[CB_MAX], ix[CB_MAX];
        memcpy(ty, P->cb_type, sizeof(ty)); memcpy(ix, P->cb_idx, sizeof(ix));
        P->processed = 1; P->ncb = 0;
        int recyc = P->recyclable;
        for (int k = 0; k < n; k++) {
            if (ty[k] == CB_RESUME) resume(o, ix[k]);
            else if (ty[k] == CB_CHECK) cond_check(o, ix[k]);
        }
        if (recyc) { o->procs[e.idx].in_use = 0; o->freelist[o->nfree++] = e.idx; }
        break;
    }
    case EV_COND: {
        Cond *C = &o->conds[e.idx];
        int n = C->ncb, ty[CB_MAX], ix[CB_MAX];
        memcpy(ty, C->cb_type, sizeof(ty)); memcpy(ix, C->cb_idx, sizeof(ix));
        C->processed = 1; C->ncb = 0;
        for (int k = 0; k < n; k++) {
            if (ty[k] == CB_BUILD) cond_remove_checks(o, e.idx);
            else if (ty[k] == CB_CHECK) cond_check(o, ix[k]);
            else if (ty[k] == CB_STOP) { o->stop = 1; break; }
        }
        break;
    }
    }
}
static void run_loop(Oracle *o) {
    o->stop = 0;
    long long start = o->nevents;
    while (!o->stop) {
        if (o->hn == 0) { fprintf(stderr, "oracle: empty schedule\n"); abort(); }
        if (o->event_budget > 0 && o->nevents - start > o->event_budget) { o->budget_hit = 1; return; }
        env_step(o);
    }
}
static void run_until_time(Oracle *o, double at) {
    if (at <= o->now) return;
    schedule(o, EV_UNTIL, 0, URGENT, at - o->now);
    run_loop(o);
}
static void run_until_cond(Oracle *o, int c) {
    if (o->conds[c].processed) return;
    cond_add_cb(o, c, CB_STOP, 0);
    run_loop(o);
}

/* ------------------------------------------------------------------ build */
static void build_static(Oracle *o) {
    int N = o->N, T = o->T;
    o->nbr_ptr = calloc(N + 1, sizeof(int)); o->tgt_ptr = calloc(N + 1, sizeof(int));
    int ne = 0, nt = 0;
    for (int i = 0; i < N; i++) {
        for (int j = 0; j < N; j++) if (i != j && euclid(o->nx[j], o->ny[j], o->nx[i], o->ny[i]) <= o->com_range) ne++;
        for (int t = 0; t < T; t++) if (euclid(o->nx[i], o->ny[i], o->tx[t], o->ty[t]) <= o->sen_range) nt++;
    }
    o->nbr_idx = malloc(sizeof(int) * (ne + 1)); o->tgt_idx = malloc(sizeof(int) * (nt + 1));
    ne = nt = 0;
    o->direct = calloc(N, sizeof(int)); o->direct_list = malloc(sizeof(int) * (N + 1)); o->ndirect = 0;
    for (int i = 0; i < N; i++) {
        o->nbr_ptr[i] = ne; o->tgt_ptr[i] = nt;
        for (int j = 0; j < N; j++) if (i != j && euclid(o->nx[j], o->ny[j], o->nx[i], o->ny[i]) <= o->com_range) o->nbr_idx[ne++] = j;
        for (int t = 0; t < T; t++) if (euclid(o->nx[i], o->ny[i], o->tx[t], o->ty[t]) <= o->sen_range) o->tgt_idx[nt++] = t;
        if (euclid(o->bsx, o->bsy, o->nx[i], o->ny[i]) <= o->com_range) { o->direct[i] = 1; o->direct_list[o->ndirect++] = i; }
    }
    o->nbr_ptr[N] = ne; o->tgt_ptr[N] = nt;
    /* Network.__init__ frame / density, Network.py:16-27 */
    o->frame[0] = o->frame[1] = o->bsx; o->frame[2] = o->frame[3] = o->bsy;
    for (int i = 0; i < N; i++) {
        o->frame[0] = fmin(o->frame[0], o->nx[i]); o->frame[1] = fmax(o->frame[1], o->nx[i]);
        o->frame[2] = fmin(o->frame[2], o->ny[i]); o->frame[3] = fmax(o->frame[3], o->ny[i]);
    }
    o->nodes_density = N / ((o->frame[1] - o->frame[0]) * (o->frame[3] - o->frame[2]));
}

/* node_par: capacity, threshold, com_range, sen_range, prob_gp, package_size, er, et, efs, emp, max_time
   mc_par  : capacity, threshold, velocity, pm, charging_range, alpha, beta, epsilon */
Oracle *orc_create(int N, int T, const double *node_xy, const double *target_xy, const double *bs_xy,
                   const double *node_par, int M, const double *mc_par, int map_size, double warm_up) {
    Oracle *o = calloc(1, sizeof(Oracle));
    o->N = N; o->T = T; o->M = M; o->S = map_size; o->warm_up = warm_up;
    o->nx = malloc(sizeof(double) * N); o->ny = malloc(sizeof(double) * N);
    o->tx = malloc(sizeof(double) * (T + 1)); o->ty = malloc(sizeof(double) * (T + 1));
    for (int i = 0; i < N; i++) { o->nx[i] = node_xy[2 * i]; o->ny[i] = node_xy[2 * i + 1]; }
    for (int t = 0; t < T; t++) { o->tx[t] = target_xy[2 * t]; o->ty[t] = target_xy[2 * t + 1]; }
    o->bsx = bs_xy[0]; o->bsy = bs_xy[1];
    o->capacity = node_par[0]; o->threshold = node_par[1]; o->com_range = node_par[2]; o->sen_range = node_par[3];
    o->prob_gp = node_par[4]; o->package_size = node_par[5]; o->er = node_par[6]; o->et = node_par[7];
    o->efs = node_par[8]; o->emp = node_par[9]; o->max_time = node_par[10];
    if (o->prob_gp < 1.0) { fprintf(stderr, "oracle: prob_gp < 1 needs MT19937 parity (Q12); unsupported\n"); free(o); return NULL; }
    if (M > 0) memcpy(o->mcpar, mc_par, sizeof(double) * 8);
    o->eps_env = 1e-9;
    build_static(o);
    o->energy = malloc(sizeof(double) * N); o->rr = malloc(sizeof(double) * N); o->cs = malloc(sizeof(double) * N);
    o->log_energy = malloc(sizeof(double) * N); o->logbuf = malloc(sizeof(double) * N * 10);
    o->loglen = malloc(sizeof(int) * N); o->status = malloc(sizeof(int) * N); o->level = malloc(sizeof(int) * N);
    o->targets_active = malloc(T + 1);
    o->hcap = 1024; o->heap = malloc(sizeof(Ev) * o->hcap);
    o->pcap = 1024; o->procs = malloc(sizeof(Proc) * o->pcap); o->freelist = malloc(sizeof(int) * o->pcap);
    o->ccap = 1024; o->conds = malloc(sizeof(Cond) * o->ccap);
    o->mc = calloc(M > 0 ? M : 1, sizeof(MC));
    for (int a = 0; a < M; a++) o->mc[a].conn = malloc(sizeof(int) * (N + 1));
    o->agent_proc = malloc(sizeof(int) * (M + 1)); o->excl = calloc(M + 1, sizeof(double));
    o->prev_fit_min = calloc(M + 1, sizeof(double)); o->agents_action = calloc(3 * (M + 1), sizeof(double));
    return o;
}
void orc_destroy(Oracle *o) {
    if (!o) return;
    free(o->nx); free(o->ny); free(o->tx); free(o->ty);
    free(o->nbr_ptr); free(o->nbr_idx); free(o->tgt_ptr); free(o->tgt_idx); free(o->direct); free(o->direct_list);
    free(o->energy); free(o->rr); free(o->cs); free(o->log_energy); free(o->logbuf); free(o->loglen);
    free(o->status); free(o->level); free(o->targets_active); free(o->heap); free(o->procs); free(o->freelist);
    free(o->conds);
    for (int a = 0; a < o->M; a++) free(o->mc[a].conn);
    free(o->mc); free(o->agent_proc); free(o->excl); free(o->prev_fit_min); free(o->agents_action);
    free(o);
}

/* NetworkIO.makeNetwork + Node.__init__ + simpy.Environment() */
static void make_network(Oracle *o) {
    int N = o->N;
    for (int i = 0; i < N; i++) {
        o->energy[i] = o->capacity; o->rr[i] = 0; o->cs[i] = 0; o->log_energy[i] = 0; o->loglen[i] = 0;
        o->status[i] = 1; o->level[i] = -1;
        check_status(o, i);
    }
    for (int t = 0; t < o->T; t++) o->targets_active[t] = 1;
    o->alive = 1;
    o->hn = 0; o->eid = 0; o->now = 0; o->nprocs = 0; o->nfree = 0; o->nconds = 0; o->stop = 0; o->budget_hit = 0;
}

/* runner/test_network.py logic: only Network.operate, no chargers, no reward process */
void orc_start_network_only(Oracle *o) {
    make_network(o);
    o->netop_proc = new_proc(o, P_NETOP, 0, 0);
}
void orc_run_until(Oracle *o, double t) { run_until_time(o, t); }
int orc_netop_done(Oracle *o) { return o->procs[o->netop_proc].processed; }

/* ------------------------------------------------------------------ WRSN layer */
static void down_mapping(Oracle *o, double x, double y, double *out) {       /* WRSN.py:86-88 */
    out[0] = (x - o->frame[0]) / (o->frame[1] - o->frame[0]);
    out[1] = (y - o->frame[2]) / (o->frame[3] - o->frame[2]);
}
static double gfunc(double x, double h) { return exp(x * x / (-2 * pow(h, 2.0))); }  /* WRSN.py:16-18 */

void orc_get_state(Oracle *o, int agent_id, double *out) {                   /* WRSN.py:130-186 */
    int S = o->S, N = o->N;
    MC *ag = &o->mc[agent_id];
    double unit = 1.0 / S;
    double *c = malloc(sizeof(double) * S), *gx = malloc(sizeof(double) * S), *gy = malloc(sizeof(double) * S);
    {   /* np.arange(unit/2, 1.0, unit): numpy fills a[i] = start + i*delta with delta = (start+step) - start */
        double start = unit / 2, delta = (start + unit) - start;
        for (int i = 0; i < S; i++) c[i] = start + i * delta;
    }
    size_t SS = (size_t)S * S;
    memset(out, 0, sizeof(double) * 4 * SS);
    double W = o->frame[1] - o->frame[0], H = o->frame[3] - o->frame[2];
    double co[2];
    for (int n = 0; n < N; n++) {
        if (o->status[n] == 0) continue;
        down_mapping(o, o->nx[n], o->ny[n], co);
        double hX = ag->range / W, hY = ag->range / H;
        double w = (o->cs[n] / (ag->alpha / pow(ag->beta, 2.0))) / ((o->energy[n] - o->threshold) / (o->capacity - o->threshold));
        for (int i = 0; i < S; i++) { gx[i] = gfunc(c[i] - co[0], hX); gy[i] = gfunc(c[i] - co[1], hY); }
        for (int i = 0; i < S; i++) { double wi = w * gx[i]; for (int j = 0; j < S; j++) out[(size_t)i * S + j] += wi * gy[j]; }
    }
    {
        down_mapping(o, ag->x, ag->y, co);
        double tmp = fmin(H, W);
        double hX = 0.5 * tmp / W, hY = 0.5 * tmp / H;
        double w = ag->energy / ag->capacity;
        for (int i = 0; i < S; i++) { gx[i] = gfunc(c[i] - co[0], hX); gy[i] = gfunc(c[i] - co[1], hY); }
        for (int i = 0; i < S; i++) { double wi = w * gx[i]; for (int j = 0; j < S; j++) out[SS + (size_t)i * S + j] += wi * gy[j]; }
    }
    for (int a = 0; a < o->M; a++) {
        MC *an = &o->mc[a];
        if (a == agent_id) continue;
        if (!an->type_charging) continue;
        down_mapping(o, an->cpa[0], an->cpa[1], co);
        double hX = an->range / W, hY = an->range / H;
        double w = an->cpa[2] / o->charging_time_max;
        for (int i = 0; i < S; i++) { gx[i] = gfunc(c[i] - co[0], hX); gy[i] = gfunc(c[i] - co[1], hY); }
        for (int i = 0; i < S; i++) { double wi = w * gx[i]; for (int j = 0; j < S; j++) out[2 * SS + (size_t)i * S + j] += wi * gy[j]; }
    }
    for (int a = 0; a < o->M; a++) {
        MC *an = &o->mc[a];
        if (a == agent_id) continue;
        if (an->type_charging) continue;
        down_mapping(o, an->cpa[0], an->cpa[1], co);
        double hX = an->range / W, hY = an->range / H;
        double w = euclid(an->x, an->y, an->cpa[0], ag->cpa[1]) / an->velocity;      /* Q5: observer's y */
        for (int i = 0; i < S; i++) { gx[i] = gfunc(c[i] - co[0], hX); gy[i] = gfunc(c[i] - co[1], hY); }
        for (int i = 0; i < S; i++) for (int j = 0; j < S; j++) out[3 * SS + (size_t)i * S + j] += gx[i] * gy[j] * w / o->moving_time_max;
    }
    free(c); free(gx); free(gy);
}

/* get_network_fitness, WRSN.py:188-220: returns min over targets (what get_reward uses); per-target values to `out` if non-NULL */
double orc_fitness(Oracle *o, double *out) {
    int N = o->N, T = o->T;
    double *node_t = malloc(sizeof(double) * N);
    int *t1 = malloc(sizeof(int) * ((size_t)N * 16 + 16)), *t2 = malloc(sizeof(int) * ((size_t)N * 16 + 16));
    int n1 = 0, n2 = 0;
    for (int i = 0; i < N; i++) node_t[i] = -1;
    for (int k = 0; k < o->ndirect; k++) {
        int i = o->direct_list[k];
        if (o->status[i] == 1) {
            t1[n1++] = i;
            node_t[i] = (o->cs[i] == 0) ? INFINITY : (o->energy[i] - o->threshold) / o->cs[i];
        }
    }
    while (n1 > 0) {
        for (int a = 0; a < n1; a++) {
            int i = t1[a];
            for (int e = o->nbr_ptr[i]; e < o->nbr_ptr[i + 1]; e++) {
                int j = o->nbr_idx[e];
                if (o->status[j] != 1) continue;
                double lt = (o->cs[j] == 0) ? INFINITY : (o->energy[j] - o->threshold) / o->cs[j];
                if (node_t[j] == -1 || (node_t[i] > node_t[j] && lt > node_t[j])) {
                    t2[n2++] = j;
                    node_t[j] = fmin(lt, node_t[i]);
                }
            }
        }
        int *t = t1; t1 = t2; t2 = t; n1 = n2; n2 = 0;
    }
    double mn = INFINITY;
    double *tt = malloc(sizeof(double) * (T + 1));
    for (int t = 0; t < T; t++) tt[t] = 0;
    for (int i = 0; i < N; i++)
        for (int e = o->tgt_ptr[i]; e < o->tgt_ptr[i + 1]; e++) {
            int t = o->tgt_idx[e];
            if (node_t[i] > tt[t]) tt[t] = node_t[i];
        }
    for (int t = 0; t < T; t++) { if (tt[t] < mn) mn = tt[t]; if (out) out[t] = tt[t]; }
    free(node_t); free(t1); free(t2); free(tt);
    return mn;
}

static int scan_decider(Oracle *o) {                                         /* WRSN.py:321-322 */
    for (int a = 0; a < o->M; a++) {
        MC *m = &o->mc[a];
        if (euclid(m->x, m->y, m->cpa[0], m->cpa[1]) < o->eps_env && m->cpa[2] == 0) return a;
    }
    return -1;
}

/* request layout (doubles): [0] agent_id (-1 None, -2 implicit None/Q7), [1] terminal, [2] reward, [3..5] action, [6] now, [7] budget_hit */
void orc_reset(Oracle *o, double *req, double *state_out) {                  /* WRSN.py:41-83 */
    make_network(o);
    o->netop_proc = new_proc(o, P_NETOP, 0, 0);
    o->ur_proc = new_proc(o, P_UR, 0, 0);
    o->netp_cond = new_cond(o, 1, OP_PROC, o->netop_proc, OP_PROC, o->ur_proc);
    for (int a = 0; a < o->M; a++) {
        MC *m = &o->mc[a];
        int *conn = m->conn;
        memset(m, 0, sizeof(*m)); m->conn = conn;
        m->x = o->bsx; m->y = o->bsy;
        m->capacity = o->mcpar[0]; m->threshold = o->mcpar[1]; m->velocity = o->mcpar[2]; m->pm = o->mcpar[3];
        m->range = o->mcpar[4]; m->alpha = o->mcpar[5]; m->beta = o->mcpar[6]; m->epsilon = o->mcpar[7];
        m->energy = m->capacity; m->status = 1; m->charging_rate = 0;
        mc_check_status(m);
        m->type_charging = 0; m->nconn = 0;
        m->cpa[0] = o->bsx; m->cpa[1] = o->bsy; m->cpa[2] = 0;
    }
    o->moving_time_max = euclid(o->frame[0], o->frame[2], o->frame[1], o->frame[3]) / o->mcpar[2];
    o->charging_time_max = (o->capacity - o->threshold) / (o->mcpar[5] / pow(o->mcpar[6], 2.0));
    o->avg_nodes_agent = o->nodes_density * M_PI * pow(o->mcpar[4], 2.0);
    run_until_time(o, o->warm_up);
    int term = o->alive == 1 ? 0 : 1;
    double fit = orc_fitness(o, NULL);
    double dm[2];
    for (int a = 0; a < o->M; a++) {
        down_mapping(o, o->bsx, o->bsy, dm);
        o->agents_action[3 * a] = dm[0]; o->agents_action[3 * a + 1] = dm[1]; o->agents_action[3 * a + 2] = 0;
        int p = new_proc(o, P_OPSTEP, a, 0);
        o->procs[p].d[0] = o->mc[a].cpa[0]; o->procs[p].d[1] = o->mc[a].cpa[1]; o->procs[p].d[2] = o->mc[a].cpa[2];
        o->agent_proc[a] = p;
        o->prev_fit_min[a] = fit;
        o->excl[a] = 0.0;
    }
    int id = scan_decider(o);
    req[0] = id; req[1] = term; req[2] = id >= 0 ? 0.0 : NAN; req[6] = o->now; req[7] = 0;
    for (int k = 0; k < 3; k++) req[3 + k] = id >= 0 ? o->agents_action[3 * id + k] : NAN;
    if (id >= 0 && state_out) orc_get_state(o, id, state_out);
}

void orc_step(Oracle *o, int agent_id, const double *input_action, double *req, double *state_out, double *prev_state_out) {
    if (agent_id >= 0) {                                                     /* WRSN.py:290-305 */
        double act[3], phy[3];
        for (int k = 0; k < 3; k++) act[k] = fmin(fmax(input_action[k], 0.0), 1.0);
        for (int k = 0; k < 3; k++) o->agents_action[3 * agent_id + k] = act[k];
        phy[0] = act[0] * (o->frame[1] - o->frame[0]) + o->frame[0];
        phy[1] = act[1] * (o->frame[3] - o->frame[2]) + o->frame[2];
        phy[2] = o->charging_time_max * act[2];
        int p = new_proc(o, P_OPSTEP, agent_id, 0);
        o->procs[p].d[0] = phy[0]; o->procs[p].d[1] = phy[1]; o->procs[p].d[2] = phy[2];
        o->agent_proc[agent_id] = p;
        if (prev_state_out) orc_get_state(o, agent_id, prev_state_out);
        o->prev_fit_min[agent_id] = orc_fitness(o, NULL);
        o->excl[agent_id] = 0;
    }
    int gt = OP_COND, gi = o->netp_cond, watched = 0;                        /* WRSN.py:307-311 */
    for (int a = 0; a < o->M; a++)
        if (o->mc[a].status != 0) { gi = new_cond(o, 0, gt, gi, OP_PROC, o->agent_proc[a]); gt = OP_COND; watched++; }
    o->budget_hit = 0;
    if (watched == 0) {
        /* every charger dead: the reference spins forever (Q1); report it instead */
        req[0] = -1; req[1] = (o->alive == 0); req[2] = NAN; req[3] = req[4] = req[5] = NAN; req[6] = o->now; req[7] = 1;
        o->budget_hit = 1;
        return;
    }
    run_until_cond(o, gi);
    req[6] = o->now; req[7] = o->budget_hit;
    if (o->alive == 0) { req[0] = -1; req[1] = 1; req[2] = NAN; req[3] = req[4] = req[5] = NAN; return; }
    int id = scan_decider(o);
    if (id < 0) { req[0] = -2; req[1] = 0; req[2] = NAN; req[3] = req[4] = req[5] = NAN; return; }   /* Q7 */
    double fit = orc_fitness(o, NULL);                                       /* get_reward, WRSN.py:222-227 */
    double term_all = fit - o->prev_fit_min[id];
    double term_excl = o->excl[id] / o->avg_nodes_agent;
    req[0] = id; req[1] = 0;
    req[2] = (term_all * 0.8 + 0.2 * term_excl) / (o->charging_time_max + o->moving_time_max);
    for (int k = 0; k < 3; k++) req[3 + k] = o->agents_action[3 * id + k];
    if (state_out) orc_get_state(o, id, state_out);
}

/* ------------------------------------------------------------------ accessors */
double orc_now(Oracle *o) { return o->now; }
int orc_alive(Oracle *o) { return o->alive; }
void orc_set_event_budget(Oracle *o, long long n) { o->event_budget = n; }
long long orc_nevents(Oracle *o) { return o->nevents; }
void orc_get_nodes(Oracle *o, double *energy, double *cs, double *rr, double *log_energy, int *status, int *level) {
    for (int i = 0; i < o->N; i++) {
        if (energy) energy[i] = o->energy[i];
        if (cs) cs[i] = o->cs[i];
        if (rr) rr[i] = o->rr[i];
        if (log_energy) log_energy[i] = o->log_energy[i];
        if (status) status[i] = o->status[i];
        if (level) level[i] = o->level[i];
    }
}
void orc_get_targets_active(Oracle *o, unsigned char *out) { memcpy(out, o->targets_active, o->T); }
/* per charger: x, y, energy, status, cpa0, cpa1, cpa2, type_charging, nconn, excl */
void orc_get_mc(Oracle *o, double *out) {
    for (int a = 0; a < o->M; a++) {
        MC *m = &o->mc[a];
        double *r = out + 10 * a;
        r[0] = m->x; r[1] = m->y; r[2] = m->energy; r[3] = m->status; r[4] = m->cpa[0]; r[5] = m->cpa[1]; r[6] = m->cpa[2];
        r[7] = m->type_charging; r[8] = m->nconn; r[9] = o->excl[a];
    }
}
/* frame[4], moving_time_max, charging_time_max, avg_nodes_agent, nodes_density */
void orc_get_consts(Oracle *o, double *out) {
    for (int k = 0; k < 4; k++) out[k] = o->frame[k];
    out[4] = o->moving_time_max; out[5] = o->charging_time_max; out[6] = o->avg_nodes_agent; out[7] = o->nodes_density;
}
int orc_get_static(Oracle *o, int *nbr_ptr, int *nbr_idx, int *tgt_ptr, int *tgt_idx, int *direct) {
    if (nbr_ptr) memcpy(nbr_ptr, o->nbr_ptr, sizeof(int) * (o->N + 1));
    if (nbr_idx) memcpy(nbr_idx, o->nbr_idx, sizeof(int) * o->nbr_ptr[o->N]);
    if (tgt_ptr) memcpy(tgt_ptr, o->tgt_ptr, sizeof(int) * (o->N + 1));
    if (tgt_idx) memcpy(tgt_idx, o->tgt_idx, sizeof(int) * o->tgt_ptr[o->N]);
    if (direct) memcpy(direct, o->direct, sizeof(int) * o->N);
    return o->nbr_ptr[o->N];
}
/* test-only: overwrite node i's energy (the tests place energies on binade edges in both simulators) */
void orc_set_node_energy(Oracle *o, int i, double e) { o->energy[i] = e; }
void orc_set_mc_energy(Oracle *o, int a, double e) { o->mc[a].energy = e; }
