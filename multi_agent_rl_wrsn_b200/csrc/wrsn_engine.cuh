/*
 * wrsn_engine.cuh — per-environment simulation engine of the batched WRSN simulator.
 *
 * One CTA advances one environment.  The environment's working set (node rows, event clock,
 * charger records) lives in shared memory for the duration of a launch; thread 0 (the
 * "leader") owns the discrete-event clock, every thread owns the nodes  i = tid, tid+G, ...
 *
 * What is reproduced (reference file:line):
 *   Network.operate / setLevels / check_targets        physical_env/network/Network.py:37-85
 *   Node.operate / send_package / receive_package /
 *   find_receiver / check_status / charger_(dis)connection   physical_env/network/Node.py:45-151
 *   MobileCharger.operate_step / move / move_step /
 *   recharge / charge / charge_step / checkStatus       physical_env/mc/MobileCharger.py:34-140
 *   WRSN.reset / step / update_reward / get_network_fitness / get_reward / translate
 *                                                       rl_env/WRSN.py:41-127,188-227,289-330
 *   and, underneath, SimPy 4.0.1's ordering rule (time, priority, insertion counter) with URGENT
 *   process starts and NORMAL timeouts / completions / conditions, and the nested AnyOf chain of
 *   WRSN.step with its check-callback removal.
 *
 * How it differs from the reference's shape (B200-first, not a translation):
 *   - the N per-node generator processes collapse into ONE block event per half second, executed
 *     node-parallel;
 *   - the per-packet multi-hop recursion collapses into a routing tree (receiver per node) with
 *     per-node relay counts, recomputed only after a death; a node's tick is then the ordered
 *     replay of ITS OWN fp64 operation sequence (relayed packets of lower ids, top-up, own packets,
 *     relayed packets of higher ids), evaluated in closed form when it stays inside one binade
 *     (sub_chain below) — bit-identical to the sequential reference;
 *   - a tick in which some node might die takes an exact serial path (leader thread);
 *   - every charger generator tree is one flat state machine ("process slot") with one pending
 *     event.
 *
 * The same source compiles for the device (nvcc, sm_100a) and, with WRSN_HOST_EMU, as plain
 * single-lane C++ used ONLY by tests/ to check the event logic on a box without a GPU.
 */
/* NOTE: no include guard — this file is included once per group-size specialisation, inside a namespace, after
 * wrsn_layout.h, with WRSN_GFIX defined: 32 = one warp per environment (every barrier is a __syncwarp, every
 * reduction a shuffle tree), 0 = any multiple of 32 threads (__syncthreads), 1 = the tests' single-lane host build. */
#ifndef WRSN_GFIX
#error "define WRSN_GFIX before including wrsn_engine.cuh"
#endif

#undef WRSN_D
#undef WRSN_DI
#undef WRSN_NOINLINE
#undef WRSN_GSZ
#if defined(WRSN_HOST_EMU)
#define WRSN_D static inline
#define WRSN_DI static inline
#define WRSN_NOINLINE static
#else
#define WRSN_D __device__ static
#define WRSN_DI __device__ __forceinline__ static      /* takes the register-resident clock by reference: must inline */
#define WRSN_NOINLINE __device__ __noinline__ static   /* cold or shared code kept out of the hot loop's I-cache footprint */
#endif
#if WRSN_GFIX
#define WRSN_GSZ(c) WRSN_GFIX
#else
#define WRSN_GSZ(c) ((c).G)
#endif
/* Who stores the replicated scalar state (clock, charger records)?  Every thread computes it redundantly.  With one
 * warp per environment ALL lanes store (same value, same address, one converged instruction: no branch, no
 * divergence at the following barrier); with several warps only thread 0 does (a second warp could otherwise read
 * a value the first one has already replaced). */
#undef WRSN_LEAD
#if WRSN_GFIX == 32
#define WRSN_LEAD(c) true
#else
#define WRSN_LEAD(c) ((c).tid == 0)
#endif

#undef WRSN_LDG                                     /* read-only scenario data (CSR graph, flags): the non-coherent L1 path */
#if defined(WRSN_HOST_EMU)
#define WRSN_LDG(p) (*(p))
#else
#define WRSN_LDG(p) __ldg(p)
#endif

#undef WRSN_SMEM_BASE
#if defined(WRSN_HOST_EMU)
#define WRSN_SMEM_BASE wrsn_smem_host              /* set per environment by the emulation driver */
#else
#define WRSN_SMEM_BASE (reinterpret_cast<char *>(wrsn_smem_u4))
#endif

/* cycle counters of the profiling builds (tools/build_prof.sh): -DWRSN_PROF=1 counts serial ticks / batches / BFS / fitness,
 * -DWRSN_PROF=2 charger events / lazy replays / event-path grid events / the slot scan, into hdr[WRSN_H_PROF1..4] */
#undef WRSN_PROF_BEGIN
#undef WRSN_PROF_END
#undef WRSN_PROFB_BEGIN
#undef WRSN_PROFB_END
#if defined(WRSN_PROF) && !defined(WRSN_HOST_EMU)
#define WRSN_PROF_T0_() const long long prof_t0_ = clock64()
#define WRSN_PROF_ADD_(c, slot) do { if ((c).tid == 0) (c).hdr[slot] += (double)(clock64() - prof_t0_); } while (0)
#else
#define WRSN_PROF_T0_() do { } while (0)
#define WRSN_PROF_ADD_(c, slot) do { } while (0)
#endif
#if defined(WRSN_PROF) && WRSN_PROF == 1
#define WRSN_PROF_BEGIN() WRSN_PROF_T0_()
#define WRSN_PROF_END(c, slot) WRSN_PROF_ADD_(c, slot)
#else
#define WRSN_PROF_BEGIN() do { } while (0)
#define WRSN_PROF_END(c, slot) do { } while (0)
#endif
#if defined(WRSN_PROF) && WRSN_PROF == 2
#define WRSN_PROFB_BEGIN() WRSN_PROF_T0_()
#define WRSN_PROFB_END(c, slot) WRSN_PROF_ADD_(c, slot)
#else
#define WRSN_PROFB_BEGIN() do { } while (0)
#define WRSN_PROFB_END(c, slot) do { } while (0)
#endif
#undef WRSN_PROFC_BEGIN
#undef WRSN_PROFC_END
#if defined(WRSN_PROF) && WRSN_PROF == 3                /* inside the batches: pass 1 / all-at-once pass 2 / cycle loop / update_reward */
#define WRSN_PROFC_BEGIN(v) const long long v = clock64()
#define WRSN_PROFC_END(c, slot, v) do { if ((c).tid == 0) (c).hdr[slot] += (double)(clock64() - v); } while (0)
#else
#define WRSN_PROFC_BEGIN(v) do { } while (0)
#define WRSN_PROFC_END(c, slot, v) do { } while (0)
#endif

/* ------------------------------------------------------------------ context
 * The environment's shared-memory image is addressed as 32-bit offsets from the CTA's dynamic shared memory (SArr):
 * the compiler then knows the address space (LDS / STS with immediate offsets instead of generic 64-bit loads), the
 * context stays small, and nothing has to be re-derived from 64-bit pointers in the hot loop. */
#undef WRSN_M
#if defined(WRSN_HOST_EMU)
#define WRSN_M inline
#else
#define WRSN_M __device__ __forceinline__
#endif
template <typename T>
struct SArr {
    uint32_t off;
    WRSN_M T *ptr() const { return reinterpret_cast<T *>(WRSN_SMEM_BASE + off); }
    WRSN_M operator T *() const { return ptr(); }
    template <typename I> WRSN_M T &operator[](I i) const { return ptr()[i]; }
};

struct Ctx {
    int tid, G;
    SArr<double> spec;                               /* [WRSN_SPEC_MAX][WRSN_SPEC_LEN] irregular nodes of the current batch.  First: every
                                                        other field then sits at the offset at which ptxas allocates the cold entry
                                                        points (fitness, BFS) without extra registers (-Xptxas -v) */
    int N, T, M, W, Tw, Npad, n_slot, scr_len;
    /* shared-memory image */
    SArr<double> hdr, mc, proc;
    SArr<double> energy, rr, cs, esend, logc;
    SArr<uint16_t> nbef, naft, own;
    SArr<int16_t> level, parent;
    SArr<uint8_t> status;
    SArr<uint32_t> tact, conn;
    SArr<double> scr0, scr1;
    SArr<int> bcast;
    SArr<double> red;
    SArr<double> par;                                /* scenario constants, copied next to the state */
    SArr<double> pairs;                              /* see wrsn_layout.h: s_pairs */
    SArr<double> exptab;                             /* 2^(j/64), j = 0..63 (wrsn_exp_b) */
    /* global, per environment */
    double *logtick, *ring;
    char *gscratch;
    /* global, per scenario */
    const double *nx, *ny, *bs_esend, *nbr_dist, *nbr_esend;
    const int32_t *nbr_ptr, *tgt_ptr, *nbr_idx, *tgt_idx;
    const uint8_t *direct;
};

enum { WRSN_URGENT = 0, WRSN_NORMAL = 1 };
enum { K_NONE = 0, K_NET, K_UR, K_NODES, K_UNTIL, K_SLOT, K_COND };
enum {   /* program counter of a charger process slot */
    PC_OP_INIT = 1, PC_MOVE_INIT, PC_MS_INIT, PC_MS_FIRE, PC_MS_DONE, PC_MOVE_DEADWAIT, PC_MOVE_DONE,
    PC_RC_INIT, PC_RC_FIRE, PC_RC_DONE, PC_CH_INIT, PC_CS_INIT, PC_CS_FIRE, PC_CS_DONE, PC_CH_DEADWAIT,
    PC_CH_DONE, PC_OP_DONE
};

WRSN_D void ctx_bind(Ctx &c, const wrsn_dims &d, const WrsnLayout &L, const char *scen_row, char *state_row, int tid, int G) {
    c.tid = tid; c.G = G;
    {   /* the scenario's own counts (d.N / d.T are the batch's largest), read from the GLOBAL row: the shared copy below is only
           visible after the caller's first barrier */
        const double *gpar = (const double *)(scen_row + L.soff[WRSN_S_PAR]);
        c.N = (int)gpar[WRSN_P_NNODES]; c.T = (int)gpar[WRSN_P_NTARGETS];
    }
    c.M = d.M; c.W = d.W; c.Tw = d.Tw; c.Npad = d.Npad; c.n_slot = d.n_slot;
    c.scr_len = L.scr_len;
    c.hdr.off = (uint32_t)L.off[WRSN_F_HDR]; c.mc.off = (uint32_t)L.off[WRSN_F_MC]; c.proc.off = (uint32_t)L.off[WRSN_F_PROC];
    c.energy.off = (uint32_t)L.off[WRSN_F_ENERGY]; c.rr.off = (uint32_t)L.off[WRSN_F_RR]; c.cs.off = (uint32_t)L.off[WRSN_F_CS];
    c.esend.off = (uint32_t)L.off[WRSN_F_ESEND]; c.logc.off = (uint32_t)L.off[WRSN_F_LOGC];
    c.nbef.off = (uint32_t)L.off[WRSN_F_NBEF]; c.naft.off = (uint32_t)L.off[WRSN_F_NAFT];
    c.level.off = (uint32_t)L.off[WRSN_F_LEVEL]; c.parent.off = (uint32_t)L.off[WRSN_F_PARENT];
    c.status.off = (uint32_t)L.off[WRSN_F_STATUS]; c.tact.off = (uint32_t)L.off[WRSN_F_TACT]; c.conn.off = (uint32_t)L.off[WRSN_F_CONN];
    c.own.off = (uint32_t)L.s_own; c.scr0.off = (uint32_t)L.s_scr0; c.scr1.off = (uint32_t)L.s_scr1;
    c.bcast.off = (uint32_t)L.s_bcast; c.red.off = (uint32_t)L.s_red; c.par.off = (uint32_t)L.s_par; c.spec.off = (uint32_t)L.s_spec; c.exptab.off = (uint32_t)L.s_exptab; c.pairs.off = (uint32_t)L.s_pairs;
    c.logtick = (double *)(state_row + L.off[WRSN_F_LOGTICK]);
    c.ring = (double *)(state_row + L.off[WRSN_F_RING]);
    c.gscratch = state_row + L.off[WRSN_F_SCRATCH];
    {
        const double *gpar = (const double *)(scen_row + L.soff[WRSN_S_PAR]);
        for (int k = tid; k < WRSN_P_LEN; k += G) c.par[k] = gpar[k];   /* visible after the caller's first barrier */
#if !defined(WRSN_HOST_EMU)
        for (int k = tid; k < 64; k += G) c.exptab[k] = wrsn_exp2_tab[k];
#endif
    }
    c.nx = (const double *)(scen_row + L.soff[WRSN_S_NX]);
    c.ny = (const double *)(scen_row + L.soff[WRSN_S_NY]);
    c.bs_esend = (const double *)(scen_row + L.soff[WRSN_S_BS_ESEND]);
    c.nbr_dist = (const double *)(scen_row + L.soff[WRSN_S_NBR_DIST]);
    c.nbr_esend = (const double *)(scen_row + L.soff[WRSN_S_NBR_ESEND]);
    c.nbr_ptr = (const int32_t *)(scen_row + L.soff[WRSN_S_NBR_PTR]);
    c.tgt_ptr = (const int32_t *)(scen_row + L.soff[WRSN_S_TGT_PTR]);
    c.nbr_idx = (const int32_t *)(scen_row + L.soff[WRSN_S_NBR_IDX]);
    c.tgt_idx = (const int32_t *)(scen_row + L.soff[WRSN_S_TGT_IDX]);
    c.direct = (const uint8_t *)(scen_row + L.soff[WRSN_S_DIRECT]);
}

/* the targets of word w of a target bitmask: Tw comes from the batch's largest scenario, so the trailing words of a smaller
 * scenario hold no target (empty mask: neither active nor dead) */
WRSN_DI uint32_t tact_word_mask(const Ctx &c, int w) {
    const int bits = c.T - 32 * w;
    return bits >= 32 ? 0xffffffffu : (bits <= 0 ? 0u : ((1u << bits) - 1u));
}

/* 32-bit shared-memory addressing for the hot loop: on the device an address is the byte offset inside the CTA's shared
 * window (ld.shared / st.shared with a register address: no generic pointers, nothing to re-derive inside the loop); in
 * the host emulation it is the offset from the environment's image. */
#if !defined(WRSN_HOST_EMU)
typedef uint32_t saddr_t;
WRSN_DI saddr_t saddr_of(const void *p) { return (saddr_t)__cvta_generic_to_shared(p); }
WRSN_DI double lds64(saddr_t a) { double v; asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a)); return v; }
WRSN_DI void sts64(saddr_t a, double v) { asm volatile("st.shared.f64 [%0], %1;" :: "r"(a), "d"(v) : "memory"); }
#else
typedef size_t saddr_t;
WRSN_DI saddr_t saddr_of(const void *p) { return (saddr_t)((const char *)p - WRSN_SMEM_BASE); }
WRSN_DI double lds64(saddr_t a) { return *(const double *)(WRSN_SMEM_BASE + a); }
WRSN_DI void sts64(saddr_t a, double v) { *(double *)(WRSN_SMEM_BASE + a) = v; }
#endif

/* ------------------------------------------------------------------ group primitives */
WRSN_D void gsync(const Ctx &c) {
#if defined(WRSN_HOST_EMU)
    (void)c;
#elif WRSN_GFIX == 32
    (void)c; __syncwarp();
#else
    (void)c; __syncthreads();
#endif
}

#if !defined(WRSN_HOST_EMU)
WRSN_NOINLINE double warp_sum(double v) {            /* one copy, five unrolled shuffle steps (called once per reduction) */
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
WRSN_NOINLINE double warp_min(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
#endif

WRSN_D double red_sum(const Ctx &c, double v) {
#if defined(WRSN_HOST_EMU)
    (void)c; return v;
#elif WRSN_GFIX == 32
    (void)c; return warp_sum(v);
#else
    v = warp_sum(v);
    __syncthreads();
    if ((c.tid & 31) == 0) c.red[c.tid >> 5] = v;
    __syncthreads();
    double s = 0.0;
    for (int k = 0; k < (c.G >> 5); k++) s += c.red[k];
    return s;
#endif
}
WRSN_D double red_min(const Ctx &c, double v) {
#if defined(WRSN_HOST_EMU)
    (void)c; return v;
#elif WRSN_GFIX == 32
    (void)c; return warp_min(v);
#else
    v = warp_min(v);
    __syncthreads();
    if ((c.tid & 31) == 0) c.red[c.tid >> 5] = v;
    __syncthreads();
    double s = c.red[0];
    for (int k = 1; k < (c.G >> 5); k++) s = fmin(s, c.red[k]);
    return s;
#endif
}
/* sums of TWO values over the environment's threads with ONE barrier: the per-warp partial sums are exchanged through
 * alternating halves of c.red (`buf` flips at every call), so the writes of call r+1 cannot meet the reads of call r; the
 * reads of call r-1 are over because every thread has passed call r's barrier since.  The caller puts one barrier before
 * the first call of a sequence (other users of c.red) and keeps `buf` in a register.  `red` is saddr_of(c.red): the hot
 * loop calls these with registers only.
 * ptxas gives every shuffle a divergent-warp fallback (BRA.DIV to a WARPSYNC / ENDCOLLECTIVE copy at the end of the
 * function) because it cannot prove that the warp arrives converged at the entry of a __noinline__ function; a
 * __syncwarp() in front does not change that.  The fallback is never taken (every lane of every warp calls these) and sits
 * outside the loop's instruction stream. */
WRSN_DI void red_sum2(saddr_t red, int tid, int G, double &a, double &b, int &buf) {
#if defined(WRSN_HOST_EMU)
    (void)red; (void)tid; (void)G; (void)a; (void)b; (void)buf;
#else
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
#if WRSN_GFIX != 32
    const saddr_t x = red + 128u * (uint32_t)buf;
    buf ^= 1;
    const int nw = G >> 5;
    if ((tid & 31) == 0) { sts64(x + 16u * (uint32_t)(tid >> 5), a); sts64(x + 16u * (uint32_t)(tid >> 5) + 8u, b); }
    __syncthreads();
    a = lds64(x); b = lds64(x + 8u);
    for (int k = 1; k < nw; k++) { a += lds64(x + 16u * (uint32_t)k); b += lds64(x + 16u * (uint32_t)k + 8u); }
#else
    (void)red; (void)tid; (void)G; (void)buf;
#endif
#endif
}
WRSN_DI void red_sum1(saddr_t red, int tid, int G, double &a, int &buf) {
#if defined(WRSN_HOST_EMU)
    (void)red; (void)tid; (void)G; (void)a; (void)buf;
#else
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
#if WRSN_GFIX != 32
    const saddr_t x = red + 128u * (uint32_t)buf;
    buf ^= 1;
    const int nw = G >> 5;
    if ((tid & 31) == 0) sts64(x + 8u * (uint32_t)(tid >> 5), a);
    __syncthreads();
    a = lds64(x);
    for (int k = 1; k < nw; k++) a += lds64(x + 8u * (uint32_t)k);
#else
    (void)red; (void)tid; (void)G; (void)buf;
#endif
#endif
}
WRSN_D bool red_or_warp(int v) {                    /* over the calling warp only (no barrier) */
#if defined(WRSN_HOST_EMU)
    return v != 0;
#else
    return __any_sync(0xffffffffu, v != 0);
#endif
}
WRSN_D int red_or(const Ctx &c, int v) {
#if defined(WRSN_HOST_EMU)
    (void)c; return v ? 1 : 0;
#elif WRSN_GFIX == 32
    (void)c; return __any_sync(0xffffffffu, v) ? 1 : 0;
#else
    (void)c; return __syncthreads_or(v) ? 1 : 0;
#endif
}
WRSN_D void atomic_or_u32(uint32_t *p, uint32_t v) {
#if !defined(WRSN_HOST_EMU)
    atomicOr(p, v);
#else
    *p |= v;
#endif
}
WRSN_D void atomic_add_i32(int *p, int v) {
#if !defined(WRSN_HOST_EMU)
    atomicAdd(p, v);
#else
    *p += v;
#endif
}
WRSN_D int atomic_add_ret_i32(int *p, int v) {
#if !defined(WRSN_HOST_EMU)
    return atomicAdd(p, v);
#else
    const int o = *p; *p += v; return o;
#endif
}
WRSN_D void atomic_max_nonneg(double *p, double v) {      /* v >= 0: order of the bit patterns == order of the values */
#if !defined(WRSN_HOST_EMU)
    atomicMax((long long *)p, __double_as_longlong(v));
#else
    if (v > *p) *p = v;
#endif
}

WRSN_D int wrsn_ctz(uint32_t v) {
#if !defined(WRSN_HOST_EMU)
    return __ffs((int)v) - 1;
#else
    return __builtin_ctz(v);
#endif
}
WRSN_D int wrsn_popc(uint32_t v) {
#if !defined(WRSN_HOST_EMU)
    return __popc(v);
#else
    return __builtin_popcount(v);
#endif
}

/* num / den for den > 0 and num >= 0.  A zero numerator (a node without traffic: energyCS == 0) would send CUDA's fp64
 * division down its special-case subroutine for the whole warp; the quotient is the (signed) zero itself. */
WRSN_D double div_pos(double num, double den) { return num == 0.0 ? num : num / den; }

/* ------------------------------------------------------------------ bounded-error fp64 helpers of the REWARD path
 * WRSN.update_reward (WRSN.py:100-127) only feeds `reward` (tolerance 1e-6 relative, SURVEY App. B L5): it is never read
 * back by the simulation.  Its N divisions, N exponentials, one square root per simulated second therefore do not need
 * IEEE rounding, they need few instructions: hardware seed (MUFU.RCP64H / RSQ64H) + Newton steps, and a table-driven
 * exponential.  All three are within a few 1e-14 relative of the exact result (the tests hold the reward at 1e-9).  Nothing
 * that is part of the simulated state (energies, energyCS, charger records) goes through these. */
#if !defined(WRSN_HOST_EMU)
WRSN_D double wrsn_fma(double a, double b, double c) { return __fma_rn(a, b, c); }
WRSN_D double wrsn_rcp(double d) {                  /* 1 / d, d > 0 with d and 1 / d normal (d <= 2^1022): <= 2 ulp;
                                                        the seed flushes a subnormal 1 / d to zero */
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
    double e = __fma_rn(-d, r, 1.0);
    r = __fma_rn(r, e, r);
    e = __fma_rn(-d, r, 1.0);
    return __fma_rn(r, e, r);
}
WRSN_D double wrsn_rsqrt(double v) {                /* 1 / sqrt(v), v > 0 normal: <= 2 ulp */
    double r;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(v));
    double e = __fma_rn(-v, r * r, 1.0);
    r = __fma_rn(r * 0.5, e, r);
    e = __fma_rn(-v, r * r, 1.0);
    return __fma_rn(r * 0.5, e, r);
}
/* exp(z) for |z| < 700, relative error <= 1e-13: z = (64 n + j) ln2/64 + r, |r| <= ln2/128;
 * exp(z) = 2^n * 2^(j/64) * (1 + r + r^2/2 + r^3/6 + r^4/24) — table of 64 doubles in shared memory (c.exptab, copied from
 * wrsn_exp2_tab at kernel start), four FMAs.  The caller's z is a z-score of N values: |z| <= sqrt(N - 1). */
WRSN_DI double wrsn_exp_tab(saddr_t tab, double z) {
    const double t = __fma_rn(z, 92.33248261689366, 6755399441055744.0);          /* 64 / ln2; 1.5 * 2^52: the integer lands in the low word */
    const int k = __double2loint(t);
    const double r = __fma_rn(t - 6755399441055744.0, -0.010830424696249145, z); /* ln2 / 64 */
    double p = __fma_rn(r, 1.0 / 24.0, 1.0 / 6.0);
    p = __fma_rn(p, r, 0.5);
    p = __fma_rn(p, r, 1.0);
    p = __fma_rn(p, r, 1.0);
    const double y = p * lds64(tab + 8u * (uint32_t)(k & 63));
    return __hiloint2double(__double2hiint(y) + ((k >> 6) << 20), __double2loint(y));
}
#else
WRSN_D double wrsn_fma(double a, double b, double c) { return a * b + c; }
WRSN_D double wrsn_rcp(double d) { return 1.0 / d; }
WRSN_D double wrsn_rsqrt(double v) { return 1.0 / sqrt(v); }
#endif
WRSN_DI double wrsn_exp_b(saddr_t tab, double z) {  /* tab = saddr_of(c.exptab) */
#if defined(WRSN_HOST_EMU)
    (void)tab; return exp(z);
#else
    return wrsn_exp_tab(tab, z);
#endif
}


WRSN_NOINLINE double euclid2(double ax, double ay, double bx, double by) {
    /* scipy.spatial.distance.euclidean == sqrt(dot(u - v, u - v)) for 2-vectors */
    double dx = ax - bx, dy = ay - by;
    return sqrt(dx * dx + dy * dy);
}

/* ------------------------------------------------------------------ exact replay of a node's subtraction chain
 * n_single times (e -= a) followed by n_pair times (e -= b; e -= a), evaluated sequentially in fp64 by the
 * reference.  Inside one binade [2^k, 2^(k+1)) every representable value is a multiple of u = 2^(k-52), so
 * "e - x" rounds to e - rint(x/u)*u (ties aside): each step removes a fixed integer number of ulps and the
 * whole chain is one exact integer multiply.  The result must lie strictly above 2^k: a chain that ends exactly on
 * 2^k has a last step whose exact value may fall below 2^k, where the spacing is u/2, and round to 2^k - u/2.  If the
 * chain would reach 2^k or leave the binade (or x/u is an exact tie) the literal loop runs instead.  Order of the
 * steps does not matter while the result stays above 2^k. */
WRSN_D double wrsn_pow2_biased(int biased) {       /* 2^(biased - 1023) for 1 <= biased <= 2046 */
    uint64_t b = (uint64_t)biased << 52;
#if !defined(WRSN_HOST_EMU)
    return __longlong_as_double((long long)b);
#else
    double r; memcpy(&r, &b, 8); return r;
#endif
}
WRSN_D int wrsn_biased_exp(double e) {
#if !defined(WRSN_HOST_EMU)
    return (int)((((unsigned long long)__double_as_longlong(e)) >> 52) & 0x7ffull);
#else
    uint64_t b; memcpy(&b, &e, 8); return (int)((b >> 52) & 0x7ffull);
#endif
}
WRSN_NOINLINE double sub_chain_literal(double e, double a, int n_single, double b, int n_pair) {
    for (int k = 0; k < n_single; k++) e -= a;
    for (int k = 0; k < n_pair; k++) { e -= b; e -= a; }
    return e;
}
/* the closed form alone: NaN when the chain would reach 2^k or leave the binade, has an exact tie, or e is out of range */
WRSN_D double sub_chain_fast(double e, double a, int n_single, double b, int n_pair) {
    int n_a = n_single + n_pair;
    if (n_a == 0) return e;
    int ex = wrsn_biased_exp(e);
    if (e > 0.0 && ex > 60 && ex < 1900) {
        double lo = wrsn_pow2_biased(ex);
        double inv_u = wrsn_pow2_biased(2098 - ex), u = wrsn_pow2_biased(ex - 52);
        double qa = a * inv_u, qb = b * inv_u;
        double ra = rint(qa), rb = rint(qb);
        bool tie = (fabs(qa - ra) == 0.5) || (n_pair > 0 && fabs(qb - rb) == 0.5);
        double total = ra * (double)n_a + rb * (double)n_pair;
        if (!tie && total < 4503599627370496.0) {
            double r = e - total * u;
            if (r > lo) return r;
        }
    }
    return NAN;
}
WRSN_D double sub_chain(double e, double a, int n_single, double b, int n_pair) {
    int n_a = n_single + n_pair;
    if (n_a == 0) return e;
    int ex = wrsn_biased_exp(e);                     /* e in [2^(ex-1023), 2^(ex-1022)), u = 2^(ex-1075) */
    if (e > 0.0 && ex > 60 && ex < 1900) {
        double lo = wrsn_pow2_biased(ex);
        double inv_u = wrsn_pow2_biased(2098 - ex), u = wrsn_pow2_biased(ex - 52);
        double qa = a * inv_u, qb = b * inv_u;       /* exact scalings */
        double ra = rint(qa), rb = rint(qb);
        bool tie = (fabs(qa - ra) == 0.5) || (n_pair > 0 && fabs(qb - rb) == 0.5);
        double total = ra * (double)n_a + rb * (double)n_pair;
        if (!tie && total < 4503599627370496.0) {    /* < 2^52 ulps: products and sum are exact integers */
            double r = e - total * u;
            if (r > lo) return r;
        }
    }
    return sub_chain_literal(e, a, n_single, b, n_pair);
}

/* ------------------------------------------------------------------ event clock
 * While run_loop() is active the clock lives in REGISTERS, identical in every thread of the environment: all
 * threads execute the (scalar) clock and charger logic redundantly from broadcast shared-memory loads, thread 0
 * alone stores.  Nothing is broadcast through shared memory and no thread waits for a leader.  Outside
 * run_loop() the clock is the hdr row (the *_h helpers, leader only).
 * An event's position in SimPy's queue is (time, priority, insertion counter); priority and counter are folded
 * into one double key = priority * 2^40 + counter, a pending time of +inf means "nothing pending". */
#define WRSN_KEY_NORMAL 1099511627776.0            /* 2^40 */

struct Clk {
    double now, seq, nev;
    double net_t, net_key, ur_t, ur_key, nodes_t, nodes_key, until_t, until_key;
    int net_state, nodes_phase, stop;
    int work;                                        /* work units of this launch (see run_loop: the step budget) */
    int nobatch_once;                                /* the batch kernel could not batch the pending second: event by event, once */
    int mc_idx;                                      /* earliest pending charger-slot (< n_slot) / condition (>= n_slot) event */
    double mc_t, mc_key, mc_other_t;                 /* its position; earliest time among the OTHER slot / condition events */
};

WRSN_D double *slot_of(Ctx &c, int s) { return c.proc + s * WRSN_PR_LEN; }
WRSN_D int *slot_i(double *p) { return (int *)p; }
WRSN_D double *mc_of(Ctx &c, int a) { return c.mc + a * WRSN_MC_LEN; }
WRSN_DI double take_seq(Clk &k) { double s = k.seq; k.seq = s + 1.0; return s; }
WRSN_D double take_seq_h(Ctx &c) { double s = c.hdr[WRSN_H_SEQ]; c.hdr[WRSN_H_SEQ] = s + 1.0; return s; }
WRSN_DI bool ev_before(double t, double key, double bt, double bkey) { return t < bt || (t == bt && key < bkey); }

WRSN_DI void clk_load(Ctx &c, Clk &k) {
    const double *h = c.hdr;
    k.now = h[WRSN_H_NOW]; k.seq = h[WRSN_H_SEQ]; k.nev = 0.0;
    k.net_t = h[WRSN_H_NET_ON] != 0.0 ? h[WRSN_H_NET_T] : INFINITY; k.net_key = WRSN_KEY_NORMAL + h[WRSN_H_NET_SEQ];
    k.net_state = (int)h[WRSN_H_NET_STATE];
    k.ur_t = h[WRSN_H_UR_ON] != 0.0 ? h[WRSN_H_UR_T] : INFINITY; k.ur_key = WRSN_KEY_NORMAL + h[WRSN_H_UR_SEQ];
    k.nodes_t = h[WRSN_H_NODES_T]; k.nodes_key = WRSN_KEY_NORMAL + h[WRSN_H_NODES_SEQ]; k.nodes_phase = (int)h[WRSN_H_NODES_PHASE];
    k.until_t = h[WRSN_H_UNTIL_ON] != 0.0 ? h[WRSN_H_UNTIL_T] : INFINITY; k.until_key = h[WRSN_H_UNTIL_SEQ];   /* URGENT */
    k.stop = 0; k.work = 0; k.nobatch_once = h[WRSN_H_NOBATCH_ONCE] != 0.0 ? 1 : 0; k.mc_idx = -1; k.mc_t = INFINITY; k.mc_key = 0.0; k.mc_other_t = INFINITY;
}
WRSN_DI void clk_store(Ctx &c, const Clk &k) {
    gsync(c);
    if (c.tid == 0) {
        double *h = c.hdr;
        h[WRSN_H_NOW] = k.now; h[WRSN_H_SEQ] = k.seq; h[WRSN_H_NEVENTS] += k.nev;
        h[WRSN_H_NET_ON] = k.net_t < INFINITY ? 1.0 : 0.0; if (k.net_t < INFINITY) h[WRSN_H_NET_T] = k.net_t;
        h[WRSN_H_NET_SEQ] = k.net_key - WRSN_KEY_NORMAL; h[WRSN_H_NET_STATE] = k.net_state;
        h[WRSN_H_UR_ON] = k.ur_t < INFINITY ? 1.0 : 0.0; if (k.ur_t < INFINITY) h[WRSN_H_UR_T] = k.ur_t;
        h[WRSN_H_UR_SEQ] = k.ur_key - WRSN_KEY_NORMAL;
        h[WRSN_H_NODES_T] = k.nodes_t; h[WRSN_H_NODES_SEQ] = k.nodes_key - WRSN_KEY_NORMAL; h[WRSN_H_NODES_PHASE] = k.nodes_phase;
        h[WRSN_H_UNTIL_ON] = k.until_t < INFINITY ? 1.0 : 0.0; if (k.until_t < INFINITY) h[WRSN_H_UNTIL_T] = k.until_t;
        h[WRSN_H_UNTIL_SEQ] = k.until_key;
        h[WRSN_H_NOBATCH_ONCE] = k.nobatch_once ? 1.0 : 0.0;
    }
    gsync(c);
}

/* earliest pending slot / condition event and the earliest time among the others (all threads, broadcast loads) */
WRSN_DI void mc_scan(Ctx &c, Clk &k) {
    int bi = -1;
    double bt = INFINITY, bkey = 0.0, ot = INFINITY;
    const int ns = c.n_slot;
#pragma unroll 1
    for (int s = 0; s < ns; s++) {
        const double *p = c.proc + s * WRSN_PR_LEN;
        const bool lazy = ((const int *)p)[WRSN_PRI_LAZY] != 0;
        const double t = lazy ? p[WRSN_PR_TINT] : p[WRSN_PR_T];   /* a lazy slot next matters when its run of spans ends */
        if (t < INFINITY) {
            const double key = lazy ? WRSN_KEY_NORMAL * 2.0 : p[WRSN_PR_KEY];
            if (ev_before(t, key, bt, bkey)) { ot = bt; bi = s; bt = t; bkey = key; }
            else ot = fmin(ot, t);
        }
    }
    const double *h = c.hdr;
    const int nch = (int)h[WRSN_H_CHAIN_N];
#pragma unroll 1
    for (int j = 0; j < nch; j++) {
        const double t = h[WRSN_H_COND_T + j];
        if (t < INFINITY) {
            const double key = h[WRSN_H_COND_KEY + j];
            if (ev_before(t, key, bt, bkey)) { ot = bt; bi = ns + j; bt = t; bkey = key; }
            else ot = fmin(ot, t);
        }
    }
    k.mc_idx = bi; k.mc_t = bt; k.mc_key = bkey; k.mc_other_t = ot;
}

/* ------------------------------------------------------------------ Node.log ring: leave the "all ten entries equal
 * logc" shortcut (entries were not written while it held) */
WRSN_NOINLINE void leave_uniform(Ctx &c) {
    bool uni = c.hdr[WRSN_H_LOG_UNIFORM] >= 10.0 && c.hdr[WRSN_H_LOG_LEN] >= 10.0;
    if (uni)
        for (int i = c.tid; i < c.N; i += WRSN_GSZ(c)) {
            double v = c.logc[i];
            for (int k = 0; k < WRSN_RING; k++) c.ring[(size_t)k * c.Npad + i] = v;
        }
    gsync(c);
    if (c.tid == 0) c.hdr[WRSN_H_LOG_UNIFORM] = 0.0;
    gsync(c);
}

/* Routing tree for the current `level` / `status` rows: receiver of every node (Node.find_receiver :92-100, first
 * nearest alive neighbour of lower level; the base station for direct nodes), its transmit cost, the relay counts and
 * the per-tick log_energy.  With fresh levels every reached node has a receiver; with STALE levels (Network.operate
 * has stopped, later deaths) a chain can end at a node without receiver: that node still pays the receive cost of what
 * its children send, forwards nothing (e_send = 0) and sends nothing itself — as the reference does. */
WRSN_NOINLINE void build_tree(Ctx &c) {
    const int N = c.N;
    int *cnt = (int *)c.scr0.ptr();                       /* 2 ints per node: relayed packets from lower / higher ids */
    for (int i = c.tid; i < N; i += WRSN_GSZ(c)) {
        cnt[2 * i] = 0; cnt[2 * i + 1] = 0;
        int par = -1; double es = 0.0;
        if (c.status[i] == 1 && c.level[i] >= 1) {
            if (c.direct[i]) { par = -2; es = c.bs_esend[i]; }
            else {
                double bd = 0.0; int lv = c.level[i];
                for (int e = c.nbr_ptr[i]; e < c.nbr_ptr[i + 1]; e++) {
                    int j = c.nbr_idx[e];
                    if (c.level[j] < lv && c.status[j] == 1) {
                        double dd = c.nbr_dist[e];
                        if (par < 0 || dd < bd) { par = j; bd = dd; es = c.nbr_esend[e]; }   /* np.argmin: first minimum */
                    }
                }
            }
        }
        c.parent[i] = (int16_t)par; c.esend[i] = es;
    }
    gsync(c);
    /* relay counts: every packet of source s crosses its ancestors up to the base station (or the chain's end) */
    for (int s = c.tid; s < N; s += WRSN_GSZ(c)) {
        int ow = c.own[s];
        if (c.status[s] != 1 || ow == 0 || c.parent[s] == -1) continue;
        for (int h = c.parent[s]; h >= 0; h = c.parent[h]) atomic_add_i32(&cnt[2 * h + (s < h ? 0 : 1)], ow);
    }
    gsync(c);
    const double er = c.par[WRSN_P_ERECV];
    for (int i = c.tid; i < N; i += WRSN_GSZ(c)) {
        int nb = cnt[2 * i], na = cnt[2 * i + 1];
        c.nbef[i] = (uint16_t)nb; c.naft[i] = (uint16_t)na;
        double lg = 0.0, es = c.esend[i];
        if (c.status[i] == 1) {
            for (int k = 0; k < nb; k++) { lg += es; lg += er; }
            int ow = c.parent[i] != -1 ? (int)c.own[i] : 0;
            for (int k = 0; k < ow; k++) lg += es;
            for (int k = 0; k < na; k++) { lg += es; lg += er; }
        }
        c.logc[i] = lg;
    }
    gsync(c);
}

/* ------------------------------------------------------------------ Network.setLevels + check_targets (Network.py:37-66,84),
 * then the routing tree the drain tick replays. */
WRSN_NOINLINE void do_bfs(Ctx &c) {
    WRSN_PROF_BEGIN();
    leave_uniform(c);
    const int N = c.N;
    for (int i = c.tid; i < N; i += WRSN_GSZ(c)) c.level[i] = (c.status[i] == 1 && c.direct[i]) ? 1 : -1;
    for (int w = c.tid; w < c.Tw; w += WRSN_GSZ(c)) c.tact[w] = 0u;
    gsync(c);
    for (int cur = 1;; cur++) {
        int any = 0;
        for (int i = c.tid; i < N; i += WRSN_GSZ(c)) {
            if (c.level[i] != cur) continue;
            for (int e = c.tgt_ptr[i]; e < c.tgt_ptr[i + 1]; e++) {
                int t = c.tgt_idx[e];
                atomic_or_u32(&c.tact[t >> 5], 1u << (t & 31));
            }
            for (int e = c.nbr_ptr[i]; e < c.nbr_ptr[i + 1]; e++) {
                int j = c.nbr_idx[e];
                if (c.status[j] == 1 && c.level[j] == -1) { c.level[j] = (int16_t)(cur + 1); any = 1; }
            }
        }
        gsync(c);
        if (!red_or(c, any)) break;
    }
    /* alive = min(targets_active) */
    int dead_t = 0;
    for (int w = c.tid; w < c.Tw; w += WRSN_GSZ(c)) {
        if ((c.tact[w] & tact_word_mask(c, w)) != tact_word_mask(c, w)) dead_t = 1;
    }
    dead_t = red_or(c, dead_t);
    build_tree(c);
    if (c.tid == 0) {
        c.hdr[WRSN_H_ALIVE] = dead_t ? 0.0 : 1.0;
        c.hdr[WRSN_H_BFS_DIRTY] = 0.0;
        c.hdr[WRSN_H_NBFS] += 1.0;
    }
    gsync(c);
    WRSN_PROF_END(c, WRSN_H_PROF3);
}

/* ------------------------------------------------------------------ Node.operate, k+0.5 tick (Node.py:57-62,92-132) */
WRSN_D void check_status_node(Ctx &c, int i) {     /* Node.py:148-151 */
    if (c.energy[i] <= c.par[WRSN_P_THR]) { c.status[i] = 0; c.cs[i] = 0.0; }
}

/* exact serial tick: packet by packet, hop by hop, as the reference does it (leader only) */
/* Starts with packet k0 of source s0 and handles `max_packets` packets at most (a whole tick: 0, 0, false, INT_MAX);
 * `begun`: the turn of s0 has begun already (its top-up is done). */
WRSN_NOINLINE int drain_serial(Ctx &c, int s0, int k0, bool begun, int max_packets) {
    const int N = c.N;
    const double thr = c.par[WRSN_P_THR], cap = c.par[WRSN_P_CAP], er = c.par[WRSN_P_ERECV];
    int deaths = 0;
    double *lt = c.scr1;                             /* this tick's log_energy, in shared memory: the leader adds to it at every hop;
                                                        the caller zeroes it before and copies it to the record afterwards */
    for (int i = s0; i < N && max_packets > 0; i++) {
        if (c.status[i] == 0) continue;
        const bool resumed = i == s0 && begun;
        if (!resumed) c.energy[i] = fmin(c.energy[i] + c.rr[i] * 0.5, cap);
        int ow = c.own[i];
        for (int k = resumed ? k0 : 0; k < ow && max_packets > 0; k++, max_packets--) {
            int h = i; bool pay_recv = false;
            for (;;) {
                /* one hop; the node's energy lives in a register from the receive to the death check (the leader is alone
                   here, and every shared-memory access is ~30 dependent cycles on this single thread) */
                double e = c.energy[h];
                if (pay_recv) {                      /* receive_package */
                    if (e - thr < er) {
                        c.energy[h] = thr;
                        if (c.status[h] == 1) deaths++;
                        c.status[h] = 0; c.cs[h] = 0.0;          /* check_status: energy == threshold */
                        break;
                    }
                    e -= er;
                }
                /* send_package: find_receiver() = the tree's receiver unless that node died earlier in this very tick
                   (a death can only remove candidates, never bring a nearer one), then the literal neighbour scan */
                int recv = c.parent[h]; double es = c.esend[h];
                if (recv >= 0 && c.status[recv] != 1) {
                    recv = -1; es = 0.0;
                    double bd = 0.0; int lv = c.level[h];
                    for (int q = c.nbr_ptr[h]; q < c.nbr_ptr[h + 1]; q++) {
                        int j = c.nbr_idx[q];
                        if (c.level[j] < lv && c.status[j] == 1) {
                            double dd = c.nbr_dist[q];
                            if (recv < 0 || dd < bd) { recv = j; bd = dd; es = c.nbr_esend[q]; }
                        }
                    }
                }
                bool sent = false;
                if (recv != -1) {
                    if (e - thr < es) e = thr;
                    else { e -= es; sent = true; }
                }
                c.energy[h] = e;
                if (sent || pay_recv) {
                    double l = lt[h];
                    if (sent) l += es;
                    if (pay_recv) l += er;
                    lt[h] = l;
                }
                if (e <= thr) {                      /* check_status */
                    if (c.status[h] == 1) deaths++;
                    c.status[h] = 0; c.cs[h] = 0.0;
                }
                if (!sent || recv == -2) break;
                h = recv; pay_recv = true;
            }
        }
    }
    return deaths;
}

/* ------------------------------------------------------------------ death tick in pieces
 * A death tick must replay packets one by one — but only around the death.  Until the first node fails nothing is
 * irregular: all packets of the sources before the death packet (s*, k*) are applied node-parallel in the exact
 * three-step closed form (relays of lower sources, top-up, own packets, relays of higher sources — restricted to the
 * sources < s*, plus the first k* packets of s*).  The death packet itself runs through the literal hop code.  After it
 * the routing is rebuilt (same rule as the reference's find_receiver on the stale levels) and, if no node is endangered
 * under the remaining load, the remaining packets are applied in closed form as well; otherwise the rest of the tick is
 * replayed serially.  (s*, k*) is found by replaying, literally and on one thread, the operation sequence of every
 * ENDANGERED node alone (a node the no-death closed form leaves within the slack of the threshold): before the first
 * death no other node can fail.  The per-tick log_energy is accumulated in the same order (piece 1, death packet,
 * piece 2). */
#define WRSN_MAX_ENDANGERED 4
WRSN_D void count_relays(Ctx &c, uint32_t *cnt, int s_lo, int k_lo, int s_hi, int k_hi) {
    /* relays per node from the packets (s, k) with (s_lo, k_lo) <= (s, k) < (s_hi, k_hi), split by s < node / s > node */
    const int N = c.N, G = WRSN_GSZ(c);
    for (int i = c.tid; i < N; i += G) { cnt[2 * i] = 0u; cnt[2 * i + 1] = 0u; }
    gsync(c);
    for (int s = c.tid; s < N; s += G) {
        int ow = c.own[s];
        if (c.status[s] != 1 || ow == 0 || c.parent[s] == -1 || s < s_lo || s > s_hi) continue;
        int first = s == s_lo ? k_lo : 0, last = s == s_hi ? k_hi : ow;
        if (last > ow) last = ow;
        const int n = last - first;
        if (n <= 0) continue;
        for (int h = c.parent[s]; h >= 0; h = c.parent[h]) {
#if !defined(WRSN_HOST_EMU)
            atomicAdd(&cnt[2 * h + (s < h ? 0 : 1)], (uint32_t)n);
#else
            cnt[2 * h + (s < h ? 0 : 1)] += (uint32_t)n;
#endif
        }
    }
    gsync(c);
}

WRSN_NOINLINE int drain_pieces(Ctx &c) {           /* returns the number of deaths, or -1: nothing changed, use drain_serial */
    const int N = c.N, G = WRSN_GSZ(c);
    const double thr = c.par[WRSN_P_THR], cap = c.par[WRSN_P_CAP], er = c.par[WRSN_P_ERECV];
    const double slack = 1e-6;
    uint32_t *cnt = (uint32_t *)c.scr0.ptr();
    double *lt = c.scr1;                             /* zeroed by the caller */
    int *bc = c.bcast;                               /* [0] number of endangered nodes, [1..4] their ids, [5] s*, [6] k*, [7] deaths */
    if (c.tid == 0) { bc[0] = 0; bc[5] = N; bc[6] = 0; bc[7] = 0; }
    gsync(c);
    /* endangered nodes under the full load of the tick */
    for (int i = c.tid; i < N; i += G) {
        if (c.status[i] != 1) continue;
        const double e = c.energy[i], es = c.esend[i], rr = c.rr[i];
        const int nb = c.nbef[i], na = c.naft[i];
        const int ow = c.parent[i] != -1 ? (int)c.own[i] : 0;
        bool end = false;
        const double e1 = sub_chain(e, es, 0, er, nb);
        if (nb > 0 && !(e1 - thr >= slack)) end = true;
        const double e2 = fmin(e1 + rr * 0.5, cap);
        const double e3 = sub_chain(e2, es, ow, er, na);
        if (ow + na > 0 && !(e3 - thr >= slack)) end = true;
        if (end) {
#if !defined(WRSN_HOST_EMU)
            const int slot = atomicAdd(&bc[0], 1);
#else
            const int slot = bc[0]++;
#endif
            if (slot < WRSN_MAX_ENDANGERED) bc[1 + slot] = i;
        }
    }
    gsync(c);
    const int n_end = bc[0];
    if (n_end < 1 || n_end > WRSN_MAX_ENDANGERED) return -1;
    /* the first packet at which an endangered node fails or is left at the threshold: its own operation sequence, literally */
    for (int q = 0; q < n_end; q++) {
        const int h = bc[1 + q];
        for (int s = c.tid; s < N; s += G) {         /* packets of source s that pass through h */
            uint32_t w = 0u;
            if (c.status[s] == 1 && s != h && c.parent[s] != -1) {
                int hops = 0;
                for (int a = c.parent[s]; a >= 0 && hops++ <= N; a = c.parent[a]) if (a == h) { w = c.own[s]; break; }
            }
            cnt[s] = w;
        }
        gsync(c);
        if (c.tid == 0) {
            double e = c.energy[h];
            const double es = c.esend[h];
            const bool can_send = c.parent[h] != -1;
            int fs = N, fk = 0;
            for (int s2 = 0; s2 < N && fs == N; s2++) {
                if (s2 == h) {
                    e = fmin(e + c.rr[h] * 0.5, cap);
                    const int ow = c.own[h];
                    for (int k = 0; k < ow; k++) {
                        if (can_send) { if (e - thr < es) { fs = s2; fk = k; break; } e -= es; }
                        if (e <= thr) { fs = s2; fk = k; break; }
                    }
                } else {
                    const int w = (int)cnt[s2];
                    for (int k = 0; k < w; k++) {
                        if (e - thr < er) { fs = s2; fk = k; break; }
                        e -= er;
                        if (can_send) { if (e - thr < es) { fs = s2; fk = k; break; } e -= es; }
                        if (e <= thr) { fs = s2; fk = k; break; }
                    }
                }
            }
            if (fs < bc[5] || (fs == bc[5] && fk < bc[6])) { bc[5] = fs; bc[6] = fk; }
        }
        gsync(c);
    }
    const int s_star = bc[5], k_star = bc[6];
    if (s_star >= N) return -1;                      /* nobody fails after all (slack): the caller's serial path settles it */
    /* piece 1: every packet before (s*, k*) */
    count_relays(c, cnt, 0, 0, s_star, k_star);
    for (int j = c.tid; j < N; j += G) {
        if (c.status[j] != 1) continue;
        const int cb = (int)cnt[2 * j], ca = (int)cnt[2 * j + 1];
        const int ow_full = c.parent[j] != -1 ? (int)c.own[j] : 0;
        const int ow = j < s_star ? ow_full : (j == s_star ? (k_star < ow_full ? k_star : ow_full) : 0);
        const double es = c.esend[j];
        const double e1 = sub_chain(c.energy[j], es, 0, er, cb);
        const double e2 = j <= s_star ? fmin(e1 + c.rr[j] * 0.5, cap) : e1;
        c.energy[j] = sub_chain(e2, es, ow, er, ca);
        double lg = 0.0;
        for (int k = 0; k < cb; k++) { lg += es; lg += er; }
        for (int k = 0; k < ow; k++) lg += es;
        for (int k = 0; k < ca; k++) { lg += es; lg += er; }
        lt[j] = lg;
    }
    gsync(c);
    /* the death packet, literally */
    if (c.tid == 0) bc[7] = drain_serial(c, s_star, k_star, true, 1);
    gsync(c);
    /* piece 2: new receivers (stale or fresh levels alike: Node.find_receiver), remaining packets */
    build_tree(c);                                   /* parent / esend of the survivors; its counts are not used here */
    count_relays(c, cnt, s_star, k_star + 1, N - 1, 1 << 30);
    int end2 = 0;
    for (int j = c.tid; j < N; j += G) {
        if (c.status[j] != 1) continue;
        const int cb = (int)cnt[2 * j], ca = (int)cnt[2 * j + 1];
        const int ow_full = c.parent[j] != -1 ? (int)c.own[j] : 0;
        int ow = j > s_star ? ow_full : (j == s_star ? ow_full - (k_star + 1) : 0);
        if (ow < 0) ow = 0;
        const double es = c.esend[j];
        const double e1 = sub_chain(c.energy[j], es, 0, er, cb);
        if (cb > 0 && !(e1 - thr >= slack)) end2 = 1;
        const double e2 = j > s_star ? fmin(e1 + c.rr[j] * 0.5, cap) : e1;
        const double e3 = sub_chain(e2, es, ow, er, ca);
        if (ow + ca > 0 && !(e3 - thr >= slack)) end2 = 1;
        /* stash the result; committed below if nobody is endangered */
        ((double *)c.gscratch)[j] = e3;
    }
    gsync(c);
    if (red_or(c, end2)) {                           /* a second death is possible: the rest of the tick literally */
        if (c.tid == 0) bc[7] += drain_serial(c, s_star, k_star + 1, true, 1 << 30);
        gsync(c);
        return bc[7];
    }
    for (int j = c.tid; j < N; j += G) {
        if (c.status[j] != 1) continue;
        const int cb = (int)cnt[2 * j], ca = (int)cnt[2 * j + 1];
        const int ow_full = c.parent[j] != -1 ? (int)c.own[j] : 0;
        int ow = j > s_star ? ow_full : (j == s_star ? ow_full - (k_star + 1) : 0);
        if (ow < 0) ow = 0;
        const double es = c.esend[j];
        c.energy[j] = ((double *)c.gscratch)[j];
        double lg = lt[j];
        for (int k = 0; k < cb; k++) { lg += es; lg += er; }
        for (int k = 0; k < ow; k++) lg += es;
        for (int k = 0; k < ca; k++) { lg += es; lg += er; }
        lt[j] = lg;
    }
    gsync(c);
    return bc[7];
}

WRSN_D void ev_nodes_drain(Ctx &c) {
    const int N = c.N;
    const double thr = c.par[WRSN_P_THR], cap = c.par[WRSN_P_CAP], er = c.par[WRSN_P_ERECV];
    const double slack = 1e-6;
    if (c.hdr[WRSN_H_BFS_DIRTY] != 0.0) {            /* a death after Network.operate stopped: levels stay stale (as in the
                                                        reference), only the receivers / relay counts are rebuilt */
        leave_uniform(c);
        build_tree(c);
        if (c.tid == 0) { c.hdr[WRSN_H_BFS_DIRTY] = 0.0; c.hdr[WRSN_H_NSTALE] += 1.0; }
        gsync(c);
    }
    int slow = 0;
    _Pragma("unroll 1")
    for (int i = c.tid; i < N; i += WRSN_GSZ(c)) {
        if (c.status[i] != 1) continue;
        double e = c.energy[i], es = c.esend[i];
        int nb = c.nbef[i], na = c.naft[i];
        int ow = c.parent[i] != -1 ? (int)c.own[i] : 0;
        const double rr = c.rr[i];
        double e3 = NAN;
        if (rr == 0.0) {
            /* no top-up in between: the two chains are one multiset of subtractions; inside a binade their order does not
               matter (sub_chain), so one closed form serves both — NaN when it would reach the binade's floor or leave it */
            e3 = sub_chain_fast(e, es, ow, er, nb + na);
            if (e3 == e3 && nb + ow + na > 0 && !(e3 - thr >= slack)) slow = 1;   /* e1 >= e3: the first check is implied */
        }
        if (e3 != e3) {
            double e1 = sub_chain(e, es, 0, er, nb);
            if (nb > 0 && !(e1 - thr >= slack)) slow = 1;
            double e2 = fmin(e1 + rr * 0.5, cap);
            e3 = sub_chain(e2, es, ow, er, na);
            if (ow + na > 0 && !(e3 - thr >= slack)) slow = 1;
        }
        c.scr0[i] = e3;
    }
    gsync(c);
    slow = red_or(c, slow);
    if (!slow) {
        _Pragma("unroll 1")
        for (int i = c.tid; i < N; i += WRSN_GSZ(c))
            if (c.status[i] == 1) c.energy[i] = c.scr0[i];
        gsync(c);
        return;
    }
    leave_uniform(c);
    WRSN_PROF_BEGIN();
    for (int i = c.tid; i < N; i += WRSN_GSZ(c)) c.scr1[i] = 0.0;
    gsync(c);
    const int pieces = c.hdr[WRSN_H_OPT_NOBATCH] != 0.0 ? -1 : drain_pieces(c);   /* (the test switch also forces the plain serial tick) */
    if (c.tid == 0) {
        const int deaths = pieces >= 0 ? pieces : drain_serial(c, 0, 0, false, 1 << 30);
        c.bcast[7] = deaths;
        c.hdr[WRSN_H_LOG_LITERAL] = 1.0;
        c.hdr[WRSN_H_NSLOW] += 1.0;
        if (pieces >= 0) c.hdr[WRSN_H_NSPLIT] += 1.0;
        if (deaths > 0) c.hdr[WRSN_H_BFS_DIRTY] = 1.0;
    }
    gsync(c);
    if (c.bcast[7] > 0) build_tree(c);               /* receivers of the survivors (levels as they are; Network.setLevels follows at
                                                        k+1.1 if Network.operate is still running) */
    for (int i = c.tid; i < N; i += WRSN_GSZ(c)) c.logtick[i] = c.scr1[i];
    gsync(c);
    WRSN_PROF_END(c, WRSN_H_PROF1);
}

/* ------------------------------------------------------------------ Node.operate, k+1.0 tick (Node.py:65-77) */
WRSN_D void ev_nodes_book(Ctx &c) {
    const int N = c.N;
    const double cap = c.par[WRSN_P_CAP];
    const int L = (int)c.hdr[WRSN_H_LOG_LEN], head = (int)c.hdr[WRSN_H_LOG_HEAD];
    const bool literal = c.hdr[WRSN_H_LOG_LITERAL] != 0.0;
    const bool uni = !literal && L >= WRSN_RING && c.hdr[WRSN_H_LOG_UNIFORM] >= 10.0;
    _Pragma("unroll 1")
    for (int i = c.tid; i < N; i += WRSN_GSZ(c)) {
        if (c.status[i] != 1) continue;
        c.energy[i] = fmin(c.energy[i] + c.rr[i] * 0.5, cap);
        double lg = literal ? c.logtick[i] : c.logc[i];
        if (L < WRSN_RING) {
            c.cs[i] = (c.cs[i] * (double)L + lg) / (double)(L + 1);
            c.ring[(size_t)L * c.Npad + i] = lg;
        } else {
            double old = uni ? lg : c.ring[(size_t)head * c.Npad + i];
            c.cs[i] = div_pos(c.cs[i] * (double)L - old + lg, (double)L);
            if (!uni) c.ring[(size_t)head * c.Npad + i] = lg;
        }
    }
    gsync(c);
    if (c.tid == 0) {
        if (L < WRSN_RING) c.hdr[WRSN_H_LOG_LEN] = L + 1;
        else c.hdr[WRSN_H_LOG_HEAD] = (head + 1) % WRSN_RING;
        if (literal) { c.hdr[WRSN_H_LOG_UNIFORM] = 0.0; c.hdr[WRSN_H_LOG_LITERAL] = 0.0; }
        else if (c.hdr[WRSN_H_LOG_UNIFORM] < 1e9) c.hdr[WRSN_H_LOG_UNIFORM] += 1.0;
        c.hdr[WRSN_H_NTICKS] += 1.0;
    }
    gsync(c);
}

/* ------------------------------------------------------------------ WRSN.update_reward (WRSN.py:100-127) */
WRSN_D double charge_rate_to(Ctx &c, const double *m, int node) {   /* alpha / (d + beta) ** 2 */
    double t = euclid2(c.nx[node], c.ny[node], m[WRSN_MC_X], m[WRSN_MC_Y]) + c.par[WRSN_P_MC_BETA];
    return c.par[WRSN_P_MC_ALPHA] / (t * t);
}

/* the softmax priority + incentive sums; only reached when some incentive sum is non-empty */
WRSN_NOINLINE double drain_node(double e, double rr, double es, double er, int nb, int ow, int na, double cap);
WRSN_NOINLINE void catch_up_for_reward(Ctx &c, double t_reward);

WRSN_D bool reward_pairs(Ctx &c) {                 /* is there any (charging charger, connected alive node) pair? */
    bool any = false;
    for (int a = 0; a < c.M; a++) {
        const double *m = c.mc + a * WRSN_MC_LEN;
        if (m[WRSN_MC_STATUS] == 0.0 || m[WRSN_MC_TYPE] == 0.0 || m[WRSN_MC_NCONN] == 0.0) continue;
        const uint32_t *cm = c.conn + a * c.W;
        for (int w = 0; w < c.W; w++)
            for (uint32_t bits = cm[w]; bits; bits &= bits - 1u)
                if (c.status[32 * w + wrsn_ctz(bits)] == 1) any = true;
    }
    return any;
}

/* per-slot flags of a thread (slot s = node tid + s * G, reward_loop below): one bit mask per flag on the device
 * (registers; the launcher keeps N <= 9 * threads), byte arrays in the host emulation (one "thread" owns all N nodes there) */
#undef WRSN_EMU_MAXN
#if defined(WRSN_HOST_EMU)
#define WRSN_EMU_MAXN 32768
#endif
#undef WRSN_FLAGS_DECL
#undef WRSN_FL_GET
#undef WRSN_FL_SET
#undef WRSN_FL_CLR
#if defined(WRSN_HOST_EMU)
#define WRSN_FLAGS_DECL(name) static thread_local uint8_t name[WRSN_EMU_MAXN]; memset(name, 0, (size_t)NPT)
#define WRSN_FL_GET(name, s) (name[s] != 0)
#define WRSN_FL_SET(name, s) (name[s] = 1)
#define WRSN_FL_CLR(name, s) (name[s] = 0)
#else
#define WRSN_FLAGS_DECL(name) uint32_t name = 0u
#define WRSN_FL_GET(name, s) (((name) >> (s)) & 1u)
#define WRSN_FL_SET(name, s) ((name) |= 1u << (s))
#define WRSN_FL_CLR(name, s) ((name) &= ~(1u << (s)))
#endif

WRSN_D int nan_payload(double d) {
#if !defined(WRSN_HOST_EMU)
    return __double2loint(d);
#else
    uint64_t b; memcpy(&b, &d, 8); return (int)(uint32_t)b;
#endif
}
WRSN_D double nan_with_payload(int slot) {
    const uint64_t b = 0x7ff8000000000000ull | (uint64_t)(uint32_t)slot;
#if !defined(WRSN_HOST_EMU)
    return __longlong_as_double((long long)b);
#else
    double r; memcpy(&r, &b, 8); return r;
#endif
}

/* the table entry's arithmetic for a node at energy e: inside e's binade [lo, 2 lo) the chain of relayed packets of lower
 * ids, the own packets + relays of higher ids and the top-up  min(e + energyRR * 0.5, cap)  move e by D1, D2 and H — whole
 * numbers of ulps — as long as glo <= e <= ghi at the start of the second (both top-ups, both chains).  glo keeps one ulp
 * above lo + D1 + D2: a chain that ends exactly on lo may round to lo - u/2 (see sub_chain).  No closed form: glo = +inf. */
struct SpecTerms { double D1, D2, H, glo, ghi; };
WRSN_DI SpecTerms spec_terms(double e, double es, double er, double rr, int nb, int ow, int na) {
    const int n_a = nb + ow + na, n_b = nb + na;
    SpecTerms s = {0.0, 0.0, 0.0, INFINITY, -INFINITY};
    const int ex = wrsn_biased_exp(e);
    if (e > 0.0 && ex > 60 && ex < 1900) {
        const double lo = wrsn_pow2_biased(ex), inv_u = wrsn_pow2_biased(2098 - ex), u = wrsn_pow2_biased(ex - 52);
        const double qa = es * inv_u, qb = er * inv_u, qh = (rr * 0.5) * inv_u;
        const double ra = rint(qa), rb = rint(qb), rh = rint(qh);
        const bool tie = (n_a > 0 && fabs(qa - ra) == 0.5) || (n_b > 0 && fabs(qb - rb) == 0.5) || fabs(qh - rh) == 0.5;
        const double K1 = (ra + rb) * (double)nb, K2 = ra * (double)(ow + na) + rb * (double)na;
        if (!tie && K1 + K2 < 1125899906842624.0 && rh < 1125899906842624.0 && rr >= 0.0) {
            s.D1 = K1 * u; s.D2 = K2 * u; s.H = rh * u;
            s.glo = lo + (s.D1 + s.D2) + u; s.ghi = (lo + lo) - (s.H + s.H) - (u + u);
        }
    }
    return s;
}
/* table entry of node i at energy e (reward_loop / spec_second) */
WRSN_NOINLINE void spec_entry(Ctx &c, int i, int slot, double e) {
    double *sp = c.spec + slot * WRSN_SPEC_LEN;
    const int ow = c.parent[i] != -1 ? (int)c.own[i] : 0;
    const SpecTerms s = spec_terms(e, c.esend[i], c.par[WRSN_P_ERECV], c.rr[i], c.nbef[i], ow, c.naft[i]);
    sp[0] = s.D1; sp[1] = s.D2; sp[2] = s.H; sp[3] = s.glo; sp[4] = s.ghi; sp[5] = (double)i;
}

/* one table node, one second: [the previous second's k+1.0 top-up,] [this second's k+0.5 tick] on c.energy[i] */
WRSN_NOINLINE void spec_second(Ctx &c, int t, int book, int drain) {
    const double *sp = c.spec + t * WRSN_SPEC_LEN;
    const int i = (int)sp[5];
    const double cap = c.par[WRSN_P_CAP];
    double e = c.energy[i];
    if (e >= sp[3] && e <= sp[4]) {                  /* inside the guards: whole ulps */
        const double H = sp[2];
        if (book) e = fmin(e + H, cap);
        if (drain) e = fmin((e - sp[0]) + H, cap) - sp[1];
    } else {
        const double rr = c.rr[i];
        if (book) e = fmin(e + rr * 0.5, cap);
        if (drain) {
            const int ow = c.parent[i] != -1 ? (int)c.own[i] : 0;
            e = drain_node(e, rr, c.esend[i], c.par[WRSN_P_ERECV], c.nbef[i], ow, c.naft[i], cap);
        }
        spec_entry(c, i, t, e);                      /* e.g. the node has left the binade its entry was made for: a new one */
    }
    c.energy[i] = e;
}

/* Node.py:75 with log[0] == log_energy, for the slots whose energyCS has not reached its fixed point yet (cold: a node gets
 * there after one or two applications) */
WRSN_NOINLINE double cs_step(double cs, double lg) { return div_pos(cs * (double)WRSN_RING - lg + lg, (double)WRSN_RING); }

WRSN_NOINLINE double charge_rate_fast(Ctx &c, const double *m, int i) {   /* alpha / (d + beta)^2, reward path (few ulps) */
    const double dx = c.nx[i] - m[WRSN_MC_X], dy = c.ny[i] - m[WRSN_MC_Y], d2 = wrsn_fma(dx, dx, dy * dy);
    const double t = (d2 > 0.0 ? d2 * wrsn_rsqrt(d2) : 0.0) + c.par[WRSN_P_MC_BETA];
    return c.par[WRSN_P_MC_ALPHA] * wrsn_rcp(t * t);
}

/* the incentive sums of one tick (WRSN.py:113-126), one thread per charger; q_n / tot are the softmax weights.  (General form:
 * reward_loop handles up to WRSN_PAIR_MAX pairs by list and comes here beyond that.) */
WRSN_NOINLINE void reward_incentives(Ctx &c, double tot) {
    const double thr = c.par[WRSN_P_THR], cap = c.par[WRSN_P_CAP];
    const double inv_tot = wrsn_rcp(tot), ab2 = c.par[WRSN_P_MC_AB2], inv_ab2 = wrsn_rcp(ab2);
    for (int a2 = c.tid; a2 < c.M; a2 += WRSN_GSZ(c)) {
        double *m = c.mc + (size_t)a2 * WRSN_MC_LEN;
        if (m[WRSN_MC_STATUS] != 0.0 && m[WRSN_MC_TYPE] != 0.0) {
            double incentive = 0.0;
            const uint32_t *cm = c.conn + (size_t)a2 * c.W;
            for (int w = 0; w < c.W; w++) {
                for (uint32_t bits = cm[w]; bits; bits &= bits - 1u) {
                    const int i = 32 * w + wrsn_ctz(bits);
                    if (c.status[i] != 1) continue;
                    const double ec = c.energy[i] - c.cs[i];
                    double e_with = cap;             /* max(ec + rate, capacity) with rate <= alpha / beta^2 */
                    if (ec + ab2 > cap) e_with = fmax(ec + charge_rate_fast(c, m, i), cap);
                    incentive += (c.scr0[i] * inv_tot) * (e_with - (ec < thr ? ec : thr)) * inv_ab2;
                }
            }
            m[WRSN_MC_EXCL] += incentive;
        }
    }
}

WRSN_NOINLINE bool node_in_incentive(Ctx &c, int i) {   /* does an incentive sum read node i? */
    bool in = false;
    for (int a = 0; a < c.M; a++) {
        const double *m = c.mc + a * WRSN_MC_LEN;
        if (m[WRSN_MC_STATUS] != 0.0 && m[WRSN_MC_TYPE] != 0.0 && ((c.conn[a * c.W + (i >> 5)] >> (i & 31)) & 1u)) in = true;
    }
    return in;
}

/* the table nodes of one second of a batch: the previous second's k+1.0 top-up (`book`) and this second's k+0.5 tick
 * (`drain`), as many threads as there are entries */
WRSN_NOINLINE void spec_phase(Ctx &c, int n_spec, int book, int drain) {
    const double cap = c.par[WRSN_P_CAP];
    const double *spec = c.spec.ptr();
    for (int t = c.tid; t < n_spec; t += WRSN_GSZ(c)) {
        const double *sp = spec + t * WRSN_SPEC_LEN;
        const int i = (int)sp[5];
        double en = c.energy[i];
        if (en >= sp[3] && en <= sp[4]) {            /* inside the guards: whole ulps (see spec_second) */
            const double H = sp[2];
            if (book) { en = en + H; en = en < cap ? en : cap; }
            if (drain) { en = (en - sp[0]) + H; en = (en < cap ? en : cap) - sp[1]; }
            c.energy[i] = en;
        } else spec_second(c, t, book, drain);
    }
}

/* the incentive sums of one tick from the pair list (built by reward_loop): one thread per pair computes its term, one
 * thread per charger adds its terms in node order */
WRSN_NOINLINE void pairs_phase(Ctx &c, double tot, int n_pairs) {
    const int G = WRSN_GSZ(c), tid = c.tid;
    if (n_pairs > WRSN_PAIR_MAX) { if (tid < c.M) reward_incentives(c, tot); return; }
    const double thr = c.par[WRSN_P_THR], cap = c.par[WRSN_P_CAP], ab2 = c.par[WRSN_P_MC_AB2];
    const double inv_tot = wrsn_rcp(tot), inv_ab2 = wrsn_rcp(ab2);
    double *pair_term = c.pairs.ptr();
    const int *pair_ids = (const int *)(pair_term + WRSN_PAIR_MAX), *pair_seg = pair_ids + 2 * WRSN_PAIR_MAX;
    for (int p = tid; p < n_pairs; p += G) {
        const int a2 = pair_ids[2 * p], i = pair_ids[2 * p + 1];
        const double ec = c.energy[i] - c.cs[i];
        double e_with = cap;                         /* max(ec + rate, capacity) with rate <= alpha / beta^2 */
        if (ec + ab2 > cap) e_with = fmax(ec + charge_rate_fast(c, c.mc + a2 * WRSN_MC_LEN, i), cap);
        pair_term[p] = (c.scr0[i] * inv_tot) * (e_with - (ec < thr ? ec : thr)) * inv_ab2;
    }
    gsync(c);
    for (int a2 = tid; a2 < c.M; a2 += G) {
        const int p0 = pair_seg[2 * a2], p1 = pair_seg[2 * a2 + 1];
        if (p1 > p0) {
            double incentive = 0.0;
            for (int p = p0; p < p1; p++) incentive += pair_term[p];
            c.mc[a2 * WRSN_MC_LEN + WRSN_MC_EXCL] += incentive;
        }
    }
}

/* ------------------------------------------------------------------ the hot loop: update_reward second by second
 * `n_cycles` consecutive update_reward ticks (WRSN.py:100-127) on the node rows in shared memory.
 * batch == 0 (event path): one tick on the node rows as they are.
 * batch != 0 (whole-cycle batches, nodes_batch): the grid events around every tick are applied on the way — the k+1.0
 *   bookkeeping of the PREVIOUS second (second top-up; energyCS towards its fixed point), then this second's k+0.5
 *   drain, then the tick; the bookkeeping of the last second follows the loop.  A regular node (energyRR == 0, inside
 *   its binade: dec[i] is its per-second decrement) costs one subtraction per second.  The few irregular ones — charged
 *   nodes above all — are listed in a table (c.spec, built by nodes_batch: dec[i] = NaN carrying the table slot); thread
 *   t < n_spec owns entry t, keeps it in registers and works on the shared-memory copy of the node's energy: inside a
 *   binade the relay / own-packet chains and the two top-ups  min(e + energyRR * 0.5, capacity)  each move the energy by a
 *   fixed whole number of ulps (sub_chain's argument; D1, D2, H of the table), so the second is four exact additions
 *   and two minima while the energy stays between the table's guards, and the literal tick (spec_second) otherwise.
 *   The incentive sums work the same way: thread p < n_pairs owns the p-th (charging charger, connected alive node)
 *   pair.
 * Thread tid owns the nodes i = tid, tid + G, ... (slot s = node tid + s * G) and walks them in a ROLLED loop: energy in
 * c.energy, energyCS in c.cs, the per-second decrement in c.scr1, x_n in c.scr0 (overwritten in place by the softmax
 * numerator of the nodes the incentive sums read; nobody else touches a slot's scr0 before the barrier of the tot sum).
 * Rolled, not unrolled into registers: the unrolled slots (one instantiation per slot count) were 31 KB of code that the
 * instruction caches could not hold next to the event code of the other environments on the SM; the rolled loop is one
 * function of about 15 KB for every group size and pays a few shared-memory loads and stores per slot and second (DESIGN
 * §4.1 has the measurement).  Per-slot flags stay in registers.  Nothing in the per-node passes goes through the context
 * record (it sits in the kernel's stack frame): 32-bit shared-memory addresses and registers, computed before the loop.
 * Arithmetic of the tick itself: x_n = energyCS / (energy - threshold + eps) by reciprocal (wrsn_rcp), mean and variance
 * from one pass (sum and sum of squares; two passes when the variance is small against mean^2), 1 / std by wrsn_rsqrt,
 * the softmax numerators by wrsn_exp_b — see the note at those helpers.  A dead node enters the sums with x_n = 0 and
 * its softmax numerator enters tot.  The event path and the batches run this very code, so they produce the same bits
 * (tests: batches == event path). */

/* the (charging charger, connected alive node) pairs of the incentive sums, charger by charger in node order (thread 0
 * builds the list; every thread gets the count) */
WRSN_NOINLINE int reward_pair_list(Ctx &c) {
    double *pair_term = c.pairs.ptr();
    int *pair_ids = (int *)(pair_term + WRSN_PAIR_MAX), *pair_seg = pair_ids + 2 * WRSN_PAIR_MAX;
    if (c.tid == 0) {
        int np = 0;
        for (int a = 0; a < c.M; a++) {
            const double *m = c.mc + a * WRSN_MC_LEN;
            pair_seg[2 * a] = np;
            if (m[WRSN_MC_STATUS] != 0.0 && m[WRSN_MC_TYPE] != 0.0) {
                const uint32_t *cm = c.conn + a * c.W;
                for (int w = 0; w < c.W; w++)
                    for (uint32_t bits = cm[w]; bits; bits &= bits - 1u) {
                        const int i = 32 * w + wrsn_ctz(bits);
                        if (c.status[i] != 1) continue;
                        if (np < WRSN_PAIR_MAX) { pair_ids[2 * np] = a; pair_ids[2 * np + 1] = i; }
                        np++;
                    }
            }
            pair_seg[2 * a + 1] = np;
        }
        c.bcast[8] = np;
    }
    gsync(c);
    return c.bcast[8];
}

/* the textbook two-pass variance sum (np.std) over x_n in scr0, for a tick whose one-pass variance cancels (cold).  Flips
 * the reduction buffer once: the caller does the same with its copy of `buf`. */
WRSN_NOINLINE double reward_two_pass(const Ctx &c, double mean, int buf) {
    const int G = WRSN_GSZ(c);
    const saddr_t a_x = saddr_of(c.scr0.ptr() + c.tid);
    double q = 0.0;
    for (int i = c.tid, o = 0; i < c.N; i += G, o += 8 * G) { const double u = lds64(a_x + o) - mean; q = wrsn_fma(u, u, q); }
    red_sum1(saddr_of(c.red.ptr()), c.tid, G, q, buf);
    return q;
}

WRSN_NOINLINE void reward_loop(Ctx &c, int batch, int n_cycles, double t_reward, int watched, int n_spec) {
    const int N = c.N, G = WRSN_GSZ(c), tid = c.tid, M = c.M;
#if defined(WRSN_HOST_EMU)
    const int NPT = N;                               /* (WRSN_FLAGS_DECL) */
#endif
    const double thr = c.par[WRSN_P_THR], eps = c.par[WRSN_P_EPSENV], inv_n = c.par[WRSN_P_INVN], cap = c.par[WRSN_P_CAP];
    const double ab2 = c.par[WRSN_P_MC_AB2], inv_ab2 = wrsn_rcp(ab2);
    /* this thread's first node in each row; slot s is 8 * s * G bytes further */
    const saddr_t a_e = saddr_of(c.energy.ptr() + tid), a_cs = saddr_of(c.cs.ptr() + tid), a_x = saddr_of(c.scr0.ptr() + tid);
    const saddr_t a_dec = saddr_of(c.scr1.ptr() + tid), a_logc = saddr_of(c.logc.ptr() + tid);
    const saddr_t a_tab = saddr_of(c.exptab.ptr()), a_red = saddr_of(c.red.ptr());
    const int step = 8 * G;
    WRSN_FLAGS_DECL(f_ok); WRSN_FLAGS_DECL(f_inc); WRSN_FLAGS_DECL(f_special); WRSN_FLAGS_DECL(f_unfixed);
    int any_inc = 0, any_unfixed = 0, buf = 0;
    gsync(c);
    _Pragma("unroll 1")
    for (int i = tid, s = 0; i < N; i += G, s++) {
        if (c.status[i] == 0) continue;
        WRSN_FL_SET(f_ok, s);
        if (node_in_incentive(c, i)) { WRSN_FL_SET(f_inc, s); any_inc = 1; }
        if (batch) {
            WRSN_FL_SET(f_unfixed, s); any_unfixed = 1;
            if (c.scr1[i] != c.scr1[i]) WRSN_FL_SET(f_special, s);
        }
    }
    any_inc = red_or(c, any_inc);                    /* (uniform over the environment: it decides about barriers) */
    const int n_pairs = reward_pair_list(c);
    const bool listed = n_pairs <= WRSN_PAIR_MAX && n_pairs <= G && M <= G;   /* one thread per pair, one per charger */
    const bool own_pair = listed && tid < n_pairs;
    saddr_t a_pe = 0, a_pc = 0, a_pq = 0, a_pt = 0, a_excl = 0, a_seg = 0;
    int p_node = 0, seg_n = 0;
    const double *p_mc = nullptr;
    {
        double *pair_term = c.pairs.ptr();
        const int *pair_ids = (const int *)(pair_term + WRSN_PAIR_MAX), *pair_seg = pair_ids + 2 * WRSN_PAIR_MAX;
        if (own_pair) {
            p_mc = c.mc + pair_ids[2 * tid] * WRSN_MC_LEN; p_node = pair_ids[2 * tid + 1];
            a_pe = saddr_of(c.energy.ptr() + p_node); a_pc = saddr_of(c.cs.ptr() + p_node); a_pq = saddr_of(c.scr0.ptr() + p_node);
            a_pt = saddr_of(pair_term + tid);
        }
        if (listed && tid < M) {
            seg_n = pair_seg[2 * tid + 1] - pair_seg[2 * tid];
            a_seg = saddr_of(pair_term + pair_seg[2 * tid]);
            a_excl = saddr_of(c.mc.ptr() + tid * WRSN_MC_LEN + WRSN_MC_EXCL);
        }
    }
    /* this thread's table entry (t = tid; more entries than threads: the rest through spec_second) */
    const bool own_spec = tid < n_spec, more_spec = n_spec > G;
    double sD1 = 0.0, sD2 = 0.0, sH = 0.0, sLo = INFINITY, sHi = -INFINITY;
    saddr_t a_spec_e = 0;
    const saddr_t a_sp = saddr_of(c.spec.ptr() + tid * WRSN_SPEC_LEN);
    if (own_spec) {
        sD1 = lds64(a_sp); sD2 = lds64(a_sp + 8); sH = lds64(a_sp + 16); sLo = lds64(a_sp + 24); sHi = lds64(a_sp + 32);
        a_spec_e = saddr_of(c.energy.ptr() + (int)lds64(a_sp + 40));
    }
    _Pragma("unroll 1")
    for (int j = 0; j < n_cycles; j++) {
        if (watched) { catch_up_for_reward(c, t_reward + (double)j); gsync(c); }
        if (n_spec > 0) {                            /* the table nodes: the previous second's top-up, this second's tick */
            if (own_spec) {
                double en = lds64(a_spec_e);
                if (en >= sLo && en <= sHi) {
                    if (j > 0) { en = en + sH; en = en < cap ? en : cap; }
                    en = (en - sD1) + sH;
                    sts64(a_spec_e, (en < cap ? en : cap) - sD2);
                } else {
                    spec_second(c, tid, j > 0, 1);   /* literal second; the entry may have been rebuilt */
                    sD1 = lds64(a_sp); sD2 = lds64(a_sp + 8); sH = lds64(a_sp + 16); sLo = lds64(a_sp + 24); sHi = lds64(a_sp + 32);
                }
            }
            if (more_spec) { _Pragma("unroll 1") for (int t = tid + G; t < n_spec; t += G) spec_second(c, t, j > 0, 1); }
            gsync(c);
        }
        if (j > 0 && red_or_warp(any_unfixed)) {     /* energyCS towards its fixed point (bookkeeping of the previous second;
                                                        cold: a node gets there after one or two applications) */
            any_unfixed = 0;
            _Pragma("unroll 1")
            for (int i = tid, s = 0, o = 0; i < N; i += G, s++, o += step) {
                if (WRSN_FL_GET(f_unfixed, s)) {
                    const double cs = lds64(a_cs + o), nx = cs_step(cs, lds64(a_logc + o));
                    if (nx == cs) WRSN_FL_CLR(f_unfixed, s);
                    else { sts64(a_cs + o, nx); any_unfixed = 1; }
                }
            }
        }
        double s1 = 0.0, s2 = 0.0;
        _Pragma("unroll 1")
        for (int i = tid, s = 0, o = 0; i < N; i += G, s++, o += step) {
            double x = 0.0;                          /* dead node: energy = capacity, energyCS = 0 */
            if (WRSN_FL_GET(f_ok, s)) {
                double e = lds64(a_e + o);
                if (batch && !WRSN_FL_GET(f_special, s)) { e = e - lds64(a_dec + o); sts64(a_e + o, e); }
                x = lds64(a_cs + o) * wrsn_rcp(e - thr + eps);
            }
            sts64(a_x + o, x);
            s1 += x; s2 = wrsn_fma(x, x, s2);
        }
        red_sum2(a_red, tid, G, s1, s2, buf);
        const double mean = s1 * inv_n;
        double var = wrsn_fma(s2, inv_n, -(mean * mean));
        if (!(var > 1e-3 * (mean * mean))) {         /* cancellation: the textbook two passes (np.std) */
            var = reward_two_pass(c, mean, buf) * inv_n;
            buf ^= 1;
        }
        const double a = var > 0.0 ? wrsn_rsqrt(var) : 1.0 / eps;       /* std == 0 -> std = epsilon (:104-105) */
        double tot = 0.0;
        _Pragma("unroll 1")
        for (int i = tid, s = 0, o = 0; i < N; i += G, s++, o += step) {
            const double q = wrsn_exp_b(a_tab, (lds64(a_x + o) - mean) * a);
            tot += q;
            if (WRSN_FL_GET(f_inc, s)) sts64(a_x + o, q);   /* what the incentive sums read */
        }
        red_sum1(a_red, tid, G, tot, buf);           /* (its barrier also publishes the stores above) */
        if (WRSN_GFIX == 32) gsync(c);
        if (tot == 0.0) tot = eps;
        if (n_pairs > 0) {
            if (listed) {
                if (own_pair) {
                    const double ec = lds64(a_pe) - lds64(a_pc);
                    double e_with = cap;             /* max(ec + rate, capacity) with rate <= alpha / beta^2 */
                    if (ec + ab2 > cap) e_with = fmax(ec + charge_rate_fast(c, p_mc, p_node), cap);
                    sts64(a_pt, (lds64(a_pq) * wrsn_rcp(tot)) * (e_with - (ec < thr ? ec : thr)) * inv_ab2);
                }
                gsync(c);
                if (seg_n > 0) {
                    double incentive = 0.0;
                    _Pragma("unroll 1")
                    for (int p = 0; p < seg_n; p++) incentive += lds64(a_seg + 8 * p);
                    sts64(a_excl, lds64(a_excl) + incentive);
                }
            } else pairs_phase(c, tot, n_pairs);
        }
        if (any_inc || n_spec > 0 || watched || WRSN_GFIX != 32) gsync(c);
    }
    if (batch) {                                     /* bookkeeping of the last second */
        if (n_spec > 0) spec_phase(c, n_spec, 1, 0);
        _Pragma("unroll 1")
        for (int i = tid, s = 0, o = 0; i < N; i += G, s++, o += step)
            if (WRSN_FL_GET(f_unfixed, s)) sts64(a_cs + o, cs_step(lds64(a_cs + o), lds64(a_logc + o)));
        gsync(c);
    }
}

WRSN_D void ev_update_reward(Ctx &c) {
    if (reward_pairs(c)) reward_loop(c, 0, 1, 0.0, 0, 0);   /* otherwise every incentive sum is empty: excl += 0 */
}

/* ------------------------------------------------------------------ WRSN.get_network_fitness (WRSN.py:188-220) -> min */
WRSN_NOINLINE double do_fitness(Ctx &c, double *per_target /* global, may be NULL */) {
    const int N = c.N;
    const double thr = c.par[WRSN_P_THR];
    double *node_t = c.scr0, *lt = c.scr1;
    WRSN_PROF_BEGIN();
    for (int i = c.tid; i < N; i += WRSN_GSZ(c)) {
        double l = 0.0;
        if (c.status[i] == 1) l = (c.cs[i] == 0.0) ? INFINITY : (c.energy[i] - thr) / c.cs[i];
        lt[i] = l;
    }
    gsync(c);
    /* start from the bottleneck of the node's own routing path (receiver by receiver to the base station): a real
       path, hence a valid lower bound of the widest one and usually the widest already, so the relaxation below has
       little or nothing left to do instead of walking the network depth hop by hop */
    for (int i = c.tid; i < N; i += WRSN_GSZ(c)) {
        double v = -1.0;
        if (c.status[i] == 1) {
            if (c.parent[i] == -2) v = lt[i];                      /* direct node: its receiver is the base station */
            else {
                /* (shared memory only: an alive node whose receiver is the base station, parent == -2, is a direct node) */
                double mn = lt[i];
                int h = c.parent[i], hops = 0;
                while (h >= 0 && hops++ < N) {
                    if (c.status[h] != 1) { h = -1; break; }     /* a death the tree does not know yet */
                    mn = fmin(mn, lt[h]);
                    h = c.parent[h];
                }
                if (h == -2) v = mn;
            }
        }
        node_t[i] = v;
    }
    gsync(c);
    for (;;) {                                       /* widest path to the base station; only min / max, so any order is exact */
        int changed = 0;
        for (int i = c.tid; i < N; i += WRSN_GSZ(c)) {
            if (c.status[i] != 1 || c.parent[i] == -2) continue;     /* dead, or direct (receiver = base station) */
            double best = -1.0;
            const int e1 = WRSN_LDG(c.nbr_ptr + i + 1);
            for (int e = WRSN_LDG(c.nbr_ptr + i); e < e1; e++) {
                int j = WRSN_LDG(c.nbr_idx + e);
                if (c.status[j] == 1) { double v = node_t[j]; if (v > best) best = v; }
            }
            if (best >= 0.0) {
                double nv = fmin(lt[i], best);
                if (nv > node_t[i]) { node_t[i] = nv; changed = 1; }
            }
        }
        gsync(c);
        if (!red_or(c, changed)) break;
    }
    double *tt = c.scr1;                             /* lt no longer needed */
    gsync(c);
    for (int t = c.tid; t < c.T; t += WRSN_GSZ(c)) tt[t] = 0.0;
    gsync(c);
    for (int i = c.tid; i < N; i += WRSN_GSZ(c)) {
        double v = node_t[i];
        if (v <= 0.0) continue;
        for (int e = c.tgt_ptr[i]; e < c.tgt_ptr[i + 1]; e++) atomic_max_nonneg(&tt[c.tgt_idx[e]], v);
    }
    gsync(c);
    double mn = INFINITY;
    for (int t = c.tid; t < c.T; t += WRSN_GSZ(c)) {
        double v = tt[t];
        if (per_target) per_target[t] = v;
        mn = fmin(mn, v);
    }
    mn = red_min(c, mn);
    gsync(c);
    WRSN_PROF_END(c, WRSN_H_PROF4);
    return mn;
}

/* ------------------------------------------------------------------ chargers (MobileCharger.py) */
/* all threads: bitmask of nodes with d(node, (x, y)) <= charging_range */
WRSN_NOINLINE void near_mask(Ctx &c, double x, double y, uint32_t *mask) {
    gsync(c);                                        /* `mask` may be a charger's connection mask that another warp is still
                                                        reading (reward_pairs / rr_invariant of the previous event) */
    for (int w = c.tid; w < c.W; w += WRSN_GSZ(c)) mask[w] = 0u;
    gsync(c);
    const double R = c.par[WRSN_P_MC_R];
    for (int i = c.tid; i < c.N; i += WRSN_GSZ(c))
        if (euclid2(c.nx[i], c.ny[i], x, y) <= R) atomic_or_u32(&mask[i >> 5], 1u << (i & 31));
    gsync(c);
}

#define WRSN_FOR_BITS(mask, W, i)                                              \
    for (int w_ = 0; w_ < (W); w_++)                                           \
        for (uint32_t bits_ = (mask)[w_]; bits_; bits_ &= bits_ - 1u)          \
            for (int i = 32 * w_ + wrsn_ctz(bits_), once_ = 1; once_; once_ = 0)

WRSN_D double charge_rate_xy(Ctx &c, double mx, double my, int node) {   /* alpha / (d + beta) ** 2 */
    double t = euclid2(c.nx[node], c.ny[node], mx, my) + c.par[WRSN_P_MC_BETA];
    return c.par[WRSN_P_MC_ALPHA] / (t * t);
}

/* schedule the slot's next event (all threads keep the clock, thread 0 stores) */
WRSN_DI void slot_sched(Ctx &c, Clk &k, double *p, int pc, int prio, double delay) {
    double t = k.now + delay, key = take_seq(k) + (prio ? WRSN_KEY_NORMAL : 0.0);
    if (WRSN_LEAD(c)) { slot_i(p)[WRSN_PRI_PC] = pc; p[WRSN_PR_T] = t; p[WRSN_PR_KEY] = key; }
}

WRSN_DI void cond_check(Ctx &c, Clk &k, int j) {   /* simpy Condition._check for AnyOf (all threads; state read before) */
    double *h = c.hdr;
    if (h[WRSN_H_COND_TRIG + j] != 0.0) return;
    double s = take_seq(k);
    gsync(c);
    if (WRSN_LEAD(c)) { h[WRSN_H_COND_TRIG + j] = 1.0; h[WRSN_H_COND_T + j] = k.now; h[WRSN_H_COND_KEY + j] = WRSN_KEY_NORMAL + s; }
    gsync(c);
}
WRSN_D void cond_check_h(Ctx &c, int j) {          /* leader-only variant used while building the chain */
    double *h = c.hdr;
    if (h[WRSN_H_COND_TRIG + j] != 0.0) return;
    h[WRSN_H_COND_TRIG + j] = 1.0;
    h[WRSN_H_COND_T + j] = h[WRSN_H_NOW]; h[WRSN_H_COND_KEY + j] = WRSN_KEY_NORMAL + take_seq_h(c);
}

/* ------------------------------------------------------------------ lazy charger spans
 * A charger in the middle of a move repeats, once per second, "move_step fires; move() updates the remaining time and
 * starts the next move_step" (MobileCharger.move :85-96); a charger charging where no alive node is in range repeats
 * "charge_step fires; charge() counts the time down and starts the next charge_step" (:59-72, :40-50).  These events
 * read and write only the charger's own record, so they commute with every grid event and with the other chargers.
 * slot_ff() replays such a run of spans in registers — the reference's arithmetic, operation by operation, three
 * insertion counters per span — up to a time limit, or (commit = false) just finds the instant at which the run ends
 * (arrival, exhaustion, end of the charge, or a charge span landing exactly on the node grid, where the reference's
 * insertion order against the grid events would matter).  Everything else about the slot stays with ev_slot(). */
WRSN_DI bool on_grid(double t) {
    const double f = floor(t);
    return t == f || t == f + 0.5 || t == f + 0.1;
}

WRSN_DI bool conn_has_alive(Ctx &c, int a) {
    const double *m = c.mc + a * WRSN_MC_LEN;
    if (m[WRSN_MC_NCONN] == 0.0) return false;
    const uint32_t *cm = c.conn + a * c.W;
    for (int w = 0; w < c.W; w++)
        for (uint32_t bits = cm[w]; bits; bits &= bits - 1u)
            if (c.status[32 * w + wrsn_ctz(bits)] == 1) return true;
    return false;
}

/* A charging charger disconnects and reconnects its nodes once per span (charge_step :40-50, Node.charger_connection /
 * charger_disconnection :134-146): energyRR -= r, then energyRR += r with the same r.  If that leaves every connected
 * alive node's energyRR exactly where it was — always the case for a node charged by this charger alone: (r - r) + r —
 * the spans of the charge are private to the charger (its own energy and countdown) and can be replayed lazily: the
 * charging rate, re-accumulated from zero over the same alive nodes in the same order, repeats as well.  A death, or
 * another charger connecting to / disconnecting from a shared node, ends the run (wake_lazy_*). */
WRSN_DI bool rr_invariant(Ctx &c, int a) {
    const double *m = c.mc + a * WRSN_MC_LEN;
    if (m[WRSN_MC_NCONN] == 0.0) return true;
    const double mx = m[WRSN_MC_X], my = m[WRSN_MC_Y];
    const uint32_t *cm = c.conn + a * c.W;
    for (int w = 0; w < c.W; w++)
        for (uint32_t bits = cm[w]; bits; bits &= bits - 1u) {
            const int i = 32 * w + wrsn_ctz(bits);
            if (c.status[i] == 0) continue;
            const double r = charge_rate_xy(c, mx, my, i), rr = c.rr[i];
            if ((rr - r) + r != rr) return false;
        }
    return true;
}

/* may the pending event of slot s start a lazy run?  0 no, 1 private, 2 private except that update_reward reads the
 * charger's position every second (SURVEY Q2: the orphan process of agent 0 marks it "charging", with the nodes around
 * the base station connected, while it is moving): update_reward then brings the slot up to date first. */
WRSN_D int slot_lazy_ok(Ctx &c, double ur_t, double ur_key, int s) {
    const double *p = slot_of(c, s);
    const int *pi = (const int *)p;
    const int pc = pi[WRSN_PRI_PC];
    if (pc != PC_MS_FIRE && pc != PC_CS_FIRE) return 0;
    const int a = pi[WRSN_PRI_AGENT];
    for (int q = 0; q < c.n_slot; q++)               /* a second running process of the same charger shares its record */
        if (q != s && slot_i(slot_of(c, q))[WRSN_PRI_USED] != 0 && slot_i(slot_of(c, q))[WRSN_PRI_AGENT] == a &&
            slot_of(c, q)[WRSN_PR_T] < INFINITY) return 0;
    const double *m = c.mc + a * WRSN_MC_LEN;
    if (pc == PC_CS_FIRE) return rr_invariant(c, a) ? 1 : 0;
    if (m[WRSN_MC_TYPE] == 0.0 || !conn_has_alive(c, a)) return 1;
    /* spans that fire at the very instant of an update_reward: from the second such span on update_reward always comes
       first (its timeout was inserted earlier); the first one must already be in that order */
    if (p[WRSN_PR_T] == ur_t && p[WRSN_PR_KEY] < ur_key) return 0;
    return 2;
}

/* replay spans of slot s whose event time is < limit; returns the number replayed and, in *t_end, the time of the span
 * event at which the run stops being private (or +inf if the limit came first).
 * mode FF_DRY: nothing is stored.  FF_ALL: every thread of the environment makes the same call, the leader stores.
 * FF_OWN: only the calling thread works on this slot (other threads replay other slots at the same time) and stores;
 * the caller puts barriers around the whole group of calls. */
enum { FF_DRY = 0, FF_ALL = 1, FF_OWN = 2 };
WRSN_D void atomic_add_f64(double *p, double v) {
#if !defined(WRSN_HOST_EMU)
    atomicAdd(p, v);
#else
    *p += v;
#endif
}
WRSN_NOINLINE int slot_ff(Ctx &c, int s, double limit, int mode, double *t_end) {
    double *p = slot_of(c, s);
    const int a = slot_i(p)[WRSN_PRI_AGENT], pc = slot_i(p)[WRSN_PRI_PC];
    double *m = mc_of(c, a);
    const double *par = c.par.ptr();
    const double thr = par[WRSN_P_MC_THR];
    const bool store = mode == FF_OWN || (mode == FF_ALL && WRSN_LEAD(c));
    double tf = p[WRSN_PR_T];
    int n = 0;
    *t_end = INFINITY;
    if (pc == PC_MS_FIRE) {
        const double v = par[WRSN_P_MC_V], pm = par[WRSN_P_MC_PM], pmv = par[WRSN_P_MC_PMV];
        const double destx = p[WRSN_PR_DESTX], desty = p[WRSN_PR_DESTY], vx = p[WRSN_PR_VX], vy = p[WRSN_PR_VY], total = p[WRSN_PR_TOTAL];
        double x = m[WRSN_MC_X], y = m[WRSN_MC_Y], en = m[WRSN_MC_ENERGY];
        double mt = p[WRSN_PR_MT], span = p[WRSN_PR_SPAN], svx = p[WRSN_PR_SVX], svy = p[WRSN_PR_SVY];
        /* Far from the destination and from exhaustion a span is always 1 s: min(mt, 1.0, (energy - threshold) / (pm v))
           with mt >= 1 and energy - threshold >= pm v (x / y >= 1 exactly when x >= y).  Then neither the square root nor
           the two divisions are needed to know the span, and the remaining time `mt` is only needed once, for the
           position the replay stops at (it is a pure function of the position: move :91).  `far` is a safe margin above
           v^2; anything closer takes the literal arithmetic. */
        const double ux = vx / total, uy = vy / total;                            /* move_step :77 (vec / total) * span */
        const double far = v * v * 1.000001;
        bool mt_known = true;
        while (tf < limit) {
            /* (a span that fires exactly on the node grid is still private: a moving charger is not "charging", so no
               grid event reads or writes its record; slot_try_lazy() refuses runs whose LAST event lands on the grid) */
            const double x1 = x + svx, y1 = y + svy, en1 = en - pm * span * v;     /* move_step :77-78 */
            if (mt_known) { if (mt - span <= 0.0) { *t_end = tf; break; } }       /* move :95 (unknown mt: > 1 = span) */
            if (en1 <= thr) { *t_end = tf; break; }                               /* arrival / exhaustion: ev_slot's business */
            const double dx = destx - x1, dy = desty - y1, d2 = dx * dx + dy * dy;
            double span2;
            if (d2 > far && en1 - thr >= pmv) { span2 = 1.0; mt_known = false; }
            else {
                mt = sqrt(d2) / v; mt_known = true;                               /* move :91-94 */
                span2 = fmin(fmin(mt, 1.0), (en1 - thr) / pmv);
            }
            x = x1; y = y1; en = en1; span = span2;
            svx = ux * span2; svy = uy * span2;
            tf = tf + span2; n++;
        }
        if (!mt_known) mt = euclid2(destx, desty, x, y) / v;
        if (mode != FF_DRY && n > 0) {
            if (mode == FF_ALL) gsync(c);
            if (store) {
                m[WRSN_MC_X] = x; m[WRSN_MC_Y] = y; m[WRSN_MC_ENERGY] = en;
                p[WRSN_PR_MT] = mt; p[WRSN_PR_SPAN] = span; p[WRSN_PR_SVX] = svx; p[WRSN_PR_SVY] = svy;
            }
        }
    } else {                                         /* PC_CS_FIRE: a charge whose disconnect / reconnect pairs change nothing */
        double en = m[WRSN_MC_ENERGY], cpa2 = m[WRSN_MC_CPA2], tmp = p[WRSN_PR_CHTMP], span = p[WRSN_PR_CHSPAN];
        const double rate = m[WRSN_MC_RATE];
        const bool jumps = c.hdr[WRSN_H_OPT_NOBATCH] != 1.0;                      /* (test switch: every span literally) */
        while (tf < limit) {
            if (on_grid(tf)) { *t_end = tf; break; }
            /* m one-second spans at once.  While the span stays 1.0 every step subtracts the same `rate` from the energy (the
               same integer number of ulps inside a binade: sub_chain), 1.0 from the two countdowns (exact below 2^53) and adds
               1.0 to the event time (exact inside the time's binade, where on_grid() cannot change either: the fraction of
               tf is preserved).  m is cut so that all of that holds and none of the loop's exits can fire inside the jump;
               whatever is left runs through the literal step below. */
            if (span == 1.0 && tmp > 2.0 && tmp < 1073741824.0 && cpa2 < 4503599627370496.0 && jumps) {
                const double fl = floor(tmp);
                double m = fl == tmp ? tmp - 1.0 : fl;                             /* spans of 1.0 before the last, shorter one */
                m = fmin(m, floor(limit - tf));                                    /* (inf - tf = inf) */
                const int ext = wrsn_biased_exp(tf);
                if (tf > 0.0 && ext > 60 && ext < 1100) m = fmin(m, floor(wrsn_pow2_biased(ext + 1) - tf)); else m = 0.0;
                double en_m = en;
                if (rate != 0.0) {
                    const int ex = wrsn_biased_exp(en);
                    if (en > 0.0 && ex > 60 && ex < 1900) {
                        const double lo = wrsn_pow2_biased(ex), inv_u = wrsn_pow2_biased(2098 - ex), u = wrsn_pow2_biased(ex - 52);
                        const double q = rate * inv_u, rq = rint(q);
                        const double room = en - fmax(lo, thr);
                        if (fabs(q - rq) == 0.5 || !(rq > 0.0) || !(room > 0.0)) m = 0.0;
                        else {
                            m = fmin(m, floor(room / (rq * u)) - 1.0);
                            if (m >= 2.0 && rq * m < 4503599627370496.0) en_m = en - (rq * m) * u; else m = 0.0;
                        }
                    } else m = 0.0;
                }
                if (m >= 2.0) {
                    en = en_m; cpa2 = cpa2 >= m ? cpa2 - m : 0.0; tmp = tmp - m;
                    span = fmin(tmp, 1.0);
                    tf = (tf + (m - 1.0)) + span; n += (int)m;
                    continue;
                }
            }
            const double en1 = en - rate * span;                                   /* charge_step :45 */
            const double cpa21 = fmax(0.0, cpa2 - span);                           /* :46 */
            const double tmp1 = tmp - span;                                        /* charge :69 */
            if (tmp1 == 0.0 || en1 <= thr) { *t_end = tf; break; }
            en = en1; cpa2 = cpa21; tmp = tmp1; span = fmin(tmp1, 1.0);            /* :63-68 (the rate is 0 there: no energy limiter, Q3) */
            tf = tf + span; n++;
        }
        if (mode != FF_DRY && n > 0) {
            if (mode == FF_ALL) gsync(c);
            if (store) {
                m[WRSN_MC_ENERGY] = en; m[WRSN_MC_CPA2] = cpa2; m[WRSN_MC_CHTIME] = tmp;
                p[WRSN_PR_CHTMP] = tmp; p[WRSN_PR_CHSPAN] = span;
            }
        }
    }
    if (mode != FF_DRY && n > 0) {
        /* every span drew three insertion counters (completion of the step, start of the next one, its timeout); they are
           owed until the slot wakes up: only the ORDER of pending events matters, and a lazy slot has none that ties */
        if (store) { p[WRSN_PR_T] = tf; p[WRSN_PR_OWED] += 3.0 * (double)n; }
        if (mode == FF_OWN) atomic_add_f64(&c.hdr[WRSN_H_NLAZY], (double)n);
        else if (store) c.hdr[WRSN_H_NLAZY] += (double)n;
        if (mode == FF_ALL) gsync(c);
    }
    return n;
}

/* after an event of slot s: if its next event starts a private run of at least one span, make the slot lazy */
WRSN_NOINLINE void slot_try_lazy(Ctx &c, double ur_t, double ur_key, int s) {
    double *p = slot_of(c, s);
    if (!(p[WRSN_PR_T] < INFINITY)) return;
    const int kind = slot_lazy_ok(c, ur_t, ur_key, s);
    if (kind == 0) return;
    double t_end;
    const int n = slot_ff(c, s, INFINITY, FF_DRY, &t_end);
    if (n < 1 || on_grid(t_end)) return;             /* arrival / exhaustion on the grid: its order against the grid events
                                                        of that instant is decided by insertion counters — event by event */
    gsync(c);
    if (WRSN_LEAD(c)) { slot_i(p)[WRSN_PRI_LAZY] = kind; p[WRSN_PR_TINT] = t_end; p[WRSN_PR_OWED] = 0.0; }
    gsync(c);
}

/* bring a lazy slot up to date: replay its spans before `limit`; wake = it becomes an ordinary slot again, and its
 * pending event gets the last of the insertion counters its spans drew (returned: how many the clock owes) */
WRSN_NOINLINE double slot_catch_up_core(Ctx &c, int s, double limit, bool wake, double seq) {
    double *p = slot_of(c, s);
    double t_end;
    slot_ff(c, s, limit, FF_ALL, &t_end);
    if (!wake) return 0.0;
    const double owed = p[WRSN_PR_OWED];
    gsync(c);
    if (WRSN_LEAD(c)) {
        slot_i(p)[WRSN_PRI_LAZY] = 0;
        if (owed > 0.0) { p[WRSN_PR_KEY] = WRSN_KEY_NORMAL + (seq + owed - 1.0); p[WRSN_PR_OWED] = 0.0; }
    }
    gsync(c);
    return owed;
}
WRSN_DI void slot_catch_up(Ctx &c, Clk &k, int s, double limit, bool wake) {
    const double owed = slot_catch_up_core(c, s, limit, wake, k.seq);
    k.seq += owed; k.nev += owed;
}
/* bring several lazy slots up to date at once, one thread per slot (they stay lazy): kind 2 = the slots whose position
 * update_reward reads, 1 = every lazy slot */
WRSN_D void catch_up_many(Ctx &c, double limit, int kind) {
    bool any = false;
    for (int q = 0; q < c.n_slot; q++) any = any || slot_i(slot_of(c, q))[WRSN_PRI_LAZY] >= kind;
    if (!any) return;
    gsync(c);
    for (int q = c.tid; q < c.n_slot; q += WRSN_GSZ(c))
        if (slot_i(slot_of(c, q))[WRSN_PRI_LAZY] >= kind) { double t_end; slot_ff(c, q, limit, FF_OWN, &t_end); }
    gsync(c);
}
/* update_reward is about to read the chargers' positions */
WRSN_NOINLINE void catch_up_for_reward(Ctx &c, double t_reward) { catch_up_many(c, t_reward, 2); }

/* a death: every lazy run ends (the alive set of a charge, hence its rate, changes from the next connection on) */
WRSN_DI void wake_lazy_all(Ctx &c, Clk &k) {
    for (int q = 0; q < c.n_slot; q++)
        if (slot_i(slot_of(c, q))[WRSN_PRI_LAZY] != 0) slot_catch_up(c, k, q, k.now, true);
}
/* charger `a` (slot s, not lazy) is about to change the energyRR of its connected nodes: lazy charges that share one of
 * them must re-validate rr_invariant() at the new value */
WRSN_DI void wake_lazy_sharing(Ctx &c, Clk &k, int s, int a) {
    const uint32_t *cm = c.conn + a * c.W;
    for (int q = 0; q < c.n_slot; q++) {
        const int *qi = slot_i(slot_of(c, q));
        if (q == s || qi[WRSN_PRI_LAZY] == 0 || qi[WRSN_PRI_PC] != PC_CS_FIRE) continue;
        const uint32_t *cq = c.conn + qi[WRSN_PRI_AGENT] * c.W;
        uint32_t both = 0u;
        for (int w = 0; w < c.W; w++) both |= cm[w] & cq[w];
        if (both) slot_catch_up(c, k, q, k.now, true);
    }
}

/* Events of one charger process slot, starting with the pending one.  Zero-delay follow-up events of the same slot
 * (process start / completion hops of the generator tree) are executed back to back as long as NO other event of the
 * environment is due at the current instant (`other_t` > now): then the (time, priority, counter) order would pick
 * them next anyway; every hop still draws its insertion counter, so later ties resolve as in the reference. */
WRSN_DI void ev_slot(Ctx &c, Clk &k, int s, double other_t) {
    double *p = slot_of(c, s);
    const int a = slot_i(p)[WRSN_PRI_AGENT];
    double *m = mc_of(c, a);
    uint32_t *cm = c.conn + (size_t)a * c.W;
    const double *par = c.par.ptr();
    const bool lead = WRSN_LEAD(c);
    for (;;) {
        const int pc = slot_i(p)[WRSN_PRI_PC];
        k.nev += 1.0;
        bool again = false;                          /* the slot's next event is due now */
        int nx_pc = 0, nx_prio = 0;                  /* the slot's next event: scheduled at ONE site below */
        double nx_delay = 0.0;
        switch (pc) {
        case PC_OP_INIT: {                           /* MobileCharger.operate_step :105-132, up to the first yield */
            const double dx = p[WRSN_PR_PHY0], dy = p[WRSN_PR_PHY1], ct = p[WRSN_PR_PHY2];
            uint32_t *near = (uint32_t *)c.scr1.ptr();
            near_mask(c, dx, dy, near);
            const double pm = par[WRSN_P_MC_PM], beta = par[WRSN_P_MC_BETA], alpha = par[WRSN_P_MC_ALPHA];
            double used = euclid2(dx, dy, m[WRSN_MC_X], m[WRSN_MC_Y]) * pm;
            double tmp = 0.0;
            WRSN_FOR_BITS(near, c.W, i) {
                if (c.status[i] == 1) {
                    double t = euclid2(dx, dy, c.nx[i], c.ny[i]) + beta;
                    tmp += alpha / (t * t);
                }
            }
            used += tmp * ct;
            used += euclid2(dx, dy, par[WRSN_P_BSX], par[WRSN_P_BSY]) * pm;
            const bool detour = used > m[WRSN_MC_ENERGY] - par[WRSN_P_MC_THR] - par[WRSN_P_MC_CAP200];
            gsync(c);
            if (lead) {
                m[WRSN_MC_CPA0] = dx; m[WRSN_MC_CPA1] = dy; m[WRSN_MC_CPA2] = ct; m[WRSN_MC_TYPE] = 0.0;
                slot_i(p)[WRSN_PRI_STAGE] = detour ? 1 : 3;
                p[WRSN_PR_DESTX] = detour ? par[WRSN_P_BSX] : dx; p[WRSN_PR_DESTY] = detour ? par[WRSN_P_BSY] : dy;
            }
            { nx_pc = PC_MOVE_INIT; nx_prio = WRSN_URGENT; nx_delay = 0.0; } again = true;
            break;
        }
        case PC_MOVE_INIT:                           /* MobileCharger.move :82-84, then the loop head :85-94 */
        case PC_MS_DONE: {                           /* back from move_step :95-96, then the loop head */
            const double destx = p[WRSN_PR_DESTX], desty = p[WRSN_PR_DESTY], v = par[WRSN_P_MC_V];
            const double mx = m[WRSN_MC_X], my = m[WRSN_MC_Y];
            double mt, vx, vy, total, en = m[WRSN_MC_ENERGY], st = m[WRSN_MC_STATUS];
            if (pc == PC_MOVE_INIT) {
                mt = euclid2(destx, desty, mx, my) / v; vx = destx - mx; vy = desty - my; total = mt;
            } else {
                mt = p[WRSN_PR_MT] - p[WRSN_PR_SPAN]; vx = p[WRSN_PR_VX]; vy = p[WRSN_PR_VY]; total = p[WRSN_PR_TOTAL];
                if (en <= par[WRSN_P_MC_THR]) { st = 0.0; en = par[WRSN_P_MC_THR]; }      /* checkStatus */
            }
            gsync(c);
            if (lead) {
                m[WRSN_MC_ENERGY] = en; m[WRSN_MC_STATUS] = st;
                if (pc == PC_MOVE_INIT) { p[WRSN_PR_VX] = vx; p[WRSN_PR_VY] = vy; p[WRSN_PR_TOTAL] = total; }
            }
            if (mt <= 0.0) {
                if (lead) p[WRSN_PR_MT] = mt;
                { nx_pc = PC_MOVE_DONE; nx_prio = WRSN_NORMAL; nx_delay = 0.0; } again = true;
            } else if (st == 0.0) {
                if (lead) p[WRSN_PR_MT] = mt;
                { nx_pc = PC_MOVE_DEADWAIT; nx_prio = WRSN_NORMAL; nx_delay = mt; }
            } else {
                mt = euclid2(destx, desty, mx, my) / v;
                double span = fmin(fmin(mt, 1.0), (en - par[WRSN_P_MC_THR]) / par[WRSN_P_MC_PMV]);
                if (lead) {
                    p[WRSN_PR_MT] = mt; p[WRSN_PR_SPAN] = span;
                    p[WRSN_PR_SVX] = vx / total * span; p[WRSN_PR_SVY] = vy / total * span;
                }
                { nx_pc = PC_MS_INIT; nx_prio = WRSN_URGENT; nx_delay = 0.0; } again = true;
            }
            break;
        }
        case PC_MS_INIT: {                           /* move_step :76 */
            const double span = p[WRSN_PR_SPAN];
            gsync(c);
            { nx_pc = PC_MS_FIRE; nx_prio = WRSN_NORMAL; nx_delay = span; } again = span == 0.0;
            break;
        }
        case PC_MS_FIRE: {                           /* move_step :77-78 */
            const double x = m[WRSN_MC_X] + p[WRSN_PR_SVX], y = m[WRSN_MC_Y] + p[WRSN_PR_SVY];
            const double en = m[WRSN_MC_ENERGY] - par[WRSN_P_MC_PM] * p[WRSN_PR_SPAN] * par[WRSN_P_MC_V];
            gsync(c);
            if (lead) { m[WRSN_MC_X] = x; m[WRSN_MC_Y] = y; m[WRSN_MC_ENERGY] = en; }
            { nx_pc = PC_MS_DONE; nx_prio = WRSN_NORMAL; nx_delay = 0.0; } again = true;
            break;
        }
        case PC_MOVE_DEADWAIT:
            gsync(c);
            { nx_pc = PC_MOVE_DONE; nx_prio = WRSN_NORMAL; nx_delay = 0.0; } again = true;
            break;
        case PC_MOVE_DONE: {                         /* back in operate_step */
            const bool detour = slot_i(p)[WRSN_PRI_STAGE] == 1;
            const double ct = p[WRSN_PR_PHY2];
            gsync(c);
            if (detour) { nx_pc = PC_RC_INIT; nx_prio = WRSN_URGENT; nx_delay = 0.0; }
            else {
                if (lead) { m[WRSN_MC_TYPE] = 1.0; p[WRSN_PR_CHTMP] = ct; }
                { nx_pc = PC_CH_INIT; nx_prio = WRSN_URGENT; nx_delay = 0.0; }
            }
            again = true;
            break;
        }
        case PC_RC_INIT: {                           /* recharge :99-103 */
            const bool at_bs = euclid2(m[WRSN_MC_X], m[WRSN_MC_Y], par[WRSN_P_BSX], par[WRSN_P_BSY]) <= par[WRSN_P_MC_EPS];
            gsync(c);
            if (lead && at_bs) { m[WRSN_MC_X] = par[WRSN_P_BSX]; m[WRSN_MC_Y] = par[WRSN_P_BSY]; m[WRSN_MC_ENERGY] = par[WRSN_P_MC_CAP]; }
            { nx_pc = PC_RC_FIRE; nx_prio = WRSN_NORMAL; nx_delay = 0.0; } again = true;
            break;
        }
        case PC_RC_FIRE:
            gsync(c);
            { nx_pc = PC_RC_DONE; nx_prio = WRSN_NORMAL; nx_delay = 0.0; } again = true;
            break;
        case PC_RC_DONE: {
            const double dx = p[WRSN_PR_PHY0], dy = p[WRSN_PR_PHY1];
            gsync(c);
            if (lead) { slot_i(p)[WRSN_PRI_STAGE] = 3; p[WRSN_PR_DESTX] = dx; p[WRSN_PR_DESTY] = dy; }
            { nx_pc = PC_MOVE_INIT; nx_prio = WRSN_URGENT; nx_delay = 0.0; } again = true;
            break;
        }
        case PC_CH_INIT:                             /* charge :53-58, then the loop head :59-68 */
        case PC_CS_DONE: {                           /* back from charge_step :69-71, then the loop head */
            double tmp, en = m[WRSN_MC_ENERGY], st = m[WRSN_MC_STATUS];
            const double rate = m[WRSN_MC_RATE];
            if (pc == PC_CH_INIT) {
                tmp = p[WRSN_PR_CHTMP];
                near_mask(c, m[WRSN_MC_X], m[WRSN_MC_Y], cm);
                int n = 0;
                for (int w = 0; w < c.W; w++) n += wrsn_popc(cm[w]);
                gsync(c);
                if (lead) m[WRSN_MC_NCONN] = n;
            } else {
                tmp = p[WRSN_PR_CHTMP] - p[WRSN_PR_CHSPAN];
                if (en <= par[WRSN_P_MC_THR]) { st = 0.0; en = par[WRSN_P_MC_THR]; }      /* checkStatus */
                gsync(c);
                if (lead) { m[WRSN_MC_ENERGY] = en; m[WRSN_MC_STATUS] = st; }
            }
            if (lead) { p[WRSN_PR_CHTMP] = tmp; m[WRSN_MC_CHTIME] = tmp; }
            if (tmp == 0.0) { { nx_pc = PC_CH_DONE; nx_prio = WRSN_NORMAL; nx_delay = 0.0; } again = true; }
            else if (st == 0.0) {
                if (lead) m[WRSN_MC_CPA2] = 0.0;
                { nx_pc = PC_CH_DEADWAIT; nx_prio = WRSN_NORMAL; nx_delay = tmp; }
            } else {
                double span = fmin(tmp, 1.0);
                if (rate != 0.0) span = fmin(span, (en - par[WRSN_P_MC_THR]) / rate);
                if (lead) p[WRSN_PR_CHSPAN] = span;
                { nx_pc = PC_CS_INIT; nx_prio = WRSN_URGENT; nx_delay = 0.0; } again = true;
            }
            break;
        }
        case PC_CS_INIT:                             /* charge_step :40-44 + Node.charger_connection :134-139 */
        case PC_CS_FIRE: {                           /* charge_step :45-50 + Node.charger_disconnection :141-146 */
            const double mx = m[WRSN_MC_X], my = m[WRSN_MC_Y], span = p[WRSN_PR_CHSPAN];
            double rate = m[WRSN_MC_RATE], en = m[WRSN_MC_ENERGY], cpa2 = m[WRSN_MC_CPA2];
            const bool connect = pc == PC_CS_INIT;
            if (!connect) { en = en - rate * span; cpa2 = fmax(0.0, cpa2 - span); }
            /* lazy charges of other chargers that share a node re-validate when this event changes energyRR for good:
               the first connection, the last disconnection, or a disconnect / reconnect pair that does not restore the
               value.  A "quiet" pair (the charge goes on and rr_invariant holds) leaves them alone. */
            bool quiet;
            if (connect) quiet = slot_i(p)[WRSN_PRI_SPARE] != 0;
            else quiet = (p[WRSN_PR_CHTMP] - span != 0.0) && en > par[WRSN_P_MC_THR] && rr_invariant(c, a);
            if (!quiet) wake_lazy_sharing(c, k, s, a);
            gsync(c);
            if (lead) slot_i(p)[WRSN_PRI_SPARE] = (!connect && quiet) ? 1 : 0;
            WRSN_FOR_BITS(cm, c.W, i) {
                if (c.status[i] == 0) continue;
                double r = charge_rate_xy(c, mx, my, i);
                if (lead) c.rr[i] = connect ? c.rr[i] + r : c.rr[i] - r;
                rate = connect ? rate + r : rate - r;
            }
            if (!connect) rate = 0.0;
            if (lead) { m[WRSN_MC_RATE] = rate; m[WRSN_MC_ENERGY] = en; m[WRSN_MC_CPA2] = cpa2; }
            if (connect) { { nx_pc = PC_CS_FIRE; nx_prio = WRSN_NORMAL; nx_delay = span; } again = span == 0.0; }
            else { { nx_pc = PC_CS_DONE; nx_prio = WRSN_NORMAL; nx_delay = 0.0; } again = true; }
            break;
        }
        case PC_CH_DEADWAIT:
            gsync(c);
            { nx_pc = PC_CH_DONE; nx_prio = WRSN_NORMAL; nx_delay = 0.0; } again = true;
            break;
        case PC_CH_DONE:                             /* operate_step returns */
            gsync(c);
            { nx_pc = PC_OP_DONE; nx_prio = WRSN_NORMAL; nx_delay = 0.0; } again = true;
            break;
        case PC_OP_DONE: {                           /* the process event itself: callbacks = condition checks */
            const bool current = slot_i(p)[WRSN_PRI_CURRENT] != 0;
            const int nch = (int)c.hdr[WRSN_H_CHAIN_N], det = (int)c.hdr[WRSN_H_CHAIN_DETACH];
            gsync(c);
            if (lead) { p[WRSN_PR_T] = INFINITY; slot_i(p)[WRSN_PRI_PROCESSED] = 1; if (!current) slot_i(p)[WRSN_PRI_USED] = 0; }
            for (int j = 0; j < nch; j++)
                if ((int)c.hdr[WRSN_H_CHAIN_SLOT + j] == s && j > det) cond_check(c, k, j);
            break;
        }
        default:
            if (lead) { c.hdr[WRSN_H_ERR] = 2.0; p[WRSN_PR_T] = INFINITY; }
            k.stop = 1;
            break;
        }
        if (nx_pc) slot_sched(c, k, p, nx_pc, nx_prio, nx_delay);
        gsync(c);
        if (!again || !(other_t > k.now)) break;
    }
}

/* a condition event of the AnyOf chain */
WRSN_DI void ev_cond(Ctx &c, Clk &k, int j) {
    double *h = c.hdr;
    const int nch = (int)h[WRSN_H_CHAIN_N];
    double det = h[WRSN_H_CHAIN_DETACH];
    k.nev += 1.0;
    /* _build_value: remove the check callbacks of this condition and, recursively, of the nested ones */
    if ((double)j > det) det = (double)j;
    gsync(c);
    if (WRSN_LEAD(c)) { h[WRSN_H_COND_T + j] = INFINITY; h[WRSN_H_CHAIN_DETACH] = det; }
    gsync(c);
    if (j + 1 < nch) { if ((double)(j + 1) > det) cond_check(c, k, j + 1); }
    else k.stop = 1;                                 /* StopSimulation */
}

/* ------------------------------------------------------------------ whole-cycle batches
 * While no charger event, no death and no active update_reward lies ahead, one simulated second of the grid is the
 * same five events over and over: drain (k+0.5), update_reward / Network.operate exit check / bookkeeping (k+1.0),
 * Network.operate connectivity (k+1.1, levels unchanged).  Nobody looks at the node rows in between, so n such cycles
 * are applied at once, node-parallel, with the reference's fp64 results:
 *   - a node that is not being charged (energyRR == 0) loses the same integer number of ulps every cycle while it
 *     stays inside its binade (see sub_chain), so n cycles are ONE exact multiply-subtract;
 *   - any other node replays its cycles one by one in registers;
 *   - energyCS under a constant per-second consumption reaches the fixed point of (cs*10 - lg + lg)/10 after one or
 *     two applications; the loop stops there.
 * A batch never contains a cycle the event-by-event path would send down the serial (possible death) path: the
 * number of cycles is cut to the safe prefix and the rest runs event by event.
 * Returns the number of cycles applied (0: nothing changed). */
WRSN_NOINLINE int replay_cycles(double e, double rr, double es, double er, int nb, int ow, int na, double thr, double cap,
                                int n, double *e_out) {
    const double slack = 1e-6;
    int done = 0;
    for (; done < n; done++) {
        const double e1 = sub_chain(e, es, 0, er, nb);
        if (nb > 0 && !(e1 - thr >= slack)) break;
        const double e2 = fmin(e1 + rr * 0.5, cap);
        const double e3 = sub_chain(e2, es, ow, er, na);
        if (ow + na > 0 && !(e3 - thr >= slack)) break;
        e = fmin(e3 + rr * 0.5, cap);
    }
    *e_out = e;
    return done;
}

/* one node's k+0.5 tick on the fast path (no death possible): relayed packets of lower ids, top-up, own packets,
 * relayed packets of higher ids */
WRSN_NOINLINE double drain_node(double e, double rr, double es, double er, int nb, int ow, int na, double cap) {
    const double e1 = sub_chain(e, es, 0, er, nb);
    const double e2 = fmin(e1 + rr * 0.5, cap);
    return sub_chain(e2, es, ow, er, na);
}

/* the per-cycle decrement dec = K u of a node without top-up (energyRR == 0) and with traffic: inside e's binade [lo, 2 lo)
 * every cycle removes the same K whole ulps (sub_chain).  *m_out: how many cycles may be applied as  e - dec * m  (at most
 * n_max); the count keeps one cycle of margin above lo and above the threshold.  NaN (and *m_out = 0): replay cycle by cycle. */
WRSN_DI double batch_dec(double e, double es, double er, int nb, int ow, int na, double thr, int n_max, int *m_out) {
    const double slack = 1e-6;
    const int n_a = nb + ow + na, n_b = nb + na;
    double dec = NAN;
    int m = 0;
    const int ex = wrsn_biased_exp(e);
    if (e > 0.0 && ex > 60 && ex < 1900) {
        const double lo = wrsn_pow2_biased(ex), inv_u = wrsn_pow2_biased(2098 - ex), u = wrsn_pow2_biased(ex - 52);
        const double qa = es * inv_u, qb = er * inv_u;
        const double ra = rint(qa), rb = rint(qb);
        const bool tie = (fabs(qa - ra) == 0.5) || (n_b > 0 && fabs(qb - rb) == 0.5);
        const double K = ra * (double)n_a + rb * (double)n_b;      /* ulps per cycle */
        if (!tie && K * (double)n_max < 4503599627370496.0) {
            dec = K * u;
            if (K == 0.0) m = n_max;
            else {
                const double room = e - fmax(lo, thr + 2.0 * slack);
                double q = room > 0.0 ? floor(room / dec) - 1.0 : 0.0;
                q = fmin(fmax(q, 0.0), (double)n_max);
                m = (int)q;
                if (m > 0) { const double r = e - dec * (double)m; if (!(r >= lo) || !(r - thr >= slack)) m = 0; }
            }
        }
    }
    if (m == 0) dec = NAN;
    *m_out = m;
    return dec;
}

/* `n_active_max`: cap on the cycles of a batch in which update_reward is active (the step budget's granularity);
 * returns the cycles applied, + 2^30 when they were of the active kind */
/* KIND 0: any batch; 2: only batches of the active kind (the batch kernel: the all-at-once branch is not even compiled in) */
template <int KIND>
WRSN_NOINLINE int nodes_batch(Ctx &c, int n_max, int ur_on, double t_reward, int n_active_max) {
    const int N = c.N;
    const double thr = c.par[WRSN_P_THR], cap = c.par[WRSN_P_CAP], er = c.par[WRSN_P_ERECV];
    const double *h = c.hdr;
    WRSN_PROF_BEGIN();
    if (h[WRSN_H_OPT_NOBATCH] == 1.0 || h[WRSN_H_BFS_DIRTY] != 0.0 || h[WRSN_H_LOG_LITERAL] != 0.0 ||
        h[WRSN_H_LOG_LEN] < (double)WRSN_RING || h[WRSN_H_LOG_UNIFORM] < 10.0) return 0;
    const bool active = KIND == 2 ? true : (ur_on && reward_pairs(c));    /* update_reward looks at every node every second */
    if (active && n_max > n_active_max) n_max = n_active_max;
    int *bc = c.bcast;                               /* [0]: entries of the table of irregular nodes (active batches) */
    if (active) { gsync(c); if (c.tid == 0) bc[0] = 0; gsync(c); }
    /* pass 1: per node, the per-cycle decrement (scr1; NaN = replay cycle by cycle) and the number of safe cycles */
    WRSN_PROFC_BEGIN(pc1);
    int n_safe = n_max;
    _Pragma("unroll 1")
    for (int i = c.tid; i < N; i += WRSN_GSZ(c)) {
        if (c.status[i] != 1) continue;
        const double e = c.energy[i], es = c.esend[i], rr = c.rr[i];
        const int nb = c.nbef[i], na = c.naft[i];
        const int ow = c.parent[i] != -1 ? (int)c.own[i] : 0;
        const int n_a = nb + ow + na, n_b = nb + na;
        double dec = NAN;
        int m = 0;
        if (rr == 0.0 && n_a == 0) { dec = 0.0; m = n_max; }
        else if (rr == 0.0) dec = batch_dec(e, es, er, nb, ow, na, thr, n_max, &m);
        if (dec != dec) {                            /* charged, near a binade edge or near the threshold: literal cycles */
            /* without any charging the node loses at most `cons` per cycle (plus a few ulps of rounding); if that cannot
               bring it within a joule of the threshold, no cycle of the batch can take the serial path because of it */
            const double cons = ((double)n_a * es + (double)n_b * er) * 1.000001 + 1e-9;
            if (e - thr - 1.0 > cons * (double)n_safe) m = n_safe;
            else { double e_end; m = replay_cycles(e, rr, es, er, nb, ow, na, thr, cap, n_safe, &e_end); }
        }
        if (active && dec != dec) {
            /* table entry (reward_loop / spec_second): inside e's binade the chain of relayed packets of lower ids, the
               own packets + relays of higher ids and the top-up  min(e + energyRR * 0.5, cap)  move e by D1, D2 and H — whole
               numbers of ulps — as long as e stays between the guards for the whole second (both top-ups, both chains) */
            const int slot = atomic_add_ret_i32(&bc[0], 1);
            if (slot < WRSN_SPEC_MAX) { spec_entry(c, i, slot, e); dec = nan_with_payload(slot); }
        }
        c.scr1[i] = dec;
        if (m < n_safe) n_safe = m;
    }
    gsync(c);
    n_safe = (int)red_min(c, (double)n_safe);
    WRSN_PROFC_END(c, WRSN_H_PROF1, pc1);
    if (n_safe <= 0) return 0;
    const int n_spec = active ? bc[0] : 0;
    if (n_spec > WRSN_SPEC_MAX) return 0;            /* more irregular nodes than the table holds: this second event by event */
    const double L = (double)WRSN_RING;
    WRSN_PROFC_BEGIN(pc2);
    if (KIND != 2 && !active) {
        /* pass 2: all cycles at once */
        _Pragma("unroll 1")
        for (int i = c.tid; i < N; i += WRSN_GSZ(c)) {
            if (c.status[i] != 1) continue;
            const double dec = c.scr1[i];
            if (dec == dec) c.energy[i] = c.energy[i] - dec * (double)n_safe;
            else {
                double e_end;
                const int nb = c.nbef[i], na = c.naft[i];
                const int ow = c.parent[i] != -1 ? (int)c.own[i] : 0;
                replay_cycles(c.energy[i], c.rr[i], c.esend[i], er, nb, ow, na, thr, cap, n_safe, &e_end);
                c.energy[i] = e_end;
            }
            const double lg = c.logc[i];
            double cs = c.cs[i];
            for (int t = 0; t < n_safe; t++) {       /* Node.py:75 with log[0] == log_energy */
                const double nx = div_pos(cs * L - lg + lg, L);
                if (nx == cs) break;
                cs = nx;
            }
            c.cs[i] = cs;
        }
        gsync(c);
        WRSN_PROFC_END(c, WRSN_H_PROF2, pc2);
    } else {
        /* pass 2: cycle by cycle, because update_reward reads every node at every k+1.0 (before the bookkeeping): the
           drain, the tick and the previous second's bookkeeping in one pass over the nodes per second (reward_loop) */
        int watched = 0;                             /* is there a lazy move whose position update_reward reads (Q2)? */
        for (int q = 0; q < c.n_slot; q++) watched |= slot_i(slot_of(c, q))[WRSN_PRI_LAZY] == 2 ? 1 : 0;
        reward_loop(c, 1, n_safe, t_reward, watched, n_spec);
        WRSN_PROFC_END(c, WRSN_H_PROF3, pc2);
    }
    if (c.tid == 0) {
        double *hw = c.hdr;
        hw[WRSN_H_LOG_HEAD] = (double)(((int)hw[WRSN_H_LOG_HEAD] + n_safe) % WRSN_RING);
        if (hw[WRSN_H_LOG_UNIFORM] < 1e9) hw[WRSN_H_LOG_UNIFORM] = fmin(hw[WRSN_H_LOG_UNIFORM] + (double)n_safe, 1e9);
        hw[WRSN_H_NTICKS] += (double)n_safe;
        hw[WRSN_H_NBATCH] += (double)n_safe;
    }
    gsync(c);
    WRSN_PROF_END(c, WRSN_H_PROF2);
    return n_safe + (active ? (1 << 30) : 0);
}

/* ------------------------------------------------------------------ the event loop: env.run(...) */
/* Whole cycles strictly before the next charger / condition / until event, seen from the k+0.5 drain of the node block at
 * `gt`: the canonical pending set is {drain now, update_reward and the exit check of Network.operate at +0.5 (in that
 * order)}.  Returns how many (0: this second runs event by event). */
WRSN_DI int batch_window(Ctx &c, const Clk &k, double gt, double maxtime) {
    const double H = fmin(fmin(k.mc_t, k.until_t), maxtime - 2.0);
    const bool ur_on = k.ur_t < INFINITY, net_on = k.net_t < INFINITY;
    if (!(gt + 1.0 <= H && (!net_on || (k.net_state == 2 && k.net_t == gt + 0.5 && c.hdr[WRSN_H_ALIVE] != 0.0)) &&
          (!ur_on || (k.ur_t == gt + 0.5 && (!net_on || k.ur_key < k.net_key))))) return 0;
    const double span = fmin(H - gt, 1048576.0);
    int n = (int)span;
    while (n > 0 && !(gt + (double)n <= H)) n--;
    return n;
}
/* the clock after `batched` cycles: every cycle drew its insertion counters in the order drain, [update_reward,] [exit
 * check,] bookkeeping, [connectivity] (Network.operate may have ended, Q1) */
WRSN_DI void batch_commit(Clk &k, double gt, int batched) {
    const bool ur_on = k.ur_t < INFINITY, net_on = k.net_t < INFINITY;
    const double nb = (double)batched;
    const double per = 2.0 + (ur_on ? 1.0 : 0.0) + (net_on ? 2.0 : 0.0);
    double s0 = k.seq + per * (nb - 1.0);
    if (ur_on) { s0 += 1.0; k.ur_key = WRSN_KEY_NORMAL + s0; k.ur_t += nb; }
    if (net_on) { s0 += 1.0; k.net_key = WRSN_KEY_NORMAL + (s0 + 2.0); k.net_t += nb; }
    k.nodes_key = WRSN_KEY_NORMAL + (s0 + 1.0);
    k.seq += per * nb; k.nev += per * nb - 1.0;
    k.nodes_t = gt + nb;
    k.now = net_on ? (k.net_t - 1.0) + 0.1 : gt + (nb - 0.5);
}
WRSN_D bool batch_ready(Ctx &c) {                   /* the preconditions nodes_batch checks first (cheap: header fields) */
    const double *h = c.hdr;
    return !(h[WRSN_H_OPT_NOBATCH] == 1.0 || h[WRSN_H_BFS_DIRTY] != 0.0 || h[WRSN_H_LOG_LITERAL] != 0.0 ||
             h[WRSN_H_LOG_LEN] < (double)WRSN_RING || h[WRSN_H_LOG_UNIFORM] < 10.0);
}
WRSN_D bool any_watched(Ctx &c) {                   /* a lazy move whose position update_reward reads (Q2)? */
    bool w = false;
    for (int q = 0; q < c.n_slot; q++) w = w || slot_i(slot_of(c, q))[WRSN_PRI_LAZY] == 2;
    return w;
}
#define WRSN_SPLIT_MIN_CYCLES 4                     /* shorter active batches are not worth a launch of their own */

/* `budget` > 0: stop at an event boundary once the launch has done that many work units (one per event handled, plus
 * one per simulated second in which update_reward is active — the expensive kind) and return 1: the clock is stored
 * as it is, the pending run(until) / AnyOf chain stay pending, and the next launch continues where this one stopped.
 * A launch then lasts as long as the budget allows, not as long as its slowest environment's whole step.
 * `split` != 0 (the events kernel of a split step, wrsn_dims.step_rounds): additionally stop — return 2 — in front of a
 * batch of the active kind; the batch kernel (run_batches) takes it from there.  The hot second-by-second loop then runs in
 * launches that contain nothing else: its code stays in the SMs' instruction caches instead of competing with the event
 * machinery of the environments next door (profiles/r02*_icache.md). */
WRSN_DI int run_loop(Ctx &c, int budget, int split, int *work = nullptr) {
    Clk k;
    clk_load(c, k);
    k.work = 0;
    const double maxtime = c.par[WRSN_P_MAXTIME];
    bool rescan = true;
    int interrupted = 0;
    for (long guard = 0; guard < 400000000L; guard++) {
        if (budget > 0 && k.work >= budget) { interrupted = 1; break; }
        k.work++;
        if (rescan) { WRSN_PROFB_BEGIN(); mc_scan(c, k); rescan = false; WRSN_PROFB_END(c, WRSN_H_PROF4); }
        /* earliest of the grid items (Network.operate, update_reward, the node block, run(until=t)) */
        int gk = K_NODES;
        double gt = k.nodes_t, gkey = k.nodes_key;
        if (ev_before(k.net_t, k.net_key, gt, gkey)) { gk = K_NET; gt = k.net_t; gkey = k.net_key; }
        if (ev_before(k.ur_t, k.ur_key, gt, gkey)) { gk = K_UR; gt = k.ur_t; gkey = k.ur_key; }
        if (ev_before(k.until_t, k.until_key, gt, gkey)) { gk = K_UNTIL; gt = k.until_t; gkey = k.until_key; }
        if (ev_before(k.mc_t, k.mc_key, gt, gkey)) {
            k.now = k.mc_t;
            if (k.mc_idx < c.n_slot) {
                const int s = k.mc_idx;
                { WRSN_PROFB_BEGIN();
                if (slot_i(slot_of(c, s))[WRSN_PRI_LAZY] != 0) slot_catch_up(c, k, s, k.mc_t, true);   /* its run of private spans ends now */
                WRSN_PROFB_END(c, WRSN_H_PROF2); }
                double other = fmin(fmin(k.mc_other_t, k.nodes_t), fmin(fmin(k.net_t, k.ur_t), k.until_t));
                { WRSN_PROFB_BEGIN();
                ev_slot(c, k, s, other);
                slot_try_lazy(c, k.ur_t, k.ur_key, s);
                WRSN_PROFB_END(c, WRSN_H_PROF1); }
            } else ev_cond(c, k, k.mc_idx - c.n_slot);
            rescan = true;
        } else {
            if (gk == K_NODES) {
                int batched = 0;
                if (k.nodes_phase == 1 && !k.nobatch_once) {
                    const int n = batch_window(c, k, gt, maxtime);
                    if (n > 0) {
                        const bool ur_on = k.ur_t < INFINITY;
                        if (split && n >= WRSN_SPLIT_MIN_CYCLES && ur_on && batch_ready(c) && reward_pairs(c) && !any_watched(c)) {
                            interrupted = 2;             /* the batch kernel's: nothing of this event has happened yet */
                            break;
                        }
                        k.now = gt;
                        const int cap_active = budget > 0 ? (budget - k.work > 8 ? budget - k.work : 8) : n;
                        batched = nodes_batch<0>(c, n, ur_on ? 1 : 0, gt + 0.5, cap_active);
                        if (batched >= (1 << 30)) { batched -= 1 << 30; k.work += batched; }
                        if (batched > 0) { k.nev += 1.0; batch_commit(k, gt, batched); }
                    }
                }
                if (!batched) {
                    WRSN_PROFB_BEGIN();
                    k.now = gt; k.nev += 1.0;
                    if (k.nodes_phase == 1) {
                        k.nobatch_once = 0;
                        ev_nodes_drain(c); k.nodes_phase = 2;
                        if (c.hdr[WRSN_H_BFS_DIRTY] != 0.0) { wake_lazy_all(c, k); rescan = true; }
                    }
                    else { ev_nodes_book(c); k.nodes_phase = 1; }
                    k.nodes_t = gt + 0.5; k.nodes_key = WRSN_KEY_NORMAL + take_seq(k);
                    WRSN_PROFB_END(c, WRSN_H_PROF3);
                }
            } else if (gk == K_NET) {                /* Network.operate :74-80 */
                k.now = gt; k.nev += 1.0;
                if (k.net_state == 1) {
                    if (c.hdr[WRSN_H_BFS_DIRTY] != 0.0) do_bfs(c);
                    k.net_t = gt + 0.9; k.net_key = WRSN_KEY_NORMAL + take_seq(k); k.net_state = 2;
                } else if (c.hdr[WRSN_H_ALIVE] == 0.0 || gt >= maxtime) k.net_t = INFINITY;
                else { k.net_t = gt + 0.1; k.net_key = WRSN_KEY_NORMAL + take_seq(k); k.net_state = 1; }
            } else if (gk == K_UR) {
                k.now = gt; k.nev += 1.0;
                WRSN_PROFB_BEGIN();
                catch_up_for_reward(c, gt);
                ev_update_reward(c);
                WRSN_PROFB_END(c, WRSN_H_PROF3);
                k.ur_t = gt + 1.0; k.ur_key = WRSN_KEY_NORMAL + take_seq(k);
            } else {                                 /* K_UNTIL */
                k.now = gt; k.nev += 1.0;
                k.until_t = INFINITY; k.stop = 1;
            }
        }
        if (k.stop) break;
    }
    /* whoever looks at the chargers next (decider scan, observation, the next step) sees them as of now */
    { WRSN_PROFB_BEGIN();
    catch_up_many(c, k.now, 1);
    WRSN_PROFB_END(c, WRSN_H_PROF2); }
    clk_store(c, k);
    if (work) *work = k.work;                        /* (the rule rollout's launch-wide budget) */
    return interrupted;
}

/* The batch kernel of a split step: as long as the environment's next event is the k+0.5 drain of the node block in
 * front of a batch of the active kind, apply it (at most `budget` simulated seconds per launch).  Returns 2 when the
 * budget ran out in front of another such batch, 1 when anything else is next (the events kernel's).  A second that
 * cannot be batched (a possible death, more irregular nodes than the table holds) goes back with `nobatch_once` set. */
WRSN_DI int run_batches(Ctx &c, int budget) {
    Clk k;
    clk_load(c, k);
    k.work = 0;
    mc_scan(c, k);                                   /* (nothing in here moves a charger event) */
    const double maxtime = c.par[WRSN_P_MAXTIME];
    int ret = 1;
    for (int guard = 0; guard < 1000000; guard++) {
        int gk = K_NODES;
        double gt = k.nodes_t, gkey = k.nodes_key;
        if (ev_before(k.net_t, k.net_key, gt, gkey)) gk = K_NET;
        if (ev_before(k.ur_t, k.ur_key, gt, gkey)) gk = K_UR;
        if (ev_before(k.until_t, k.until_key, gt, gkey)) gk = K_UNTIL;
        if (gk != K_NODES || ev_before(k.mc_t, k.mc_key, gt, gkey) || k.nodes_phase != 1 || k.nobatch_once) break;
        const int n = batch_window(c, k, gt, maxtime);
        if (n < WRSN_SPLIT_MIN_CYCLES || !(k.ur_t < INFINITY) || !batch_ready(c) || !reward_pairs(c) || any_watched(c)) break;
        if (k.work >= budget) { ret = 2; break; }
        k.now = gt;
        int batched = nodes_batch<2>(c, n, 1, gt + 0.5, budget - k.work > 8 ? budget - k.work : 8);
        if (batched >= (1 << 30)) batched -= 1 << 30;
        if (batched <= 0) { k.nobatch_once = 1; break; }
        k.work += batched;
        k.nev += 1.0;
        batch_commit(k, gt, batched);
    }
    clk_store(c, k);
    return ret;
}

/* ------------------------------------------------------------------ entry points (one environment) */

/* NetworkIO.makeNetwork + the t = 0 starts of Network.operate / update_reward / Node.operate */
WRSN_D void entry_init_network(Ctx &c, int with_reward) {
    for (int i = c.tid; i < c.Npad; i += WRSN_GSZ(c)) {
        bool real = i < c.N;
        c.energy[i] = real ? c.par[WRSN_P_CAP] : 0.0;
        c.rr[i] = 0.0; c.cs[i] = 0.0; c.esend[i] = 0.0; c.logc[i] = 0.0;
        c.nbef[i] = 0; c.naft[i] = 0; c.level[i] = -1; c.parent[i] = -1;
        c.status[i] = real ? 1 : 0;
        c.logtick[i] = 0.0;
        for (int k = 0; k < WRSN_RING; k++) c.ring[(size_t)k * c.Npad + i] = 0.0;
    }
    for (int w = c.tid; w < c.Tw; w += WRSN_GSZ(c)) c.tact[w] = tact_word_mask(c, w);
    for (int w = c.tid; w < (c.M > 0 ? c.M : 1) * c.W; w += WRSN_GSZ(c)) c.conn[w] = 0u;
    for (int k = c.tid; k < WRSN_H_LEN; k += WRSN_GSZ(c)) c.hdr[k] = 0.0;
    for (int k = c.tid; k < (c.M > 0 ? c.M : 1) * WRSN_MC_LEN; k += WRSN_GSZ(c)) c.mc[k] = 0.0;
    for (int k = c.tid; k < c.n_slot * WRSN_PR_LEN; k += WRSN_GSZ(c)) c.proc[k] = (k % WRSN_PR_LEN) == WRSN_PR_T ? INFINITY : 0.0;
    for (int j = c.tid; j < WRSN_MAX_MC; j += WRSN_GSZ(c)) c.hdr[WRSN_H_COND_T + j] = INFINITY;
    gsync(c);
    for (int i = c.tid; i < c.N; i += WRSN_GSZ(c)) check_status_node(c, i);   /* Node.__init__ :43 */
    if (c.tid == 0) {
        double *h = c.hdr;
        h[WRSN_H_ALIVE] = 1.0; h[WRSN_H_BFS_DIRTY] = 1.0; h[WRSN_H_CHAIN_DETACH] = -1.0;
        /* scheduling order at t = 0: Network.operate's timeout(0.1), update_reward's timeout(1.0), the nodes'
           timeout(0.5) (the process starts themselves are URGENT events at t = 0 and have all run) */
        h[WRSN_H_NET_ON] = 1.0; h[WRSN_H_NET_T] = 1.0 / 10.0; h[WRSN_H_NET_SEQ] = take_seq_h(c); h[WRSN_H_NET_STATE] = 1.0;
        if (with_reward) { h[WRSN_H_UR_ON] = 1.0; h[WRSN_H_UR_T] = 1.0; h[WRSN_H_UR_SEQ] = take_seq_h(c); }
        h[WRSN_H_NODES_T] = 0.5; h[WRSN_H_NODES_SEQ] = take_seq_h(c); h[WRSN_H_NODES_PHASE] = 1.0;
    }
    gsync(c);
}

/* env.run(until=t) */
WRSN_D void entry_run_until(Ctx &c, double at) {
    if (!(at > c.hdr[WRSN_H_NOW])) return;
    gsync(c);
    if (c.tid == 0) {
        c.hdr[WRSN_H_UNTIL_ON] = 1.0; c.hdr[WRSN_H_UNTIL_T] = at; c.hdr[WRSN_H_UNTIL_SEQ] = take_seq_h(c);
    }
    gsync(c);
    run_loop(c, 0, 0);
}

WRSN_D int scan_decider(Ctx &c) {                  /* WRSN.py:321-322 */
    for (int a = 0; a < c.M; a++) {
        const double *m = mc_of(c, a);
        if (euclid2(m[WRSN_MC_X], m[WRSN_MC_Y], m[WRSN_MC_CPA0], m[WRSN_MC_CPA1]) < c.par[WRSN_P_EPSENV] &&
            m[WRSN_MC_CPA2] == 0.0) return a;
    }
    return -1;
}

/* leader: env.process(agent.operate_step(phy)) */
WRSN_D int new_slot_h(Ctx &c, int agent, double phy0, double phy1, double phy2) {
    int s = -1;
    for (int k = 0; k < c.n_slot; k++) if (slot_i(slot_of(c, k))[WRSN_PRI_USED] == 0) { s = k; break; }
    if (s < 0) { c.hdr[WRSN_H_ERR] = 3.0; return -1; }
    double *p = slot_of(c, s);
    for (int k = 0; k < WRSN_PR_LEN; k++) p[k] = 0.0;
    int *pi = slot_i(p);
    pi[WRSN_PRI_USED] = 1; pi[WRSN_PRI_CURRENT] = 1; pi[WRSN_PRI_AGENT] = agent; pi[WRSN_PRI_PC] = PC_OP_INIT;
    p[WRSN_PR_PHY0] = phy0; p[WRSN_PR_PHY1] = phy1; p[WRSN_PR_PHY2] = phy2;
    p[WRSN_PR_T] = c.hdr[WRSN_H_NOW]; p[WRSN_PR_KEY] = take_seq_h(c);       /* URGENT */
    return s;
}


/* the rest of WRSN.reset after env.run(until=warm_up) (WRSN.py:44-83) */
WRSN_D void entry_reset_finish(Ctx &c, ReqOut *r) {
    if (c.tid == 0) {
        for (int a = 0; a < c.M; a++) {
            double *m = mc_of(c, a);
            for (int k = 0; k < WRSN_MC_LEN; k++) m[k] = 0.0;
            m[WRSN_MC_X] = c.par[WRSN_P_BSX]; m[WRSN_MC_Y] = c.par[WRSN_P_BSY];
            m[WRSN_MC_ENERGY] = c.par[WRSN_P_MC_CAP]; m[WRSN_MC_STATUS] = 1.0;
            if (m[WRSN_MC_ENERGY] <= c.par[WRSN_P_MC_THR]) { m[WRSN_MC_STATUS] = 0.0; m[WRSN_MC_ENERGY] = c.par[WRSN_P_MC_THR]; }
            m[WRSN_MC_CPA0] = c.par[WRSN_P_BSX]; m[WRSN_MC_CPA1] = c.par[WRSN_P_BSY]; m[WRSN_MC_CPA2] = 0.0;
            m[WRSN_MC_SLOT] = -1.0;
        }
        for (int k = 0; k < c.n_slot * WRSN_PR_LEN; k++) c.proc[k] = (k % WRSN_PR_LEN) == WRSN_PR_T ? INFINITY : 0.0;
        for (int j = 0; j < WRSN_MAX_MC; j++) c.hdr[WRSN_H_COND_T + j] = INFINITY;
        for (int w = 0; w < c.M * c.W; w++) c.conn[w] = 0u;
        c.hdr[WRSN_H_CHAIN_N] = 0.0; c.hdr[WRSN_H_CHAIN_DETACH] = -1.0; c.hdr[WRSN_H_HANG] = 0.0;
    }
    gsync(c);
    double fit = do_fitness(c, (double *)0);
    if (c.tid == 0) {
        c.hdr[WRSN_H_FIT_MIN] = fit;
        const double f0 = c.par[WRSN_P_F0], f1 = c.par[WRSN_P_F1], f2 = c.par[WRSN_P_F2], f3 = c.par[WRSN_P_F3];
        for (int a = 0; a < c.M; a++) {
            double *m = mc_of(c, a);
            m[WRSN_MC_ACT0] = (c.par[WRSN_P_BSX] - f0) / (f1 - f0);          /* down_mapping :86-88 */
            m[WRSN_MC_ACT1] = (c.par[WRSN_P_BSY] - f2) / (f3 - f2);
            m[WRSN_MC_ACT2] = 0.0;
            m[WRSN_MC_SLOT] = new_slot_h(c, a, m[WRSN_MC_CPA0], m[WRSN_MC_CPA1], m[WRSN_MC_CPA2]);
            m[WRSN_MC_PREVFIT] = fit; m[WRSN_MC_EXCL] = 0.0;
        }
        int id = scan_decider(c);
        r->agent = id; r->terminal = c.hdr[WRSN_H_ALIVE] == 1.0 ? 0 : 1; r->now = c.hdr[WRSN_H_NOW];
        r->reward = id >= 0 ? 0.0 : NAN; r->detail[0] = r->detail[1] = id >= 0 ? 0.0 : NAN;
        for (int k = 0; k < 3; k++) r->act[k] = id >= 0 ? mc_of(c, id)[WRSN_MC_ACT0 + k] : NAN;
        r->flags = c.hdr[WRSN_H_ERR] != 0.0 ? 2 : 0;
        if (id >= 0) c.hdr[WRSN_H_NDECISIONS] += 1.0;
    }
    gsync(c);
}

/* WRSN.step (WRSN.py:289-330) */
/* `budget`: see run_loop.  A step that ran out of budget returns agent = -4 ("in flight") and hdr[INFLIGHT] = 1; the
 * next call for this environment ignores agent_id / input_action and continues the same env.run(until=general_process). */
WRSN_D void entry_in_flight(Ctx &c, ReqOut *r, int code) {       /* the request record of a step that continues later */
    if (c.tid == 0) {
        c.hdr[WRSN_H_INFLIGHT] = (double)code; c.hdr[WRSN_H_NRESUME] += 1.0;
        r->now = c.hdr[WRSN_H_NOW]; r->flags = c.hdr[WRSN_H_ERR] != 0.0 ? 2 : 0; r->agent = -4; r->terminal = 0;
        r->reward = NAN; r->detail[0] = r->detail[1] = NAN;
        for (int k = 0; k < 3; k++) r->act[k] = NAN;
    }
    gsync(c);
}

/* the batch kernel of a split step (wrsn_dims.step_rounds): only for environments with hdr[INFLIGHT] == 2 */
WRSN_D void entry_batches(Ctx &c, ReqOut *r, int budget) {
    const int code = run_batches(c, budget > 0 ? budget : (1 << 30));
    gsync(c);
    entry_in_flight(c, r, code);
}

/* `work` (may be NULL): the work units the call used, for a caller that spreads one budget over several steps */
WRSN_D void entry_step(Ctx &c, int agent_id, const double *input_action, ReqOut *r, int budget, int split, int *work = nullptr) {
    const bool resume = c.hdr[WRSN_H_INFLIGHT] != 0.0;
    gsync(c);
    if (c.tid == 0 && !resume) {
        double *h = c.hdr;
        if (agent_id >= 0 && agent_id < c.M) {       /* :290-305 */
            double *m = mc_of(c, agent_id);
            double act[3];
            for (int k = 0; k < 3; k++) act[k] = fmin(fmax(input_action[k], 0.0), 1.0);   /* np.clip */
            for (int k = 0; k < 3; k++) m[WRSN_MC_ACT0 + k] = act[k];
            const double f0 = c.par[WRSN_P_F0], f1 = c.par[WRSN_P_F1], f2 = c.par[WRSN_P_F2], f3 = c.par[WRSN_P_F3];
            double phy0 = act[0] * (f1 - f0) + f0;                                        /* translate :95-98 */
            double phy1 = act[1] * (f3 - f2) + f2;
            double phy2 = c.par[WRSN_P_CTM] * act[2];
            int old = (int)m[WRSN_MC_SLOT];
            if (old >= 0) {
                int *po = slot_i(slot_of(c, old));
                po[WRSN_PRI_CURRENT] = 0;
                po[WRSN_PRI_LAZY] = 0;               /* two processes now share this charger's record: no private runs */
                if (po[WRSN_PRI_PROCESSED] != 0) po[WRSN_PRI_USED] = 0;
            }
            m[WRSN_MC_SLOT] = new_slot_h(c, agent_id, phy0, phy1, phy2);
            m[WRSN_MC_PREVFIT] = h[WRSN_H_FIT_MIN];   /* the network has not moved since the last request (refreshed at every request
                                                         that leaves the environment steppable: a decider's, an implicit None's) */
            m[WRSN_MC_EXCL] = 0.0;
        } else if (agent_id >= c.M) h[WRSN_H_ERR] = 4.0;
        /* general_process = net_process | p_0 | p_1 ... over chargers with status != 0 (:307-310) */
        int n = 0;
        h[WRSN_H_CHAIN_DETACH] = -1.0;
        for (int a = 0; a < c.M; a++) {
            const double *m = mc_of(c, a);
            if (m[WRSN_MC_STATUS] == 0.0) continue;
            int s = (int)m[WRSN_MC_SLOT];
            h[WRSN_H_CHAIN_SLOT + n] = s; h[WRSN_H_COND_TRIG + n] = 0.0; h[WRSN_H_COND_T + n] = INFINITY;
            if (s >= 0 && slot_i(slot_of(c, s))[WRSN_PRI_PROCESSED] != 0) cond_check_h(c, n);   /* operand already processed */
            n++;
        }
        h[WRSN_H_CHAIN_N] = n;
        h[WRSN_H_HANG] = n == 0 ? 1.0 : 0.0;
    }
    gsync(c);
    const int watched = (int)c.hdr[WRSN_H_CHAIN_N];
    int interrupted = 0;
    if (watched > 0) interrupted = run_loop(c, budget, split, work);
    else if (work) *work = 0;
    gsync(c);
    if (interrupted) { entry_in_flight(c, r, interrupted); return; }
    int id = -1;
    if (!(watched == 0 || c.hdr[WRSN_H_ALIVE] == 0.0)) { id = scan_decider(c); if (id < 0) id = -2; }   /* all threads */
    double fit = 0.0;
    if (id >= 0 || id == -2) fit = do_fitness(c, (double *)0);   /* get_reward :222-227; after an implicit None (time has moved, no
                                                                   decider) only the cached minimum is refreshed: the next step(agent,
                                                                   action) reads get_network_fitness() as of now (:303) */
    if (c.tid == 0) {
        c.hdr[WRSN_H_INFLIGHT] = 0.0;
        r->now = c.hdr[WRSN_H_NOW];
        r->flags = (watched == 0 ? 1 : 0) | (c.hdr[WRSN_H_ERR] != 0.0 ? 2 : 0);
        r->agent = id;
        r->terminal = (c.hdr[WRSN_H_ALIVE] == 0.0) ? 1 : 0;
        if (id >= 0) {
            double *m = mc_of(c, id);
            c.hdr[WRSN_H_FIT_MIN] = fit;
            double term_all = fit - m[WRSN_MC_PREVFIT];
            double term_excl = m[WRSN_MC_EXCL] / c.par[WRSN_P_AVGNA];
            r->reward = (term_all * 0.8 + 0.2 * term_excl) / (c.par[WRSN_P_CTM] + c.par[WRSN_P_MTM]);
            r->detail[0] = term_all; r->detail[1] = term_excl;
            for (int k = 0; k < 3; k++) r->act[k] = m[WRSN_MC_ACT0 + k];
            c.hdr[WRSN_H_NDECISIONS] += 1.0;
        } else {
            if (id == -2) c.hdr[WRSN_H_FIT_MIN] = fit;
            r->reward = NAN; r->detail[0] = r->detail[1] = NAN;
            for (int k = 0; k < 3; k++) r->act[k] = NAN;
        }
    }
    gsync(c);
}
