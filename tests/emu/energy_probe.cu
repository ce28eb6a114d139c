/*
 * energy_probe.cu — TEST INFRASTRUCTURE (tests/test_energy_chains.py, tests/test_charger_spans.py).  Scalar entry points into
 * the engine's exact energy arithmetic and its lazy charger spans, so that the closed forms can be compared with literal fp64
 * chains one case at a time.
 *
 * Built twice by the test, never by the package:
 *   - g++ -x c++ with the flags of tests/emu/Makefile: wrsn_engine.cuh under WRSN_HOST_EMU, WRSN_GFIX 1 (the host build);
 *   - nvcc with the library's flags (__graft_entry__.NVCC_FLAGS): the whole of wrsn_kernels.cu, so the probe kernel calls the
 *     g32:: functions with the device's rint, FMA contraction settings and code generation that the library ships.
 *
 * probe_run(op, x, y, n): row k of x (PROBE_IN doubles) -> row k of y (PROBE_OUT doubles).  On the device x and y are device
 * pointers.  The ops and their row layouts are listed in probe_one.
 */
#if defined(__CUDACC__)
#include "wrsn_kernels.cu"
#define PROBE_NS g32
#define PROBE_D __device__
#else
#define WRSN_HOST_EMU 1
#include <stdio.h>
#include <stdlib.h>

#include "wrsn_launch.h"
static thread_local char *wrsn_smem_host = nullptr;
#define WRSN_GFIX 1
namespace host1 {
#include "wrsn_engine.cuh"
}
#define PROBE_NS host1
#define PROBE_D
#endif

#define PROBE_IN 10
#define PROBE_OUT 8

enum { OP_SUB_CHAIN = 0, OP_SUB_CHAIN_FAST, OP_SUB_CHAIN_LITERAL, OP_DRAIN_NODE, OP_REPLAY_CYCLES, OP_SPEC_TERMS, OP_BATCH_DEC,
       OP_RCP, OP_RSQRT, OP_EXP_TAB, OP_CHARGE_RUN, OP_MOVE_SPAN };

/* tab: the exp table in shared memory (device), unused on the host */
template <typename Tab>
PROBE_D static void probe_one(int op, const double *x, double *y, Tab tab) {
    using namespace PROBE_NS;
    for (int k = 0; k < PROBE_OUT; k++) y[k] = 0.0;
    switch (op) {
    case OP_SUB_CHAIN:                               /* e, a, n_single, b, n_pair */
        y[0] = sub_chain(x[0], x[1], (int)x[2], x[3], (int)x[4]); break;
    case OP_SUB_CHAIN_FAST:
        y[0] = sub_chain_fast(x[0], x[1], (int)x[2], x[3], (int)x[4]); break;
    case OP_SUB_CHAIN_LITERAL:
        y[0] = sub_chain_literal(x[0], x[1], (int)x[2], x[3], (int)x[4]); break;
    case OP_DRAIN_NODE:                              /* e, rr, es, er, nb, ow, na, cap */
        y[0] = drain_node(x[0], x[1], x[2], x[3], (int)x[4], (int)x[5], (int)x[6], x[7]); break;
    case OP_REPLAY_CYCLES: {                         /* e, rr, es, er, nb, ow, na, thr, cap, n -> e_out, cycles done */
        double e_out = 0.0;
        y[1] = (double)replay_cycles(x[0], x[1], x[2], x[3], (int)x[4], (int)x[5], (int)x[6], x[7], x[8], (int)x[9], &e_out);
        y[0] = e_out;
        break;
    }
    case OP_SPEC_TERMS: {                            /* e, es, er, rr, nb, ow, na -> D1, D2, H, glo, ghi */
        const SpecTerms s = spec_terms(x[0], x[1], x[2], x[3], (int)x[4], (int)x[5], (int)x[6]);
        y[0] = s.D1; y[1] = s.D2; y[2] = s.H; y[3] = s.glo; y[4] = s.ghi;
        break;
    }
    case OP_BATCH_DEC: {                             /* e, es, er, nb, ow, na, thr, n_max -> dec, m */
        int m = -1;
        y[0] = batch_dec(x[0], x[1], x[2], (int)x[3], (int)x[4], (int)x[5], x[6], (int)x[7], &m);
        y[1] = (double)m;
        break;
    }
    case OP_CHARGE_RUN: {                            /* en, rate, thr, tmp, cpa2, span, tf, limit, jumps -> en, cpa2, tmp, span, tf,
                                                        n, t_end (+inf: the limit came first) */
        ChargeRun r = { x[0], x[4], x[3], x[5], x[6] };
        double t_end = INFINITY;
        const int n = charge_run(r, x[1], x[2], x[7], x[8] != 0.0, &t_end);
        y[0] = r.en; y[1] = r.cpa2; y[2] = r.tmp; y[3] = r.span; y[4] = r.tf; y[6] = (double)n; y[7] = t_end;
        break;
    }
    case OP_MOVE_SPAN:                               /* d2, en1, thr, v, pmv -> 1 if the span is taken as 1 s unseen */
        y[0] = move_span_is_one(x[0], move_far(x[3]), x[1], x[2], x[4]) ? 1.0 : 0.0; break;
#if defined(__CUDACC__)
    case OP_RCP: y[0] = wrsn_rcp(x[0]); break;
    case OP_RSQRT: y[0] = wrsn_rsqrt(x[0]); break;
    case OP_EXP_TAB: y[0] = wrsn_exp_tab(tab, x[0]); break;
#endif
    default: y[0] = NAN; y[5] = 1.0; break;      /* y[5] = 1: not available in this build */
    }
}

#if defined(__CUDACC__)
__global__ void k_probe(int op, const double *x, double *y, int n) {
    __shared__ double tab[64];
    for (int j = threadIdx.x; j < 64; j += blockDim.x) tab[j] = wrsn_exp2_tab[j];
    __syncthreads();
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) probe_one(op, x + (size_t)k * PROBE_IN, y + (size_t)k * PROBE_OUT, g32::saddr_of(tab));
}

extern "C" int probe_run(int op, const double *x, double *y, int n) {
    if (n <= 0) return 0;
    k_probe<<<(n + 127) / 128, 128>>>(op, x, y, n);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { fprintf(stderr, "probe_run: %s\n", cudaGetErrorString(e)); return 1; }
    return 0;
}
#else
extern "C" int probe_run(int op, const double *x, double *y, int n) {
    for (int k = 0; k < n; k++) probe_one(op, x + (size_t)k * PROBE_IN, y + (size_t)k * PROBE_OUT, 0);
    return 0;
}
#endif
