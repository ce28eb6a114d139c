/*
 * wrsn_launch.h — the parameters of one launch of the environment kernel (wrsn_env_kernel.cuh: env_run), shared by the CUDA
 * library and the tests' host emulation.
 */
#pragma once
#include "wrsn_layout.h"

enum { MODE_INIT = 0, MODE_RUN_UNTIL, MODE_RESET_FINISH, MODE_RESTORE_RESET, MODE_STEP, MODE_FITNESS, MODE_K_BFS,
       MODE_K_DRAIN, MODE_K_BOOK, MODE_K_REWARD, MODE_STEP_BATCH };

struct KParams {
    wrsn_dims d;
    WrsnLayout L;
    const char *scen;
    const int32_t *scen_id;
    char *state;
    const char *snap;
    const uint8_t *mask;
    int mask_mode;                                   /* 0: mask[] (or all); 1: rows with req.agent_id >= 0; 2: rows with req.agent_id < 0 */
    const double *t_until;
    const int32_t *agent_in;
    const double *action_in;
    wrsn_request req;
    double *fitness, *fit_min;
    int with_reward;
    int resume_only;                                 /* later rounds of a split step: only rows whose step is in flight (agent_id == -4) */
    const int32_t *order;                            /* MODE_STEP: row taken by CTA k (k_step_order), or NULL = k */
};
