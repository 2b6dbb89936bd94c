// snake_step.cuh -- device-side types shared by the kernels and the C-ABI host code.
#pragma once
#include <stdint.h>

#include "../../include/snake_b200.h"

#define NB SNK_NB
#define NJ SNK_NJ
#define NC SNK_NC
#define ND SNK_NDOF
#define NROW (NJ + 3 * NC)
// word of the device counters that accumulates the joint-limit rows active at the end of the ticks (snk_joint_limit_stats): behind the
// 8 statistics / hand-out words and the 64 words of the exact kernel's hand-out scheduler, so that no kernel's word is shared
#define SNK_CTR_LIMIT_ROWS (8 + 64)

// Model tables in fp32, resident in global memory (read through the read-only path; every
// access is either warp-uniform or one element per lane, so they live in L1 after first touch).
struct DevTables {
    float jR0[NJ][9];
    float jt[NJ][3];
    float jax[NJ][3];
    float jdamp[NJ];
    float mass[NB];
    float com[NB][3];
    float Ic[NB][9];
    float ccen[NC][3];
    float cax[NC][3];
    float cfr[NC][9];
    float crad[NC], chl[NC], cend[NC], cmar[NC], cbrk[NC];
    float hpt[NB][3];
    float fzax[3];
    float rootm;
    int cbody[NC];
    int hbody[NB];
};

// Task/solver parameters in fp32, passed by value to the kernels.
struct KParams {
    float dt, inv_dt, g[3], kp, kd, maximp, sf, alpha, beta, gamma, edt, mu, aniso[3], kl, ka, erp2, slop, resthr, sthr /* sqrt(resthr), computed on the host so that the solver reads it from the constant bank */,
        maxvel, errthr, hthr, tang, donepen, colf, colpen;
    int iters, maxticks, gait, cone, tjoint, stale, altmotor, actdim, exact;
};
