// snake_step.cu -- fused SnakeGymEnv.step() for N environments, one warp per environment (sm_100a).
//
// One launch = one SubprocVecEnv.step(): clip + createAction, the data-dependent 0..41-tick loop of
// {PD motor rows, articulated-body forward dynamics, cylinder-vs-plane contacts, projected
// Gauss-Seidel}, observation, reward, termination and auto-reset, written straight into the
// caller's (torch) buffers.  All intermediate state of an environment lives in its warp's slice of
// shared memory and in registers for the whole env-step; HBM sees 256 B of state in, 256 B out, the
// action row in, and obs/reward/done out.
//
// Lane roles change by phase (DESIGN.md section 5):
//   kinematic / velocity / acceleration chains : every lane walks the 16-joint chain redundantly in
//       registers (no shared-memory round trip per joint); lane b keeps body b's result
//   bias forces                                 : lane = body
//   articulated inertias (backward pass)        : lane = element of the 6x6 matrices, 4 stages/joint
//   constraint rows (J, M^-1 J^T, rhs)          : lane = collision cylinder (32 cylinders = 32 lanes);
//       lanes 0..15 additionally own one motor row; each lane runs the O(n) impulse response of its rows
//   projected Gauss-Seidel                      : BLOCK form with exact in-block coupling (same iterates as the row-by-row
//       sweep, see pgs_* below): lane = row of the current block of <= 32 rows (16 motor rows | 32 normal rows | 2 x 16 friction
//       pairs); J.dv of all rows of the block at once (lane = row, no reduction), the rows then follow each other through the
//       block's Delassus entries A = J M^-1 J^T (one broadcast shuffle per row on the serial chain instead of a five-level
//       butterfly), the velocity update of the whole block at the end (lane = DoF)
//
// Reference call sites replaced: SnakeGymEnv.py:33-50,82-103; snake.py:209-306,336-341;
// ppo/multiprocessing_env.py:11-16; physics per SURVEY.md Appendix A (see oracle/snake_oracle.c,
// whose row order, clamping and residual rule this kernel reproduces).
#include "snake_dev.cuh"
#define WARPS_PER_CTA 1
#define CTAS_PER_SM 9
#define JS 23
#define APACK (1 + NC * (NC - 1) / 2 + 3)
#define A_OFF(i) ((i) * NC - ((i) * ((i) + 1)) / 2)

struct WarpMemPgs {
    float s[SNK_STATE_STRIDE];
    float Rw[NB][9];
    float pw[NB][3];
    float nu[ND];
    float nuF[ND];
    float target[NJ];
    float Jf[2 * NC][JS];  // Jacobians of the friction rows (2c, 2c + 1 of contact c), padded to JS words: lane = row reads are bank-conflict free
    float B[NROW][ND];
    float rhs[NROW];
    float invD[NROW];
    float dvs[32];         // the solver's velocity change (lane = DoF keeps it in a register; this is the copy the rows read)
    float dl[32];          // impulse changes of the block just solved (lane = row), read by the velocity update
    // Three lifetimes share one region: what only the forward dynamics and the row set-up read (joint frames, articulated quantities;
    // fk() rewrites Rj after every tick), inside it the forward-dynamics workspace and then the staging rows of the normal Jacobians,
    // and finally -- once the rows exist and every lane holds its normal row in registers -- the Delassus blocks of the solver.
    union {
        struct {
            float Rj[NB][9];
            float U[NB][6];
            float Dinv[NB];
            float uu[NB];
            float IA0inv[36];
            union {
                struct {       // forward-dynamics workspace: dead once the unconstrained velocity nu and U, Dinv, uu, IA0inv exist
                    float v[NB][6];
                    float cb[NB][6];
                    float pA[NB][6];
                    float IA[NB][36];
                    float X[36];
                    float Ia[36];
                    float Tm[36];
                    float pa[6];
                };
                float Jn[NC][JS];  // Jacobians of the normal rows while the rows are built
            };
        };
        struct {           // in-block Delassus entries, packed upper triangles: entry (i, j > i) = J_j . B_i at A_OFF(i) + j - i (one pad
            float An[APACK];   // word in front, so that the finished lanes j <= i of a step read inside the array); the motor block
            float Af[2][APACK]; // needs none (J = unit vector: B itself)
        };
    };
};

static_assert((sizeof(WarpMemPgs) * WARPS_PER_CTA + 1024) * CTAS_PER_SM <= 233472, "CTAS_PER_SM CTAs of the warp-per-env kernel must fit into the 228 KB of an SM");

// ---------------------------------------------------------------------------------------------
// response of the generalized velocity to a unit impulse (oracle: impulse_response): spatial impulse
// f6 on body b (b < 0: none) and/or unit torque impulse at joint jm (0: none).  Runs per lane; every
// lane walks all 16 joints so the shared-memory reads are warp-uniform broadcasts.
// ---------------------------------------------------------------------------------------------
template <class WM>
__device__ __forceinline__ void impulse_response_body(const WM& W, const DevTables* __restrict__ T, int b, const float* f6, int jm,
                                                      float* out /* ND, shared or local */) {
    float u[NB];
    float p[6] = {0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int i = NB - 1; i >= 1; i--) {
        if (i == b) {
#pragma unroll
            for (int k = 0; k < 6; k++) p[k] -= f6[k];
        }
        float ax[3] = {__ldg(&T->jax[i - 1][0]), __ldg(&T->jax[i - 1][1]), __ldg(&T->jax[i - 1][2])};
        float r[3] = {__ldg(&T->jt[i - 1][0]), __ldg(&T->jt[i - 1][1]), __ldg(&T->jt[i - 1][2])};
        u[i] = ((i == jm) ? 1.f : 0.f) - dot3(ax, p);
        float s = u[i] * W.Dinv[i], pa[6], pp[6];
#pragma unroll
        for (int k = 0; k < 6; k++) pa[k] = p[k] + W.U[i][k] * s;
        xfrc(W.Rj[i], r, pa, pp);
#pragma unroll
        for (int k = 0; k < 6; k++) p[k] = pp[k];
    }
    if (b == 0) {
#pragma unroll
        for (int k = 0; k < 6; k++) p[k] -= f6[k];
    }
    float a[6];
#pragma unroll
    for (int r = 0; r < 6; r++) {
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < 6; k++) s -= W.IA0inv[6 * r + k] * p[k];
        a[r] = s;
        out[r] = s;
    }
#pragma unroll
    for (int i = 1; i < NB; i++) {
        float ax[3] = {__ldg(&T->jax[i - 1][0]), __ldg(&T->jax[i - 1][1]), __ldg(&T->jax[i - 1][2])};
        float r[3] = {__ldg(&T->jt[i - 1][0]), __ldg(&T->jt[i - 1][1]), __ldg(&T->jt[i - 1][2])};
        float ac[6];
        xmot(W.Rj[i], r, a, ac);
        float s = u[i];
#pragma unroll
        for (int k = 0; k < 6; k++) s -= W.U[i][k] * ac[k];
        float qdd = s * W.Dinv[i];
        out[6 + i - 1] = qdd;
        a[0] = ac[0] + ax[0] * qdd; a[1] = ac[1] + ax[1] * qdd; a[2] = ac[2] + ax[2] * qdd;
        a[3] = ac[3]; a[4] = ac[4]; a[5] = ac[5];
    }
}

__device__ __noinline__ void impulse_response(const WarpMemPgs& W, const DevTables* __restrict__ T, int b, const float* f6, int jm,
                                              float* out /* ND, shared or local */) {
    impulse_response_body(W, T, b, f6, jm, out);
}

// 6x6 SPD inverse by Cholesky, all in registers (every lane computes the same thing)
__device__ void sym6_inverse(const float* A /* shared */, float* Ainv /* registers, 36 */) {
    float L[36];
#pragma unroll
    for (int k = 0; k < 36; k++) L[k] = 0.f;
#pragma unroll
    for (int j = 0; j < 6; j++) {
        float d = A[6 * j + j];
#pragma unroll
        for (int k = 0; k < j; k++) d -= L[6 * j + k] * L[6 * j + k];
        d = sqrtf(d);
        L[6 * j + j] = d;
        float id = 1.f / d;
#pragma unroll
        for (int i = j + 1; i < 6; i++) {
            float s = A[6 * i + j];
#pragma unroll
            for (int k = 0; k < j; k++) s -= L[6 * i + k] * L[6 * j + k];
            L[6 * i + j] = s * id;
        }
    }
#pragma unroll
    for (int c = 0; c < 6; c++) {
        float y[6], x[6];
#pragma unroll
        for (int i = 0; i < 6; i++) {
            float s = (i == c) ? 1.f : 0.f;
#pragma unroll
            for (int k = 0; k < i; k++) s -= L[6 * i + k] * y[k];
            y[i] = s / L[6 * i + i];
        }
#pragma unroll
        for (int i = 5; i >= 0; i--) {
            float s = y[i];
#pragma unroll
            for (int k = i + 1; k < 6; k++) s -= L[6 * k + i] * x[k];
            x[i] = s / L[6 * i + i];
        }
#pragma unroll
        for (int i = 0; i < 6; i++) Ainv[6 * i + c] = x[i];
    }
}

// ---------------------------------------------------------------------------------------------
// one physics tick (oracle: forward_dynamics + tick).  Returns the PGS iteration count.
// ---------------------------------------------------------------------------------------------
// passes 1-3 of the articulated-body algorithm (oracle: forward_dynamics): W.nu = unconstrained generalized velocity; W.U, Dinv, uu,
// IA0inv are kept for the impulse responses
template <class WM>
__device__ __forceinline__ void pgs_dynamics(WM& W, const DevTables* __restrict__ T, const KParams& P, int lane) {
    const float dt = P.dt;
    // ---- pass 1: velocity chain (every lane, registers), lane b keeps v_b ----
    float vcur[6], vm[6];
    {
        float w[3] = {W.s[SNK_S_OMEGA], W.s[SNK_S_OMEGA + 1], W.s[SNK_S_OMEGA + 2]};
        float vv[3] = {W.s[SNK_S_VEL], W.s[SNK_S_VEL + 1], W.s[SNK_S_VEL + 2]};
        m3tv(W.Rw[0], w, vcur);
        m3tv(W.Rw[0], vv, vcur + 3);
    }
#pragma unroll
    for (int k = 0; k < 6; k++) vm[k] = vcur[k];
#pragma unroll 1
    for (int i = 1; i < NB; i++) {
        float r[3] = {__ldg(&T->jt[i - 1][0]), __ldg(&T->jt[i - 1][1]), __ldg(&T->jt[i - 1][2])};
        float vn[6];
        xmot(W.Rj[i], r, vcur, vn);
        float qd = W.s[SNK_S_QD + i - 1];
        vn[0] += __ldg(&T->jax[i - 1][0]) * qd; vn[1] += __ldg(&T->jax[i - 1][1]) * qd; vn[2] += __ldg(&T->jax[i - 1][2]) * qd;
#pragma unroll
        for (int k = 0; k < 6; k++) vcur[k] = vn[k];
        if (lane == i) {
#pragma unroll
            for (int k = 0; k < 6; k++) vm[k] = vn[k];
        }
    }
    // ---- bias forces, lane = body ----
    if (lane < NB) {
        const int b = lane;
        float m = __ldg(&T->mass[b]);
        float c[3] = {__ldg(&T->com[b][0]), __ldg(&T->com[b][1]), __ldg(&T->com[b][2])};
        float Ic[9];
#pragma unroll
        for (int k = 0; k < 9; k++) Ic[k] = __ldg(&T->Ic[b][k]);
        float cbv[6] = {0, 0, 0, 0, 0, 0};
        if (b > 0) {
            float qd = W.s[SNK_S_QD + b - 1];
            float sq[3] = {__ldg(&T->jax[b - 1][0]) * qd, __ldg(&T->jax[b - 1][1]) * qd, __ldg(&T->jax[b - 1][2]) * qd};
            cross3(vm, sq, cbv);
            cross3(vm + 3, sq, cbv + 3);
        }
        // h = I v (rigid inertia at the body origin): h_lin = m (v + w x c), h_ang = Ic w + c x h_lin
        float wc[3], vc[3], hl[3], ha[3], t[3];
        cross3(vm, c, wc);
        vc[0] = vm[3] + wc[0]; vc[1] = vm[4] + wc[1]; vc[2] = vm[5] + wc[2];
        hl[0] = m * vc[0]; hl[1] = m * vc[1]; hl[2] = m * vc[2];
        float Iw[3];
        m3v(Ic, vm, Iw);
        cross3(c, hl, t);
        ha[0] = Iw[0] + t[0]; ha[1] = Iw[1] + t[1]; ha[2] = Iw[2] + t[2];
        float p[6], t1[3], t2[3];
        cross3(vm, ha, t1); cross3(vm + 3, hl, t2);
        p[0] = t1[0] + t2[0]; p[1] = t1[1] + t2[1]; p[2] = t1[2] + t2[2];
        cross3(vm, hl, p + 3);
        // gravity + velocity damping
        float gb[3], fg[3], ng[3], Fd[3], Td[3], nd[3];
        m3tv(W.Rw[b], P.g, gb);
        fg[0] = m * gb[0]; fg[1] = m * gb[1]; fg[2] = m * gb[2];
        cross3(c, fg, ng);
        float nv = sqrtf(dot3(vc, vc)), nw = sqrtf(dot3(vm, vm));
        float kl = P.kl + P.kl * nv, ka = P.ka + P.ka * nw;
#pragma unroll
        for (int k = 0; k < 3; k++) { Fd[k] = -m * vc[k] * kl; Td[k] = -Iw[k] * ka; }
        cross3(c, Fd, nd);
#pragma unroll
        for (int k = 0; k < 3; k++) { p[k] -= ng[k] + Td[k] + nd[k]; p[3 + k] -= fg[k] + Fd[k]; }
#pragma unroll
        for (int k = 0; k < 6; k++) { W.v[b][k] = vm[k]; W.cb[b][k] = cbv[k]; W.pA[b][k] = p[k]; }
    }
    // rigid spatial inertias at the body origins -> IA, lane = element
    for (int idx = lane; idx < NB * 36; idx += 32) {
        int b = idx / 36, e = idx - b * 36, r = e / 6, cc = e - r * 6;
        float m = __ldg(&T->mass[b]);
        const float* c = T->com[b];
        float val;
        if (r < 3 && cc < 3) { // Ic - m [c]x[c]x = Ic + m (c.c 1 - c c^T)
            float c0 = __ldg(c), c1 = __ldg(c + 1), c2 = __ldg(c + 2);
            float cr = (r == 0) ? c0 : (r == 1) ? c1 : c2, ccv = (cc == 0) ? c0 : (cc == 1) ? c1 : c2;
            val = __ldg(&T->Ic[b][3 * r + cc]) + m * (((r == cc) ? (c0 * c0 + c1 * c1 + c2 * c2) : 0.f) - cr * ccv);
        } else if (r >= 3 && cc >= 3) {
            val = (r == cc) ? m : 0.f;
        } else { // m [c]x (upper right), -m [c]x (lower left)
            int a = (r < 3) ? r : r - 3, d = (cc < 3) ? cc : cc - 3;
            float sgn = (r < 3) ? 1.f : -1.f;
            float cx = 0.f;
            if (a != d) {
                int k3 = 3 - a - d; // the remaining index
                float ck = __ldg(c + k3);
                // [c]x[a][d] = -eps(a,d,k) c_k
                bool even = ((a == 0 && d == 1) || (a == 1 && d == 2) || (a == 2 && d == 0));
                cx = even ? -ck : ck;
            }
            val = sgn * m * cx;
        }
        (&W.IA[0][0])[idx] = val;
    }
    __syncwarp();
    // ---- pass 2: articulated inertias, lane = matrix element ----
#pragma unroll 1
    for (int i = NB - 1; i >= 1; i--) {
        const float ax0 = __ldg(&T->jax[i - 1][0]), ax1 = __ldg(&T->jax[i - 1][1]), ax2 = __ldg(&T->jax[i - 1][2]);
        const float r0 = __ldg(&T->jt[i - 1][0]), r1 = __ldg(&T->jt[i - 1][1]), r2 = __ldg(&T->jt[i - 1][2]);
        // stage A: U = IA ax (lanes 0..5); X (all lanes, 36 elements)
        if (lane < 6) W.U[i][lane] = W.IA[i][6 * lane] * ax0 + W.IA[i][6 * lane + 1] * ax1 + W.IA[i][6 * lane + 2] * ax2;
        for (int e = lane; e < 36; e += 32) {
            int a = e / 6, c = e - 6 * a;
            int a3 = (a < 3) ? a : a - 3, c3 = (c < 3) ? c : c - 3;
            float val;
            if (a < 3 && c >= 3) val = 0.f;
            else if ((a < 3) == (c < 3)) val = W.Rj[i][3 * c3 + a3]; // E = Rj^T
            else { // -(E rx)[a3][c3],  rx = [[0,-r2,r1],[r2,0,-r0],[-r1,r0,0]]
                float e0 = W.Rj[i][a3], e1 = W.Rj[i][3 + a3], e2 = W.Rj[i][6 + a3]; // row a3 of E
                float v0 = e1 * r2 - e2 * r1, v1 = -e0 * r2 + e2 * r0, v2 = e0 * r1 - e1 * r0;
                val = -((c3 == 0) ? v0 : (c3 == 1) ? v1 : v2);
            }
            W.X[e] = val;
        }
        __syncwarp();
        const float D = ax0 * W.U[i][0] + ax1 * W.U[i][1] + ax2 * W.U[i][2];
        const float Dinv = 1.f / D;
        const float tau = -__ldg(&T->jdamp[i - 1]) * W.s[SNK_S_QD + i - 1];
        const float uu = tau - (ax0 * W.pA[i][0] + ax1 * W.pA[i][1] + ax2 * W.pA[i][2]);
        if (lane == 0) { W.Dinv[i] = Dinv; W.uu[i] = uu; }
        // stage B: Ia = IA - U U^T / D
        for (int e = lane; e < 36; e += 32) {
            int a = e / 6, c = e - 6 * a;
            W.Ia[e] = W.IA[i][e] - W.U[i][a] * W.U[i][c] * Dinv;
        }
        __syncwarp();
        // stage C: Tm = Ia X ; pa = pA + Ia cb + U uu / D (lanes 0..5)
        for (int e = lane; e < 36; e += 32) {
            int a = e / 6, c = e - 6 * a;
            float z = 0.f;
#pragma unroll
            for (int k = 0; k < 6; k++) z += W.Ia[6 * a + k] * W.X[6 * k + c];
            W.Tm[e] = z;
        }
        if (lane < 6) {
            float z = W.pA[i][lane] + W.U[i][lane] * uu * Dinv;
#pragma unroll
            for (int k = 0; k < 6; k++) z += W.Ia[6 * lane + k] * W.cb[i][k];
            W.pa[lane] = z;
        }
        __syncwarp();
        // stage D: IA[i-1] += X^T Tm ; pA[i-1] += X* pa
        for (int e = lane; e < 36; e += 32) {
            int a = e / 6, c = e - 6 * a;
            float z = 0.f;
#pragma unroll
            for (int k = 0; k < 6; k++) z += W.X[6 * k + a] * W.Tm[6 * k + c];
            W.IA[i - 1][e] += z;
        }
        if (lane < 6) { // force transform = X^T applied to pa
            float z = 0.f;
#pragma unroll
            for (int k = 0; k < 6; k++) z += W.X[6 * k + lane] * W.pa[k];
            W.pA[i - 1][lane] += z;
        }
        __syncwarp();
    }
    // ---- base: IA0^-1 (registers, every lane), shared copy for the impulse responses ----
    float Ainv[36];
    sym6_inverse(W.IA[0], Ainv);
    for (int e = lane; e < 36; e += 32) {
        float val = 0.f;
#pragma unroll
        for (int k = 0; k < 36; k++) if (k == e) val = Ainv[k];
        W.IA0inv[e] = val;
    }
    // ---- pass 3: acceleration chain (every lane), unconstrained velocity ----
    {
        float a[6];
#pragma unroll
        for (int r = 0; r < 6; r++) {
            float z = 0.f;
#pragma unroll
            for (int k = 0; k < 6; k++) z -= Ainv[6 * r + k] * W.pA[0][k];
            a[r] = z;
        }
        float wxv[3];
        cross3(W.v[0], W.v[0] + 3, wxv);
        {
            float al = 0.f;
#pragma unroll
            for (int r = 0; r < 6; r++) if (lane == r) al = a[r] + ((r >= 3) ? wxv[(r >= 3) ? r - 3 : 0] : 0.f);
            if (lane < 6) W.nu[lane] = W.v[0][lane] + dt * al;
        }
        float myqdd = 0.f;
#pragma unroll 1
        for (int i = 1; i < NB; i++) {
            float r[3] = {__ldg(&T->jt[i - 1][0]), __ldg(&T->jt[i - 1][1]), __ldg(&T->jt[i - 1][2])};
            float ac[6];
            xmot(W.Rj[i], r, a, ac);
            float z = W.uu[i];
#pragma unroll
            for (int k = 0; k < 6; k++) { ac[k] += W.cb[i][k]; z -= W.U[i][k] * ac[k]; }
            float qdd = z * W.Dinv[i];
            a[0] = ac[0] + __ldg(&T->jax[i - 1][0]) * qdd; a[1] = ac[1] + __ldg(&T->jax[i - 1][1]) * qdd;
            a[2] = ac[2] + __ldg(&T->jax[i - 1][2]) * qdd;
            a[3] = ac[3]; a[4] = ac[4]; a[5] = ac[5];
            if (lane == i - 1) myqdd = qdd;
        }
        if (lane < NJ) W.nu[6 + lane] = W.s[SNK_S_QD + lane] + dt * myqdd;
    }
    __syncwarp();

}

// velocity update with the solver's dv (lane = DoF), joint feedback (lam_m: lane j's motor impulse), semi-implicit Euler
template <class WM>
__device__ __forceinline__ void pgs_finish(WM& W, const DevTables* __restrict__ T, const KParams& P, int lane, float dv, float lam_m) {
    const float dt = P.dt;
    const bool dof = lane < ND;
    // ---- velocity update, joint feedback, semi-implicit Euler ----
    if (dof) { float x = W.nu[lane] + dv; x = (x > P.maxvel) ? P.maxvel : x; W.nuF[lane] = (x < -P.maxvel) ? -P.maxvel : x; } // NaN passes through
    __syncwarp();
    float wnew[3], vnew[3];
    m3v(W.Rw[0], W.nuF, wnew);
    m3v(W.Rw[0], W.nuF + 3, vnew);
    float fz;
    {
        float vo[3] = {W.s[SNK_S_VEL], W.s[SNK_S_VEL + 1], W.s[SNK_S_VEL + 2]};
        float nv = sqrtf(dot3(vo, vo)), f[3], zw[3], fzax[3] = {__ldg(&T->fzax[0]), __ldg(&T->fzax[1]), __ldg(&T->fzax[2])};
        float rm = __ldg(&T->rootm);
#pragma unroll
        for (int k = 0; k < 3; k++) f[k] = rm * P.g[k] - rm * vo[k] * (P.kl + P.kl * nv) - rm * (vnew[k] - vo[k]) * P.inv_dt;
        m3v(W.Rw[0], fzax, zw);
        fz = dot3(zw, f);
    }
    float qn[4];
    {
        float ang = sqrtf(dot3(wnew, wnew)), sc;
        if (ang < 0.001f) sc = 0.5f * dt - dt * dt * dt * 0.020833333333f * ang * ang;
        else sc = sinf(0.5f * ang * dt) / ang;
        float ax[3] = {wnew[0] * sc, wnew[1] * sc, wnew[2] * sc};
        float cw = cosf(ang * dt * 0.5f);
        const float* q = W.s + SNK_S_QUAT;
        float x = cw * q[0] + ax[0] * q[3] + ax[1] * q[2] - ax[2] * q[1];
        float y = cw * q[1] + ax[1] * q[3] + ax[2] * q[0] - ax[0] * q[2];
        float z = cw * q[2] + ax[2] * q[3] + ax[0] * q[1] - ax[1] * q[0];
        float w = cw * q[3] - ax[0] * q[0] - ax[1] * q[1] - ax[2] * q[2];
        float in = 1.f / sqrtf(x * x + y * y + z * z + w * w);
        qn[0] = x * in; qn[1] = y * in; qn[2] = z * in; qn[3] = w * in;
    }
    __syncwarp(); // all lanes have read the old state
    if (lane < NJ) {
        float qd = W.nuF[6 + lane];
        W.s[SNK_S_TAU + lane] = lam_m * P.inv_dt;
        W.s[SNK_S_QD + lane] = qd;
        W.s[SNK_S_Q + lane] += qd * dt;
    }
    if (lane == 16) W.s[SNK_S_FZ] = fz;
    if (lane >= 17 && lane < 20) {
        int k = lane - 17;
        W.s[SNK_S_VEL + k] = vnew[k]; W.s[SNK_S_OMEGA + k] = wnew[k]; W.s[SNK_S_POS + k] += vnew[k] * dt;
    }
    if (lane >= 20 && lane < 24) W.s[SNK_S_QUAT + lane - 20] = qn[lane - 20];
    __syncwarp();
}

// ---------------------------------------------------------------------------------------------
// joint-limit rows (snk_set_joint_limits; oracle: tick with set_joint_limits, btMultiBodyJointLimitConstraint of A.1): two unilateral
// rows per joint, row 2j = +e_(6+j) at the lower limit (penetration q_j + angle) and row 2j + 1 = -e_(6+j) at the upper one
// (penetration angle - q_j), set up like contact normals.  Both rows reuse the motor row of their joint: response s B_j, inverse
// effective mass invD_j, in-block Delassus entry A(r_i, r_k) = s_i s_k B_(j_i)[6 + j_k].
// ---------------------------------------------------------------------------------------------
// right-hand sides of joint j's two rows; q = q_j at the start of the tick, nu = its post-ABA velocity, iD = invD_j
__device__ __forceinline__ void limit_rows_rhs(float q, float nu, float angle, const KParams& P, float iD, float& r_lo, float& r_up) {
    float pen = q + angle, verr = -nu, perr = 0.f;
    if (pen > 0.f) verr -= pen * P.inv_dt; else perr = -pen * P.erp2 * P.inv_dt;
    r_lo = (verr + perr) * iD;
    pen = angle - q; verr = nu; perr = 0.f;
    if (pen > 0.f) verr -= pen * P.inv_dt; else perr = -pen * P.erp2 * P.inv_dt;
    r_up = (verr + perr) * iD;
}

// One sweep over the 32 limit rows in row order, between the motor block and the normal rows (lambda >= 0, no upper bound).  Lane =
// joint owns BOTH of its rows: the upper row follows the lower one on the same lane (its w is -(w + A d_lo), A = B_j[6 + j]), and since
// the two rows differ only in sign, the later joints see their net impulse change d_lo - d_up -- one broadcast shuffle per joint, a
// 16-step serial chain for 32 rows.  Branch free like the motor block (tick).  B: the motor rows' responses (B[j], j < NJ); dvs / dl: the
// shared copies of dv and of the block's impulse changes; dv, res: this lane's velocity change (lane = DoF) and residual, updated.
__device__ __forceinline__ void pgs_limit_block(const float (*B)[ND], float* dvs, float* dl, int lane, float r_lo, float r_up, float iD, float Dg,
                                                float& lam_lo, float& lam_up, float& dv, float& res) {
    const bool dof = lane < ND;
    const int ld = dof ? lane : 0;
    const int lm = lane & (NJ - 1);
    float w = dvs[6 + lm], dlo_mine = 0.f, dup_mine = 0.f;
    float bn = B[0][6 + lm]; // A of the coming step, fetched one step ahead of the chain
#pragma unroll 4
    for (int i = 0; i < NJ; i++) {
        const float a = bn;
        bn = B[i < NJ - 1 ? i + 1 : i][6 + lm];
        const float d0 = r_lo - w * iD;            // lower row of joint i
        const float s0 = lam_lo + d0;
        const bool n0 = s0 < 0.f;
        const float slo = n0 ? 0.f : s0, dlo = n0 ? -lam_lo : d0;
        const float wu = -fmaf(a, dlo, w);         // upper row: J = -e, after the lower row's update
        const float d1 = r_up - wu * iD;
        const float s1 = lam_up + d1;
        const bool n1 = s1 < 0.f;
        const float sup = n1 ? 0.f : s1, dup = n1 ? -lam_up : d1;
        const float di = __shfl_sync(FULL, dlo - dup, i);
        const bool mine = lane == i;
        lam_lo = mine ? slo : lam_lo; lam_up = mine ? sup : lam_up;
        dlo_mine = mine ? dlo : dlo_mine; dup_mine = mine ? dup : dup_mine;
        w = fmaf(a, di, w);
    }
    dl[lane] = dlo_mine - dup_mine;
    __syncwarp();
    if (dof) { // dv += sum_j B_j (d_2j - d_2j+1)
#pragma unroll
        for (int i = 0; i < NJ; i++) dv = fmaf(B[i][ld], dl[i], dv);
        dvs[lane] = dv;
    }
    const float r0 = dlo_mine * Dg, r1 = dup_mine * Dg;
    res = fmaxf(res, fmaxf(r0 * r0, r1 * r1));
    __syncwarp();
}

// limit rows with lambda > 0 at the end of the tick (lanes >= NJ hold none)
__device__ __forceinline__ unsigned limit_rows_active(float lam_lo, float lam_up) {
    return __popc(__ballot_sync(FULL, lam_lo > 0.f)) + __popc(__ballot_sync(FULL, lam_up > 0.f));
}

// the record of the warp-per-env kernel with the joint-limit rows on (snk_lim_env_kernel): the limit angle, and the rows active at the
// end of the ticks so far
struct WarpMemPgsLim : WarpMemPgs {
    float lim_angle;
    unsigned lim_active;
};
static_assert((sizeof(WarpMemPgsLim) * WARPS_PER_CTA + 1024) * CTAS_PER_SM <= 233472, "CTAS_PER_SM CTAs of the limit-row kernel must fit into an SM");

// LIM: with the joint-limit rows at +-lim_angle; *lim_active (shared) accumulates the rows active at the end of the tick
template <bool LIM>
__device__ int tick_pgs(WarpMemPgs& W, const DevTables* __restrict__ T, const KParams& P, int lane, float lim_angle, unsigned* lim_active) {
    pgs_dynamics(W, T, P, lane);
    // ---- constraint rows ----
    float lam_m = 0.f, lam_n = 0.f; // motor / normal impulses owned by this lane (motor row = joint, normal row = cylinder)
    if (lane < NJ) { // motor row of joint lane+1 (A.4)
        const int j = lane;
        const float zero6[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        impulse_response(W, T, -1, zero6, j + 1, W.B[j]);
        float D = W.B[j][6 + j];
        float q = W.s[SNK_S_Q + j], qd = W.nu[6 + j];
        float vt = P.kp * (W.target[j] - q) * P.inv_dt + qd + P.kd * (0.f - qd);
        W.invD[j] = 1.f / D; W.rhs[j] = (vt - qd) / D;
    }
    bool active;
    {
        const int c = lane;
        const int b = __ldg(&T->cbody[c]);
        float cax[3] = {__ldg(&T->cax[c][0]), __ldg(&T->cax[c][1]), __ldg(&T->cax[c][2])};
        float ccen[3] = {__ldg(&T->ccen[c][0]), __ldg(&T->ccen[c][1]), __ldg(&T->ccen[c][2])};
        float axw[3], cw[3], p[3];
        m3v(W.Rw[b], cax, axw);
        m3v(W.Rw[b], ccen, cw);
        float eh = __ldg(&T->cend[c]) * __ldg(&T->chl[c]);
        float az = axw[2], nn = fmaxf(1.f - az * az, 1e-12f);
        float inv = 1.f / sqrtf(nn), rad = __ldg(&T->crad[c]);
        p[0] = W.pw[b][0] + cw[0] + eh * axw[0] + rad * (az * axw[0] * inv);
        p[1] = W.pw[b][1] + cw[1] + eh * axw[1] + rad * (az * axw[1] * inv);
        p[2] = W.pw[b][2] + cw[2] + eh * axw[2] + rad * ((az * axw[2] - 1.f) * inv);
        float dist = p[2] - __ldg(&T->cmar[c]);
        active = dist < __ldg(&T->cbrk[c]);
        p[2] = dist;
        float Rl[9], cfr[9];
#pragma unroll
        for (int k = 0; k < 9; k++) cfr[k] = __ldg(&T->cfr[c][k]);
        m3m3(W.Rw[b], cfr, Rl);
        if (!active) { // a separated contact: all-zero rows are no-ops of the block solver below
#pragma unroll 1
            for (int f = 0; f < 3; f++) {
                const int r = (f == 0) ? c : NC + 2 * c + (f - 1);
                float* Jz = (f == 0) ? W.Jn[c] : W.Jf[2 * c + (f - 1)];
#pragma unroll 1
                for (int k = 0; k < ND; k++) { Jz[k] = 0.f; W.B[NJ + r][k] = 0.f; }
                W.invD[NJ + r] = 0.f; W.rhs[NJ + r] = 0.f;
            }
        }
#pragma unroll 1
        for (int f = 0; f < 3; f++) {
            if (!active) break;
            float d[3] = {0.f, 0.f, 1.f};
            if (f > 0) {
                float t[3] = {(f == 2) ? 1.f : 0.f, (f == 1) ? -1.f : 0.f, 0.f}, loc[3];
                m3tv(Rl, t, loc);
                loc[0] *= P.aniso[0]; loc[1] *= P.aniso[1]; loc[2] *= P.aniso[2];
                m3v(Rl, loc, d);
            }
            const int r = (f == 0) ? c : NC + 2 * c + (f - 1); // B / rhs rows are NJ + r
            float* Jr = (f == 0) ? W.Jn[c] : W.Jf[2 * c + (f - 1)];
            float* Br = W.B[NJ + r];
            float rel[3] = {p[0] - W.pw[0][0], p[1] - W.pw[0][1], p[2] - W.pw[0][2]}, rxd[3], jb[6];
            cross3(rel, d, rxd);
            m3tv(W.Rw[0], rxd, jb);
            m3tv(W.Rw[0], d, jb + 3);
#pragma unroll
            for (int k = 0; k < 6; k++) Jr[k] = jb[k];
#pragma unroll 1
            for (int j = 1; j < NB; j++) {
                float val = 0.f;
                if (j <= b) {
                    float ax[3] = {__ldg(&T->jax[j - 1][0]), __ldg(&T->jax[j - 1][1]), __ldg(&T->jax[j - 1][2])}, aw[3];
                    m3v(W.Rw[j], ax, aw);
                    float ro[3] = {p[0] - W.pw[j][0], p[1] - W.pw[j][1], p[2] - W.pw[j][2]}, t[3];
                    cross3(ro, d, t);
                    val = dot3(aw, t);
                }
                Jr[6 + j - 1] = val;
            }
            float f6[6], db[3], pb[3], ro[3] = {p[0] - W.pw[b][0], p[1] - W.pw[b][1], p[2] - W.pw[b][2]};
            m3tv(W.Rw[b], d, db);
            m3tv(W.Rw[b], ro, pb);
            cross3(pb, db, f6);
            f6[3] = db[0]; f6[4] = db[1]; f6[5] = db[2];
            impulse_response(W, T, b, f6, 0, Br);
            float D = 0.f, vrel = 0.f;
#pragma unroll 1
            for (int k = 0; k < ND; k++) { D += Jr[k] * Br[k]; vrel += Jr[k] * W.nu[k]; }
            float iD = 1.f / D, rh;
            if (f == 0) {
                float pen = dist + P.slop, verr = -vrel, perr = 0.f;
                if (pen > 0.f) verr -= pen * P.inv_dt; else perr = -pen * P.erp2 * P.inv_dt;
                rh = (verr + perr) * iD;
            } else rh = -vrel * iD;
            W.invD[NJ + r] = iD; W.rhs[NJ + r] = rh;
        }
    }
    __syncwarp();

    // ---- in-block Delassus entries A(i, j) = J_j . B_i for the rows j > i of the same block (lane = row j) ----
    // the lane of contact c keeps the Jacobian of its normal row in registers from here on: the staging rows share their shared memory
    // with the Delassus blocks written next
    float Jn[ND];
#pragma unroll
    for (int k = 0; k < ND; k++) Jn[k] = W.Jn[lane][k];
    __syncwarp();
    {
        float Jr[ND];
#pragma unroll
        for (int k = 0; k < ND; k++) Jr[k] = Jn[k];
#pragma unroll 1
        for (int i = 0; i < NC - 1; i++) {
            const float* Bi = W.B[NJ + i];
            float a0 = 0.f, a1 = 0.f;
#pragma unroll
            for (int k = 0; k < ND; k += 2) { a0 = fmaf(Jr[k], Bi[k], a0); a1 = fmaf(Jr[k + 1], Bi[k + 1], a1); }
            if (lane > i) W.An[A_OFF(i) + lane - i] = a0 + a1;
        }
#pragma unroll 1
        for (int fb = 0; fb < 2; fb++) {
#pragma unroll
            for (int k = 0; k < ND; k++) Jr[k] = W.Jf[32 * fb + lane][k];
#pragma unroll 1
            for (int i = 0; i < NC - 1; i++) {
                const float* Bi = W.B[NJ + NC + 32 * fb + i];
                float a0 = 0.f, a1 = 0.f;
#pragma unroll
                for (int k = 0; k < ND; k += 2) { a0 = fmaf(Jr[k], Bi[k], a0); a1 = fmaf(Jr[k + 1], Bi[k + 1], a1); }
                if (lane > i) W.Af[fb][A_OFF(i) + lane - i] = a0 + a1;
            }
        }
    }

    // ---- projected Gauss-Seidel in BLOCK form ----
    // The sweep visits the rows in Bullet's order (motor rows, normal rows, friction pairs: oracle tick()), and every row sees the
    // impulses of all rows before it -- but the rows of a block of <= 32 are handled together: (1) w = J dv for every row of the
    // block at once, lane = row; (2) the rows in order: the lane of row i turns its w into the impulse change d_i, one shuffle
    // broadcasts it, and the later rows j of the block add A(i, j) d_i to their w (what the velocity update of row i would have
    // done to J_j dv); (3) dv += sum_i B_i d_i for the whole block, lane = DoF.  The serial chain per row is clamp + shuffle + fma
    // instead of a shared-memory load, a five-level shuffle butterfly and the clamp; everything on it is branch free (a
    // data-dependent branch would split the warp in front of the next shuffle).
    const bool dof = lane < ND;
    const int ld = dof ? lane : 0;
    const int lm = lane & (NJ - 1);
    float dv = 0.f;
    float lam_fa[2] = {0.f, 0.f}, lam_fb[2] = {0.f, 0.f}; // friction impulses of contact 16 fb + lane / 2 (both lanes of the pair hold both)
    W.dvs[lane] = 0.f;
    // the rows' effective masses D (for the residual) are recovered from 1 / D; an all-zero row has D = 0
    const float m_rhs = W.rhs[lm], m_iD = W.invD[lm], m_Dg = (m_iD != 0.f) ? 1.f / m_iD : 0.f;
    const float n_rhs = W.rhs[NJ + lane], n_iD = W.invD[NJ + lane], n_Dg = (n_iD != 0.f) ? 1.f / n_iD : 0.f;
    const int pa = lane & ~1; // the lane pair (pa, pa + 1) holds the two friction rows of one contact
    float fa_rhs[2], fa_iD[2], fa_Dg[2], fb_rhs[2], fb_iD[2], fb_Dg[2];
#pragma unroll
    for (int fb = 0; fb < 2; fb++) {
        const int r = NJ + NC + 32 * fb + pa;
        fa_rhs[fb] = W.rhs[r]; fa_iD[fb] = W.invD[r]; fa_Dg[fb] = (fa_iD[fb] != 0.f) ? 1.f / fa_iD[fb] : 0.f;
        fb_rhs[fb] = W.rhs[r + 1]; fb_iD[fb] = W.invD[r + 1]; fb_Dg[fb] = (fb_iD[fb] != 0.f) ? 1.f / fb_iD[fb] : 0.f;
    }
    const float maximp = P.maximp, mu = P.mu;
    const bool cone = P.cone != 0;
    float l_rhs_lo = 0.f, l_rhs_up = 0.f, lam_lo = 0.f, lam_up = 0.f; // limit rows of joint lm (lane = joint)
    if constexpr (LIM) limit_rows_rhs(W.s[SNK_S_Q + lm], W.nu[6 + lm], lim_angle, P, m_iD, l_rhs_lo, l_rhs_up);
    __syncwarp();
    int it = 0;
#pragma unroll 1
    for (;; it++) {
        float res = 0.f;
        {   // ---- motor rows (J = unit vector of joint j: w = dv[6 + j], A(i, j) = B_i[6 + j]) ----
            const bool rev = P.altmotor && !(it & 1);
            float w = W.dvs[6 + lm], lam = lam_m, dmine = 0.f;
            float bn = W.B[rev ? NJ - 1 : 0][6 + lm]; // A(i, j) of the coming step, fetched one step ahead of the chain
#pragma unroll 4
            for (int s = 0; s < NJ; s++) {
                const int i = rev ? NJ - 1 - s : s;
                const float a = bn;
                const int inext = rev ? (i > 0 ? i - 1 : 0) : (i < NJ - 1 ? i + 1 : i);
                bn = W.B[inext][6 + lm];
                const float d0 = m_rhs - w * m_iD;
                const float sum0 = lam + d0;
                const bool lo = sum0 < -maximp, hi = sum0 > maximp; // both false for a NaN: it passes through, as in the oracle
                const float sum = lo ? -maximp : (hi ? maximp : sum0);
                const float d = lo ? (-maximp - lam) : (hi ? (maximp - lam) : d0);
                const float di = __shfl_sync(FULL, d, i);
                const bool mine = lane == i;
                lam = mine ? sum : lam; dmine = mine ? d : dmine;
                w = fmaf(a, di, w);
            }
            lam_m = lam;
            W.dl[lane] = dmine;
            __syncwarp();
            if (dof) {
#pragma unroll
                for (int i = 0; i < NJ; i++) dv = fmaf(W.B[i][ld], W.dl[i], dv);
                W.dvs[lane] = dv;
            }
            const float rr = dmine * m_Dg;
            res = fmaxf(res, rr * rr);
            __syncwarp();
        }
        if constexpr (LIM) pgs_limit_block(W.B, W.dvs, W.dl, lane, l_rhs_lo, l_rhs_up, m_iD, m_Dg, lam_lo, lam_up, dv, res);
        {   // ---- normal rows, lane = contact ----
            float w0 = 0.f, w1 = 0.f;
#pragma unroll
            for (int k = 0; k < ND; k += 2) { w0 = fmaf(Jn[k], W.dvs[k], w0); w1 = fmaf(Jn[k + 1], W.dvs[k + 1], w1); }
            float w = w0 + w1, lam = lam_n, dmine = 0.f;
            // rolled (4 rows per trip: the whole sweep stays in the instruction caches); the Delassus entry of a row is fetched one row
            // ahead of the chain; A(i, lane) sits at An[aoff + lane] with aoff = A_OFF(i) - i, which grows by NC - i - 2 per row
            const float* Ap = W.An + lane;
            int aoff = 0;
            float an = Ap[0];
#pragma unroll 4
            for (int i = 0; i < NC; i++) {
                const float a = an;
                aoff += NC - i - 2;
                an = Ap[i < NC - 2 ? aoff : 0]; // rows NC - 2 and NC - 1 have nothing left to fetch
                const float d0 = n_rhs - w * n_iD;
                const float sum0 = lam + d0;
                const bool neg = sum0 < 0.f;
                const float sum = neg ? 0.f : sum0, d = neg ? -lam : d0;
                const float di = __shfl_sync(FULL, d, i);
                const bool mine = lane == i;
                lam = mine ? sum : lam; dmine = mine ? d : dmine;
                w = fmaf(a, di, w); // the last row's entry is a dummy: no row is left to read w
            }
            lam_n = lam;
            W.dl[lane] = dmine;
            __syncwarp();
            if (dof) {
                float x0 = 0.f, x1 = 0.f;
#pragma unroll
                for (int i = 0; i < NC; i += 2) { x0 = fmaf(W.B[NJ + i][ld], W.dl[i], x0); x1 = fmaf(W.B[NJ + i + 1][ld], W.dl[i + 1], x1); }
                dv += x0 + x1;
                W.dvs[lane] = dv;
            }
            const float rr = dmine * n_Dg;
            res = fmaxf(res, rr * rr);
            __syncwarp();
        }
#pragma unroll
        for (int fb = 0; fb < 2; fb++) { // ---- friction pairs of contacts 16 fb .. 16 fb + 15 ----
            // lanes 2p and 2p + 1 both carry BOTH rows of contact 16 fb + p (w_a, w_b and the two impulses), so the cone projection
            // needs no exchange between lanes: the only shuffles on the chain broadcast the pair's (da, db)
            const float* Ja = W.Jf[32 * fb + pa];
            const float* Jb = W.Jf[32 * fb + pa + 1];
            float wa = 0.f, wb = 0.f;
#pragma unroll
            for (int k = 0; k < ND; k++) { const float x = W.dvs[k]; wa = fmaf(Ja[k], x, wa); wb = fmaf(Jb[k], x, wb); }
            float la = lam_fa[fb], lb = lam_fb[fb], da_mine = 0.f, db_mine = 0.f;
            const float lim = mu * __shfl_sync(FULL, lam_n, 16 * fb + (lane >> 1));
            const float* Af = W.Af[fb];
            const float a_rhs = fa_rhs[fb], a_iD = fa_iD[fb], b_rhs = fb_rhs[fb], b_iD = fb_iD[fb];
            // rolled, two contacts per trip; the four Delassus entries of a step are fetched one step ahead: A(2p, pa), A(2p, pa + 1) at
            // Af[o0 + pa], Af[o0 + pa + 1] with o0 = A_OFF(2p) - 2p, and A(2p + 1, .) at o1 = A_OFF(2p + 1) - 2p - 1 = o0 + NC - 2p - 2
            const float* Aq = Af + pa;
            int o0 = 0;
            float a00 = Aq[0], a01 = Aq[1], a10 = Aq[NC - 2], a11 = Aq[NC - 1];
#pragma unroll 2
            for (int p = 0; p < NC / 2; p++) {
                const float c00 = a00, c01 = a01, c10 = a10, c11 = a11;
                o0 += 2 * NC - 4 * p - 5; // A_OFF(2p + 2) - (2p + 2) - (A_OFF(2p) - 2p)
                {
                    const int q0 = p < NC / 2 - 1 ? o0 : 0, q1 = p < NC / 2 - 1 ? o0 + NC - 2 * p - 4 : 0; // nothing left to fetch for the last pair
                    a00 = Aq[q0]; a01 = Aq[q0 + 1]; a10 = Aq[q1]; a11 = Aq[q1 + 1];
                }
                float sa = la + (a_rhs - wa * a_iD), sb = lb + (b_rhs - wb * b_iD);
                if (cone) { // implicit cone: s <- s min(1, lim / |s|) (0/0 and lim/0 resolve to 1 through fminf, a NaN stays a NaN)
                    float rs;
                    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(rs) : "f"(fmaf(sa, sa, sb * sb)));
                    const float sc = fminf(1.f, lim * rs);
                    sa *= sc; sb *= sc;
                } else {
                    sa = fminf(fmaxf(sa, -lim), lim);
                    sb = fminf(fmaxf(sb, -lim), lim);
                }
                const float da0 = sa - la, db0 = sb - lb;
                const float da = __shfl_sync(FULL, da0, 2 * p), db = __shfl_sync(FULL, db0, 2 * p);
                const bool mine = (lane >> 1) == p;
                la = mine ? sa : la; lb = mine ? sb : lb; da_mine = mine ? da0 : da_mine; db_mine = mine ? db0 : db_mine;
                wa = fmaf(c00, da, fmaf(c10, db, wa)); // after the last pair nothing reads wa / wb: its entries are dummies
                wb = fmaf(c01, da, fmaf(c11, db, wb));
            }
            lam_fa[fb] = la; lam_fb[fb] = lb;
            W.dl[lane] = (lane & 1) ? db_mine : da_mine;
            __syncwarp();
            if (dof) {
                float x0 = 0.f, x1 = 0.f;
                const int rb = NJ + NC + 32 * fb;
#pragma unroll
                for (int i = 0; i < 32; i += 2) { x0 = fmaf(W.B[rb + i][ld], W.dl[i], x0); x1 = fmaf(W.B[rb + i + 1][ld], W.dl[i + 1], x1); }
                dv += x0 + x1;
                W.dvs[lane] = dv;
            }
            const float rr = fmaf(da_mine, fa_Dg[fb], db_mine * fb_Dg[fb]);
            res = fmaxf(res, rr * rr);
            __syncwarp();
        }
        res = __uint_as_float(__reduce_max_sync(FULL, __float_as_uint(res))); // res >= 0: the bit patterns order like the values
        if (res <= P.resthr || it >= P.iters - 1) break;
    }
    if constexpr (LIM) {
        const unsigned na = limit_rows_active(lam_lo, lam_up);
        if (lane == 0) *lim_active += na;
    }

    pgs_finish(W, T, P, lane, dv, lam_m);
    return it + 1;
}

__device__ __forceinline__ int tick(WarpMemPgs& W, const DevTables* __restrict__ T, const KParams& P, int lane) {
    return tick_pgs<false>(W, T, P, lane, 0.f, nullptr);
}
__device__ __forceinline__ int tick(WarpMemPgsLim& W, const DevTables* __restrict__ T, const KParams& P, int lane) {
    return tick_pgs<true>(W, T, P, lane, W.lim_angle, &W.lim_active);
}

// ---------------------------------------------------------------------------------------------
// kernels: the env-step template instantiated for this solver variant
// ---------------------------------------------------------------------------------------------
#include "snake_task.cuh"

// reset / observe.  mode 0 = masked soft reset (+ optional obs of every env), 1 = initialise everything, 2 = observe only.
// HBM bound (256 B record in, 224 B observation row out, the record of a reset environment written back), so the layout is chosen
// for bytes in flight: SIXTEEN threads per environment, thread j < 14 owns the j-th 16-byte word of the observation row -- four
// state slots in, one aligned float4 out, a warp writes 512 consecutive bytes -- and threads 14, 15 own the eight slots that are not
// part of the observation in the slot map below; a reset environment's record is written as sixteen ALIGNED 16-byte words, one per
// thread.  (One thread per slot, the first version, kept 4 B per thread in flight and reached 40 % of the copy bandwidth; writing the
// record back as unaligned scalars, the second, 11 %.)  Observation index -> state slot (snake.py:209-217): q 0..15 <- 13..28,
// qd 16..31 <- 29..44, applied torque 32..47 <- 45..60, base position 48..50 <- 0..2, quaternion 51..54 <- 3..6, Fz 55 <- 61.
__device__ __forceinline__ int reset_slot_of(int j, int c) { // state slot of component c of 16-byte word j (j = 14, 15: the non-observed slots)
    if (j < 12) return SNK_S_Q + 4 * j + c;
    if (j == 12) return c;                                  // pos.xyz, quat.x
    if (j == 13) return (c < 3) ? 4 + c : SNK_S_FZ;         // quat.yzw, Fz
    if (j == 14) return SNK_S_VEL + c;                      // vel.xyz, omega.x
    return (c < 2) ? SNK_S_OMEGA + 1 + c : SNK_S_RET + (c - 2); // omega.yz, return, length
}
__global__ void __launch_bounds__(256) snk_reset_kernel(const KParams P, float* __restrict__ state, const uint8_t* __restrict__ mask, float* __restrict__ obs,
                                                        int64_t n, int mode) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t env = idx >> 4;
    const int j = (int)(idx & 15);
    if (env >= n) return;
    const bool hit = (mode == 1) || (mode == 0 && (!mask || mask[env]));
    float* s = state + env * SNK_STATE_STRIDE;
    const bool stale = P.stale && mode == 0; // Q9: the torque / Fz slots (45..61) survive a soft reset
    // (a) the record of a reset environment: thread j writes its ALIGNED 16-byte word j (slots 4j..4j+3) -- a constant, except for the
    //     words that hold surviving slots (44..63), which are read, cleared around them and written back
    if (hit) {
        float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
        if (j == 1) w.z = 1.f;                       // slot 6 = quat.w
        if (stale && j >= 11) {
            w = reinterpret_cast<const float4*>(s)[j];
            if (j == 11) w.x = 0.f;                  // slot 44 = qd[15]
            if (j == 15) { w.z = 0.f; w.w = 0.f; }   // slots 62, 63 = return, length
        }
        reinterpret_cast<float4*>(s)[j] = w;
    }
    // (b) the observation row: thread j < 14 builds its 16-byte word from the PRE-reset record and the reset rule (thread (a) of a
    //     surviving slot rewrites the value it read, so the two roles never disagree)
    if (obs && j < 14) {
        float v[4];
#pragma unroll
        for (int c = 0; c < 4; c++) {
            const int k = reset_slot_of(j, c);
            const bool keep = (k >= SNK_S_TAU && k <= SNK_S_FZ) && stale;
            v[c] = (hit && !keep) ? ((k == SNK_S_QUAT + 3) ? 1.f : 0.f) : ((mode == 1) ? 0.f : s[k]);
        }
        *reinterpret_cast<float4*>(obs + env * SNK_OBS_DIM + 4 * j) = make_float4(v[0], v[1], v[2], v[3]);
    }
}

// ---------------------------------------------------------------------------------------------
// Self-collision clearance (SURVEY.md Q11 / 8f rank 3).  The reference loads the snake with
// URDF_USE_SELF_COLLISION (snake.py:93): Bullet then tests every pair of links except parent-child pairs, i.e.
// every pair of the 32 cylinders that are not consecutive along the chain (465 pairs).  The step kernels omit
// those pairs because they cannot touch at the joint angles the task reaches (|q| <= pi/6 + the 0.5 rad
// termination); this kernel is the counter that proves it for a given batch state: per environment, a LOWER
// BOUND of the smallest distance between two non-consecutive cylinders -- for every pair the best separation
//   gap(d) = d.(cB - cA) - support_A(d) - support_B(-d),  support(d) = h |d.a| + r sqrt(1 - (d.a)^2)
// over nine candidate directions d (the two axes, both signs; the centre line; the centre line with each axis
// projected out; the common normal, both signs).  Any unit d gives a valid bound, so the result can only
// under-estimate the true distance.  One warp per environment, lanes over pairs.
// ---------------------------------------------------------------------------------------------
struct WarpMemFk {
    float s[SNK_STATE_STRIDE];
    float Rw[NB][9];
    float pw[NB][3];
    float Rj[NB][9];
    float cc[NC][3]; // cylinder centres, world
    float ca[NC][3]; // cylinder axes, world
};
#define CLR_WARPS 4

__device__ __forceinline__ float cyl_support(const float* d, const float* a, float h, float r) {
    const float t = dot3(d, a);
    return h * fabsf(t) + r * sqrtf(fmaxf(0.f, 1.f - t * t));
}

__global__ void __launch_bounds__(CLR_WARPS * 32)
snk_self_clearance_kernel(const DevTables* __restrict__ T, const float* __restrict__ state, float* __restrict__ out, int64_t n) {
    __shared__ WarpMemFk Ws[CLR_WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t env = (int64_t)blockIdx.x * CLR_WARPS + warp;
    if (env >= n) return;
    WarpMemFk& W = Ws[warp];
    const float* gs = state + env * SNK_STATE_STRIDE;
    W.s[lane] = gs[lane];
    W.s[lane + 32] = gs[lane + 32];
    __syncwarp();
    fk(W, T, lane);
    { // lane = cylinder
        const int b = __ldg(&T->cbody[lane]);
        float c[3] = {__ldg(&T->ccen[lane][0]), __ldg(&T->ccen[lane][1]), __ldg(&T->ccen[lane][2])}, cw[3];
        float a[3] = {__ldg(&T->cax[lane][0]), __ldg(&T->cax[lane][1]), __ldg(&T->cax[lane][2])}, aw[3];
        m3v(W.Rw[b], c, cw);
        m3v(W.Rw[b], a, aw);
#pragma unroll
        for (int k = 0; k < 3; k++) { W.cc[lane][k] = W.pw[b][k] + cw[k]; W.ca[lane][k] = aw[k]; }
    }
    __syncwarp();
    float best = 3.0e38f;
#pragma unroll 1
    for (int i = 0; i < NC - 2; i++) {
        const float hi = __ldg(&T->chl[i]), ri = __ldg(&T->crad[i]);
#pragma unroll 1
        for (int j = i + 2 + lane; j < NC; j += 32) {
            const float hj = __ldg(&T->chl[j]), rj = __ldg(&T->crad[j]);
            const float* ai = W.ca[i];
            const float* aj = W.ca[j];
            const float dc[3] = {W.cc[j][0] - W.cc[i][0], W.cc[j][1] - W.cc[i][1], W.cc[j][2] - W.cc[i][2]};
            float cand[9][3];
            int nc = 0;
#pragma unroll
            for (int k = 0; k < 3; k++) { cand[0][k] = ai[k]; cand[1][k] = -ai[k]; cand[2][k] = aj[k]; cand[3][k] = -aj[k]; }
            nc = 4;
            const float nd = sqrtf(dot3(dc, dc));
            if (nd > 1e-9f) { for (int k = 0; k < 3; k++) cand[nc][k] = dc[k] / nd; nc++; }
            for (int w = 0; w < 2; w++) { // centre line with one axis projected out
                const float* ax = w ? aj : ai;
                const float t = dot3(ax, dc);
                float pr[3] = {dc[0] - ax[0] * t, dc[1] - ax[1] * t, dc[2] - ax[2] * t};
                const float np_ = sqrtf(dot3(pr, pr));
                if (np_ > 1e-9f) { for (int k = 0; k < 3; k++) cand[nc][k] = pr[k] / np_; nc++; }
            }
            float x[3];
            cross3(ai, aj, x);
            const float nx = sqrtf(dot3(x, x));
            if (nx > 1e-9f) {
                for (int k = 0; k < 3; k++) { cand[nc][k] = x[k] / nx; cand[nc + 1][k] = -x[k] / nx; }
                nc += 2;
            }
            float g = -3.0e38f;
            for (int q = 0; q < nc; q++) g = fmaxf(g, dot3(cand[q], dc) - cyl_support(cand[q], ai, hi, ri) - cyl_support(cand[q], aj, hj, rj));
            best = fminf(best, g);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = fminf(best, __shfl_xor_sync(FULL, best, o));
    if (lane == 0) out[env] = best;
}

cudaError_t snk_launch_self_clearance(const DevTables* T, const float* state, float* out, int64_t n, cudaStream_t st) {
    dim3 grid((unsigned)((n + CLR_WARPS - 1) / CLR_WARPS)), block(CLR_WARPS * 32);
    snk_self_clearance_kernel<<<grid, block, 0, st>>>(T, state, out, n);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// launch wrappers used by the C-ABI host code (snake_abi.cu)
// ---------------------------------------------------------------------------------------------
size_t snk_pgs_smem_bytes() { return sizeof(WarpMemPgs) * WARPS_PER_CTA; }

cudaError_t snk_pgs_configure() {
    cudaError_t e = cudaFuncSetAttribute(snk_env_kernel<WarpMemPgs, false, WARPS_PER_CTA, CTAS_PER_SM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)snk_pgs_smem_bytes());
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(snk_env_kernel<WarpMemPgs, true, WARPS_PER_CTA, CTAS_PER_SM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)snk_pgs_smem_bytes());
}

cudaError_t snk_pgs_launch_step(const DevTables* T, const KParams& P, float* state, const float* actions, float* obs, float* rew, uint8_t* done,
                            int32_t* ticks, unsigned long long* counters, int64_t n, cudaStream_t st, float* tick_obs, float* tick_links) {
    dim3 grid((unsigned)((n + WARPS_PER_CTA - 1) / WARPS_PER_CTA)), block(WARPS_PER_CTA * 32);
    snk_env_kernel<WarpMemPgs, false, WARPS_PER_CTA, CTAS_PER_SM><<<grid, block, snk_pgs_smem_bytes(), st>>>(T, P, state, actions, obs, rew, done, ticks, counters, n, 0,
                                                                                                    tick_obs, tick_links);
    return cudaGetLastError();
}

cudaError_t snk_pgs_launch_tick(const DevTables* T, const KParams& P, float* state, const float* targets, unsigned long long* counters, int64_t n,
                            int n_ticks, cudaStream_t st) {
    dim3 grid((unsigned)((n + WARPS_PER_CTA - 1) / WARPS_PER_CTA)), block(WARPS_PER_CTA * 32);
    snk_env_kernel<WarpMemPgs, true, WARPS_PER_CTA, CTAS_PER_SM><<<grid, block, snk_pgs_smem_bytes(), st>>>(T, P, state, targets, nullptr, nullptr, nullptr, nullptr, counters, n, n_ticks);
    return cudaGetLastError();
}

// the same env-step with the joint-limit rows at +-lim_angle (snk_set_joint_limits); counters[SNK_CTR_LIMIT_ROWS] accumulates the rows active at the end
// of the ticks (snk_joint_limit_stats)
template <bool RAW>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, CTAS_PER_SM)
snk_lim_env_kernel(const DevTables* __restrict__ T, const KParams P, float* __restrict__ state, const float* __restrict__ in,
                   float* __restrict__ obs, float* __restrict__ rew, uint8_t* __restrict__ done, int32_t* __restrict__ ticks,
                   unsigned long long* __restrict__ counters, int64_t n, int n_ticks, float* __restrict__ tick_obs, float* __restrict__ tick_links,
                   float lim_angle) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t env = (int64_t)blockIdx.x * WARPS_PER_CTA + warp;
    if (env >= n) return;
    WarpMemPgsLim& W = reinterpret_cast<WarpMemPgsLim*>(smem_raw)[warp];
    if (lane == 0) { W.lim_angle = lim_angle; W.lim_active = 0; } // visible behind env_step's first __syncwarp
    env_step<WarpMemPgsLim, RAW>(W, lane, env, T, P, state, in, obs, rew, done, ticks, counters, n_ticks, tick_obs, tick_links);
    if (lane == 0 && counters && W.lim_active) atomicAdd(&counters[SNK_CTR_LIMIT_ROWS], (unsigned long long)W.lim_active);
}

size_t snk_pgs_lim_smem_bytes() { return sizeof(WarpMemPgsLim) * WARPS_PER_CTA; }

cudaError_t snk_pgs_lim_configure() {
    cudaError_t e = cudaFuncSetAttribute(snk_lim_env_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)snk_pgs_lim_smem_bytes());
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(snk_lim_env_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)snk_pgs_lim_smem_bytes());
}

cudaError_t snk_pgs_lim_launch_step(const DevTables* T, const KParams& P, float lim_angle, float* state, const float* actions, float* obs, float* rew,
                                    uint8_t* done, int32_t* ticks, unsigned long long* counters, int64_t n, cudaStream_t st, float* tick_obs,
                                    float* tick_links) {
    dim3 grid((unsigned)((n + WARPS_PER_CTA - 1) / WARPS_PER_CTA)), block(WARPS_PER_CTA * 32);
    snk_lim_env_kernel<false><<<grid, block, snk_pgs_lim_smem_bytes(), st>>>(T, P, state, actions, obs, rew, done, ticks, counters, n, 0, tick_obs,
                                                                             tick_links, lim_angle);
    return cudaGetLastError();
}

cudaError_t snk_pgs_lim_launch_tick(const DevTables* T, const KParams& P, float lim_angle, float* state, const float* targets,
                                    unsigned long long* counters, int64_t n, int n_ticks, cudaStream_t st) {
    dim3 grid((unsigned)((n + WARPS_PER_CTA - 1) / WARPS_PER_CTA)), block(WARPS_PER_CTA * 32);
    snk_lim_env_kernel<true><<<grid, block, snk_pgs_lim_smem_bytes(), st>>>(T, P, state, targets, nullptr, nullptr, nullptr, nullptr, counters, n,
                                                                            n_ticks, nullptr, nullptr, lim_angle);
    return cudaGetLastError();
}

cudaError_t snk_launch_reset(const KParams& P, float* state, const uint8_t* mask, float* obs, int64_t n, int mode, cudaStream_t st) {
    int64_t total = n * 16;
    dim3 grid((unsigned)((total + 255) / 256)), block(256);
    snk_reset_kernel<<<grid, block, 0, st>>>(P, state, mask, obs, n, mode);
    return cudaGetLastError();
}

// Bullet's literal tick: the same tick on the persistent manifolds' contact set (snk_set_bullet_tick)
#include "snake_pgs_manifold.cuh"
