// snake_pgs_manifold.cuh -- Bullet's literal tick (snk_set_bullet_tick): the warp-per-environment Bullet-order tick of snake_pgs.cu
// (motor rows relaxed inside the PGS, deviation D4 of DESIGN.md lifted) on the contact set of Bullet's persistent manifolds with warm
// starting (deviation D1 lifted).  Oracle twin: tick_bt in tests/oracle_bt/bullet_tick_oracle.c.
// Included at the end of snake_pgs.cu: it reuses that file's forward dynamics (pgs_dynamics), impulse response and finish.
//
// Per tick, lane roles:
//   manifold update            : lane = cylinder; the port of man_update / man_sort_cached (snake_manifold.cuh) on this kernel's tables,
//                                cache layout byte for byte that of snk_set_manifold (SNK_MAN_STRIDE floats per environment)
//   point compaction           : a warp prefix sum over the per-cylinder counts gives each cached point its index in the oracle's
//                                cylinder-major order
//   rows                       : lanes over points, rounds of 32 points; a point = one normal row + one friction pair, one impulse response
//                                per row.  The tail of the last round is zero rows, which are no-ops of the block solver
//   block Gauss-Seidel         : the motor block of snake_pgs.cu, then ceil(NP / 32) normal blocks and ceil(NP / 16) friction blocks, each
//                                with its packed Delassus triangle; the warm start acts on dv before the first sweep
//   write-back                 : lane = cylinder, the normal impulse of each of its points into the slot (only a tick that runs touches
//                                the caches: the height test of the env-step comes after the tick, as in the oracle)
//
// Storage: every row of the up to 128 points lives in the warp's shared memory (no global scratch, no persistent grid): 100.8 KB per
// warp, one warp per CTA, 2 CTAs per SM.
#pragma once

#define BT_SLOTS 4
#define BT_SLOT_W 8                         // lp.x lp.y lp.z dist | anchor.x anchor.y impulse_n spare (snake_manifold.cuh)
#define BT_CYL_W (BT_SLOTS * BT_SLOT_W)
#define BT_NP (BT_SLOTS * NC)               // contact points at most
#define BT_NR (NJ + 3 * BT_NP)              // rows at most: motors, normals, friction pairs
#define BT_NBN (BT_NP / 32)                 // normal blocks at most
#define BT_NBF (BT_NP / 16)                 // friction blocks at most
#define BT_CTAS_PER_SM 2
static_assert(NC * BT_CYL_W + NC == SNK_MAN_STRIDE, "the cache layout of include/snake_b200.h (snk_get_manifold_cache) is this one");
static_assert(NC == 32, "lane = cylinder");

struct WarpMemBt {
    float s[SNK_STATE_STRIDE];
    float Rw[NB][9];
    float pw[NB][3];
    float nu[ND];
    float nuF[ND];
    float target[NJ];
    float J[3 * BT_NP][JS];  // contact row r: normal row of point p at r = p, friction rows at r = BT_NP + 2p, BT_NP + 2p + 1
    float B[BT_NR][ND];      // motor row j at j, contact row r at NJ + r (rhs, invD alike)
    float rhs[BT_NR];
    float invD[BT_NR];
    float lam[3 * BT_NP];    // contact impulses (index r)
    float dvs[32];
    float dl[32];
    union {
        struct {
            float Rj[NB][9];
            float U[NB][6];
            float Dinv[NB];
            float uu[NB];
            float IA0inv[36];
            union {
                struct {       // forward-dynamics workspace (pgs_dynamics)
                    float v[NB][6];
                    float cb[NB][6];
                    float pA[NB][6];
                    float IA[NB][36];
                    float X[36];
                    float Ia[36];
                    float Tm[36];
                    float pa[6];
                };
                struct {       // the tick's points while the rows are built: world position, distance; warm-start impulse; cylinder
                    float pp[BT_NP][4];
                    float pwarm[BT_NP];
                    int pcyl[BT_NP];
                };
            };
        };
        float A[BT_NBN + BT_NBF][APACK]; // in-block Delassus triangles (as An / Af of WarpMemPgs): normal blocks, then friction blocks
    };
};
static_assert((sizeof(WarpMemBt) + 1024) * BT_CTAS_PER_SM <= 233472, "BT_CTAS_PER_SM CTAs of the Bullet-tick kernel must fit into an SM");

__device__ __noinline__ void impulse_response(const WarpMemBt& W, const DevTables* __restrict__ T, int b, const float* f6, int jm, float* out) {
    impulse_response_body(W, T, b, f6, jm, out);
}

// btPersistentManifold::sortCachedPoints (oracle: man_sort_cached): the slot a new point replaces in a full cache
__device__ __forceinline__ int bt_sort_cached(const float (&mc)[BT_CYL_W], const float* lp, float dist) {
    int deepest = -1;
    float maxpen = dist;
#pragma unroll
    for (int i = 0; i < BT_SLOTS; i++)
        if (mc[i * BT_SLOT_W + 3] < maxpen) { deepest = i; maxpen = mc[i * BT_SLOT_W + 3]; }
    float res[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int p0 = (k == 0) ? 1 : 0, p1 = (k == 3) ? 2 : 3, p2 = (k < 2) ? 2 : 1; // {1,3,2},{0,3,2},{0,3,1},{0,2,1}
        if (deepest == k) continue;
        float a[3], b[3], cr[3];
#pragma unroll
        for (int q = 0; q < 3; q++) { a[q] = lp[q] - mc[p0 * BT_SLOT_W + q]; b[q] = mc[p1 * BT_SLOT_W + q] - mc[p2 * BT_SLOT_W + q]; }
        cross3(a, b, cr);
        res[k] = dot3(cr, cr);
    }
    int best = 0;
    float bestr = res[0];
#pragma unroll
    for (int k = 1; k < 4; k++) if (res[k] > bestr) { bestr = res[k]; best = k; }
    return best;
}

// One collision-detection pass of cylinder c (oracle: manifold_update; port of man_update): R, pb = world frame of the cylinder's body,
// mc = its 4 slots (registers: every slot index is a compile-time constant), n = its point count.  Returns the new count.
__device__ __forceinline__ int bt_man_update(const DevTables* __restrict__ T, int c, const float* R, const float* pb, float (&mc)[BT_CYL_W], int n) {
    const float brk = __ldg(&T->cbrk[c]), mar = __ldg(&T->cmar[c]), rad = __ldg(&T->crad[c]), hl = __ldg(&T->chl[c]);
    float F[9];
#pragma unroll
    for (int k = 0; k < 9; k++) F[k] = __ldg(&T->cfr[c][k]);
    // world-z of the body-frame hull vertex ccen + F (r sin t, r cos t, +-hl):  z0 + g0 r sin t + g1 r cos t +- g2 hl
    const float g0 = R[6] * F[0] + R[7] * F[3] + R[8] * F[6];
    const float g1 = R[6] * F[1] + R[7] * F[4] + R[8] * F[7];
    const float g2 = R[6] * F[2] + R[7] * F[5] + R[8] * F[8];
    float bestv = g1, bs = 0.f, bc = 1.f; // vertex 0: sin 0 = 0, cos 0 = 1
#pragma unroll 4
    for (int i = 1; i < 32; i++) {
        float sn, cs;
        sincospif((float)i * (1.f / 16.f), &sn, &cs); // 2 pi i / 32
        const float v = g0 * sn + g1 * cs;
        if (v < bestv) { bestv = v; bs = sn; bc = cs; }
    }
    const float zend = (-hl * g2 <= hl * g2) ? -hl : hl; // the rim z = -L/2 comes first in the hull (ties go to it)
    const float vl[3] = {rad * bs, rad * bc, zend};
    float vb[3], rv[3];
#pragma unroll
    for (int k = 0; k < 3; k++) vb[k] = __ldg(&T->ccen[c][k]) + F[3 * k] * vl[0] + F[3 * k + 1] * vl[1] + F[3 * k + 2] * vl[2];
    m3v(R, vb, rv);
    const float rel[3] = {rv[0], rv[1], rv[2] - mar}; // localGetSupportingVertex adds the margin along the query direction -n
    const float dist = pb[2] + rel[2];
    if (dist < brk) {
        float lp[3];
        m3tv(R, rel, lp);
        int idx = -1;
        float shortest = brk * brk;
#pragma unroll
        for (int i = 0; i < BT_SLOTS; i++)
            if (i < n) {
                const float d[3] = {mc[i * BT_SLOT_W] - lp[0], mc[i * BT_SLOT_W + 1] - lp[1], mc[i * BT_SLOT_W + 2] - lp[2]};
                const float d2 = dot3(d, d);
                if (d2 < shortest) { shortest = d2; idx = i; }
            }
        float imp = 0.f;
        if (idx >= 0) { // replaceContactPoint keeps the cached impulse
#pragma unroll
            for (int i = 0; i < BT_SLOTS; i++) if (idx == i) imp = mc[i * BT_SLOT_W + 6];
        } else if (n < BT_SLOTS) idx = n++;
        else idx = bt_sort_cached(mc, lp, dist);
        const float ax = pb[0] + rel[0], ay = pb[1] + rel[1];
#pragma unroll
        for (int i = 0; i < BT_SLOTS; i++)
            if (idx == i) {
                mc[i * BT_SLOT_W] = lp[0]; mc[i * BT_SLOT_W + 1] = lp[1]; mc[i * BT_SLOT_W + 2] = lp[2]; mc[i * BT_SLOT_W + 3] = dist;
                mc[i * BT_SLOT_W + 4] = ax; mc[i * BT_SLOT_W + 5] = ay; mc[i * BT_SLOT_W + 6] = imp; mc[i * BT_SLOT_W + 7] = 0.f;
            }
    }
#pragma unroll
    for (int i = BT_SLOTS - 1; i >= 0; i--) // refreshContactPoints
        if (i < n) {
            float w[3];
            const float l[3] = {mc[i * BT_SLOT_W], mc[i * BT_SLOT_W + 1], mc[i * BT_SLOT_W + 2]};
            m3v(R, l, w);
            const float pos[3] = {pb[0] + w[0], pb[1] + w[1], pb[2] + w[2]};
            mc[i * BT_SLOT_W + 3] = pos[2];
            const float dx = mc[i * BT_SLOT_W + 4] - pos[0], dy = mc[i * BT_SLOT_W + 5] - pos[1];
            if (pos[2] > brk || dx * dx + dy * dy > brk * brk) { // removeContactPoint: the last point takes the slot
                const int last = n - 1;
#pragma unroll
                for (int q = 0; q < BT_SLOT_W; q++) {
                    float v = mc[i * BT_SLOT_W + q];
#pragma unroll
                    for (int l2 = i + 1; l2 < BT_SLOTS; l2++) if (last == l2) v = mc[l2 * BT_SLOT_W + q];
                    mc[i * BT_SLOT_W + q] = v;
                }
                n--;
            }
        }
    return n;
}

// ---------------------------------------------------------------------------------------------
// one physics tick (oracle: tick with the bullet switch on).  cache: this environment's SNK_MAN_STRIDE floats.  Returns the PGS
// iteration count; *np_out = cached points of the tick.  LIM: with the joint-limit rows at +-lim_angle (snake_pgs.cu: pgs_limit_block)
// after the motor rows; *lim_active accumulates the limit rows active at the end of the tick.
// ---------------------------------------------------------------------------------------------
template <bool LIM>
__device__ int tick_bt(WarpMemBt& W, const DevTables* __restrict__ T, const KParams& P, int lane, float* __restrict__ cache, float warm, int* np_out,
                       float lim_angle, unsigned* lim_active) {
    pgs_dynamics(W, T, P, lane);

    // ---- manifolds, lane = cylinder; the forward-dynamics workspace is dead from here on and holds the point table ----
    const int cyl = lane;
    int ncyl, base, NP;
    {
        const int b = __ldg(&T->cbody[cyl]);
        float mc[BT_CYL_W];
#pragma unroll
        for (int k = 0; k < BT_CYL_W; k++) mc[k] = 0.f;
        float4* gc = reinterpret_cast<float4*>(cache + cyl * BT_CYL_W);
        const int n_old = (int)cache[NC * BT_CYL_W + cyl];
#pragma unroll
        for (int q = 0; q < BT_SLOTS; q++)
            if (q < n_old) {
                const float4 u = gc[2 * q], v = gc[2 * q + 1];
                mc[8 * q] = u.x; mc[8 * q + 1] = u.y; mc[8 * q + 2] = u.z; mc[8 * q + 3] = u.w;
                mc[8 * q + 4] = v.x; mc[8 * q + 5] = v.y; mc[8 * q + 6] = v.z; mc[8 * q + 7] = v.w;
            }
        ncyl = bt_man_update(T, cyl, W.Rw[b], W.pw[b], mc, n_old);
#pragma unroll
        for (int q = 0; q < BT_SLOTS; q++)
            if (q < ncyl) {
                gc[2 * q] = make_float4(mc[8 * q], mc[8 * q + 1], mc[8 * q + 2], mc[8 * q + 3]);
                gc[2 * q + 1] = make_float4(mc[8 * q + 4], mc[8 * q + 5], mc[8 * q + 6], mc[8 * q + 7]);
            }
        if (ncyl != n_old) cache[NC * BT_CYL_W + cyl] = (float)ncyl;
        // cylinder-major point order: exclusive prefix sum of the counts
        int incl = ncyl;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += t;
        }
        base = incl - ncyl;
        NP = __shfl_sync(FULL, incl, 31);
#pragma unroll
        for (int q = 0; q < BT_SLOTS; q++)
            if (q < ncyl) {
                const float l[3] = {mc[8 * q], mc[8 * q + 1], mc[8 * q + 2]};
                float w[3];
                m3v(W.Rw[b], l, w);
                const int p = base + q;
                W.pp[p][0] = W.pw[b][0] + w[0]; W.pp[p][1] = W.pw[b][1] + w[1]; W.pp[p][2] = W.pw[b][2] + w[2]; W.pp[p][3] = mc[8 * q + 3];
                W.pwarm[p] = mc[8 * q + 6] * warm;
                W.pcyl[p] = cyl;
            }
    }
    __syncwarp();

    // ---- constraint rows ----
    if (lane < NJ) { // motor row of joint lane+1 (A.4)
        const int j = lane;
        const float zero6[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        impulse_response(W, T, -1, zero6, j + 1, W.B[j]);
        float D = W.B[j][6 + j];
        float q = W.s[SNK_S_Q + j], qd = W.nu[6 + j];
        float vt = P.kp * (W.target[j] - q) * P.inv_dt + qd + P.kd * (0.f - qd);
        W.invD[j] = 1.f / D; W.rhs[j] = (vt - qd) / D;
    }
    const int nbn = (NP + 31) >> 5, nbf = (NP + 15) >> 4;
#pragma unroll 1
    for (int rnd = 0; rnd < nbn; rnd++) { // lanes over points, 32 per round
        const int pt = 32 * rnd + lane;
        if (pt >= NP) { // the tail of the last block: all-zero rows are no-ops of the block solver
#pragma unroll 1
            for (int f = 0; f < 3; f++) {
                const int r = (f == 0) ? pt : BT_NP + 2 * pt + (f - 1);
#pragma unroll 1
                for (int k = 0; k < ND; k++) { W.J[r][k] = 0.f; W.B[NJ + r][k] = 0.f; }
                W.invD[NJ + r] = 0.f; W.rhs[NJ + r] = 0.f;
            }
            continue;
        }
        const int c = W.pcyl[pt];
        const int b = __ldg(&T->cbody[c]);
        const float p[3] = {W.pp[pt][0], W.pp[pt][1], W.pp[pt][2]}, dist = W.pp[pt][3];
        float Rl[9], cfr[9];
#pragma unroll
        for (int k = 0; k < 9; k++) cfr[k] = __ldg(&T->cfr[c][k]);
        m3m3(W.Rw[b], cfr, Rl);
#pragma unroll 1
        for (int f = 0; f < 3; f++) {
            float d[3] = {0.f, 0.f, 1.f};
            if (f > 0) {
                float t[3] = {(f == 2) ? 1.f : 0.f, (f == 1) ? -1.f : 0.f, 0.f}, loc[3];
                m3tv(Rl, t, loc);
                loc[0] *= P.aniso[0]; loc[1] *= P.aniso[1]; loc[2] *= P.aniso[2];
                m3v(Rl, loc, d);
            }
            const int r = (f == 0) ? pt : BT_NP + 2 * pt + (f - 1);
            float* Jr = W.J[r];
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
    // impulses: the normal rows start at the cached impulse x warm factor (zero rows at 0), the friction rows at 0
#pragma unroll 1
    for (int r = lane; r < 32 * nbn; r += 32) W.lam[r] = (r < NP) ? W.pwarm[r] : 0.f;
#pragma unroll 1
    for (int r = lane; r < 32 * nbf; r += 32) W.lam[BT_NP + r] = 0.f;
    __syncwarp();

    const bool dof = lane < ND;
    const int ld = dof ? lane : 0;
    const int lm = lane & (NJ - 1);
    float dv = 0.f;
    if (warm > 0.f && dof) { // warm start (A.5): the effect of the starting impulses acts on dv before the first sweep
#pragma unroll 1
        for (int p = 0; p < NP; p++) dv += W.B[NJ + p][ld] * W.lam[p];
    }
    // ---- in-block Delassus entries A(i, j) = J_j . B_i for the rows j > i of the same block (lane = row j); the point table is dead ----
#pragma unroll 1
    for (int g = 0; g < nbn + nbf; g++) {
        const int r0 = (g < nbn) ? 32 * g : BT_NP + 32 * (g - nbn);
        float* Ag = W.A[(g < nbn) ? g : BT_NBN + (g - nbn)];
        float Jr[ND];
#pragma unroll
        for (int k = 0; k < ND; k++) Jr[k] = W.J[r0 + lane][k];
#pragma unroll 1
        for (int i = 0; i < 31; i++) {
            const float* Bi = W.B[NJ + r0 + i];
            float a0 = 0.f, a1 = 0.f;
#pragma unroll
            for (int k = 0; k < ND; k += 2) { a0 = fmaf(Jr[k], Bi[k], a0); a1 = fmaf(Jr[k + 1], Bi[k + 1], a1); }
            if (lane > i) Ag[A_OFF(i) + lane - i] = a0 + a1;
        }
    }

    // ---- projected Gauss-Seidel in block form (snake_pgs.cu: tick), rows in Bullet's order: motors, normals, friction pairs ----
    float lam_m = 0.f;
    W.dvs[lane] = dof ? dv : 0.f;
    const float m_rhs = W.rhs[lm], m_iD = W.invD[lm], m_Dg = (m_iD != 0.f) ? 1.f / m_iD : 0.f;
    const int pa = lane & ~1; // the lane pair (pa, pa + 1) holds the two friction rows of one point
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
            float bn = W.B[rev ? NJ - 1 : 0][6 + lm];
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
#pragma unroll 1
        for (int g = 0; g < nbn; g++) { // ---- normal rows of points 32 g .. 32 g + 31, lane = point ----
            const int row = 32 * g + lane;
            const float n_rhs = W.rhs[NJ + row], n_iD = W.invD[NJ + row], n_Dg = (n_iD != 0.f) ? 1.f / n_iD : 0.f;
            const float* Jn = W.J[row];
            float w0 = 0.f, w1 = 0.f;
#pragma unroll
            for (int k = 0; k < ND; k += 2) { w0 = fmaf(Jn[k], W.dvs[k], w0); w1 = fmaf(Jn[k + 1], W.dvs[k + 1], w1); }
            float w = w0 + w1, lam = W.lam[row], dmine = 0.f;
            const float* Ap = W.A[g] + lane;
            int aoff = 0;
            float an = Ap[0];
#pragma unroll 4
            for (int i = 0; i < 32; i++) {
                const float a = an;
                aoff += 32 - i - 2;
                an = Ap[i < 30 ? aoff : 0];
                const float d0 = n_rhs - w * n_iD;
                const float sum0 = lam + d0;
                const bool neg = sum0 < 0.f;
                const float sum = neg ? 0.f : sum0, d = neg ? -lam : d0;
                const float di = __shfl_sync(FULL, d, i);
                const bool mine = lane == i;
                lam = mine ? sum : lam; dmine = mine ? d : dmine;
                w = fmaf(a, di, w);
            }
            W.lam[row] = lam;
            W.dl[lane] = dmine;
            __syncwarp();
            if (dof) {
                float x0 = 0.f, x1 = 0.f;
                const int rb = NJ + 32 * g;
#pragma unroll
                for (int i = 0; i < 32; i += 2) { x0 = fmaf(W.B[rb + i][ld], W.dl[i], x0); x1 = fmaf(W.B[rb + i + 1][ld], W.dl[i + 1], x1); }
                dv += x0 + x1;
                W.dvs[lane] = dv;
            }
            const float rr = dmine * n_Dg;
            res = fmaxf(res, rr * rr);
            __syncwarp();
        }
#pragma unroll 1
        for (int fb = 0; fb < nbf; fb++) { // ---- friction pairs of points 16 fb .. 16 fb + 15 ----
            // lanes 2p and 2p + 1 both carry BOTH rows of point 16 fb + p, so the cone projection needs no exchange between lanes
            const int ra = BT_NP + 32 * fb + pa, rb = ra + 1;
            const float a_rhs = W.rhs[NJ + ra], a_iD = W.invD[NJ + ra], b_rhs = W.rhs[NJ + rb], b_iD = W.invD[NJ + rb];
            const float a_Dg = (a_iD != 0.f) ? 1.f / a_iD : 0.f, b_Dg = (b_iD != 0.f) ? 1.f / b_iD : 0.f;
            const float* Ja = W.J[ra];
            const float* Jb = W.J[rb];
            float wa = 0.f, wb = 0.f;
#pragma unroll
            for (int k = 0; k < ND; k++) { const float x = W.dvs[k]; wa = fmaf(Ja[k], x, wa); wb = fmaf(Jb[k], x, wb); }
            float la = W.lam[ra], lb = W.lam[rb], da_mine = 0.f, db_mine = 0.f;
            const float lim = mu * W.lam[16 * fb + (lane >> 1)];
            const float* Aq = W.A[BT_NBN + fb] + pa;
            int o0 = 0;
            float a00 = Aq[0], a01 = Aq[1], a10 = Aq[30], a11 = Aq[31];
#pragma unroll 2
            for (int p = 0; p < 16; p++) {
                const float c00 = a00, c01 = a01, c10 = a10, c11 = a11;
                o0 += 2 * 32 - 4 * p - 5; // A_OFF(2p + 2) - (2p + 2) - (A_OFF(2p) - 2p)
                {
                    const int q0 = p < 15 ? o0 : 0, q1 = p < 15 ? o0 + 32 - 2 * p - 4 : 0; // nothing left to fetch for the last pair
                    a00 = Aq[q0]; a01 = Aq[q0 + 1]; a10 = Aq[q1]; a11 = Aq[q1 + 1];
                }
                float sa = la + (a_rhs - wa * a_iD), sb = lb + (b_rhs - wb * b_iD);
                if (cone) { // implicit cone: s <- s min(1, lim / |s|)
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
                wa = fmaf(c00, da, fmaf(c10, db, wa));
                wb = fmaf(c01, da, fmaf(c11, db, wb));
            }
            W.lam[BT_NP + 32 * fb + lane] = (lane & 1) ? lb : la;
            W.dl[lane] = (lane & 1) ? db_mine : da_mine;
            __syncwarp();
            if (dof) {
                float x0 = 0.f, x1 = 0.f;
                const int rb0 = NJ + BT_NP + 32 * fb;
#pragma unroll
                for (int i = 0; i < 32; i += 2) { x0 = fmaf(W.B[rb0 + i][ld], W.dl[i], x0); x1 = fmaf(W.B[rb0 + i + 1][ld], W.dl[i + 1], x1); }
                dv += x0 + x1;
                W.dvs[lane] = dv;
            }
            const float rr = fmaf(da_mine, a_Dg, db_mine * b_Dg);
            res = fmaxf(res, rr * rr);
            __syncwarp();
        }
        res = __uint_as_float(__reduce_max_sync(FULL, __float_as_uint(res))); // res >= 0: the bit patterns order like the values
        if (res <= P.resthr || it >= P.iters - 1) break;
    }
    if constexpr (LIM) *lim_active += limit_rows_active(lam_lo, lam_up);
    // the normal impulses go back into the slots (m_appliedImpulse), lane = cylinder
#pragma unroll
    for (int q = 0; q < BT_SLOTS; q++)
        if (q < ncyl) cache[cyl * BT_CYL_W + q * BT_SLOT_W + 6] = W.lam[base + q];
    pgs_finish(W, T, P, lane, dv, lam_m);
    *np_out = NP;
    return it + 1;
}

// ---------------------------------------------------------------------------------------------
// kernel: snk_env_kernel's task logic (snake_task.cuh) around tick_bt, one warp (= one CTA) per environment.  RAW = false: one
// SubprocVecEnv.step (tick_obs / tick_links: the mode='test' info stream, either may be null); RAW = true: n_ticks raw ticks with
// targets[N,16].  cache: [N][SNK_MAN_STRIDE].  counters[7] accumulates the cached points over the ticks (snk_manifold_stats); with LIM
// (the joint-limit rows at +-lim_angle) counters[SNK_CTR_LIMIT_ROWS] the limit rows active at the end of the ticks (snk_joint_limit_stats).
// ---------------------------------------------------------------------------------------------
template <bool RAW, bool LIM>
__device__ __forceinline__ void bt_env_step(WarpMemBt& W, int lane, int64_t env, const DevTables* __restrict__ T, const KParams P, float* __restrict__ state, const float* __restrict__ in,
                                            float* __restrict__ obs, float* __restrict__ rew, uint8_t* __restrict__ done, int32_t* __restrict__ ticks,
                                            unsigned long long* __restrict__ counters, int n_ticks, float* __restrict__ tick_obs,
                                            float* __restrict__ tick_links, float* __restrict__ cache, float warm, float lim_angle) {
    unsigned lim_active = 0;
    float* mc = cache + env * SNK_MAN_STRIDE;
    float* gs = state + env * SNK_STATE_STRIDE;
    W.s[lane] = gs[lane];
    W.s[lane + 32] = gs[lane + 32];
    if (lane < NJ) {
        float tgt;
        if (RAW) tgt = in[env * NJ + lane];
        else { // checkBound (SnakeGymEnv.py:82-88) + createAction (snake.py:247-269) + scaling (snake.py:223-225)
            int k = -1;
            if (P.gait == 0) { if (!(lane & 1)) k = lane >> 1; }
            else if (P.gait == 1) { if (lane & 1) k = lane >> 1; }
            else k = lane;
            float a = (k >= 0) ? in[env * P.actdim + k] : 0.f;
            a = (a < -1.f) ? -1.f : a;
            a = (a > 1.f) ? 1.f : a;
            tgt = a * P.sf;
        }
        W.target[lane] = tgt;
    }
    __syncwarp();
    const float xprev = W.s[SNK_S_POS];
    float height = fk(W, T, lane);
    int counter = 0, iters = 0;
    unsigned long long points = 0;
    bool end_height = false;
    if (RAW) {
        for (int t = 0; t < n_ticks; t++) {
            int np;
            iters += tick_bt<LIM>(W, T, P, lane, mc, warm, &np, LIM ? lim_angle : 0.f, LIM ? &lim_active : nullptr);
            points += (unsigned long long)np;
            counter++;
            height = fk(W, T, lane);
        }
    } else {
        for (;;) { // snake.py:284-304
            float e2 = 0.f;
#pragma unroll 1
            for (int j = 0; j < NJ; j++) { float d = W.target[j] - W.s[SNK_S_Q + j]; e2 += d * d; }
            if (!(sqrtf(e2) > P.errthr)) break;
            int np;
            iters += tick_bt<LIM>(W, T, P, lane, mc, warm, &np, LIM ? lim_angle : 0.f, LIM ? &lim_active : nullptr);
            points += (unsigned long long)np;
            height = fk(W, T, lane);
            if (tick_obs) { // mode='test' info stream (snake.py:291-292): the observation after this tick
                float* to = tick_obs + (env * P.maxticks + counter) * SNK_OBS_DIM;
                to[lane] = obs_of(W, lane);
                if (lane + 32 < SNK_OBS_DIM) to[lane + 32] = obs_of(W, lane + 32);
            }
            if (tick_links && lane < NB) { // snake.py:293,138-146: [x0..x16 | y0..y16 | z0..z16], lane = link
                const int b = __ldg(&T->hbody[lane]);
                float* tl = tick_links + (env * P.maxticks + counter) * (3 * NB);
#pragma unroll
                for (int k = 0; k < 3; k++)
                    tl[k * NB + lane] = W.pw[b][k] + W.Rw[b][3 * k] * __ldg(&T->hpt[lane][0]) + W.Rw[b][3 * k + 1] * __ldg(&T->hpt[lane][1]) +
                                        W.Rw[b][3 * k + 2] * __ldg(&T->hpt[lane][2]);
            }
            counter++;
            if (height > P.hthr) { end_height = true; break; }
            if (counter >= P.maxticks) break;
        }
    }
    if (lane == 0 && counters && points) atomicAdd(&counters[7], points);
    if constexpr (LIM) { if (lane == 0 && counters && lim_active) atomicAdd(&counters[SNK_CTR_LIMIT_ROWS], (unsigned long long)lim_active); }
    if (RAW) {
        gs[lane] = W.s[lane];
        gs[lane + 32] = W.s[lane + 32];
        if (lane == 0 && counters) { atomicAdd(&counters[0], (unsigned long long)counter); atomicAdd(&counters[1], (unsigned long long)iters); }
        return;
    }
    const bool bad = __any_sync(FULL, !isfinite(W.s[lane]) || !isfinite(W.s[lane + 32]));
    // reward (SnakeGymEnv.py:90-97, snake.py:336-341) and termination (SnakeGymEnv.py:99-103), every lane
    float energy = 0.f;
#pragma unroll 1
    for (int j = 0; j < NJ; j++) energy += W.s[SNK_S_QD + j] * W.s[SNK_S_TAU + j] * P.edt;
    float r = P.alpha * (W.s[SNK_S_POS] - xprev) + ((fabsf(W.s[SNK_S_FZ]) > P.colf) ? P.colpen : 0.f) - P.beta * fabsf(W.s[SNK_S_POS + 1] - 0.f) -
              P.gamma * energy;
    bool d = (fabsf(obs_of(W, P.tjoint)) > P.tang) || (height > P.hthr) || end_height;
    if (bad) { d = true; r = P.donepen; }
    else if (d) r += P.donepen;
    __syncwarp();
    if (bad) { // force-reset: the environment restarts like a hard reset, its caches (impulses of this step not finite) emptied
        W.s[lane] = 0.f; W.s[lane + 32] = 0.f;
#pragma unroll 1
        for (int k = 4 * lane; k < SNK_MAN_STRIDE; k += 128) *reinterpret_cast<float4*>(mc + k) = make_float4(0.f, 0.f, 0.f, 0.f);
        __syncwarp();
    }
    if (lane == 0) { W.s[SNK_S_RET] += r; W.s[SNK_S_LEN] += 1.f; }
    __syncwarp();
    if (d) { soft_reset(W, P, lane); __syncwarp(); } // in-step reset + worker reset: post-reset obs (multiprocessing_env.py:14-15)
    float* go = obs + env * SNK_OBS_DIM;
    go[lane] = obs_of(W, lane);
    if (lane + 32 < SNK_OBS_DIM) go[lane + 32] = obs_of(W, lane + 32);
    gs[lane] = W.s[lane];
    gs[lane + 32] = W.s[lane + 32];
    if (lane == 0) {
        rew[env] = r;
        done[env] = d ? 1 : 0;
        if (ticks) ticks[env] = counter;
        if (counters) {
            atomicAdd(&counters[0], (unsigned long long)counter);
            atomicAdd(&counters[1], (unsigned long long)iters);
            if (d) atomicAdd(&counters[2], 1ull);
            if (bad) atomicAdd(&counters[3], 1ull);
        }
    }
}

template <bool RAW>
__global__ void __launch_bounds__(32, BT_CTAS_PER_SM)
snk_bt_env_kernel(const DevTables* __restrict__ T, const KParams P, float* __restrict__ state, const float* __restrict__ in,
                  float* __restrict__ obs, float* __restrict__ rew, uint8_t* __restrict__ done, int32_t* __restrict__ ticks,
                  unsigned long long* __restrict__ counters, int64_t n, int n_ticks, float* __restrict__ tick_obs, float* __restrict__ tick_links,
                  float* __restrict__ cache, float warm) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int64_t env = blockIdx.x;
    if (env >= n) return;
    WarpMemBt& W = *reinterpret_cast<WarpMemBt*>(smem_raw);
    bt_env_step<RAW, false>(W, lane, env, T, P, state, in, obs, rew, done, ticks, counters, n_ticks, tick_obs, tick_links, cache, warm, 0.f);
}

// Bullet's literal tick with the joint-limit rows (snk_set_joint_limits together with snk_set_bullet_tick)
template <bool RAW>
__global__ void __launch_bounds__(32, BT_CTAS_PER_SM)
snk_bt_lim_env_kernel(const DevTables* __restrict__ T, const KParams P, float* __restrict__ state, const float* __restrict__ in,
                      float* __restrict__ obs, float* __restrict__ rew, uint8_t* __restrict__ done, int32_t* __restrict__ ticks,
                      unsigned long long* __restrict__ counters, int64_t n, int n_ticks, float* __restrict__ tick_obs, float* __restrict__ tick_links,
                      float* __restrict__ cache, float warm, float lim_angle) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int64_t env = blockIdx.x;
    if (env >= n) return;
    WarpMemBt& W = *reinterpret_cast<WarpMemBt*>(smem_raw);
    bt_env_step<RAW, true>(W, lane, env, T, P, state, in, obs, rew, done, ticks, counters, n_ticks, tick_obs, tick_links, cache, warm, lim_angle);
}

size_t snk_bt_smem_bytes() { return sizeof(WarpMemBt); }

cudaError_t snk_bt_configure() {
    cudaError_t e = cudaFuncSetAttribute(snk_bt_env_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)snk_bt_smem_bytes());
    if (e == cudaSuccess) e = cudaFuncSetAttribute(snk_bt_env_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)snk_bt_smem_bytes());
    if (e == cudaSuccess) e = cudaFuncSetAttribute(snk_bt_lim_env_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)snk_bt_smem_bytes());
    if (e == cudaSuccess) e = cudaFuncSetAttribute(snk_bt_lim_env_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)snk_bt_smem_bytes());
    return e;
}

// lim: the joint-limit rows' angle, 0 = off (the kernels without them)
cudaError_t snk_bt_launch_step(const DevTables* T, const KParams& P, float* state, float* cache, float warm, float lim, const float* actions, float* obs,
                               float* rew, uint8_t* done, int32_t* ticks, unsigned long long* counters, int64_t n, cudaStream_t st, float* tick_obs,
                               float* tick_links) {
    if (lim > 0.f)
        snk_bt_lim_env_kernel<false><<<(unsigned)n, 32, snk_bt_smem_bytes(), st>>>(T, P, state, actions, obs, rew, done, ticks, counters, n, 0, tick_obs,
                                                                                   tick_links, cache, warm, lim);
    else
        snk_bt_env_kernel<false><<<(unsigned)n, 32, snk_bt_smem_bytes(), st>>>(T, P, state, actions, obs, rew, done, ticks, counters, n, 0, tick_obs, tick_links,
                                                                               cache, warm);
    return cudaGetLastError();
}

cudaError_t snk_bt_launch_tick(const DevTables* T, const KParams& P, float* state, float* cache, float warm, float lim, const float* targets,
                               unsigned long long* counters, int64_t n, int n_ticks, cudaStream_t st) {
    if (lim > 0.f)
        snk_bt_lim_env_kernel<true><<<(unsigned)n, 32, snk_bt_smem_bytes(), st>>>(T, P, state, targets, nullptr, nullptr, nullptr, nullptr, counters, n,
                                                                                  n_ticks, nullptr, nullptr, cache, warm, lim);
    else
        snk_bt_env_kernel<true><<<(unsigned)n, 32, snk_bt_smem_bytes(), st>>>(T, P, state, targets, nullptr, nullptr, nullptr, nullptr, counters, n, n_ticks,
                                                                              nullptr, nullptr, cache, warm);
    return cudaGetLastError();
}
