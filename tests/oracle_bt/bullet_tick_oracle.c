/*
 * bullet_tick_oracle.c -- Bullet's literal tick in the CPU oracle.   TEST INFRASTRUCTURE.
 *
 * The twin of snk_set_bullet_tick (bullet_envs_b200/csrc/snake_pgs_manifold.cuh): the Bullet-order tick of oracle/snake_oracle.c
 * (motor rows relaxed inside the projected Gauss-Seidel, deviation D4 of DESIGN.md lifted) on the contact set of that file's persistent
 * manifolds (deviation D1 lifted), normal impulses warm-started.  This file includes the oracle unchanged and adds, with the oracle's
 * helpers (forward_dynamics, impulse_response, manifold_update, contact_dirs, contact_jacobian, finish_tick):
 *   tick_bt      -- tick() with the contact set of the caches: every cached point of every cylinder, cylinder-major (tick_exact's
 *                   order); rows = motors, joint-limit rows if on, all normal rows, all friction pairs; the normal rows start at the
 *                   cached impulse x warm (its effect B lambda added to dv before the first sweep); the three impulses of each point
 *                   go back into its slot after the solve;
 *   bt_env_step  -- env_step_traced with tick_bt;
 *   PFX(bt_set) / PFX(bt_step_range) / PFX(bt_step) / PFX(bt_step_trace) / PFX(bt_tick) -- entry points; while the switch is off the
 *                   step and tick entry points are the oracle's own.
 * The switch is on while the handle owns caches and the exact tick's manifolds (PFX(set_manifold)) are off.
 * Build: tests/bullet_tick_oracle.py (fp64 and, with -DSNK_REAL_FLOAT, fp32 into one library).
 */
#include "../../oracle/snake_oracle.c"

static int bt_on(const Handle* h) { return h->M != NULL && !h->P.manifold; }

static void tick_bt(const Tables* T, const Par* P, real* s, const Kin* K, const real* target, TickInfo* info) {
    const real dt = P->dt;
    Aba A;
    real nu[ND];
    forward_dynamics(T, P, s, K, &A, nu);

    /* ---- constraint rows (A.3 step 5): motors, then contact normals, then friction pairs ---- */
    /* NP contact points: one per cylinder (D1; point c = cylinder c), or with the Bullet tick every cached point of every cylinder's
     * manifold, cylinder-major (tick_exact's order); normal row of point c = NJ + c, its friction pair NJ + NP + 2c, NJ + NP + 2c + 1 */
    enum { NPMAX = MAN_SLOTS * NC, NRMAX = NJ + 3 * NPMAX };
    static __thread real J[NRMAX][ND], B[NRMAX][ND];
    static __thread real rhs[NRMAX], invD[NRMAX], Dg[NRMAX], lam[NRMAX];
    static __thread real cp[NPMAX][3], cd[NPMAX][3][3], pdist[NPMAX];
    static __thread int active[NPMAX], pcyl[NPMAX], pslot[NPMAX];
    const int use_man = info->man != NULL;
    int NP = NC;
    const real maximp = P->maxf * dt;
    for (int j = 0; j < NJ; j++) { /* A.4 */
        memset(J[j], 0, sizeof J[j]);
        J[j][6 + j] = 1;
        impulse_response(T, K, &A, -1, NULL, j + 1, B[j]);
        Dg[j] = B[j][6 + j];
        invD[j] = 1 / Dg[j];
        real q = s[SNK_S_Q + j], qd = nu[6 + j];
        real vt = P->kp * (target[j] - q) / dt + qd + P->kd * (0 - qd); /* erp = 1, target velocity 0 */
        rhs[j] = (vt - qd) * invD[j];
        lam[j] = 0;
    }
    int ncontacts = 0;
    if (use_man) {
        NP = 0;
        for (int c = 0; c < NC; c++) {
            Manifold* m = &info->man[c];
            manifold_update(T, K, c, m);
            const int b = T->cbody[c];
            for (int i = 0; i < m->n; i++, NP++) {
                real w[3];
                m3v(K->Rw[b], m->pt[i].lp, w);
                for (int k = 0; k < 3; k++) cp[NP][k] = K->pw[b][k] + w[k];
                pdist[NP] = m->pt[i].dist; pcyl[NP] = c; pslot[NP] = i;
                contact_dirs(T, P, K, c, cd[NP]);
            }
        }
    }
    for (int c = 0; c < NP; c++) { /* A.5 with deviation D1, or the cached points */
        int b = T->cbody[use_man ? pcyl[c] : c];
        real* p = cp[c];
        real dist;
        real (*dirs)[3] = cd[c];
        int r0 = NJ + c, r1 = NJ + NP + 2 * c, r2 = r1 + 1;
        if (use_man) { active[c] = 1; dist = pdist[c]; }
        else active[c] = contact_geometry(T, P, K, c, p, &dist, dirs);
        lam[r0] = lam[r1] = lam[r2] = 0;
        if (!active[c]) continue;
        ncontacts++;
        int rows[3] = {r0, r1, r2};
        for (int f = 0; f < 3; f++) {
            int r = rows[f];
            const real* d = dirs[f];
            contact_jacobian(T, K, b, p, d, J[r]);
            real f6[6], db[3], pb[3], ro[3];
            m3tv(K->Rw[b], d, db);
            for (int k = 0; k < 3; k++) ro[k] = p[k] - K->pw[b][k];
            m3tv(K->Rw[b], ro, pb);
            v3cross(pb, db, f6);
            f6[3] = db[0]; f6[4] = db[1]; f6[5] = db[2];
            impulse_response(T, K, &A, b, f6, 0, B[r]);
            real D = 0, vrel = 0;
            for (int k = 0; k < ND; k++) { D += J[r][k] * B[r][k]; vrel += J[r][k] * nu[k]; }
            Dg[r] = D; invD[r] = 1 / D;
            if (f == 0) {
                real pen = dist + P->slop, verr = -vrel, perr = 0;
                if (pen > 0) verr -= pen / dt; else perr = -pen * P->erp2 / dt;
                rhs[r] = (verr + perr) * invD[r];
            } else {
                rhs[r] = -vrel * invD[r];
            }
        }
    }

    /* joint-limit rows (oracle-only switch; btMultiBodyJointLimitConstraint, A.1): two unilateral rows per joint, +e_j at the lower
     * and -e_j at the upper limit, set up like contacts (speculative while the joint is inside its range) */
    real rhsl[2 * NJ], laml[2 * NJ];
    if (P->limits)
        for (int j = 0; j < NJ; j++)
            for (int side = 0; side < 2; side++) {
                const real sgn = side ? (real)-1 : (real)1;
                const real pen = side ? (P->limit_angle - s[SNK_S_Q + j]) : (s[SNK_S_Q + j] + P->limit_angle);
                real verr = -sgn * nu[6 + j], perr = 0;
                if (pen > 0) verr -= pen / dt; else perr = -pen * P->erp2 / dt;
                rhsl[2 * j + side] = (verr + perr) * invD[j];
                laml[2 * j + side] = 0;
            }

    /* ---- projected Gauss-Seidel (A.3 step 6) ---- */
    real dv[ND];
    memset(dv, 0, sizeof dv);
    if (use_man && P->warm > 0) /* warm start (A.5): the cached normal impulse x warmstartingFactor, applied before the first sweep */
        for (int c = 0; c < NP; c++) {
            lam[NJ + c] = info->man[pcyl[c]].pt[pslot[c]].imp[0] * P->warm;
            for (int k = 0; k < ND; k++) dv[k] += B[NJ + c][k] * lam[NJ + c];
        }
    int it = 0;
    for (;; it++) {
        real res = 0;
        for (int jj = 0; jj < NJ; jj++) {
            int j = (P->altmotor && !(it & 1)) ? NJ - 1 - jj : jj;
            real d = rhs[j] - dv[6 + j] * invD[j];
            real sum = lam[j] + d;
            if (sum < -maximp) { d = -maximp - lam[j]; lam[j] = -maximp; }
            else if (sum > maximp) { d = maximp - lam[j]; lam[j] = maximp; }
            else lam[j] = sum;
            for (int k = 0; k < ND; k++) dv[k] += B[j][k] * d;
            real rr = d * Dg[j];
            if (rr * rr > res) res = rr * rr;
        }
        if (P->limits)
            for (int r = 0; r < 2 * NJ; r++) {
                const int j = r >> 1;
                const real sgn = (r & 1) ? (real)-1 : (real)1;
                real d = rhsl[r] - sgn * dv[6 + j] * invD[j];
                real sum = laml[r] + d;
                if (sum < 0) { d = -laml[r]; laml[r] = 0; } else laml[r] = sum;
                for (int k = 0; k < ND; k++) dv[k] += sgn * B[j][k] * d;
                real rr = d * Dg[j];
                if (rr * rr > res) res = rr * rr;
            }
        for (int c = 0; c < NP; c++) {
            if (!active[c]) continue;
            int r = NJ + c;
            real jd = 0;
            for (int k = 0; k < ND; k++) jd += J[r][k] * dv[k];
            real d = rhs[r] - jd * invD[r];
            real sum = lam[r] + d;
            if (sum < 0) { d = -lam[r]; lam[r] = 0; } else lam[r] = sum;
            for (int k = 0; k < ND; k++) dv[k] += B[r][k] * d;
            real rr = d * Dg[r];
            if (rr * rr > res) res = rr * rr;
        }
        for (int c = 0; c < NP; c++) {
            if (!active[c]) continue;
            int ra = NJ + NP + 2 * c, rb = ra + 1;
            real lim = P->mu * lam[NJ + c];
            real ja = 0, jb = 0;
            for (int k = 0; k < ND; k++) { ja += J[ra][k] * dv[k]; jb += J[rb][k] * dv[k]; }
            real da = rhs[ra] - ja * invD[ra], db = rhs[rb] - jb * invD[rb];
            real sa = lam[ra] + da, sb = lam[rb] + db;
            if (P->cone) { /* implicit cone: radial projection onto the disc of radius mu*lambda_n */
                real n2 = sa * sa + sb * sb;
                if (n2 > lim * lim) { real sc = lim * RSQRT(n2); sa *= sc; sb *= sc; }
            } else {
                if (sa < -lim) sa = -lim; else if (sa > lim) sa = lim;
                if (sb < -lim) sb = -lim; else if (sb > lim) sb = lim;
            }
            da = sa - lam[ra]; db = sb - lam[rb];
            lam[ra] = sa; lam[rb] = sb;
            for (int k = 0; k < ND; k++) dv[k] += B[ra][k] * da + B[rb][k] * db;
            real rr = da * Dg[ra] + db * Dg[rb];
            if (rr * rr > res) res = rr * rr;
        }
        if (res <= P->resthr || it >= P->iters - 1) break;
    }
    info->iterations = it + 1;
    info->contacts = ncontacts;
    if (P->limits) for (int r = 0; r < 2 * NJ; r++) if (laml[r] > 0) info->limit_active++;
    if (use_man) /* the impulses go back into the cache (m_appliedImpulse, m_appliedImpulseLateral1/2) */
        for (int c = 0; c < NP; c++) {
            ManPt* q = &info->man[pcyl[c]].pt[pslot[c]];
            q->imp[0] = lam[NJ + c]; q->imp[1] = lam[NJ + NP + 2 * c]; q->imp[2] = lam[NJ + NP + 2 * c + 1];
        }

    real tau[NJ];
    for (int k = 0; k < ND; k++) nu[k] += dv[k];
    for (int j = 0; j < NJ; j++) tau[j] = lam[j] / dt;
    finish_tick(T, P, s, K, nu, tau);
}

static void bt_env_step(Handle* h, int64_t* cnt, real* s, const real* action, real* obs, real* rew, uint8_t* done, int32_t* ticks_out,
                            real* trace_obs, real* trace_links) {
    const Par* P = &h->P;
    const Tables* T = &h->T;
    real a16[NJ], target[NJ];
    /* checkBound (SnakeGymEnv.py:82-88) + createAction (snake.py:247-269) */
    for (int j = 0; j < NJ; j++) a16[j] = 0;
    for (int k = 0; k < P->actdim; k++) {
        real a = action[k];
        if (a < -1) a = -1;
        if (a > 1) a = 1;
        int j = (P->gait == 0) ? 2 * k : (P->gait == 1) ? 2 * k + 1 : k;
        a16[j] = a;
    }
    for (int j = 0; j < NJ; j++) target[j] = a16[j] * P->sf; /* snake.py:223-225 */
    const real xprev = s[SNK_S_POS]; /* self._observation[48], vec-wrapper semantics (Q8) */

    Kin K;
    fk(T, s, &K);
    int counter = 0, end_height = 0;
    for (;;) { /* snake.py:284-304 */
        real e2 = 0;
        for (int j = 0; j < NJ; j++) { real d = target[j] - s[SNK_S_Q + j]; e2 += d * d; }
        if (!(SQRT(e2) > P->errthr)) break;
        TickInfo ti;
        ti.man = h->M ? h->M + ((s - h->S) / SNK_STATE_STRIDE) * NC : NULL;
        ti.limit_active = 0; ti.lam_out = NULL;
        tick_bt(T, P, s, &K, target, &ti);
        cnt[0] += 1; cnt[1] += ti.iterations;
        if (ti.man) { __sync_fetch_and_add(&h->man_points, (int64_t)ti.contacts); __sync_fetch_and_add(&h->man_ticks, (int64_t)1); }
        if (ti.limit_active) __sync_fetch_and_add(&h->limit_active, (int64_t)ti.limit_active);
        fk(T, s, &K);
        if (trace_obs) observe(s, trace_obs + (size_t)counter * SNK_OBS_DIM);            /* snake.py:291-292 */
        if (trace_links) link_positions(T, &K, trace_links + (size_t)counter * 3 * NB);   /* snake.py:293 */
        counter++;
        if (K.height > P->hthr) { end_height = 1; break; }
        if (counter >= P->maxticks) break; /* `counter > 40` */
    }
    int bad = !finite_state(s);
    real o[SNK_OBS_DIM];
    observe(s, o);
    /* calculateReward (SnakeGymEnv.py:90-97), calculateEnergy (snake.py:336-341) */
    real energy = 0;
    for (int j = 0; j < NJ; j++) energy += o[NJ + j] * o[2 * NJ + j] * P->edt;
    real r = P->alpha * (o[48] - xprev) + ((FABS(o[55]) > P->colf) ? P->colpen : 0) - P->beta * FABS(o[49] - 0) - P->gamma * energy;
    /* checkTermination (SnakeGymEnv.py:99-103) */
    int d = (FABS(o[P->tjoint]) > P->tang) || (K.height > P->hthr) || end_height;
    if (bad) { /* force-reset: restarts like a hard reset, contact caches emptied (their impulses of this step are not finite) */
        d = 1; r = P->donepen; cnt[3] += 1; for (int k = 0; k < SNK_STATE_STRIDE; k++) s[k] = 0; s[SNK_S_QUAT + 3] = 1;
        if (h->M) memset(h->M + ((s - h->S) / SNK_STATE_STRIDE) * NC, 0, NC * sizeof(Manifold));
    }
    else if (d) r += P->donepen;
    s[SNK_S_RET] += r; s[SNK_S_LEN] += 1;
    if (d) { /* in-step reset + worker reset: returned obs is the post-reset one */
        cnt[2] += 1;
        soft_reset(P, s);
        observe(s, o);
    }
    for (int k = 0; k < SNK_OBS_DIM; k++) obs[k] = o[k];
    *rew = r; *done = (uint8_t)d;
    if (ticks_out) *ticks_out = counter;
}

/* on = 1: Bullet's literal tick with warm-start factor `warm`, empty caches; on = 0: back to the handle's own tick, caches freed.
 * Refused while the exact tick's manifolds are on. */
int PFX(bt_set)(Handle* h, int on, double warm) {
    if ((on != 0 && on != 1) || !(warm >= 0) || h->P.manifold) return SNK_E_ARG;
    free(h->M); h->M = NULL;
    h->P.warm = on ? (real)warm : 0;
    if (on) { h->M = (Manifold*)calloc((size_t)h->n * NC, sizeof(Manifold)); if (!h->M) return SNK_E_NOMEM; }
    h->man_points = h->man_ticks = 0;
    return 0;
}

int PFX(bt_step_range)(Handle* h, int64_t e0, int64_t e1, const real* actions, real* obs, real* rew, uint8_t* done, int32_t* ticks) {
    if (!bt_on(h)) return PFX(step_range)(h, e0, e1, actions, obs, rew, done, ticks);
    int64_t cnt[4] = {0, 0, 0, 0};
    for (int64_t e = e0; e < e1; e++)
        bt_env_step(h, cnt, h->S + e * SNK_STATE_STRIDE, actions + e * h->P.actdim, obs + e * SNK_OBS_DIM, rew + e, done + e,
                    ticks ? ticks + e : NULL, NULL, NULL);
    for (int k = 0; k < 4; k++) __atomic_fetch_add(&h->counters[k], cnt[k], __ATOMIC_RELAXED);
    return 0;
}
int PFX(bt_step)(Handle* h, const real* actions, real* obs, real* rew, uint8_t* done, int32_t* ticks) {
    return PFX(bt_step_range)(h, 0, h->n, actions, obs, rew, done, ticks);
}

int PFX(bt_step_trace)(Handle* h, const real* actions, real* obs, real* rew, uint8_t* done, int32_t* ticks, real* tick_obs, real* tick_links) {
    if (!bt_on(h)) return PFX(step_trace)(h, actions, obs, rew, done, ticks, tick_obs, tick_links);
    int64_t cnt[4] = {0, 0, 0, 0};
    const size_t mt = (size_t)h->P.maxticks;
    for (int64_t e = 0; e < h->n; e++)
        bt_env_step(h, cnt, h->S + e * SNK_STATE_STRIDE, actions + e * h->P.actdim, obs + e * SNK_OBS_DIM, rew + e, done + e,
                    ticks ? ticks + e : NULL, tick_obs ? tick_obs + (size_t)e * mt * SNK_OBS_DIM : NULL,
                    tick_links ? tick_links + (size_t)e * mt * 3 * NB : NULL);
    for (int k = 0; k < 4; k++) __atomic_fetch_add(&h->counters[k], cnt[k], __ATOMIC_RELAXED);
    return 0;
}

int PFX(bt_tick)(Handle* h, const real* targets, int32_t n_ticks, int32_t* iters_out) {
    if (!bt_on(h)) return PFX(tick)(h, targets, n_ticks, iters_out);
    for (int64_t e = 0; e < h->n; e++) {
        real* s = h->S + e * SNK_STATE_STRIDE;
        TickInfo ti = {0, 0, NULL, 0, NULL};
        ti.man = h->M + e * NC;
        for (int t = 0; t < n_ticks; t++) {
            Kin K;
            fk(&h->T, s, &K);
            tick_bt(&h->T, &h->P, s, &K, targets + e * NJ, &ti);
            h->counters[0] += 1; h->counters[1] += ti.iterations;
            h->man_points += ti.contacts; h->man_ticks += 1;
        }
        h->limit_active += ti.limit_active;
        if (iters_out) iters_out[e] = ti.iterations;
    }
    return 0;
}
