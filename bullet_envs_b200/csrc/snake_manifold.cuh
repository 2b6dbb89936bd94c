// snake_manifold.cuh -- the env-step with Bullet's PERSISTENT CONTACT MANIFOLDS and contact warm starting (SURVEY.md 8f rank 2,
// Appendix A.5; oracle twin: tick_exact with `manifold` on, manifold_update / man_sort_cached in oracle/snake_oracle.c).
//
// What changes against the benchmarked tick (snake_exact_core.cuh, deviation D1 of DESIGN.md): per collision cylinder the contact
// is not the analytic lowest rim point but what btConvexPlaneCollisionAlgorithm + btPersistentManifold produce -- every tick the
// support vertex of the 32-gon hull (64 vertices, collision margin along -n) becomes a contact point when it is closer than the
// breaking threshold; it replaces the cached point within the threshold of it (keeping that point's impulse) or takes a free slot,
// else sortCachedPoints picks the slot (never the deepest point, largest area); every cached point is then refreshed from its
// body-frame position and dropped when its distance or its tangential drift from the anchor exceeds the threshold.  Up to 4 points
// per cylinder = up to 128 contact points per environment (a sliding snake carries ~33, a resting one up to ~62), and the normal
// impulses of the previous tick warm-start the solver (x warm_factor; Bullet: 0.1).  The caches survive soft resets (Q10).
//
// Data placement.  128 points x 20 words do not fit on chip next to 255 other environments, so this variant keeps the row table in
// GLOBAL memory: every resident thread owns a slice of a scratch array laid out [warp][point][float4 word][lane] (a warp's 32
// lanes on 512 consecutive bytes; ~100 MB are live at a time, most of it in L2), streamed through a per-thread cp.async ring in shared
// memory by the solver sweeps (below), and the per-environment caches live in HBM as 32 cylinders x 4 slots x 8 floats + 32 counts =
// 4 224 B (only the occupied slots move).  No tensor memory, so no warp-convergence requirement: a thread leaves its solver loop
// when ITS residual falls below the threshold.  One environment per thread, persistent grid; as in the benchmarked kernel the unit
// the lanes of a warp share is one physics tick, and a thread whose env-step has ended takes the next environment from a global
// counter.  Measured and profiled in DESIGN.md section 5 / profiles/README.md (1.1 M env-steps/s at 262 144 environments).
// The same loop (man_run) also runs the traced step (snk_step_trace) and the fused linear-policy rollout (snk_rollout_linear).
#pragma once
#include "snake_exact_core.cuh"

#define MAN_SLOTS 4
#define MAN_NP (MAN_SLOTS * NC)
#define MAN_SLOT_W 8                                     // lp.x lp.y lp.z dist | anchor.x anchor.y impulse_n spare
#define MAN_CYL_W (MAN_SLOTS * MAN_SLOT_W)               // 32 floats per cylinder
#define MAN_STRIDE (NC * MAN_CYL_W + NC)                 // floats per environment; the last NC words hold the point counts
static_assert(MAN_STRIDE == SNK_MAN_STRIDE, "the cache layout of include/snake_b200.h (snk_get_manifold_cache) is this one");
#define MAN_ROW_V4 5                                     // float4 words per contact point in the scratch table
#define MAN_WARP_V4 (MAN_NP * MAN_ROW_V4 * 32)           // float4 words per warp of the scratch table
#define MAN_HULL 32

__constant__ float cHullS[MAN_HULL], cHullC[MAN_HULL];   // sin / cos of 2 pi i / 32: Bullet's cylinder hull, first vertex at (0, r)

// the scratch table of one thread: word v of point k at rows[(k * MAN_ROW_V4 + v) * 32]
//   v0 = (ln, r.x, r.y, r.z)   v1 = (invD_n, rhs_n invD_n, -, -)   v2 = (d1.xyz, invD_1)   v3 = (d2.xyz, invD_2)   v4 = (la, lb, rhs_1 invD_1, rhs_2 invD_2)
//   (the normal sweep reads v0, v1, the friction sweep v0, v2, v3, v4: 32 + 64 bytes per point and sweep)
// (pass 1 parks its temporaries in v0..v2 exactly like ex_tick)
struct ManRows {
    float4* rows;
    __device__ __forceinline__ float4& at(int k, int v) const { return rows[(k * MAN_ROW_V4 + v) * 32]; }
};

// The solver sweeps stream the row table through a per-thread RING in shared memory filled by cp.async (LDGSTS, L2 -> shared memory
// without a register round trip): MAN_RING rows are in flight per thread, which hides the L2 latency that a one-row-ahead register
// prefetch cannot (the first version of this kernel spent 70 % of its time waiting for exactly these loads).  Ring word v of slot s of
// thread t: ring[(s * MAN_ROW_V4 + v) * MAN_THREADS + t] -- consecutive threads on consecutive 16 B words, conflict free.
#define MAN_THREADS 128
#ifndef MAN_MINB
#define MAN_MINB 2
#endif
#ifndef MAN_RING
#define MAN_RING 6
#endif
#define MAN_RING_BYTES (MAN_RING * MAN_ROW_V4 * MAN_THREADS * 16)
__device__ __forceinline__ void man_cp16(float4* smem_dst, const float4* gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void man_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void man_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// btPersistentManifold::sortCachedPoints: the slot a new point replaces in a full cache (oracle: man_sort_cached)
__device__ __forceinline__ int man_sort_cached(const float (&mc)[MAN_CYL_W], V3 lp, float dist) {
    int deepest = -1;
    float maxpen = dist;
#pragma unroll
    for (int i = 0; i < MAN_SLOTS; i++)
        if (mc[i * MAN_SLOT_W + 3] < maxpen) { deepest = i; maxpen = mc[i * MAN_SLOT_W + 3]; }
    float res[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int p0 = (k == 0) ? 1 : 0, p1 = (k == 3) ? 2 : 3, p2 = (k < 2) ? 2 : 1; // {1,3,2},{0,3,2},{0,3,1},{0,2,1}
        if (deepest == k) continue;
        const V3 a = lp - mk(mc[p0 * MAN_SLOT_W], mc[p0 * MAN_SLOT_W + 1], mc[p0 * MAN_SLOT_W + 2]);
        const V3 b = mk(mc[p1 * MAN_SLOT_W], mc[p1 * MAN_SLOT_W + 1], mc[p1 * MAN_SLOT_W + 2]) -
                     mk(mc[p2 * MAN_SLOT_W], mc[p2 * MAN_SLOT_W + 1], mc[p2 * MAN_SLOT_W + 2]);
        const V3 cr = cross(a, b);
        res[k] = dot(cr, cr);
    }
    int best = 0;
    float bestr = res[0];
#pragma unroll
    for (int k = 1; k < 4; k++) if (res[k] > bestr) { bestr = res[k]; best = k; }
    return best;
}

// One collision-detection pass of cylinder c (oracle: manifold_update).  R / pb: frame of the cylinder's body (pb relative to the base
// origin), p0: base origin (world).  mc: the cylinder's 4 slots, n: its point count.  Every slot index below is a compile-time constant
// (unrolled loops, selects instead of pointers), so that the 32 words stay in REGISTERS: as a dynamically indexed local array they cost
// 16 GB of local-memory traffic per launch and 33 KB of the L1 that the state records and caches need.
__device__ __forceinline__ void man_update(const ExTables& T, int c, const M3& R, V3 pb, V3 p0, float (&mc)[MAN_CYL_W], int& n) {
    const float brk = T.cbrk[c], mar = T.cmar[c], rad = T.crad[c], hl = fabsf(T.ceh[c]);
    const float* F = T.cfr[c];
    // world-z of the body-frame vector ccen + cfr (r sin t, r cos t, +-hl):  z0 + g.x r sin t + g.y r cos t +- g.z hl
    const float g0 = R.m[6] * F[0] + R.m[7] * F[3] + R.m[8] * F[6];
    const float g1 = R.m[6] * F[1] + R.m[7] * F[4] + R.m[8] * F[7];
    const float g2 = R.m[6] * F[2] + R.m[7] * F[5] + R.m[8] * F[8];
    int best = 0;
    float bestv = g1; // vertex 0: sin 0 = 0, cos 0 = 1
#pragma unroll 4
    for (int i = 1; i < MAN_HULL; i++) {
        const float v = g0 * cHullS[i] + g1 * cHullC[i];
        if (v < bestv) { bestv = v; best = i; }
    }
    const float zend = (-hl * g2 <= hl * g2) ? -hl : hl; // the rim z = -L/2 comes first in the hull (ties go to it)
    const V3 vl = mk(rad * cHullS[best], rad * cHullC[best], zend);
    const V3 vb = ld3(T.ccen[c]) + mk(F[0] * vl.x + F[1] * vl.y + F[2] * vl.z, F[3] * vl.x + F[4] * vl.y + F[5] * vl.z, F[6] * vl.x + F[7] * vl.y + F[8] * vl.z);
    const V3 rv = mul(R, vb);
    const V3 rel = mk(rv.x, rv.y, rv.z - mar); // localGetSupportingVertex adds the margin along the query direction -n
    const float dist = p0.z + pb.z + rel.z;
    if (dist < brk) {
        const V3 lp = mulT(R, rel);
        int idx = -1;
        float shortest = brk * brk;
#pragma unroll
        for (int i = 0; i < MAN_SLOTS; i++)
            if (i < n) {
                const V3 d = mk(mc[i * MAN_SLOT_W] - lp.x, mc[i * MAN_SLOT_W + 1] - lp.y, mc[i * MAN_SLOT_W + 2] - lp.z);
                const float d2 = dot(d, d);
                if (d2 < shortest) { shortest = d2; idx = i; }
            }
        float imp = 0.f;
        if (idx >= 0) { // replaceContactPoint keeps the cached impulse
#pragma unroll
            for (int i = 0; i < MAN_SLOTS; i++) if (idx == i) imp = mc[i * MAN_SLOT_W + 6];
        } else if (n < MAN_SLOTS) idx = n++;
        else idx = man_sort_cached(mc, lp, dist);
        const float ax = p0.x + pb.x + rel.x, ay = p0.y + pb.y + rel.y;
#pragma unroll
        for (int i = 0; i < MAN_SLOTS; i++)
            if (idx == i) {
                mc[i * MAN_SLOT_W] = lp.x; mc[i * MAN_SLOT_W + 1] = lp.y; mc[i * MAN_SLOT_W + 2] = lp.z; mc[i * MAN_SLOT_W + 3] = dist;
                mc[i * MAN_SLOT_W + 4] = ax; mc[i * MAN_SLOT_W + 5] = ay; mc[i * MAN_SLOT_W + 6] = imp; mc[i * MAN_SLOT_W + 7] = 0.f;
            }
    }
#pragma unroll
    for (int i = MAN_SLOTS - 1; i >= 0; i--) // refreshContactPoints
        if (i < n) {
            const V3 w = mul(R, mk(mc[i * MAN_SLOT_W], mc[i * MAN_SLOT_W + 1], mc[i * MAN_SLOT_W + 2]));
            const V3 pos = p0 + pb + w;
            mc[i * MAN_SLOT_W + 3] = pos.z;
            const float dx = mc[i * MAN_SLOT_W + 4] - pos.x, dy = mc[i * MAN_SLOT_W + 5] - pos.y;
            if (pos.z > brk || dx * dx + dy * dy > brk * brk) { // removeContactPoint: the last point takes the slot
                const int last = n - 1;
#pragma unroll
                for (int q = 0; q < MAN_SLOT_W; q++) {
                    float v = mc[i * MAN_SLOT_W + q];
#pragma unroll
                    for (int l = i + 1; l < MAN_SLOTS; l++) if (last == l) v = mc[l * MAN_SLOT_W + q];
                    mc[i * MAN_SLOT_W + q] = v;
                }
                n--;
            }
        }
}

// -----------------------------------------------------------------------------------------------
// One physics tick with persistent manifolds; the structure and every formula outside the contact generation are those of ex_tick.
// `cache` = this environment's MAN_STRIDE floats.  Returns like ex_tick; out->contacts = cached points of the tick.
// -----------------------------------------------------------------------------------------------
template <bool CONE>
__device__ void man_tick(const ExTables& T, const KParams& P, const ManRows& R, float4* __restrict__ ring, float* __restrict__ cache, float warm, ExEnv& e, const float* __restrict__ tg,
                         bool abort_on_height, bool* aborted, ExTickOut* out) {
    const float dt = P.dt, inv_dt = P.inv_dt;
    const V3 p0 = ld3(e.pos);
    // ------------------------------------------------------------------ pass 1: tip-ward (ex_tick), contacts from the manifolds
    ExCursor c;
    c.R = quat_to_m3(e.quat);
    c.p = mk(0.f, 0.f, 0.f);
    c.w = ld3(e.omg); c.v = ld3(e.vel);
    c.al = mk(0.f, 0.f, 0.f); c.acc = mk(0.f, 0.f, 0.f);
    V3 wJ = mk(0.f, 0.f, 0.f), vJ = mk(0.f, 0.f, 0.f);
    V3 h = mk(0.f, 0.f, 0.f), F0 = h, N0 = h;
    S3 J; J.xx = J.xy = J.xz = J.yy = J.yz = J.zz = 0.f;
    float hsum = 0.f, err2n = 0.f;
    // the height test comes first: an aborted tick must not touch the caches
    if (abort_on_height) {
        const float hgt = ex_height(T, e);
        if (hgt > P.hthr) { *aborted = true; out->height = hgt; out->iterations = 0; out->contacts = 0; out->err2_next = 0.f; return; }
    }
    *aborted = false;
    int np = 0;
#pragma unroll 1
    for (int i = 0; i < NB; i++) {
        if (i > 0) {
            const int j = i - 1;
            const float q = slot(e, SNK_S_Q + j), qd = slot(e, SNK_S_QD + j), tgj = tg[j];
            float qds = P.kp * (tgj - q) * inv_dt;
            qds = ex_clamp(qds, P.maxvel);
            const float qdd = (qds - qd) * inv_dt;
            const float en = tgj - (q + dt * qds);
            err2n += en * en;
            V3 d = mul(c.R, ld3(T.jt[j]));
            V3 wxd = cross(c.w, d);
            c.acc = c.acc + cross(c.al, d) + cross(c.w, wxd);
            c.v = c.v + wxd;
            vJ = vJ + cross(wJ, d);
            c.p = c.p + d;
            c.R = mul(c.R, joint_rot(T, j, q));
            V3 a = mul(c.R, ld3(T.jax[j]));
            V3 wq = a * qd;
            c.al = c.al + a * qdd + cross(c.w, wq);
            c.w = c.w + wq;
            wJ = wJ + a * qds;
        }
        {
            const float m = T.mass[i];
            V3 rc = mul(c.R, ld3(T.com[i]));
            V3 cc = c.p + rc;
            S3 Iw = world_inertia(T, i, c.R);
            V3 wxr = cross(c.w, rc);
            V3 vc = c.v + wxr;
            V3 ac = c.acc + cross(c.al, rc) + cross(c.w, wxr);
            V3 F, N;
            body_wrench(T, P, i, Iw, c.w, c.al, vc, ac, &F, &N);
            F0 = F0 + F;
            N0 = N0 + cross(cc, F) + N;
            h = h + cc * m;
            const float c2 = dot(cc, cc);
            J.xx += Iw.xx + m * (c2 - cc.x * cc.x); J.yy += Iw.yy + m * (c2 - cc.y * cc.y); J.zz += Iw.zz + m * (c2 - cc.z * cc.z);
            J.xy += Iw.xy - m * cc.x * cc.y; J.xz += Iw.xz - m * cc.x * cc.z; J.yz += Iw.yz - m * cc.y * cc.z;
            hsum += p0.z + c.p.z + c.R.m[6] * T.hpt[i][0] + c.R.m[7] * T.hpt[i][1] + c.R.m[8] * T.hpt[i][2];
        }
#pragma unroll 1
        for (int k = T.cstart[i]; k < T.cstart[i + 1]; k++) {
            float mc[MAN_CYL_W];
            float4* gc = reinterpret_cast<float4*>(cache + k * MAN_CYL_W);
            int n = (int)cache[NC * MAN_CYL_W + k];
            const int n_old = n;
            // only the occupied slots move: a sliding snake holds about one point per cylinder (32 B of the cylinder's 128 B)
#pragma unroll
            for (int q = 0; q < MAN_SLOTS; q++)
                if (q < n_old) {
                    const float4 u = gc[2 * q], v = gc[2 * q + 1];
                    mc[8 * q] = u.x; mc[8 * q + 1] = u.y; mc[8 * q + 2] = u.z; mc[8 * q + 3] = u.w;
                    mc[8 * q + 4] = v.x; mc[8 * q + 5] = v.y; mc[8 * q + 6] = v.z; mc[8 * q + 7] = v.w;
                }
            man_update(T, k, c.R, c.p, p0, mc, n);
#pragma unroll
            for (int q = 0; q < MAN_SLOTS; q++)
                if (q < n) {
                    gc[2 * q] = make_float4(mc[8 * q], mc[8 * q + 1], mc[8 * q + 2], mc[8 * q + 3]);
                    gc[2 * q + 1] = make_float4(mc[8 * q + 4], mc[8 * q + 5], mc[8 * q + 6], mc[8 * q + 7]);
                }
            if (n != n_old) cache[NC * MAN_CYL_W + k] = (float)n;
            if (n == 0) continue;
            M3 cf, Rl;
#pragma unroll
            for (int q9 = 0; q9 < 9; q9++) cf.m[q9] = T.cfr[k][q9];
            Rl = mul(c.R, cf);
            V3 l1 = mk(-Rl.m[3] * P.aniso[0], -Rl.m[4] * P.aniso[1], -Rl.m[5] * P.aniso[2]);
            V3 l2 = mk(Rl.m[0] * P.aniso[0], Rl.m[1] * P.aniso[1], Rl.m[2] * P.aniso[2]);
            V3 d1 = mul(Rl, l1), d2 = mul(Rl, l2);
#pragma unroll
            for (int s = 0; s < MAN_SLOTS; s++) {
                if (s >= n) break;
                const V3 rp = mul(c.R, mk(mc[s * MAN_SLOT_W], mc[s * MAN_SLOT_W + 1], mc[s * MAN_SLOT_W + 2])); // point relative to the body origin
                const V3 pc = c.p + rp;
                const V3 uJ = vJ + cross(wJ, rp);
                // temporaries: v0 = (uJ.x | pc), v1 = (d1 | d2.x), v2 = (d2.y d2.z | uJ.y uJ.z), v3 = (dist, warm-start impulse, -, -)
                R.at(np, 0) = make_float4(uJ.x, pc.x, pc.y, pc.z);
                R.at(np, 1) = make_float4(d1.x, d1.y, d1.z, d2.x);
                R.at(np, 2) = make_float4(d2.y, d2.z, uJ.y, uJ.z);
                R.at(np, 3) = make_float4(mc[s * MAN_SLOT_W + 3], mc[s * MAN_SLOT_W + 6] * warm, 0.f, 0.f);
                np++;
            }
        }
    }
    out->height = hsum * (1.f / NB);
    out->err2_next = err2n;

    // ------------------------------------------------------------------ free rigid motion about C (ex_tick)
    const float invM = T.inv_mtot, M = T.mtot;
    const V3 hc = h * invM;
    {
        const float h2 = dot(hc, hc);
        J.xx -= M * (h2 - hc.x * hc.x); J.yy -= M * (h2 - hc.y * hc.y); J.zz -= M * (h2 - hc.z * hc.z);
        J.xy += M * hc.x * hc.y; J.xz += M * hc.x * hc.z; J.yz += M * hc.y * hc.z;
    }
    S3 Ji;
    {
        const float c00 = J.yy * J.zz - J.yz * J.yz, c01 = J.xz * J.yz - J.xy * J.zz, c02 = J.xy * J.yz - J.xz * J.yy;
        const float det = J.xx * c00 + J.xy * c01 + J.xz * c02;
        const float id = 1.f / det;
        Ji.xx = c00 * id; Ji.xy = c01 * id; Ji.xz = c02 * id;
        Ji.yy = (J.xx * J.zz - J.xz * J.xz) * id; Ji.yz = (J.xy * J.xz - J.xx * J.yz) * id; Ji.zz = (J.xx * J.yy - J.xy * J.xy) * id;
    }
    const V3 NC0 = N0 - cross(hc, F0);
    const V3 alf = mul(Ji, NC0) * -1.f;
    const V3 aC = F0 * -invM;
    const V3 w0 = ld3(e.omg), v0 = ld3(e.vel);
    const V3 wf = w0 + alf * dt;
    const V3 VC = v0 + cross(w0, hc) + aC * dt;

    // ------------------------------------------------------------------ rows; the warm start goes into (dw, dV) on the way
    V3 dw = mk(0.f, 0.f, 0.f), dV = mk(0.f, 0.f, 0.f);
#pragma unroll 1
    for (int k = 0; k < np; k++) {
        const float4 t0 = R.at(k, 0), t1 = R.at(k, 1), t2 = R.at(k, 2), t3 = R.at(k, 3);
        const V3 uJ = mk(t0.x, t2.z, t2.w);
        const float dist = t3.x, ln0 = t3.y;
        const V3 r = mk(t0.y - hc.x, t0.z - hc.y, t0.w - hc.z);
        const V3 d1 = mk(t1.x, t1.y, t1.z), d2 = mk(t1.w, t2.x, t2.y);
        const V3 vp = VC + cross(wf, r) + uJ;
        const V3 rn = mk(r.y, -r.x, 0.f);
        const V3 Jn = mul(Ji, rn);
        const float Dn = invM + dot(rn, Jn);
        const float iDn = 1.f / Dn;
        const float pen = dist + P.slop;
        float verr = -vp.z, perr = 0.f;
        if (pen > 0.f) verr -= pen * inv_dt; else perr = -pen * P.erp2 * inv_dt;
        const float rhsn = (verr + perr) * iDn;
        const V3 r1 = cross(r, d1), r2 = cross(r, d2);
        const V3 J1 = mul(Ji, r1), J2 = mul(Ji, r2);
        const float D1 = dot(d1, d1) * invM + dot(r1, J1), D2 = dot(d2, d2) * invM + dot(r2, J2);
        const float iD1 = 1.f / D1, iD2 = 1.f / D2;
        R.at(k, 0) = make_float4(ln0, r.x, r.y, r.z);
        R.at(k, 1) = make_float4(iDn, rhsn, 0.f, 0.f);
        R.at(k, 2) = make_float4(d1.x, d1.y, d1.z, iD1);
        R.at(k, 3) = make_float4(d2.x, d2.y, d2.z, iD2);
        R.at(k, 4) = make_float4(0.f, 0.f, -dot(d1, vp) * iD1, -dot(d2, vp) * iD2);
        // warm start (A.5): the cached normal impulse x warm factor acts before the first sweep
        dw = dw + Jn * ln0;
        dV.z = fmaf(ln0, invM, dV.z);
    }

    // ------------------------------------------------------------------ projected Gauss-Seidel (row formulas of ex_tick)
    const float sthr = P.sthr, mu = P.mu;
    int sweeps = 0;
#pragma unroll 1
    for (int it = 0; it < P.iters; it++) {
        float viol = 0.f;
        // normal rows: words v0, v1 of MAN_RING - 1 rows ahead are on their way into the ring while row k is on the (dw, dV) chain
        __threadfence_block(); // the asynchronous copies below must see this thread's own stores of the previous phase (ln, la, lb)
#pragma unroll
        for (int k = 0; k < MAN_RING - 1; k++) {
            if (k < np) { man_cp16(ring + (k * MAN_ROW_V4) * MAN_THREADS, &R.at(k, 0)); man_cp16(ring + (k * MAN_ROW_V4 + 1) * MAN_THREADS, &R.at(k, 1)); }
            man_commit();
        }
        int sk = 0; // ring slot of row k; row k + MAN_RING - 1 goes into the slot row k - 1 has just left
#pragma unroll 1
        for (int k = 0; k < np; k++) {
            {
                const int kn = k + MAN_RING - 1, sn = (sk == 0) ? MAN_RING - 1 : sk - 1;
                if (kn < np) { man_cp16(ring + (sn * MAN_ROW_V4) * MAN_THREADS, &R.at(kn, 0)); man_cp16(ring + (sn * MAN_ROW_V4 + 1) * MAN_THREADS, &R.at(kn, 1)); }
                man_commit();
                man_wait<MAN_RING - 1>();
            }
            const float4 x0 = ring[(sk * MAN_ROW_V4) * MAN_THREADS], x1 = ring[(sk * MAN_ROW_V4 + 1) * MAN_THREADS];
            sk = (sk == MAN_RING - 1) ? 0 : sk + 1;
            const float ln = x0.x, rx = x0.y, ry = x0.z, idn = x1.x;
            const float p = ln + x1.y;
            float jd = fmaf(dw.x, ry, dV.z);
            jd = fmaf(-dw.y, rx, jd);
            const float sum = fmaxf(fmaf(-jd, idn, p), 0.f);
            const float dd = sum - ln;
            R.at(k, 0).x = sum;
            const float t1 = ry * dd, t2 = -rx * dd;
            dw.x = fmaf(Ji.xx, t1, fmaf(Ji.xy, t2, dw.x));
            dw.y = fmaf(Ji.xy, t1, fmaf(Ji.yy, t2, dw.y));
            dw.z = fmaf(Ji.xz, t1, fmaf(Ji.yz, t2, dw.z));
            dV.z = fmaf(dd, invM, dV.z);
            viol = fmaxf(viol, fmaf(-sthr, idn, fabsf(dd)));
        }
        man_wait<0>();
        __threadfence_block();
        // friction pairs: all five words of a row
#pragma unroll
        for (int k = 0; k < MAN_RING - 1; k++) {
            if (k < np) {
#pragma unroll
                for (int v = 0; v < MAN_ROW_V4; v++) if (v != 1) man_cp16(ring + (k * MAN_ROW_V4 + v) * MAN_THREADS, &R.at(k, v));
            }
            man_commit();
        }
        sk = 0;
#pragma unroll 1
        for (int k = 0; k < np; k++) {
            {
                const int kn = k + MAN_RING - 1, sn = (sk == 0) ? MAN_RING - 1 : sk - 1;
                if (kn < np) {
#pragma unroll
                    for (int v = 0; v < MAN_ROW_V4; v++) if (v != 1) man_cp16(ring + (sn * MAN_ROW_V4 + v) * MAN_THREADS, &R.at(kn, v));
                }
                man_commit();
                man_wait<MAN_RING - 1>();
            }
            const float4* rk = ring + (sk * MAN_ROW_V4) * MAN_THREADS;
            sk = (sk == MAN_RING - 1) ? 0 : sk + 1;
            const float4 x0 = rk[0], x2 = rk[2 * MAN_THREADS], x3 = rk[3 * MAN_THREADS], x4 = rk[4 * MAN_THREADS];
            const float rx = x0.y, ry = x0.z, rz = x0.w, la = x4.x, lb = x4.y;
            const float pa = la + x4.z, pb = lb + x4.w, lim = mu * x0.x;
            const float ux = fmaf(dw.y, rz, fmaf(-dw.z, ry, dV.x));
            const float uy = fmaf(dw.z, rx, fmaf(-dw.x, rz, dV.y));
            const float uz = fmaf(dw.x, ry, fmaf(-dw.y, rx, dV.z));
            const float g1 = fmaf(x2.x, ux, fmaf(x2.y, uy, x2.z * uz));
            const float g2 = fmaf(x3.x, ux, fmaf(x3.y, uy, x3.z * uz));
            float sa = fmaf(-g1, x2.w, pa), sb = fmaf(-g2, x3.w, pb);
            if (CONE) {
                const float sc = fminf(1.f, lim * ex_rsqrt_fast(fmaf(sa, sa, sb * sb)));
                sa *= sc; sb *= sc;
            } else {
                sa = fminf(fmaxf(sa, -lim), lim);
                sb = fminf(fmaxf(sb, -lim), lim);
            }
            const float da = sa - la, db = sb - lb;
            *reinterpret_cast<float2*>(&R.at(k, 4).x) = make_float2(sa, sb);
            const float fx = fmaf(x3.x, db, x2.x * da), fy = fmaf(x3.y, db, x2.y * da), fz = fmaf(x3.z, db, x2.z * da);
            const float tx = fmaf(-rz, fy, ry * fz), ty = fmaf(-rx, fz, rz * fx), tz = fmaf(-ry, fx, rx * fy);
            dV.x = fmaf(fx, invM, dV.x); dV.y = fmaf(fy, invM, dV.y); dV.z = fmaf(fz, invM, dV.z);
            dw.x = fmaf(Ji.xx, tx, fmaf(Ji.xy, ty, fmaf(Ji.xz, tz, dw.x)));
            dw.y = fmaf(Ji.xy, tx, fmaf(Ji.yy, ty, fmaf(Ji.yz, tz, dw.y)));
            dw.z = fmaf(Ji.xz, tx, fmaf(Ji.yz, ty, fmaf(Ji.zz, tz, dw.z)));
            viol = fmaxf(viol, fmaf(-sthr * x2.w, x3.w, fabsf(fmaf(da, x3.w, db * x2.w))));
        }
        man_wait<0>();
        sweeps++;
        if (viol <= 0.f) break;
    }
    out->iterations = sweeps;
    out->contacts = np;

    // ------------------------------------------------------------------ new base velocity (ex_tick)
    const V3 wN_u = wf + dw;
    const V3 vN_u = (VC + dV) - cross(wN_u, hc);
    const V3 al0 = (wN_u - w0) * inv_dt;
    const V3 a0 = (vN_u - v0) * inv_dt;
    const M3 R0 = quat_to_m3(e.quat);
    V3 wb = mulT(R0, wN_u), vb = mulT(R0, vN_u);
    wb = mk(ex_clamp(wb.x, P.maxvel), ex_clamp(wb.y, P.maxvel), ex_clamp(wb.z, P.maxvel));
    vb = mk(ex_clamp(vb.x, P.maxvel), ex_clamp(vb.y, P.maxvel), ex_clamp(vb.z, P.maxvel));
    const V3 wN = mul(R0, wb), vN = mul(R0, vb);

    // ------------------------------------------------------------------ pass 2: base-ward, torques; impulses back into the caches
    {
        V3 SF = mk(0.f, 0.f, 0.f), SN = SF;
        int pend = np;
#pragma unroll 1
        for (int i = NB - 1; i >= 0; i--) {
            // the points of body i are the last ones not consumed yet (cylinder-major order of pass 1)
            int cnt = 0;
#pragma unroll 1
            for (int k = T.cstart[i]; k < T.cstart[i + 1]; k++) cnt += (int)cache[NC * MAN_CYL_W + k];
            const int pbeg = pend - cnt;
            {   // write the solved normal impulses into the slots (m_appliedImpulse)
                int q = pbeg;
#pragma unroll 1
                for (int k = T.cstart[i]; k < T.cstart[i + 1]; k++) {
                    const int n = (int)cache[NC * MAN_CYL_W + k];
                    for (int s = 0; s < n; s++, q++) cache[k * MAN_CYL_W + s * MAN_SLOT_W + 6] = R.at(q, 0).x;
                }
            }
            if (i == 0) break; // body 0 has no joint above it: only its impulses had to go back
            const int j = i - 1;
            const float q = slot(e, SNK_S_Q + j), qd = slot(e, SNK_S_QD + j), tgj = tg[j];
            float qds = P.kp * (tgj - q) * inv_dt;
            qds = ex_clamp(qds, P.maxvel);
            const float qdd = (qds - qd) * inv_dt;
            V3 rc = mul(c.R, ld3(T.com[i]));
            V3 cc = c.p + rc;
            S3 Iw = world_inertia(T, i, c.R);
            V3 wxr = cross(c.w, rc);
            V3 vc = c.v + wxr;
            V3 ac = c.acc + cross(c.al, rc) + cross(c.w, wxr) + a0 + cross(al0, cc);
            V3 F, N;
            body_wrench(T, P, i, Iw, c.w, c.al + al0, vc, ac, &F, &N);
            SF = SF + F;
            SN = SN + cross(cc, F) + N;
#pragma unroll 1
            for (int k = pbeg; k < pend; k++) {
                const float4 x0 = R.at(k, 0), x2 = R.at(k, 2), x3 = R.at(k, 3), x4 = R.at(k, 4);
                V3 f = mk(fmaf(x3.x, x4.y, x2.x * x4.x), fmaf(x3.y, x4.y, x2.y * x4.x), fmaf(x3.z, x4.y, fmaf(x2.z, x4.x, x0.x))) * inv_dt;
                V3 r = mk(x0.y + hc.x, x0.z + hc.y, x0.w + hc.z);
                SF = SF - f;
                SN = SN - cross(r, f);
            }
            pend = pbeg;
            V3 a = mul(c.R, ld3(T.jax[j]));
            const float tau = dot(a, SN - cross(c.p, SF)) + T.jdamp[j] * qd;
            slot(e, SNK_S_TAU + j) = tau;
            slot(e, SNK_S_QD + j) = qds;
            slot(e, SNK_S_Q + j) = q + qds * dt;
            V3 wq = a * qd;
            c.w = c.w - wq;
            c.al = c.al - a * qdd - cross(c.w, wq);
            c.R = mulBT(c.R, joint_rot(T, j, q));
            V3 d = mul(c.R, ld3(T.jt[j]));
            V3 wxd = cross(c.w, d);
            c.p = c.p - d;
            c.v = c.v - wxd;
            c.acc = c.acc - cross(c.al, d) - cross(c.w, wxd);
        }
    }

    // ------------------------------------------------------------------ finish (ex_tick)
    {
        const float nv = sqrtf(dot(v0, v0));
        const float rm = T.rootm, kl = P.kl + P.kl * nv;
        V3 f = mk(rm * P.g[0] - rm * v0.x * kl - rm * (vN.x - v0.x) * inv_dt, rm * P.g[1] - rm * v0.y * kl - rm * (vN.y - v0.y) * inv_dt,
                  rm * P.g[2] - rm * v0.z * kl - rm * (vN.z - v0.z) * inv_dt);
        slot(e, SNK_S_FZ) = dot(mul(R0, ld3(T.fzax)), f);
    }
    e.vel[0] = vN.x; e.vel[1] = vN.y; e.vel[2] = vN.z;
    e.omg[0] = wN.x; e.omg[1] = wN.y; e.omg[2] = wN.z;
    e.pos[0] += vN.x * dt; e.pos[1] += vN.y * dt; e.pos[2] += vN.z * dt;
    {
        const float ang = sqrtf(dot(wN, wN));
        float sc, sn, cw;
        ex_sincos(0.5f * ang * dt, &sn, &cw);
        if (ang < 0.001f) sc = 0.5f * dt - dt * dt * dt * 0.020833333333f * ang * ang;
        else sc = sn / ang;
        const float ax = wN.x * sc, ay = wN.y * sc, az = wN.z * sc;
        const float* q = e.quat;
        float x = cw * q[0] + ax * q[3] + ay * q[2] - az * q[1];
        float y = cw * q[1] + ay * q[3] + az * q[0] - ax * q[2];
        float z = cw * q[2] + az * q[3] + ax * q[1] - ay * q[0];
        float w = cw * q[3] - ax * q[0] - ay * q[1] - az * q[2];
        const float in = ex_rsqrt(x * x + y * y + z * z + w * w);
        e.quat[0] = x * in; e.quat[1] = y * in; e.quat[2] = z * in; e.quat[3] = w * in;
    }
}

// -----------------------------------------------------------------------------------------------
// The persistent loop of one thread with persistent manifolds; thread = environment, persistent grid.
//   TRACE: the mode='test' info stream (snk_step_trace) -- after every tick an environment takes, its observation goes to
//          tick_obs[env][tick][56] and its link positions to tick_links[env][tick][51] (an aborted tick writes nothing); the
//          arithmetic is that of the plain step, so obs / rew / done / ticks and the caches are bit-identical to it.
//   ROLL:  A.n_steps env-steps with a linear policy per environment (snk_rollout_linear): the thread keeps its environment for the
//          whole rollout and starts the next env-step at once when one ends (policy_targets turns the observation into the next
//          targets), so no lane waits for its warp; only the return (and the optional policy-input trace) leaves the chip.
// counters: [0] ticks, [1] PGS sweeps, [2] dones, [3] non-finite resets, [4] next environment to hand out, [7] cached points.
// -----------------------------------------------------------------------------------------------
struct ManTgt { // the joint targets of the env-step in flight: the environment's 64 B row of the handle's target scratch array
    float* tg;
    __device__ __forceinline__ float& tgt(int j) const { return tg[j]; }
};

template <bool CONE, bool TRACE, bool ROLL>
__device__ __forceinline__ void man_run(const KParams& P, float* __restrict__ state, float* __restrict__ tgt_scratch, float* __restrict__ cache,
                                        float4* __restrict__ scratch, float warm, const float* __restrict__ actions, float* __restrict__ obs,
                                        float* __restrict__ rew, uint8_t* __restrict__ done, int32_t* __restrict__ ticks,
                                        unsigned long long* __restrict__ counters, int64_t n, float* __restrict__ tick_obs,
                                        float* __restrict__ tick_links, const RolloutArgs& A) {
    const int lane = threadIdx.x & 31;
    const int64_t gw = ((int64_t)blockIdx.x * MAN_THREADS + threadIdx.x) >> 5;
    ManRows R;
    R.rows = scratch + gw * MAN_WARP_V4 + lane;
    extern __shared__ __align__(16) unsigned char man_smem[];
    float4* ring = reinterpret_cast<float4*>(man_smem) + threadIdx.x;
    unsigned long long c_ticks = 0, c_iters = 0;
    unsigned c_done = 0, c_bad = 0;
    unsigned long long c_points = 0; // cached contact points summed over the ticks (counters[7]: snk_manifold_stats)
    // The unit the lanes of a warp share is ONE PHYSICS TICK, as in the benchmarked kernel: a thread whose environment has finished its
    // tick loop writes the outputs and takes the next environment (first its own index, then a global counter) while the other lanes
    // keep ticking -- a plain `for env { for tick }` nest would make every warp wait for its longest env-step at the end of the inner loop.
    const int64_t tid = (int64_t)blockIdx.x * MAN_THREADS + threadIdx.x, T0 = (int64_t)gridDim.x * MAN_THREADS;
    ExEnv e;
    e.st = state; e.tid = lane;
    ManTgt G;
    G.tg = tgt_scratch;
    float* mc = cache;
    ExRun run;
    int64_t env = -1;
    bool have = false, first = true;
    int t = 0;       // ROLL: env-step of the rollout in flight
    float ret = 0.f; // ROLL: sum of its rewards so far
#pragma unroll 1
    for (;;) {
        if (!have) {
            const int64_t cand = first ? tid : T0 + (int64_t)atomicAdd(&counters[4], 1ull);
            first = false;
            if (cand >= n) break;
            env = cand; have = true;
            e.st = state + env * SNK_STATE_STRIDE;
            G.tg = tgt_scratch + env * NJ;
            mc = cache + env * MAN_STRIDE;
            if (ROLL) {
                t = 0;
                ex_load_base(e);
                policy_targets(P, G, e, A, env, n, 0);
            } else {
                load_targets(P, G, actions + env * P.actdim);
                ex_load_base(e);
            }
            ex_step_begin(P, G, e, &run);
        }
        bool fin = !(sqrtf(run.e2) > P.errthr); // checkFeedback (snake.py:228-235); true at once: a zero-tick step (Q5)
        if (!fin) {
            bool aborted;
            ExTickOut to;
            man_tick<CONE>(cT, P, R, ring, mc, warm, e, G.tg, run.counter > 0, &aborted, &to);
            if (aborted) { run.end_height = true; run.height = to.height; run.have_height = true; fin = true; } // the previous tick lifted the snake
            else {
                run.iters += to.iterations;
                c_points += (unsigned long long)to.contacts;
                run.counter++;
                run.e2 = to.err2_next;
                fin = run.counter >= P.maxticks || !(sqrtf(run.e2) > P.errthr);
                if (TRACE) { // the tick went through: snake.py:291-293
                    const int64_t row = env * P.maxticks + (run.counter - 1);
                    if (tick_obs) {
                        float* to_ = tick_obs + row * SNK_OBS_DIM;
#pragma unroll 1
                        for (int k = 0; k < SNK_OBS_DIM; k++) to_[k] = ex_obs_of(e, k);
                    }
                    if (tick_links) ex_link_positions(cT, e, tick_links + row * (3 * NB));
                }
            }
        }
        if (fin) {
            ExStepOut o;
            ex_step_end(cT, P, e, run, &o);
            if (ROLL) {
                c_ticks += (unsigned long long)o.ticks; c_iters += (unsigned long long)o.iters; c_done += o.done; c_bad += o.bad;
                ret = (t == 0) ? o.rew : ret + o.rew;
                if (++t < A.n_steps) { // the next env-step of the same environment starts at once, from the observation just made
                    policy_targets(P, G, e, A, env, n, t);
                    ex_step_begin(P, G, e, &run);
                } else {
                    A.returns[env] = ret;
                    have = false;
                }
            } else {
                rew[env] = o.rew;
                done[env] = (uint8_t)o.done;
                if (ticks) ticks[env] = o.ticks;
                float* go = obs + env * SNK_OBS_DIM;
#pragma unroll 1
                for (int k = 0; k < SNK_OBS_DIM; k += 4)
                    *reinterpret_cast<float4*>(go + k) = make_float4(ex_obs_of(e, k), ex_obs_of(e, k + 1), ex_obs_of(e, k + 2), ex_obs_of(e, k + 3));
                c_ticks += (unsigned long long)o.ticks; c_iters += (unsigned long long)o.iters; c_done += o.done; c_bad += o.bad;
                have = false;
            }
        }
    }
    if (c_ticks) atomicAdd(&counters[0], c_ticks);
    if (c_iters) atomicAdd(&counters[1], c_iters);
    if (c_done) atomicAdd(&counters[2], (unsigned long long)c_done);
    if (c_bad) atomicAdd(&counters[3], (unsigned long long)c_bad);
    if (c_points) atomicAdd(&counters[7], c_points);
}

// kernel: one SubprocVecEnv.step() of N environments with persistent manifolds
template <bool CONE>
__global__ void __launch_bounds__(MAN_THREADS, MAN_MINB)
snk_man_step_kernel(const KParams P, float* __restrict__ state, float* __restrict__ tgt_scratch, float* __restrict__ cache, float4* __restrict__ scratch,
                    float warm, const float* __restrict__ actions, float* __restrict__ obs, float* __restrict__ rew, uint8_t* __restrict__ done,
                    int32_t* __restrict__ ticks, unsigned long long* __restrict__ counters, int64_t n) {
    man_run<CONE, false, false>(P, state, tgt_scratch, cache, scratch, warm, actions, obs, rew, done, ticks, counters, n, nullptr, nullptr, RolloutArgs());
}

// the same env-step with the mode='test' info stream (snk_step_trace); tick_obs / tick_links: [N][max_ticks][56] / [51], either may be null
template <bool CONE>
__global__ void __launch_bounds__(MAN_THREADS, MAN_MINB)
snk_man_step_trace_kernel(const KParams P, float* __restrict__ state, float* __restrict__ tgt_scratch, float* __restrict__ cache, float4* __restrict__ scratch,
                          float warm, const float* __restrict__ actions, float* __restrict__ obs, float* __restrict__ rew, uint8_t* __restrict__ done,
                          int32_t* __restrict__ ticks, unsigned long long* __restrict__ counters, int64_t n, float* __restrict__ tick_obs,
                          float* __restrict__ tick_links) {
    man_run<CONE, true, false>(P, state, tgt_scratch, cache, scratch, warm, actions, obs, rew, done, ticks, counters, n, tick_obs, tick_links, RolloutArgs());
}

// A.n_steps env-steps with a linear policy per environment (snk_rollout_linear); A.queue / A.done_steps are not used: a thread keeps its
// environment, and the threads do not wait for each other, so neither a ready queue nor a cooperative launch is needed
template <bool CONE>
__global__ void __launch_bounds__(MAN_THREADS, MAN_MINB)
snk_man_rollout_kernel(const KParams P, float* __restrict__ state, float* __restrict__ tgt_scratch, float* __restrict__ cache, float4* __restrict__ scratch,
                       float warm, const RolloutArgs A, unsigned long long* __restrict__ counters, int64_t n) {
    man_run<CONE, false, true>(P, state, tgt_scratch, cache, scratch, warm, nullptr, nullptr, nullptr, nullptr, nullptr, counters, n, nullptr, nullptr, A);
}

// the cache half of a hard reset (snk_clear_manifold): the MAN_STRIDE floats of every environment whose mask byte is non-zero (all: mask null)
__global__ void snk_man_clear_kernel(float* __restrict__ cache, const uint8_t* __restrict__ mask, int64_t n) {
    const int64_t words = n * (MAN_STRIDE / 4), stride = (int64_t)gridDim.x * blockDim.x;
#pragma unroll 1
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < words; i += stride)
        if (!mask || mask[i / (MAN_STRIDE / 4)]) reinterpret_cast<float4*>(cache)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
}

// input check of snk_set_manifold_cache: *bad += environments of `cache` whose NC count words are not all integers in 0..MAN_SLOTS (a larger
// count would make pass 1 write more than MAN_NP rows into the next warp's slice of the row table, and pass 2 impulses beyond the slots)
__global__ void snk_man_check_kernel(const float* __restrict__ cache, int64_t n, unsigned long long* __restrict__ bad) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    unsigned cnt = 0;
#pragma unroll 1
    for (int64_t env = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; env < n; env += stride) {
        const float* c = cache + env * MAN_STRIDE + NC * MAN_CYL_W;
        bool ok = true;
#pragma unroll 1
        for (int k = 0; k < NC; k++) { const float v = c[k]; ok &= v >= 0.f && v <= (float)MAN_SLOTS && v == truncf(v); } // NaN fails
        cnt += ok ? 0u : 1u;
    }
    if (cnt) atomicAdd(bad, (unsigned long long)cnt);
}
