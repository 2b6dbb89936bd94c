// snake_exact.cu -- fused SnakeGymEnv.step() for N environments, one environment per THREAD (sm_100a).
//
// This is the kernel the reference configuration runs on (motor force = inf, kd = 1, so the motor
// rows are equalities and only the 6 rigid degrees of freedom of the chain are unknown; see
// snake_exact_core.cuh for the algorithm and oracle/snake_oracle.c:tick_exact for its CPU twin).
//
// One launch = one SubprocVecEnv.step(): clip + createAction, the data-dependent 0..41-tick loop,
// observation, reward, termination, auto-reset.  The grid is persistent, one CTA of EIGHT warps per SM, each lane
// owning one environment at a time (256 environments in flight per SM, two warps on every scheduler).  The
// per-environment working set is the contact-row table (32 contacts x 17 words, re-read by every solver sweep), and what
// bounds the kernel is how many of those tables fit on chip.  snk_hyb_step_kernel spreads every table over the three
// on-chip memories of a Blackwell SM (RowsH in snake_exact_core.cuh):
//   8 words per contact in TENSOR MEMORY (tcgen05.ld/st 32x32b: TMEM lane = thread; warps w and w + 4 share lane quadrant
//                       w and take 256 of its 512 columns each),
//   7 words per contact in shared memory ([contact][lane] columns, conflict free, 28 KB per warp = 224 KB per CTA),
//   2 words per contact in registers (64 of the thread's 255; the normal sweep that reads them is fully unrolled).
// The lock-step unit of a warp is ONE PHYSICS TICK, not one env-step: a lane whose environment has
// finished its tick loop writes its outputs and takes the next environment from a global counter while
// the other lanes keep ticking, so the 0..41 spread of tick counts costs no idle lanes.
//
// Other data: base state and loop progress in registers, joint state in the environment's 256 B record
// of the handle's [N][64] state array and the joint targets in its 64 B row of the handle's target scratch
// array (both L1/L2 resident while the lane owns the environment), model tables in constant memory at
// warp-uniform addresses.
//
// Reference call sites replaced: SnakeGymEnv.py:33-50,82-103; snake.py:209-306,336-341;
// ppo/multiprocessing_env.py:11-16; snake_gait_test.py:96-104 (raw ticks).
#include <cuda_runtime.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>

#include "snake_exact_core.cuh"

__constant__ ExTables cT;

#define FULL 0xffffffffu

// joint targets of one environment: checkBound (SnakeGymEnv.py:82-88) + createAction (snake.py:247-269)
// + scaling (snake.py:223-225)
template <class Rows>
__device__ __forceinline__ void load_targets(const KParams& P, const Rows& R, const float* __restrict__ act) {
#pragma unroll
    for (int j = 0; j < NJ; j++) R.tgt(j) = 0.f;
#pragma unroll 1
    for (int k4 = 0; k4 < P.actdim; k4 += 4) { // act_dim is 8 or 16: the row is read as 16 B vectors (it may live in mapped host memory)
        const float4 v = *reinterpret_cast<const float4*>(act + k4);
        const float av[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int k = k4 + q;
            float a = av[q];
            a = (a < -1.f) ? -1.f : a; // checkBound's comparisons: a NaN passes through (SnakeGymEnv.py:84-87)
            a = (a > 1.f) ? 1.f : a;
            const int j = (P.gait == 0) ? 2 * k : (P.gait == 1) ? 2 * k + 1 : k;
            R.tgt(j) = a * P.sf;
        }
    }
}

// SPLIT HAND-OUT of one CTA (HandOut::split_total, set up by snk_hyb_step_kernel; n_a = 0: off).  With n = k L + r environments on L
// lanes, whole env-steps leave r lanes with k + 1 of them and the others with k: the launch ends on a last wave that
// only r lanes take part in.  Instead the r SHORTEST env-steps are cut in two at a tick boundary: r lanes (n_a of
// them in this CTA, the same in every warp) START with the first part of one, park it -- the state record is in global memory
// anyway, the seven words of ExRun go to `run_words` -- and carry on with whole env-steps; when the whole env-steps have run out,
// the lanes of the same CTA that become free finish the parked ones.  Every lane then carries k env-steps and about r / L of one
// (r <= L / 2: one part each for 2 r lanes; r > L / 2: the L - r other lanes finish several short second parts each).
// Parking and resuming never cross a CTA, so the protocol needs no co-residency of CTAs; a lane never blocks its warp on a flag
// (it retries once per tick), and the arithmetic of a tick does not depend on which lane runs it: results are bit-identical.
struct SplitCta {
    int n_a;                // entries (= a-part lanes) of this CTA
    int a_idx;              // this thread's entry within the CTA, or -1
    int64_t first;          // global index of the CTA's first entry; entry i sits at position pos0 + i of the hand-out order
    int64_t pos0;           // n - split_total: the whole env-steps are the positions [0, pos0)
    int frac_q8;            // an a-part ends after max(1, predicted ticks * frac_q8 / 256) ticks
    const uint8_t* bucket;  // predicted tick counts (snk_exact_predict_kernel)
    int* bnext;             // the CTA's claim counter for parked env-steps (zeroed per launch)
    int* flags;             // per entry (zeroed per launch): 1 parked, 2 finished inside its a-part
    float* run_words;       // per entry 8 words
};

// Reward, done and ticks of an environment are 4 + 1 + 4 bytes in three arrays, written when the environment finishes -- in the
// longest-first order, i.e. scattered over the arrays in time.  With ordinary stores the 32-byte sector around such a word has
// left the L2 (500 MB of records and observation rows stream through it per launch) long before its neighbours arrive, and every
// word becomes a read-modify-write of a sector in DRAM (about 190 of the 998 B/env ncu measured).  The three arrays together are
// 9 MB at 2^20 environments: their stores carry an L2 evict-last policy, so the sectors stay in the 126 MB L2 until they are full.
__device__ __forceinline__ uint64_t l2_keep_policy() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void st_keep_f32(float* a, float v, uint64_t pol) { asm volatile("st.global.L2::cache_hint.f32 [%0], %1, %2;" ::"l"(a), "f"(v), "l"(pol) : "memory"); }
__device__ __forceinline__ void st_keep_s32(int32_t* a, int32_t v, uint64_t pol) { asm volatile("st.global.L2::cache_hint.s32 [%0], %1, %2;" ::"l"(a), "r"(v), "l"(pol) : "memory"); }
__device__ __forceinline__ void st_keep_u8(uint8_t* a, int v, uint64_t pol) { asm volatile("st.global.L2::cache_hint.u8 [%0], %1, %2;" ::"l"(a), "r"(v), "l"(pol) : "memory"); }

// The persistent loop of one warp.  counters: [0] ticks, [1] PGS sweeps, [2] dones, [3] non-finite resets,
// [4] next environment to hand out.
// TRACE: the mode='test' info stream (snake.py:275-278,292-293): after every physics tick the observation goes to
// tick_obs[env][tick][56] and the link positions to tick_links[env][tick][51] (max_ticks rows per environment).
template <bool CONE, class Rows, bool TRACE = false, bool SPLIT = false>
__device__ __forceinline__ void run_warp(const KParams& P, Rows R, float* __restrict__ state, float* __restrict__ tgt_scratch, const float* __restrict__ actions,
                                         float* __restrict__ obs, float* __restrict__ rew, uint8_t* __restrict__ done, int32_t* __restrict__ ticks,
                                         unsigned long long* __restrict__ counters, const int32_t* __restrict__ order, int64_t n,
                                         int64_t first_base, int64_t dyn_base, float* __restrict__ tick_obs = nullptr,
                                         float* __restrict__ tick_links = nullptr, int pool = 0, int64_t n_long = -1, int64_t dyn_base_short = 0,
                                         bool flag_rows = false, const SplitCta* split = nullptr) {
    // Hand-out positions: the warp's first 32 are static, [first_base, first_base + 32), laid out warp-major over the
    // grid by the caller so that a batch smaller than the grid's lanes spreads over all SMs (one warp per scheduler
    // before a second one anywhere); every later position comes from a global counter, which starts at dyn_base.
    // TWO POOLS (HandOut below): positions [0, n_long) are the long pool, [n_long, n) the short pool; a warp draws from its own pool
    // (counter [4] / [6]) and moves over to the other one when its own is exhausted.  n_long < 0: one pool.
    const bool split_on = SPLIT && split && split->n_a > 0; // SPLIT = false: everything below that concerns the split hand-out folds away
    const bool one_pool = n_long < 0 || split_on;
    if (n_long < 0) n_long = n;
    if (split_on) n_long = split->pos0; // one pool: the whole env-steps
    int64_t a_start = (split_on && split->a_idx >= 0) ? split->pos0 + split->first + split->a_idx : -1; // first of all: the lane's a-part
    int a_entry = -1, susp_at = 0; // a-part in progress: its entry, and the tick count at which it parks
    int claim = -1;                // parked env-step this lane has claimed and waits for
    bool b_done = !split_on;       // nothing (more) to claim
    const int lane = R.lane;
    const unsigned lt_mask = (1u << lane) - 1u;
    ExEnv e; // a lane without an environment computes (masked) on record 0 in the rest pose
    e.st = state;
    e.tid = lane;
#pragma unroll
    for (int k = 0; k < 3; k++) { e.pos[k] = 0.f; e.vel[k] = 0.f; e.omg[k] = 0.f; e.quat[k] = 0.f; }
    e.quat[3] = 1.f;
    R.tg = tgt_scratch + n * NJ; // ... and on the spare (all-zero) target row behind the last environment
    ExRun run;
    run.xprev = 0.f; run.e2 = 0.f; run.height = 0.f; run.counter = 0; run.iters = 0; run.end_height = false; run.have_height = false;
    int64_t env = -1;
    bool have = false;
    unsigned long long c_ticks = 0, c_iters = 0;
    unsigned c_done = 0, c_bad = 0;
    bool first = first_base >= 0; // a negative first_base: no static wave
#pragma unroll 1
    for (;;) {
        // ---- lanes without an environment take the next ones (first: the static positions, then the global counter)
        unsigned need = __ballot_sync(FULL, !have && a_start < 0 && claim < 0);
        unsigned fixed = __ballot_sync(FULL, a_start >= 0); // lanes that start on their a-part draw nothing from the counters
#pragma unroll 1
        for (int attempt = 0; attempt < 2 && (need | fixed); attempt++) { // second attempt: the other pool, once the warp's own is exhausted
            unsigned long long base = (unsigned long long)first_base;
            if (!first && need) {
                if (lane == 0) base = (unsigned long long)(pool ? dyn_base_short : dyn_base) + atomicAdd(&counters[pool ? 6 : 4], (unsigned long long)__popc(need));
                base = __shfl_sync(FULL, base, 0);
            }
            first = false;
            if (!have && claim < 0) {
                const bool apart = a_start >= 0;
                const int64_t cand = apart ? a_start : (int64_t)base + __popc(need & lt_mask);
                if (apart || cand < (pool ? n : n_long)) {
                    env = order ? (int64_t)order[cand] : cand; have = true; // longest-first order when the batch exceeds the lanes
                    e.st = state + env * SNK_STATE_STRIDE;
                    R.tg = tgt_scratch + env * NJ;
                    load_targets(P, R, actions + env * P.actdim);
                    ex_load_base(e);
                    ex_step_begin(P, R, e, &run);
                    if (apart) {
                        a_entry = (int)(split->first + split->a_idx);
                        susp_at = max(1, ((int)split->bucket[env] * split->frac_q8) >> 8);
                        a_start = -1;
                    }
                }
            }
            need = __ballot_sync(FULL, !have && claim < 0);
            fixed = 0u;
            if (one_pool) break;
            if (need) pool ^= 1;           // positions beyond the pool's end were drawn: it is empty, go on with the other one
        }
        if (split_on) { // the whole env-steps have run out for this lane: finish a parked one of the CTA
            if (!have && claim < 0 && !b_done) {
                const int j = atomicAdd(split->bnext, 1);
                if (j < split->n_a) claim = (int)split->first + j; else b_done = true;
            }
            if (claim >= 0) {
                const int f = *reinterpret_cast<volatile int*>(split->flags + claim);
                if (f == 1) { // parked: its record, target row and run words were written before the flag
                    __threadfence_block();
                    env = (int64_t)order[split->pos0 + claim]; have = true;
                    e.st = state + env * SNK_STATE_STRIDE;
                    R.tg = tgt_scratch + env * NJ;
                    ex_load_base(e);
                    const volatile float* rw = split->run_words + (int64_t)claim * 8;
                    run.xprev = rw[0]; run.e2 = rw[1]; run.height = rw[2];
                    run.counter = __float_as_int(rw[3]); run.iters = __float_as_int(rw[4]);
                    const int bits = __float_as_int(rw[5]);
                    run.end_height = (bits & 1) != 0; run.have_height = (bits & 2) != 0;
                    claim = -1;
                } else if (f == 2) claim = -1; // it ended inside its a-part: claim another one in the next round
            }
            if (!__any_sync(FULL, have || claim >= 0 || !b_done)) break;
        } else if (!__any_sync(FULL, have)) break;
        __syncwarp();
        const int tick0 = run.counter;
        const bool finished = ex_step_advance<CONE>(cT, P, R, e, have, &run); // every lane of the warp ticks together
        if (TRACE && have && run.counter > tick0) { // this lane's environment took a tick: snake.py:291-293
            const int64_t row = env * P.maxticks + tick0;
            if (tick_obs) {
                float* to = tick_obs + row * SNK_OBS_DIM;
#pragma unroll 1
                for (int k = 0; k < SNK_OBS_DIM; k++) to[k] = ex_obs_of(e, k);
            }
            if (tick_links) ex_link_positions(cT, e, tick_links + row * (3 * NB));
        }
        if (finished) {
            ExStepOut o;
            ex_step_end(cT, P, e, run, &o);
            const uint64_t keep = l2_keep_policy();
            st_keep_f32(rew + env, o.rew, keep);
            st_keep_u8(done + env, o.done, keep);
            float* go = obs + env * SNK_OBS_DIM; // 224 B row, 16 B aligned: 14 full-sector vector stores
#pragma unroll 1
            for (int k = 0; k < SNK_OBS_DIM; k += 4)
                *reinterpret_cast<float4*>(go + k) = make_float4(ex_obs_of(e, k), ex_obs_of(e, k + 1), ex_obs_of(e, k + 2), ex_obs_of(e, k + 3));
            // flag_rows (snk_step_host_f64): ticks[env] doubles as the environment's "row ready" flag for host threads that convert
            // the results while the launch is still running -- it goes out last, behind a system-wide fence
            if (flag_rows) __threadfence_system();
            if (ticks) st_keep_s32(ticks + env, o.ticks, keep);
            c_ticks += (unsigned long long)o.ticks; c_iters += (unsigned long long)o.iters; c_done += o.done; c_bad += o.bad;
            have = false;
            if (a_entry >= 0) { *reinterpret_cast<volatile int*>(split->flags + a_entry) = 2; a_entry = -1; } // nothing left to park
        }
        if (have && a_entry >= 0 && run.counter >= susp_at) { // end of the a-part: park the env-step for another lane of the CTA
            ex_store_base(e);
            volatile float* rw = split->run_words + (int64_t)a_entry * 8;
            rw[0] = run.xprev; rw[1] = run.e2; rw[2] = run.height;
            rw[3] = __int_as_float(run.counter); rw[4] = __int_as_float(run.iters);
            rw[5] = __int_as_float((run.end_height ? 1 : 0) | (run.have_height ? 2 : 0));
            __threadfence_block();
            *reinterpret_cast<volatile int*>(split->flags + a_entry) = 1;
            have = false; a_entry = -1;
        }
        __syncwarp();
    }
    // one atomic per warp and counter
#pragma unroll
    for (int sft = 16; sft > 0; sft >>= 1) {
        c_ticks += __shfl_xor_sync(FULL, c_ticks, sft); c_iters += __shfl_xor_sync(FULL, c_iters, sft);
        c_done += __shfl_xor_sync(FULL, c_done, sft); c_bad += __shfl_xor_sync(FULL, c_bad, sft);
    }
    if (lane == 0) {
        atomicAdd(&counters[0], c_ticks);
        atomicAdd(&counters[1], c_iters);
        if (c_done) atomicAdd(&counters[2], (unsigned long long)c_done);
        if (c_bad) atomicAdd(&counters[3], (unsigned long long)c_bad);
    }
}

// ---------------------------------------------------------------------------------------------
// n_steps env-steps per launch with a linear policy per environment (snk_rollout_linear; ARS rollouts,
// ars/train.py:74-116).  A lane keeps its environment for the whole rollout: after every env-step it turns
// the observation it would have returned into the next action, a = W_env ((obs + noise - mean) * inv_std),
// so nothing but the return (and the optional observation trace) leaves the chip between steps.
// ---------------------------------------------------------------------------------------------
struct RolloutArgs {
    const float* weights;  // [N, act_dim, 56]
    const float* mean;     // [56] or null
    const float* inv_std;  // [56] or null
    const float* noise;    // [n_steps, N, 56] or null
    float* returns;        // [N]
    float* trace;          // [n_steps, N, 56] or null
    int n_steps;
    int32_t* queue;        // [N * (n_steps - 1)] ready queue, -1 = not pushed yet (handle owned)
    int32_t* done_steps;   // [N] env-steps finished so far in this rollout (handle owned, zeroed per call)
};

template <class Rows>
__device__ __forceinline__ void policy_targets(const KParams& P, const Rows& R, const ExEnv& e, const RolloutArgs& A, int64_t env, int64_t n, int t) {
    float x[SNK_OBS_DIM];
    const int64_t row = ((int64_t)t * n + env) * SNK_OBS_DIM;
#pragma unroll
    for (int k = 0; k < SNK_OBS_DIM; k++) {
        float v = ex_obs_of(e, k);
        if (A.noise) v += A.noise[row + k];
        if (A.trace) A.trace[row + k] = v;
        x[k] = (v - (A.mean ? A.mean[k] : 0.f)) * (A.inv_std ? A.inv_std[k] : 1.f);
    }
#pragma unroll
    for (int j = 0; j < NJ; j++) R.tgt(j) = 0.f;
#pragma unroll 1
    for (int k = 0; k < P.actdim; k++) {
        const float4* w = reinterpret_cast<const float4*>(A.weights + (env * P.actdim + k) * SNK_OBS_DIM); // 224 B rows: 16 B aligned
        float acc = 0.f;
#pragma unroll
        for (int q = 0; q < SNK_OBS_DIM / 4; q++) { // same summation order as the oracle (sequential over the 56 inputs)
            const float4 wq = w[q];
            acc = fmaf(wq.x, x[4 * q], acc); acc = fmaf(wq.y, x[4 * q + 1], acc); acc = fmaf(wq.z, x[4 * q + 2], acc); acc = fmaf(wq.w, x[4 * q + 3], acc);
        }
        float a = acc;
        a = (a < -1.f) ? -1.f : a; // checkBound's comparisons (SnakeGymEnv.py:84-87)
        a = (a > 1.f) ? 1.f : a;
        const int j = (P.gait == 0) ? 2 * k : (P.gait == 1) ? 2 * k + 1 : k;
        R.tgt(j) = a * P.sf;
    }
}

// Work distribution of the rollout.  The unit handed to a lane is ONE env-step of one environment; an
// environment whose step has finished (and that has steps left) is pushed onto a ready queue in global memory
// and taken by whichever lane frees up next, so the lanes stay busy for any ratio of environments to lanes
// (a lane that kept its environment for the whole rollout would leave the last partial wave of rollouts on a
// mostly idle GPU).  Tickets: ticket k < N is environment k's first step; ticket k >= N is the (k - N)-th push.
// A lane holding a ticket whose queue slot is still empty polls it once per loop iteration -- it never blocks
// the warp.  Ordering: the pushing lane fences its state-record stores before the push; the popping lane
// fences (which also invalidates its SM's L1) after seeing the entry and before loading the record.
// counters: [4] tickets handed out, [5] pushes done.
template <bool CONE, class Rows>
__device__ __forceinline__ void run_rollout_warp(const KParams& P, Rows R, float* __restrict__ state, float* __restrict__ tgt_scratch, const RolloutArgs A,
                                                 unsigned long long* __restrict__ counters, int64_t n, int64_t first_base, int64_t dyn_base) {
    const int lane = R.lane;
    const unsigned lt_mask = (1u << lane) - 1u;
    const bool sticky = n <= (int64_t)gridDim.x * (int64_t)blockDim.x; // as many lanes as environments: no ready queue needed
    const long long total = sticky ? (long long)n : (long long)n * A.n_steps; // tickets that will ever be served
    ExEnv e;
    e.st = state;
    e.tid = lane;
#pragma unroll
    for (int k = 0; k < 3; k++) { e.pos[k] = 0.f; e.vel[k] = 0.f; e.omg[k] = 0.f; e.quat[k] = 0.f; }
    e.quat[3] = 1.f;
    R.tg = tgt_scratch + n * NJ;
    ExRun run;
    run.xprev = 0.f; run.e2 = 0.f; run.height = 0.f; run.counter = 0; run.iters = 0; run.end_height = false; run.have_height = false;
    int64_t env = -1;
    long long ticket = -1;    // >= 0: waiting for that ticket's environment
    bool have = false, exhausted = false, first = true;
    int t = 0;
    unsigned long long c_ticks = 0, c_iters = 0;
    unsigned c_done = 0, c_bad = 0;
#pragma unroll 1
    for (;;) {
        // ---- idle lanes draw tickets
        const unsigned need = __ballot_sync(FULL, !have && ticket < 0 && !exhausted);
        if (first) { // static first tickets, warp-major over the grid (see run_warp); the counter starts at dyn_base <= n
            first = false;
            const long long k = (long long)first_base + lane;
            if (k < n) ticket = k;
        } else if (need) {
            unsigned long long base = 0;
            if (lane == 0) base = (unsigned long long)dyn_base + atomicAdd(&counters[4], (unsigned long long)__popc(need));
            base = __shfl_sync(FULL, base, 0);
            if (!have && ticket < 0 && !exhausted) {
                const long long k = (long long)base + __popc(need & lt_mask);
                if (k < total) ticket = k; else exhausted = true;
            }
        }
        // ---- lanes with a ticket look whether its environment is ready
        if (ticket >= 0) {
            long long cand = -1;
            if (ticket < n) cand = ticket;
            else cand = *reinterpret_cast<volatile int32_t*>(A.queue + (ticket - n));
            if (cand >= 0) {
                __threadfence(); // acquire: the previous owner's stores to the record, returns[] and done_steps[]
                env = cand; have = true; ticket = -1;
                e.st = state + env * SNK_STATE_STRIDE;
                R.tg = tgt_scratch + env * NJ;
                t = A.done_steps[env];
                ex_load_base(e);
                policy_targets(P, R, e, A, env, n, t);
                ex_step_begin(P, R, e, &run);
            }
        }
        if (!__any_sync(FULL, have)) {
            if (__all_sync(FULL, exhausted && ticket < 0)) break;
            __nanosleep(500); // every lane of this warp waits for a push
            continue;
        }
        __syncwarp();
        if (ex_step_advance<CONE>(cT, P, R, e, have, &run)) {
            ExStepOut o;
            ex_step_end(cT, P, e, run, &o);
            A.returns[env] = (t == 0) ? o.rew : A.returns[env] + o.rew;
            c_ticks += (unsigned long long)o.ticks; c_iters += (unsigned long long)o.iters; c_done += o.done; c_bad += o.bad;
            A.done_steps[env] = t + 1;
            if (t + 1 < A.n_steps && sticky) {
                // every environment has a lane of its own (n <= lanes of the grid): the lane keeps it for the whole rollout -- no
                // hand-over latency, and its state record and weight rows stay in this SM's caches
                t = t + 1;
                policy_targets(P, R, e, A, env, n, t);
                ex_step_begin(P, R, e, &run);
            } else {
                if (t + 1 < A.n_steps) {
                    __threadfence(); // release the record before the environment becomes visible to other lanes
                    const unsigned long long p = atomicAdd(&counters[5], 1ull);
                    *reinterpret_cast<volatile int32_t*>(A.queue + p) = (int32_t)env;
                }
                have = false;
            }
        }
        __syncwarp();
    }
#pragma unroll
    for (int sft = 16; sft > 0; sft >>= 1) {
        c_ticks += __shfl_xor_sync(FULL, c_ticks, sft); c_iters += __shfl_xor_sync(FULL, c_iters, sft);
        c_done += __shfl_xor_sync(FULL, c_done, sft); c_bad += __shfl_xor_sync(FULL, c_bad, sft);
    }
    if (lane == 0) {
        atomicAdd(&counters[0], c_ticks);
        atomicAdd(&counters[1], c_iters);
        if (c_done) atomicAdd(&counters[2], (unsigned long long)c_done);
        if (c_bad) atomicAdd(&counters[3], (unsigned long long)c_bad);
    }
}

// ---------------------------------------------------------------------------------------------
// The benchmarked kernel: 8 warps per CTA, one CTA per SM, every warp's rows spread over tensor memory, shared memory
// and registers (RowsH).  Warps w and w + 4 run on scheduler w and share TMEM lane quadrant w.
// ---------------------------------------------------------------------------------------------
#define HWARPS 8
struct StepSmemH {
    RowsHybStore w[HWARPS];
    uint32_t tmem_base;
};

__device__ __forceinline__ uint32_t hyb_tmem_alloc(StepSmemH& S, int warp) {
    if (warp == 0) { // the whole tensor memory of the SM: 512 columns x 128 lanes
        const uint32_t dst = (uint32_t)__cvta_generic_to_shared(&S.tmem_base);
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;");
    return S.tmem_base;
}
__device__ __forceinline__ void hyb_tmem_free(uint32_t tbase, int warp) {
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tbase), "r"(512));
}
__device__ __forceinline__ RowsH hyb_rows(StepSmemH& S, uint32_t tbase, int warp, int lane) {
    RowsH R;
    R.taddr = tbase + ((uint32_t)(32 * (warp & 3)) << 16) + 256u * (uint32_t)(warp >> 2);
    R.s = &S.w[warp];
    R.lane = lane;
    R.tg = nullptr;
    return R;
}

struct HandOut {       // two-pool hand-out of a launch (see snk_hyb_step_kernel); short_warps = 0: one pool, plain longest-first
    int64_t n_long;    // positions [0, n_long) of the longest-first order are the long pool, [n_long, n) the short pool
    int short_warps;   // warps (in warp-major order over the grid) that draw from the short pool
    int flag_rows;     // != 0: ticks[env] is written last, behind a system fence (the host reads finished rows during the launch)
    // split hand-out (SplitCta): the split_total shortest env-steps are run in two parts by two lanes of a CTA; 0 = off
    int split_total, split_frac_q8;
    const uint8_t* bucket;
    int* split_buf;    // [SPLIT_CTAS] claim counters, [SPLIT_MAX] flags, [SPLIT_MAX][8] run words (handle owned; counters and flags zeroed per launch)
};
#define SPLIT_CTAS 256
#define SPLIT_MAX (SPLIT_CTAS * HWARPS * 32)

// TRACE = true: the same kernel with the mode='test' info stream (snk_step_trace) -- a separate instantiation, so the
// benchmarked one carries no trace code, and the traced step returns bit for bit what the plain step returns.
template <bool CONE, bool TRACE, bool SPLIT = false>
__global__ void __launch_bounds__(HWARPS * 32, 1)
snk_hyb_step_kernel(const KParams P, float* __restrict__ state, float* __restrict__ tgt_scratch, const float* __restrict__ actions, float* __restrict__ obs,
                    float* __restrict__ rew, uint8_t* __restrict__ done, int32_t* __restrict__ ticks, unsigned long long* __restrict__ counters,
                    const int32_t* __restrict__ order, int64_t n, int active_warps, int spread, const HandOut H, float* __restrict__ tick_obs,
                    float* __restrict__ tick_links) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    StepSmemH& S = *reinterpret_cast<StepSmemH*>(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t tbase = hyb_tmem_alloc(S, warp);
    // first wave (SNK_EXACT_SPREAD): warp-major over the grid (default) -- a batch smaller than the grid's lanes puts one warp on every
    // scheduler of every SM before any scheduler gets a second one (warps w and w + 4 share scheduler w); 0 = CTA-major; 2 = no static
    // wave, everything from the global counter (ablations)
    int64_t first_base = (spread == 2) ? -1 : (spread ? ((int64_t)warp * gridDim.x + blockIdx.x) * 32 : ((int64_t)blockIdx.x * active_warps + warp) * 32);
    int64_t dyn_base = (spread == 2) ? 0 : min((int64_t)gridDim.x * active_warps * 32, n);
    // Balanced hand-out (HandOut, computed by the launcher): with n = k L + r environments on L lanes, r lanes run k + 1 env-steps and
    // the others k.  The `short` warps -- the first ones in warp-major order, i.e. one per scheduler on every SM before a second one
    // anywhere -- run the k + 1 and draw them from the SHORTEST (k + 1) r environments of the longest-first order, the other warps draw
    // their k from the longest ones: every lane then carries about the same number of ticks, and the launch ends with the short warps
    // alone on their schedulers instead of with every warp half empty.
    int pool = 0;
    int64_t dyn_short = 0;
    if (H.short_warps > 0) {
        const int64_t gw = (int64_t)warp * gridDim.x + blockIdx.x;
        const int64_t long_warps = (int64_t)gridDim.x * active_warps - H.short_warps;
        if (gw < H.short_warps) { pool = 1; first_base = H.n_long + gw * 32; }
        else first_base = (gw - H.short_warps) * 32;
        dyn_base = min(long_warps * 32, H.n_long);
        dyn_short = H.n_long + min((int64_t)H.short_warps * 32, n - H.n_long);
        if (first_base >= (pool ? n : H.n_long)) first_base = n; // nothing static for this warp: it starts with the counters
    }
    SplitCta sp;
    sp.n_a = 0;
    if (SPLIT && H.split_total > 0) { // entries are dealt out CTA by CTA, inside a CTA warp by warp (every warp gets the same number of a-part lanes)
        const int q = H.split_total / (int)gridDim.x, rm = H.split_total % (int)gridDim.x;
        sp.n_a = q + ((int)blockIdx.x < rm ? 1 : 0);
        sp.first = (int64_t)blockIdx.x * q + min((int)blockIdx.x, rm);
        sp.pos0 = n - H.split_total;
        sp.a_idx = (lane * HWARPS + warp < sp.n_a) ? lane * HWARPS + warp : -1;
        sp.frac_q8 = H.split_frac_q8;
        sp.bucket = H.bucket;
        sp.bnext = H.split_buf + blockIdx.x;
        sp.flags = H.split_buf + SPLIT_CTAS;
        sp.run_words = reinterpret_cast<float*>(H.split_buf + SPLIT_CTAS + SPLIT_MAX);
        first_base = -1; dyn_base = 0; // no static wave: the lanes without an a-part draw their first env-step from the counter
    }
    if (warp < active_warps) // SNK_EXACT_WARPS (ablation): the other warps take no environments
        run_warp<CONE, RowsH, TRACE, SPLIT>(P, hyb_rows(S, tbase, warp, lane), state, tgt_scratch, actions, obs, rew, done, ticks, counters, order, n, first_base,
                                            dyn_base, tick_obs, tick_links, pool, H.short_warps > 0 ? H.n_long : -1, dyn_short, H.flag_rows != 0, &sp);
    hyb_tmem_free(tbase, warp);
}

// n_ticks raw ticks with explicit targets[N,16] (snk_tick; gait script): every environment runs the same number of ticks, so the
// assignment is static (thread = environment), 256 environments per CTA
template <bool CONE>
__global__ void __launch_bounds__(HWARPS * 32, 1)
snk_hyb_tick_kernel(const KParams P, float* __restrict__ state, const float* __restrict__ targets, unsigned long long* __restrict__ counters, int64_t n,
                    int n_ticks) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    StepSmemH& S = *reinterpret_cast<StepSmemH*>(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t tbase = hyb_tmem_alloc(S, warp);
    RowsH R = hyb_rows(S, tbase, warp, lane);
    const int64_t env = (int64_t)blockIdx.x * (HWARPS * 32) + threadIdx.x;
    const bool live = env < n;
    ExEnv e;
    e.st = state + (live ? env : 0) * SNK_STATE_STRIDE;
    e.tid = lane;
    R.tg = const_cast<float*>(targets) + (live ? env : 0) * NJ; // the caller's row itself (only read here)
    ex_load_base(e);
    int iters = 0;
#pragma unroll 1
    for (int t = 0; t < n_ticks; t++) {
        bool ab;
        ExTickOut to;
        ex_tick<CONE>(cT, P, R, e, live, false, &ab, &to);
        iters += to.iterations;
    }
    if (live) {
        ex_store_base(e);
        if (counters) {
            atomicAdd(&counters[0], (unsigned long long)n_ticks);
            atomicAdd(&counters[1], (unsigned long long)iters);
        }
    }
    hyb_tmem_free(tbase, warp);
}

template <bool CONE>
__global__ void __launch_bounds__(HWARPS * 32, 1)
snk_hyb_rollout_kernel(const KParams P, float* __restrict__ state, float* __restrict__ tgt_scratch, const RolloutArgs A,
                       unsigned long long* __restrict__ counters, int64_t n) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    StepSmemH& S = *reinterpret_cast<StepSmemH*>(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t tbase = hyb_tmem_alloc(S, warp);
    const int64_t first_base = ((int64_t)warp * gridDim.x + blockIdx.x) * 32;
    const int64_t dyn_base = min((int64_t)gridDim.x * HWARPS * 32, n);
    run_rollout_warp<CONE>(P, hyb_rows(S, tbase, warp, lane), state, tgt_scratch, A, counters, n, first_base, dyn_base);
    hyb_tmem_free(tbase, warp);
}

// ---------------------------------------------------------------------------------------------
// Longest-first hand-out order.  The tick count of an env-step is known before it runs: with the motor
// rows imposed exactly the joint error shrinks by (1 - kp) per tick, so ticks = ceil(log(thr / |e|) /
// log(1 - kp)).  When the batch is larger than the lanes of the persistent grid, environments are handed out
// in descending predicted tick count (counting sort, 64 buckets), so the launch ends on the short jobs
// instead of on a half-empty GPU waiting for a 30-tick straggler.  Results do not depend on the order.
// ---------------------------------------------------------------------------------------------
#define SCHED_BUCKETS 64

__global__ void snk_exact_predict_kernel(const KParams P, const float* __restrict__ state, const float* __restrict__ actions, int64_t n,
                                         uint8_t* __restrict__ bucket, unsigned* __restrict__ hist) {
    __shared__ unsigned cnt[SCHED_BUCKETS];
    if (threadIdx.x < SCHED_BUCKETS) cnt[threadIdx.x] = 0u;
    __syncthreads();
    const int64_t env = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (env < n) {
        float tgt[NJ];
#pragma unroll
        for (int j = 0; j < NJ; j++) tgt[j] = 0.f;
        for (int k4 = 0; k4 < P.actdim; k4 += 4) { // 16-byte loads (the rows may live in mapped host memory: few, wide PCIe reads)
            const float4 v = *reinterpret_cast<const float4*>(actions + env * P.actdim + k4);
            const float av[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int k = k4 + q;
                float a = av[q];
                a = (a < -1.f) ? -1.f : a;
                a = (a > 1.f) ? 1.f : a;
                const int j = (P.gait == 0) ? 2 * k : (P.gait == 1) ? 2 * k + 1 : k;
#pragma unroll
                for (int jj = 0; jj < NJ; jj++) if (jj == j) tgt[jj] = a * P.sf;
            }
        }
        const float* q = state + env * SNK_STATE_STRIDE + SNK_S_Q;
        float e2 = 0.f;
#pragma unroll
        for (int j = 0; j < NJ; j++) { const float d = tgt[j] - q[j]; e2 += d * d; }
        const float err = sqrtf(e2);
        int k = 0;
        if (err > P.errthr) { // a NaN error compares false: zero ticks, as in the step itself
            const float shrink = 1.f - P.kp;
            k = (shrink > 0.f && shrink < 1.f) ? (int)ceilf(__logf(P.errthr / err) / __logf(shrink)) : 1;
            k = max(1, min(k, min(P.maxticks, SCHED_BUCKETS - 1)));
        }
        bucket[env] = (uint8_t)k;
        atomicAdd(&cnt[k], 1u);
    }
    __syncthreads();
    if (threadIdx.x < SCHED_BUCKETS && cnt[threadIdx.x]) atomicAdd(&hist[threadIdx.x], cnt[threadIdx.x]);
}

__global__ void snk_exact_order_kernel(int64_t n, const uint8_t* __restrict__ bucket, const unsigned* __restrict__ hist,
                                       unsigned* __restrict__ cursor, int32_t* __restrict__ order) {
    __shared__ unsigned cnt[SCHED_BUCKETS], base[SCHED_BUCKETS];
    if (threadIdx.x < SCHED_BUCKETS) cnt[threadIdx.x] = 0u;
    __syncthreads();
    const int64_t env = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned b = 0, my = 0;
    if (env < n) { b = bucket[env]; my = atomicAdd(&cnt[b], 1u); }
    __syncthreads();
    if (threadIdx.x < SCHED_BUCKETS) {
        unsigned off = 0; // environments in longer buckets come first
        for (int j = threadIdx.x + 1; j < SCHED_BUCKETS; j++) off += hist[j];
        base[threadIdx.x] = off + (cnt[threadIdx.x] ? atomicAdd(&cursor[threadIdx.x], cnt[threadIdx.x]) : 0u);
    }
    __syncthreads();
    if (env < n) order[base[b] + my] = (int32_t)env;
}

#ifndef SNK_SCREEN
#include "snake_manifold.cuh"
#endif

#ifdef SNK_SCREEN
// tools/screen_variants.py compiles this file with -DSNK_SCREEN: only the benchmarked kernel, for a look at its SASS
template __global__ void snk_hyb_step_kernel<true, false>(const KParams, float*, float*, const float*, float*, float*, uint8_t*, int32_t*, unsigned long long*,
                                                           const int32_t*, int64_t, int, int, const HandOut, float*, float*);
#else
// ---------------------------------------------------------------------------------------------
// launch wrappers used by the C-ABI host code (snake_abi.cu)
// ---------------------------------------------------------------------------------------------
#define MAX_DEVICES 64
// Process-wide configuration, written under g_mu by snk_exact_configure (i.e. by snk_create) and read by the launchers.
// The per-device figures are indexed by the CUDA device ordinal; the ablation switches come from the environment once per create.
static std::mutex g_mu;
static int g_sms[MAX_DEVICES];
static bool g_no_sort = false;   // SNK_EXACT_ORDER=index disables the longest-first hand-out (ablation)
static int g_spread = 3;         // SNK_EXACT_SPREAD: first-wave hand-out policy (see snk_hyb_step_kernel; 1 and 3 are both warp-major)
static int g_active_warps = 0;   // SNK_EXACT_WARPS=1..8 forces the number of working warps per SM (0: all HWARPS)
static bool g_balance = true;    // SNK_EXACT_BALANCE=0 disables the two-pool (balanced) hand-out (ablation)
static bool g_split = true;      // SNK_EXACT_SPLIT=0 disables the split hand-out (env-steps run in two parts; the two pools take over)
static int g_split_frac_q8 = 154; // SNK_EXACT_SPLIT_FRAC (percent; default: chosen per launch): share of an env-step's predicted ticks in its first part
static bool g_split_frac_forced = false;
static int g_split_kmax = 4;       // SNK_EXACT_SPLIT_KMAX: split only up to this many whole env-steps per lane (beyond, the two pools do as well or better)
static int g_split_min_pct = 3;    // SNK_EXACT_SPLIT_MINPCT: ... and only if the idle lanes of the last wave are at least this share of the batch

size_t snk_exact_split_buf_bytes() { return (size_t)(SPLIT_CTAS + SPLIT_MAX + SPLIT_MAX * 8) * sizeof(int); }

const char* snk_exact_variant() {
    return "8 warps/SM, rows in TMEM (8 words) + shared memory (7) + registers (2), 256 envs/SM";
}

// The model tables live in one __constant__ symbol per device: all live handles of a process must share one
// model.  Returns cudaErrorInvalidValue (reported by snk_create) when `host_tables` differs from the tables of
// the handles that are alive.
static ExTables g_tables;
static int g_live_handles = 0;

void snk_exact_release() {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_live_handles > 0) g_live_handles--;
}

template <class K>
static cudaError_t set_smem(K kernel, size_t bytes) { return cudaFuncSetAttribute((const void*)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes); }

cudaError_t snk_exact_configure(const ExTables* host_tables) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_live_handles > 0 && memcmp(&g_tables, host_tables, sizeof(ExTables)) != 0) return cudaErrorInvalidValue;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= MAX_DEVICES) return cudaErrorInvalidDevice;
    memcpy(&g_tables, host_tables, sizeof(ExTables));
    const char* so = getenv("SNK_EXACT_ORDER");
    g_no_sort = so && so[0] == 'i';
    const char* sp = getenv("SNK_EXACT_SPREAD");
    g_spread = (sp && sp[0] >= '0' && sp[0] <= '3') ? sp[0] - '0' : 3;
    const char* bl = getenv("SNK_EXACT_BALANCE");
    g_balance = !(bl && bl[0] == '0');
    const char* spl = getenv("SNK_EXACT_SPLIT");
    g_split = !(spl && spl[0] == '0');
    const char* spf = getenv("SNK_EXACT_SPLIT_FRAC");
    g_split_frac_forced = spf && atoi(spf) >= 5 && atoi(spf) <= 95;
    g_split_frac_q8 = g_split_frac_forced ? atoi(spf) * 256 / 100 : 154;
    const char* skm = getenv("SNK_EXACT_SPLIT_KMAX");
    g_split_kmax = (skm && atoi(skm) >= 0) ? atoi(skm) : 4;
    const char* smp = getenv("SNK_EXACT_SPLIT_MINPCT");
    g_split_min_pct = (smp && atoi(smp) >= 0) ? atoi(smp) : 3;
    const char* w = getenv("SNK_EXACT_WARPS");
    g_active_warps = (w && atoi(w) >= 1 && atoi(w) <= HWARPS) ? atoi(w) : 0;
    e = cudaMemcpyToSymbol(cT, host_tables, sizeof(ExTables));
    if (e == cudaSuccess) { // Bullet's 32-gon cylinder hull (snake_manifold.cuh): vertex i at angle 2 pi i / 32 from the link's y axis
        float hs[MAN_HULL], hcs[MAN_HULL];
        for (int i = 0; i < MAN_HULL; i++) { const double th = 2.0 * 3.14159265358979323846 / MAN_HULL * i; hs[i] = (float)sin(th); hcs[i] = (float)cos(th); }
        e = cudaMemcpyToSymbol(cHullS, hs, sizeof hs);
        if (e == cudaSuccess) e = cudaMemcpyToSymbol(cHullC, hcs, sizeof hcs);
    }
    if (e == cudaSuccess) e = set_smem(snk_hyb_step_kernel<true, false>, sizeof(StepSmemH));
    if (e == cudaSuccess) e = set_smem(snk_hyb_step_kernel<false, false>, sizeof(StepSmemH));
    if (e == cudaSuccess) e = set_smem(snk_hyb_step_kernel<true, false, true>, sizeof(StepSmemH));
    if (e == cudaSuccess) e = set_smem(snk_hyb_step_kernel<false, false, true>, sizeof(StepSmemH));
    if (e == cudaSuccess) e = set_smem(snk_hyb_step_kernel<true, true>, sizeof(StepSmemH));
    if (e == cudaSuccess) e = set_smem(snk_hyb_step_kernel<false, true>, sizeof(StepSmemH));
    if (e == cudaSuccess) e = set_smem(snk_hyb_tick_kernel<true>, sizeof(StepSmemH));
    if (e == cudaSuccess) e = set_smem(snk_hyb_tick_kernel<false>, sizeof(StepSmemH));
    if (e == cudaSuccess) e = set_smem(snk_hyb_rollout_kernel<true>, sizeof(StepSmemH));
    if (e == cudaSuccess) e = set_smem(snk_hyb_rollout_kernel<false>, sizeof(StepSmemH));
    if (e == cudaSuccess) e = set_smem(snk_man_step_kernel<true>, MAN_RING_BYTES);
    if (e == cudaSuccess) e = set_smem(snk_man_step_kernel<false>, MAN_RING_BYTES);
    if (e == cudaSuccess) e = set_smem(snk_man_step_trace_kernel<true>, MAN_RING_BYTES);
    if (e == cudaSuccess) e = set_smem(snk_man_step_trace_kernel<false>, MAN_RING_BYTES);
    if (e == cudaSuccess) e = set_smem(snk_man_rollout_kernel<true>, MAN_RING_BYTES);
    if (e == cudaSuccess) e = set_smem(snk_man_rollout_kernel<false>, MAN_RING_BYTES);
    // MAN_MINB CTAs x MAN_RING_BYTES of ring per SM and the rest of the 256 KB as L1 (state records, contact caches, local arrays): the
    // carveout is requested explicitly, otherwise it depends on which kernel ran before (a larger one costs L1: 3 CTAs x 60 KB ran 277 ms
    // against 228 ms for 2 x 60 KB at 262 144 environments)
    {
        int pct = (int)((MAN_MINB * (MAN_RING_BYTES + 1024) * 100 + 233471) / 233472);
        if (getenv("SNK_MAN_CARVEOUT")) pct = atoi(getenv("SNK_MAN_CARVEOUT"));
        if (pct > 100) pct = 100;
        const void* man_kernels[] = {(const void*)snk_man_step_kernel<true>, (const void*)snk_man_step_kernel<false>, (const void*)snk_man_step_trace_kernel<true>,
                                     (const void*)snk_man_step_trace_kernel<false>, (const void*)snk_man_rollout_kernel<true>, (const void*)snk_man_rollout_kernel<false>};
        for (const void* k : man_kernels)
            if (e == cudaSuccess) e = cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
    }
    if (e != cudaSuccess) return e;
    e = cudaDeviceGetAttribute(&g_sms[dev], cudaDevAttrMultiProcessorCount, dev);
    if (e == cudaSuccess) g_live_handles++;
    return e;
}

static int cur_dev() { int d = 0; cudaGetDevice(&d); return (d >= 0 && d < MAX_DEVICES) ? d : 0; }

// sched = {bucket[n] u8, order[n] i32} owned by the handle (null: hand out in index order); hist/cursor are the
// 2 x 64 words after the 8 counters (zeroed with them)
cudaError_t snk_exact_launch_step(const KParams& P, float* state, float* tgt_scratch, const float* actions, float* obs, float* rew, uint8_t* done,
                                  int32_t* ticks, unsigned long long* counters, uint8_t* bucket, int32_t* order, int64_t n, cudaStream_t st,
                                  int* launches, int flag_rows, int* split_buf) {
    const int dev = cur_dev(), sms = g_sms[dev];
    const int aw = g_active_warps ? g_active_warps : HWARPS;
    const int lanes = sms * aw * 32;
    const int32_t* use_order = nullptr;
    *launches = 1;
    if (bucket && order && n > lanes && !g_no_sort) {
        unsigned* hist = reinterpret_cast<unsigned*>(counters + 8);
        unsigned* cursor = hist + SCHED_BUCKETS;
        dim3 g((unsigned)((n + 255) / 256)), b(256);
        snk_exact_predict_kernel<<<g, b, 0, st>>>(P, state, actions, n, bucket, hist);
        snk_exact_order_kernel<<<g, b, 0, st>>>(n, bucket, hist, cursor, order);
        use_order = order;
        *launches = 3;
    }
    // a small batch gets one CTA per warp of environments: all SMs before a second warp per SM
    const int64_t want = g_spread ? (n + EB - 1) / EB : (n + aw * 32 - 1) / (aw * 32);
    dim3 grid((unsigned)(want < sms ? want : sms)), block(HWARPS * 32);
    HandOut H;
    H.n_long = n; H.short_warps = 0; H.flag_rows = flag_rows;
    H.split_total = 0; H.split_frac_q8 = g_split_frac_q8; H.bucket = bucket; H.split_buf = split_buf;
    if (use_order && g_balance && g_split && split_buf && aw == HWARPS && (int)grid.x == sms && sms <= SPLIT_CTAS) {
        // n = k L + r: the r shortest env-steps are run in two parts (SplitCta).  Model (tools/handout_sim.py, 131 072 environments =
        // 3.46 L): 110.2 warp iterations with the two pools below, 107.0 split, 104.3 ideal.  Measured on B200 (ms per step, split /
        // two pools): 50 000 envs 12.1 / 14.6, 62 000 13.7 / 15.3, 100 000 21.2 / 22.7, 131 072 27.8 / 29.2, 162 918 34.9 / 35.3,
        // 200 000 42.4 / 42.1 -- from five whole env-steps per lane on the two pools do as well, and without the 3 % gate the large
        // batches lose a little (2^20: 214.9 / 214.2), so: k <= 4 and (L - r) / n >= 3 %.
        const int64_t L = (int64_t)grid.x * aw * 32, k = n / L, r = n - k * L;
        if (k >= 1 && k <= g_split_kmax && 16 * r >= L && 100 * (L - r) >= g_split_min_pct * n) {
            H.split_total = (int)r;
            // share of the first part: with r <= L / 2 one part per lane, about half each (the lanes without a first part start on
            // the LONGEST whole env-steps, so a little more than half balances: 60 %, measured); with r > L / 2 the L - r other
            // lanes finish several second parts each, and the parts even out at r / L (+ 10 points for the same reason)
            if (!g_split_frac_forced) H.split_frac_q8 = 2 * r <= L ? 154 : (int)((r * 256) / L) + 26 > 230 ? 230 : (int)((r * 256) / L) + 26;
        }
    }
    if (H.split_total > 0) {
        cudaError_t me = cudaMemsetAsync(split_buf, 0, (size_t)(SPLIT_CTAS + H.split_total) * sizeof(int), st);
        if (me != cudaSuccess) return me; // (a memset node, not a kernel: `launches` stays)
    } else if (use_order && g_balance && (g_spread == 1 || g_spread == 3)) { // n = k L + r: r lanes (whole warps) run k + 1 env-steps, taken from the shortest
        const int64_t L = (int64_t)grid.x * aw * 32, k = n / L, r = n - k * L;
        // Worth it when plain longest-first would end on a long, thinly populated last wave: L - r idle lanes for one env-step out
        // of n / L per lane, i.e. a loss of about (L - r) / n.  Measured on B200 (ms per step, balanced / plain): 100 000 envs
        // 22.6 / 23.0, 131 072 29.1 / 30.2, 200 000 42.0 / 44.8, 262 144 53.3 / 53.6 -- but 524 288 109.1 / 106.6: over many waves
        // the lanes drift away from the k / k + 1 split and the pools only disturb the longest-first order, so it is used for
        // (L - r) / n >= 3 % only.
        if (k >= 1 && r > 0 && 100 * (L - r) >= 3 * n) {
            H.short_warps = (int)((r + 31) / 32);
            const int64_t n_short = H.short_warps * 32LL * (k + 1);
            H.n_long = n_short < n ? n - n_short : 0;
        }
    }
    // the split hand-out is an instantiation of its own: the plain one, which runs the large batches, carries none of its code
#define SNK_LAUNCH_HYB(C, SP) snk_hyb_step_kernel<C, false, SP><<<grid, block, sizeof(StepSmemH), st>>>(P, state, tgt_scratch, actions, obs, rew, done, ticks, counters, use_order, n, aw, g_spread, H, nullptr, nullptr)
    if (H.split_total > 0) { if (P.cone) SNK_LAUNCH_HYB(true, true); else SNK_LAUNCH_HYB(false, true); }
    else { if (P.cone) SNK_LAUNCH_HYB(true, false); else SNK_LAUNCH_HYB(false, false); }
#undef SNK_LAUNCH_HYB
    return cudaGetLastError();
}

// persistent manifolds (snake_manifold.cuh): grid and scratch size of a device, and the step launch
static int man_grid(int dev) { return g_sms[dev] * MAN_MINB; }
size_t snk_man_scratch_bytes() { return (size_t)man_grid(cur_dev()) * (MAN_THREADS / 32) * MAN_WARP_V4 * sizeof(float4); }
size_t snk_man_cache_floats() { return MAN_STRIDE; }
cudaError_t snk_man_launch_step(const KParams& P, float* state, float* tgt_scratch, float* cache, void* scratch, float warm, const float* actions, float* obs,
                                float* rew, uint8_t* done, int32_t* ticks, unsigned long long* counters, int64_t n, cudaStream_t st) {
    const int64_t want = (n + MAN_THREADS - 1) / MAN_THREADS;
    const int full = man_grid(cur_dev());
    dim3 grid((unsigned)(want < full ? want : full)), block(MAN_THREADS);
    if (P.cone) snk_man_step_kernel<true><<<grid, block, MAN_RING_BYTES, st>>>(P, state, tgt_scratch, cache, (float4*)scratch, warm, actions, obs, rew, done, ticks, counters, n);
    else snk_man_step_kernel<false><<<grid, block, MAN_RING_BYTES, st>>>(P, state, tgt_scratch, cache, (float4*)scratch, warm, actions, obs, rew, done, ticks, counters, n);
    return cudaGetLastError();
}

cudaError_t snk_man_launch_step_trace(const KParams& P, float* state, float* tgt_scratch, float* cache, void* scratch, float warm, const float* actions,
                                      float* obs, float* rew, uint8_t* done, int32_t* ticks, unsigned long long* counters, int64_t n, float* tick_obs,
                                      float* tick_links, cudaStream_t st) {
    const int64_t want = (n + MAN_THREADS - 1) / MAN_THREADS;
    const int full = man_grid(cur_dev());
    dim3 grid((unsigned)(want < full ? want : full)), block(MAN_THREADS);
    if (P.cone) snk_man_step_trace_kernel<true><<<grid, block, MAN_RING_BYTES, st>>>(P, state, tgt_scratch, cache, (float4*)scratch, warm, actions, obs, rew, done, ticks, counters, n, tick_obs, tick_links);
    else snk_man_step_trace_kernel<false><<<grid, block, MAN_RING_BYTES, st>>>(P, state, tgt_scratch, cache, (float4*)scratch, warm, actions, obs, rew, done, ticks, counters, n, tick_obs, tick_links);
    return cudaGetLastError();
}

// at most man_grid(dev) CTAs, like the step: the handle's row tables (man_scratch) are indexed by global warp
cudaError_t snk_man_launch_rollout(const KParams& P, float* state, float* tgt_scratch, float* cache, void* scratch, float warm, const float* weights,
                                   const float* mean, const float* inv_std, const float* noise, int n_steps, float* returns, float* trace,
                                   unsigned long long* counters, int64_t n, cudaStream_t st) {
    RolloutArgs A;
    A.weights = weights; A.mean = mean; A.inv_std = inv_std; A.noise = noise; A.returns = returns; A.trace = trace; A.n_steps = n_steps;
    A.queue = nullptr; A.done_steps = nullptr;
    const int64_t want = (n + MAN_THREADS - 1) / MAN_THREADS;
    const int full = man_grid(cur_dev());
    dim3 grid((unsigned)(want < full ? want : full)), block(MAN_THREADS);
    if (P.cone) snk_man_rollout_kernel<true><<<grid, block, MAN_RING_BYTES, st>>>(P, state, tgt_scratch, cache, (float4*)scratch, warm, A, counters, n);
    else snk_man_rollout_kernel<false><<<grid, block, MAN_RING_BYTES, st>>>(P, state, tgt_scratch, cache, (float4*)scratch, warm, A, counters, n);
    return cudaGetLastError();
}

cudaError_t snk_man_launch_clear(float* cache, const uint8_t* mask, int64_t n, cudaStream_t st) {
    const int64_t blocks = (n * (MAN_STRIDE / 4) + 255) / 256;
    snk_man_clear_kernel<<<(unsigned)(blocks < 65536 ? blocks : 65536), 256, 0, st>>>(cache, mask, n);
    return cudaGetLastError();
}

cudaError_t snk_man_launch_check(const float* cache, int64_t n, unsigned long long* bad, cudaStream_t st) {
    const int64_t blocks = (n + 255) / 256;
    snk_man_check_kernel<<<(unsigned)(blocks < 4096 ? blocks : 4096), 256, 0, st>>>(cache, n, bad);
    return cudaGetLastError();
}

cudaError_t snk_exact_launch_step_trace(const KParams& P, float* state, float* tgt_scratch, const float* actions, float* obs, float* rew, uint8_t* done,
                                        int32_t* ticks, unsigned long long* counters, int64_t n, float* tick_obs, float* tick_links, cudaStream_t st) {
    // the benchmarked kernel's TRACE instantiation: same arithmetic, same bits as snk_step
    const int dev = cur_dev();
    const int64_t warps = (n + EB - 1) / EB;
    dim3 grid((unsigned)(warps < g_sms[dev] ? warps : g_sms[dev])), block(HWARPS * 32);
    HandOut H;
    H.n_long = n; H.short_warps = 0; H.flag_rows = 0;
    if (P.cone) snk_hyb_step_kernel<true, true><<<grid, block, sizeof(StepSmemH), st>>>(P, state, tgt_scratch, actions, obs, rew, done, ticks, counters, nullptr, n, HWARPS, 1, H, tick_obs, tick_links);
    else snk_hyb_step_kernel<false, true><<<grid, block, sizeof(StepSmemH), st>>>(P, state, tgt_scratch, actions, obs, rew, done, ticks, counters, nullptr, n, HWARPS, 1, H, tick_obs, tick_links);
    return cudaGetLastError();
}

// The rollout kernel's lanes wait for environments that other CTAs push onto the ready queue, so its whole grid must be
// resident at once: it is launched COOPERATIVELY (one CTA per SM at most), which makes the driver either co-schedule every
// CTA or refuse the launch (cudaErrorCooperativeLaunchTooLarge under an SM-limited context) -- it can never hang on a CTA
// that did not get an SM.  Two rollouts on one device (two handles / streams) are serialised by the driver.
cudaError_t snk_exact_launch_rollout(const KParams& P, float* state, float* tgt_scratch, const float* weights, const float* mean, const float* inv_std,
                                     const float* noise, int n_steps, float* returns, float* trace, int32_t* queue, int32_t* done_steps,
                                     unsigned long long* counters, int64_t n, cudaStream_t st) {
    RolloutArgs A;
    A.weights = weights; A.mean = mean; A.inv_std = inv_std; A.noise = noise; A.returns = returns; A.trace = trace; A.n_steps = n_steps;
    A.queue = queue; A.done_steps = done_steps;
    const int dev = cur_dev(), sms = g_sms[dev];
    const int64_t want = (n + EB - 1) / EB;
    KParams Pc = P;
    void* args[] = {(void*)&Pc, (void*)&state, (void*)&tgt_scratch, (void*)&A, (void*)&counters, (void*)&n};
    int per_sm = 0;
    const void* k = P.cone ? (const void*)snk_hyb_rollout_kernel<true> : (const void*)snk_hyb_rollout_kernel<false>;
    cudaError_t e = P.cone ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, snk_hyb_rollout_kernel<true>, HWARPS * 32, sizeof(StepSmemH))
                           : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, snk_hyb_rollout_kernel<false>, HWARPS * 32, sizeof(StepSmemH));
    if (e != cudaSuccess) return e;
    if (per_sm < 1) return cudaErrorCooperativeLaunchTooLarge;
    dim3 grid((unsigned)(want < sms ? want : sms)), block(HWARPS * 32);
    return cudaLaunchCooperativeKernel(k, grid, block, args, sizeof(StepSmemH), st);
}

cudaError_t snk_exact_launch_tick(const KParams& P, float* state, const float* targets, unsigned long long* counters, int64_t n,
                                  int n_ticks, cudaStream_t st) {
    dim3 grid((unsigned)((n + HWARPS * 32 - 1) / (HWARPS * 32))), block(HWARPS * 32);
    if (P.cone) snk_hyb_tick_kernel<true><<<grid, block, sizeof(StepSmemH), st>>>(P, state, targets, counters, n, n_ticks);
    else snk_hyb_tick_kernel<false><<<grid, block, sizeof(StepSmemH), st>>>(P, state, targets, counters, n, n_ticks);
    return cudaGetLastError();
}

#ifdef SNK_PHASE_CLOCKS
// phase clocks of the current device (see ExPhaseClock): copies the [SNK_CLK_WARPS][SNK_CLK_PHASES] cycle sums to `out` (may be null), then
// zeroes them when `reset` is set.  Synchronises the device.
extern "C" int snk_phase_clocks(unsigned long long* out, int reset) {
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess && out) e = cudaMemcpyFromSymbol(out, snk_phase_clk, sizeof(snk_phase_clk));
    if (e == cudaSuccess && reset) {
        static unsigned long long zero[SNK_CLK_WARPS][SNK_CLK_PHASES];
        e = cudaMemcpyToSymbol(snk_phase_clk, zero, sizeof(zero));
    }
    return (int)e;
}
#endif
#endif // SNK_SCREEN
