// snake_task.cuh -- the env-step kernel template: task logic of SnakeGymEnv.step() around a
// per-warp physics tick.  WM is the warp's shared-memory record of one solver variant; it must
// provide s[64], target[16], Rw, pw, Rj and an overload  int tick(WM&, const DevTables*, const KParams&, int lane).
#pragma once
#include "snake_dev.cuh"

// ---------------------------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------------------------
template <class WM>
__device__ __forceinline__ float obs_of(const WM& W, int k) { // snake.py:209-217
    if (k < 16) return W.s[SNK_S_Q + k];
    if (k < 32) return W.s[SNK_S_QD + k - 16];
    if (k < 48) return W.s[SNK_S_TAU + k - 32];
    if (k < 51) return W.s[SNK_S_POS + k - 48];
    if (k < 55) return W.s[SNK_S_QUAT + k - 51];
    return W.s[SNK_S_FZ];
}

template <class WM>
__device__ __forceinline__ void soft_reset(WM& W, const KParams& P, int lane) { // snake.py:119-127
    for (int k = lane; k < SNK_STATE_STRIDE; k += 32) {
        bool keep = (k >= SNK_S_TAU && k <= SNK_S_FZ) && P.stale;
        if (!keep) W.s[k] = (k == SNK_S_QUAT + 3) ? 1.f : 0.f;
    }
}

// One env-step (or n_ticks raw ticks) of environment env on its warp's record W.  RAW = false: one SubprocVecEnv.step.  RAW = true:
// n_ticks raw ticks with targets[N,16] (gait script).  P is taken by value like the kernel parameter it is: passed by reference it
// changes the code generated for the existing kernels.
template <class WM, bool RAW>
__device__ __forceinline__ void env_step(WM& W, int lane, int64_t env, const DevTables* __restrict__ T, const KParams P, float* __restrict__ state,
                                         const float* __restrict__ in, float* __restrict__ obs, float* __restrict__ rew, uint8_t* __restrict__ done,
                                         int32_t* __restrict__ ticks, unsigned long long* __restrict__ counters, int n_ticks,
                                         float* __restrict__ tick_obs, float* __restrict__ tick_links) {
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
            a = (a < -1.f) ? -1.f : a; // checkBound's comparisons: a NaN passes through (SnakeGymEnv.py:84-87)
            a = (a > 1.f) ? 1.f : a;
            tgt = a * P.sf;
        }
        W.target[lane] = tgt;
    }
    __syncwarp();
    const float xprev = W.s[SNK_S_POS];
    float height = fk(W, T, lane);
    int counter = 0, iters = 0;
    bool end_height = false;
    if (RAW) {
        for (int t = 0; t < n_ticks; t++) {
            iters += tick(W, T, P, lane);
            counter++;
            height = fk(W, T, lane);
        }
    } else {
        for (;;) { // snake.py:284-304
            float e2 = 0.f;
#pragma unroll 1
            for (int j = 0; j < NJ; j++) { float d = W.target[j] - W.s[SNK_S_Q + j]; e2 += d * d; }
            if (!(sqrtf(e2) > P.errthr)) break;
            iters += tick(W, T, P, lane);
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
    if (bad) { W.s[lane] = 0.f; W.s[lane + 32] = 0.f; __syncwarp(); }
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

template <class WM, bool RAW, int WARPS, int MINB>
__global__ void __launch_bounds__(WARPS * 32, MINB)
snk_env_kernel(const DevTables* __restrict__ T, const KParams P, float* __restrict__ state, const float* __restrict__ in,
                float* __restrict__ obs, float* __restrict__ rew, uint8_t* __restrict__ done, int32_t* __restrict__ ticks,
                unsigned long long* __restrict__ counters, int64_t n, int n_ticks, float* __restrict__ tick_obs = nullptr,
                float* __restrict__ tick_links = nullptr) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t env = (int64_t)blockIdx.x * WARPS + warp;
    if (env >= n) return;
    WM& W = reinterpret_cast<WM*>(smem_raw)[warp];
    env_step<WM, RAW>(W, lane, env, T, P, state, in, obs, rew, done, ticks, counters, n_ticks, tick_obs, tick_links);
}

