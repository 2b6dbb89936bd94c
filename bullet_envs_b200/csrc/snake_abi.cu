// snake_abi.cu -- the extern "C" boundary declared in include/snake_b200.h (host side).
//
// Owns: the [N,64] fp32 state array, the fp32 model tables, four device counters and (for the
// *_host entry points) pinned staging buffers plus their device twins.  Everything else belongs to
// the caller.  No CPU fallback: every entry point either enqueues CUDA work or fails.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <time.h>

#include <atomic>
#include <new>
#include <vector>

#include "snake_host.h"

// warp-per-env kernel with Bullet-order motor rows (snake_pgs.cu)
cudaError_t snk_pgs_configure();
cudaError_t snk_pgs_launch_step(const DevTables* T, const KParams& P, float* state, const float* actions, float* obs, float* rew, uint8_t* done,
                                int32_t* ticks, unsigned long long* counters, int64_t n, cudaStream_t st, float* tick_obs = nullptr,
                                float* tick_links = nullptr);
cudaError_t snk_pgs_launch_tick(const DevTables* T, const KParams& P, float* state, const float* targets, unsigned long long* counters, int64_t n,
                                int n_ticks, cudaStream_t st);
// thread-per-env kernel with the motor rows eliminated (snake_exact.cu)
cudaError_t snk_exact_configure(const ExTables* host_tables);
void snk_exact_release();
const char* snk_exact_variant();
cudaError_t snk_exact_launch_step(const KParams& P, float* state, float* tgt_scratch, const float* actions, float* obs, float* rew, uint8_t* done,
                                  int32_t* ticks, unsigned long long* counters, uint8_t* bucket, int32_t* order, int64_t n, cudaStream_t st,
                                  int* launches, int flag_rows, int* split_buf);
bool snk_exact_row_flags_supported();
size_t snk_exact_split_buf_bytes();
cudaError_t snk_exact_launch_rollout(const KParams& P, float* state, float* tgt_scratch, const float* weights, const float* mean, const float* inv_std,
                                     const float* noise, int n_steps, float* returns, float* trace, int32_t* queue, int32_t* done_steps,
                                     unsigned long long* counters, int64_t n, cudaStream_t st);
cudaError_t snk_exact_launch_step_trace(const KParams& P, float* state, float* tgt_scratch, const float* actions, float* obs, float* rew, uint8_t* done,
                                        int32_t* ticks, unsigned long long* counters, int64_t n, float* tick_obs, float* tick_links, cudaStream_t st);
cudaError_t snk_exact_launch_tick(const KParams& P, float* state, const float* targets, unsigned long long* counters, int64_t n,
                                  int n_ticks, cudaStream_t st);
// persistent contact manifolds + warm starting (snake_manifold.cuh, compiled into snake_exact.cu)
size_t snk_man_scratch_bytes();
size_t snk_man_cache_floats();
cudaError_t snk_man_launch_step(const KParams& P, float* state, float* tgt_scratch, float* cache, void* scratch, float warm, const float* actions, float* obs,
                                float* rew, uint8_t* done, int32_t* ticks, unsigned long long* counters, int64_t n, cudaStream_t st);
cudaError_t snk_man_launch_step_trace(const KParams& P, float* state, float* tgt_scratch, float* cache, void* scratch, float warm, const float* actions,
                                      float* obs, float* rew, uint8_t* done, int32_t* ticks, unsigned long long* counters, int64_t n, float* tick_obs,
                                      float* tick_links, cudaStream_t st);
cudaError_t snk_man_launch_rollout(const KParams& P, float* state, float* tgt_scratch, float* cache, void* scratch, float warm, const float* weights,
                                   const float* mean, const float* inv_std, const float* noise, int n_steps, float* returns, float* trace,
                                   unsigned long long* counters, int64_t n, cudaStream_t st);
cudaError_t snk_man_launch_clear(float* cache, const uint8_t* mask, int64_t n, cudaStream_t st);
cudaError_t snk_man_launch_check(const float* cache, int64_t n, unsigned long long* bad, cudaStream_t st);
// generalised advantage estimation (snake_gae.cu)
cudaError_t snk_launch_gae(const float* rewards, const uint8_t* dones, const float* values, const float* next_value, float gamma, float tau,
                           float* returns, float* advantages, int T, int64_t n, cudaStream_t st);
// self-collision clearance counter (snake_pgs.cu)
cudaError_t snk_launch_self_clearance(const DevTables* T, const float* state, float* out, int64_t n, cudaStream_t st);
// reset / observe (snake_pgs.cu)
cudaError_t snk_launch_reset(const KParams& P, float* state, const uint8_t* mask, float* obs, int64_t n, int mode, cudaStream_t st);

#define NCOUNTERS (8 + 64) // 8 counters + 2 x 64 32-bit words of the hand-out scheduler (histogram, cursors)

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, const char* detail = "") {
    snprintf(g_err, sizeof g_err, fmt, detail);
    return code;
}
#define CU(call)                                                                  \
    do {                                                                          \
        cudaError_t e_ = (call);                                                  \
        if (e_ != cudaSuccess) return fail(SNK_E_CUDA, #call ": %s", cudaGetErrorString(e_)); \
    } while (0)

struct snk_handle {
    int device;
    int64_t n;
    bool exact;                   // thread-per-env kernel with the motor rows eliminated (else warp-per-env, Bullet-order rows)
    KParams P;
    DevTables* T;                 // device: general model tables (warp-per-env kernel, clearance counter)
    float* state;                 // device [n][64]
    float* tgt;                   // device [n + 1][16]: joint targets of the env-step in flight (exact kernel; row n stays zero)
    uint8_t* bucket;              // device [n]: predicted tick count of the coming env-step (exact kernel)
    int32_t* order;               // device [n]: longest-first hand-out order
    int* split_buf;               // device: claim counters, flags and run words of the split hand-out (exact kernel)
    int32_t* roll_queue;          // device: ready queue of snk_rollout_linear, n * (steps - 1) entries (grown on demand)
    size_t roll_queue_len;
    unsigned long long* counters; // device [NCOUNTERS]: ticks, sweeps, dones, non-finite, work-queue head
    int64_t launches;
    // persistent contact manifolds (snk_set_manifold): per-environment caches, the resident threads' row tables, warm-start factor
    bool manifold;
    float* man_cache;             // device [n][MAN_STRIDE]
    void* man_scratch;            // device, snk_man_scratch_bytes()
    unsigned long long* man_bad;  // device, 1 word: result of the count-word check of snk_set_manifold_cache
    float man_warm;
    // staging for the *_host entry points (allocated on first use)
    cudaEvent_t ev_dev;           // recorded after every state-touching launch on a caller stream; the *_host entry points
    bool ev_valid;                // make their own stream wait on it (a device-path call may still be in flight)
    cudaStream_t hstream;
    float *h_act, *h_obs, *h_rew; // pinned
    uint8_t *h_done, *h_mask;
    int32_t* h_ticks;
    float *d_act, *d_obs, *d_rew; // device twins
    uint8_t *d_done, *d_mask;
    int32_t* d_ticks;
    bool staged;
    cudaEvent_t ev_chunk[16];     // one per chunk of the pipelined float64 host path
    int n_ev_chunk;
};

// Ordering between the caller's streams (device-path entry points, asynchronous) and the handle's own stream (host-path entry
// points, synchronous): a device-path call records ev_dev behind its work, a host-path call waits for it before touching the state.
static void mark_device_work(snk_handle* h, cudaStream_t st) {
    if (st == h->hstream && h->hstream) return;
    // a caller capturing its stream into a CUDA graph (the device-path entry points are capturable: no allocation, no synchronisation):
    // an event recorded inside a capture cannot be waited for outside of it, so nothing is recorded -- after replaying such a graph
    // the caller synchronises before mixing in *_host calls
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cap) == cudaSuccess && cap != cudaStreamCaptureStatusNone) return;
    if (!h->ev_valid) { if (cudaEventCreateWithFlags(&h->ev_dev, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); return; } h->ev_valid = true; }
    cudaEventRecord(h->ev_dev, st);
}
static void wait_device_work(snk_handle* h) {
    if (h->ev_valid && h->hstream) cudaStreamWaitEvent(h->hstream, h->ev_dev, 0);
}

// the exact kernel moves action / observation / weight rows as 16-byte vectors (rows are 32, 64 and 224 bytes long, so an aligned
// base pointer makes every row aligned): a misaligned pointer would fault inside the kernel and poison the context
static inline bool aligned16(const void* p) { return ((uintptr_t)p & 15u) == 0; }

// One env-step of the environments [off, off + cnt) (default: all).  act / obs / rew / done / ticks point at the rows of environment
// `off`.  The per-launch scheduler words of `counters` must be zero; the statistics words [0..3] accumulate.
static cudaError_t launch_step(snk_handle* h, const float* act, float* obs, float* rew, uint8_t* done, int32_t* ticks, cudaStream_t st, int64_t off = 0,
                               int64_t cnt = -1, int flag_rows = 0) {
    if (cnt < 0) cnt = h->n;
    int launches = 1;
    cudaError_t e = h->manifold ? snk_man_launch_step(h->P, h->state + off * SNK_STATE_STRIDE, h->tgt + off * NJ,
                                                      h->man_cache + off * (int64_t)snk_man_cache_floats(), h->man_scratch, h->man_warm, act, obs, rew, done,
                                                      ticks, h->counters, cnt, st)
                    : h->exact ? snk_exact_launch_step(h->P, h->state + off * SNK_STATE_STRIDE, h->tgt + off * NJ, act, obs, rew, done, ticks, h->counters,
                                                     h->bucket + off, h->order + off, cnt, st, &launches, flag_rows, h->split_buf)
                             : snk_pgs_launch_step(h->T, h->P, h->state + off * SNK_STATE_STRIDE, act, obs, rew, done, ticks, h->counters, cnt, st);
    h->launches += launches;
    mark_device_work(h, st);
    return e;
}

#include "snake_hostpool.h"
#include "snake_rowflags.h"

template <class F>
static void parallel_chunks(size_t n, F f, size_t serial_below = (size_t)1 << 16) { HostPool::get().run(n, std::function<void(size_t, size_t)>(f), serial_below); }
// Touch every page of a caller buffer that is about to be overwritten completely (the fresh arrays numpy hands over are untouched
// anonymous memory: 470 MB of observations are 115 000 page faults).  Called while the GPU works on the first chunk, so that the faults
// are not taken inside the widening of the last chunk, which nothing hides.  SNK_HOST_PREFAULT=0 disables it.
static void prefault_output(void* p, size_t bytes) {
    static int on = -1;
    if (on < 0) { const char* e = getenv("SNK_HOST_PREFAULT"); on = !(e && e[0] == '0'); }
    if (!on || bytes < ((size_t)1 << 20)) return;
    const size_t page = 4096;
    volatile char* base = (volatile char*)p;
    parallel_chunks((bytes + page - 1) / page, [=](size_t i0, size_t i1) { for (size_t i = i0; i < i1; i++) base[i * page] = 0; });
}

extern "C" {

const char* snk_last_error(void) { return g_err; }

const char* snk_build_info(void) {
    return "snake_b200 sm_100a; fused env-step kernels: thread-per-env (motor rows eliminated) and warp-per-env (Bullet-order PGS); built " __DATE__ " " __TIME__;
}

const char* snk_kernel_variant(void) { return snk_exact_variant(); }

int snk_default_params(snk_params* p) {
    if (!p) return fail(SNK_E_ARG, "snk_default_params: null pointer%s");
    memset(p, 0, sizeof *p);
    p->dt = 1.0 / 240.0; p->gravity[2] = -9.8;
    p->motor_kp = 0.1; p->motor_kd = 1.0; p->motor_max_force = INFINITY;
    p->scaling_factor = 3.14159265358979323846 / 6.0;
    p->alpha = 1.0; p->beta = 0.01; p->gamma = 0.1; p->energy_dt = 0.01;
    p->friction = 2.0; p->aniso[0] = 1.0; p->aniso[1] = 0.1; p->aniso[2] = 0.01;
    p->lin_damping = 0.04; p->ang_damping = 0.04; p->erp2 = 0.08; p->linear_slop = 1e-5; p->residual_threshold = 1e-7;
    p->max_coord_vel = 100.0; p->err_threshold = 0.05; p->height_threshold = 0.1; p->term_angle = 0.5;
    p->done_penalty = -5.0; p->collision_force = 10.0; p->collision_penalty = -10.0;
    p->solver_iterations = 50; p->max_ticks = 41; p->gait_selection = 1; p->cone_friction = 1; p->term_joint = 9;
    p->stale_obs_on_reset = 1; p->alternate_motor_order = 1; p->motor_solver = 2;
    return 0;
}

int snk_create(const snk_model* model, const snk_params* params, int64_t n_envs, int device, snk_handle** out) {
    if (!model || !params || !out) return fail(SNK_E_ARG, "snk_create: null pointer%s");
    if (n_envs <= 0) return fail(SNK_E_ARG, "snk_create: n_envs must be positive%s");
    if (n_envs > 0x7fffffffLL) return fail(SNK_E_ARG, "snk_create: at most 2^31 - 1 environments per handle (32-bit hand-out order); shard over handles%s");
    if (params->term_joint < 0 || params->term_joint >= SNK_OBS_DIM) return fail(SNK_E_ARG, "snk_create: term_joint out of range%s");
    if (params->solver_iterations < 1 || params->max_ticks < 0) return fail(SNK_E_ARG, "snk_create: bad iteration/tick limits%s");
    if (!(params->dt > 0)) return fail(SNK_E_ARG, "snk_create: dt must be positive%s");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(SNK_E_NODEV, "snk_create: no CUDA device (%s); this library has no CPU fallback", cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(SNK_E_ARG, "snk_create: device index out of range%s");
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail(SNK_E_NODEV, "snk_create: kernels are built for sm_100a only, found %s", prop.name);
    if (params->motor_solver < 0 || params->motor_solver > 2) return fail(SNK_E_ARG, "snk_create: motor_solver must be 0, 1 or 2%s");
    snk_handle* h = new (std::nothrow) snk_handle();
    if (!h) return fail(SNK_E_NOMEM, "snk_create: out of host memory%s");
    memset(h, 0, sizeof *h);
    h->device = device; h->n = n_envs;
    snk_to_kparams(params, &h->P);
    cudaError_t err = cudaSuccess;
    if (h->P.exact) { // thread-per-env kernel: tables in constant memory, state as [slot][env]
        ExTables xt;
        if (snk_to_extables(model, &xt)) { delete h; return fail(SNK_E_ARG, "snk_create: model layout not supported by the exact motor solver%s"); }
        err = snk_exact_configure(&xt);
        if (err == cudaErrorInvalidValue) { delete h; return fail(SNK_E_ARG, "snk_create: the exact motor solver keeps one model per process; destroy the handles of the other model first%s"); }
        h->exact = true;
        if (err == cudaSuccess) err = cudaMalloc(&h->bucket, (size_t)n_envs);
        if (err == cudaSuccess) err = cudaMalloc(&h->order, (size_t)n_envs * sizeof(int32_t));
        if (err == cudaSuccess) err = cudaMalloc(&h->split_buf, snk_exact_split_buf_bytes());
        if (err == cudaSuccess) err = cudaMalloc(&h->tgt, (size_t)(n_envs + 1) * NJ * sizeof(float));
        if (err == cudaSuccess) err = cudaMemset(h->tgt, 0, (size_t)(n_envs + 1) * NJ * sizeof(float));
    } else {
        err = snk_pgs_configure();
    }
    {
        DevTables host_tables;
        snk_to_tables(model, &host_tables);
        if (err == cudaSuccess) err = cudaMalloc(&h->T, sizeof(DevTables));
        if (err == cudaSuccess) err = cudaMemcpy(h->T, &host_tables, sizeof host_tables, cudaMemcpyHostToDevice);
    }
    if (err == cudaSuccess) err = cudaMalloc(&h->state, (size_t)n_envs * SNK_STATE_STRIDE * sizeof(float));
    if (err == cudaSuccess) err = cudaMalloc(&h->counters, NCOUNTERS * sizeof(unsigned long long));
    if (err == cudaSuccess) err = cudaMemset(h->counters, 0, NCOUNTERS * sizeof(unsigned long long));
    if (err == cudaSuccess) err = snk_launch_reset(h->P, h->state, nullptr, nullptr, h->n, 1, 0);
    if (err == cudaSuccess) err = cudaDeviceSynchronize();
    if (err != cudaSuccess) {
        if (h->exact) snk_exact_release();
        cudaFree(h->man_cache); cudaFree(h->man_scratch); cudaFree(h->man_bad);
    cudaFree(h->T); cudaFree(h->state); cudaFree(h->counters); cudaFree(h->bucket); cudaFree(h->order); cudaFree(h->split_buf); cudaFree(h->tgt);
        delete h;
        return fail(SNK_E_CUDA, "snk_create: %s", cudaGetErrorString(err));
    }
    h->launches = 1;
    *out = h;
    return 0;
}

int snk_destroy(snk_handle* h) {
    if (!h) return 0;
    cudaSetDevice(h->device);
    if (h->hstream && !h->staged) { cudaStreamSynchronize(h->hstream); cudaStreamDestroy(h->hstream); }
    if (h->staged) {
        cudaStreamSynchronize(h->hstream);
        cudaFreeHost(h->h_act); cudaFreeHost(h->h_obs); cudaFreeHost(h->h_rew); cudaFreeHost(h->h_done); cudaFreeHost(h->h_ticks);
        cudaFreeHost(h->h_mask);
        cudaFree(h->d_act); cudaFree(h->d_obs); cudaFree(h->d_rew); cudaFree(h->d_done); cudaFree(h->d_ticks); cudaFree(h->d_mask);
        cudaStreamDestroy(h->hstream);
    }
    if (h->ev_valid) cudaEventDestroy(h->ev_dev);
    for (int c = 0; c < h->n_ev_chunk; c++) cudaEventDestroy(h->ev_chunk[c]);
    if (h->exact) snk_exact_release();
    cudaFree(h->T); cudaFree(h->state); cudaFree(h->counters); cudaFree(h->bucket); cudaFree(h->order); cudaFree(h->split_buf); cudaFree(h->roll_queue); cudaFree(h->tgt);
    cudaFree(h->man_cache); cudaFree(h->man_scratch); cudaFree(h->man_bad);
    delete h;
    return 0;
}

int64_t snk_num_envs(const snk_handle* h) { return h ? h->n : 0; }
int snk_action_dim(const snk_handle* h) { return h ? h->P.actdim : 0; }
int snk_device(const snk_handle* h) { return h ? h->device : -1; }
int64_t snk_launch_count(const snk_handle* h) { return h ? h->launches : 0; }

int snk_reset(snk_handle* h, const uint8_t* mask_dev, float* obs_dev, void* stream) {
    if (!h) return fail(SNK_E_ARG, "snk_reset: null handle%s");
    if (obs_dev && !aligned16(obs_dev)) return fail(SNK_E_ARG, "snk_reset: obs must be 16-byte aligned%s");
    CU(cudaSetDevice(h->device));
    CU(snk_launch_reset(h->P, h->state, mask_dev, obs_dev, h->n, 0, (cudaStream_t)stream));
    h->launches++;
    mark_device_work(h, (cudaStream_t)stream);
    return 0;
}

int snk_observe(snk_handle* h, float* obs_dev, void* stream) {
    if (!h || !obs_dev) return fail(SNK_E_ARG, "snk_observe: null pointer%s");
    if (!aligned16(obs_dev)) return fail(SNK_E_ARG, "snk_observe: obs must be 16-byte aligned%s");
    CU(cudaSetDevice(h->device));
    CU(snk_launch_reset(h->P, h->state, nullptr, obs_dev, h->n, 2, (cudaStream_t)stream));
    h->launches++;
    mark_device_work(h, (cudaStream_t)stream); // a later *_host call must not overwrite the state under this read
    return 0;
}

int snk_step(snk_handle* h, const float* actions_dev, float* obs_dev, float* rew_dev, uint8_t* done_dev, int32_t* ticks_dev, void* stream) {
    if (!h || !actions_dev || !obs_dev || !rew_dev || !done_dev) return fail(SNK_E_ARG, "snk_step: null pointer%s");
    if (!aligned16(actions_dev) || !aligned16(obs_dev)) return fail(SNK_E_ARG, "snk_step: actions and obs must be 16-byte aligned%s");
    CU(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    CU(cudaMemsetAsync(h->counters, 0, NCOUNTERS * sizeof(unsigned long long), st));
    CU(launch_step(h, actions_dev, obs_dev, rew_dev, done_dev, ticks_dev, st));
    return 0;
}

int snk_step_trace(snk_handle* h, const float* actions_dev, float* obs_dev, float* rew_dev, uint8_t* done_dev, int32_t* ticks_dev,
                   float* tick_obs_dev, float* tick_links_dev, void* stream) {
    if (!h || !actions_dev || !obs_dev || !rew_dev || !done_dev || !ticks_dev)
        return fail(SNK_E_ARG, "snk_step_trace: null pointer (ticks_dev is required: it says how many trace rows are valid)%s");
    if (!aligned16(actions_dev) || !aligned16(obs_dev)) return fail(SNK_E_ARG, "snk_step_trace: actions and obs must be 16-byte aligned%s");
    CU(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    CU(cudaMemsetAsync(h->counters, 0, NCOUNTERS * sizeof(unsigned long long), st));
    if (h->manifold) CU(snk_man_launch_step_trace(h->P, h->state, h->tgt, h->man_cache, h->man_scratch, h->man_warm, actions_dev, obs_dev, rew_dev, done_dev,
                                                  ticks_dev, h->counters, h->n, tick_obs_dev, tick_links_dev, st));
    else if (h->exact) CU(snk_exact_launch_step_trace(h->P, h->state, h->tgt, actions_dev, obs_dev, rew_dev, done_dev, ticks_dev, h->counters, h->n, tick_obs_dev,
                                                 tick_links_dev, st));
    else CU(snk_pgs_launch_step(h->T, h->P, h->state, actions_dev, obs_dev, rew_dev, done_dev, ticks_dev, h->counters, h->n, st, tick_obs_dev,
                                tick_links_dev));
    h->launches++;
    mark_device_work(h, st);
    return 0;
}

int snk_rollout_linear(snk_handle* h, const float* weights_dev, const float* mean_dev, const float* inv_std_dev, const float* noise_dev,
                       int32_t n_steps, float* returns_dev, float* obs_trace_dev, void* stream) {
    if (!h || !weights_dev || !returns_dev || n_steps < 1) return fail(SNK_E_ARG, "snk_rollout_linear: bad argument%s");
    if (!h->exact) return fail(SNK_E_ARG, "snk_rollout_linear: only with the exact motor solver (motor force = inf, kd = 1)%s");
    if (!aligned16(weights_dev)) return fail(SNK_E_ARG, "snk_rollout_linear: weights must be 16-byte aligned%s");
    CU(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (h->manifold) { // one environment per thread for the whole rollout: no ready queue, no hand-out order
        CU(cudaMemsetAsync(h->counters, 0, NCOUNTERS * sizeof(unsigned long long), st));
        CU(snk_man_launch_rollout(h->P, h->state, h->tgt, h->man_cache, h->man_scratch, h->man_warm, weights_dev, mean_dev, inv_std_dev, noise_dev, n_steps,
                                  returns_dev, obs_trace_dev, h->counters, h->n, st));
        h->launches++;
        mark_device_work(h, st);
        return 0;
    }
    const size_t qlen = (size_t)h->n * (size_t)(n_steps > 1 ? n_steps - 1 : 1);
    if (qlen > h->roll_queue_len) { // grow the ready queue (first call, or a longer rollout than before)
        CU(cudaStreamSynchronize(st));
        cudaFree(h->roll_queue); h->roll_queue = nullptr; h->roll_queue_len = 0;
        CU(cudaMalloc(&h->roll_queue, qlen * sizeof(int32_t)));
        h->roll_queue_len = qlen;
    }
    CU(cudaMemsetAsync(h->counters, 0, NCOUNTERS * sizeof(unsigned long long), st));
    CU(cudaMemsetAsync(h->roll_queue, 0xff, qlen * sizeof(int32_t), st));        // -1: not pushed yet
    CU(cudaMemsetAsync(h->order, 0, (size_t)h->n * sizeof(int32_t), st));          // env-steps done (the step kernel's order[] is rebuilt per step)
    CU(snk_exact_launch_rollout(h->P, h->state, h->tgt, weights_dev, mean_dev, inv_std_dev, noise_dev, n_steps, returns_dev, obs_trace_dev, h->roll_queue,
                                h->order, h->counters, h->n, st));
    h->launches++;
    mark_device_work(h, st);
    return 0;
}

int snk_set_manifold(snk_handle* h, int on, double warm_start) {
    if (!h) return fail(SNK_E_ARG, "snk_set_manifold: null handle%s");
    if (on && !h->exact) return fail(SNK_E_ARG, "snk_set_manifold: only with the exact motor solver (motor force = inf, kd = 1)%s");
    if (!(warm_start >= 0.0)) return fail(SNK_E_ARG, "snk_set_manifold: warm_start must be >= 0%s");
    CU(cudaSetDevice(h->device));
    CU(cudaDeviceSynchronize()); // the caches of a step in flight are about to be cleared or freed
    if (!on) {
        cudaFree(h->man_cache); cudaFree(h->man_scratch); cudaFree(h->man_bad);
        h->man_cache = nullptr; h->man_scratch = nullptr; h->man_bad = nullptr; h->manifold = false;
        return 0;
    }
    const size_t cache_bytes = (size_t)h->n * snk_man_cache_floats() * sizeof(float);
    if (!h->man_cache) {
        if (cudaMalloc(&h->man_cache, cache_bytes) != cudaSuccess || cudaMalloc(&h->man_scratch, snk_man_scratch_bytes()) != cudaSuccess ||
            cudaMalloc(&h->man_bad, sizeof(unsigned long long)) != cudaSuccess) {
            cudaGetLastError();
            cudaFree(h->man_cache); cudaFree(h->man_scratch); cudaFree(h->man_bad);
            h->man_cache = nullptr; h->man_scratch = nullptr; h->man_bad = nullptr; h->manifold = false;
            return fail(SNK_E_NOMEM, "snk_set_manifold: out of device memory (4 224 B per environment + 388 MB of row tables)%s");
        }
    }
    CU(cudaMemset(h->man_cache, 0, cache_bytes)); // empty caches, like a freshly loaded world
    h->man_warm = (float)warm_start;
    h->manifold = true;
    return 0;
}

int snk_get_manifold_cache(snk_handle* h, float* cache_dev, void* stream) {
    if (!h || !cache_dev) return fail(SNK_E_ARG, "snk_get_manifold_cache: null pointer%s");
    if (!h->manifold) return fail(SNK_E_ARG, "snk_get_manifold_cache: persistent manifolds are off (snk_set_manifold)%s");
    CU(cudaSetDevice(h->device));
    CU(cudaMemcpyAsync(cache_dev, h->man_cache, (size_t)h->n * SNK_MAN_STRIDE * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    mark_device_work(h, (cudaStream_t)stream);
    return 0;
}

int snk_set_manifold_cache(snk_handle* h, const float* cache_dev, void* stream) {
    if (!h || !cache_dev) return fail(SNK_E_ARG, "snk_set_manifold_cache: null pointer%s");
    if (!h->manifold) return fail(SNK_E_ARG, "snk_set_manifold_cache: persistent manifolds are off (snk_set_manifold)%s");
    CU(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long bad = 0;
    CU(cudaMemsetAsync(h->man_bad, 0, sizeof bad, st));
    CU(snk_man_launch_check(cache_dev, h->n, h->man_bad, st));
    h->launches++;
    CU(cudaMemcpyAsync(&bad, h->man_bad, sizeof bad, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (bad) {
        static thread_local char msg[128];
        snprintf(msg, sizeof msg, "%llu environment(s) with a point count that is not an integer in 0..4", bad);
        return fail(SNK_E_ARG, "snk_set_manifold_cache: %s; the caches are unchanged", msg);
    }
    CU(cudaMemcpyAsync(h->man_cache, cache_dev, (size_t)h->n * SNK_MAN_STRIDE * sizeof(float), cudaMemcpyDeviceToDevice, st));
    mark_device_work(h, st);
    return 0;
}

int snk_clear_manifold(snk_handle* h, const uint8_t* mask_dev, void* stream) {
    if (!h) return fail(SNK_E_ARG, "snk_clear_manifold: null handle%s");
    if (!h->manifold) return fail(SNK_E_ARG, "snk_clear_manifold: persistent manifolds are off (snk_set_manifold)%s");
    CU(cudaSetDevice(h->device));
    CU(snk_man_launch_clear(h->man_cache, mask_dev, h->n, (cudaStream_t)stream));
    h->launches++;
    mark_device_work(h, (cudaStream_t)stream);
    return 0;
}

int snk_gae(int device, const float* rewards_dev, const uint8_t* dones_dev, const float* values_dev, const float* next_value_dev, double gamma,
            double tau, float* returns_dev, float* advantages_dev, int32_t n_steps, int64_t n_envs, void* stream) {
    if (!rewards_dev || !dones_dev || !values_dev || !next_value_dev || !returns_dev) return fail(SNK_E_ARG, "snk_gae: null pointer%s");
    if (n_steps < 1 || n_envs < 1) return fail(SNK_E_ARG, "snk_gae: n_steps and n_envs must be positive%s");
    CU(cudaSetDevice(device));
    CU(snk_launch_gae(rewards_dev, dones_dev, values_dev, next_value_dev, (float)gamma, (float)tau, returns_dev, advantages_dev, n_steps, n_envs,
                      (cudaStream_t)stream));
    return 0;
}

int snk_tick(snk_handle* h, const float* targets_dev, int32_t n_ticks, void* stream) {
    if (!h || !targets_dev || n_ticks < 0) return fail(SNK_E_ARG, "snk_tick: bad argument%s");
    if (h->manifold) return fail(SNK_E_ARG, "snk_tick: not available with persistent manifolds (snk_set_manifold); use snk_step%s");
    CU(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    CU(cudaMemsetAsync(h->counters, 0, NCOUNTERS * sizeof(unsigned long long), st));
    if (h->exact) CU(snk_exact_launch_tick(h->P, h->state, targets_dev, h->counters, h->n, n_ticks, st));
    else CU(snk_pgs_launch_tick(h->T, h->P, h->state, targets_dev, h->counters, h->n, n_ticks, st));
    h->launches++;
    mark_device_work(h, st);
    return 0;
}

static int ensure_stream(snk_handle* h) {
    if (!h->hstream) CU(cudaStreamCreateWithFlags(&h->hstream, cudaStreamNonBlocking));
    return 0;
}

static int ensure_staging(snk_handle* h) {
    if (h->staged) return 0;
    size_t n = (size_t)h->n;
    int rc0 = ensure_stream(h);
    if (rc0) return rc0;
    CU(cudaMallocHost(&h->h_act, n * NJ * sizeof(float)));
    CU(cudaMallocHost(&h->h_obs, n * SNK_OBS_DIM * sizeof(float)));
    CU(cudaMallocHost(&h->h_rew, n * sizeof(float)));
    CU(cudaMallocHost(&h->h_done, n));
    CU(cudaMallocHost(&h->h_mask, n));
    CU(cudaMallocHost(&h->h_ticks, n * sizeof(int32_t)));
    CU(cudaMalloc(&h->d_act, n * NJ * sizeof(float)));
    CU(cudaMalloc(&h->d_obs, n * SNK_OBS_DIM * sizeof(float)));
    CU(cudaMalloc(&h->d_rew, n * sizeof(float)));
    CU(cudaMalloc(&h->d_done, n));
    CU(cudaMalloc(&h->d_mask, n));
    CU(cudaMalloc(&h->d_ticks, n * sizeof(int32_t)));
    h->staged = true;
    return 0;
}

// true when `p` is page-locked host memory known to CUDA (cudaMallocHost / cudaHostRegister / torch pinned):
// such a buffer is the DMA source/target itself and needs no staging copy
static bool is_pinned(const void* p, void** dev = nullptr) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    if (dev) *dev = a.devicePointer;
    return a.type == cudaMemoryTypeHost;
}

// SNK_HOST_ZEROCOPY=0 disables the mapped-host-memory path of snk_step_host (ablation)
static bool zero_copy_enabled() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("SNK_HOST_ZEROCOPY"); v = !(e && e[0] == '0'); }
    return v != 0;
}

int snk_step_host(snk_handle* h, const float* actions_host, float* obs_host, float* rew_host, uint8_t* done_host, int32_t* ticks_host) {
    if (!h || !actions_host || !obs_host || !rew_host || !done_host) return fail(SNK_E_ARG, "snk_step_host: null pointer%s");
    CU(cudaSetDevice(h->device));
    void *da = nullptr, *dob = nullptr, *dr = nullptr, *dd = nullptr, *dt = nullptr;
    const bool pa = is_pinned(actions_host, &da), po = is_pinned(obs_host, &dob), pr = is_pinned(rew_host, &dr), pd = is_pinned(done_host, &dd),
               pt = ticks_host && is_pinned(ticks_host, &dt);
    if (zero_copy_enabled() && pa && po && pr && pd && (!ticks_host || pt) && da && dob && dr && dd && (!ticks_host || dt) && aligned16(da) &&
        aligned16(dob)) { // (a misaligned pinned buffer takes the staged path below)
        // Every caller buffer is page-locked and mapped: the kernel reads the 32 B action row of an environment straight from
        // host memory when a lane takes it and posts the observation row / reward / done / ticks straight back over PCIe when
        // the environment finishes, spread over the whole launch -- no copy before or after the kernel.
        int rc0 = ensure_stream(h);
        if (rc0) return rc0;
        wait_device_work(h);
        cudaStream_t zs = h->hstream;
        CU(cudaMemsetAsync(h->counters, 0, NCOUNTERS * sizeof(unsigned long long), zs));
        CU(launch_step(h, (const float*)da, (float*)dob, (float*)dr, (uint8_t*)dd, (int32_t*)dt, zs));
        CU(cudaStreamSynchronize(zs));
        return 0;
    }
    int rc = ensure_staging(h);
    if (rc) return rc;
    wait_device_work(h);
    size_t n = (size_t)h->n, na = n * h->P.actdim * sizeof(float);
    cudaStream_t st = h->hstream;
    // pageable caller buffers go through the handle's pinned staging buffers; pinned ones are DMA sources / targets themselves
    if (!pa) memcpy(h->h_act, actions_host, na);
    CU(cudaMemcpyAsync(h->d_act, pa ? actions_host : h->h_act, na, cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(h->counters, 0, NCOUNTERS * sizeof(unsigned long long), st));
    CU(launch_step(h, h->d_act, h->d_obs, h->d_rew, h->d_done, h->d_ticks, st));
    CU(cudaMemcpyAsync(po ? obs_host : h->h_obs, h->d_obs, n * SNK_OBS_DIM * sizeof(float), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(pr ? rew_host : h->h_rew, h->d_rew, n * sizeof(float), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(pd ? done_host : h->h_done, h->d_done, n, cudaMemcpyDeviceToHost, st));
    if (ticks_host) CU(cudaMemcpyAsync(pt ? ticks_host : h->h_ticks, h->d_ticks, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (!po) memcpy(obs_host, h->h_obs, n * SNK_OBS_DIM * sizeof(float));
    if (!pr) memcpy(rew_host, h->h_rew, n * sizeof(float));
    if (!pd) memcpy(done_host, h->h_done, n);
    if (ticks_host && !pt) memcpy(ticks_host, h->h_ticks, n * sizeof(int32_t));
    return 0;
}

// The call the reference's numpy callers make (ppo/train.py:122, ars/train.py:99): float64 arrays in and out, as
// SubprocVecEnv.step returns them.  Actions are narrowed into the handle's page-locked buffer, the kernel runs on the
// mapped page-locked buffers (see snk_step_host), and the results are widened into the caller's arrays by a few threads.
// SNK_HOST_FLAGS=0: snk_step_host_f64 takes the chunk-pipelined path even where the flag-driven one is available (ablation)
static bool row_flags_enabled() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("SNK_HOST_FLAGS"); v = !(e && e[0] == '0'); }
    return v != 0;
}

// snk_step_host_f64, flag-driven: ONE launch for the whole batch, writing into the handle's mapped page-locked buffers; the kernel
// posts an environment's ticks word last, behind a system-wide fence (HandOut::flag_rows), and the host threads -- each owning a
// contiguous range of environments -- widen every row into the caller's float64 arrays as soon as its ticks word turns up, while
// the launch is still running.  Only the narrowing of the actions (before the launch) and the rows of the last few lanes to finish
// are not hidden behind the kernel, and the batch is not cut into smaller launches (each of which would pay its own last wave).
static int step_host_f64_flags(snk_handle* h, const double* actions_host, double* obs_host, double* rew_host, uint8_t* done_host, int32_t* ticks_host) {
    const size_t n = (size_t)h->n, ad = (size_t)h->P.actdim;
    cudaStream_t st = h->hstream;
    float* ha = h->h_act;
    int32_t* ht = h->h_ticks;
    const size_t grain = 4096; // environments; below it the calling thread works alone
    parallel_chunks(n, [=](size_t b, size_t e) {
        for (size_t i = b * ad; i < e * ad; i++) ha[i] = (float)actions_host[i];
        for (size_t i = b; i < e; i++) ht[i] = -1; // "row not there yet" (tick counts are 0...41)
    }, grain);
    CU(cudaMemsetAsync(h->counters, 0, NCOUNTERS * sizeof(unsigned long long), st));
    CU(launch_step(h, h->h_act, h->h_obs, h->h_rew, h->h_done, h->h_ticks, st, 0, -1, 1));
    RowSink sink;
    sink.obs_src = h->h_obs; sink.rew_src = h->h_rew; sink.done_src = h->h_done; sink.ticks_src = h->h_ticks;
    sink.obs = obs_host; sink.rew = rew_host; sink.done = done_host; sink.ticks = ticks_host; sink.obs_dim = SNK_OBS_DIM;
    static int nt = -1; // SNK_HOST_NT=0: plain stores for the widened rows (ablation)
    if (nt < 0) { const char* e = getenv("SNK_HOST_NT"); nt = !(e && e[0] == '0'); }
    sink.stream = nt != 0;
    std::atomic<int> launch_state{ROWS_IN_FLIGHT};
    std::atomic<int> sync_error{(int)cudaSuccess};
    static int prefault = -1;
    if (prefault < 0) { const char* e = getenv("SNK_HOST_PREFAULT"); prefault = !(e && e[0] == '0'); }
    parallel_chunks(n, [&](size_t b, size_t e) {
        rows_widen_as_posted(sink, b, e, launch_state, /* leader: the calling thread, which has the CUDA context */ b == 0, prefault && (e - b) >= grain,
            [&]() { const cudaError_t q = cudaStreamQuery(st); if (q == cudaSuccess) return 1; if (q == cudaErrorNotReady) return 0; sync_error.store((int)q); return -1; },
            [&]() { const cudaError_t q = cudaStreamSynchronize(st); if (q == cudaSuccess) return 1; sync_error.store((int)q); return -1; });
    }, grain);
    const cudaError_t e_sync = cudaStreamSynchronize(st);
    if (launch_state.load() == ROWS_LAUNCH_FAILED || e_sync != cudaSuccess)
        return fail(SNK_E_CUDA, "snk_step_host_f64: the env-step launch failed: %s", cudaGetErrorString(e_sync != cudaSuccess ? e_sync : (cudaError_t)sync_error.load()));
    if (launch_state.load() == ROWS_MISSING) return fail(SNK_E_CUDA, "snk_step_host_f64: the launch finished without posting every row%s");
    return 0;
}

int snk_step_host_f64(snk_handle* h, const double* actions_host, double* obs_host, double* rew_host, uint8_t* done_host, int32_t* ticks_host) {
    if (!h || !actions_host || !obs_host || !rew_host || !done_host) return fail(SNK_E_ARG, "snk_step_host_f64: null pointer%s");
    CU(cudaSetDevice(h->device));
    int rc = ensure_staging(h);
    if (rc) return rc;
    wait_device_work(h);
    if (zero_copy_enabled() && row_flags_enabled() && h->exact && !h->manifold && snk_exact_row_flags_supported())
        return step_host_f64_flags(h, actions_host, obs_host, rew_host, done_host, ticks_host);
    const size_t n = (size_t)h->n, ad = (size_t)h->P.actdim;
    cudaStream_t st = h->hstream;
    // (Kernels without row flags -- Bullet-order rows, persistent manifolds, the ablation layouts.)  The batch goes through in a few chunks of environments, pipelined: while the GPU steps chunk c the host threads narrow the
    // actions of chunk c + 1, and while it steps chunk c + 1 they widen the results of chunk c into the caller's arrays -- only the
    // first narrowing and the last widening are not hidden behind the kernel (SNK_HOST_CHUNKS, default 4 from 2^18 environments).
    static int cfg_chunks = -1;
    if (cfg_chunks < 0) { const char* e = getenv("SNK_HOST_CHUNKS"); cfg_chunks = (e && atoi(e) >= 1 && atoi(e) <= 16) ? atoi(e) : 4; }
    const int chunks = (n >= ((size_t)1 << 18)) ? cfg_chunks : 1;
    if (h->n_ev_chunk < chunks) {
        for (int c = h->n_ev_chunk; c < chunks; c++) CU(cudaEventCreateWithFlags(&h->ev_chunk[c], cudaEventDisableTiming));
        h->n_ev_chunk = chunks;
    }
    const bool zc = zero_copy_enabled();
    CU(cudaMemsetAsync(h->counters, 0, NCOUNTERS * sizeof(unsigned long long), st));
    size_t lo[17]; // chunk boundaries, multiples of 32 environments (row pointers stay 16-byte aligned)
    for (int c = 0; c <= chunks; c++) {
        size_t x = (n * (size_t)c / (size_t)chunks + 31) / 32 * 32;
        lo[c] = (c == chunks || x > n) ? n : x;
    }
    for (int c = 0; c < chunks; c++) {
        const size_t b = lo[c], e = lo[c + 1];
        if (e <= b) { CU(cudaEventRecord(h->ev_chunk[c], st)); continue; }
        float* ha = h->h_act;
        parallel_chunks((e - b) * ad, [=](size_t i0, size_t i1) { for (size_t i = b * ad + i0; i < b * ad + i1; i++) ha[i] = (float)actions_host[i]; });
        if (c > 0) { // the hand-out words are per launch ([7] is a statistic of the manifold kernel: it accumulates like [0..3])
            CU(cudaMemsetAsync(h->counters + 4, 0, 3 * sizeof(unsigned long long), st));
            CU(cudaMemsetAsync(h->counters + 8, 0, (NCOUNTERS - 8) * sizeof(unsigned long long), st));
        }
        if (zc) {
            CU(launch_step(h, h->h_act + b * ad, h->h_obs + b * SNK_OBS_DIM, h->h_rew + b, h->h_done + b, h->h_ticks + b, st, (int64_t)b, (int64_t)(e - b)));
        } else {
            CU(cudaMemcpyAsync(h->d_act + b * ad, h->h_act + b * ad, (e - b) * ad * sizeof(float), cudaMemcpyHostToDevice, st));
            CU(launch_step(h, h->d_act + b * ad, h->d_obs + b * SNK_OBS_DIM, h->d_rew + b, h->d_done + b, h->d_ticks + b, st, (int64_t)b, (int64_t)(e - b)));
            CU(cudaMemcpyAsync(h->h_obs + b * SNK_OBS_DIM, h->d_obs + b * SNK_OBS_DIM, (e - b) * SNK_OBS_DIM * sizeof(float), cudaMemcpyDeviceToHost, st));
            CU(cudaMemcpyAsync(h->h_rew + b, h->d_rew + b, (e - b) * sizeof(float), cudaMemcpyDeviceToHost, st));
            CU(cudaMemcpyAsync(h->h_done + b, h->d_done + b, e - b, cudaMemcpyDeviceToHost, st));
            CU(cudaMemcpyAsync(h->h_ticks + b, h->d_ticks + b, (e - b) * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        }
        CU(cudaEventRecord(h->ev_chunk[c], st));
    }
    prefault_output(obs_host, n * SNK_OBS_DIM * sizeof(double)); // the GPU is busy with the first chunk for tens of milliseconds
    prefault_output(rew_host, n * sizeof(double));
    for (int c = 0; c < chunks; c++) {
        const size_t b = lo[c], e = lo[c + 1];
        CU(cudaEventSynchronize(h->ev_chunk[c]));
        if (e <= b) continue;
        const float* ho = h->h_obs;
        parallel_chunks((e - b) * SNK_OBS_DIM, [=](size_t i0, size_t i1) { for (size_t i = b * SNK_OBS_DIM + i0; i < b * SNK_OBS_DIM + i1; i++) obs_host[i] = (double)ho[i]; });
        const float* hr = h->h_rew;
        parallel_chunks(e - b, [=](size_t i0, size_t i1) { for (size_t i = b + i0; i < b + i1; i++) rew_host[i] = (double)hr[i]; });
        memcpy(done_host + b, h->h_done + b, e - b);
        if (ticks_host) memcpy(ticks_host + b, h->h_ticks + b, (e - b) * sizeof(int32_t));
    }
    CU(cudaStreamSynchronize(st));
    return 0;
}

int snk_reset_host(snk_handle* h, const uint8_t* mask_host, float* obs_host) {
    if (!h) return fail(SNK_E_ARG, "snk_reset_host: null handle%s");
    CU(cudaSetDevice(h->device));
    int rc = ensure_staging(h);
    if (rc) return rc;
    wait_device_work(h);
    size_t n = (size_t)h->n;
    cudaStream_t st = h->hstream;
    if (mask_host) {
        memcpy(h->h_mask, mask_host, n);
        CU(cudaMemcpyAsync(h->d_mask, h->h_mask, n, cudaMemcpyHostToDevice, st));
    }
    CU(snk_launch_reset(h->P, h->state, mask_host ? h->d_mask : nullptr, obs_host ? h->d_obs : nullptr, h->n, 0, st));
    h->launches++;
    if (obs_host) CU(cudaMemcpyAsync(h->h_obs, h->d_obs, n * SNK_OBS_DIM * sizeof(float), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (obs_host) memcpy(obs_host, h->h_obs, n * SNK_OBS_DIM * sizeof(float));
    return 0;
}

int snk_self_clearance(snk_handle* h, float* clearance_dev, void* stream) {
    if (!h || !clearance_dev) return fail(SNK_E_ARG, "snk_self_clearance: null pointer%s");
    CU(cudaSetDevice(h->device));
    CU(snk_launch_self_clearance(h->T, h->state, clearance_dev, h->n, (cudaStream_t)stream));
    h->launches++;
    mark_device_work(h, (cudaStream_t)stream);
    return 0;
}

int snk_get_state(snk_handle* h, float* state_dev, void* stream) {
    if (!h || !state_dev) return fail(SNK_E_ARG, "snk_get_state: null pointer%s");
    CU(cudaSetDevice(h->device));
    CU(cudaMemcpyAsync(state_dev, h->state, (size_t)h->n * SNK_STATE_STRIDE * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    mark_device_work(h, (cudaStream_t)stream);
    return 0;
}

int snk_set_state(snk_handle* h, const float* state_dev, void* stream) {
    if (!h || !state_dev) return fail(SNK_E_ARG, "snk_set_state: null pointer%s");
    CU(cudaSetDevice(h->device));
    CU(cudaMemcpyAsync(h->state, state_dev, (size_t)h->n * SNK_STATE_STRIDE * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    mark_device_work(h, (cudaStream_t)stream);
    return 0;
}

int snk_last_counters(snk_handle* h, int64_t out[4]) {
    if (!h || !out) return fail(SNK_E_ARG, "snk_last_counters: null pointer%s");
    CU(cudaSetDevice(h->device));
    unsigned long long tmp[4];
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(tmp, h->counters, sizeof tmp, cudaMemcpyDeviceToHost));
    for (int k = 0; k < 4; k++) out[k] = (int64_t)tmp[k];
    return 0;
}

int snk_manifold_stats(snk_handle* h, int64_t out[2]) {
    if (!h || !out) return fail(SNK_E_ARG, "snk_manifold_stats: null pointer%s");
    if (!h->manifold) return fail(SNK_E_ARG, "snk_manifold_stats: persistent manifolds are off (snk_set_manifold)%s");
    CU(cudaSetDevice(h->device));
    unsigned long long tmp[8];
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(tmp, h->counters, sizeof tmp, cudaMemcpyDeviceToHost));
    out[0] = (int64_t)tmp[7]; out[1] = (int64_t)tmp[0];
    return 0;
}

} // extern "C"
