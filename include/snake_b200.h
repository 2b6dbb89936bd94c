/*
 * snake_b200.h -- C ABI of the B200-native batched snake simulator.
 *
 * This is the drop-in boundary for the one hot path of vinits5/bullet-envs ("snakeRL"):
 * SnakeGymEnv.step() = clip -> Snake.step (variable tick loop of PyBullet stepSimulation)
 * -> observation -> reward -> termination -> auto-reset, for N independent environments.
 * Everything behind these entry points is hand-written sm_100a CUDA; there is no CPU
 * fallback in this library (the CPU restatement lives in oracle/ and is test-only).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no C++/torch types.
 *   - every function returns 0 on success or a negative SNK_E_* code; the message is
 *     available from snk_last_error() (thread-local, never NULL).
 *   - pointers named *_dev are device pointers on the handle's device, owned by the caller
 *     (torch allocates them); pointers named *_host are host pointers.  The handle owns only
 *     its internal state array and constant tables.  snk_step() allocates nothing.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream); all work is
 *     enqueued on it, no hidden synchronisation except in the *_host entry points.  snk_step, snk_reset, snk_tick and snk_gae
 *     allocate nothing and never synchronise, so they may be captured into a CUDA graph (synchronise after replaying such a
 *     graph before calling a *_host entry point on the same handle).
 *   - layouts are row-major fp32: actions [N, act_dim], obs [N, 56], reward [N], done [N] u8.
 *   - actions, obs and weights pointers must be 16-byte aligned (rows move as 16-byte vectors); anything a device or
 *     pinned allocator returns is.  A misaligned pointer is refused with SNK_E_ARG (snk_step_host stages it instead).
 *
 * Reference interfaces replaced (file:line under /root/reference):
 *   snk_create      <- SnakeGymEnv.__init__ (SnakeGymEnv.py:5-26), Snake.__init__/reset(hardReset=True)
 *                      /setDynamics (snake.py:14-32, 86-107), SubprocVecEnv.__init__
 *                      (ppo/multiprocessing_env.py:97-117)
 *   snk_destroy     <- SubprocVecEnv.close (ppo/multiprocessing_env.py:140-150)
 *   snk_reset       <- SubprocVecEnv.reset (ppo/multiprocessing_env.py:130-133) ->
 *                      SnakeGymEnv.reset (SnakeGymEnv.py:28-31) -> Snake.reset(False) (snake.py:86-101,119-127)
 *   snk_step        <- SubprocVecEnv.step_async/step_wait + worker auto-reset
 *                      (ppo/multiprocessing_env.py:7-16,119-128) -> SnakeGymEnv.step (SnakeGymEnv.py:33-50)
 *                      -> Snake.step (snake.py:274-306) -> pybullet.setJointMotorControlArray +
 *                      stepSimulation (snake.py:219-225,286) + getObservation (snake.py:209-217)
 *   snk_step_host   <- the same call made with numpy arrays (ppo/train.py:122, ars/train.py:99)
 *   snk_tick        <- raw setJointMotorControlArray + stepSimulation loop of the gait script
 *                      (snake_gait_test.py:96-104)
 *   snk_step_trace  <- the same step in mode='test': Snake.step's per-tick step_internal_observations / link_positions
 *                      (snake.py:275-278,292-293,138-146) returned through info (SnakeGymEnv.py:43-44; read by ppo/test.py:93-105)
 *   snk_observe     <- Snake.getObservation (snake.py:209-217)
 *   snk_set_manifold <- the contact model of pybullet.stepSimulation itself (persistent manifolds, warm starting): snake.py:92-93,286
 *   snk_rollout_linear <- ARS rollout with a linear policy per environment: ars/train.py:74-116 (test_envs)
 *                      with policy() = W x (ars/train.py:40-41), normalisation (ars/train.py:152-169, statistics
 *                      frozen for the rollout) and the state noise of ars/train.py:81,90 supplied by the caller
 *   snk_self_clearance <- loadURDF(..., flags=URDF_USE_SELF_COLLISION) (snake.py:93): the pairs Bullet would test
 *   snk_get_state / snk_set_state <- resetBasePositionAndOrientation / resetJointState
 *                      (snake.py:119-127) generalised to arbitrary states (parity harness)
 */
#ifndef SNAKE_B200_H
#define SNAKE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SNK_NB 17            /* rigid bodies after merging the 33 fixed joints        */
#define SNK_NJ 16            /* revolute joints = motors (snake.py:16)                 */
#define SNK_NC 32            /* collision cylinders (snake.urdf: 2 per module)         */
#define SNK_NDOF 22          /* 6 floating-base + 16 joint velocities                  */
#define SNK_OBS_DIM 56       /* snake.py:163-164                                       */
#define SNK_STATE_STRIDE 64  /* floats per environment in the state array (256 B)      */

/* offsets inside one environment's state record (fp32 on device, fp64 in the oracle) */
#define SNK_S_POS 0          /* base (kdl_dummy_root) origin, world                    */
#define SNK_S_QUAT 3         /* base orientation xyzw                                  */
#define SNK_S_VEL 7          /* base linear velocity, world                            */
#define SNK_S_OMEGA 10       /* base angular velocity, world                           */
#define SNK_S_Q 13           /* 16 joint angles                                        */
#define SNK_S_QD 29          /* 16 joint velocities                                    */
#define SNK_S_TAU 45         /* 16 last applied motor torques (persist over soft reset, Q9) */
#define SNK_S_FZ 61          /* last joint-0 reaction Fz (persists over soft reset)    */
#define SNK_S_RET 62         /* running return of the current episode                  */
#define SNK_S_LEN 63         /* env-steps taken in the current episode                 */

#define SNK_E_ARG (-1)
#define SNK_E_CUDA (-2)
#define SNK_E_NOMEM (-3)
#define SNK_E_NODEV (-4)

/* Merged rigid-body model of snake.urdf (built by bullet_envs_b200/urdf_model.py). */
typedef struct snk_model {
    double joint_R0[SNK_NJ][9];    /* joint frame (q=0) axes in parent-body frame, row-major */
    double joint_t[SNK_NJ][3];     /* joint origin in parent-body frame                     */
    double joint_axis[SNK_NJ][3];  /* rotation axis in the child frame                      */
    double joint_damping[SNK_NJ];  /* URDF <dynamics damping>, explicit torque -d*qd        */
    double body_mass[SNK_NB];
    double body_com[SNK_NB][3];    /* in body frame                                         */
    double body_inertia[SNK_NB][9];/* about the COM, body-frame axes, row-major             */
    double cyl_center[SNK_NC][3];  /* body frame                                            */
    double cyl_axis[SNK_NC][3];    /* unit, body frame                                      */
    double cyl_fric_R[SNK_NC][9];  /* collision-link axes in body frame (anisotropic friction) */
    double cyl_radius[SNK_NC];
    double cyl_halflen[SNK_NC];
    double cyl_end[SNK_NC];        /* +1/-1: which rim carries the contact point            */
    double cyl_margin[SNK_NC];     /* collision margin (0.001)                              */
    double cyl_break[SNK_NC];      /* contact breaking threshold                            */
    double height_pt[SNK_NB][3];   /* points averaged by checkSnakeHeight, body frame       */
    double fz_axis[3];             /* z axis of URDF link `base` in body-0 frame            */
    double root_mass;              /* mass of kdl_dummy_root (joint-0 reaction force)       */
    int32_t cyl_body[SNK_NC];
    int32_t height_body[SNK_NB];
} snk_model;

/* Task + solver parameters.  The defaults are the reference's task settings and PyBullet's documented world defaults (DESIGN.md
 * section 3).  The tick underneath is this project's restatement of Bullet, not Bullet itself -- one contact point per cylinder and
 * no persistent manifold (D1), no joint-limit / self-collision rows (D3: limit rows are a switch of the Bullet-order kernels,
 * snk_set_joint_limits, off by default), and with motor_solver = 2 the motor rows imposed exactly
 * instead of relaxed by 50 sweeps (D4); DESIGN.md section 4 measures each.  No PyBullet was available to pin it against. */
typedef struct snk_params {
    double dt;                  /* 1/240: Snake.setTimeSteps is never called (snake.py:271-272) */
    double gravity[3];          /* (0,0,-9.8) snake.py:8,91                                     */
    double motor_kp;            /* 0.1  PyBullet POSITION_CONTROL default                      */
    double motor_kd;            /* 1.0  PyBullet POSITION_CONTROL default                      */
    double motor_max_force;     /* inf  snake.py:26-27                                          */
    double scaling_factor;      /* pi/6 snake.py:41,63                                          */
    double alpha, beta, gamma;  /* 1, 0.01, 0.1  SnakeGymEnv.py:14-16                           */
    double energy_dt;           /* 0.01 snake.py:9,339                                          */
    double friction;            /* 2 (link) x 1 (plane) snake.py:104-106                        */
    double aniso[3];            /* (1,0.1,0.01) snake.py:25                                     */
    double lin_damping;         /* 0.04 btMultiBody default                                     */
    double ang_damping;         /* 0.04                                                         */
    double erp2;                /* 0.08                                                         */
    double linear_slop;         /* 1e-5                                                         */
    double residual_threshold;  /* 1e-7 leastSquaresResidualThreshold                           */
    double max_coord_vel;       /* 100                                                          */
    double err_threshold;       /* 0.05 snake.py:232                                            */
    double height_threshold;    /* 0.1  snake.py:238                                            */
    double term_angle;          /* 0.5  SnakeGymEnv.py:100                                      */
    double done_penalty;        /* -5   SnakeGymEnv.py:40                                       */
    double collision_force;     /* 10   SnakeGymEnv.py:94                                       */
    double collision_penalty;   /* -10  SnakeGymEnv.py:94                                       */
    int32_t solver_iterations;  /* 50                                                           */
    int32_t max_ticks;          /* 41: loop breaks when counter > 40 (snake.py:303)             */
    int32_t gait_selection;     /* 1    snake.py:62,247-269                                     */
    int32_t cone_friction;      /* 1 = implicit cone, 0 = pyramid                               */
    int32_t term_joint;         /* 9    SnakeGymEnv.py:100                                      */
    int32_t stale_obs_on_reset; /* 1 = torque/Fz slots keep last tick's values after reset (Q9) */
    int32_t alternate_motor_order; /* 1 = Bullet's `iteration & 1 ? j : n-1-j` motor row order  */
    int32_t motor_solver;       /* 0 = motor rows relaxed inside the PGS in Bullet's order (A.4);
                                   1 = motor rows imposed exactly (needs force = inf, kd = 1);
                                   2 = auto: 1 when admissible, else 0  (DESIGN.md section 4, D4)   */
} snk_params;

typedef struct snk_handle snk_handle;

/* Fill *p with the reference defaults listed above. */
int snk_default_params(snk_params* p);

int snk_create(const snk_model* model, const snk_params* params, int64_t n_envs, int device,
               snk_handle** out);
int snk_destroy(snk_handle* h);

int64_t snk_num_envs(const snk_handle* h);
int snk_action_dim(const snk_handle* h);
int snk_device(const snk_handle* h);

/* Soft reset (snake.py:119-127) of the environments whose mask byte is non-zero (all when
 * mask_dev is NULL); when obs_dev is non-NULL the observation of EVERY environment is written. */
int snk_reset(snk_handle* h, const uint8_t* mask_dev, float* obs_dev, void* stream);

/* One SubprocVecEnv.step over all N environments: one kernel launch. ticks_dev may be NULL. */
int snk_step(snk_handle* h, const float* actions_dev, float* obs_dev, float* rew_dev,
             uint8_t* done_dev, int32_t* ticks_dev, void* stream);

/* Same call with HOST buffers: H2D of the actions, the step kernel, D2H of obs/rew/done/ticks
 * through the handle's pinned staging buffers, then a stream synchronise.  ticks_host may be NULL. */
int snk_step_host(snk_handle* h, const float* actions_host, float* obs_host, float* rew_host,
                  uint8_t* done_host, int32_t* ticks_host);
int snk_reset_host(snk_handle* h, const uint8_t* mask_host, float* obs_host);

/* snk_step_host with the reference's own dtypes: float64 actions in, float64 obs / reward out, exactly the arrays
 * SubprocVecEnv.step exchanges with ppo/train.py:122 and ars/train.py:99 (np.stack of the workers' float64 results,
 * ppo/multiprocessing_env.py:126-128).  The narrowing / widening runs on a few host threads (SNK_HOST_THREADS); with the default
 * kernel the batch is one launch that posts every environment's row into page-locked memory as the environment finishes, its ticks
 * word last, and the threads widen the rows into the caller's arrays while the launch is still running.  Synchronous: the arrays are
 * complete on return. */
int snk_step_host_f64(snk_handle* h, const double* actions_host, double* obs_host, double* rew_host,
                      uint8_t* done_host, int32_t* ticks_host);

/* snk_step plus the mode='test' info stream of the reference (snake.py:275-278,292-293; SnakeGymEnv.py:43-44): for every
 * physics tick k < ticks_dev[e] of environment e, the observation after that tick (info['internal_observations'][k]) goes to
 * tick_obs_dev[e][k][0..55] and the world COM positions of URDF links arange(0,49,3) (info['link_positions'][k],
 * Snake.getLinkPositions, snake.py:138-146) to tick_links_dev[e][k][0..50], laid out [x0..x16 | y0..y16 | z0..z16].
 * Both arrays hold params.max_ticks (41) rows per environment; rows k >= ticks_dev[e] are left untouched.  Either trace
 * pointer may be NULL; ticks_dev is required.  An analysis path (a handful of environments): not the benchmarked kernel. */
#define SNK_LINK_POS_DIM 51
int snk_step_trace(snk_handle* h, const float* actions_dev, float* obs_dev, float* rew_dev, uint8_t* done_dev,
                   int32_t* ticks_dev, float* tick_obs_dev, float* tick_links_dev, void* stream);

/* n_steps env-steps in ONE launch with a linear policy per environment (ARS, SURVEY.md 8f rank 1): before every
 * step   x = obs (+ noise[t, env, :])   xn = (x - mean) * inv_std   action = W_env xn   (then clipped as in snk_step),
 * where obs is the observation the previous step returned (the post-reset one after a done, exactly what the
 * vector wrapper feeds back, ars/train.py:99-110).  weights_dev [N, act_dim, 56]; mean_dev / inv_std_dev [56] or
 * NULL (identity); noise_dev [n_steps, N, 56] or NULL; returns_dev [N] receives the sum of the n_steps rewards;
 * obs_trace_dev [n_steps, N, 56] or NULL receives every x the policy saw (for the caller's running statistics).
 * Only with the exact motor solver (the reference configuration).  State persists as after n_steps snk_step calls.  With persistent
 * manifolds on (snk_set_manifold) the manifold kernel runs the rollout, caches included. */
int snk_rollout_linear(snk_handle* h, const float* weights_dev, const float* mean_dev, const float* inv_std_dev,
                       const float* noise_dev, int32_t n_steps, float* returns_dev, float* obs_trace_dev, void* stream);

/* Bullet's persistent contact manifolds and contact warm starting (SURVEY.md 8f rank 2 / Appendix A.5; what
 * pybullet.loadURDF + stepSimulation do for the snake's 32 collision cylinders, snake.py:92-93,286): on != 0 switches the
 * handle's snk_step / snk_step_host* to the manifold kernel -- per cylinder the support vertex of the 32-gon hull feeds a
 * 4-slot contact cache with Bullet's add / replace / refresh / breaking rules (up to 128 contact points per environment), and
 * the cached normal impulses x warm_start (Bullet: 0.1; 0 = off) start the solver.  The call (re)allocates and CLEARS the caches
 * (4 224 B per environment + 388 MB of row tables per device); they survive soft resets like Bullet's (Q10).  on == 0 returns to
 * the default one-point-per-cylinder tick (deviation D1) and frees the memory.  Only with the exact motor solver.  While it is on,
 * snk_step, snk_step_host*, snk_step_trace and snk_rollout_linear run the manifold kernels; snk_tick is refused.  An environment
 * whose state goes non-finite in an env-step (counter word 3 of snk_last_counters) restarts like a hard reset: its caches are emptied
 * with the force-reset, so no cached impulse of that step warm-starts the next one.  Synchronises the device. */
int snk_set_manifold(snk_handle* h, int on, double warm_start);

/* Bullet's literal tick: Bullet-order motor rows (relaxed inside the projected Gauss-Seidel, as with motor_solver = 0) together with
 * the persistent manifolds and warm starting of snk_set_manifold -- the one configuration that is stepSimulation's own tick (DESIGN.md
 * section 4: deviations D1 and D4 both lifted).  Works on any handle: while it is on the handle's motor_solver is not consulted (the
 * default parameters have an unlimited motor force, so Bullet-order rows are always admissible).  on != 0 (re)allocates and CLEARS
 * the caches (4 224 B per environment, layout SNK_MAN_STRIDE below); on == 0 frees them and returns to the handle's own solver.
 * warm_start: factor of the cached normal impulses that start the solver (Bullet: 0.1; 0 = off; < 0 is refused).  While it is on,
 * snk_step, snk_step_host*, snk_step_trace and snk_tick run the Bullet-tick kernel, the cache entry points and snk_manifold_stats
 * work, and snk_rollout_linear is refused.  A non-finite force-reset empties that environment's caches, as with snk_set_manifold
 * (snk_tick has no non-finite check and leaves them).  Refused (SNK_E_ARG) while snk_set_manifold is on, and snk_set_manifold is refused
 * while this is on.  Synchronises the device.  on == 0 is refused on a handle with the exact motor solver while snk_set_joint_limits is on. */
int snk_set_bullet_tick(snk_handle* h, int on, double warm_start);

/* Joint-limit rows (btMultiBodyJointLimitConstraint, which pybullet.loadURDF gives every revolute joint of snake.urdf at +-1.57 rad):
 * on != 0 adds two unilateral rows per joint at -angle and +angle to every kernel of this handle with Bullet-order motor rows -- the
 * warp-per-env kernel when motor_solver resolves to 0, and Bullet's literal tick whenever snk_set_bullet_tick is on (either order).
 * Every sweep solves them after the motor rows and before the contact rows; impulses >= 0, no warm start.  Inert while the joints stay
 * inside the limits (outputs bit-identical to the rows off).  Refused (SNK_E_ARG) when angle is not a finite number > 0, and on a
 * handle with the exact motor solver while the Bullet tick is off (its unlimited-force motor equalities admit no limit rows).  on == 0
 * always succeeds.  Allocates nothing, does not synchronise; takes effect from the next launch. */
int snk_set_joint_limits(snk_handle* h, int on, double angle);
/* out[0] = joint-limit rows with a positive impulse at the end of a tick, summed over the environments and physics ticks of the last
 * step launch; out[1] = those ticks (the oracle's row_stats()[1] counts the same rows).  SNK_E_ARG while the limits are off.
 * Synchronises the device. */
int snk_joint_limit_stats(snk_handle* h, int64_t out[2]);

/* The contact caches of the persistent manifolds: SNK_MAN_STRIDE floats per environment, [N][SNK_MAN_STRIDE].  Cylinder c (0..31)
 * owns the floats [32 c, 32 c + 32): 4 slots of 8 words, slot s at 32 c + 8 s = (body-frame point x, y, z, distance to the ground
 * plane, world anchor x, y, normal impulse of the last tick, 0).  The same layout serves snk_set_bullet_tick.  Float 1024 + c holds the number of occupied slots of cylinder c, an
 * integer 0..4 stored as a float; slots at and beyond it are unused.  The caches are simulator state: a checkpoint that should resume
 * bit for bit needs them next to snk_get_state. */
#define SNK_MAN_STRIDE 1056
/* Copy the caches out to cache_dev [N][SNK_MAN_STRIDE] (device memory).  Asynchronous on `stream`, capturable.  SNK_E_ARG when
 * persistent manifolds are off. */
int snk_get_manifold_cache(snk_handle* h, float* cache_dev, void* stream);
/* Copy cache_dev [N][SNK_MAN_STRIDE] (device memory) into the caches.  The count words are checked first (a kernel, then a
 * synchronisation of `stream`): if any of them is not an integer in 0..4, SNK_E_ARG is returned and the caches are left untouched.
 * SNK_E_ARG when persistent manifolds are off. */
int snk_set_manifold_cache(snk_handle* h, const float* cache_dev, void* stream);
/* Empty the caches of the environments whose mask byte is non-zero (all when mask_dev is NULL): the contact half of a hard reset
 * (a rebuilt world has no cached points).  Asynchronous on `stream`, capturable.  SNK_E_ARG when persistent manifolds are off. */
int snk_clear_manifold(snk_handle* h, const uint8_t* mask_dev, void* stream);
/* out[0] = cached contact points summed over the physics ticks of the last step launch, out[1] = those ticks (their ratio is the
 * mean number of contact rows-triples per tick; the oracle's row_stats).  Synchronises the device. */
int snk_manifold_stats(snk_handle* h, int64_t out[2]);

/* Generalised advantage estimation over a device-resident rollout (SURVEY.md 8f rank 1, PPO half): compute_gae of ppo/agent.py:14-22
 * as one kernel.  rewards_dev / values_dev / returns_dev / advantages_dev are [T, N] fp32 row-major (time major, as RolloutBuffer
 * stores what ppo/train.py:131-136 appends), dones_dev [T, N] u8 (mask = 1 - done, ppo/train.py:134), next_value_dev [N] = V of the
 * state after the last step (ppo/train.py:170-171).  returns_dev receives gae + V (what compute_gae returns), advantages_dev (may be
 * NULL) the gae itself (= returns - values, ppo/train.py:178).  Stateless: no handle; runs on `device`. */
int snk_gae(int device, const float* rewards_dev, const uint8_t* dones_dev, const float* values_dev, const float* next_value_dev,
            double gamma, double tau, float* returns_dev, float* advantages_dev, int32_t n_steps, int64_t n_envs, void* stream);

/* Raw physics ticks with explicit joint targets [N,16] (gait script, snake_gait_test.py:96-104);
 * no task logic.  n_ticks ticks are run with the same targets. */
int snk_tick(snk_handle* h, const float* targets_dev, int32_t n_ticks, void* stream);

/* Observation of the current state (snake.py:209-217) without stepping. */
int snk_observe(snk_handle* h, float* obs_dev, void* stream);

/* Self-collision clearance of the current state (SURVEY.md Q11): clearance_dev[e] = a lower bound, in metres, of the
 * smallest distance between two cylinders of environment e that Bullet would test under URDF_USE_SELF_COLLISION
 * (snake.py:93: all link pairs except parent-child, i.e. the 465 pairs of non-consecutive cylinders).  The step
 * kernels do not generate self-contacts (deviation D3); a positive clearance over a run proves none was missed.
 * Bullet's hulls are 32-gons inscribed in these cylinders plus a 0.001 margin each. */
int snk_self_clearance(snk_handle* h, float* clearance_dev, void* stream);

/* Copy the [N, SNK_STATE_STRIDE] fp32 state array out of / into the handle (device pointers). */
int snk_get_state(snk_handle* h, float* state_dev, void* stream);
int snk_set_state(snk_handle* h, const float* state_dev, void* stream);

/* Per-launch counters of the last snk_step (device-side sums, read back synchronously):
 * out[0] = total physics ticks, out[1] = total PGS iterations, out[2] = dones,
 * out[3] = environments whose state went non-finite and were force-reset: done with reward done_penalty and the reset pose, and
 *          with persistent manifolds on (snk_set_manifold, snk_set_bullet_tick) their contact caches emptied, as a hard reset does. */
int snk_last_counters(snk_handle* h, int64_t out[4]);

/* Number of kernels this library has launched on this handle since creation. */
int64_t snk_launch_count(const snk_handle* h);

const char* snk_last_error(void);
const char* snk_build_info(void);
/* Row layout / warp configuration of the thread-per-environment env-step kernel the library launches. */
const char* snk_kernel_variant(void);

#ifdef __cplusplus
}
#endif
#endif /* SNAKE_B200_H */
