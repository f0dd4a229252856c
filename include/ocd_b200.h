/*
 * ocd_b200.h -- C ABI of the B200-native batched MPC engine (libocd_b200.so).
 *
 * Drop-in boundary for ONE hot path of avikj/L4DC-MPC-OCD: the planner inner loop
 * (NaivePlanner.generate_plan) and the receding-horizon episode loop that
 * MPC_ORD.eval_weights runs serially.  The reference has no FFI of its own (it is pure
 * Python on TensorFlow); each entry point below therefore names the reference *Python*
 * interface it replaces (paths relative to the reference checkout).  INTEGRATION.md shows
 * the ctypes stub a reference maintainer would add.
 *
 * Conventions
 *   - Plain C types only: pointers, sizes, the two POD structs below.  No torch types.
 *   - Unless a function name ends in _host, every data pointer is a DEVICE pointer owned by
 *     the caller; work is enqueued on `stream` (a cudaStream_t passed as void*) and the call
 *     returns without synchronising.  No hidden allocation, no global mutable state: calls
 *     on distinct streams are thread-safe.
 *   - Layout is structure-of-arrays with the batch index fastest: a "[C][4][B]" array holds
 *     element (c, k, b) at ((c*4)+k)*B + b.  float32 / int32 device data throughout (the reference
 *     computes in float32: car.py:55, linear_reward_car.py:34).
 *   - Car 0 is the planning ("robot") car; cars 1..C-1 are the other cars.
 *   - Return value: 0 on success, a negative OCD_E* code otherwise (ocd_strerror()).  Nothing
 *     throws or exits across the ABI.  There is NO CPU fallback: without a CUDA device every
 *     compute entry point returns OCD_ECUDA.
 *   - Environment variables read (never written) at call time, for tests and tuning:
 *     OCD_KERNEL_FORM=throughput|latency|wide|tp forces a kernel form (see ocd_kernel_form; all forms
 *     give bit-identical results); OCD_RUNTIME_H=1 runs H = 15 / 50 on the runtime-horizon kernels instead of
 *     their compile-time specialisations; OCD_HOST_CHUNKS="w0,w1,..." sets the chunk weights of
 *     ocd_solve_batch_host's copy/compute pipeline and OCD_HOST_THREADS=<n> its staging-copy threads (default: the
 *     cores in the calling process's affinity mask, at most 8).
 */
#ifndef OCD_B200_H
#define OCD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OCD_ABI_VERSION 3
#define OCD_MAX_LANES   4
#define OCD_MAX_OTHER   7     /* other cars per world (C <= 8)            */
#define OCD_MAX_PLAN    16    /* FixedPlanCar plan length                 */
#define OCD_MAX_H       64    /* planning horizon                         */
#define OCD_MAX_STARTS  6
#define OCD_LBFGS_MAX_H 16    /* horizon limit of the opt-in L-BFGS optimiser     */

enum {
    OCD_OK       = 0,
    OCD_EINVAL   = -1,   /* bad argument (NULL pointer, B < 0, bad shape)          -> Python ValueError */
    OCD_EUNSUP   = -2,   /* H / C / L outside the supported range                                      */
    OCD_ECUDA    = -3,   /* CUDA runtime error (no device, launch failure)                             */
    OCD_ENOMEM   = -4    /* allocation failure in an ocd_ctx                                           */
};

/* Planner + world constants.
 * Replaces the constructor state of NaivePlanner (interact_drive/planner/naive_planner.py:19-30),
 * CarWorld.dt / lanes (interact_drive/world.py:18-37,143-159) and ThreeLaneTestCar
 * (experiments/merging.py:20-30). */
typedef struct {
    int32_t H;            /* horizon (naive_planner.py:24)                                         */
    int32_t C;            /* cars in the world, robot included                                      */
    int32_t L;            /* lanes; feature count K = L + 4 (merging.py:61-83)                      */
    int32_t n_iter;       /* SGD steps per start (naive_planner.py:151)                             */
    int32_t num_lanes;    /* fence threshold 0.05*num_lanes (merging.py:80)                         */
    int32_t other_mode;   /* 0: other cars keep velocity; 1: known controls (naive_planner.py:53-66)*/
    int32_t extra_inits;  /* 3 more starts with a0 = friction*v^2 (naive_planner.py:112-116)        */
    int32_t math_mode;    /* 0: MUFU intrinsics (sin/cos/ex2/rcp.approx); 1: IEEE div + libdevice   */
    int32_t optimizer;    /* 0: the reference's fixed-budget SGD (naive_planner.py:151-153);
                           * 1: L-BFGS, at most n_iter iterations per start (opt-in; see ocd_solve_batch) */
    int32_t reserved;     /* must be 0                                                              */
    /* Python floats in the reference; kept as doubles and cast to float32 at the point of
     * use exactly as TensorFlow does (e.g. dt**2 is squared in double, then cast).            */
    double  lr;           /* learning_rate (naive_planner.py:20,28)                                 */
    double  dt;           /* world.dt                                                               */
    double  friction;     /* robot friction (car.py:33)                                             */
    double  target_speed; /* merging.py:29                                                          */
    double  lane_x[OCD_MAX_LANES];  /* lane median x (world.py:149-159 via StraightLane.p[0])       */
} ocd_params;

/* The scripted cars and the replanning world for the episode driver.
 * Replaces FixedControlCar / FixedVelocityCar / FixedPlanCar state
 * (interact_drive/car/fixed_control_car.py:12-36, fixed_velocity_car.py:18-24,
 * fixed_plan_car.py:13-39) and ReplanningCarWorld (experiments/replanning_world.py:11-36). */
typedef struct {
    int32_t n_other;                        /* must equal params.C - 1                               */
    int32_t critical_t;                     /* 0: plain CarWorld; >0: teleport when world.t == it    */
    int32_t kind[OCD_MAX_OTHER];            /* 0 fixed control / fixed velocity, 1 fixed plan        */
    int32_t plan_len[OCD_MAX_OTHER];
    float   init_state[OCD_MAX_OTHER][4];   /* used when other_init == NULL                          */
    float   friction[OCD_MAX_OTHER];        /* 0 for FixedVelocityCar, 0.2 default for FixedPlanCar  */
    float   control[OCD_MAX_OTHER][2];      /* fixed control / default_control                       */
    float   plan[OCD_MAX_OTHER][OCD_MAX_PLAN][2];
    float   teleport_state[4];              /* replanning_world.py:34: [10, 0, 0, 0]                 */
} ocd_scenario;

int         ocd_abi_version(void);
const char *ocd_strerror(int code);
/* number of starts S: 3, or 6 with extra_inits (naive_planner.py:107-118) */
int         ocd_num_starts(const ocd_params *p);
/* number of CUDA devices visible to the library (0 if none / no driver) */
int         ocd_device_count(void);

/* car_dynamics_step / next_car_state (interact_drive/simulation_utils.py:9-21,73-123) and
 * Car.step (interact_drive/car/car.py:76-87), for B cars at once.
 * friction_b may be NULL (then `friction` is used for every car). */
int ocd_dynamics_step_batch(const float *state /*[4][B]*/, const float *control /*[2][B]*/,
                            float dt, float friction, const float *friction_b /*[B] or NULL*/,
                            float *next_state /*[4][B]*/, int64_t B, void *stream);

/* The smooth helpers of interact_drive/math_utils.py, evaluated with the kernels' precise math for
 * B points (kind selects the function; p0, p1 are its parameters):
 *   OCD_SMOOTH_F          _f(x, shape=p0)                        math_utils.py:7-31
 *   OCD_SMOOTH_THRESHOLD  smooth_threshold(threshold=p0, width=p1, c=5)(z)   math_utils.py:59-97
 *   OCD_SMOOTH_BUMP       smooth_bump(start=p0, end=p1)(z)        math_utils.py:135-180 */
enum { OCD_SMOOTH_F = 0, OCD_SMOOTH_THRESHOLD = 1, OCD_SMOOTH_BUMP = 2 };
int ocd_smooth_batch(int kind, const float *z /*[B]*/, double p0, double p1, float *out /*[B]*/,
                     int64_t B, void *stream);

/* ThreeLaneTestCar.features (experiments/merging.py:32-83) for B world states. */
int ocd_features_batch(const ocd_params *p, const float *world /*[C][4][B]*/,
                       float *phi /*[K][B]*/, int64_t B, void *stream);

/* NaivePlanner.reward_func == mpc_reward (interact_drive/planner/naive_planner.py:32-79) and its
 * gradient with respect to the controls (what tf.GradientTape / optimizer.minimize obtain).
 * other_controls: [C-1][H][2][Bo] with Bo == 1 (shared) or Bo == B; required iff other_mode == 1.
 * weights: [K][Bw]; weight_idx[b] in [0,Bw) selects the vector of problem b; with
 * weight_idx == NULL, Bw must be 1 (shared) or B (one per problem). */
int ocd_reward_grad_batch(const ocd_params *p, const float *world /*[C][4][B]*/,
                          const float *controls /*[H][2][B]*/,
                          const float *other_controls, int64_t Bo,
                          const float *weights, int64_t Bw, const int32_t *weight_idx,
                          float *reward /*[B]*/, float *grad /*[H][2][B] or NULL*/,
                          int64_t B, void *stream);

/* Which form of the planner kernel a batch of B problems (episode != 0: B worlds of ocd_episode_batch) would run:
 * the throughput form (warp votes skip inactive feature blocks), the latency form (straight-line sweep, for small
 * batches), the wide form (the same under a register cap, for large batches) or the time-parallel form (eight
 * lanes per start, for the smallest).  All forms give bit-identical results; the choice follows measurements on
 * B200 (DESIGN.md) and can be forced with the environment variable OCD_KERNEL_FORM=throughput|latency|wide|tp.
 * Pure host logic (no CUDA call).  -> OCD_FORM_* or a negative status. */
enum { OCD_FORM_THROUGHPUT = 0, OCD_FORM_LATENCY = 1, OCD_FORM_WIDE = 2, OCD_FORM_TIME_PARALLEL = 3 };
int ocd_kernel_form(const ocd_params *p, int64_t B, int episode);

/* Jacobian of the horizon-summed features with respect to the controls: what the reference's inverse
 * optimal control classes take from tf.GradientTape -- segment_loss's d r / d u = J^T w
 * (interact_drive/reward_design/first_order_ioc.py:62-91) and segment_jacobian / total_jacobian
 * (:213-268).  Row i is the gradient of sum_t phi_i(s_{t+1}) with TensorFlow's gradient conventions,
 * i.e. ocd_reward_grad_batch with weights = e_i; other cars as in ocd_reward_grad_batch.
 * Outputs: phi_sum [K][B], jac [K][H][2][B]. */
int ocd_feature_jacobian_batch(const ocd_params *p, const float *world /*[C][4][B]*/,
                               const float *controls /*[H][2][B]*/,
                               const float *other_controls, int64_t Bo,
                               float *phi_sum /*[K][B]*/, float *jac /*[K][H][2][B]*/,
                               int64_t B, void *stream);

/* Hessians of the horizon-summed features with respect to the controls: what the reference's second-order inverse
 * optimal control takes from TensorFlow as t.jacobian(gradients, controls)
 * (interact_drive/reward_design/second_order_ioc.py:80-152, LocalCIOC.compute_total_augmented_loss).  The reward is
 * linear in the weights, so the Hessian of the reward is sum_k w_k hess[k] and CIOC's likelihood and its weight
 * gradient need nothing beyond these K matrices and ocd_feature_jacobian_batch's K rows.  Exact second derivatives
 * (hyper-dual arithmetic in float32, libdevice transcendentals), TensorFlow's branch conventions at clip / min / max /
 * where; other cars as in ocd_reward_grad_batch.  Output: hess [K][2H][2H][B], symmetric in the two control
 * indices (flat index 2 t + c for control c of step t). */
int ocd_feature_hessian_batch(const ocd_params *p, const float *world /*[C][4][B]*/,
                              const float *controls /*[H][2][B]*/,
                              const float *other_controls, int64_t Bo,
                              float *hess /*[K][2H][2H][B]*/, int64_t B, void *stream);

/* NaivePlanner.generate_plan (interact_drive/planner/naive_planner.py:81-164) + Keras SGD
 * (call sites :28,:153): S starts x n_iter gradient steps, final loss per start, first-minimum
 * argmin.  cur_speed ([B] or NULL -> world's robot speed) feeds the extra_inits starts (:114-116).
 * With params.optimizer == 1 each start is minimised by L-BFGS instead (two-loop recursion with 4
 * correction pairs, Armijo backtracking, first step of length lr; H <= OCD_LBFGS_MAX_H; precise math).
 * That stands in for the reference's never-enabled `use_lbfgs` branch (naive_planner.py:127-149, TFP's
 * lbfgs_minimize): same role, its own semantics -- there is nothing in the reference to pin it to.
 * Outputs: plan [H][2][B] (the selected start), losses [S][B], best [B];
 * all_plans [S][H][2][B] optional. */
int ocd_solve_batch(const ocd_params *p, const float *world /*[C][4][B]*/,
                    const float *other_controls, int64_t Bo,
                    const float *weights, int64_t Bw, const int32_t *weight_idx,
                    const float *cur_speed,
                    float *plan, float *losses, int32_t *best, float *all_plans,
                    int64_t B, void *stream);

/* Vector-Jacobian product of ocd_solve_batch's plan with respect to the weights and the initial world: given
 * plan_bar = d loss / d plan, weights_bar[k][b] = d loss / d w_k of problem b's weight vector and world_bar = d loss /
 * d world, for the fixed-budget SGD plan (optimizer == 0; L-BFGS's line search is not differentiable: OCD_EUNSUP).
 * The derivative follows the start ocd_solve_batch picked (best, its output) through the n_iter SGD steps
 * (naive_planner.py:151-153) and through the start itself (the extra-init starts depend on the robot's speed when
 * cur_speed is NULL); the argmin over starts, clip masks and min / max selections have zero derivative almost
 * everywhere.  The other cars enter world_bar through the planner's prediction of them (naive_planner.py:53-66).
 * Nothing is summed across problems: with a shared or indexed weight table the caller adds the rows of weights_bar
 * that use the same vector.  Inputs as for ocd_solve_batch (the same params, world, weights, other controls and
 * cur_speed); world_bar may be NULL.  workspace: device memory of at least ocd_solve_vjp_workspace_bytes() bytes
 * (n_iter * H * 2 * B floats: the recomputed iterates); too small -> OCD_EINVAL.
 * Outputs: weights_bar [K][B], world_bar [C][4][B] or NULL. */
int ocd_solve_vjp_workspace_bytes(const ocd_params *p, int64_t B, size_t *bytes);
int ocd_solve_vjp_batch(const ocd_params *p, const float *world /*[C][4][B]*/,
                        const float *other_controls, int64_t Bo,
                        const float *weights, int64_t Bw, const int32_t *weight_idx,
                        const float *cur_speed,
                        const int32_t *best /*[B], from ocd_solve_batch*/, const float *plan_bar /*[H][2][B]*/,
                        float *weights_bar /*[K][B]*/, float *world_bar /*[C][4][B] or NULL*/,
                        void *workspace, size_t workspace_bytes, int64_t B, void *stream);

/* The receding-horizon episode of MPC_ORD.eval_weights_for_init
 * (interact_drive/reward_design/mpc_ord.py:87-103): T times CarWorld.step
 * (interact_drive/world.py:79-109; ReplanningCarWorld.step experiments/replanning_world.py:29-36),
 * each step = one full MPC solve for the robot (PlannerCar._get_next_control,
 * interact_drive/car/planner_car.py:54-85) + scripted-car stepping, accumulating the TRUE-weight
 * reward of the past state.  One launch for all B worlds and all T steps.
 *   robot_init   [4][B]
 *   other_init   [C-1][4][B] or NULL (NULL: scenario->init_state for every world)
 *   plan_weights [K][Bw] + weight_idx as above (the candidate weights the planner optimises)
 *   true_weights [K]     (device) designer weights used for the return
 *   unlucky_idx  [B] or NULL: car index teleported at world.t == critical_t (0 = none)
 *   t0           world step index of the first step (0 after reset); FixedPlanCar plans and the
 *                teleport are indexed by t0 + i
 *   returns      [B]   sum over the T steps of true_weights . features(past_state)
 *   traj_controls [T][2][B], traj_best [T][B], traj_states [T][C][4][B] (past states): optional
 *   final_world  [C][4][B] optional: world state after the last step
 * With T == 1 this is exactly one CarWorld.step for B worlds. */
int ocd_episode_batch(const ocd_params *p, const ocd_scenario *sc,
                      const float *robot_init, const float *other_init,
                      const float *plan_weights, int64_t Bw, const int32_t *weight_idx,
                      const float *true_weights, const int32_t *unlucky_idx,
                      int32_t t0, int32_t T,
                      float *returns, float *traj_controls, int32_t *traj_best,
                      float *traj_states, float *final_world,
                      int64_t B, void *stream);

/* Vector-Jacobian product of ocd_episode_batch's returns: given returns_bar = d loss / d returns,
 *   plan_weights_bar [K][B]         d loss / d (world b's planning weight vector)
 *   robot_init_bar   [4][B] or NULL d loss / d robot_init
 *   true_weights_bar [K][B] or NULL d loss / d true_weights, per world (returns_bar[b] * sum_t features(past state))
 * for the fixed-budget SGD planner (optimizer == 1: OCD_EUNSUP).  The derivative follows the episode's own
 * trajectory: traj_states [T][C][4][B], traj_best [T][B] and traj_controls [T][2][B] are what ocd_episode_batch
 * wrote for the same params, scenario, weights and T.  Every step contributes the Jacobian of its applied control with
 * respect to the weights and the robot's state (the solve VJP of the winning start, seeded on plan[0]) and the
 * simulator step's; the scripted cars depend on neither, and the argmin over starts, clip masks and min / max
 * selections are not differentiated.  Nothing is summed across worlds.  workspace: device memory of at least
 * min_bytes from ocd_episode_vjp_workspace_bytes (the Jacobian rows and the iterates of one step); full_bytes holds
 * the iterates of all T steps at once, so fewer launches; anything in between is used as far as it goes, with the
 * same results.  Too small -> OCD_EINVAL.  T == 0 writes zeros. */
int ocd_episode_vjp_workspace_bytes(const ocd_params *p, int32_t T, int64_t B, size_t *min_bytes, size_t *full_bytes);
int ocd_episode_vjp_batch(const ocd_params *p, const ocd_scenario *sc,
                          const float *plan_weights, int64_t Bw, const int32_t *weight_idx,
                          const float *true_weights, int32_t T,
                          const float *traj_states /*[T][C][4][B]*/, const int32_t *traj_best /*[T][B]*/,
                          const float *traj_controls /*[T][2][B]*/, const float *returns_bar /*[B]*/,
                          float *plan_weights_bar /*[K][B]*/, float *robot_init_bar /*[4][B] or NULL*/,
                          float *true_weights_bar /*[K][B] or NULL*/,
                          void *workspace, size_t workspace_bytes, int64_t B, void *stream);

/* ---- host-buffer convenience layer (what a Python/ctypes caller without torch uses) ---------
 * An ocd_ctx owns a device, a stream, pinned staging buffers and device buffers that grow on
 * demand.  The *_host calls take HOST pointers with the same layouts as above, copy in, run the
 * same kernels, copy out and synchronise before returning. */
typedef struct ocd_ctx ocd_ctx;
int  ocd_ctx_create(int device, ocd_ctx **out);
void ocd_ctx_destroy(ocd_ctx *ctx);

/* Page-lock a caller-owned host array in place (cudaHostRegister) / undo it.  A steady-state caller that reuses its
 * ordinary (pageable) input and output arrays registers them once; the *_host calls then copy from / into them
 * directly, exactly as for arrays allocated page-locked, instead of staging every call through the context's pinned
 * area with host memcpys (which is what bounds eight ranks sharing one host's cores).  The caller must unregister before
 * freeing the memory.  -> OCD_OK, OCD_EINVAL (null / zero bytes) or OCD_ECUDA (not lockable, already registered). */
int ocd_host_register(void *ptr, size_t bytes);
int ocd_host_unregister(void *ptr);

int ocd_solve_batch_host(ocd_ctx *ctx, const ocd_params *p, const float *world,
                         const float *other_controls, int64_t Bo,
                         const float *weights, int64_t Bw, const int32_t *weight_idx,
                         const float *cur_speed,
                         float *plan, float *losses, int32_t *best, int64_t B);

/* The same solve for a receding-horizon caller, which applies plan[0] and discards the rest
 * (PlannerCar._get_next_control returns plan[0]: interact_drive/car/planner_car.py:80-85): only the first control
 * [2][B] travels back (8 B per solve instead of 8 H), and losses / best are optional (NULL: not copied). */
int ocd_solve_first_host(ocd_ctx *ctx, const ocd_params *p, const float *world,
                         const float *other_controls, int64_t Bo,
                         const float *weights, int64_t Bw, const int32_t *weight_idx,
                         const float *cur_speed,
                         float *first_control /*[2][B]*/, float *losses /*[S][B] or NULL*/,
                         int32_t *best /*[B] or NULL*/, int64_t B);

/* final_world [C][4][B] or NULL.  Repeated calls with the same shapes and constants (a CMA-ES run makes one per
 * generation) replay a CUDA graph of copy-in / kernel / copy-out captured on the first of them. */
int ocd_episode_batch_host(ocd_ctx *ctx, const ocd_params *p, const ocd_scenario *sc,
                           const float *robot_init, const float *other_init,
                           const float *plan_weights, int64_t Bw, const int32_t *weight_idx,
                           const float *true_weights, const int32_t *unlucky_idx,
                           int32_t t0, int32_t T, float *returns, float *final_world, int64_t B);

/* FP32 FMA micro-benchmark used by bench.py to measure the roofline denominator in the same
 * job: runs `iters` dependent-free FMA rounds on every SM, returns achieved FLOP/s in *flops. */
int ocd_fp32_peak(int iters, double *flops, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* OCD_B200_H */
