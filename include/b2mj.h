/* b2mj.h -- C ABI of the B200-native batched physics path.
 *
 * Drop-in boundary for the one hot path of ChenDavidTimothy/mujoco-template.  The
 * reference has no FFI of its own: its "operator API" for this path is the set of
 * third-party `mujoco` symbols it calls.  Each entry point below names the reference
 * call site(s) it replaces (paths relative to the reference repo root).
 *
 * Conventions
 *  - extern "C", plain pointers and sizes, no torch / C++ types.
 *  - All state arrays are SoA with the env index fastest: element (k, e) of an array
 *    with leading dimension `dim` lives at  base[k * nenv + e].  Precision is fixed per
 *    batch (B2_F64 or B2_F32); pointers are `void*` and must match it.
 *  - Pointers may be device memory or page-locked host memory mapped into the device
 *    address space (the single-env `Env` uses the latter for zero-copy NumPy views).
 *  - Calls are asynchronous on `stream` (a cudaStream_t passed as void*; NULL = legacy
 *    default stream) unless stated otherwise.  Device memory is allocated in b2_model_create /
 *    b2_batch_create (model images, warp-engine scratch) and on the FIRST call of the entry points
 *    that need extra buffers (b2_control_tick / b2_step_lazy: shadow state; b2_step_host: staging;
 *    b2_lqr_set_gain); b2_step, b2_rollout, b2_rollout_feedback, b2_forward, b2_linearize, b2_linearize_sensors,
 *    b2_linearize_rollout and b2_jacobian never allocate.
 *  - No process-wide model state: a model's constants live in per-model device images handed to
 *    every launch, so batches of different models can be driven from different threads and streams,
 *    and a captured CUDA graph replays with the model it was captured with.  One b2_batch must not be
 *    used from two threads at once (its scratch is per batch).
 *  - Every function returns B2_OK (0) or a negative error code; b2_last_error() returns
 *    a thread-local message.  There is no CPU fallback: without a CUDA device every
 *    compute entry point fails with B2_ERR_CUDA.
 */
#ifndef B2MJ_H
#define B2MJ_H
#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif

#define B2_OK 0
#define B2_ERR_ARG (-1)      /* -> ConfigError */
#define B2_ERR_BLOB (-2)     /* -> ConfigError (malformed / version mismatch) */
#define B2_ERR_CAPACITY (-3) /* -> ConfigError (model larger than any compiled size class) */
#define B2_ERR_CUDA (-4)     /* -> TemplateError */
#define B2_ERR_LINEARIZE (-5) /* -> LinearizationError */

#define B2_F64 64
#define B2_F32 32

/* per-env status bits written to b2_state.flags (replaces upstream's silent
 * mj_checkPos/Vel/Acc auto-reset, SURVEY.md section 5) */
#define B2_FLAG_BAD_QPOS 1
#define B2_FLAG_BAD_QVEL 2
#define B2_FLAG_BAD_QACC 4
#define B2_FLAG_OVERFLOW 8 /* contact / constraint-row capacity of the size class exceeded */

/* Jacobian kinds for b2_jacobian (reference mujoco_template/jacobians.py:12-23) */
#define B2_JAC_SITE 0
#define B2_JAC_BODY 1
#define B2_JAC_BODYCOM 2
#define B2_JAC_SUBTREECOM 3

typedef struct b2_model b2_model; /* opaque: compiled model constants (mj.MjModel's role) */
typedef struct b2_batch b2_batch; /* opaque: nenv envs of one model on one device (mj.MjData's role) */

/* SoA state of a batch; qacc_warmstart and flags may be NULL.  (mj.MjData.qpos/qvel/ctrl/
 * qacc_warmstart, reference mujoco_template/state_utils.py:9-31) */
typedef struct b2_state {
  void* qpos;           /* (nq, nenv) */
  void* qvel;           /* (nv, nenv) */
  void* ctrl;           /* (nu, nenv) */
  void* qacc_warmstart; /* (nv, nenv) or NULL (treated as zeros, not written) */
  int* flags;           /* (nenv) int32 status bits, OR-ed in; or NULL */
} b2_state;

/* optional derived outputs of the forward pass that PRECEDES the last integration
 * (MuJoCo semantics: derived arrays lag the state by one step).  Any pointer may be NULL.
 * (mj.MjData.xpos/xipos/geom_xpos/site_xpos/subtree_com/qacc read by
 *  reference mujoco_template/observations.py:132-164 and logging.py probes) */
typedef struct b2_derived {
  void* xpos;        /* (nbody*3, nenv) */
  void* xquat;       /* (nbody*4, nenv) */
  void* xipos;       /* (nbody*3, nenv) */
  void* geom_xpos;   /* (ngeom*3, nenv) */
  void* site_xpos;   /* (nsite*3, nenv) */
  void* subtree_com; /* (nbody*3, nenv) */
  void* qacc;        /* (nv, nenv) */
  void* qfrc_bias;   /* (nv, nenv) */
  int* ncon;         /* (nenv) active contacts */
  int* nefc;         /* (nenv) constraint rows */
  int* solver_iter;  /* (nenv) Newton iterations */
  void* sensordata;  /* (nsensordata, nenv) mjData.sensordata (reference observations.py:117-127) */
} b2_derived;

/* Replaces mj.MjModel.from_xml_path/from_xml_string (reference mujoco_template/model.py:22-31):
 * the host compiler (mujoco_template/mjcf.py) produces `blob`; see include/b2_model_layout.h. */
int b2_model_create(const void* blob, size_t nbytes, b2_model** out);
void b2_model_destroy(b2_model* model);
/* update the actuator-disable mask (opt.disableactuator, reference model.py:77-105); nu ints */
int b2_model_set_actuator_disabled(b2_model* model, const int* disabled, int nu);

/* Replaces mj.MjData(model) (reference model.py:14-20).  Allocates scratch only. */
int b2_batch_create(const b2_model* model, int nenv, int device, int precision, b2_batch** out);
void b2_batch_destroy(b2_batch* batch);

/* Replaces mj.mj_step (reference mujoco_template/model.py:56-57, driven by env.py:190):
 * advances every env `nsteps` steps with ctrl held constant.  `derived` may be NULL. */
int b2_step(b2_batch* batch, const b2_state* state, int nsteps, const b2_derived* derived, void* stream);

/* Open-loop rollout of every env (upstream mujoco.rollout's role; sampling planners, shooting, the forward pass of iLQR):
 * for t = 0 .. nsteps-1, state.ctrl <- ctrl_seq[t]; one mj_step; record.  Exactly the loop
 *     state.ctrl <- ctrl_seq[t]; b2_step(batch, state, 1, t == nsteps-1 ? derived : NULL)
 * with the state recorded after each call.  On the lane engine it is one launch that keeps every env in registers.
 * ctrl_seq    (nsteps, nu, nenv), element (t, a, e) at base[(t*nu + a)*nenv + e]; NULL = hold state.ctrl (b2_step's case)
 * qpos_traj   (nsteps, nq, nenv): the state after step t (mj_step's qpos), may be NULL
 * qvel_traj   (nsteps, nv, nenv): likewise, may be NULL
 * sensor_traj (nsteps, nsensordata, nenv): the sensordata step t leaves (the forward pass of the pre-step state,
 *             as mj_step leaves it); may be NULL; ignored when the model has no sensors
 * derived     as in b2_step: the derived arrays of the LAST step; may be NULL.
 * After the call state.qpos / qvel / qacc_warmstart hold the final state, state.ctrl holds ctrl_seq[nsteps-1] and
 * flags are OR-ed as the loop ORs them.  Controls outside ctrlrange are clamped inside the physics; ctrl_seq is not
 * modified.  A diverged env is flagged and frozen from the step that detects it: its remaining qpos / qvel rows repeat
 * the state it is frozen in, its remaining sensor rows are NaN (no forward pass ran).  nsteps < 1: B2_ERR_ARG. */
int b2_rollout(b2_batch* batch, const b2_state* state, int nsteps, const void* ctrl_seq, void* qpos_traj, void* qvel_traj,
               void* sensor_traj, const b2_derived* derived, void* stream);

/* Replaces mj.mj_forward (reference model.py:53-54, env.py:157): no integration. */
int b2_forward(b2_batch* batch, const b2_state* state, const b2_derived* derived, void* stream);

/* Replaces mj.mjd_transitionFD(model, data, eps, centered, A, B, None, None)
 * (reference mujoco_template/linearization.py:16-35).  A: (2nv, 2nv, nenv), B: (2nv, nu, nenv),
 * element (r, c, e) at base[(r * ncols + c) * nenv + e].  State is not modified. */
int b2_linearize(b2_batch* batch, const b2_state* state, double eps, int centered, void* A, void* B, void* stream);

/* Replaces mj.mjd_transitionFD(model, data, eps, centered, A, B, C, D) with the sensor Jacobians: b2_linearize's (A, B)
 * plus C = d sensordata / dx (nsensordata, 2nv, nenv) and D = d sensordata / du (nsensordata, nu, nenv), same layout, from
 * the same rollouts in the same launch.  A rollout's reading is the sensordata of its forward pass at the perturbed input
 * state (RK4: the first stage); readings are differenced by plain subtraction (framequat components too), control columns
 * follow B's ctrlrange rules.  Any of A, B, C, D may be NULL, but not all four.  Without sensors this is b2_linearize.
 * State is not modified; never allocates. */
int b2_linearize_sensors(b2_batch* batch, const b2_state* state, double eps, int centered, void* A, void* B, void* C, void* D,
                         void* stream);

/* Linearisation along a rollout (iLQR / DDP, time-varying LQR about a nominal trajectory, the linear model of MPC): the
 * transition and sensor Jacobians at every step of an open-loop control sequence.  Exactly the loop, on a COPY s of state,
 *     X[0] <- s
 *     for t = 0 .. nsteps-1:  s.ctrl <- ctrl_seq[t];  b2_linearize_sensors(s, eps, centered, A[t], B[t], C[t], D[t]);
 *                             b2_step(s, 1);  X[t+1] <- s
 * On the lane engine it is two launches for any nsteps: the nominal rollout, then the FD of every step at once.
 * ctrl_seq    (nsteps, nu, nenv) as in b2_rollout; NULL = hold state.ctrl
 * A, B        (nsteps, 2nv, 2nv, nenv), (nsteps, 2nv, nu, nenv): b2_linearize's layout with the step outermost
 * C, D        (nsteps, nsensordata, 2nv, nenv), (nsteps, nsensordata, nu, nenv); ignored when the model has no sensors.
 *             Any of A, B, C, D may be NULL, but not all four.
 * qpos_traj   (nsteps+1, nq, nenv), required: row 0 is x0, row t+1 the state after step t -- the nominal the FD reads
 * qvel_traj   (nsteps+1, nv, nenv), required: likewise
 * warm_traj   (nsteps+1, nv, nenv): the qacc_warmstart each step starts from (row 0: state.qacc_warmstart); required when
 *             state.qacc_warmstart is non-NULL, ignored when it is NULL (every step then starts from zeros, as b2_step)
 * sensor_traj (nsteps, nsensordata, nenv): the nominal reading of step t, as b2_rollout records it; may be NULL; ignored
 *             when the model has no sensors
 * State is not modified, except that flags get every bit the loop would set OR-ed in.  A diverged env is frozen from the
 * step that detects it, as in b2_rollout: its remaining state and warm rows repeat the frozen state, its remaining sensor
 * rows are NaN, and its later Jacobians are the FD about the frozen state.  Offsets are 64-bit; never allocates; capturable
 * in a CUDA graph.  nsteps < 1, a NULL qpos_traj / qvel_traj, a NULL warm_traj with a warm start, or all four Jacobians
 * NULL: B2_ERR_ARG; eps <= 0: B2_ERR_LINEARIZE. */
int b2_linearize_rollout(b2_batch* batch, const b2_state* state, int nsteps, const void* ctrl_seq, double eps, int centered,
                         void* A, void* B, void* C, void* D, void* qpos_traj, void* qvel_traj, void* warm_traj, void* sensor_traj,
                         void* stream);

/* Closed-loop rollout under a time-varying LQR law (the forward pass of iLQR / DDP, time-varying LQR tracking of a nominal
 * trajectory).  Exactly the loop, for t = 0 .. nsteps-1,
 *     state.ctrl <- clip(ctrl_nom[t] + alpha[e] k[t] - K[t] [qpos (-) qpos_nom[t] ; qvel - qvel_nom[t]], ctrlrange);
 *     b2_step(batch, state, 1, t == nsteps-1 ? derived : NULL)
 * with the state recorded after each step as in b2_rollout.  (-) is b2_differentiate_pos(dt = 1, qpos_nom[t] -> qpos): the
 * tangent-space deviation of b2_lqr_control and of b2_linearize's A.  Clipping applies to ctrl-limited actuators only.
 * ctrl_nom    (nsteps, nu, nenv), required
 * qpos_nom    (>= nsteps, nq, nenv), qvel_nom (>= nsteps, nv, nenv): row t is the nominal state of step t; required.  Rows
 *             0 .. nsteps-1 are read, so b2_linearize_rollout's (nsteps+1)-row trajectories serve as they are.
 * K           (nsteps, nu, 2nv, nenv): b2_tvlqr's layout; required
 * k           (nsteps, nu, nenv): feedforward terms; NULL = zero
 * alpha       (nenv): step size per env (an iLQR line search is per env), in the batch's precision; NULL = 1
 * ctrl_traj   (nsteps, nu, nenv): the control applied at step t; may be NULL
 * qpos_traj, qvel_traj, sensor_traj, derived: as in b2_rollout; may be NULL.
 * State, flags, derived arrays and diverged envs behave as in b2_rollout; a frozen env's remaining ctrl_traj rows are NaN and
 * its state.ctrl keeps the last control it was given (otherwise state.ctrl holds the control of step nsteps-1).  On the
 * lane engine it is one launch; offsets are 64-bit; never allocates; capturable in a CUDA graph.  nsteps < 1, a NULL
 * required pointer or a model without actuators: B2_ERR_ARG. */
int b2_rollout_feedback(b2_batch* batch, const b2_state* state, int nsteps, const void* ctrl_nom, const void* qpos_nom,
                        const void* qvel_nom, const void* K, const void* k, const void* alpha, void* ctrl_traj, void* qpos_traj,
                        void* qvel_traj, void* sensor_traj, const b2_derived* derived, void* stream);

/* Replaces mj.mj_jacSite / mj_jacBody / mj_jacBodyCom / mj_jacSubtreeCom
 * (reference mujoco_template/jacobians.py:44,55,67,79).  jacp/jacr: (3, nv, nenv); jacr may be NULL. */
int b2_jacobian(b2_batch* batch, const b2_state* state, int kind, int objid, void* jacp, void* jacr, void* stream);

/* Replaces mj.mj_inverse + the dense actuator moment (reference mujoco_template/setpoints.py:23-48, steady_ctrl0):
 * qfrc_inverse (nv, nenv) = M qacc + bias - passive - constraint for the prescribed qacc (nv, nenv; NULL = zeros);
 * actuator_moment (nu*nv, nenv), row-major nu x nv per env, may be NULL.  State is not modified. */
int b2_inverse(b2_batch* batch, const b2_state* state, const void* qacc, void* qfrc_inverse, void* actuator_moment, void* stream);

/* On-device LQR control tick (SURVEY.md 8f row 2).  Replaces the per-step arithmetic of the reference's LQR
 * controllers (reference examples/drone/controllers/lqr.py:227-278, examples/humanoid/controllers/lqr.py:153-170):
 * ctrl = clip(ctrl_ref - K [mj_differentiatePos(qpos_ref -> qpos); qvel], ctrlrange) for every env in one launch.
 * b2_lqr_set_gain (synchronous) uploads K (nu x 2nv, row-major), qpos_ref (nq), ctrl_ref (nu), given in double. */
int b2_lqr_set_gain(b2_batch* batch, const double* K, const double* qpos_ref, const double* ctrl_ref);
int b2_lqr_control(b2_batch* batch, const b2_state* state, void* stream);

/* One control tick of the reference's step loop (mujoco_template/env.py:177-191: controller, then (A, B) for a
 * needs_linearization controller, then mj_step) for the whole batch: with use_lqr != 0 the control law set by
 * b2_lqr_set_gain produces the controls (written to state.ctrl); A/B as in b2_linearize at those controls; then one
 * step as in b2_step.  The kernels evaluate the control law themselves, so there is no controller launch.
 * derived == NULL on an Euler model: the step rides in the FD launch (the thread that owns an env's velocity / control
 * columns shares its position stage with the step) plus a small commit launch; the derived arrays of that step can
 * still be obtained afterwards with b2_refresh_derived.  Otherwise: FD launch, then step launch. */
int b2_control_tick(b2_batch* batch, const b2_state* state, const b2_derived* derived, int use_lqr, double eps,
                    int centered, void* A, void* B, void* stream);

/* One mj_step (reference mujoco_template/model.py:56-57) without derived outputs, keeping the pre-step state so that
 * b2_refresh_derived can still produce them on demand: writing ~100 derived reals per env costs more HBM traffic than
 * the step itself, and a rollout that only consumes the state (Env.step(return_obs=False)) never reads them. */
int b2_step_lazy(b2_batch* batch, const b2_state* state, void* stream);

/* Derived arrays of the last b2_control_tick(derived = NULL) / b2_step_lazy: exactly what mj_step leaves in mjData after
 * that step (the forward pass of the pre-step state, which the call kept).  Error if there is no such call. */
int b2_refresh_derived(b2_batch* batch, const b2_derived* derived, void* stream);

/* Replace mj.mj_integratePos / mj.mj_differentiatePos (reference linearization.py:10-13,55,67). */
int b2_integrate_pos(b2_batch* batch, void* qpos, const void* qvel, double dt, void* stream);
int b2_differentiate_pos(b2_batch* batch, void* qvel_out, double dt, const void* qpos1, const void* qpos2, void* stream);

/* End-to-end variant with HOST buffers (pageable or pinned): copies qpos/qvel/ctrl[/warm]
 * host->device, runs `nsteps` steps (optionally one linearization first, as
 * reference env.py:178-190 does per control tick), copies qpos/qvel[/warm][/A,B] back, and
 * synchronises.  A/B may be NULL.  `linearize` is a bit set: B2_HOST_LINEARIZE computes (A, B) before the step;
 * B2_HOST_LQR evaluates the control law of b2_lqr_set_gain on the device first -- host_state.ctrl is then an OUTPUT
 * (the controls that were applied) instead of an input.  host_A / host_B that are page-locked and device-mapped
 * (cudaHostAlloc, cudaHostRegister, torch pin_memory()) are written by the FD kernel directly, with no staging copy in
 * HBM; any other host memory goes through a staged device buffer.  Used by bench.py's e2e leg. */
#define B2_HOST_LINEARIZE 1
#define B2_HOST_LQR 2
#define B2_HOST_ASYNC 4
int b2_step_host(b2_batch* batch, const b2_state* host_state, int nsteps, int linearize, double eps, void* host_A,
                 void* host_B, void* stream);
/* With B2_HOST_ASYNC in `linearize`, b2_step_host returns as soon as its copy / compute pipeline is queued (on streams the
 * batch owns); the host buffers belong to the library until b2_step_host_wait(batch) returns, which is also when their
 * contents are the step's results.  One call in flight per batch.  Two batches driven alternately -- wait(a), submit(a),
 * wait(b), submit(b), ... -- keep the device-to-host link busy with one batch's (A, B) while the other computes
 * (bench.py's e2e leg: the env batch as two half-batches, each a closed loop through its own host buffers). */
int b2_step_host_wait(b2_batch* batch);

/* Measured CUDA-core FMA throughput (TFLOP/s, 2 flops per FMA) of `device` for B2_F64 / B2_F32:
 * the FP-pipe roofline denominator (MEASURED_PEAKS.json only has HBM and bf16 tensor peaks).
 * Synchronous. */
int b2_fp_peak(int precision, int device, double* tflops);

int b2_stream_synchronize(b2_batch* batch, void* stream);

/* b2_lqr_control with a gain of its own for every env (time-varying LQR): K_env is a DEVICE array (nu, 2nv, nenv), env
 * fastest -- the layout b2_dlqr writes -- and qpos_ref / ctrl_ref are those of b2_lqr_set_gain. */
int b2_lqr_control_env(b2_batch* batch, const b2_state* state, const void* K_env, void* stream);

/* Random-rollout controller on the device (BASELINE.json configs #3 / #4: "batched random controls ... generated on
 * device"): ctrl[a, e] ~ U(lo, hi), i.i.d. per call, env and actuator (Philox4x32-10 keyed by (seed, env); the per-env
 * draw counter lives in the batch, so a captured CUDA graph replays with fresh numbers).  With reset_qpos != NULL the
 * same launch applies a rollout driver's episode reset first: an env whose qpos[watch_row] < watch_min restarts from its
 * column of reset_qpos (nq, nenv) / reset_qvel (nv, nenv; NULL = zeros).  Fills the role of a reference Controller
 * (control.py:18-32) for a batch; writes state.ctrl (and the reset states) in place. */
int b2_random_controls(b2_batch* batch, const b2_state* state, double lo, double hi, unsigned long long seed, int watch_row,
                       double watch_min, const void* reset_qpos, const void* reset_qvel, void* stream);

/* Batched discrete-time LQR synthesis on the device: for every env e the stabilising solution P_e of the DARE
 *     P = A'PA - A'PB (R + B'PB)^-1 B'PA + Q
 * and the gain K_e = (R + B'PB)^-1 B'PA (u = -K x) from that env's own (A_e, B_e) -- what the reference's example
 * controllers compute once per system on the host (scipy.linalg.solve_discrete_are + solve:
 * examples/drone/controllers/lqr.py:350-378, examples/humanoid/controllers/lqr.py:114-115).  A (nx, nx, nenv) and
 * B (nx, nu, nenv) are DEVICE arrays in the layout b2_linearize writes (env fastest); K (nu, nx, nenv) and
 * P (nx, nx, nenv) likewise; Q (nx x nx) and R (nu x nu) are HOST arrays, row-major, shared by all envs.  Structured
 * doubling iteration, at most `max_doublings` (2^k Riccati steps), stopped when the relative change of P is <= tol.
 * status (device, nenv ints, may be NULL): doublings used, negative if a pivot underflowed.  Not tied to a batch. */
int b2_dlqr(int device, int precision, const void* A, const void* B, const double* Q, const double* R, int nx, int nu, int nenv,
            int max_doublings, double tol, void* K, void* P, int* status, void* stream);

/* Finite-horizon time-varying LQR about a trajectory, batched: the Riccati backward pass of TV-LQR, iLQR and DDP (without
 * second-order dynamics terms) for every env from its own (A_t, B_t), t = 0 .. nsteps-1.  Deviations are in A's tangent
 * space, dx = [q (-) qbar ; v - vbar] (nx = 2nv for b2_linearize_rollout's output), du = u - ubar, and u = -K dx as in
 * b2_dlqr.  The cost is
 *     J = sum_t [1/2 dx_t'Q dx_t + q_t'dx_t + 1/2 du_t'R du_t + r_t'du_t] + 1/2 dx_T'Qf dx_T + q_T'dx_T
 * and, from P = Qf, s = q_T, for t = nsteps-1 .. 0:
 *     Qx = q_t + A's   Qu = r_t + B's   Qxx = Q + A'PA   Quu = R + B'PB   Qux = B'PA
 *     K_t = (Quu + reg I)^-1 Qux,   k_t = -(Quu + reg I)^-1 Qu          (Cholesky of Quu + reg I)
 *     P <- Qxx + K'Quu K - K'Qux - Qux'K  (symmetrised),   s <- Qx - K'Qu - K'Quu k + Qux'k
 *     dV0 += k'Qu,   dV1 += 1/2 k'Quu k
 * so that the closed-loop control is ubar_t + alpha k_t - K_t dx_t (b2_rollout_feedback), and for a linear system
 * alpha dV0 + alpha^2 dV1 is the change of J that step size alpha brings.  reg = 0 without q / r is plain TV-LQR; for a
 * constant (A, B) and a long horizon K_0 and P0 approach b2_dlqr's K and P.
 * DEVICE arrays, env fastest (element (t, i, j, e) at base[((t*rows + i)*cols + j)*nenv + e]):
 *     A (nsteps, nx, nx, nenv), B (nsteps, nx, nu, nenv)  -- b2_linearize_rollout's layout, read in place
 *     q (nsteps+1, nx, nenv), r (nsteps, nu, nenv)         -- may be NULL (zeros)
 *     K (nsteps, nu, nx, nenv) required;  k (nsteps, nu, nenv), P0 (nx, nx, nenv), dV (2, nenv) may be NULL
 *     status (nenv ints, may be NULL): 0, or -(t+1) when Quu_t + reg I is not positive definite (the first such t from the
 *     end); that env's rows <= t of K and k, its P0 and its dV are then NaN.
 * Q, Qf (nx x nx) and R (nu x nu): HOST arrays, row-major, shared by all envs; kept on the device by content as b2_dlqr
 * keeps its weights, so that repeated calls neither allocate nor copy and can be captured in a CUDA graph.  One launch:
 * a thread per env for (nx, nu) = (2, 1), (4, 1), (4, 2), otherwise a warp per env with its matrices in shared memory.
 * Offsets are 64-bit.  Not tied to a batch.  nsteps, nx, nu or nenv < 1, reg < 0, a bad precision or a NULL A, B, Q, R, Qf
 * or K: B2_ERR_ARG; an (nx, nu) whose workspace exceeds an SM's shared memory: B2_ERR_CAPACITY. */
int b2_tvlqr(int device, int precision, int nsteps, int nx, int nu, int nenv, const void* A, const void* B, const double* Q,
             const double* R, const double* Qf, const void* q, const void* r, double reg, void* K, void* k, void* P0, void* dV,
             int* status, void* stream);

/* Batched recorder sink: one CSV row per selected env and step, in the reference's column layout
 * (reference logging.py:81-247: time_s, qpos.., qvel.., ctrl.., probe columns).  A recorder is a column table
 * { array base (device pointer into a (dim, nenv) state / derived array of the batch), row } plus a selection of env
 * indices; b2_recorder_record gathers one step into `out_slot` (ncol x nsel reals of the batch's precision, env fastest)
 * in ONE launch, on `stream`, without a host synchronisation.  kind 0: array row, 1: the `time` argument, 2: NaN (the
 * `ctrl[none]` column of a model without actuators). */
typedef struct b2_recorder b2_recorder;
typedef struct b2_record_col { const void* base; int row; int kind; } b2_record_col;
int b2_recorder_create(b2_batch* batch, const b2_record_col* cols, int ncol, const int* env_index, int nsel, b2_recorder** out);
int b2_recorder_record(b2_recorder* rec, double time, void* out_slot, void* stream);
void b2_recorder_destroy(b2_recorder* rec);
/* Diagnostic: histogram of the warp engine's queue keys of the last b2_step (16 bins: Newton rounds of the step before,
 * capped at 7; + 8 when the env had constraint rows that couple two branches of the tree).  Synchronises `stream`. */
int b2_warp_queue_histogram(b2_batch* batch, int* hist16, void* stream);
/* number of kernels launched by this library in the calling process (bench gpu_launches) */
long long b2_launch_count(void);
/* size class the model was mapped to: 0 tiny, 1 small, 2 large */
int b2_batch_size_class(const b2_batch* batch);
/* "generic" / "generic-warp" (runtime model image, any MJCF in the subset) or the name of the compiled-in
 * model-specialised kernel set the batch runs on (selected by blob hash; env B2_DISABLE_SPEC=1
 * forces generic) */
const char* b2_batch_kernel_variant(const b2_batch* batch);
const char* b2_last_error(void);
const char* b2_version(void);

#ifdef __cplusplus
}
#endif
#endif
