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
 *    b2_lqr_set_gain); b2_step, b2_forward, b2_linearize, b2_linearize_sensors and b2_jacobian never allocate.
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
