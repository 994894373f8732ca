// What the kernel translation units export: one table of launchers per precision from the generic units, and the
// model-specialised kernel sets that the generated units register at load time (b2_model_create looks a model up by the
// FNV-1a hash of its blob).  All launchers return a cudaError_t as int; count envs, env stride N.
#pragma once
#include <cstddef>
#include <cstdint>

#include "../../include/b2_model_layout.h"
#include "../../include/b2mj.h"

namespace b2 {

// The model-dependent lane-engine launchers, which both the generic and the specialised kernel sets provide.  image / cls:
// the generic kernels' model image and size class; a specialised set ignores both.
struct LaneKernels {
  // gain != null: the control law of b2_lqr_set_gain is evaluated inside the kernel (ctrl becomes an output of step)
  // park != null: the kernel also copies the pre-step state there (b2_step_lazy)
  int (*step)(const void* image, int cls, const b2_state* st, const b2_derived* out, int count, int N, int nsteps, const void* gain,
              const b2_state* park, void* stream);
  // ntask: FD tasks per env (fd_task_count of the model)
  // shadow != null (Euler models): the FD launch also advances every env into the shadow arrays (see k_linearize)
  int (*linearize)(const void* image, int cls, const b2_state* st, int count, int N, int ntask, double eps, int centered, void* A,
                   void* B, const void* gain, const b2_state* shadow, void* stream);
  // b2_linearize_sensors: (A, B) and the sensor Jacobians dsdx / dsdu from the same rollouts.  A specialised set has it only
  // for models with sensors; null otherwise (the call is then b2_linearize)
  int (*linearize_sensors)(const void* image, int cls, const b2_state* st, int count, int N, int ntask, double eps, int centered,
                           void* A, void* B, void* dsdx, void* dsdu, void* stream);
  int (*jacobian)(const void* image, int cls, const b2_state* st, int N, int kind, int objid, void* jacp, void* jacr, void* stream);
  // b2_rollout: per-step controls and the recorded trajectory of every env in one launch (k_rollout)
  int (*rollout)(const void* image, int cls, const b2_state* st, const b2_derived* out, int N, int nsteps, const void* ctrl_seq,
                 void* qpos_traj, void* qvel_traj, void* sensor_traj, void* stream);
  // b2_linearize_rollout: the nominal trajectory (k_nominal_traj), then the FD of every step in one launch
  // (k_linearize_traj); dsdx / dsdu non-null selects the sensor variant, which a specialised set has only for models with
  // sensors
  int (*linearize_rollout)(const void* image, int cls, const b2_state* st, int N, int ntask, int nsteps, const void* ctrl_seq, double eps,
                           int centered, void* A, void* B, void* dsdx, void* dsdu, void* qpos_traj, void* qvel_traj, void* warm_traj,
                           void* sensor_traj, void* stream);
  // b2_rollout_feedback: the time-varying LQR law in front of every step of a rollout, in one launch (k_rollout_feedback)
  int (*rollout_feedback)(const void* image, int cls, const b2_state* st, const b2_derived* out, int N, int nsteps, const void* ctrl_nom,
                          const void* qpos_nom, const void* qvel_nom, const void* K, const void* k, const void* alpha, void* ctrl_traj,
                          void* qpos_traj, void* qvel_traj, void* sensor_traj, void* stream);
};

// The generic kernels of one precision (b2_kernels_impl.cuh).
struct Kernels {
  LaneKernels generic;
  int (*inverse)(const void* image, int cls, const b2_state* st, int N, const void* qacc, void* qfrc, void* moment, void* stream);
  int (*lqr_control)(const void* image, int cls, const b2_state* st, int count, int N, const void* gain, void* stream);
  int (*lqr_control_env)(const void* image, int cls, const b2_state* st, int count, int N, const void* gain, const void* K_env,
                         void* stream);
  int (*integrate_pos)(const void* image, int cls, void* qpos, const void* qvel, double dt, int N, void* stream);
  int (*differentiate_pos)(const void* image, int cls, void* out, double dt, const void* q1, const void* q2, int N, void* stream);
  // model-independent
  int (*commit_state)(const b2_state* st, const b2_state* shadow, int count, int N, int nq, int nv, int nu, void* stream);
  int (*random_controls)(const b2_state* st, int N, int nq, int nv, int nu, double lo, double hi, unsigned long long seed, void* ctr,
                         int watch_row, double watch_min, const void* reset_qpos, const void* reset_qvel, void* stream);
  int (*record_rows)(const void* cols, int ncol, const int* env_index, int nsel, int N, double time, void* out, void* stream);
  int (*dare)(const void* A, const void* B, const void* qr, int nx, int nu, int N, int max_doublings, double tol, void* K, void* P,
              int* status, void* stream);
  double (*fma_peak)(void* stream);
  // the lane engine's model image of a size class: size, and fill on the host
  size_t (*image_bytes)(int cls);
  void (*image_fill)(int cls, const b2m_view* v, const int* disabled, void* host);
  // warp engine (large models)
  int (*warp_plan)(const b2m_view* v, int N, int* out_wpb, int* out_blocks);
  size_t (*warp_scratch_bytes)(const b2m_view* v, int slots);
  size_t (*warp_image_bytes)();
  void (*warp_image_fill)(const b2m_view* v, const int* disabled, void* host);
  size_t (*warp_sort_bytes)(int N);
  int (*warp_step)(const void* image, const b2m_view* v, const b2_state* st, const b2_derived* out, int N, int nsteps, void* jscratch,
                   void* counter, void* sortbuf, int wpb, int blocks, const b2_state* park, void* stream);
  int (*warp_linearize)(const void* image, const b2m_view* v, const b2_state* st, int N, double eps, int centered, void* A, void* B,
                        void* jscratch, void* counter, int wpb, int blocks, void* stream);
  // b2_tvlqr (model-independent): W = Q, R, Qf on the device; returns cudaErrorInvalidValue when one env's workspace does not
  // fit the shared memory of an SM
  int (*tvlqr)(const void* A, const void* B, const void* W, const void* q, const void* r, int nsteps, int nx, int nu, int N, double reg,
               void* K, void* k, void* P0, void* dV, int* status, void* stream);
  // one step's law of b2_rollout_feedback on the lane engine's model image (the warp engine's loop): pointers at step t's rows
  int (*tvlqr_law)(const void* image, int cls, const b2_state* st, int N, const void* ubar, const void* qbar, const void* vbar,
                   const void* K, const void* k, const void* alpha, void* ctrl_row, void* stream);
  // b2_traj_cost on the lane engine's model image: W = Q, R, Qf on the device (the b2_tvlqr block); one launch
  int (*traj_cost)(const void* image, int cls, int N, int nsteps, const void* qpos, const void* qvel, const void* ctrl, const void* qref,
                   const void* vref, const void* uref, const void* W, void* J, void* q, void* r, void* stream);
};
extern const Kernels kernels_f64, kernels_f32;

struct SpecKernels {
  const char* name;
  uint64_t blob_hash;
  size_t blob_size;
  LaneKernels lane[2];  // [0] FP64, [1] FP32
};

void register_spec(const SpecKernels* k);
const SpecKernels* find_spec(uint64_t hash, size_t size);

inline uint64_t fnv1a(const void* data, size_t n) {
  const unsigned char* p = (const unsigned char*)data;
  uint64_t h = 1469598103934665603ull;
  for (size_t i = 0; i < n; i++) { h ^= p[i]; h *= 1099511628211ull; }
  return h;
}

}  // namespace b2
