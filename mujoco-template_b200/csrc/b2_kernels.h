// Host-callable launchers exported by the per-precision kernel translation units.
#pragma once
#include "../../include/b2_model_layout.h"
#include "../../include/b2mj.h"

namespace b2 {
#define B2_DECL(SUF)                                                                                                       \
  double b2k_fma_peak##SUF(void* stream);                                                                                  \
  int b2k_warp_plan##SUF(const b2m_view* v, int N, int* out_wpb, int* out_blocks);                                        \
  size_t b2k_warp_scratch_bytes##SUF(const b2m_view* v, int slots);                                                        \
  size_t b2k_warp_image_bytes##SUF();                                                                                      \
  void b2k_warp_image_fill##SUF(const b2m_view* v, const int* disabled, void* host);                                       \
  size_t b2k_warp_sort_bytes##SUF(int N);                                                                                  \
  int b2k_warp_step##SUF(const void* image, const b2m_view* v, const b2_state* st, const b2_derived* out, int N, int nsteps, void* jscratch, void* counter,  \
                         void* sortbuf, int wpb, int blocks, const b2_state* park, void* stream);                                                                   \
  int b2k_warp_linearize##SUF(const void* image, const b2m_view* v, const b2_state* st, int N, double eps, int centered, void* A, void* B, void* jscratch,  \
                              void* counter, int wpb, int blocks, void* stream);                                                        \
  size_t b2k_image_bytes##SUF(int cls);                                                                                    \
  void b2k_image_fill##SUF(int cls, const b2m_view* v, const int* disabled, void* host);                                   \
  int b2k_step##SUF(const void* image, int cls, const b2_state* st, const b2_derived* out, int count, int N, int nsteps, const void* gain, const b2_state* park, void* stream);                  \
  int b2k_linearize##SUF(const void* image, int cls, const b2_state* st, int count, int N, int ntask, double eps, int centered, void* A, void* B,         \
                         const void* gain, const b2_state* shadow, void* stream);                                                                                    \
  int b2k_linearize_sensors##SUF(const void* image, int cls, const b2_state* st, int count, int N, int ntask, double eps, int centered, void* A,  \
                                 void* B, void* dsdx, void* dsdu, void* stream);                                                                         \
  int b2k_commit_state##SUF(const b2_state* st, const b2_state* shadow, int count, int N, int nq, int nv, int nu, void* stream); \
  int b2k_jacobian##SUF(const void* image, int cls, const b2_state* st, int N, int kind, int objid, void* jacp, void* jacr, void* stream);    \
  int b2k_inverse##SUF(const void* image, int cls, const b2_state* st, int N, const void* qacc, void* qfrc, void* moment, void* stream);     \
  int b2k_lqr_control##SUF(const void* image, int cls, const b2_state* st, int count, int N, const void* gain, void* stream);                           \
  int b2k_dare##SUF(const void* A, const void* B, const void* qr, int nx, int nu, int N, int max_doublings, double tol, void* K, void* P, \
                    int* status, void* stream);                                                                            \
  int b2k_lqr_control_env##SUF(const void* image, int cls, const b2_state* st, int count, int N, const void* gain, const void* K_env, void* stream); \
  int b2k_random_controls##SUF(const b2_state* st, int N, int nq, int nv, int nu, double lo, double hi, unsigned long long seed, void* ctr, \
                               int watch_row, double watch_min, const void* reset_qpos, const void* reset_qvel, void* stream);             \
  int b2k_record_rows##SUF(const void* cols, int ncol, const int* env_index, int nsel, int N, double time, void* out, void* stream); \
  int b2k_integrate_pos##SUF(const void* image, int cls, void* qpos, const void* qvel, double dt, int N, void* stream);                       \
  int b2k_differentiate_pos##SUF(const void* image, int cls, void* out, double dt, const void* q1, const void* q2, int N, void* stream); \
  int b2k_rollout##SUF(const void* image, int cls, const b2_state* st, const b2_derived* out, int N, int nsteps, const void* ctrl_seq, \
                       void* qpos_traj, void* qvel_traj, void* sensor_traj, void* stream);
B2_DECL(_f64)
B2_DECL(_f32)
#undef B2_DECL
}  // namespace b2
