// Kernel templates of the lane engine, parameterised on <arithmetic type T, capacities D,
// model provider M>.  Instantiated by the generic translation units (runtime provider, one per
// precision) and by the generated per-model translation units (static providers).
//
// SoA layout: element (k, e) of a (dim, nenv) array is base[k * nenv + e]; a warp reads 32
// consecutive envs of one component -> fully coalesced 256 B (FP64) transactions.
#pragma once
#include <cuda_runtime.h>

#include <type_traits>

#include "../../include/b2mj.h"
#include "b2_engine.cuh"

// block size of the FD kernel and the minimum resident blocks per SM requested for it (caps registers per thread); the
// generated translation units of small models set their own
#ifndef B2_LIN_THREADS
#define B2_LIN_THREADS 128
#endif
#ifndef B2_LIN_MIN_BLOCKS
#define B2_LIN_MIN_BLOCKS 1
#endif

namespace b2 {

// Runtime providers keep the model image in shared memory and fill it from the per-model image in device memory the launch
// passes (`image`); static providers (generated, everything folded into the instruction stream) have no load().
template <class M> B2_DEV auto model_load(const void* image, int) -> decltype(M::load(image)) { M::load(image); }
template <class M> B2_DEV void model_load(const void*, long) {}

template <typename T> struct StateDev { T *qpos, *qvel, *ctrl, *warm; int* flags; };
template <typename T> struct DerivedDev { T *xpos, *xquat, *xipos, *geom_xpos, *site_xpos, *subtree_com, *qacc, *qfrc_bias, *sensordata; int *ncon, *nefc, *solver_iter; };

template <typename T>
static inline StateDev<T> to_dev(const b2_state* s) {
  StateDev<T> d;
  if (!s) { d.qpos = d.qvel = d.ctrl = d.warm = nullptr; d.flags = nullptr; return d; }
  d.qpos = (T*)s->qpos; d.qvel = (T*)s->qvel; d.ctrl = (T*)s->ctrl; d.warm = (T*)s->qacc_warmstart; d.flags = s->flags;
  return d;
}
template <typename T>
static inline DerivedDev<T> to_dev(const b2_derived* o) {
  DerivedDev<T> d;
  memset(&d, 0, sizeof(d));
  if (o) {
    d.xpos = (T*)o->xpos; d.xquat = (T*)o->xquat; d.xipos = (T*)o->xipos; d.geom_xpos = (T*)o->geom_xpos;
    d.site_xpos = (T*)o->site_xpos; d.subtree_com = (T*)o->subtree_com; d.qacc = (T*)o->qacc;
    d.qfrc_bias = (T*)o->qfrc_bias; d.sensordata = (T*)o->sensordata; d.ncon = o->ncon; d.nefc = o->nefc; d.solver_iter = o->solver_iter;
  }
  return d;
}

template <typename T, class D, class M>
B2_DEV void load_state(LaneEnv<T, D, M>& env, const StateDev<T>& st, int N, int e) {  // N: env stride (leading dimension)
  B2_UNROLL
  for (int k = 0; k < M::nq(); k++) env.qpos[k] = st.qpos[(size_t)k * N + e];
  B2_UNROLL
  for (int k = 0; k < M::nv(); k++) env.qvel[k] = st.qvel[(size_t)k * N + e];
  B2_UNROLL
  for (int k = 0; k < M::nu(); k++) env.ctrl[k] = st.ctrl[(size_t)k * N + e];
  B2_UNROLL
  for (int k = 0; k < M::nv(); k++) env.warm[k] = st.warm ? st.warm[(size_t)k * N + e] : T(0);
}
template <typename T, class D, class M>
B2_DEV void store_derived(LaneEnv<T, D, M>& env, const DerivedDev<T>& o, int N, int e) {
  if (o.sensordata && M::nsensor() > 0) {
    T sd[D::NSD];
    env.sensors(sd);
    B2_UNROLL
    for (int k = 0; k < M::nsensordata(); k++) o.sensordata[(size_t)k * N + e] = sd[k];
  }
  if (o.xpos) { B2_UNROLL for (int k = 0; k < 3 * M::nbody(); k++) o.xpos[(size_t)k * N + e] = env.xpos[k]; }
  if (o.xquat) { B2_UNROLL for (int k = 0; k < 4 * M::nbody(); k++) o.xquat[(size_t)k * N + e] = env.xquat[k]; }
  if (o.xipos) { B2_UNROLL for (int k = 0; k < 3 * M::nbody(); k++) o.xipos[(size_t)k * N + e] = env.xipos[k]; }
  if (o.geom_xpos) {
    B2_UNROLL
    for (int g = 0; g < M::ngeom(); g++) { T p[3], R[9]; env.geom_pose(g, p, R); for (int k = 0; k < 3; k++) o.geom_xpos[(size_t)(3 * g + k) * N + e] = p[k]; }
  }
  if (o.site_xpos) {
    B2_UNROLL
    for (int s = 0; s < M::nsite(); s++) { T p[3], R[9]; env.site_pose(s, p, R); for (int k = 0; k < 3; k++) o.site_xpos[(size_t)(3 * s + k) * N + e] = p[k]; }
  }
  if (o.subtree_com) { B2_UNROLL for (int k = 0; k < 3 * M::nbody(); k++) o.subtree_com[(size_t)k * N + e] = env.com[k]; }
  if (o.qacc) { B2_UNROLL for (int k = 0; k < M::nv(); k++) o.qacc[(size_t)k * N + e] = env.qacc[k]; }
  if (o.qfrc_bias) { B2_UNROLL for (int k = 0; k < M::nv(); k++) o.qfrc_bias[(size_t)k * N + e] = env.f_bias[k]; }
  if (o.ncon) o.ncon[e] = env.ncon;
  if (o.nefc) o.nefc[e] = env.nefc;
  if (o.solver_iter) o.solver_iter[e] = env.niter;
}

// u = clip(u_ref - K [qpos (-) qpos_ref ; qvel], ctrlrange) for one env whose state is in registers.
// gain: K (nu x 2nv row-major), then qpos_ref (nq), then ctrl_ref (nu), shared by all envs.
template <typename T, class D, class M>
B2_DEV void lqr_law(const LaneEnv<T, D, M>& env, const T* q, const T* v, const T* __restrict__ gain, T* u_out) {
  const int nq = M::nq(), nv = M::nv(), nu = M::nu();
  T qr[D::NQ], x[2 * D::NV];
  B2_UNROLL
  for (int k = 0; k < nq; k++) qr[k] = gain[nu * 2 * nv + k];
  env.differentiate_pos(x, T(1), qr, q);
  B2_UNROLL
  for (int k = 0; k < nv; k++) x[nv + k] = v[k];
  B2_UNROLL
  for (int a = 0; a < nu; a++) {
    T u = gain[nu * 2 * nv + nq + a];
    B2_UNROLL
    for (int k = 0; k < 2 * nv; k++) u -= gain[a * 2 * nv + k] * x[k];
    if (M::actuator_ctrllimited(a)) u = tclip(u, M::actuator_ctrlrange(2 * a), M::actuator_ctrlrange(2 * a + 1));
    u_out[a] = u;
  }
}

// nsteps x mj_step with ctrl held; nsteps == 0 means mj_forward (no integration).
// The step loop is rolled: one inlined copy of the physics per kernel.
template <typename T, class D, class M>
__global__ void __launch_bounds__(128, 1) k_step(StateDev<T> st, DerivedDev<T> out, int want_derived, int count, int N, int nsteps, const T* __restrict__ gain,
                                                 StateDev<T> park, const void* image = nullptr) {
  model_load<M>(image, 0);
  // count envs are processed; N is the env stride of the SoA arrays (count < N for a chunk of a larger batch)
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= count) return;
  RowStore<T, D> rows;
  LaneEnv<T, D, M> env(rows);
  // Register-starved static models (LaneEnv::kLateMass: the drone) compute mass matrix and actuator moments in the
  // acceleration stage (see LaneEnv): 2 % faster and no spill write-back left in the DRAM traffic of the launch.
  // (Measured on top of it and dropped, profiles/ab_drone_late_r03l.txt: every stage re-loading the state it consumes
  // from the SoA arrays instead of holding it, +4 %; reading the warm start only when the step has constraint rows, +2 %.)
  constexpr bool kLate = LaneEnv<T, D, M>::kLateMass;
  load_state(env, st, N, e);
  if (gain) {  // device-resident control law (b2_control_tick): ctrl is an output of this launch
    lqr_law(env, env.qpos, env.qvel, gain, env.ctrl);
    B2_UNROLL
    for (int k = 0; k < M::nu(); k++) st.ctrl[(size_t)k * N + e] = env.ctrl[k];
  }
  if (park.qpos) {  // b2_step_lazy: keep the pre-step state (it is in registers anyway) for b2_refresh_derived
    B2_UNROLL
    for (int k = 0; k < M::nq(); k++) park.qpos[(size_t)k * N + e] = env.qpos[k];
    B2_UNROLL
    for (int k = 0; k < M::nv(); k++) { park.qvel[(size_t)k * N + e] = env.qvel[k]; park.warm[(size_t)k * N + e] = env.warm[k]; }
    B2_UNROLL
    for (int k = 0; k < M::nu(); k++) park.ctrl[(size_t)k * N + e] = env.ctrl[k];
  }
  const int total = nsteps > 0 ? nsteps : 1;
  B2_NOUNROLL
  for (int s = 0; s < total; s++) {
    env.check_state();
    // a diverged env (NaN or |x| > 1e10: upstream would silently reset it) is flagged and frozen: stepping it on would
    // only burn the Newton iteration cap on a meaningless state, and hold up the other 31 lanes of its warp
    if (env.flags & 3) {
      if (st.flags) st.flags[e] |= env.flags;
      return;
    }
    env.template forward_position<kLate>();
    env.forward_velocity();
    env.template forward_acc<kLate>();
    B2_UNROLL
    for (int k = 0; k < M::nv(); k++) if (!(fabs(env.qacc[k]) <= T(1e10))) env.flags |= 4;
    if (want_derived && s == total - 1) store_derived(env, out, N, e);
    if (nsteps > 0) { if (M::integrator() == 1) env.rk4(); else env.euler(); }
  }
  if (nsteps > 0) {
    B2_UNROLL
    for (int k = 0; k < M::nq(); k++) st.qpos[(size_t)k * N + e] = env.qpos[k];
    B2_UNROLL
    for (int k = 0; k < M::nv(); k++) st.qvel[(size_t)k * N + e] = env.qvel[k];
  }
  // qacc_warmstart <- qacc at the end of the constraint stage (upstream mj_fwdConstraint: "save result for next step
  // warmstart"), i.e. by mj_forward too -- which is why mjd_transitionFD saves and restores it around every rollout
  if (st.warm) { B2_UNROLL for (int k = 0; k < M::nv(); k++) st.warm[(size_t)k * N + e] = env.warm[k]; }
  if (st.flags && env.flags) st.flags[e] |= env.flags;
}
// Host launchers of k_step, k_linearize and k_jacobian, shared by the generic and the generated translation units: they
// own the block size and the grid.  image: the runtime provider's model image (null for a static provider).
// (Deduced return types: a launcher, and with it its kernel, is instantiated where it is called rather than at the end of
// the translation unit, so the kernels keep their place in the module; cicc's inlining, and so the SASS of the other
// kernels of the module, depends on that order.)
template <typename T, class D, class M>
auto launch_step(const void* image, const b2_state* st, const b2_derived* out, int count, int N, int nsteps, const void* gain,
                 const b2_state* park, void* stream) {
  const int threads = 128, blocks = (count + threads - 1) / threads;
  k_step<T, D, M><<<blocks, threads, 0, (cudaStream_t)stream>>>(to_dev<T>(st), to_dev<T>(out), out != nullptr, count, N, nsteps, (const T*)gain,
                                                                to_dev<T>(park), image);
  return (int)cudaGetLastError();
}

// The nominal state of a thread's env is re-read from the SoA arrays at the start of every rollout (L1/L2 hits) rather
// than held in registers: ~14 fewer live registers across the physics, which is what the 168-register budget of three
// resident blocks is short of.  The controls are the exception (they may come from the control law, not from st.ctrl).
// (The addresses are left to the compiler: the specialised cartpole kernel keeps all six in registers already, and
// per-thread base pointers with a stride of their own raised the drone group thread's spill loads; see DESIGN.md §3.)
template <typename T>
struct NominalInMemory {
  static constexpr bool kSens = false;
  StateDev<T> st;
  int N, e;
  const T* u0;
  B2_DEV void set(const T* qpos, const T* qvel, const T* warm, int n, int ee) {
    st.qpos = (T*)qpos; st.qvel = (T*)qvel; st.warm = (T*)warm; st.ctrl = nullptr; st.flags = nullptr; N = n; e = ee;
  }
  B2_DEV T q(int k) const { return __ldg(st.qpos + (size_t)k * N + e); }
  B2_DEV T v(int k) const { return __ldg(st.qvel + (size_t)k * N + e); }
  B2_DEV T u(int k) const { return u0[k]; }
  B2_DEV T w(int k) const { return st.warm ? __ldg(st.warm + (size_t)k * N + e) : T(0); }
};
// ... plus the outputs of the sensor Jacobians (k_linearize<..., SENS = true>) and fd_column's place in them.  (Kept in the
// accessor rather than as arguments and locals of fd_column: the instantiations without sensors then compile to exactly
// the code they had before the sensor variant existed.)
template <typename T>
struct NominalWithSensors : NominalInMemory<T> {
  static constexpr bool kSens = true;
  T *dsdx, *dsdu;
  mutable T* col;      // entry (0, c, e) of the current column in dsdx / dsdu, or null
  mutable int ncol;    // columns of that array
};

// One column of the FD linearisation for env e -- c < nv: tangent-space position column, c < 2nv: velocity column, else
// control column c - 2nv -- or, with nominal = true, the unperturbed step itself, which leaves the advanced state in
// env.qpos / env.qvel / env.warm.  nom: accessor of the env's nominal state.
// With S::kSens (NominalWithSensors) the same rollouts also give the column of the sensor Jacobians, nom.dsdx =
// d sensordata / dx (nsensordata, 2nv, N) for state columns and nom.dsdu = d sensordata / du (nsensordata, nu, N) for
// control columns (either may be null).
template <typename T, class D, class M, class S>
B2_DEV void fd_column(LaneEnv<T, D, M>& env, const S& nom, int c, bool nominal,
                      T eps, T inv_eps, int centered, int N, int e, T* A, T* B, int& last) {
  constexpr int NQ = D::NQ, NV = D::NV;
  const int nq = M::nq(), nv = M::nv(), nu = M::nu(), ndx = 2 * nv;
  T s1[NQ + NV], s2[NQ + NV], col[2 * NV];  // the two end points of the difference quotient
  // Without quaternion coordinates (nq == nv) the tangent difference is a plain subtraction: the end points are summed with
  // their signs as they arrive (fma with +-1: the same value as s2 - s1) instead of being kept apart by selects.
  const bool scalar_only = nq == nv;
  T dacc[2 * NV];
  B2_UNROLL
  for (int k = 0; k < 2 * nv; k++) dacc[k] = 0;
  // The column, decided once: which sides of the quotient exist (ctrlrange one-sidedness as mjd_transitionFD) ...
  bool fwd = !nominal, back = !nominal && centered != 0;
  if (!nominal && c >= ndx) {
    const int i = c - ndx;
    int lim = 0;
    T lo = 0, hi = 0, u = 0;
    B2_UNROLL
    for (int a = 0; a < nu; a++)
      if (a == i) { lim = M::actuator_ctrllimited(a); lo = M::actuator_ctrlrange(2 * a); hi = M::actuator_ctrlrange(2 * a + 1); u = nom.u(a); }
    fwd = !lim || (u >= lo && u <= hi && u + eps >= lo && u + eps <= hi);
    back = (centered || !fwd) && (!lim || (u - eps >= lo && u - eps <= hi && u >= lo && u <= hi));
  }
  // ... and so its rollouts: the first is the plus side (minus when only that exists), the second the opposite side
  // (centred) or the nominal step (one-sided); the env advance is one nominal rollout.  slot: the perturbed entry of
  // [dq; v; u] (the column index itself), -1 for none.  to2 / sg: the rollout's end and sign in the quotient (plus -> s2,
  // minus -> s1, the nominal step -> whichever end the one-sided quotient is missing).
  const bool both = fwd && back;
  const int nroll = nominal ? 1 : (fwd || back ? 2 : 0);
  int slot = nominal ? -1 : c;
  T delta = fwd ? eps : -eps;
  // Stage skips under Euler: a rollout at the nominal qpos (velocity / control columns, the advance) reuses the position
  // stage of the thread's previous rollout when that one also ran at the nominal qpos (last: the thread's last column
  // with rollouts, -1 before the first), and at the nominal qvel too (control columns, the advance) its velocity stage.
  // bit 0: skip the position stage, bit 1: the velocity stage; for this column's first rollout, then for the rest.
  const bool euler = M::integrator() == 0;
  const bool reuse_pos = euler && (nominal || c >= nv), reuse_vel = euler && (nominal || c >= ndx);
  int skip = (reuse_pos && last >= nv ? 1 : 0) | (reuse_vel && last >= ndx ? 2 : 0);
  const int skip_rest = (reuse_pos ? 1 : 0) | (reuse_vel ? 2 : 0);
  if (nroll > 0) last = c;
  // SENS: the column's sensor entries live in the output array itself, not in registers (the group thread of the drone is
  // at the 255-register limit already).  Each (r, c, e) entry has one owning thread: its first rollout stores the reading
  // with its sign, its second adds its own and scales, so the entry is (s2 - s1) * ih -- the plain difference quotient,
  // with no tangent-space handling (framequat components included), as upstream mjd_stepFD differences sensordata.
  const T ih = both ? T(0.5) * inv_eps : inv_eps;
  if constexpr (S::kSens) {
    nom.col = nullptr;
    if (!nominal) {
      nom.col = c < ndx ? nom.dsdx : nom.dsdu;
      nom.ncol = c < ndx ? ndx : nu;
      if (nom.col) nom.col += (size_t)(c < ndx ? c : c - ndx) * N + e;
    }
  }
  // rolled rollout loop: the physics is instantiated once; all array indices stay static
  B2_NOUNROLL
  for (int ro = 0; ro < nroll; ro++) {
    // the nominal state, then the perturbation as one update of entry `slot`
    if (scalar_only) {
      B2_UNROLL
      for (int k = 0; k < nq; k++) { T x = nom.q(k); if (k == slot) x += delta; env.qpos[k] = x; }
    } else {
      B2_UNROLL
      for (int k = 0; k < nq; k++) env.qpos[k] = nom.q(k);
      if ((unsigned)slot < (unsigned)nv) {
        T dp[NV];
        B2_UNROLL
        for (int k = 0; k < nv; k++) dp[k] = (k == slot) ? T(1) : T(0);
        env.integrate_pos(env.qpos, dp, delta);
      }
    }
    B2_UNROLL
    for (int k = 0; k < nv; k++) { T x = nom.v(k); if (nv + k == slot) x += delta; env.qvel[k] = x; env.warm[k] = nom.w(k); }
    B2_UNROLL
    for (int k = 0; k < nu; k++) { T x = nom.u(k); if (ndx + k == slot) x += delta; env.ctrl[k] = x; }
    // one mj_step
    if (!(skip & 1)) env.forward_position();
    if (!(skip & 2)) env.forward_velocity();
    env.forward_acc();
    B2_UNROLL
    for (int k = 0; k < nv; k++) if (!(fabs(env.qacc[k]) <= T(1e10))) env.flags |= 4;
    const bool to2 = (ro == 0) == fwd;
    const T sg = to2 ? T(1) : T(-1);
    if constexpr (S::kSens) {
      // this rollout's sensordata: its forward pass at the perturbed input state, before integration (RK4: the first stage,
      // as mj_step leaves it).  sensors() uses spat as scratch; nothing the skipped stages reuse lives there -- the
      // velocity stage's only use of it is as bias_forces' scratch.
      if (nom.col) {
        T sd[D::NSD];
        env.sensors(sd);
        B2_UNROLL
        for (int r = 0; r < M::nsensordata(); r++) {
          T* p = nom.col + (size_t)r * nom.ncol * N;
          *p = ro == 0 ? sg * sd[r] : fma(sg, sd[r], *p) * ih;
        }
      }
    }
    if (M::integrator() == 1) env.rk4(); else env.euler();
    if (scalar_only) {
      B2_UNROLL
      for (int k = 0; k < 2 * nv; k++) dacc[k] = fma(sg, k < nv ? env.qpos[k < nv ? k : 0] : env.qvel[k >= nv ? k - nv : 0], dacc[k]);
    } else {
      B2_UNROLL
      for (int k = 0; k < nq + nv; k++) {
        const T val = k < nq ? env.qpos[k < nq ? k : 0] : env.qvel[k >= nq ? k - nq : 0];
        if (to2) s2[k] = val; else s1[k] = val;
      }
    }
    // the second rollout
    skip = skip_rest;
    delta = -delta;
    if (!both) slot = -1;
  }
  if (nominal) return;
  if (nroll > 0) {
    // difference quotient with the reciprocal step (1 / (2 eps) = 0.5 / eps exactly): no division per entry
    if (scalar_only) {
      B2_UNROLL
      for (int k = 0; k < 2 * nv; k++) col[k] = dacc[k] * ih;
    } else {
      env.differentiate_pos(col, T(1), s1, s2);
      B2_UNROLL
      for (int k = 0; k < nv; k++) { col[k] *= ih; col[nv + k] = (s2[nq + k] - s1[nq + k]) * ih; }
    }
  } else {
    B2_UNROLL
    for (int k = 0; k < ndx; k++) col[k] = 0;
    if constexpr (S::kSens) {
      if (nom.col) { B2_UNROLL for (int r = 0; r < M::nsensordata(); r++) nom.col[(size_t)r * nom.ncol * N] = 0; }
    }
  }
  if (c < ndx) { if (A) { B2_UNROLL for (int r = 0; r < ndx; r++) A[((size_t)r * ndx + c) * N + e] = col[r]; } }
  else if (B) { B2_UNROLL for (int r = 0; r < ndx; r++) B[((size_t)r * nu + (c - ndx)) * N + e] = col[r]; }
}

// Centred / one-sided finite differences of one step.  Columns 0..nv-1 perturb tangent-space position, nv..2nv-1
// velocity, 2nv..2nv+nu-1 control.  Replaces mjd_transitionFD (reference mujoco_template/linearization.py:16-35): state
// and qacc_warmstart of every rollout start from the saved nominal values; control columns fall back to one-sided
// differences at the ctrlrange bounds.
// Work split: under Euler the velocity and control columns all share the position stage of the nominal qpos, so a
// thread takes a group of up to B2_FD_GROUP of them, runs that stage once and then their rollouts (tasks 0..groups-1,
// launched first: they are the longest); each position column is a thread of its own (two full rollouts).  Larger
// groups save more position stages but serialise more rollouts in one thread.  RK4 models have nothing to share between
// columns: one thread per (env, column).  fd_task_count (b2_model_dev.cuh) gives the threads per env.
// (Splitting the launch into a kernel for the groups and one for the position columns, each with its own register budget,
// was measured on the cartpole tick and rejected: profiles/ab_cartpole_lin_split_r03c.txt.)
// SENS (b2_linearize_sensors): the rollouts also produce the sensor Jacobians dsdx (nsensordata, 2nv, N) and dsdu
// (nsensordata, nu, N), layout as A / B; launched with gain == nullptr and no shadow (no control law, no env advance).
template <typename T, class D, class M, bool SENS = false>
__global__ void __launch_bounds__(B2_LIN_THREADS, B2_LIN_MIN_BLOCKS) k_linearize(StateDev<T> st, int count, int N, T eps, int centered, T* A, T* B, const T* __restrict__ gain,
                                                                                 StateDev<T> shadow, const void* image = nullptr, T* dsdx = nullptr, T* dsdu = nullptr) {
  model_load<M>(image, 0);
  const int nq = M::nq(), nv = M::nv(), nu = M::nu(), ndx = 2 * nv;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int ntask = fd_task_count(M::integrator(), nv, nu);
  const long long total = (long long)count * ntask;
  if (idx >= total) return;
  // count envs, env stride N; task-major.  32-bit division when the launch fits (a 64-bit one is ~100 instructions)
  int e, task;
  if (total <= 0x7fffffffLL) { const unsigned u = (unsigned)idx; task = (int)(u / (unsigned)count); e = (int)(u - (unsigned)task * (unsigned)count); }
  else { task = (int)(idx / count); e = (int)(idx % count); }
  RowStore<T, D> rows;
  LaneEnv<T, D, M> env(rows);
  T u0[D::NU];
  if (gain) {  // device-resident control law: linearise about the controls it produces (k_step applies the same law)
    T q[D::NQ], v[D::NV];
    B2_UNROLL
    for (int k = 0; k < nq; k++) q[k] = st.qpos[(size_t)k * N + e];
    B2_UNROLL
    for (int k = 0; k < nv; k++) v[k] = st.qvel[(size_t)k * N + e];
    lqr_law(env, q, v, gain, u0);
  } else {
    B2_UNROLL
    for (int k = 0; k < nu; k++) u0[k] = st.ctrl[(size_t)k * N + e];
  }
  typedef typename std::conditional<SENS, NominalWithSensors<T>, NominalInMemory<T>>::type Nominal;
  Nominal nom;
  nom.set(st.qpos, st.qvel, st.warm, N, e);
  nom.u0 = u0;
  if constexpr (SENS) { nom.dsdx = dsdx; nom.dsdu = dsdu; }
  const bool grouped = M::integrator() == 0;  // not a constant expression for the runtime provider
  const int groups = fd_group_count(nv, nu);
  int c0 = task, c1 = task + 1;
  if (grouped) {
    if (task < groups) { c0 = nv + task * B2_FD_GROUP; c1 = c0 + B2_FD_GROUP < ndx + nu ? c0 + B2_FD_GROUP : ndx + nu; }
    else { c0 = task - groups; c1 = c0 + 1; }
  }
  // shadow.qpos != null (grouped form only): the thread of the velocity / control columns also advances the env -- its
  // position stage is the step's -- and leaves the new state in the shadow arrays (the other threads of the env still
  // read the nominal state); k_commit_state swaps the two afterwards
  const bool advance = grouped && task == 0 && shadow.qpos != nullptr;
  int last = -1;
  const T inv_eps = T(1) / eps;
  // mj_checkPos / mj_checkVel once on the nominal state (an eps perturbation of a finite state is finite)
  B2_UNROLL
  for (int k = 0; k < nq; k++) env.qpos[k] = nom.q(k);
  B2_UNROLL
  for (int k = 0; k < nv; k++) env.qvel[k] = nom.v(k);
  env.check_state();
  // a diverged env is flagged and frozen, as in k_step: its "advanced" state is the state it has (one copy of the stores)
  const bool frozen = advance && (env.flags & 3) != 0;
  B2_NOUNROLL
  for (int c = c0; c < c1 + (advance ? 1 : 0) && !frozen; c++) {
    const bool nominal = c == c1;  // the advance comes after the group's columns, on the same position stage
    fd_column(env, nom, nominal ? ndx + nu : c, nominal, eps, inv_eps, centered, N, e, A, B, last);
  }
  if (advance) {
    B2_UNROLL
    for (int k = 0; k < nq; k++) shadow.qpos[(size_t)k * N + e] = frozen ? nom.q(k) : env.qpos[k];
    B2_UNROLL
    for (int k = 0; k < nv; k++) { shadow.qvel[(size_t)k * N + e] = frozen ? nom.v(k) : env.qvel[k]; shadow.warm[(size_t)k * N + e] = frozen ? nom.w(k) : env.warm[k]; }
    B2_UNROLL
    for (int k = 0; k < nu; k++) shadow.ctrl[(size_t)k * N + e] = u0[k];
  }
  if (st.flags && env.flags) atomicOr(st.flags + e, env.flags);
}
// ntask: FD threads per env, fd_task_count of the model (an argument: a runtime provider's accessors read shared memory).
// The block size is the one the kernel's __launch_bounds__ were compiled for.
template <typename T, class D, class M, bool SENS = false>
auto launch_linearize(const void* image, const b2_state* st, int count, int N, int ntask, double eps, int centered, void* A, void* B,
                      const void* gain, const b2_state* shadow, void* dsdx, void* dsdu, void* stream) {
  const long long total = (long long)count * ntask;
  const int blocks = (int)((total + B2_LIN_THREADS - 1) / B2_LIN_THREADS);
  k_linearize<T, D, M, SENS><<<blocks, B2_LIN_THREADS, 0, (cudaStream_t)stream>>>(to_dev<T>(st), count, N, (T)eps, centered, (T*)A, (T*)B, (const T*)gain,
                                                                                  to_dev<T>(shadow), image, (T*)dsdx, (T*)dsdu);
  return (int)cudaGetLastError();
}

// After a launch that advanced envs into the shadow arrays: swap state and shadow (rows of count elements, row stride N).
// The state arrays then hold the new state and the shadow the pre-step one, from which b2_refresh_derived can still
// produce the derived arrays mj_step would have left behind.
template <typename T>
__global__ void __launch_bounds__(256) k_commit_state(StateDev<T> st, StateDev<T> shadow, int count, int N, int nq, int nv, int nu) {
  // blockIdx.y: row of the concatenated [qpos; qvel; warm; ctrl]; x: envs (two per thread, 16-byte accesses when aligned)
  int row = blockIdx.y;
  T *a, *b;
  bool swap = true;
  if (row < nq) { a = st.qpos; b = shadow.qpos; }
  else if ((row -= nq) < nv) { a = st.qvel; b = shadow.qvel; }
  else if ((row -= nv) < nv) { a = st.warm; b = shadow.warm; if (!a) return; }
  else { row -= nv; a = st.ctrl; b = shadow.ctrl; swap = false; }  // applied controls: both sides keep them
  a += (size_t)row * N; b += (size_t)row * N;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
    const T x = a[i];
    a[i] = b[i];
    if (swap) b[i] = x;
  }
}

// point Jacobians from the current qpos (mj_jacSite/Body/BodyCom/SubtreeCom)
template <typename T, class D, class M>
__global__ void __launch_bounds__(128) k_jacobian(StateDev<T> st, int N, int kind, int objid, T* jacp, T* jacr, const void* image = nullptr) {
  model_load<M>(image, 0);
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N) return;
  RowStore<T, D> rows;
  LaneEnv<T, D, M> env(rows);
  const int nv = M::nv();
  B2_UNROLL
  for (int k = 0; k < M::nq(); k++) env.qpos[k] = st.qpos[(size_t)k * N + e];
  env.kinematics();
  env.com_frame();
  T jp[3 * D::NV], jr[3 * D::NV];
  B2_UNROLL
  for (int k = 0; k < 3 * nv; k++) { jp[k] = 0; jr[k] = 0; }
  auto put = [&](int d, const T* p, const T* r) {
    for (int a = 0; a < 3; a++) { jp[a * nv + d] = p[a]; jr[a * nv + d] = r[a]; }
  };
  if (kind == B2_JAC_SITE) { T sp[3], sR[9]; env.compute_site_pose(objid, sp, sR); env.for_jac(M::site_bodyid(objid), sp, put); }
  else if (kind == B2_JAC_BODY) env.for_jac(objid, env.xpos + 3 * objid, put);
  else if (kind == B2_JAC_BODYCOM) env.for_jac(objid, env.xipos + 3 * objid, put);
  else {
    B2_NOUNROLL
    for (int b = objid; b < M::nbody(); b++) {
      if (b > objid && M::body_parentid(b) < objid) break;
      const T mass = M::body_mass(b);
      env.for_jac(b, env.xipos + 3 * b, [&](int d, const T* p, const T*) {
        for (int a = 0; a < 3; a++) jp[a * nv + d] += p[a] * mass;
      });
    }
    const T inv = T(1) / M::body_subtreemass(objid);
    B2_UNROLL
    for (int k = 0; k < 3 * nv; k++) jp[k] *= inv;
  }
  if (jacp) { B2_UNROLL for (int k = 0; k < 3 * nv; k++) jacp[(size_t)k * N + e] = jp[k]; }
  if (jacr) { B2_UNROLL for (int k = 0; k < 3 * nv; k++) jacr[(size_t)k * N + e] = jr[k]; }
}
template <typename T, class D, class M>
auto launch_jacobian(const void* image, const b2_state* st, int N, int kind, int objid, void* jacp, void* jacr, void* stream) {
  const int threads = 128, blocks = (N + threads - 1) / threads;
  k_jacobian<T, D, M><<<blocks, threads, 0, (cudaStream_t)stream>>>(to_dev<T>(st), N, kind, objid, (T*)jacp, (T*)jacr, image);
  return (int)cudaGetLastError();
}

// mj_inverse for a prescribed acceleration (steady_ctrl0: reference mujoco_template/setpoints.py:23-30);
// optionally exports the dense actuator moment matrix (nu x nv) of every env
template <typename T, class D, class M>
__global__ void __launch_bounds__(128) k_inverse(StateDev<T> st, int N, const T* qacc, T* qfrc, T* moment, const void* image = nullptr) {
  model_load<M>(image, 0);
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N) return;
  RowStore<T, D> rows;
  LaneEnv<T, D, M> env(rows);
  load_state(env, st, N, e);
  T acc[D::NV], out[D::NV];
  for (int k = 0; k < M::nv(); k++) acc[k] = qacc ? qacc[(size_t)k * N + e] : T(0);
  env.inverse(acc, out);
  for (int k = 0; k < M::nv(); k++) qfrc[(size_t)k * N + e] = out[k];
  if (moment) for (int k = 0; k < M::nu() * M::nv(); k++) moment[(size_t)k * N + e] = env.act_moment[k];
}

// Fused LQR control tick for every env: u = clip(u_ref - K [qpos (-) qpos_ref ; qvel], ctrlrange), where (-) is the
// tangent-space difference (mj_differentiatePos, so free-joint quaternions are handled).  One launch replaces
// the per-step controller arithmetic of the reference's LQR controllers
// (reference examples/drone/controllers/lqr.py:227-278, examples/humanoid/controllers/lqr.py:153-170).
// gain: K (nu x 2nv row-major), then qpos_ref (nq), then ctrl_ref (nu), shared by all envs.
template <typename T, class D, class M>
__global__ void __launch_bounds__(128) k_lqr_control(StateDev<T> st, int count, int N, const T* __restrict__ gain, const void* image = nullptr) {
  model_load<M>(image, 0);
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= count) return;
  RowStore<T, D> rows;
  LaneEnv<T, D, M> env(rows);
  T q[D::NQ], v[D::NV], u[D::NU];
  for (int k = 0; k < M::nq(); k++) q[k] = st.qpos[(size_t)k * N + e];
  for (int k = 0; k < M::nv(); k++) v[k] = st.qvel[(size_t)k * N + e];
  lqr_law(env, q, v, gain, u);
  for (int a = 0; a < M::nu(); a++) st.ctrl[(size_t)a * N + e] = u[a];
}

// The same law with a gain of its own for every env (time-varying LQR: K_e re-synthesised from the env's latest (A, B) by
// b2_dlqr): K_env (nu, 2nv, N) env fastest; qpos_ref / ctrl_ref from the shared gain block.
template <typename T, class D, class M>
__global__ void __launch_bounds__(128) k_lqr_control_env(StateDev<T> st, int count, int N, const T* __restrict__ gain, const T* __restrict__ K_env,
                                                         const void* image = nullptr) {
  model_load<M>(image, 0);
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= count) return;
  RowStore<T, D> rows;
  LaneEnv<T, D, M> env(rows);
  const int nq = M::nq(), nv = M::nv(), nu = M::nu();
  T q[D::NQ], v[D::NV], u[D::NU], g[D::NU * 2 * D::NV + D::NQ + D::NU];
  for (int k = 0; k < nu * 2 * nv; k++) g[k] = K_env[(size_t)k * N + e];
  for (int k = 0; k < nq + nu; k++) g[nu * 2 * nv + k] = gain[nu * 2 * nv + k];
  for (int k = 0; k < nq; k++) q[k] = st.qpos[(size_t)k * N + e];
  for (int k = 0; k < nv; k++) v[k] = st.qvel[(size_t)k * N + e];
  lqr_law(env, q, v, g, u);
  for (int a = 0; a < nu; a++) st.ctrl[(size_t)a * N + e] = u[a];
}

// Random-rollout controller (BASELINE configs #3 / #4: controls U(lo, hi) i.i.d. per step, env and actuator, drawn on the
// device) fused with the episode reset a batched rollout driver applies: an env whose qpos[watch_row] has dropped below
// watch_min starts again from its row of reset_qpos / reset_qvel.  Philox4x32-10 keyed by (seed, env), counter = the env's
// own draw count (kept in ctr[], so a captured graph replays with fresh numbers).  One launch instead of five tensor ops.
B2_DEV void philox4x32_10(unsigned c0, unsigned c1, unsigned c2, unsigned c3, unsigned k0, unsigned k1, unsigned* out) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const unsigned hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0, hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const unsigned n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
template <typename T>
__global__ void __launch_bounds__(256) k_random_controls(StateDev<T> st, int N, int nq, int nv, int nu, T lo, T hi, unsigned long long seed,
                                                         unsigned* __restrict__ ctr, int watch_row, T watch_min,
                                                         const T* __restrict__ reset_qpos, const T* __restrict__ reset_qvel) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N) return;
  if (reset_qpos && st.qpos[(size_t)watch_row * N + e] < watch_min) {
    for (int k = 0; k < nq; k++) st.qpos[(size_t)k * N + e] = reset_qpos[(size_t)k * N + e];
    for (int k = 0; k < nv; k++) st.qvel[(size_t)k * N + e] = reset_qvel ? reset_qvel[(size_t)k * N + e] : T(0);
  }
  const unsigned draw = ctr[e];
  ctr[e] = draw + 1;
  for (int a = 0; a < nu; a += 2) {
    unsigned r[4];
    philox4x32_10(draw, (unsigned)(a >> 1), (unsigned)e, 0u, (unsigned)seed, (unsigned)(seed >> 32), r);
    // 53-bit uniform in [0, 1) from two words each
    const double u0 = ((double)(((unsigned long long)(r[0] >> 5) << 26) | (r[1] >> 6))) * (1.0 / 9007199254740992.0);
    const double u1 = ((double)(((unsigned long long)(r[2] >> 5) << 26) | (r[3] >> 6))) * (1.0 / 9007199254740992.0);
    st.ctrl[(size_t)a * N + e] = lo + (hi - lo) * (T)u0;
    if (a + 1 < nu) st.ctrl[(size_t)(a + 1) * N + e] = lo + (hi - lo) * (T)u1;
  }
}

// Recorder gather (reference logging.py:81-247 rows for a selection of envs): blockIdx.y = column, x = selected envs.
struct RecordColDev { const void* base; int row; int kind; };
template <typename T>
__global__ void __launch_bounds__(128) k_record_rows(const RecordColDev* __restrict__ cols, const int* __restrict__ env_index, int nsel,
                                                     int N, T time, T* out) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x, c = blockIdx.y;
  if (j >= nsel) return;
  const RecordColDev col = cols[c];
  T v;
  if (col.kind == 0) v = static_cast<const T*>(col.base)[(size_t)col.row * N + env_index[j]];
  else v = col.kind == 1 ? time : T(__int_as_float(0x7fc00000));
  out[(size_t)c * nsel + j] = v;
}

template <typename T, class D, class M>
__global__ void __launch_bounds__(128) k_integrate_pos(T* qpos, const T* qvel, T dt, int N, const void* image = nullptr) {
  model_load<M>(image, 0);
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N) return;
  RowStore<T, D> rows;
  LaneEnv<T, D, M> env(rows);
  for (int k = 0; k < M::nq(); k++) env.qpos[k] = qpos[(size_t)k * N + e];
  for (int k = 0; k < M::nv(); k++) env.qvel[k] = qvel[(size_t)k * N + e];
  env.integrate_pos(env.qpos, env.qvel, dt);
  for (int k = 0; k < M::nq(); k++) qpos[(size_t)k * N + e] = env.qpos[k];
}
template <typename T, class D, class M>
__global__ void __launch_bounds__(128) k_differentiate_pos(T* out, T dt, const T* q1, const T* q2, int N, const void* image = nullptr) {
  model_load<M>(image, 0);
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N) return;
  RowStore<T, D> rows;
  LaneEnv<T, D, M> env(rows);
  T a[D::NQ], b[D::NQ];
  for (int k = 0; k < M::nq(); k++) { a[k] = q1[(size_t)k * N + e]; b[k] = q2[(size_t)k * N + e]; }
  env.differentiate_pos(env.qvel, dt, a, b);
  for (int k = 0; k < M::nv(); k++) out[(size_t)k * N + e] = env.qvel[k];
}

// Open-loop rollout (b2_rollout): for s = 0 .. nsteps-1, ctrl <- ctrl_seq[s] (when given), one mj_step, record.  The same
// result as a loop of k_step launches with nsteps = 1, with the state in registers across all steps: ctrl_seq
// (nsteps, nu, N), qpos_traj (nsteps, nq, N), qvel_traj (nsteps, nv, N), sensor_traj (nsteps, nsensordata, N); any of them
// may be null.  A row of sensor_traj is the reading of step s's forward pass (before integration, as mj_step leaves it).
// A diverged env is frozen from the step that detects it, as in k_step; its remaining state rows repeat the state it is
// frozen in (the one the loop would leave in the state arrays) and its remaining sensor rows are NaN (no forward pass ran).
// Kept apart from k_step (its own arguments, per-step I/O and frozen-env handling) so k_step's instantiations stay as they are.
template <typename T, class D, class M>
__global__ void __launch_bounds__(128, 1) k_rollout(StateDev<T> st, DerivedDev<T> out, int want_derived, int N, int nsteps,
                                                    const T* __restrict__ ctrl_seq, T* qpos_traj, T* qvel_traj, T* sensor_traj,
                                                    const void* image = nullptr) {
  model_load<M>(image, 0);
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N) return;
  RowStore<T, D> rows;
  LaneEnv<T, D, M> env(rows);
  constexpr bool kLate = LaneEnv<T, D, M>::kLateMass;
  const int nq = M::nq(), nv = M::nv(), nu = M::nu(), nsd = M::nsensor() > 0 ? M::nsensordata() : 0;
  load_state(env, st, N, e);
  int s = 0;
  B2_NOUNROLL
  for (; s < nsteps; s++) {
    if (ctrl_seq) { B2_UNROLL for (int k = 0; k < nu; k++) env.ctrl[k] = ctrl_seq[((size_t)s * nu + k) * N + e]; }
    env.check_state();
    if (env.flags & 3) break;
    env.template forward_position<kLate>();
    env.forward_velocity();
    env.template forward_acc<kLate>();
    B2_UNROLL
    for (int k = 0; k < nv; k++) if (!(fabs(env.qacc[k]) <= T(1e10))) env.flags |= 4;
    if (sensor_traj && nsd > 0) {
      T sd[D::NSD];
      env.sensors(sd);
      B2_UNROLL
      for (int k = 0; k < nsd; k++) sensor_traj[((size_t)s * nsd + k) * N + e] = sd[k];
    }
    if (want_derived && s == nsteps - 1) store_derived(env, out, N, e);
    if (M::integrator() == 1) env.rk4(); else env.euler();
    if (qpos_traj) { B2_UNROLL for (int k = 0; k < nq; k++) qpos_traj[((size_t)s * nq + k) * N + e] = env.qpos[k]; }
    if (qvel_traj) { B2_UNROLL for (int k = 0; k < nv; k++) qvel_traj[((size_t)s * nv + k) * N + e] = env.qvel[k]; }
  }
  // frozen at step s (s == nsteps when the env never diverged)
  B2_NOUNROLL
  for (int r = s; r < nsteps; r++) {
    if (qpos_traj) { B2_UNROLL for (int k = 0; k < nq; k++) qpos_traj[((size_t)r * nq + k) * N + e] = env.qpos[k]; }
    if (qvel_traj) { B2_UNROLL for (int k = 0; k < nv; k++) qvel_traj[((size_t)r * nv + k) * N + e] = env.qvel[k]; }
    if (sensor_traj && nsd > 0) { B2_UNROLL for (int k = 0; k < nsd; k++) sensor_traj[((size_t)r * nsd + k) * N + e] = T(__int_as_float(0x7fc00000)); }
  }
  B2_UNROLL
  for (int k = 0; k < nq; k++) st.qpos[(size_t)k * N + e] = env.qpos[k];
  B2_UNROLL
  for (int k = 0; k < nv; k++) st.qvel[(size_t)k * N + e] = env.qvel[k];
  if (st.warm) { B2_UNROLL for (int k = 0; k < nv; k++) st.warm[(size_t)k * N + e] = env.warm[k]; }
  // the loop leaves the last control row in state.ctrl, frozen envs included
  if (ctrl_seq) { B2_UNROLL for (int k = 0; k < nu; k++) st.ctrl[(size_t)k * N + e] = ctrl_seq[((size_t)(nsteps - 1) * nu + k) * N + e]; }
  if (st.flags && env.flags) st.flags[e] |= env.flags;
}
template <typename T, class D, class M>
auto launch_rollout(const void* image, const b2_state* st, const b2_derived* out, int N, int nsteps, const void* ctrl_seq, void* qpos_traj,
                    void* qvel_traj, void* sensor_traj, void* stream) {
  const int threads = 128, blocks = (N + threads - 1) / threads;
  k_rollout<T, D, M><<<blocks, threads, 0, (cudaStream_t)stream>>>(to_dev<T>(st), to_dev<T>(out), out != nullptr, N, nsteps, (const T*)ctrl_seq,
                                                                   (T*)qpos_traj, (T*)qvel_traj, (T*)sensor_traj, image);
  return (int)cudaGetLastError();
}

// Linearisation along a rollout (b2_linearize_rollout), launch 1 of 2: the nominal trajectory.  k_rollout's step loop,
// reading x0 from the state and writing nothing back to it but flags: row 0 of qpos_traj (nsteps+1, nq, N), qvel_traj and
// warm_traj (nsteps+1, nv, N) is x0, row s+1 the state after step s, and row s of warm_traj the qacc_warmstart step s starts
// from.  warm_traj null: no warm start, every step starts from zeros as b2_step does without one.  sensor_traj
// (nsteps, nsensordata, N) as in k_rollout.  A diverged env is frozen as in k_rollout: its remaining state and warm rows
// repeat the state it is frozen in, its remaining sensor rows are NaN.  (A kernel of its own, so k_rollout stays as it is.)
template <typename T, class D, class M>
__global__ void __launch_bounds__(128, 1) k_nominal_traj(StateDev<T> st, int N, int nsteps, const T* __restrict__ ctrl_seq, T* qpos_traj,
                                                         T* qvel_traj, T* warm_traj, T* sensor_traj, const void* image = nullptr) {
  model_load<M>(image, 0);
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N) return;
  RowStore<T, D> rows;
  LaneEnv<T, D, M> env(rows);
  constexpr bool kLate = LaneEnv<T, D, M>::kLateMass;
  const int nq = M::nq(), nv = M::nv(), nu = M::nu(), nsd = M::nsensor() > 0 ? M::nsensordata() : 0;
  load_state(env, st, N, e);
  auto store_row = [&](int r) {
    B2_UNROLL
    for (int k = 0; k < nq; k++) qpos_traj[((size_t)r * nq + k) * N + e] = env.qpos[k];
    B2_UNROLL
    for (int k = 0; k < nv; k++) qvel_traj[((size_t)r * nv + k) * N + e] = env.qvel[k];
    if (warm_traj) { B2_UNROLL for (int k = 0; k < nv; k++) warm_traj[((size_t)r * nv + k) * N + e] = env.warm[k]; }
  };
  store_row(0);
  int s = 0;
  B2_NOUNROLL
  for (; s < nsteps; s++) {
    if (ctrl_seq) { B2_UNROLL for (int k = 0; k < nu; k++) env.ctrl[k] = ctrl_seq[((size_t)s * nu + k) * N + e]; }
    if (!warm_traj) { B2_UNROLL for (int k = 0; k < nv; k++) env.warm[k] = T(0); }
    env.check_state();
    if (env.flags & 3) break;
    env.template forward_position<kLate>();
    env.forward_velocity();
    env.template forward_acc<kLate>();
    B2_UNROLL
    for (int k = 0; k < nv; k++) if (!(fabs(env.qacc[k]) <= T(1e10))) env.flags |= 4;
    if (sensor_traj && nsd > 0) {
      T sd[D::NSD];
      env.sensors(sd);
      B2_UNROLL
      for (int k = 0; k < nsd; k++) sensor_traj[((size_t)s * nsd + k) * N + e] = sd[k];
    }
    if (M::integrator() == 1) env.rk4(); else env.euler();
    store_row(s + 1);
  }
  // frozen at step s (s == nsteps when the env never diverged)
  B2_NOUNROLL
  for (int r = s; r < nsteps; r++) {
    store_row(r + 1);
    if (sensor_traj && nsd > 0) { B2_UNROLL for (int k = 0; k < nsd; k++) sensor_traj[((size_t)r * nsd + k) * N + e] = T(__int_as_float(0x7fc00000)); }
  }
  if (st.flags && env.flags) st.flags[e] |= env.flags;
}

// Launch 2 of 2: the FD columns of every step of the nominal trajectory in one launch, one thread per (task, step, env) --
// k_linearize's task decomposition and fd_column, task-major (the long group tasks of Euler models start first), then step,
// env fastest.  A thread's nominal state is row t of the trajectory arrays, its controls row t of ctrl_seq (null: the
// state's held controls); its outputs are step t of A (nsteps, 2nv, 2nv, N), B (nsteps, 2nv, nu, N) and, with SENS,
// dsdx (nsteps, nsensordata, 2nv, N) and dsdu (nsteps, nsensordata, nu, N).  No control law, no env advance.
template <typename T, class D, class M, bool SENS = false>
__global__ void __launch_bounds__(B2_LIN_THREADS, B2_LIN_MIN_BLOCKS) k_linearize_traj(StateDev<T> st, int N, int nsteps, T eps, int centered,
                                                                                      const T* __restrict__ ctrl_seq, T* qpos_traj, T* qvel_traj,
                                                                                      T* warm_traj, T* A, T* B, T* dsdx, T* dsdu,
                                                                                      const void* image = nullptr) {
  model_load<M>(image, 0);
  const int nq = M::nq(), nv = M::nv(), nu = M::nu(), ndx = 2 * nv;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int ntask = fd_task_count(M::integrator(), nv, nu);
  const long long per_task = (long long)nsteps * N, total = per_task * ntask;
  if (idx >= total) return;
  // 32-bit division when the launch fits (a 64-bit one is ~100 instructions)
  int e, t, task;
  if (total <= 0x7fffffffLL) {
    const unsigned u = (unsigned)idx, r = u % (unsigned)per_task;
    task = (int)(u / (unsigned)per_task); t = (int)(r / (unsigned)N); e = (int)(r - (unsigned)t * (unsigned)N);
  } else {
    const long long r = idx % per_task;
    task = (int)(idx / per_task); t = (int)(r / N); e = (int)(r - (long long)t * N);
  }
  RowStore<T, D> rows;
  LaneEnv<T, D, M> env(rows);
  T u0[D::NU];
  B2_UNROLL
  for (int k = 0; k < nu; k++) u0[k] = ctrl_seq ? ctrl_seq[((size_t)t * nu + k) * N + e] : st.ctrl[(size_t)k * N + e];
  typedef typename std::conditional<SENS, NominalWithSensors<T>, NominalInMemory<T>>::type Nominal;
  Nominal nom;
  nom.set(qpos_traj + (size_t)t * nq * N, qvel_traj + (size_t)t * nv * N, warm_traj ? warm_traj + (size_t)t * nv * N : nullptr, N, e);
  nom.u0 = u0;
  if constexpr (SENS) {
    const size_t nsd = M::nsensordata();
    nom.dsdx = dsdx ? dsdx + (size_t)t * nsd * ndx * N : nullptr;
    nom.dsdu = dsdu ? dsdu + (size_t)t * nsd * nu * N : nullptr;
  }
  T* At = A ? A + (size_t)t * ndx * ndx * N : nullptr;
  T* Bt = B ? B + (size_t)t * ndx * nu * N : nullptr;
  const bool grouped = M::integrator() == 0;  // not a constant expression for the runtime provider
  const int groups = fd_group_count(nv, nu);
  int c0 = task, c1 = task + 1;
  if (grouped) {
    if (task < groups) { c0 = nv + task * B2_FD_GROUP; c1 = c0 + B2_FD_GROUP < ndx + nu ? c0 + B2_FD_GROUP : ndx + nu; }
    else { c0 = task - groups; c1 = c0 + 1; }
  }
  int last = -1;
  const T inv_eps = T(1) / eps;
  // mj_checkPos / mj_checkVel once on the nominal state, as k_linearize does
  B2_UNROLL
  for (int k = 0; k < nq; k++) env.qpos[k] = nom.q(k);
  B2_UNROLL
  for (int k = 0; k < nv; k++) env.qvel[k] = nom.v(k);
  env.check_state();
  B2_NOUNROLL
  for (int c = c0; c < c1; c++) fd_column(env, nom, c, false, eps, inv_eps, centered, N, e, At, Bt, last);
  if (st.flags && env.flags) atomicOr(st.flags + e, env.flags);
}
// Both launches of b2_linearize_rollout.  ntask: FD tasks per env (fd_task_count of the model).  The FD launch is skipped
// when there is no Jacobian to write.
template <typename T, class D, class M, bool SENS = false>
auto launch_linearize_rollout(const void* image, const b2_state* st, int N, int ntask, int nsteps, const void* ctrl_seq, double eps,
                              int centered, void* A, void* B, void* dsdx, void* dsdu, void* qpos_traj, void* qvel_traj, void* warm_traj,
                              void* sensor_traj, void* stream) {
  const StateDev<T> s = to_dev<T>(st);
  k_nominal_traj<T, D, M><<<(N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(s, N, nsteps, (const T*)ctrl_seq, (T*)qpos_traj, (T*)qvel_traj,
                                                                             (T*)warm_traj, (T*)sensor_traj, image);
  cudaError_t rc = cudaGetLastError();
  if (rc != cudaSuccess || !(A || B || dsdx || dsdu)) return (int)rc;
  const long long total = (long long)nsteps * N * ntask;
  const unsigned blocks = (unsigned)((total + B2_LIN_THREADS - 1) / B2_LIN_THREADS);
  k_linearize_traj<T, D, M, SENS><<<blocks, B2_LIN_THREADS, 0, (cudaStream_t)stream>>>(s, N, nsteps, (T)eps, centered, (const T*)ctrl_seq,
                                                                                        (T*)qpos_traj, (T*)qvel_traj, (T*)warm_traj, (T*)A,
                                                                                        (T*)B, (T*)dsdx, (T*)dsdu, image);
  return (int)cudaGetLastError();
}


// u = clip(ubar + alpha k - K [q (-) qbar ; v - vbar], ctrlrange) for one env whose state is in registers: the
// time-varying law of b2_rollout_feedback.  (-) is mj_differentiatePos(qbar -> q), as in lqr_law.  ubar (nu, N), qbar
// (nq, N), vbar (nv, N), K (nu, 2nv, N) and k (nu, N; may be null) are one step's rows, env fastest.
template <typename T, class D, class M>
B2_DEV void tvlqr_law(const LaneEnv<T, D, M>& env, const T* q, const T* v, const T* __restrict__ ubar, const T* __restrict__ qbar,
                      const T* __restrict__ vbar, const T* __restrict__ K, const T* __restrict__ k, T alpha, int N, int e, T* u_out) {
  const int nq = M::nq(), nv = M::nv(), nu = M::nu();
  T qr[D::NQ], x[2 * D::NV];
  B2_UNROLL
  for (int i = 0; i < nq; i++) qr[i] = qbar[(size_t)i * N + e];
  env.differentiate_pos(x, T(1), qr, q);
  B2_UNROLL
  for (int i = 0; i < nv; i++) x[nv + i] = v[i] - vbar[(size_t)i * N + e];
  B2_UNROLL
  for (int a = 0; a < nu; a++) {
    T u = ubar[(size_t)a * N + e];
    if (k) u += alpha * k[(size_t)a * N + e];
    B2_UNROLL
    for (int j = 0; j < 2 * nv; j++) u -= K[((size_t)a * 2 * nv + j) * N + e] * x[j];
    if (M::actuator_ctrllimited(a)) u = tclip(u, M::actuator_ctrlrange(2 * a), M::actuator_ctrlrange(2 * a + 1));
    u_out[a] = u;
  }
}

// Closed-loop rollout (b2_rollout_feedback): for s = 0 .. nsteps-1, ctrl <- tvlqr_law at step s's rows of the nominal
// trajectory and gains, one mj_step, record -- k_rollout's step loop with the law in front of each step.  ctrl_nom
// (nsteps, nu, N), qpos_nom / qvel_nom (>= nsteps rows of nq / nv), K (nsteps, nu, 2nv, N), k (nsteps, nu, N) or null,
// alpha (N) or null (1); ctrl_traj (nsteps, nu, N) records the applied controls, the other trajectories as in k_rollout.
// A diverged env is frozen as in k_rollout; its remaining control rows are NaN, and state.ctrl keeps the last control it
// was given.  A kernel of its own, so k_rollout stays as it is.
template <typename T, class D, class M>
__global__ void __launch_bounds__(128, 1) k_rollout_feedback(StateDev<T> st, DerivedDev<T> out, int want_derived, int N, int nsteps,
                                                             const T* __restrict__ ctrl_nom, const T* __restrict__ qpos_nom,
                                                             const T* __restrict__ qvel_nom, const T* __restrict__ K, const T* __restrict__ k,
                                                             const T* __restrict__ alpha, T* ctrl_traj, T* qpos_traj, T* qvel_traj,
                                                             T* sensor_traj, const void* image = nullptr) {
  model_load<M>(image, 0);
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N) return;
  RowStore<T, D> rows;
  LaneEnv<T, D, M> env(rows);
  constexpr bool kLate = LaneEnv<T, D, M>::kLateMass;
  const int nq = M::nq(), nv = M::nv(), nu = M::nu(), nsd = M::nsensor() > 0 ? M::nsensordata() : 0;
  load_state(env, st, N, e);
  const T a = alpha ? alpha[e] : T(1);
  int s = 0;
  B2_NOUNROLL
  for (; s < nsteps; s++) {
    env.check_state();
    if (env.flags & 3) break;
    tvlqr_law(env, env.qpos, env.qvel, ctrl_nom + (size_t)s * nu * N, qpos_nom + (size_t)s * nq * N, qvel_nom + (size_t)s * nv * N,
              K + (size_t)s * nu * 2 * nv * N, k ? k + (size_t)s * nu * N : nullptr, a, N, e, env.ctrl);
    if (ctrl_traj) { B2_UNROLL for (int i = 0; i < nu; i++) ctrl_traj[((size_t)s * nu + i) * N + e] = env.ctrl[i]; }
    env.template forward_position<kLate>();
    env.forward_velocity();
    env.template forward_acc<kLate>();
    B2_UNROLL
    for (int i = 0; i < nv; i++) if (!(fabs(env.qacc[i]) <= T(1e10))) env.flags |= 4;
    if (sensor_traj && nsd > 0) {
      T sd[D::NSD];
      env.sensors(sd);
      B2_UNROLL
      for (int i = 0; i < nsd; i++) sensor_traj[((size_t)s * nsd + i) * N + e] = sd[i];
    }
    if (want_derived && s == nsteps - 1) store_derived(env, out, N, e);
    if (M::integrator() == 1) env.rk4(); else env.euler();
    if (qpos_traj) { B2_UNROLL for (int i = 0; i < nq; i++) qpos_traj[((size_t)s * nq + i) * N + e] = env.qpos[i]; }
    if (qvel_traj) { B2_UNROLL for (int i = 0; i < nv; i++) qvel_traj[((size_t)s * nv + i) * N + e] = env.qvel[i]; }
  }
  // frozen at step s (s == nsteps when the env never diverged)
  const T nan = T(__int_as_float(0x7fc00000));
  B2_NOUNROLL
  for (int r = s; r < nsteps; r++) {
    if (qpos_traj) { B2_UNROLL for (int i = 0; i < nq; i++) qpos_traj[((size_t)r * nq + i) * N + e] = env.qpos[i]; }
    if (qvel_traj) { B2_UNROLL for (int i = 0; i < nv; i++) qvel_traj[((size_t)r * nv + i) * N + e] = env.qvel[i]; }
    if (sensor_traj && nsd > 0) { B2_UNROLL for (int i = 0; i < nsd; i++) sensor_traj[((size_t)r * nsd + i) * N + e] = nan; }
    if (ctrl_traj) { B2_UNROLL for (int i = 0; i < nu; i++) ctrl_traj[((size_t)r * nu + i) * N + e] = nan; }
  }
  B2_UNROLL
  for (int i = 0; i < nq; i++) st.qpos[(size_t)i * N + e] = env.qpos[i];
  B2_UNROLL
  for (int i = 0; i < nv; i++) st.qvel[(size_t)i * N + e] = env.qvel[i];
  if (st.warm) { B2_UNROLL for (int i = 0; i < nv; i++) st.warm[(size_t)i * N + e] = env.warm[i]; }
  B2_UNROLL
  for (int i = 0; i < nu; i++) st.ctrl[(size_t)i * N + e] = env.ctrl[i];
  if (st.flags && env.flags) st.flags[e] |= env.flags;
}
template <typename T, class D, class M>
auto launch_rollout_feedback(const void* image, const b2_state* st, const b2_derived* out, int N, int nsteps, const void* ctrl_nom,
                             const void* qpos_nom, const void* qvel_nom, const void* K, const void* k, const void* alpha, void* ctrl_traj,
                             void* qpos_traj, void* qvel_traj, void* sensor_traj, void* stream) {
  const int threads = 128, blocks = (N + threads - 1) / threads;
  k_rollout_feedback<T, D, M><<<blocks, threads, 0, (cudaStream_t)stream>>>(
      to_dev<T>(st), to_dev<T>(out), out != nullptr, N, nsteps, (const T*)ctrl_nom, (const T*)qpos_nom, (const T*)qvel_nom, (const T*)K,
      (const T*)k, (const T*)alpha, (T*)ctrl_traj, (T*)qpos_traj, (T*)qvel_traj, (T*)sensor_traj, image);
  return (int)cudaGetLastError();
}

// One step's law of b2_rollout_feedback on its own (the warp engine runs the loop on the host: this launch, one warp
// step, row copies): state.ctrl <- tvlqr_law, also written to ctrl_row (nu, N) when given.  An env whose state fails
// mj_checkPos / mj_checkVel is the one the step freezes: its ctrl is left alone and its ctrl_row is NaN.
template <typename T, class D, class M>
__global__ void __launch_bounds__(128) k_tvlqr_law(StateDev<T> st, int N, const T* __restrict__ ubar, const T* __restrict__ qbar,
                                                   const T* __restrict__ vbar, const T* __restrict__ K, const T* __restrict__ k,
                                                   const T* __restrict__ alpha, T* ctrl_row, const void* image = nullptr) {
  model_load<M>(image, 0);
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N) return;
  RowStore<T, D> rows;
  LaneEnv<T, D, M> env(rows);
  const int nu = M::nu();
  for (int i = 0; i < M::nq(); i++) env.qpos[i] = st.qpos[(size_t)i * N + e];
  for (int i = 0; i < M::nv(); i++) env.qvel[i] = st.qvel[(size_t)i * N + e];
  env.check_state();
  if (env.flags & 3) {
    if (ctrl_row) for (int i = 0; i < nu; i++) ctrl_row[(size_t)i * N + e] = T(__int_as_float(0x7fc00000));
    return;
  }
  T u[D::NU];
  tvlqr_law(env, env.qpos, env.qvel, ubar, qbar, vbar, K, k, alpha ? alpha[e] : T(1), N, e, u);
  for (int i = 0; i < nu; i++) {
    st.ctrl[(size_t)i * N + e] = u[i];
    if (ctrl_row) ctrl_row[(size_t)i * N + e] = u[i];
  }
}

}  // namespace b2
