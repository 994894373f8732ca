// Kernels of the warp engine (one env per warp, workspace in shared memory).
#pragma once
#include "b2_kernel_templates.cuh"
#include "b2_warp_engine.cuh"

// Register budget (__maxnreg__): an SM sub-partition has 16 K registers, so 168 registers per thread allow three resident
// warps per scheduler (12 per SM), 128 allow four.  The kernel is latency-bound: 128 registers (about 100 B of spills per
// thread) with lock-step blocks of four warps measured +18 % over 168 registers with blocks of two on the humanoid
// (round 2, gpurun A/B: 5.89e6 -> 6.98e6 env-steps/s; 112 and 96 registers spill too much).
#ifndef B2_WARP_MAXNREG
#define B2_WARP_MAXNREG 128
#endif
#ifndef B2_WARP_MAXNREG_RUNTIME
#define B2_WARP_MAXNREG_RUNTIME 200  // runtime sizes keep ~40 workspace pointers live: fewer registers only spill them
#endif
#define B2_WARP_REGS(M) (M::Dims::STATIC ? B2_WARP_MAXNREG : B2_WARP_MAXNREG_RUNTIME)

namespace b2 {

// position-dependent derived outputs (exported before their storage is reused: WarpEnv::forward)
template <typename T, class M>
B2_DEV void warp_store_position(const WarpEnv<T, M>& env, const DerivedDev<T>& o, int N, int e) {
  const int lane = env.lane;
  if (o.xpos) WFOR(k, 3 * env.mdl.nbody()) o.xpos[(size_t)k * N + e] = env.xpos[k];
  if (o.xquat) WFOR(k, 4 * env.mdl.nbody()) o.xquat[(size_t)k * N + e] = env.xquat[k];
  if (o.xipos) WFOR(k, 3 * env.mdl.nbody()) o.xipos[(size_t)k * N + e] = env.xipos[k];
  if (o.geom_xpos) WFOR(k, 3 * env.mdl.ngeom()) o.geom_xpos[(size_t)k * N + e] = env.geom_xpos[k];
  if (o.subtree_com) WFOR(k, 3 * env.mdl.nbody()) o.subtree_com[(size_t)k * N + e] = env.com[k];
}
// outputs of the acceleration stage
template <typename T, class M>
B2_DEV void warp_store_solution(const WarpEnv<T, M>& env, const DerivedDev<T>& o, int N, int e) {
  const int lane = env.lane;
  if (o.qacc) WFOR(k, env.mdl.nv()) o.qacc[(size_t)k * N + e] = env.qacc[k];
  if (o.qfrc_bias) WFOR(k, env.mdl.nv()) o.qfrc_bias[(size_t)k * N + e] = env.f_bias[k];
  if (lane == 0) {
    if (o.ncon) o.ncon[e] = env.ncon;
    if (o.nefc) o.nefc[e] = env.nefc;
    if (o.solver_iter) o.solver_iter[e] = env.niter;
  }
}

// Cost-ordered work queue.  The warps of a lock-step block leave the Newton loop together, i.e. a block pays for the
// slowest of its envs; an env's Newton iteration count changes slowly from step to step, so the envs are handed out in
// descending order of the count of their previous step (counting sort into kCostBins bins: histogram, then a scatter
// that reserves a range per block and bin): block mates then need about the same number of rounds, and the expensive
// envs start first.  Which env a warp runs has no effect on that env's result.
#ifndef B2_WARP_COST_BINS
#define B2_WARP_COST_BINS 64
#endif
constexpr int kCostBins = B2_WARP_COST_BINS;  // 16: (coupled rows?, Newton rounds); 64: ... x four buckets of the row count (+1 %)
template <int BINS>
__global__ void __launch_bounds__(256) k_cost_hist(const int* __restrict__ cost, int N, int* hist) {
  __shared__ int h[BINS];
  if (threadIdx.x < BINS) h[threadIdx.x] = 0;
  __syncthreads();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
    const int c = cost[i];
    atomicAdd(&h[c < BINS - 1 ? (c > 0 ? c : 0) : BINS - 1], 1);
  }
  __syncthreads();
  if (threadIdx.x < BINS && h[threadIdx.x]) atomicAdd(&hist[threadIdx.x], h[threadIdx.x]);
}
template <int BINS>
__global__ void __launch_bounds__(256) k_cost_scatter(const int* __restrict__ cost, int N, const int* __restrict__ hist, int* cursor, int* perm) {
  __shared__ int base[BINS], cnt[BINS], off[BINS];
  if (threadIdx.x < BINS) {  // descending cost: bin b starts after all bins above it
    int s = 0;
    for (int b = BINS - 1; b > (int)threadIdx.x; b--) s += hist[b];
    base[threadIdx.x] = s;
  }
  for (int i0 = blockIdx.x * blockDim.x; i0 < N; i0 += gridDim.x * blockDim.x) {
    if (threadIdx.x < BINS) cnt[threadIdx.x] = 0;
    __syncthreads();
    const int i = i0 + threadIdx.x;
    int b = 0, r = 0;
    if (i < N) {
      const int c = cost[i];
      b = c < BINS - 1 ? (c > 0 ? c : 0) : BINS - 1;
      r = atomicAdd(&cnt[b], 1);
    }
    __syncthreads();
    if (threadIdx.x < BINS) off[threadIdx.x] = cnt[threadIdx.x] ? atomicAdd(&cursor[threadIdx.x], cnt[threadIdx.x]) : 0;
    __syncthreads();
    if (i < N) perm[base[b] + off[b] + r] = i;
    __syncthreads();
  }
}

// nsteps x mj_step (nsteps == 0: mj_forward), one env per warp, persistent over envs: the first gridDim * wpb envs are
// assigned statically, the rest through an atomic work queue (env costs differ with contacts and Newton iterations).
// The warps of a block run their envs stage by stage behind the block barrier (WarpEnv::forward), so that one
// instruction fetch serves all of them; warps without an env of their own at the tail of the batch recompute the last env
// and discard the result, so that every warp reaches every barrier.
template <typename T, class M>
__global__ void __maxnreg__(B2_WARP_REGS(M)) k_warp_step_ls(const WarpImage<T>* __restrict__ img, StateDev<T> st, DerivedDev<T> out,
                                                            int want_derived, int N, int nsteps, T* jscratch, int* queue,
                                                            const int* __restrict__ perm, int* cost, StateDev<T> park) {
  extern __shared__ double b2_smem[];
  __shared__ int s_next;
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  const int gw = blockIdx.x * wpb + wib, nw = gridDim.x * wpb;
  WarpEnv<T, M> env;
  env.mdl.img = img;
  const int ws_reals = warp_ws_reals(env.mdl.nq(), env.mdl.nv(), env.mdl.nu(), env.mdl.nbody(), env.mdl.njnt(), env.mdl.ngeom(), env.mdl.ntendon());
  env.bind(img, reinterpret_cast<T*>(b2_smem) + (size_t)wib * ws_reals, jscratch + (size_t)gw * warp_slot_reals(env.mdl.nv()));
  const int total = nsteps > 0 ? nsteps : 1;
  int first = blockIdx.x * wpb;
  while (first < N) {
    const bool mine = first + wib < N;
    const int slot = mine ? first + wib : N - 1;
    const int e = perm ? perm[slot] : slot;  // cost-ordered queue (see k_cost_scatter)
    WFOR(k, env.mdl.nq()) env.qpos[k] = st.qpos[(size_t)k * N + e];
    WFOR(k, env.mdl.nv()) { env.qvel[k] = st.qvel[(size_t)k * N + e]; env.warm[k] = st.warm ? st.warm[(size_t)k * N + e] : T(0); }
    WFOR(k, env.mdl.nu()) env.ctrl[k] = st.ctrl[(size_t)k * N + e];
    env.flags = 0;
    __syncwarp();
    if (park.qpos && mine) {  // b2_step_lazy: keep the pre-step state for b2_refresh_derived (no copy launches)
      WFOR(k, env.mdl.nq()) park.qpos[(size_t)k * N + e] = env.qpos[k];
      WFOR(k, env.mdl.nv()) { park.qvel[(size_t)k * N + e] = env.qvel[k]; park.warm[(size_t)k * N + e] = env.warm[k]; }
      WFOR(k, env.mdl.nu()) park.ctrl[(size_t)k * N + e] = env.ctrl[k];
    }
    bool frozen = false;  // diverged env: flagged and left as it is (see k_step); its warp keeps pace on the rest pose
    for (int s = 0; s < total; s++) {
      env.check_state();
      if (!frozen && (env.flags & 3)) {
        frozen = true;
        if (mine && st.flags && lane == 0) st.flags[e] |= env.flags;
        WFOR(k, env.mdl.nq()) env.qpos[k] = env.mdl.qpos0(k);
        WFOR(k, env.mdl.nv()) { env.qvel[k] = 0; env.warm[k] = 0; }
        WFOR(k, env.mdl.nu()) env.ctrl[k] = 0;
        __syncwarp();
      }
      const bool store = want_derived && s == total - 1 && mine && !frozen;
      env.forward([&] { if (store) warp_store_position(env, out, N, e); });
      env.check_acc();
      if (store) warp_store_solution(env, out, N, e);
      env.stage_sync();
      if (nsteps > 0) env.euler();
    }
    if (mine && !frozen) {
      if (nsteps > 0) {
        WFOR(k, env.mdl.nq()) st.qpos[(size_t)k * N + e] = env.qpos[k];
        WFOR(k, env.mdl.nv()) st.qvel[(size_t)k * N + e] = env.qvel[k];
      }
      if (st.warm) WFOR(k, env.mdl.nv()) st.warm[(size_t)k * N + e] = env.warm[k];  // by mj_forward too (mj_fwdConstraint saves it)
      if (st.flags && env.flags && lane == 0) st.flags[e] |= env.flags;
    }
    // queue key of the next step: Newton rounds of this one, envs whose rows couple two branches of the tree (merged
    // ancestor lists: longer factorisation sweeps) in the upper half of the bins.  (The measured cycle count of the env's
    // constraint stage as the key, in 16 K / 32 K-cycle bins, was 4 % slower: 7.7e6 against 8.0e6 env-steps/s; the clock
    // also counts the time the warp waits for its SM's other warps.)
    if (mine && cost && lane == 0) {
      int key = ((env.nefc && env.rows_cross) ? 8 : 0) + (env.niter < 7 ? env.niter : 7);
      if (kCostBins == 64) key = key * 4 + (env.nefc < 12 ? 0 : (env.nefc < 24 ? 1 : (env.nefc < 36 ? 2 : 3)));
      cost[e] = frozen ? 0 : key;
    }
    if (threadIdx.x == 0) s_next = nw + atomicAdd(queue, wpb);
    __syncthreads();
    first = s_next;
    __syncthreads();
  }
}

// FD linearisation on the warp engine (large models): the work items are (column, env) pairs -- column-major, so that the
// warps of a lock-step block run the same kind of column -- and an item is two full rollouts of one step from the
// nominal state: plus / minus for a centred column, plus (or minus) and the nominal step where a control sits at its
// range bound (mjd_transitionFD's one-sidedness, as k_linearize).  Every rollout restores qacc_warmstart.  The columns go
// to A (2nv x 2nv x N) and B (2nv x nu x N), env fastest.  extra = 2 (nq + nv) reals per warp hold the two end states.
template <typename T, class M>
__global__ void __maxnreg__(B2_WARP_REGS(M)) k_warp_linearize(const WarpImage<T>* __restrict__ img, StateDev<T> st, int N, T eps, int centered,
                                                              T* A, T* B, T* jscratch, int* queue) {
  extern __shared__ double b2_smem[];
  __shared__ int s_next;
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  const int gw = blockIdx.x * wpb + wib, nw = gridDim.x * wpb;
  WarpEnv<T, M> env;
  env.mdl.img = img;
  const int nq = env.mdl.nq(), nv = env.mdl.nv(), nu = env.mdl.nu(), ndx = 2 * nv, ncol = ndx + nu;
  const int ws_reals = warp_ws_reals(nq, nv, nu, env.mdl.nbody(), env.mdl.njnt(), env.mdl.ngeom(), env.mdl.ntendon());
  const int extra = 2 * (nq + nv);
  T* base = reinterpret_cast<T*>(b2_smem) + (size_t)wib * (ws_reals + extra);
  env.bind(img, base, jscratch + (size_t)gw * warp_slot_reals(nv));
  T* ends[2] = {base + ws_reals, base + ws_reals + nq + nv};  // [0]: minus side (s1), [1]: plus side (s2)
  const int total = N * ncol;
  int flags_all = 0;
  int first = blockIdx.x * wpb;
  while (first < total) {
    const bool mine = first + wib < total;
    const int item = mine ? first + wib : total - 1;
    const int c = item / N, e = item - c * N;
    int kind, i;
    bool fwd = true, back = centered != 0;
    if (c < nv) { kind = 1; i = c; }
    else if (c < ndx) { kind = 2; i = c - nv; }
    else {
      kind = 3; i = c - ndx;
      const T u = st.ctrl[(size_t)i * N + e], lo = env.mdl.actuator_ctrlrange(2 * i), hi = env.mdl.actuator_ctrlrange(2 * i + 1);
      const bool lim = env.mdl.actuator_ctrllimited(i) != 0;
      fwd = !lim || (u >= lo && u <= hi && u + eps >= lo && u + eps <= hi);
      back = (centered || !fwd) && (!lim || (u - eps >= lo && u - eps <= hi && u >= lo && u <= hi));
    }
    // two rollouts per item whatever the column needs, so that all warps of a block meet at every barrier
    for (int side = 1; side >= 0; side--) {
      const T delta = side ? (fwd ? eps : T(0)) : (back ? -eps : T(0));
      WFOR(k, nq) env.qpos[k] = st.qpos[(size_t)k * N + e];
      WFOR(k, nv) { env.qvel[k] = st.qvel[(size_t)k * N + e] + ((kind == 2 && k == i) ? delta : T(0)); env.warm[k] = st.warm ? st.warm[(size_t)k * N + e] : T(0); }
      WFOR(k, nu) env.ctrl[k] = st.ctrl[(size_t)k * N + e] + ((kind == 3 && k == i) ? delta : T(0));
      env.flags = 0;
      __syncwarp();
      if (kind == 1 && lane == 0) {  // tangent-space step along dof i (mj_integratePos of a unit vector)
        const int j = env.mdl.dof_jntid(i), pa = env.mdl.jnt_qposadr(j), d = i - env.mdl.jnt_dofadr(j);
        if (env.mdl.jnt_type(j) == JNT_FREE && d >= 3) {
          T q[4] = {env.qpos[pa + 3], env.qpos[pa + 4], env.qpos[pa + 5], env.qpos[pa + 6]}, w[3] = {0, 0, 0};
          w[d - 3] = 1;
          quat_integrate(q, w, delta);
          for (int k = 0; k < 4; k++) env.qpos[pa + 3 + k] = q[k];
        } else env.qpos[pa + (env.mdl.jnt_type(j) == JNT_FREE ? d : 0)] += delta;
      }
      __syncwarp();
      env.check_state();
      env.forward([] {});
      env.check_acc();
      env.stage_sync();
      env.euler();
      flags_all |= env.flags;
      T* dst = ends[side];
      WFOR(k, nq) dst[k] = env.qpos[k];
      WFOR(k, nv) dst[nq + k] = env.qvel[k];
      __syncwarp();
    }
    if (mine) {
      const T* s1 = ends[0];
      const T* s2 = ends[1];
      const T ih = (fwd && back) ? T(0.5) / eps : ((fwd || back) ? T(1) / eps : T(0));
      T* out = c < ndx ? A + ((size_t)c) * N + e : B + ((size_t)(c - ndx)) * N + e;
      const size_t rs = (size_t)(c < ndx ? ndx : nu) * N;  // row stride
      if (c < ndx ? A != nullptr : B != nullptr) {
        WFOR(j, env.mdl.njnt()) {
          const int pa = env.mdl.jnt_qposadr(j), va = env.mdl.jnt_dofadr(j);
          if (env.mdl.jnt_type(j) == JNT_FREE) {
            T neg[4] = {s1[pa + 3], -s1[pa + 4], -s1[pa + 5], -s1[pa + 6]}, q2[4] = {s2[pa + 3], s2[pa + 4], s2[pa + 5], s2[pa + 6]}, dq[4], rv[3];
            quat_mul(dq, neg, q2);
            quat_to_vel(rv, dq, T(1));
            for (int k = 0; k < 3; k++) { out[(va + k) * rs] = (s2[pa + k] - s1[pa + k]) * ih; out[(va + 3 + k) * rs] = rv[k] * ih; }
          } else out[va * rs] = (s2[pa] - s1[pa]) * ih;
        }
        WFOR(k, nv) out[(nv + k) * rs] = (s2[nq + k] - s1[nq + k]) * ih;
      }
      if (st.flags && flags_all && lane == 0) atomicOr(st.flags + e, flags_all);
    }
    flags_all = 0;
    __syncwarp();
    if (threadIdx.x == 0) s_next = nw + atomicAdd(queue, wpb);
    __syncthreads();
    first = s_next;
    __syncthreads();
  }
}

}  // namespace b2
