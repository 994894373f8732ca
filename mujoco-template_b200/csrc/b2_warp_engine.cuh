// Warp-cooperative rigid-body engine ("warp engine": one env per warp) for large models.
//
// Same physics as the lane engine (b2_engine.cuh) -- what the reference reaches through
// mj.mj_step (reference mujoco_template/model.py:56-57) -- but one env is spread over the 32
// lanes of a warp: tree passes run level by level with one body per lane, the packed mass matrix
// and the Newton Hessian are updated with one entry group per lane, constraint rows and contact
// candidates are distributed over lanes, reductions use warp shuffles.  The per-env workspace
// (poses, inertias, motion axes, packed M / L'DL / H, force vectors, contact and row metadata)
// lives in shared memory; only the dense constraint Jacobian J (nefc x nv) sits in an
// L2-resident global scratch slot owned by the warp (together with the per-row vectors).
//
// Supported model features: free / hinge / slide joints, joint-transmission actuators, fixed
// tendons, plane / sphere / capsule geoms, semi-implicit Euler.  Anything else (fluid forces, site
// transmissions, box / ellipsoid geoms, RK4) is routed to the lane engine by the host.
#pragma once
#include "b2_math.cuh"
#include "b2_model_dev.cuh"

namespace b2 {

// lane-strided loop; almost always a single trip, so it is kept rolled: unrolled by four the kernel is 10 % larger and,
// being bound by instruction fetch, 2.6 % slower
#define WFOR(i, n) _Pragma("unroll 1") for (int i = lane; i < (n); i += 32)

// out of line (as are the other helpers with many call sites below): the kernel is bound by instruction fetch, a butterfly of
// five dependent shuffles gains nothing from being inlined 50 times
template <typename T> __device__ __noinline__ T warp_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
B2_DEV int tri(int i, int j) { return i * (i + 1) / 2 + j; }  // packed lower triangle, j <= i

// Everything a warp-engine kernel reads about one model, as ONE global-memory object owned by the b2_model (per device and
// precision) and passed to the kernels by pointer -- no process-wide device symbols, so batches of different large models
// can run concurrently on different streams.  Lanes read the model with lane-dependent indices, which the constant cache
// would serialise (one address per cycle); read-only global loads are gathered by L1 instead.
//  * tri_row / tri_col / tri_ij: inverse of tri() for matrices up to 32 x 32.
template <typename T>
struct WarpImage {
  DevModel<T, DimsLarge> model;
  unsigned char tri_row[528], tri_col[528];
  unsigned short tri_ij[544];  // per packed entry e: row | col << 8 | (col is row itself or an ancestor of it) << 15
};

template <typename T>
inline void fill_warp_image(WarpImage<T>& img, const b2m_view& v, const int* actuator_disabled) {
  fill_dev_model(img.model, v, actuator_disabled);
  auto tri_h = [](int i, int j) { return i * (i + 1) / 2 + j; };
  int e = 0;
  for (int i = 0; i < 32; i++) for (int j = 0; j <= i; j++) { img.tri_row[e] = (unsigned char)i; img.tri_col[e] = (unsigned char)j; e++; }
  for (int x = 0; x < 544; x++) img.tri_ij[x] = 0;
  e = 0;
  for (int i = 0; i < 32; i++)
    for (int j = 0; j <= i; j++) {
      bool anc = false;
      if (i < v.nv) for (int a = i; a >= 0; a = v.dof_parentid[a]) if (a == j) { anc = true; break; }
      img.tri_ij[e++] = (unsigned short)(i | (j << 8) | (anc ? 0x8000 : 0));
    }
}

// Model providers of the warp engine: an object that holds the image pointer; every field is a member accessor.
// DimsRuntime reads the sizes from the image (any model of the large class); DimsStatic<...> makes them compile-time
// constants, so that every workspace offset and loop bound folds (used when a model's sizes match an instantiated
// kernel: the humanoid).  The field VALUES always come from the image.
struct DimsRuntime { static constexpr bool STATIC = false; };
template <int NQ_, int NV_, int NU_, int NB_, int NJ_, int NG_, int NT_, int DEPTH_>
struct DimsStatic {
  static constexpr bool STATIC = true;
  static constexpr int NQ = NQ_, NV = NV_, NU = NU_, NB = NB_, NJ = NJ_, NG = NG_, NT = NT_, DEPTH = DEPTH_;
};
template <typename T>
struct ImageModelBase {
  typedef DimsLarge D;
  const WarpImage<T>* img;
#define X(name) B2_DEV int name() const { return __ldg(&img->model.name); }
  B2_MODEL_INT_SCALARS(X)
#undef X
#define X(name) B2_DEV T name() const { return __ldg(&img->model.name); }
  B2_MODEL_REAL_SCALARS(X)
#undef X
#define X(name, cap) B2_DEV int name(int i) const { return __ldg(&img->model.name[i]); }
  B2_MODEL_INT_ARRAYS(X)
#undef X
#define X(name, cap) B2_DEV T name(int i) const { return __ldg(&img->model.name[i]); }
  B2_MODEL_REAL_ARRAYS(X)
#undef X
  B2_DEV void untri(int e, int& i, int& j) const { i = __ldg(&img->tri_row[e]); j = __ldg(&img->tri_col[e]); }
};
template <typename T, class DM>
struct ImageModel : ImageModelBase<T> {
  typedef DM Dims;
  B2_DEV int nq() const { return DM::NQ; }
  B2_DEV int nv() const { return DM::NV; }
  B2_DEV int nu() const { return DM::NU; }
  B2_DEV int nbody() const { return DM::NB; }
  B2_DEV int njnt() const { return DM::NJ; }
  B2_DEV int ngeom() const { return DM::NG; }
  B2_DEV int ntendon() const { return DM::NT; }
  B2_DEV int maxdepth() const { return DM::DEPTH; }
};
template <typename T>
struct ImageModel<T, DimsRuntime> : ImageModelBase<T> { typedef DimsRuntime Dims; };

struct WarpCaps { static constexpr int NCON = 32, NEFC = 128; };
// reals of global scratch one resident warp owns: J (NEFC x nv), six row vectors, the contact records (dist, pos, frame) and
// the int metadata of contacts and rows (counted as one real each)
// ... and the env's merged ancestor lists (32 counts + 32 x 32 byte indices, see WarpEnv::merge_branches): 1152 B
__host__ __device__ inline size_t warp_slot_reals(int nv) {
  return (size_t)WarpCaps::NEFC * (nv + 6) + 13 * WarpCaps::NCON + WarpCaps::NCON + WarpCaps::NEFC + 320;
}

// Shared-memory workspace of one env (offsets in reals).  How many warps an SM holds is decided by this size (and by the
// registers), and the kernel is latency-bound, so arrays share storage wherever their live ranges allow:
//   P  live across stages: state, packed M, bias / passive force, tendons, subtree CoM, cinert, cdof
//   X  one region used three times over:
//      A  kinematics   xpos xquat xipos xmat ximat xanchor xaxis geom_xpos geom_z   (dead once collide + com_frame ran)
//      B  dynamics     crb buf6 cvel cdof_dot cacc                                   (mass matrix, velocities, RNE)
//      C  solve        LDp dinv hdinv + nine nv-vectors                              (factorisations, Newton, Euler)
// The stage order of forward() follows from it (collide right after kinematics, the first factorisation after RNE).
struct WarpLayout {
  int qpos, qvel, ctrl, warm, Mp, f_bias, f_passive, ten_len, ten_J, com, cinert, cdof, X, total;
  int xpos, xquat, xipos, xmat, ximat, xanchor, xaxis, geom_xpos, geom_z;
  int crb, buf6, cvel, cdof_dot, cacc;
  int LDp, dinv, hdinv, f_smooth, f_con, a_smooth, qacc, Ma, Mv, grad, Mgrad, search;
  __host__ __device__ constexpr WarpLayout(int nq, int nv, int nu, int nb, int nj, int ng, int nt)
      : qpos(0), qvel(qpos + nq), ctrl(qvel + nv), warm(ctrl + nu), Mp(warm + nv), f_bias(Mp + nv * (nv + 1) / 2),
        f_passive(f_bias + nv), ten_len(f_passive + nv), ten_J(ten_len + nt), com(ten_J + nt * nv), cinert(com + 3 * nb),
        cdof(cinert + 10 * nb), X(cdof + 6 * nv), total(0),
        xpos(X), xquat(xpos + 3 * nb), xipos(xquat + 4 * nb), xmat(xipos + 3 * nb), ximat(xmat + 9 * nb), xanchor(ximat + 9 * nb),
        xaxis(xanchor + 3 * nj), geom_xpos(xaxis + 3 * nj), geom_z(geom_xpos + 3 * ng),
        crb(X), buf6(crb + 10 * nb), cvel(buf6 + 6 * (nv > nb ? nv : nb)), cdof_dot(cvel + 6 * nb), cacc(cdof_dot + 6 * nv),
        LDp(X), dinv(LDp + nv * (nv + 1) / 2), hdinv(dinv + nv), f_smooth(hdinv + nv), f_con(f_smooth + nv), a_smooth(f_con + nv),
        qacc(a_smooth + nv), Ma(qacc + nv), Mv(Ma + nv), grad(Mv + nv), Mgrad(grad + nv), search(Mgrad + nv) {
    int endA = geom_z + 3 * ng, endB = cacc + 6 * nb, endC = search + nv;
    total = endA > endB ? endA : endB;
    if (endC > total) total = endC;
  }
};
// number of T elements of shared memory one env needs
__host__ __device__ inline int warp_ws_reals(int nq, int nv, int nu, int nb, int nj, int ng, int nt) {
  return WarpLayout(nq, nv, nu, nb, nj, ng, nt).total;
}

// In-place L'DL of the packed matrix in LDp (tree sparsity, mj_factorM).  Pivot k (leaves first): lane l owns the l-th
// proper ancestor i_l of k (nearest first), keeps row k's entry L[k, i_l] and its quotient t_l = L[k, i_l] / d_k in registers,
// and updates row i_l: L[i_l, i_{l+s}] -= t_l * L[k, i_{l+s}] for s = 0 .. m-1-l, the row-k value and the column index
// coming from lane l+s by shuffle.  Nothing in the update loop waits on memory except its own read-modify-write, and the
// next pivot's ancestor list is fetched while this one is being worked on (the kernel is latency-bound: the plan-driven
// version of r01 spent 9 % of all stall samples on its load -> load -> FMA -> store chain).
// The ancestor lists come either from the model image (the kinematic tree: int entries, read-only path) or from the env's
// scratch slot (the tree with the branches its constraint rows couple merged: byte entries, WarpEnv::merge_branches).
B2_DEV int anc_load(const int* p) { return __ldg(p); }
B2_DEV int anc_load(const unsigned char* p) { return *p; }
template <typename T, typename IDX>
__device__ __noinline__ void factor_LD_impl(int nv, const int* __restrict__ nanc, const IDX* __restrict__ anclist, T* LDp, T* dinv, int lane) {
  // The (l, s) pairs of a pivot form a triangle, and chains are short (humanoid: m <= 14): the warp is folded into 32 / W
  // groups of W > m lanes, every group holds the same row-k registers, and group h takes the offsets s = h, h + 32 / W, ...
  // -- a quarter (m < 8) or half (m < 16) of the sweeps of the one-group form, every entry still updated exactly once per
  // pivot with the same operands (bit-identical).
  constexpr int LS = DimsLarge::NV;  // stride of the ancestor lists
  int m = anc_load(nanc + nv - 1);
  int wl = m < 8 ? 3 : (m < 16 ? 4 : 5);  // log2 W
  int i = (lane & ((1 << wl) - 1)) < m ? anc_load(anclist + (nv - 1) * LS + (lane & ((1 << wl) - 1))) : 0;
#pragma unroll 1
  for (int k = nv - 1; k >= 0; k--) {
    // prefetch the next pivot's list (independent of this pivot's arithmetic)
    const int mn = k > 0 ? anc_load(nanc + k - 1) : 0;
    const int wln = mn < 8 ? 3 : (mn < 16 ? 4 : 5);
    const int ln = lane & ((1 << wln) - 1);
    const int in = (k > 0 && ln < mn) ? anc_load(anclist + (k - 1) * LS + ln) : 0;
    const int l = lane & ((1 << wl) - 1), h = lane >> wl, hs = 32 >> wl;
    const int kk = tri(k, 0);
    const T dkk = LDp[kk + k];
    const T rk = l < m ? LDp[kk + i] : T(1);
    const T q = rk / dkk;  // l < m: t_l; lane m (group 0, W > m): 1 / d_k
    if (lane == m) dinv[k] = q;
    if (m) {
      const int rowbase = tri(i, 0);
#ifndef B2_WARP_PAIRFOLD  // measured 2.6 % slower than the plain sweeps (gpurun A/B, profiles/ab_hum_pairfold_r03g.txt): off
      if (true) {
#else
      if (wl < 5) {
#endif
#pragma unroll 2
        for (int s = h; s - h < m; s += hs) {
          const T rks = __shfl_sync(0xffffffffu, rk, l + s);  // group 0 holds the row; l + s < m <= W there when it is used
          const int js = __shfl_sync(0xffffffffu, i, l + s);
          if (l + s < m) LDp[rowbase + js] -= q * rks;
        }
      } else {
        // Long ancestor sets (16 <= m <= 31: merged trees) leave no room for lane groups; instead sweep s (m - s pairs,
        // lanes 0 .. m-s-1) runs together with sweep m-1-s (s + 1 pairs, lanes m-s .. m): m + 1 lanes busy, half the sweeps.
        // A lane of the second group works for row l' = lane - (m - s) at offset m-1-s, i.e. on column lane - 1; the row's
        // quotient and base come by shuffle.
        const int half = (m + 1) >> 1;
#pragma unroll 1
        for (int s = 0; s < half; s++) {
          const int nA = m - s;
          const bool inA = lane < nA, inB = (m - 1 - s != s) && lane >= nA && lane <= m;
          const int lrow = inA ? lane : (lane - nA) & 31, lcol = (inA ? lane + s : lane - 1) & 31;
          const T rks = __shfl_sync(0xffffffffu, rk, lcol);
          const int js = __shfl_sync(0xffffffffu, i, lcol);
          const T ql = __shfl_sync(0xffffffffu, q, lrow);
          const int rb = __shfl_sync(0xffffffffu, rowbase, lrow);
          if (inA || inB) LDp[rb + js] -= ql * rks;
        }
      }
      if (lane < m) LDp[kk + i] = q;
    }
    __syncwarp();
    m = mn; i = in; wl = wln;
  }
}

// x <- (L'DL)^-1 x with x_l in a register of lane l (nv <= 32): column sweeps by shuffle, no shared-memory traffic for x
// and no warp barrier per column; the L entries of a column are loaded ahead of the value they multiply.
// anc: this lane's proper-ancestor mask (kinematic tree or merged, matching the factor in LDp)
template <typename T>
__device__ __noinline__ void solve_LD_impl(int nv, unsigned anc, const T* LDp, const T* dinv, T* x, int lane) {
  const int rowbase = tri(lane < nv ? lane : 0, 0);
  T xl = lane < nv ? x[lane] : T(0);
  // x <- L^-T x : dof i (leaves first) pushes x_i into its ancestors j: x_j -= L[i,j] x_i.  Lane j needs bit j of anc(i),
  // i.e. "i is a descendant of j": read from lane i's mask by shuffle.
#pragma unroll 1
  for (int i = nv - 1; i > 0; i--) {
    const unsigned anci = __shfl_sync(0xffffffffu, anc, i);
    const bool on = (anci >> lane) & 1u;
    const T l = on ? LDp[tri(i, 0) + lane] : T(0);
    const T xi = __shfl_sync(0xffffffffu, xl, i);
    xl -= l * xi;
  }
  xl *= lane < nv ? dinv[lane] : T(0);
  // x <- L^-1 x : dof j (root first) pushes x_j into its descendants i: x_i -= L[i,j] x_j; lane i owns row i.
#pragma unroll 1
  for (int j = 0; j < nv - 1; j++) {
    const bool on = (anc >> j) & 1u;
    const T l = on ? LDp[rowbase + j] : T(0);
    const T xj = __shfl_sync(0xffffffffu, xl, j);
    xl -= l * xj;
  }
  if (lane < nv) x[lane] = xl;
  __syncwarp();
}

// one evaluation of the exact piecewise-quadratic line-search objective (seven call sites share this copy);
// out = {alpha, cost, d1, d2}
template <typename T>
__device__ __noinline__ void ls_eval_impl(const T* Jaref, const T* Jv, const T* row_D, int nefc, int lane, T qg0, T qg1, T qg2,
                                          T alpha, T* out) {

    T q0 = 0, q1 = 0, q2 = 0;
    WFOR(i, nefc) {
      if (Jaref[i] + alpha * Jv[i] < 0) {
        const T dj = row_D[i] * Jaref[i];
        q0 += T(0.5) * Jaref[i] * dj; q1 += Jv[i] * dj; q2 += T(0.5) * Jv[i] * row_D[i] * Jv[i];
      }
    }
    q0 = qg0 + warp_sum(q0); q1 = qg1 + warp_sum(q1); q2 = qg2 + warp_sum(q2);
    T d2 = 2 * q2;
  if (d2 <= 0) d2 = Num<T>::minval();
  out[0] = alpha; out[1] = alpha * alpha * q2 + alpha * q1 + q0; out[2] = 2 * alpha * q2 + q1; out[3] = d2;
  }

// r = M v with the packed lower triangle Mp (one row per lane); out = J v [- sub] (one constraint row per lane)
template <typename T>
__device__ __noinline__ void mul_M_impl(const T* Mp, T* r, const T* v, int nv, int lane) {
  WFOR(i, nv) {
    T s = 0;
    for (int j = 0; j < nv; j++) s += (j <= i ? Mp[tri(i, j)] : Mp[tri(j, i)]) * v[j];
    r[i] = s;
  }
  __syncwarp();
}
template <typename T>
__device__ __noinline__ void mul_J_impl(const T* J, T* out, const T* v, const T* sub, int nefc, int nv, int lane) {
  WFOR(i, nefc) {
    T s = 0;
    for (int k = 0; k < nv; k++) s += J[i * nv + k] * v[k];
    out[i] = sub ? s - sub[i] : s;
  }
  __syncwarp();
}
template <typename T> __device__ __noinline__ void make_frame_shared(T* fr) { make_frame(fr); }

template <typename T, class M>
struct WarpEnv {
  M mdl;
  int lane, ncon, nefc, niter, flags;
  T *qpos, *qvel, *ctrl, *warm;
  T *xpos, *xquat, *xmat, *xipos, *ximat, *xanchor, *xaxis, *cdof_dot, *cvel;
  T *geom_xpos, *geom_z, *com, *cinert, *crb, *cdof, *cacc;
  T *Mp, *LDp, *dinv, *hdinv, *ten_len, *ten_J;
  T *f_bias, *f_passive, *f_smooth, *f_con, *a_smooth, *qacc, *Ma, *Mv, *grad, *Mgrad, *search, *buf6;
  T *con_dist, *con_pos, *con_frame, *row_pos, *row_margin, *row_D, *row_aref, *Jaref, *Jv;
  int *con_pair, *row_meta;  // row_meta = type | id << 8
  T* J;                      // global scratch, NEFC * nv
  T cost, gauss, qg0, qg1, qg2;
  int ls_iter;
  unsigned active_sig[(WarpCaps::NEFC + 31) / 32];  // active-row bit set the factor in LDp was built for
  bool hess_valid;
  // Sparsity of the Newton Hessian H = M + J' D J.  A row that touches one root-to-leaf chain (a limit, a contact with the
  // world or between a body and its own ancestor) keeps M's tree pattern.  A row that couples two branches (foot against
  // the other shin, hand on a thigh) adds fill between their chains: the env then factorises H over the MERGED tree --
  // tree_mask / amask are this lane's proper-ancestor masks in the kinematic tree and in the merged one, dyn_nanc /
  // dyn_list the merged ancestor lists in the scratch slot (merge_branches) -- instead of falling back to a dense
  // Cholesky (round 1 and the first half of round 2: 17 % of the executed instructions once humanoids lie on the floor).
  bool rows_cross;
  unsigned tree_mask, amask;
  int* dyn_nanc;
  unsigned char* dyn_list;

  // base: this env's shared-memory workspace (WarpLayout); jscratch: the warp's global scratch slot
  B2_DEV void bind(const WarpImage<T>* image, T* base, T* jscratch) {
    mdl.img = image;
    const int nv = mdl.nv();
    const WarpLayout L(mdl.nq(), nv, mdl.nu(), mdl.nbody(), mdl.njnt(), mdl.ngeom(), mdl.ntendon());
    qpos = base + L.qpos; qvel = base + L.qvel; ctrl = base + L.ctrl; warm = base + L.warm; Mp = base + L.Mp;
    f_bias = base + L.f_bias; f_passive = base + L.f_passive; ten_len = base + L.ten_len; ten_J = base + L.ten_J;
    com = base + L.com; cinert = base + L.cinert; cdof = base + L.cdof;
    xpos = base + L.xpos; xquat = base + L.xquat; xipos = base + L.xipos; xmat = base + L.xmat; ximat = base + L.ximat;
    xanchor = base + L.xanchor; xaxis = base + L.xaxis; geom_xpos = base + L.geom_xpos; geom_z = base + L.geom_z;
    crb = base + L.crb; buf6 = base + L.buf6; cvel = base + L.cvel; cdof_dot = base + L.cdof_dot; cacc = base + L.cacc;
    LDp = base + L.LDp; dinv = base + L.dinv; hdinv = base + L.hdinv; f_smooth = base + L.f_smooth; f_con = base + L.f_con;
    a_smooth = base + L.a_smooth; qacc = base + L.qacc; Ma = base + L.Ma; Mv = base + L.Mv; grad = base + L.grad;
    Mgrad = base + L.Mgrad; search = base + L.search;
    // per-row data lives in the warp's global scratch slot (L1/L2 resident): J, then six row vectors
    J = jscratch;
    T* rv = jscratch + WarpCaps::NEFC * nv;
    row_pos = rv; row_margin = rv + WarpCaps::NEFC; row_D = rv + 2 * WarpCaps::NEFC; row_aref = rv + 3 * WarpCaps::NEFC;
    Jaref = rv + 4 * WarpCaps::NEFC; Jv = rv + 5 * WarpCaps::NEFC;
    T* cb = rv + 6 * WarpCaps::NEFC;  // contact records: written by collide, read by make_rows (once per step each)
    con_dist = cb; con_pos = cb + WarpCaps::NCON; con_frame = cb + 4 * WarpCaps::NCON;
    con_pair = reinterpret_cast<int*>(cb + 13 * WarpCaps::NCON); row_meta = con_pair + WarpCaps::NCON;
    dyn_nanc = reinterpret_cast<int*>(cb + 13 * WarpCaps::NCON + WarpCaps::NCON + WarpCaps::NEFC);
    dyn_list = reinterpret_cast<unsigned char*>(dyn_nanc + 32);
    lane = threadIdx.x & 31;
    tree_mask = lane < nv ? ((unsigned)mdl.dof_anc(lane)) & ~(1u << lane) : 0u;
    amask = tree_mask;
    rows_cross = false;
    ncon = nefc = niter = flags = 0;
  }
  B2_DEV bool dof_is_anc(int i, int j) const { return (((unsigned)mdl.dof_anc(i)) >> j) & 1u; }
  B2_DEV bool in_subtree(int root, int b) const { return (((unsigned)mdl.body_anc(b)) >> root) & 1u; }

  // ------------------------------------------------------------------ position stage
  B2_DEV void kinematics() {
    const int nb = mdl.nbody();
    if (lane == 0) {
      for (int k = 0; k < 3; k++) { xpos[k] = 0; xipos[k] = 0; }
      xquat[0] = 1; xquat[1] = xquat[2] = xquat[3] = 0;
      quat_to_mat(xmat, xquat); quat_to_mat(ximat, xquat);
    }
    __syncwarp();
    for (int level = 1; level <= mdl.maxdepth(); level++) {
      const int i = lane;
      if (i < nb && mdl.body_depth(i) == level) {
        T p[3], q[4];
        const int ja = mdl.body_jntadr(i), jn = mdl.body_jntnum(i), pid = mdl.body_parentid(i);
        if (jn == 1 && mdl.jnt_type(ja) == JNT_FREE) {
          const int qa = mdl.jnt_qposadr(ja);
          for (int k = 0; k < 3; k++) p[k] = qpos[qa + k];
          for (int k = 0; k < 4; k++) q[k] = qpos[qa + 3 + k];
          normalize4(q);
          for (int k = 0; k < 3; k++) { xanchor[3 * ja + k] = p[k]; xaxis[3 * ja + k] = mdl.jnt_axis(3 * ja + k); }
        } else {
          T bpos[3] = {mdl.body_pos(3 * i), mdl.body_pos(3 * i + 1), mdl.body_pos(3 * i + 2)};
          T bquat[4] = {mdl.body_quat(4 * i), mdl.body_quat(4 * i + 1), mdl.body_quat(4 * i + 2), mdl.body_quat(4 * i + 3)};
          if (pid) {
            T pm[9], pq[4];
            for (int k = 0; k < 9; k++) pm[k] = xmat[9 * pid + k];
            for (int k = 0; k < 4; k++) pq[k] = xquat[4 * pid + k];
            mat_vec(p, pm, bpos);
            for (int k = 0; k < 3; k++) p[k] += xpos[3 * pid + k];
            quat_mul(q, pq, bquat);
          } else {
            for (int k = 0; k < 3; k++) p[k] = bpos[k];
            for (int k = 0; k < 4; k++) q[k] = bquat[k];
          }
          for (int j = ja; j < ja + jn; j++) {
            T anchor[3], axis[3];
            const int qa = mdl.jnt_qposadr(j);
            T jaxis[3] = {mdl.jnt_axis(3 * j), mdl.jnt_axis(3 * j + 1), mdl.jnt_axis(3 * j + 2)};
            T jpos[3] = {mdl.jnt_pos(3 * j), mdl.jnt_pos(3 * j + 1), mdl.jnt_pos(3 * j + 2)};
            quat_rot(axis, jaxis, q);
            quat_rot(anchor, jpos, q);
            for (int k = 0; k < 3; k++) anchor[k] += p[k];
            const T disp = qpos[qa] - mdl.qpos0(qa);
            if (mdl.jnt_type(j) == JNT_SLIDE) {
              for (int k = 0; k < 3; k++) p[k] += axis[k] * disp;
            } else {
              T ql[4], off[3];
              quat_axis_angle(ql, jaxis, disp);
              quat_mul(q, q, ql);
              quat_rot(off, jpos, q);
              for (int k = 0; k < 3; k++) p[k] = anchor[k] - off[k];
            }
            for (int k = 0; k < 3; k++) { xanchor[3 * j + k] = anchor[k]; xaxis[3 * j + k] = axis[k]; }
          }
        }
        normalize4(q);
        T m9[9], qi[4], ip[3];
        quat_to_mat(m9, q);
        for (int k = 0; k < 3; k++) xpos[3 * i + k] = p[k];
        for (int k = 0; k < 4; k++) xquat[4 * i + k] = q[k];
        for (int k = 0; k < 9; k++) xmat[9 * i + k] = m9[k];
        T ipos[3] = {mdl.body_ipos(3 * i), mdl.body_ipos(3 * i + 1), mdl.body_ipos(3 * i + 2)};
        T iquat[4] = {mdl.body_iquat(4 * i), mdl.body_iquat(4 * i + 1), mdl.body_iquat(4 * i + 2), mdl.body_iquat(4 * i + 3)};
        mat_vec(ip, m9, ipos);
        for (int k = 0; k < 3; k++) xipos[3 * i + k] = ip[k] + p[k];
        quat_mul(qi, q, iquat);
        quat_to_mat(m9, qi);
        for (int k = 0; k < 9; k++) ximat[9 * i + k] = m9[k];
      }
      __syncwarp();
    }
    WFOR(g, mdl.ngeom()) {
      const int b = mdl.geom_bodyid(g);
      T gp[3] = {mdl.geom_pos(3 * g), mdl.geom_pos(3 * g + 1), mdl.geom_pos(3 * g + 2)};
      T gq[4] = {mdl.geom_quat(4 * g), mdl.geom_quat(4 * g + 1), mdl.geom_quat(4 * g + 2), mdl.geom_quat(4 * g + 3)};
      T bm[9], bq[4], r[3], q[4], m9[9];
      for (int k = 0; k < 9; k++) bm[k] = xmat[9 * b + k];
      for (int k = 0; k < 4; k++) bq[k] = xquat[4 * b + k];
      mat_vec(r, bm, gp);
      for (int k = 0; k < 3; k++) geom_xpos[3 * g + k] = r[k] + xpos[3 * b + k];
      quat_mul(q, bq, gq);
      quat_to_mat(m9, q);
      geom_z[3 * g] = m9[2]; geom_z[3 * g + 1] = m9[5]; geom_z[3 * g + 2] = m9[8];
    }
    __syncwarp();
  }

  // subtree centres of mass, com-frame inertias, motion axes
  B2_DEV void com_frame() {
    const int nb = mdl.nbody();
    WFOR(i, nb) {
      T s[3] = {0, 0, 0};
      for (int j = i; j < nb; j++)
        if (in_subtree(i, j)) { const T mj = mdl.body_mass(j); for (int k = 0; k < 3; k++) s[k] += xipos[3 * j + k] * mj; }
      if (mdl.body_subtreemass(i) < Num<T>::minval()) { for (int k = 0; k < 3; k++) s[k] = xipos[3 * i + k]; }
      else { const T inv = T(1) / tmax(Num<T>::minval(), mdl.body_subtreemass(i)); for (int k = 0; k < 3; k++) s[k] *= inv; }
      for (int k = 0; k < 3; k++) com[3 * i + k] = s[k];
    }
    __syncwarp();
    WFOR(i, nb) {
      T ci[10];
      if (i == 0) { for (int k = 0; k < 10; k++) ci[k] = 0; }
      else {
        const int r = mdl.body_rootid(i);
        T off[3], inertia[3] = {mdl.body_inertia(3 * i), mdl.body_inertia(3 * i + 1), mdl.body_inertia(3 * i + 2)}, im[9];
        for (int k = 0; k < 3; k++) off[k] = xipos[3 * i + k] - com[3 * r + k];
        for (int k = 0; k < 9; k++) im[k] = ximat[9 * i + k];
        inert_about(ci, inertia, im, off, mdl.body_mass(i));
      }
      for (int k = 0; k < 10; k++) cinert[10 * i + k] = ci[k];
    }
    WFOR(j, mdl.njnt()) {
      const int b = mdl.jnt_bodyid(j), r = mdl.body_rootid(b);
      T* cd = cdof + 6 * mdl.jnt_dofadr(j);
      T off[3], ax[3];
      for (int k = 0; k < 3; k++) off[k] = com[3 * r + k] - xanchor[3 * j + k];
      const int t = mdl.jnt_type(j);
      if (t == JNT_FREE) {
        for (int k = 0; k < 18; k++) cd[k] = 0;
        cd[3] = 1; cd[10] = 1; cd[17] = 1;
        for (int a = 0; a < 3; a++) {
          T c3[3];
          ax[0] = xmat[9 * b + a]; ax[1] = xmat[9 * b + a + 3]; ax[2] = xmat[9 * b + a + 6];
          cross3(c3, ax, off);
          T* c = cd + 18 + 6 * a;
          c[0] = ax[0]; c[1] = ax[1]; c[2] = ax[2]; c[3] = c3[0]; c[4] = c3[1]; c[5] = c3[2];
        }
      } else if (t == JNT_SLIDE) {
        cd[0] = cd[1] = cd[2] = 0;
        for (int k = 0; k < 3; k++) cd[3 + k] = xaxis[3 * j + k];
      } else {
        T c3[3];
        for (int k = 0; k < 3; k++) ax[k] = xaxis[3 * j + k];
        cross3(c3, ax, off);
        for (int k = 0; k < 3; k++) { cd[k] = ax[k]; cd[3 + k] = c3[k]; }
      }
    }
    WFOR(t, mdl.ntendon()) {
      T L = 0;
      for (int k = 0; k < mdl.nv(); k++) ten_J[t * mdl.nv() + k] = 0;
      for (int w = mdl.tendon_adr(t); w < mdl.tendon_adr(t) + mdl.tendon_num(t); w++) {
        const int j = mdl.wrap_jntid(w);
        L += mdl.wrap_coef(w) * qpos[mdl.jnt_qposadr(j)];
        ten_J[t * mdl.nv() + mdl.jnt_dofadr(j)] = mdl.wrap_coef(w);
      }
      ten_len[t] = L;
    }
    __syncwarp();
  }

  // composite inertias (subtree sums) and the packed lower-triangular mass matrix
  B2_DEV void mass_matrix() {
    const int nb = mdl.nbody(), nv = mdl.nv();
    WFOR(i, nb) {
      T s[10];
      for (int k = 0; k < 10; k++) s[k] = cinert[10 * i + k];
      if (i > 0)
        for (int j = nb - 1; j > i; j--)   // children accumulate from the last body backwards, as upstream's reverse pass
          if (in_subtree(i, j)) for (int k = 0; k < 10; k++) s[k] += cinert[10 * j + k];
      for (int k = 0; k < 10; k++) crb[10 * i + k] = s[k];
    }
    __syncwarp();
    WFOR(d, nv) {
      T b6[6], c[10], cd[6];
      const int b = mdl.dof_bodyid(d);
      for (int k = 0; k < 10; k++) c[k] = crb[10 * b + k];
      for (int k = 0; k < 6; k++) cd[k] = cdof[6 * d + k];
      inert_mul(b6, c, cd);
      for (int k = 0; k < 6; k++) buf6[6 * d + k] = b6[k];
    }
    __syncwarp();
    const int np = nv * (nv + 1) / 2;
    WFOR(e, np) {
      int i, j;
      mdl.untri(e, i, j);
      T v = 0;
      if (dof_is_anc(i, j)) { for (int k = 0; k < 6; k++) v += cdof[6 * j + k] * buf6[6 * i + k]; }
      if (i == j) v = mdl.dof_armature(i) + v;
      Mp[e] = v;
    }
    __syncwarp();
  }

  // in-place L'DL of the packed matrix in LDp (tree sparsity): per pivot k all ancestor pairs at once
  B2_DEV void factor_LD() { factor_LD_impl<T, int>(mdl.nv(), mdl.img->model.dof_nanc, mdl.img->model.dof_anclist, LDp, dinv, lane); }
  B2_DEV void solve_LD(T* x) { solve_LD_impl<T>(mdl.nv(), tree_mask, LDp, dinv, x, lane); }
  // the Newton Hessian's factor and solve: over the merged tree when a row couples two branches
  B2_DEV void factor_H(T* H) {
    if (rows_cross) factor_LD_impl<T, unsigned char>(mdl.nv(), dyn_nanc, dyn_list, H, hdinv, lane);
    else factor_LD_impl<T, int>(mdl.nv(), mdl.img->model.dof_nanc, mdl.img->model.dof_anclist, H, hdinv, lane);
  }
  B2_DEV void solve_H(const T* H, T* x) { solve_LD_impl<T>(mdl.nv(), rows_cross ? amask : tree_mask, H, hdinv, x, lane); }
  // a constraint row couples the chains `chains` (bit set of dofs): every dof of the union gets the union's lower dofs as
  // ancestors
  B2_DEV void couple(unsigned chains) {
    rows_cross = true;
    if ((chains >> lane) & 1u) amask |= chains & ((1u << lane) - 1u);
  }
  // Symbolic factorisation of the merged pattern (eliminating dof k, leaves first, makes its ancestors a clique) and the
  // compact ancestor lists the numeric factorisation walks (nearest ancestor first), written to the scratch slot.
  B2_DEV void merge_branches() {
    const int nv = mdl.nv();
#pragma unroll 1
    for (int k = nv - 1; k > 0; k--) {
      const unsigned mk = __shfl_sync(0xffffffffu, amask, k);
      if ((mk >> lane) & 1u) amask |= mk & ((1u << lane) - 1u);
    }
#pragma unroll 1
    for (int k = 0; k < nv; k++) {
      const unsigned mk = __shfl_sync(0xffffffffu, amask, k);
      if (lane == 0) dyn_nanc[k] = __popc(mk);
      if ((mk >> lane) & 1u) dyn_list[k * 32 + __popc(mk >> (lane + 1))] = (unsigned char)lane;  // bits set only below k <= 31
    }
    __syncwarp();
  }
  B2_DEV void mul_M(T* r, const T* v) { mul_M_impl<T>(Mp, r, v, mdl.nv(), lane); }

  // Jacobian column of dof d for a point on `body` at offset `off` from the root's subtree CoM; false if d does not move body
  B2_DEV bool jac_col(int last, int d, const T* off, T* jp) const {
    if (last < 0 || d > last || !dof_is_anc(last, d)) return false;
    T c[6];
    for (int k = 0; k < 6; k++) c[k] = cdof[6 * d + k];
    cross3(jp, c, off);
    jp[0] += c[3]; jp[1] += c[4]; jp[2] += c[5];
    return true;
  }
  B2_DEV int last_dof(int body) const {
    while (body && !mdl.body_dofnum(body)) body = mdl.body_parentid(body);
    return body ? mdl.body_dofadr(body) + mdl.body_dofnum(body) - 1 : -1;
  }

  // ------------------------------------------------------------------ collision + rows
  // candidate pairs are tested 32 at a time; contacts are appended in pair order (ballot prefix)
  B2_DEV void collide() {
    ncon = 0;
    const int np = mdl.npair();
    for (int base = 0; base < np; base += 32) {
      const int p = base + lane;
      int cnt = 0;
      T cd[2], cpos[6], cfr[12];
      if (p < np) {
        const int g1 = mdl.pair_geom1(p), g2 = mdl.pair_geom2(p);
        const T margin = mdl.pair_margin(p);
        T p1[3], p2[3], z1[3], z2[3], d[3];
        for (int k = 0; k < 3; k++) { p1[k] = geom_xpos[3 * g1 + k]; p2[k] = geom_xpos[3 * g2 + k]; z1[k] = geom_z[3 * g1 + k]; z2[k] = geom_z[3 * g2 + k]; d[k] = p2[k] - p1[k]; }
        const int t1 = mdl.geom_type(g1), t2 = mdl.geom_type(g2);
        const T r1 = mdl.geom_size(3 * g1), l1 = mdl.geom_size(3 * g1 + 1), r2 = mdl.geom_size(3 * g2), l2 = mdl.geom_size(3 * g2 + 1);
        auto emit = [&](T dist, const T* pos, const T* n, const T* hint) {
          cd[cnt] = dist;
          for (int k = 0; k < 3; k++) { cpos[3 * cnt + k] = pos[k]; cfr[6 * cnt + k] = n[k]; cfr[6 * cnt + 3 + k] = hint ? hint[k] : T(0); }
          cnt++;
        };
        auto plane_sphere = [&](const T* sp, T radius, const T* hint) {
          T dd[3] = {sp[0] - p1[0], sp[1] - p1[1], sp[2] - p1[2]};
          const T c = dot3(dd, z1);
          if (c > margin + radius) return;
          const T dist = c - radius, s = -dist / 2 - radius;
          T pos[3] = {sp[0] + z1[0] * s, sp[1] + z1[1] * s, sp[2] + z1[2] * s};
          emit(dist, pos, z1, hint);
        };
        auto sphere_sphere = [&](const T* a, T ra, const T* b, T rb) -> int {
          T n[3] = {b[0] - a[0], b[1] - a[1], b[2] - a[2]};
          const T dsq = dot3(n, n), lim = margin + ra + rb;
          if (dsq > lim * lim) return 0;
          const T c = normalize3(n);
          const T dist = c - ra - rb;
          if (c < Num<T>::minval()) { cross3(n, z1, z2); normalize3(n); }
          const T s = ra + T(0.5) * dist;
          T pos[3] = {a[0] + n[0] * s, a[1] + n[1] * s, a[2] + n[2] * s};
          emit(dist, pos, n, nullptr);
          return 1;
        };
        if (t1 == GEOM_PLANE) {
          if (dot3(d, z1) <= margin + mdl.geom_rbound(g2)) {
            if (t2 == GEOM_SPHERE) plane_sphere(p2, r2, nullptr);
            else if (t2 == GEOM_CAPSULE) {
              T e[3];
              for (int k = 0; k < 3; k++) e[k] = p2[k] + z2[k] * l2;
              plane_sphere(e, r2, z2);
              for (int k = 0; k < 3; k++) e[k] = p2[k] - z2[k] * l2;
              plane_sphere(e, r2, z2);
            }
          }
        } else {
          const T bound = margin + mdl.geom_rbound(g1) + mdl.geom_rbound(g2);
          if (dot3(d, d) <= bound * bound) {
            if (t1 == GEOM_SPHERE && t2 == GEOM_SPHERE) sphere_sphere(p1, r1, p2, r2);
            else if (t1 == GEOM_SPHERE && t2 == GEOM_CAPSULE) {
              T v[3] = {-d[0], -d[1], -d[2]};
              const T x = tclip(dot3(z2, v), -l2, l2);
              for (int k = 0; k < 3; k++) v[k] = p2[k] + z2[k] * x;
              sphere_sphere(p1, r1, v, r2);
            } else if (t1 == GEOM_CAPSULE && t2 == GEOM_CAPSULE) {
              T dif[3] = {-d[0], -d[1], -d[2]}, v1[3], v2[3];
              const T ma = dot3(z1, z1), mb = -dot3(z1, z2), mc = dot3(z2, z2), u = -dot3(z1, dif), w = dot3(z2, dif);
              const T det = ma * mc - mb * mb;
              if (fabs(det) >= Num<T>::minval()) {
                T x1 = (mc * u - mb * w) / det, x2 = (ma * w - mb * u) / det;
                if (x1 > l1) { x1 = l1; x2 = (w - mb * l1) / mc; }
                else if (x1 < -l1) { x1 = -l1; x2 = (w + mb * l1) / mc; }
                if (x2 > l2) { x2 = l2; x1 = tclip((u - mb * l2) / ma, -l1, l1); }
                else if (x2 < -l2) { x2 = -l2; x1 = tclip((u + mb * l2) / ma, -l1, l1); }
                for (int k = 0; k < 3; k++) { v1[k] = p1[k] + z1[k] * x1; v2[k] = p2[k] + z2[k] * x2; }
                sphere_sphere(v1, r1, v2, r2);
              } else {
                int n = 0;
                for (int side = 1; side >= -1 && n < 2; side -= 2) {
                  const T x = tclip((w - side * mb * l1) / mc, -l2, l2);
                  for (int k = 0; k < 3; k++) { v1[k] = p1[k] + z1[k] * (side * l1); v2[k] = p2[k] + z2[k] * x; }
                  n += sphere_sphere(v1, r1, v2, r2);
                }
                for (int side = 1; side >= -1 && n < 2; side -= 2) {
                  const T x = tclip((u - side * mb * l2) / ma, -l1, l1);
                  for (int k = 0; k < 3; k++) { v2[k] = p2[k] + z2[k] * (side * l2); v1[k] = p1[k] + z1[k] * x; }
                  n += sphere_sphere(v1, r1, v2, r2);
                }
              }
            }
          }
        }
      }
      // exclusive prefix of per-lane contact counts (0..2) keeps pair order
      int incl = cnt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
      const int total = __shfl_sync(0xffffffffu, incl, 31);
      const int start = ncon + incl - cnt;
      for (int c = 0; c < cnt; c++) {
        const int slot = start + c;
        if (slot < WarpCaps::NCON) {
          T fr[9];
          for (int k = 0; k < 6; k++) fr[k] = cfr[6 * c + k];
          make_frame_shared(fr);
          con_dist[slot] = cd[c]; con_pair[slot] = p;
          for (int k = 0; k < 3; k++) con_pos[3 * slot + k] = cpos[3 * c + k];
          for (int k = 0; k < 9; k++) con_frame[9 * slot + k] = fr[k];
        }
      }
      ncon += total;
      if (ncon > WarpCaps::NCON) { ncon = WarpCaps::NCON; flags |= 8; }
    }
    __syncwarp();
  }

  // limit rows (joints, then tendons) followed by contact rows; J rows are written one dof per lane
  B2_DEV void make_rows() {
    const int nv = mdl.nv();
    nefc = 0;
    rows_cross = false;
    amask = tree_mask;
    auto zero_row = [&](int r) { WFOR(k, nv) J[r * nv + k] = 0; };
    // joint limits: sequential over joints keeps upstream row order; the test itself is uniform
    for (int j = 0; j < mdl.njnt(); j++) {
      if (!mdl.jnt_limited(j) || mdl.jnt_type(j) < JNT_SLIDE) continue;
      const T value = qpos[mdl.jnt_qposadr(j)], margin = mdl.jnt_margin(j);
      for (int side = -1; side <= 1; side += 2) {
        const T dist = side * (mdl.jnt_range(2 * j + (side + 1) / 2) - value);
        if (dist < margin) {
          if (nefc >= WarpCaps::NEFC) { flags |= 8; continue; }
          const int r = nefc++;
          zero_row(r);
          __syncwarp();
          if (lane == 0) { row_meta[r] = ROW_LIMIT_JOINT | (j << 8); row_pos[r] = dist; row_margin[r] = margin; J[r * nv + mdl.jnt_dofadr(j)] = T(-side); }
        }
      }
    }
    for (int t = 0; t < mdl.ntendon(); t++) {
      if (!mdl.tendon_limited(t)) continue;
      const T value = ten_len[t], margin = mdl.tendon_margin(t);
      for (int side = -1; side <= 1; side += 2) {
        const T dist = side * (mdl.tendon_range(2 * t + (side + 1) / 2) - value);
        if (dist < margin) {
          if (nefc >= WarpCaps::NEFC) { flags |= 8; continue; }
          const int r = nefc++;
          // a fixed tendon couples the dofs of its joints: chain-compatible if they are ancestors of one another
          bool chain = true;
          unsigned chains = 0;
          for (int w = mdl.tendon_adr(t); w < mdl.tendon_adr(t) + mdl.tendon_num(t); w++) {
            const int d1 = mdl.jnt_dofadr(mdl.wrap_jntid(w));
            chains |= (unsigned)mdl.dof_anc(d1);
            for (int u = mdl.tendon_adr(t); u < w; u++) {
              const int d2 = mdl.jnt_dofadr(mdl.wrap_jntid(u));
              if (!(d1 >= d2 ? dof_is_anc(d1, d2) : dof_is_anc(d2, d1))) chain = false;
            }
          }
          if (!chain) couple(chains);
          WFOR(k, nv) J[r * nv + k] = -side * ten_J[t * nv + k];
          if (lane == 0) { row_meta[r] = ROW_LIMIT_TENDON | (t << 8); row_pos[r] = dist; row_margin[r] = margin; }
        }
      }
    }
    for (int c = 0; c < ncon; c++) {
      const int p = con_pair[c];
      const T incl = mdl.pair_margin(p) - mdl.pair_gap(p), dist = con_dist[c];
      if (dist >= incl) continue;
      const int dim = mdl.pair_dim(p), nrow = dim == 1 ? 1 : 4;
      if (nefc + nrow > WarpCaps::NEFC) { flags |= 8; break; }
      const int r0 = nefc;
      nefc += nrow;
      const int b1 = mdl.geom_bodyid(mdl.pair_geom1(p)), b2 = mdl.geom_bodyid(mdl.pair_geom2(p));
      const int last1 = last_dof(b1), last2 = last_dof(b2);
      if (last1 >= 0 && last2 >= 0 && !(last1 >= last2 ? dof_is_anc(last1, last2) : dof_is_anc(last2, last1)))
        couple((unsigned)mdl.dof_anc(last1) | (unsigned)mdl.dof_anc(last2));
      const T mu = mdl.pair_friction(2 * p);
      T fr[9], pos[3], off1[3], off2[3];
      for (int k = 0; k < 9; k++) fr[k] = con_frame[9 * c + k];
      for (int k = 0; k < 3; k++) { pos[k] = con_pos[3 * c + k]; off1[k] = pos[k] - com[3 * mdl.body_rootid(b1) + k]; off2[k] = pos[k] - com[3 * mdl.body_rootid(b2) + k]; }
      WFOR(d, nv) {
        T acc[4] = {0, 0, 0, 0}, jp[3];
        // body 1 enters with a minus sign, then body 2 with a plus sign (same accumulation order as the lane engine)
        for (int pass = 0; pass < 2; pass++) {
          const T sgn = pass ? T(1) : T(-1);
          if (!jac_col(pass ? last2 : last1, d, pass ? off2 : off1, jp)) continue;
          const T jn = sgn * dot3(fr, jp);
          if (dim == 1) { acc[0] += jn; continue; }
          const T j1 = sgn * dot3(fr + 3, jp), j2 = sgn * dot3(fr + 6, jp);
          acc[0] += jn + mu * j1; acc[1] += jn - mu * j1; acc[2] += jn + mu * j2; acc[3] += jn - mu * j2;
        }
        for (int k = 0; k < nrow; k++) J[(r0 + k) * nv + d] = acc[k];
      }
      if (lane < nrow) { row_meta[r0 + lane] = (dim == 1 ? ROW_CONTACT_1 : ROW_CONTACT_PYR) | (c << 8); row_pos[r0 + lane] = dist; row_margin[r0 + lane] = incl; }
    }
    __syncwarp();
    if (rows_cross) merge_branches();
  }

  static B2_DEV T impedance(const T* si, T pos, T margin) {
    const T lo = T(0.0001), hi = T(0.9999);
    const T dmin = tclip(si[0], lo, hi), dmax = tclip(si[1], lo, hi), width = tmax(Num<T>::minval(), si[2]);
    const T mid = tclip(si[3], lo, hi), power = tmax(T(1), si[4]);
    if (dmin == dmax || width <= Num<T>::minval()) return T(0.5) * (dmin + dmax);
    T x = (pos - margin) / width;
    if (x < 0) x = -x;
    if (x >= 1) return dmax;
    if (x == 0) return dmin;
    T y;
    if (power == 1) y = x;
    else if (x <= mid) y = (T(1) / pow(mid, power - 1)) * pow(x, power);
    else y = T(1) - (T(1) / pow(T(1) - mid, power - 1)) * pow(T(1) - x, power);
    return dmin + y * (dmax - dmin);
  }
  B2_DEV void row_params() {
    const int nv = mdl.nv();
    WFOR(i, nefc) {
      T sr[2], si[5], diag;
      const int type = row_meta[i] & 255, id = row_meta[i] >> 8;
      T mu = 0;
      if (type == ROW_LIMIT_JOINT) {
        for (int k = 0; k < 2; k++) sr[k] = mdl.jnt_solref(2 * id + k);
        for (int k = 0; k < 5; k++) si[k] = mdl.jnt_solimp(5 * id + k);
        diag = mdl.dof_invweight0(mdl.jnt_dofadr(id));
      } else if (type == ROW_LIMIT_TENDON) {
        for (int k = 0; k < 2; k++) sr[k] = mdl.tendon_solref(2 * id + k);
        for (int k = 0; k < 5; k++) si[k] = mdl.tendon_solimp(5 * id + k);
        diag = mdl.tendon_invweight0(id);
      } else {
        const int p = con_pair[id];
        for (int k = 0; k < 2; k++) sr[k] = mdl.pair_solref(2 * p + k);
        for (int k = 0; k < 5; k++) si[k] = mdl.pair_solimp(5 * p + k);
        const T tran = mdl.body_invweight0(2 * mdl.geom_bodyid(mdl.pair_geom1(p))) + mdl.body_invweight0(2 * mdl.geom_bodyid(mdl.pair_geom2(p)));
        mu = mdl.pair_friction(2 * p);
        diag = (type == ROW_CONTACT_1) ? tran : tran + mu * mu * tran;
      }
      const T pos = row_pos[i], margin = row_margin[i];
      const T imp = impedance(si, pos, margin);
      const T dmax = tclip(si[1], T(0.0001), T(0.9999));
      T K, B;
      if (sr[0] > 0) {
        const T tc = tmax(sr[0], 2 * mdl.timestep()), dr = sr[1];
        K = T(1) / tmax(Num<T>::minval(), dmax * dmax * tc * tc * dr * dr);
        B = T(2) / tmax(Num<T>::minval(), dmax * tc);
      } else {
        K = -sr[0] / tmax(Num<T>::minval(), dmax * dmax);
        B = -sr[1] / tmax(Num<T>::minval(), dmax);
      }
      T reg = tmax(Num<T>::minval(), (T(1) - imp) * diag / imp);
      if (type == ROW_CONTACT_PYR) reg = 2 * mu * mu * reg;  // all four edges share pos/margin, hence the same value
      row_D[i] = T(1) / reg;
      T vel = 0;
      for (int k = 0; k < nv; k++) vel += J[i * nv + k] * qvel[k];
      row_aref[i] = -B * vel - K * imp * (pos - margin);
    }
    __syncwarp();
  }

  // ------------------------------------------------------------------ velocity stage
  B2_DEV void velocities() {
    const int nb = mdl.nbody();
    if (lane < 6) cvel[lane] = 0;
    __syncwarp();
    for (int level = 1; level <= mdl.maxdepth(); level++) {
      const int i = lane;
      if (i < nb && mdl.body_depth(i) == level) {
        T v[6], cd[6], cdd[6];
        const int da = mdl.body_dofadr(i), dn = mdl.body_dofnum(i), p = mdl.body_parentid(i);
        for (int k = 0; k < 6; k++) v[k] = cvel[6 * p + k];
        if (dn == 6 && mdl.jnt_type(mdl.dof_jntid(da)) == JNT_FREE) {
          for (int k = 0; k < 18; k++) cdof_dot[6 * da + k] = 0;
          for (int k = 0; k < 6; k++) {
            T t = 0;
            for (int q = 0; q < 3; q++) t += cdof[6 * (da + q) + k] * qvel[da + q];
            v[k] += t;
          }
          for (int q = 3; q < 6; q++) {
            for (int k = 0; k < 6; k++) cd[k] = cdof[6 * (da + q) + k];
            cross_motion(cdd, v, cd);
            for (int k = 0; k < 6; k++) cdof_dot[6 * (da + q) + k] = cdd[k];
          }
          for (int k = 0; k < 6; k++) {
            T t = 0;
            for (int q = 3; q < 6; q++) t += cdof[6 * (da + q) + k] * qvel[da + q];
            v[k] += t;
          }
        } else {
          for (int j = 0; j < dn; j++) {
            for (int k = 0; k < 6; k++) cd[k] = cdof[6 * (da + j) + k];
            cross_motion(cdd, v, cd);
            for (int k = 0; k < 6; k++) { cdof_dot[6 * (da + j) + k] = cdd[k]; v[k] += cd[k] * qvel[da + j]; }
          }
        }
        for (int k = 0; k < 6; k++) cvel[6 * i + k] = v[k];
      }
      __syncwarp();
    }
  }

  B2_DEV void passive_forces() {
    const int nv = mdl.nv();
    WFOR(d, nv) {
      const int j = mdl.dof_jntid(d);
      T f = 0;
      const T st = mdl.jnt_stiffness(j);
      if (st != 0 && mdl.jnt_type(j) >= JNT_SLIDE) { const int pa = mdl.jnt_qposadr(j); f -= st * (qpos[pa] - mdl.qpos_spring(pa)); }
      f -= mdl.dof_damping(d) * qvel[d];
      f_passive[d] = f;
    }
    __syncwarp();
    for (int t = 0; t < mdl.ntendon(); t++) {
      const T st = mdl.tendon_stiffness(t), dm = mdl.tendon_damping(t);
      if (st == 0 && dm == 0) continue;
      T frc = 0, vel = 0;
      const T lo = mdl.tendon_lengthspring(2 * t), hi = mdl.tendon_lengthspring(2 * t + 1), L = ten_len[t];
      if (L > hi) frc = st * (hi - L); else if (L < lo) frc = st * (lo - L);
      for (int k = 0; k < nv; k++) vel += ten_J[t * nv + k] * qvel[k];
      frc -= dm * vel;
      WFOR(k, nv) f_passive[k] += ten_J[t * nv + k] * frc;
      __syncwarp();
    }
  }

  // recursive Newton-Euler without accelerations
  B2_DEV void bias_forces() {
    const int nb = mdl.nbody(), nv = mdl.nv();
    if (lane < 6) cacc[lane] = lane < 3 ? T(0) : -mdl.gravity(lane - 3);
    __syncwarp();
    for (int level = 1; level <= mdl.maxdepth(); level++) {
      const int i = lane;
      if (i < nb && mdl.body_depth(i) == level) {
        const int da = mdl.body_dofadr(i), p = mdl.body_parentid(i);
        T t[6] = {0, 0, 0, 0, 0, 0};
        for (int j = 0; j < mdl.body_dofnum(i); j++)
          for (int k = 0; k < 6; k++) t[k] += cdof_dot[6 * (da + j) + k] * qvel[da + j];
        for (int k = 0; k < 6; k++) cacc[6 * i + k] = cacc[6 * p + k] + t[k];
      }
      __syncwarp();
    }
    T* cfrc_body = buf6;  // 6 per body (nb <= nv + 1 is not guaranteed; buf6 holds 6*nv >= 6*(nb-1); world slot unused)
    WFOR(i, nb) {
      if (i == 0) continue;
      T ci[10], a[6], v[6], f[6], t[6], t1[6];
      for (int k = 0; k < 10; k++) ci[k] = cinert[10 * i + k];
      for (int k = 0; k < 6; k++) { a[k] = cacc[6 * i + k]; v[k] = cvel[6 * i + k]; }
      inert_mul(f, ci, a);
      inert_mul(t, ci, v);
      cross_force(t1, v, t);
      for (int k = 0; k < 6; k++) cfrc_body[6 * (i - 1) + k] = f[k] + t1[k];
    }
    __syncwarp();
    // subtree force sums land in crb's storage (dead after the mass matrix): 6 per body
    T* cfrc = crb;
    WFOR(i, nb) {
      if (i == 0) continue;
      T s[6];
      for (int k = 0; k < 6; k++) s[k] = cfrc_body[6 * (i - 1) + k];
      for (int j = nb - 1; j > i; j--)
        if (in_subtree(i, j)) for (int k = 0; k < 6; k++) s[k] += cfrc_body[6 * (j - 1) + k];
      for (int k = 0; k < 6; k++) cfrc[6 * i + k] = s[k];
    }
    __syncwarp();
    WFOR(d, nv) {
      T s = 0;
      const int b = mdl.dof_bodyid(d);
      for (int k = 0; k < 6; k++) s += cdof[6 * d + k] * cfrc[6 * b + k];
      f_bias[d] = s;
    }
    __syncwarp();
  }

  B2_DEV void smooth_dynamics() {
    const int nv = mdl.nv();
    WFOR(d, nv) {
      T fa = 0;
      for (int a = 0; a < mdl.nu(); a++) {
        const int jid = mdl.actuator_trnid(a);
        if (mdl.jnt_dofadr(jid) != d) continue;
        T u = ctrl[a];
        if (mdl.actuator_ctrllimited(a)) u = tclip(u, mdl.actuator_ctrlrange(2 * a), mdl.actuator_ctrlrange(2 * a + 1));
        const T gear = mdl.actuator_gear(6 * a);
        const T len = qpos[mdl.jnt_qposadr(jid)] * gear, vel = gear * qvel[d];
        T force = mdl.actuator_gainprm(a) * u + mdl.actuator_biasprm(3 * a) + mdl.actuator_biasprm(3 * a + 1) * len + mdl.actuator_biasprm(3 * a + 2) * vel;
        if (mdl.actuator_forcelimited(a)) force = tclip(force, mdl.actuator_forcerange(2 * a), mdl.actuator_forcerange(2 * a + 1));
        if (mdl.actuator_disabled(a)) force = 0;
        fa += gear * force;
      }
      T fs = f_passive[d] - f_bias[d];
      fs += fa;
      f_smooth[d] = fs; a_smooth[d] = fs;
    }
    __syncwarp();
    solve_LD(a_smooth);
  }

  // ------------------------------------------------------------------ Newton solver
  // J v for all rows: one row per lane
  B2_DEV void mul_J(T* out, const T* v, const T* sub) { mul_J_impl<T>(J, out, v, sub, nefc, mdl.nv(), lane); }
  B2_DEV T row_cost(const T* jar) {
    T c = 0;
    WFOR(i, nefc) if (jar[i] < 0) c += T(0.5) * row_D[i] * jar[i] * jar[i];
    return warp_sum(c);
  }
  B2_DEV T dotv(const T* a, const T* b) {
    T s = 0;
    WFOR(k, mdl.nv()) s += a[k] * b[k];
    return warp_sum(s);
  }
  struct LsPoint { T alpha, cost, d1, d2; };
  B2_DEV void ls_eval(T alpha, LsPoint& p) {
    ls_iter++;
    ls_eval_impl<T>(Jaref, Jv, row_D, nefc, lane, qg0, qg1, qg2, alpha, &p.alpha);
  }
  B2_DEV int ls_bracket(LsPoint& p, const LsPoint* cand, LsPoint& pnext) {
    int flag = 0;
    for (int i = 0; i < 3; i++) {
      if (p.d1 < 0 && cand[i].d1 < 0 && p.d1 < cand[i].d1) { p = cand[i]; flag = 1; }
      else if (p.d1 > 0 && cand[i].d1 > 0 && p.d1 > cand[i].d1) { p = cand[i]; flag = 2; }
    }
    if (flag) ls_eval(p.alpha - p.d1 / p.d2, pnext);
    return flag;
  }
  B2_DEV T line_search() {
    const int nv = mdl.nv();
    LsPoint p0, p1, p2, pmid, p1n, p2n;
    ls_iter = 0;
    const T sn = sqrt(dotv(search, search));
    if (sn < Num<T>::minval()) return 0;
    const T scale = T(1) / (mdl.meaninertia() * T(nv > 1 ? nv : 1));
    const T gtol = mdl.tolerance() * mdl.ls_tolerance() * sn / scale;
    mul_M(Mv, search);
    mul_J(Jv, search, nullptr);
    qg0 = gauss; qg1 = dotv(search, Ma) - dotv(f_smooth, search); qg2 = T(0.5) * dotv(search, Mv);
    ls_eval(0, p0);
    ls_eval(p0.alpha - p0.d1 / p0.d2, p1);
    if (p0.cost < p1.cost) p1 = p0;
    if (fabs(p1.d1) < gtol) return p1.alpha;
    const int dir = p1.d1 < 0 ? 1 : -1;
    bool p2up = false;
    const int maxls = mdl.ls_iterations();
    while (p1.d1 * dir <= -gtol && ls_iter < maxls) {
      p2 = p1; p2up = true;
      ls_eval(p1.alpha - p1.d1 / p1.d2, p1);
      if (fabs(p1.d1) < gtol) return p1.alpha;
    }
    if (ls_iter >= maxls || !p2up) return p1.alpha;
    p2n = p1;
    ls_eval(p1.alpha - p1.d1 / p1.d2, p1n);
    while (ls_iter < maxls) {
      ls_eval(T(0.5) * (p1.alpha + p2.alpha), pmid);
      LsPoint cand[3] = {p1n, p2n, pmid};
      T best = 0; int bi = -1;
      for (int i = 0; i < 3; i++)
        if (fabs(cand[i].d1) < gtol && (bi == -1 || cand[i].cost < best)) { best = cand[i].cost; bi = i; }
      if (bi >= 0) return cand[bi].alpha;
      const int b1 = ls_bracket(p1, cand, p1n), b2 = ls_bracket(p2, cand, p2n);
      if (!b1 && !b2) return pmid.alpha;
    }
    if (p1.cost <= p2.cost && p1.cost < p0.cost) return p1.alpha;
    if (p2.cost <= p1.cost && p2.cost < p0.cost) return p2.alpha;
    return 0;
  }
  // cost, constraint force and gradient at the current iterate ...
  B2_DEV void newton_gradient() {
    const int nv = mdl.nv();
    cost = row_cost(Jaref);
    WFOR(k, nv) {
      T f = 0;
      for (int i = 0; i < nefc; i++) if (Jaref[i] < 0) f += J[i * nv + k] * (-row_D[i] * Jaref[i]);
      f_con[k] = f;
    }
    __syncwarp();
    T g = 0;
    WFOR(k, nv) { g += (Ma[k] - f_smooth[k]) * (qacc[k] - a_smooth[k]); grad[k] = Ma[k] - f_smooth[k] - f_con[k]; }
    gauss = T(0.5) * warp_sum(g);
    cost += gauss;
  }
  // ... and the Newton direction H^-1 grad (H = M + J' D_active J).  Only called when the iterate is not accepted as
  // converged: the round that detects convergence needs cost and gradient but no direction, which saves one of the
  // ~4.5 Hessian factorisations of a humanoid step (same iterates, bit for bit).
  B2_DEV void newton_direction() {
    const int nv = mdl.nv(), np = nv * (nv + 1) / 2;
    // Hessian, packed lower triangle in LDp: each lane owns entries e = lane, lane + 32, ...
    // It only depends on the active set: when no row changed state since the last refresh the
    // factor in LDp is still valid (bit-identical to refactoring) and is reused.
    T* H = LDp;
    unsigned sig[(WarpCaps::NEFC + 31) / 32];
    bool same = hess_valid;
#pragma unroll
    for (int w = 0; w < (WarpCaps::NEFC + 31) / 32; w++) {
      const int r = w * 32 + lane;
      sig[w] = __ballot_sync(0xffffffffu, r < nefc && Jaref[r] < 0);
      same = same && sig[w] == active_sig[w];
      active_sig[w] = sig[w];
    }
    hess_valid = true;
    if (!same) {
    {
      // rows outer, entries inner: each lane accumulates its packed entries e = lane + 32 t in registers while the
      // active rows are visited in increasing order (the summation order of the scalar algorithm)
      constexpr int EPL = 17;  // ceil(32 * 33 / 2 / 32)
      T h[EPL];
      int ij[EPL];  // row | col << 8 of this lane's entries, -1 beyond the end (skipping the entries outside the tree
                    // pattern when every row is a chain row was measured 2.7 % slower: the predicate costs more than the FMAs)
#pragma unroll
      for (int t = 0; t < EPL; t++) {
        ij[t] = lane + 32 * t < np ? (int)__ldg(&mdl.img->tri_ij[lane + 32 * t]) & 0x7fff : -1;
        h[t] = lane + 32 * t < np ? Mp[lane + 32 * t] : T(0);
      }
#pragma unroll 1
      for (int w = 0; w < (WarpCaps::NEFC + 31) / 32; w++) {
        for (unsigned bits = w == 0 ? sig[0] : (w == 1 ? sig[1] : (w == 2 ? sig[2] : sig[3])); bits; bits &= bits - 1) {
          const int r = w * 32 + __ffs(bits) - 1;
          const T* Jr = J + r * nv;
          const T d = row_D[r];
#ifndef B2_WARP_HESS_GATHER
          // the row is read once, one dof per lane, and its entries travel by shuffle instead of being gathered from the
          // scratch slot entry by entry: +2 % at 4.7 contacts per env, +5 % at 7.7 (gpurun A/B, round 2)
          const T jl = lane < nv ? Jr[lane] : T(0), djl = d * jl;
#pragma unroll
          for (int t = 0; t < EPL; t++) {
            const int a = ij[t] >= 0 ? ij[t] & 255 : 0, b = ij[t] >= 0 ? ij[t] >> 8 : 0;
            const T pa = __shfl_sync(0xffffffffu, djl, a), pb = __shfl_sync(0xffffffffu, jl, b);
            if (ij[t] >= 0) h[t] += pa * pb;
          }
#else
#pragma unroll
          for (int t = 0; t < EPL; t++) {
            if (ij[t] >= 0) {
              h[t] += (d * Jr[ij[t] & 255]) * Jr[ij[t] >> 8];
            }
          }
#endif
        }
      }
#pragma unroll
      for (int t = 0; t < EPL; t++) if (lane + 32 * t < np) H[lane + 32 * t] = h[t];
    }
    __syncwarp();
    // H has the sparsity of the (merged) tree: the tree-sparse L'DL of mj_factorM factorises it
    factor_H(H);
    }  // !same
    WFOR(k, nv) Mgrad[k] = grad[k];
    __syncwarp();
    solve_H(H, Mgrad);
  }
  // Lock step: the warps of a block run the same stage at the same time, separated by block barriers, so that one
  // instruction fetch from L2 serves all of them.  The kernel is bound by instruction-fetch bandwidth: its 276 KB of
  // SASS cannot stay in the 32 KB L1.5 instruction cache, and two resident warps per SM already reach 69 % of the
  // throughput of eight that run out of phase.  The Newton loop runs free (no barrier per round): measured on the
  // humanoid (200-step rollout, blocks of four warps, cost-ordered queue) 7.44e6 env-steps/s against 7.30e6 with a barrier
  // in every round -- the loop's code is small enough to stay in the instruction cache, and a warp no longer waits for its
  // block mates.  The lock-step group is the whole block and the barrier is barrier 0: a register-valued barrier id makes
  // ptxas reserve all 16 barriers per block, which caps an SM at four blocks whatever the registers and shared memory
  // would allow (ncu "Block Limit Barriers", profiles/ncu_hum_step_r01j.txt).
  B2_DEV void stage_sync() const { __syncthreads(); }
  B2_DEV void constrained_acceleration() {
    const int nv = mdl.nv();
    niter = 0;
    bool done = false;
    if (!nefc) {
      WFOR(k, nv) { qacc[k] = a_smooth[k]; warm[k] = a_smooth[k]; f_con[k] = 0; }
      __syncwarp();
      return;
    }
    row_params();
    hess_valid = false;
    WFOR(k, nv) qacc[k] = warm[k];
    __syncwarp();
    mul_J(Jaref, qacc, row_aref);
    T cw = row_cost(Jaref);
    mul_M(Ma, qacc);
    T g = 0;
    WFOR(k, nv) g += T(0.5) * (Ma[k] - f_smooth[k]) * (qacc[k] - a_smooth[k]);
    cw += warp_sum(g);
    mul_J(Jv, a_smooth, row_aref);
    const T cs = row_cost(Jv);
    if (cw > cs) {
      WFOR(k, nv) qacc[k] = a_smooth[k];
      WFOR(i, nefc) Jaref[i] = Jv[i];
      __syncwarp();
      mul_M(Ma, qacc);
    }
    const T scale = T(1) / (mdl.meaninertia() * T(nv > 1 ? nv : 1));
    T old = 0;
    bool first = true;
    while (!done) {
      newton_gradient();
      if (!first) {
        const T gn = dotv(grad, grad);
        niter++;
        if (scale * (old - cost) < mdl.tolerance() || scale * sqrt(gn) < mdl.tolerance()) done = true;
      }
      if (!done && niter >= mdl.iterations()) done = true;  // iteration cap: the iterate stands, no further search
      if (!done) {
        newton_direction();
        first = false;
        WFOR(k, nv) search[k] = -Mgrad[k];
        __syncwarp();
      }
      if (!done) {
        const T alpha = line_search();
        if (alpha == 0) done = true;
        else {
          WFOR(k, nv) { qacc[k] += alpha * search[k]; Ma[k] += alpha * Mv[k]; }
          WFOR(i, nefc) Jaref[i] += alpha * Jv[i];
          __syncwarp();
          old = cost;
        }
      }
    }
    WFOR(k, nv) warm[k] = qacc[k];
    __syncwarp();
  }

  // ------------------------------------------------------------------ forward + Euler
  // after_position(): called once the position-dependent arrays (xpos .. geom_xpos, com) are complete and before their
  // storage is reused -- the kernels export the derived outputs there.
  template <class F>
  B2_DEV void forward(F&& after_position) {
    const int nv = mdl.nv(), np = nv * (nv + 1) / 2;
    kinematics();
    stage_sync();
    collide();
    stage_sync();
    com_frame();
    after_position();
    stage_sync();
    make_rows();
    stage_sync();
    mass_matrix();  // from here on region X holds the dynamics arrays
    stage_sync();
    velocities();
    passive_forces();
    stage_sync();
    bias_forces();
    WFOR(e, np) LDp[e] = Mp[e];  // ... and from here on the factor and the solver vectors
    __syncwarp();
    stage_sync();
    factor_LD();
    stage_sync();
    smooth_dynamics();
    stage_sync();
    constrained_acceleration();
  }
  B2_DEV void check_state() {
    int bad = 0;
    WFOR(k, mdl.nq()) if (!(fabs(qpos[k]) <= T(1e10))) bad |= 1;
    WFOR(k, mdl.nv()) if (!(fabs(qvel[k]) <= T(1e10))) bad |= 2;
    flags |= __reduce_or_sync(0xffffffffu, bad);
  }
  B2_DEV void check_acc() {
    int bad = 0;
    WFOR(k, mdl.nv()) if (!(fabs(qacc[k]) <= T(1e10))) bad |= 4;
    flags |= __reduce_or_sync(0xffffffffu, bad);
  }
  B2_DEV void euler() {
    const int nv = mdl.nv(), np = nv * (nv + 1) / 2;
    const T h = mdl.timestep();
    T* acc = grad;
    if (!mdl.has_dofdamping()) { WFOR(k, nv) acc[k] = qacc[k]; __syncwarp(); }
    else {
      WFOR(k, nv) acc[k] = f_smooth[k] + f_con[k];
      __syncwarp();
      // implicit joint damping: (M + h diag(damping))^-1.  (Building this factor in the same sweep as M's, two matrices per
      // pivot, was measured 2.3 % slower: tools/ab_run.sh, round 2.)
      WFOR(e, np) LDp[e] = Mp[e];
      __syncwarp();
      WFOR(k, nv) LDp[tri(k, k)] += h * mdl.dof_damping(k);
      __syncwarp();
      factor_LD();
      solve_LD(acc);
    }
    WFOR(k, nv) qvel[k] += acc[k] * h;
    __syncwarp();
    WFOR(j, mdl.njnt()) {
      const int pa = mdl.jnt_qposadr(j), va = mdl.jnt_dofadr(j);
      if (mdl.jnt_type(j) == JNT_FREE) {
        T q[4], w[3];
        for (int k = 0; k < 3; k++) qpos[pa + k] += h * qvel[va + k];
        for (int k = 0; k < 4; k++) q[k] = qpos[pa + 3 + k];
        for (int k = 0; k < 3; k++) w[k] = qvel[va + 3 + k];
        quat_integrate(q, w, h);
        for (int k = 0; k < 4; k++) qpos[pa + 3 + k] = q[k];
      } else qpos[pa] += h * qvel[va];
    }
    __syncwarp();
  }
};

}  // namespace b2
