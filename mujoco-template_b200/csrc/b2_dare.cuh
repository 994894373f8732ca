// Batched discrete-time LQR synthesis on the device (SURVEY.md section 8f row 2): the gain the reference's example
// controllers compute once per system on the host with scipy.linalg.solve_discrete_are
// (reference examples/drone/controllers/lqr.py:350-378, examples/humanoid/controllers/lqr.py:114-115), for every env of a
// batch from its own FD linearisation (A, B) -- the arrays b2_linearize / b2_control_tick write, in their SoA layout.
//
// One warp per env, all matrices of the env in shared memory.  The DARE  P = A'PA - A'PB (R + B'PB)^-1 B'PA + Q  is solved
// by the structure-preserving doubling iteration (k doublings = 2^k steps of the Riccati recursion, quadratic convergence):
//     W = I + G H;   [V1 V2] = W^-1 [A G];   H <- H + A' H V1;   G <- G + A V2 A';   A <- A V1        (G0 = B R^-1 B', H0 = Q)
// W^-1 [A G] by Gauss-Jordan elimination with partial pivoting on the augmented nx x 3nx block; afterwards
//     K = (R + B'PB)^-1 B'PA      (u = -K x).
// Work per doubling: five nx^3 products and one nx x 3nx elimination; nx = 4 (cartpole), 12 (drone), 54 (humanoid).
#pragma once
#include "b2_math.cuh"

namespace b2 {

// shared-memory reals one env needs: A, G, H, the augmented [W | V1 V2] block (3 nx^2) and two scratch matrices
__host__ __device__ inline size_t dare_ws_reals(int nx, int nu) { return (size_t)8 * nx * nx + (size_t)2 * nx * nu + (size_t)2 * nu * nu + 32; }

template <typename T>
B2_DEV void dare_matmul(T* C, const T* X, bool tx, const T* Y, bool ty, int n, int lane) {
  // C (n x n) = op(X) op(Y), one entry per lane and sweep (C is write-only: it may hold anything, NaN included)
  for (int e = lane; e < n * n; e += 32) {
    const int i = e / n, j = e - i * n;
    T s = 0;
    for (int k = 0; k < n; k++) s += (tx ? X[k * n + i] : X[i * n + k]) * (ty ? Y[j * n + k] : Y[k * n + j]);
    C[e] = s;
  }
  __syncwarp();
}

// In-place Gauss-Jordan with partial pivoting on M (n rows, w columns, the first n of them the matrix to invert): on return the
// trailing w - n columns hold inverse * (their old content).  Returns false when a pivot underflows.
template <typename T>
B2_DEV bool dare_gauss_jordan(T* M, int n, int w, int lane) {
  for (int c = 0; c < n; c++) {
    // pivot search over rows c..n-1 of column c (warp arg-max)
    T best = -1; int row = c;
    for (int r = c + lane; r < n; r += 32) { const T a = fabs(M[r * w + c]); if (a > best) { best = a; row = r; } }
    for (int o = 16; o > 0; o >>= 1) {
      const T ob = __shfl_xor_sync(0xffffffffu, best, o); const int orow = __shfl_xor_sync(0xffffffffu, row, o);
      if (ob > best || (ob == best && orow < row)) { best = ob; row = orow; }
    }
    if (!(best > Num<T>::minval())) return false;
    if (row != c) for (int k = lane; k < w; k += 32) { const T t = M[c * w + k]; M[c * w + k] = M[row * w + k]; M[row * w + k] = t; }
    __syncwarp();
    const T inv = T(1) / M[c * w + c];
    __syncwarp();
    for (int k = lane; k < w; k += 32) M[c * w + k] *= inv;
    __syncwarp();
    // eliminate column c from every other row: entries (r, k), k > c (column c itself is not needed again)
    for (int e = lane; e < n * (w - c - 1); e += 32) {
      const int r = e / (w - c - 1), k = c + 1 + e - r * (w - c - 1);
      if (r != c) M[r * w + k] -= M[r * w + c] * M[c * w + k];
    }
    __syncwarp();
  }
  return true;
}

// A (nx, nx, N), B (nx, nu, N), K (nu, nx, N), P (nx, nx, N): env fastest (element (i, j, e) at [(i * cols + j) * N + e]).
// Q (nx x nx), R (nu x nu), Rinv (nu x nu): row-major, shared by all envs.  status[e]: doublings used, negated on failure.
template <typename T>
__global__ void __launch_bounds__(128) k_dare(const T* __restrict__ Ag, const T* __restrict__ Bg, const T* __restrict__ Q,
                                              const T* __restrict__ R, const T* __restrict__ Rinv, int nx, int nu, int N,
                                              int max_doublings, T tol, T* Kg, T* Pg, int* status) {
  extern __shared__ double b2_dare_smem[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, e = blockIdx.x * (blockDim.x >> 5) + wib;
  if (e >= N) return;
  const int nn = nx * nx;
  T* ws = reinterpret_cast<T*>(b2_dare_smem) + (size_t)wib * dare_ws_reals(nx, nu);
  T *A = ws, *G = A + nn, *H = G + nn, *M = H + nn /* nx x 3nx */, *T1 = M + 3 * nn, *T2 = T1 + nn, *Bm = T2 + nn /* nx x nu */,
    *BR = Bm + nx * nu /* nx x nu: B Rinv, later P B */, *S = BR + nx * nu /* nu x 2nu */;
#ifdef B2_DARE_POISON  // debugging aid: every read of workspace the kernel has not written shows up as a failed env
  for (int k = lane; k < (int)dare_ws_reals(nx, nu); k += 32) ws[k] = T(__int_as_float(0x7fc00000));
  __syncwarp();
#endif
  for (int k = lane; k < nn; k += 32) { A[k] = Ag[(size_t)k * N + e]; H[k] = Q[k]; }
  for (int k = lane; k < nx * nu; k += 32) Bm[k] = Bg[(size_t)k * N + e];
  __syncwarp();
  // G0 = B Rinv B'
  for (int k = lane; k < nx * nu; k += 32) {
    const int i = k / nu, a = k - i * nu;
    T s = 0;
    for (int b = 0; b < nu; b++) s += Bm[i * nu + b] * Rinv[b * nu + a];
    BR[k] = s;
  }
  __syncwarp();
  for (int k = lane; k < nn; k += 32) {
    const int i = k / nx, j = k - i * nx;
    T s = 0;
    for (int a = 0; a < nu; a++) s += BR[i * nu + a] * Bm[j * nu + a];
    G[k] = s;
  }
  __syncwarp();
  int used = 0;
  bool ok = true;
  for (int it = 0; it < max_doublings; it++) {
    // M = [I + G H | A | G]
    dare_matmul(T1, G, false, H, false, nx, lane);
    for (int k = lane; k < nn; k += 32) {
      const int i = k / nx, j = k - i * nx;
      M[i * 3 * nx + j] = T1[k] + (i == j ? T(1) : T(0));
      M[i * 3 * nx + nx + j] = A[k];
      M[i * 3 * nx + 2 * nx + j] = G[k];
    }
    __syncwarp();
    ok = dare_gauss_jordan(M, nx, 3 * nx, lane);
    if (!ok) break;
    // T1 = V1, T2 = V2 (contiguous copies)
    for (int k = lane; k < nn; k += 32) { const int i = k / nx, j = k - i * nx; T1[k] = M[i * 3 * nx + nx + j]; T2[k] = M[i * 3 * nx + 2 * nx + j]; }
    __syncwarp();
    // H <- H + A' (H V1): M[0..nn) = H V1, then accumulate; track the change of H
    dare_matmul(M, H, false, T1, false, nx, lane);
    T dmax = 0, hmax = 0;
    for (int k = lane; k < nn; k += 32) {
      const int i = k / nx, j = k - i * nx;
      T s = 0;
      for (int q = 0; q < nx; q++) s += A[q * nx + i] * M[q * nx + j];
      M[nn + k] = s;  // increment, symmetrised below
    }
    __syncwarp();
    for (int k = lane; k < nn; k += 32) {
      const int i = k / nx, j = k - i * nx;
      const T inc = T(0.5) * (M[nn + k] + M[nn + j * nx + i]);
      const T h = H[k] + inc;
      dmax = fmax(dmax, fabs(inc)); hmax = fmax(hmax, fabs(h));
      M[2 * nn + k] = h;
    }
    __syncwarp();
    for (int k = lane; k < nn; k += 32) H[k] = M[2 * nn + k];
    // G <- G + A V2 A': M[0..nn) = A V2, then (A V2) A' symmetrised
    dare_matmul(M, A, false, T2, false, nx, lane);
    dare_matmul(M + nn, M, false, A, true, nx, lane);
    for (int k = lane; k < nn; k += 32) { const int i = k / nx, j = k - i * nx; G[k] += T(0.5) * (M[nn + k] + M[nn + j * nx + i]); }
    // A <- A V1
    dare_matmul(M, A, false, T1, false, nx, lane);
    for (int k = lane; k < nn; k += 32) A[k] = M[k];
    __syncwarp();
    for (int o = 16; o > 0; o >>= 1) { dmax = fmax(dmax, __shfl_xor_sync(0xffffffffu, dmax, o)); hmax = fmax(hmax, __shfl_xor_sync(0xffffffffu, hmax, o)); }
    used = it + 1;
    if (it >= 3 && dmax <= tol * fmax(hmax, T(1))) break;
  }
  // P = H; K = (R + B'PB)^-1 B'PA with the ORIGINAL A (re-read)
  for (int k = lane; k < nn; k += 32) { Pg[(size_t)k * N + e] = H[k]; A[k] = Ag[(size_t)k * N + e]; }
  __syncwarp();
  for (int k = lane; k < nx * nu; k += 32) {  // BR = P B (nx x nu)
    const int i = k / nu, a = k - i * nu;
    T s = 0;
    for (int q = 0; q < nx; q++) s += H[i * nx + q] * Bm[q * nu + a];
    BR[k] = s;
  }
  __syncwarp();
  // augmented [R + B'PB | B'PA] : nu x (nu + nx), in M
  const int w = nu + nx;
  for (int k = lane; k < nu * nu; k += 32) {
    const int a = k / nu, b = k - a * nu;
    T s = R[k];
    for (int q = 0; q < nx; q++) s += Bm[q * nu + a] * BR[q * nu + b];
    M[a * w + b] = s;
  }
  for (int k = lane; k < nu * nx; k += 32) {
    const int a = k / nx, j = k - a * nx;
    T s = 0;
    for (int q = 0; q < nx; q++) s += BR[q * nu + a] * A[q * nx + j];  // (P B)' A = B' P A (P symmetric)
    M[a * w + nu + j] = s;
  }
  __syncwarp();
  ok = dare_gauss_jordan(M, nu, w, lane) && ok;
  for (int k = lane; k < nu * nx; k += 32) { const int a = k / nx, j = k - a * nx; Kg[(size_t)k * N + e] = M[a * w + nu + j]; }
  if (lane == 0 && status) status[e] = ok ? used : -used - 1;
  (void)S;
}

}  // namespace b2

namespace b2 {

// Thread-per-env variant for small systems (pendulum 2 x 1, cartpole 4 x 1, ...): compile-time sizes, every matrix in
// registers, same iteration and stopping rule as k_dare.  A warp per 4 x 4 system leaves 30 lanes idle; this form
// synthesises the gains of 65,536 cartpoles in a fraction of a millisecond, which makes re-synthesis at every control tick
// (time-varying LQR from the tick's own (A, B)) affordable.
template <typename T, int N>
B2_DEV void small_mul(T* C, const T* X, const T* Y) {  // C = X Y
#pragma unroll
  for (int i = 0; i < N; i++)
#pragma unroll
    for (int j = 0; j < N; j++) {
      T s = 0;
#pragma unroll
      for (int k = 0; k < N; k++) s += X[i * N + k] * Y[k * N + j];
      C[i * N + j] = s;
    }
}
template <typename T, int N>
B2_DEV void small_mul_tn(T* C, const T* X, const T* Y) {  // C = X' Y
#pragma unroll
  for (int i = 0; i < N; i++)
#pragma unroll
    for (int j = 0; j < N; j++) {
      T s = 0;
#pragma unroll
      for (int k = 0; k < N; k++) s += X[k * N + i] * Y[k * N + j];
      C[i * N + j] = s;
    }
}
template <typename T, int N>
B2_DEV void small_mul_nt(T* C, const T* X, const T* Y) {  // C = X Y'
#pragma unroll
  for (int i = 0; i < N; i++)
#pragma unroll
    for (int j = 0; j < N; j++) {
      T s = 0;
#pragma unroll
      for (int k = 0; k < N; k++) s += X[i * N + k] * Y[j * N + k];
      C[i * N + j] = s;
    }
}
// Gauss-Jordan with partial pivoting on [W | R1 R2] (N x N and two N x N right-hand sides), fully unrolled: the row swap is a
// chain of selects, so that no index is a run-time value and everything stays in registers.
template <typename T, int N, int RHS>
B2_DEV bool small_solve(T* W, T* R) {  // R: N x (RHS) row-major, overwritten by W^-1 R
  bool ok = true;
#pragma unroll
  for (int c = 0; c < N; c++) {
    // bring the largest |W[r][c]|, r >= c, to row c
#pragma unroll
    for (int r = c + 1; r < N; r++) {
      const bool sw = fabs(W[r * N + c]) > fabs(W[c * N + c]);
#pragma unroll
      for (int k = 0; k < N; k++) { const T a = W[c * N + k], b = W[r * N + k]; W[c * N + k] = sw ? b : a; W[r * N + k] = sw ? a : b; }
#pragma unroll
      for (int k = 0; k < RHS; k++) { const T a = R[c * RHS + k], b = R[r * RHS + k]; R[c * RHS + k] = sw ? b : a; R[r * RHS + k] = sw ? a : b; }
    }
    if (!(fabs(W[c * N + c]) > Num<T>::minval())) ok = false;
    const T inv = T(1) / W[c * N + c];
#pragma unroll
    for (int k = 0; k < N; k++) W[c * N + k] *= inv;
#pragma unroll
    for (int k = 0; k < RHS; k++) R[c * RHS + k] *= inv;
#pragma unroll
    for (int r = 0; r < N; r++) {
      if (r == c) continue;
      const T f = W[r * N + c];
#pragma unroll
      for (int k = 0; k < N; k++) W[r * N + k] -= f * W[c * N + k];
#pragma unroll
      for (int k = 0; k < RHS; k++) R[r * RHS + k] -= f * R[c * RHS + k];
    }
  }
  return ok;
}

template <typename T, int NX, int NU>
__global__ void __launch_bounds__(64) k_dare_small(const T* __restrict__ Ag, const T* __restrict__ Bg, const T* __restrict__ Q,
                                                   const T* __restrict__ R, const T* __restrict__ Rinv, int N, int max_doublings, T tol,
                                                   T* Kg, T* Pg, int* status) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N) return;
  constexpr int NN = NX * NX;
  T A0[NN], A[NN], G[NN], H[NN], B[NX * NU];
#pragma unroll
  for (int k = 0; k < NN; k++) { A0[k] = Ag[(size_t)k * N + e]; A[k] = A0[k]; H[k] = Q[k]; }
#pragma unroll
  for (int k = 0; k < NX * NU; k++) B[k] = Bg[(size_t)k * N + e];
  {  // G0 = B Rinv B'
    T BR[NX * NU];
#pragma unroll
    for (int i = 0; i < NX; i++)
#pragma unroll
      for (int a = 0; a < NU; a++) { T s = 0;
#pragma unroll
        for (int b = 0; b < NU; b++) s += B[i * NU + b] * Rinv[b * NU + a];
        BR[i * NU + a] = s; }
#pragma unroll
    for (int i = 0; i < NX; i++)
#pragma unroll
      for (int j = 0; j < NX; j++) { T s = 0;
#pragma unroll
        for (int a = 0; a < NU; a++) s += BR[i * NU + a] * B[j * NU + a];
        G[i * NX + j] = s; }
  }
  int used = 0;
  bool ok = true;
#pragma unroll 1
  for (int it = 0; it < max_doublings; it++) {
    T W[NN], V[NX * 2 * NX];  // V = [A | G] -> W^-1 [A | G]
    small_mul<T, NX>(W, G, H);
#pragma unroll
    for (int i = 0; i < NX; i++) {
      W[i * NX + i] += T(1);
#pragma unroll
      for (int j = 0; j < NX; j++) { V[i * 2 * NX + j] = A[i * NX + j]; V[i * 2 * NX + NX + j] = G[i * NX + j]; }
    }
    ok = small_solve<T, NX, 2 * NX>(W, V);
    if (!ok) break;
    T V1[NN], V2[NN], t1[NN], t2[NN];
#pragma unroll
    for (int i = 0; i < NX; i++)
#pragma unroll
      for (int j = 0; j < NX; j++) { V1[i * NX + j] = V[i * 2 * NX + j]; V2[i * NX + j] = V[i * 2 * NX + NX + j]; }
    small_mul<T, NX>(t1, H, V1);
    small_mul_tn<T, NX>(t2, A, t1);  // A' H V1
    T dmax = 0, hmax = 0;
#pragma unroll
    for (int i = 0; i < NX; i++)
#pragma unroll
      for (int j = 0; j < NX; j++) {
        const T inc = T(0.5) * (t2[i * NX + j] + t2[j * NX + i]);
        t1[i * NX + j] = H[i * NX + j] + inc;
        dmax = fmax(dmax, fabs(inc)); hmax = fmax(hmax, fabs(t1[i * NX + j]));
      }
#pragma unroll
    for (int k = 0; k < NN; k++) H[k] = t1[k];
    small_mul<T, NX>(t1, A, V2);
    small_mul_nt<T, NX>(t2, t1, A);  // A V2 A'
#pragma unroll
    for (int i = 0; i < NX; i++)
#pragma unroll
      for (int j = 0; j < NX; j++) t1[i * NX + j] = G[i * NX + j] + T(0.5) * (t2[i * NX + j] + t2[j * NX + i]);
#pragma unroll
    for (int k = 0; k < NN; k++) G[k] = t1[k];
    small_mul<T, NX>(t1, A, V1);
#pragma unroll
    for (int k = 0; k < NN; k++) A[k] = t1[k];
    used = it + 1;
    if (it >= 3 && dmax <= tol * fmax(hmax, T(1))) break;
  }
#pragma unroll
  for (int k = 0; k < NN; k++) Pg[(size_t)k * N + e] = H[k];
  // K = (R + B'PB)^-1 B'P A0
  T PB[NX * NU], S[NU * NU], RH[NU * NX];
#pragma unroll
  for (int i = 0; i < NX; i++)
#pragma unroll
    for (int a = 0; a < NU; a++) { T s = 0;
#pragma unroll
      for (int q = 0; q < NX; q++) s += H[i * NX + q] * B[q * NU + a];
      PB[i * NU + a] = s; }
#pragma unroll
  for (int a = 0; a < NU; a++) {
#pragma unroll
    for (int b = 0; b < NU; b++) { T s = R[a * NU + b];
#pragma unroll
      for (int q = 0; q < NX; q++) s += B[q * NU + a] * PB[q * NU + b];
      S[a * NU + b] = s; }
#pragma unroll
    for (int j = 0; j < NX; j++) { T s = 0;
#pragma unroll
      for (int q = 0; q < NX; q++) s += PB[q * NU + a] * A0[q * NX + j];
      RH[a * NX + j] = s; }
  }
  ok = small_solve<T, NU, NX>(S, RH) && ok;
#pragma unroll
  for (int k = 0; k < NU * NX; k++) Kg[(size_t)k * N + e] = RH[k];
  if (status) status[e] = ok ? used : -used - 1;
}

}  // namespace b2

namespace b2 {

// ---- Finite-horizon time-varying LQR / the backward pass of iLQR (b2_tvlqr, see include/b2mj.h for the recursion).
// A (nsteps, nx, nx, N), B (nsteps, nx, nu, N), q (nsteps+1, nx, N), r (nsteps, nu, N), K (nsteps, nu, nx, N),
// k (nsteps, nu, N), P0 (nx, nx, N), dV (2, N): env fastest.  W: Q (nx x nx), R (nu x nu), Qf (nx x nx), row-major, shared
// by all envs.  q, r, k, P0, dV and status may be null.  A step whose Quu + reg I is not positive definite gets NaN gains;
// they make P, and so every earlier step, NaN as well, so only the first failure (the largest t) is recorded.

// Thread per env for the sizes k_dare_small covers: every matrix in registers, nu <= 2 (closed-form Cholesky).
template <typename T, int NX, int NU>
__global__ void __launch_bounds__(64) k_tvlqr_small(const T* __restrict__ Ag, const T* __restrict__ Bg, const T* __restrict__ W,
                                                    const T* __restrict__ qg, const T* __restrict__ rg, int nsteps, int N, T reg, T* Kg,
                                                    T* kg, T* P0g, T* dVg, int* status) {
  static_assert(NU == 1 || NU == 2, "closed-form Cholesky");
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N) return;
  constexpr int NN = NX * NX;
  const T *Q = W, *R = W + NN, *Qf = W + NN + NU * NU;
  const T nan = T(__int_as_float(0x7fc00000));
  T P[NN], s[NX];
#pragma unroll
  for (int k = 0; k < NN; k++) P[k] = Qf[k];
#pragma unroll
  for (int i = 0; i < NX; i++) s[i] = qg ? qg[((size_t)nsteps * NX + i) * N + e] : T(0);
  T dv0 = 0, dv1 = 0;
  int failed = 0;
#pragma unroll 1
  for (int t = nsteps - 1; t >= 0; t--) {
    T A[NN], B[NX * NU], PA[NN], PB[NX * NU];
#pragma unroll
    for (int k = 0; k < NN; k++) A[k] = Ag[((size_t)t * NN + k) * N + e];
#pragma unroll
    for (int k = 0; k < NX * NU; k++) B[k] = Bg[((size_t)t * NX * NU + k) * N + e];
    small_mul<T, NX>(PA, P, A);
#pragma unroll
    for (int i = 0; i < NX; i++)
#pragma unroll
      for (int a = 0; a < NU; a++) { T v = 0;
#pragma unroll
        for (int j = 0; j < NX; j++) v += P[i * NX + j] * B[j * NU + a];
        PB[i * NU + a] = v; }
    T Qx[NX], Qu[NU], Quu[NU * NU], Qux[NU * NX];
#pragma unroll
    for (int i = 0; i < NX; i++) { T v = qg ? qg[((size_t)t * NX + i) * N + e] : T(0);
#pragma unroll
      for (int j = 0; j < NX; j++) v += A[j * NX + i] * s[j];
      Qx[i] = v; }
#pragma unroll
    for (int a = 0; a < NU; a++) {
      T v = rg ? rg[((size_t)t * NU + a) * N + e] : T(0);
#pragma unroll
      for (int j = 0; j < NX; j++) v += B[j * NU + a] * s[j];
      Qu[a] = v;
#pragma unroll
      for (int b = 0; b < NU; b++) { T w = R[a * NU + b];
#pragma unroll
        for (int j = 0; j < NX; j++) w += B[j * NU + a] * PB[j * NU + b];
        Quu[a * NU + b] = w; }
#pragma unroll
      for (int i = 0; i < NX; i++) { T w = 0;
#pragma unroll
        for (int j = 0; j < NX; j++) w += B[j * NU + a] * PA[j * NX + i];
        Qux[a * NX + i] = w; }
    }
    small_mul_tn<T, NX>(P, A, PA);  // P <- Qxx = Q + A'PA
#pragma unroll
    for (int k = 0; k < NN; k++) P[k] += Q[k];
    // K = (Quu + reg I)^-1 Qux, k = -(Quu + reg I)^-1 Qu by the Cholesky factor L L' of Quu + reg I (lower triangle)
    T K[NU * NX], kk[NU];
    bool ok;
    if constexpr (NU == 1) {
      const T d = Quu[0] + reg;
      ok = d > T(0);
      const T inv = T(1) / d;
#pragma unroll
      for (int i = 0; i < NX; i++) K[i] = inv * Qux[i];
      kk[0] = -inv * Qu[0];
    } else {
      const T l11 = sqrt(Quu[0] + reg), l21 = Quu[2] / l11, d2 = Quu[3] + reg - l21 * l21, l22 = sqrt(d2);
      ok = Quu[0] + reg > T(0) && d2 > T(0);
      auto solve = [&](T y1, T y2, T& x1, T& x2) {
        const T z1 = y1 / l11, z2 = (y2 - l21 * z1) / l22;
        x2 = z2 / l22; x1 = (z1 - l21 * x2) / l11;
      };
#pragma unroll
      for (int i = 0; i < NX; i++) solve(Qux[i], Qux[NX + i], K[i], K[NX + i]);
      solve(-Qu[0], -Qu[1], kk[0], kk[1]);
    }
    if (!ok) {
      if (!failed) failed = t + 1;
#pragma unroll
      for (int k = 0; k < NU * NX; k++) K[k] = nan;
#pragma unroll
      for (int a = 0; a < NU; a++) kk[a] = nan;
    }
    // P <- Qxx + K'(Quu K - Qux) - Qux'K (symmetrised);  s <- Qx - K'(Qu + Quu k) + Qux'k
    T M[NU * NX], w[NU];
#pragma unroll
    for (int a = 0; a < NU; a++) {
      T v = Qu[a];
#pragma unroll
      for (int b = 0; b < NU; b++) v += Quu[a * NU + b] * kk[b];
      w[a] = v;
      dv0 += kk[a] * Qu[a];
      dv1 += T(0.5) * kk[a] * (v - Qu[a]);
#pragma unroll
      for (int i = 0; i < NX; i++) { T m = -Qux[a * NX + i];
#pragma unroll
        for (int b = 0; b < NU; b++) m += Quu[a * NU + b] * K[b * NX + i];
        M[a * NX + i] = m; }
    }
    T Pn[NN];
#pragma unroll
    for (int i = 0; i < NX; i++) {
#pragma unroll
      for (int j = 0; j < NX; j++) { T v = P[i * NX + j];
#pragma unroll
        for (int a = 0; a < NU; a++) v += K[a * NX + i] * M[a * NX + j] - Qux[a * NX + i] * K[a * NX + j];
        Pn[i * NX + j] = v; }
      T v = Qx[i];
#pragma unroll
      for (int a = 0; a < NU; a++) v += Qux[a * NX + i] * kk[a] - K[a * NX + i] * w[a];
      s[i] = v;
    }
#pragma unroll
    for (int i = 0; i < NX; i++)
#pragma unroll
      for (int j = 0; j < NX; j++) P[i * NX + j] = T(0.5) * (Pn[i * NX + j] + Pn[j * NX + i]);
#pragma unroll
    for (int k = 0; k < NU * NX; k++) Kg[((size_t)t * NU * NX + k) * N + e] = K[k];
    if (kg) {
#pragma unroll
      for (int a = 0; a < NU; a++) kg[((size_t)t * NU + a) * N + e] = kk[a];
    }
  }
  if (P0g) {
#pragma unroll
    for (int k = 0; k < NN; k++) P0g[(size_t)k * N + e] = P[k];
  }
  if (dVg) { dVg[e] = dv0; dVg[(size_t)N + e] = dv1; }
  if (status) status[e] = -failed;
}

// shared-memory reals one env of k_tvlqr needs: P, A, a scratch nx x nx; B, P B (later Quu K - Qux), Qux, K; Quu and its
// Cholesky factor; s, Qx; Qu, k, Qu + Quu k
__host__ __device__ inline size_t tvlqr_ws_reals(int nx, int nu) {
  return ((size_t)3 * nx * nx + (size_t)4 * nx * nu + (size_t)2 * nu * nu + 2 * (size_t)nx + 3 * (size_t)nu + 1) & ~(size_t)1;
}

// Warp per env, the env's matrices in shared memory; wpb (= blockDim.x / 32) consecutive envs per block.  The block stages
// A_t, B_t, q_t and r_t of its envs together, env fastest, so that a load of one matrix element of wpb envs uses whole
// 32-byte sectors (FP64, wpb = 4) where a warp loading its own env alone would use a quarter of each.
template <typename T>
__global__ void __launch_bounds__(128) k_tvlqr(const T* __restrict__ Ag, const T* __restrict__ Bg, const T* __restrict__ W,
                                               const T* __restrict__ qg, const T* __restrict__ rg, int nsteps, int nx, int nu, int N, T reg,
                                               T* Kg, T* kg, T* P0g, T* dVg, int* status) {
  extern __shared__ double b2_tvlqr_smem[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  const int e0 = blockIdx.x * wpb, e = e0 + wib;
  const bool active = e < N;
  const int nn = nx * nx, xu = nx * nu, uu = nu * nu;
  const size_t per = tvlqr_ws_reals(nx, nu);
  T* ws = reinterpret_cast<T*>(b2_tvlqr_smem) + (size_t)wib * per;
  T *P = ws, *A = P + nn, *S = A + nn, *Bm = S + nn, *PB = Bm + xu, *Qux = PB + xu, *K = Qux + xu, *Quu = K + xu, *L = Quu + uu,
    *s = L + uu, *Qx = s + nx, *Qu = Qx + nx, *kk = Qu + nu, *w = kk + nu;
  const T *Q = W, *R = W + nn, *Qf = W + nn + uu;
  const T nan = T(__int_as_float(0x7fc00000));
  // q_t and r_t are staged into Qx and Qu
  auto stage = [&](const T* src, int off, int count) {
    T* base = reinterpret_cast<T*>(b2_tvlqr_smem);
    for (int idx = threadIdx.x; idx < count * wpb; idx += blockDim.x) {
      const int j = idx % wpb, k = idx / wpb;
      if (e0 + j < N) base[(size_t)j * per + off + k] = src ? src[(size_t)k * N + e0 + j] : T(0);
    }
  };
  stage(qg ? qg + (size_t)nsteps * nx * N : nullptr, (int)(s - ws), nx);
  for (int k = lane; k < nn; k += 32) P[k] = Qf[k];
  T dv0 = 0, dv1 = 0;
  int failed = 0;
  for (int t = nsteps - 1; t >= 0; t--) {
    __syncthreads();  // every warp is done with the previous step's A, B, Qx, Qu
    stage(Ag + (size_t)t * nn * N, (int)(A - ws), nn);
    stage(Bg + (size_t)t * xu * N, (int)(Bm - ws), xu);
    stage(qg ? qg + (size_t)t * nx * N : nullptr, (int)(Qx - ws), nx);
    stage(rg ? rg + (size_t)t * nu * N : nullptr, (int)(Qu - ws), nu);
    __syncthreads();
    if (!active) continue;
    dare_matmul(S, P, false, A, false, nx, lane);  // S = P A
    for (int x = lane; x < xu; x += 32) {  // PB = P B
      const int i = x / nu, a = x - i * nu;
      T v = 0;
      for (int j = 0; j < nx; j++) v += P[i * nx + j] * Bm[j * nu + a];
      PB[x] = v;
    }
    __syncwarp();
    for (int x = lane; x < xu; x += 32) {  // Qux = B'PA
      const int a = x / nx, i = x - a * nx;
      T v = 0;
      for (int j = 0; j < nx; j++) v += Bm[j * nu + a] * S[j * nx + i];
      Qux[x] = v;
    }
    for (int x = lane; x < uu; x += 32) {  // Quu = R + B'PB
      const int a = x / nu, b = x - a * nu;
      T v = R[x];
      for (int j = 0; j < nx; j++) v += Bm[j * nu + a] * PB[j * nu + b];
      Quu[x] = v;
    }
    for (int i = lane; i < nx + nu; i += 32) {  // Qx = q + A's, Qu = r + B's
      T v = 0;
      if (i < nx) { for (int j = 0; j < nx; j++) v += A[j * nx + i] * s[j]; Qx[i] += v; }
      else { const int a = i - nx; for (int j = 0; j < nx; j++) v += Bm[j * nu + a] * s[j]; Qu[a] += v; }
    }
    for (int x = lane; x < nn; x += 32) {  // P <- Qxx = Q + A'PA
      const int i = x / nx, j = x - i * nx;
      T v = Q[x];
      for (int q = 0; q < nx; q++) v += A[q * nx + i] * S[q * nx + j];
      P[x] = v;
    }
    __syncwarp();
    // Cholesky L L' = Quu + reg I, column by column (lower triangle)
    bool ok = true;
    for (int c = 0; c < nu; c++) {
      T d = Quu[c * nu + c] + reg;
      for (int k = 0; k < c; k++) d -= L[c * nu + k] * L[c * nu + k];
      ok = ok && d > T(0);
      const T lcc = sqrt(d);
      for (int i = c + 1 + lane; i < nu; i += 32) {
        T v = Quu[i * nu + c];
        for (int k = 0; k < c; k++) v -= L[i * nu + k] * L[c * nu + k];
        L[i * nu + c] = v / lcc;
      }
      if (lane == 0) L[c * nu + c] = lcc;
      __syncwarp();
    }
    // K = L'^-1 L^-1 Qux and k = -L'^-1 L^-1 Qu: one right-hand side per lane, solved in place
    for (int c = lane; c <= nx; c += 32) {
      T* y = c < nx ? K + c : kk;
      const int ys = c < nx ? nx : 1;
      for (int a = 0; a < nu; a++) {
        T v = c < nx ? Qux[a * nx + c] : -Qu[a];
        for (int b = 0; b < a; b++) v -= L[a * nu + b] * y[b * ys];
        y[a * ys] = ok ? v / L[a * nu + a] : nan;
      }
      for (int a = nu - 1; a >= 0; a--) {
        T v = y[a * ys];
        for (int b = a + 1; b < nu; b++) v -= L[b * nu + a] * y[b * ys];
        y[a * ys] = ok ? v / L[a * nu + a] : nan;
      }
    }
    if (!ok && !failed) failed = t + 1;
    __syncwarp();
    for (int x = lane; x < xu; x += 32) {  // PB <- Quu K - Qux
      const int a = x / nx, i = x - a * nx;
      T v = -Qux[x];
      for (int b = 0; b < nu; b++) v += Quu[a * nu + b] * K[b * nx + i];
      PB[x] = v;
    }
    for (int a = lane; a < nu; a += 32) {  // w = Qu + Quu k
      T v = Qu[a];
      for (int b = 0; b < nu; b++) v += Quu[a * nu + b] * kk[b];
      w[a] = v;
    }
    __syncwarp();
    for (int x = lane; x < nn; x += 32) {  // S = Qxx + K'(Quu K - Qux) - Qux'K
      const int i = x / nx, j = x - i * nx;
      T v = P[x];
      for (int a = 0; a < nu; a++) v += K[a * nx + i] * PB[a * nx + j] - Qux[a * nx + i] * K[a * nx + j];
      S[x] = v;
    }
    for (int i = lane; i < nx; i += 32) {  // s = Qx - K'w + Qux'k
      T v = Qx[i];
      for (int a = 0; a < nu; a++) v += Qux[a * nx + i] * kk[a] - K[a * nx + i] * w[a];
      s[i] = v;
    }
    for (int a = 0; a < nu; a++) { dv0 += kk[a] * Qu[a]; dv1 += T(0.5) * kk[a] * (w[a] - Qu[a]); }
    for (int x = lane; x < xu; x += 32) Kg[((size_t)t * xu + x) * N + e] = K[x];
    if (kg) for (int a = lane; a < nu; a += 32) kg[((size_t)t * nu + a) * N + e] = kk[a];
    __syncwarp();
    for (int x = lane; x < nn; x += 32) { const int i = x / nx, j = x - i * nx; P[x] = T(0.5) * (S[x] + S[j * nx + i]); }
    __syncwarp();
  }
  if (!active) return;
  if (P0g) for (int x = lane; x < nn; x += 32) P0g[(size_t)x * N + e] = P[x];
  if (lane == 0) {
    if (dVg) { dVg[e] = dv0; dVg[(size_t)N + e] = dv1; }
    if (status) status[e] = -failed;
  }
}

}  // namespace b2
