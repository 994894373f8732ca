// Generic (runtime-model) instantiation of the lane-engine kernels for ONE arithmetic type.
// Included by b2_kernels_f64.cu and b2_kernels_f32.cu with B2_REAL / B2_SUFFIX defined; each
// translation unit owns its own __constant__ model images (one per size class), so the two
// precisions do not share the 64 KB constant bank.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>

#include "b2_kernel_templates.cuh"
#include "b2_kernels.h"
#include "b2_warp_kernels.cuh"
#include "b2_dare.cuh"

namespace b2 {

typedef B2_REAL real;

// The generic kernels read the model from a copy in shared memory, filled at kernel start from the model's image in device
// memory (one per model, device and precision, owned by the b2_model and passed to every launch).  Nothing about a model is
// process-wide device state: two models of one size class can run on different streams and from different threads, and a
// captured CUDA graph replays with the image it was captured with.  (Round 1 kept one image per size class in __constant__
// memory, swapped under a lock -- a graph replay could then run with another model's constants.)
__shared__ DevModel<real, DimsTiny> s_model_tiny;
__shared__ DevModel<real, DimsSmall> s_model_small;
__shared__ DevModel<real, DimsLarge> s_model_large;

template <class D> struct SharedImage;
template <> struct SharedImage<DimsTiny> { static B2_DEV DevModel<real, DimsTiny>& get() { return s_model_tiny; } };
template <> struct SharedImage<DimsSmall> { static B2_DEV DevModel<real, DimsSmall>& get() { return s_model_small; } };
template <> struct SharedImage<DimsLarge> { static B2_DEV DevModel<real, DimsLarge>& get() { return s_model_large; } };

// provider that reads the shared-memory image: uniform addresses (one broadcast read per warp), any model of the size class
template <class DD>
struct RuntimeModel {
  typedef DD D;
  static B2_DEV void load(const void* image) {  // whole block, before anything else (and before any thread returns)
    static_assert(sizeof(DevModel<real, D>) % 4 == 0, "model image is copied in 32-bit words");
    const unsigned* src = reinterpret_cast<const unsigned*>(image);
    unsigned* dst = reinterpret_cast<unsigned*>(&SharedImage<D>::get());
    for (int i = threadIdx.x; i < (int)(sizeof(DevModel<real, D>) / 4); i += blockDim.x) dst[i] = __ldg(src + i);
    __syncthreads();
  }
#define X(name) static B2_DEV int name() { return SharedImage<D>::get().name; }
  B2_MODEL_INT_SCALARS(X)
#undef X
#define X(name) static B2_DEV real name() { return SharedImage<D>::get().name; }
  B2_MODEL_REAL_SCALARS(X)
#undef X
#define X(name, cap) static B2_DEV int name(int i) { return SharedImage<D>::get().name[i]; }
  B2_MODEL_INT_ARRAYS(X)
#undef X
#define X(name, cap) static B2_DEV real name(int i) { return SharedImage<D>::get().name[i]; }
  B2_MODEL_REAL_ARRAYS(X)
#undef X
};

// register-resident FMA chain: measures the CUDA-core FP pipe peak the roofline is quoted against
__global__ void __launch_bounds__(256) k_fma_peak(real* out, int iters, real a, real b) {
  real x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
  for (int i = 0; i < iters; i++) {
    x0 = x0 * a + b; x1 = x1 * a + b; x2 = x2 * a + b; x3 = x3 * a + b;
    x4 = x4 * a + b; x5 = x5 * a + b; x6 = x6 * a + b; x7 = x7 * a + b;
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}

#define B2_DISPATCH(cls, CALL)                         \
  switch (cls) {                                       \
    case 0: { typedef DimsTiny DD; CALL; break; }      \
    case 1: { typedef DimsSmall DD; CALL; break; }     \
    default: { typedef DimsLarge DD; CALL; break; }    \
  }

#define B2_CAT_(a, b) a##b
#define B2_CAT(a, b) B2_CAT_(a, b)
#define B2_FN(name) B2_CAT(name, B2_SUFFIX)

// the lane engine's model image of a size class: size, and fill on the host (uploaded once per model by the C-ABI layer)
size_t B2_FN(b2k_image_bytes)(int cls) {
  size_t n = 0;
  B2_DISPATCH(cls, n = sizeof(DevModel<real, DD>));
  return n;
}
void B2_FN(b2k_image_fill)(int cls, const b2m_view* v, const int* disabled, void* host) {
  B2_DISPATCH(cls, fill_dev_model(*reinterpret_cast<DevModel<real, DD>*>(host), *v, disabled));
}
// returns measured TFLOP/s (2 flops per FMA) or a negative cudaError
double B2_FN(b2k_fma_peak)(void* stream) {
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int threads = 256, blocks = sms * 8, iters = 1 << 15;
  real* out = nullptr;
  if (cudaMalloc(&out, sizeof(real) * threads * blocks) != cudaSuccess) return -1;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  cudaStream_t s = (cudaStream_t)stream;
  k_fma_peak<<<blocks, threads, 0, s>>>(out, iters, (real)0.999999, (real)1e-7);
  float best = 1e30f;
  for (int rep = 0; rep < 5; rep++) {
    cudaEventRecord(e0, s);
    k_fma_peak<<<blocks, threads, 0, s>>>(out, iters, (real)0.999999, (real)1e-7);
    cudaEventRecord(e1, s);
    cudaEventSynchronize(e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    if (ms < best) best = ms;
  }
  cudaError_t err = cudaGetLastError();
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(out);
  if (err != cudaSuccess) return -(double)err;
  const double flops = 2.0 * 8.0 * iters * (double)threads * blocks;
  return flops / (best * 1e-3) / 1e12;
}
int B2_FN(b2k_step)(const void* image, int cls, const b2_state* st, const b2_derived* out, int count, int N, int nsteps, const void* gain,
                    const b2_state* park, void* stream) {
  const int threads = 128, blocks = (count + threads - 1) / threads;
  B2_DISPATCH(cls, (k_step<real, DD, RuntimeModel<DD>><<<blocks, threads, 0, (cudaStream_t)stream>>>(
                       to_dev<real>(st), to_dev<real>(out), out != nullptr, count, N, nsteps, (const real*)gain, to_dev<real>(park), image)));
  return (int)cudaGetLastError();
}
// ---- warp engine (large models): launch geometry and per-warp scratch are sized by the host
// Sizes with a compiled-in kernel variant (every workspace offset and loop bound a constant): the humanoid's.
typedef DimsStatic<28, 27, 21, 17, 22, 20, 2, 6> DimsHumanoid;
static int view_maxdepth(const b2m_view* v) {
  int best = 0;
  for (int i = 1; i < v->nbody; i++) {
    int depth = 0;
    for (int j = i; j > 0; j = v->body_parentid[j]) depth++;
    if (depth > best) best = depth;
  }
  return best;
}
static bool dims_are_humanoid(const b2m_view* v) {
  if (const char* x = getenv("B2_WARP_STATIC_DIMS")) if (x[0] == '0') return false;
  typedef DimsHumanoid H;
  return v->nq == H::NQ && v->nv == H::NV && v->nu == H::NU && v->nbody == H::NB && v->njnt == H::NJ && v->ngeom == H::NG &&
         v->ntendon == H::NT && view_maxdepth(v) == H::DEPTH;
}
#define B2_WARP_DIMS(v, CALL)                                          \
  if (dims_are_humanoid(v)) { typedef ImageModel<real, DimsHumanoid> WM; CALL; } \
  else { typedef ImageModel<real, DimsRuntime> WM; CALL; }

// lock-step mode of the warp kernels (WarpEnv::forward<LS>): 1 = every stage and every Newton round behind the block
// barrier, 2 = stages only (the Newton loop runs free), 0 = none.  Measured on the humanoid (200-step rollout, blocks of four
// warps, cost-ordered queue): mode 2 7.44e6 env-steps/s, mode 1 7.30e6 -- the Newton loop's code is small enough to stay
// in the instruction cache, and a warp no longer waits for its block mates in every round.
#ifndef B2_WARP_LS_MODE
#define B2_WARP_LS_MODE 2
#endif
static int warp_ws_reals_of(const b2m_view* v) { return warp_ws_reals(v->nq, v->nv, v->nu, v->nbody, v->njnt, v->ngeom, v->ntendon); }
static size_t warp_block_smem(const b2m_view* v, int wpb, int extra_reals) {
  size_t extra = 0;
  if (const char* x = getenv("B2_WARP_EXTRA_SMEM")) extra = (size_t)atoi(x);  // tuning: lowers the resident blocks per SM
  return extra + (size_t)wpb * ((size_t)warp_ws_reals_of(v) + extra_reals) * sizeof(real);
}
static int warp_wpb() {  // warps (envs) per lock-step block: 4 x 128 registers = 16 resident warps per SM, four to a fetch
  int wpb = 4;
  if (const char* x = getenv("B2_WARP_LS_WPB")) { const int w = atoi(x); if (w >= 1 && w <= 8) wpb = w; }
  return wpb;
}
template <class K>
static int warp_occupancy(K kern, int wpb, size_t smem, int* per_sm) {
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -1;
  // the whole L1 / shared-memory array as shared memory: the workspace per env decides how many warps an SM holds
  cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, kern, wpb * 32, smem) != cudaSuccess || *per_sm < 1) return -1;
  return 0;
}
size_t B2_FN(b2k_warp_image_bytes)() { return sizeof(WarpImage<real>); }
void B2_FN(b2k_warp_image_fill)(const b2m_view* v, const int* disabled, void* host) {
  fill_warp_image(*reinterpret_cast<WarpImage<real>*>(host), *v, disabled);
}
// chooses warps-per-block / grid so that every SM is filled; returns the number of warp slots (scratch slots)
int B2_FN(b2k_warp_plan)(const b2m_view* v, int N, int* out_wpb, int* out_blocks) {
  int dev = 0, sms = 0, smem_max = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  int wpb = warp_wpb();
  while (wpb > 1 && warp_block_smem(v, wpb, 0) + 1024 > (size_t)smem_max) wpb--;
  const size_t smem = warp_block_smem(v, wpb, 0);
  int per_sm = 0, rc = 0;
  B2_WARP_DIMS(v, (rc = warp_occupancy(k_warp_step_ls<real, WM, B2_WARP_LS_MODE>, wpb, smem, &per_sm)));
  if (rc) return -1;
  int blocks = sms * per_sm;
  const int need = (N + wpb - 1) / wpb;
  if (blocks > need) blocks = need;
  if (getenv("B2_WARP_DEBUG")) fprintf(stderr, "[b2mj] warp plan: %d warps/block, %d blocks/SM, %zu B shared memory/block, static dims %d\n", wpb, per_sm, smem, (int)dims_are_humanoid(v));
  *out_wpb = wpb; *out_blocks = blocks;
  return blocks * wpb;
}
size_t B2_FN(b2k_warp_scratch_bytes)(const b2m_view* v, int slots) {
  return (size_t)slots * warp_slot_reals(v->nv) * sizeof(real);
}
// bytes of the cost-ordered queue's buffers behind the work-queue counter: [hist | cursor] (2 kCostBins ints), cost[N], perm[N]
size_t B2_FN(b2k_warp_sort_bytes)(int N) { return (2 * kCostBins + 2 * (size_t)N) * sizeof(int); }
int B2_FN(b2k_warp_step)(const void* image, const b2m_view* v, const b2_state* st, const b2_derived* out, int N, int nsteps, void* jscratch,
                         void* counter, void* sortbuf, int wpb, int blocks, const b2_state* park, void* stream) {
  const size_t smem = warp_block_smem(v, wpb, 0);
  cudaStream_t s = (cudaStream_t)stream;
  // envs are handed out through a work queue: the first gridDim * wpb statically, the rest by atomic counter
  cudaError_t e = cudaMemsetAsync(counter, 0, sizeof(int), s);
  if (e != cudaSuccess) return (int)e;
  int *cost = nullptr, *perm = nullptr;
  if (sortbuf && wpb > 1 && nsteps > 0) {  // lock-step blocks: order the queue by the envs' last Newton iteration counts
    int* hist = (int*)sortbuf;
    cost = hist + 2 * kCostBins; perm = cost + N;
    if ((e = cudaMemsetAsync(hist, 0, 2 * kCostBins * sizeof(int), s)) != cudaSuccess) return (int)e;
    int sb = (N + 255) / 256;
    if (sb > 148 * 4) sb = 148 * 4;
    k_cost_hist<kCostBins><<<sb, 256, 0, s>>>(cost, N, hist);
    k_cost_scatter<kCostBins><<<sb, 256, 0, s>>>(cost, N, hist, hist + kCostBins, perm);
  }
  B2_WARP_DIMS(v, (k_warp_step_ls<real, WM, B2_WARP_LS_MODE><<<blocks, wpb * 32, smem, s>>>(
                      (const WarpImage<real>*)image, to_dev<real>(st), to_dev<real>(out), out != nullptr, N, nsteps, (real*)jscratch, (int*)counter,
                      perm, cost, to_dev<real>(park))));
  return (int)cudaGetLastError();
}
// FD linearisation on the warp engine: same scratch slots as the step plan (wpb warps per block)
int B2_FN(b2k_warp_linearize)(const void* image, const b2m_view* v, const b2_state* st, int N, double eps, int centered, void* A, void* B,
                              void* jscratch, void* counter, int wpb, int blocks, void* stream) {
  const size_t smem = warp_block_smem(v, wpb, 2 * (v->nq + v->nv));
  int per_sm = 0, dev = 0, sms = 0, rc = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  B2_WARP_DIMS(v, (rc = warp_occupancy(k_warp_linearize<real, WM, B2_WARP_LS_MODE>, wpb, smem, &per_sm)));
  if (rc) return (int)cudaErrorLaunchOutOfResources;
  if (blocks > sms * per_sm) blocks = sms * per_sm;  // persistent: never more blocks than fit at once (scratch slots are per block)
  cudaError_t e = cudaMemsetAsync(counter, 0, sizeof(int), (cudaStream_t)stream);
  if (e != cudaSuccess) return (int)e;
  B2_WARP_DIMS(v, (k_warp_linearize<real, WM, B2_WARP_LS_MODE><<<blocks, wpb * 32, smem, (cudaStream_t)stream>>>(
                      (const WarpImage<real>*)image, to_dev<real>(st), N, (real)eps, centered, (real*)A, (real*)B, (real*)jscratch, (int*)counter)));
  return (int)cudaGetLastError();
}
int B2_FN(b2k_linearize)(const void* image, int cls, const b2_state* st, int count, int N, int ncol, double eps, int centered, void* A, void* B,
                         const void* gain, const b2_state* shadow, void* stream) {
  const int threads = 128;
  const long long total = (long long)count * ncol;  // ncol: FD tasks per env (b2_capi: nv + 1 under Euler, else 2nv + nu)
  const int blocks = (int)((total + threads - 1) / threads);
  B2_DISPATCH(cls, (k_linearize<real, DD, RuntimeModel<DD>><<<blocks, threads, 0, (cudaStream_t)stream>>>(
                       to_dev<real>(st), count, N, (real)eps, centered, (real*)A, (real*)B, (const real*)gain, to_dev<real>(shadow), image)));
  return (int)cudaGetLastError();
}
// (A, B) and the sensor Jacobians from the same rollouts (k_linearize<..., SENS = true>); no control law, no env advance
int B2_FN(b2k_linearize_sensors)(const void* image, int cls, const b2_state* st, int count, int N, int ncol, double eps, int centered, void* A,
                                 void* B, void* dsdx, void* dsdu, void* stream) {
  const int threads = 128;
  const long long total = (long long)count * ncol;
  const int blocks = (int)((total + threads - 1) / threads);
  const b2_state* no_shadow = nullptr;
  B2_DISPATCH(cls, (k_linearize<real, DD, RuntimeModel<DD>, 0, true><<<blocks, threads, 0, (cudaStream_t)stream>>>(
                       to_dev<real>(st), count, N, (real)eps, centered, (real*)A, (real*)B, nullptr, to_dev<real>(no_shadow), image,
                       (real*)dsdx, (real*)dsdu)));
  return (int)cudaGetLastError();
}
int B2_FN(b2k_commit_state)(const b2_state* st, const b2_state* shadow, int count, int N, int nq, int nv, int nu, void* stream) {
  int bx = (count + 255) / 256;
  if (bx > 148 * 8) bx = 148 * 8;
  k_commit_state<real><<<dim3(bx, nq + 2 * nv + nu), 256, 0, (cudaStream_t)stream>>>(to_dev<real>(st), to_dev<real>(shadow), count, N, nq, nv, nu);
  return (int)cudaGetLastError();
}
int B2_FN(b2k_jacobian)(const void* image, int cls, const b2_state* st, int N, int kind, int objid, void* jacp, void* jacr, void* stream) {
  const int threads = 128, blocks = (N + threads - 1) / threads;
  B2_DISPATCH(cls, (k_jacobian<real, DD, RuntimeModel<DD>><<<blocks, threads, 0, (cudaStream_t)stream>>>(
                       to_dev<real>(st), N, kind, objid, (real*)jacp, (real*)jacr, image)));
  return (int)cudaGetLastError();
}
int B2_FN(b2k_inverse)(const void* image, int cls, const b2_state* st, int N, const void* qacc, void* qfrc, void* moment, void* stream) {
  const int threads = 128, blocks = (N + threads - 1) / threads;
  B2_DISPATCH(cls, (k_inverse<real, DD, RuntimeModel<DD>><<<blocks, threads, 0, (cudaStream_t)stream>>>(
                       to_dev<real>(st), N, (const real*)qacc, (real*)qfrc, (real*)moment, image)));
  return (int)cudaGetLastError();
}
int B2_FN(b2k_lqr_control)(const void* image, int cls, const b2_state* st, int count, int N, const void* gain, void* stream) {
  const int threads = 128, blocks = (count + threads - 1) / threads;
  B2_DISPATCH(cls, (k_lqr_control<real, DD, RuntimeModel<DD>><<<blocks, threads, 0, (cudaStream_t)stream>>>(
                       to_dev<real>(st), count, N, (const real*)gain, image)));
  return (int)cudaGetLastError();
}
// batched DARE / LQR gains: one warp per env, as many warps per block as the shared-memory workspace allows (at most four)
int B2_FN(b2k_dare)(const void* A, const void* B, const void* qr /* device: Q, R, Rinv */, int nx, int nu, int N, int max_doublings,
                    double tol, void* K, void* P, int* status, void* stream) {
  const real* qd = (const real*)qr;
  // small systems: one env per thread, compile-time sizes (B2_DARE_WARP=1 forces the warp kernel)
  const char* force_warp = getenv("B2_DARE_WARP");
  if (!(force_warp && force_warp[0] == '1')) {
#define B2_DARE_SMALL(NX_, NU_)                                                                                                   \
    if (nx == NX_ && nu == NU_) {                                                                                                 \
      k_dare_small<real, NX_, NU_><<<(N + 63) / 64, 64, 0, (cudaStream_t)stream>>>((const real*)A, (const real*)B, qd, qd + nx * nx, \
                                                                                  qd + nx * nx + nu * nu, N, max_doublings, (real)tol,   \
                                                                                  (real*)K, (real*)P, status);                     \
      return (int)cudaGetLastError();                                                                                             \
    }
    B2_DARE_SMALL(2, 1) B2_DARE_SMALL(4, 1) B2_DARE_SMALL(4, 2)
#undef B2_DARE_SMALL
  }
  int dev = 0, smem_max = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  const size_t per = dare_ws_reals(nx, nu) * sizeof(real);
  int wpb = (int)((size_t)smem_max / per);
  if (wpb < 1) return (int)cudaErrorInvalidValue;  // nx too large for one SM's shared memory
  if (wpb > 4) wpb = 4;
  cudaError_t e = cudaFuncSetAttribute(k_dare<real>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(per * wpb));
  if (e != cudaSuccess) return (int)e;
  const real* q = (const real*)qr;
  k_dare<real><<<(N + wpb - 1) / wpb, wpb * 32, per * wpb, (cudaStream_t)stream>>>(
      (const real*)A, (const real*)B, q, q + nx * nx, q + nx * nx + nu * nu, nx, nu, N, max_doublings, (real)tol, (real*)K, (real*)P, status);
  return (int)cudaGetLastError();
}
int B2_FN(b2k_lqr_control_env)(const void* image, int cls, const b2_state* st, int count, int N, const void* gain, const void* K_env, void* stream) {
  const int threads = 128, blocks = (count + threads - 1) / threads;
  B2_DISPATCH(cls, (k_lqr_control_env<real, DD, RuntimeModel<DD>><<<blocks, threads, 0, (cudaStream_t)stream>>>(
                       to_dev<real>(st), count, N, (const real*)gain, (const real*)K_env, image)));
  return (int)cudaGetLastError();
}
int B2_FN(b2k_random_controls)(const b2_state* st, int N, int nq, int nv, int nu, double lo, double hi, unsigned long long seed, void* ctr,
                               int watch_row, double watch_min, const void* reset_qpos, const void* reset_qvel, void* stream) {
  k_random_controls<real><<<(N + 255) / 256, 256, 0, (cudaStream_t)stream>>>(to_dev<real>(st), N, nq, nv, nu, (real)lo, (real)hi, seed,
                                                                             (unsigned*)ctr, watch_row, (real)watch_min,
                                                                             (const real*)reset_qpos, (const real*)reset_qvel);
  return (int)cudaGetLastError();
}
int B2_FN(b2k_record_rows)(const void* cols, int ncol, const int* env_index, int nsel, int N, double time, void* out, void* stream) {
  const int threads = 128;
  k_record_rows<real><<<dim3((nsel + threads - 1) / threads, ncol), threads, 0, (cudaStream_t)stream>>>(
      (const RecordColDev*)cols, env_index, nsel, N, (real)time, (real*)out);
  return (int)cudaGetLastError();
}
int B2_FN(b2k_integrate_pos)(const void* image, int cls, void* qpos, const void* qvel, double dt, int N, void* stream) {
  const int threads = 128, blocks = (N + threads - 1) / threads;
  B2_DISPATCH(cls, (k_integrate_pos<real, DD, RuntimeModel<DD>><<<blocks, threads, 0, (cudaStream_t)stream>>>(
                       (real*)qpos, (const real*)qvel, (real)dt, N, image)));
  return (int)cudaGetLastError();
}
int B2_FN(b2k_differentiate_pos)(const void* image, int cls, void* out, double dt, const void* q1, const void* q2, int N, void* stream) {
  const int threads = 128, blocks = (N + threads - 1) / threads;
  B2_DISPATCH(cls, (k_differentiate_pos<real, DD, RuntimeModel<DD>><<<blocks, threads, 0, (cudaStream_t)stream>>>(
                       (real*)out, (real)dt, (const real*)q1, (const real*)q2, N, image)));
  return (int)cudaGetLastError();
}

}  // namespace b2
