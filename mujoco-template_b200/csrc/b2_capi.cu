// C-ABI of the B200-native batched physics path (see include/b2mj.h for the contract and the
// reference call sites each entry point replaces).  Host-only logic: model bookkeeping,
// the models' device images, launches, and the host-buffer (e2e) variant.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "../../include/b2mj.h"
#include "b2_kernels.h"
#include "b2_model_dev.cuh"

namespace {
thread_local std::string g_err;
std::atomic<long long> g_launches{0};
std::atomic<unsigned long long> g_serial{1};

int fail(int code, const std::string& msg) { g_err = msg; return code; }
int cuda_fail(cudaError_t e, const char* what) {
  return fail(B2_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
// counts one launch; rc is the launcher's cudaError_t
int launched(int rc, const char* what) {
  g_launches++;
  return rc ? cuda_fail((cudaError_t)rc, what) : B2_OK;
}
const b2::Kernels* kernels(int precision) { return precision == B2_F64 ? &b2::kernels_f64 : &b2::kernels_f32; }
}  // namespace

struct b2_model {
  std::vector<unsigned char> blob;
  b2m_view v;
  std::vector<int> disabled;
  int cls;
  unsigned long long serial;
  const b2::SpecKernels* spec;  // model-specialised kernels, or nullptr (generic kernels)
  const b2::LaneKernels* lane[2];  // [0] FP64, [1] FP32: the lane-engine launchers of spec, or the generic ones
  // The model's images in device memory, per device and precision: [.][.][0] the lane engine's (DevModel of the model's
  // size class), [.][.][1] the warp engine's (constants + factorisation work lists).  Kernels get them by pointer, so
  // nothing about a model is process-wide device state: batches of different models are independent of each other on
  // any stream and thread, and a captured graph keeps the image it was captured with.
  mutable std::mutex image_mu;
  mutable void* image[16][2][2] = {};
  mutable unsigned long long image_serial[16][2][2] = {};
  mutable std::vector<std::pair<int, void*>> retired_images;  // (device, pointer) replaced after a disable-mask change
};

namespace b2 {
static std::vector<const SpecKernels*>& spec_table() {
  static std::vector<const SpecKernels*> t;
  return t;
}
void register_spec(const SpecKernels* k) { spec_table().push_back(k); }
const SpecKernels* find_spec(uint64_t hash, size_t size) {
  const char* off = getenv("B2_DISABLE_SPEC");
  if (off && off[0] == '1') return nullptr;
  for (const SpecKernels* k : spec_table())
    if (k->blob_hash == hash && k->blob_size == size) return k;
  return nullptr;
}
}  // namespace b2

static void set_spec(b2_model* m, const b2::SpecKernels* spec) {
  m->spec = spec;
  m->lane[0] = spec ? &spec->lane[0] : &b2::kernels_f64.generic;
  m->lane[1] = spec ? &spec->lane[1] : &b2::kernels_f32.generic;
}

struct HostStepKey {
  void *qpos, *qvel, *ctrl, *warm, *A, *B;
  int nsteps, linearize;
  double eps;
  unsigned long long model_serial;
};

struct b2_batch {
  const b2_model* model;
  int nenv, device, precision;
  int pi;  // 0 FP64, 1 FP32: index of the model's per-precision kernels and images
  const b2::Kernels* k;  // the generic kernels of this precision
  size_t esz;
  // device staging for b2_step_host
  void *d_qpos = nullptr, *d_qvel = nullptr, *d_ctrl = nullptr, *d_warm = nullptr, *d_A = nullptr, *d_B = nullptr;
  // warp engine (large models), decided in b2_batch_create
  bool warp = false;
  int warp_wpb = 0, warp_blocks = 0, warp_slots = 0;
  void* d_jscratch = nullptr;
  void* d_warp_counter = nullptr;  // inside d_jscratch
  void* d_warp_sort = nullptr;     // inside d_jscratch: cost-ordered queue (hist / cursor, cost[N], perm[N])
  void* d_shadow = nullptr;        // shadow state of the FD launch that also advances the envs (b2_control_tick)
  bool shadow_has_prestep = false;
  void* d_gain = nullptr;  // LQR gain block: K, qpos_ref, ctrl_ref
  void* d_rng_ctr = nullptr;  // b2_random_controls: draw counter per env
  cudaStream_t pipe[3] = {nullptr, nullptr, nullptr};  // copy/compute pipeline of b2_step_host
  cudaEvent_t pipe_ev[3] = {nullptr, nullptr, nullptr};
  bool pipe_ready = false;
  cudaGraphExec_t host_graph = nullptr;  // captured pipeline, valid for host_key
  HostStepKey host_key;
  int host_graph_launches = 0;
};

// The warp engine covers the feature set of large articulated models (humanoid); everything else
// in the large size class runs on the lane engine.
static bool warp_engine_supports(const b2m_view& v) {
  const char* off = getenv("B2_DISABLE_WARP");
  if (off && off[0] == '1') return false;
  if (v.integrator != 0 || v.has_fluid || v.nbody > 32 || v.nv > 32 || v.nsite != 0 || v.nsensor != 0) return false;
  for (int a = 0; a < v.nu; a++) if (v.actuator_trntype[a] != b2::TRN_JOINT) return false;
  for (int g = 0; g < v.ngeom; g++) {
    const int t = v.geom_type[g];
    if (t != b2::GEOM_PLANE && t != b2::GEOM_SPHERE && t != b2::GEOM_CAPSULE) {
      bool collides = false;
      for (int p = 0; p < v.npair; p++) collides = collides || v.pair_geom1[p] == g || v.pair_geom2[p] == g;
      if (collides) return false;
    }
  }
  return true;
}

// decide whether the batch runs on the large-model warp engine; plan its launch and scratch
static int prepare_warp(b2_batch* b) {
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
  if (b->model->cls != 2 || !warp_engine_supports(b->model->v)) return B2_OK;
  int wpb = 0, blocks = 0;
  const int slots = b->k->warp_plan(&b->model->v, b->nenv, &wpb, &blocks);
  if (slots <= 0) return B2_OK;  // not enough shared memory: stay on the lane engine
  const size_t bytes = b->k->warp_scratch_bytes(&b->model->v, slots);
  // + the work-queue counter of the persistent kernel + the buffers of the cost-ordered queue
  const size_t sort_bytes = b->k->warp_sort_bytes(b->nenv);
  e = cudaMalloc(&b->d_jscratch, bytes + 256 + sort_bytes);
  if (e != cudaSuccess) return cuda_fail(e, "warp-engine scratch cudaMalloc");
  b->d_warp_counter = (char*)b->d_jscratch + bytes;
  b->d_warp_sort = (char*)b->d_warp_counter + 256;
  if ((e = cudaMemset(b->d_warp_sort, 0, sort_bytes)) != cudaSuccess) return cuda_fail(e, "warp-engine queue cudaMemset");
  b->warp = true; b->warp_wpb = wpb; b->warp_blocks = blocks; b->warp_slots = slots;
  return B2_OK;
}
// The model's image for this batch's device and precision (kind 0: lane engine, 1: warp engine): uploaded on first use
// (b2_batch_create does that for the kinds the batch will launch) and again after a disable-mask change.
static int image_of(b2_batch* b, int kind, const void** out) {
  const b2_model* m = b->model;
  const int pi = b->pi, dev = b->device;
  std::lock_guard<std::mutex> lock(m->image_mu);
  if (!m->image[dev][pi][kind] || m->image_serial[dev][pi][kind] != m->serial) {
    const size_t bytes = kind == 1 ? b->k->warp_image_bytes() : b->k->image_bytes(m->cls);
    std::vector<unsigned char> host(bytes);
    if (kind == 1) b->k->warp_image_fill(&m->v, m->disabled.data(), host.data());
    else b->k->image_fill(m->cls, &m->v, m->disabled.data(), host.data());
    void* d = nullptr;
    cudaError_t e = cudaMalloc(&d, bytes);
    if (e != cudaSuccess) return cuda_fail(e, "model image cudaMalloc");
    if ((e = cudaMemcpy(d, host.data(), bytes, cudaMemcpyHostToDevice)) != cudaSuccess) { cudaFree(d); return cuda_fail(e, "model image upload"); }
    if (m->image[dev][pi][kind]) m->retired_images.emplace_back(dev, m->image[dev][pi][kind]);  // kernels in flight may still read it
    m->image[dev][pi][kind] = d;
    m->image_serial[dev][pi][kind] = m->serial;
  }
  *out = m->image[dev][pi][kind];
  return B2_OK;
}
// Every launch starts here: selects the batch's device and hands out its model's current lane-engine image and, when the
// batch runs on the warp engine and `warp` is given, its warp-engine image.
static int batch_images(b2_batch* b, const void** lane, const void** warp = nullptr) {
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
  int rc = image_of(b, 0, lane);
  if (!rc && warp && b->warp) rc = image_of(b, 1, warp);
  return rc;
}
// the warp engine takes the launches it supports, unless the model has specialised kernels
static bool on_warp_engine(const b2_batch* b) { return b->warp && !b->model->spec; }

#define B2_CHECK_STATE(fn)                                                                         \
  if (!b || !st || !st->qpos || !st->qvel || (b->model->v.nu && !st->ctrl)) return fail(B2_ERR_ARG, fn ": null batch/state pointer")

extern "C" {

const char* b2_last_error(void) { return g_err.c_str(); }
const char* b2_version(void) { return "b2mj 0.1 (sm_100a lane engine)"; }
long long b2_launch_count(void) { return g_launches.load(); }

int b2_model_create(const void* blob, size_t nbytes, b2_model** out) {
  if (!blob || !out) return fail(B2_ERR_ARG, "b2_model_create: null argument");
  b2_model* m = new (std::nothrow) b2_model();
  if (!m) return fail(B2_ERR_ARG, "out of host memory");
  m->blob.assign((const unsigned char*)blob, (const unsigned char*)blob + nbytes);
  int rc = b2m_view_init(&m->v, m->blob.data(), nbytes);
  if (rc) { delete m; return fail(B2_ERR_BLOB, "b2_model_create: malformed model blob (code " + std::to_string(rc) + ")"); }
  const b2m_view& v = m->v;
  if (b2::model_fits<b2::DimsTiny>(v)) m->cls = 0;
  else if (b2::model_fits<b2::DimsSmall>(v)) m->cls = 1;
  else if (b2::model_fits<b2::DimsLarge>(v)) m->cls = 2;
  else { delete m; return fail(B2_ERR_CAPACITY, "b2_model_create: model exceeds the largest compiled size class"); }
  m->disabled.assign(v.actuator_disabled, v.actuator_disabled + v.nu);
  m->serial = g_serial.fetch_add(1);
  set_spec(m, b2::find_spec(b2::fnv1a(blob, nbytes), nbytes));
  *out = m;
  return B2_OK;
}
void b2_model_destroy(b2_model* m) {
  if (!m) return;
  int cur = 0;
  cudaGetDevice(&cur);
  for (int d = 0; d < 16; d++)
    for (int p = 0; p < 2; p++)
      for (int k = 0; k < 2; k++)
        if (m->image[d][p][k]) { cudaSetDevice(d); cudaFree(m->image[d][p][k]); }
  for (auto& r : m->retired_images) { cudaSetDevice(r.first); cudaFree(r.second); }
  cudaSetDevice(cur);
  delete m;
}

int b2_model_set_actuator_disabled(b2_model* m, const int* disabled, int nu) {
  if (!m || (nu && !disabled) || nu != m->v.nu) return fail(B2_ERR_ARG, "b2_model_set_actuator_disabled: bad arguments");
  // an unchanged mask keeps the images: launches never upload one then (an upload cannot run inside a graph capture)
  if (std::equal(disabled, disabled + nu, m->disabled.begin())) return B2_OK;
  m->disabled.assign(disabled, disabled + nu);
  m->serial = g_serial.fetch_add(1);  // the device images are rebuilt on their next use
  for (int i = 0; i < nu; i++)
    if (disabled[i] != m->v.actuator_disabled[i]) set_spec(m, nullptr);  // the specialisation bakes the mask in
  return B2_OK;
}

int b2_batch_create(const b2_model* model, int nenv, int device, int precision, b2_batch** out) {
  if (!model || !out || nenv < 1) return fail(B2_ERR_ARG, "b2_batch_create: bad arguments");
  if (precision != B2_F64 && precision != B2_F32) return fail(B2_ERR_ARG, "b2_batch_create: precision must be 64 or 32");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) return fail(B2_ERR_CUDA, "b2_batch_create: no CUDA device (this path has no CPU fallback)");
  if (device < 0 || device >= ndev || device >= 16) return fail(B2_ERR_ARG, "b2_batch_create: device index out of range");
  b2_batch* b = new (std::nothrow) b2_batch();
  if (!b) return fail(B2_ERR_ARG, "out of host memory");
  b->model = model; b->nenv = nenv; b->device = device; b->precision = precision;
  b->pi = precision == B2_F64 ? 0 : 1; b->k = kernels(precision); b->esz = precision == B2_F64 ? 8 : 4;
  // everything the step path needs on the device is set up here, so that b2_step / b2_linearize only launch: the model's
  // images (shared by all batches of the model on this device) and, for large models, the warp engine's plan and scratch
  const void *lane = nullptr, *warp = nullptr;
  int rc = prepare_warp(b);
  if (rc || (rc = batch_images(b, &lane, &warp))) { b2_batch_destroy(b); return rc; }
  *out = b;
  return B2_OK;
}
void b2_batch_destroy(b2_batch* b) {
  if (!b) return;
  void* p[] = {b->d_qpos, b->d_qvel, b->d_ctrl, b->d_warm, b->d_A, b->d_B, b->d_jscratch, b->d_gain, b->d_shadow, b->d_rng_ctr};
  for (void* q : p) if (q) cudaFree(q);
  if (b->host_graph) cudaGraphExecDestroy(b->host_graph);
  if (b->pipe_ready) { for (cudaStream_t st : b->pipe) cudaStreamDestroy(st); for (cudaEvent_t ev : b->pipe_ev) cudaEventDestroy(ev); }
  delete b;
}
int b2_batch_size_class(const b2_batch* b) { return b ? b->model->cls : -1; }
const char* b2_batch_kernel_variant(const b2_batch* b) {
  if (!b) return "";
  if (b->model->spec) return b->model->spec->name;
  return b->warp ? "generic-warp" : "generic";
}

static int do_lqr_control(b2_batch* b, const b2_state* st, int count, void* stream) {
  const void* lane = nullptr;
  int rc = batch_images(b, &lane);
  if (rc) return rc;
  return launched(b->k->lqr_control(lane, b->model->cls, st, count, b->nenv, b->d_gain, stream), "b2_lqr_control launch");
}

// count envs (a leading chunk of the arrays `st` points at; the env stride is always b->nenv)
static int do_step(b2_batch* b, const b2_state* st, int count, int nsteps, const b2_derived* derived, void* stream,
                   const void* gain = nullptr, const b2_state* park = nullptr) {
  const void *lane = nullptr, *warp = nullptr;
  int rc = batch_images(b, &lane, &warp);
  if (rc) return rc;
  const b2_model* m = b->model;
  if (on_warp_engine(b) && count == b->nenv) {
    // the warp engine has no in-kernel control law: separate launch
    if (gain && (rc = do_lqr_control(b, st, count, stream))) return rc;
    if (b->warp_wpb > 1 && nsteps > 0) g_launches += 2;  // the queue's histogram and scatter kernels
    rc = b->k->warp_step(warp, &m->v, st, derived, b->nenv, nsteps, b->d_jscratch, b->d_warp_counter, b->d_warp_sort, b->warp_wpb,
                         b->warp_blocks, park, stream);
  } else {
    rc = m->lane[b->pi]->step(lane, m->cls, st, derived, count, b->nenv, nsteps, gain, park, stream);
  }
  return launched(rc, "step launch");
}
// b2_rollout.  Lane engine (specialised or generic kernels): one k_rollout launch.  Warp engine: the contract's loop itself,
// one warp step per control row -- a humanoid step of a full batch takes milliseconds, so a launch per step costs nothing,
// and every step re-orders the warp engine's cost-ordered queue as b2_step does.
static int do_rollout(b2_batch* b, const b2_state* st, int nsteps, const void* ctrl_seq, void* qpos_traj, void* qvel_traj, void* sensor_traj,
                      const b2_derived* derived, void* stream) {
  const b2_model* m = b->model;
  const b2m_view& v = m->v;
  const void* lane = nullptr;
  int rc = batch_images(b, &lane);
  if (rc) return rc;
  if (on_warp_engine(b)) {  // the warp engine runs no model with sensors: sensor_traj is null here
    const size_t N = (size_t)b->nenv, es = b->esz, ctrl_bytes = v.nu * N * es, qpos_bytes = v.nq * N * es, qvel_bytes = v.nv * N * es;
    cudaStream_t s = (cudaStream_t)stream;
    for (int t = 0; t < nsteps; t++) {
      cudaError_t e = cudaSuccess;
      if (ctrl_seq && ctrl_bytes) e = cudaMemcpyAsync(st->ctrl, (const char*)ctrl_seq + t * ctrl_bytes, ctrl_bytes, cudaMemcpyDefault, s);
      if (e != cudaSuccess) return cuda_fail(e, "b2_rollout: control row copy");
      if ((rc = do_step(b, st, b->nenv, 1, t == nsteps - 1 ? derived : nullptr, stream))) return rc;
      if (qpos_traj) e = cudaMemcpyAsync((char*)qpos_traj + t * qpos_bytes, st->qpos, qpos_bytes, cudaMemcpyDefault, s);
      if (e == cudaSuccess && qvel_traj) e = cudaMemcpyAsync((char*)qvel_traj + t * qvel_bytes, st->qvel, qvel_bytes, cudaMemcpyDefault, s);
      if (e != cudaSuccess) return cuda_fail(e, "b2_rollout: trajectory row copy");
    }
    return B2_OK;
  }
  rc = m->lane[b->pi]->rollout(lane, m->cls, st, derived, b->nenv, nsteps, ctrl_seq, qpos_traj, qvel_traj, sensor_traj, stream);
  return launched(rc, "rollout launch");
}
// C / D (b2_linearize_sensors): the sensor Jacobians from the same rollouts; either one non-null selects the sensor variant
// of the FD kernel, which has no control law and no env advance
static int do_linearize(b2_batch* b, const b2_state* st, int count, double eps, int centered, void* A, void* B, void* stream,
                        const void* gain = nullptr, const b2_state* shadow = nullptr, void* C = nullptr, void* D = nullptr) {
  const bool sensors = C || D;
  const void *lane = nullptr, *warp = nullptr;
  int rc = batch_images(b, &lane, &warp);
  if (rc) return rc;
  const b2_model* m = b->model;
  // large models on the warp engine: one warp per (column, env) rollout pair (the warp engine runs no model with sensors)
  if (on_warp_engine(b) && count == b->nenv && !gain && !shadow && !sensors) {
    rc = b->k->warp_linearize(warp, &m->v, st, b->nenv, eps, centered, A, B, b->d_jscratch, b->d_warp_counter, b->warp_wpb, b->warp_blocks,
                              stream);
    return launched(rc, "warp linearize launch");
  }
  // FD tasks per env: see k_linearize (Euler: one thread per group of velocity / control columns + one per position column)
  const int ntask = b2::fd_task_count(m->v.integrator, m->v.nv, m->v.nu);
  const b2::LaneKernels* lk = m->lane[b->pi];
  rc = sensors ? lk->linearize_sensors(lane, m->cls, st, count, b->nenv, ntask, eps, centered, A, B, C, D, stream)
               : lk->linearize(lane, m->cls, st, count, b->nenv, ntask, eps, centered, A, B, gain, shadow, stream);
  return launched(rc, "linearize launch");
}
// b2_linearize_rollout.  Lane engine: the nominal rollout, then one FD launch over every (step, env).  Warp engine (no
// sensors): the contract's loop itself on the trajectory rows, which serve as the working state -- a humanoid FD launch
// takes milliseconds, so a launch pair per step costs nothing.  warm_traj is null exactly when the state has no warm start.
static int do_linearize_rollout(b2_batch* b, const b2_state* st, int nsteps, const void* ctrl_seq, double eps, int centered, void* A, void* B,
                                void* C, void* D, void* qpos_traj, void* qvel_traj, void* warm_traj, void* sensor_traj, void* stream) {
  const b2_model* m = b->model;
  const b2m_view& v = m->v;
  const void* lane = nullptr;
  int rc = batch_images(b, &lane);
  if (rc) return rc;
  if (on_warp_engine(b)) {
    const size_t N = (size_t)b->nenv, es = b->esz, ndx = 2 * (size_t)v.nv, qpos_bytes = v.nq * N * es, qvel_bytes = v.nv * N * es;
    const size_t ctrl_bytes = v.nu * N * es, A_bytes = ndx * ndx * N * es, B_bytes = ndx * v.nu * N * es;
    cudaStream_t s = (cudaStream_t)stream;
    // row t of the trajectories as a state, with the controls of step t (the warp kernels only read state.ctrl)
    auto row = [&](int t) {
      return b2_state{(char*)qpos_traj + t * qpos_bytes, (char*)qvel_traj + t * qvel_bytes,
                      ctrl_seq ? (char*)ctrl_seq + t * ctrl_bytes : st->ctrl, warm_traj ? (char*)warm_traj + t * qvel_bytes : nullptr, st->flags};
    };
    auto copy_row = [&](const b2_state& dst, const b2_state& src) {
      cudaError_t e = cudaMemcpyAsync(dst.qpos, src.qpos, qpos_bytes, cudaMemcpyDefault, s);
      if (e == cudaSuccess) e = cudaMemcpyAsync(dst.qvel, src.qvel, qvel_bytes, cudaMemcpyDefault, s);
      if (e == cudaSuccess && warm_traj) e = cudaMemcpyAsync(dst.qacc_warmstart, src.qacc_warmstart, qvel_bytes, cudaMemcpyDefault, s);
      return e == cudaSuccess ? B2_OK : cuda_fail(e, "b2_linearize_rollout: trajectory row copy");
    };
    if ((rc = copy_row(row(0), *st))) return rc;
    for (int t = 0; t < nsteps; t++) {
      const b2_state x = row(t);
      if ((A || B) && (rc = do_linearize(b, &x, b->nenv, eps, centered, A ? (char*)A + t * A_bytes : nullptr, B ? (char*)B + t * B_bytes : nullptr, stream)))
        return rc;
      b2_state next = row(t + 1);
      next.ctrl = x.ctrl;
      if ((rc = copy_row(next, x)) || (rc = do_step(b, &next, b->nenv, 1, nullptr, stream))) return rc;
    }
    return B2_OK;
  }
  const int ntask = b2::fd_task_count(v.integrator, v.nv, v.nu);
  rc = m->lane[b->pi]->linearize_rollout(lane, m->cls, st, b->nenv, ntask, nsteps, ctrl_seq, eps, centered, A, B, C, D, qpos_traj, qvel_traj,
                                         warm_traj, sensor_traj, stream);
  if (A || B || C || D) g_launches++;  // the FD launch
  return launched(rc, "linearize_rollout launch");
}
// b2_rollout_feedback.  Lane engine: one k_rollout_feedback launch.  Warp engine: the contract's loop itself, as do_rollout
// runs it, with a law launch (which also records the control row) in front of every warp step.
static int do_rollout_feedback(b2_batch* b, const b2_state* st, int nsteps, const void* ctrl_nom, const void* qpos_nom, const void* qvel_nom,
                               const void* K, const void* k, const void* alpha, void* ctrl_traj, void* qpos_traj, void* qvel_traj,
                               void* sensor_traj, const b2_derived* derived, void* stream) {
  const b2_model* m = b->model;
  const b2m_view& v = m->v;
  const void* lane = nullptr;
  int rc = batch_images(b, &lane);
  if (rc) return rc;
  if (on_warp_engine(b)) {  // no sensors on the warp engine
    const size_t N = (size_t)b->nenv, es = b->esz, ctrl_bytes = v.nu * N * es, qpos_bytes = v.nq * N * es, qvel_bytes = v.nv * N * es;
    const size_t K_bytes = ctrl_bytes * 2 * v.nv;
    cudaStream_t s = (cudaStream_t)stream;
    for (int t = 0; t < nsteps; t++) {
      rc = b->k->tvlqr_law(lane, m->cls, st, b->nenv, (const char*)ctrl_nom + t * ctrl_bytes, (const char*)qpos_nom + t * qpos_bytes,
                           (const char*)qvel_nom + t * qvel_bytes, (const char*)K + t * K_bytes, k ? (const char*)k + t * ctrl_bytes : nullptr,
                           alpha, ctrl_traj ? (char*)ctrl_traj + t * ctrl_bytes : nullptr, stream);
      if ((rc = launched(rc, "b2_rollout_feedback: law launch"))) return rc;
      if ((rc = do_step(b, st, b->nenv, 1, t == nsteps - 1 ? derived : nullptr, stream))) return rc;
      cudaError_t e = cudaSuccess;
      if (qpos_traj) e = cudaMemcpyAsync((char*)qpos_traj + t * qpos_bytes, st->qpos, qpos_bytes, cudaMemcpyDefault, s);
      if (e == cudaSuccess && qvel_traj) e = cudaMemcpyAsync((char*)qvel_traj + t * qvel_bytes, st->qvel, qvel_bytes, cudaMemcpyDefault, s);
      if (e != cudaSuccess) return cuda_fail(e, "b2_rollout_feedback: trajectory row copy");
    }
    return B2_OK;
  }
  rc = m->lane[b->pi]->rollout_feedback(lane, m->cls, st, derived, b->nenv, nsteps, ctrl_nom, qpos_nom, qvel_nom, K, k, alpha, ctrl_traj,
                                        qpos_traj, qvel_traj, sensor_traj, stream);
  return launched(rc, "rollout_feedback launch");
}

int b2_step(b2_batch* b, const b2_state* st, int nsteps, const b2_derived* derived, void* stream) {
  B2_CHECK_STATE("b2_step");
  if (nsteps < 1) return fail(B2_ERR_ARG, "b2_step: nsteps must be >= 1");
  return do_step(b, st, b->nenv, nsteps, derived, stream);
}

int b2_rollout(b2_batch* b, const b2_state* st, int nsteps, const void* ctrl_seq, void* qpos_traj, void* qvel_traj, void* sensor_traj,
               const b2_derived* derived, void* stream) {
  B2_CHECK_STATE("b2_rollout");
  if (nsteps < 1) return fail(B2_ERR_ARG, "b2_rollout: nsteps must be >= 1");
  const b2m_view& v = b->model->v;
  return do_rollout(b, st, nsteps, v.nu ? ctrl_seq : nullptr, qpos_traj, qvel_traj, v.nsensordata ? sensor_traj : nullptr, derived, stream);
}

int b2_forward(b2_batch* b, const b2_state* st, const b2_derived* derived, void* stream) {
  B2_CHECK_STATE("b2_forward");
  return do_step(b, st, b->nenv, 0, derived, stream);
}

int b2_linearize(b2_batch* b, const b2_state* st, double eps, int centered, void* A, void* B, void* stream) {
  B2_CHECK_STATE("b2_linearize");
  if (!(eps > 0)) return fail(B2_ERR_LINEARIZE, "b2_linearize: eps must be > 0");
  if (!A && !B) return fail(B2_ERR_ARG, "b2_linearize: A and B are both NULL");
  return do_linearize(b, st, b->nenv, eps, centered, A, B, stream);
}

int b2_linearize_sensors(b2_batch* b, const b2_state* st, double eps, int centered, void* A, void* B, void* C, void* D, void* stream) {
  B2_CHECK_STATE("b2_linearize_sensors");
  if (!(eps > 0)) return fail(B2_ERR_LINEARIZE, "b2_linearize_sensors: eps must be > 0");
  if (!A && !B && !C && !D) return fail(B2_ERR_ARG, "b2_linearize_sensors: A, B, C and D are all NULL");
  const b2m_view& v = b->model->v;
  // without sensors (or without C / D to fill) this is b2_linearize; the warp engine only runs models without sensors
  if (v.nsensordata == 0 || (!C && !D)) return (A || B) ? do_linearize(b, st, b->nenv, eps, centered, A, B, stream) : B2_OK;
  if (!b->model->lane[b->pi]->linearize_sensors) return fail(B2_ERR_ARG, "b2_linearize_sensors: specialised kernel set has no sensor variant");
  return do_linearize(b, st, b->nenv, eps, centered, A, B, stream, nullptr, nullptr, C, D);
}

int b2_linearize_rollout(b2_batch* b, const b2_state* st, int nsteps, const void* ctrl_seq, double eps, int centered, void* A, void* B, void* C,
                         void* D, void* qpos_traj, void* qvel_traj, void* warm_traj, void* sensor_traj, void* stream) {
  if (nsteps < 1) return fail(B2_ERR_ARG, "b2_linearize_rollout: nsteps must be >= 1");
  if (!qpos_traj || !qvel_traj) return fail(B2_ERR_ARG, "b2_linearize_rollout: qpos_traj and qvel_traj are required");
  if (st && st->qacc_warmstart && !warm_traj) return fail(B2_ERR_ARG, "b2_linearize_rollout: warm_traj is required with a warm start");
  if (!A && !B && !C && !D) return fail(B2_ERR_ARG, "b2_linearize_rollout: A, B, C and D are all NULL");
  if (!(eps > 0)) return fail(B2_ERR_LINEARIZE, "b2_linearize_rollout: eps must be > 0");
  B2_CHECK_STATE("b2_linearize_rollout");
  const b2m_view& v = b->model->v;
  const bool sens = v.nsensordata != 0;
  return do_linearize_rollout(b, st, nsteps, v.nu ? ctrl_seq : nullptr, eps, centered, A, B, sens ? C : nullptr, sens ? D : nullptr,
                              qpos_traj, qvel_traj, st->qacc_warmstart ? warm_traj : nullptr, sens ? sensor_traj : nullptr, stream);
}

int b2_rollout_feedback(b2_batch* b, const b2_state* st, int nsteps, const void* ctrl_nom, const void* qpos_nom, const void* qvel_nom,
                        const void* K, const void* k, const void* alpha, void* ctrl_traj, void* qpos_traj, void* qvel_traj, void* sensor_traj,
                        const b2_derived* derived, void* stream) {
  if (nsteps < 1) return fail(B2_ERR_ARG, "b2_rollout_feedback: nsteps must be >= 1");
  if (!ctrl_nom || !qpos_nom || !qvel_nom || !K) return fail(B2_ERR_ARG, "b2_rollout_feedback: ctrl_nom, qpos_nom, qvel_nom and K are required");
  B2_CHECK_STATE("b2_rollout_feedback");
  const b2m_view& v = b->model->v;
  if (v.nu == 0) return fail(B2_ERR_ARG, "b2_rollout_feedback: the model has no actuators");
  return do_rollout_feedback(b, st, nsteps, ctrl_nom, qpos_nom, qvel_nom, K, k, alpha, ctrl_traj, qpos_traj, qvel_traj,
                             v.nsensordata ? sensor_traj : nullptr, derived, stream);
}

int b2_jacobian(b2_batch* b, const b2_state* st, int kind, int objid, void* jacp, void* jacr, void* stream) {
  if (!b || !st || !st->qpos) return fail(B2_ERR_ARG, "b2_jacobian: null batch/state pointer");
  const b2m_view& v = b->model->v;
  const int limit = kind == B2_JAC_SITE ? v.nsite : v.nbody;
  if (kind < B2_JAC_SITE || kind > B2_JAC_SUBTREECOM || objid < 0 || objid >= limit)
    return fail(B2_ERR_ARG, "b2_jacobian: kind/objid out of range");
  const void* lane = nullptr;
  int rc = batch_images(b, &lane);
  if (rc) return rc;
  rc = b->model->lane[b->pi]->jacobian(lane, b->model->cls, st, b->nenv, kind, objid, jacp, jacr, stream);
  return launched(rc, "b2_jacobian launch");
}

int b2_inverse(b2_batch* b, const b2_state* st, const void* qacc, void* qfrc_inverse, void* actuator_moment, void* stream) {
  B2_CHECK_STATE("b2_inverse");
  if (!qfrc_inverse) return fail(B2_ERR_ARG, "b2_inverse: qfrc_inverse is NULL");
  const void* lane = nullptr;
  int rc = batch_images(b, &lane);  // one-shot setup call: always the generic kernels
  if (rc) return rc;
  return launched(b->k->inverse(lane, b->model->cls, st, b->nenv, qacc, qfrc_inverse, actuator_moment, stream), "b2_inverse launch");
}

int b2_lqr_set_gain(b2_batch* b, const double* K, const double* qpos_ref, const double* ctrl_ref) {
  if (!b || !K || !qpos_ref || !ctrl_ref) return fail(B2_ERR_ARG, "b2_lqr_set_gain: null pointer");
  const b2m_view& v = b->model->v;
  if (v.nu == 0) return fail(B2_ERR_ARG, "b2_lqr_set_gain: model has no actuators");
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
  const size_t n = (size_t)v.nu * 2 * v.nv + v.nq + v.nu;
  std::vector<unsigned char> host(n * b->esz);
  for (size_t i = 0; i < n; i++) {
    const double x = i < (size_t)v.nu * 2 * v.nv ? K[i] : (i < (size_t)v.nu * 2 * v.nv + v.nq ? qpos_ref[i - (size_t)v.nu * 2 * v.nv] : ctrl_ref[i - (size_t)v.nu * 2 * v.nv - v.nq]);
    if (b->precision == B2_F64) ((double*)host.data())[i] = x; else ((float*)host.data())[i] = (float)x;
  }
  if (!b->d_gain && (e = cudaMalloc(&b->d_gain, n * b->esz))) return cuda_fail(e, "b2_lqr_set_gain: cudaMalloc");
  if ((e = cudaMemcpy(b->d_gain, host.data(), n * b->esz, cudaMemcpyHostToDevice))) return cuda_fail(e, "b2_lqr_set_gain: copy");
  return B2_OK;
}

int b2_lqr_control(b2_batch* b, const b2_state* st, void* stream) {
  B2_CHECK_STATE("b2_lqr_control");
  if (!b->d_gain) return fail(B2_ERR_ARG, "b2_lqr_control: call b2_lqr_set_gain first");
  return do_lqr_control(b, st, b->nenv, stream);
}

// Shadow state arrays of a batch (same shapes as the caller's): target of the env advance that rides in the FD launch.
static int shadow_state(b2_batch* b, b2_state* out) {
  const b2m_view& v = b->model->v;
  const size_t N = (size_t)b->nenv, es = b->esz, nu1 = v.nu ? v.nu : 1;
  if (!b->d_shadow) {
    cudaError_t e = cudaSetDevice(b->device);
    if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
    e = cudaMalloc(&b->d_shadow, (v.nq + 2 * (size_t)v.nv + nu1) * N * es);
    if (e != cudaSuccess) return cuda_fail(e, "shadow state cudaMalloc");
  }
  char* p = (char*)b->d_shadow;
  *out = b2_state{p, p + v.nq * N * es, p + (v.nq + v.nv) * N * es, p + (v.nq + v.nv + nu1) * N * es, nullptr};
  return B2_OK;
}

// One control tick: [LQR law] -> (A, B) at the new controls -> one step (reference env.py:177-191 order).  The kernels
// evaluate the control law themselves (no controller launch).
//  * derived == NULL and an Euler model: ONE physics launch.  The FD thread that owns an env's velocity / control columns
//    has already run the position stage of the nominal state, so it also does the step (one more rollout instead of a
//    k_step launch that cannot fill the GPU at this batch size) and writes the new state to the batch's shadow arrays;
//    k_commit_state then swaps state and shadow.  The pre-step state stays in the shadow, so b2_refresh_derived can
//    still produce the derived arrays of this tick on demand.
//  * otherwise: FD kernel, then step kernel (which exports the derived arrays).
int b2_control_tick(b2_batch* b, const b2_state* st, const b2_derived* derived, int use_lqr, double eps, int centered,
                    void* A, void* B, void* stream) {
  B2_CHECK_STATE("b2_control_tick");
  if (!(eps > 0)) return fail(B2_ERR_LINEARIZE, "b2_control_tick: eps must be > 0");
  if (!A && !B) return fail(B2_ERR_ARG, "b2_control_tick: A and B are both NULL");
  if (use_lqr && !b->d_gain) return fail(B2_ERR_ARG, "b2_control_tick: call b2_lqr_set_gain first");
  const void* gain = use_lqr ? b->d_gain : nullptr;
  const b2m_view& v = b->model->v;
  b->shadow_has_prestep = false;
  if (on_warp_engine(b)) {
    // large models: control-law launch, FD on the warp engine, step on the warp engine.  Without a `derived`
    // argument the pre-step state is parked in the shadow arrays for b2_refresh_derived, as in the fused form.
    int rc;
    if (gain && (rc = do_lqr_control(b, st, b->nenv, stream))) return rc;
    if ((rc = do_linearize(b, st, b->nenv, eps, centered, A, B, stream))) return rc;
    if (!derived && st->qacc_warmstart) {  // the step kernel parks the pre-step state itself
      b2_state shadow;
      if ((rc = shadow_state(b, &shadow)) || (rc = do_step(b, st, b->nenv, 1, nullptr, stream, nullptr, &shadow))) return rc;
      b->shadow_has_prestep = true;
      return B2_OK;
    }
    return do_step(b, st, b->nenv, 1, derived, stream);
  }
  if (!derived && v.integrator == 0 && st->qacc_warmstart && (v.nu == 0 || st->ctrl)) {
    b2_state shadow;
    int rc = shadow_state(b, &shadow);
    if (rc) return rc;
    if ((rc = do_linearize(b, st, b->nenv, eps, centered, A, B, stream, gain, &shadow))) return rc;
    if ((rc = launched(b->k->commit_state(st, &shadow, b->nenv, b->nenv, v.nq, v.nv, v.nu, stream), "commit launch"))) return rc;
    b->shadow_has_prestep = true;
    return B2_OK;
  }
  int rc = do_linearize(b, st, b->nenv, eps, centered, A, B, stream, gain);
  if (rc) return rc;
  return do_step(b, st, b->nenv, 1, derived, stream, gain);
}

int b2_step_lazy(b2_batch* b, const b2_state* st, void* stream) {
  B2_CHECK_STATE("b2_step_lazy");
  if (!st->qacc_warmstart) return fail(B2_ERR_ARG, "b2_step_lazy: state.qacc_warmstart is required");
  int rc;
  // the step kernel (lane or warp engine) has the pre-step state at hand and writes it to the shadow arrays itself
  b2_state shadow;
  if ((rc = shadow_state(b, &shadow))) return rc;
  if ((rc = do_step(b, st, b->nenv, 1, nullptr, stream, nullptr, &shadow))) return rc;
  b->shadow_has_prestep = true;
  return B2_OK;
}

// Derived arrays (xpos, ..., sensordata) of the last b2_control_tick that ran without a `derived` argument: what mj_step
// leaves in mjData after that step, i.e. the forward pass of the PRE-step state, which the tick kept in its shadow arrays.
int b2_refresh_derived(b2_batch* b, const b2_derived* derived, void* stream) {
  if (!b || !derived) return fail(B2_ERR_ARG, "b2_refresh_derived: null pointer");
  if (!b->shadow_has_prestep) return fail(B2_ERR_ARG, "b2_refresh_derived: no control tick without derived outputs to refresh");
  b2_state shadow;
  int rc = shadow_state(b, &shadow);
  if (rc) return rc;
  return do_step(b, &shadow, b->nenv, 0, derived, stream);
}

int b2_integrate_pos(b2_batch* b, void* qpos, const void* qvel, double dt, void* stream) {
  if (!b || !qpos || !qvel) return fail(B2_ERR_ARG, "b2_integrate_pos: null pointer");
  const void* lane = nullptr;
  int rc = batch_images(b, &lane);
  if (rc) return rc;
  return launched(b->k->integrate_pos(lane, b->model->cls, qpos, qvel, dt, b->nenv, stream), "b2_integrate_pos launch");
}

int b2_differentiate_pos(b2_batch* b, void* out, double dt, const void* q1, const void* q2, void* stream) {
  if (!b || !out || !q1 || !q2) return fail(B2_ERR_ARG, "b2_differentiate_pos: null pointer");
  if (dt == 0) return fail(B2_ERR_ARG, "b2_differentiate_pos: dt must be nonzero");
  const void* lane = nullptr;
  int rc = batch_images(b, &lane);
  if (rc) return rc;
  return launched(b->k->differentiate_pos(lane, b->model->cls, out, dt, q1, q2, b->nenv, stream), "b2_differentiate_pos launch");
}

// Host-buffer step.  The env range is cut into chunks that flow through a small pool of streams:
// H2D of chunk c+1 and D2H of chunk c-1 overlap the kernels of chunk c (both copy engines busy).
int b2_step_host(b2_batch* b, const b2_state* hs, int nsteps, int linearize, double eps, void* host_A, void* host_B, void* stream) {
  if (!b || !hs || !hs->qpos || !hs->qvel || (b->model->v.nu && !hs->ctrl)) return fail(B2_ERR_ARG, "b2_step_host: null pointer");
  if (nsteps < 1) return fail(B2_ERR_ARG, "b2_step_host: nsteps must be >= 1");
  const bool lqr = (linearize & B2_HOST_LQR) != 0;  // ctrl is produced on the device by the b2_lqr_set_gain law and copied back
  const bool async = (linearize & B2_HOST_ASYNC) != 0;  // return once the pipeline is queued; b2_step_host_wait completes it
  linearize &= B2_HOST_LINEARIZE;
  if (lqr && !b->d_gain) return fail(B2_ERR_ARG, "b2_step_host: B2_HOST_LQR needs b2_lqr_set_gain first");
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
  const b2m_view& v = b->model->v;
  const size_t N = (size_t)b->nenv, es = b->esz, nx = 2 * (size_t)v.nv, nu1 = v.nu ? v.nu : 1;
  auto need = [&](void** p, size_t bytes) -> cudaError_t { return *p ? cudaSuccess : cudaMalloc(p, bytes); };
  if ((e = need(&b->d_qpos, v.nq * N * es)) || (e = need(&b->d_qvel, v.nv * N * es)) || (e = need(&b->d_ctrl, nu1 * N * es)) ||
      (e = need(&b->d_warm, v.nv * N * es)))
    return cuda_fail(e, "b2_step_host: cudaMalloc");
  // (A, B) are 8 (2nv)(2nv + nu) bytes per env against 8 (nq + 2nv) of state -- 89 % of the bytes that go back to the host for
  // the cartpole.  When the caller's buffers are page-locked and mapped into this device's address space (cudaHostAlloc /
  // cudaHostRegister under unified addressing: torch's pin_memory()), the FD kernel stores its columns straight into them --
  // coalesced 256 B rows over PCIe while the kernel is still computing -- instead of staging them in HBM and copying
  // afterwards.  B2_HOST_STAGED=1 keeps the staged form.
  void *map_A = nullptr, *map_B = nullptr;
  bool direct = linearize && host_A && (host_B || !v.nu);
  if (const char* x = getenv("B2_HOST_STAGED")) if (x[0] == '1') direct = false;
  if (direct) {
    auto mapped = [&](void* host, void** dev) {
      cudaPointerAttributes at;
      if (cudaPointerGetAttributes(&at, host) != cudaSuccess) { cudaGetLastError(); return false; }
      if (at.type != cudaMemoryTypeHost || !at.devicePointer) return false;
      *dev = at.devicePointer;
      return true;
    };
    direct = mapped(host_A, &map_A) && (!host_B || mapped(host_B, &map_B));
  }
  if (linearize && !direct && ((e = need(&b->d_A, nx * nx * N * es)) || (e = need(&b->d_B, nx * nu1 * N * es)))) return cuda_fail(e, "b2_step_host: cudaMalloc");
  // chunking: warp-engine batches and small batches go through in one piece
  // two chunks measured best at N = 65536 (1.72e8 vs 1.55e8 with 4, 0.94e8 with 16): every extra chunk adds ~11 copy nodes
  // (an async call overlaps with the other batch's call instead: one chunk measured best there, 1.93e8 vs 1.89e8)
  const int nchunk = (b->warp || N < 4096 || async) ? 1 : 2;
  if (!b->pipe_ready) {
    for (int i = 0; i < 3; i++) if ((e = cudaStreamCreateWithFlags(&b->pipe[i], cudaStreamNonBlocking))) return cuda_fail(e, "cudaStreamCreate");
    for (int i = 0; i < 3; i++) if ((e = cudaEventCreateWithFlags(&b->pipe_ev[i], cudaEventDisableTiming))) return cuda_fail(e, "cudaEventCreate");
    b->pipe_ready = true;
  }
  // The whole copy/compute pipeline is captured once into a CUDA graph (the host buffers of a
  // rollout loop are the same every step) and replayed with a single launch afterwards.
  HostStepKey key;
  memset(&key, 0, sizeof(key));
  key.qpos = hs->qpos; key.qvel = hs->qvel; key.ctrl = hs->ctrl; key.warm = hs->qacc_warmstart; key.A = host_A; key.B = host_B;
  key.nsteps = nsteps; key.linearize = linearize | (lqr ? B2_HOST_LQR : 0) | (nchunk << 8) | (direct ? 1 << 16 : 0); key.eps = eps; key.model_serial = b->model->serial;
  if (b->host_graph && memcmp(&key, &b->host_key, sizeof(key)) != 0) {
    cudaGraphExecDestroy(b->host_graph);
    b->host_graph = nullptr;
  }
  cudaStream_t s0 = b->pipe[0];
  if (!b->host_graph) {
    const size_t pitch = N * es;
    auto copy_rows = [&](void* dst, const void* src, size_t e0, size_t cnt, size_t rows, cudaMemcpyKind kind, cudaStream_t s) {
      return cudaMemcpy2DAsync((char*)dst + e0 * es, pitch, (const char*)src + e0 * es, pitch, cnt * es, rows, kind, s);
    };
    const long long launches_before = g_launches.load();
    if ((e = cudaStreamBeginCapture(s0, cudaStreamCaptureModeThreadLocal))) return cuda_fail(e, "cudaStreamBeginCapture");
    int err = B2_OK;
    // fork the side streams off the capturing stream
    if (!(e = cudaEventRecord(b->pipe_ev[0], s0)))
      for (int i = 1; i < 3 && !e; i++) e = cudaStreamWaitEvent(b->pipe[i], b->pipe_ev[0], 0);
    const size_t per = (N + nchunk - 1) / nchunk;
    for (int c = 0; c < nchunk && !e && !err; c++) {
      const size_t e0 = (size_t)c * per;
      if (e0 >= N) break;
      const size_t cnt = (e0 + per <= N) ? per : N - e0;
      cudaStream_t s = b->pipe[c % 3];
      if ((e = copy_rows(b->d_qpos, hs->qpos, e0, cnt, v.nq, cudaMemcpyHostToDevice, s)) ||
          (e = copy_rows(b->d_qvel, hs->qvel, e0, cnt, v.nv, cudaMemcpyHostToDevice, s)) ||
          (v.nu && !lqr && (e = copy_rows(b->d_ctrl, hs->ctrl, e0, cnt, v.nu, cudaMemcpyHostToDevice, s))))
        break;
      if (hs->qacc_warmstart) e = copy_rows(b->d_warm, hs->qacc_warmstart, e0, cnt, v.nv, cudaMemcpyHostToDevice, s);
      else e = cudaMemset2DAsync((char*)b->d_warm + e0 * es, pitch, 0, cnt * es, v.nv, s);
      if (e) break;
      b2_state ds = {(char*)b->d_qpos + e0 * es, (char*)b->d_qvel + e0 * es, (char*)b->d_ctrl + e0 * es, (char*)b->d_warm + e0 * es, nullptr};
      const void* gain = lqr ? b->d_gain : nullptr;
      void* out_A = direct ? (char*)map_A + e0 * es : (char*)b->d_A + e0 * es;
      void* out_B = direct ? (map_B ? (char*)map_B + e0 * es : nullptr) : (char*)b->d_B + e0 * es;
      if (linearize && (err = do_linearize(b, &ds, (int)cnt, eps, 1, out_A, out_B, s, gain))) break;
      if ((err = do_step(b, &ds, (int)cnt, nsteps, nullptr, s, gain))) break;
      if ((e = copy_rows(hs->qpos, b->d_qpos, e0, cnt, v.nq, cudaMemcpyDeviceToHost, s)) ||
          (e = copy_rows(hs->qvel, b->d_qvel, e0, cnt, v.nv, cudaMemcpyDeviceToHost, s)))
        break;
      if (hs->qacc_warmstart && (e = copy_rows(hs->qacc_warmstart, b->d_warm, e0, cnt, v.nv, cudaMemcpyDeviceToHost, s))) break;
      if (lqr && (e = copy_rows(hs->ctrl, b->d_ctrl, e0, cnt, v.nu, cudaMemcpyDeviceToHost, s))) break;
      if (linearize && !direct && host_A && (e = copy_rows(host_A, b->d_A, e0, cnt, nx * nx, cudaMemcpyDeviceToHost, s))) break;
      if (linearize && !direct && host_B && v.nu && (e = copy_rows(host_B, b->d_B, e0, cnt, nx * v.nu, cudaMemcpyDeviceToHost, s))) break;
    }
    // join the side streams back
    for (int i = 1; i < 3; i++) {
      cudaError_t e2 = cudaEventRecord(b->pipe_ev[i], b->pipe[i]);
      if (!e2) e2 = cudaStreamWaitEvent(s0, b->pipe_ev[i], 0);
      if (!e) e = e2;
    }
    cudaGraph_t graph = nullptr;
    cudaError_t ec = cudaStreamEndCapture(s0, &graph);
    if (err) { if (graph) cudaGraphDestroy(graph); return err; }
    if (e || ec) { if (graph) cudaGraphDestroy(graph); return cuda_fail(e ? e : ec, "b2_step_host: pipeline capture"); }
    e = cudaGraphInstantiate(&b->host_graph, graph, 0);
    cudaGraphDestroy(graph);
    if (e) { b->host_graph = nullptr; return cuda_fail(e, "cudaGraphInstantiate"); }
    b->host_key = key;
    b->host_graph_launches = (int)(g_launches.load() - launches_before);
    g_launches -= b->host_graph_launches;  // counted per replay below
  }
  // order after work the caller queued on `stream`, then replay
  if ((e = cudaStreamSynchronize((cudaStream_t)stream))) return cuda_fail(e, "b2_step_host: synchronize");
  if ((e = cudaGraphLaunch(b->host_graph, s0))) return cuda_fail(e, "cudaGraphLaunch");
  g_launches += b->host_graph_launches;
  if (async) return B2_OK;
  e = cudaStreamSynchronize(s0);
  return e ? cuda_fail(e, "b2_step_host: synchronize") : B2_OK;
}

int b2_step_host_wait(b2_batch* b) {
  if (!b) return fail(B2_ERR_ARG, "b2_step_host_wait: null batch");
  if (!b->pipe_ready) return B2_OK;  // nothing was ever queued
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
  e = cudaStreamSynchronize(b->pipe[0]);
  return e ? cuda_fail(e, "b2_step_host_wait: synchronize") : B2_OK;
}

int b2_lqr_control_env(b2_batch* b, const b2_state* st, const void* K_env, void* stream) {
  B2_CHECK_STATE("b2_lqr_control_env");
  if (!b->d_gain) return fail(B2_ERR_ARG, "b2_lqr_control_env: call b2_lqr_set_gain first (qpos_ref / ctrl_ref come from it)");
  if (!K_env) return fail(B2_ERR_ARG, "b2_lqr_control_env: K_env is NULL");
  const void* lane = nullptr;
  int rc = batch_images(b, &lane);
  if (rc) return rc;
  return launched(b->k->lqr_control_env(lane, b->model->cls, st, b->nenv, b->nenv, b->d_gain, K_env, stream), "b2_lqr_control_env launch");
}

int b2_random_controls(b2_batch* b, const b2_state* st, double lo, double hi, unsigned long long seed, int watch_row, double watch_min,
                       const void* reset_qpos, const void* reset_qvel, void* stream) {
  B2_CHECK_STATE("b2_random_controls");
  const b2m_view& v = b->model->v;
  if (v.nu == 0) return fail(B2_ERR_ARG, "b2_random_controls: model has no actuators");
  if (reset_qpos && (watch_row < 0 || watch_row >= v.nq)) return fail(B2_ERR_ARG, "b2_random_controls: watch_row out of range");
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
  if (!b->d_rng_ctr) {
    if ((e = cudaMalloc(&b->d_rng_ctr, sizeof(unsigned) * (size_t)b->nenv)) || (e = cudaMemset(b->d_rng_ctr, 0, sizeof(unsigned) * (size_t)b->nenv)))
      return cuda_fail(e, "b2_random_controls: draw counters");
  }
  return launched(b->k->random_controls(st, b->nenv, v.nq, v.nv, v.nu, lo, hi, seed, b->d_rng_ctr, watch_row, watch_min, reset_qpos, reset_qvel, stream),
                  "b2_random_controls launch");
}

}  // extern "C"

// The weight blocks of b2_dlqr (Q, R, R^-1) and b2_tvlqr (Q, R, Qf), converted to the call's precision, live on the device for
// as long as the process does, keyed by their contents: repeated calls with the same weights (a controller that
// re-synthesises its gains every tick, an iLQR iteration) neither allocate nor copy, and the calls can be captured into a
// CUDA graph once the block exists.  The calling thread's current device must be `device`.
static int resident_weights(int device, int precision, int nx, int nu, const std::vector<double>& vals, const char* who, void** out) {
  const size_t esz = precision == B2_F64 ? 8 : 4;
  std::vector<unsigned char> host(vals.size() * esz);
  for (size_t i = 0; i < vals.size(); i++) {
    if (precision == B2_F64) ((double*)host.data())[i] = vals[i]; else ((float*)host.data())[i] = (float)vals[i];
  }
  static std::mutex mu;
  static std::vector<std::pair<std::vector<unsigned char>, void*>> cache;  // key: bytes, then device, precision and sizes
  std::vector<unsigned char> key(host);
  const int head[4] = {device, precision, nx, nu};
  key.insert(key.end(), (const unsigned char*)head, (const unsigned char*)head + sizeof(head));
  std::lock_guard<std::mutex> lock(mu);
  for (auto& kv : cache) if (kv.first == key) { *out = kv.second; return B2_OK; }
  void* d = nullptr;
  cudaError_t e;
  if ((e = cudaMalloc(&d, host.size())) != cudaSuccess) return cuda_fail(e, (std::string(who) + ": cudaMalloc").c_str());
  if ((e = cudaMemcpy(d, host.data(), host.size(), cudaMemcpyHostToDevice)) != cudaSuccess) {
    cudaFree(d);
    return cuda_fail(e, (std::string(who) + ": upload").c_str());
  }
  if (cache.size() >= 64) { cudaFree(cache.front().second); cache.erase(cache.begin()); }
  cache.emplace_back(std::move(key), d);
  *out = d;
  return B2_OK;
}

extern "C" {

// Batched discrete LQR synthesis (see include/b2mj.h).  Q, R are host arrays shared by all envs; R is inverted here.
int b2_dlqr(int device, int precision, const void* A, const void* B, const double* Q, const double* R, int nx, int nu, int nenv,
            int max_doublings, double tol, void* K, void* P, int* status, void* stream) {
  if (!A || !B || !Q || !R || !K || !P || nx < 1 || nu < 1 || nu > nx || nenv < 1 || max_doublings < 1 || !(tol > 0))
    return fail(B2_ERR_ARG, "b2_dlqr: bad arguments");
  if (precision != B2_F64 && precision != B2_F32) return fail(B2_ERR_ARG, "b2_dlqr: precision must be 64 or 32");
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
  // Rinv by Gauss-Jordan with partial pivoting (nu x nu, host)
  std::vector<double> aug((size_t)nu * 2 * nu, 0.0);
  for (int i = 0; i < nu; i++) { for (int j = 0; j < nu; j++) aug[(size_t)i * 2 * nu + j] = R[i * nu + j]; aug[(size_t)i * 2 * nu + nu + i] = 1.0; }
  for (int c = 0; c < nu; c++) {
    int piv = c;
    for (int r = c + 1; r < nu; r++) if (std::abs(aug[(size_t)r * 2 * nu + c]) > std::abs(aug[(size_t)piv * 2 * nu + c])) piv = r;
    if (!(std::abs(aug[(size_t)piv * 2 * nu + c]) > 1e-300)) return fail(B2_ERR_ARG, "b2_dlqr: R is singular");
    if (piv != c) for (int k = 0; k < 2 * nu; k++) std::swap(aug[(size_t)c * 2 * nu + k], aug[(size_t)piv * 2 * nu + k]);
    const double inv = 1.0 / aug[(size_t)c * 2 * nu + c];
    for (int k = 0; k < 2 * nu; k++) aug[(size_t)c * 2 * nu + k] *= inv;
    for (int r = 0; r < nu; r++) if (r != c) { const double f = aug[(size_t)r * 2 * nu + c]; for (int k = 0; k < 2 * nu; k++) aug[(size_t)r * 2 * nu + k] -= f * aug[(size_t)c * 2 * nu + k]; }
  }
  std::vector<double> qr(Q, Q + (size_t)nx * nx);
  qr.insert(qr.end(), R, R + (size_t)nu * nu);
  for (int i = 0; i < nu; i++) qr.insert(qr.end(), aug.begin() + (size_t)i * 2 * nu + nu, aug.begin() + (size_t)(i + 1) * 2 * nu);
  void* dqr = nullptr;
  if (int rc = resident_weights(device, precision, nx, nu, qr, "b2_dlqr", &dqr)) return rc;
  const int rc = kernels(precision)->dare(A, B, dqr, nx, nu, nenv, max_doublings, tol, K, P, status, stream);
  g_launches++;
  if (rc == (int)cudaErrorInvalidValue) return fail(B2_ERR_CAPACITY, "b2_dlqr: nx too large for the shared-memory workspace of one SM");
  return rc ? cuda_fail((cudaError_t)rc, "b2_dlqr launch") : B2_OK;
}

// Finite-horizon time-varying LQR / iLQR backward pass (see include/b2mj.h).  Q, R, Qf are host arrays shared by all envs.
int b2_tvlqr(int device, int precision, int nsteps, int nx, int nu, int nenv, const void* A, const void* B, const double* Q, const double* R,
             const double* Qf, const void* q, const void* r, double reg, void* K, void* k, void* P0, void* dV, int* status, void* stream) {
  if (nsteps < 1 || nx < 1 || nu < 1 || nenv < 1) return fail(B2_ERR_ARG, "b2_tvlqr: nsteps, nx, nu and nenv must be >= 1");
  if (!(reg >= 0)) return fail(B2_ERR_ARG, "b2_tvlqr: reg must be >= 0");
  if (precision != B2_F64 && precision != B2_F32) return fail(B2_ERR_ARG, "b2_tvlqr: precision must be 64 or 32");
  if (!A || !B || !Q || !R || !Qf || !K) return fail(B2_ERR_ARG, "b2_tvlqr: A, B, Q, R, Qf and K are required");
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
  std::vector<double> w(Q, Q + (size_t)nx * nx);
  w.insert(w.end(), R, R + (size_t)nu * nu);
  w.insert(w.end(), Qf, Qf + (size_t)nx * nx);
  void* dw = nullptr;
  if (int rc = resident_weights(device, precision, nx, nu, w, "b2_tvlqr", &dw)) return rc;
  const int rc = kernels(precision)->tvlqr(A, B, dw, q, r, nsteps, nx, nu, nenv, reg, K, k, P0, dV, status, stream);
  g_launches++;
  if (rc == (int)cudaErrorInvalidValue) return fail(B2_ERR_CAPACITY, "b2_tvlqr: nx, nu too large for the shared-memory workspace of one SM");
  return rc ? cuda_fail((cudaError_t)rc, "b2_tvlqr launch") : B2_OK;
}

struct b2_recorder {
  b2_batch* batch;
  void* d_cols;
  int* d_index;
  int ncol, nsel;
};

int b2_recorder_create(b2_batch* b, const b2_record_col* cols, int ncol, const int* env_index, int nsel, b2_recorder** out) {
  if (!b || !cols || !env_index || !out || ncol < 1 || nsel < 1 || ncol > 65535) return fail(B2_ERR_ARG, "b2_recorder_create: bad arguments");
  for (int c = 0; c < ncol; c++)
    if (cols[c].kind < 0 || cols[c].kind > 2 || (cols[c].kind == 0 && (!cols[c].base || cols[c].row < 0)))
      return fail(B2_ERR_ARG, "b2_recorder_create: bad column " + std::to_string(c));
  for (int j = 0; j < nsel; j++)
    if (env_index[j] < 0 || env_index[j] >= b->nenv) return fail(B2_ERR_ARG, "b2_recorder_create: env index out of range");
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
  b2_recorder* r = new (std::nothrow) b2_recorder();
  if (!r) return fail(B2_ERR_ARG, "out of host memory");
  r->batch = b; r->ncol = ncol; r->nsel = nsel; r->d_cols = nullptr; r->d_index = nullptr;
  static_assert(sizeof(b2_record_col) == 16, "column table layout is shared with the kernel");
  if ((e = cudaMalloc(&r->d_cols, sizeof(b2_record_col) * ncol)) || (e = cudaMalloc((void**)&r->d_index, sizeof(int) * nsel)) ||
      (e = cudaMemcpy(r->d_cols, cols, sizeof(b2_record_col) * ncol, cudaMemcpyHostToDevice)) ||
      (e = cudaMemcpy(r->d_index, env_index, sizeof(int) * nsel, cudaMemcpyHostToDevice))) {
    b2_recorder_destroy(r);
    return cuda_fail(e, "b2_recorder_create");
  }
  *out = r;
  return B2_OK;
}
int b2_recorder_record(b2_recorder* r, double time, void* out_slot, void* stream) {
  if (!r || !out_slot) return fail(B2_ERR_ARG, "b2_recorder_record: null pointer");
  cudaError_t e = cudaSetDevice(r->batch->device);
  if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
  return launched(r->batch->k->record_rows(r->d_cols, r->ncol, r->d_index, r->nsel, r->batch->nenv, time, out_slot, stream),
                  "b2_recorder_record launch");
}
void b2_recorder_destroy(b2_recorder* r) {
  if (!r) return;
  if (r->d_cols) cudaFree(r->d_cols);
  if (r->d_index) cudaFree(r->d_index);
  delete r;
}

int b2_warp_queue_histogram(b2_batch* b, int* hist16, void* stream) {
  if (!b || !hist16) return fail(B2_ERR_ARG, "b2_warp_queue_histogram: null pointer");
  if (!b->warp) return fail(B2_ERR_ARG, "b2_warp_queue_histogram: batch does not run on the warp engine's ordered queue");
  cudaError_t e = cudaSetDevice(b->device);
  if (!e) e = cudaStreamSynchronize((cudaStream_t)stream);
  int bins[64] = {0};
  if (!e) e = cudaMemcpy(bins, b->d_warp_sort, 64 * sizeof(int), cudaMemcpyDeviceToHost);
  if (e) return cuda_fail(e, "b2_warp_queue_histogram");
  for (int k = 0; k < 16; k++) hist16[k] = bins[4 * k] + bins[4 * k + 1] + bins[4 * k + 2] + bins[4 * k + 3];  // row-count buckets folded
  return B2_OK;
}

int b2_fp_peak(int precision, int device, double* tflops) {
  if (!tflops || (precision != B2_F64 && precision != B2_F32)) return fail(B2_ERR_ARG, "b2_fp_peak: bad arguments");
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
  const double v = kernels(precision)->fma_peak(nullptr);
  g_launches += 6;
  if (v < 0) return fail(B2_ERR_CUDA, "b2_fp_peak: kernel failed");
  *tflops = v;
  return B2_OK;
}

int b2_stream_synchronize(b2_batch* b, void* stream) {
  if (b) cudaSetDevice(b->device);
  cudaError_t e = cudaStreamSynchronize((cudaStream_t)stream);
  return e ? cuda_fail(e, "cudaStreamSynchronize") : B2_OK;
}

}  // extern "C"
