// Registry of model-specialised kernel sets (generated translation units register themselves
// at load time; b2_model_create looks a model up by the FNV-1a hash of its blob).
#pragma once
#include <cstddef>
#include <cstdint>

#include "../../include/b2mj.h"

namespace b2 {

struct SpecKernels {
  const char* name;
  uint64_t blob_hash;
  size_t blob_size;
  // [0] FP64, [1] FP32; count envs, env stride N
  // gain != null: the control law of b2_lqr_set_gain is evaluated inside the kernel (ctrl becomes an output of step)
  // park != null: the kernel also copies the pre-step state there (b2_step_lazy)
  int (*step[2])(const b2_state* st, const b2_derived* out, int count, int N, int nsteps, const void* gain, const b2_state* park,
                 void* stream);
  // shadow != null (Euler models): the FD launch also advances every env into the shadow arrays (see k_linearize)
  int (*linearize[2])(const b2_state* st, int count, int N, double eps, int centered, void* A, void* B, const void* gain,
                      const b2_state* shadow, void* stream);
  int (*jacobian[2])(const b2_state* st, int N, int kind, int objid, void* jacp, void* jacr, void* stream);
  // b2_linearize_sensors: (A, B) and the sensor Jacobians dsdx / dsdu from the same rollouts.  Emitted only for models with
  // sensors; null otherwise (the call is then b2_linearize)
  int (*linearize_sensors[2])(const b2_state* st, int count, int N, double eps, int centered, void* A, void* B, void* dsdx,
                              void* dsdu, void* stream);
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
