"""Emit model-specialised CUDA translation units (static model providers).

For a compiled model this writes ``csrc/generated/spec_<name>.cu``: a provider class whose
accessors return compile-time constants (function-local ``constexpr`` tables), exact-size
capacity constants, launchers for the step / linearize / jacobian / rollout kernels instantiated with that
provider, and a registrar keyed by the FNV-1a hash of the model blob.  ``libb2mj.so`` picks the
specialised kernels automatically when ``b2_model_create`` sees a blob with a registered hash;
any other model runs on the generic kernels.

Run by ``__graft_entry__.build()`` for the example models before ``make``.
"""

from __future__ import annotations

import os

import numpy as np

from . import _layout

# (field, kind) in the order of the X-macro lists in csrc/b2_model_dev.cuh
INT_SCALARS = ("nq", "nv", "nu", "nbody", "njnt", "ngeom", "nsite", "ntendon", "npair", "integrator", "iterations",
               "ls_iterations", "has_fluid", "has_dofdamping", "maxdepth", "nsensor", "nsensordata")
REAL_SCALARS = ("timestep", "density", "viscosity", "tolerance", "ls_tolerance", "meaninertia")
INT_ARRAYS = ("body_parentid", "body_rootid", "body_jntnum", "body_jntadr", "body_dofnum", "body_dofadr", "body_anc",
              "body_depth", "jnt_type",
              "jnt_qposadr", "jnt_dofadr", "jnt_bodyid", "jnt_limited", "dof_bodyid", "dof_jntid", "dof_parentid", "dof_anc",
              "dof_nanc", "dof_anclist",
              "geom_type", "geom_bodyid", "site_bodyid", "tendon_adr", "tendon_num", "tendon_limited", "wrap_jntid",
              "actuator_trntype", "actuator_trnid", "actuator_ctrllimited", "actuator_forcelimited", "actuator_disabled",
              "pair_geom1", "pair_geom2", "pair_dim", "sensor_type", "sensor_objtype", "sensor_objid", "sensor_adr",
              "sensor_dim")
REAL_ARRAYS = ("gravity", "wind", "body_pos", "body_quat", "body_ipos", "body_iquat", "body_mass", "body_subtreemass",
               "body_inertia", "body_invweight0", "jnt_pos", "jnt_axis", "jnt_stiffness", "jnt_range", "jnt_margin",
               "jnt_solref", "jnt_solimp", "qpos0", "qpos_spring", "dof_armature", "dof_damping", "dof_invweight0",
               "geom_size", "geom_rbound", "geom_pos", "geom_quat", "site_pos", "site_quat", "tendon_range",
               "tendon_margin", "tendon_solref", "tendon_solimp", "tendon_invweight0", "tendon_stiffness",
               "tendon_damping", "tendon_lengthspring", "wrap_coef", "actuator_gear", "actuator_ctrlrange",
               "actuator_forcerange", "actuator_gainprm", "actuator_biasprm", "pair_margin", "pair_gap", "pair_friction",
               "pair_solref", "pair_solimp", "sensor_cutoff")

# FD kernel block shape for small models (nv <= 2): (threads per block, min resident blocks per SM).  64 x 4 lets ptxas use
# 253 registers -- the cartpole FD kernel then has no spills at all -- at 8 warps per SM, in blocks small enough that the last
# wave of the launch is short: 36.4 us against 38.6 us for 128 x 3 (168 registers, 320 B of spills, 12 warps); explicit caps
# in between (184 / 200 / 216 registers at 9-11 warps) are all slower (round 2, profiles/ab_cartpole_lin_shapes_r02k.txt).
# Larger models keep the kernel's default, 128 x 1.
SMALL_LIN_SHAPE = (64, 4)

_MAX_CONTACTS = {(0, 2): 1, (0, 3): 2, (0, 6): 4, (0, 4): 1, (2, 2): 1, (2, 3): 1, (3, 3): 2}


def fnv1a(data: bytes) -> int:
    h = 1469598103934665603
    for b in data:
        h = ((h ^ b) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return h


def _values(c: dict, name: str) -> np.ndarray:
    if name == "dof_anc":
        out = []
        for i in range(int(c["nv"])):
            mask, j = 0, i
            while j >= 0:
                mask |= 1 << j
                j = int(c["dof_parentid"][j])
            out.append(mask - (1 << 32) if mask >= (1 << 31) else mask)
        return np.array(out, dtype=np.int64)
    if name in ("dof_nanc", "dof_anclist"):
        nv = int(c["nv"])
        stride = max(1, nv)  # generated Dims use exact sizes: NV == nv
        counts, flat = [], [0] * (stride * stride)
        for i in range(nv):
            n, j = 0, int(c["dof_parentid"][i])
            while j >= 0:
                flat[i * stride + n] = j
                n += 1
                j = int(c["dof_parentid"][j])
            counts.append(n)
        return np.array(counts if name == "dof_nanc" else flat, dtype=np.int64)
    if name in ("body_anc", "body_depth"):
        masks, depths = [], []
        for i in range(int(c["nbody"])):
            mask, depth, j = 1 << i, 0, i
            while j > 0:
                j = int(c["body_parentid"][j])
                mask |= 1 << j
                depth += 1
            masks.append(mask - (1 << 32) if mask >= (1 << 31) else mask)
            depths.append(depth)
        return np.array(masks if name == "body_anc" else depths, dtype=np.int64)
    if name == "pair_friction":
        return np.asarray(c["pair_friction"], dtype=float).reshape(-1, 5)[:, :2].ravel()
    return np.asarray(c[name]).ravel()


def _lit(x: float) -> str:
    s = repr(float(x))
    if s in ("inf", "-inf", "nan"):
        raise ValueError("non-finite model constant")
    return s if ("." in s or "e" in s or "E" in s) else s + ".0"


def emit_spec(compiled: dict, name: str) -> str:
    c = compiled
    blob = _layout.pack(c)
    nb, nj, nq, nv, nu = (int(c[k]) for k in ("nbody", "njnt", "nq", "nv", "nu"))
    ng, ns, nt, nw, npair = (int(c[k]) for k in ("ngeom", "nsite", "ntendon", "nwrap", "npair"))
    ncon = 0
    for p in range(npair):
        key = (int(c["geom_type"][c["pair_geom1"][p]]), int(c["geom_type"][c["pair_geom2"][p]]))
        ncon += _MAX_CONTACTS.get(key, 1)
    nefc = 2 * int(np.sum(c["jnt_limited"])) + 2 * int(np.sum(c["tendon_limited"])) + 4 * ncon
    one = lambda n: max(1, n)  # noqa: E731
    L: list[str] = []
    A = L.append
    A(f"// GENERATED by mujoco_template/_specialize.py for model '{name}' -- do not edit.")
    A("// Static model provider: every accessor folds to a compile-time constant after unrolling.")
    A("#define B2_STATIC_MODEL 1")
    lin_threads, lin_blocks = SMALL_LIN_SHAPE if nv <= 2 else (128, 1)
    A(f"#define B2_LIN_THREADS {lin_threads}")
    A(f"#define B2_LIN_MIN_BLOCKS {lin_blocks}")
    # the sensor-Jacobian FD launcher exists only for models with sensors (the others' C-ABI call is b2_linearize), so the
    # generated sources of sensorless models do not change with it
    has_sensors = int(c["nsensordata"]) > 0
    A('#include "../b2_kernel_templates.cuh"')
    A('#include "../b2_kernels.h"')
    A("")
    A("namespace b2 {")
    A("namespace {")
    A("struct SDims {")
    A(f"  static constexpr int NB = {one(nb)}, NJ = {one(nj)}, NQ = {one(nq)}, NV = {one(nv)}, NU = {one(nu)}, NG = {one(ng)}, "
      f"NS = {one(ns)}, NT = {one(nt)}, NW = {one(nw)}, NPAIR = {one(npair)}, NCON = {one(ncon)}, NEFC = {one(nefc)}, "
      f"NSEN = {one(int(c['nsensor']))}, NSD = {one(int(c['nsensordata']))};")
    A("};")
    A("template <typename T>")
    A("struct SModel {")
    for k in INT_SCALARS:
        val = int(max(_values(c, "body_depth"))) if k == "maxdepth" else int(c[k])
        A(f"  static B2_DEV constexpr int {k}() {{ return {val}; }}")
    for k in REAL_SCALARS:
        A(f"  static B2_DEV constexpr T {k}() {{ return T({_lit(c[k])}); }}")
    for k in INT_ARRAYS:
        v = _values(c, k)
        body = ", ".join(str(int(x)) for x in v) if v.size else "0"
        A(f"  static B2_DEV int {k}(int i) {{ static constexpr int t[{one(v.size)}] = {{{body}}}; return t[i]; }}")
    for k in REAL_ARRAYS:
        v = _values(c, k)
        body = ", ".join(_lit(x) for x in v) if v.size else "0.0"
        A(f"  static B2_DEV T {k}(int i) {{ static constexpr T t[{one(v.size)}] = {{{body}}}; return t[i]; }}")
    A("};")
    A("")
    # launchers with the LaneKernels signatures (b2_kernels.h): b2_kernel_templates.cuh's launch_* own block size and grid;
    # the static provider needs no model image, and the caller passes the FD task count
    lane = "const void*, int, const b2_state* st"
    for T, suf in (("double", ""), ("float", "32")):
        M = f"{T}, SDims, SModel<{T}>"
        A(f"int spec_step{suf}({lane}, const b2_derived* out, int count, int N, int nsteps, const void* gain, const b2_state* park, void* stream) {{")
        A(f"  return launch_step<{M}>(nullptr, st, out, count, N, nsteps, gain, park, stream);")
        A("}")
        A(f"int spec_linearize{suf}({lane}, int count, int N, int ntask, double eps, int centered, void* A, void* B, const void* gain, const b2_state* shadow, void* stream) {{")
        A(f"  return launch_linearize<{M}>(nullptr, st, count, N, ntask, eps, centered, A, B, gain, shadow, nullptr, nullptr, stream);")
        A("}")
        if has_sensors:
            # (A, B) plus the sensor Jacobians from the same rollouts: no control law, no advance
            A(f"int spec_linearize_sensors{suf}({lane}, int count, int N, int ntask, double eps, int centered, void* A, void* B, void* dsdx, void* dsdu, void* stream) {{")
            A(f"  return launch_linearize<{M}, true>(nullptr, st, count, N, ntask, eps, centered, A, B, nullptr, nullptr, dsdx, dsdu, stream);")
            A("}")
        A(f"int spec_jacobian{suf}({lane}, int N, int kind, int objid, void* jacp, void* jacr, void* stream) {{")
        A(f"  return launch_jacobian<{M}>(nullptr, st, N, kind, objid, jacp, jacr, stream);")
        A("}")
    # the rollout kernels come after all the others: cicc's inlining, and so the other kernels' code, depends on kernel order
    for T, suf in (("double", ""), ("float", "32")):
        A(f"int spec_rollout{suf}({lane}, const b2_derived* out, int N, int nsteps, const void* ctrl_seq, void* qpos_traj, void* qvel_traj, void* sensor_traj, void* stream) {{")
        A(f"  return launch_rollout<{T}, SDims, SModel<{T}>>(nullptr, st, out, N, nsteps, ctrl_seq, qpos_traj, qvel_traj, sensor_traj, stream);")
        A("}")
    # ... and the linearisation along a rollout after them; its sensor variant only for models with sensors (the C-ABI
    # passes no dsdx / dsdu for a model without)
    for T, suf in (("double", ""), ("float", "32")):
        M = f"{T}, SDims, SModel<{T}>"
        A(f"int spec_linearize_rollout{suf}({lane}, int N, int ntask, int nsteps, const void* ctrl_seq, double eps, int centered, void* A, void* B, void* dsdx, void* dsdu, void* qpos_traj, void* qvel_traj, void* warm_traj, void* sensor_traj, void* stream) {{")
        call = "(nullptr, st, N, ntask, nsteps, ctrl_seq, eps, centered, A, B, {}, qpos_traj, qvel_traj, warm_traj, sensor_traj, stream);"
        if has_sensors:
            A(f"  if (dsdx || dsdu) return launch_linearize_rollout<{M}, true>" + call.format("dsdx, dsdu"))
        A(f"  return launch_linearize_rollout<{M}>" + call.format("nullptr, nullptr"))
        A("}")
    # ... and the closed-loop rollout last
    for T, suf in (("double", ""), ("float", "32")):
        A(f"int spec_rollout_feedback{suf}({lane}, const b2_derived* out, int N, int nsteps, const void* ctrl_nom, const void* qpos_nom, const void* qvel_nom, const void* K, const void* k, const void* alpha, void* ctrl_traj, void* qpos_traj, void* qvel_traj, void* sensor_traj, void* stream) {{")
        A(f"  return launch_rollout_feedback<{T}, SDims, SModel<{T}>>(nullptr, st, out, N, nsteps, ctrl_nom, qpos_nom, qvel_nom, K, k, alpha, ctrl_traj, qpos_traj, qvel_traj, sensor_traj, stream);")
        A("}")
    lanes = []
    for suf in ("", "32"):
        sens = f"spec_linearize_sensors{suf}" if has_sensors else "nullptr"
        lanes.append(f"{{spec_step{suf}, spec_linearize{suf}, {sens}, spec_jacobian{suf}, spec_rollout{suf}, spec_linearize_rollout{suf}, "
                     f"spec_rollout_feedback{suf}}}")
    A(f'const SpecKernels kSpec = {{"{name}", 0x{fnv1a(blob):016x}ull, {len(blob)}, {{{lanes[0]}, {lanes[1]}}}}};')
    A("struct Registrar { Registrar() { register_spec(&kSpec); } } registrar;")
    A("}  // namespace")
    A("}  // namespace b2")
    return "\n".join(L) + "\n"


def write_specs(models: dict[str, dict], outdir: str) -> list[str]:
    """models: name -> compiled dict.  Returns the written paths (only rewrites changed files)."""
    os.makedirs(outdir, exist_ok=True)
    paths = []
    for name, compiled in models.items():
        text = emit_spec(compiled, name)
        path = os.path.join(outdir, f"spec_{name}.cu")
        old = open(path).read() if os.path.exists(path) else None
        if old != text:
            with open(path, "w") as fh:
                fh.write(text)
        paths.append(path)
    return paths


# ------------------------------------------------------------------ run-time specialisation of a user's model
JIT_MAX_NV = 8  # beyond this the fully unrolled kernels stop paying (registers, compile time): generic / warp engine


def jit_specialize(model, name: str | None = None, cache_dir: str | None = None, verbose: bool = False) -> str | None:
    """Compile model-specialised (register-resident) kernels for ``model`` with nvcc and register them with the
    loaded ``libb2mj.so``; later ``b2_model_create`` calls on the same blob pick them up (``kernel_variant`` then
    reports ``name``).  The example models ship pre-compiled; this gives any other small model of the MJCF subset the
    same kernels (reference ``Env.from_xml_path`` compiles the model at load time too: ``mujoco_template/env.py:99-143``).

    Returns the path of the shared object, or ``None`` when the model is too large (nv > JIT_MAX_NV).  The object is
    cached under ``cache_dir`` (default ``$B2_SPEC_CACHE`` or ``~/.cache/b2mj``) keyed by the blob hash, so the
    ~1 minute compile happens once per model."""
    import ctypes
    import shutil
    import subprocess

    from . import _capi

    c = model._c if hasattr(model, "_c") else model
    if int(c["nv"]) > JIT_MAX_NV:
        return None
    blob = _layout.pack(c)
    csrc = os.path.normpath(os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "csrc"))
    flags = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC",
             "--expt-relaxed-constexpr", "-shared"]
    name_hint = name
    # The cache key covers everything the object depends on: the model, the generated source (kernel launch shape, spec
    # ABI), the engine headers it includes and the compiler flags -- an object built against an older library is never
    # picked up after an update.
    source = emit_spec(c, name or "jit")
    h = fnv1a(blob)
    for path in sorted(os.listdir(csrc)):
        if path.endswith((".cuh", ".h")) or path in ("ptx_fold.py", "fold_build.py"):
            with open(os.path.join(csrc, path), "rb") as fh:
                h = fnv1a(fh.read() + h.to_bytes(8, "little"))
    h = fnv1a(source.encode() + " ".join(flags).encode() + h.to_bytes(8, "little"))
    key = f"{fnv1a(blob):016x}_{len(blob)}_{h:016x}"
    name = name_hint or f"jit_{key[:8]}"
    cache_dir = cache_dir or os.environ.get("B2_SPEC_CACHE") or os.path.join(os.path.expanduser("~"), ".cache", "b2mj")
    os.makedirs(cache_dir, exist_ok=True)
    so = os.path.join(cache_dir, f"spec_{key}.so")
    if not os.path.exists(so):
        import tempfile

        nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
        # private temporaries (several ranks may compile the same model at once), published by an atomic rename
        fd, cu = tempfile.mkstemp(prefix=f"spec_{key}_", suffix=".cu", dir=cache_dir)
        with os.fdopen(fd, "w") as fh:
            fh.write(emit_spec(c, name))
        tmp_so, obj = cu[:-3] + ".so.tmp", cu[:-3] + ".o"
        # compile through fold_build.py (exact zeros / ones of the model folded on the PTX, as for the built-in models),
        # then link
        import sys

        cflags = [f for f in flags if f != "-shared"] + ["-I", os.path.join(csrc, "generated")]
        r = subprocess.run([sys.executable, os.path.join(csrc, "fold_build.py"), nvcc, cu, obj] + cflags, capture_output=True, text=True)
        if r.returncode == 0:
            r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", tmp_so, obj], capture_output=True, text=True)
        if r.returncode != 0:
            from .exceptions import ConfigError

            for leftover in (cu, tmp_so, obj):
                if os.path.exists(leftover):
                    os.remove(leftover)
            raise ConfigError("jit_specialize: nvcc failed\n" + r.stderr[-2000:])
        os.replace(tmp_so, so)
        os.remove(cu)
        os.remove(obj)
        if verbose:
            print(f"jit_specialize: built {so}")
    _capi.lib()  # libb2mj.so must be loaded (globally) first: the object's registrar calls b2::register_spec
    _LOADED.setdefault(so, ctypes.CDLL(so, mode=ctypes.RTLD_GLOBAL))
    return so


_LOADED: dict = {}
