"""TEST INFRASTRUCTURE ONLY -- ctypes front-end of the CPU oracle (oracle/mjstep_oracle.c).

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline legs may
import this module; the product package (``mujoco-template_b200/``) never does.

PARITY UNPINNED against a live MuJoCo except for the humanoid's inverse dynamics (published tutorial output:
tests/test_published_values.py); see the mjstep_oracle.c header and DESIGN.md section 5.
"""

from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_dp = C.POINTER(C.c_double)


def build(force: bool = False, variant: str = "strict") -> str:
    """strict: -O2 -ffp-contract=off, the parity oracle.  count: the op-counting build (orc_count.h).  Both are built
    in the tree by ``__graft_entry__.build()``; this rebuilds them when a source is newer."""
    target = {"strict": "liborc.so", "count": "liborc_count.so"}[variant]
    so = os.path.join(_HERE, target)
    src = [os.path.join(_HERE, f) for f in ("mjstep_oracle.c", "orc_math.h", "orc_count.h")]
    src.append(os.path.join(_HERE, "..", "include", "b2_model_layout.h"))
    stale = not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src)
    if force or stale:
        subprocess.run(["make", "-C", _HERE, "-B", target], check=True, capture_output=True)
    return so


def _load_fast() -> C.CDLL:
    """fast: -O3 -march=native with contraction, ONLY for bench.py's CPU arm.  Compiled for the CPU of the host that
    runs it, in a temporary directory (the source tree may be read-only) that is removed once the library is loaded."""
    with tempfile.TemporaryDirectory(prefix="orc_fast_") as tmp:
        so = os.path.join(tmp, "liborc_fast.so")
        subprocess.run(["make", "-C", _HERE, "-B", f"FAST_DIR={tmp}", so], check=True, capture_output=True)
        return C.CDLL(so)


_LIBS: dict[str, C.CDLL] = {}


def lib(variant: str = "strict") -> C.CDLL:
    global _LIB
    if variant != "strict":
        if variant not in _LIBS:
            _LIBS[variant] = _declare(_load_fast() if variant == "fast" else C.CDLL(build(variant=variant)))
            if variant == "count":
                _LIBS[variant].orc_count_read.argtypes = [C.POINTER(C.c_ulonglong)]
        return _LIBS[variant]
    if _LIB is None:
        _LIB = _declare(C.CDLL(build()))
    return _LIB


def _declare(L: C.CDLL) -> C.CDLL:
    if True:
        L.orc_model_create.restype = C.c_void_p
        L.orc_model_create.argtypes = [C.c_char_p, C.c_size_t]
        L.orc_model_free.argtypes = [C.c_void_p]
        L.orc_model_nsensordata.argtypes = [C.c_void_p]
        L.orc_data_create.restype = C.c_void_p
        L.orc_data_create.argtypes = [C.c_void_p]
        L.orc_data_free.argtypes = [C.c_void_p]
        L.orc_reset.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.orc_forward.argtypes = [C.c_void_p, C.c_void_p]
        L.orc_step.argtypes = [C.c_void_p, C.c_void_p]
        L.orc_transition_fd.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_int, _dp, _dp]
        L.orc_inverse.argtypes = [C.c_void_p, C.c_void_p, _dp, _dp]
        L.orc_integrate_pos.argtypes = [C.c_void_p, _dp, _dp, C.c_double]
        L.orc_differentiate_pos.argtypes = [C.c_void_p, _dp, C.c_double, _dp, _dp]
        L.orc_jac.argtypes = [C.c_void_p, C.c_void_p, _dp, _dp, _dp, C.c_int]
        for fn in ("orc_jac_site", "orc_jac_body", "orc_jac_bodycom"):
            getattr(L, fn).argtypes = [C.c_void_p, C.c_void_p, _dp, _dp, C.c_int]
        L.orc_jac_subtreecom.argtypes = [C.c_void_p, C.c_void_p, _dp, C.c_int]
        L.orc_ptr.restype = _dp
        L.orc_ptr.argtypes = [C.c_void_p, C.c_char_p]
        L.orc_get_time.restype = C.c_double
        L.orc_get_time.argtypes = [C.c_void_p]
        L.orc_set_time.argtypes = [C.c_void_p, C.c_double]
        for fn in ("orc_ncon", "orc_nefc", "orc_solver_iter", "orc_warnings"):
            getattr(L, fn).argtypes = [C.c_void_p]
        L.orc_get_contact.argtypes = [C.c_void_p, C.c_int, _dp]
        L.orc_setconst_check.restype = C.c_double
        L.orc_setconst_check.argtypes = [C.c_void_p, _dp, _dp, _dp]
        L.orc_batch_rollout.argtypes = [C.c_void_p, C.c_int, _dp, _dp, _dp, _dp, C.c_int, C.c_int, C.c_double,
                                        _dp, _dp, C.c_int]
    return L


def op_count(blob: bytes, dims: dict, qpos, qvel, ctrl, *, linearize: bool = False, warm_steps: int = 1) -> dict:
    """Algorithmic operation count of one mj_step (or one mjd_transitionFD + step) of the oracle on the given state:
    runs `warm_steps` uncounted steps first (so that qacc_warmstart is a realistic one), then counts one.  Weights as in
    SURVEY.md section 8(d): add / mul / div / sqrt = 1 flop, transcendental call = 20."""
    om = OracleModel(blob, dims, variant="count")
    od = OracleData(om)
    od.qpos[:] = qpos; od.qvel[:] = qvel
    if od.ctrl.size:
        od.ctrl[:] = ctrl
    for _ in range(warm_steps):
        od.step()
    L = om._L
    L.orc_count_reset()
    if linearize:
        od.transition_fd(1e-6, True)
    od.step()
    c = (C.c_ulonglong * 5)()
    L.orc_count_read(c)
    add, mul, div, sq, tr = (int(x) for x in c)
    return {"add": add, "mul": mul, "div": div, "sqrt": sq, "transcendental": tr, "flops": add + mul + div + sq + 20 * tr,
            "ncon": int(od.ncon), "nefc": int(od.nefc), "solver_iter": int(od.solver_iter)}


def _p(a: np.ndarray | None):
    return None if a is None else a.ctypes.data_as(_dp)


class OracleModel:
    def __init__(self, blob: bytes, dims: dict, variant: str = "strict"):
        self._L = lib(variant)
        self.h = self._L.orc_model_create(blob, len(blob))
        if not self.h:
            raise RuntimeError("oracle rejected model blob")
        self.dims = {k: int(dims[k]) for k in ("nq", "nv", "nu", "nbody", "njnt", "ngeom", "nsite", "ntendon")}
        self.dims["nsensordata"] = int(self._L.orc_model_nsensordata(self.h))

    def __del__(self):
        if getattr(self, "h", None):
            self._L.orc_model_free(self.h)
            self.h = None

    def setconst(self):
        d = self.dims
        dof = np.zeros(d["nv"]); body = np.zeros(2 * d["nbody"]); ten = np.zeros(max(1, d["ntendon"]))
        mean = self._L.orc_setconst_check(self.h, _p(dof), _p(body), _p(ten))
        return mean, dof, body.reshape(-1, 2), ten[: d["ntendon"]]

    def batch_rollout(self, qpos, qvel, ctrl, warm=None, nsteps=1, lin=False, eps=1e-6, nthreads=1, want_ab=False):
        """AoS batch: qpos (N,nq), qvel (N,nv), ctrl (N,nu). Arrays are advanced in place."""
        d = self.dims
        N = qpos.shape[0]
        assert qpos.flags.c_contiguous and qvel.flags.c_contiguous and ctrl.flags.c_contiguous
        if warm is None:
            warm = np.zeros((N, d["nv"]))
        A = B = None
        if lin and want_ab:
            A = np.zeros((N, 2 * d["nv"], 2 * d["nv"])); B = np.zeros((N, 2 * d["nv"], d["nu"]))
        self._L.orc_batch_rollout(self.h, N, _p(qpos), _p(qvel), _p(ctrl), _p(warm), int(nsteps), int(bool(lin)),
                                  float(eps), _p(A), _p(B), int(nthreads))
        return warm, A, B


class OracleData:
    """mjData-like view: ``qpos``/``qvel``/``ctrl``... are NumPy views of the C arrays."""

    _SIZES = dict(qpos="nq", qvel="nv", ctrl="nu", qacc="nv", qacc_warmstart="nv", qfrc_bias="nv", qfrc_passive="nv",
                  qfrc_actuator="nv", qfrc_smooth="nv", qacc_smooth="nv", qfrc_constraint="nv")

    def __init__(self, model: OracleModel):
        self.model = model
        self._L = model._L
        self.h = self._L.orc_data_create(model.h)
        d = model.dims
        for name, key in self._SIZES.items():
            setattr(self, name, self._view(name, (d[key],)))
        nb, ng, ns, nv = d["nbody"], d["ngeom"], d["nsite"], d["nv"]
        self.xpos = self._view("xpos", (nb, 3)); self.xquat = self._view("xquat", (nb, 4))
        self.xmat = self._view("xmat", (nb, 9)); self.xipos = self._view("xipos", (nb, 3))
        self.ximat = self._view("ximat", (nb, 9)); self.subtree_com = self._view("subtree_com", (nb, 3))
        self.geom_xpos = self._view("geom_xpos", (ng, 3)); self.geom_xmat = self._view("geom_xmat", (ng, 9))
        self.site_xpos = self._view("site_xpos", (ns, 3)); self.site_xmat = self._view("site_xmat", (ns, 9))
        self.qM = self._view("qM", (nv, nv)); self.cvel = self._view("cvel", (nb, 6))
        self.actuator_force = self._view("actuator_force", (d["nu"],))
        self.actuator_moment = self._view("actuator_moment", (d["nu"], nv))
        self.sensordata = self._view("sensordata", (d["nsensordata"],)); self.cacc = self._view("cacc", (nb, 6))
        self.reset()

    def _view(self, name: str, shape):
        n = int(np.prod(shape))
        if n == 0:
            return np.zeros(shape)
        ptr = self._L.orc_ptr(self.h, name.encode())
        return np.ctypeslib.as_array(ptr, shape=(n,)).reshape(shape)

    def __del__(self):
        if getattr(self, "h", None):
            self._L.orc_data_free(self.h)
            self.h = None

    @property
    def time(self) -> float:
        return self._L.orc_get_time(self.h)

    @time.setter
    def time(self, t: float) -> None:
        self._L.orc_set_time(self.h, float(t))

    @property
    def ncon(self) -> int:
        return self._L.orc_ncon(self.h)

    @property
    def nefc(self) -> int:
        return self._L.orc_nefc(self.h)

    @property
    def solver_iter(self) -> int:
        return self._L.orc_solver_iter(self.h)

    @property
    def warnings(self) -> int:
        return self._L.orc_warnings(self.h)

    def efc(self, name: str):
        nefc, nv = self.nefc, self.model.dims["nv"]
        n = nefc * nv if name == "efc_J" else nefc
        if n == 0:
            return np.zeros((0, nv) if name == "efc_J" else 0)
        a = np.ctypeslib.as_array(self._L.orc_ptr(self.h, name.encode()), shape=(n,)).copy()
        return a.reshape(nefc, nv) if name == "efc_J" else a

    def contacts(self):
        out = []
        buf = np.zeros(16)
        for k in range(self.ncon):
            self._L.orc_get_contact(self.h, k, _p(buf))
            out.append(dict(dist=buf[0], pos=buf[1:4].copy(), frame=buf[4:13].copy().reshape(3, 3), dim=int(buf[13]),
                            geom1=int(buf[14]), geom2=int(buf[15])))
        return out

    def reset(self, key: int = -1) -> None:
        self._L.orc_reset(self.model.h, self.h, int(key))

    def forward(self) -> None:
        self._L.orc_forward(self.model.h, self.h)

    def step(self, n: int = 1) -> None:
        for _ in range(n):
            self._L.orc_step(self.model.h, self.h)

    def transition_fd(self, eps: float = 1e-6, centered: bool = True):
        d = self.model.dims
        A = np.zeros((2 * d["nv"], 2 * d["nv"])); B = np.zeros((2 * d["nv"], d["nu"]))
        self._L.orc_transition_fd(self.model.h, self.h, float(eps), int(centered), _p(A), _p(B) if d["nu"] else None)
        return A, B

    def inverse(self, qacc: np.ndarray) -> np.ndarray:
        """mj_inverse at the current (qpos, qvel) for the given qacc; also refreshes ``actuator_moment``."""
        out = np.zeros(self.model.dims["nv"])
        a = np.ascontiguousarray(qacc, dtype=float)
        self._L.orc_inverse(self.model.h, self.h, _p(a), _p(out))
        return out

    def integrate_pos(self, qpos: np.ndarray, qvel: np.ndarray, dt: float) -> np.ndarray:
        q = np.array(qpos, dtype=float); v = np.ascontiguousarray(qvel, dtype=float)
        self._L.orc_integrate_pos(self.model.h, _p(q), _p(v), float(dt))
        return q

    def differentiate_pos(self, dt: float, qpos1: np.ndarray, qpos2: np.ndarray) -> np.ndarray:
        out = np.zeros(self.model.dims["nv"])
        q1 = np.ascontiguousarray(qpos1, dtype=float); q2 = np.ascontiguousarray(qpos2, dtype=float)
        self._L.orc_differentiate_pos(self.model.h, _p(out), float(dt), _p(q1), _p(q2))
        return out

    def jac(self, kind: str, objid: int):
        nv = self.model.dims["nv"]
        jp = np.zeros((3, nv)); jr = np.zeros((3, nv))
        if kind == "subtreecom":
            self._L.orc_jac_subtreecom(self.model.h, self.h, _p(jp), int(objid))
            return jp, None
        getattr(self._L, f"orc_jac_{kind}")(self.model.h, self.h, _p(jp), _p(jr), int(objid))
        return jp, jr
