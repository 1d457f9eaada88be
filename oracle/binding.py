"""ctypes wrapper around oracle/liboracle.so — TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py (cpu_baseline / --impl reference) may import this.
The product package momentum_b200 never does.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
import sys
import tempfile
from typing import Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "liboracle.so")
_lib = None
_native = None

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


def build(force: bool = False) -> str:
    src = [os.path.join(_HERE, f) for f in ("ik_oracle_capi.cpp", "ik_oracle.hpp", "Makefile")]
    if force or not os.path.exists(_LIB_PATH) or any(os.path.getmtime(s) > os.path.getmtime(_LIB_PATH) for s in src):
        subprocess.check_call(["make", "-C", _HERE, "-s", "-B"])
    return _LIB_PATH


def native_lib():
    """The -march=native / fast-math build for bench.py's CPU arm. Always rebuilt by the process that times it (a copy built on
    another host may use instructions this one lacks), into a temporary directory so that the source tree is never written; falls
    back to the portable checker build if the compile fails."""
    global _native
    if _native is None:
        tmp = tempfile.mkdtemp(prefix="oracle_native_")
        try:
            path = os.path.join(tmp, "liboracle_native.so")
            subprocess.check_call(["make", "-C", _HERE, "-s", "-B", "native", f"NATIVE_OUT={path}"])
            _native = _bind(C.CDLL(path))  # the mapping outlives the file, so the directory can go at once
            _native.is_native = True
        except Exception as e:  # noqa: BLE001
            print(f"[oracle] native build unavailable ({e}); timing the portable build", file=sys.stderr, flush=True)
            _native = lib()
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
    return _native


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        _lib = _bind(C.CDLL(_LIB_PATH))
    return _lib


def _bind(L):
    if True:  # (keeps the declaration block at its historical indentation)
        L.orc_rig_create.restype = C.c_void_p
        L.orc_rig_create.argtypes = [C.c_int, _ip, _dp, _dp, C.c_int, _ip, _ip, _dp, _dp]
        L.orc_rig_add_limit.argtypes = [C.c_void_p, C.c_int, C.c_double, _ip, _dp]
        L.orc_rig_destroy.argtypes = [C.c_void_p]
        L.orc_fn_create.restype = C.c_void_p
        L.orc_fn_create.argtypes = [C.c_void_p, C.c_int]
        L.orc_fn_destroy.argtypes = [C.c_void_p]
        L.orc_fn_set_trust_region_radius.argtypes = [C.c_void_p, C.c_double]
        L.orc_fn_set_trust_region_radius.restype = None
        L.orc_fn_add_joint_ef.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_double, C.c_int, _ip, _dp, _dp, _dp]
        L.orc_fn_add_state_ef.argtypes = [C.c_void_p, C.c_double, C.c_int, C.c_double, C.c_double, _dp, _dp, _dp]
        L.orc_fn_add_limit_ef.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_double]
        L.orc_fn_set_half_plane.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.orc_fn_add_model_parameters_ef.argtypes = [C.c_void_p, C.c_double, _dp, _dp]
        L.orc_fn_set_targets.argtypes = [C.c_void_p, C.c_int, _dp]
        L.orc_fn_set_cweights.argtypes = [C.c_void_p, C.c_int, _dp]
        L.orc_fn_set_weight.argtypes = [C.c_void_p, C.c_int, C.c_double]
        L.orc_fn_set_enabled.argtypes = [C.c_void_p, C.POINTER(C.c_uint8)]
        L.orc_fn_actual_parameters.argtypes = [C.c_void_p]
        L.orc_fn_get_error.restype = C.c_double
        L.orc_fn_get_error.argtypes = [C.c_void_p, _dp]
        L.orc_fn_jacobian_rows.argtypes = [C.c_void_p]
        L.orc_fn_get_jacobian.restype = C.c_double
        L.orc_fn_get_jacobian.argtypes = [C.c_void_p, _dp, _dp, _dp, _ip]
        L.orc_fn_get_jtjr.restype = C.c_double
        L.orc_fn_get_jtjr.argtypes = [C.c_void_p, _dp, _dp, _dp]
        L.orc_fn_fk.argtypes = [C.c_void_p, _dp, _dp, _dp, _dp]
        L.orc_solve.restype = C.c_double
        L.orc_solve.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int, _dp, _ip, _dp]
        L.orc_solve_batch.restype = C.c_double
        L.orc_solve_batch.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int, _dp,
                                      C.POINTER(_dp), C.c_int, _dp, _ip, _dp]
        L.orc_hardware_threads.restype = C.c_int
        L.orc_online_qr.argtypes = [C.c_int, C.c_int, C.c_int, C.c_double, _dp, _dp, C.c_int, _ip, _dp, _dp]
    return L


def _d(a):
    a = np.ascontiguousarray(a, np.float64)
    return a, a.ctypes.data_as(_dp)


def _i(a):
    a = np.ascontiguousarray(a, np.int32)
    return a, a.ctypes.data_as(_ip)


class OracleFunction:
    """Single-instance SkeletonSolverFunctionT<T> + GaussNewtonSolverT<T> restatement.

    ``error_functions`` are the spec objects of momentum_b200.character; per-instance data (targets)
    is taken from batch index ``b`` (default 0) and can be switched with :meth:`select_instance`.
    """

    def __init__(self, character, error_functions: Sequence, dtype: str = "float32", instance: int = 0, native: bool = False):
        # native=True: the -march=native timing build (bench.py CPU arm only); parity checks always use the portable checker build
        L = self._L = native_lib() if native else lib()
        self.ch = character
        self.efs = list(error_functions)
        self.dtype = 0 if dtype in ("float32", "f32", np.float32) else 1
        keep = []
        pa, pp = _i(character.parents)
        of, op = _d(character.offsets)
        pr, prp = _d(character.prerot)
        ou, oup = _i(character.pt_outer)
        inn, inp = _i(character.pt_inner)
        va, vap = _d(character.pt_vals)
        po, pop = _d(character.pt_offsets)
        self.rig = L.orc_rig_create(character.num_joints, pp, op, prp, character.num_params, oup, inp, vap, pop)
        for lim in character.limits:
            ii, ff = lim.packed()
            ia, iap = _i(ii)
            fa, fap = _d(ff)
            L.orc_rig_add_limit(self.rig, int(lim.type), float(lim.weight), iap, fap)
        self.fn = L.orc_fn_create(self.rig, self.dtype)
        for ef in self.efs:
            k = ef.kind
            if k in (0, 1, 2):
                pa, pp = _i(ef.parents)
                cw, cwp = _d(ef.weights)
                inst_off = getattr(ef, "instance_offsets", None)  # offsets per batch element: this oracle object is then tied to `instance`
                of, op = _d(ef.offsets if inst_off is None else np.asarray(inst_off)[instance])
                self.instanced = getattr(self, "instanced", False) or inst_off is not None
                tg, tgp = _d(np.asarray(ef.targets)[instance])
                L.orc_fn_add_joint_ef(self.fn, k, float(ef.weight), float(ef.loss_alpha), float(ef.loss_c), len(ef.parents), pp, cwp, op, tgp)
            elif k == 3:
                pw, pwp = _d(ef.pos_weights)
                rw, rwp = _d(ef.rot_weights)
                tg, tgp = _d(np.asarray(ef.targets)[instance])
                L.orc_fn_add_state_ef(self.fn, float(ef.weight), int(ef.rotation_error_type), float(ef.pos_wgt), float(ef.rot_wgt), pwp, rwp, tgp)
            elif k == 4:
                L.orc_fn_add_limit_ef(self.fn, float(ef.weight), float(ef.loss_alpha), float(ef.loss_c))
            elif k == 5:
                pa, pp = _i(ef.parents)
                cw, cwp = _d(ef.weights)
                of, op = _d(ef.offsets)
                tg, tgp = _d(np.asarray(ef.targets)[instance])
                idx = L.orc_fn_add_joint_ef(self.fn, k, float(ef.weight), float(ef.loss_alpha), float(ef.loss_c), len(ef.parents), pp, cwp, op, tgp)
                L.orc_fn_set_half_plane(self.fn, idx, int(bool(ef.above)))
            elif k == 6:
                tw, twp = _d(ef.target_weights)
                tg, tgp = _d(np.asarray(ef.targets)[instance])
                L.orc_fn_add_model_parameters_ef(self.fn, float(ef.weight), tgp, twp)
            else:
                raise ValueError(k)
        self.n = character.num_params

    def __del__(self):
        try:
            L = self._L
            if getattr(self, "fn", None):
                L.orc_fn_destroy(self.fn)
                self.fn = None
            if getattr(self, "rig", None):
                L.orc_rig_destroy(self.rig)
                self.rig = None
        except Exception:
            pass

    def select_instance(self, b: int):
        L = self._L
        if getattr(self, "instanced", False):
            raise ValueError("error functions with per-instance offsets: build one OracleFunction per instance")
        for idx, ef in enumerate(self.efs):
            if ef.kind in (0, 1, 2, 3, 5, 6):
                tg, tgp = _d(np.asarray(ef.targets)[b])
                L.orc_fn_set_targets(self.fn, idx, tgp)

    def set_enabled_parameters(self, enabled):
        e = np.ascontiguousarray(np.asarray(enabled, bool).astype(np.uint8))
        assert e.size == self.n
        self._L.orc_fn_set_enabled(self.fn, e.ctypes.data_as(C.POINTER(C.c_uint8)))

    @property
    def actual_parameters(self):
        return self._L.orc_fn_actual_parameters(self.fn)

    def get_error(self, params) -> float:
        p, pp = _d(params)
        return self._L.orc_fn_get_error(self.fn, pp)

    def get_jacobian(self, params):
        """Returns (error, J [rows, n] , residual [rows], rows) — J as a numpy (rows x n) view of the
        reference's column-major storage."""
        L = self._L
        rows = L.orc_fn_jacobian_rows(self.fn)
        p, pp = _d(params)
        jac = np.zeros((self.n, rows), np.float64)
        res = np.zeros(rows, np.float64)
        ar = C.c_int(0)
        err = L.orc_fn_get_jacobian(self.fn, pp, jac.ctypes.data_as(_dp), res.ctypes.data_as(_dp), C.byref(ar))
        return err, jac.T, res, ar.value

    def get_jtjr(self, params):
        """(error, JtJ [ap, ap] lower triangle, Jtr [ap]) as solver_function.cpp:74-121."""
        L = self._L
        ap = self.actual_parameters
        p, pp = _d(params)
        H = np.zeros((ap, ap), np.float64)
        g = np.zeros(ap, np.float64)
        err = L.orc_fn_get_jtjr(self.fn, pp, H.ctypes.data_as(_dp), g.ctypes.data_as(_dp))
        return err, H.T, g  # column-major -> numpy [row, col]

    def fk(self, params):
        J = self.ch.num_joints
        p, pp = _d(params)
        xf = np.zeros((J, 8)); ra = np.zeros((J, 9)); ta = np.zeros((J, 9))
        self._L.orc_fn_fk(self.fn, pp, xf.ctypes.data_as(_dp), ra.ctypes.data_as(_dp), ta.ctypes.data_as(_dp))
        # axes returned column-major per joint -> [J, row, col]
        return xf, ra.reshape(J, 3, 3).transpose(0, 2, 1), ta.reshape(J, 3, 3).transpose(0, 2, 1)

    def solve(self, params, *, min_iterations=1, max_iterations=2, threshold=1.0, regularization=0.05, do_line_search=False,
              use_block_jtj=False, subset_solver=False, qr_solver=False, trust_region_qr=False, trust_region_radius=1.0):
        """GaussNewtonSolverT::solve. Returns (error, params, iterations, error_history)."""
        self._L.orc_fn_set_trust_region_radius(self.fn, C.c_double(trust_region_radius))
        p = np.ascontiguousarray(params, np.float64).copy()
        hist = np.zeros(max(1, max_iterations), np.float64)
        it = C.c_int(0)
        err = self._L.orc_solve(self.fn, min_iterations, max_iterations, threshold, regularization, int(do_line_search), int(use_block_jtj),
                              3 if trust_region_qr else (2 if qr_solver else int(subset_solver)), p.ctypes.data_as(_dp), C.byref(it), hist.ctypes.data_as(_dp))
        return err, p, it.value, hist[: it.value].copy()

    def solve_batch(self, params, *, threads=1, min_iterations=1, max_iterations=2, threshold=1.0, regularization=0.05,
                    do_line_search=False, use_block_jtj=False, subset_solver=False, instances: Optional[slice] = None, final_errors=True, qr_solver=False):
        """One solver per instance over ``threads`` host threads (tensor_ik.cpp:127). Returns dict."""
        P = np.ascontiguousarray(params, np.float64).copy()
        B = P.shape[0]
        sl = instances if instances is not None else slice(0, B)
        tg_arrays, ptrs = [], (_dp * len(self.efs))()
        for idx, ef in enumerate(self.efs):
            if ef.kind in (0, 1, 2, 3, 5, 6):
                a = np.ascontiguousarray(np.asarray(ef.targets)[sl], np.float64)
                assert a.shape[0] == B, (a.shape, B)
                tg_arrays.append(a)
                ptrs[idx] = a.ctypes.data_as(_dp)
            else:
                ptrs[idx] = None
        errs = np.zeros(B); fin = np.zeros(B); its = np.zeros(B, np.int32)
        secs = self._L.orc_solve_batch(self.fn, min_iterations, max_iterations, threshold, regularization, int(do_line_search), int(use_block_jtj),
                                     2 if qr_solver else int(subset_solver), B, P.ctypes.data_as(_dp), ptrs, int(threads), errs.ctypes.data_as(_dp),
                                     its.ctypes.data_as(_ip), fin.ctypes.data_as(_dp) if final_errors else None)
        return {"params": P, "errors": errs, "final_errors": fin, "iterations": its, "seconds": secs}


def online_qr(A, b, lam=0.0, chunks=None, dtype="float64"):
    """OnlineHouseholderQR (math/online_householder_qr.cpp): rows of A added chunk by chunk; returns (result(), At_times_b())."""
    A = np.ascontiguousarray(A, np.float64); b = np.ascontiguousarray(b, np.float64)
    rows, n = A.shape
    ch = np.ascontiguousarray(chunks if chunks is not None else [rows], np.int32)
    assert ch.sum() == rows
    x = np.zeros(n); g = np.zeros(n)
    lib().orc_online_qr(0 if dtype == "float32" else 1, rows, n, float(lam), A.ctypes.data_as(_dp), b.ctypes.data_as(_dp), len(ch), ch.ctypes.data_as(_ip),
                        x.ctypes.data_as(_dp), g.ctypes.data_as(_dp))
    return x, g


def hardware_threads() -> int:
    return lib().orc_hardware_threads()
