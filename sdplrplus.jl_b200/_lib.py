"""ctypes binding of libsdplrp_b200.so -- the C-ABI declared in include/sdplrp_b200.h.

This is the Python equivalent of the Julia `ccall` shim (julia/SDPLRPlusB200.jl,
INTEGRATION.md).  There is no CPU fallback: if the shared library is missing the
import fails loudly, and on a machine without a CUDA device `Handle()` raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsdplrp_b200.so")

# ids of include/sdplrp_b200.h
MAT_R, MAT_G, MAT_D, MAT_W0, MAT_W1, MAT_CR, MAT_CD, MAT_S0, MAT_Y0 = 0, 1, 2, 3, 4, 5, 6, 16, 48
(VEC_LAMBDA, VEC_LAMBDA_UB, VEC_B, VEC_PVIO_RAW, VEC_Y, VEC_PVIO_LB, VEC_A_RD, VEC_A_DD, VEC_S_NZVAL,
 VEC_TRIUS_NZVAL) = range(10)
ERR_ASYMMETRIC = -4
ERR_NO_DEVICE = -6

_p_i64 = C.POINTER(C.c_int64)
_p_f64 = C.POINTER(C.c_double)
_p_u8 = C.POINTER(C.c_uint8)
_H = C.c_void_p

BLOCK_TRIPLETS, BLOCK_CSC, BLOCK_DIAG, BLOCK_EDGES, BLOCK_IDENTITY = range(5)


class Block(C.Structure):
    """sdplrp_block (include/sdplrp_b200.h): one structured block of the sparse list."""
    _fields_ = [("kind", C.c_int64), ("on_device", C.c_int64), ("count", C.c_int64), ("first_gid", C.c_int64), ("nnz", C.c_int64),
                ("I", C.c_void_p), ("J", C.c_void_p), ("V", C.c_void_p)]


# name -> argtypes (restype is always int32 unless listed in _SPECIAL)
_SIGNATURES = {
    "sdplrp_nccl_unique_id": [C.c_void_p],
    "sdplrp_create": [C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.POINTER(_H)],
    "sdplrp_destroy": [_H],
    "sdplrp_synchronize": [_H],
    "sdplrp_set_option": [_H, C.c_char_p, C.c_double],
    "sdplrp_preprocess": [_H, C.c_int64, C.c_int64, C.c_int64, _p_i64, _p_i64, _p_i64, _p_f64, _p_i64],
    "sdplrp_preprocess_device": [_H, C.c_int64, C.c_int64, C.c_int64, _p_i64, C.c_void_p, C.c_void_p, C.c_void_p, _p_i64],
    "sdplrp_preprocess_blocks": [_H, C.c_int64, C.c_int64, C.c_int64, C.POINTER(Block)],
    "sdplrp_halo_stats": [_H, _p_i64],
    "sdplrp_pattern_sizes": [_H, _p_i64, _p_i64, _p_i64],
    "sdplrp_value_free_weight": [_H, _p_f64],
    "sdplrp_pattern_export": [_H, _p_i64, _p_i64, _p_i64, _p_i64, _p_f64, _p_f64, _p_i64, _p_i64, _p_i64],
    "sdplrp_add_symlowrank": [_H, C.c_int64, C.c_int64, _p_f64, _p_f64],
    "sdplrp_set_problem": [_H, _p_f64, _p_u8],
    "sdplrp_set_rank": [_H, C.c_int32, C.c_int32],
    "sdplrp_set_sigma": [_H, C.c_double],
    "sdplrp_get_sigma": [_H, _p_f64],
    "sdplrp_get_obj": [_H, _p_f64],
    "sdplrp_upload_mat": [_H, C.c_int32, _p_f64],
    "sdplrp_download_mat": [_H, C.c_int32, _p_f64],
    "sdplrp_upload_mat_slice": [_H, C.c_int32, _p_f64],
    "sdplrp_download_mat_slice": [_H, C.c_int32, _p_f64],
    "sdplrp_upload_vec": [_H, C.c_int32, _p_f64, C.c_int64],
    "sdplrp_download_vec": [_H, C.c_int32, _p_f64, C.c_int64],
    "sdplrp_A_uu": [_H, C.c_int32, _p_f64],
    "sdplrp_A_uv": [_H, C.c_int32, C.c_int32, _p_f64],
    "sdplrp_At_preprocess": [_H, _p_f64],
    "sdplrp_At_left": [_H, C.c_int32, C.c_int32],
    "sdplrp_At_right": [_H, _p_f64, _p_f64, C.c_int64],
    "sdplrp_f": [_H, _p_f64, _p_f64],
    "sdplrp_g": [_H, _p_f64, _p_f64],
    "sdplrp_fg": [_H, _p_f64],
    "sdplrp_lbfgs_dir": [_H, _p_f64],
    "sdplrp_use_gradient_direction": [_H],
    "sdplrp_linesearch_coeffs": [_H, _p_f64],
    "sdplrp_step": [_H, C.c_double, _p_f64],
    "sdplrp_step_g": [_H, C.c_double, _p_f64],
    "sdplrp_lbfgs_update": [_H, C.c_double],
    "sdplrp_lbfgs_clear": [_H],
    "sdplrp_dual_update": [_H],
    "sdplrp_armijo_eval": [_H, _p_f64, C.c_int32, _p_f64, _p_f64],
    "sdplrp_lanczos": [_H, C.c_int64, _p_f64, C.c_uint64, C.c_int32, _p_f64, _p_f64, _p_i64],
    "sdplrp_tridiag_mineig": [_p_f64, _p_f64, C.c_int64, _p_f64],
    "sdplrp_dual_obj": [_H, C.c_double, C.c_int64, _p_f64, C.c_uint64, _p_f64, _p_f64, _p_i64],
    "sdplrp_S_eigval": [_H, C.c_int64, C.c_int64, C.c_double, C.c_int64, _p_f64, C.c_uint64, _p_f64, _p_f64, _p_i64, _p_i64],
    "sdplrp_dual_obj_highprecision": [_H, C.c_double, _p_f64, C.c_uint64, _p_f64, _p_f64, _p_i64],
    "sdplrp_dimacs_errors": [_H, C.c_double, C.c_double, _p_f64, C.c_uint64, _p_f64],
    "sdplrp_dense_symeig": [_p_f64, C.c_int64, _p_f64, _p_f64],
    "sdplrp_set_profiling": [_H, C.c_int32],
    "sdplrp_section_times": [_H, _p_f64, _p_i64],
    "sdplrp_launch_count": [_H, _p_i64],
    "sdplrp_row_range": [_H, _p_i64, _p_i64],
}


class Config(C.Structure):
    """sdplrp_config (include/sdplrp_b200.h): BurerMonteiroConfig with 8-byte fields."""
    _fields_ = ([(k, C.c_double) for k in ("ptol", "gtol", "objtol", "sigma_0", "sigmafac", "maxtime", "printfreq", "fprec",
                                            "prior_trace_bound", "alpha_max")] +
                [(k, C.c_int64) for k in ("maxmajoriter", "maxiter", "numlbfgsvecs", "rankupd_tol", "printlevel", "gtol_relative",
                                           "ptol_relative", "objtol_relative", "eval_DIMACS_errs", "eigval_highprecision")] +
                [("seed", C.c_uint64)])


class Result(C.Structure):
    """sdplrp_result (include/sdplrp_b200.h)."""
    _fields_ = ([(k, C.c_double) for k in ("sigma", "grad_norm", "primal_vio", "obj", "L", "max_dual_value", "min_duality_gap",
                                            "totaltime", "dual_time", "primaltime", "DIMACS_time")] +
                [("DIMACS_errs", C.c_double * 6)] +
                [(k, C.c_int64) for k in ("iter", "majoriter", "lanczos_steps", "r", "status")])


_SIGNATURES.update({
    "sdplrp_config_default": [C.POINTER(Config)],
    "sdplrp_solve": [_H, C.POINTER(Config), C.c_int64, _p_f64, _p_f64, C.c_double, C.c_double, C.POINTER(Result), _p_f64],
    "sdplrp_pick_alpha": [_p_f64, C.c_double, _p_f64, _p_f64],
    "sdplrp_iterate": [_H, C.c_int64, C.c_double, C.c_int32, C.c_int32, _p_f64],
    "sdplrp_fill_uniform": [_H, C.c_int32, C.c_uint64],
    "sdplrp_round_hyperplane": [_H, C.c_int64, _p_f64, C.c_uint64, _p_f64, _p_f64, _p_f64, _p_i64, _p_f64],
    "sdplrp_round_local_search": [_H, C.c_int64, _p_f64, C.c_uint64, C.c_int64, _p_f64, _p_f64, _p_f64, _p_f64, _p_i64, _p_i64, _p_i64,
                                  _p_f64],
})

_SPECIAL = {
    "sdplrp_version": ([], C.c_int32),
    "sdplrp_error_string": ([C.c_int32], C.c_char_p),
    "sdplrp_last_error": ([_H], C.c_char_p),
    "sdplrp_stream": ([_H], C.c_void_p),
}
EXPORTED_SYMBOLS = sorted(list(_SIGNATURES) + list(_SPECIAL))

_lib = None


def load():
    """Load the shared library (built by __graft_entry__.build() / csrc/Makefile)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback for the SDPLRPlus hot path)")
    lib = C.CDLL(LIB_PATH)
    for name, argtypes in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = C.c_int32
    for name, (argtypes, restype) in _SPECIAL.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = restype
    _lib = lib
    return lib


class SdplrpError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"sdplrp error {code}: {message}")
        self.code = code


def _f64(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a, a.ctypes.data_as(_p_f64)


def _i64(a):
    a = np.ascontiguousarray(a, dtype=np.int64)
    return a, a.ctypes.data_as(_p_i64)


class Handle:
    """One GPU's solver context (sdplrp_handle).  Thin, 1:1 with the C ABI."""

    def __init__(self, device=0, rank=0, world=1, nccl_id=None):
        self.lib = load()
        self._h = _H()
        idbuf = None
        if nccl_id is not None:
            idbuf = C.create_string_buffer(bytes(nccl_id), 128)
        rc = self.lib.sdplrp_create(device, rank, world, idbuf, C.byref(self._h))
        if rc != 0:
            self._h = _H()
            raise SdplrpError(rc, self.lib.sdplrp_error_string(rc).decode())
        self.n = self.m = self.r = 0
        self.rank, self.world = rank, world

    # -- plumbing ---------------------------------------------------------
    def _check(self, rc, allow=()):
        if rc != 0 and rc not in allow:
            raise SdplrpError(rc, self.lib.sdplrp_last_error(self._h).decode())
        return rc

    def set_option(self, key, value):
        """Tuning knobs of include/sdplrp_b200.h ("relabel" must be set before preprocess)."""
        self._check(self.lib.sdplrp_set_option(self._h, str(key).encode(), float(value)))

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self.lib.sdplrp_destroy(self._h)
            self._h = _H()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def nccl_unique_id():
        buf = C.create_string_buffer(128)
        rc = load().sdplrp_nccl_unique_id(buf)
        if rc != 0:
            raise SdplrpError(rc, "ncclGetUniqueId failed")
        return buf.raw

    def synchronize(self):
        self._check(self.lib.sdplrp_synchronize(self._h))

    @property
    def stream(self):
        return self.lib.sdplrp_stream(self._h)

    # -- preprocessing ------------------------------------------------------
    def preprocess(self, n, m, mat_off, I1, J1, V, gids1, allow_asymmetric=False):
        mat_off, p_off = _i64(mat_off)
        I1, pI = _i64(I1)
        J1, pJ = _i64(J1)
        V, pV = _f64(V)
        gids1, pG = _i64(gids1)
        nA = len(gids1)
        rc = self.lib.sdplrp_preprocess(self._h, n, m, nA, p_off, pI, pJ, pV, pG)
        self._check(rc, allow=(ERR_ASYMMETRIC,) if allow_asymmetric else ())
        self.n, self.m, self.nA = int(n), int(m), int(nA)
        return rc

    def preprocess_device(self, n, m, mat_off, dI, dJ, dV, gids1, allow_asymmetric=False):
        """sdplrp_preprocess_device: dI / dJ (int64, 1-based) and dV (float64) are CUDA tensors on the handle's GPU (anything
        with data_ptr(), e.g. torch); mat_off / gids1 are host arrays.  The caller's stream must have finished writing them."""
        mat_off, p_off = _i64(mat_off)
        gids1, pG = _i64(gids1)
        nA = len(gids1)
        rc = self.lib.sdplrp_preprocess_device(self._h, n, m, nA, p_off, C.c_void_p(int(dI.data_ptr())), C.c_void_p(int(dJ.data_ptr())),
                                               C.c_void_p(int(dV.data_ptr())), pG)
        self._check(rc, allow=(ERR_ASYMMETRIC,) if allow_asymmetric else ())
        self.n, self.m, self.nA = int(n), int(m), int(nA)
        return rc

    def preprocess_blocks(self, n, m, blocks, allow_asymmetric=False):
        """sdplrp_preprocess_blocks.  `blocks`: list of dicts {kind, first_gid, count=, I=, J=, V=}; the arrays are numpy arrays
        (host) or objects with data_ptr() (device tensors: on_device is set).  For BLOCK_CSC: I = rowval, J = colptr."""
        arr = (Block * len(blocks))()
        keep = []   # the arrays must outlive the call
        nA = 0
        for k, b in enumerate(blocks):
            kind = int(b["kind"])
            dev = False
            ptrs = {}
            sizes = {}
            for name, dt in (("I", np.int64), ("J", np.int64), ("V", np.float64)):
                a = b.get(name)
                if a is None:
                    ptrs[name] = None
                    continue
                if hasattr(a, "data_ptr"):
                    dev = True
                    ptrs[name] = int(a.data_ptr()); sizes[name] = int(a.numel())
                    keep.append(a)
                else:
                    a = np.ascontiguousarray(a, dtype=dt)
                    keep.append(a)
                    ptrs[name] = a.ctypes.data; sizes[name] = int(a.size)
            if kind in (BLOCK_TRIPLETS, BLOCK_CSC):
                count, nnz = 1, sizes.get("V", 0)
            elif kind == BLOCK_IDENTITY:
                count, nnz = 1, 0
            else:
                count = int(b["count"]) if "count" in b else sizes.get("I", 0)
                nnz = 0
            arr[k] = Block(kind, int(dev), count, int(b["first_gid"]), nnz, ptrs["I"], ptrs["J"], ptrs["V"])
            nA += count
        rc = self.lib.sdplrp_preprocess_blocks(self._h, n, m, len(blocks), arr)
        self._check(rc, allow=(ERR_ASYMMETRIC,) if allow_asymmetric else ())
        self.n, self.m, self.nA = int(n), int(m), int(nA)
        return rc

    def pattern_sizes(self):
        a, b, c = C.c_int64(), C.c_int64(), C.c_int64()
        self._check(self.lib.sdplrp_pattern_sizes(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def value_free_weight(self):
        """The weight v the gather pass CD = C*D factors out of C (option "obj_value_free"); 0.0 when it reads C's values."""
        v = C.c_double()
        self._check(self.lib.sdplrp_value_free_weight(self._h, C.byref(v)))
        return v.value

    def pattern_export(self):
        nnzT, nnzF, Ec = self.pattern_sizes()
        n, nA = self.n, self.nA
        out = {
            "triu_colptr": np.zeros(n + 1, np.int64), "triu_rowval": np.zeros(nnzT, np.int64),
            "matptr": np.zeros(nA + 1, np.int64), "nzind": np.zeros(Ec, np.int64),
            "nzval_one": np.zeros(Ec, np.float64), "nzval_two": np.zeros(Ec, np.float64),
            "full_colptr": np.zeros(n + 1, np.int64), "full_rowval": np.zeros(nnzF, np.int64),
            "mapped": np.zeros(nnzF, np.int64),
        }
        order = ["triu_colptr", "triu_rowval", "matptr", "nzind", "nzval_one", "nzval_two", "full_colptr",
                 "full_rowval", "mapped"]
        ptrs = [out[k].ctypes.data_as(_p_f64 if out[k].dtype == np.float64 else _p_i64) for k in order]
        self._check(self.lib.sdplrp_pattern_export(self._h, *ptrs))
        return out

    def add_symlowrank(self, gid1, B, D):
        B = np.asfortranarray(B, dtype=np.float64)
        D = np.ascontiguousarray(D, dtype=np.float64)
        assert B.shape[0] == self.n and B.shape[1] == D.shape[0]
        self._check(self.lib.sdplrp_add_symlowrank(self._h, gid1, B.shape[1], B.ctypes.data_as(_p_f64),
                                                    D.ctypes.data_as(_p_f64)))

    def set_problem(self, b, is_ineq=None):
        b, pb = _f64(b)
        pq = None
        if is_ineq is not None:
            q = np.ascontiguousarray(is_ineq, dtype=np.uint8)
            pq = q.ctypes.data_as(_p_u8)
        self._check(self.lib.sdplrp_set_problem(self._h, pb, pq))

    # -- state ------------------------------------------------------------
    def set_rank(self, r, numlbfgsvecs):
        self._check(self.lib.sdplrp_set_rank(self._h, int(r), int(numlbfgsvecs)))
        self.r, self.hist = int(r), int(numlbfgsvecs)

    @property
    def sigma(self):
        v = C.c_double()
        self._check(self.lib.sdplrp_get_sigma(self._h, C.byref(v)))
        return v.value

    @sigma.setter
    def sigma(self, s):
        self._check(self.lib.sdplrp_set_sigma(self._h, float(s)))

    @property
    def obj(self):
        v = C.c_double()
        self._check(self.lib.sdplrp_get_obj(self._h, C.byref(v)))
        return v.value

    def upload_mat(self, mat_id, Rt):
        """Rt is r x n (Julia column-major == numpy (n, r) C-order)."""
        a = np.ascontiguousarray(Rt, dtype=np.float64)
        assert a.size == self.n * self.r, (a.shape, self.n, self.r)
        self._check(self.lib.sdplrp_upload_mat(self._h, mat_id, a.ctypes.data_as(_p_f64)))

    def upload_mat_slice(self, mat_id, Rt):
        """Several GPUs: rank q reads rows [q*S, (q+1)*S) of the full-size (n, r) array, S = ceil(n / world); the rest comes over NVLink."""
        a = np.ascontiguousarray(Rt, dtype=np.float64)
        assert a.size == self.n * self.r, (a.shape, self.n, self.r)
        self._check(self.lib.sdplrp_upload_mat_slice(self._h, mat_id, a.ctypes.data_as(_p_f64)))

    def download_mat_slice(self, mat_id, out):
        """Several GPUs: rank q writes rows [q*S, (q+1)*S) of the caller's full-size (n, r) array `out`."""
        assert out.flags.c_contiguous and out.dtype == np.float64 and out.size == self.n * self.r
        self._check(self.lib.sdplrp_download_mat_slice(self._h, mat_id, out.ctypes.data_as(_p_f64)))

    def download_mat(self, mat_id):
        """Returns the matrix as a numpy (n, r) C-order array (== Julia r x n column-major)."""
        a = np.empty((self.n, self.r), np.float64)
        self._check(self.lib.sdplrp_download_mat(self._h, mat_id, a.ctypes.data_as(_p_f64)))
        return a

    def upload_vec(self, vec_id, v):
        v, p = _f64(v)
        self._check(self.lib.sdplrp_upload_vec(self._h, vec_id, p, v.size))

    def download_vec(self, vec_id, length):
        a = np.empty(length, np.float64)
        self._check(self.lib.sdplrp_download_vec(self._h, vec_id, a.ctypes.data_as(_p_f64), length))
        return a

    # -- operators ----------------------------------------------------------
    def A_uu(self, U_id=MAT_R):
        out = np.empty(self.m + 1, np.float64)
        self._check(self.lib.sdplrp_A_uu(self._h, U_id, out.ctypes.data_as(_p_f64)))
        return out

    def A_uv(self, U_id, V_id):
        out = np.empty(self.m + 1, np.float64)
        self._check(self.lib.sdplrp_A_uv(self._h, U_id, V_id, out.ctypes.data_as(_p_f64)))
        return out

    def At_preprocess(self, y=None):
        if y is None:
            self._check(self.lib.sdplrp_At_preprocess(self._h, None))
        else:
            y, p = _f64(y)
            assert y.size == self.m + 1
            self._check(self.lib.sdplrp_At_preprocess(self._h, p))

    def At_left(self, X_id, Y_id):
        self._check(self.lib.sdplrp_At_left(self._h, X_id, Y_id))

    def At_right(self, x):
        """x: (n,) or (n, ncols) -> S @ x (+ low rank)."""
        x = np.asarray(x, np.float64)
        one = x.ndim == 1
        x2 = np.asfortranarray(x.reshape(-1, 1) if one else x)
        assert x2.shape[0] == self.n
        y = np.empty(x2.shape, np.float64, order="F")
        self._check(self.lib.sdplrp_At_right(self._h, x2.ctypes.data_as(_p_f64), y.ctypes.data_as(_p_f64), x2.shape[1]))
        return y[:, 0] if one else y

    # -- fused iteration ------------------------------------------------------
    def f(self):
        L, obj = C.c_double(), C.c_double()
        self._check(self.lib.sdplrp_f(self._h, C.byref(L), C.byref(obj)))
        return L.value, obj.value

    def g(self):
        a, b = C.c_double(), C.c_double()
        self._check(self.lib.sdplrp_g(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def fg(self):
        out = (C.c_double * 4)()
        self._check(self.lib.sdplrp_fg(self._h, out))
        return out[0], out[1], out[2], out[3]

    def lbfgs_dir(self):
        d = C.c_double()
        self._check(self.lib.sdplrp_lbfgs_dir(self._h, C.byref(d)))
        return d.value

    def use_gradient_direction(self):
        self._check(self.lib.sdplrp_use_gradient_direction(self._h))

    def linesearch_coeffs(self):
        out = (C.c_double * 5)()
        self._check(self.lib.sdplrp_linesearch_coeffs(self._h, out))
        return np.array(out[:], dtype=np.float64)

    def step(self, alpha, want_obj=True):
        o = C.c_double()
        self._check(self.lib.sdplrp_step(self._h, float(alpha), C.byref(o) if want_obj else None))
        return o.value

    def step_g(self, alpha):
        """step + g in one call -> (obj, ||G||_F^2, ||pvio||_2^2)"""
        out = (C.c_double * 3)()
        self._check(self.lib.sdplrp_step_g(self._h, float(alpha), out))
        return out[0], out[1], out[2]

    def lbfgs_update(self, alpha):
        self._check(self.lib.sdplrp_lbfgs_update(self._h, float(alpha)))

    def lbfgs_clear(self):
        self._check(self.lib.sdplrp_lbfgs_clear(self._h))

    def dual_update(self):
        self._check(self.lib.sdplrp_dual_update(self._h))

    def armijo_eval(self, alphas):
        a, pa = _f64(alphas)
        L = np.empty(a.size, np.float64)
        s = C.c_double()
        self._check(self.lib.sdplrp_armijo_eval(self._h, pa, a.size, L.ctypes.data_as(_p_f64), C.byref(s)))
        return L, s.value

    # -- dual bound -----------------------------------------------------------
    def lanczos(self, q, v0=None, seed=0, reorth=False):
        q = int(max(1, min(q, self.n - 1)))
        alpha, beta = np.zeros(q), np.zeros(q)
        iters = C.c_int64()
        pv = None
        if v0 is not None:
            v0, pv = _f64(v0)
            assert v0.size == self.n
        self._check(self.lib.sdplrp_lanczos(self._h, q, pv, int(seed), int(bool(reorth)), alpha.ctypes.data_as(_p_f64),
                                             beta.ctypes.data_as(_p_f64), C.byref(iters)))
        return alpha, beta, iters.value

    def dual_obj(self, trace_bound, it, v0=None, seed=0):
        d, e, s = C.c_double(), C.c_double(), C.c_int64()
        pv = None
        if v0 is not None:
            v0, pv = _f64(v0)
        self._check(self.lib.sdplrp_dual_obj(self._h, float(trace_bound), int(it), pv, int(seed), C.byref(d), C.byref(e),
                                              C.byref(s)))
        return d.value, e.value, s.value

    def S_eigval(self, nevs=1, ncv=None, tol=0.0, maxiter=10 ** 6, v0=None, seed=0):
        """SDP_S_eigval(var, aux, nevs, true; which=:SA, ncv, tol, maxiter) on the S last assembled ->
        (eigenvalues ascending, residual bounds, matvecs, restarts)"""
        ncv = min(100, self.n) if ncv is None else int(ncv)
        ev, bd = np.zeros(int(nevs)), np.zeros(int(nevs))
        mv, rs = C.c_int64(), C.c_int64()
        pv = None
        if v0 is not None:
            v0, pv = _f64(v0)
            assert v0.size == self.n
        self._check(self.lib.sdplrp_S_eigval(self._h, int(nevs), ncv, float(tol), int(maxiter), pv, int(seed),
                                              ev.ctypes.data_as(_p_f64), bd.ctypes.data_as(_p_f64), C.byref(mv), C.byref(rs)))
        return ev, bd, mv.value, rs.value

    def dual_obj_highprecision(self, trace_bound, v0=None, seed=0):
        d, e, s = C.c_double(), C.c_double(), C.c_int64()
        pv = None
        if v0 is not None:
            v0, pv = _f64(v0)
        self._check(self.lib.sdplrp_dual_obj_highprecision(self._h, float(trace_bound), pv, int(seed), C.byref(d), C.byref(e),
                                                            C.byref(s)))
        return d.value, e.value, s.value

    def dimacs_errors(self, normb, normC, v0=None, seed=0):
        errs = np.zeros(6)
        pv = None
        if v0 is not None:
            v0, pv = _f64(v0)
        self._check(self.lib.sdplrp_dimacs_errors(self._h, float(normb), float(normC), pv, int(seed), errs.ctypes.data_as(_p_f64)))
        return errs

    def iterate(self, k, alpha_max=1.0, use_armijo=False, update_history=True):
        """k inner iterations inside the library -> (L, obj, ||G||^2, ||pvio||^2, alpha) of the last one"""
        out = (C.c_double * 5)()
        self._check(self.lib.sdplrp_iterate(self._h, int(k), float(alpha_max), int(bool(use_armijo)), int(bool(update_history)), out))
        return tuple(out)

    def fill_uniform(self, mat_id, seed):
        """mat <- U(-1,1) from the counter-based device generator (same matrix for any GPU count / vertex order)"""
        self._check(self.lib.sdplrp_fill_uniform(self._h, int(mat_id), int(seed)))

    def round_hyperplane(self, K, G=None, seed=0):
        """sdplrp_round_hyperplane: K hyperplane roundings x_k = sign(R g_k) of the current R ->
        dict(obj (K,), sum (K,), best (0-based), best_x (n,) of +-1.0, G_used (K, r))"""
        K = int(K)
        pg = None
        if G is not None:
            G, pg = _f64(G)
            assert G.size == K * self.r, (G.shape, K, self.r)
        G_used = np.empty((K, self.r), np.float64)
        obj, tot, x = np.empty(K), np.empty(K), np.empty(self.n)
        best = C.c_int64()
        self._check(self.lib.sdplrp_round_hyperplane(self._h, K, pg, int(seed), G_used.ctypes.data_as(_p_f64), obj.ctypes.data_as(_p_f64),
                                                      tot.ctypes.data_as(_p_f64), C.byref(best), x.ctypes.data_as(_p_f64)))
        return {"obj": obj, "sum": tot, "best": best.value - 1, "best_x": x, "G_used": G_used}

    def round_local_search(self, K, G=None, seed=0, max_rounds=1000):
        """sdplrp_round_local_search: the K hyperplane roundings of round_hyperplane, each refined by one-flip descent ->
        dict(obj_round (K,) before the descent, obj (K,), sum (K,), flips (K,), rounds (K,; -1 = stopped by max_rounds),
        best (0-based), best_x (n,) of +-1.0, G_used (K, r))"""
        K = int(K)
        pg = None
        if G is not None:
            G, pg = _f64(G)
            assert G.size == K * self.r, (G.shape, K, self.r)
        G_used = np.empty((K, self.r), np.float64)
        obj0, obj, tot, x = np.empty(K), np.empty(K), np.empty(K), np.empty(self.n)
        flips, rounds = np.empty(K, np.int64), np.empty(K, np.int64)
        best = C.c_int64()
        self._check(self.lib.sdplrp_round_local_search(
            self._h, K, pg, int(seed), int(max_rounds), G_used.ctypes.data_as(_p_f64), obj0.ctypes.data_as(_p_f64),
            obj.ctypes.data_as(_p_f64), tot.ctypes.data_as(_p_f64), flips.ctypes.data_as(_p_i64), rounds.ctypes.data_as(_p_i64),
            C.byref(best), x.ctypes.data_as(_p_f64)))
        return {"obj_round": obj0, "obj": obj, "sum": tot, "flips": flips, "rounds": rounds, "best": best.value - 1, "best_x": x,
                "G_used": G_used}

    def solve(self, cfg, r, Rt0=None, lambda0=None, normb=1.0, normC=1.0):
        """sdplrp_solve: the native outer loop -> (Result, best_lambda[m+1])"""
        pr = pl = None
        if Rt0 is not None:
            Rt0, pr = _f64(Rt0)
            assert Rt0.size == self.n * int(r)
        if lambda0 is not None:
            lambda0, pl = _f64(lambda0)
            assert lambda0.size == self.m
        res = Result()
        best = np.zeros(self.m + 1)
        self._check(self.lib.sdplrp_solve(self._h, C.byref(cfg), int(r), pr, pl, float(normb), float(normC), C.byref(res),
                                           best.ctypes.data_as(_p_f64)))
        self.r = int(res.r)
        return res, best

    SECTIONS = ["lbfgs_dir", "ls_pass", "ls_coeff", "step", "s_assemble", "spmm", "norms", "lbfgs_update", "a_uu", "f_finish",
                "lanczos", "comm", "grad", "tail"]

    def set_profiling(self, on):
        self._check(self.lib.sdplrp_set_profiling(self._h, int(bool(on))))

    def section_times(self):
        """{section: (milliseconds, count)} accumulated since the last call (CUDA events on the handle's stream)."""
        k = len(self.SECTIONS)
        ms = np.zeros(k); cnt = np.zeros(k, np.int64)
        self._check(self.lib.sdplrp_section_times(self._h, ms.ctypes.data_as(_p_f64), cnt.ctypes.data_as(_p_i64)))
        return {name: (float(ms[i]), int(cnt[i])) for i, name in enumerate(self.SECTIONS)}

    def launch_count(self):
        c = C.c_int64()
        self._check(self.lib.sdplrp_launch_count(self._h, C.byref(c)))
        return c.value

    def halo_stats(self):
        a = np.zeros(7, np.int64)
        self._check(self.lib.sdplrp_halo_stats(self._h, a.ctypes.data_as(_p_i64)))
        return dict(zip(("active", "own_rows", "own_nnz", "hub_ghosts", "tail_ghosts", "hub_rows_sent", "tail_rows_sent"), (int(x) for x in a)))

    def row_range(self):
        lo, hi = C.c_int64(), C.c_int64()
        self._check(self.lib.sdplrp_row_range(self._h, C.byref(lo), C.byref(hi)))
        return lo.value, hi.value


def tridiag_mineig(d, e):
    d, pd = _f64(d)
    e, pe = _f64(e if len(e) else np.zeros(1))
    out = C.c_double()
    rc = load().sdplrp_tridiag_mineig(pd, pe, d.size, C.byref(out))
    if rc != 0:
        raise SdplrpError(rc, "tridiag_mineig: bad argument")
    return out.value


def dense_symeig(A):
    """Ascending eigenvalues and eigenvectors (columns) of a small dense symmetric matrix (host helper of the ABI)."""
    A, pa = _f64(A)
    k = A.shape[0]
    ev, Q = np.zeros(k), np.zeros((k, k))
    rc = load().sdplrp_dense_symeig(pa, k, ev.ctypes.data_as(_p_f64), Q.ctypes.data_as(_p_f64))
    if rc != 0:
        raise SdplrpError(rc, "dense_symeig: bad argument")
    return ev, Q


def default_config():
    cfg = Config()
    rc = load().sdplrp_config_default(C.byref(cfg))
    if rc != 0:
        raise SdplrpError(rc, "config_default")
    return cfg


def pick_alpha_native(bq, alpha_max=1.0):
    """sdplrp_pick_alpha: root selection of linesearch! on the host (C++); raises ArithmeticError like the reference."""
    bq, pb = _f64(bq)
    a, v = C.c_double(), C.c_double()
    rc = load().sdplrp_pick_alpha(pb, float(alpha_max), C.byref(a), C.byref(v))
    if rc == -7:
        raise ArithmeticError(f"Error: cubic[1] = {bq[1]} should be less than 0.")
    if rc != 0:
        raise SdplrpError(rc, "pick_alpha: bad argument")
    return a.value, v.value
