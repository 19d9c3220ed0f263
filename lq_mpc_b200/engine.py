"""ctypes binding of the C ABI in include/lqmpc_b200.h + a thin tensor-level wrapper.

PyTorch is used here only for device memory, streams and (elsewhere) torch.distributed; every computation is done
by the hand-written sm_100a kernels in `_lib/liblqmpc_b200.so`.  There is NO CPU path: if the library or a CUDA
device is missing, every entry point raises.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LQMPC_LIB") or os.path.join(_PKG, "_lib", "liblqmpc_b200.so")   # LQMPC_LIB: A/B builds (scripts/unit_variants.sh)

FLAG_UNSTABLE = 1
FLAG_QP_ACTIVE = 2
FLAG_QP_MAXITER = 4
FLAG_DARE_NOCONV = 8
FLAG_NONFINITE = 16
FLAG_BOUND_INVALID = 32
FLAG_LYAP_NOCONV = 64
FLAG_EIG_NOCONV = 128
FLAG_CHOL_FAIL = 256
FLAG_DOMAIN_ERROR = 512
FLAG_TAIL_UNCERTIFIED = 1024
FLAG_ASCENT_MAXITER = 2048

WORST_NORMS = {"f": 0, "2": 1, "max": 2}   # norm_type of lqmpc_worst_case_batch / lqmpc_worst_case_sup_batch

RADIX_MAX_SEL = 32          # LQMPC_RADIX_MAX_SEL: selectors per lqmpc_column_radix_histogram call

_c_double_p = ctypes.POINTER(ctypes.c_double)
_c_int32_p = ctypes.POINTER(ctypes.c_int32)
_vp = ctypes.c_void_p
_i64 = ctypes.c_int64
_int = ctypes.c_int

# name -> (restype, argtypes); the single source of truth for the symbols include/lqmpc_b200.h declares
ABI = {
    "lqmpc_abi_version": (_int, []),
    "lqmpc_supported_dims": (ctypes.c_char_p, []),
    "lqmpc_create": (_int, [ctypes.POINTER(_vp), _int, _vp]),
    "lqmpc_destroy": (None, [_vp]),
    "lqmpc_last_error": (ctypes.c_char_p, [_vp]),
    "lqmpc_sync": (_int, [_vp]),
    "lqmpc_set_problem": (_int, [_vp, _int, _int] + [_vp] * 7 + [_int]),
    "lqmpc_get_prepared": (_int, [_vp, _vp, _i64]),
    "lqmpc_eval_batch": (_int, [_vp, _i64, _vp, _vp, _vp, _int, _int, _int] + [_vp] * 7),
    "lqmpc_eval_seeded": (_int, [_vp, ctypes.c_uint64, _i64, _i64, ctypes.c_double, ctypes.c_double, _int, _int] + [_vp] * 5),
    "lqmpc_eval_batch_host": (_int, [_vp, _i64, _vp, _vp, _vp, _int, _int, _int, _vp, _vp, _vp, _vp, _i64]),
    "lqmpc_set_problem_tiled": (_int, [_vp, _int, _int] + [_vp] * 5 + [_int]),
    "lqmpc_get_prepared_tiled": (_int, [_vp, _vp, _i64]),
    "lqmpc_eval_batch_tiled": (_int, [_vp, _i64, _vp, _vp, _vp, _int, _int] + [_vp] * 5),
    "lqmpc_eval_batch_tiled_host": (_int, [_vp, _i64, _vp, _vp, _vp, _int, _int, _vp, _vp, _vp, _vp, _i64]),
    "lqmpc_set_references": (_int, [_vp, _int, _vp, _vp]),
    "lqmpc_set_input_polytope": (_int, [_vp, _int, _vp]),
    "lqmpc_mpc_solve_batch": (_int, [_vp, _i64, _vp, _vp, _int, _int] + [_vp] * 6),
    "lqmpc_simulate_batch": (_int, [_vp, _i64, _vp, _vp, _int, _int] + [_vp] * 7),
    "lqmpc_simulate_inf_batch": (_int, [_vp, _i64, _vp, _vp, _int, _int] + [_vp] * 5),
    "lqmpc_eval_grad_batch": (_int, [_vp, _i64, _vp, _vp, _vp, _int] + [_vp] * 6),
    "lqmpc_worst_case_batch": (_int, [_vp, _i64, _vp, _vp, _vp, _int, ctypes.c_double, ctypes.c_double, _int, _int,
                                      ctypes.c_double] + [_vp] * 7),
    "lqmpc_ratio_sup_batch": (_int, [_vp, _i64, _vp, _vp, _int] + [_vp] * 7),
    "lqmpc_worst_case_sup_batch": (_int, [_vp, _i64, _vp, _vp, _int, ctypes.c_double, ctypes.c_double, _int, _int,
                                          ctypes.c_double] + [_vp] * 7),
    "lqmpc_simulate_inf_grad_batch": (_int, [_vp, _i64, _vp, _vp, _int, _int] + [_vp] * 8),
    "lqmpc_worst_case_inf_batch": (_int, [_vp, _i64, _vp, _vp, _int, _int, _vp, _vp, ctypes.c_double, ctypes.c_double,
                                          _int, _int, ctypes.c_double] + [_vp] * 7),
    "lqmpc_bounds_fields": (_int, []),
    "lqmpc_bounds_batch": (_int, [_vp, _i64, _vp, _vp, _int, _vp, _vp, ctypes.c_double, ctypes.c_double, _vp,
                                  ctypes.c_double, _vp, _vp, _vp, _vp, _vp, ctypes.c_double, ctypes.c_double,
                                  ctypes.c_double, _int] + [_vp] * 9),
    "lqmpc_mpc_solve_range": (_int, [_vp, _i64, _vp, _vp, _int, _int, _int] + [_vp] * 6),
    "lqmpc_bounds_range": (_int, [_vp, _i64, _vp, _vp, _int, _int, _vp, _vp, ctypes.c_double, ctypes.c_double, _vp,
                                  ctypes.c_double, _vp, _vp, _vp, _vp, _vp, ctypes.c_double, ctypes.c_double,
                                  ctypes.c_double, _int] + [_vp] * 9),
    "lqmpc_dlqr_batch": (_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "lqmpc_column_stats": (_int, [_vp, _vp, _int, _i64, _i64, _vp]),
    "lqmpc_column_sqdev": (_int, [_vp, _vp, _int, _i64, _i64, _vp, _vp]),
    "lqmpc_column_moments": (_int, [_vp, _vp, _int, _i64, _i64, _vp]),
    "lqmpc_column_radix_histogram": (_int, [_vp, _vp, _int, _i64, _i64, _int, _int, _vp, _vp]),
    "lqmpc_column_radix_select": (_int, [_vp, _vp, _int, _int, _int, _vp, _vp]),
    "lqmpc_column_argext": (_int, [_vp, _vp, _int, _i64, _i64, _i64, _vp, _vp]),
    "lqmpc_sample_error_grid": (_int, [_vp, ctypes.c_uint64, _int, _int, _int, _i64, _i64, _int, _vp, _i64, _int, _vp,
                                       _vp]),
    "lqmpc_fp64_peak": (_int, [_vp, _c_double_p]),
    "lqmpc_fp64_tensor_peak": (_int, [_vp, _c_double_p]),
    "lqmpc_launch_count": (_i64, [_vp]),
}

# order of `enum BoundField` in csrc/bounds.cuh (rows of the `detail` output of lqmpc_bounds_batch)
BOUND_FIELDS = ['alpha', 'beta', 'xi', 'eta', 'bound', 'E_psi', 'E_u', 'E_psi_u', 'theta_u', 'theta_x_u', 'C_K',
                'rho_K', 'gamma', 'rho_gamma', 'L_V', 'N_0', 'omega_N1', 'omega_N0d5', 'err_th', 'N_min', 'h',
                'epsilon_K', 'norm_A', 'norm_B', 'norm_K', 'norm_Gamma', 'norm_Phi', 'min_H', 'rho_cl', 'bar_u',
                'bar_d_u']

_lib = None


class EngineError(RuntimeError):
    pass


def load_library(path: Optional[str] = None):
    """dlopen the engine and bind every ABI symbol. Raises (never falls back) when the library is missing."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise EngineError(
            "lq_mpc_b200: CUDA engine %s not built (run `python -c 'import __graft_entry__ as g; g.build()'`). "
            "There is no CPU fallback." % p)
    lib = ctypes.CDLL(p)
    for name, (res, args) in ABI.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing: loud by design
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib


def _np_f64(a, shape=None):
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float64))
    if shape is not None:
        a = a.reshape(shape)
    return a


def _ptr(t):
    """Device/host pointer of a torch tensor or numpy array (None -> NULL)."""
    if t is None:
        return None
    if isinstance(t, np.ndarray):
        return t.ctypes.data
    return t.data_ptr()


def _streamed(fn):
    """Run a public Engine method with the engine's stream as torch's CURRENT stream: staging copies (`_dev`), output
    allocations (caching-allocator stream ownership) and the kernels the C ABI enqueues then share one stream order,
    whichever stream the Engine was created on."""
    import functools

    @functools.wraps(fn)
    def wrapper(self, *a, **k):
        with self.torch.cuda.stream(self._stream):
            return fn(self, *a, **k)
    return wrapper


class Engine:
    """One engine context per (device, stream). Not thread-safe."""

    def __init__(self, device: int = 0, stream=None):
        import torch
        if not torch.cuda.is_available():
            raise EngineError("lq_mpc_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.torch = torch
        self.lib = load_library()
        self.device = torch.device("cuda", device)
        torch.cuda.set_device(self.device)
        torch.zeros(1, device=self.device)  # make sure the primary context exists
        self._stream = stream if stream is not None else torch.cuda.current_stream(self.device)
        h = _vp()
        rc = self.lib.lqmpc_create(ctypes.byref(h), device, _vp(self._stream.cuda_stream))
        if rc != 0:
            raise EngineError("lqmpc_create failed with code %d" % rc)
        self._h = h
        self.n = self.m = 0

    # ------------------------------------------------------------------------------------------------ plumbing
    def close(self):
        if getattr(self, "_h", None):
            self.lib.lqmpc_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            msg = self.lib.lqmpc_last_error(self._h)
            raise EngineError("%s failed (%d): %s" % (what, rc, msg.decode() if msg else ""))

    def sync(self):
        self._check(self.lib.lqmpc_sync(self._h), "lqmpc_sync")

    @property
    def launch_count(self) -> int:
        return int(self.lib.lqmpc_launch_count(self._h))

    def supported_dims(self):
        return [tuple(int(v) for v in s.split("x")) for s in self.lib.lqmpc_supported_dims().decode().split(",")]

    def _dev(self, a):
        """numpy / tensor -> contiguous float64 CUDA tensor on this engine's device."""
        torch = self.torch
        if isinstance(a, torch.Tensor):
            t = a.to(device=self.device, dtype=torch.float64)
        else:
            t = torch.from_numpy(_np_f64(a)).to(self.device)
        return t.contiguous()

    # ------------------------------------------------------------------------------------------------ problem
    def set_problem(self, A, B, Q, R, P=None, u_lo=None, u_hi=None, N_opc: int = 30):
        A = _np_f64(A)
        n = A.shape[0]
        B = _np_f64(B, (n, -1))
        m = B.shape[1]
        Q = _np_f64(Q, (n, n))
        R = _np_f64(R, (m, m))
        P = Q if P is None else _np_f64(P, (n, n))
        lo = None if u_lo is None else _np_f64(u_lo, (m,))
        hi = None if u_hi is None else _np_f64(u_hi, (m,))
        rc = self.lib.lqmpc_set_problem(self._h, n, m, _ptr(A), _ptr(B), _ptr(Q), _ptr(R), _ptr(P), _ptr(lo),
                                        _ptr(hi), int(N_opc))
        self._check(rc, "lqmpc_set_problem")
        self._poly_bar = None                       # lqmpc_set_problem clears an installed input polytope
        self.n, self.m = n, m
        self.A, self.B, self.Q, self.R, self.P = A, B, Q, R, P
        self.u_lo, self.u_hi = lo, hi
        self.N_opc = int(N_opc)
        return self

    # ------------------------------------------------------------------------------------------------ K4
    TILED_DIMS = ((32, 8), (16, 4))

    @_streamed
    def set_problem_tiled(self, A, B, Q, R, P=None, N_opc: int = 30):
        """Large-n path (K4; n x m in TILED_DIMS): unconstrained law, array-of-matrices operands."""
        A = _np_f64(A)
        n = A.shape[0]
        B = _np_f64(B, (n, -1))
        m = B.shape[1]
        Q = _np_f64(Q, (n, n))
        R = _np_f64(R, (m, m))
        P = Q if P is None else _np_f64(P, (n, n))
        rc = self.lib.lqmpc_set_problem_tiled(self._h, n, m, _ptr(A), _ptr(B), _ptr(Q), _ptr(R), _ptr(P), int(N_opc))
        self._check(rc, "lqmpc_set_problem_tiled")
        self.tn, self.tm = n, m
        return self

    def prepared_tiled(self):
        out = np.zeros(self.tn * self.tn)
        self._check(self.lib.lqmpc_get_prepared_tiled(self._h, _ptr(out), out.size), "lqmpc_get_prepared_tiled")
        return {"Pexp": out.reshape(self.tn, self.tn)}

    @_streamed
    def eval_batch_tiled(self, dA, dB, x0, N_min: int, N_max: int, want=("J", "rho", "ratio", "flags")):
        """dA [S][n][n], dB [S][n][m], x0 [S][n] (array of matrices, device or host). Returns [H][S] device tensors
        plus the contiguous `table` like eval_batch."""
        torch = self.torch
        n, m = self.tn, self.tm
        dA, dB, x0 = self._dev(dA), self._dev(dB), self._dev(x0)
        S = x0.shape[0]
        if dA.numel() != n * n * S or dB.numel() != n * m * S or x0.numel() != n * S:
            raise ValueError("operand shapes do not match (n, m, S)")
        H = N_max - N_min + 1
        names = [k for k in ("J", "rho", "ratio", "V_N") if k in want]
        table = torch.empty((len(names) * H, S), dtype=torch.float64, device=self.device)
        out = {k: table[i * H:(i + 1) * H] for i, k in enumerate(names)}
        out["table"], out["table_rows"] = table, [(k, N_min + h) for k in names for h in range(H)]
        if "flags" in want:
            out["flags"] = torch.empty((H, S), dtype=torch.int32, device=self.device)
        rc = self.lib.lqmpc_eval_batch_tiled(self._h, S, _ptr(dA), _ptr(dB), _ptr(x0), N_min, N_max,
                                             _ptr(out.get("J")), _ptr(out.get("rho")), _ptr(out.get("ratio")),
                                             _ptr(out.get("V_N")), _ptr(out.get("flags")))
        self._check(rc, "lqmpc_eval_batch_tiled")
        return out

    @_streamed
    def eval_batch_tiled_host(self, dA, dB, x0, N_min: int, N_max: int, out=None, chunk: int = 16384):
        """eval_batch_tiled from/to HOST buffers (numpy arrays or CPU tensors [S][n*n] ..., ideally pinned), chunked
        with copies overlapping the kernels. `out` may hold preallocated host tensors J/rho/ratio/flags [H][S]."""
        torch = self.torch
        S = x0.shape[0]
        H = N_max - N_min + 1
        if out is None:
            out = {"J": torch.empty((H, S), dtype=torch.float64).pin_memory(),
                   "rho": torch.empty((H, S), dtype=torch.float64).pin_memory(),
                   "ratio": torch.empty((H, S), dtype=torch.float64).pin_memory(),
                   "flags": torch.empty((H, S), dtype=torch.int32).pin_memory()}
        rc = self.lib.lqmpc_eval_batch_tiled_host(self._h, S, _ptr(dA), _ptr(dB), _ptr(x0), N_min, N_max,
                                                  _ptr(out.get("J")), _ptr(out.get("rho")), _ptr(out.get("ratio")),
                                                  _ptr(out.get("flags")), chunk)
        self._check(rc, "lqmpc_eval_batch_tiled_host")
        return out

    def prepared(self):
        n = self.n
        out = np.zeros(2 * n * n + 4)
        self._check(self.lib.lqmpc_get_prepared(self._h, _ptr(out), out.size), "lqmpc_get_prepared")
        return {"Pexp": out[:n * n].reshape(n, n).copy(), "Qinv": out[n * n:2 * n * n].reshape(n, n).copy(),
                "maxQ": out[2 * n * n], "minQ": out[2 * n * n + 1], "maxR": out[2 * n * n + 2],
                "minR": out[2 * n * n + 3]}

    # ------------------------------------------------------------------------------------------------ K1
    @_streamed
    def eval_batch(self, dA, dB, x0, N_min: int, N_max: int, T: int = 0, want=("J", "rho", "ratio", "flags")):
        """dA [n*n][S], dB [n*m][S], x0 [n][S] (SoA, device). Returns dict of [H][S] device tensors."""
        torch = self.torch
        n, m = self.n, self.m
        dA, dB, x0 = self._dev(dA), self._dev(dB), self._dev(x0)
        S = dA.shape[-1]
        if dA.numel() != n * n * S or dB.numel() != n * m * S or x0.numel() != n * S:
            raise ValueError("operand shapes do not match (n, m, S)")
        H = N_max - N_min + 1
        out = {}
        names = [k for k in ("J", "rho", "ratio", "V_N", "J_T") if k in want]
        # one allocation: out["table"] is the column-contiguous [len(names)*H][S] result table K5 reduces directly
        table = torch.empty((len(names) * H, S), dtype=torch.float64, device=self.device)
        for i, k in enumerate(names):
            out[k] = table[i * H:(i + 1) * H]
        out["table"], out["table_rows"] = table, [(k, N_min + h) for k in names for h in range(H)]
        if "flags" in want:
            out["flags"] = torch.empty((H, S), dtype=torch.int32, device=self.device)
        if "K0" in want:
            out["K0"] = torch.empty((H, m * n, S), dtype=torch.float64, device=self.device)
        rc = self.lib.lqmpc_eval_batch(self._h, S, _ptr(dA), _ptr(dB), _ptr(x0), N_min, N_max, T,
                                       _ptr(out.get("J")), _ptr(out.get("rho")), _ptr(out.get("ratio")),
                                       _ptr(out.get("V_N")), _ptr(out.get("J_T")), _ptr(out.get("flags")),
                                       _ptr(out.get("K0")))
        self._check(rc, "lqmpc_eval_batch")
        return out

    @_streamed
    def eval_seeded(self, seed: int, first: int, S: int, e_A: float, e_B: float, N_min: int, N_max: int,
                    want=("moments",)):
        """K1 on seeded synthetic samples drawn in the kernel (global sample indices [first, first + S)).
        want: any of "J", "rho", "ratio", "flags" (device tensors [H][S]; J/rho/ratio are rows of one `table`) and
        "moments" (device [3H][6]: max, min, n_finite, n_nonfinite, mean, M2 per column of {J, rho, ratio})."""
        torch = self.torch
        H = N_max - N_min + 1
        out = {}
        tables = any(k in want for k in ("J", "rho", "ratio"))
        if tables:
            table = torch.empty((3 * H, S), dtype=torch.float64, device=self.device)
            out["table"] = table
            out["J"], out["rho"], out["ratio"] = table[:H], table[H:2 * H], table[2 * H:]
        if "flags" in want:
            out["flags"] = torch.empty((H, S), dtype=torch.int32, device=self.device)
        if "moments" in want:
            out["moments"] = torch.empty((3 * H, 6), dtype=torch.float64, device=self.device)
        rc = self.lib.lqmpc_eval_seeded(self._h, int(seed), int(first), int(S), float(e_A), float(e_B), N_min, N_max,
                                        _ptr(out.get("J")), _ptr(out.get("rho")), _ptr(out.get("ratio")),
                                        _ptr(out.get("flags")), _ptr(out.get("moments")))
        self._check(rc, "lqmpc_eval_seeded")
        return out

    @_streamed
    def eval_batch_host(self, dA, dB, x0, N_min: int, N_max: int, out=None, chunk: int = 1 << 20):
        """Same as eval_batch but from/to HOST buffers (numpy arrays or CPU tensors, ideally pinned), pipelined in
        chunks with copies overlapping compute. `out` may hold preallocated host arrays J/rho/ratio/flags [H][S]."""
        torch = self.torch
        n, m = self.n, self.m
        S = dA.shape[-1]
        H = N_max - N_min + 1
        if out is None:
            out = {"J": torch.empty((H, S), dtype=torch.float64).pin_memory(),
                   "rho": torch.empty((H, S), dtype=torch.float64).pin_memory(),
                   "ratio": torch.empty((H, S), dtype=torch.float64).pin_memory(),
                   "flags": torch.empty((H, S), dtype=torch.int32).pin_memory()}
        rc = self.lib.lqmpc_eval_batch_host(self._h, S, _ptr(dA), _ptr(dB), _ptr(x0), N_min, N_max, 0,
                                            _ptr(out.get("J")), _ptr(out.get("rho")), _ptr(out.get("ratio")),
                                            _ptr(out.get("flags")), chunk)
        self._check(rc, "lqmpc_eval_batch_host")
        return out

    # ------------------------------------------------------------------------------------------------ K2
    def set_references(self, x_ref=None, u_ref=None):
        """Shared references of the following mpc_solve_batch / simulate_batch calls: x_ref (n, >=N), u_ref (m, >=N);
        None / all-zero clears them (the reference's callers always pass zeros)."""
        xr = None if x_ref is None else _np_f64(x_ref, (self.n, -1))
        ur = None if u_ref is None else _np_f64(u_ref, (self.m, -1))
        if xr is not None and not xr.any():
            xr = None
        if ur is not None and not ur.any():
            ur = None
        if xr is None and ur is None:
            self._check(self.lib.lqmpc_set_references(self._h, 0, None, None), "lqmpc_set_references")
            return self
        cols = (xr if xr is not None else ur).shape[1]
        if xr is not None and ur is not None and xr.shape[1] != ur.shape[1]:
            cols = min(xr.shape[1], ur.shape[1])
            xr, ur = np.ascontiguousarray(xr[:, :cols]), np.ascontiguousarray(ur[:, :cols])
        self._check(self.lib.lqmpc_set_references(self._h, cols, _ptr(xr), _ptr(ur)), "lqmpc_set_references")
        return self

    def set_input_polytope(self, F_u=None, bar_u: float = -1.0, bar_d_u: float = -1.0):
        """General input polytope F_u u <= 1 (p x m) for the following K2 / K3 calls; None clears it (box of
        set_problem). set_problem also clears it. bar_u / bar_d_u (utils.py:592-650, vertex maxima) become the defaults
        of bounds_batch while the polytope is installed."""
        if F_u is None:
            self._check(self.lib.lqmpc_set_input_polytope(self._h, 0, None), "lqmpc_set_input_polytope")
            self._poly_bar = None
            return self
        F = _np_f64(F_u)
        if F.ndim != 2 or F.shape[1] != self.m:
            raise EngineError("F_u must be (p, m) with m = %d input columns, got %r" % (self.m, F.shape))
        self._check(self.lib.lqmpc_set_input_polytope(self._h, F.shape[0], _ptr(F)), "lqmpc_set_input_polytope")
        self._poly_bar = None
        if bar_u >= 0.0 and bar_d_u >= 0.0:
            self._poly_bar = (float(bar_u), float(bar_d_u))
        return self

    def references(self, x_ref=None, u_ref=None):
        """`with eng.references(x_ref, u_ref): ...` — set for the K2 calls inside, cleared on exit."""
        eng = self

        class _Scope:
            def __enter__(self_inner):
                eng.set_references(x_ref, u_ref)
                return eng

            def __exit__(self_inner, *exc):
                eng.set_references(None, None)
                return False
        return _Scope()

    def _opt_dev(self, a):
        return None if a is None else self._dev(a)

    @_streamed
    def mpc_solve_batch(self, dA, dB, N: int, pts=None, x0=None, S: Optional[int] = None,
                        want=("V", "u0", "M_V", "flags")):
        """Batched LQ_MPC_Controller.solve. dA/dB: [n*n][S]/[n*m][S] or None (true model; give S).
        pts: (npts, n) states shared by all samples, or x0: [n][S] one state per sample."""
        torch = self.torch
        n, m = self.n, self.m
        dA, dB = self._opt_dev(dA), self._opt_dev(dB)
        if S is None:
            S = dA.shape[-1] if dA is not None else (x0.shape[-1] if x0 is not None else 1)
        if pts is None:
            pts_d = None
        elif isinstance(pts, torch.Tensor):
            pts_d = self._dev(pts).reshape(-1, n)
        else:
            pts_d = self._dev(np.asarray(pts, dtype=np.float64).reshape(-1, n))
        x0_d = self._opt_dev(x0)
        P = pts_d.shape[0] if pts_d is not None else 1
        out = {}
        if "V" in want:
            out["V"] = torch.empty((P, S), dtype=torch.float64, device=self.device)
        if "u0" in want:
            out["u0"] = torch.empty((P, m, S), dtype=torch.float64, device=self.device)
        if "M_V" in want:
            out["M_V"] = torch.empty((S,), dtype=torch.float64, device=self.device)
        if "flags" in want:
            out["flags"] = torch.empty((P, S), dtype=torch.int32, device=self.device)
        rc = self.lib.lqmpc_mpc_solve_batch(self._h, S, _ptr(dA), _ptr(dB), int(N), P if pts_d is not None else 0,
                                            _ptr(pts_d), _ptr(x0_d), _ptr(out.get("V")), _ptr(out.get("u0")),
                                            _ptr(out.get("M_V")), _ptr(out.get("flags")))
        self._check(rc, "lqmpc_mpc_solve_batch")
        return out

    @_streamed
    def mpc_solve_range(self, dA, dB, N_min: int, N_max: int, pts=None, x0=None, S: Optional[int] = None,
                        want=("V", "u0", "M_V", "flags")):
        """mpc_solve_batch for every horizon N_min..N_max in one call: V [H][P][S], u0 [H][P][m][S], M_V [H][S],
        flags [H][P][S] (slot h = N - N_min), bit-identical to H calls of mpc_solve_batch."""
        torch = self.torch
        n, m = self.n, self.m
        dA, dB = self._opt_dev(dA), self._opt_dev(dB)
        if S is None:
            S = dA.shape[-1] if dA is not None else (x0.shape[-1] if x0 is not None else 1)
        if pts is None:
            pts_d = None
        elif isinstance(pts, torch.Tensor):
            pts_d = self._dev(pts).reshape(-1, n)
        else:
            pts_d = self._dev(np.asarray(pts, dtype=np.float64).reshape(-1, n))
        x0_d = self._opt_dev(x0)
        P = pts_d.shape[0] if pts_d is not None else 1
        H = int(N_max) - int(N_min) + 1
        if H < 1:
            raise ValueError("N_max < N_min")
        out = {}
        if "V" in want:
            out["V"] = torch.empty((H, P, S), dtype=torch.float64, device=self.device)
        if "u0" in want:
            out["u0"] = torch.empty((H, P, m, S), dtype=torch.float64, device=self.device)
        if "M_V" in want:
            out["M_V"] = torch.empty((H, S), dtype=torch.float64, device=self.device)
        if "flags" in want:
            out["flags"] = torch.empty((H, P, S), dtype=torch.int32, device=self.device)
        rc = self.lib.lqmpc_mpc_solve_range(self._h, S, _ptr(dA), _ptr(dB), int(N_min), int(N_max),
                                            P if pts_d is not None else 0, _ptr(pts_d), _ptr(x0_d),
                                            _ptr(out.get("V")), _ptr(out.get("u0")), _ptr(out.get("M_V")),
                                            _ptr(out.get("flags")))
        self._check(rc, "lqmpc_mpc_solve_range")
        return out

    @_streamed
    def simulate_batch(self, dA, dB, N: int, T: int, x0_shared=None, x0=None, S: Optional[int] = None,
                       want=("J_T", "flags", "n_active")):
        """Batched LQ_MPC_Simulator.simulate. x0_shared: (n,) one state for all samples, or x0: [n][S]."""
        torch = self.torch
        n, m = self.n, self.m
        dA, dB = self._opt_dev(dA), self._opt_dev(dB)
        if S is None:
            S = dA.shape[-1] if dA is not None else (x0.shape[-1] if x0 is not None else 1)
        if x0_shared is None:
            xs = None
        elif isinstance(x0_shared, torch.Tensor):               # already staged by the caller (no per-call H2D copy)
            xs = self._dev(x0_shared).reshape(n)
        else:
            xs = self._dev(np.asarray(x0_shared, dtype=np.float64).reshape(n))
        x0_d = self._opt_dev(x0)
        out = {}
        if "J_T" in want:
            out["J_T"] = torch.empty((S,), dtype=torch.float64, device=self.device)
        if "X" in want:
            out["X"] = torch.empty((T + 1, n, S), dtype=torch.float64, device=self.device)
        if "U" in want:
            out["U"] = torch.empty((T, m, S), dtype=torch.float64, device=self.device)
        if "flags" in want:
            out["flags"] = torch.empty((S,), dtype=torch.int32, device=self.device)
        if "n_active" in want:
            out["n_active"] = torch.empty((S,), dtype=torch.int32, device=self.device)
        rc = self.lib.lqmpc_simulate_batch(self._h, S, _ptr(dA), _ptr(dB), int(N), int(T), _ptr(xs), _ptr(x0_d),
                                           _ptr(out.get("J_T")), _ptr(out.get("X")), _ptr(out.get("U")),
                                           _ptr(out.get("flags")), _ptr(out.get("n_active")))
        self._check(rc, "lqmpc_simulate_batch")
        return out

    @_streamed
    def simulate_inf_batch(self, dA, dB, N: int, T_max: int = 1000, x0_shared=None, x0=None, S: Optional[int] = None,
                           want=("J_inf", "T_cert", "flags")):
        """Infinite-horizon cost of the simulate_batch closed loop (lqmpc_simulate_inf_batch): J_inf [S] (+inf:
        unstable, NaN: not certified within T_max steps), T_cert [S] (the certified step, -1 when there is none),
        flags [S]. x0_shared: (n,) one state for all samples, or x0: [n][S]. Regulation only."""
        torch = self.torch
        n = self.n
        dA, dB = self._opt_dev(dA), self._opt_dev(dB)
        if S is None:
            S = dA.shape[-1] if dA is not None else (x0.shape[-1] if x0 is not None else 1)
        if x0_shared is None:
            xs = None
        elif isinstance(x0_shared, torch.Tensor):
            xs = self._dev(x0_shared).reshape(n)
        else:
            xs = self._dev(np.asarray(x0_shared, dtype=np.float64).reshape(n))
        x0_d = self._opt_dev(x0)
        out = {}
        if "J_inf" in want:
            out["J_inf"] = torch.empty((S,), dtype=torch.float64, device=self.device)
        if "T_cert" in want:
            out["T_cert"] = torch.empty((S,), dtype=torch.int32, device=self.device)
        if "flags" in want:
            out["flags"] = torch.empty((S,), dtype=torch.int32, device=self.device)
        rc = self.lib.lqmpc_simulate_inf_batch(self._h, S, _ptr(dA), _ptr(dB), int(N), int(T_max), _ptr(xs),
                                               _ptr(x0_d), _ptr(out.get("J_inf")), _ptr(out.get("T_cert")),
                                               _ptr(out.get("flags")))
        self._check(rc, "lqmpc_simulate_inf_batch")
        return out

    # ------------------------------------------------------------------------------------------------ worst case
    def _worst_operands(self, dA, dB, x0=None):
        n, m = self.n, self.m
        dA, dB = self._dev(dA), self._dev(dB)
        x0 = None if x0 is None else self._dev(x0)
        S = dA.shape[-1]
        if dA.numel() != n * n * S or dB.numel() != n * m * S or (x0 is not None and x0.numel() != n * S):
            raise ValueError("operand shapes do not match (n, m, S)")
        return dA, dB, x0, S

    @_streamed
    def eval_grad_batch(self, dA, dB, x0, N: int):
        """J_inf of the unconstrained law (as eval_batch at one horizon N) and its exact gradient in the model error
        (lqmpc_eval_grad_batch). dA [n*n][S], dB [n*m][S], x0 [n][S]. Returns device tensors J, rho, ratio [S],
        gA [n*n][S] = dJ/d(dA), gB [n*m][S] = dJ/d(dB) (NaN where unstable or failed) and flags [S]."""
        torch = self.torch
        n, m = self.n, self.m
        dA, dB, x0, S = self._worst_operands(dA, dB, x0)
        f64 = dict(dtype=torch.float64, device=self.device)
        out = {k: torch.empty((S,), **f64) for k in ("J", "rho", "ratio")}
        out["gA"], out["gB"] = torch.empty((n * n, S), **f64), torch.empty((n * m, S), **f64)
        out["flags"] = torch.empty((S,), dtype=torch.int32, device=self.device)
        rc = self.lib.lqmpc_eval_grad_batch(self._h, S, _ptr(dA), _ptr(dB), _ptr(x0), int(N), _ptr(out["J"]),
                                            _ptr(out["rho"]), _ptr(out["ratio"]), _ptr(out["gA"]), _ptr(out["gB"]),
                                            _ptr(out["flags"]))
        self._check(rc, "lqmpc_eval_grad_batch")
        return out

    @_streamed
    def worst_case_batch(self, dA, dB, x0, N: int, e_A: float, e_B: float, norm: str = "f", max_iter: int = 200,
                         tol: float = 1e-8):
        """Projected ascent of J_inf from every sample over {||dA|| <= e_A, ||dB|| <= e_B} (lqmpc_worst_case_batch);
        norm: "f" (Frobenius), "2" (spectral) or "max" (entrywise). Operands as eval_grad_batch. Returns device tensors
        dA [n*n][S], dB [n*m][S] (the final perturbation), J, rho, ratio [S], iters [S] (accepted steps) and flags [S]
        (FLAG_UNSTABLE: the set holds a destabilising error, J = +inf; FLAG_ASCENT_MAXITER: budget exhausted)."""
        torch = self.torch
        n, m = self.n, self.m
        if norm not in WORST_NORMS:
            raise ValueError("norm must be one of %s" % sorted(WORST_NORMS))
        dA, dB, x0, S = self._worst_operands(dA, dB, x0)
        f64 = dict(dtype=torch.float64, device=self.device)
        out = {"dA": torch.empty((n * n, S), **f64), "dB": torch.empty((n * m, S), **f64)}
        out.update({k: torch.empty((S,), **f64) for k in ("J", "rho", "ratio")})
        out["iters"] = torch.empty((S,), dtype=torch.int32, device=self.device)
        out["flags"] = torch.empty((S,), dtype=torch.int32, device=self.device)
        rc = self.lib.lqmpc_worst_case_batch(self._h, S, _ptr(dA), _ptr(dB), _ptr(x0), int(N), float(e_A), float(e_B),
                                             WORST_NORMS[norm], int(max_iter), float(tol), _ptr(out["dA"]),
                                             _ptr(out["dB"]), _ptr(out["J"]), _ptr(out["rho"]), _ptr(out["ratio"]),
                                             _ptr(out["iters"]), _ptr(out["flags"]))
        self._check(rc, "lqmpc_worst_case_batch")
        return out

    @_streamed
    def ratio_sup_batch(self, dA, dB, N: int, grad: bool = False):
        """The worst performance ratio over every initial state, gamma = sup_x0 J_inf(x0) / V_expert(x0) =
        lambda_max(S, P_exp), at each model error (lqmpc_ratio_sup_batch). dA [n*n][S], dB [n*m][S]. Returns device
        tensors gamma [S], x_worst [n][S] (the state attaining it, x_worst'P_exp x_worst = 1), gap [S] (relative
        eigengap (lambda_1 - lambda_2) / lambda_1), rho [S] and flags [S]; with grad also gA [n*n][S] = dgamma/d(dA) and
        gB [n*m][S] = dgamma/d(dB) (exact where gap > 0; NaN where unstable or failed)."""
        torch = self.torch
        n, m = self.n, self.m
        dA, dB, _, S = self._worst_operands(dA, dB)
        f64 = dict(dtype=torch.float64, device=self.device)
        out = {k: torch.empty((S,), **f64) for k in ("gamma", "gap", "rho")}
        out["x_worst"] = torch.empty((n, S), **f64)
        out["flags"] = torch.empty((S,), dtype=torch.int32, device=self.device)
        if grad:
            out["gA"], out["gB"] = torch.empty((n * n, S), **f64), torch.empty((n * m, S), **f64)
        rc = self.lib.lqmpc_ratio_sup_batch(self._h, S, _ptr(dA), _ptr(dB), int(N), _ptr(out["gamma"]),
                                            _ptr(out["x_worst"]), _ptr(out["gap"]), _ptr(out["rho"]),
                                            _ptr(out.get("gA")), _ptr(out.get("gB")), _ptr(out["flags"]))
        self._check(rc, "lqmpc_ratio_sup_batch")
        return out

    @_streamed
    def worst_case_sup_batch(self, dA, dB, N: int, e_A: float, e_B: float, norm: str = "f", max_iter: int = 200,
                             tol: float = 1e-8):
        """Projected ascent of gamma (ratio_sup_batch) from every sample over {||dA|| <= e_A, ||dB|| <= e_B}
        (lqmpc_worst_case_sup_batch): the joint worst case over the model error and the initial state, to a stationary
        point. Settings and flags as worst_case_batch. Returns device tensors dA [n*n][S], dB [n*m][S], gamma [S],
        x_worst [n][S], rho [S], iters [S] and flags [S]."""
        torch = self.torch
        n, m = self.n, self.m
        if norm not in WORST_NORMS:
            raise ValueError("norm must be one of %s" % sorted(WORST_NORMS))
        dA, dB, _, S = self._worst_operands(dA, dB)
        f64 = dict(dtype=torch.float64, device=self.device)
        out = {"dA": torch.empty((n * n, S), **f64), "dB": torch.empty((n * m, S), **f64),
               "gamma": torch.empty((S,), **f64), "x_worst": torch.empty((n, S), **f64),
               "rho": torch.empty((S,), **f64)}
        out["iters"] = torch.empty((S,), dtype=torch.int32, device=self.device)
        out["flags"] = torch.empty((S,), dtype=torch.int32, device=self.device)
        rc = self.lib.lqmpc_worst_case_sup_batch(self._h, S, _ptr(dA), _ptr(dB), int(N), float(e_A), float(e_B),
                                                 WORST_NORMS[norm], int(max_iter), float(tol), _ptr(out["dA"]),
                                                 _ptr(out["dB"]), _ptr(out["gamma"]), _ptr(out["x_worst"]),
                                                 _ptr(out["rho"]), _ptr(out["iters"]), _ptr(out["flags"]))
        self._check(rc, "lqmpc_worst_case_sup_batch")
        return out

    def _inf_operands(self, dA, dB, x0_shared, x0):
        n = self.n
        dA, dB, _, S = self._worst_operands(dA, dB)
        if (x0_shared is None) == (x0 is None):
            raise ValueError("give exactly one of x0_shared / x0")
        xs = None if x0_shared is None else self._dev(x0_shared).reshape(n)
        x0 = None if x0 is None else self._dev(x0)
        if x0 is not None and x0.numel() != n * S:
            raise ValueError("operand shapes do not match (n, m, S)")
        return dA, dB, xs, x0, S

    @_streamed
    def simulate_inf_grad_batch(self, dA, dB, N: int, T_max: int = 1000, x0_shared=None, x0=None, grad: bool = True):
        """J_inf of the input-constrained closed loop (as simulate_inf_batch) and its exact gradient in the model error
        (lqmpc_simulate_inf_grad_batch). dA [n*n][S], dB [n*m][S]; x0_shared: (n,) one state for all samples, or x0:
        [n][S]. Returns device tensors J_inf [S] (+inf: unstable, NaN: not certified within T_max steps), T_cert [S],
        rho [S] = rho(A + B K0), flags [S] and, with grad, gA [n*n][S] = dJ_inf/d(dA), gB [n*m][S] = dJ_inf/d(dB)
        (NaN where J_inf is not finite or a failure flag is set). Box only, regulation only."""
        torch = self.torch
        n, m = self.n, self.m
        dA, dB, xs, x0, S = self._inf_operands(dA, dB, x0_shared, x0)
        f64 = dict(dtype=torch.float64, device=self.device)
        out = {"J_inf": torch.empty((S,), **f64), "T_cert": torch.empty((S,), dtype=torch.int32, device=self.device),
               "rho": torch.empty((S,), **f64), "flags": torch.empty((S,), dtype=torch.int32, device=self.device)}
        if grad:
            out["gA"], out["gB"] = torch.empty((n * n, S), **f64), torch.empty((n * m, S), **f64)
        rc = self.lib.lqmpc_simulate_inf_grad_batch(self._h, S, _ptr(dA), _ptr(dB), int(N), int(T_max), _ptr(xs),
                                                    _ptr(x0), _ptr(out["J_inf"]), _ptr(out["T_cert"]),
                                                    _ptr(out["rho"]), _ptr(out.get("gA")), _ptr(out.get("gB")),
                                                    _ptr(out["flags"]))
        self._check(rc, "lqmpc_simulate_inf_grad_batch")
        return out

    @_streamed
    def worst_case_inf_batch(self, dA, dB, N: int, e_A: float, e_B: float, norm: str = "f", max_iter: int = 200,
                             tol: float = 1e-8, T_max: int = 1000, x0_shared=None, x0=None):
        """Projected ascent of the input-constrained closed loop's J_inf (simulate_inf_grad_batch) from every sample
        over {||dA|| <= e_A, ||dB|| <= e_B} (lqmpc_worst_case_inf_batch), to a stationary point. Settings as
        worst_case_batch, operands as simulate_inf_grad_batch. Returns device tensors dA [n*n][S], dB [n*m][S] (the
        final perturbation), J_inf, T_cert, rho, iters [S] and flags [S] (FLAG_UNSTABLE: a destabilising error, J_inf =
        +inf; FLAG_ASCENT_MAXITER: budget exhausted; a start with another failure flag is returned as it is)."""
        torch = self.torch
        n, m = self.n, self.m
        if norm not in WORST_NORMS:
            raise ValueError("norm must be one of %s" % sorted(WORST_NORMS))
        dA, dB, xs, x0, S = self._inf_operands(dA, dB, x0_shared, x0)
        f64 = dict(dtype=torch.float64, device=self.device)
        i32 = dict(dtype=torch.int32, device=self.device)
        out = {"dA": torch.empty((n * n, S), **f64), "dB": torch.empty((n * m, S), **f64),
               "J_inf": torch.empty((S,), **f64), "T_cert": torch.empty((S,), **i32), "rho": torch.empty((S,), **f64),
               "iters": torch.empty((S,), **i32), "flags": torch.empty((S,), **i32)}
        rc = self.lib.lqmpc_worst_case_inf_batch(self._h, S, _ptr(dA), _ptr(dB), int(N), int(T_max), _ptr(xs),
                                                 _ptr(x0), float(e_A), float(e_B), WORST_NORMS[norm], int(max_iter),
                                                 float(tol), _ptr(out["dA"]), _ptr(out["dB"]), _ptr(out["J_inf"]),
                                                 _ptr(out["T_cert"]), _ptr(out["rho"]), _ptr(out["iters"]),
                                                 _ptr(out["flags"]))
        self._check(rc, "lqmpc_worst_case_inf_batch")
        return out

    # ------------------------------------------------------------------------------------------------ K3
    @_streamed
    def bounds_batch(self, dA, dB, N: int, e_A, e_B, M_V, x, p, V_expert: float, K=None, S: Optional[int] = None,
                     bar_u: float = -1.0, bar_d_u: float = -1.0, strict_reference: bool = True, want_K=False,
                     want_P=False):
        """Batched energy_decreasing + energy_bound + J_bound. e_A/e_B/M_V: python scalars or [S] arrays;
        x: (n,) shared or [n][S]; K: None (-> -K_dlqr per sample), (m,n)/(m*n,) shared, or [m*n][S] (u = +Kx)."""
        torch = self.torch
        n, m = self.n, self.m
        dA, dB = self._opt_dev(dA), self._opt_dev(dB)
        if S is None:
            S = dA.shape[-1] if dA is not None else 1

        def per_sample(v):
            if np.isscalar(v) or (hasattr(v, "ndim") and v.ndim == 0):
                return None, float(v)
            return self._dev(v).reshape(S), 0.0

        eA_d, eA_s = per_sample(e_A)
        eB_d, eB_s = per_sample(e_B)
        MV_d, MV_s = per_sample(M_V)
        x_arr = x if isinstance(x, torch.Tensor) else np.asarray(x, dtype=np.float64)
        x_sh = x_ps = None
        if int(np.prod(x_arr.shape)) == n:          # one state shared by every sample
            x_sh = self._dev(x_arr).reshape(n)
        else:
            x_ps = self._dev(x_arr).reshape(n, S)
        K_sh = K_ps = None
        if K is not None:
            K_arr = K if isinstance(K, torch.Tensor) else np.asarray(K, dtype=np.float64)
            if K_arr.size == m * n:
                K_sh = self._dev(K_arr).reshape(m * n)
            else:
                K_ps = self._dev(K_arr).reshape(m * n, S)
        NF = int(self.lib.lqmpc_bounds_fields())
        assert NF == len(BOUND_FIELDS)
        detail = torch.empty((NF, S), dtype=torch.float64, device=self.device)
        flags = torch.empty((S,), dtype=torch.int32, device=self.device)
        K_out = torch.empty((m * n, S), dtype=torch.float64, device=self.device) if want_K else None
        P_out = torch.empty((n * n, S), dtype=torch.float64, device=self.device) if want_P else None
        p3 = _np_f64(p, (3,))
        if getattr(self, "_poly_bar", None) is not None and (bar_u < 0.0 or bar_d_u < 0.0):
            bar_u, bar_d_u = self._poly_bar
        rc = self.lib.lqmpc_bounds_batch(self._h, S, _ptr(dA), _ptr(dB), int(N), _ptr(eA_d), _ptr(eB_d), eA_s, eB_s,
                                         _ptr(MV_d), MV_s, _ptr(x_sh), _ptr(x_ps), _ptr(K_ps), _ptr(K_sh), _ptr(p3),
                                         float(V_expert), float(bar_u), float(bar_d_u), int(bool(strict_reference)),
                                         None, None, None, None, None, _ptr(detail), _ptr(K_out), _ptr(P_out),
                                         _ptr(flags))
        self._check(rc, "lqmpc_bounds_batch")
        out = {k: detail[i] for i, k in enumerate(BOUND_FIELDS)}
        out["flags"] = flags
        if want_K:
            out["K"] = K_out
        if want_P:
            out["P"] = P_out
        return out

    @_streamed
    def bounds_range(self, dA, dB, N_min: int, N_max: int, e_A, e_B, M_V, x, p, V_expert: float, K=None,
                     S: Optional[int] = None, bar_u: float = -1.0, bar_d_u: float = -1.0, strict_reference: bool = True,
                     want_K=False, want_P=False, detail: bool = True):
        """bounds_batch for every horizon N_min..N_max in one call. M_V: scalar, [S] (shared by every horizon) or
        [H][S]. Returns [H][S] tensors per field (slot h = N - N_min) and flags [H][S]; K / P [..][S] once. With
        detail=False only alpha, beta, xi, eta, bound and flags are produced (no [H][fields][S] table)."""
        torch = self.torch
        n, m = self.n, self.m
        dA, dB = self._opt_dev(dA), self._opt_dev(dB)
        if S is None:
            S = dA.shape[-1] if dA is not None else 1
        H = int(N_max) - int(N_min) + 1
        if H < 1:
            raise ValueError("N_max < N_min")

        def per_sample(v, name, rows=1):
            """scalar -> (None, v); [S] (or [rows][S]) -> contiguous device vector of rows * S entries."""
            if np.isscalar(v) or (hasattr(v, "ndim") and v.ndim == 0):
                return None, float(v)
            t = self._dev(v)
            if rows > 1 and t.numel() == S:                  # one [S] vector shared by every horizon
                t = t.reshape(1, S).expand(rows, S).contiguous()
            if t.numel() != rows * S:
                raise ValueError("%s must be a scalar or hold %s entries, got %d"
                                 % (name, "S = %d" % S if rows == 1 else "S or H * S = %d" % (rows * S), t.numel()))
            return t.reshape(-1), 0.0

        eA_d, eA_s = per_sample(e_A, "e_A")
        eB_d, eB_s = per_sample(e_B, "e_B")
        MV_d, MV_s = per_sample(M_V, "M_V", rows=H)
        x_arr = x if isinstance(x, torch.Tensor) else np.asarray(x, dtype=np.float64)
        x_sh = x_ps = None
        if int(np.prod(x_arr.shape)) == n:
            x_sh = self._dev(x_arr).reshape(n)
        else:
            x_ps = self._dev(x_arr).reshape(n, S)
        K_sh = K_ps = None
        if K is not None:
            K_arr = K if isinstance(K, torch.Tensor) else np.asarray(K, dtype=np.float64)
            if int(np.prod(K_arr.shape)) == m * n:
                K_sh = self._dev(K_arr).reshape(m * n)
            else:
                K_ps = self._dev(K_arr).reshape(m * n, S)
        NF = int(self.lib.lqmpc_bounds_fields())
        assert NF == len(BOUND_FIELDS)
        out = {}
        if detail:
            table = torch.empty((H, NF, S), dtype=torch.float64, device=self.device)
            out.update({k: table[:, i] for i, k in enumerate(BOUND_FIELDS)})
            ptrs = [None] * 5
        else:
            table = None
            core = torch.empty((5, H, S), dtype=torch.float64, device=self.device)
            for i, k in enumerate(("alpha", "beta", "xi", "eta", "bound")):
                out[k] = core[i]
            ptrs = [core[i] for i in range(5)]
        flags = torch.empty((H, S), dtype=torch.int32, device=self.device)
        K_out = torch.empty((m * n, S), dtype=torch.float64, device=self.device) if want_K else None
        P_out = torch.empty((n * n, S), dtype=torch.float64, device=self.device) if want_P else None
        p3 = _np_f64(p, (3,))
        if getattr(self, "_poly_bar", None) is not None and (bar_u < 0.0 or bar_d_u < 0.0):
            bar_u, bar_d_u = self._poly_bar
        rc = self.lib.lqmpc_bounds_range(self._h, S, _ptr(dA), _ptr(dB), int(N_min), int(N_max), _ptr(eA_d),
                                         _ptr(eB_d), eA_s, eB_s, _ptr(MV_d), MV_s, _ptr(x_sh), _ptr(x_ps), _ptr(K_ps),
                                         _ptr(K_sh), _ptr(p3), float(V_expert), float(bar_u), float(bar_d_u),
                                         int(bool(strict_reference)), *[_ptr(t) for t in ptrs], _ptr(table),
                                         _ptr(K_out), _ptr(P_out), _ptr(flags))
        self._check(rc, "lqmpc_bounds_range")
        out["flags"] = flags
        if want_K:
            out["K"] = K_out
        if want_P:
            out["P"] = P_out
        return out

    @_streamed
    def dlqr_batch(self, dA=None, dB=None, S: Optional[int] = None):
        """Batched control.dlqr: returns K [m*n][S] (u = -Kx), P [n*n][S], flags [S]."""
        torch = self.torch
        n, m = self.n, self.m
        dA, dB = self._opt_dev(dA), self._opt_dev(dB)
        if S is None:
            S = dA.shape[-1] if dA is not None else 1
        K = torch.empty((m * n, S), dtype=torch.float64, device=self.device)
        P = torch.empty((n * n, S), dtype=torch.float64, device=self.device)
        fl = torch.empty((S,), dtype=torch.int32, device=self.device)
        self._check(self.lib.lqmpc_dlqr_batch(self._h, S, _ptr(dA), _ptr(dB), _ptr(K), _ptr(P), _ptr(fl)),
                    "lqmpc_dlqr_batch")
        return {"K": K, "P": P, "flags": fl}

    # ------------------------------------------------------------------------------------------------ K5
    @_streamed
    def column_stats_raw(self, table):
        """table: [cols][S] device tensor (rows contiguous). Returns [cols][5] = max, min, sum, n_finite, n_bad."""
        torch = self.torch
        t = self._dev(table)
        if t.ndim == 1:
            t = t.reshape(1, -1)
        cols, S = t.shape
        if S == 0:
            return torch.tensor([[-np.inf, np.inf, 0.0, 0.0, 0.0]] * cols, dtype=torch.float64, device=self.device)
        stats = torch.empty((cols, 5), dtype=torch.float64, device=self.device)
        self._check(self.lib.lqmpc_column_stats(self._h, _ptr(t), cols, S, S, _ptr(stats)), "lqmpc_column_stats")
        return stats

    @_streamed
    def column_moments_raw(self, table):
        """table: [cols][S] device tensor. Returns device [cols][6] = max, min, n_finite, n_nonfinite, mean, M2."""
        torch = self.torch
        t = self._dev(table)
        if t.ndim == 1:
            t = t.reshape(1, -1)
        cols, S = t.shape
        if S == 0:                                   # nothing to reduce (and no valid device pointer to pass)
            return torch.tensor([[-np.inf, np.inf, 0.0, 0.0, np.nan, np.nan]] * cols, dtype=torch.float64,
                                device=self.device)
        out = torch.empty((cols, 6), dtype=torch.float64, device=self.device)
        self._check(self.lib.lqmpc_column_moments(self._h, _ptr(t), cols, S, S, _ptr(out)), "lqmpc_column_moments")
        return out

    @_streamed
    def column_sqdev_raw(self, table, mean):
        torch = self.torch
        t = self._dev(table)
        if t.ndim == 1:
            t = t.reshape(1, -1)
        cols, S = t.shape
        mean = self._dev(mean).reshape(cols)
        if S == 0:
            return torch.zeros((cols,), dtype=torch.float64, device=self.device)
        out = torch.empty((cols,), dtype=torch.float64, device=self.device)
        self._check(self.lib.lqmpc_column_sqdev(self._h, _ptr(t), cols, S, S, _ptr(mean), _ptr(out)),
                    "lqmpc_column_sqdev")
        return out

    def _table_view(self, table):
        """[cols][S] table -> (tensor, cols, S, ld). A float64 CUDA tensor on this device whose rows are contiguous is
        used in place (row stride = ld, storage offset kept), anything else is staged as a contiguous copy."""
        torch = self.torch
        t = table
        if isinstance(t, torch.Tensor) and t.ndim == 1:
            t = t.reshape(1, -1)
        if not (isinstance(t, torch.Tensor) and t.device == self.device and t.dtype == torch.float64 and t.ndim == 2
                and (t.stride(1) == 1 or t.shape[1] <= 1) and (t.shape[0] <= 1 or t.stride(0) >= t.shape[1])):
            t = self._dev(table)
            if t.ndim == 1:
                t = t.reshape(1, -1)
        cols, S = t.shape
        return t, cols, S, (int(t.stride(0)) if cols > 1 else S)

    @_streamed
    def column_radix_histogram_raw(self, table, prefix, pass_: int):
        """One radix pass (lqmpc_column_radix_histogram): prefix device int64 [cols][nsel] (the uint64 key prefixes,
        nsel <= RADIX_MAX_SEL). Returns device int64 [cols][nsel][256]."""
        torch = self.torch
        t, cols, S, ld = self._table_view(table)
        nsel = prefix.shape[1]
        hist = torch.empty((cols, nsel, 256), dtype=torch.int64, device=self.device)
        self._check(self.lib.lqmpc_column_radix_histogram(self._h, _ptr(t) if S else None, cols, S, ld, nsel,
                                                          int(pass_), _ptr(prefix), _ptr(hist)),
                    "lqmpc_column_radix_histogram")
        return hist

    @_streamed
    def column_radix_select_raw(self, hist, pass_: int, rank, prefix):
        """Digit pick of one radix pass (lqmpc_column_radix_select): updates rank and prefix [cols][nsel] in place."""
        cols, nsel = rank.shape
        self._check(self.lib.lqmpc_column_radix_select(self._h, _ptr(hist), cols, nsel, int(pass_), _ptr(rank),
                                                       _ptr(prefix)), "lqmpc_column_radix_select")

    @_streamed
    def column_argext_raw(self, table, index_base: int = 0):
        """Returns device (val [cols][2] = {max, min} of the finite entries, idx [cols][2] int64 = index_base + the
        lowest position attaining each; -1 and -inf / +inf for a column without a finite entry)."""
        torch = self.torch
        t, cols, S, ld = self._table_view(table)
        val = torch.empty((cols, 2), dtype=torch.float64, device=self.device)
        idx = torch.empty((cols, 2), dtype=torch.int64, device=self.device)
        self._check(self.lib.lqmpc_column_argext(self._h, _ptr(t) if S else None, cols, S, ld, int(index_base),
                                                 _ptr(val), _ptr(idx)), "lqmpc_column_argext")
        return val, idx

    # ------------------------------------------------------------------------------------------------ K6
    @_streamed
    def sample_error_grid(self, seed: int, which: int, rows: int, cols: int, N_sys: int, levels, n_boundary: int,
                          norm_type: str = "f", j_first: int = 0, want_stats: bool = False):
        """Device-side `random_matrix` grid (utils.py:779-847 restated, seeded): returns the SoA tensor
        [rows*cols][N_sys*n_err] (== the reference's (rows, cols, N_sys, n_err) array in C order)."""
        torch = self.torch
        lev = _np_f64(levels)
        n_err = lev.size
        out = torch.empty((rows * cols, N_sys * n_err), dtype=torch.float64, device=self.device)
        st = np.zeros(2, dtype=np.int64) if want_stats else None
        rc = self.lib.lqmpc_sample_error_grid(self._h, int(seed), int(which), rows, cols, N_sys, j_first, n_err,
                                              _ptr(lev), int(n_boundary), {"f": 0, "2": 1}[norm_type], _ptr(out),
                                              None if st is None else st.ctypes.data)
        self._check(rc, "lqmpc_sample_error_grid")
        return (out, {"rejected": int(st[0]), "projected": int(st[1])}) if want_stats else out

    def fp64_tensor_peak(self) -> float:
        v = ctypes.c_double(0.0)
        self._check(self.lib.lqmpc_fp64_tensor_peak(self._h, ctypes.byref(v)), "lqmpc_fp64_tensor_peak")
        return float(v.value)

    def fp64_peak(self) -> float:
        v = ctypes.c_double(0.0)
        self._check(self.lib.lqmpc_fp64_peak(self._h, ctypes.byref(v)), "lqmpc_fp64_peak")
        return float(v.value)
