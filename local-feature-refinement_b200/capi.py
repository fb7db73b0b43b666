"""ctypes binding of include/lfr.h.

`load_b200()` loads the product library (csrc/liblfr_b200.so) and fails loudly
when it is missing: there is no CPU fallback.  The same struct definitions also
bind the CPU oracle's library, but that is done only by tests/ and bench.py's
baseline legs (see tests/oracle_util.py), never from this package.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

from .graph import EDGE_DTYPE, Problem

HERE = os.path.dirname(os.path.abspath(__file__))
B200_LIB_PATH = os.path.join(HERE, "csrc", "liblfr_b200.so")
HOST_LIB_PATH = os.path.join(HERE, "csrc", "liblfr_host.so")

LFR_OK = 0
# lfr_options.debug_flags (include/lfr.h)
DBG_FORCE_SMEM_CHOLESKY, DBG_NO_TILE, DBG_NO_ZERO_COPY, DBG_PROFILE = 0x1, 0x2, 0x8, 0x10
TERM_NAMES = {0: "skipped", 1: "gradient_tol", 2: "parameter_tol", 3: "function_tol",
              4: "min_radius", 5: "no_convergence", 6: "failure", 7: "empty"}


class LfrProblem(C.Structure):
    _fields_ = [
        ("n_nodes", C.c_uint32), ("n_components", C.c_uint32), ("n_edges", C.c_uint64),
        ("row_ptr", C.c_void_p), ("edges", C.c_void_p), ("track", C.c_void_p),
        ("comp", C.c_void_p), ("is_root", C.c_void_p), ("comp_ptr", C.c_void_p),
        ("comp_nodes", C.c_void_p),
    ]


class LfrOptions(C.Structure):
    _fields_ = [
        ("bound", C.c_double), ("cauchy_a", C.c_double), ("tukey_a", C.c_double),
        ("tukey_variant", C.c_int32), ("max_num_iterations", C.c_int32),
        ("max_num_consecutive_invalid_steps", C.c_int32),
        ("max_num_line_search_step_size_iterations", C.c_int32),
        ("function_tolerance", C.c_double), ("gradient_tolerance", C.c_double),
        ("parameter_tolerance", C.c_double), ("initial_trust_region_radius", C.c_double),
        ("max_trust_region_radius", C.c_double), ("min_trust_region_radius", C.c_double),
        ("min_relative_decrease", C.c_double), ("min_lm_diagonal", C.c_double),
        ("max_lm_diagonal", C.c_double), ("line_search_sufficient_function_decrease", C.c_double),
        ("max_line_search_step_contraction", C.c_double),
        ("min_line_search_step_contraction", C.c_double), ("min_line_search_step_size", C.c_double),
        ("n_threads", C.c_int32), ("device", C.c_int32), ("linear_solver", C.c_int32),
        ("debug_flags", C.c_int32),
    ]


class LfrStats(C.Structure):
    _fields_ = [
        ("iterations", C.c_void_p), ("termination", C.c_void_p), ("initial_cost", C.c_void_p),
        ("final_cost", C.c_void_p), ("total_iterations", C.c_uint64),
        ("total_line_search_steps", C.c_uint64), ("n_solved", C.c_uint32),
        ("n_kernel_launches", C.c_uint32), ("h2d_ms", C.c_double), ("kernel_ms", C.c_double),
        ("d2h_ms", C.c_double), ("total_ms", C.c_double),
    ]


class LfrMultiInfo(C.Structure):
    _fields_ = [("kernel_ms", C.c_double * 16), ("total_ms", C.c_double * 16), ("n_slots", C.c_uint32 * 16),
                ("n_edges", C.c_uint64 * 16), ("zero_copy", C.c_int32), ("reserved", C.c_int32)]


#: every symbol include/lfr.h declares
ABI_SYMBOLS = [
    "lfr_abi_version", "lfr_backend", "lfr_last_error", "lfr_options_default", "lfr_solve", "lfr_solve_multi", "lfr_shutdown", "lfr_host_alloc", "lfr_host_free",
    "lfr_plan_create", "lfr_plan_solve", "lfr_plan_download", "lfr_plan_num_launches",
    "lfr_plan_traffic", "lfr_plan_destroy", "lfr_debug_edge_eval",
]


def _ptr(a: Optional[np.ndarray]) -> Optional[int]:
    return None if a is None else a.ctypes.data


class Library:
    """One loaded implementation of include/lfr.h."""

    def __init__(self, path: str):
        if not os.path.exists(path):
            raise RuntimeError(
                "lfr: %s is missing — build it first (python __graft_entry__.py build); "
                "there is no CPU fallback" % path)
        self.path = path
        self.lib = C.CDLL(path)
        L = self.lib
        L.lfr_abi_version.restype = C.c_int
        L.lfr_backend.restype = C.c_char_p
        L.lfr_last_error.restype = C.c_char_p
        L.lfr_options_default.argtypes = [C.POINTER(LfrOptions)]
        L.lfr_options_default.restype = None
        L.lfr_solve.argtypes = [C.POINTER(LfrProblem), C.POINTER(LfrOptions), C.c_void_p, C.POINTER(LfrStats)]
        L.lfr_solve.restype = C.c_int
        L.lfr_solve_multi.argtypes = [C.POINTER(LfrProblem), C.POINTER(LfrOptions), C.c_void_p, C.c_int32, C.c_void_p,
                                      C.POINTER(LfrStats), C.POINTER(LfrMultiInfo)]
        L.lfr_solve_multi.restype = C.c_int
        L.lfr_plan_create.argtypes = [C.POINTER(LfrProblem), C.POINTER(LfrOptions), C.c_void_p,
                                      C.POINTER(C.c_void_p)]
        L.lfr_plan_create.restype = C.c_int
        L.lfr_plan_solve.argtypes = [C.c_void_p, C.c_void_p]
        L.lfr_plan_solve.restype = C.c_int
        L.lfr_plan_download.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(LfrStats)]
        L.lfr_plan_download.restype = C.c_int
        L.lfr_plan_num_launches.argtypes = [C.c_void_p]
        L.lfr_plan_num_launches.restype = C.c_int
        L.lfr_plan_traffic.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        L.lfr_plan_traffic.restype = C.c_int
        L.lfr_plan_destroy.argtypes = [C.c_void_p]
        L.lfr_plan_destroy.restype = None
        L.lfr_debug_edge_eval.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                          C.POINTER(LfrOptions), C.c_void_p, C.c_void_p, C.c_void_p]
        L.lfr_debug_edge_eval.restype = C.c_int
        if L.lfr_abi_version() != 1:
            raise RuntimeError("lfr: ABI version mismatch in %s" % path)

    @property
    def backend(self) -> str:
        return self.lib.lfr_backend().decode()

    def last_error(self) -> str:
        return (self.lib.lfr_last_error() or b"").decode()

    def check(self, rc: int, what: str) -> None:
        if rc != LFR_OK:
            raise RuntimeError("lfr: %s failed (%d): %s" % (what, rc, self.last_error()))

    def default_options(self, **overrides) -> LfrOptions:
        o = LfrOptions()
        self.lib.lfr_options_default(C.byref(o))
        for k, v in overrides.items():
            if not hasattr(o, k):
                raise AttributeError("lfr_options has no field %r" % k)
            setattr(o, k, v)
        return o

    # -- problem marshalling ---------------------------------------------------
    @staticmethod
    def marshal(p: Problem):
        g = p.graph
        arrays = dict(
            row_ptr=np.ascontiguousarray(g.row_ptr, dtype=np.uint32),
            edges=np.ascontiguousarray(g.edges, dtype=EDGE_DTYPE),
            track=np.ascontiguousarray(p.track, dtype=np.uint32),
            comp=np.ascontiguousarray(p.comp, dtype=np.uint32),
            is_root=np.ascontiguousarray(p.is_root, dtype=np.uint8),
            comp_ptr=np.ascontiguousarray(p.comp_ptr, dtype=np.uint32),
            comp_nodes=np.ascontiguousarray(p.comp_nodes, dtype=np.uint32),
        )
        s = LfrProblem(
            n_nodes=g.n_nodes, n_components=p.n_components, n_edges=g.n_edges,
            row_ptr=_ptr(arrays["row_ptr"]), edges=_ptr(arrays["edges"]), track=_ptr(arrays["track"]),
            comp=_ptr(arrays["comp"]), is_root=_ptr(arrays["is_root"]), comp_ptr=_ptr(arrays["comp_ptr"]),
            comp_nodes=_ptr(arrays["comp_nodes"]),
        )
        return s, arrays   # keep `arrays` alive while `s` is in use

    @staticmethod
    def make_stats(n_components: int):
        bufs = dict(
            iterations=np.zeros(n_components, dtype=np.int32),
            termination=np.zeros(n_components, dtype=np.int32),
            initial_cost=np.zeros(n_components, dtype=np.float64),
            final_cost=np.zeros(n_components, dtype=np.float64),
        )
        st = LfrStats(iterations=_ptr(bufs["iterations"]), termination=_ptr(bufs["termination"]),
                      initial_cost=_ptr(bufs["initial_cost"]), final_cost=_ptr(bufs["final_cost"]))
        return st, bufs

    @staticmethod
    def stats_dict(st: LfrStats, bufs: dict) -> dict:
        d = dict(bufs)
        for k in ("total_iterations", "total_line_search_steps", "n_solved", "n_kernel_launches",
                  "h2d_ms", "kernel_ms", "d2h_ms", "total_ms"):
            d[k] = getattr(st, k)
        return d

    def solve(self, p: Problem, options: Optional[LfrOptions] = None,
              positions: Optional[np.ndarray] = None):
        """lfr_solve: returns (positions [N,2] float64, stats dict)."""
        s, keep = self.marshal(p)
        o = options if options is not None else self.default_options()
        N = p.graph.n_nodes
        pos = np.zeros((N, 2), dtype=np.float64) if positions is None else \
            np.ascontiguousarray(positions, dtype=np.float64).reshape(N, 2).copy()
        st, bufs = self.make_stats(p.n_components)
        rc = self.lib.lfr_solve(C.byref(s), C.byref(o), _ptr(pos), C.byref(st))
        self.check(rc, "lfr_solve")
        del keep
        return pos, self.stats_dict(st, bufs)

    def solve_multi(self, p: Problem, devices, options: Optional[LfrOptions] = None,
                    positions: Optional[np.ndarray] = None, pinned: bool = False):
        """lfr_solve_multi: one call, several GPUs.  pinned=True page-locks the edge array and the
        position array first (torch), which lets every device pull only its own components' edges.
        Returns (positions [N,2], stats dict incl. per-device `multi` info)."""
        s, keep = self.marshal(p)
        o = options if options is not None else self.default_options()
        N = p.graph.n_nodes
        pos = np.zeros((N, 2), dtype=np.float64) if positions is None else \
            np.ascontiguousarray(positions, dtype=np.float64).reshape(N, 2).copy()
        holders = []
        pos_ptr = _ptr(pos)
        if pinned:
            import torch
            e_pin = torch.empty(max(keep["edges"].nbytes, 16), dtype=torch.uint8).pin_memory()
            e_pin.numpy()[:keep["edges"].nbytes] = keep["edges"].view(np.uint8).reshape(-1)
            s.edges = e_pin.data_ptr()
            p_pin = torch.zeros(max(2 * N, 2), dtype=torch.float64).pin_memory()
            p_pin.numpy()[:2 * N] = pos.reshape(-1)
            pos_ptr = p_pin.data_ptr()
            holders = [e_pin, p_pin]
        dev = np.ascontiguousarray(list(devices), dtype=np.int32)
        st, bufs = self.make_stats(p.n_components)
        info = LfrMultiInfo()
        rc = self.lib.lfr_solve_multi(C.byref(s), C.byref(o), dev.ctypes.data, int(dev.shape[0]), pos_ptr,
                                      C.byref(st), C.byref(info))
        self.check(rc, "lfr_solve_multi")
        if pinned:
            pos = holders[1].numpy()[:2 * N].reshape(N, 2).copy()
        d = self.stats_dict(st, bufs)
        n = int(dev.shape[0])
        d["multi"] = dict(devices=dev.tolist(), kernel_ms=list(info.kernel_ms)[:n], total_ms=list(info.total_ms)[:n],
                          n_slots=list(info.n_slots)[:n], n_edges=list(info.n_edges)[:n], zero_copy=int(info.zero_copy))
        del keep, holders
        return pos, d

    def edge_eval(self, edges: np.ndarray, kind: np.ndarray, xs: np.ndarray, xd: np.ndarray,
                  options: Optional[LfrOptions] = None):
        n = int(edges.shape[0])
        edges = np.ascontiguousarray(edges, dtype=EDGE_DTYPE)
        kind = np.ascontiguousarray(kind, dtype=np.uint8)
        xs = np.ascontiguousarray(xs, dtype=np.float64)
        xd = np.ascontiguousarray(xd, dtype=np.float64)
        r = np.zeros((n, 2)); jac = np.zeros((n, 4)); rho = np.zeros((n, 3))
        o = options if options is not None else self.default_options()
        rc = self.lib.lfr_debug_edge_eval(_ptr(edges), _ptr(kind), n, _ptr(xs), _ptr(xd), C.byref(o),
                                          _ptr(r), _ptr(jac), _ptr(rho))
        self.check(rc, "lfr_debug_edge_eval")
        return r, jac, rho


class Plan:
    """Device-resident problem (lfr_plan_*), used by bench.py's `value` leg."""

    def __init__(self, lib: Library, p: Problem, options: Optional[LfrOptions] = None,
                 positions: Optional[np.ndarray] = None):
        self.lib = lib
        self.problem = p
        s, keep = lib.marshal(p)
        o = options if options is not None else lib.default_options()
        init = None if positions is None else np.ascontiguousarray(positions, dtype=np.float64)
        h = C.c_void_p()
        lib.check(lib.lib.lfr_plan_create(C.byref(s), C.byref(o), _ptr(init), C.byref(h)), "lfr_plan_create")
        self.handle = h

    def solve(self, stream: int = 0) -> None:
        self.lib.check(self.lib.lib.lfr_plan_solve(self.handle, C.c_void_p(stream)), "lfr_plan_solve")

    def download(self, stream: int = 0):
        N = self.problem.graph.n_nodes
        pos = np.zeros((N, 2), dtype=np.float64)
        st, bufs = Library.make_stats(self.problem.n_components)
        self.lib.check(self.lib.lib.lfr_plan_download(self.handle, C.c_void_p(stream), _ptr(pos), C.byref(st)),
                       "lfr_plan_download")
        return pos, Library.stats_dict(st, bufs)

    def num_launches(self) -> int:
        return int(self.lib.lib.lfr_plan_num_launches(self.handle))

    def traffic(self, stream: int = 0):
        a, b = C.c_uint64(), C.c_uint64()
        self.lib.check(self.lib.lib.lfr_plan_traffic(self.handle, C.c_void_p(stream), C.byref(a), C.byref(b)),
                       "lfr_plan_traffic")
        return int(a.value), int(b.value)

    def close(self) -> None:
        if self.handle:
            self.lib.lib.lfr_plan_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_b200: Optional[Library] = None


def load_b200() -> Library:
    """The product library.  Raises if it has not been built."""
    global _b200
    if _b200 is None:
        _b200 = Library(B200_LIB_PATH)
        if _b200.backend != "b200":
            raise RuntimeError("lfr: %s is not the b200 backend" % B200_LIB_PATH)
    return _b200


_host: Optional[C.CDLL] = None


def load_host() -> C.CDLL:
    """The CPU-only host utilities (csrc/liblfr_host.so: protobuf wire codec, include/lfr_wire.h, and the
    host graph stage, include/lfr_host.h).  No CUDA dependency."""
    global _host
    if _host is None:
        if not os.path.exists(HOST_LIB_PATH):
            raise RuntimeError("lfr: %s is missing — build it first (python __graft_entry__.py build)" % HOST_LIB_PATH)
        _host = C.CDLL(HOST_LIB_PATH)
    return _host
