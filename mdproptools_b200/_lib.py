"""ctypes binding of libmdprop_b200.so (the C ABI declared in include/mdprop_b200.h).

There is no CPU fallback: importing the package works anywhere (so that host-only helpers and the
CPU test-suite can run), but the first call that needs the device raises ``MdpropError`` when the shared
library is missing or no sm_100 GPU is present.
"""
from __future__ import annotations

import ctypes
import os
import threading
from ctypes import POINTER, c_char_p, c_double, c_int, c_int32, c_int64, c_uint64, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmdprop_b200.so")

MDP_PAIR_NO_CULL = 1
MDP_PAIR_NO_SORT = 2


class MdpropError(RuntimeError):
    pass


_lib = None
_lib_lock = threading.Lock()

_PROTOS = {
    "mdp_version": (c_int, []),
    "mdp_last_error": (c_char_p, []),
    "mdp_ctx_create": (c_int, [c_int, POINTER(c_void_p)]),
    "mdp_ctx_destroy": (None, [c_void_p]),
    "mdp_ctx_scratch_bytes": (c_int64, [c_void_p]),
    "mdp_ctx_set_scratch_limit": (c_int, [c_void_p, c_int64]),
    "mdp_ctx_launch_count": (c_int64, [c_void_p]),
    "mdp_ctx_pair_stats": (c_int, [c_void_p, POINTER(c_int64)]),
    "mdp_ctx_timing": (c_int, [c_void_p, c_int]),
    "mdp_ctx_timing_read": (c_int, [c_void_p, c_int, POINTER(c_double), POINTER(c_int64)]),
    "mdp_bin_edges": (c_int, [c_double, c_int, POINTER(c_double)]),
    "mdp_pair_hist": (c_int, [c_void_p, c_int,
                              c_int64, c_void_p, c_void_p, c_int64, c_int,
                              c_int64, c_void_p, c_void_p, c_int64, c_int,
                              POINTER(c_double), c_double, POINTER(c_double), c_int, c_double,
                              c_void_p, c_int, c_void_p]),
    "mdp_hist_reduce": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, POINTER(c_int32), c_int, c_void_p,
                                c_void_p]),
    "mdp_unique_pair_keys": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p]),
    "mdp_list_group": (c_int, [c_void_p, c_int, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "mdp_hydration_count": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, POINTER(c_double),
                                    c_int64, c_void_p, c_double, c_void_p, c_void_p, c_void_p, c_void_p]),
    "mdp_cluster_members": (c_int, [c_void_p, c_int, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_double, c_double,
                                    c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "mdp_shell_search": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_int64, c_void_p, POINTER(c_double), c_double, c_double,
                                 c_int, c_int, c_void_p, c_int64, c_void_p, c_void_p]),
    "mdp_pair_list": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_int64, c_void_p, POINTER(c_double), c_double,
                              c_double, c_int, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_int, c_void_p]),
    "mdp_segment_com": (c_int, [c_void_p, c_int, c_int, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p,
                                c_void_p, c_void_p, c_void_p, c_void_p]),
    "mdp_msd_single_origin": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_double, POINTER(c_int64), c_int,
                                      c_void_p, c_void_p, c_void_p]),
    "mdp_msd_interval": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_double, c_int, c_void_p, c_void_p]),
    "mdp_msd_all_origins": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_double, POINTER(c_int64), c_int, c_int,
                                    c_void_p, c_void_p]),
    "mdp_charge_flux": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_void_p,
                                POINTER(c_int64), c_int, c_double, c_double, c_void_p, c_int64, c_int64, c_void_p]),
    "mdp_xcorr_unbiased": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "mdp_xcorr_fft": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "mdp_cross_msd_fft": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_int, POINTER(c_int64), c_int64, c_void_p,
                                  c_void_p]),
    "mdp_group_acf_fft": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_int, POINTER(c_int64), c_int64, c_void_p, c_void_p]),
    "mdp_structure_factor": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_int64, c_int, POINTER(c_double), c_int64,
                                     POINTER(c_int32), c_int, POINTER(c_int64), c_void_p, c_void_p]),
    "mdp_sk_rho": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_int64, c_int, POINTER(c_double), c_int64, POINTER(c_int32),
                           c_void_p, c_int64, c_int64, c_void_p]),
    "mdp_isf_fft": (c_int, [c_void_p, c_int, c_int64, c_int64, c_void_p, c_int, POINTER(c_int32), c_int, POINTER(c_int64), c_int64,
                            c_void_p, c_void_p]),
    "mdp_orient_series": (c_int, [c_void_p, c_int, c_int64, c_void_p, POINTER(c_double), c_int, c_int64, POINTER(c_int32), c_void_p,
                                  c_int64, c_int64, c_void_p]),
    "mdp_cumtrapz": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_double, c_double, c_int, c_void_p, c_void_p]),
    "mdp_bitmask_fill": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "mdp_bitmask_autocorr": (c_int, [c_void_p, c_int64, c_int, c_int64, c_void_p, c_void_p, c_void_p]),
    "mdp_survival_runs": (c_int, [c_void_p, c_int64, c_int, c_int64, c_void_p, c_void_p, c_void_p]),
    "mdp_axis_density": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_double, c_int, POINTER(c_double), c_double,
                                 c_double, c_int, c_void_p, c_void_p, c_void_p]),
    "mdp_ols_sums": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "mdp_dump_scan": (c_int64, [c_char_p, c_int64, POINTER(c_int64), c_int64]),
    "mdp_dump_header": (c_int, [c_char_p, c_int64, POINTER(c_double), c_char_p, c_int]),
    "mdp_dump_parse": (c_int, [c_char_p, c_int64, POINTER(c_char_p), c_int, c_void_p, c_int64, POINTER(c_double),
                               c_int]),
    "mdp_dump_parse_device": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int,
                                      POINTER(c_int), c_int, c_int, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p]),
    "mdp_dump_parse_batch": (c_int, [c_int, POINTER(c_char_p), POINTER(c_int64), POINTER(c_char_p), c_int, c_void_p, c_int64,
                                     c_int64, POINTER(c_double), c_int]),
}

EXPORTED_SYMBOLS = tuple(_PROTOS)

PAIR_NO_CULL, PAIR_NO_SORT, PAIR_TRICLINIC, PAIR_F64 = 1, 2, 4, 16   # flags of mdp_pair_hist / mdp_pair_list
SK_NLIM, SK_MAX_CLASSES, SK_EPS = 1024, 64, 1e-5       # mdp_structure_factor: Miller bound, classes, accuracy (csrc/sk_phase.h)
ORIENT_KINDS = {"bond": 0, "bisector": 1, "normal": 2}  # mdp_orient_series: vector kinds (csrc/orient.h)


def lib() -> ctypes.CDLL:
    """Load the shared library (building it in-tree first if the sources are newer and nvcc exists)."""
    global _lib
    with _lib_lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                try:
                    from . import build as _build
                    _build.build()
                except Exception as exc:  # noqa: BLE001
                    raise MdpropError(
                        f"libmdprop_b200.so is missing and could not be built ({exc}); run "
                        "`python -m mdproptools_b200.build` -- there is no CPU fallback") from exc
            try:
                cdll = ctypes.CDLL(LIB_PATH)
            except OSError as exc:
                raise MdpropError(f"cannot load {LIB_PATH}: {exc}") from exc
            for name, (res, args) in _PROTOS.items():
                fn = getattr(cdll, name)
                fn.restype = res
                fn.argtypes = args
            _lib = cdll
    return _lib


def last_error() -> str:
    msg = lib().mdp_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        raise MdpropError(f"{what or 'libmdprop_b200'} failed (rc={rc}): {last_error()}")


class Context:
    """One mdp_ctx per (process, device)."""

    _instances: dict[int, "Context"] = {}
    _lock = threading.Lock()         # the file pipeline's producer thread and the caller may both ask first

    def __init__(self, device: int):
        h = c_void_p()
        check(lib().mdp_ctx_create(int(device), ctypes.byref(h)), "mdp_ctx_create")
        self.handle = h
        self.device = int(device)

    @classmethod
    def get(cls, device: int | None = None) -> "Context":
        import torch

        if not torch.cuda.is_available():
            raise MdpropError("no CUDA device is visible: mdproptools_b200 has no CPU fallback")
        if device is None:
            device = torch.cuda.current_device()
        ctx = cls._instances.get(device)
        if ctx is None:
            with cls._lock:
                ctx = cls._instances.get(device)
                if ctx is None:
                    ctx = cls._instances[device] = Context(device)
        return ctx

    def launch_count(self) -> int:
        return int(lib().mdp_ctx_launch_count(self.handle))

    def scratch_bytes(self) -> int:
        return int(lib().mdp_ctx_scratch_bytes(self.handle))

    def timing(self, enable: bool) -> None:
        check(lib().mdp_ctx_timing(self.handle, 1 if enable else 0), "mdp_ctx_timing")

    def timing_read(self, tag: int):
        """(total milliseconds, launches) of the kernels recorded under ``tag`` since the last read."""
        ms, n = c_double(), c_int64()
        check(lib().mdp_ctx_timing_read(self.handle, int(tag), ctypes.byref(ms), ctypes.byref(n)), "mdp_ctx_timing_read")
        return float(ms.value), int(n.value)

    def pair_stats(self) -> dict:
        out = (c_int64 * 4)()
        check(lib().mdp_ctx_pair_stats(self.handle, out), "mdp_ctx_pair_stats")
        return {"items": int(out[0]), "nominal_tile_pairs": int(out[1]), "pair_evals": int(out[2]),
                "exact_path_pairs": int(out[3])}    # pairs k_pair_fast settled in fp64 (0 for the all-fp64 kernel)


def ptr(t):
    """device pointer of a torch tensor (or None)."""
    return None if t is None else c_void_p(t.data_ptr())


def stream_ptr():
    import torch

    return c_void_p(torch.cuda.current_stream().cuda_stream)


def dptr(a: np.ndarray):
    return a.ctypes.data_as(POINTER(c_double))


_EDGES: dict = {}


def bin_edges(ddr: float, nb: int) -> np.ndarray:
    """Host-only: exact rsq thresholds of bin(rsq) = int(sqrt(rsq)/ddr) (rdf_cn.py:68,85).  Cached per (ddr, nb); the
    returned array is read-only."""
    key = (float(ddr), int(nb))
    e = _EDGES.get(key)
    if e is None:
        e = np.empty(nb + 1, dtype=np.float64)
        check(lib().mdp_bin_edges(float(ddr), int(nb), dptr(e)), "mdp_bin_edges")
        e.setflags(write=False)
        if len(_EDGES) > 64:
            _EDGES.clear()
        _EDGES[key] = e
    return e
