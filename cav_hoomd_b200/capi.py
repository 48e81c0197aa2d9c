"""ctypes binding of include/cavb200.h (libcavb200.so) -- no torch, no CUDA runtime of its own.

This is the Python host layer above the C ABI.  It never falls back to a CPU implementation: if
the shared library is missing or there is no CUDA device, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CAVB200_LIB") or os.path.join(_HERE, "lib", "libcavb200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "cavb200.h")


class CavbError(RuntimeError):
    """A libcavb200 call returned a non-zero cudaError_t."""

    def __init__(self, code: int, what: str, where: str):
        super().__init__(f"{where}: CUDA error {code}: {what}")
        self.code = code


class Params(C.Structure):
    """struct cavb200_params == cavity_force_params (reference src/CavityForceCompute.h:28-54)."""

    _fields_ = [("omegac", C.c_double), ("couplstr", C.c_double), ("K", C.c_double), ("phmass", C.c_double)]

    @classmethod
    def make(cls, omegac: float, couplstr: float, phmass: float = 1.0) -> "Params":
        # K = phmass * omegac * omegac, left to right (src/CavityForceCompute.h:38-42)
        return cls(omegac, couplstr, phmass * omegac * omegac, phmass)


class BussiArgs(C.Structure):
    """struct cavb200_bussi_args."""

    _fields_ = [("kT", C.c_double), ("tau", C.c_double), ("deltaT", C.c_double), ("dof", C.c_double),
                ("r_normal", C.c_double), ("gamma_draw", C.c_double)]


class LangevinArgs(C.Structure):
    """struct cavb200_langevin_args: the cavity mode's Langevin bath, the draws of ONE step two (r uniform in [-1, 1])."""

    _fields_ = [("gamma", C.c_double), ("kT", C.c_double), ("r", C.c_double * 3)]

    @classmethod
    def make(cls, gamma: float, kT: float, r) -> "LangevinArgs":
        return cls(gamma, kT, (C.c_double * 3)(*[float(x) for x in r]))


_vp = C.c_void_p
_u32 = C.c_uint32
_u64 = C.c_uint64
_dbl = C.c_double
_PP = C.POINTER(Params)
_BP = C.POINTER(BussiArgs)
_LP = C.POINTER(LangevinArgs)
_dp = C.POINTER(C.c_double)

_SIGNATURES = {
    "cavb200_version": (C.c_int, []),
    "cavb200_create": (C.c_int, [C.POINTER(_vp), C.c_int]),
    "cavb200_destroy": (C.c_int, [_vp]),
    "cavb200_error_string": (C.c_char_p, [C.c_int]),
    "cavb200_launch_count": (_u64, [_vp]),
    "cavb200_fault_count": (_u64, [_vp]),
    "cavb200_debug_stamps": (C.c_int, [_vp, C.POINTER(C.c_uint64), _u32]),
    "cavb200_debug_delay": (C.c_int, [_vp, _u64, _vp]),
    "cavb200_debug_fp64_peak": (C.c_int, [_vp, _dp]),
    "cavb200_debug_launch_ring": (C.c_int, [_vp, C.c_int, C.POINTER(C.c_uint64), _u32, C.POINTER(C.c_uint64)]),
    "cavb200_set_tuning": (C.c_int, [_vp, C.c_char_p, C.c_int]),
    "cavb200_get_tuning": (C.c_int, [_vp, C.c_char_p, C.POINTER(C.c_int)]),
    "cavb200_force": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _u32, _dbl, _dbl, _dbl, _u32, _PP, _vp]),
    "cavb200_force_read": (C.c_int, [_vp, _dp, _dp, C.POINTER(C.c_int32), _vp]),
    "cavb200_bussi": (C.c_int, [_vp, _vp, _vp, _u32, _u32, _BP, _vp]),
    "cavb200_bussi_ke": (C.c_int, [_vp, _vp, _vp, _u32, _u32, _vp]),
    "cavb200_bussi_read": (C.c_int, [_vp, _dp, _vp]),
    "cavb200_bussi_reset": (C.c_int, [_vp, _vp]),
    "cavb200_step": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _u32, _dbl, _dbl, _dbl, _u32, _PP, _u32, _u32, _BP, _vp]),
    "cavb200_nve_kick_drift": (C.c_int, [_vp, _vp, _vp, _vp, _u32, _dbl, _vp]),
    "cavb200_nve_half_kick": (C.c_int, [_vp, _vp, _vp, _u32, _dbl, _vp]),
    "cavb200_nvt_step_one": (C.c_int, [_vp, _vp, _vp, _vp, _u32, _dbl, _u32, _u32, _BP, _vp]),
    "cavb200_nvt_step_two": (C.c_int, [_vp, _vp, _vp, _u32, _dbl, _u32, _u32, _vp]),
    "cavb200_nve_kick_drift_wrap": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _u32, _dbl, _dbl, _dbl, _dbl, _vp]),
    "cavb200_nvt_step_one_wrap": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _u32, _dbl, _dbl, _dbl, _dbl, _u32, _u32, _BP, _vp]),
    "cavb200_nvt_step_one_rank1_wrap": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _u32, _dbl, _dbl, _dbl, _dbl, _u32, _dbl,
                                                  _u32, _u32, _BP, _vp]),
    "cavb200_md_step_one_wrap": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _u32, _dbl, _dbl, _dbl, _dbl, _u32, _PP, _u32, _u32,
                                           _BP, _vp]),
    "cavb200_md_step_fused_wrap": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _u32, _dbl, _dbl, _dbl, _dbl, _u32, _PP, _u32,
                                             _u32, _BP, _vp]),
    "cavb200_force_rank1": (C.c_int, [_vp, _vp, _vp, _vp, _u32, _dbl, _dbl, _dbl, _u32, _PP, _vp]),
    "cavb200_rank1_read": (C.c_int, [_vp, _dp, _dp, C.POINTER(C.c_int32), C.POINTER(_u32), _vp]),
    "cavb200_net_force_add_rank1": (C.c_int, [_vp, _vp, _vp, _vp, _u32, _u32, _dbl, _vp]),
    "cavb200_nvt_step_one_rank1": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _u32, _dbl, _u32, _dbl, _u32, _u32, _BP, _vp]),
    "cavb200_md_step_one": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _u32, _dbl, _dbl, _dbl, _dbl, _u32, _PP, _u32, _u32, _BP,
                                      _vp]),
    "cavb200_md_step_fused": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _u32, _dbl, _dbl, _dbl, _dbl, _u32, _PP, _u32, _u32, _BP,
                                        _vp]),
    "cavb200_nvt_step_two_rank1": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _u32, _dbl, _u32, _dbl, _u32, _u32, _vp]),
    "cavb200_nvt_step_two_rank1_bath": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _u32, _dbl, _u32, _dbl, _u32, _u32, _LP, _vp]),
    "cavb200_nvt_step_one_rank1_wrap_bath": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _u32, _dbl, _dbl, _dbl, _dbl, _u32,
                                                       _dbl, _u32, _u32, _BP, _vp]),
    "cavb200_md_step_one_wrap_bath": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _u32, _dbl, _dbl, _dbl, _dbl, _u32, _PP, _u32,
                                                _u32, _BP, _vp]),
    "cavb200_md_step_fused_wrap_bath": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _u32, _dbl, _dbl, _dbl, _dbl, _u32, _PP,
                                                  _u32, _u32, _BP, _LP, _vp]),
    "cavb200_group_set": (C.c_int, [_vp, _vp, _u32, _u32, _vp]),
    "cavb200_rank1_reindex": (C.c_int, [_vp, _vp, _u32, _u32, _vp]),
    "cavb200_track_open": (C.c_int, [_vp, _u32]),
    "cavb200_track_set_reference": (C.c_int, [_vp, _vp]),
    "cavb200_track_record": (C.c_int, [_vp, _u64, _vp, _u32, _vp]),
    "cavb200_track_read": (C.c_int, [_vp, _dp, _u32, C.POINTER(_u32), C.POINTER(_u64), _vp]),
    "cavb200_rhok": (C.c_int, [_vp, _vp, _u32, _u64, _u32, _u32, _vp, _u32, _vp, _vp]),
    "cavb200_rhok_f32": (C.c_int, [_vp, _vp, _u64, _u32, _u32, _vp, _u32, _vp, _vp]),
    "cavb200_fkt": (C.c_int, [_vp, _vp, _u32, _u32, _u32, _u32, _vp, _vp]),
    "cavb200_fkt_track_open": (C.c_int, [_vp, _dp, _u32, _u32, _u32, _u32]),
    "cavb200_fkt_track_step": (C.c_int, [_vp, _vp, _u32, _u64, _u32, _vp]),
    "cavb200_fkt_track_read": (C.c_int, [_vp, _dp, _u32, C.POINTER(_u32), C.POINTER(_u64), _vp]),
    "cavb200_shard_nccl_unique_id": (C.c_int, [_vp]),
    "cavb200_shard_init_nccl": (C.c_int, [_vp, _vp, C.c_int, C.c_int]),
    "cavb200_shard_mailbox_export": (C.c_int, [_vp, _vp]),
    "cavb200_shard_mailbox_open": (C.c_int, [_vp, _vp, C.c_int, C.c_int]),
    "cavb200_shard_set_mode": (C.c_int, [_vp, C.c_int]),
    "cavb200_shard_step": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _u32, _u64, _dbl, _dbl, _dbl, _u32, _PP, _u32, _u32,
                                     _BP, _vp]),
    "cavb200_step_host_submit": (C.c_int, [_vp, _u32, _vp, _vp, _vp, _vp, _vp, _u32, _dbl, _dbl, _dbl, _u32, _PP, _u32, _u32,
                                           _BP]),
    "cavb200_step_host_wait": (C.c_int, [_vp, _u32, _dp, _dp]),
    "cavb200_step_host_submit_ex": (C.c_int, [_vp, _u32, _vp, _vp, _vp, _vp, _vp, _u32, _dbl, _dbl, _dbl, _u32, _PP, _u32,
                                              _u32, _BP, _u32]),
    "cavb200_step_host_wait_ex": (C.c_int, [_vp, _u32, _dp, _dp, _dp]),
    "cavb200_step_host": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _u32, _dbl, _dbl, _dbl, _u32, _PP, _u32, _u32, _BP,
                                    _dp, _dp]),
    "cavb200_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "cavb200_dev_alloc": (C.c_int, [C.POINTER(_vp), _u64]),
    "cavb200_dev_free": (C.c_int, [_vp]),
    "cavb200_host_alloc": (C.c_int, [C.POINTER(_vp), _u64]),
    "cavb200_host_free": (C.c_int, [_vp]),
    "cavb200_memcpy_h2d": (C.c_int, [_vp, _vp, _u64, _vp]),
    "cavb200_memcpy_d2h": (C.c_int, [_vp, _vp, _u64, _vp]),
    "cavb200_memcpy_d2d": (C.c_int, [_vp, _vp, _u64, _vp]),
    "cavb200_memset": (C.c_int, [_vp, C.c_int, _u64, _vp]),
    "cavb200_stream_create": (C.c_int, [C.POINTER(_vp)]),
    "cavb200_stream_destroy": (C.c_int, [_vp]),
    "cavb200_stream_sync": (C.c_int, [_vp]),
    "cavb200_device_sync": (C.c_int, []),
    "cavb200_event_create": (C.c_int, [C.POINTER(_vp)]),
    "cavb200_event_destroy": (C.c_int, [_vp]),
    "cavb200_event_record": (C.c_int, [_vp, _vp]),
    "cavb200_event_elapsed_ms": (C.c_int, [_vp, _vp, C.POINTER(C.c_float)]),
    "cavb200_graph_begin": (C.c_int, [_vp]),
    "cavb200_graph_end": (C.c_int, [_vp, C.POINTER(_vp)]),
    "cavb200_graph_launch": (C.c_int, [_vp, _vp]),
    "cavb200_graph_destroy": (C.c_int, [_vp]),
}

_lib = None


def load() -> C.CDLL:
    """Load libcavb200.so (built in-tree by `make lib` / __graft_entry__.build()).  Raises if absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FileNotFoundError(
                f"{LIB_PATH} not built: run `make lib` (or __graft_entry__.build()). There is no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            if os.environ.get("CAVB200_LIB") and not hasattr(lib, name):
                continue  # A/B runs of tools/ against an older build of the library
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(code: int, where: str) -> None:
    if code != 0:
        raise CavbError(code, load().cavb200_error_string(code).decode(), where)


def device_count() -> int:
    n = C.c_int(0)
    code = load().cavb200_device_count(C.byref(n))
    return n.value if code == 0 else 0


# ---------------------------------------------------------------------------------------------
# device / pinned-host buffers
# ---------------------------------------------------------------------------------------------
class DeviceArray:
    """A typed device allocation (cudaMalloc through the library)."""

    def __init__(self, shape, dtype):
        self.shape = tuple(int(s) for s in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        self.dtype = np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape, dtype=np.int64)) * self.dtype.itemsize
        p = _vp()
        check(load().cavb200_dev_alloc(C.byref(p), self.nbytes), "cavb200_dev_alloc")
        self.ptr = p.value

    @classmethod
    def from_numpy(cls, a: np.ndarray, stream=None) -> "DeviceArray":
        a = np.ascontiguousarray(a)
        d = cls(a.shape, a.dtype)
        d.upload(a, stream)
        return d

    def upload(self, a: np.ndarray, stream=None) -> None:
        a = np.ascontiguousarray(a, dtype=self.dtype)
        assert a.nbytes == self.nbytes, (a.nbytes, self.nbytes)
        check(load().cavb200_memcpy_h2d(self.ptr, a.ctypes.data, self.nbytes, stream), "cavb200_memcpy_h2d")
        check(load().cavb200_stream_sync(stream), "cavb200_stream_sync")

    def numpy(self, stream=None) -> np.ndarray:
        out = np.empty(self.shape, self.dtype)
        if self.nbytes:
            check(load().cavb200_memcpy_d2h(out.ctypes.data, self.ptr, self.nbytes, stream), "cavb200_memcpy_d2h")
            check(load().cavb200_stream_sync(stream), "cavb200_stream_sync")
        return out

    def fill_bytes(self, value: int, stream=None) -> None:
        check(load().cavb200_memset(self.ptr, value, self.nbytes, stream), "cavb200_memset")

    def offset(self, nbytes: int) -> int:
        return self.ptr + int(nbytes)

    def free(self) -> None:
        if getattr(self, "ptr", None):
            load().cavb200_dev_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class PinnedArray:
    """Page-locked host memory exposed as a NumPy array (cudaMallocHost through the library)."""

    def __init__(self, shape, dtype):
        self.shape = tuple(int(s) for s in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        self.dtype = np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape, dtype=np.int64)) * self.dtype.itemsize
        p = _vp()
        check(load().cavb200_host_alloc(C.byref(p), self.nbytes), "cavb200_host_alloc")
        self.ptr = p.value
        buf = (C.c_char * max(self.nbytes, 1)).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape, dtype=np.int64))).reshape(self.shape)

    @classmethod
    def from_numpy(cls, a: np.ndarray) -> "PinnedArray":
        p = cls(a.shape, a.dtype)
        p.array[...] = a
        return p

    def free(self) -> None:
        if getattr(self, "ptr", None):
            self.array = None
            load().cavb200_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Stream:
    def __init__(self):
        p = _vp()
        check(load().cavb200_stream_create(C.byref(p)), "cavb200_stream_create")
        self.ptr = p.value

    def sync(self):
        check(load().cavb200_stream_sync(self.ptr), "cavb200_stream_sync")

    def __del__(self):
        try:
            if self.ptr:
                load().cavb200_stream_destroy(self.ptr)
        except Exception:
            pass


class Event:
    def __init__(self):
        p = _vp()
        check(load().cavb200_event_create(C.byref(p)), "cavb200_event_create")
        self.ptr = p.value

    def record(self, stream=None):
        check(load().cavb200_event_record(self.ptr, stream), "cavb200_event_record")

    def elapsed_ms_since(self, start: "Event") -> float:
        ms = C.c_float(0)
        check(load().cavb200_event_elapsed_ms(start.ptr, self.ptr, C.byref(ms)), "cavb200_event_elapsed_ms")
        return float(ms.value)

    def __del__(self):
        try:
            if self.ptr:
                load().cavb200_event_destroy(self.ptr)
        except Exception:
            pass


def _ptr(x):
    if x is None:
        return None
    if isinstance(x, (DeviceArray, PinnedArray)):
        return x.ptr
    if isinstance(x, np.ndarray):
        return x.ctypes.data
    return int(x)


# ---------------------------------------------------------------------------------------------
# handle
# ---------------------------------------------------------------------------------------------
class Handle:
    """cavb200_handle: owns the device workspace; bound to one device."""

    def __init__(self, device: int = 0):
        self.lib = load()
        h = _vp()
        check(self.lib.cavb200_create(C.byref(h), device), "cavb200_create")
        self.h = h.value
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.cavb200_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- tuning / counters -------------------------------------------------------------------
    def set_tuning(self, **kw):
        for k, v in kw.items():
            check(self.lib.cavb200_set_tuning(self.h, k.encode(), int(v)), f"cavb200_set_tuning({k})")

    def get_tuning(self, key: str) -> int:
        v = C.c_int(0)
        check(self.lib.cavb200_get_tuning(self.h, key.encode(), C.byref(v)), f"cavb200_get_tuning({key})")
        return v.value

    def debug_stamps(self, n_ctas: int) -> np.ndarray:
        out = np.zeros((n_ctas, 8), dtype=np.uint64)
        check(self.lib.cavb200_debug_stamps(self.h, out.ctypes.data_as(C.POINTER(C.c_uint64)), n_ctas),
              "cavb200_debug_stamps")
        return out

    def debug_delay(self, ns: int, stream=None):
        check(self.lib.cavb200_debug_delay(self.h, int(ns), stream), "cavb200_debug_delay")

    def debug_fp64_peak(self) -> float:
        """FP64 fused multiply-adds per second of the device (DFMA microbenchmark)."""
        v = C.c_double(0.0)
        check(self.lib.cavb200_debug_fp64_peak(self.h, C.byref(v)), "cavb200_debug_fp64_peak")
        return float(v.value)

    def debug_launch_ring(self, reset: bool = False, read: bool = True):
        """-> (ring uint64[2048, 2] of {start, end} ns, epoch of the last launch); tuning stamps = 2."""
        out = np.zeros((2048, 2), dtype=np.uint64)
        ep = C.c_uint64(0)
        check(self.lib.cavb200_debug_launch_ring(self.h, int(reset), out.ctypes.data_as(C.POINTER(C.c_uint64)) if read else None,
                                                 2048 if read else 0, C.byref(ep)), "cavb200_debug_launch_ring")
        return out, int(ep.value)

    @property
    def launch_count(self) -> int:
        return int(self.lib.cavb200_launch_count(self.h))

    @property
    def fault_count(self) -> int:
        return int(self.lib.cavb200_fault_count(self.h))

    # -- cavity force ------------------------------------------------------------------------
    def force(self, pos, charge, image, force, N, box, L_typeid, params: Params, stream=None):
        check(self.lib.cavb200_force(self.h, _ptr(pos), _ptr(charge), _ptr(image), _ptr(force), N, box[0], box[1],
                                     box[2], L_typeid & 0xFFFFFFFF, C.byref(params), stream), "cavb200_force")

    def force_read(self, stream=None):
        en = (C.c_double * 3)()
        dip = (C.c_double * 3)()
        ph = C.c_int32(0)
        check(self.lib.cavb200_force_read(self.h, en, dip, C.byref(ph), stream), "cavb200_force_read")
        return np.array(en[:]), np.array(dip[:]), int(ph.value)

    # -- Bussi ---------------------------------------------------------------------------------
    def bussi(self, vel, group_idx, group_first, n, args: BussiArgs, stream=None):
        check(self.lib.cavb200_bussi(self.h, _ptr(vel), _ptr(group_idx), group_first, n, C.byref(args), stream),
              "cavb200_bussi")

    def bussi_ke(self, vel, group_idx, group_first, n, stream=None):
        check(self.lib.cavb200_bussi_ke(self.h, _ptr(vel), _ptr(group_idx), group_first, n, stream), "cavb200_bussi_ke")

    def bussi_read(self, stream=None):
        out = (C.c_double * 5)()
        check(self.lib.cavb200_bussi_read(self.h, out, stream), "cavb200_bussi_read")
        return dict(ke=out[0], alpha=out[1], instantaneous=out[2], cumulative=out[3], err=out[4])

    def bussi_reset(self, stream=None):
        check(self.lib.cavb200_bussi_reset(self.h, stream), "cavb200_bussi_reset")

    # -- fused step ----------------------------------------------------------------------------
    def step(self, pos, charge, image, force, vel, N, box, L_typeid, params, group_first, n_group, bussi, stream=None):
        check(self.lib.cavb200_step(self.h, _ptr(pos), _ptr(charge), _ptr(image), _ptr(force), _ptr(vel), N, box[0],
                                    box[1], box[2], L_typeid & 0xFFFFFFFF, C.byref(params), group_first, n_group,
                                    C.byref(bussi), stream), "cavb200_step")

    def step_host(self, pos, charge, image, force, vel, N, box, L_typeid, params, group_first, n_group, bussi):
        en = (C.c_double * 3)()
        bo = (C.c_double * 5)()
        check(self.lib.cavb200_step_host(self.h, _ptr(pos), _ptr(charge), _ptr(image), _ptr(force), _ptr(vel), N,
                                         box[0], box[1], box[2], L_typeid & 0xFFFFFFFF, C.byref(params), group_first,
                                         n_group, C.byref(bussi), en, bo), "cavb200_step_host")
        return np.array(en[:]), dict(ke=bo[0], alpha=bo[1], instantaneous=bo[2], cumulative=bo[3], err=bo[4])

    def step_host_submit(self, slot, pos, charge, image, force, vel, N, box, L_typeid, params, group_first, n_group,
                         bussi):
        check(self.lib.cavb200_step_host_submit(self.h, slot, _ptr(pos), _ptr(charge), _ptr(image), _ptr(force),
                                                _ptr(vel), N, box[0], box[1], box[2], L_typeid & 0xFFFFFFFF,
                                                C.byref(params), group_first, n_group, C.byref(bussi)),
              "cavb200_step_host_submit")

    HOST_KEEP_CHARGE, HOST_KEEP_IMAGE, HOST_RANK1_RESULT = 1, 2, 4

    def step_host_submit_ex(self, slot, pos, charge, image, force, vel, N, box, L_typeid, params, group_first, n_group,
                            bussi, flags):
        check(self.lib.cavb200_step_host_submit_ex(self.h, slot, _ptr(pos), _ptr(charge), _ptr(image), _ptr(force),
                                                   _ptr(vel), N, box[0], box[1], box[2], L_typeid & 0xFFFFFFFF,
                                                   C.byref(params), group_first, n_group, C.byref(bussi), flags),
              "cavb200_step_host_submit_ex")

    def step_host_wait_ex(self, slot):
        """-> (energies[3], bussi dict, rank1 dict {Dq[2], F_L[3], photon_idx})"""
        en, bo, r1 = (C.c_double * 3)(), (C.c_double * 5)(), (C.c_double * 6)()
        check(self.lib.cavb200_step_host_wait_ex(self.h, slot, en, bo, r1), "cavb200_step_host_wait_ex")
        return (np.array(en[:]), dict(ke=bo[0], alpha=bo[1], instantaneous=bo[2], cumulative=bo[3], err=bo[4]),
                dict(Dq=np.array(r1[0:2]), F_L=np.array(r1[2:5]), photon_idx=int(r1[5])))

    def step_host_wait(self, slot):
        en = (C.c_double * 3)()
        bo = (C.c_double * 5)()
        check(self.lib.cavb200_step_host_wait(self.h, slot, en, bo), "cavb200_step_host_wait")
        return np.array(en[:]), dict(ke=bo[0], alpha=bo[1], instantaneous=bo[2], cumulative=bo[3], err=bo[4])

    # -- NVE harness ------------------------------------------------------------------------------
    def nve_kick_drift(self, pos, vel, force, N, dt, stream=None, image=None, box=None):
        """image / box given: the drift is followed by the box wrap + image update (cavb200_nve_kick_drift_wrap)."""
        if image is not None:
            check(self.lib.cavb200_nve_kick_drift_wrap(self.h, _ptr(pos), _ptr(vel), _ptr(force), _ptr(image), N, dt,
                                                       box[0], box[1], box[2], stream), "cavb200_nve_kick_drift_wrap")
            return
        check(self.lib.cavb200_nve_kick_drift(self.h, _ptr(pos), _ptr(vel), _ptr(force), N, dt, stream),
              "cavb200_nve_kick_drift")

    def nvt_step_one(self, pos, vel, force, N, dt, group_first, n_group, bussi=None, stream=None, image=None, box=None):
        b = C.byref(bussi) if bussi is not None else None
        if image is not None:
            check(self.lib.cavb200_nvt_step_one_wrap(self.h, _ptr(pos), _ptr(vel), _ptr(force), _ptr(image), N, dt, box[0],
                                                     box[1], box[2], group_first, n_group, b, stream),
                  "cavb200_nvt_step_one_wrap")
            return
        check(self.lib.cavb200_nvt_step_one(self.h, _ptr(pos), _ptr(vel), _ptr(force), N, dt, group_first, n_group,
                                            b, stream), "cavb200_nvt_step_one")

    def nvt_step_two(self, vel, force, N, dt, group_first, n_group, stream=None):
        check(self.lib.cavb200_nvt_step_two(self.h, _ptr(vel), _ptr(force), N, dt, group_first, n_group, stream),
              "cavb200_nvt_step_two")

    # -- rank-1 cavity force (SURVEY.md 8f.2) ---------------------------------------------------
    def force_rank1(self, pos, charge, image, N, box, L_typeid, params: Params, stream=None):
        check(self.lib.cavb200_force_rank1(self.h, _ptr(pos), _ptr(charge), _ptr(image), N, box[0], box[1], box[2],
                                           L_typeid & 0xFFFFFFFF, C.byref(params), stream), "cavb200_force_rank1")

    def rank1_read(self, stream=None):
        dq, fl = (C.c_double * 2)(), (C.c_double * 3)()
        ph, nl = C.c_int32(0), C.c_uint32(0)
        check(self.lib.cavb200_rank1_read(self.h, dq, fl, C.byref(ph), C.byref(nl), stream), "cavb200_rank1_read")
        return np.array(dq[:]), np.array(fl[:]), int(ph.value), int(nl.value)

    def net_force_add_rank1(self, net_force, charge, pos, N, L_typeid, couplstr, stream=None):
        check(self.lib.cavb200_net_force_add_rank1(self.h, _ptr(net_force), _ptr(charge), _ptr(pos), N,
                                                   L_typeid & 0xFFFFFFFF, couplstr, stream),
              "cavb200_net_force_add_rank1")

    # bath=: the cavity mode's Langevin bath (cavb200_*_bath).  Step one takes bath=True (the photon's kick adds the bath
    # force the last step two stored); step two and the fused step take the LangevinArgs of the step two they perform.
    # The bath entry points exist for the wrapped steps only.
    def nvt_step_one_rank1(self, pos, vel, force_other, charge, N, dt, L_typeid, couplstr, group_first, n_group,
                           bussi=None, stream=None, image=None, box=None, bath=False):
        if bath and image is None:
            raise ValueError("the photon bath comes with the box wrap only (image=, box=)")
        if image is not None:
            fn = self.lib.cavb200_nvt_step_one_rank1_wrap_bath if bath else self.lib.cavb200_nvt_step_one_rank1_wrap
            check(fn(self.h, _ptr(pos), _ptr(vel), _ptr(force_other), _ptr(charge), _ptr(image), N, dt, box[0], box[1],
                     box[2], L_typeid & 0xFFFFFFFF, couplstr, group_first, n_group,
                     C.byref(bussi) if bussi is not None else None, stream),
                  fn.__name__)
            return
        check(self.lib.cavb200_nvt_step_one_rank1(self.h, _ptr(pos), _ptr(vel), _ptr(force_other), _ptr(charge), N, dt,
                                                  L_typeid & 0xFFFFFFFF, couplstr, group_first, n_group,
                                                  C.byref(bussi) if bussi is not None else None, stream),
              "cavb200_nvt_step_one_rank1")

    def md_step_one(self, pos, vel, force_other, charge, image, N, dt, box, L_typeid, params, group_first, n_group,
                    bussi=None, stream=None, wrap=False, bath=False):
        if bath and not wrap:
            raise ValueError("the photon bath comes with the box wrap only (wrap=True)")
        fn = self.lib.cavb200_md_step_one_wrap_bath if bath else (
            self.lib.cavb200_md_step_one_wrap if wrap else self.lib.cavb200_md_step_one)
        check(fn(self.h, _ptr(pos), _ptr(vel), _ptr(force_other), _ptr(charge), _ptr(image), N,
                                           dt, box[0], box[1], box[2], L_typeid & 0xFFFFFFFF, C.byref(params), group_first,
                                           n_group, C.byref(bussi) if bussi is not None else None, stream),
              "cavb200_md_step_one")

    def md_step_fused(self, pos, vel, force_other, charge, image, N, dt, box, L_typeid, params, group_first, n_group,
                      bussi=None, stream=None, wrap=False, bath=None):
        """bath: LangevinArgs of the deferred step two (the previous step's draws)."""
        bussi_p = C.byref(bussi) if bussi is not None else None
        if bath is not None:
            if not wrap:
                raise ValueError("the photon bath comes with the box wrap only (wrap=True)")
            check(self.lib.cavb200_md_step_fused_wrap_bath(self.h, _ptr(pos), _ptr(vel), _ptr(force_other), _ptr(charge),
                                                           _ptr(image), N, dt, box[0], box[1], box[2],
                                                           L_typeid & 0xFFFFFFFF, C.byref(params), group_first, n_group,
                                                           bussi_p, C.byref(bath), stream),
                  "cavb200_md_step_fused_wrap_bath")
            return
        fn = self.lib.cavb200_md_step_fused_wrap if wrap else self.lib.cavb200_md_step_fused
        check(fn(self.h, _ptr(pos), _ptr(vel), _ptr(force_other), _ptr(charge), _ptr(image), N,
                                             dt, box[0], box[1], box[2], L_typeid & 0xFFFFFFFF, C.byref(params),
                                             group_first, n_group, bussi_p, stream),
              "cavb200_md_step_fused")

    def nvt_step_two_rank1(self, vel, force_other, charge, pos, N, dt, L_typeid, couplstr, group_first, n_group,
                           stream=None, bath=None):
        """bath: LangevinArgs of this step two."""
        if bath is not None:
            check(self.lib.cavb200_nvt_step_two_rank1_bath(self.h, _ptr(vel), _ptr(force_other), _ptr(charge), _ptr(pos),
                                                           N, dt, L_typeid & 0xFFFFFFFF, couplstr, group_first, n_group,
                                                           C.byref(bath), stream),
                  "cavb200_nvt_step_two_rank1_bath")
            return
        check(self.lib.cavb200_nvt_step_two_rank1(self.h, _ptr(vel), _ptr(force_other), _ptr(charge), _ptr(pos), N, dt,
                                                  L_typeid & 0xFFFFFFFF, couplstr, group_first, n_group, stream),
              "cavb200_nvt_step_two_rank1")

    # -- index-list groups and particle sorts ----------------------------------------------------
    GROUP_MASK = 0xFFFFFFFF  # CAVB200_GROUP_MASK: pass as group_first to thermostat the mask of the last group_set

    def group_set(self, group_idx, n, N, stream=None):
        """Build the handle's group mask from the device index list group_idx (uint32[n]) of N particles (blocking)."""
        check(self.lib.cavb200_group_set(self.h, _ptr(group_idx), n, N, stream), "cavb200_group_set")

    def rank1_reindex(self, pos, N, L_typeid, stream=None):
        """After a permutation of the particle arrays: move the photon index of the last rank-1 result (blocking)."""
        check(self.lib.cavb200_rank1_reindex(self.h, _ptr(pos), N, L_typeid & 0xFFFFFFFF, stream), "cavb200_rank1_reindex")

    # -- device-side trackers (SURVEY.md 8f.4) --------------------------------------------------
    TRACK_FIELDS = ("timestep", "dx", "dy", "dz", "qx", "qy", "qz", "harmonic", "coupling", "dipole_self", "autocorr",
                    "cavity_ke", "group_ke", "alpha", "reservoir", "photon_idx")

    def track_open(self, capacity: int):
        check(self.lib.cavb200_track_open(self.h, capacity), "cavb200_track_open")

    def track_set_reference(self, stream=None):
        check(self.lib.cavb200_track_set_reference(self.h, stream), "cavb200_track_set_reference")

    def track_record(self, timestep: int, vel, N: int, stream=None):
        check(self.lib.cavb200_track_record(self.h, timestep, _ptr(vel), N, stream), "cavb200_track_record")

    def track_read(self, max_records: int, stream=None):
        """-> (records float64[n, 16] oldest first, total appended since open)"""
        out = np.zeros((max(max_records, 1), 16), dtype=np.float64)
        n, total = C.c_uint32(0), C.c_uint64(0)
        check(self.lib.cavb200_track_read(self.h, out.ctypes.data_as(_dp), max_records, C.byref(n), C.byref(total), stream),
              "cavb200_track_read")
        return out[:n.value], int(total.value)

    def nve_half_kick(self, vel, force, N, dt, stream=None):
        check(self.lib.cavb200_nve_half_kick(self.h, _ptr(vel), _ptr(force), N, dt, stream), "cavb200_nve_half_kick")

    # -- F(k,t) ----------------------------------------------------------------------------------
    def rhok(self, pos, stride, frame_stride, N, T, kvec, K, rho, stream=None):
        check(self.lib.cavb200_rhok(self.h, _ptr(pos), stride, frame_stride, N, T, _ptr(kvec), K, _ptr(rho), stream),
              "cavb200_rhok")

    def rhok_f32(self, pos_xyz, frame_stride, N, T, kvec, K, rho, stream=None):
        check(self.lib.cavb200_rhok_f32(self.h, _ptr(pos_xyz), frame_stride, N, T, _ptr(kvec), K, _ptr(rho), stream),
              "cavb200_rhok_f32")

    def fkt(self, rho, T, K, n_origins, n_lags, out, stream=None):
        check(self.lib.cavb200_fkt(self.h, _ptr(rho), T, K, n_origins, n_lags, _ptr(out), stream), "cavb200_fkt")

    # -- F(k,t) tracker without snapshots -----------------------------------------------------------
    FKT_RECORD, FKT_ADD_REFERENCE = 1, 2  # CAVB200_FKT_RECORD, CAVB200_FKT_ADD_REFERENCE

    def fkt_track_open(self, kvec, max_references: int, capacity: int, N: int):
        """kvec: host wave vectors [K, 3].  Blocking; drops every stored reference and empties the ring."""
        k = np.ascontiguousarray(kvec, dtype=np.float64).reshape(-1, 3)
        check(self.lib.cavb200_fkt_track_open(self.h, k.ctypes.data_as(_dp), k.shape[0], max_references, capacity, N),
              "cavb200_fkt_track_open")
        self._fkt_words = 2 + int(max_references) + 2 * k.shape[0]

    def fkt_track_step(self, pos, N: int, timestep: int, flags: int, stream=None):
        check(self.lib.cavb200_fkt_track_step(self.h, _ptr(pos), N, timestep, flags, stream), "cavb200_fkt_track_step")

    def fkt_track_read(self, max_records: int, stream=None):
        """-> (records float64[n, 2 + max_references + 2K] oldest first, total appended since open)"""
        words = getattr(self, "_fkt_words", 1)
        out = np.zeros((max(max_records, 1), words), dtype=np.float64)
        n, total = C.c_uint32(0), C.c_uint64(0)
        check(self.lib.cavb200_fkt_track_read(self.h, out.ctypes.data_as(_dp), max_records, C.byref(n), C.byref(total),
                                              stream), "cavb200_fkt_track_read")
        return out[:n.value], int(total.value)

    # -- sharded ---------------------------------------------------------------------------------
    def nccl_unique_id(self) -> bytes:
        buf = (C.c_char * 128)()
        check(self.lib.cavb200_shard_nccl_unique_id(buf), "cavb200_shard_nccl_unique_id")
        return bytes(buf)

    def shard_init_nccl(self, unique_id: bytes, rank: int, nranks: int):
        buf = (C.c_char * 128).from_buffer_copy(unique_id)
        check(self.lib.cavb200_shard_init_nccl(self.h, buf, rank, nranks), "cavb200_shard_init_nccl")

    def shard_mailbox_export(self) -> bytes:
        buf = (C.c_char * 64)()
        check(self.lib.cavb200_shard_mailbox_export(self.h, buf), "cavb200_shard_mailbox_export")
        return bytes(buf)

    def shard_mailbox_open(self, handles: list, rank: int, nranks: int):
        blob = b"".join(handles)
        buf = (C.c_char * len(blob)).from_buffer_copy(blob)
        check(self.lib.cavb200_shard_mailbox_open(self.h, buf, rank, nranks), "cavb200_shard_mailbox_open")

    def shard_set_mode(self, mode: int):
        check(self.lib.cavb200_shard_set_mode(self.h, mode), "cavb200_shard_set_mode")

    def shard_step(self, pos, charge, image, force, vel, N_local, index_offset, box, L_typeid, params, group_first,
                   n_group, bussi, stream=None):
        check(self.lib.cavb200_shard_step(self.h, _ptr(pos), _ptr(charge), _ptr(image), _ptr(force), _ptr(vel), N_local,
                                          index_offset, box[0], box[1], box[2], L_typeid & 0xFFFFFFFF, C.byref(params),
                                          group_first, n_group, C.byref(bussi), stream), "cavb200_shard_step")

    # -- graphs ----------------------------------------------------------------------------------
    def graph_capture(self, stream, fn):
        """Capture the calls made by fn() on `stream` into an executable graph."""
        check(self.lib.cavb200_graph_begin(stream), "cavb200_graph_begin")
        try:
            fn()
        finally:
            g = _vp()
            code = self.lib.cavb200_graph_end(stream, C.byref(g))
        check(code, "cavb200_graph_end")
        return g.value

    def graph_launch(self, graph, stream):
        check(self.lib.cavb200_graph_launch(graph, stream), "cavb200_graph_launch")

    def graph_destroy(self, graph):
        self.lib.cavb200_graph_destroy(graph)


def sync():
    check(load().cavb200_device_sync(), "cavb200_device_sync")
