"""Bridge registry: loads the native sm_100a library and exposes its C ABI.

Counterpart of /root/reference/mpi4jax/_src/xla_bridge/__init__.py:1-174, which
imports the nanobind modules, checks the MPI ABI, fans ``set_logging`` out to every
extension and registers 12 XLA FFI targets per platform.  Here there is one shared
library (``mpi4jax_b200/_native/libb2mpi.so``) bound through ``ctypes``; the "targets"
are the ``b2_*`` entry points listed in ``csrc/b2_runtime.h``.  There is no MPI, so
the ABI check degenerates to a build-info record (``NATIVE_ABI_INFO``).

``HAS_CUDA_EXT`` is True when the library could be loaded (it loads on GPU-less
hosts too: the CUDA driver is resolved lazily).  Ops on CUDA tensors fail loudly
when it is False -- there is no silent PyTorch fallback on the GPU path.
"""

from __future__ import annotations

import ctypes
import os
import sys
from ctypes import (
    CFUNCTYPE,
    POINTER,
    Structure,
    c_char_p,
    c_double,
    c_float,
    c_int,
    c_longlong,
    c_size_t,
    c_void_p,
)
from pathlib import Path

from ..decorators import env_flag
from . import codes  # noqa: F401

_LIB_PATH = Path(__file__).resolve().parents[2] / "_native" / "libb2mpi.so"

HAS_CUDA_EXT = False
HAS_XPU_EXT = False  # the reference has an Intel XPU bridge; B200 does not
CUDA_EXT_ERROR = ""
lib = None


class B2HaloDesc(Structure):
    _fields_ = [
        ("nfields", c_int),
        ("field", c_void_p * 8),
        ("kind", c_int * 8),
        ("ny", c_int),
        ("nx", c_int),
        ("pitch", c_int),
        ("west", c_int),
        ("east", c_int),
        ("south", c_int),
        ("north", c_int),
        ("sw", c_int),
        ("se", c_int),
        ("nw", c_int),
        ("ne", c_int),
        ("periodic_x", c_int),
        ("at_east_wall", c_int),
        ("at_north_wall", c_int),
    ]


class B2Strided(Structure):
    """Layout of a non-contiguous input of a data-movement collective (csrc/b2_runtime.h)."""
    _fields_ = [
        ("nd", c_int),
        ("esize", c_int),
        ("shape", c_longlong * 4),
        ("stride", c_longlong * 4),
        ("blk_stride", c_longlong),
    ]


class B2SweParams(Structure):
    _fields_ = [
        ("ny", c_int),
        ("nx", c_int),
        ("pitch", c_int),
        ("dx", c_float),
        ("dy", c_float),
        ("dt", c_float),
        ("gravity", c_float),
        ("viscosity", c_float),
        ("rdx", c_float),
        ("rdy", c_float),
        ("ab_a", c_float),
        ("ab_b", c_float),
        ("first_step", c_int),
        ("south_wall", c_int),
        ("north_wall", c_int),
        ("coriolis", c_void_p),
        ("c_gx", c_float), ("c_gy", c_float),        # folded constants, see csrc/b2_swe_body.cuh
        ("c_nux", c_float), ("c_nuy", c_float),
        ("c_fx", c_float), ("c_fy", c_float),
    ]


class B2SweState(Structure):
    _fields_ = [(name, c_void_p) for name in
                ("h0", "h1", "u", "v", "dh", "du", "dv", "fe", "fn", "q", "ke", "fe2", "fn2", "u1", "v1")]


class B2SweCA(Structure):
    _fields_ = [(name, c_void_p) for name in ("hx", "upx", "vpx", "uppx", "vppx")] + [
        ("epitch", c_int), ("cb1", c_int)]


class B2StatusRecord(Structure):
    _fields_ = [
        ("source", c_int),
        ("tag", c_int),
        ("count_bytes", c_longlong),
        ("error", c_int),
        ("ready", c_int),
    ]


_PRINT_CB = CFUNCTYPE(None, c_char_p)


def _py_print(msg: bytes) -> None:
    # routed through sys.stdout so pytest's capsys / notebooks see native log lines
    sys.stdout.write(msg.decode("utf-8", "replace") + "\n")
    sys.stdout.flush()


_print_cb_keepalive = _PRINT_CB(_py_print)

_SIGNATURES = {
    "b2_version": (c_char_p, []),
    "b2_last_error": (c_char_p, []),
    "b2_set_logging": (None, [c_int]),
    "b2_get_logging": (c_int, []),
    "b2_set_print_callback": (None, [_PRINT_CB]),
    "b2_launch_count": (c_int, []),
    "b2_init": (c_int, [c_int]),
    "b2_multicast_supported": (c_int, [c_int]),
    "b2_vmm_supported": (c_int, [c_int]),
    "b2_granularity": (c_size_t, [c_int, c_int]),
    "b2_seg_create": (c_void_p, [c_int, c_int, c_int, c_size_t, c_int]),
    "b2_seg_export_fd": (c_int, [c_void_p]),
    "b2_seg_import_fd": (c_int, [c_void_p, c_int, c_int]),
    "b2_seg_ipc_handle": (c_int, [c_void_p, c_void_p]),
    "b2_seg_import_ipc": (c_int, [c_void_p, c_int, c_void_p]),
    "b2_seg_ptr": (c_void_p, [c_void_p, c_int]),
    "b2_seg_bytes": (c_size_t, [c_void_p]),
    "b2_seg_destroy": (c_int, [c_void_p]),
    "b2_mc_create": (c_void_p, [c_int, c_int, c_size_t]),
    "b2_mc_export_fd": (c_int, [c_void_p]),
    "b2_mc_import": (c_void_p, [c_int, c_int, c_size_t]),
    "b2_mc_add_device": (c_int, [c_void_p]),
    "b2_mc_bind": (c_int, [c_void_p, c_void_p]),
    "b2_mc_ptr": (c_void_p, [c_void_p]),
    "b2_mc_destroy": (c_int, [c_void_p]),
    "b2_layout_bytes": (c_size_t, [c_int, c_size_t, c_size_t, c_size_t]),
    "b2_comm_create": (c_void_p, [c_int, c_int, c_int, c_void_p, c_size_t, c_size_t, c_size_t, c_double]),
    "b2_comm_set_stage": (c_int, [c_void_p, c_void_p, c_void_p]),
    "b2_comm_stage_half": (c_size_t, [c_void_p]),
    "b2_comm_set_tuning": (c_int, [c_void_p, c_longlong, c_longlong, c_longlong, c_int]),
    "b2_comm_set_option": (c_int, [c_void_p, c_char_p, c_longlong]),
    "b2_comm_get_option": (c_longlong, [c_void_p, c_char_p]),
    "b2_comm_check_error": (c_int, [c_void_p, c_char_p, c_int]),
    "b2_comm_destroy": (c_int, [c_void_p]),
    "b2_stage_need": (c_size_t, [c_int, c_int, c_size_t]),
    "b2_barrier": (c_int, [c_void_p, c_void_p]),
    "b2_allreduce": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_void_p]),
    "b2_allreduce_sym": (c_int, [c_void_p, c_void_p, c_size_t, c_int, c_void_p]),
    "b2_reduce": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_void_p]),
    "b2_scan": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_void_p]),
    # (comm, in, out, count = elements per block, dtype, op, algo, stream)
    "b2_reduce_scatter": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_void_p]),
    "b2_allgather": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, POINTER(B2Strided), c_void_p]),
    "b2_alltoall": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, POINTER(B2Strided), c_void_p]),
    "b2_bcast": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_int, POINTER(B2Strided), c_void_p]),
    "b2_gather": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_int, POINTER(B2Strided), c_void_p]),
    "b2_scatter": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_int, POINTER(B2Strided), c_void_p]),
    "b2_status_alloc": (POINTER(B2StatusRecord), []),
    "b2_status_free": (None, [POINTER(B2StatusRecord)]),
    "b2_send": (c_int, [c_void_p, c_void_p, c_size_t, c_int, c_int, c_void_p]),
    "b2_recv": (c_int, [c_void_p, c_void_p, c_size_t, c_int, c_int, POINTER(B2StatusRecord), c_void_p]),
    "b2_sendrecv": (
        c_int,
        [c_void_p, c_void_p, c_size_t, c_int, c_int, c_void_p, c_size_t, c_int, c_int,
         POINTER(B2StatusRecord), c_void_p],
    ),
    "b2_abi_info": (c_int, [POINTER(c_int), c_int]),
    "b2_gemm_allreduce": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "b2_halo_exchange": (c_int, [c_void_p, POINTER(B2HaloDesc), c_void_p]),
    "b2_swe_multistep_ca": (
        c_int,
        [c_void_p, POINTER(B2SweParams), POINTER(B2SweState), POINTER(B2SweCA), POINTER(B2HaloDesc), c_int, c_int,
         c_void_p],
    ),
    "b2_swe_ca_timeline": (None, [c_void_p, c_int]),
    "b2_swe_ca_init": (
        c_int,
        [c_void_p, POINTER(B2SweParams), POINTER(B2SweState), POINTER(B2SweCA), POINTER(B2HaloDesc), c_void_p],
    ),
    "b2_swe_multistep": (
        c_int,
        [c_void_p, POINTER(B2SweParams), POINTER(B2SweState), POINTER(B2HaloDesc), c_int, c_int, c_void_p],
    ),
}


#: must equal B2_ABI_VERSION in csrc/b2_common.h
ABI_VERSION = 11
_ABI_FIELDS = ("abi_version", "sizeof_status_record", "sizeof_halo_desc", "sizeof_swe_params",
               "sizeof_swe_state", "sizeof_error_record", "max_ranks", "p2p_nslot", "sizeof_swe_ca")


def _abi_expected() -> dict:
    return {"abi_version": ABI_VERSION, "sizeof_status_record": ctypes.sizeof(B2StatusRecord),
            "sizeof_halo_desc": ctypes.sizeof(B2HaloDesc), "sizeof_swe_params": ctypes.sizeof(B2SweParams),
            "sizeof_swe_state": ctypes.sizeof(B2SweState), "sizeof_swe_ca": ctypes.sizeof(B2SweCA)}


def _abi_native(handle) -> dict:
    buf = (c_int * len(_ABI_FIELDS))()
    n = handle.b2_abi_info(buf, len(_ABI_FIELDS))
    return {k: int(buf[i]) for i, k in enumerate(_ABI_FIELDS[:n])}


def _abi_mismatch(handle) -> str:
    """'' if the ctypes mirrors match the structs compiled into the library, else a description
    (counterpart of the reference's import-time MPI ABI check, xla_bridge/__init__.py:23-89)."""
    have = _abi_native(handle)
    bad = [f"{k}: library {have.get(k)} != python {v}" for k, v in _abi_expected().items() if have.get(k) != v]
    return "; ".join(bad)


def _load() -> None:
    global lib, HAS_CUDA_EXT, CUDA_EXT_ERROR
    if not _LIB_PATH.exists():
        CUDA_EXT_ERROR = f"{_LIB_PATH} does not exist"
        return
    try:
        handle = ctypes.CDLL(str(_LIB_PATH))
        for name, (restype, argtypes) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = restype
            fn.argtypes = argtypes
        handle.b2_set_print_callback(_print_cb_keepalive)
    except (OSError, AttributeError) as exc:  # pragma: no cover - build problems
        CUDA_EXT_ERROR = f"{type(exc).__name__}: {exc}"
        return
    problem = _abi_mismatch(handle)
    if problem and any("native.build" in a or a.endswith("build.py") for a in getattr(sys, "orig_argv", [])):
        CUDA_EXT_ERROR = f"stale library ({problem}); rebuilding"     # `python -m ...native.build` itself
        return
    if problem and not env_flag("MPI4JAX_B200_SKIP_ABI_CHECK", False):
        raise RuntimeError(
            f"mpi4jax_b200: {_LIB_PATH} does not match this Python package ({problem}). The library is "
            "stale: rebuild it with `python setup.py build_ext --inplace` (or set "
            "MPI4JAX_B200_SKIP_ABI_CHECK=1 to load it anyway, at your own risk)."
        )
    lib = handle
    HAS_CUDA_EXT = True


_load()

# python-level logging flag (the CPU backend logs from Python with the same format)
_logging = False


def set_logging(enable: bool) -> None:
    """Enable/disable the per-call debug log on every backend
    (reference: xla_bridge/__init__.py:114-125)."""
    global _logging
    _logging = bool(enable)
    if HAS_CUDA_EXT:
        lib.b2_set_logging(1 if enable else 0)


def get_logging() -> bool:
    """Whether the per-call debug log is on (also set by ``MPI4JAX_B200_DEBUG=1`` at import)."""
    return _logging


def last_error() -> str:
    return lib.b2_last_error().decode() if HAS_CUDA_EXT else ""


def launch_count() -> int:
    """Number of native kernels launched by this process (all communicators)."""
    return int(lib.b2_launch_count()) if HAS_CUDA_EXT else 0


NATIVE_ABI_INFO = {
    "library": str(_LIB_PATH),
    "loaded": HAS_CUDA_EXT,
    "version": lib.b2_version().decode() if HAS_CUDA_EXT else None,
    "arch": "sm_100a",
    "sizeof_status_record": ctypes.sizeof(B2StatusRecord),
    "sizeof_halo_desc": ctypes.sizeof(B2HaloDesc),
    "python": _abi_expected(),
    "native": _abi_native(lib) if HAS_CUDA_EXT else None,
}

# reference: MPI4JAX_DEBUG is read at import (xla_bridge/__init__.py:128-129)
set_logging(env_flag("MPI4JAX_B200_DEBUG", False) or env_flag("MPI4JAX_DEBUG", False))
