"""Shared helpers of the op layer.

Counterpart of /root/reference/mpi4jax/_src/utils.py:1-174: the ``NOTSET`` sentinel,
the lazily created default communicator (a private clone of ``COMM_WORLD``), the
token-argument rejection, dtype support table and the capability probes.  What the
reference needs in addition -- MPI handle casts and hashable wrappers so that comm/op
can be static primitive parameters, and the ordered JAX effect -- has no equivalent
here: ops are ordinary Python calls that enqueue kernels on the current CUDA stream,
and **stream order is program order**, which is exactly the guarantee the ordered
effect token provides inside ``jax.jit`` (utils.py:45-53).  The same holds inside
``mpi4jax_b200.jit`` (CUDA-graph capture preserves stream order).
"""

from __future__ import annotations

from typing import Any, Optional

import numpy as np
import torch

from . import comm as _comm
from .native import codes

class _NotSet:
    """Sentinel type of ``NOTSET`` (prints nicely in signatures and generated docs)."""

    __slots__ = ()

    def __repr__(self) -> str:
        return "NOTSET"


NOTSET = _NotSet()

_default_comm: Optional[_comm.Comm] = None


def get_default_comm() -> _comm.Comm:
    """A private clone of COMM_WORLD, so library traffic cannot interleave with the
    user's own messages (reference: utils.py:17-27, docs/sharp-bits.rst:74-135)."""
    global _default_comm
    if _default_comm is None or _default_comm._freed:
        _default_comm = _comm.get_world().Clone()
    return _default_comm


def raise_if_token_is_set(token: Any) -> None:
    if token is not NOTSET:
        raise RuntimeError(
            "Explicit token management is not supported for mpi4jax>=0.8.0. "
            "Tokens are now managed automatically and must not be passed "
            "as arguments to collective operations anymore.\n"
            "That is, please adjust your code like this:\n"
            "     # For mpi4jax<0.8.0:\n"
            "     result, token = mpi4jax.allgather(x, token=token)\n"
            "     # For mpi4jax>=0.8.0:\n"
            "     result = mpi4jax.allgather(x)"
        )


# dtypes with a wire representation.  The reference supports 14 numpy dtypes and NOT
# float16/bfloat16 (utils.py:101-128); both 16-bit floats are supported here (fp32
# accumulation inside the fused reduce kernels); float128 has no GPU representation.
SUPPORTED_DTYPES = tuple(codes.DTYPE_CODE)


def check_dtype(t: torch.Tensor) -> None:
    if t.dtype not in codes.DTYPE_CODE:
        raise RuntimeError(f"Unknown MPI type for dtype {t.dtype}")


def as_tensor(x: Any, comm: _comm.Comm) -> torch.Tensor:
    """Accept tensors, numpy arrays and Python scalars (scalars become 0-d tensors, as in
    the reference's tests, e.g. tests/collective_ops/test_allreduce.py:35-54).  Non-tensor
    inputs are placed on the communicator's device."""
    if isinstance(x, torch.Tensor):
        return x
    if isinstance(x, np.ndarray):
        t = torch.from_numpy(np.ascontiguousarray(x))
    elif isinstance(x, (bool, int, float, complex, np.generic)):
        t = torch.tensor(x)
        if t.dtype == torch.float64 and isinstance(x, float):
            t = t.to(torch.get_default_dtype())
    else:
        t = torch.as_tensor(x)
    return t.to(comm.device)


_functorch = torch._C._functorch


def needs_autograd(*tensors) -> bool:
    """True when an op must go through its ``torch.autograd.Function`` (reverse-mode graph
    recording, or any active torch.func transform: vmap / grad / jvp / vjp).  Otherwise ops
    call their backend directly -- ``Function.apply`` alone costs ~25 us, an order of
    magnitude more than a small-message collective."""
    if _functorch.peek_interpreter_stack() is not None:
        return True
    if torch.is_grad_enabled():
        for t in tensors:
            if t.requires_grad:
                return True
    return torch.autograd.forward_ad._current_level >= 0


def carries_grad(t: torch.Tensor) -> bool:
    """True when dropping ``t`` from the graph would lose a gradient: reverse-mode recording is on
    for it, or it is the grad-tracking wrapper of an active torch.func transform."""
    if _functorch.is_gradtrackingtensor(t):
        return True
    return bool(torch.is_grad_enabled() and t.requires_grad)


def backend_of(t: torch.Tensor) -> str:
    return "cuda" if t.is_cuda else "cpu"


def has_cuda_support() -> bool:
    """True when the native sm_100a library is loaded (reference: utils.py:159-165)."""
    from . import native

    return bool(native.HAS_CUDA_EXT)


def has_sycl_support() -> bool:
    """Always False: the reference's Intel XPU bridge (utils.py:168-174) is out of scope
    for a B200-native framework."""
    return False


def check_rank(value: int, comm: _comm.Comm, opname: str, what: str, allow_any: bool = False) -> None:
    """Fail fast on an out-of-range peer rank, like the reference's abort_on_error path does
    when MPI reports MPI_ERR_RANK (mpi_ops_common.h:60-78; exercised by
    tests/collective_ops/test_common.py:60-88): prints
    ``r<rank> | MPI_<Op> returned error code 6: ... - aborting`` and aborts (or raises
    MPIError when MPI4JAX_B200_ABORT_ON_ERROR=0)."""
    if allow_any and value == _comm.ANY_SOURCE:
        return
    if value == _comm.PROC_NULL:          # MPI: communication with PROC_NULL is a no-op
        return
    if 0 <= value < comm.Get_size():
        return
    from .backends.cuda import abort_or_raise

    abort_or_raise(
        f"r{comm.Get_rank()} | MPI_{opname} returned error code 6: invalid {what} rank {value} "
        f"(communicator size {comm.Get_size()}) - aborting", 6)


def fold(parts, op) -> torch.Tensor:
    """``((x_0 (+) x_1) (+) x_2) ...`` with a user-defined operator, on the device."""
    acc = parts[0]
    for part in parts[1:]:
        acc = op.function(acc, part)
        if not isinstance(acc, torch.Tensor) or acc.shape != parts[0].shape:
            raise TypeError("a user-defined reduction must return a tensor of its operands' shape")
    return acc.to(parts[0].dtype)


def comm_reserve(nbytes: int, *, comm: Optional[_comm.Comm] = None) -> None:
    """Pre-size the GPU staging buffers of ``comm`` (default communicator if None) for collectives
    of up to ``nbytes`` per rank (alltoall, scatter and reduce_scatter: per block), so that no later
    call has to grow them.  Growth is collective and
    impossible during CUDA-graph capture; ``mpi4jax_b200.jit`` avoids it by running a function once
    eagerly, ``comm_reserve`` is the explicit alternative.  A no-op on CPU communicators."""
    if comm is None:
        comm = get_default_comm()
    if comm.device.type == "cuda":
        native_comm = comm._native_comm()
        if hasattr(native_comm, "reserve"):
            native_comm.reserve(int(nbytes))


def symmetric_empty(shape, dtype=None, *, comm: Optional[_comm.Comm] = None):
    """Uninitialised tensor in the SYMMETRIC heap of ``comm``: the same allocation on every rank, mapped
    into every peer GPU and bound to an NVSwitch multicast object.  Collectives on ordinary tensors stage
    their payload through such memory (one local copy in, one out); :func:`allreduce_` on a symmetric
    tensor skips both.  Collective (every rank must call it with the same shape and dtype); the memory is
    released with the communicator.  On a CPU communicator this is ``torch.empty``.

    Extension: the reference hands device pointers of XLA buffers to MPI (mpi_xla_bridge_cuda.cpp) and
    has no notion of registered / symmetric memory."""
    import torch

    if comm is None:
        comm = get_default_comm()
    dtype = dtype or torch.float32
    if comm.device.type != "cuda":
        return torch.empty(shape, dtype=dtype)
    return comm._native_comm().symmetric_empty(shape, dtype)


def allreduce_(x, op=None, *, comm: Optional[_comm.Comm] = None):
    """SUM-allreduce ``x`` IN PLACE and return it.  ``x`` must come from :func:`symmetric_empty` (or be a
    contiguous view of such a tensor) and be float32 / bfloat16 / float16; the sum is formed inside the
    NVSwitch (``multimem.ld_reduce``, fp32 accumulation) and written back through it, without staging
    copies.  Not differentiable.  On a CPU communicator: an ordinary in-place allreduce."""
    from . import comm as _c

    if comm is None:
        comm = get_default_comm()
    if op is not None and op is not _c.SUM:
        raise NotImplementedError("allreduce_ reduces with MPI.SUM only (what the switch implements)")
    if comm.device.type != "cuda" or not x.is_cuda:
        from .collective_ops.allreduce import allreduce as _allreduce

        x.copy_(_allreduce(x, _c.SUM, comm=comm))
        return x
    return comm._native_comm().allreduce_inplace(x)

