"""``torch.library`` registration of the 12 ops -- the traceable frontend.

The reference's ops are JAX *primitives*: abstract-eval rules give shapes, an ordered effect
threads a token through every custom call so XLA keeps them in program order
(/root/reference/mpi4jax/_src/utils.py:45-53, jax_compat.py:82-100, e.g. allreduce.py:87-111).
The torch analogue: every op is a ``torch.library.custom_op`` with a fake (meta) kernel =
the abstract-eval rule, and is registered as an **ORDERED effectful op**
(``torch._higher_order_ops.effects``), which makes AOTAutograd thread effect tokens through
them exactly like JAX does -- ``send`` (no result) and ``barrier`` (no operands) can neither be
dead-code-eliminated nor reordered inside ``torch.compile(fullgraph=True)``.

The eager/CUDA-graph path (``mpi4jax_b200.jit``) does not need any of this; it is provided so
that functions using the ops can be traced by ``torch.compile`` / ``torch.export``:

    from mpi4jax_b200 import compiled as mc
    f = torch.compile(lambda x: mc.allreduce(x, MPI.SUM, comm=comm), fullgraph=True)

Communicators and reduction ops travel through the graph as plain integers (comm id, op code),
the counterpart of the reference's int64 handle attributes.
"""

from __future__ import annotations

from typing import Optional

import torch
from torch.library import custom_op

from . import comm as _comm_mod
from .collective_ops import _dispatch
from .comm import ANY_SOURCE, ANY_TAG, SUM, Comm, as_op
from .native import codes
from .utils import get_default_comm

def _register(comm: Optional[Comm]) -> int:
    """Communicator -> integer graph attribute.  No registration side effect here: Dynamo defers
    Python side effects of a traced frame until after the graph has run, so the lookup table must
    exist beforehand -- it is the registry every ``Comm`` enters at construction."""
    comm = comm or get_default_comm()
    return comm._id


def _c(comm_id: int) -> Comm:
    for comm in list(_comm_mod._comm_registry):
        if comm._id == comm_id:
            return comm
    raise RuntimeError(f"mpi4jax_b200: communicator #{comm_id} no longer exists (it was freed or garbage "
                       "collected after the function using it was compiled)")


def _st(status_id: int):
    """Status id -> object (0 = no status requested)."""
    if status_id == 0:
        return None
    st = _comm_mod._status_registry.get(status_id)
    if st is None:
        raise RuntimeError(f"mpi4jax_b200: Status #{status_id} was garbage collected after the function "
                           "using it was compiled; keep a reference to it")
    return st


# ---------------------------------------------------------------- op definitions
@custom_op("mpi4jax_b200::allreduce", mutates_args=())
def _allreduce(x: torch.Tensor, op: int, comm_id: int) -> torch.Tensor:
    return _dispatch.allreduce(_c(comm_id), x.contiguous(), op, codes.ALGO_AUTO)


@_allreduce.register_fake
def _(x, op, comm_id):
    return torch.empty_like(x, memory_format=torch.contiguous_format)


def _allreduce_setup(ctx, inputs, output):
    _, ctx.op, ctx.comm_id = inputs


def _allreduce_backward(ctx, g):
    if ctx.op != SUM.code:
        raise NotImplementedError("The adjoint of allreduce is only defined for SUM")
    return g, None, None            # transpose of allreduce(SUM) = identity on the local cotangent


_allreduce.register_autograd(_allreduce_backward, setup_context=_allreduce_setup)


@custom_op("mpi4jax_b200::reduce_scatter", mutates_args=())
def _reduce_scatter(x: torch.Tensor, op: int, comm_id: int) -> torch.Tensor:
    return _dispatch.reduce_scatter(_c(comm_id), x.contiguous(), op, codes.ALGO_AUTO)


@_reduce_scatter.register_fake
def _(x, op, comm_id):
    return x.new_empty(x.shape[1:])


def _reduce_scatter_setup(ctx, inputs, output):
    _, ctx.op, ctx.comm_id = inputs


def _reduce_scatter_backward(ctx, g):
    if ctx.op != SUM.code:
        raise NotImplementedError("The adjoint of reduce_scatter is only defined for SUM")
    comm = _c(ctx.comm_id)
    return torch.ops.mpi4jax_b200.allgather(g.contiguous(), ctx.comm_id, comm.Get_size()), None, None


_reduce_scatter.register_autograd(_reduce_scatter_backward, setup_context=_reduce_scatter_setup)


@custom_op("mpi4jax_b200::allgather", mutates_args=())
def _allgather(x: torch.Tensor, comm_id: int, size: int) -> torch.Tensor:
    return _dispatch.allgather(_c(comm_id), x.contiguous())


@_allgather.register_fake
def _(x, comm_id, size):
    return x.new_empty((size, *x.shape))


def _allgather_setup(ctx, inputs, output):
    _, ctx.comm_id, _ = inputs


def _allgather_backward(ctx, g):
    # adjoint of allgather = reduce-scatter of the cotangent (here: allreduce + own slice)
    total = torch.ops.mpi4jax_b200.allreduce(g.contiguous(), SUM.code, ctx.comm_id)
    return total[_c(ctx.comm_id).Get_rank()], None, None


_allgather.register_autograd(_allgather_backward, setup_context=_allgather_setup)


@custom_op("mpi4jax_b200::alltoall", mutates_args=())
def _alltoall(x: torch.Tensor, comm_id: int) -> torch.Tensor:
    return _dispatch.alltoall(_c(comm_id), x.contiguous())


@_alltoall.register_fake
def _(x, comm_id):
    return torch.empty_like(x, memory_format=torch.contiguous_format)


def _alltoall_setup(ctx, inputs, output):
    _, ctx.comm_id = inputs


def _alltoall_backward(ctx, g):
    return torch.ops.mpi4jax_b200.alltoall(g.contiguous(), ctx.comm_id), None      # self-adjoint up to the swap


_alltoall.register_autograd(_alltoall_backward, setup_context=_alltoall_setup)


@custom_op("mpi4jax_b200::bcast", mutates_args=())
def _bcast(x: torch.Tensor, root: int, comm_id: int) -> torch.Tensor:
    out = _dispatch.bcast(_c(comm_id), x.contiguous(), root)
    return out.clone() if out.data_ptr() == x.data_ptr() else out   # custom ops may not alias inputs


@_bcast.register_fake
def _(x, root, comm_id):
    return torch.empty_like(x, memory_format=torch.contiguous_format)


def _bcast_setup(ctx, inputs, output):
    _, ctx.root, ctx.comm_id = inputs


def _bcast_backward(ctx, g):
    # adjoint of bcast = sum of the cotangents on the root, nothing elsewhere
    total = torch.ops.mpi4jax_b200.reduce(g.contiguous(), SUM.code, ctx.root, ctx.comm_id)
    if _c(ctx.comm_id).Get_rank() == ctx.root:
        return total, None, None
    return torch.zeros_like(g), None, None


_bcast.register_autograd(_bcast_backward, setup_context=_bcast_setup)


@custom_op("mpi4jax_b200::scan", mutates_args=())
def _scan(x: torch.Tensor, op: int, comm_id: int) -> torch.Tensor:
    return _dispatch.scan(_c(comm_id), x.contiguous(), op)


@_scan.register_fake
def _(x, op, comm_id):
    return torch.empty_like(x, memory_format=torch.contiguous_format)


@custom_op("mpi4jax_b200::reduce", mutates_args=())
def _reduce(x: torch.Tensor, op: int, root: int, comm_id: int) -> torch.Tensor:
    comm = _c(comm_id)
    out = _dispatch.reduce(comm, x.contiguous(), op, root)
    return out if comm.Get_rank() == root else x.clone()


@_reduce.register_fake
def _(x, op, root, comm_id):
    return torch.empty_like(x, memory_format=torch.contiguous_format)


@custom_op("mpi4jax_b200::gather_root", mutates_args=())
def _gather_root(x: torch.Tensor, root: int, comm_id: int, size: int) -> torch.Tensor:
    return _dispatch.gather(_c(comm_id), x.contiguous(), root)


@_gather_root.register_fake
def _(x, root, comm_id, size):
    return x.new_empty((size, *x.shape))


@custom_op("mpi4jax_b200::gather_leaf", mutates_args=())
def _gather_leaf(x: torch.Tensor, root: int, comm_id: int) -> torch.Tensor:
    _dispatch.gather(_c(comm_id), x.contiguous(), root)
    return x.clone()


@_gather_leaf.register_fake
def _(x, root, comm_id):
    return torch.empty_like(x, memory_format=torch.contiguous_format)


@custom_op("mpi4jax_b200::scatter", mutates_args=())
def _scatter(x: torch.Tensor, root: int, comm_id: int, is_root: bool) -> torch.Tensor:
    shape = tuple(x.shape[1:]) if is_root else tuple(x.shape)
    return _dispatch.scatter(_c(comm_id), x.contiguous(), root, shape, x.dtype)


@_scatter.register_fake
def _(x, root, comm_id, is_root):
    return x.new_empty(tuple(x.shape[1:]) if is_root else tuple(x.shape))


@custom_op("mpi4jax_b200::barrier", mutates_args=())
def _barrier(comm_id: int) -> None:
    _dispatch.barrier(_c(comm_id))


@_barrier.register_fake
def _(comm_id):
    return None


@custom_op("mpi4jax_b200::send", mutates_args=())
def _send(x: torch.Tensor, dest: int, tag: int, comm_id: int) -> None:
    _dispatch.send(_c(comm_id), x.contiguous(), dest, tag)


@_send.register_fake
def _(x, dest, tag, comm_id):
    return None


@custom_op("mpi4jax_b200::recv", mutates_args=())
def _recv(template: torch.Tensor, source: int, tag: int, comm_id: int, status_id: int) -> torch.Tensor:
    return _dispatch.recv(_c(comm_id), template, source, tag, _st(status_id))


@_recv.register_fake
def _(template, source, tag, comm_id, status_id):
    return torch.empty_like(template, memory_format=torch.contiguous_format)


@custom_op("mpi4jax_b200::sendrecv", mutates_args=())
def _sendrecv(sendbuf: torch.Tensor, recvbuf: torch.Tensor, source: int, dest: int, sendtag: int,
              recvtag: int, comm_id: int, status_id: int) -> torch.Tensor:
    return _dispatch.sendrecv(_c(comm_id), sendbuf.contiguous(), recvbuf, source, dest, sendtag, recvtag,
                              _st(status_id))


@_sendrecv.register_fake
def _(sendbuf, recvbuf, source, dest, sendtag, recvtag, comm_id, status_id):
    return torch.empty_like(recvbuf, memory_format=torch.contiguous_format)


def _sendrecv_setup(ctx, inputs, output):
    sendbuf, _, ctx.source, ctx.dest, ctx.sendtag, ctx.recvtag, ctx.comm_id, _ = inputs
    ctx.send_meta = (tuple(sendbuf.shape), sendbuf.dtype, sendbuf.device)


def _sendrecv_backward(ctx, g):
    # transpose: the cotangent of what was received travels back to where it came from
    # (the reference swaps source and dest the same way, sendrecv.py:277-292)
    shape, dtype, device = ctx.send_meta
    template = torch.empty(shape, dtype=dtype, device=device)
    back = torch.ops.mpi4jax_b200.sendrecv(g.contiguous(), template, ctx.dest, ctx.source,
                                           max(ctx.recvtag, 0), ctx.sendtag, ctx.comm_id, 0)
    return back, None, None, None, None, None, None, None


_sendrecv.register_autograd(_sendrecv_backward, setup_context=_sendrecv_setup)


ALL_OPS = ("allreduce", "reduce_scatter", "allgather", "alltoall", "bcast", "scan", "reduce", "gather_root", "gather_leaf",
           "scatter", "barrier", "send", "recv", "sendrecv")
ORDERED_EFFECT = False
try:  # the ordered effect: AOTAutograd threads a token through these ops in program order
    from torch._higher_order_ops.effects import _EffectType, _register_effectful_op

    for _name in ALL_OPS:
        _register_effectful_op(f"mpi4jax_b200::{_name}", _EffectType.ORDERED)
    ORDERED_EFFECT = True
except Exception:  # pragma: no cover - private API moved; ops then still rely on "has side effects"
    pass


# ---------------------------------------------------------------- public, traceable wrappers
class compiled:
    """Namespace of ``torch.compile``-traceable ops (static arguments are plain Python values)."""

    @staticmethod
    def allreduce(x, op, *, comm=None):
        return torch.ops.mpi4jax_b200.allreduce(x, as_op(op).code, _register(comm))

    @staticmethod
    def reduce_scatter(x, op, *, comm=None):
        """``x`` of shape ``(nproc, ...)`` -> this rank's reduced block (SUM is differentiable)."""
        return torch.ops.mpi4jax_b200.reduce_scatter(x, as_op(op).code, _register(comm))

    @staticmethod
    def allgather(x, *, comm=None):
        comm = comm or get_default_comm()     # plain attribute reads only: this code is traced by Dynamo
        return torch.ops.mpi4jax_b200.allgather(x, comm._id, comm.Get_size())

    @staticmethod
    def alltoall(x, *, comm=None):
        return torch.ops.mpi4jax_b200.alltoall(x, _register(comm))

    @staticmethod
    def bcast(x, root, *, comm=None):
        return torch.ops.mpi4jax_b200.bcast(x, int(root), _register(comm))

    @staticmethod
    def scan(x, op, *, comm=None):
        return torch.ops.mpi4jax_b200.scan(x, as_op(op).code, _register(comm))

    @staticmethod
    def reduce(x, op, root, *, comm=None):
        return torch.ops.mpi4jax_b200.reduce(x, as_op(op).code, int(root), _register(comm))

    @staticmethod
    def gather(x, root, *, comm=None):
        comm = comm or get_default_comm()
        if comm.Get_rank() == root:
            return torch.ops.mpi4jax_b200.gather_root(x, int(root), comm._id, comm.Get_size())
        return torch.ops.mpi4jax_b200.gather_leaf(x, int(root), comm._id)

    @staticmethod
    def scatter(x, root, *, comm=None):
        comm = comm or get_default_comm()
        return torch.ops.mpi4jax_b200.scatter(x, int(root), comm._id, comm.Get_rank() == root)

    @staticmethod
    def barrier(*, comm=None):
        torch.ops.mpi4jax_b200.barrier(_register(comm))

    @staticmethod
    def send(x, dest, *, tag=0, comm=None):
        torch.ops.mpi4jax_b200.send(x, int(dest), int(tag), _register(comm))

    @staticmethod
    def recv(x, source=ANY_SOURCE, *, tag=ANY_TAG, comm=None, status=None):
        """``status``: an ``MPI.Status`` filled when the compiled function runs (as under ``jax.jit`` in
        the reference, tests/collective_ops/test_send_and_recv.py:113-153); keep it alive."""
        return torch.ops.mpi4jax_b200.recv(x, int(source), int(tag), _register(comm),
                                           0 if status is None else status._id)

    @staticmethod
    def sendrecv(sendbuf, recvbuf, source, dest, *, sendtag=0, recvtag=ANY_TAG, comm=None, status=None):
        return torch.ops.mpi4jax_b200.sendrecv(sendbuf, recvbuf, int(source), int(dest), int(sendtag),
                                               int(recvtag), _register(comm), 0 if status is None else status._id)
