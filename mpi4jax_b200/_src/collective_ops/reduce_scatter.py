"""reduce_scatter -- ``MPI_Reduce_scatter_block``: rank r receives ``op`` over all ranks q of ``x_q[r]``.

Extension: mpi4jax has no reduce-scatter.  Every rank passes ``x`` of shape ``(nproc, *S)`` and
receives shape ``S``; it moves ``(P-1)/P`` of the input per rank where ``allreduce(x)[rank]`` moves
all of it.  GPU implementation: LL push, one-shot pull and in-switch (NVLS) kernels
(csrc/b2_reduce_scatter.cuh, b2_collectives.cu).  Autograd for SUM: the adjoint is the allgather of
the cotangent, the derivative is the reduce-scatter of the tangent.
"""

from __future__ import annotations

import torch

from ..comm import OP_TYPES, SUM, Comm, Op, as_op
from ..native import codes
from ..utils import (NOTSET, as_tensor, check_dtype, fold, get_default_comm, needs_autograd,
                     raise_if_token_is_set)
from ..validation import enforce_types
from . import _dispatch

ALGORITHMS = ("auto", "ll", "oneshot", "nvls")


def _require_sum(op: Op, what: str) -> None:
    if op is not SUM:
        raise NotImplementedError(f"The {what} of reduce_scatter for {op.name} is not defined")


class _ReduceScatter(torch.autograd.Function):
    @staticmethod
    def forward(x, op, comm, algo):
        return _dispatch.reduce_scatter(comm, x, op.code, algo)

    @staticmethod
    def setup_context(ctx, inputs, output):
        _, ctx.op, ctx.comm, ctx.algo = inputs

    @staticmethod
    def backward(ctx, g):
        _require_sum(ctx.op, "adjoint")
        from .allgather import allgather      # the differentiable op: works under torch.func too

        return allgather(g.contiguous(), comm=ctx.comm), None, None, None

    @staticmethod
    def jvp(ctx, x_t, *_):
        _require_sum(ctx.op, "derivative")
        return _ReduceScatter.apply(x_t.contiguous(), ctx.op, ctx.comm, ctx.algo)

    @staticmethod
    def vmap(info, in_dims, x, op, comm, algo):
        # keep the (nproc, ...) axis in front: (B, P, *S) -> (P, B, *S), reduced as one message -> (B, *S)
        return _ReduceScatter.apply(x.movedim(in_dims[0], 1).contiguous(), op, comm, algo), 0


@enforce_types(op=OP_TYPES, comm=(type(None), Comm))
def reduce_scatter(x, op, *, comm=None, token=NOTSET, algorithm="auto"):
    """Perform a reduce-scatter operation (``MPI_Reduce_scatter_block``).

    Every rank passes ``x`` of shape ``(nproc, ...)`` with the same shape and dtype; rank ``r``
    receives the reduction with ``op`` over all ranks of their ``x[r]``.  Extension: the reference
    has no reduce-scatter.

    Arguments:
        x: input of shape ``(nproc, ...)``.
        op: the reduction operator (e.g. ``mpi4jax_b200.MPI.SUM``).
        comm: the communicator (defaults to a clone of ``COMM_WORLD``).
        algorithm: GPU transport -- ``"auto"`` (the allreduce size thresholds), ``"ll"``,
            ``"oneshot"`` or ``"nvls"``.

    Returns:
        Tensor: this rank's reduced block, shape ``x.shape[1:]`` and the dtype of ``x``.
    """
    raise_if_token_is_set(token)
    if comm is None:
        comm = get_default_comm()
    op = as_op(op)
    if algorithm not in ALGORITHMS:
        raise ValueError(f"reduce_scatter: algorithm must be one of {ALGORITHMS}, got {algorithm!r}")
    x = as_tensor(x, comm)
    check_dtype(x)
    if x.dim() == 0 or x.shape[0] != comm.Get_size():
        raise ValueError("Reduce_scatter input must have shape (nproc, ...)")
    algo = codes.ALGO_BY_NAME[algorithm]
    if op.code is None:                      # MPI.Op.Create: exchange the blocks natively, fold on the device
        if needs_autograd(x):
            raise NotImplementedError(f"The derivative of reduce_scatter for {op.name} is not defined")
        return fold(list(_dispatch.alltoall(comm, x.contiguous()).unbind(0)), op)
    if not needs_autograd(x):
        return _dispatch.reduce_scatter(comm, x, op.code, algo)
    return _ReduceScatter.apply(x, op, comm, algo)
