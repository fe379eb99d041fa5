"""mpi4jax_b200 -- Blackwell-native communication primitives with the API of mpi4jax.

Public namespace (reference: /root/reference/mpi4jax/__init__.py:9-41): the 12 ops and the
two capability probes, plus what replaces the pieces JAX/mpi4py provided there:

* ``MPI``      communicators, reduction ops, Status, ANY_SOURCE/ANY_TAG (``mpi4py.MPI`` stand-in)
* ``jit``      CUDA-graph capture of a function containing ops (``jax.jit`` stand-in)
* ``flush``    drain all pending communication (``jax.effects_barrier`` stand-in)
* ``linear_transpose`` / autograd / ``torch.func`` transforms work through the ops
"""

from ._version import __version__  # noqa: F401
from ._src import (  # noqa: F401
    allgather,
    allreduce,
    alltoall,
    barrier,
    bcast,
    allreduce_,
    comm_reserve,
    flush,
    gather,
    has_cuda_support,
    has_sycl_support,
    recv,
    reduce,
    reduce_scatter,
    scan,
    scatter,
    send,
    send_with_grad,
    sendrecv,
    symmetric_empty,
)
from . import MPI  # noqa: F401
from ._src.jit import jit, linear_transpose  # noqa: F401
from ._src.compile_ops import compiled  # noqa: F401  (torch.library / torch.compile frontend)

effects_barrier = flush

__all__ = [
    "allgather", "allreduce", "alltoall", "barrier", "bcast", "gather", "recv", "reduce",
    "scan", "scatter", "send", "sendrecv", "has_cuda_support", "has_sycl_support",
    "MPI", "jit", "compiled", "flush", "effects_barrier", "linear_transpose", "send_with_grad", "comm_reserve",
    "symmetric_empty", "allreduce_", "reduce_scatter",
]
