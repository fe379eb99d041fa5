"""Host-staged transport for CUDA tensors: D2H -> CPU backend (gloo) -> H2D.

This is the reference's *default* GPU mode (``MPI4JAX_USE_CUDA_MPI`` unset/falsy:
mpi_xla_bridge_cuda.cpp copies every buffer through host memory around the MPI call,
e.g. :185-206) and the only way to reach a rank outside the local NVLink domain.  Here it is the
fallback, never the default on one node:

* chosen automatically when the ranks of a communicator span several hosts (the native transport
  needs peer-mapped HBM, i.e. one NVLink domain), with a one-time warning;
* forced by ``MPI4JAX_B200_TRANSPORT=host`` or the reference's ``MPI4JAX_USE_CUDA_MPI=0``.

Same method surface as ``backends.cuda.NativeComm`` for the 12 ops; the fused / B200-only entry
points (halo exchange, GEMM+allreduce) raise.  Ops synchronise the stream and block the host, so
they cannot be captured into CUDA graphs: ``mpi4jax_b200.jit`` runs such functions eagerly.
"""

from __future__ import annotations

from typing import Optional

import torch

from ..comm import Comm, MPIError, Status
from . import cpu as _cpu

#: set once any communicator uses this transport (``jit`` then stops capturing graphs)
ACTIVE = False


class HostStagedComm:
    """GPU side of a communicator whose traffic is staged through pinned host memory."""

    has_nvls = False

    def __init__(self, comm: Comm, reason: str = ""):
        global ACTIVE
        ACTIVE = True
        self.comm = comm
        self.reason = reason
        self.handle = None

    # -- staging -----------------------------------------------------------------------
    @staticmethod
    def _down(x: torch.Tensor) -> torch.Tensor:
        """Device -> host (stream-ordered: ``.cpu()`` waits for the producer kernels of ``x``)."""
        return x.detach().cpu() if x.device.type != "cpu" else x.detach()

    @staticmethod
    def _up(y: Optional[torch.Tensor], like: torch.Tensor) -> Optional[torch.Tensor]:
        if y is None:
            return None
        return y.to(like.device, non_blocking=False) if like.device.type != "cpu" else y

    def _unsupported(self, what: str):
        raise MPIError(f"{what} needs the native NVLink transport, but this communicator uses host "
                       f"staging ({self.reason or 'requested'}); use the 12 primitives instead")

    # -- lifecycle (NativeComm surface) ---------------------------------------------
    def flush(self) -> None:
        if torch.cuda.is_available():
            torch.cuda.synchronize()

    def check_device_error(self) -> None:
        pass

    def destroy(self) -> None:
        pass

    def set_tuning(self, *a, **k) -> None:
        pass

    # -- the 12 ops ------------------------------------------------------------------
    def barrier(self) -> None:
        self.flush()                      # the reference: stream sync, then MPI_Barrier (cuda.cpp:75-86)
        _cpu.barrier(self.comm)

    def allreduce(self, x, op_code: int, algo: int = 0):
        return self._up(_cpu.allreduce(self.comm, self._down(x), op_code), x)

    def reduce(self, x, op_code: int, root: int):
        return self._up(_cpu.reduce(self.comm, self._down(x), op_code, root), x)

    def scan(self, x, op_code: int):
        return self._up(_cpu.scan(self.comm, self._down(x), op_code), x)

    def allgather(self, x):
        return self._up(_cpu.allgather(self.comm, self._down(x)), x)

    def reduce_scatter(self, x, op_code: int, algo: int = 0):
        return self._up(_cpu.reduce_scatter(self.comm, self._down(x), op_code), x)

    def alltoall(self, x):
        return self._up(_cpu.alltoall(self.comm, self._down(x)), x)

    def bcast(self, x, root: int):
        out = _cpu.bcast(self.comm, self._down(x), root)
        return x if self.comm.rank == root else self._up(out, x)

    def gather(self, x, root: int):
        return self._up(_cpu.gather(self.comm, self._down(x), root), x)

    def scatter(self, x, root: int, out_shape, dtype):
        return self._up(_cpu.scatter(self.comm, self._down(x), root, out_shape, dtype), x)

    def send(self, x, dest: int, tag: int) -> None:
        _cpu.send(self.comm, self._down(x), dest, tag)

    def recv(self, template, source: int, tag: int, status: Optional[Status] = None):
        host = torch.empty(template.shape, dtype=template.dtype)
        return self._up(_cpu.recv(self.comm, host, source, tag, status), template)

    def sendrecv(self, sendbuf, recv_template, source: int, dest: int, sendtag: int, recvtag: int,
                 status: Optional[Status] = None):
        host = torch.empty(recv_template.shape, dtype=recv_template.dtype)
        out = _cpu.sendrecv(self.comm, self._down(sendbuf), host, source, dest, sendtag, recvtag, status)
        return self._up(out, recv_template)

    # -- B200-only entry points ---------------------------------------------------------
    def gemm_allreduce(self, *a, **k):
        self._unsupported("the fused GEMM + allreduce kernel")

    def halo_exchange(self, *a, **k):
        self._unsupported("the fused halo-exchange kernel")
