"""Backend dispatch for the 12 ops: CUDA tensors -> native kernels, CPU tensors -> gloo.

This is the analogue of the per-platform lowering registration each reference op does
(``register_lowering(..., platform="cpu"|"cuda"|"xpu")``, e.g.
/root/reference/mpi4jax/_src/collective_ops/allreduce.py:162-173): one op, several
device back ends, chosen by where the operand lives.
"""

from __future__ import annotations

from typing import Optional

import torch

from .. import native
from ..backends import cpu as _cpu
from ..comm import Comm, Status
from ..native import codes


def _log(comm: Comm, opname: str, details: str):
    if native.get_logging():
        return _cpu.log_call(comm.rank, opname, details)
    return None


_is_wrapped = torch._C._functorch.is_functorch_wrapped_tensor


def _plain(x: torch.Tensor) -> torch.Tensor:
    """Backends need real storage (the CUDA path takes raw pointers).  A torch.func wrapper here
    means an op's autograd rule called the backend directly instead of going through a
    ``torch.autograd.Function`` (which peels the transform levels) -- caught on every backend so the
    CPU suite sees it too."""
    if _is_wrapped(x):
        raise RuntimeError("mpi4jax_b200 internal error: a torch.func-wrapped tensor reached the "
                           "communication backend; use run_opaque() / a differentiable op in the rule")
    return x


class _Opaque(torch.autograd.Function):
    """Runs ``fn(x)`` with the torch.func transform levels peeled off ``x``."""

    @staticmethod
    def forward(fn, x):
        out = fn(x)
        return x.new_empty(0) if out is None else out

    @staticmethod
    def setup_context(ctx, inputs, output):
        pass

    @staticmethod
    def backward(ctx, g):
        raise NotImplementedError("higher-order derivatives through this communication rule are not defined")

    @staticmethod
    def vmap(info, in_dims, fn, x):
        return _Opaque.apply(fn, x), in_dims[1]     # rank-wise elementwise rules: the batch rides along


def run_opaque(fn, x: torch.Tensor):
    """Call a non-differentiable backend function from inside an autograd rule (where ``x`` may be a
    GradTrackingTensor / BatchedTensor of an active torch.func transform)."""
    if _is_wrapped(x) or torch._C._functorch.peek_interpreter_stack() is not None:
        return _Opaque.apply(fn, x)
    return fn(x)


def _is_cuda(*tensors) -> bool:
    return any(t is not None and t.is_cuda for t in tensors)


def barrier(comm: Comm) -> None:
    if comm.device.type == "cuda":
        comm._native_comm().barrier()
        return
    done = _log(comm, "Barrier", "")
    _cpu.barrier(comm)
    if done:
        done()


def allreduce(comm: Comm, x: torch.Tensor, op_code: int, algo: int = codes.ALGO_AUTO) -> torch.Tensor:
    _plain(x)
    if x.is_cuda:
        return comm._native_comm().allreduce(x, op_code, algo)
    done = _log(comm, "Allreduce", f"with {x.numel()} items")
    out = _cpu.allreduce(comm, x, op_code)
    if done:
        done()
    return out


def reduce(comm: Comm, x: torch.Tensor, op_code: int, root: int) -> Optional[torch.Tensor]:
    _plain(x)
    if x.is_cuda:
        return comm._native_comm().reduce(x, op_code, root)
    done = _log(comm, "Reduce", f"with {x.numel()} items to root {root}")
    out = _cpu.reduce(comm, x, op_code, root)
    if done:
        done()
    return out


def scan(comm: Comm, x: torch.Tensor, op_code: int) -> torch.Tensor:
    _plain(x)
    if x.is_cuda:
        return comm._native_comm().scan(x, op_code)
    done = _log(comm, "Scan", f"with {x.numel()} items")
    out = _cpu.scan(comm, x, op_code)
    if done:
        done()
    return out


def allgather(comm: Comm, x: torch.Tensor) -> torch.Tensor:
    _plain(x)
    if x.is_cuda:
        return comm._native_comm().allgather(x)
    done = _log(comm, "Allgather", f"sending {x.numel() * x.element_size()} bytes")
    out = _cpu.allgather(comm, x)
    if done:
        done()
    return out


def alltoall(comm: Comm, x: torch.Tensor) -> torch.Tensor:
    _plain(x)
    if x.is_cuda:
        return comm._native_comm().alltoall(x)
    done = _log(comm, "Alltoall", f"with {x.numel()} items")
    out = _cpu.alltoall(comm, x)
    if done:
        done()
    return out


def reduce_scatter(comm: Comm, x: torch.Tensor, op_code: int, algo: int = codes.ALGO_AUTO) -> torch.Tensor:
    _plain(x)
    if x.is_cuda:
        return comm._native_comm().reduce_scatter(x, op_code, algo)
    done = _log(comm, "Reduce_scatter_block", f"with {x[0].numel() if x.dim() else 0} items per rank")
    out = _cpu.reduce_scatter(comm, x, op_code)
    if done:
        done()
    return out


def bcast(comm: Comm, x: torch.Tensor, root: int) -> torch.Tensor:
    _plain(x)
    if x.is_cuda:
        return comm._native_comm().bcast(x, root)
    done = _log(comm, "Bcast", f"{x.numel()} items from root {root}")
    out = _cpu.bcast(comm, x, root)
    if done:
        done()
    return out


def gather(comm: Comm, x: torch.Tensor, root: int) -> Optional[torch.Tensor]:
    _plain(x)
    if x.is_cuda:
        return comm._native_comm().gather(x, root)
    done = _log(comm, "Gather", f"{x.numel()} items to root {root}")
    out = _cpu.gather(comm, x, root)
    if done:
        done()
    return out


def scatter(comm: Comm, x: torch.Tensor, root: int, out_shape, dtype) -> torch.Tensor:
    _plain(x)
    if x.is_cuda:
        return comm._native_comm().scatter(x, root, out_shape, dtype)
    done = _log(comm, "Scatter", f"from root {root}")
    out = _cpu.scatter(comm, x, root, out_shape, dtype)
    if done:
        done()
    return out


def send(comm: Comm, x: torch.Tensor, dest: int, tag: int) -> None:
    _plain(x)
    if x.is_cuda:
        comm._native_comm().send(x, dest, tag)
        return
    done = _log(comm, "Send", f"{x.numel()} items to {dest} with tag {tag}")
    _cpu.send(comm, x, dest, tag)
    if done:
        done()


def recv(comm: Comm, template: torch.Tensor, source: int, tag: int,
         status: Optional[Status]) -> torch.Tensor:
    if template.is_cuda:
        return comm._native_comm().recv(template, source, tag, status)
    done = _log(comm, "Recv", f"{template.numel()} items from {source} with tag {tag}")
    out = _cpu.recv(comm, template, source, tag, status)
    if done:
        done()
    return out


def sendrecv(comm: Comm, sendbuf: torch.Tensor, recv_template: torch.Tensor, source: int,
             dest: int, sendtag: int, recvtag: int, status: Optional[Status]) -> torch.Tensor:
    if sendbuf.is_cuda != recv_template.is_cuda:
        raise ValueError("sendrecv: sendbuf and recvbuf must live on the same device type")
    if sendbuf.is_cuda:
        return comm._native_comm().sendrecv(sendbuf, recv_template, source, dest, sendtag,
                                            recvtag, status)
    done = _log(comm, "Sendrecv", f"<{source} (tag {recvtag}) / >{dest} (tag {sendtag})")
    out = _cpu.sendrecv(comm, sendbuf, recv_template, source, dest, sendtag, recvtag, status)
    if done:
        done()
    return out
