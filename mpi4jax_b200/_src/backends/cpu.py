"""CPU backend: the 12 ops on host tensors over ``torch.distributed`` (gloo).

Role: what the reference's CPU bridge (mpi_xla_bridge_cpu.cpp, one blocking MPI call
per op) is to its GPU bridge -- the correctness path that runs anywhere, including the
GPU-less CI box.  The image has no MPI, so gloo carries the bytes; semantics follow MPI:

* collectives move raw bytes (every dtype incl. bool/complex) with ``all_gather`` /
  ``broadcast`` and reduce locally in rank order (deterministic, all 10 ops);
* point-to-point keeps MPI matching semantics on top of gloo's FIFO channels: each
  message is a (header, payload) pair, the receiver keeps an unexpected-message queue
  per source, so tags may be consumed out of order, ``ANY_SOURCE`` / ``ANY_TAG`` work
  and ``Status`` is filled.  Sends are eager (``isend``) for every size, completed at
  ``flush()``; self-sends never touch the network.
"""

from __future__ import annotations

import time
from collections import deque
from typing import Optional

import torch
import torch.distributed as dist

from ..comm import ANY_SOURCE, ANY_TAG, Comm, Status
from ..native import codes

_HDR_WORDS = 4  # tag, nbytes, dtype code (informational), magic
_MAGIC = 0x6232_6D70  # "b2mp"


def _bytes_view(x: torch.Tensor) -> torch.Tensor:
    return x.contiguous().reshape(-1).view(torch.uint8)


def reduce_stack(stack: torch.Tensor, op_code: int) -> torch.Tensor:
    """Reduce ``stack`` (P, *shape) over dim 0 with MPI op semantics, in rank order."""
    dt = stack.dtype
    if stack.shape[0] == 1:
        return stack[0].clone()     # a single contribution passes through unchanged (as in MPI)
    if dt == torch.bool:
        if op_code in (codes.SUM, codes.MAX, codes.LOR, codes.BOR):
            return stack.any(dim=0)
        if op_code in (codes.PROD, codes.MIN, codes.LAND, codes.BAND):
            return stack.all(dim=0)
        if op_code in (codes.LXOR, codes.BXOR):
            return (stack.to(torch.int32).sum(dim=0) % 2).to(torch.bool)
    is_float = dt.is_floating_point
    is_cplx = dt.is_complex
    if op_code == codes.SUM:
        acc_dt = torch.float32 if dt in (torch.float16, torch.bfloat16) else dt
        acc = stack[0].to(acc_dt).clone()
        for q in range(1, stack.shape[0]):
            acc += stack[q].to(acc_dt)
        return acc.to(dt)
    if op_code == codes.PROD:
        acc_dt = torch.float32 if dt in (torch.float16, torch.bfloat16) else dt
        acc = stack[0].to(acc_dt).clone()
        for q in range(1, stack.shape[0]):
            acc *= stack[q].to(acc_dt)
        return acc.to(dt)
    if is_cplx:
        raise NotImplementedError("only SUM and PROD are defined for complex dtypes")
    if op_code == codes.MIN:
        return stack.amin(dim=0) if not is_float else torch.min(stack, dim=0).values
    if op_code == codes.MAX:
        return stack.amax(dim=0) if not is_float else torch.max(stack, dim=0).values
    if is_float:
        raise NotImplementedError("logical/bitwise reductions need an integer or bool dtype")
    if op_code == codes.LAND:
        return (stack != 0).all(dim=0).to(dt)
    if op_code == codes.LOR:
        return (stack != 0).any(dim=0).to(dt)
    if op_code == codes.LXOR:
        return ((stack != 0).to(torch.int32).sum(dim=0) % 2).to(dt)
    wide = stack.to(torch.int64) if dt in (torch.uint16, torch.uint32, torch.uint64) else stack
    acc = wide[0].clone()
    for q in range(1, stack.shape[0]):
        if op_code == codes.BAND:
            acc &= wide[q]
        elif op_code == codes.BOR:
            acc |= wide[q]
        else:
            acc ^= wide[q]
    return acc.to(dt)


class CpuState:
    """Per-communicator host-side p2p state (unexpected queues, pending sends)."""

    def __init__(self, comm: Comm):
        self.comm = comm
        self.pending: list = []                      # (work, keepalive tensors)
        self.unexpected = [deque() for _ in range(comm.size)]   # per source: (tag, payload)
        self.self_queue: deque = deque()

    def prune(self) -> None:
        self.pending = [(w, k) for (w, k) in self.pending if not w.is_completed()]

    def flush(self) -> None:
        for work, _ in self.pending:
            work.wait()
        self.pending.clear()


# ---------------------------------------------------------------------------
# collectives
# ---------------------------------------------------------------------------
def _allgather_bytes(comm: Comm, x: torch.Tensor) -> list:
    flat = _bytes_view(x)
    if comm.size == 1:
        return [flat.clone()]
    outs = [torch.empty_like(flat) for _ in range(comm.size)]
    dist.all_gather(outs, flat, group=comm._group)
    return comm._in_rank_order(outs)


def _gather_stack(comm: Comm, x: torch.Tensor) -> torch.Tensor:
    parts = _allgather_bytes(comm, x)
    return torch.stack([p.view(x.dtype).reshape(x.shape) for p in parts], dim=0)


def barrier(comm: Comm) -> None:
    dist.barrier(group=comm._group)


def allreduce(comm: Comm, x: torch.Tensor, op_code: int) -> torch.Tensor:
    return reduce_stack(_gather_stack(comm, x), op_code)


def reduce(comm: Comm, x: torch.Tensor, op_code: int, root: int) -> Optional[torch.Tensor]:
    stack = _gather_stack(comm, x)
    return reduce_stack(stack, op_code) if comm.rank == root else None


def scan(comm: Comm, x: torch.Tensor, op_code: int) -> torch.Tensor:
    stack = _gather_stack(comm, x)
    return reduce_stack(stack[: comm.rank + 1], op_code)


def allgather(comm: Comm, x: torch.Tensor) -> torch.Tensor:
    return _gather_stack(comm, x)


def alltoall(comm: Comm, x: torch.Tensor) -> torch.Tensor:
    # x: (P, *S).  Everybody gathers everything and keeps its column (correctness path).
    stack = _gather_stack(comm, x)            # (P_src, P_dst, *S)
    return stack[:, comm.rank].clone()


def reduce_scatter(comm: Comm, x: torch.Tensor, op_code: int) -> torch.Tensor:
    # x: (P, *S).  The blocks travel as an alltoall, then the P received blocks are reduced in rank order.
    return reduce_stack(alltoall(comm, x), op_code)


def bcast(comm: Comm, x: torch.Tensor, root: int) -> torch.Tensor:
    buf = _bytes_view(x).clone()
    if comm.size > 1:
        dist.broadcast(buf, src=comm._global(root), group=comm._group)
    return buf.view(x.dtype).reshape(x.shape)


def gather(comm: Comm, x: torch.Tensor, root: int) -> Optional[torch.Tensor]:
    stack = _gather_stack(comm, x)
    return stack if comm.rank == root else None


def scatter(comm: Comm, x: torch.Tensor, root: int, out_shape, dtype) -> torch.Tensor:
    # root holds (P, *S); others pass a template of shape S
    numel = 1
    for s in out_shape:
        numel *= s
    nbytes = numel * torch.empty((), dtype=dtype).element_size()
    if comm.rank == root:
        buf = _bytes_view(x).clone()
    else:
        buf = torch.empty(nbytes * comm.size, dtype=torch.uint8)
    if comm.size > 1:
        dist.broadcast(buf, src=comm._global(root), group=comm._group)
    mine = buf[comm.rank * nbytes : (comm.rank + 1) * nbytes].clone()
    return mine.view(dtype).reshape(out_shape)


# ---------------------------------------------------------------------------
# point to point
# ---------------------------------------------------------------------------
def send(comm: Comm, x: torch.Tensor, dest: int, tag: int) -> None:
    st = comm._cpu()
    payload = _bytes_view(x).clone()
    if dest == comm.rank:
        st.self_queue.append((tag, payload))
        return
    hdr = torch.tensor([tag, payload.numel(), codes.DTYPE_CODE.get(x.dtype, -1), _MAGIC],
                       dtype=torch.int64)
    g = comm._global(dest)
    w1 = dist.isend(hdr, dst=g, group=comm._group)
    st.pending.append((w1, hdr))
    if payload.numel() > 0:
        w2 = dist.isend(payload, dst=g, group=comm._group)
        st.pending.append((w2, payload))
    st.prune()


def _pull_one(comm: Comm, source: int):
    """Blocking receive of the next (tag, payload) from ``source`` (rank in comm)."""
    hdr = torch.empty(_HDR_WORDS, dtype=torch.int64)
    dist.recv(hdr, src=comm._global(source), group=comm._group)
    if int(hdr[3]) != _MAGIC:
        raise RuntimeError("mpi4jax_b200 CPU p2p protocol error (foreign traffic on the group?)")
    payload = torch.empty(int(hdr[1]), dtype=torch.uint8)
    if payload.numel() > 0:
        dist.recv(payload, src=comm._global(source), group=comm._group)
    return int(hdr[0]), payload


def _match(queue: deque, tag: int):
    for k, (t, payload) in enumerate(queue):
        if tag == ANY_TAG or t == tag:
            del queue[k]
            return t, payload
    return None


def recv_bytes(comm: Comm, source: int, tag: int):
    """Blocking matched receive of one message: returns ``(source, tag, payload uint8 tensor)``."""
    st = comm._cpu()
    got = None
    src = source
    if source == comm.rank or (source == ANY_SOURCE and st.self_queue):
        got = _match(st.self_queue, tag)
        if got is not None:
            src = comm.rank
        elif source == comm.rank:
            raise RuntimeError("recv from self: no matching message was sent (would deadlock)")
    if got is None and source != ANY_SOURCE:
        got = _match(st.unexpected[source], tag)
        while got is None:
            t, payload = _pull_one(comm, source)
            if tag == ANY_TAG or t == tag:
                got = (t, payload)
            else:
                st.unexpected[source].append((t, payload))
    if got is None:
        # ANY_SOURCE: first look at what already arrived, then take whoever sends next
        for q in range(comm.size):
            got = _match(st.unexpected[q], tag)
            if got is not None:
                src = q
                break
        while got is None:
            hdr = torch.empty(_HDR_WORDS, dtype=torch.int64)
            g = dist.recv(hdr, src=None, group=comm._group)
            q = comm._ranks.index(g)
            payload = torch.empty(int(hdr[1]), dtype=torch.uint8)
            if payload.numel() > 0:
                dist.recv(payload, src=g, group=comm._group)
            if tag == ANY_TAG or int(hdr[0]) == tag:
                got, src = (int(hdr[0]), payload), q
            else:
                st.unexpected[q].append((int(hdr[0]), payload))
    t, payload = got
    return src, t, payload


def recv(comm: Comm, template: torch.Tensor, source: int, tag: int,
         status: Optional[Status]) -> torch.Tensor:
    src, t, payload = recv_bytes(comm, source, tag)
    want = template.numel() * template.element_size()
    if payload.numel() != want:
        # same rule as the GPU transport (csrc/b2_p2p.cu: B2_ERR_TRUNCATE): the template fixes the message
        # size.  (MPI would accept a shorter message; the reference never relies on that, and a
        # transport-dependent answer is worse than a strict one.)
        raise RuntimeError(
            f"message size mismatch: received {payload.numel()} bytes into a {want}-byte buffer "
            "(send and recv must agree on the size, docs/sharp-bits.md)")
    out = torch.empty(template.shape, dtype=template.dtype)
    out.reshape(-1).view(torch.uint8)[:] = payload
    if status is not None:
        status._set(src, t, payload.numel(), template.element_size())
    return out


def send_object(comm: Comm, obj, dest: int, tag: int) -> None:
    """Pickle-based message (mpi4py's lower-case ``comm.send``)."""
    import pickle

    send(comm, torch.frombuffer(bytearray(pickle.dumps(obj)), dtype=torch.uint8), dest, tag)


def recv_object(comm: Comm, source: int, tag: int, status: Optional[Status]):
    import pickle

    src, t, payload = recv_bytes(comm, source, tag)
    if status is not None:
        status._set(src, t, payload.numel(), 1)
    return pickle.loads(payload.numpy().tobytes())


def sendrecv(comm: Comm, sendbuf: torch.Tensor, recv_template: torch.Tensor, source: int,
             dest: int, sendtag: int, recvtag: int, status: Optional[Status]) -> torch.Tensor:
    send(comm, sendbuf, dest, sendtag)         # eager -> cannot deadlock against the recv
    return recv(comm, recv_template, source, recvtag, status)


def log_call(rank: int, opname: str, details: str):
    """Debug trace with the reference's line format (mpi_ops_common.h:154-206)."""
    import random
    import string

    ident = "".join(random.choices(string.ascii_letters + string.digits, k=8))
    prefix = f"r{rank} | {ident} | MPI_{opname}"
    print(f"{prefix} {details}".rstrip(), flush=True)
    t0 = time.perf_counter()

    def done(code: int = 0):
        print(f"{prefix} done with code {code} ({time.perf_counter() - t0:.2e}s)", flush=True)

    return done
