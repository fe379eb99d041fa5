"""Port of /root/reference/tests/collective_ops/test_barrier.py."""

import time

import torch

import mpi4jax_b200 as m
from mpi4jax_b200 import MPI

comm = MPI.COMM_WORLD


def _path_of_rank0(path):
    """rank 0's file name -> all ranks (uint8 bcast through the public op)."""
    buf = torch.zeros(4096, dtype=torch.uint8)
    if comm.Get_rank() == 0:
        raw = str(path).encode()
        buf[: len(raw)] = torch.tensor(list(raw), dtype=torch.uint8)
    buf = m.bcast(buf.to(comm.device), 0, comm=comm).cpu()
    return bytes(buf[buf != 0].tolist()).decode()


def test_barrier(device, tmp_path):
    """Ranks append lines before/after a barrier to one file; all 'start' lines must precede
    all 'done' lines."""
    rank, size = comm.Get_rank(), comm.Get_size()
    # a file of this run's own (a fixed name in the shared temp directory may belong to another user)
    write_to = _path_of_rank0(tmp_path / f"barrier-{device.type}.txt")
    if rank == 0:
        with open(write_to, "w"):
            pass
    comm.Barrier()
    time.sleep(rank * 0.2)
    with open(write_to, "a") as f:
        f.write(f"r{rank} | start\n")
    m.barrier()
    m.flush()       # the barrier is stream-ordered; flush makes it a host rendezvous
    with open(write_to, "a") as f:
        f.write(f"r{rank} | done\n")
    time.sleep(0.2)
    m.barrier()
    m.flush()
    comm.Barrier()
    with open(write_to) as f:
        outputs = f.readlines()
    assert len(outputs) == size * 2
    assert all(o.endswith("start\n") for o in outputs[:size])
    assert all(o.endswith("done\n") for o in outputs[size:])


def test_barrier_jit(device):
    def f(x):
        m.barrier()
        y = x + 1
        m.barrier()
        return y

    fj = m.jit(f)
    x = torch.zeros(3, device=device)
    for _ in range(3):
        assert torch.equal(fj(x), x + 1)
