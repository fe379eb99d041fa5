"""Capabilities beyond the reference's rule set that round 1's review asked for: adjoints of the
rooted ops and scan (the reference raises for them), user-defined reduction operators
(``MPI.Op.Create``; the reference forwards any ``MPI.Op`` handle, allreduce.py:104), ``PROC_NULL``
peers, communicator duplication on sub-communicators, staging reservation."""

import pytest
import torch

import mpi4jax_b200 as m
from mpi4jax_b200 import MPI

comm = MPI.COMM_WORLD
rank, size = comm.Get_rank(), comm.Get_size()


def _leaf(device, *shape):
    return (torch.arange(float(torch.Size(shape).numel()), device=device).reshape(shape) + rank).requires_grad_()


@pytest.mark.parametrize("root", sorted({0, size - 1}))
def test_reduce_vjp_is_a_broadcast_from_the_root(device, root):
    x = _leaf(device, 3, 2)
    w = torch.arange(6.0, device=device).reshape(3, 2) + 1
    out = m.reduce(x, MPI.SUM, root, comm=comm)
    loss = (out * w).sum() if rank == root else (out * 0.5).sum()      # non-root: out is x itself
    loss.backward()
    want = w if rank == root else w + 0.5
    assert torch.equal(x.grad, want)


def test_scan_vjp_is_the_suffix_sum(device):
    x = _leaf(device, 4)
    w = torch.full((4,), float(rank + 1), device=device)
    (m.scan(x, MPI.SUM, comm=comm) * w).sum().backward()
    want = sum(float(q + 1) for q in range(rank, size))       # ranks r .. P-1 see x_r with unit weight
    assert torch.allclose(x.grad, torch.full((4,), want, device=device))


@pytest.mark.parametrize("root", sorted({0, size - 1}))
def test_gather_and_scatter_are_adjoint(device, root):
    x = _leaf(device, 2, 3)
    out = m.gather(x, root, comm=comm)
    if rank == root:
        w = torch.arange(float(size * 6), device=device).reshape(size, 2, 3)
        (out * w).sum().backward()
        assert torch.equal(x.grad, w[rank])
    else:
        (out * 2.0).sum().backward()            # the root's cotangent block for this rank + own pass-through
        w = torch.arange(float(size * 6), device=device).reshape(size, 2, 3)
        assert torch.equal(x.grad, w[rank] + 2.0)
    # scatter: the root's input gradient stacks every rank's cotangent
    src = (torch.arange(float(size * 4), device=device).reshape(size, 4)).requires_grad_() if rank == root else \
        torch.empty(4, device=device).requires_grad_()
    blk = m.scatter(src, root, comm=comm)
    (blk * float(rank + 1)).sum().backward()
    if rank == root:
        want = torch.stack([torch.full((4,), float(q + 1), device=device) for q in range(size)])
        assert torch.equal(src.grad, want)
    else:
        assert torch.equal(src.grad, torch.zeros(4, device=device))


def test_non_sum_rules_still_raise(device):
    x = _leaf(device, 3)
    with pytest.raises(NotImplementedError):
        m.reduce(x, MPI.MAX, 0, comm=comm)
    with pytest.raises(NotImplementedError):
        m.scan(x, MPI.PROD, comm=comm)


def test_plain_send_of_a_tensor_that_requires_grad_raises(device):
    x = _leaf(device, 3)
    with pytest.raises(NotImplementedError, match="send_with_grad"):
        m.send(x, rank, comm=comm)
    m.send(x.detach(), rank, tag=5, comm=comm)       # explicit detach is the sanctioned way
    got = m.recv(torch.empty(3, device=device), rank, tag=5, comm=comm)
    assert torch.equal(got, x.detach())


def test_user_defined_operator(device):
    """MPI.Op.Create: a non-commutative 2x2 matrix product, folded in rank order on every rank."""
    matmul = MPI.Op.Create(lambda a, b: a @ b, commute=False)
    assert not matmul.Is_commutative()
    x = torch.tensor([[1.0, float(rank + 1)], [0.0, 1.0]], device=device)        # shear by rank + 1
    want_all = torch.tensor([[1.0, float(size * (size + 1) // 2)], [0.0, 1.0]], device=device)
    assert torch.equal(m.allreduce(x, matmul, comm=comm), want_all)
    want_scan = torch.tensor([[1.0, float((rank + 1) * (rank + 2) // 2)], [0.0, 1.0]], device=device)
    assert torch.equal(m.scan(x, matmul, comm=comm), want_scan)
    got = m.reduce(x, matmul, size - 1, comm=comm)
    assert torch.equal(got, want_all if rank == size - 1 else x)
    hypot = MPI.Op.Create(lambda a, b: torch.sqrt(a * a + b * b))
    v = torch.tensor([3.0, 0.0], device=device)
    assert torch.allclose(m.allreduce(v, hypot, comm=comm), torch.tensor([3.0 * size ** 0.5, 0.0], device=device))
    assert comm.allreduce(3, op=MPI.Op.Create(lambda a, b: a * b)) == 3 ** size      # object API, too


def test_proc_null_peers_are_no_ops(device):
    x = torch.full((5,), float(rank), device=device)
    m.send(x, MPI.PROC_NULL, comm=comm)
    st = MPI.Status()
    keep = torch.full((5,), -7.0, device=device)
    got = m.recv(keep, MPI.PROC_NULL, comm=comm, status=st)
    assert torch.equal(got, keep) and st.Get_source() == MPI.PROC_NULL and st.Get_count() == 0
    # open chain: the ends talk to PROC_NULL on one side (the boundary idiom of MPI stencil codes)
    up = rank + 1 if rank + 1 < size else MPI.PROC_NULL
    down = rank - 1 if rank > 0 else MPI.PROC_NULL
    got = m.sendrecv(x, keep, source=down, dest=up, comm=comm)
    assert torch.equal(got, keep if rank == 0 else torch.full((5,), float(rank - 1), device=device))


def test_dup_and_split_on_a_sub_communicator_do_not_involve_other_ranks(device):
    """Clone / Split on a sub-communicator are collective over ITS members only; the default
    communicator (a lazy world clone) still works afterwards."""
    sub = comm.Split(rank // 2, rank)
    if rank < 2:                                   # only the first pair duplicates / re-splits
        dup = sub.Clone()
        again = dup.Split(0, -dup.Get_rank())      # reversed order inside the pair
        got = m.allreduce(torch.ones(3, device=device), MPI.SUM, comm=again)
        assert torch.equal(got, torch.full((3,), float(sub.Get_size()), device=device))
        assert again.Get_rank() == sub.Get_size() - 1 - sub.Get_rank()
        # key order, not launch order, numbers the ranks: order-sensitive results follow it
        mine = torch.tensor([float(again.Get_rank())], device=device)
        assert torch.equal(m.allgather(mine, comm=again)[:, 0], torch.arange(float(again.Get_size()), device=device))
        assert again.allgather(again.Get_rank()) == list(range(again.Get_size()))
        again.Free()
        dup.Free()
    total = m.allreduce(torch.ones(2, device=device), MPI.SUM)          # default comm: every rank
    assert torch.equal(total, torch.full((2,), float(size), device=device))
    sub.Free()


def test_comm_reserve(device):
    m.comm_reserve(1 << 20, comm=comm)
    x = torch.ones(1 << 18, device=device)
    assert torch.equal(m.allreduce(x, MPI.SUM, comm=comm), x * size)


def test_strided_inputs_are_packed_by_the_collective_itself(device):
    """Non-contiguous inputs (transposes, slices) of the data-movement collectives: on CUDA the
    strides go to the native kernel, which gathers while it stages (no ``.contiguous()`` copy
    kernel in front, cf. the reference's regression tests/collective_ops/test_alltoall.py:43-65)."""
    base = torch.arange(float(size * 6 * 10), device=device).reshape(size, 6, 10) + 1000.0 * rank
    views = {
        "transposed": base.transpose(1, 2),                 # (size, 10, 6), inner stride 10
        "sliced": base[:, ::2, 1:9:3],                      # (size, 3, 3)
        "lead_stride": base.transpose(0, 1)[:size] if size <= 6 else base,     # block stride != block size
    }
    for name, x in views.items():
        assert x.shape[0] == size
        want = x.contiguous()
        got = m.alltoall(x, comm=comm)
        ref = m.alltoall(want, comm=comm)
        assert torch.equal(got, ref), ("alltoall", name)
        assert torch.equal(m.allgather(x[0], comm=comm), m.allgather(want[0], comm=comm)), ("allgather", name)
        root = size - 1
        g, gr = m.gather(x[0], root, comm=comm), m.gather(want[0], root, comm=comm)
        assert torch.equal(g, gr) or rank != root, ("gather", name)
        sc = m.scatter(x if rank == root else torch.empty_like(want[0]), root, comm=comm)
        scr = m.scatter(want if rank == root else torch.empty_like(want[0]), root, comm=comm)
        assert torch.equal(sc, scr), ("scatter", name)
    for dtype in (torch.uint8, torch.bfloat16, torch.float64, torch.complex128):
        t = (torch.arange(size * 8 * 4, device=device).reshape(size, 8, 4) % 13 + rank).to(dtype).transpose(1, 2)
        assert torch.equal(m.alltoall(t, comm=comm), m.alltoall(t.contiguous(), comm=comm)), dtype


@pytest.mark.parametrize("nbytes", [1 << 12, 3 << 20])
def test_large_rooted_ops_and_scan(device, nbytes):
    """Sizes on both sides of the switch-over to the multicast paths (bcast by multimem.st, reduce by
    multimem.ld_reduce on the root, two-phase scan) -- closed-form results, root = last rank."""
    n = nbytes // 4
    base = (torch.arange(n, device=device) % 97).float()
    x = base + rank
    root = size - 1
    b = m.bcast(x if rank == root else torch.empty_like(x), root, comm=comm)
    assert torch.equal(b, base + root)
    r = m.reduce(x, MPI.SUM, root, comm=comm)
    assert torch.equal(r, base * size + size * (size - 1) / 2 if rank == root else x)
    s = m.scan(x, MPI.SUM, comm=comm)
    assert torch.equal(s, base * (rank + 1) + rank * (rank + 1) / 2)
    s = m.scan((x % 5).to(torch.int32), MPI.MAX, comm=comm)
    want = torch.stack([((base + q) % 5).to(torch.int32) for q in range(rank + 1)]).max(0).values
    assert torch.equal(s, want)
    xb = (torch.arange(n, device=device) % 7 + rank).to(torch.bfloat16)
    rb = m.reduce(xb, MPI.SUM, 0, comm=comm)
    if rank == 0:
        assert torch.equal(rb.float(), (torch.arange(n, device=device) % 7).float() * size + size * (size - 1) / 2)


@pytest.fixture
def comm_on_device(device, monkeypatch):
    """COMM_WORLD, or for the CPU case on a machine with a GPU a clone of it that lives on the CPU
    (symmetric_empty allocates on its communicator's device)."""
    if device.type == comm.device.type:
        yield comm
        return
    monkeypatch.setenv("MPI4JAX_B200_DEVICE", "cpu")
    cpu_comm = comm.Clone()
    yield cpu_comm
    cpu_comm.Free()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("n", [4, 1000, 70_000, (1 << 20) + 8])
def test_symmetric_tensor_allreduce_in_place(device, comm_on_device, dtype, n):
    """Extension: tensors allocated in the symmetric heap are reduced in place inside the NVSwitch
    (no staging copy in, none out).  The reference has no registered-memory notion to compare with;
    the oracle is the functional allreduce of the same values."""
    comm2 = comm_on_device
    x = m.symmetric_empty((n,), dtype, comm=comm2)
    vals = (torch.arange(n, device=device, dtype=torch.float32) % 13 + rank).to(dtype)
    x.copy_(vals)
    want = m.allreduce(vals, MPI.SUM, comm=comm2)
    if device.type == "cuda" and size > 1 and (n * x.element_size()) % 16:
        with pytest.raises(Exception, match="16"):
            m.allreduce_(x, comm=comm2)
        m.flush()
        return
    out = m.allreduce_(x, comm=comm2)
    assert out.data_ptr() == x.data_ptr()
    assert torch.equal(out, want)
    # a contiguous, 16-byte aligned view is fine too; twice in a row reuses the barrier epochs
    if n >= 1000:
        view = x[8: 8 + 64]
        before = view.clone()
        m.allreduce_(view, comm=comm2)
        assert torch.equal(view.float(), before.float() * size)
    with pytest.raises(NotImplementedError):
        m.allreduce_(x, MPI.MAX, comm=comm2)


def test_allreduce_inplace_rejects_ordinary_cuda_tensors(device):
    if device.type != "cuda" or size == 1:
        pytest.skip("only the GPU transport distinguishes symmetric memory (and only with peers)")
    with pytest.raises(ValueError, match="symmetric_empty"):
        m.allreduce_(torch.ones(64, device=device), comm=comm)

