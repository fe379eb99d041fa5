"""reduce_scatter (MPI_Reduce_scatter_block): rank r receives op over all ranks q of x_q[r].

Every rank builds every rank's input from a generator seeded by (seed, q), so the exact expected
result is computed locally by folding in rank order in the accumulate type (fp32 for f16 / bf16),
as the kernels do."""

import re

import numpy as np
import pytest
import torch
from torch.func import grad, jvp, vjp, vmap

import mpi4jax_b200 as m
from mpi4jax_b200 import MPI
from mpi4jax_b200._src.backends import host_staged
from mpi4jax_b200._src.native import codes

comm = MPI.COMM_WORLD
rank = comm.Get_rank()
size = comm.Get_size()

FLOATS = (torch.float32, torch.float64, torch.float16, torch.bfloat16)
INTS = (torch.int8, torch.int16, torch.int32, torch.int64, torch.uint8, torch.uint16, torch.uint32, torch.uint64)
ARITH = ("SUM", "PROD", "MIN", "MAX")
LOGICAL = ("LAND", "LOR", "LXOR", "BAND", "BOR", "BXOR")
VALID = ([(dt, op) for dt in FLOATS for op in ARITH] + [(dt, op) for dt in INTS for op in ARITH + LOGICAL]
         + [(torch.bool, op) for op in ARITH + LOGICAL]
         + [(dt, op) for dt in (torch.complex64, torch.complex128) for op in ("SUM", "PROD")])


def make_input(q, shape, dtype, seed=0):
    """Rank q's input of shape (size, *shape), identical wherever it is built."""
    g = torch.Generator().manual_seed(1000 * seed + q)
    full = (size, *shape)
    if dtype == torch.bool:
        return torch.randint(0, 2, full, generator=g).bool()
    if dtype.is_complex:
        return torch.complex(torch.randn(full, generator=g), torch.randn(full, generator=g)).to(dtype)
    if dtype.is_floating_point:
        return torch.randn(full, generator=g).to(dtype)
    return torch.randint(0, 4, full, generator=g).to(dtype)


def _np_apply(opname, a, b):
    if opname in ("LAND", "LOR", "LXOR"):
        f = {"LAND": np.logical_and, "LOR": np.logical_or, "LXOR": np.logical_xor}[opname]
        return f(a != 0, b != 0).astype(a.dtype)
    return {"SUM": np.add, "PROD": np.multiply, "MIN": np.minimum, "MAX": np.maximum, "BAND": np.bitwise_and,
            "BOR": np.bitwise_or, "BXOR": np.bitwise_xor}[opname](a, b).astype(a.dtype)


def expected(shape, dtype, opname, seed=0, block=None):
    """Fold block `block` (default: this rank's) of every rank's input in rank order."""
    block = rank if block is None else block
    parts = [make_input(q, shape, dtype, seed)[block] for q in range(size)]
    if size == 1:
        return parts[0]
    if dtype == torch.bool:
        bool_op = {"SUM": "LOR", "MAX": "LOR", "BOR": "LOR", "PROD": "LAND", "MIN": "LAND", "BAND": "LAND",
                   "BXOR": "LXOR"}.get(opname, opname)
        acc = parts[0].numpy()
        for p in parts[1:]:
            acc = _np_apply(bool_op, acc.astype(np.uint8), p.numpy().astype(np.uint8)).astype(bool)
        return torch.from_numpy(acc)
    if dtype.is_floating_point or dtype.is_complex:
        acc_dt = torch.float32 if dtype in (torch.float16, torch.bfloat16) else dtype
        acc = parts[0].to(acc_dt)
        for p in parts[1:]:
            p = p.to(acc_dt)
            if opname == "SUM":
                acc = acc + p
            elif opname == "PROD":
                acc = acc * p
            elif opname == "MIN":
                acc = torch.where((p < acc) | torch.isnan(p), p, acc)
            else:
                acc = torch.where((p > acc) | torch.isnan(p), p, acc)
        return acc.to(dtype)
    acc = parts[0].numpy()
    for p in parts[1:]:
        acc = _np_apply(opname, acc, p.numpy())
    return torch.from_numpy(acc)


def _cpu_unsupported(device, dtype, opname):
    # torch has no CPU add / min / max kernels for uint16 / uint32 / uint64 (the gloo backend reduces with torch)
    return (device.type == "cpu" and size > 1 and dtype in (torch.uint16, torch.uint32, torch.uint64)
            and opname in ("SUM", "MIN", "MAX"))


def test_reduce_scatter(device):
    x = make_input(rank, (3, 2), torch.float32).to(device)
    _x = x.clone()
    res = m.reduce_scatter(x, MPI.SUM)
    assert res.shape == (3, 2) and res.dtype == torch.float32 and res.device == x.device
    assert torch.equal(res.cpu(), expected((3, 2), torch.float32, "SUM"))
    assert torch.equal(x, _x)


def test_reduce_scatter_scalar_blocks(device):
    x = torch.arange(size, dtype=torch.int64, device=device) * 10 + rank      # x_q[r] = 10 r + q
    res = m.reduce_scatter(x, MPI.SUM)
    assert res.shape == ()
    assert res.item() == 10 * rank * size + sum(range(size))


def test_reduce_scatter_single_rank(device):
    """P = 1: a copy of x[0] on every transport that exists at one rank."""
    solo = comm.Split(rank, 0)
    try:
        x = torch.randn(1, 5, 3, device=device)
        for algorithm in ("auto", "oneshot", "ll"):
            res = m.reduce_scatter(x, MPI.SUM, comm=solo, algorithm=algorithm)
            assert torch.equal(res, x[0])
            assert res.data_ptr() != x.data_ptr()
        assert torch.equal(m.reduce_scatter(x.to(torch.int32), MPI.MAX, comm=solo), x[0].to(torch.int32))
    finally:
        m.flush()
        solo.Free()


def test_reduce_scatter_shape_errors(device):
    with pytest.raises(ValueError, match=re.escape("Reduce_scatter input must have shape (nproc, ...)")):
        m.reduce_scatter(torch.ones(size + 1, 2, device=device), MPI.SUM)
    with pytest.raises(ValueError, match=re.escape("Reduce_scatter input must have shape (nproc, ...)")):
        m.reduce_scatter(torch.tensor(1.0, device=device), MPI.SUM)
    with pytest.raises(ValueError, match="algorithm"):
        m.reduce_scatter(torch.ones(size, 2, device=device), MPI.SUM, algorithm="twoshot")


@pytest.mark.parametrize("dtype,opname", VALID, ids=[f"{str(d)[6:]}-{o}" for d, o in VALID])
def test_reduce_scatter_ops_dtypes(device, dtype, opname):
    if _cpu_unsupported(device, dtype, opname):
        pytest.skip("torch has no CPU kernel for this unsigned dtype / op")
    x = make_input(rank, (7,), dtype, seed=1).to(device)
    res = m.reduce_scatter(x, getattr(MPI, opname))
    assert res.dtype == dtype and res.shape == (7,)
    want = expected((7,), dtype, opname, seed=1)
    if dtype.is_complex and opname == "PROD":      # the device may contract the complex product into FMAs
        torch.testing.assert_close(res.cpu(), want, rtol=1e-5, atol=1e-5)
    else:
        assert torch.equal(res.cpu(), want)


def test_reduce_scatter_invalid_op_dtype(device):
    if device.type == "cpu" and size == 1:
        pytest.skip("the CPU backend passes a single contribution through unchecked, as for allreduce")
    with pytest.raises(NotImplementedError):
        m.reduce_scatter(torch.ones(size, 4, device=device), MPI.BAND)
    with pytest.raises(NotImplementedError):
        m.reduce_scatter(torch.ones(size, 4, dtype=torch.complex64, device=device), MPI.MAX)


@pytest.mark.parametrize("dtype,shape", [(torch.float16, (3,)), (torch.int8, (5,)), (torch.float32, (1, 3)),
                                         (torch.bfloat16, (1000, 7)), (torch.int32, (4099,))])
def test_reduce_scatter_odd_block_sizes(device, dtype, shape):
    """Blocks that are not a multiple of 16 bytes: every block after the first starts unaligned."""
    x = make_input(rank, shape, dtype, seed=2).to(device)
    for algorithm in ("auto", "oneshot", "ll"):
        res = m.reduce_scatter(x, MPI.SUM, algorithm=algorithm)
        assert torch.equal(res.cpu(), expected(shape, dtype, "SUM", seed=2)), algorithm


@pytest.mark.gpu
@pytest.mark.parametrize("mib", [4, 64])
def test_reduce_scatter_large(mib):
    """Blocks that span many chunks and CTAs (every transport that applies)."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    dev = comm.device
    n = (mib << 20) // 4 // size                       # mib MiB of float32 input per rank
    base = torch.arange(n, dtype=torch.float32, device=dev) % 1024
    x = torch.stack([base * (q + 1) + rank for q in range(size)])      # x_r[q] = (q + 1) * base + r
    want = base * (rank + 1) * size + sum(range(size))
    algos = ["auto", "oneshot"] + (["nvls"] if size > 2 and comm._native_comm().has_nvls else [])
    for algorithm in algos:
        assert torch.equal(m.reduce_scatter(x, MPI.SUM, algorithm=algorithm), want), algorithm
    xi = x.to(torch.int32)
    assert torch.equal(m.reduce_scatter(xi, MPI.MAX), (base * (rank + 1) + size - 1).to(torch.int32))


@pytest.mark.parametrize("algorithm", ["ll", "oneshot"])
@pytest.mark.parametrize("dtype,opname", [(torch.float32, "SUM"), (torch.bfloat16, "SUM"), (torch.float16, "PROD"),
                                          (torch.int32, "MAX"), (torch.float64, "MIN")])
def test_reduce_scatter_matches_allreduce(device, algorithm, dtype, opname):
    """Both fold in rank order: bitwise equal to block `rank` of an allreduce on the same transport."""
    shape = (3, 333)
    x = make_input(rank, shape, dtype, seed=3).to(device)
    op = getattr(MPI, opname)
    res = m.reduce_scatter(x, op, algorithm=algorithm)
    ref = m.allreduce(x, op, algorithm=algorithm)[rank]
    assert torch.equal(res, ref)
    assert torch.equal(res.cpu(), expected(shape, dtype, opname, seed=3))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_reduce_scatter_nvls(device, dtype):
    if device.type == "cuda" and (size < 3 or not comm._native_comm().has_nvls):
        pytest.skip("the in-switch transport needs NVLS multicast and more than 2 ranks")
    shape = (64, 1024)
    x = make_input(rank, shape, dtype, seed=4).to(device)
    res = m.reduce_scatter(x, MPI.SUM, algorithm="nvls")
    tol = {torch.float32: 1e-5, torch.bfloat16: 1e-2, torch.float16: 2e-3}[dtype]
    ref = m.allreduce(x, MPI.SUM, algorithm="nvls")[rank]
    torch.testing.assert_close(res.float(), ref.float(), rtol=tol, atol=tol)
    torch.testing.assert_close(res.cpu().float(), expected(shape, dtype, "SUM", seed=4).float(), rtol=tol, atol=tol)


@pytest.mark.gpu
def test_reduce_scatter_invalid_transport_is_an_error(monkeypatch):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    monkeypatch.setenv("MPI4JAX_B200_ABORT_ON_ERROR", "0")
    dev = comm.device
    with pytest.raises(MPI.MPIError, match="NVLS"):
        m.reduce_scatter(torch.ones(size, 4096, device=dev), MPI.MAX, algorithm="nvls")
    with pytest.raises(MPI.MPIError, match="LL algorithm"):
        m.reduce_scatter(torch.ones(size, 1 << 20, device=dev), MPI.SUM, algorithm="ll")
    x = torch.ones(size, 8, device=dev)              # the communicator still works afterwards
    assert torch.equal(m.reduce_scatter(x, MPI.SUM), torch.full((8,), float(size), device=dev))


def test_reduce_scatter_user_defined_op(device):
    """MPI.Op.Create: a non-commutative 2x2 matrix product, folded in rank order."""
    matmul = MPI.Op.Create(lambda a, b: a @ b, commute=False)
    # x_q[r] = shear by (q + 1) * (r + 1)
    x = torch.stack([torch.tensor([[1.0, float((rank + 1) * (r + 1))], [0.0, 1.0]]) for r in range(size)])
    res = m.reduce_scatter(x.to(device), matmul)
    want = torch.tensor([[1.0, float((rank + 1) * size * (size + 1) // 2)], [0.0, 1.0]])
    assert torch.equal(res.cpu(), want)
    # non-commutative: a rotation by 90 degrees from every rank, a shear from rank q; rank order matters
    rot = torch.tensor([[0.0, -1.0], [1.0, 0.0]])
    mats = [torch.tensor([[1.0, float(q + 1)], [0.0, 1.0]]) @ rot for q in range(size)]
    want = mats[0]
    for q in range(1, size):
        want = want @ mats[q]
    y = torch.stack([mats[rank]] * size).to(device)
    assert torch.equal(m.reduce_scatter(y, matmul).cpu(), want)


def test_reduce_scatter_jit(device):
    shape = (5, 17)
    f = m.jit(lambda t: m.reduce_scatter(t, MPI.SUM))
    x = make_input(rank, shape, torch.float32).to(device)
    for seed in range(3):  # eager warm-up, capture, replay -- new data every call
        x.copy_(make_input(rank, shape, torch.float32, seed=seed))
        assert torch.equal(f(x).cpu(), expected(shape, torch.float32, "SUM", seed=seed))


def test_reduce_scatter_jit_alternating_with_allreduce(device):
    """One graph that alternates reduce_scatter and allreduce on the LL path: the two share the LL
    buffers and the ticket parity."""
    shape = (64,)

    def body(t):
        outs = []
        for k in range(4):
            outs.append(m.reduce_scatter(t + k, MPI.SUM, algorithm="ll"))
            outs.append(m.allreduce(t + k, MPI.SUM, algorithm="ll"))
        return outs

    f = m.jit(body)
    x = make_input(rank, shape, torch.float32).to(device).round()
    for seed in range(3):
        x.copy_(make_input(rank, shape, torch.float32, seed=seed).round())
        outs = f(x)
        total = sum(make_input(q, shape, torch.float32, seed=seed).round() for q in range(size))
        for k in range(4):
            assert torch.equal(outs[2 * k].cpu(), total[rank] + k * size), (seed, k)
            assert torch.equal(outs[2 * k + 1].cpu(), total + k * size), (seed, k)


def test_reduce_scatter_grad(device):
    x = make_input(rank, (4,), torch.float64).to(device)
    w = torch.arange(4, dtype=torch.float64, device=device) + rank

    def loss(t):
        return (m.reduce_scatter(t, MPI.SUM) * w).sum()

    g = grad(loss)(x)
    want = m.allgather(w)            # d loss_q / d x_r[q] = w_q: the VJP is the allgather of the cotangent
    assert torch.equal(g, want)
    xr = x.clone().requires_grad_(True)
    loss(xr).backward()
    assert torch.equal(xr.grad, want)


def test_reduce_scatter_vjp_jvp(device):
    x = make_input(rank, (2, 3), torch.float32).to(device)
    ct = torch.full((2, 3), float(rank + 1), device=device)
    res, pullback = vjp(lambda t: m.reduce_scatter(t, MPI.SUM), x)
    assert torch.equal(res, m.reduce_scatter(x, MPI.SUM))
    (g,) = pullback(ct)
    assert torch.equal(g, m.allgather(ct))
    tan = make_input(rank, (2, 3), torch.float32, seed=7).to(device)
    res, t_out = jvp(lambda t: m.reduce_scatter(t, MPI.SUM), (x,), (tan,))
    assert torch.equal(res, m.reduce_scatter(x, MPI.SUM))
    assert torch.equal(t_out, m.reduce_scatter(tan, MPI.SUM))


def test_reduce_scatter_non_sum_grad_raises(device):
    x = torch.ones(size, 3, device=device, requires_grad=True)
    y = m.reduce_scatter(x, MPI.MAX)
    with pytest.raises(NotImplementedError):
        y.sum().backward()
    with pytest.raises(NotImplementedError):
        jvp(lambda t: m.reduce_scatter(t, MPI.MIN), (x.detach(),), (x.detach(),))


def test_reduce_scatter_vmap(device):
    batch = torch.stack([make_input(rank, (3,), torch.float32, seed=s) for s in range(4)]).to(device)  # (B, P, 3)
    res = vmap(lambda t: m.reduce_scatter(t, MPI.SUM))(batch)
    assert res.shape == (4, 3)
    for s in range(4):
        assert torch.equal(res[s].cpu(), expected((3,), torch.float32, "SUM", seed=s))
    res2 = vmap(lambda t: m.reduce_scatter(t, MPI.SUM), in_dims=1)(batch.movedim(0, 1))
    assert torch.equal(res2, res)


def test_compiled_reduce_scatter_and_grad(device):
    from mpi4jax_b200 import compiled as mc

    w = torch.arange(3, dtype=torch.float32, device=device) + rank
    f = torch.compile(lambda t: (mc.reduce_scatter(t * 2, MPI.SUM, comm=comm) * w).sum(),
                      backend="aot_eager", fullgraph=True)
    x = make_input(rank, (3,), torch.float32).to(device).round().requires_grad_(True)
    y = f(x)
    assert torch.equal(y.detach(), (2 * m.reduce_scatter(x.detach(), MPI.SUM) * w).sum())
    y.backward()
    assert torch.equal(x.grad, 2 * m.allgather(w))
    assert mc.reduce_scatter(torch.empty(size, 4, 5, device=device), MPI.SUM, comm=comm).shape == (4, 5)


def test_reduce_scatter_host_staged(device, monkeypatch):
    monkeypatch.setattr(host_staged, "ACTIVE", host_staged.ACTIVE)      # restore the flag afterwards
    hs = host_staged.HostStagedComm(comm.Clone(), "unit test")
    try:
        x = make_input(rank, (6,), torch.float32, seed=5).to(device)
        res = hs.reduce_scatter(x, codes.SUM)
        assert res.device == x.device
        assert torch.equal(res.cpu(), expected((6,), torch.float32, "SUM", seed=5))
        b = make_input(rank, (5,), torch.bool, seed=5).to(device)
        assert torch.equal(hs.reduce_scatter(b, codes.LXOR).cpu(), expected((5,), torch.bool, "LXOR", seed=5))
    finally:
        hs.comm.Free()


def test_reduce_scatter_debug_log(capsys, device):
    from mpi4jax_b200._src.native import set_logging

    x = torch.ones(size, 4, device=device)
    m.reduce_scatter(x, MPI.SUM)
    m.flush()
    capsys.readouterr()
    set_logging(True)
    try:
        res = m.reduce_scatter(x, MPI.SUM)
        m.flush()
    finally:
        set_logging(False)
    out = capsys.readouterr().out
    assert re.search(rf"r{rank} \| \w{{8}} \| MPI_Reduce_scatter_block( \(\w+\))? with 4 items per rank", out), out
    assert re.search(rf"r{rank} \| \w{{8}} \| MPI_Reduce_scatter_block( \(\w+\))? done with code 0", out), out
    assert torch.equal(res, torch.full((4,), float(size), device=device))
