"""Device-timed sweeps for the BASELINE.json collective configs:

* allreduce 1 KB - 1 GB, fp32 + bf16, every transport (ll / oneshot / twoshot / nvls / auto)
  next to NCCL on the same box                                   (configs 2)
* reduce_scatter 1 KB - 1 GB input per rank, fp32 SUM, every transport (ll / oneshot / nvls / auto)
  next to NCCL reduce_scatter_tensor; the allreduce fp32 rows at the same size are the cost of the
  allreduce + slice workaround
* allgather and alltoall 1 KB - 1 GB per-rank payload vs NCCL     (config 4)
* bcast, reduce, gather, scatter (root = last rank) vs NCCL, scan (no NCCL counterpart)
* sendrecv ring, halo exchange latency

Timing: ``reps`` back-to-back ops captured in ONE CUDA graph, one replay timed with CUDA
events on the launching stream (barrier + synchronize before), max over ranks -- i.e. the
kernels' time, not the Python launch path.  Bus bandwidth uses the NCCL-tests conventions:
allreduce S/t*2(P-1)/P, allgather/alltoall/reduce_scatter (P-1)/P * total/t.

    python -m mpi4jax_b200.run -n 8 bench/collectives_sweep.py [--max-bytes 1073741824] [--out f.json]
"""

import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ.setdefault("MPI4JAX_B200_ABORT_ON_ERROR", "0")

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import mpi4jax_b200 as m  # noqa: E402
from mpi4jax_b200 import MPI  # noqa: E402
from mpi4jax_b200.utils import max_over_ranks  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--max-bytes", type=int, default=1 << 30)
ap.add_argument("--out", default="gpurun_out/collectives_sweep.json")
ap.add_argument("--quick", action="store_true", help="every fourth size")
ap.add_argument("--skip-allreduce-algos", action="store_true", help="time only the automatic choice")
ap.add_argument("--only-allreduce", action="store_true", help="stop after the allreduce tables")
ap.add_argument("--only-reduce-scatter", action="store_true",
                help="only the fp32 allreduce table and the reduce_scatter table")
ap.add_argument("--only-p2p", action="store_true", help="only the p2p ring, barrier and halo lines")
ap.add_argument("--max-blocks", type=int, default=0, help="override the collective grid cap")
ap.add_argument("--nvls-pipeline", type=int, default=-1, help="0 / 1: software pipelining of the NVLS allreduce")
ap.add_argument("--min-bytes", type=int, default=1 << 10)
ns = ap.parse_args()

comm = MPI.COMM_WORLD
rank, size = comm.Get_rank(), comm.Get_size()
dev = comm.device
nccl = None
try:
    nccl = dist.new_group(backend="nccl")
    t = torch.ones(8, device=dev)
    dist.all_reduce(t, group=nccl)
    torch.cuda.synchronize()
except Exception as exc:  # pragma: no cover
    if rank == 0:
        print("NCCL comparison unavailable:", exc)
    nccl = None
nc = comm._native_comm()
has_nvls = nc.has_nvls
if ns.max_blocks:
    nc.set_tuning(max_blocks=ns.max_blocks)
if ns.nvls_pipeline >= 0:
    nc.set_option("nvls_pipeline", ns.nvls_pipeline)


def reps_for(nbytes):
    return 50 if nbytes <= (1 << 16) else 20 if nbytes <= (1 << 22) else 5 if nbytes <= (1 << 27) else 3


def time_graph(fn, reps):
    """fn() enqueues ONE op; returns us per op (device time, max over ranks)."""
    fn()
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side), torch.cuda.graph(g, stream=side, capture_error_mode="thread_local"):
        for _ in range(reps):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    g.replay()
    torch.cuda.synchronize()
    best = None
    for _ in range(3):
        comm.Barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        g.replay()
        e.record()
        e.synchronize()
        us = s.elapsed_time(e) * 1e3 / reps
        best = us if best is None else min(best, us)
    del g
    return max_over_ranks(best, comm)


def time_eager(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    best = None
    for _ in range(3):
        comm.Barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(reps):
            fn()
        e.record()
        e.synchronize()
        us = s.elapsed_time(e) * 1e3 / reps
        best = us if best is None else min(best, us)
    return max_over_ranks(best, comm)


def time_nccl(fn, reps):
    try:
        return time_graph(fn, reps)
    except Exception:
        torch.cuda.synchronize()
        return time_eager(fn, max(reps, 10))


sizes = [] if ns.only_p2p else [1 << k for k in range(10, 31, 2 if ns.quick else 1) if ns.min_bytes <= (1 << k) <= ns.max_bytes]
result = {"world": size, "nvls": has_nvls, "allreduce": {}, "allgather": {}, "alltoall": {}, "p2p": {}}
# what the numbers were measured on: the card and its power limit, read in the same run
result["gpu"] = torch.cuda.get_device_name(dev) if dev.type == "cuda" else "cpu"
try:
    import subprocess

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30)
    result["nvidia_smi_name_power_limit_max_sm_clock"] = q.stdout.strip().splitlines() or q.stderr.strip()[:120]
except Exception as exc:  # pragma: no cover
    result["nvidia_smi_name_power_limit_max_sm_clock"] = f"unavailable: {exc}"[:120]

# ---------------------------------------------------------------- allreduce
sym_pool = None
if sizes and size > 1 and dev.type == "cuda":
    sym_pool = m.symmetric_empty((max(sizes),), torch.uint8, comm=comm)
for dtype, dname in ((torch.float32, "fp32"),) + (() if ns.only_reduce_scatter else ((torch.bfloat16, "bf16"),)):
    table = {}
    for nbytes in sizes:
        x = torch.ones(nbytes // torch.empty((), dtype=dtype).element_size(), dtype=dtype, device=dev)
        row = {}
        reps = reps_for(nbytes)
        for algo in (("auto",) if ns.skip_allreduce_algos else ("auto", "ll", "oneshot", "twoshot", "nvls")):
            if algo == "ll" and nbytes > (64 << 10):
                continue
            if algo == "nvls" and not has_nvls:
                continue
            if algo == "oneshot" and size > 2 and nbytes > (1 << 27):
                continue
            try:
                us = time_graph(lambda: m.allreduce(x, MPI.SUM, comm=comm, algorithm=algo), reps)
                row[algo] = {"us": round(us, 2), "busbw": round(nbytes / us / 1e3 * 2 * (size - 1) / size, 1)}
            except Exception as exc:
                row[algo] = {"error": str(exc)[:120]}
        if nccl is not None:
            us = time_nccl(lambda: dist.all_reduce(x, group=nccl), reps)
            row["nccl"] = {"us": round(us, 2), "busbw": round(nbytes / us / 1e3 * 2 * (size - 1) / size, 1)}
        if sym_pool is not None and has_nvls and nbytes >= 16:
            # the same reduction on a SYMMETRIC tensor, in place (no staging copies): mpi4jax_b200.allreduce_
            xs = sym_pool[: nbytes].view(dtype)
            xs.fill_(1)
            try:
                us = time_graph(lambda: m.allreduce_(xs, comm=comm), reps)
                row["sym"] = {"us": round(us, 2), "busbw": round(nbytes / us / 1e3 * 2 * (size - 1) / size, 1)}
            except Exception as exc:
                row["sym"] = {"error": str(exc)[:120]}
        table[str(nbytes)] = row
        if rank == 0:
            print(dname, nbytes, {k: (v.get("us"), v.get("busbw")) for k, v in row.items()}, flush=True)
        del x
    result["allreduce"][dname] = table

# ---------------------------------------------------------------- reduce_scatter (input per rank = nbytes)
result["reduce_scatter"] = {}
for nbytes in ([] if ns.only_allreduce else sizes):
    if nbytes < 4 * size:
        continue
    blk = nbytes // 4 // size
    x = torch.ones(size, blk, device=dev)
    tot = x.numel() * 4
    reps = reps_for(nbytes)
    row = {}
    for algo in ("auto", "ll", "oneshot", "nvls"):
        if algo == "ll" and 2 * blk * 4 > (128 << 10):
            continue
        if algo == "nvls" and not has_nvls:
            continue
        try:
            us = time_graph(lambda: m.reduce_scatter(x, MPI.SUM, comm=comm, algorithm=algo), reps)
            row[algo] = {"us": round(us, 2), "busbw": round(tot * (size - 1) / size / us / 1e3, 1)}
        except Exception as exc:
            row[algo] = {"error": str(exc)[:120]}
    if nccl is not None:
        out = torch.empty(blk, device=dev)
        flat = x.reshape(-1)
        us = time_nccl(lambda: dist.reduce_scatter_tensor(out, flat, group=nccl), reps)
        row["nccl"] = {"us": round(us, 2), "busbw": round(tot * (size - 1) / size / us / 1e3, 1)}
        del out, flat
    result["reduce_scatter"][str(nbytes)] = row
    if rank == 0:
        print("reduce_scatter", nbytes, {k: (v.get("us"), v.get("busbw")) for k, v in row.items()}, flush=True)
    del x

if ns.only_allreduce or ns.only_reduce_scatter:
    if rank == 0:
        os.makedirs(os.path.dirname(ns.out) or ".", exist_ok=True)
        with open(ns.out, "w") as f:
            json.dump(result, f, indent=1)
    m.flush()
    sys.exit(0)

# ---------------------------------------------------------------- allgather / alltoall (per-rank payload = nbytes)
for nbytes in sizes:
    if nbytes * size > (8 << 30):
        continue
    reps = reps_for(nbytes * size // 2)
    x = torch.ones(nbytes // 4, device=dev)
    row = {}
    us = time_graph(lambda: m.allgather(x, comm=comm), reps)
    row["ours"] = {"us": round(us, 2), "busbw": round(nbytes * (size - 1) / us / 1e3, 1)}
    if nccl is not None:
        out = torch.empty(size * x.numel(), device=dev)
        us = time_nccl(lambda: dist.all_gather_into_tensor(out, x, group=nccl), reps)
        row["nccl"] = {"us": round(us, 2), "busbw": round(nbytes * (size - 1) / us / 1e3, 1)}
        del out
    result["allgather"][str(nbytes)] = row
    if nbytes >= size * 4:
        y = torch.ones(size, nbytes // 4 // size, device=dev)        # total payload = nbytes per rank
        tot = y.numel() * 4
        row2 = {}
        us = time_graph(lambda: m.alltoall(y, comm=comm), reps)
        row2["ours"] = {"us": round(us, 2), "busbw": round(tot * (size - 1) / size / us / 1e3, 1)}
        if nccl is not None:
            out = torch.empty_like(y)
            us = time_nccl(lambda: dist.all_to_all_single(out, y, group=nccl), reps)
            row2["nccl"] = {"us": round(us, 2), "busbw": round(tot * (size - 1) / size / us / 1e3, 1)}
            del out
        result["alltoall"][str(nbytes)] = row2
        del y
    if rank == 0:
        print("allgather/alltoall", nbytes, row, result["alltoall"].get(str(nbytes)), flush=True)
    del x

# ---------------------------------------------------------------- rooted ops + scan (per-rank payload = nbytes)
result.update({"bcast": {}, "reduce": {}, "gather": {}, "scatter": {}, "scan": {}})
root = size - 1
for nbytes in [b for b in sizes if b >= 1 << 10][::1 if ns.quick else 2]:
    reps = reps_for(nbytes)
    x = torch.ones(nbytes // 4, device=dev)
    rows = {k: {} for k in ("bcast", "reduce", "scan")}
    us = time_graph(lambda: m.bcast(x, root, comm=comm), reps)
    rows["bcast"]["ours"] = {"us": round(us, 2), "gbs": round(nbytes / us / 1e3, 1)}
    us = time_graph(lambda: m.reduce(x, MPI.SUM, root, comm=comm), reps)
    rows["reduce"]["ours"] = {"us": round(us, 2), "gbs": round(nbytes / us / 1e3, 1)}
    us = time_graph(lambda: m.scan(x, MPI.SUM, comm=comm), reps)
    rows["scan"]["ours"] = {"us": round(us, 2), "gbs": round(nbytes / us / 1e3, 1)}
    if nccl is not None:
        y = x.clone()
        us = time_nccl(lambda: dist.broadcast(y, src=root, group=nccl), reps)
        rows["bcast"]["nccl"] = {"us": round(us, 2), "gbs": round(nbytes / us / 1e3, 1)}
        us = time_nccl(lambda: dist.reduce(y, dst=root, group=nccl), reps)
        rows["reduce"]["nccl"] = {"us": round(us, 2), "gbs": round(nbytes / us / 1e3, 1)}
        del y
    for k in rows:
        result[k][str(nbytes)] = rows[k]
    if nbytes * size <= (2 << 30):
        rows2 = {"gather": {}, "scatter": {}}
        us = time_graph(lambda: m.gather(x, root, comm=comm), reps)
        rows2["gather"]["ours"] = {"us": round(us, 2), "gbs": round(nbytes * (size - 1) / us / 1e3, 1)}
        big = torch.ones(size, nbytes // 4, device=dev) if rank == root else x
        us = time_graph(lambda: m.scatter(big, root, comm=comm), reps)
        rows2["scatter"]["ours"] = {"us": round(us, 2), "gbs": round(nbytes * (size - 1) / us / 1e3, 1)}
        if nccl is not None:
            try:
                outs = [torch.empty_like(x) for _ in range(size)] if rank == root else None
                us = time_eager(lambda: dist.gather(x, outs, dst=root, group=nccl), max(reps, 5))
                rows2["gather"]["nccl"] = {"us": round(us, 2), "gbs": round(nbytes * (size - 1) / us / 1e3, 1)}
                ins = [torch.ones_like(x) for _ in range(size)] if rank == root else None
                y = torch.empty_like(x)
                us = time_eager(lambda: dist.scatter(y, ins, src=root, group=nccl), max(reps, 5))
                rows2["scatter"]["nccl"] = {"us": round(us, 2), "gbs": round(nbytes * (size - 1) / us / 1e3, 1)}
                del outs, ins, y
            except Exception as exc:  # pragma: no cover
                rows2["gather"]["nccl"] = {"error": str(exc)[:100]}
        for k in rows2:
            result[k][str(nbytes)] = rows2[k]
        del big
    if rank == 0:
        print("rooted", nbytes, {k: v for k, v in rows.items()}, {k: result[k].get(str(nbytes)) for k in ("gather", "scatter")},
              flush=True)
    del x

# ---------------------------------------------------------------- p2p ring + halo
for nbytes in (8, 4096, 1 << 16, 1 << 20, 1 << 24, 1 << 28):
    x = torch.ones(max(nbytes // 4, 1), device=dev)
    us = time_graph(lambda: m.sendrecv(x, x, source=(rank - 1) % size, dest=(rank + 1) % size, comm=comm),
                    reps_for(nbytes))
    result["p2p"][str(nbytes)] = {"us": round(us, 2), "gbs": round(nbytes / us / 1e3, 1)}
us = time_graph(lambda: m.barrier(comm=comm), 50)
result["barrier_us"] = round(us, 2)
if size in (1, 2, 4, 6, 8, 16):
    from mpi4jax_b200.models import ShallowWaterConfig, ShallowWaterModel

    mod = ShallowWaterModel(ShallowWaterConfig.for_resolution(4096, 4096), comm=comm, device=dev)
    for nf in (2, 4):
        fields = [mod.fe, mod.fn, mod.q, mod.ke][:nf]
        kinds = ["u", "v", "h", "h"][:nf]
        us = time_graph(lambda: mod.enforce_boundaries(fields, kinds), 50)
        result[f"halo{nf}_us"] = round(us, 2)
if rank == 0:
    print("p2p", result["p2p"], "barrier", result["barrier_us"], "halo", result.get("halo2_us"), result.get("halo4_us"))
    os.makedirs(os.path.dirname(ns.out) or ".", exist_ok=True)
    with open(ns.out, "w") as f:
        json.dump(result, f, indent=1)
m.flush()
