"""Headline benchmark (driver contract): shallow-water steps/s on a 4096x4096 grid.

BASELINE.json metric: "allreduce bus GB/s vs message size and shallow_water.py steps/sec
(whole box, device-timed, max over ranks) at 1/2/4/8 B200".  ``value`` is the shallow-water
throughput (defined for every N, including N=1); the allreduce bus-bandwidth sweep (N>1)
is reported in the extra key ``allreduce_busbw_gbs``.

    python bench.py --gpus N --steps K --warmup W            # N=1 directly
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   # N>1
    python bench.py --impl reference                          # reference arm
    python bench.py ... --dump-outputs DIR                    # + the state after the last timed step, DIR/*.npy

* device-timed with CUDA events on the launching stream, barrier + synchronize on both
  sides, max over ranks; W untimed warm-up steps, exactly K timed steps;
* strong scaling: the global 4096x4096 grid is fixed, ranks split it 2 x (N/2);
* the timed region launches only this repo's kernels (5 fused stencil + 4 fused halo
  exchange kernels per model step, replayed from a CUDA graph);
* ``e2e``: the same K steps through the public API, in chunks of ``e2e_chunk_steps`` model
  steps (the reference's ``do_multistep(state, 100)`` call granularity); every chunk copies
  the model state host->device from pinned memory and reads the surface-height snapshot back
  device->host, timed by the wall clock between barriers.
"""

from __future__ import annotations

import argparse
import json
import math
import os
import sys
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

GRID = 4096
# published reference numbers (BASELINE.md): 3600x1800 grid on Tesla P100, derived steps/s
BASELINE_STEPS_PER_S = {1: 80.0, 2: 129.0}


def reference_arm() -> int:
    """The unmodified reference cannot be installed offline: it needs mpicc, mpi4py,
    nanobind and jax at build time (see DESIGN.md, 'Reference arm')."""
    why = ("mpi4jax cannot be installed offline in this image: pip --no-index fails on "
           "mpi4py>=3.0.1 (not in /opt/wheelhouse); with --no-deps setup.py raises 'Building "
           "mpi4jax requires mpi4py and nanobind'; jax, mpicc and an MPI library are absent too")
    try:
        sys.path.insert(0, os.path.join(REPO, "baseline", "_ref"))
        import mpi4jax  # noqa: F401

        why = "baseline/_ref/mpi4jax imports, but no MPI launcher / jax runtime exists to run it"
    except Exception:
        pass
    if int(os.environ.get("RANK", "0")) == 0:          # one line per job, also under torchrun
        print(json.dumps({"impl": "reference", "unavailable": why}))
    return 0


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--grid", type=int, default=GRID)
    ap.add_argument("--no-sweep", action="store_true", help="skip the allreduce sweep extras")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the model state after the last timed step to DIR/<field>.npy (see dump_outputs)")
    ns = ap.parse_args()
    if ns.steps < 1:
        ap.error("--steps must be at least 1")
    if ns.impl == "reference":
        return reference_arm()

    world = int(os.environ.get("WORLD_SIZE", "1"))
    if ns.gpus > 1 and world == 1:
        # convenience: `python bench.py --gpus N` without torchrun -> launch the ranks ourselves
        from mpi4jax_b200.run import launch

        code, _ = launch(ns.gpus, [os.path.abspath(__file__), *sys.argv[1:]])
        return code

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        print(json.dumps({"metric": "shallow_water_steps_per_sec", "value": None,
                          "error": "no CUDA device"}))
        return 1
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank % torch.cuda.device_count())
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("cpu:gloo,cuda:nccl")

    import mpi4jax_b200 as m
    from mpi4jax_b200 import MPI
    from mpi4jax_b200._src import native
    from mpi4jax_b200.models import ShallowWaterConfig, ShallowWaterModel
    from mpi4jax_b200.utils import ClockSampler, flush_l2, max_over_ranks

    comm = MPI.COMM_WORLD
    rank, size = comm.Get_rank(), comm.Get_size()
    K, W = ns.steps, max(ns.warmup, 3)
    dev = comm.device

    # ---- correctness on THIS job's ranks before anything is timed --------------------------------
    checks = correctness_checks(m, MPI, comm, dev)

    model = ShallowWaterModel(ShallowWaterConfig.for_resolution(ns.grid, ns.grid), comm=comm, device=dev,
                              backend="native")
    model.step(first_step=True)

    # ---- CUDA graphs: chunk of C steps (+ remainder) -------------------------------------
    C = min(50, K)
    graphs = {}

    def graph_for(n):
        if n not in graphs:
            fn = m.jit(lambda: model.multistep(n, first_step=False), warmup=0)
            before = native.launch_count()
            fn()                                    # capture (+ one replay)
            graphs[n] = (fn, native.launch_count() - before)
        return graphs[n]

    def run_steps(n_total):
        launches = 0
        full, rem = divmod(n_total, C)
        for _ in range(full):
            fn, per = graph_for(C)
            fn()
            launches += per
        if rem:
            fn, per = graph_for(rem)
            fn()
            launches += per
        return launches

    graph_for(C)
    if K % C:
        graph_for(K % C)
    run_steps(W)                                    # untimed warm-up steps
    model.reset()
    model.step(first_step=True)
    run_steps(W)
    run_steps(K)                                    # the exact replay sequence of the timed region, once untimed

    # ---- device-timed region: exactly K steps ---------------------------------------------
    flush_l2(dev)
    torch.cuda.synchronize()
    comm.Barrier()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(gpu_index=torch.cuda.current_device(), period_s=0.005, first_delay_s=0.003) as clocks:
        torch.cuda.synchronize()
        # The timed window is K steps ON THE DEVICE.  A short spin kernel first: while the GPU sits in it
        # the host enqueues everything below (barrier kernel, start event, the graph launches), so what
        # runs between the two events is the replayed steps and not this process' Python / launch
        # latency (measured before: 20 steps at 8 GPUs took 817 us in the window, 32 us per step in the
        # device timeline -- the rest was the host getting from `start.record()` to `cudaGraphLaunch`
        # while eight `nvidia-smi` clock queries started next to it; the clocks are now read through
        # in-process NVML, and the end-to-end number below accounts for launch latency separately).
        torch.cuda._sleep(int(4e7))                 # ~20 ms at 1.9 GHz: also covers a descheduled rank process
        # device-side barrier on the stream right before the start event: the ranks' timed windows
        # open together on the GPUs, whatever skew the host-side barrier left between the processes
        m.barrier(comm=comm)
        start.record()
        gpu_launches = run_steps(K)
        end.record()
        torch.cuda.synchronize()
        # the state the timed steps left, before the untimed steps below advance it
        timed_state = [t.clone() for t in model.state] if ns.dump_outputs else None
        if start.elapsed_time(end) < 400:           # keep the GPU under load long enough to sample
            t_end = time.time() + 0.5
            while time.time() < t_end:
                run_steps(C)
            torch.cuda.synchronize()
    comm.Barrier()
    ms = max_over_ranks(start.elapsed_time(end), comm)
    steps_per_s = K / (ms * 1e-3)
    nproc_y, nproc_x, ny_local, nx_local, pipeline = (model.nproc_y, model.nproc_x, model.ny_local, model.nx_local,
                                                      model.pipeline)
    finite = bool(torch.isfinite(model.h).all().item())
    mass = model.total_mass().item()
    checks["finite"] = finite
    checks["total_mass"] = mass

    # ---- end to end through the public API: the reference's solve loop -------------------------
    # (examples/shallow_water.py:414-463) with the initial condition in pinned HOST memory: upload
    # it, first (Euler) step, then K - 1 steps in `do_multistep` chunks; after every chunk the
    # surface-height snapshot is copied to the host and read there.  Wall clock between barriers.
    chunk = min(100, max(1, K - 1))
    model.reset()
    torch.cuda.synchronize()
    host_ic = [t.detach().cpu().pin_memory() for t in (model.h, model.u, model.v)]
    host_h = torch.empty_like(host_ic[0]).pin_memory()
    h2d = sum(t.numel() * t.element_size() for t in host_ic)
    d2h = host_h.numel() * host_h.element_size()
    step_chunk, _ = graph_for(chunk)
    tail = (K - 1) % chunk
    step_tail = graph_for(tail)[0] if tail else None

    def e2e_run():
        model.load_initial_condition(*host_ic)      # pinned host -> device: h, u, v (+ frame storage, collective)
        model.step(first_step=True)
        nsnap = 0
        for fn in [step_chunk] * ((K - 1) // chunk) + ([step_tail] if tail else []):
            fn()                                    # public API: jit(model.multistep)(chunk)
            host_h.copy_(model.h, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            _ = float(host_h[1, 1])                 # the host consumes the snapshot
            nsnap += 1
        if nsnap == 0:
            host_h.copy_(model.h, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            nsnap = 1
        return nsnap

    e2e_run()
    torch.cuda.synchronize()
    comm.Barrier()
    t0 = time.perf_counter()
    nsnap = e2e_run()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    comm.Barrier()
    e2e_s = max_over_ranks(t1 - t0, comm)
    e2e_value = K / e2e_s

    # ---- extras: the reference-style USER program (BASELINE config 3) --------------------------
    # the same discrete system written with torch arithmetic and the PUBLIC sendrecv / send / recv
    # ops in the reference's message order (models/shallow_water.py, backend="ops"), under jit
    ops_rate = None
    try:
        ops_model = ShallowWaterModel(ShallowWaterConfig.for_resolution(ns.grid, ns.grid), comm=comm, device=dev,
                                      backend="ops")
        ops_model.step(first_step=True)
        n_ops = 5
        ops_fn = m.jit(lambda: ops_model.multistep(n_ops, first_step=False), warmup=1)
        ops_fn()
        ops_fn()
        torch.cuda.synchronize()
        comm.Barrier()
        s0, e0 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        m.barrier(comm=comm)
        s0.record()
        ops_fn()
        ops_fn()
        e0.record()
        torch.cuda.synchronize()
        ops_ms = max_over_ranks(s0.elapsed_time(e0), comm) / (2 * n_ops)
        ops_rate = {"steps_per_s": round(1e3 / ops_ms, 1), "ms_per_step": round(ops_ms, 4),
                    "note": "backend='ops': torch stencils + public sendrecv/send/recv (48 p2p ops per step at 8 "
                            "ranks, as the reference issues them), captured by mpi4jax_b200.jit"}
        del ops_model, ops_fn
    except Exception as exc:  # pragma: no cover
        ops_rate = {"error": str(exc)[:200]}

    # ---- extras: allreduce bus bandwidth sweep (N > 1) -----------------------------------------
    sweep = None
    if size > 1 and not ns.no_sweep:
        sweep = allreduce_sweep(m, MPI, comm, dev)

    if rank == 0:
        base = BASELINE_STEPS_PER_S.get(size, BASELINE_STEPS_PER_S[2] if size > 1 else None)
        out = {
            "metric": "shallow_water_steps_per_sec",
            "value": round(steps_per_s, 2),
            "unit": "steps/s",
            "n_gpus": size,
            "steps": K,
            "warmup": W,
            "ms_per_step": round(ms / K, 5),
            "higher_is_better": True,
            "scaling": "strong",
            "vs_baseline": round(steps_per_s / base, 2) if base else None,
            "dtype": "fp32",
            "data": "synthetic (the reference's analytic jet initial condition)",
            "impl": "ours",
            "config": {
                "model": "examples/shallow_water.py (non-linear shallow water, C-grid, AB2)",
                "global_batch": f"{ns.grid}x{ns.grid} grid (the demo's 1800 km x 900 km domain)",
                "seq_len": None,
                "parallelism": f"2-D domain decomposition {nproc_y}x{nproc_x}",
                "l2": ("L2 flushed before the timed region; per-rank state "
                       f"{13 * ny_local * nx_local * 4 / 2**20:.0f} MiB vs 126 MiB L2"),
                "graph_chunk_steps": C,
                "kernel_path": pipeline,
                "baseline_note": ("vs_baseline divides by the reference's published P100 numbers for "
                                  "a 3600x1800 grid (80 steps/s at n=1, 129 at n=2), this run uses "
                                  "the 2.6x larger 4096x4096 grid named in BASELINE.json"),
            },
            "gpu_launches": int(gpu_launches),
            "clocks": clocks.summary(),
            "e2e": {
                "value": round(e2e_value, 2),
                "unit": "steps/s",
                "h2d_bytes_per_step": int(h2d // K),
                "d2h_bytes_per_step": int(d2h * nsnap // K),
                "e2e_chunk_steps": chunk,
                "note": ("solve loop through the public API: initial condition (h, u, v) H2D from pinned memory once "
                         f"({h2d} B), Euler step + K-1 steps in jit(multistep) chunks, surface-height snapshot "
                         "D2H + host read after every chunk"),
            },
            "checks": checks,
        }
        out["public_ops_shallow_water"] = ops_rate
        if sweep is not None:
            out["allreduce_busbw_gbs"] = sweep
        print(json.dumps(out))
    if ns.dump_outputs:
        dump_outputs(ns.dump_outputs, model, timed_state)
    m.flush()
    return 0


DUMP_SAMPLE = 1 << 21          # values per field: 6 float32 fields of 8 MiB, 48 MiB in all
DUMP_SEED = 0


def dump_outputs(directory, model, state):
    """Write ``state`` (h, u, v, dh, du, dv: what ``model.multistep`` leaves a caller) as
    ``directory/<field>.npy`` in float32, so that two builds can be compared output for output.
    Each field is the global (ny + 2, nx + 2) array including its halo ring, gathered on rank 0.
    A field of more than DUMP_SAMPLE values is written as the values at DUMP_SAMPLE sorted flat
    indices drawn without replacement by numpy's default_rng(DUMP_SEED): the same indices for
    every run on the same grid, whatever the number of GPUs."""
    import numpy as np

    index = None
    for name, local in zip(model.state._fields, state):
        field = model.gather_global(local)          # collective: every rank takes part
        if field is None:
            continue
        arr = field.float().cpu().numpy()
        if arr.size > DUMP_SAMPLE:
            if index is None:
                index = np.sort(np.random.default_rng(DUMP_SEED).choice(arr.size, DUMP_SAMPLE, replace=False))
            arr = arr.reshape(-1)[index]
        os.makedirs(directory, exist_ok=True)
        np.save(os.path.join(directory, f"{name}.npy"), arr)


def correctness_checks(m, MPI, comm, dev):
    """Every native transport on this job's ranks against closed-form / fp32 torch results, and the
    shallow-water kernels against the public-ops (torch + sendrecv) implementation of the same
    discrete system.  Returns {name: max abs error (0.0 = exact)}; raises nothing -- the numbers
    are reported under ``checks`` and ``checks_ok``."""
    import torch

    from mpi4jax_b200._src.native import codes
    from mpi4jax_b200.models import ShallowWaterConfig, ShallowWaterModel

    rank, size = comm.Get_rank(), comm.Get_size()
    out = {}

    def err(got, want):
        return float((got.double() - want.double()).abs().max().item())

    tot = size * (size - 1) / 2
    x = torch.arange(1 << 16, device=dev, dtype=torch.float32) % 251 + rank
    base = torch.arange(1 << 16, device=dev, dtype=torch.float32) % 251
    if size > 1:
        nc = comm._native_comm()
        algos = [("ll", codes.ALGO_LL, 1 << 12), ("oneshot", codes.ALGO_ONESHOT, 1 << 16),
                 ("twoshot", codes.ALGO_TWOSHOT, 1 << 16)]
        if nc.has_nvls:
            algos.append(("nvls", codes.ALGO_NVLS, 1 << 16))
        for name, algo, n in algos:
            got = nc.allreduce(x[:n], codes.SUM, algo)
            out[f"allreduce_{name}_f32"] = err(got, base[:n] * size + tot)
        xb = (torch.arange(1 << 16, device=dev) % 7 + rank).to(torch.bfloat16)
        want = ((torch.arange(1 << 16, device=dev) % 7).float() * size + tot)
        out["allreduce_auto_bf16"] = err(m.allreduce(xb, MPI.SUM, comm=comm).float(), want.to(torch.bfloat16).float())
    out["allreduce_auto_f32"] = err(m.allreduce(x, MPI.SUM, comm=comm), base * size + tot)
    out["allreduce_max_i32"] = err(m.allreduce(torch.full((1000,), rank, device=dev, dtype=torch.int32), MPI.MAX,
                                               comm=comm), torch.full((1000,), size - 1, device=dev))
    small = torch.arange(4096, device=dev, dtype=torch.float32) + 1000.0 * rank
    ag = m.allgather(small, comm=comm)
    out["allgather"] = max(err(ag[q], small - 1000.0 * rank + 1000.0 * q) for q in range(size))
    a2a_in = torch.stack([small + 7.0 * q for q in range(size)])
    a2a = m.alltoall(a2a_in, comm=comm)
    out["alltoall"] = max(err(a2a[q], small - 1000.0 * rank + 1000.0 * q + 7.0 * rank) for q in range(size))
    for root in sorted({0, size - 1}):
        b = m.bcast(small if rank == root else torch.empty_like(small), root, comm=comm)
        out[f"bcast_root{root}"] = err(b, small - 1000.0 * rank + 1000.0 * root)
        r = m.reduce(small, MPI.SUM, root, comm=comm)
        if rank == root:
            out[f"reduce_root{root}"] = err(r, (small - 1000.0 * rank) * size + 1000.0 * tot)
        g = m.gather(small, root, comm=comm)
        if rank == root:
            out[f"gather_root{root}"] = max(err(g[q], small - 1000.0 * rank + 1000.0 * q) for q in range(size))
        sc = m.scatter(a2a_in if rank == root else torch.empty_like(small), root, comm=comm)
        out[f"scatter_root{root}"] = err(sc, small - 1000.0 * rank + 1000.0 * root + 7.0 * rank)
    sc = m.scan(small, MPI.SUM, comm=comm)
    out["scan"] = err(sc, (small - 1000.0 * rank) * (rank + 1) + 1000.0 * rank * (rank + 1) / 2)
    nxt, prv = (rank + 1) % size, (rank - 1) % size
    ring = m.sendrecv(small, torch.empty_like(small), source=prv, dest=nxt, comm=comm)
    out["sendrecv_ring"] = err(ring, small - 1000.0 * rank + 1000.0 * prv)
    big = torch.arange(1 << 22, device=dev, dtype=torch.float32) + rank
    ring = m.sendrecv(big, torch.empty_like(big), source=prv, dest=nxt, sendtag=3, recvtag=3, comm=comm)
    out["sendrecv_ring_16MiB"] = err(ring, big - rank + prv)
    m.barrier(comm=comm)
    # rooted results exist on one rank only: share the worst value (public allreduce, MAX)
    keys = sorted(set(k for k in out) | {f"{op}_root{r}" for op in ("reduce", "gather") for r in {0, size - 1}})
    vec = torch.tensor([out.get(k, 0.0) for k in keys], device=dev, dtype=torch.float64)
    vec = m.allreduce(vec, MPI.MAX, comm=comm)
    out = {k: float(v) for k, v in zip(keys, vec.tolist())}

    # shallow water: native kernels (communication-avoiding schedule and the stand-alone kernels)
    # vs the model written with the public ops, 10 steps on a small grid of this decomposition
    cfg = ShallowWaterConfig(nx=96 * max(1, size // 2), ny=64)
    ops = ShallowWaterModel(cfg, comm=comm, device=dev, backend="ops")
    ops.multistep(10)
    for pipe in ("ca", "standalone"):
        nat = ShallowWaterModel(cfg, comm=comm, device=dev, backend="native", pipeline=pipe)
        nat.multistep(10)
        worst = 0.0
        for name, a, b in zip(nat.state._fields, nat.state, ops.state):
            scale = b.abs().max().item() + 1e-30
            worst = max(worst, (a - b).abs().max().item() / scale / (2e-4 if name in "huv" else 2e-3))
        worst = float(m.allreduce(torch.tensor(worst, device=dev, dtype=torch.float64), MPI.MAX, comm=comm).item())
        out[f"swe_{pipe}_vs_ops_rel_to_tol"] = worst          # < 1: within tests/test_examples.py's tolerances
    ca = ShallowWaterModel(cfg, comm=comm, device=dev, backend="native", pipeline="ca")
    sa = ShallowWaterModel(cfg, comm=comm, device=dev, backend="native", pipeline="standalone")
    ca.multistep(10)
    sa.multistep(10)
    same = all(torch.equal(a, b) for a, b in zip(ca.state, sa.state))
    same = bool(m.allreduce(torch.tensor(int(same), device=dev), MPI.MIN, comm=comm).item())
    out["swe_ca_bitwise_equals_standalone"] = same
    exact = [k for k in out if k.startswith(("allreduce", "allgather", "alltoall", "bcast", "reduce", "gather",
                                              "scatter", "scan", "sendrecv"))]
    out["checks_ok"] = bool(all(out[k] == 0.0 for k in exact) and same
                            and out["swe_ca_vs_ops_rel_to_tol"] < 1 and out["swe_standalone_vs_ops_rel_to_tol"] < 1)
    m.flush()
    return out


def allreduce_sweep(m, MPI, comm, dev):
    """Device-timed allreduce bus bandwidth (GB/s), fp32 and bf16, CUDA-graph replays so the
    number is the kernels' and not the Python launch path's; max over ranks."""
    import torch

    from mpi4jax_b200.utils import max_over_ranks

    size = comm.Get_size()
    res = {}
    for dtype, name in ((torch.float32, "fp32"), (torch.bfloat16, "bf16")):
        row = {}
        for nbytes in (1 << 10, 1 << 14, 1 << 17, 1 << 20, 1 << 23, 1 << 26, 1 << 28, 1 << 30):
            x = torch.ones(nbytes // x_size(dtype), dtype=dtype, device=dev)
            reps = 20 if nbytes <= (1 << 23) else 5
            f = m.jit(lambda t: [m.allreduce(t, MPI.SUM, comm=comm) for _ in range(reps)][-1],
                      warmup=1, donate_outputs=True, static_inputs=True)
            f(x)
            f(x)
            torch.cuda.synchronize()
            comm.Barrier()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            f(x)
            e.record()
            e.synchronize()
            us = max_over_ranks(s.elapsed_time(e), comm) * 1e3 / reps
            row[str(nbytes)] = {"us": round(us, 2),
                                "busbw": round(nbytes / us / 1e3 * 2 * (size - 1) / size, 1)}
            del f, x
        res[name] = row
    # the same reduction on SYMMETRIC tensors, in place (mpi4jax_b200.symmetric_empty / allreduce_): no
    # staging copies around the in-switch reduction
    if size > 1 and comm._native_comm().has_nvls:
        pool = m.symmetric_empty((1 << 30,), torch.uint8, comm=comm)
        row = {}
        for nbytes in (1 << 10, 1 << 14, 1 << 17, 1 << 20, 1 << 23, 1 << 26, 1 << 28, 1 << 30):
            x = pool[:nbytes].view(torch.float32)
            x.fill_(1.0)
            reps = 20 if nbytes <= (1 << 23) else 5

            def body(t, reps=reps):
                for _ in range(reps):
                    m.allreduce_(t, comm=comm)
                return t

            f = m.jit(body, warmup=1, donate_outputs=True, static_inputs=True)
            f(x)
            f(x)
            x.fill_(1.0)
            torch.cuda.synchronize()
            comm.Barrier()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            f(x)
            e.record()
            e.synchronize()
            us = max_over_ranks(s.elapsed_time(e), comm) * 1e3 / reps
            row[str(nbytes)] = {"us": round(us, 2),
                                "busbw": round(nbytes / us / 1e3 * 2 * (size - 1) / size, 1)}
            del f
        res["fp32_symmetric_inplace"] = row
    return res


def x_size(dtype):
    import torch

    return torch.empty((), dtype=dtype).element_size()


if __name__ == "__main__":
    sys.exit(main())
